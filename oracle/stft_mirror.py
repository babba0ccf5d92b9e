"""Float64 mirror of the STFT / ISTFT kernels (csrc/stft.cu), with an error bound per output.  Oracle: test infrastructure only.

``stft_f64`` is the rfft of ``x * hann`` (float64 window, zeros past ``x_len``) of every frame of a ragged batch, framed the
way ``stft_kernel`` frames it; ``istft_f64`` is ``sum_j w * irfft(m X)_j`` over the frames that cover a sample, divided by the
float32 window sum-square that librosa accumulates (``stft_np.window_sumsquare``), exactly 0 where that sum is <= FLT_MIN
and past the natural length ``1024 + 256 (N - 1)``.  ``power_f64`` is ``|X|^2`` of a complex64 spectrum (``dvae_power``).
Everything runs in torch on the tensors' device: the large references of the GPU tests are computed on the GPU.

The bounds are first-order rounding-error bounds derived from the kernels' own operations, with the second-order term as a
gamma factor ``c / (1 - c)``.  Every path from an input value to an output of a Cooley-Tukey FFT meets exactly one node per
level and carries a weight of modulus one, so an error of at most ``c u |node|`` at every node of a level adds at most
``c u sum |input|`` to every output (the element bound, relative to the frame's 1-norm), and, the levels being scaled unitary
maps, at most ``c u ||output||_2`` to the output vector (the frame bound; Higham, Accuracy and Stability of Numerical
Algorithms, section 24.1, made there for radix 2 and repeated here per radix-8 pass and for the split step).  u = 2^-24.

Operation by operation (line numbers of csrc/stft.cu):

* ``cadd`` / ``csub`` / ``cadd_mi`` / ``cadd_pi`` (97-108): one rounding per component, ``u |result|``.
* ``cmul`` (93-95), FMA-contracted as nvcc does by default: per component ``u |inner product| + u |result|``; the inner
  product is one of ``a.x b.x, a.y b.y`` (real part) and one of ``a.x b.y, a.y b.x`` (imaginary part), a vector of modulus
  ``<= |a| |b|``, so ``|cmul - ab| <= 2u |a| |b|``.
* ``fft8`` (111-125): three add levels, plus on the odd outputs ``s (o.x +- o.y)``: one add, one multiply and the rounded
  constant ``s = fl(1/sqrt 2)``.
* ``twiddle_powers`` (147-155): table values ``g_tw`` rounded from double (52) have error ``<= u``; ``w^k`` for k <= 7 is built
  by up to three chained ``cmul``: errors e1 = u, e2 = 2 e1 + 2u, e3 = e2 + e1 + 2u, e4 = 2 e2 + 2u, e5 = e4 + e1 + 2u,
  e6 = e4 + e2 + 2u, e7 = e4 + e3 + 2u = 19u; the pass's own ``cmul`` (171, 187) adds 2u.
* split step (304-325): ``W^k = W^t (cr, ci)`` (table u, constant u, ``cmul`` 2u); ``s``, ``d``, ``W^k d``, the final add.
  The 2 x 2 map ``(Z_k, conj Z_512-k) -> (X_k, conj X_512-k)`` is unitary for 0 < k < 256 and sqrt 2 times one at k = 0, so
  the FFT's error reaches X at most sqrt 2 times over.
* window (54, 289): ``fl(hann)`` and the packed multiply, 2u relative per sample.
* P (310, 314): ``fma(r.x, r.x, r.y r.y)``: 2u of ``|X_hat|^2``, plus the X error carried through, plus an absolute floor
  of 2^-148 for subnormal results (the build has no ``-ftz``).
* ISTFT (395-466): the masked product (401-403, 2u), the pre-processing ``s``, ``d``, ``conj W^k d``, ``s + i wd``, the same
  512-point FFT, the window multiply (364, 432; the 1 / 1024 is a power of two), the float32 overlap-add of up to four terms
  in ascending frame order (441), and the multiplication by ``fl(1 / wss)`` (67, 454, 460).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import stft_np

F64 = torch.float64
U = 2.0 ** -24                   # FP32 rounding, round to nearest
FLOOR = 2.0 ** -149              # the smallest subnormal: absolute error of a rounding into the subnormal range <= FLOOR / 2
N_FFT, HALF, F, HOP = 1024, 512, 513, 256
FLT_MIN = float(np.finfo(np.float32).tiny)

ADD = U                                                     # cadd / csub / cadd_mi / cadd_pi (97-108)
CMUL = 2 * U                                                # cmul with FMA contraction (93-95)
TABLE = U                                                   # g_tw[k] = (float) exp(-2 pi i k / 1024) from double (52)
SQRT_HALF = abs(float(np.float32(math.sqrt(0.5))) - math.sqrt(0.5)) / math.sqrt(0.5)  # s = 0.70710678f (112): 0.29u
CONST = U                                                   # cr / ci of the split step (319-320, 410-413)


def _powers():
    e = [0.0, TABLE]
    e.append(2 * e[1] + CMUL)                               # w^2 = w w
    e.append(e[2] + e[1] + CMUL)                            # w^3 = w^2 w
    e.append(2 * e[2] + CMUL)                               # w^4 = w^2 w^2
    e.append(e[4] + e[1] + CMUL)                            # w^5 = w^4 w
    e.append(e[4] + e[2] + CMUL)                            # w^6 = w^4 w^2
    e.append(e[4] + e[3] + CMUL)                            # w^7 = w^4 w^3
    return max(e)


W_POW = _powers()                                           # twiddle_powers (147-155): 19u
FFT8 = 3 * ADD + ADD + U + SQRT_HALF                        # fft8 (111-125), odd outputs: 3 adds, s (o.x + o.y), the product by s
TWIDDLE = CMUL + W_POW                                      # a[k] * w^k between the passes (171, 187)
FFT512 = 3 * FFT8 + 2 * TWIDDLE                             # fft512 (163-198)
WINDOW = TABLE + U                                          # fl(hann) (54) and the packed multiply (289 / 432)
W_SPLIT = TABLE + CONST + CMUL                              # W^k = W^t (cr, ci) (324 / 414)
SQ2 = math.sqrt(2.0)

# STFT, per bin and relative to the frame's sum |x w|: the window, the FFT (reaching X at most sqrt 2 times over), the split
# step's s (u |s| / 2 <= u S), d (likewise), W^k d (cmul and the twiddle, times |d| / 2 <= S) and its final add (u |X|)
C_ELEM = WINDOW + SQ2 * FFT512 + (ADD + ADD + CMUL + W_SPLIT + ADD)
# STFT, per frame and relative to ||X||_2 (>= ||Z||_2 = sqrt 512 ||x w||_2, and ||rfft e||_2 <= sqrt 1024 ||e||_2)
C_FRAME = SQ2 * (WINDOW + FFT512 + ADD + ADD + CMUL + W_SPLIT) + ADD
# ISTFT pre-processing of bin pair (k, 512 - k) (405-418): s, d (u each), conj W^k d (cmul + twiddle), s + i wd (u |zb|, |zb|
# <= 2 (|X_k| + |X_512-k|)), relative to |X_k| + |X_512-k|
PRE = ADD + ADD + CMUL + W_SPLIT + 2 * ADD
MASK = U + U                                                # mk = mask * scale, mk * X (401-403)
C_IRFFT = SQ2 * FFT512 + PRE                                # per sample of a frame, relative to sum |H| / 1024
RECIP = U + U                                               # fl(1 / wss) in the table (67), r = v * inv (454, 460)


def gamma(c):
    """First-order coefficient ``c`` (a multiple of u) -> ``c / (1 - c)``: the second-order terms included."""
    return c / (1.0 - c)


def hann(device=None):
    return torch.tensor(stft_np.hann_periodic(N_FFT), dtype=F64, device=device)


def _i64(a, device):
    return torch.as_tensor(np.asarray(a.cpu() if torch.is_tensor(a) else a, dtype=np.int64), device=device)


def frames_f64(x, x_off, x_len, fr_off, hop, n0, n1):
    """Frames n0 .. n1-1 of the batch as ``stft_kernel`` reads them: utterance u's frame i starts at sample
    ``x_off[u] + i hop`` and reads zeros at and past ``x_len[u]``; float64 ``[n1 - n0][1024]``."""
    dev = x.device
    n = torch.arange(n0, n1, device=dev, dtype=torch.int64)
    u = torch.searchsorted(fr_off[1:], n, right=True)
    s0 = (n - fr_off[u]) * hop
    q = s0[:, None] + torch.arange(N_FFT, device=dev, dtype=torch.int64)[None, :]
    live = q < x_len[u][:, None].to(torch.int64)
    idx = torch.where(live, x_off[u][:, None] + q, torch.zeros_like(q))
    return torch.where(live, x[idx].to(F64), torch.zeros((), dtype=F64, device=dev))


def stft_f64(x, x_off, x_len, fr_off, hop=HOP, chunk=8192):
    """``(X [NT][513] complex128, P [NT][513], elem [NT][513], frame [NT], p_bound [NT][513])`` of the frames ``fr_off``
    (prefix offsets, ``B + 1``) of the signals ``x[x_off[u] : x_off[u] + x_len[u]]``.

    ``elem``: ``|X_hat_k - X_k| <= gamma(C_ELEM) sum_n |x_n w_n|`` for every bin; ``frame``: ``||X_hat - X||_2 <=
    gamma(C_FRAME) ||X||_2`` for every frame; ``p_bound``: ``|P_hat - |X|^2|`` for the P the kernel derives from its X."""
    dev = x.device
    x_off, x_len, fr_off = _i64(x_off, dev), _i64(x_len, dev), _i64(fr_off, dev)
    NT = int(fr_off[-1])
    w = hann(dev)
    X = torch.empty((NT, F), dtype=torch.complex128, device=dev)
    S = torch.empty(NT, dtype=F64, device=dev)
    for n0 in range(0, NT, chunk):
        n1 = min(NT, n0 + chunk)
        v = frames_f64(x, x_off, x_len, fr_off, hop, n0, n1) * w
        X[n0:n1] = torch.fft.rfft(v, dim=1)
        S[n0:n1] = v.abs().sum(1)
    absX = X.abs()
    elem = (gamma(C_ELEM) * S + gamma(C_ELEM) * FLOOR)[:, None].expand(NT, F)
    frame = gamma(C_FRAME) * torch.linalg.vector_norm(X, dim=1) + math.sqrt(F) * gamma(C_ELEM) * FLOOR
    P = absX * absX
    return X, P, elem, frame, p_bound(absX, elem)


def p_bound(absX, e):
    """``|fma(r.x, r.x, r.y r.y) - |X|^2|`` for ``|r - X| <= e``: the X error carried through, 2u of the result, the floor."""
    return 2 * absX * e + e * e + gamma(2 * U) * (absX + e) ** 2 + 2 * FLOOR


HYPOT = 3 * 2.0 ** -23           # hypotf: 3 ulp (CUDA C++ Programming Guide, single-precision mathematical functions)


def power_f64(X):
    """``(P, bound)`` of ``dvae_power`` (nmf.cu: ``a = hypotf(x, y); P = a * a``) on a complex64 spectrum: ``|X|^2`` in
    float64 and ``(2 HYPOT + u) |X|^2`` (second order included) plus the subnormal floor."""
    a = X.to(torch.complex128).abs()
    P = a * a
    return P, ((1 + HYPOT) ** 2 * (1 + U) - 1) * P + 2 * FLOOR


_WSS = {}


def window_sumsquare32(N, device):
    """librosa's float32 window sum-square of N frames (``stft_np.window_sumsquare``) as float64 values."""
    key = (N, str(device))
    if key not in _WSS:
        _WSS[key] = torch.tensor(stft_np.window_sumsquare(N, N_FFT, HOP).astype(np.float64), device=device)
    return _WSS[key]


def istft_f64(X, fr_off, y_off, y_len, total, mask=None, mask_scale=1.0, chunk=8192):
    """``(y [total] float64, bound [total], written [total] bool)`` of ``dvae_istft_f32`` (``mask`` None) or
    ``dvae_istft_masked_f32`` on ``X [NT][ld]`` complex64 (``mask [NT][ld]`` float32, ``mask_scale`` as the kernel receives
    it, a float32).  ``written``: the samples ``y_off[u] .. y_off[u] + y_len[u] - 1`` the kernel stores; ``y`` and ``bound``
    are 0 elsewhere.  Where the bound is 0 (sample 0, past the natural length) the kernel must store exactly 0."""
    dev = X.device
    fr_off_h = np.asarray(fr_off.cpu() if torch.is_tensor(fr_off) else fr_off, np.int64)
    y_off_h = np.asarray(y_off.cpu() if torch.is_tensor(y_off) else y_off, np.int64)
    y_len_h = np.asarray(y_len.cpu() if torch.is_tensor(y_len) else y_len, np.int64)
    NT = int(fr_off_h[-1])
    w = hann(dev)
    scale = float(np.float32(mask_scale))
    frames = torch.empty((NT, N_FFT), dtype=F64, device=dev)
    e = torch.empty(NT, dtype=F64, device=dev)
    c_frame = C_IRFFT + (MASK if mask is not None else 0.0)
    for n0 in range(0, NT, chunk):
        n1 = min(NT, n0 + chunk)
        Y = X[n0:n1, :F].to(torch.complex128)
        if mask is not None:
            Y = Y * (mask[n0:n1, :F].to(F64) * scale)
        Y[:, 0] = Y[:, 0].real                                          # irfft ignores Im of DC and Nyquist
        Y[:, HALF] = Y[:, HALF].real
        a = Y.abs()
        A = a[:, 0] + a[:, HALF] + 2 * a[:, 1:HALF].sum(1)              # 1-norm of the Hermitian-extended spectrum
        frames[n0:n1] = torch.fft.irfft(Y, n=N_FFT, dim=1)
        e[n0:n1] = c_frame * A / N_FFT
    y = torch.zeros(total, dtype=F64, device=dev)
    bound = torch.zeros(total, dtype=F64, device=dev)
    written = torch.zeros(total, dtype=torch.bool, device=dev)
    g = gamma(4 * U + WINDOW + RECIP)                                   # slack for the second-order terms
    for u in range(len(y_len_h)):
        f0, N, L, o = int(fr_off_h[u]), int(fr_off_h[u + 1] - fr_off_h[u]), int(y_len_h[u]), int(y_off_h[u])
        if L <= 0:
            continue
        written[o:o + L] = True
        if N == 0:
            continue
        nat = N_FFT + HOP * (N - 1)
        fr = frames[f0:f0 + N] * w                                      # w irfft(m X)_j
        acc = torch.zeros((N + 3, HOP), dtype=F64, device=dev)
        mag = torch.zeros_like(acc)                                     # sum_j |w y_j|
        err = torch.zeros_like(acc)                                     # sum_j w e_j
        cnt = torch.zeros_like(acc)
        ew = e[f0:f0 + N, None] * w[None, :]
        for c in range(4):
            sl = slice(HOP * c, HOP * (c + 1))
            acc[c:c + N] += fr[:, sl]
            mag[c:c + N] += fr[:, sl].abs()
            err[c:c + N] += ew[:, sl]
            cnt[c:c + N] += 1
        acc, mag, err, cnt = acc.reshape(-1), mag.reshape(-1), err.reshape(-1), cnt.reshape(-1)
        wss = window_sumsquare32(N, dev)
        live = wss > FLT_MIN
        inv = torch.where(live, 1.0 / torch.where(live, wss, torch.ones_like(wss)), torch.zeros_like(wss))
        yy = acc * inv
        # per frame: irfft error times w, window rounding; the float32 overlap-add: cnt - 1 additions after the exact first one
        b = (err + WINDOW * mag + (cnt - 1) * ADD * mag) * inv
        b = (b + RECIP * yy.abs()) * (1 + g) + torch.where(live, 2 * FLOOR * inv, torch.zeros_like(inv))
        m = min(L, nat)
        y[o:o + m] = yy[:m]
        bound[o:o + m] = b[:m]
    return y, bound, written
