"""The STFT, the power spectrum and both ISTFT kernels (csrc/stft.cu, ``dvae_power``) against float64, element by element.

* ``dvae_stft_f32``: every bin inside the element bound of the float64 mirror (``oracle/stft_mirror.py``: the frame's
  ``sum |x w|`` times a constant derived from the kernel's operations), every frame inside the norm-wise bound
  ``C2 u ||X||_2``, every P inside its bound; even and odd ``x_off`` (vector and scalar loads), hops 128 / 256 / 307 / 512 /
  1024, ``ld`` 513 / 520 / 528, ``P = NULL``, zero-frame utterances and frames past the signal, and a ragged steady-state
  batch in which every CTA loops at least three times and the proportional utterance guess misses.
* ``dvae_istft_f32`` / ``dvae_istft_masked_f32``: every sample inside the mirror's bound (per-frame irfft error, the mask
  and window roundings, the float32 overlap-add, the reciprocal of the window sum-square), exactly 0 where the window
  sum-square is <= FLT_MIN and past the natural length, sentinels around every output untouched.
* Exact checks: an utterance's rows / samples do not depend on the batch around it, its offset parity, ``ld``, ``P``, the
  ISTFT's segmentation (B = 1, 7, 70, 600) or the batch order; the masked kernel equals the plain one on the mask product.

No max-normalised tolerance: a quiet frame, a quiet bin or an edge sample is held to its own bound.  The largest
error / bound ratio per (kernel, output, family) is printed at the end of the module.
"""
import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth
from dvae_b200.engine import RaggedBatch, _p, _stream
from oracle import stft_mirror as sm
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu
F = 513
SENT = -7.0
RATIOS = {}                                     # (kernel, output, family) -> largest |gpu - f64| / bound
P_REL60 = []                                    # speech: largest |P_gpu - P| / P over bins within 60 dB of their frame's peak
LENS = [768, 1023, 1024, 1025, 1279, 1280, 1281, 16000, 33333, 48000, 48001, 96000]


@pytest.fixture(scope="module", autouse=True)
def _ratio_table():
    yield
    if RATIOS:
        print("\nlargest |gpu - f64| / bound")
        for (kern, out, fam), r in sorted(RATIOS.items()):
            print("  %-14s %-6s %-10s %9.3g" % (kern, out, fam, r))
    if P_REL60:
        print("speech: largest relative error of P over bins within 60 dB of their frame's peak: %.3g" % max(P_REL60))


def _check(kern, out, fam, got, ref, bound):
    """``|got - ref| <= bound`` for every element (complex: the modulus of the difference); 0 bound means exactly equal."""
    got, ref = torch.as_tensor(got).to(DEV), torch.as_tensor(ref).to(DEV)
    dt = torch.complex128 if (got.is_complex() or ref.is_complex()) else torch.float64
    got, ref = got.to(dt), ref.to(dt)
    bound = torch.as_tensor(bound).to(DEV, torch.float64).expand(got.shape)
    err = (got - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / torch.where(bound > 0, bound, torch.full_like(bound, 1e-300)))
    ratio = torch.where(torch.isfinite(got.abs() if got.is_complex() else got), ratio, torch.full_like(ratio, np.inf))
    r = float(ratio.max()) if ratio.numel() else 0.0
    RATIOS[(kern, out, fam)] = max(RATIOS.get((kern, out, fam), 0.0), r)
    if not r <= 1.0:
        i = int(torch.argmax(ratio.reshape(-1)))
        idx = np.unravel_index(i, tuple(ratio.shape))
        pytest.fail("%s %s [%s]: |gpu - f64| / bound = %.3g at %s (gpu %r, f64 %r, bound %.3g)"
                    % (kern, out, fam, r, idx, complex(got.reshape(-1)[i]), complex(ref.reshape(-1)[i]), float(bound.reshape(-1)[i])))


# --------------------------------------------------------------------------------------------- signal families
def _speech(T, seed):
    out, pos, k = np.zeros(T, np.float32), 0, 0
    while pos < T:                                   # synth utterances at several SNRs, end to end
        x, _, _ = synth.synth_utterance(seed + k, 3.0, (-5.0, 5.0, 20.0)[k % 3])
        n = min(T - pos, len(x))
        out[pos:pos + n] = x[:n]
        pos, k = pos + n, k + 1
    if seed % 2:                                     # 16-bit PCM values k / 32768
        out = (np.clip(np.round(out * 32768.0), -32768, 32767) / 32768.0).astype(np.float32)
    return out


def _tonal(T, seed):
    n = np.arange(T)
    kind = seed % 6
    if kind == 0:
        k0 = (1, 100, 200, 255, 256, 300, 511)[seed // 6 % 7]       # bin-centred: every other bin is 0 in float64
        return np.cos(2 * np.pi * k0 * n / 1024).astype(np.float32)
    if kind == 1:
        return np.ones(T, np.float32)                                 # DC
    if kind == 2:
        return np.where(n % 2 == 0, 1.0, -1.0).astype(np.float32)     # Nyquist
    if kind == 3:
        x = np.zeros(T, np.float32)
        x[(seed * 37) % 256::256] = 1.0                               # one impulse per hop
        return x
    if kind == 4:
        return np.sin(2 * np.pi * 200.5 * n / 1024).astype(np.float32) * np.float32(0.5)
    return np.where(np.random.default_rng(seed).random(T) < 0.5, -1.0, 1.0).astype(np.float32)   # full-scale +-1 noise


def _tiny(T, seed):
    return (_speech(T, seed) * np.float32((1e-20, 3e-22, 1e-30)[seed % 3])).astype(np.float32)


def _dynamic(T, seed):
    x = _speech(T, seed)
    if seed % 2:
        x *= np.float32(1e-5)                                         # -100 dB, packed between full-scale neighbours
    elif T > 8000:
        x[:T // 2] = 0.0                                              # digital silence, then a full-scale burst whose first
        x[T // 2 + 3000:] = 0.0                                       # frames only graze it with the window tail
        x[T // 2:T // 2 + 3000] = np.where(x[T // 2:T // 2 + 3000] < 0, -1.0, 1.0)
    return x.astype(np.float32)


FAMILIES = {"speech": _speech, "tonal": _tonal, "tiny": _tiny, "dynamic": _dynamic}


def _n_frames(T, hop):
    """The shim's frame count (stft.py: end padding by one hop unless the length is a whole number of windows)."""
    q = (T / 16000) / 64e-3 / (hop / 1024)
    Tp = T + hop if np.ceil(q) != int(q) else T
    return max(0, 1 + (Tp - 1024) // hop) if Tp >= 1024 else 1


# --------------------------------------------------------------------------------------------- STFT driver
def _pack(xs, odd, gap=3):
    """Concatenate the signals with sentinel gaps; ``odd``: every offset odd (the scalar-load path), else even."""
    off, pos = [], gap
    for x in xs:
        if (pos % 2 == 1) != odd:
            pos += 1
        off.append(pos)
        pos += len(x) + gap
    flat = np.full(pos + gap, 0.25, np.float32)                      # samples past x_len must never be read as signal
    for o, x in zip(off, xs):
        flat[o:o + len(x)] = x
    return torch.from_numpy(flat).to(DEV), np.array(off, np.int64)


def _stft(flat, off, lens, nfr, hop=256, ld=520, want_p=True):
    B = len(lens)
    fr_off = np.zeros(B + 1, np.int64)
    np.cumsum(nfr, out=fr_off[1:])
    NT = int(fr_off[-1])
    X = torch.full((NT + 1, ld), complex(SENT, SENT), dtype=torch.complex64, device=DEV)
    P = torch.full((NT + 1, ld), SENT, device=DEV) if want_p else None
    x_off = torch.from_numpy(off).to(DEV)
    x_len = torch.tensor(lens, dtype=torch.int32, device=DEV)
    fo = torch.from_numpy(fr_off).to(DEV)
    _lib.call("dvae_stft_f32", _p(flat), _p(x_off), _p(x_len), B, _p(X), _p(P), _p(fo), NT, 1024, hop, ld, _stream())
    torch.cuda.synchronize()
    assert bool((X[NT] == complex(SENT, SENT)).all()) and bool((X[:, F:] == complex(SENT, SENT)).all())
    if want_p:
        assert bool((P[NT] == SENT).all()) and bool((P[:, F:] == SENT).all())
    return X[:NT, :F], (P[:NT, :F] if want_p else None), fr_off


def _stft_check(fam, flat, off, lens, nfr, hop, ld=520, want_p=True, kern="stft"):
    X, P, fr_off = _stft(flat, off, lens, nfr, hop, ld, want_p)
    Xr, Pr, eb, fb, pb = sm.stft_f64(flat, off, lens, fr_off, hop)
    _check(kern, "X", fam, X, Xr, eb)
    _check(kern, "frame", fam, torch.linalg.vector_norm(X.to(torch.complex128) - Xr, dim=1), 0.0, fb)
    if want_p:
        _check(kern, "P", fam, P, Pr, pb)
    return X, P, fr_off


@pytest.mark.parametrize("fam", sorted(FAMILIES))
@pytest.mark.parametrize("hop,odd", [(256, False), (256, True), (128, True), (307, False), (512, True), (1024, False)])
def test_stft_against_f64(fam, hop, odd):
    """Every length of LENS at one hop, the shim's frame count, plus a zero-frame entry and one with more frames than
    its signal covers; all offsets even or all odd."""
    xs = [FAMILIES[fam](T, 7 * i + hop) for i, T in enumerate(LENS)] + [FAMILIES[fam](2000, 5), FAMILIES[fam](1500, 6)]
    lens = [len(x) for x in xs]
    nfr = [_n_frames(T, hop) for T in LENS] + [0, _n_frames(1500, hop) + 9]
    flat, off = _pack(xs, odd)
    X, P, fr_off = _stft_check(fam, flat, off, lens, nfr, hop)
    if fam == "speech":                             # what the Itakura-Saito cost sees: P relative to P, bin by bin
        Pr = sm.stft_f64(flat, off, lens, fr_off, hop)[1]
        live = (Pr >= 1e-6 * Pr.amax(1, keepdim=True)) & (Pr > 0)
        P_REL60.append(float(((P.double() - Pr).abs() / Pr)[live].max()))
    if hop == 256 and fam == "speech":
        # the same utterances at the other offset parity, at ld 513 and without P: bit-identical rows
        flat2, off2 = _pack(xs, not odd)
        X2, _, _ = _stft(flat2, off2, lens, nfr, hop, ld=513, want_p=False)
        assert torch.equal(X, X2)
        X3, P3, _ = _stft_check(fam, flat, off, lens, nfr, hop, ld=528)
        assert torch.equal(X, X3) and torch.equal(P, P3)


def test_stft_shim_hop_percent():
    """``stft(..., hop_percent=0.3)`` (hop 307: aligned and misaligned frames alternate) and 0.5 through the shim."""
    from dvae_b200.packages.processing.stft import stft
    for hp, T in ((0.3, 33333), (0.5, 16000), (0.125, 20001)):
        x = _speech(T, 3)
        got = stft(x, fs=16000, wlen_sec=64e-3, win="hann", hop_percent=hp, center=False, pad_at_end=True)
        hop = int(hp * 1024)
        N = got.shape[1]
        Xr, _, eb, fb, _ = sm.stft_f64(torch.from_numpy(x).to(DEV), [0], [T], [0, N], hop)
        g = torch.from_numpy(np.ascontiguousarray(got.T)).to(DEV)
        _check("stft(shim)", "X", "speech", g, Xr, eb)
        _check("stft(shim)", "frame", "speech", torch.linalg.vector_norm(g.to(torch.complex128) - Xr, dim=1), 0.0, fb)


def _steady_batch():
    """Three 60 s utterances among many 0.1 s ones and zero-frame entries: NT >= 12 000 frames, every CTA of
    the 888-CTA grid loops at least three times, and the proportional utterance guess misses almost everywhere."""
    xs, nfr = [], []
    rng = np.random.default_rng(4)
    for i in range(420):
        if i in (100, 250, 400):
            T = 960000
        elif i % 37 == 5:
            T = 0
        else:
            T = 1600
        xs.append(_speech(T, i) if T else np.zeros(0, np.float32))
        nfr.append(0 if T == 0 else _n_frames(T, 256))
    return xs, nfr, rng


def test_stft_steady_state_ragged_batch():
    xs, nfr, _ = _steady_batch()
    lens = [len(x) for x in xs]
    flat, off = _pack(xs, False)
    NT = sum(nfr)
    n_pass = (NT + 3) // 4
    assert NT >= 12000 and n_pass >= 3 * 888 and n_pass % 888
    X, P, fr_off = _stft_check("speech*", flat, off, lens, nfr, 256)
    for u in (0, 100, 101, 250, 419):                              # alone, at an odd offset: the same rows
        f, o = _pack([xs[u]], True)
        Xu, Pu, _ = _stft(f, o, [lens[u]], [nfr[u]], 256)
        assert torch.equal(Xu, X[fr_off[u]:fr_off[u + 1]]) and torch.equal(Pu, P[fr_off[u]:fr_off[u + 1]])


def test_stft_split_twiddles_are_unbiased():
    """The split step's constant twiddles (W^k = W^t (cr[j], ci[j]), j = 1..3): the component of the error along the
    derivative of X_k by W^k, ``D_k = (X_k - conj X_512-k) / 2``, estimated by least squares over many full-scale frames,
    stays within the rounding of one twiddle (table u, constant u, cmul 2u).  A wrong constant shows up here even when it
    stays under the frame bounds: its error is proportional to D_k in every frame."""
    xs = [_tonal(48000, 6 * i + 5) for i in range(6)] + [_speech(48000, i) for i in range(6)]
    lens = [len(x) for x in xs]
    nfr = [_n_frames(T, 256) for T in lens]
    flat, off = _pack(xs, False)
    X, _, fr_off = _stft(flat, off, lens, nfr, 256)
    Xr = sm.stft_f64(flat, off, lens, fr_off, 256)[0]
    E = X.to(torch.complex128) - Xr
    for j in range(1, 4):
        k = torch.arange(64 * j, 64 * j + 64, device=DEV)
        k = k[k > 0]
        D = (Xr[:, k] - Xr[:, 512 - k].conj()) / 2
        G = (E[:, k] - E[:, 512 - k].conj()) / 2                      # a twiddle error rho adds rho D_k here
        rho = complex((D.conj() * G).sum() / (D.abs() ** 2).sum())
        RATIOS[("stft", "rho[%d]" % j, "split")] = abs(rho) / sm.W_SPLIT
        assert abs(rho) <= sm.W_SPLIT, "split twiddle group %d: error component along D_k = %.3g u" % (j, abs(rho) / sm.U)


@pytest.mark.parametrize("fam", ["tonal", "tiny"])
def test_power_against_f64(fam):
    xs = [FAMILIES[fam](T, 3 * i) for i, T in enumerate(LENS[:9])]
    lens = [len(x) for x in xs]
    flat, off = _pack(xs, False)
    X, _, _ = _stft(flat, off, lens, [_n_frames(T, 256) for T in lens], 256)
    Xs = X.contiguous()
    P = torch.full((Xs.numel() + 5,), SENT, device=DEV)
    _lib.call("dvae_power", _p(Xs), _p(P), Xs.numel(), _stream())
    torch.cuda.synchronize()
    assert bool((P[Xs.numel():] == SENT).all())
    Pr, pb = sm.power_f64(Xs.reshape(-1))
    _check("power", "P", fam, P[:Xs.numel()], Pr, pb)


# --------------------------------------------------------------------------------------------- ISTFT
N_SET = [0, 1, 2, 3, 4, 5, 185]


def _shapes():
    out = []
    for N in N_SET:
        nat = 1024 + 256 * (N - 1) if N else 0
        for L in sorted({1, 255, 256, 1023, 1024, 1025, max(1, nat - 1), max(1, nat), nat + 1, nat + 3000}):
            out.append((N, L))
    return out


SHAPES = _shapes()


def _spectra(fam, shapes, seed):
    """(X [NT][520] complex64, mask [NT][520] or None, mask_scale, fr_off) of one ISTFT input family."""
    nfr = [N for N, _ in shapes]
    fr_off = np.zeros(len(nfr) + 1, np.int64)
    np.cumsum(nfr, out=fr_off[1:])
    NT = int(fr_off[-1])
    gen = torch.Generator(device=DEV).manual_seed(seed)
    X = torch.zeros((NT, 520), dtype=torch.complex64, device=DEV)
    if fam in ("roundtrip", "wiener"):
        xs = [_speech(1024 + 256 * max(N - 1, 0) + 100, seed + i) for i, N in enumerate(nfr)]
        flat, off = _pack(xs, False)
        Xs, _, _ = _stft(flat, off, [len(x) for x in xs], nfr, 256)
        X[:, :F] = Xs
    elif fam == "random":                                           # no STFT of anything; Im at DC and Nyquist nonzero
        lvl = 10.0 ** (torch.randint(-4, 2, (NT, 1), device=DEV, generator=gen).float())
        X[:, :F] = torch.complex(torch.randn((NT, F), device=DEV, generator=gen), torch.randn((NT, F), device=DEV, generator=gen)) * lvl
    else:                                                           # sparse: one live bin per frame
        k = torch.randint(0, F, (NT,), device=DEV, generator=gen)
        X[torch.arange(NT, device=DEV), k] = torch.complex(torch.randn(NT, device=DEV, generator=gen),
                                                          torch.randn(NT, device=DEV, generator=gen))
    mask, scale = None, 1.0
    if fam == "wiener":
        R = 25 if seed % 2 else 30
        mask = torch.rand((NT, 520), device=DEV, generator=gen) * R          # WFs-like sums in [0, R]
        mask[torch.rand((NT, 520), device=DEV, generator=gen) < 0.1] = 0.0   # exact zeros
        late = torch.rand((NT, 520), device=DEV, generator=gen) < 0.2
        mask[late] = 1e-12 * R                                               # a late-run state
        scale = 1.0 / R
    elif fam in ("random", "sparse"):
        mask = torch.rand((NT, 520), device=DEV, generator=gen)
    return X, mask, scale, fr_off


def _layout(shapes, order=None, gap=5):
    """y_off of every utterance with sentinel gaps; ``order``: the order of the utterances in memory (non-monotone y_off)."""
    order = range(len(shapes)) if order is None else order
    y_off, pos = np.zeros(len(shapes), np.int64), gap
    for u in order:
        y_off[u] = pos
        pos += shapes[u][1] + gap
    return y_off, pos + gap


def _istft(X, mask, scale, fr_off, y_off, lens, total):
    y = torch.full((total,), SENT, device=DEV)
    B = len(lens)
    fo = torch.from_numpy(fr_off).to(DEV)                            # held until the kernel has run
    yo = torch.from_numpy(y_off).to(DEV)
    yl = torch.tensor(lens, dtype=torch.int32, device=DEV)
    args = (_p(fo), B, _p(y), _p(yo), _p(yl), int(max(lens)), 1024, 256, X.shape[1], _stream())
    if mask is None:
        _lib.call("dvae_istft_f32", _p(X), *args)
    else:
        _lib.call("dvae_istft_masked_f32", _p(X), _p(mask), float(scale), *args)
    torch.cuda.synchronize()
    return y


def _istft_check(fam, kern, X, mask, scale, fr_off, shapes, order=None):
    lens = [L for _, L in shapes]
    y_off, total = _layout(shapes, order)
    y = _istft(X, mask, scale, fr_off, y_off, lens, total)
    yr, b, written = sm.istft_f64(X, fr_off, y_off, lens, total, mask, scale)
    assert bool((y[~written] == SENT).all()), "%s wrote outside its utterances" % kern
    _check(kern, "y", fam, y[written], yr[written], b[written])
    return y, y_off


@pytest.mark.parametrize("fam", ["roundtrip", "wiener", "random", "sparse"])
@pytest.mark.parametrize("masked", [False, True])
def test_istft_against_f64(fam, masked):
    """Every (N, y_len) of SHAPES in one batch (B = 70): each sample inside its bound, exact zeros at sample 0 and past
    the natural length, sentinels untouched."""
    X, mask, scale, fr_off = _spectra(fam, SHAPES, 11)
    if not masked:
        if mask is not None:                                        # the plain kernel on the mask product
            mk = mask * np.float32(scale)
            X = torch.complex(mk * X.real, mk * X.imag)
        mask = None
    _istft_check(fam, "istft_masked" if masked else "istft", X, mask, scale, fr_off, SHAPES)


def _rows(y, y_off, shapes):
    return [y[o:o + L] for o, (_, L) in zip(y_off, shapes)]


@pytest.mark.parametrize("masked", [False, True])
def test_istft_is_independent_of_segmentation_and_order(masked):
    """An utterance's samples are bit-identical at B = 1 (most segments), B = 7, B = 70 and B = 600 (one CTA per
    utterance), after permuting the batch with non-monotone y_off, and in the plain kernel on the mask product."""
    fam = "random"
    X, mask, scale, fr_off = _spectra(fam, SHAPES, 12)
    if not masked:
        mask = None
    y, y_off = _istft_check(fam, "istft_masked" if masked else "istft", X, mask, scale, fr_off, SHAPES)
    ref = _rows(y, y_off, SHAPES)

    def sub(idx):
        shapes = [SHAPES[i] for i in idx]
        rows = torch.cat([torch.arange(fr_off[i], fr_off[i + 1]) for i in idx]) if len(idx) else torch.zeros(0, dtype=torch.long)
        rows = rows.to(DEV, torch.long) if len(rows) else torch.zeros(1, dtype=torch.long, device=DEV)   # N = 0: a dummy row
        fo = np.zeros(len(idx) + 1, np.int64)
        np.cumsum([s[0] for s in shapes], out=fo[1:])
        return shapes, X[rows].contiguous(), (None if mask is None else mask[rows].contiguous()), fo

    for idx in [[i] for i in range(len(SHAPES))] + [list(range(i, min(i + 7, len(SHAPES)))) for i in range(0, len(SHAPES), 7)]:
        shapes, Xs, ms, fo = sub(idx)
        y_off_s, total = _layout(shapes)
        ys = _istft(Xs, ms, scale, fo, y_off_s, [L for _, L in shapes], total)
        for i, r in zip(idx, _rows(ys, y_off_s, shapes)):
            assert torch.equal(r, ref[i]), "utterance %d (N, y_len = %s) differs at B = %d" % (i, SHAPES[i], len(idx))
    perm = np.random.default_rng(3).permutation(len(SHAPES))
    idx = list(perm) + list(np.random.default_rng(4).integers(0, len(SHAPES), 600 - len(SHAPES)))   # B = 600, shuffled
    shapes, Xs, ms, fo = sub(idx)
    order = np.random.default_rng(5).permutation(len(idx))          # memory order unrelated to the batch order
    y_off_s, total = _layout(shapes, order)
    ys = _istft(Xs, ms, scale, fo, y_off_s, [L for _, L in shapes], total)
    written = torch.zeros(total, dtype=torch.bool, device=DEV)
    for i, o, (_, L), r in zip(idx, y_off_s, shapes, _rows(ys, y_off_s, shapes)):
        assert torch.equal(r, ref[i]), "utterance %d differs at B = 600, permuted" % i
        written[o:o + L] = True
    assert bool((ys[~written] == SENT).all())
    if masked:                                                       # the plain kernel on the mask product, B = 1 and B = 70
        mk = mask * np.float32(scale)
        Xm = torch.complex(mk * X.real, mk * X.imag)
        lens = [L for _, L in SHAPES]
        y2 = _istft(Xm, None, 1.0, fr_off, y_off, lens, int(y.numel()))
        assert torch.equal(y2, y)
        for i in [k for k, (N, _) in enumerate(SHAPES) if N in (1, 3, 185)]:    # short N and the most segments, B = 1
            shapes, _, _, fo = sub([i])
            Xs = Xm[fr_off[i]:fr_off[i + 1]].contiguous()
            y_off_s, total = _layout(shapes)
            ys = _istft(Xs, None, 1.0, fo, y_off_s, [SHAPES[i][1]], total)
            assert torch.equal(_rows(ys, y_off_s, shapes)[0], ref[i])
