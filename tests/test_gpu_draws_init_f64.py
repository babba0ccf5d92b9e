"""The random draws and the EM starting state against a host Philox and float64, element by element.

* ``box_muller`` (csrc/common.cuh, through ``dvae_box_muller_f32``): every one of the 2^24 uniforms of each word, the other
  word at fixed values, inside the bound of ``oracle/philox_np.box_muller_f64`` (``__logf``, ``sqrtf``, the FP32 angle,
  ``__sincosf``, the FP32 product) and finite.  The module prints how often ``__logf(u1) > 0`` (a NaN radius) or ``= 0`` (a
  zero radius) occurred for ``u1 < 1``.
* ``dvae_rng_dump``, both kernels: uniforms bit-exact with the host Philox, normals inside the bound, every element; ragged
  ``L``, chain counts up to 128, negative and extreme utterance ids, frame indices up to 2^20 - 1, ``iter0 + it`` wrapping
  past 2^32, per-frame ``iter0_frame``, a misaligned output and 65 536 iterations.
* ``dvae_nmf_init``: W, H and g bit-exact with the host restatement (zero-frame utterances first / middle / last, repeated and
  negative ids, K 1 / 10 / 16, F 33 / 513, the ``eps`` clamp); ``dvae_nmf_vb`` within ``gamma_K Vb`` of float64 ``W H``.
* ``McemEngine.init_parameters`` (M1, M2, M2v3, the IBM-conditioned M2): the chain start Z (FP32 encoder mean) inside the
  float64 forward's bound, repeated bit-exactly over the chains; ``ybias`` inside its bound; ``kscale`` equal to the host
  restatement of ``row_scale_kernel``.
* ``dvae_mlp_fwd`` across its 2^18-row chunks: an encoder with labels over 600 000 rows and a decoder with label row
  divisors that do not divide 2^18, every element against float64, boundary rows alone bit-identical, pad columns untouched.

The largest error / bound ratio per (kernel, output, family) is printed at the end of the module.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth, tc
from dvae_b200.engine import (McemConfig, McemEngine, PackedMlp, RaggedBatch, VaeWeights, _ld_for, _p, _stream, mlp_forward,
                              stft_batch)
from oracle import philox_np as ph
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
SENT = -7.0
SEED = 0x0123456789ABCDEF                       # both key words nonzero
RATIOS = {}                                     # (kernel, output, family) -> largest |gpu - f64| / bound
LOGF = {"u1 < 1": 0, "logf > 0": 0, "logf = 0": 0}


@pytest.fixture(scope="module", autouse=True)
def _ratio_table():
    yield
    if RATIOS:
        print("\nlargest |gpu - f64| / bound")
        for (kern, out, fam), r in sorted(RATIOS.items()):
            print("  %-16s %-8s %-22s %9.3g" % (kern, out, fam, r))
    if LOGF["u1 < 1"]:
        print("box_muller over %d words with u1 < 1: __logf(u1) > 0 (NaN radius) %d times, = 0 (zero radius) %d times"
              % (LOGF["u1 < 1"], LOGF["logf > 0"], LOGF["logf = 0"]))


def _check(kern, out, fam, got, ref, bound):
    """``|got - ref| <= bound`` for every element; a non-finite ``got`` fails."""
    got = torch.as_tensor(got).to(DEV, torch.float64)
    ref = torch.as_tensor(ref).to(DEV, torch.float64)
    bound = torch.as_tensor(bound).to(DEV, torch.float64).expand(got.shape)
    err = (got - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / torch.where(bound > 0, bound, torch.full_like(bound, 1e-300)))
    ratio = torch.where(torch.isfinite(got), ratio, torch.full_like(ratio, np.inf))
    r = float(ratio.max()) if ratio.numel() else 0.0
    RATIOS[(kern, out, fam)] = max(RATIOS.get((kern, out, fam), 0.0), r)
    if not r <= 1.0:
        i = int(torch.argmax(ratio.reshape(-1)))
        idx = np.unravel_index(i, tuple(ratio.shape))
        pytest.fail("%s %s [%s]: |gpu - f64| / bound = %.3g at %s (gpu %r, f64 %r, bound %.3g)"
                    % (kern, out, fam, r, idx, float(got.reshape(-1)[i]), float(ref.reshape(-1)[i]), float(bound.reshape(-1)[i])))


def _dev_u32(a):
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, np.uint32)).view(np.int32)).to(DEV)


# --------------------------------------------------------------------------------------------- Box-Muller
FIXED = {"a": [0x00000000, 0x3FFFFF80, 0x80000000, 0xFFFFFFFF],             # the angle word: u2 ~ 0, 1/4, 1/2, 1
         "b": [0x00000000, 0x80000000, 0xFFFFFE00, 0xFFFFFFFF]}             # the radius word: u1 ~ 0, 1/2, 1 - 2^-23, 1


@pytest.mark.parametrize("sweep", ["a", "b"])
def test_box_muller_every_uniform(sweep):
    """All 2^24 values of ``a >> 8`` (radius) or ``b >> 8`` (angle), the low byte varied, the other word fixed."""
    k = np.arange(1 << 24, dtype=np.uint32)
    words = (k << np.uint32(8)) | ((k * np.uint32(0x9E)) & np.uint32(0xFF))
    wd = _dev_u32(words)
    n = words.size
    n0 = torch.empty(n, device=DEV)
    n1 = torch.empty(n, device=DEV)
    for other in FIXED[sweep]:
        fixed = np.full(n, other, np.uint32)
        a, b = (words, fixed) if sweep == "a" else (fixed, words)
        ad, bd = (wd, _dev_u32(fixed)) if sweep == "a" else (_dev_u32(fixed), wd)
        _lib.call("dvae_box_muller_f32", _p(ad), _p(bd), _p(n0), _p(n1), n, _stream())
        torch.cuda.synchronize()
        below = torch.from_numpy(ph.u01(a) < 1).to(DEV)
        LOGF["u1 < 1"] += int(below.sum())
        LOGF["logf > 0"] += int((below & torch.isnan(n0)).sum())
        LOGF["logf = 0"] += int((below & (n0 == 0) & (n1 == 0)).sum())
        r0, r1, b0, b1 = ph.box_muller_f64(a, b)
        _check("box_muller", "n0", "%s sweep" % sweep, n0, torch.from_numpy(r0), torch.from_numpy(b0))
        _check("box_muller", "n1", "%s sweep" % sweep, n1, torch.from_numpy(r1), torch.from_numpy(b1))


# --------------------------------------------------------------------------------------------- dvae_rng_dump
GID = [0, 5, -1, -2 ** 31, 2 ** 31 - 1, 123456789, 5]
FIDX = [0, 1, 2 ** 20 - 1, 777, 2 ** 19, 3, 1]
IT0F = [2 ** 32 - 1, 0, 5, 2 ** 31, 2 ** 32 - 2, 65535, 1]


def _dump(L, C_, n_iter, iter0=0, per_frame=False, misalign=False, NT=len(GID)):
    gid, idx = _dev_u32(np.asarray(GID[:NT], np.int64) & 0xFFFFFFFF), _dev_u32(FIDX[:NT])
    rng = _lib.DvaeRng()
    rng.seed, rng.iter0 = SEED, iter0 & 0xFFFFFFFF
    it0 = _dev_u32(IT0F[:NT]) if per_frame else None
    rng.iter0_frame = None if it0 is None else it0.data_ptr()
    chains = NT * C_
    n = n_iter * chains * L
    buf = torch.full((n + 8,), SENT, device=DEV)
    eps = buf[1:n + 1] if misalign else buf[:n]
    u = torch.full((n_iter * chains + 4,), SENT, device=DEV)
    _lib.call("dvae_rng_dump", C.byref(rng), _p(gid), _p(idx), NT, C_, L, n_iter, _p(eps), _p(u), _stream())
    torch.cuda.synchronize()
    assert bool((buf[n + (1 if misalign else 0):] == SENT).all()) and bool((u[n_iter * chains:] == SENT).all())
    if misalign:
        assert float(buf[0]) == SENT
    ref, bnd, uref = ph.draws_f64(SEED, GID[:NT], FIDX[:NT], C_, L, n_iter, iter0, IT0F[:NT] if per_frame else None)
    return eps.view(n_iter, chains, L), u[:n_iter * chains].view(n_iter, chains), ref, bnd, uref


# (L, C, n_iter, iter0, per-frame iter0, misaligned eps): the first four take rng_dump4_kernel, the rest the generic kernel
DUMP_CASES = [(4, 1, 9, 2 ** 32 - 4, False, False), (16, 3, 5, 0, True, False), (32, 16, 4, 2 ** 31, False, False),
              (64, 128, 3, 2 ** 32 - 1, True, False),
              (1, 1, 7, 2 ** 32 - 3, False, False), (3, 3, 5, 11, True, False), (5, 16, 4, 2 ** 32 - 2, False, False),
              (17, 128, 2, 0, True, False), (63, 5, 3, 2 ** 32 - 1, False, False), (16, 4, 6, 2 ** 32 - 5, True, True)]


@pytest.mark.parametrize("L,C_,n_iter,iter0,per_frame,misalign", DUMP_CASES)
def test_rng_dump_against_host_philox(L, C_, n_iter, iter0, per_frame, misalign):
    kern = "rng_dump4" if (L in (4, 8, 16, 32, 64) and not misalign) else "rng_dump"
    eps, u, ref, bnd, uref = _dump(L, C_, n_iter, iter0, per_frame, misalign)
    assert torch.equal(u.cpu(), torch.from_numpy(uref)), "accept uniforms differ from the host Philox"
    _check(kern, "eps", "L=%d" % L, eps, torch.from_numpy(ref), torch.from_numpy(bnd))


def test_rng_dump_65536_iterations():
    """n_iter = 65 536 is past the 16-bit grid of rng_dump4_kernel: the generic kernel, with iter0 + it wrapping."""
    eps, u, ref, bnd, uref = _dump(4, 2, 65536, 2 ** 32 - 30000, NT=2)
    assert torch.equal(u.cpu(), torch.from_numpy(uref))
    _check("rng_dump", "eps", "n_iter=65536", eps, torch.from_numpy(ref), torch.from_numpy(bnd))


def test_rng_dump_rejects_4096_chains():
    rng = _lib.DvaeRng()
    t = torch.zeros(16, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError, match="n_chains"):
        _lib.call("dvae_rng_dump", C.byref(rng), _p(t), _p(t), 1, 4096, 4, 1, _p(t), _p(t), _stream())


# --------------------------------------------------------------------------------------------- NMF start
KMAX = 16


def _nmf_init_host(seed, utt_ids, fr_off, F, K, ld, eps):
    """nmf_init_kernel restated: W [B][K][ld] (0 in the pad columns), H [NT][K], from word x of the Philox blocks."""
    utt_ids = np.asarray(utt_ids, np.int64)
    fr_off = np.asarray(fr_off, np.int64)
    B, NT = len(utt_ids), int(fr_off[-1])
    e = np.float32(eps)
    f, k = np.meshgrid(np.arange(F), np.arange(K), indexing="ij")
    W = np.zeros((B, K, ld), np.float32)
    for u in range(B):
        x = ph.mh_words(seed, utt_ids[u], f * KMAX + k, 0xFFFFFFF0, 0)[0]
        W[u, :, :F] = np.maximum(ph.u01(x), e).T
    n = np.arange(NT)
    owner = np.searchsorted(fr_off[:B], n, side="right") - 1        # the last utterance starting at or before n
    kk = np.arange(K)[None, :]
    x = ph.mh_words(seed, utt_ids[owner][:, None], (n - fr_off[owner])[:, None] * KMAX + kk, 0xFFFFFFF1, 0)[0]
    H = np.maximum(ph.u01(x), e)
    return W, H


def _vb_f64(W, H, frame_utt):
    """float64 W H per frame and the bound of the FP32 FMA chain over K (all terms positive: sum |w h| = Vb)."""
    W64, H64 = W.double(), H.double()
    K = H.shape[1]
    Vb = torch.einsum("nkf,nk->nf", W64[frame_utt.long()], H64)
    return Vb, K * U / (1 - K * U) * Vb


NMF_LENS = [0, 37, 0, 120, 1, 0, 0]
NMF_IDS = [7, -3, 7, 2 ** 31 - 1, -2 ** 31, 7, 11]


@pytest.mark.parametrize("K,F,eps", [(1, 33, 0.5), (10, 513, 0.5), (16, 513, 1e-8), (10, 33, 1e-8), (16, 33, 0.5)])
def test_nmf_init_and_vb(K, F, eps):
    ld = _ld_for(F) + 8
    b = RaggedBatch(NMF_LENS, DEV, utt_ids=NMF_IDS)
    B, NT = b.B, b.NT
    W = torch.full((B, K, ld), SENT, device=DEV)
    H = torch.full((NT + 1, K), SENT, device=DEV)
    g = torch.full((NT + 1,), SENT, device=DEV)
    _lib.call("dvae_nmf_init", SEED, _p(b.utt_ids), _p(b.fr_off), B, NT, F, K, ld, eps, _p(W), _p(H), _p(g), _stream())
    torch.cuda.synchronize()
    Wr, Hr = _nmf_init_host(SEED, NMF_IDS, b.fr_off_host, F, K, ld, eps)
    assert torch.equal(W.cpu(), torch.from_numpy(Wr)), "W differs from the host Philox"
    assert torch.equal(H[:NT].cpu(), torch.from_numpy(Hr)), "H differs from the host Philox"
    assert bool((g[:NT] == 1.0).all()) and float(H[NT, 0]) == SENT and float(g[NT]) == SENT
    if eps == 0.5:
        assert bool((W[:, :, :F] == 0.5).any()) and bool((W[:, :, :F] > 0.5).any())
    Vb = torch.full((NT + 1, ld), SENT, device=DEV)
    _lib.call("dvae_nmf_vb", _p(W), _p(H), _p(b.frame_utt), NT, F, K, ld, _p(Vb), _stream())
    torch.cuda.synchronize()
    assert bool((Vb[:, F:] == SENT).all()) and bool((Vb[NT] == SENT).all())
    ref, bound = _vb_f64(W[:, :, :F], H[:NT], b.frame_utt)
    _check("nmf_vb", "Vb", "K=%d" % K, Vb[:NT, :F], ref, bound)


# --------------------------------------------------------------------------------------------- float64 MLP forward
def _ulp_bound(t):
    """At least one FP32 ulp of every value of magnitude <= |t| (float64 in)."""
    return 2.0 ** -23 * t.abs() + 2.0 ** -149


def mlp_f64(layers, x, x2=None, div=1, block=1 << 16):
    """float64 forward of a tanh MLP (``layers``: [(W [out][in], b)] float32) on FP32 rows ``x`` [+ label rows ``x2[r // div]``]
    and the bound of ``linear_kernel``'s arithmetic: per layer an FFMA chain from 0 over K inputs (``gamma_K sum |a w|``), the
    input radii through ``sum |w| r``, the FP32 bias add, and ``tanhf`` at 2 ulp with Lipschitz constant 1.  Returns
    (out, bound) float64 on the device."""
    Ws = [(torch.as_tensor(w).to(DEV, torch.float64), torch.as_tensor(b).to(DEV, torch.float64)) for w, b in layers]
    outs, bounds = [], []
    for r0 in range(0, x.shape[0], block):
        a = x[r0:r0 + block].to(torch.float64)
        if x2 is not None:
            rows = torch.arange(r0, r0 + a.shape[0], device=DEV) // div
            a = torch.cat([a, x2[rows].to(torch.float64)], 1)
        rad = torch.zeros_like(a)
        for i, (W, bias) in enumerate(Ws):
            K = W.shape[1]
            acc = a @ W.T
            err = K * U / (1 - K * U) * ((a.abs() + rad) @ W.abs().T) + rad @ W.abs().T
            pre = acc + bias
            err = err + U * (pre.abs() + err)
            if i + 1 < len(Ws):
                a = torch.tanh(pre)
                rad = err + 2 * _ulp_bound(a.abs() + err)
            else:
                a, rad = pre, err
        outs.append(a)
        bounds.append(rad)
    return torch.cat(outs), torch.cat(bounds)


def test_mlp_fwd_tanh_epilogue_against_f64():
    """The tanh epilogue of ``linear_kernel`` on its own: a 1 x 1 layer (weight 1, bias 0: the pre-activation is the input,
    exactly) over 2^20 inputs from 1e-30 to saturation, both signs, held to ``tanhf``'s 2 ulp.  Inside the MLP bounds an
    approximate tanh can hide under the accumulated rounding of the layers around it; here it cannot."""
    mlp = PackedMlp([(np.ones((1, 1), np.float32), np.zeros(1, np.float32))], DEV)
    mag = torch.logspace(-30, np.log10(12.0), 1 << 19, dtype=torch.float64, device=DEV).float()
    x = torch.cat([mag, -mag])[:, None].contiguous()
    y = mlp_forward(mlp, x, _lib.ACT_TANH)
    torch.cuda.synchronize()
    t = torch.tanh(x.double())
    _check("mlp_fwd(tanh)", "out", "1x1 layer", y, t, 2 * _ulp_bound(t))


# --------------------------------------------------------------------------------------------- EM starting state
def _weights(kind):
    variant, y_dim = {"M1": ("M1", 0), "M2": ("M2", 1), "M2v3": ("M2v3", 1), "IBM": ("M2", 513)}[kind]
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=21, out_bias=float(np.log(0.05)))
    for key in list(sd):                                             # nonzero biases: the bias add is part of the bound
        if key.endswith("bias"):
            sd[key] = (sd[key] + np.random.default_rng(len(key)).normal(0, 0.1, sd[key].shape)).astype(np.float32)
    return sd, VaeWeights(sd, variant, torch.device(DEV)), y_dim


def _q16(x):
    return (np.clip(np.round(x * 32768.0), -32768, 32767) / 32768.0).astype(np.float32)


def _speech_batch():
    """Ragged batch with zero-frame utterances first, in the middle and last; 16-bit speech with digital silence (all-zero
    frames) and +-1 LSB noise (16-bit-quiet frames); utterances 2^40 louder and quieter (the kscale clamp)."""
    rng = np.random.default_rng(8)
    sp = lambda u, s: synth.synth_utterance(u, s, 5.0)[0]           # noqa: E731
    lsb = (rng.integers(-1, 2, 8000) / 32768.0).astype(np.float32)
    u0 = np.concatenate([_q16(sp(1, 1.5)), np.zeros(8000, np.float32), lsb, _q16(sp(2, 0.5))])
    xs = [np.zeros(0, np.float32), u0, np.zeros(0, np.float32), (sp(3, 1.0) * np.float32(2.0 ** 40)),
          (sp(4, 1.0) * np.float32(2.0 ** -40)), _q16(sp(5, 0.3)), np.zeros(0, np.float32)]
    nfr = [0 if len(x) < 1024 else 1 + (len(x) - 1024) // 256 for x in xs]
    ids = [7, 12, -5, 7, -2 ** 31, 99, 3]
    b = RaggedBatch(nfr, DEV, utt_ids=ids)
    off = np.cumsum([0] + [len(x) for x in xs])[:-1].astype(np.int64)
    flat = torch.from_numpy(np.concatenate(xs)).to(DEV)
    _, P = stft_batch(flat, torch.from_numpy(off).to(DEV), torch.tensor([len(x) for x in xs], dtype=torch.int32, device=DEV), b)
    P[:, 513:] = 0.0
    torch.cuda.synchronize()
    zero = (P[:, :513] == 0).all(1)
    assert bool(zero.any()) and bool((~zero).any())
    return b, P


def _kscale_host(P, bias_log2, F):
    """row_scale_kernel restated: ``(k, k_alt)``; k = 2^(-2c), c = clamp(rint(top) - 16, +-30), top = max_f log2 P - b over P > 0,
    2^15 without energy.  Where the float64 top is within log2f's error (1 ulp) and the FP32 subtraction of a midpoint
    n + 1/2, ``k_alt`` is the neighbouring scale, else k."""
    P64 = P[:, :F].double()
    b = bias_log2.double()[None, :]
    lg = torch.where(P64 > 0, torch.log2(P64), torch.full_like(P64, -np.inf))
    top = (lg - b).max(1).values
    err = 2.0 ** -23 * (top.abs() + b.abs().max()) + U * (top.abs() + 1.0)      # |log2 P| <= |top| + |b|
    live = torch.isfinite(top)
    topf = torch.where(live, top, torch.zeros_like(top))

    def scale(t):
        c = torch.clamp(torch.round(t) - 16.0, -30.0, 30.0)
        return torch.where(live, torch.exp2(-2.0 * c), torch.full_like(t, 32768.0))
    k = scale(topf)
    mid = torch.floor(topf) + 0.5
    near = (topf - mid).abs() <= err
    k_alt = torch.where(near, scale(torch.where(topf >= mid, mid - 0.25, mid + 0.25)), k)
    return k, k_alt


@pytest.mark.parametrize("kind", ["M1", "M2", "M2v3", "IBM"])
def test_starting_state_against_f64(kind):
    sd, w, y_dim = _weights(kind)
    b, P = _speech_batch()
    NT, F, C_ = b.NT, 513, 3
    y = None
    if y_dim:
        y = (torch.rand((NT, y_dim), generator=torch.Generator(device=DEV).manual_seed(4), device=DEV) > 0.5).float()
    X = torch.zeros((NT, 520), dtype=torch.complex64, device=DEV)
    eng = McemEngine(w, McemConfig(niter=1, sampler="tc", n_chains=C_, seed=SEED), DEV)
    eng.init_parameters(X, P, b, y)
    torch.cuda.synchronize()
    # W, H, g and Vb
    Wr, Hr = _nmf_init_host(SEED, b.utt_ids_host, b.fr_off_host, F, eng.cfg.nmf_rank, eng.ld, eng.cfg.eps)
    assert torch.equal(eng.W.cpu(), torch.from_numpy(Wr)) and torch.equal(eng.H.cpu(), torch.from_numpy(Hr))
    assert bool((eng.g == 1.0).all())
    ref, bound = _vb_f64(eng.W[:, :, :F], eng.H, b.frame_utt)
    _check("nmf_vb", "Vb", kind, eng.Vb[:, :F], ref, bound)
    # Z: the encoder mean, repeated over the chains
    enc = [(sd["encoder.hidden.%d.weight" % i], sd["encoder.hidden.%d.bias" % i]) for i in range(2)]
    enc.append((sd["encoder.sample.mu.weight"], sd["encoder.sample.mu.bias"]))
    mu, mb = mlp_f64(enc, P[:, :F], y if w.enc_takes_y else None)
    Z = eng.Z.view(NT, C_, w.z_dim)
    _check("mlp_fwd(enc)", "Z", kind, Z[:, 0], mu, mb)
    for c in range(1, C_):
        assert torch.equal(Z[:, c], Z[:, 0])
    # kscale
    img = tc.decoder_image(w)
    off = int(_lib.load().dvae_tc_image_bias_offset(w.dec_tc.ref, w.z_dim, w.tc_y_dim))
    bias_log2 = img[off:off + 4 * F].view(torch.float32)
    k, k_alt = _kscale_host(P, bias_log2, F)
    ks = eng.kscale[:NT].double()
    bad = (ks != k) & (ks != k_alt)
    assert not bool(bad.any()), "kscale differs from row_scale_kernel restated at frames %s" % torch.nonzero(bad)[:8, 0].tolist()
    assert bool((ks == 32768.0).any()) and bool((ks == 2.0 ** 60).any()) and bool((ks == 2.0 ** -60).any())
    # ybias of the label-bias decoder: W1[:, L:] y + b1
    if w.tc_label_bias:
        W1 = sd["decoder.hidden.0.weight"]
        yb, ybb = mlp_f64([(W1[:, w.z_dim:], sd["decoder.hidden.0.bias"])], y)
        _check("mlp_fwd(ybias)", "ybias", kind, eng.ybias, yb, ybb)
    else:
        assert eng.ybias is None


# --------------------------------------------------------------------------------------------- row chunks of dvae_mlp_fwd
CHUNK = 1 << 18


def _chunked(mlp, layers, x, x2, div, N, fam):
    rows = x.shape[0]
    buf = torch.full((rows, N + 5), SENT, device=DEV)
    out = buf[:, :N]
    mlp_forward(mlp, x, _lib.ACT_NONE, x2=x2, x2_row_div=div, out=out)
    torch.cuda.synchronize()
    assert bool((buf[:, N:] == SENT).all()), "dvae_mlp_fwd wrote into the pad columns"
    ref, bound = mlp_f64(layers, x, x2, div)
    _check("mlp_fwd(chunks)", "out", fam, out, ref, bound)
    chunk = CHUNK // div * div
    for cb in range(chunk, rows, chunk):                            # each boundary: a window of whole label rows, alone
        s = cb - 2 * div
        e = min(rows, cb + 2 * div)
        alone = mlp_forward(mlp, x[s:e], _lib.ACT_NONE, x2=x2[s // div:], x2_row_div=div)
        torch.cuda.synchronize()
        assert torch.equal(alone, out[s:e]), "rows %d..%d alone differ from the same rows in the chunked call" % (s, e)
    return out


def test_mlp_fwd_encoder_with_labels_over_three_chunks():
    """The M2 encoder over [x; y] on 600 000 rows: chunks of 2^18, 2^18 and 75 712 rows."""
    sd, _, _ = _weights("M2")
    layers = [(sd["encoder.hidden.%d.weight" % i], sd["encoder.hidden.%d.bias" % i]) for i in range(2)]
    layers.append((sd["encoder.sample.mu.weight"], sd["encoder.sample.mu.bias"]))
    mlp = PackedMlp(layers, DEV)
    rows = 600000
    gen = torch.Generator(device=DEV).manual_seed(6)
    x = torch.empty((rows, 513), device=DEV).exponential_(1.0, generator=gen) * 0.05
    y = torch.rand((rows, 1), device=DEV, generator=gen)
    _chunked(mlp, layers, x, y, 1, 16, "encoder, div=1")


@pytest.mark.parametrize("div", [7, 10, 30])
def test_mlp_fwd_decoder_label_rows_across_chunks(div):
    """A decoder over [z; y[r / div]] (three label columns) on 270 000 rows: the chunk is the largest multiple of div below
    2^18, and the label pointer of the second chunk is offset by whole label rows."""
    sd = synth.xavier_state_dict("M2", 513, 16, [128, 128], 3, seed=9, out_bias=float(np.log(0.05)))
    layers = [(sd["decoder.hidden.%d.weight" % i], sd["decoder.hidden.%d.bias" % i]) for i in range(2)]
    layers.append((sd["decoder.reconstruction.weight"], sd["decoder.reconstruction.bias"]))
    mlp = PackedMlp(layers, DEV)
    rows = 270000
    gen = torch.Generator(device=DEV).manual_seed(div)
    z = torch.randn((rows, 16), device=DEV, generator=gen)
    y = torch.rand(((rows + div - 1) // div, 3), device=DEV, generator=gen)
    _chunked(mlp, layers, z, y, div, 513, "decoder, div=%d" % div)
