"""Both Metropolis-Hastings samplers against a float64 replay of their own chains (oracle/mh_replay.py), every iteration of
every chain, and the packed P / Vb stream of the tensor-core sampler element by element.

The sampler runs first on Philox draws; ``dvae_rng_dump`` gives the same draws (test_gpu_vst.py pins that), and the replay
recomputes every proposal from them in float64, taking each accept decision from the sampler: kept iterations from ``Zs``,
burn-in iterations from ``a_trace`` and ``u``.  The trajectories never diverge, so nothing after a close call goes unchecked.

Per case: the kept samples, the final states, the accept counts and the emission's slot table equal the replay exactly; the
log ratio is within tau * S of the replay through the sampler's own rounding points (the "mirrored" decoder: BF16 weights,
BF16 activations from a table of the samplers' tanh.approx.bf16x2 over every BF16 input, the stream's own P' / Vb') and within the stated 0.05 + 2e-3 S of the plain FP32-weight decoder, with
S = sum_f (2 + P/Vx + P/Vx'); every decision outside the band |log u - a| <= tau * S is float64's; every emitted slot is the
mirrored decoder's 2^v of its sample to the precision of the emission word.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth, tc
from dvae_b200.engine import McemConfig, McemEngine, RaggedBatch, VaeWeights, _p, _stream
from oracle import mh_replay, stft_np
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu
KW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
F, LD, NPAD, TM = 513, 520, 528, 128
MODE_FLAGS = {0: 0, 1: tc.POLY_EX2, 2: tc.POLY_EX2 | tc.POLY_EX2_ALL}

# |a_gpu - a_mirrored| <= TAU[mode] * S.  The mirror takes the samplers' activation from a table of tanh.approx.bf16x2 over
# all BF16 inputs (it differs from the correctly rounded tanh by one BF16 ulp in 2086 of the 65280 finite inputs).  What remains:
# the FP32 sums of l(z) and l(z') (528 bins, 132 quad logarithms and reciprocals), the MUFU ex2 / lg2 / rcp approximations
# (~2^-22 relative) and, in polynomial bins, ex2_poly2 (7.5e-5 relative, largely the same for z and z': v' - v is small); and
# the pre-activations whose FP32 tensor-core accumulator and float64 value lie on opposite sides of a BF16 rounding midpoint,
# which changes one activation by one BF16 ulp (the spread between cases of one mode: case 10 6.0e-7, case 2 2.5e-5).
# Largest ratio measured over all cases on one B200 (1000 W): mode 0 2.54e-5 (case 2), mode 1 4.28e-5 (case 9), mode 2
# 1.26e-5 (case 7); TAU is twice that, rounded up.  (With the correctly rounded tanh in the mirror: 4.3e-4, 5.9e-4, 2.4e-4.)
TAU = {0: 5.1e-5, 1: 8.6e-5, 2: 2.6e-5}
# Emission: relative deviation of an emitted 2^v from the mirrored decoder's beyond the word's precision (and ex2_poly2's in
# polynomial bins), from the same midpoint flips.  Measured max 6.4e-4 (case 5); RHO is twice that.  The edge bins of the edge
# decoder sum 64 saturated (tabulated, flip-free) activations exactly, so they are held to the word's precision + ex2_poly2's
# alone (measured excess 0).
RHO = 1.3e-3
# The FP32 sampler against the plain replay: |a_gpu - a_plain| <= TAU_FP32 * S (FP32 decoder and sums).  Measured max
# 3.2e-7 (case 101); TAU_FP32 is twice that.  Its decision band is TAU_FP32 * S as well.
TAU_FP32 = 6.4e-7
WORD_REL = 2.0 ** -8            # BF16 low half (round half up) or nearest word with a given low half: half a BF16 ulp, which
                                # is 2^-8 of a value at the bottom of its binade (2^-9 only at the top)
POLY_REL = 7.5e-5               # ex2_poly2
A_PLAIN = (0.05, 2e-3)          # DESIGN section 6: |a_tc - a| <= 0.05 + 2e-3 S against the FP32 weights


# ----------------------------------------------------------------------------------------------------------- inputs
def _speech(n_frames, seed=5):
    """(P [n][513] float32, IBM [n][513], mean-power bias [513]) from a synthetic utterance, frames repeated as needed."""
    x, s, _ = synth.synth_utterance(seed, 3.0)
    X, S = stft_np.stft(x, **KW), stft_np.stft(s, **KW)
    idx = np.arange(n_frames) % X.shape[1]
    P = (np.abs(X) ** 2).T[idx].astype(np.float32)
    ibm = stft_np.clean_speech_ibm(S).T[idx].astype(np.float32)
    return P, ibm, s


def _spectra(scenario, NT, rng):
    P, ibm, s = _speech(NT)
    if scenario == "nulls":
        P[:, 100:140] *= 1e-12                                          # a spectral null, 120 dB deep
        P = np.maximum(P, 1e-30)
    elif scenario == "partials":                                         # loud partials over a floor 140 dB below them
        P = rng.gamma(1.0, 1e-12, size=(NT, F)).astype(np.float32)
        P[:, 40::64] = rng.gamma(2.0, 50.0, size=P[:, 40::64].shape).astype(np.float32)
    bias = synth.speech_prior_bias(s) if scenario == "decades" else float(np.log(np.mean(P) + 1e-30))
    return P, ibm, bias


def _edge_decoder(sd, bound=119.5):
    """Hidden-2 units 0..63 saturated at +-1 (large b2) and, in every fifth bin, W3 rows of the opposite sign on those units
    only: v = -bound exactly there (BF16-exact weights), log2(e) sum_k |W3[k][f]| = bound for those bins."""
    sign = np.where(np.arange(64) % 2, 1.0, -1.0).astype(np.float32)
    sd["decoder.hidden.1.weight"][:64] *= np.float32(0.1)
    sd["decoder.hidden.1.bias"][:64] = 8.0 * sign
    bins = np.arange(0, F, 5)
    w3 = sd["decoder.reconstruction.weight"]
    w3[bins] = 0.0
    w3[np.ix_(bins, np.arange(64))] = (-sign[None, :] * np.float32(bound / 64.0 / 1.4426950408889634)).astype(np.float32)
    return bins


def _weights(labels, L, scenario, bias, seed=3):
    variant, y_dim = {"none": ("M1", 0), "y1": ("M2", 1), "ibm": ("M2", F)}[labels]
    sd = synth.xavier_state_dict(variant, F, L, [128, 128] if L == 16 else [128], y_dim, seed=seed, out_bias=bias)
    edge = _edge_decoder(sd) if scenario == "edge" else None
    return sd, variant, y_dim, edge


def _rng_dump(eng, seed, iter0, n_iter):
    b, Cc, L = eng.batch, eng.cfg.n_chains, eng.w.z_dim
    rows = b.NT * Cc
    eps = torch.empty((n_iter, rows, L), device=DEV)
    u = torch.empty((n_iter, rows), device=DEV)
    rng = _lib.DvaeRng()
    rng.seed, rng.iter0 = seed, iter0
    _lib.call("dvae_rng_dump", C.byref(rng), _p(b.frame_gid), _p(b.frame_idx), b.NT, Cc, L, n_iter, _p(eps), _p(u), _stream())
    return eps, u


def _stream_words(eng, rows):
    """The sampler's packed stream as int32 words [rows][528] (bin 4q + j = word j of quad q)."""
    pv = next(v for k, v in eng._buf.items() if k[0] == "PVpk")
    n_tiles = (rows + TM - 1) // TM
    w = pv.view(torch.int32)[: n_tiles * (NPAD // 4) * TM * 4].view(n_tiles, NPAD // 4, TM, 4)
    return w.permute(0, 2, 1, 3).reshape(n_tiles * TM, NPAD)[:rows]


def _emission(eng, rows, keep):
    """The emitted 2^v [rows][keep + 1][513] float64: bin 2i is the BF16 low half of word i, bin 2i + 1 the whole word."""
    n_tiles = (rows + TM - 1) // TM
    w = eng.VsT.view(torch.int32)[: n_tiles * (keep + 1) * 33 * TM * 8].view(n_tiles, keep + 1, 33, TM, 8)
    w = w.permute(0, 3, 1, 2, 4).reshape(n_tiles * TM, keep + 1, 33 * 8)[:rows]
    lo = ((w.to(torch.int64) << 16) & 0xFFFFFFFF).to(torch.int32).view(torch.float32)
    hi = w.contiguous().view(torch.float32)
    return torch.stack([lo, hi], dim=-1).reshape(rows, keep + 1, NPAD)[:, :, :F].double()


_TANH = []


def _tanh_table():
    """The samplers' activation over every BF16 input (dvae_tc_tanh_bf16_table), float64 [65536] by bit pattern."""
    if not _TANH:
        bits = torch.full((65536,), -1, dtype=torch.int16, device=DEV)
        _lib.call("dvae_tc_tanh_bf16_table", _p(bits), _stream())
        _TANH.append(mh_replay.bf16_from_bits(bits))
    return _TANH[0]


def test_sampler_activation_table_is_tanh_within_one_bf16_ulp():
    """tanh.approx.bf16x2 over all 65536 BF16 inputs: odd, within one BF16 ulp of the correctly rounded tanh everywhere.  It is
    not the correctly rounded tanh (which is why the mirrored decoder indexes this table instead of calling tanh)."""
    t = _tanh_table()
    x = mh_replay.bf16_from_bits(torch.arange(65536, device=DEV))
    fin = torch.isfinite(x)
    ref = mh_replay.bf16(torch.tanh(x))
    ulp = torch.exp2(torch.floor(torch.log2(ref.abs().clamp(min=2.0 ** -126))) - 7)
    err = ((t - ref).abs() / ulp)[fin]
    assert bool(torch.isfinite(t[fin]).all()) and float(err.max()) <= 1.0
    assert torch.equal(t[fin], -t[(torch.arange(65536, device=DEV) ^ 0x8000)][fin])
    print("TANH table: %d of %d finite inputs differ from the rounded tanh by one BF16 ulp" % (int((err > 0).sum()), int(fin.sum())))


# ----------------------------------------------------------------------------------------------------------- harness
RAG, RAG_IDS = [1, 150, 37, 5, 90], [7, 3, 1000, 42, 11]     # a one-frame utterance, one across the first tile boundary
SMALL, SMALL_IDS = [3, 1, 9], [5, 900, 2]                     # x16 chains: 208 rows, the last utterance across a tile
TINY = [1, 2]                                                 # x128 chains


def _run(cid, sampler, mode, emit, L, Cc, labels, scenario, keep, burn, second, lens, ids):
    rng = np.random.default_rng(17)
    NT = sum(lens)
    P_np, ibm, bias = _spectra(scenario, NT, rng)
    sd, variant, y_dim, edge = _weights(labels, L, scenario, bias)
    w = VaeWeights(sd, variant, torch.device(DEV))
    if sampler == "tc":
        tc.decoder_image(w)
        w._tc_flags = MODE_FLAGS[mode]
    P = torch.zeros((NT, LD), device=DEV)
    P[:, :F] = torch.from_numpy(P_np).to(DEV)
    if y_dim == 1:
        y = torch.from_numpy((rng.uniform(size=(NT, 1)) > 0.5).astype(np.float32)).to(DEV)
    elif y_dim:
        y = torch.from_numpy(ibm).to(DEV)
    else:
        y = None
    seed = 1234 + 7 * cid
    cfg = McemConfig(niter=1, keep_E=keep, burn_E=burn, sampler=sampler, seed=seed, n_chains=Cc)
    eng = McemEngine(w, cfg, DEV)
    eng.init_parameters(torch.zeros((NT, LD), dtype=torch.complex64, device=DEV), P, RaggedBatch(lens, DEV, utt_ids=ids), y)
    if scenario == "nulls":                     # the noise model explains the observation, the gains of some frames collapsed
        eng.Vb.copy_(P)
        eng.g[::3] = 1e-22
        eng.g[1::6] = 1e-30
    if second:                                  # a second call: the Philox iteration counter starts at mh_iter0 != 0
        eng.sample_posterior(3, 4)
    rows = NT * Cc
    n_iter = keep + burn
    Z0, n0, iter0 = eng.Z.clone(), eng.n_accept.clone(), eng.mh_iter0
    assert iter0 == (7 if second else 0)
    a_gpu = torch.full((n_iter, rows), float("nan"), device=DEV)
    Zs = eng.sample_posterior(keep, burn, a_trace=a_gpu, emit=emit).clone().view(rows, keep, L)
    if sampler == "tc":
        tc.check_status(eng)                                            # 6: no timeout, no non-finite likelihood
    eps, u = _rng_dump(eng, seed, iter0, n_iter)
    torch.cuda.synchronize()

    fr = torch.arange(rows, device=DEV) // Cc
    g = eng.g[fr]
    y_rows = None if y is None else y[fr]
    ev = {"plain": mh_replay.plain_evaluator(mh_replay.PlainDecoder(sd, DEV), P[fr, :F], eng.Vb[fr, :F], g, y_rows)}
    dec_m = None
    if sampler == "tc":
        dec_m = mh_replay.MirroredDecoder(sd, L, DEV, label_bias=w.tc_label_bias, tanh_table=_tanh_table())
        Pp, Vbp = mh_replay.decode_stream(_stream_words(eng, rows), eng.kscale[fr])
        ybias = None if eng.ybias is None else eng.ybias[fr]
        ev["mirrored"] = mh_replay.mirrored_evaluator(dec_m, Pp, Vbp, g, None if w.tc_label_bias else y_rows, ybias)

    a64 = a_gpu.double()
    logu = torch.log(u.double())
    traj_ok = torch.ones(rows, dtype=torch.bool, device=DEV)

    def decide(it, z, zp, a):
        if it >= burn:                                                  # kept: the sample is the proposal or the old state
            kept = Zs[:, it - burn]
            acc = (kept == zp).all(1)
            traj_ok.logical_and_((kept == zp).all(1) | (kept == z).all(1))
            return acc
        return logu[it] < a64[it]                                       # burn-in: from the trace

    rep = mh_replay.replay(ev, Z0, eps, eng.cfg.var_rw, burn, decide)
    S = rep["S"]
    pairs = rows * n_iter

    # 3. against the plain FP32-weight decoder: the stated tolerance of the tensor-core path (the FP32 sampler: its own bound)
    d_plain = (a64 - rep["a"]["plain"]).abs()
    if sampler == "tc":
        bound_plain = A_PLAIN[0] + A_PLAIN[1] * S
    else:
        bound_plain = 2e-4 * (1.0 + a64.abs()) + 5e-3
    ratio_plain = float((d_plain / bound_plain).max())
    if sampler == "tc":
        # 2. against the mirrored decoder; 4. decisions outside the band are float64's
        a_ref = rep["a"]["mirrored"]
        ratio = float(((a64 - a_ref).abs() / S).max())
        band = (logu - a_ref).abs() <= TAU[mode] * S
    else:
        a_ref = rep["a"]["plain"]
        ratio = float(((a64 - a_ref).abs() / S).max())
        band = (logu - a_ref).abs() <= TAU_FP32 * S
    wrong = (rep["acc"] != (logu < a_ref)) & ~band
    # 5. the emission: every slot, against the mirrored decoder's 2^v of the slot's state
    resid = edge_resid = 0.0
    if emit:
        E = _emission(eng, rows, keep)
        poly = torch.zeros(F, dtype=torch.float64, device=DEV)
        if mode == 2:
            poly[:] = POLY_REL
        elif mode == 1:
            poly[(torch.arange(F, device=DEV) % 4) >= 2] = POLY_REL
        states = [rep["Z_burn"]] + [rep["Zp"][burn + r] for r in range(keep)]
        edge_t = None if edge is None else torch.as_tensor(edge, device=DEV)
        for s_, zz in enumerate(states):
            ref = torch.exp2(dec_m.v(zz, None if w.tc_label_bias else y_rows, None if eng.ybias is None else eng.ybias[fr]))
            excess = (E[:, s_] - ref).abs() / ref - WORD_REL - poly
            resid = max(resid, float(excess.max()))
            if edge_t is not None:
                edge_resid = max(edge_resid, float(excess[:, edge_t].max()))
    print("REPLAY case=%s %s mode=%d tau_ratio=%.3e band=%d pairs=%d emit_resid=%.3e plain_ratio=%.3f wrong=%d traj_bad=%d%s"
          % (cid, sampler, mode, ratio, int(band.sum()), pairs, resid, ratio_plain, int(wrong.sum()), int((~traj_ok).sum()),
             "" if edge is None else " edge_v=%.3f edge_resid=%.3e" % (float(dec_m.v(Z0)[:, torch.as_tensor(edge, device=DEV)].max()),
                                                                     edge_resid)))

    assert torch.isfinite(a64).all()
    # 1. trajectories, accept counts, slot table
    assert bool(traj_ok.all()), "%d chains hold a kept sample that is neither the state nor the proposal" % int((~traj_ok).sum())
    assert torch.equal(rep["Zs"], Zs)
    assert torch.equal(rep["Z_end"], eng.Z)
    assert torch.equal((eng.n_accept - n0).long(), rep["n_acc"])
    if emit:
        assert torch.equal(eng.vs_idx.view(-1, 32)[:rows, :keep].long(), rep["slot"])
    # the decisions read off Zs are the sampler's own log(u) < a_gpu, up to the error of its logarithm (__logf: MUFU)
    flip = rep["acc"][burn:] != (logu[burn:] < a64[burn:])
    assert not bool((flip & ((logu[burn:] - a64[burn:]).abs() > 2.0 ** -20 * logu[burn:].abs().clamp(min=1.0))).any())
    if sampler == "tc":
        assert ratio <= TAU[mode], ratio
        assert resid <= RHO, resid
        assert edge_resid <= 0.0, edge_resid
    else:
        assert ratio <= TAU_FP32, ratio
    assert not bool(wrong.any()), "%d decisions differ from float64 outside the band" % int(wrong.sum())
    assert ratio_plain <= 1.0, ratio_plain


#       id   mode emit   L    C  labels  scenario    keep burn second batch
TC_CASES = [
    (1,   1, True,  16,   1, "none", "speech",   31,  5, False, RAG, RAG_IDS),
    (2,   0, False, 16,   1, "none", "speech",   10, 20, False, RAG, None),
    (3,   2, True,  16,   1, "none", "edge",     10,  5, False, RAG, RAG_IDS),
    (4,   1, False, 16,   3, "y1",   "speech",   10,  5, True,  RAG, RAG_IDS),
    (5,   1, True,  16,  16, "y1",   "decades",  10,  0, False, SMALL, SMALL_IDS),
    (6,   0, True,  32,   1, "none", "nulls",    10, 10, False, RAG, RAG_IDS),
    (7,   2, False, 32,  16, "y1",   "partials",  1, 10, False, SMALL, SMALL_IDS),
    (8,   1, True,  16, 128, "none", "speech",    5,  5, False, TINY, [4, 9]),
    (9,   1, True,  16,   1, "ibm",  "speech",   10, 10, True,  RAG, RAG_IDS),
    (10,  0, False, 16,  16, "ibm",  "decades",   5,  5, False, SMALL, None),
    (11,  2, True,  16,  16, "none", "nulls",    31,  0, False, SMALL, SMALL_IDS),
    (12,  1, False, 32,   1, "y1",   "partials",  1,  0, True,  RAG, RAG_IDS),
    (13,  0, True,  32, 128, "y1",   "speech",    3,  2, False, TINY, None),
    (14,  1, True,  16,   1, "none", "partials", 10, 10, False, RAG, RAG_IDS),
    (15,  2, False, 16,   3, "ibm",  "decades",  10,  5, False, RAG, RAG_IDS),
]


@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: "tc%d-poly%d-%s-L%d-C%d-%s-%s-k%d-b%d%s" % (
    c[0], c[1], "emit" if c[2] else "noemit", c[3], c[4], c[5], c[6], c[7], c[8], "-2nd" if c[9] else ""))
def test_tc_sampler_against_float64_replay(case):
    _run(case[0], "tc", *case[1:])


FP32_CASES = [
    (101, 0, False, 16,  1, "none", "speech",  10, 10, False, RAG, RAG_IDS),
    (102, 0, False, 16,  3, "y1",   "speech",   5,  5, True,  RAG, RAG_IDS),
    (103, 0, False, 16, 16, "ibm",  "decades",  5,  3, False, SMALL, SMALL_IDS),
]


@pytest.mark.parametrize("case", FP32_CASES, ids=lambda c: "fp32-C%d-%s" % (c[4], c[5]))
def test_fp32_sampler_against_float64_replay(case):
    _run(case[0], "fp32", *case[1:])


# ----------------------------------------------------------------------------------------------------------- exp2 mode
def _image_bias_log2(w):
    """The FP32 layer-3 bias (log2 domain) inside the decoder image, as the stream kernels read it."""
    off = int(_lib.load().dvae_tc_image_bias_offset(w.dec_tc.ref, w.z_dim, w.tc_y_dim))
    assert off > 0
    return tc.decoder_image(w)[off:off + 4 * F].view(torch.float32).clone()


@pytest.mark.parametrize("env,bound,want", [(None, 119.5, tc.POLY_EX2), ("0", 119.5, 0), ("1", 119.5, tc.POLY_EX2),
                                            ("2", 119.5, tc.POLY_EX2 | tc.POLY_EX2_ALL), ("2", 120.5, 0), (None, 120.5, 0)])
def test_exp2_mode_selection_and_exponent_bound(monkeypatch, env, bound, want):
    """DVAE_TC_POLY picks the share of polynomial exponentials; a decoder whose exponent bound reaches DVAE_TC_POLY_EX2_LIMIT
    runs on MUFU only whatever is asked; the bound is log2(e) max_f sum_k |W3[k][f]| (FP32 sums of 128 terms: 2e-6)."""
    if env is None:
        monkeypatch.delenv("DVAE_TC_POLY", raising=False)
    else:
        monkeypatch.setenv("DVAE_TC_POLY", env)
    sd = synth.xavier_state_dict("M1", F, 16, [128, 128], 0, seed=3, out_bias=-3.0)
    _edge_decoder(sd, bound)
    w = VaeWeights(sd, "M1", torch.device(DEV))
    got = C.c_float(0.0)
    _lib.call("dvae_tc_decoder_exponent_bound", w.dec_tc.ref, 16, 0, C.byref(got), _stream())
    ref = 1.4426950408889634 * np.abs(sd["decoder.reconstruction.weight"].astype(np.float64)).sum(1).max()
    assert abs(got.value - ref) <= 2e-6 * ref and abs(ref - bound) < 1e-4
    tc.decoder_image(w)
    assert w._tc_flags == want


# ----------------------------------------------------------------------------------------------------------- the stream
def _integer_bias(bias):
    """Per-bin FP32 b3 whose FP32 product with log2(e) is an integer in every even quad (the stream's scale 2^-b is then a
    power of two and its words are exact), the given bias elsewhere."""
    b = np.asarray(bias, np.float32).copy()
    l2e = np.float32(1.4426950408889634)
    for f in range(F):
        if (f // 4) % 2:
            continue
        n0 = float(np.rint(b[f] * l2e))
        found = None
        for n in (n0, n0 + 1, n0 - 1, n0 + 2, n0 - 2):
            x0 = np.float32(n / 1.4426950408889634)
            for d in range(-8, 9):
                x = np.float32(x0 + np.float32(d) * np.spacing(x0))
                if float(np.float32(x * l2e)) == n:
                    found = x
                    break
            if found is not None:
                break
        assert found is not None
        b[f] = found
    return b


def _bf16_bits(x32):
    return x32.to(torch.bfloat16).view(torch.int16).to(torch.int64) & 0xFFFF


def _word_with_low_half(p32, low):
    d = (p32.view(torch.int32).to(torch.int64) & 0xFFFFFFFF) - low + 0x8000
    d = d.clamp(min=0)
    w = ((d >> 16) << 16) | low
    return torch.where((w & 0x7F800000) == 0x7F800000, w - 0x10000, w)


@pytest.mark.parametrize("n_chains,ld", [(1, LD), (3, LD), (3, 521)])
def test_packed_stream_matches_float64_restatement(n_chains, ld):
    """dvae_tc_row_scale + dvae_tc_pack_pv (tiled kernel for ld % 4 == 0, generic kernel otherwise) against a float64
    restatement of the format: k = 2^-2c per frame (c = round(max_f log2(P 2^-b)) - 16 clamped to +-30, 2^15 without energy),
    word j = P' (/ k for j >= 2) with bf16(Vb') (* k for j < 2) in its low half, Vb' floored at 2^(c - 30), padding bins
    513..527 packed as the constant 1 of the quad's scale, zero words for the tail rows of the last tile."""
    lens = [1, 150, 37, 5]
    NT = sum(lens)
    rng = np.random.default_rng(23)
    P_np, _, s = _speech(NT)
    P_np[0:10] = 0.0                                                        # frames without energy
    P_np[10:60] = rng.gamma(1.0, 1e-12, size=(50, F))                       # loud partials 140 dB over the floor
    P_np[10:60, 40::64] = rng.gamma(2.0, 50.0, size=(50, len(range(40, F, 64))))
    P_np[60] = 1e12                                                         # c clamped at +30
    P_np[61] = 1e-30                                                        # c clamped at -30
    bias = _integer_bias(synth.speech_prior_bias(s))                        # spans > 5 decades
    sd = synth.xavier_state_dict("M1", F, 16, [128, 128], 0, seed=3, out_bias=bias)
    w = VaeWeights(sd, "M1", torch.device(DEV))
    eng = McemEngine(w, McemConfig(niter=1, sampler="tc", n_chains=n_chains), DEV)
    P = torch.zeros((NT, LD), device=DEV)
    P[:, :F] = torch.from_numpy(P_np.astype(np.float32)).to(DEV)
    eng.init_parameters(torch.zeros((NT, LD), dtype=torch.complex64, device=DEV), P, RaggedBatch(lens, DEV), None)
    Vb = eng.Vb.clone()
    Vb[62:90, 200:260] = 1e-35                                              # noise variance far below the floor
    Pl = torch.zeros((NT, ld), device=DEV)
    Vl = torch.zeros((NT, ld), device=DEV)
    Pl[:, :F], Vl[:, :F] = P[:, :F], Vb[:, :F]
    img = tc.decoder_image(w)
    b = _image_bias_log2(w).double()
    integer_b = b == torch.round(b)
    assert int(integer_b.sum()) >= 256

    k = torch.full((NT,), -1.0, device=DEV)
    _lib.call("dvae_tc_row_scale", w.dec_tc.ref, _p(img), 16, 0, _p(Pl), NT, F, ld, _p(k), _stream())
    P64 = P[:, :F].double()
    lp = torch.where(P64 > 0, torch.log2(P64) - b, torch.full_like(P64, -torch.inf))
    top = lp.max(1).values
    energy = torch.isfinite(top)
    c = (torch.round(top) - 16).clamp(-30, 30)
    k_ref = torch.where(energy, torch.exp2(-2 * c), torch.full_like(top, 32768.0))
    near = (top - torch.floor(top) - 0.5).abs() < 1e-5
    assert torch.equal((k.double() == k_ref) | near, torch.ones_like(near))
    assert bool((k[~energy] == 32768.0).all()) and float(k[60]) == 2.0 ** -60 and float(k[61]) == 2.0 ** 60
    assert int((~energy).sum()) == 10

    chains = NT * n_chains
    n_tiles = (chains + TM - 1) // TM
    nbytes = int(_lib.load().dvae_tc_packed_pv_bytes(chains))
    buf = torch.full((nbytes + 4096,), 0xA5, dtype=torch.uint8, device=DEV)
    _lib.call("dvae_tc_pack_pv", w.dec_tc.ref, _p(img), 16, 0, _p(Pl), _p(Vl), _p(k), NT, n_chains, F, ld, _p(buf), _stream())
    assert bool((buf[nbytes:] == 0xA5).all()), "the packer wrote past the stream"
    words = buf[:nbytes].view(torch.int32).view(n_tiles, NPAD // 4, TM, 4).permute(0, 2, 1, 3).reshape(n_tiles * TM, NPAD)
    words = words.to(torch.int64) & 0xFFFFFFFF
    assert bool((words[chains:] == 0).all()), "tail rows of the last tile must be zero words"
    words = words[:chains]

    fr = torch.arange(chains, device=DEV) // n_chains
    kk = k.double()[fr][:, None]
    level = kk.rsqrt()
    j = torch.arange(NPAD, device=DEV) % 4
    lowq = j[None, :F] < 2
    sc = torch.exp2(-b)[None, :]
    pj = P64[fr] * sc * torch.where(lowq, 1.0, 1.0 / kk)
    vf = torch.maximum(Vb[fr, :F].double() * sc, level * 2.0 ** -30)
    vj = vf * torch.where(lowq, kk, 1.0)
    v32 = vj.to(torch.float32)
    low_ref = _bf16_bits(v32)
    low = words[:, :F] & 0xFFFF
    # bins whose 2^-b is not a power of two: the kernel's exp2f and FP32 products are a few FP32 ulps off the float64
    # value, which can move a value within 2^-20 of a BF16 rounding midpoint to the other side
    mid = ((v32.view(torch.int32).to(torch.int64) & 0xFFFF) - 0x8000).abs() <= 16
    exact = integer_b[None, :].expand_as(low)
    assert torch.equal(low[exact], low_ref[exact])
    assert bool(((low == low_ref) | (mid & ((low - low_ref).abs() <= 1)))[~exact].all())
    w_ref = _word_with_low_half(pj.to(torch.float32), low)                # the nearest word with the kernel's own low half
    assert torch.equal(words[:, :F][exact], w_ref[exact])
    assert bool((((words[:, :F] >> 16) - (w_ref >> 16)).abs() <= 1).all())
    # floored bins carry exactly the floor 2^(c - 30) (times k in bins 0, 1 of a quad)
    floored = Vb[fr, :F].double() * sc < level * 2.0 ** -30
    assert int(floored.sum()) > 0 and torch.equal(low[floored & exact], _bf16_bits((level * 2.0 ** -30 * torch.where(lowq, kk, 1.0)).expand_as(vj).to(torch.float32))[floored & exact])
    # padding bins 513..527: P' = 0 and the constant 1 of the quad's scale (k Vb' = k^(1/2) in bins 0, 1, Vb' = k^(-1/2) in 2, 3)
    jp = j[None, F:]
    pad_ref = _bf16_bits(torch.where(jp < 2, kk.sqrt(), level).expand(chains, NPAD - F).to(torch.float32))
    assert torch.equal(words[:, F:], _word_with_low_half(torch.zeros_like(pad_ref, dtype=torch.float32), pad_ref))
    # chains of a frame share the frame's words
    if n_chains > 1:
        per = words.view(NT, n_chains, NPAD)
        assert bool((per == per[:, :1]).all())
