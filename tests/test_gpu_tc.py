"""Tensor-core (tcgen05 BF16) decoder path against the FP32 CUDA path and the oracle.

Stated tolerance of the BF16 path (weights and hidden activations rounded to BF16, FP32 accumulation, MUFU
approximations for tanh / exp2 / log2 / reciprocal): decoder outputs within 1 % relative, log-acceptance values
within 0.05 absolute of FP32, enhanced-speech SI-SDR within 0.05 dB (BASELINE.json north star).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth, tc
from dvae_b200.engine import (Enhancer, InjectedDraws, McemConfig, McemEngine, RaggedBatch, VaeWeights, _p, _stream,
                              mlp_forward)
from oracle import mcem_port, stft_np
from tests.golden_io import Golden
from tests.gpu_util import DEV, engine_for, golden_draws, unfm

pytestmark = pytest.mark.gpu
KW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
IKW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False)


def test_decoder_image_layout():
    """The packed image is the documented K-major 128B-swizzled BF16 layout (checked element by element)."""
    g = Golden("full_M2")
    w = VaeWeights(g.sd, "M2", torch.device(DEV))
    img = tc.decoder_image(w).cpu().numpy()
    L, y_dim, HID, NPAD = 16, 1, 128, 528

    def elem(base, rows, n, k):
        off = base + (k >> 6) * rows * 128 + n * 128 + ((((k & 63) >> 3) ^ (n & 7)) << 4) + (k & 7) * 2
        return torch.tensor(img[off:off + 2].copy()).view(torch.bfloat16).float().item()

    def bf(x):
        return torch.tensor(np.float32(x)).to(torch.bfloat16).float().item()

    W1, b1 = g.sd["decoder.hidden.0.weight"], g.sd["decoder.hidden.0.bias"]
    W2 = g.sd["decoder.hidden.1.weight"]
    W3, b3 = g.sd["decoder.reconstruction.weight"], g.sd["decoder.reconstruction.bias"]
    for n, k in ((0, 0), (5, 3), (127, 15)):
        assert elem(0, HID, n, k) == bf(W1[n, k]) and elem(0, HID, n, k + L) == bf(W1[n, k])
    assert elem(0, HID, 9, 2 * L) == bf(W1[9, L]) and elem(0, HID, 9, 2 * L + 1) == bf(W1[9, L])
    assert elem(0, HID, 9, 2 * L + 2) == bf(b1[9]) and elem(0, HID, 9, 2 * L + 3) == 0.0
    for n, k in ((0, 0), (77, 100), (127, 127)):
        assert elem(16384, HID, n, k) == bf(W2[n, k])
    log2e = np.float32(1.4426950408889634)
    for n, k in ((0, 0), (300, 64), (512, 127)):
        assert elem(16384 + 32768, NPAD, n, k) == bf(W3[n, k] * log2e)
    assert elem(16384 + 32768, NPAD, 513, 7) == 0.0
    bias = np.frombuffer(img[16384 + 32768 + 2 * NPAD * 128:].tobytes(), np.float32)
    np.testing.assert_allclose(bias[:128], g.sd["decoder.hidden.1.bias"])
    np.testing.assert_allclose(bias[128:128 + 513], b3 * log2e, rtol=1e-6)


@pytest.mark.parametrize("variant,L,h", [("M1", 16, [128, 128]), ("M2", 16, [128, 128]), ("M1", 32, [128])])
def test_decode_tc_within_one_percent_of_fp32(variant, L, h):
    y_dim = 0 if variant == "M1" else 1
    sd = synth.xavier_state_dict(variant, 513, L, h, y_dim, seed=7, out_bias=-3.0)
    w = VaeWeights(sd, variant, torch.device(DEV))
    rows, div = 2000, 25                                   # 15.6 tiles: exercises the partial last tile
    x = torch.randn((rows, L), device=DEV, generator=torch.Generator(device=DEV).manual_seed(0))
    y = (torch.rand((rows // div, 1), device=DEV) > 0.5).float() if y_dim else None
    ref = mlp_forward(w.dec, x, _lib.ACT_EXP, x2=y, x2_row_div=div)
    out = torch.full((rows + 3, 520), -1.0, device=DEV)
    st = torch.zeros(1, dtype=torch.int32, device=DEV)
    _lib.call("dvae_decode_tc", w.dec.ref, _p(tc.decoder_image(w)), _p(x), rows, L, _p(y), y_dim, None, div, _p(out), 520, _p(st), _stream())
    assert int(st.item()) == 0
    rel = ((out[:rows, :513] - ref) / ref).abs()
    assert rel.max().item() <= 1e-2 and rel.mean().item() <= 2e-3
    assert torch.all(out[rows:] == -1.0) and torch.all(out[:rows, 513:] == -1.0)      # nothing written out of bounds


@pytest.mark.parametrize("name", ["full_M1", "full_M2", "full_M2v3", "cfg1_M1"])
def test_sampler_tc_log_acceptance_vs_oracle(name):
    g = Golden(name)
    o = mcem_port.MCEMOracle(g.variant, g.niter, *g.sched, g.var_RW, draws=mcem_port.ReplayDraws(g.draws))
    o.init_parameters(g.X, g.S, g.sd, g.K, g.eps, y=g.y)
    (kE, bE), _ = o.schedule()
    o.taps = []
    o.sample_posterior(o.Z, kE, bE)
    eng, X, P, y, batch = engine_for(g, o.schedule(), sampler="tc")
    draws = golden_draws(g, o.schedule())
    eng.init_parameters(X, P, batch, y, draws)
    N = g.X.shape[1]
    a = torch.zeros((kE + bE, N), device=DEV)
    eng.sample_posterior(kE, bE, draws, a_trace=a)
    a = a.cpu().numpy()
    tc.check_status(eng)
    same = np.ones(N, bool)
    n_dec = n_flip = 0
    Pt = torch.tensor(np.abs(g.X) ** 2)
    for it, tap in enumerate(o.taps):
        a_ref = tap["a"].numpy()
        # a 1 % error of a decoder output moves its log-likelihood term by 1 % of (1 + P/Vx): scale the bound with it
        Vx = o.g * o._decode_cols(tap["Z"]) + o.Vb
        Vxp = o.g * o._decode_cols(tap["Zp"]) + o.Vb
        scale = (2.0 + Pt / Vx + Pt / Vxp).sum(0).numpy()
        assert np.all(np.abs(a[it] - a_ref)[same] <= 0.05 + 2e-3 * scale[same]), "iteration %d" % it
        acc_gpu = np.log(tap["u"].numpy()) < a[it]
        n_dec += int(same.sum())
        n_flip += int((same & (acc_gpu != tap["acc"].numpy())).sum())
        same &= acc_gpu == tap["acc"].numpy()
    assert n_flip <= max(2, int(0.03 * n_dec)), "%d of %d decisions flipped" % (n_flip, n_dec)


@pytest.mark.parametrize("name", ["full_M1", "full_M2", "full_M2v3", "cfg1_M1"])
def test_full_run_tc_against_reference_golden(name):
    g = Golden(name)
    sched = mcem_port.MCEMOracle(g.variant, g.niter, *g.sched).schedule()
    eng, X, P, y, batch = engine_for(g, sched, sampler="tc")
    draws = golden_draws(g, sched)
    eng.init_parameters(X, P, batch, y, draws)
    cost = eng.run(draws).cpu().numpy()[:, 0]
    tc.check_status(eng)
    S_hat = unfm(eng.S_hat, g.F)
    np.testing.assert_allclose(cost, g.ref["cost"], rtol=3e-2)
    assert np.linalg.norm(S_hat - g.ref["S_hat"]) / np.linalg.norm(g.ref["S_hat"]) <= 8e-2


def test_tc_si_sdr_within_0p05_db_of_oracle_and_fp32():
    from dvae_b200.packages.models import mcem as shim_mcem
    from dvae_b200.packages.models import models as shim_models
    from dvae_b200.packages.processing.stft import istft
    x, s, _ = synth.synth_utterance(21, 1.0)
    X_ref, S_ref = stft_np.stft(x, **KW), stft_np.stft(s, **KW)
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=3, out_bias=synth.speech_prior_bias(s))
    niter = 12
    torch.manual_seed(77)
    o = mcem_port.MCEMOracle("M1", niter, 10, 30, 25, 75, 0.01)
    o.init_parameters(X_ref, S_ref, sd, 10, 1e-8)
    o.run()
    s_ref = stft_np.istft(o.S_hat, max_len=len(x), **IKW)
    ref = mcem_port.si_sdr(s_ref[800:-800], s[800:-800])
    base = mcem_port.si_sdr(x[800:-800], s[800:-800])
    assert ref > base + 1.0, "the synthetic speech prior should enhance (%.2f -> %.2f dB)" % (base, ref)
    model = shim_models.VariationalAutoencoder([513, 16, [128, 128]])
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    model.to(DEV).eval()
    sdr = {}
    for sampler in ("fp32", "tc"):
        algo = shim_mcem.MCEM_M1(niter, 10, 30, 25, 75, 0.01, rng="torch", sampler=sampler)
        torch.manual_seed(77)                                  # the reference's own draw order, same numbers
        algo.init_parameters(X=X_ref, S=S_ref, vae=model, nmf_rank=10, eps=1e-8, device=0)
        algo.run()
        s_hat = istft(algo.S_hat, max_len=len(x), **IKW)
        sdr[sampler] = mcem_port.si_sdr(s_hat[800:-800], s[800:-800])
    assert abs(sdr["tc"] - ref) <= 0.05 and abs(sdr["fp32"] - ref) <= 0.05, (sdr, ref, base)


@pytest.mark.parametrize("variant", ["M1", "M2", "M2v3"])
def test_tc_at_the_benchmark_configuration_against_the_oracle(variant):
    """bench.py's workload for one utterance: 3 s, 100 EM iterations, the reference's MH schedule (M1: 60 / 30 and 105 / 75;
    M2*: 40 / 10 and 100 / 25), sampler="tc" (sampler emission, BF16 variances), against the CPU oracle on the SAME draws
    (torch CPU generator in the reference's consumption order).  North star: SI-SDR within 0.05 dB; cost curve within 2 %."""
    from dvae_b200.packages.models import mcem as shim_mcem
    from dvae_b200.packages.models import models as shim_models
    from dvae_b200.packages.processing.stft import istft
    x, s, _ = synth.synth_utterance(1003, 3.0)
    X_ref, S_ref = stft_np.stft(x, **KW), stft_np.stft(s, **KW)
    y_dim = 0 if variant == "M1" else 1
    y = synth.energy_vad(s) if y_dim else None
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=1234, out_bias=synth.speech_prior_bias(s))
    niter = 100
    torch.manual_seed(2024)
    o = mcem_port.MCEMOracle(variant, niter, 10, 30, 25, 75, 0.01)
    o.init_parameters(X_ref, S_ref, sd, 10, 1e-8, y=y)
    cost_ref = o.run()
    s_ref = stft_np.istft(o.S_hat, max_len=len(x), **IKW)
    ref = mcem_port.si_sdr(s_ref[800:-800], s[800:-800])
    base = mcem_port.si_sdr(x[800:-800], s[800:-800])
    assert ref > base + 1.0, "the synthetic speech prior should enhance (%.2f -> %.2f dB)" % (base, ref)
    if variant == "M1":
        model, cls = shim_models.VariationalAutoencoder([513, 16, [128, 128]]), shim_mcem.MCEM_M1
    elif variant == "M2":
        model, cls = shim_models.DeepGenerativeModel([513, 1, 16, [128, 128]], None), shim_mcem.MCEM_M2
    else:
        model, cls = shim_models.DeepGenerativeModel_v3([513, 1, 16, [128, 128]]), shim_mcem.MCEM_M2v3
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()}, strict=False)
    model.to(DEV).eval()
    algo = cls(niter, 10, 30, 25, 75, 0.01, rng="torch", sampler="tc")
    torch.manual_seed(2024)
    kw = dict(X=X_ref, S=S_ref, vae=model, nmf_rank=10, eps=1e-8, device=0)
    if y_dim:
        kw["y"] = torch.tensor(y, device=DEV)
    algo.init_parameters(**kw)
    cost = algo.run()
    assert algo._engine.cfg.sampler == "tc" and ("VsT", ) == tuple(k[0] for k in algo._engine._buf if k[0] == "VsT")   # the E-steps used the sampler's emission
    s_hat = istft(algo.S_hat, max_len=len(x), **IKW)
    got = mcem_port.si_sdr(s_hat[800:-800], s[800:-800])
    assert abs(got - ref) <= 0.05, (got, ref, base)
    np.testing.assert_allclose(cost, cost_ref, rtol=2e-2)
    # the lazily exposed variances of the filter samples have the reference's shapes (mcem.py:29-34)
    R_wf = 75 if variant == "M1" else 25
    assert tuple(algo.Vs.shape) == (R_wf, 513, X_ref.shape[1]) and tuple(algo.Vx.shape) == tuple(algo.Vs.shape)


def test_tc_rejects_unsupported_shapes():
    sd = synth.xavier_state_dict("M1", 257, 16, [128, 128], 0)
    w = VaeWeights(sd, "M1", torch.device(DEV))
    with pytest.raises(ValueError):
        tc.decoder_image(w)
    sd = synth.xavier_state_dict("M1", 513, 16, [64, 64], 0)
    with pytest.raises(ValueError):
        tc.decoder_image(VaeWeights(sd, "M1", torch.device(DEV)))


@pytest.mark.parametrize("variant,keep", [("M1", 30), ("M2", 10), ("M2v3", 10)])
def test_stats_and_emit_routes_match_decode_route(variant, keep):
    """The three E-step routes (``McemEngine.route``) on the same Philox draws: (a) "decode": decode_tc + the W kernel that
    reads Vs, (b) "stats": dvae_decode_stats_tc (FP32 Vs + frame statistics in one pass), (c) "emit": the sampler's own BF16
    emission + dvae_vst_w_partials or dvae_vst_frame_stats + dvae_nmf_mstep_vst.  (b) must equal (a) to FP32 rounding; (c)
    carries the BF16 rounding of the stored variances (2^-9 relative per value + the sampler's polynomial exp2: stated
    tolerance 1.2 % per variance of the first E-step, where all three hold the same samples, and 2 % relative L2 on the M-step
    outputs of this two-iteration run, whose second E-step may already take a different accept decision here and there)."""
    y_dim = 0 if variant == "M1" else 1
    lens = [185, 37, 1, 64]                                     # ragged: partial tiles, one-frame utterance
    NT = sum(lens)
    rng = np.random.default_rng(11)
    P = torch.tensor(rng.gamma(1.0, 0.05, size=(NT, 520)).astype(np.float32)).to(DEV)
    X = torch.zeros((NT, 520), dtype=torch.complex64, device=DEV)
    y = (torch.rand((NT, 1), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4)) > 0.5).float() if y_dim else None
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=9, out_bias=float(np.log(0.05)))
    w = VaeWeights(sd, variant, torch.device(DEV))
    out = {}
    for mode, route in (("decode", "decode"), ("stats", "stats"), ("emit", "emit"), ("emit_a1a2", "emit")):
        cfg = McemConfig(niter=2, keep_E=keep, burn_E=5, keep_WF=3, burn_WF=3, sampler="tc", seed=3, w_partials=(mode == "emit"))
        eng = McemEngine(w, cfg, DEV)
        assert eng.route == "emit"                              # what these shapes run; the other routes are forced
        eng.route = route
        eng.init_parameters(X, P, RaggedBatch(lens, DEV), y)
        for it in range(2):
            eng.e_step()
            assert ((eng.wstat is not None) or (eng.wpart is not None)) == (route != "decode") and (eng.VsT is not None) == (route == "emit") and (eng.wpart is not None) == (mode == "emit")
            if it == 0:
                vs = eng.Vs.clone()
            eng.m_step(it)
        tc.check_status(eng)
        out[mode] = (vs.cpu(), eng.W.cpu().clone(), eng.H.cpu().clone(), eng.g.cpu().clone(), eng.cost.cpu().clone())
    a = out["decode"]
    for i in (1, 2, 3, 4):                            # the two W reductions of the emission path differ by summation order only
        assert ((out["emit"][i] - out["emit_a1a2"][i]).double().norm() / out["emit_a1a2"][i].double().norm()).item() <= 1e-5
    for mode, tol_vs, tol in (("stats", 1e-5, 1e-4), ("emit", 1.2e-2, 2e-2)):
        b = out[mode]
        assert ((a[0][:, :, :513] - b[0][:, :, :513]).abs() / a[0][:, :, :513]).max().item() <= tol_vs, mode
        for i, name in ((1, "W"), (2, "H"), (3, "g"), (4, "cost")):
            ref = a[i][..., :513] if i == 1 else a[i]
            got = b[i][..., :513] if i == 1 else b[i]
            if mode == "stats":
                err = ((got - ref).abs().max() / ref.abs().max()).item()
            else:
                err = ((got - ref).double().norm() / ref.double().norm()).item()
            assert err <= tol, "%s: %s differs by %g" % (mode, name, err)


@pytest.mark.parametrize("variant,keep,chains", [("M2v3", 10, 16), ("M2", 10, 2), ("M1", 30, 4)])
def test_multi_chain_emit_route_matches_stats_route(variant, keep, chains):
    """Several chains per frame, "emit" route against "stats" route: the sampler's emission + dvae_vst_w_partials + the
    windowed emission M-step kernel against the windowed FP32 decode (dvae_decode_stats_win_tc) + its M-step kernel on the
    same Philox draws.  The first E-step holds the same samples on both paths (BF16 storage: 1.2 % per variance); M-step
    outputs after it within 0.5 % relative L2, after a second iteration (accept decisions may differ here and there) within
    2 %."""
    y_dim = 0 if variant == "M1" else 1
    lens = [70, 37, 1, 20]
    NT = sum(lens)
    rng = np.random.default_rng(12)
    P = torch.tensor(rng.gamma(1.0, 0.05, size=(NT, 520)).astype(np.float32)).to(DEV)
    X = torch.zeros((NT, 520), dtype=torch.complex64, device=DEV)
    y = (torch.rand((NT, 1), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4)) > 0.5).float() if y_dim else None
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=9, out_bias=float(np.log(0.05)))
    w = VaeWeights(sd, variant, torch.device(DEV))
    out = {}
    for route in ("stats", "emit"):
        cfg = McemConfig(niter=2, keep_E=keep, burn_E=5, keep_WF=3, burn_WF=3, sampler="tc", seed=3, n_chains=chains)
        eng = McemEngine(w, cfg, DEV)
        assert eng.route == "emit"
        eng.route = route
        eng.init_parameters(X, P, RaggedBatch(lens, DEV), y)
        snap = []
        for it in range(2):
            eng.e_step()
            emit = route == "emit"
            assert (eng.VsT is not None) == emit and (eng.wpart is not None) == emit and (eng.wstat is not None) != emit and eng.R == chains * keep
            if it == 0:
                vs = eng.Vs.clone()
                assert tuple(vs.shape) == (NT, chains * keep, 520)
            eng.m_step(it)
            snap.append([t.cpu().clone() for t in (eng.W[..., :513], eng.H, eng.g, eng.Vb[:, :513], eng.cost[it])])
        tc.check_status(eng)
        out[route] = (vs.cpu(), snap)
    a, b = out["stats"], out["emit"]
    assert ((a[0][:, :, :513] - b[0][:, :, :513]).abs() / a[0][:, :, :513]).max().item() <= 1.2e-2
    for it, tol in ((0, 5e-3), (1, 2e-2)):
        for name, ref, got in zip(("W", "H", "g", "Vb", "cost"), a[1][it], b[1][it]):
            err = ((got - ref).double().norm() / ref.double().norm()).item()
            assert err <= tol, "iteration %d: %s differs by %g" % (it, name, err)


def test_sampler_handles_decoder_biases_spanning_many_decades():
    """A decoder whose output bias is tiny in part of the spectrum (a prior without energy above 3 kHz: exp(b3) ~ 1e-10 there)
    makes the sampler's bias-free variances X = Vx exp(-b3) huge in those bins.  With a fixed quad scale the four-fold products
    of the likelihood overflowed, l(z') became Inf and the affected chains never moved; the per-frame scale of
    dvae_tc_row_scale keeps them finite: no status bit, and the chains accept as often as the exact FP32 sampler's."""
    x, s, _ = synth.synth_utterance(5, 1.0)
    bias = synth.speech_prior_bias(s)
    assert bias.min() < -20.0 and bias.max() > -8.0                      # > 5 decades between bins
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=3, out_bias=bias)
    X = stft_np.stft(x, **KW)
    N = X.shape[1]
    P = torch.zeros((N, 520), device=DEV)
    P[:, :513] = torch.from_numpy(np.ascontiguousarray((np.abs(X) ** 2).T)).to(DEV)
    rate = {}
    for sampler in ("fp32", "tc"):
        w = VaeWeights(sd, "M1", torch.device(DEV))
        eng = McemEngine(w, McemConfig(niter=2, keep_E=10, burn_E=20, sampler=sampler, seed=4), DEV)
        eng.init_parameters(torch.zeros((N, 520), dtype=torch.complex64, device=DEV), P, RaggedBatch([N], DEV, utt_ids=[9]))
        for it in range(2):
            eng.e_step()
            eng.m_step(it)
        if sampler == "tc":
            tc.check_status(eng)                                         # neither a timeout nor a non-finite likelihood
            k = eng.kscale.cpu().numpy()
            assert np.all(k > 0) and np.all(np.log2(k) == np.rint(np.log2(k))) and k.min() < 1.0     # powers of two, far from 2^15
        rate[sampler] = float(eng.n_accept.sum().item()) / (N * 60)
        assert bool(torch.isfinite(eng.cost).all())
    assert rate["fp32"] > 0.3 and abs(rate["tc"] - rate["fp32"]) <= 0.03, rate


def test_sampler_and_cost_survive_collapsed_gains_and_spectral_nulls():
    """Late in a run the NMF explains noise-only frames alone: the gain g of such a frame collapses by many decades, and in
    spectral nulls both the observation and Vb lie far below the frame's level.  The sampler's quad products (four bins, including
    the observation-free padding bins whose variance is g alone) and the cost pass's products of four samples must stay finite:
    no status bit, finite cost, and the chains of those frames accept like the exact FP32 sampler's (their likelihood hardly
    depends on z: almost every proposal is accepted).  The first version of the quad trick produced NaN here (bench run, after
    ~100 EM iterations)."""
    x, s, _ = synth.synth_utterance(5, 1.0)
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=3, out_bias=float(np.log(0.05)))
    X = stft_np.stft(x, **KW)
    N = X.shape[1]
    P = torch.zeros((N, 520), device=DEV)
    P[:, :513] = torch.from_numpy(np.ascontiguousarray((np.abs(X) ** 2).T)).to(DEV)
    P[:, 100:140] *= 1e-12                                               # a spectral null, 120 dB deep
    P[:, :513].clamp_(min=1e-30)
    rate = {}
    for sampler in ("fp32", "tc"):
        w = VaeWeights(sd, "M1", torch.device(DEV))
        eng = McemEngine(w, McemConfig(niter=2, keep_E=10, burn_E=20, sampler=sampler, seed=4), DEV)
        eng.init_parameters(torch.zeros((N, 520), dtype=torch.complex64, device=DEV), P, RaggedBatch([N], DEV, utt_ids=[9]))
        for it in range(2):
            eng.Vb.copy_(P)                                              # the noise model explains the observation alone ...
            eng.g[::3] = 1e-22                                           # ... and the gain of every third frame has collapsed
            eng.g[1::6] = 1e-30
            eng.e_step()
            if sampler == "tc":
                tc.check_status(eng)                                     # neither a timeout nor a non-finite likelihood
            eng.m_step(it)
        if sampler == "tc":
            tc.check_status(eng)
        assert bool(torch.isfinite(eng.cost).all()), eng.cost
        acc = eng.n_accept.view(-1).float()
        rate[sampler] = (float(acc[::3].sum().item()) / (len(acc[::3]) * 60), float(acc.sum().item()) / (N * 60))
    assert rate["fp32"][0] > 0.5 and abs(rate["tc"][0] - rate["fp32"][0]) <= 0.05, rate
    assert abs(rate["tc"][1] - rate["fp32"][1]) <= 0.05, rate


def test_sampler_handles_140_db_of_dynamic_range_inside_a_frame():
    """Frames with a few loud partials over a floor 140 dB below them (a quiet room with a tonal source; 16-bit material reaches
    96 dB).  The geometric mean of such a frame sits near the floor, so a scale centred on it overflowed the four-fold product at
    the partials; centred 16 octaves below the loudest bin, with the Vb' floor underneath, everything stays finite and the chains
    accept like the exact FP32 sampler's."""
    rng = np.random.default_rng(3)
    N = 96
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=3, out_bias=float(np.log(0.05)))
    Pn = rng.gamma(1.0, 1e-12, size=(N, 513)).astype(np.float32)
    Pn[:, 40::64] = rng.gamma(2.0, 50.0, size=Pn[:, 40::64].shape).astype(np.float32)       # eight partials per frame
    P = torch.zeros((N, 520), device=DEV)
    P[:, :513] = torch.from_numpy(Pn).to(DEV)
    rate = {}
    for sampler in ("fp32", "tc"):
        w = VaeWeights(sd, "M1", torch.device(DEV))
        eng = McemEngine(w, McemConfig(niter=3, keep_E=10, burn_E=20, sampler=sampler, seed=4), DEV)
        eng.init_parameters(torch.zeros((N, 520), dtype=torch.complex64, device=DEV), P, RaggedBatch([N], DEV, utt_ids=[9]))
        for it in range(3):
            eng.e_step()
            if sampler == "tc":
                tc.check_status(eng)
            eng.m_step(it)
        if sampler == "tc":
            tc.check_status(eng)
        assert bool(torch.isfinite(eng.cost).all()), eng.cost
        rate[sampler] = float(eng.n_accept.sum().item()) / (N * 90)
    assert abs(rate["tc"] - rate["fp32"]) <= 0.05, rate
