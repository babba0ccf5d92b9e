"""End-to-end parity: the CUDA path against the reference's golden outputs and against the oracle.

Bit parity over a whole run is not attainable (a Metropolis-Hastings accept is a discontinuous function of an FP32
sum; one flipped decision decorrelates that frame's chain, SURVEY §7.3), so whole runs are judged on what the
north star names: enhanced-speech SI-SDR within 0.05 dB, plus the cost curve and the model parameters to a few percent.
"""
import numpy as np
import pytest
import torch

from dvae_b200 import synth
from oracle import mcem_port, stft_np
from tests.golden_io import Golden
from tests.gpu_util import DEV, engine_for, golden_draws, relerr, unfm

pytestmark = pytest.mark.gpu
KW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
IKW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False)


@pytest.mark.parametrize("name", ["tiny_M1", "tiny_M2", "tiny_M2v2", "tiny_M2v3", "full_M1", "full_M2", "full_M2v3", "cfg1_M1"])
def test_full_run_against_reference_golden(name):
    g = Golden(name)
    sched = mcem_port.MCEMOracle(g.variant, g.niter, *g.sched).schedule()
    eng, X, P, y, batch = engine_for(g, sched)
    draws = golden_draws(g, sched)
    eng.init_parameters(X, P, batch, y, draws)
    cost = eng.run(draws).cpu().numpy()[:, 0]
    F = g.F
    S_hat, N_hat = unfm(eng.S_hat, F), unfm(eng.N_hat, F)
    assert tuple(g.ref["Vs_shape"]) == (eng.R_wf, F, g.X.shape[1])
    np.testing.assert_allclose(cost, g.ref["cost"], rtol=2e-2)
    # relative L2 error of the estimates; a handful of flipped accepts moves single frames only
    def l2(a, b):
        return np.linalg.norm(a - b) / np.linalg.norm(b)
    assert l2(S_hat, g.ref["S_hat"]) <= 5e-2
    assert l2(N_hat, g.ref["N_hat"]) <= 5e-2
    assert l2(eng.W[0, :, :F].t().cpu().numpy(), g.ref["W"]) <= 5e-2
    assert l2(eng.H.t().cpu().numpy(), g.ref["H"]) <= 5e-2
    assert l2(eng.g.cpu().numpy(), g.ref["g"]) <= 5e-2
    # S_hat + N_hat = X * (mean Vs/Vx + mean Vb/Vx) = X exactly in real arithmetic
    assert relerr(S_hat + N_hat, g.X) <= 1e-5


def _si_sdr(est, ref):
    return mcem_port.si_sdr(est[800:-800], ref[800:-800])


@pytest.mark.parametrize("variant", ["M1", "M2", "M2v3"])
def test_dropin_si_sdr_within_0p05_db_of_oracle(variant):
    """The reference-signature classes with the reference's own draw order vs the oracle on a synthetic utterance."""
    from dvae_b200.packages.models import mcem as shim_mcem
    from dvae_b200.packages.models import models as shim_models
    from dvae_b200.packages.processing.stft import istft, stft
    x, s, _ = synth.synth_utterance(21, 1.0)
    X_ref, S_ref = stft_np.stft(x, **KW), stft_np.stft(s, **KW)
    X = stft(x, **KW)
    S = stft(s, **KW)
    F, N = X.shape
    y = synth.energy_vad(s) if variant != "M1" else None
    sd = synth.xavier_state_dict(variant, F, 16, [128, 128], 0 if variant == "M1" else 1, seed=3,
                                 out_bias=synth.speech_prior_bias(s))
    niter = 12
    # oracle
    torch.manual_seed(77)
    o = mcem_port.MCEMOracle(variant, niter, 10, 30, 25, 75, 0.01)
    o.init_parameters(X_ref, S_ref, sd, 10, 1e-8, y=y)
    cost_ref = o.run()
    s_ref = stft_np.istft(o.S_hat, max_len=len(x), **IKW)
    # drop-in
    if variant == "M1":
        model = shim_models.VariationalAutoencoder([F, 16, [128, 128]])
        algo = shim_mcem.MCEM_M1(niter, 10, 30, 25, 75, 0.01, rng="torch", sampler="fp32")
    elif variant == "M2":
        model = shim_models.DeepGenerativeModel([F, 1, 16, [128, 128]], None)
        algo = shim_mcem.MCEM_M2(niter, 10, 30, 25, 75, 0.01, rng="torch", sampler="fp32")
    else:
        model = shim_models.DeepGenerativeModel_v5([F, 1, 16, [128, 128]]).enc_dec_clf
        algo = shim_mcem.MCEM_M2v3(niter, 10, 30, 25, 75, 0.01, rng="torch", sampler="fp32")
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()}, strict=False)
    model.to(DEV).eval()
    torch.manual_seed(77)
    if variant == "M1":
        algo.init_parameters(X=X, S=S, vae=model, nmf_rank=10, eps=1e-8, device=0)
    else:
        algo.init_parameters(X=X, S=S, y=torch.tensor(y).to(DEV), vae=model, nmf_rank=10, eps=1e-8, device=0)
    cost = algo.run()
    assert cost.shape == (niter,) and cost.dtype == np.float64
    assert algo.S_hat.shape == (F, N) and algo.S_hat.dtype == np.complex64
    s_hat = istft(algo.S_hat, max_len=len(x), **IKW)
    d = abs(_si_sdr(s_hat, s) - _si_sdr(s_ref, s))
    assert d <= 0.05, "SI-SDR differs by %.3f dB" % d
    np.testing.assert_allclose(cost, cost_ref, rtol=2e-2)
    assert 0.02 < algo.acceptance_rate < 0.98
    # a second utterance through the same object: init_parameters resets everything
    if variant == "M1":
        algo.init_parameters(X=X[:, :50], S=S[:, :50], vae=model, nmf_rank=10, eps=1e-8, device="cuda:0")
        assert algo.run().shape == (niter,) and algo.S_hat.shape == (F, 50)


def test_enhancer_batch_matches_single_and_is_deterministic():
    """Philox draws are keyed by (utterance id, frame, iteration): batch composition must not change any result."""
    from dvae_b200.engine import Enhancer, McemConfig
    lens = [16000, 12000, 20000]
    xs = [synth.synth_utterance(30 + i, l / 16000.0)[0] for i, l in enumerate(lens)]
    P0 = np.abs(stft_np.stft(xs[0], **KW)) ** 2
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=5, out_bias=float(np.log(P0.mean())))
    cfg = McemConfig(niter=3, keep_E=4, burn_E=6, keep_WF=5, burn_WF=7, seed=11)
    enh = Enhancer(sd, "M1", cfg, device=0)
    s_all, n_all, c_all = enh.enhance(xs, utt_ids=[100, 101, 102])
    s_again, _, c_again = enh.enhance(xs, utt_ids=[100, 101, 102])
    for a, b in zip(s_all, s_again):
        assert np.array_equal(a, b)
    assert np.array_equal(c_all, c_again)
    s_one, n_one, c_one = enh.enhance([xs[1]], utt_ids=[101])
    assert np.array_equal(s_one[0], s_all[1]) and np.array_equal(n_one[0], n_all[1])
    np.testing.assert_allclose(c_one[0], c_all[1], rtol=1e-12)
    for x, s, n in zip(xs, s_all, n_all):
        assert s.shape == x.shape and s.dtype == np.float32
        assert np.max(np.abs((s + n)[800:-800] - x[800:-800])) <= 1e-4      # masks sum to one


def test_multi_chain_pools_samples():
    from dvae_b200.engine import Enhancer, McemConfig
    x = synth.synth_utterance(40, 1.0)[0]
    P0 = np.abs(stft_np.stft(x, **KW)) ** 2
    sd = synth.xavier_state_dict("M2v3", 513, 16, [128, 128], 1, seed=6, out_bias=float(np.log(P0.mean())))
    y = synth.energy_vad(synth.synth_utterance(40, 1.0)[1])
    cfg = McemConfig(niter=2, keep_E=3, burn_E=4, keep_WF=4, burn_WF=5, seed=1, n_chains=4)
    enh = Enhancer(sd, "M2v3", cfg, device=0)
    s, n, c = enh.enhance([x], y_list=[y])
    assert enh.engine.R == 12 and enh.engine.R_wf == 16
    assert np.isfinite(s[0]).all() and np.isfinite(c).all()


def test_device_vad_labels_equal_host_labels():
    """M2-info model: labels from the clean speech on the device (s_list) give the same run as host labels (y_list)."""
    from dvae_b200.engine import Enhancer, McemConfig
    lens = [16000, 13000]
    utts = [synth.synth_utterance(50 + i, l / 16000.0) for i, l in enumerate(lens)]
    xs, ss = [u[0] for u in utts], [u[1] for u in utts]
    P0 = np.abs(stft_np.stft(xs[0], **KW)) ** 2
    sd = synth.xavier_state_dict("M2v3", 513, 16, [128, 128], 1, seed=8, out_bias=float(np.log(P0.mean())))
    cfg = McemConfig(niter=2, keep_E=3, burn_E=4, keep_WF=4, burn_WF=5, seed=3)
    enh = Enhancer(sd, "M2v3", cfg, device=0)
    ys = [synth.energy_vad(s) for s in ss]
    assert 0 < ys[0].mean() < 1
    s_host, _, c_host = enh.enhance(xs, y_list=ys, utt_ids=[7, 8])
    s_host = [a.copy() for a in s_host]
    s_dev, _, c_dev = enh.enhance(xs, s_list=ss, utt_ids=[7, 8])
    for a, b in zip(s_host, s_dev):
        assert np.array_equal(a, b)
    assert np.array_equal(c_host, c_dev)


def test_process_sublist_replacement(tmp_path):
    """batch_io.process_sublist: wav files in, *_s_est.wav / *_n_est.wav out, existing outputs skipped (evaluate_ntcd_M1.py:81-214)."""
    import os
    from dvae_b200 import batch_io
    from dvae_b200.engine import Enhancer, McemConfig
    wav_dir, out_dir = str(tmp_path / "wav") + "/", str(tmp_path / "out") + "/"
    lens = [16000, 12000, 20000]
    sub = []
    for i, l in enumerate(lens):
        x = synth.synth_utterance(60 + i, l / 16000.0)[0]
        rel = "spk%d/utt%d.wav" % (i % 2, i)
        batch_io.write_wav(wav_dir + rel, x, 16000)
        sub.append((rel, "unused_clean_path"))
    x0, _ = batch_io.read_wav(wav_dir + sub[0][0])
    P0 = np.abs(stft_np.stft(x0, **KW)) ** 2
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=5, out_bias=float(np.log(P0.mean())))
    enh = Enhancer(sd, "M1", McemConfig(niter=2, keep_E=3, burn_E=4, keep_WF=4, burn_WF=5, seed=2), device=0)
    done = batch_io.process_sublist(sub, enh, wav_dir, out_dir, batch_size=2)
    assert len(done) == 3
    for (rel, _), l in zip(sub, lens):
        s, fs = batch_io.read_wav(batch_io.output_stem(out_dir, rel) + "_s_est.wav")
        n, _ = batch_io.read_wav(batch_io.output_stem(out_dir, rel) + "_n_est.wav")
        x, _ = batch_io.read_wav(wav_dir + rel)
        assert fs == 16000 and len(s) == l and len(n) == l
        assert np.max(np.abs((s + n)[800:-800] - x[800:-800])) < 2e-4          # masks sum to one; two 16-bit roundings
    assert batch_io.process_sublist(sub, enh, wav_dir, out_dir) == []           # everything exists: skipped like the reference


def test_full_size_properties_configs1():
    """BASELINE.json configs[1] size (512 x 3 s, M1, full MH schedule, 2 EM iterations): size-independent properties.

    * the two Wiener masks sum to one, so s_hat + n_hat reproduces the mixture (away from the first hop, where the
      reference's ISTFT divides by a vanishing window sum);
    * the run is bit-reproducible, and a shard of the batch (rank 1 of 2) gives bit-identical results for its utterances:
      the Philox counters are keyed by global utterance id, not by position in the batch (the shard starts on a 128-frame tile
      boundary here, 256 x 185 = 370 x 128; for other offsets see the summation-order test below);
    * the cost of every utterance is finite and does not increase from the first to the second EM iteration.
    """
    from dvae_b200.engine import Enhancer, McemConfig
    from dvae_b200.shard import shard_range
    B = 512
    xs = [np.asarray(x, np.float32) for x in synth.synth_batch(0, B, seconds=3.0)[0]]
    P0 = np.abs(stft_np.stft(xs[0], **KW)) ** 2
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=1234, out_bias=float(np.log(P0.mean())))
    cfg = McemConfig(niter=2, keep_E=30, burn_E=30, keep_WF=75, burn_WF=30, seed=7)
    enh = Enhancer(sd, "M1", cfg, device=0)
    ids = list(range(B))
    s1, n1, c1 = enh.enhance(xs, utt_ids=ids)
    s1 = [a.copy() for a in s1]
    n1 = [a.copy() for a in n1]
    worst = max(float(np.max(np.abs((s + n)[800:-800] - x[800:-800]))) for x, s, n in zip(xs, s1, n1))
    assert worst <= 1e-4, worst
    assert np.isfinite(c1).all() and np.all(c1[:, 1] <= c1[:, 0] + 1e-6)
    s2, _, c2 = enh.enhance(xs, utt_ids=ids)
    assert all(np.array_equal(a, b) for a, b in zip(s1, s2)) and np.array_equal(c1, c2)
    lo, hi = shard_range(B, 1, 2)
    s3, n3, c3 = enh.enhance(xs[lo:hi], utt_ids=ids[lo:hi])
    assert all(np.array_equal(a, b) for a, b in zip(s1[lo:hi], s3)) and all(np.array_equal(a, b) for a, b in zip(n1[lo:hi], n3))
    np.testing.assert_allclose(c3, c1[lo:hi], rtol=1e-12)


def test_multi_chain_routes_agree_end_to_end():
    """4 chains x 10 kept samples = 40 samples per frame on the tensor-core sampler, one enhancement per E-step route
    (``McemEngine.route``): "stats" (windowed fused decode + windowed M-step kernel) against "decode" (materialised decode,
    generic NMF passes) on the same draws, and "emit" (the sampler's own emission with the windowed emission M-step kernel;
    BF16 variances: looser tolerance)."""
    from dvae_b200.engine import Enhancer, McemConfig
    x = synth.synth_utterance(41, 1.2)[0]
    s_clean = synth.synth_utterance(41, 1.2)[1]
    P0 = np.abs(stft_np.stft(x, **KW)) ** 2
    sd = synth.xavier_state_dict("M2v3", 513, 16, [128, 128], 1, seed=6, out_bias=float(np.log(P0.mean())))
    y = synth.energy_vad(s_clean)
    out = {}
    for mode, route in (("win", "stats"), ("generic", "decode"), ("emit", "emit")):
        cfg = McemConfig(niter=3, keep_E=10, burn_E=5, keep_WF=25, burn_WF=5, seed=1, n_chains=4, sampler="tc")
        enh = Enhancer(sd, "M2v3", cfg, device=0)
        assert enh.engine.route == "emit"
        enh.engine.route = route
        s, n, c = enh.enhance([x], y_list=[y], utt_ids=[3])
        assert enh.engine.R == 40 and enh.engine.R_wf == 100
        out[mode] = (s[0].copy(), c.copy())
    # same draws, same decoder arithmetic up to rounding: the trajectories agree closely (no accept decision is near-tied here)
    assert np.allclose(out["win"][1], out["generic"][1], rtol=2e-4), (out["win"][1], out["generic"][1])
    err = np.linalg.norm(out["win"][0] - out["generic"][0]) / np.linalg.norm(out["generic"][0])
    assert err < 5e-3, err
    assert np.allclose(out["emit"][1], out["generic"][1], rtol=5e-3), (out["emit"][1], out["generic"][1])
    err = np.linalg.norm(out["emit"][0] - out["generic"][0]) / np.linalg.norm(out["generic"][0])
    assert err < 5e-2, err


def test_results_of_an_utterance_do_not_depend_on_its_batch_beyond_summation_order():
    """The random draws of an utterance are keyed by its global id, so the same utterance enhanced inside different batches sees
    the same numbers.  What may differ is floating-point association: the fused W-update reduction (McemConfig.w_partials) sums
    an utterance's frames in runs cut at 128-frame tile boundaries, which fall elsewhere when the utterance sits at another offset
    of the batch.  * with w_partials=False (per-frame statistics, summed per utterance in frame order) a sub-batch is bit-identical
    whatever its offset;  * with the default, a tile-aligned sub-batch is bit-identical and a misaligned one agrees to rounding
    (no accept decision flips in this short run)."""
    from dvae_b200.engine import Enhancer, McemConfig
    B = 24
    xs = [np.asarray(x, np.float32) for x in synth.synth_batch(40, B, seconds=2.0)[0]]       # 123 frames each
    P0 = np.abs(stft_np.stft(xs[0], **KW)) ** 2
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=1234, out_bias=float(np.log(P0.mean())))
    ids = list(range(500, 500 + B))
    for wp in (False, True):
        cfg = McemConfig(niter=3, keep_E=30, burn_E=10, keep_WF=25, burn_WF=10, seed=7, w_partials=wp)
        enh = Enhancer(sd, "M1", cfg, device=0)
        s1, n1, c1 = enh.enhance(xs, utt_ids=ids)
        s1 = [a.copy() for a in s1]
        lo, hi = 5, 17                                                   # 5 x 123 frames: not a multiple of 128
        s2, _, c2 = enh.enhance(xs[lo:hi], utt_ids=ids[lo:hi])
        if not wp:
            assert all(np.array_equal(a, b) for a, b in zip(s1[lo:hi], s2)) and np.array_equal(c1[lo:hi], c2)
        else:
            err = max(float(np.linalg.norm(a - b) / np.linalg.norm(a)) for a, b in zip(s1[lo:hi], s2))
            assert err <= 1e-3, err
            np.testing.assert_allclose(c2, c1[lo:hi], rtol=1e-4)
