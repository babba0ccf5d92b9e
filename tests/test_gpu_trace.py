"""The quality trace over EM iterations: McemEngine.run(checkpoints=...), Enhancer.enhance(score_at=...) and
batch_io.process_sublist(score=True, score_at=...).  A trace entry must equal the score of a separate run with that many
EM iterations bit for bit, and the traced run must return exactly what the untraced run returns."""
import numpy as np
import pytest
import torch

from dvae_b200 import batch_io, synth
from dvae_b200.engine import Enhancer, InjectedDraws, McemConfig, RaggedBatch
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu

SCORE_AT = (2, 4, 6)
CASES = {
    # tensor-core path, the sampler's emission with 10 kept samples; filter through the fused A1 decode (R = 10)
    "M1_tc_keep10": ("M1", dict(keep_E=10, burn_E=5, keep_WF=10, burn_WF=5, sampler="tc")),
    # emission with 30 kept samples; filter through the FP32 Vs scratch (R = 5 has no A1 chunk)
    "M1_tc_keep30": ("M1", dict(keep_E=30, burn_E=5, keep_WF=5, burn_WF=5, sampler="tc")),
    # exact mode; E-step and filter share the kept-sample buffer (keep_E == keep_WF)
    "M1_fp32": ("M1", dict(keep_E=5, burn_E=5, keep_WF=5, burn_WF=5, sampler="fp32")),
    # labels: the clean speech's VAD computed on the device
    "M2_vad_tc": ("M2", dict(keep_E=10, burn_E=5, keep_WF=10, burn_WF=5, sampler="tc")),
    # two chains per frame: the emission with segment partial sums, filter R = 2 x 5
    "M1_tc_2chains": ("M1", dict(keep_E=10, burn_E=5, keep_WF=5, burn_WF=5, sampler="tc", n_chains=2)),
}


def _utts():
    """Ragged: odd lengths, and one utterance of at most two 50 ms trims (its score rows are NaN)."""
    rows = [synth.synth_utterance(u, sec) for u, sec in zip(range(60, 66), (2.0, 3.0, 1.7311, 2.5, 1599 / 16000, 1.0))]
    return [r[0] for r in rows], [r[1] for r in rows]


def _enhancer(variant, kw, niter, s0):
    y_dim = 0 if variant == "M1" else 1
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=3, out_bias=synth.speech_prior_bias(s0))
    return Enhancer(sd, variant, McemConfig(niter=niter, **kw), device=DEV)


@pytest.mark.parametrize("case", list(CASES))
def test_trace_equals_separate_runs_and_leaves_the_run_untouched(case):
    variant, kw = CASES[case]
    x_list, s_list = _utts()
    call = dict(utt_ids=[7, 11, 13, 17, 19, 23], s_list=s_list if variant != "M1" else None, ref_list=s_list)
    enh = _enhancer(variant, kw, 6, s_list[0])
    s0, n0, c0, sc0 = enh.enhance(x_list, **call)
    s0, n0 = [a.copy() for a in s0], [a.copy() for a in n0]
    acc0 = enh.engine.n_accept.clone()
    s1, n1, c1, sc1, tr = enh.enhance(x_list, score_at=SCORE_AT, **call)
    assert tr.shape == (6, 3, 5) and tr.dtype == np.float64
    # the traced run returns exactly what the untraced one returns
    for u in range(6):
        assert np.array_equal(s1[u], s0[u]) and np.array_equal(n1[u], n0[u]), u
    assert np.array_equal(c1, c0)
    assert np.array_equal(sc1, sc0, equal_nan=True)
    assert torch.equal(enh.engine.n_accept, acc0)
    # niter = 6 is the call's own estimate
    assert np.array_equal(tr[:, 2], sc1[:, 0], equal_nan=True)
    # the other entries are what separate runs with fewer EM iterations return
    for k, n in enumerate(SCORE_AT[:2]):
        sep = _enhancer(variant, kw, n, s_list[0]).enhance(x_list, **call)[3]
        assert np.array_equal(tr[:, k], sep[:, 0], equal_nan=True), (case, n)
        assert np.array_equal(sep[:, 1], sc1[:, 1], equal_nan=True)
    assert np.isnan(tr[4]).all() and np.isfinite(tr[[0, 1, 3]]).all()
    assert not np.array_equal(tr[[0, 1, 3], 0], tr[[0, 1, 3], 2])
    # a trace without the last iteration, on the device
    s2, n2, c2, sc2, tr2 = enh.enhance(x_list, score_at=(4,), return_device=True, **call)
    assert tr2.is_cuda and tr2.shape == (6, 1, 5)
    assert np.array_equal(tr2.cpu().numpy()[:, 0], tr[:, 1], equal_nan=True)
    assert np.array_equal(sc2.cpu().numpy(), sc0, equal_nan=True)


def test_engine_checkpoints_callback_and_errors():
    x_list, s_list = _utts()
    enh = _enhancer("M1", CASES["M1_tc_keep10"][1], 6, s_list[0])
    eng = enh.engine
    seen = []

    def on_checkpoint(n):
        seen.append((n, eng.mh_calls, eng.mh_iter0))

    per_e, per_f = 10 + 5, 10 + 5
    eng.timing = True
    enh.enhance(x_list, utt_ids=list(range(6)), ref_list=s_list)
    plain_stages = eng.stage_times_ms()
    enh.enhance(x_list, utt_ids=list(range(6)), ref_list=s_list, score_at=(1, 3, 6))
    traced_stages = eng.stage_times_ms()
    eng.timing = False
    assert "trace" not in plain_stages and traced_stages["trace"][1] == 2          # 1 and 3 are side runs, 6 the run's own
    assert {k: v[1] for k, v in traced_stages.items() if k != "trace"} == {k: v[1] for k, v in plain_stages.items()}
    # the callback sees the side filter's counters, then the run's own filter; the counters end as without checkpoints
    lens = np.array([len(a) for a in x_list], np.int32)
    off = np.zeros(len(x_list) + 1, np.int64)
    np.cumsum((lens.astype(np.int64) + 1) // 2 * 2, out=off[1:])
    flat = np.zeros(int(off[-1]), np.float32)
    for a, o in zip(x_list, off):
        flat[o:o + len(a)] = a
    batch = RaggedBatch([synth.num_frames(int(t)) for t in lens], DEV, list(range(6)))
    enh.run_device(torch.from_numpy(flat).to(DEV), torch.from_numpy(off[:-1].copy()).to(DEV), torch.from_numpy(lens).to(DEV),
                   batch, None, int(off[-1]), int(lens.max()), checkpoints=(2, 5, 6), on_checkpoint=on_checkpoint)
    assert seen == [(2, 3, 2 * per_e + per_f), (5, 6, 5 * per_e + per_f), (6, 7, 6 * per_e + per_f)]
    assert eng.mh_calls == 7 and eng.mh_iter0 == 6 * per_e + per_f
    # argument errors, before any device work
    draws = InjectedDraws(None, None, None, None)
    with pytest.raises(ValueError):
        eng.run(draws, checkpoints=(2,))
    for bad in ((0,), (7,), (4, 2), (2, 2)):
        with pytest.raises(ValueError):
            eng.run(checkpoints=bad)
        with pytest.raises(ValueError):
            enh.enhance(x_list, ref_list=s_list, score_at=bad)
    with pytest.raises(ValueError):
        enh.enhance(x_list, score_at=(2,))                                        # no ref_list
    with pytest.raises(ValueError):
        enh.enhance(x_list, ref_list=s_list, score_at=(2,), draws=draws)


def test_process_sublist_trace_matches_enhance(tmp_path):
    wav_dir = str(tmp_path / "in")
    sub = []
    for i in range(7):
        x, s, _ = synth.synth_utterance(70 + i, (16000 + 2345 * i + (i % 2)) / 16000 if i != 5 else 1599 / 16000)
        rel = "/spk%d/utt%d.wav" % (i % 2, i)
        batch_io.write_wav(wav_dir + rel, x, 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, s, 16000)
        sub.append((rel, "/clean" + rel))
    variant, kw = CASES["M1_tc_keep10"]
    enh = _enhancer(variant, kw, 6, synth.synth_utterance(70, 1.0)[1])
    out_a, out_b = str(tmp_path / "plain"), str(tmp_path / "traced")
    stems_a = batch_io.process_sublist(sub, enh, wav_dir, out_a, batch_size=3)
    stems_b, sc, tr = batch_io.process_sublist(sub, enh, wav_dir, out_b, batch_size=3, score=True, score_at=SCORE_AT)
    assert len(stems_a) == len(stems_b) == 7 and sc.shape == (7, 2, 5) and tr.shape == (7, 3, 5)
    for rel, _ in sub:
        for suffix in ("_s_est.wav", "_n_est.wav"):
            a = open(batch_io.output_stem(out_a, rel) + suffix, "rb").read()
            b = open(batch_io.output_stem(out_b, rel) + suffix, "rb").read()
            assert a == b, (rel, suffix)
    # enhance on the same batches of the same files
    ref = []
    for lo in range(0, 7, 3):
        part = sub[lo:lo + 3]
        xs = [batch_io.read_wav(wav_dir + a)[0].astype(np.float32) for a, _ in part]
        cs = [batch_io.read_wav(wav_dir + b)[0].astype(np.float32) for _, b in part]
        ids = [batch_io.utterance_id(a) for a, _ in part]
        ref.append(enh.enhance(xs, utt_ids=ids, ref_list=cs, pcm16=True, score_at=SCORE_AT)[4])
    assert np.array_equal(tr, np.concatenate(ref), equal_nan=True)
    assert np.array_equal(tr[:, 2], sc[:, 0], equal_nan=True)
    assert np.isnan(tr[5]).all()
    again = batch_io.process_sublist(sub, enh, wav_dir, out_b, batch_size=3, score=True, score_at=SCORE_AT)
    assert again[0] == [] and again[2].shape == (0, 3, 5)
