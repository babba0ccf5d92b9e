"""Oracle labels of the M2 models computed on the device from the clean speech (Enhancer.enhance(..., s_list=, oracle_labels=)
and process_sublist(..., oracle_labels=)) against the labels of the package's per-utterance shims, computed on the whole clean
signal and cut to the frame cap, as scripts/evaluate_ntcd_M2.py:187-195 cuts them."""
import numpy as np
import pytest
import torch

from dvae_b200 import batch_io, synth
from dvae_b200.engine import Enhancer, McemConfig
from dvae_b200.packages.processing import stft as dstft
from dvae_b200.packages.processing import target as dtarget
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu
KW = dict(fs=16000, wlen_sec=64e-3, hop_percent=0.25, center=False, pad_at_end=True)
BIG = np.iinfo(np.int64).max
CFG = dict(keep_E=10, burn_E=5, keep_WF=10, burn_WF=5)


def shim_labels(mode, s):
    """The labels a user builds with the per-utterance shims: ``(y_dim, N)`` over the whole clean signal."""
    if mode == "vad":
        return dtarget.clean_speech_VAD(s, device=DEV, **KW)
    S = dstft.stft(s, win="hann", **KW)
    if mode == "ibm":
        return dtarget.clean_speech_IBM(S, device=DEV)
    return dtarget.noise_robust_clean_speech_IBM(s, S, device=DEV, **KW)


def _enhancer(mode, s0, sampler="fp32", **cfg):
    y_dim = 1 if mode == "vad" else 513
    sd = synth.xavier_state_dict("M2", 513, 16, [128, 128], y_dim, seed=3, out_bias=synth.speech_prior_bias(s0))
    return Enhancer(sd, "M2", McemConfig(sampler=sampler, **dict(CFG, **cfg)), device=DEV)


def _frame_power(s):
    N = synth.num_frames(len(s))
    y = np.zeros(synth.padded_length(len(s)))
    y[:len(s)] = s
    idx = np.arange(1024)[None, :] + 256 * np.arange(N)[:, None]
    return np.sum(y[idx] ** 2, axis=1)


# ---------------------------------------------------------------------------------------------------- 1. label equality
QUIET, LOUD = 4, 5


def _label_batch():
    """Ragged utterances and caps: one frame, short, 3 s; caps None, N, N - 1, 1, past N and two in the middle, one of them
    on an utterance whose quietest frame lies past the cap, the other on one whose loudest bin does."""
    lens = [1024, 4000, 48000, 27698, 48000, 40000, 35200, 20000]
    xs, ss = [], []
    for u, T in enumerate(lens):
        x, s, _ = synth.synth_utterance(200 + u, T / 16000)
        s = s.astype(np.float64)
        if u == QUIET:
            s[130 * 256:] *= 1e-4
        if u == LOUD:
            s[100 * 256:] *= 20.0
        xs.append(x)
        ss.append(s.astype(np.float32))
    N = [synth.num_frames(T) for T in lens]
    caps = [BIG, N[1], N[2] - 1, 1, 90, 60, BIG, N[7] + 5]
    return xs, ss, caps


def test_label_batch_covers_the_cap_cases():
    """The quiet and loud utterances make labels over the capped frames differ from the rule's labels (the VAD route before
    the truncation rule computed them over the capped frames)."""
    xs, ss, caps = _label_batch()
    p = _frame_power(ss[QUIET].astype(np.float64))
    n = caps[QUIET]
    assert np.argmin(p) >= n
    assert not np.array_equal(p[:n] > 10 ** 1.7 * p[:n].min(), (p > 10 ** 1.7 * p.min())[:n])
    S = np.abs(dstft.stft(ss[LOUD], win="hann", **KW))
    n = caps[LOUD]
    assert np.unravel_index(np.argmax(S), S.shape)[1] >= n
    assert not np.array_equal(S[:, :n] + 1e-8 > (S[:, :n].max() + 1e-8) * 10 ** -2.5, (S + 1e-8 > (S.max() + 1e-8) * 10 ** -2.5)[:, :n])


@pytest.mark.parametrize("capped", [True, False])
@pytest.mark.parametrize("mode", ["vad", "ibm", "robust_ibm"])
def test_device_labels_equal_the_shims_cut_to_the_cap(mode, capped):
    xs, ss, caps = _label_batch()
    caps = caps if capped else None
    enh = _enhancer(mode, ss[2], niter=1)
    enh.enhance(xs, s_list=ss, oracle_labels=mode, max_frames_list=caps, utt_ids=list(range(len(xs))), return_device=True)
    got = enh.engine.y.cpu().numpy()
    want = np.concatenate([shim_labels(mode, s)[:, :min(synth.num_frames(len(s)), c)].T
                           for s, c in zip(ss, caps or [BIG] * len(ss))])
    assert got.dtype == np.float32 and got.shape == want.shape and np.array_equal(got, want)
    if mode == "vad":           # the default mode of a one-label model is the same route
        enh.enhance(xs, s_list=ss, max_frames_list=caps, utt_ids=list(range(len(xs))), return_device=True)
        assert np.array_equal(enh.engine.y.cpu().numpy(), want)


# ---------------------------------------------------------------------------------------------------- 2. end to end
def _utts():
    rows = [synth.synth_utterance(u, sec) for u, sec in zip(range(60, 66), (2.0, 3.0, 1.7311, 2.5, 1599 / 16000, 1.0))]
    xs, ss = [r[0] for r in rows], [r[1] for r in rows]
    N = [synth.num_frames(len(x)) for x in xs]
    caps = [BIG, N[1] - 1, 1, 50, N[4], 30]
    return xs, ss, caps


def _callback_y(mode, ss, caps):
    return [shim_labels(mode, s)[:, :min(synth.num_frames(len(s)), c)] for s, c in zip(ss, caps)]


def _assert_same(a, b):
    assert len(a) == len(b)
    for u in range(len(a[0])):
        assert np.array_equal(a[0][u], b[0][u]) and np.array_equal(a[1][u], b[1][u]), u
    for k in range(2, len(a)):
        assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("sampler", ["fp32", "tc"])
@pytest.mark.parametrize("mode", ["vad", "ibm", "robust_ibm"])
def test_enhance_device_labels_equal_callback_labels(mode, sampler):
    xs, ss, caps = _utts()
    ids = [7, 11, 13, 17, 19, 23]
    ys = _callback_y(mode, ss, caps)
    s_copy = [s.copy() for s in ss]
    enh = _enhancer(mode, ss[0], sampler, niter=6)
    base = dict(utt_ids=ids, max_frames_list=caps)
    _assert_same(enh.enhance(xs, y_list=ys, **base), enh.enhance(xs, s_list=ss, oracle_labels=mode, **base))
    assert enh.h2d_bytes == 2 * 4 * sum((len(x) + 1) // 2 * 2 for x in xs)     # noisy + clean, no labels
    sc = dict(base, score_at=(2, 6))
    ref = enh.enhance(xs, y_list=ys, ref_list=s_copy, **sc)
    dev = enh.enhance(xs, s_list=ss, ref_list=ss, oracle_labels=mode, **sc)
    _assert_same(ref, dev)
    assert enh.h2d_bytes == 2 * 4 * sum((len(x) + 1) // 2 * 2 for x in xs)     # ref_list is s_list: the clean signals once
    stop = _enhancer(mode, ss[0], sampler, niter=12, stop_tol=0.02, stop_window=2)
    ref = stop.enhance(xs, y_list=ys, ref_list=s_copy, **base)
    dev = stop.enhance(xs, s_list=ss, ref_list=ss, oracle_labels=mode, **base)
    _assert_same(ref, dev)


# ---------------------------------------------------------------------------------------------------- 3. files
@pytest.mark.parametrize("mode, sampler", [("vad", "tc"), ("ibm", "fp32"), ("robust_ibm", "tc")])
def test_process_sublist_oracle_labels_equal_the_callback_route(tmp_path, mode, sampler):
    xs, ss, _ = _utts()
    wav_dir = str(tmp_path / "in")
    sub, cap_of = [], {}
    for u, (x, s) in enumerate(zip(xs, ss)):
        rel = "/utt%d.wav" % u
        batch_io.write_wav(wav_dir + rel, x, 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, s, 16000)
        sub.append((rel, "/clean" + rel))
        cap_of[rel] = (None, synth.num_frames(len(x)) - 1, 1, 50, None)[u % 5]
    caps = lambda a, b: cap_of[a]                                          # noqa: E731

    def labels(a, b):
        return shim_labels(mode, batch_io.read_wav(wav_dir + b)[0].astype(np.float32))

    enh = _enhancer(mode, ss[0], sampler, niter=3)
    for bs in (2, 6):
        for score in (False, True):
            outs = {}
            for route in ("callback", "oracle"):
                out_dir = str(tmp_path / ("%s_%d_%d" % (route, bs, score)))
                kw = dict(labels=labels) if route == "callback" else dict(oracle_labels=mode)
                res = batch_io.process_sublist(sub, enh, wav_dir, out_dir, batch_size=bs, max_frames=caps, score=score, **kw)
                stems = res[0] if score else res
                files = [open(st + sfx, "rb").read() for st in stems for sfx in ("_s_est.wav", "_n_est.wav")]
                outs[route] = (files, res[1] if score else None)
            assert outs["callback"][0] == outs["oracle"][0], (bs, score)
            if score:
                assert np.array_equal(outs["callback"][1], outs["oracle"][1], equal_nan=True)   # STOI of a sub-trim utterance is NaN


# ---------------------------------------------------------------------------------------------------- 4. errors
def test_errors_come_before_any_device_work(tmp_path):
    xs, ss, caps = _utts()
    one, ibm = _enhancer("vad", ss[0]), _enhancer("ibm", ss[0])
    m1 = Enhancer(synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=3), "M1", McemConfig(**CFG), device=DEV)
    ys1 = [np.ones((1, synth.num_frames(len(x))), np.float32) for x in xs]
    short = [s[:-1] for s in ss]
    cases = [
        (one, dict(s_list=ss, oracle_labels="ibm"), "gives 513 labels"),
        (one, dict(s_list=ss, oracle_labels="robust_ibm"), "gives 513 labels"),
        (ibm, dict(s_list=ss, oracle_labels="vad"), "gives 1 labels"),
        (ibm, dict(s_list=ss), "oracle_labels='ibm'"),
        (m1, dict(s_list=ss, oracle_labels="vad"), "M1"),
        (one, dict(oracle_labels="vad"), "s_list"),
        (ibm, dict(oracle_labels="ibm"), "s_list"),
        (one, dict(s_list=ss, y_list=ys1, oracle_labels="vad"), "y_list"),
        (one, dict(s_list=ss, oracle_labels="nr"), "must be one of"),
        (one, dict(s_list=short, oracle_labels="vad"), "of the utterance's length"),
        (ibm, dict(s_list=ss[:-1], oracle_labels="robust_ibm"), "of the utterance's length"),
    ]
    torch.cuda.synchronize()
    for enh, kw, what in cases:
        before = torch.cuda.memory_allocated(DEV)
        with pytest.raises(ValueError, match=what.replace("(", r"\(")):
            enh.enhance(xs, max_frames_list=caps, **kw)
        assert enh._pinned == {} and enh.engine._buf == {}, what                 # nothing staged, uploaded or allocated
        assert torch.cuda.memory_allocated(DEV) == before, what
    with pytest.raises(ValueError, match="labels callback"):
        batch_io.process_sublist([("/a.wav", "/b.wav")], one, str(tmp_path), str(tmp_path / "o"), oracle_labels="vad",
                                 labels=lambda a, b: None)
    assert one._pinned == {} and one.engine._buf == {}
