"""Device scoring of enhanced utterances: the 16-bit PCM quantiser (dvae_pcm16_f32), metrics.score_batch, the scores of
Enhancer.enhance(ref_list=...) and batch_io.process_sublist(score=True) / score_sublist."""
import os

import numpy as np
import pytest
import torch

from dvae_b200 import batch_io, synth
from dvae_b200.engine import Enhancer, McemConfig
from dvae_b200.packages import metrics as dmetrics
from oracle import mcem_port, stoi_np
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu

TOL_DB = 1e-4          # energy ratios against the float64 oracle, as tests/test_gpu_metrics.py
TOL_STOI = 1e-4        # STOI / ESTOI against the float64 oracle, as tests/test_gpu_stoi.py
CFG = dict(niter=2, keep_E=5, burn_E=5, keep_WF=5, burn_WF=5)


def _numpy_pcm16(x):
    return np.clip(np.rint(np.asarray(x, np.float64) * 32768.0), -32768, 32767).astype(np.int16)


def _pack(signals):
    """Concatenate at even offsets (the layout of Enhancer.run_device): (flat float32 host array, off int64, lens int32)."""
    lens = np.array([len(a) for a in signals], np.int32)
    off = np.zeros(len(signals) + 1, np.int64)
    np.cumsum((lens.astype(np.int64) + 1) // 2 * 2, out=off[1:])
    flat = np.zeros(int(off[-1]), np.float32)
    for a, o in zip(signals, off):
        flat[o:o + len(a)] = a
    return flat, off[:-1].copy(), lens


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _quantise(x):
    xd = _dev(x)
    pcm = torch.empty(xd.numel(), dtype=torch.int16, device=DEV)
    xq = torch.empty_like(xd)
    dmetrics.pcm16(xd, pcm, xq)
    return pcm.cpu().numpy(), xq.cpu().numpy()


def test_pcm16_matches_write_wav():
    k = np.arange(-32770, 32770, dtype=np.float64)
    rng = np.random.default_rng(11)
    x = np.concatenate([
        [1.0, -1.0, np.nextafter(1.0, 2.0), np.nextafter(-1.0, -2.0), 32767 / 32768, -32768 / 32768, 32767.5 / 32768, -32768.5 / 32768],
        [1.5, -1.5, 3e38, -3e38, 1e-40, -1e-40, 0.0, -0.0, np.inf, -np.inf],
        (k + 0.5) / 32768,                                     # every exact half step: round half to even
        rng.standard_normal(3_000_001) * 0.4,                  # a long signal, odd length: vector body and scalar tail
    ]).astype(np.float32)
    ref = _numpy_pcm16(x)
    for lo in (0, 1, 2):                                       # 16-byte aligned (vectorised) and unaligned views
        xd = _dev(x)[lo:]
        p = torch.empty(xd.numel(), dtype=torch.int16, device=DEV)
        q = torch.empty(xd.numel() + (lo > 0), dtype=torch.float32, device=DEV)[(lo > 0):]
        dmetrics.pcm16(xd, p, q)
        pcm, xq = p.cpu().numpy(), q.cpu().numpy()
        assert np.array_equal(pcm, ref[lo:]), lo
        assert np.array_equal(xq, pcm.astype(np.float32) / np.float32(32768.0)), lo
    assert pcm.dtype == np.int16
    # each output alone
    xd = _dev(x)
    p = torch.zeros(xd.numel(), dtype=torch.int16, device=DEV)
    dmetrics.pcm16(xd, p, None)
    q = torch.zeros_like(xd)
    dmetrics.pcm16(xd, None, q)
    assert np.array_equal(p.cpu().numpy(), ref) and np.array_equal(q.cpu().numpy(), ref.astype(np.float32) / np.float32(32768.0))
    # NaN maps to 0 (numpy's cast of NaN is platform-defined, so it is not part of the comparison above)
    pcm, xq = _quantise(np.array([np.nan, 0.5, -np.nan, np.nan, 0.25], np.float32))
    assert pcm.tolist() == [0, 16384, 0, 0, 8192] and xq.tolist() == [0.0, 0.5, 0.0, 0.0, 0.25]
    with pytest.raises(ValueError):
        dmetrics.pcm16(xd, None, None)
    with pytest.raises(ValueError):
        dmetrics.pcm16(xd, torch.empty(5, dtype=torch.int16, device=DEV))


def _score_set():
    """(est, x, s) triples: odd lengths, one utterance of at most 2 trims (NaN row), one of 20 s, one with silent clean speech."""
    rng = np.random.default_rng(5)
    out = []
    for u, sec in ((20, 3.0), (21, 47999 / 16000), (22, 1599 / 16000), (23, 20.0), (24, 2.5), (25, 33333 / 16000)):
        x, s, n = synth.synth_utterance(u, sec)
        if u == 24:
            s = np.zeros_like(s)
            x = n
        est = (0.7 * s + 0.2 * (x - s) + 0.01 * rng.standard_normal(len(s))).astype(np.float32)
        out.append((est, x.astype(np.float32), s.astype(np.float32)))
    return out


def test_score_batch_matches_its_parts_and_the_oracles():
    sets = _score_set()
    trim = 800
    fe, off, lens = _pack([t[0] for t in sets])
    fx, _, _ = _pack([t[1] for t in sets])
    fs_, _, _ = _pack([t[2] for t in sets])
    d_off, d_len = _dev(off), _dev(lens)
    got = dmetrics.score_batch(_dev(fe), _dev(fx), _dev(fs_), d_off, d_len, 16000).cpu().numpy()
    assert got.shape == (len(sets), 2, 5) and got.dtype == np.float64
    # exactly the existing batched metrics on the trimmed layout
    fn = (fx - fs_).astype(np.float32)
    t_off, t_len = _dev(off + trim), _dev(np.maximum(lens - 2 * trim, 0).astype(np.int32))
    for k, sig in enumerate((fe, fx)):
        er = dmetrics.energy_ratios_batch(_dev(sig), _dev(fs_), _dev(fn), t_off, t_len).cpu().numpy()
        st = dmetrics.stoi_batch(_dev(fs_), _dev(sig), t_off, t_len, 16000).cpu().numpy()
        part = np.concatenate([er, st], axis=1)
        part[lens <= 2 * trim] = np.nan
        assert np.array_equal(got[:, k], part, equal_nan=True), k
    # the float64 oracles on the trimmed signals
    for u, (est, x, s) in enumerate(sets):
        if len(s) <= 2 * trim:
            assert np.isnan(got[u]).all()
            continue
        sl = slice(trim, len(s) - trim)
        for k, sig in enumerate((est, x)):
            if u == 4:                                         # silent clean speech: no score is defined
                assert np.isnan(got[u, k]).all(), got[u, k]
                continue
            with np.errstate(all="ignore"):
                ref = mcem_port.energy_ratios(sig[sl], s[sl], (x - s)[sl])
                st = [stoi_np.stoi(s[sl], sig[sl], 16000), stoi_np.stoi(s[sl], sig[sl], 16000, extended=True)]
            assert np.allclose(got[u, k, :3], ref, rtol=0, atol=TOL_DB), (u, k, got[u, k], ref)
            assert np.allclose(got[u, k, 3:], st, rtol=0, atol=TOL_STOI), (u, k, got[u, k], st)
    # a different trim, and the result written into a caller's buffer
    out = torch.full((len(sets), 2, 5), -1.0, dtype=torch.float64, device=DEV)
    r = dmetrics.score_batch(_dev(fe), _dev(fx), _dev(fs_), d_off, d_len, 16000, trim=0, out=out)
    assert r is out and not np.isnan(out[0].cpu().numpy()).any()
    with pytest.raises(ValueError):
        dmetrics.score_batch(_dev(fe), _dev(fx)[:-2], _dev(fs_), d_off, d_len, 16000)


def _utts(u0, count):
    rows = [synth.synth_utterance(u, sec) for u, sec in zip(range(u0, u0 + count), (2.0, 3.0, 1.7311, 2.5, 1.0))]
    return [r[0] for r in rows], [r[1] for r in rows]


@pytest.mark.parametrize("variant", ["M1", "M2"])
def test_enhance_scores_do_not_perturb_and_match_score_batch(variant):
    x_list, s_list = _utts(30, 5)
    y_dim = 0 if variant == "M1" else 1
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=3, out_bias=synth.speech_prior_bias(s_list[0]))
    enh = Enhancer(sd, variant, McemConfig(**CFG), device=DEV)
    kw = dict(utt_ids=list(range(5)), s_list=s_list if y_dim else None)
    s0, n0, c0 = enh.enhance(x_list, **kw)
    s0, n0 = [a.copy() for a in s0], [a.copy() for a in n0]
    s1, n1, c1, sc1 = enh.enhance(x_list, ref_list=s_list, **kw)
    assert sc1.shape == (5, 2, 5) and sc1.dtype == np.float64
    assert enh.d2h_bytes == 2 * sum((len(a) + 1) // 2 * 2 for a in x_list) * 4 + c1.size * 8 + sc1.size * 8
    for u in range(5):
        assert np.array_equal(s1[u], s0[u]) and np.array_equal(n1[u], n0[u]), u
    assert np.array_equal(c1, c0)
    s2, n2, c2, sc2 = enh.enhance(x_list, ref_list=s_list, pcm16=True, **kw)
    total = sum((len(a) + 1) // 2 * 2 for a in x_list)
    assert enh.d2h_bytes == 2 * total * 2 + c2.size * 8 + sc2.size * 8
    for u in range(5):
        assert s2[u].dtype == np.int16 and np.array_equal(s2[u], _numpy_pcm16(s0[u])), u
        assert np.array_equal(n2[u], _numpy_pcm16(n0[u])), u
    assert np.array_equal(sc2, sc1, equal_nan=True)
    # the scores are score_batch of the 16-bit estimate against the staged mixture and clean speech
    fe, off, lens = _pack([a.astype(np.float32) / np.float32(32768.0) for a in s2])
    fx, _, _ = _pack(x_list)
    fs_, _, _ = _pack(s_list)
    ref = dmetrics.score_batch(_dev(fe), _dev(fx), _dev(fs_), _dev(off), _dev(lens), 16000).cpu().numpy()
    assert np.array_equal(sc2, ref, equal_nan=True)
    assert np.isfinite(sc2[[0, 1, 3]]).all()
    # device results: int16 estimates and the score tensor
    sd_, nd_, _, scd = enh.enhance(x_list, ref_list=s_list, pcm16=True, return_device=True, **kw)
    assert sd_.dtype == torch.int16 and nd_.dtype == torch.int16 and scd.is_cuda
    assert np.array_equal(scd.cpu().numpy(), sc2, equal_nan=True)
    with pytest.raises(ValueError):
        enh.enhance(x_list, ref_list=s_list[:4], **kw)


def test_process_sublist_score_matches_score_sublist(tmp_path):
    wav_dir = str(tmp_path / "in")
    sub = []
    for i in range(8):
        x, s, _ = synth.synth_utterance(40 + i, (16000 + 2345 * i + (i % 2)) / 16000)
        rel = "/spk%d/utt%d.wav" % (i % 2, i)
        batch_io.write_wav(wav_dir + rel, x, 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, s, 16000)
        sub.append((rel, "/clean" + rel))
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=3, out_bias=synth.speech_prior_bias(s))
    enh = Enhancer(sd, "M1", McemConfig(**CFG), device=DEV)
    out_a, out_b = str(tmp_path / "plain"), str(tmp_path / "scored")
    stems_a = batch_io.process_sublist(sub, enh, wav_dir, out_a, batch_size=3)
    stems_b, sc = batch_io.process_sublist(sub, enh, wav_dir, out_b, batch_size=3, score=True)
    assert len(stems_a) == len(stems_b) == 8 and sc.shape == (8, 2, 5)
    for rel, _ in sub:
        for suffix in ("_s_est.wav", "_n_est.wav"):
            a = open(batch_io.output_stem(out_a, rel) + suffix, "rb").read()
            b = open(batch_io.output_stem(out_b, rel) + suffix, "rb").read()
            assert a == b, (rel, suffix)
    stems_c, sc_files = batch_io.score_sublist(sub, wav_dir, out_b, device=DEV, batch_size=5)
    assert stems_c == stems_b
    assert np.array_equal(sc, sc_files, equal_nan=True)
    assert np.isfinite(sc).all()
    again, sc_again = batch_io.process_sublist(sub, enh, wav_dir, out_b, batch_size=3, score=True)
    assert again == [] and sc_again.shape == (0, 2, 5)
    os.remove(batch_io.output_stem(out_b, sub[3][0]) + "_s_est.wav")
    with pytest.raises(FileNotFoundError):
        batch_io.score_sublist(sub, wav_dir, out_b, device=DEV)
