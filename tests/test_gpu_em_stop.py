"""Per-utterance stopping of the EM loop (McemConfig.stop_tol): the stopping kernel, the row gathers, the per-frame Philox
iteration base of both samplers, and end to end: a stopped utterance returns exactly what a run with niter = n_u returns."""
import ctypes as C

import numpy as np
import pytest
import torch

from dvae_b200 import _lib, batch_io, synth, tc
from dvae_b200.engine import Enhancer, McemConfig, McemEngine, RaggedBatch, VaeWeights, _p, _stream, permute_rows, stft_batch
from tests.gpu_util import DEV
from tests.test_em_stop_host import stop_iterations

pytestmark = pytest.mark.gpu


def _flags_ref(cost, n, w, tol, B_active):
    out = np.zeros(B_active, np.uint8)
    for u in range(B_active):
        s_old = s_new = 0.0
        for k in range(n - 2 * w, n - w):
            s_old += float(cost[k, u])
        for k in range(n - w, n):
            s_new += float(cost[k, u])
        out[u] = (s_old / w - s_new / w) <= tol * abs(s_new / w)
    return out


def test_stop_check_kernel_matches_restatement():
    rng = np.random.default_rng(5)
    niter, B = 40, 300
    mats = [rng.normal(0, 1, (niter, B)) * 10 ** rng.uniform(-3, 3, B),                 # random signs and scales
            np.cumsum(-np.abs(rng.normal(0, 1, (niter, B))), axis=0) - 50.0]           # decreasing, negative
    crafted = mats[1].copy()
    crafted[7, :5] = np.nan                                                            # NaN never stops
    crafted[:, 5:9] = 4.0                                                              # flat: stops at tol = 0
    crafted[:, 9] = [6.0, 6.0, 4.0, 4.0] + [4.0] * (niter - 4)                         # the == boundary at w = 2, tol = 0.5
    mats.append(crafted)
    flags = torch.zeros(B, dtype=torch.uint8, device=DEV)
    for cost in mats:
        cd = torch.from_numpy(cost).to(DEV)
        for w in (1, 2, 5):
            for n in sorted({2 * w, 2 * w + 1, 17, niter}):
                for tol in (0.0, 1e-3, 0.5, 3.0):
                    for b_act in (B, 123):
                        flags.fill_(7)
                        _lib.call("dvae_em_stop_check", _p(cd), B, b_act, n, w, tol, _p(flags), _stream())
                        got = flags.cpu().numpy()
                        assert np.array_equal(got[:b_act], _flags_ref(cost, n, w, tol, b_act)), (w, n, tol, b_act)
                        assert (got[b_act:] == 7).all()
    with pytest.raises(ValueError):
        _lib.call("dvae_em_stop_check", _p(cd), B, B, 3, 2, 0.0, _p(flags), _stream())            # n < 2w
    with pytest.raises(ValueError):
        _lib.call("dvae_em_stop_check", _p(cd), B, B, 4, 2, float("nan"), _p(flags), _stream())


def test_permute_rows_matches_indexing():
    g = torch.Generator().manual_seed(3)
    B, n_act = 37, 29
    perm = torch.randperm(n_act, generator=g).to(torch.int32)
    arrays = [torch.randn(B, 520, dtype=torch.complex64), torch.randn(B, 10), torch.randn(B), torch.randn(B, 3),
              torch.randint(0, 1 << 30, (B,), dtype=torch.int32), torch.randn(B, 513), torch.randn(B, 10, 520)]
    srcs = [a.to(DEV) for a in arrays]
    dsts = [torch.zeros_like(a) for a in srcs]
    m = perm.to(DEV)
    permute_rows([(s, d, m, n_act, s.numel() * s.element_size() // B, 1, 0) for s, d in zip(srcs, dsts)])
    for s, d in zip(srcs, dsts):
        assert torch.equal(d[:n_act], s[perm.long().to(DEV)]) and not d[n_act:].any()
    # columns of a row-major matrix: n_rep planes of one element per row
    mat = torch.randn(9, B, dtype=torch.float64, device=DEV)
    out = torch.full_like(mat, -1.0)
    full = torch.cat([perm, torch.arange(n_act, B, dtype=torch.int32)]).to(DEV)
    permute_rows([(mat, out, full, B, 8, 6, 8 * B)])
    assert torch.equal(out[:6], mat[:6][:, full.long()]) and (out[6:] == -1).all()
    with pytest.raises(ValueError):
        permute_rows([(srcs[1], dsts[1], m, n_act, 6, 1, 0)])                  # not a multiple of 4


def _engine(variant, cfg, n_utts=3, seconds=(1.0, 0.7531, 1.25)):
    xs = [synth.synth_utterance(90 + u, sec)[0] for u, sec in zip(range(n_utts), seconds)]
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], 0, seed=3, out_bias=synth.speech_prior_bias(xs[0]))
    eng = McemEngine(VaeWeights(sd, variant, torch.device(DEV)), cfg, DEV)
    lens = np.array([len(x) for x in xs], np.int32)
    off = np.concatenate([[0], np.cumsum((lens.astype(np.int64) + 1) // 2 * 2)])
    flat = np.zeros(int(off[-1]), np.float32)
    for x, o in zip(xs, off):
        flat[o:o + len(x)] = x
    batch = RaggedBatch([synth.num_frames(int(t)) for t in lens], DEV, [4, 9, 2])
    X, P = stft_batch(torch.from_numpy(flat).to(DEV), torch.from_numpy(off[:-1].copy()).to(DEV), torch.from_numpy(lens).to(DEV), batch)
    eng.init_parameters(X, P, batch)
    return eng, batch


def test_rng_dump_with_iter0_frame_equals_group_dumps():
    _lib.load()
    batch = RaggedBatch([5, 3, 7], DEV, [11, 3, 8])
    it0 = np.array([100, 40, 7], np.int64)
    per_frame = torch.from_numpy(np.repeat(it0, batch.n_frames).astype(np.uint32)).to(DEV)
    for L, C_ in ((16, 1), (16, 3), (5, 2)):
        rows, n_iter = batch.NT * C_, 6
        eps = torch.empty(n_iter, rows, L, device=DEV)
        u = torch.empty(n_iter, rows, device=DEV)
        rng = _lib.DvaeRng(seed=77, iter0=999, iter0_frame=per_frame.data_ptr())
        _lib.call("dvae_rng_dump", C.byref(rng), _p(batch.frame_gid), _p(batch.frame_idx), batch.NT, C_, L, n_iter, _p(eps), _p(u), _stream())
        for g_, base in enumerate(it0):
            e1, u1 = torch.empty_like(eps), torch.empty_like(u)
            r1 = _lib.DvaeRng(seed=77, iter0=int(base))
            _lib.call("dvae_rng_dump", C.byref(r1), _p(batch.frame_gid), _p(batch.frame_idx), batch.NT, C_, L, n_iter, _p(e1), _p(u1), _stream())
            lo, hi = int(batch.fr_off_host[g_]) * C_, int(batch.fr_off_host[g_ + 1]) * C_
            assert torch.equal(eps[:, lo:hi], e1[:, lo:hi]) and torch.equal(u[:, lo:hi], u1[:, lo:hi]), (L, C_, g_)


@pytest.mark.parametrize("sampler,chains", [("tc", 1), ("tc", 2), ("fp32", 1)])
def test_samplers_with_iter0_frame_equal_scalar_calls(sampler, chains):
    cfg = McemConfig(niter=2, keep_E=10, burn_E=5, sampler=sampler, n_chains=chains)
    eng, batch = _engine("M1", cfg)
    emit = sampler == "tc"
    bases = np.array([300, 15, 300])                     # utterances 0 and 2 in one group, 1 in the other
    Z0, acc0 = eng.Z.clone(), eng.n_accept.clone()

    def call(iter0, per_frame):
        eng.Z.copy_(Z0)
        eng.n_accept.copy_(acc0)
        eng.mh_iter0 = iter0
        eng._iter0_frame = per_frame
        try:
            Zs = eng.sample_posterior(10, 5, emit=emit).clone()
        finally:
            eng._iter0_frame = None
        out = [Zs, eng.Z.clone(), eng.n_accept.clone()]
        if emit:
            out += [eng.vs_idx.view(-1, 32)[:batch.NT * chains].clone(), tc.vst_unpack(eng, 10)]
        return out

    mixed = call(0, torch.from_numpy(np.repeat(bases, batch.n_frames).astype(np.uint32)).to(DEV))
    by_group = {b: call(int(b), None) for b in np.unique(bases)}
    for u, b in enumerate(bases):
        lo, hi = int(batch.fr_off_host[u]), int(batch.fr_off_host[u + 1])
        for k, (m, s) in enumerate(zip(mixed, by_group[b])):
            rows = slice(lo, hi) if k in (0, 4) else slice(lo * chains, hi * chains)     # Zs and unpacked Vs: per frame
            assert torch.equal(m[rows], s[rows]), (sampler, u, k)
    assert not torch.equal(by_group[300][0], by_group[15][0])
    tc.check_status(eng)


# ---------------------------------------------------------------------------------------------------------- end to end
NITER, W = 14, 2
CASES = {
    "M1_tc_keep10": ("M1", dict(keep_E=10, burn_E=5, keep_WF=10, burn_WF=5, sampler="tc")),
    "M1_tc_keep30": ("M1", dict(keep_E=30, burn_E=5, keep_WF=5, burn_WF=5, sampler="tc")),
    "M1_fp32": ("M1", dict(keep_E=5, burn_E=5, keep_WF=5, burn_WF=5, sampler="fp32")),
    "M1_tc_2chains": ("M1", dict(keep_E=10, burn_E=5, keep_WF=5, burn_WF=5, sampler="tc", n_chains=2)),
    "M2_vad_tc": ("M2", dict(keep_E=10, burn_E=5, keep_WF=10, burn_WF=5, sampler="tc")),
    "M2_ibm513_tc": ("M2", dict(keep_E=10, burn_E=5, keep_WF=10, burn_WF=5, sampler="tc")),
}


def _utts():
    rows = [synth.synth_utterance(u, sec) for u, sec in zip(range(60, 68), (2.0, 3.0, 1.7311, 2.5, 1599 / 16000, 1.0, 1.3, 2.2))]
    return [r[0] for r in rows], [r[1] for r in rows]


def _enhancer(case, niter=NITER, **cfg_kw):
    variant, kw = CASES[case]
    x_list, s_list = _utts()
    y_dim = 513 if case == "M2_ibm513_tc" else (0 if variant == "M1" else 1)
    sd = synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=3, out_bias=synth.speech_prior_bias(s_list[0]))
    call = dict(utt_ids=[7, 11, 13, 17, 19, 23, 29, 31], ref_list=s_list)
    if y_dim == 1:
        call["s_list"] = s_list
    elif y_dim == 513:
        call["y_list"] = [(np.random.default_rng(u).random((513, synth.num_frames(len(x)))) > 0.6).astype(np.float32)
                          for u, x in enumerate(x_list)]
    cfg = McemConfig(niter=niter, **dict(dict(kw, w_partials=False), **cfg_kw))
    return Enhancer(sd, variant, cfg, device=DEV), x_list, call


def _pick_tol(cost):
    """A tolerance whose stopping counts take at least three distinct values, niter among them."""
    cands = set()
    for row in cost:
        for n in range(2 * W, NITER):
            m_old, m_new = np.mean(row[n - 2 * W:n - W]), np.mean(row[n - W:n])
            cands.add(float((m_old - m_new) / abs(m_new)))
    cands = sorted(c for c in cands if c >= 0)
    for tol in [(a + b) / 2 for a, b in zip(cands, cands[1:])]:        # between two ratios: no test sits on its boundary
        n_u = stop_iterations(cost, tol, W)
        if len(set(n_u)) >= 3 and NITER in n_u:
            return tol, n_u
    raise AssertionError("no tolerance gives three distinct stopping counts")


def _check_stopping_case(case, w_partials):
    """With w_partials=False the estimates and scores of a stopped utterance equal the niter = n_u run's bit for bit.  So does
    its cost, except on the M-step over the sampler's emission (tc, one chain): that kernel's CTAs cover frame blocks aligned
    in the batch's global frame index, so an utterance's cost is a sum of per-block partials whose cuts move with its offset;
    the cost then agrees to double rounding (its H, g and W are per-frame or per-utterance and stay bit-identical)."""
    emission_mstep = CASES[case][1]["sampler"] == "tc" and CASES[case][1].get("n_chains", 1) == 1
    enh, x_list, call = _enhancer(case, w_partials=w_partials)
    pilot = enh.enhance(x_list, **call)
    tol, n_ref = _pick_tol(pilot[2])
    enh_s, _, _ = _enhancer(case, w_partials=w_partials, stop_tol=tol, stop_window=W)
    s, n, c, sc = enh_s.enhance(x_list, **call)
    n_u = enh_s.engine.n_iter
    assert n_u.dtype.kind == "i" and np.array_equal(n_u, stop_iterations(c, tol, W)), (n_u, stop_iterations(c, tol, W))
    if not w_partials:
        assert np.array_equal(n_u, n_ref)
    for u in range(len(x_list)):
        assert np.isnan(c[u, n_u[u]:]).all() and not np.isnan(c[u, :n_u[u]]).any()
    for k in np.unique(n_u):
        enh_k, _, _ = _enhancer(case, niter=int(k), w_partials=w_partials)
        sk, nk, ck, sck = enh_k.enhance(x_list, **call)
        for u in np.flatnonzero(n_u == k):
            if not w_partials:
                assert np.array_equal(s[u], sk[u]) and np.array_equal(n[u], nk[u]), (case, u, k)
                assert np.array_equal(sc[u], sck[u], equal_nan=True), (case, u, k)
                if emission_mstep:
                    np.testing.assert_allclose(c[u, :k], ck[u], rtol=1e-12, atol=0)
                else:
                    assert np.array_equal(c[u, :k], ck[u]), (case, u, k)
            else:
                if np.linalg.norm(sk[u]) > 0:
                    assert np.linalg.norm(s[u] - sk[u]) / np.linalg.norm(sk[u]) <= 1e-3, (case, u, k)
                np.testing.assert_allclose(c[u, :k], ck[u], rtol=1e-4)
    return enh_s


@pytest.mark.parametrize("case", list(CASES))
def test_stopped_utterances_equal_runs_with_their_iteration_count(case):
    _check_stopping_case(case, False)


def test_stopping_with_fused_w_reduction_agrees_to_rounding():
    _check_stopping_case("M1_tc_keep10", True)


def test_stopping_that_cannot_trigger_is_bit_identical_and_early_exit():
    enh, x_list, call = _enhancer("M1_tc_keep10")
    s0, n0, c0, sc0 = enh.enhance(x_list, **call)
    s0, n0 = [a.copy() for a in s0], [a.copy() for a in n0]
    enh_s, _, _ = _enhancer("M1_tc_keep10", stop_tol=1e30, stop_window=NITER // 2 + 1)        # 2w > niter: never tested
    s1, n1, c1, sc1 = enh_s.enhance(x_list, **call)
    assert all(np.array_equal(a, b) for a, b in zip(s0, s1)) and all(np.array_equal(a, b) for a, b in zip(n0, n1))
    assert np.array_equal(c0, c1) and np.array_equal(sc0, sc1, equal_nan=True)
    assert (enh_s.engine.n_iter == NITER).all()
    # every utterance passes the first test (n = 2w): the loop ends there
    enh_e, _, _ = _enhancer("M1_tc_keep10", stop_tol=1e30, stop_window=3)
    enh_e.engine.timing = True
    _, _, c2, _ = enh_e.enhance(x_list, **call)
    st = enh_e.engine.stage_times_ms()
    eng = enh_e.engine
    assert (eng.n_iter == 6).all() and np.isnan(c2[:, 6:]).all() and np.array_equal(c2[:, :6], c0[:, :6])
    assert eng.mh_calls == 7 and eng.mh_iter0 == 6 * 15 + 15
    assert st["stop_check"][1] == 1 and st["mstep"][1] == 6


def test_process_sublist_with_stopping_matches_enhance(tmp_path):
    wav_dir = str(tmp_path / "in")
    sub = []
    for i in range(7):
        x, s, _ = synth.synth_utterance(70 + i, (16000 + 2345 * i + (i % 2)) / 16000)
        rel = "/spk%d/utt%d.wav" % (i % 2, i)
        batch_io.write_wav(wav_dir + rel, x, 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, s, 16000)
        sub.append((rel, "/clean" + rel))
    enh, _, _ = _enhancer("M1_tc_keep10", stop_tol=2e-3, stop_window=W)
    out = str(tmp_path / "out")
    stems, sc = batch_io.process_sublist(sub, enh, wav_dir, out, batch_size=3, score=True)
    assert len(stems) == 7 and sc.shape == (7, 2, 5)
    ref, n_all = [], []
    for lo in range(0, 7, 3):
        part = sub[lo:lo + 3]
        xs = [batch_io.read_wav(wav_dir + a)[0].astype(np.float32) for a, _ in part]
        cs = [batch_io.read_wav(wav_dir + b)[0].astype(np.float32) for _, b in part]
        ids = [batch_io.utterance_id(a) for a, _ in part]
        s_pcm, _, _, scores = enh.enhance(xs, utt_ids=ids, ref_list=cs, pcm16=True)
        ref.append(scores)
        n_all.append(enh.engine.n_iter.copy())
        for (rel, _), a in zip(part, s_pcm):
            batch_io.write_wav(str(tmp_path / "ref.wav"), a, 16000)
            assert open(batch_io.output_stem(out, rel) + "_s_est.wav", "rb").read() == open(str(tmp_path / "ref.wav"), "rb").read(), rel
    assert np.array_equal(sc, np.concatenate(ref), equal_nan=True)
    assert len(set(np.concatenate(n_all))) > 1
