"""Every M-step and statistics route against the float64 M-step (``mcem_port.m_step_f64``), element by element.

Each output of the kernels -- W, H, g, Vb, the per-utterance cost, A1 / A2 of the statistics pass and every W-update partial sum
``Wpart[seg][k][.][f]`` -- must satisfy ``|gpu - f64| <= bound`` with the bound of ``m_step_f64``'s error model (written out in
``oracle/mcem_port.py``: FP32 rounding along each kernel's longest chain of additions, the approximate reciprocal / logarithm at
their PTX bounds, propagated through the W -> H -> g passes).  No max-normalised tolerance: a quiet frame, a spectral null or a
collapsed gain is held to the same relative bound as the loudest bin.

Input families (all inside the range the kernels handle, ``mcem_port.m_step_in_range``, checked per case):
  control  the benign distribution of the older parity tests;
  late     a late-run state: P the STFT power of a synthetic utterance with a 120 dB spectral null and a run of frames 100 dB
           down, W columns spanning 1e-12 .. 1, H spanning 1e-10 .. 1e3 across frames, g collapsed to 1e-22 .. 1e-12 on every
           third frame;
  floor    a few loud partials over a floor 140 dB below them;
  spread   the samples of one bin spread over 2^+-28 around the bin's first sample (the cost passes' per-bin scale);
  bias     (emission only) a decoder output bias spanning decades, so that the stored bias-free words are far from 1.
The route each case takes is asserted from the host conditions of ``dvae_nmf_mstep`` / ``dvae_nmf_mstep_vst`` /
``dvae_vst_frame_stats`` (mirrored below), and the range limits are tested on both sides: inside, element-wise agreement;
outside, the documented outcome (agreement, or ``DVAE_STATUS_NONFINITE`` from the cost reduction), never silent garbage.
The largest error / bound ratio per (route, output, family) is printed at the end of the module, with the float32 reference's
ratio on the same inputs beside it.
"""
import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth, tc
from dvae_b200.engine import RaggedBatch, VaeWeights, _ld_for, _p, _stream
from oracle import mcem_port
from tests.gpu_util import DEV, fm, unfm

pytestmark = pytest.mark.gpu
NONFINITE = 2                                   # DVAE_STATUS_NONFINITE (include/dvae_b200.h)
SENT = 0xA5
RATIOS = {}                                     # (route, output, family) -> [largest gpu ratio, largest float32-reference ratio]

# ragged batches: one-frame utterances, 7 / 8 / 9 frames, offsets that are not multiples of 8 (short first / last hg7 blocks),
# an utterance crossing the 128-frame tile (several W segments), and a last tile holding one frame
LENS_RAW = [1, 9, 7, 8, 21]
LENS_VST = [3, 7, 9, 8, 1, 101]                 # offsets 0 3 10 19 27 28; 129 frames: the last tile holds frame 128 alone
LENS_CHAINS = {2: [3, 7, 9, 8, 1, 36], 4: [3, 7, 9, 8, 1, 4], 16: [3, 7, 9, 8, 1], 128: [1, 3, 5]}


@pytest.fixture(scope="module", autouse=True)
def _ratio_table():
    yield
    if RATIOS:
        print("\nlargest |gpu - f64| / bound (float32 reference beside it)")
        for (route, out, fam), (r, r32) in sorted(RATIOS.items()):
            print("  %-28s %-6s %-8s %9.3g %9s" % (route, out, fam, r, "-" if r32 is None else "%.3g" % r32))


# --------------------------------------------------------------------------------------------- input families
def _stft_power(N, seed):
    x, _, _ = synth.synth_utterance(seed, (N * 256 + 1024) / 16000 + 0.01)
    idx = np.arange(1024)[None, :] + 256 * np.arange(N)[:, None]
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(1024) / 1024)
    return (np.abs(np.fft.rfft(x.astype(np.float64)[idx] * w, axis=1)) ** 2).T           # (513, N)


def family(name, F, N, K, R, seed):
    """``(P (F,N), Vs (R,F,N), W (F,K), H (K,N), g (N,))`` float32 of one input family (module docstring)."""
    rng = np.random.default_rng(seed)
    P = rng.gamma(1.0, 1.0, size=(F, N)) * 0.1
    Vs = rng.gamma(2.0, 0.05, size=(R, F, N))
    W = np.maximum(rng.uniform(size=(F, K)), 1e-8)
    H = np.maximum(rng.uniform(size=(K, N)), 1e-8)
    g = rng.uniform(0.5, 1.5, size=N)
    if name == "late":
        lo, hi = F // 5, F // 5 + max(1, F // 12)
        q0, q1 = N // 3, N // 3 + max(1, N // 5)
        P = _stft_power(N, seed % 7)[:F]
        P = P / P.mean() * 0.1
        P[lo:hi] *= 1e-12                                               # 120 dB spectral null
        P[:, q0:q1] *= 1e-10                                            # a run of frames 100 dB down
        shape = np.ones((F, N))
        shape[lo:hi] = 1e-12                                            # the speech model has learnt both
        shape[:, q0:q1] = 1e-10
        Vs = Vs * shape
        W = 10.0 ** rng.uniform(-12, 0, size=(F, K))
        H = 10.0 ** rng.uniform(-10, 3, size=(K, N))
        g[::3] = 10.0 ** rng.uniform(-22, -12, size=len(g[::3]))        # collapsed gains: the NMF carries these frames alone
        H[:, ::3] = 10.0 ** rng.uniform(-1, 3, size=(K, len(g[::3])))
        g[q0:q1] = rng.uniform(0.5, 1.5, size=q1 - q0)
        H[:, q0:q1] = 10.0 ** rng.uniform(-10, -6, size=(K, q1 - q0))
    elif name == "floor":
        part = np.arange(F) % 64 == 40
        P = rng.gamma(1.0, 1e-12, size=(F, N))
        P[part] = rng.gamma(2.0, 50.0, size=P[part].shape)              # partials 140 dB above the floor
        Vs = Vs * np.where(part, 1.0, 1e-12)[None, :, None]
        W = W * 1e-6
    elif name == "spread":
        Vs[1:] = Vs[:1] * 2.0 ** rng.uniform(-28, 28, size=(R - 1, F, N))
        W = W * 1e-12
    f32 = lambda a: np.ascontiguousarray(a, np.float32)
    return f32(P), f32(Vs), f32(W), f32(H), f32(g)


def _weights(bias):
    if bias == "speech":                                                # E[f] = exp(b3[f]) spanning decades
        _, s, _ = synth.synth_utterance(5, 1.0)
        out_bias = synth.speech_prior_bias(s)
    else:
        out_bias = (np.log(0.05) + np.linspace(-1.0, 1.0, 513)).astype(np.float32)
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128], 0, seed=5, out_bias=out_bias)
    return VaeWeights(sd, "M1", torch.device(DEV))


# --------------------------------------------------------------------------------------------- routes (host conditions)
def mstep_route(F, ld, K, R, vs_ptr, max_frames, wstat):
    """The kernels ``dvae_nmf_mstep`` (nmf.cu) launches for these arguments: (W kernel, H / g / cost kernel)."""
    w = "w_from_frame_stats" if wstat else "nmf_w"
    if max_frames == 0:
        return w, None
    fast = F == 513 and ld == 520 and K <= 10 and vs_ptr % 16 == 0
    if fast and R > 30 and R % 10 == 0:
        return w, "hg6<30>" if R % 30 == 0 else "hg6<10>"
    if fast and R in (10, 30):
        return w, "hg5<%d>" % R
    return w, "hg_generic"


def vst_route(R, C, wpart):
    """``dvae_nmf_mstep_vst``: W from the partials or from A1 / A2, then hg7 (one chain per frame) or the windowed hg7w."""
    return ("w_from_partials" if wpart else "w_from_frame_stats"), ("hg7w<%d>" if C > 1 else "hg7<%d>") % R


def stats_route(R):
    return "vst_frame_stats<%d>" % (R if R in (10, 30) else 0)


# --------------------------------------------------------------------------------------------- comparison
def _score(got, ref, bound):
    got, ref, bound = (np.atleast_1d(np.asarray(a, np.float64)) for a in (got, ref, bound))
    err = np.abs(got - ref)
    ratio = np.where(err == 0, 0.0, err / np.where(bound > 0, bound, 1e-300))
    ratio[~np.isfinite(got)] = np.inf
    return ratio


def _check(route, out, fam, got, ref, bound, fails, f32=None):
    ratio = _score(got, ref, bound)
    r = float(ratio.max()) if ratio.size else 0.0
    r32 = None if f32 is None else (float(_score(f32, ref, bound).max()) if ratio.size else 0.0)
    old = RATIOS.get((route, out, fam), [0.0, None])
    RATIOS[(route, out, fam)] = [max(old[0], r), r32 if old[1] is None else max(old[1], r32 or 0.0)]
    if not r <= 1.0:
        i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
        got, ref, bound = (np.atleast_1d(np.asarray(a, np.float64)) for a in (got, ref, bound))
        fails.append("%s %s [%s]: |gpu - f64| / bound = %.3g at %s (gpu %r, f64 %r, bound %.3g)"
                     % (route, out, fam, r, i, got[i], np.broadcast_to(ref, got.shape)[i], np.broadcast_to(bound, got.shape)[i]))


def _reference(P, Vs, W, H, g, a, b, **kw):
    ref = mcem_port.m_step_f64(P[:, a:b], Vs[:, :, a:b], W, H[:, a:b], g[a:b], **kw)
    f32 = mcem_port.m_step_reference(*(torch.tensor(np.ascontiguousarray(x)) for x in
                                       (P[:, a:b], Vs[:, :, a:b], W, H[:, a:b], g[a:b])))
    return ref, {k: v.numpy() for k, v in f32.items()}


def _compare_utterances(route, fam, P, Vs, W, H, g, batch, Wd, Hd, gd, Vbd, cost, fails, seg_frames=None, chains=1,
                        stats_rel=None):
    F = P.shape[0]
    off = batch.fr_off_host
    for u in range(batch.B):
        a, b = int(off[u]), int(off[u + 1])
        kw = dict(chains=chains, stats_rel=stats_rel, segments=None if seg_frames is None else seg_frames[u])
        ref, f32 = _reference(P, Vs, W, H, g, a, b, **kw)
        assert mcem_port.m_step_in_range(ref), (fam, u, ref["vx_min"], ref["vx_max"], ref["spread_log2"])
        _check(route, "W", fam, Wd[u, :, :F].t().cpu().numpy(), ref["W"], ref["bound_W"], fails, f32["W"])
        _check(route, "H", fam, Hd[a:b].t().cpu().numpy(), ref["H"], ref["bound_H"], fails, f32["H"])
        _check(route, "g", fam, gd[a:b].cpu().numpy(), ref["g"], ref["bound_g"], fails, f32["g"])
        _check(route, "Vb", fam, unfm(Vbd[a:b], F), ref["Vb"], ref["bound_Vb"], fails, f32["Vb"])
        _check(route, "cost", fam, cost[u].item(), ref["cost"], ref["bound_cost"], fails, f32["cost"])


# --------------------------------------------------------------------------------------------- FP32-variance M-step
def _run_raw(P, Vs, W, H, g, lens, misalign=False, wstat=None):
    F, K, R = P.shape[0], W.shape[1], Vs.shape[0]
    ld = _ld_for(F)
    batch = RaggedBatch(lens, DEV)
    B, N = batch.B, batch.NT
    rows = max(N, 1)
    Pd = torch.zeros((rows, ld), device=DEV)
    Pd[:N, :F] = torch.from_numpy(np.ascontiguousarray(P.T)).to(DEV)
    flat = torch.zeros(rows * R * ld + 4, device=DEV)
    Vsd = flat[(1 if misalign else 0):][: rows * R * ld].view(rows, R, ld)       # misaligned: 4 bytes off 16
    Vsd[:N, :, :F] = torch.from_numpy(np.ascontiguousarray(Vs.transpose(2, 0, 1))).to(DEV)
    Wd = torch.zeros((B, K, ld), device=DEV)
    Wd[:, :, :F] = torch.from_numpy(np.ascontiguousarray(W.T)).to(DEV)[None]
    Hd = torch.zeros((rows, K), device=DEV)
    Hd[:N] = torch.from_numpy(np.ascontiguousarray(H.T)).to(DEV)
    gd = torch.ones(rows, device=DEV)
    gd[:N] = torch.from_numpy(g).to(DEV)
    Vbd = torch.zeros((rows, ld), device=DEV)
    if N:
        _lib.call("dvae_nmf_vb", _p(Wd), _p(Hd), _p(batch.frame_utt), N, F, K, ld, _p(Vbd), _stream())
    ws_stat = None
    if wstat is not None:
        ws_stat = torch.zeros(2 * rows * ld, device=DEV)
        ws_stat.view(2, rows, ld)[:, :N, :F] = torch.from_numpy(np.ascontiguousarray(wstat.transpose(0, 2, 1))).to(DEV)
    cost = torch.full((B,), 7.0, dtype=torch.float64, device=DEV)
    st = torch.zeros(1, dtype=torch.int32, device=DEV)
    ws = torch.empty(int(_lib.load().dvae_nmf_workspace_floats(B, K, ld, batch.max_frames)) + 2, device=DEV)
    route = mstep_route(F, ld, K, R, Vsd.data_ptr(), batch.max_frames, wstat is not None)
    _lib.call("dvae_nmf_mstep", _p(Pd), _p(Vsd), R, _p(Wd), _p(Hd), _p(gd), _p(Vbd), _p(cost), _p(batch.fr_off),
              _p(batch.frame_utt), B, N, F, K, ld, batch.max_frames, _p(ws), _p(ws_stat), _p(st), _stream())
    torch.cuda.synchronize()
    return route, batch, Wd, Hd[:N], gd[:N], Vbd[:N], cost, int(st.item())


RAW_CASES = [  # F, K, R, misaligned Vs, expected (W kernel, H / g / cost kernel)
    (33, 1, 1, False, "hg_generic"), (33, 3, 7, False, "hg_generic"), (513, 10, 1, False, "hg_generic"),
    (513, 7, 7, False, "hg_generic"), (513, 10, 10, True, "hg_generic"),
    (513, 7, 10, False, "hg5<10>"), (513, 10, 30, False, "hg5<30>"),
    (513, 10, 60, False, "hg6<30>"), (513, 7, 90, False, "hg6<30>"), (513, 10, 40, False, "hg6<10>"), (513, 3, 160, False, "hg6<10>"),
]


@pytest.mark.parametrize("fam", ["control", "late", "floor", "spread"])
@pytest.mark.parametrize("F,K,R,misalign,hg", RAW_CASES)
def test_m_step_on_fp32_variances_against_f64(F, K, R, misalign, hg, fam):
    lens = LENS_RAW if R < 100 else LENS_RAW[:4]
    P, Vs, W, H, g = family(fam, F, sum(lens), K, R, seed=F + K + R)
    route, batch, Wd, Hd, gd, Vbd, cost, st = _run_raw(P, Vs, W, H, g, lens, misalign=misalign)
    assert route == ("nmf_w", hg)
    assert st == 0
    fails = []
    _compare_utterances("%s+%s" % route, fam, P, Vs, W, H, g, batch, Wd, Hd, gd, Vbd, cost, fails)
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("fam", ["control", "late", "floor", "spread"])
@pytest.mark.parametrize("K,R", [(10, 10), (7, 30)])
def test_m_step_from_frame_statistics_against_f64(K, R, fam):
    """``dvae_nmf_mstep`` with ``wstat``: A1 / A2 are the float64 oracle's, rounded to FP32 (relative error u)."""
    lens = LENS_RAW
    P, Vs, W, H, g = family(fam, 513, sum(lens), K, R, seed=3 * K + R)
    batch = RaggedBatch(lens, DEV)
    A = np.zeros((2, 513, batch.NT))
    for u in range(batch.B):
        a, b = int(batch.fr_off_host[u]), int(batch.fr_off_host[u + 1])
        ref = mcem_port.m_step_f64(P[:, a:b], Vs[:, :, a:b], W, H[:, a:b], g[a:b])
        A[0, :, a:b], A[1, :, a:b] = ref["A1"], ref["A2"]
    route, batch, Wd, Hd, gd, Vbd, cost, st = _run_raw(P, Vs, W, H, g, lens, wstat=A.astype(np.float32))
    assert route == ("w_from_frame_stats", "hg5<%d>" % R) and st == 0
    fails = []
    _compare_utterances("%s+%s" % route, fam, P, Vs, W, H, g, batch, Wd, Hd, gd, Vbd, cost, fails, stats_rel=mcem_port.U32)
    assert not fails, "\n".join(fails)


def test_m_step_without_frames_zeroes_the_cost_and_still_updates_w():
    """``max_frames = 0``: the W pass runs (0 / 0 for every bin, as in the reference), no H / g / cost kernel, cost = 0."""
    F, K, R = 513, 10, 10
    P, Vs, W, H, g = family("control", F, 0, K, R, seed=1)
    route, batch, Wd, Hd, gd, Vbd, cost, st = _run_raw(P, Vs, W, H, g, [0, 0])
    assert route == ("nmf_w", None) and st == 0
    ref = mcem_port.m_step_reference(*(torch.tensor(x) for x in (P, Vs, W, H, g)))
    assert np.all(np.isnan(ref["W"].numpy())) and bool(torch.isnan(Wd[:, :, :F]).all())
    assert bool((Wd[:, :, F:] == 0).all())
    assert cost.tolist() == [0.0, 0.0]


# --------------------------------------------------------------------------------------------- the sampler's emission
def _emission(w, Vs, C):
    """Pack ``Vs`` (R = C x Rc, F, N) as C chain rows of Rc samples per frame (with repeated slots, as rejected proposals
    leave them) and return ``(vst, idx, Vq)``: Vq = what the kernels see, unpacked, (R, F, N) float32."""
    R, F, N = Vs.shape
    Rc, NC, ld = R // C, N * C, 520
    Vsd = torch.zeros((N, R, ld), device=DEV)
    Vsd[:, :, :F] = torch.from_numpy(np.ascontiguousarray(Vs.transpose(2, 0, 1))).to(DEV)
    img = tc.decoder_image(w)
    nbytes = int(_lib.load().dvae_vst_bytes(NC, Rc))
    vst = torch.full((nbytes + 4096,), SENT, dtype=torch.uint8, device=DEV)
    idx = torch.full(((NC + 2) * 32,), SENT, dtype=torch.uint8, device=DEV)
    _lib.call("dvae_vst_pack", w.dec.ref, _p(img), w.z_dim, w.y_dim, _p(Vsd), Rc, NC, ld, _p(vst), _p(idx), _stream())
    rng = np.random.default_rng(R + N)
    it = idx.view(-1, 32)
    rep = torch.tensor(rng.uniform(size=(NC, Rc)) < 0.2).to(DEV)
    rep[:, 0] = False
    for r in range(1, Rc):
        it[:NC, r] = torch.where(rep[:, r], it[:NC, r - 1], it[:NC, r])
    out = torch.full((NC + 1, Rc, ld), -7.0, device=DEV)
    _lib.call("dvae_vst_unpack", w.dec.ref, _p(img), w.z_dim, w.y_dim, _p(vst), _p(idx), Rc, NC, ld, _p(out), _stream())
    Vq = out[:NC, :, :F].reshape(N, R, F).permute(1, 2, 0).cpu().numpy()
    return vst, idx, np.ascontiguousarray(Vq)


def _emission_family(fam, N, K, R, seed):
    bias = "speech" if fam == "bias" else "plain"
    return _weights(bias), family("control" if fam == "bias" else fam, 513, N, K, R, seed)


EMISSION_FAMILIES = ["control", "late", "floor", "spread", "bias"]


@pytest.mark.parametrize("fam", EMISSION_FAMILIES)
@pytest.mark.parametrize("R", [1, 7, 10, 25, 30, 31])
def test_frame_statistics_against_f64(R, fam):
    """``dvae_vst_frame_stats``: A1 / A2 of every (frame, bin), compile-time R = 10 / 30 and the run-time-R instance."""
    N, K, ld = 130, 10, 520
    w, (P, Vs, W, H, g) = _emission_family(fam, N, K, R, seed=R + 17)
    vst, idx, Vq = _emission(w, Vs, 1)
    Hd = torch.from_numpy(np.ascontiguousarray(H.T)).to(DEV)
    Wd = torch.zeros((1, K, ld), device=DEV)
    Wd[0, :, :513] = torch.from_numpy(np.ascontiguousarray(W.T)).to(DEV)
    Vbd = torch.zeros((N, ld), device=DEV)
    _lib.call("dvae_nmf_vb", _p(Wd), _p(Hd), _p(torch.zeros(N, dtype=torch.int32, device=DEV)), N, 513, K, ld, _p(Vbd), _stream())
    fstat = torch.full((2 * N * ld + 64,), float("nan"), device=DEV)
    _lib.call("dvae_vst_frame_stats", w.dec.ref, _p(tc.decoder_image(w)), 16, 0, _p(vst), _p(idx), R, _p(Vbd),
              _p(torch.from_numpy(g).to(DEV)), N, ld, _p(fstat), _p(fstat[N * ld:]), _stream())
    torch.cuda.synchronize()
    assert bool(torch.isnan(fstat[2 * N * ld:]).all()) and bool(torch.isnan(fstat[: 2 * N * ld].view(2, N, ld)[..., 513:]).all())
    ref = mcem_port.m_step_f64(P, Vq, W, H, g)
    fails = []
    for i, k in enumerate(("A1", "A2")):
        _check(stats_route(R), k, fam, unfm(fstat[i * N * ld:(i + 1) * N * ld].view(N, ld), 513), ref[k], ref["bound_" + k], fails)
    assert not fails, "\n".join(fails)


def _segments_by_utterance(batch, C):
    seg_start, tile_seg, utt_seg, S = batch.segments(n_chains=C)
    cuts = seg_start.cpu().numpy() // C                                  # chain rows -> frames (a frame's chains share a tile)
    us = utt_seg.cpu().numpy()
    per = []
    for u in range(batch.B):
        a = int(batch.fr_off_host[u])
        per.append([(int(cuts[s]) - a, int(cuts[s + 1]) - a) for s in range(us[u], us[u + 1])])
    return seg_start, tile_seg, utt_seg, S, per


def _run_vst(fam, lens, K, Rc, C, wpart, seed):
    R, ld = Rc * C, 520
    batch = RaggedBatch(lens, DEV)
    B, N = batch.B, batch.NT
    w, (P, Vs, W, H, g) = _emission_family(fam, N, K, R, seed)
    vst, idx, Vq = _emission(w, Vs, C)
    img = tc.decoder_image(w)
    Pd = fm(P)
    Wd = torch.zeros((B, K, ld), device=DEV)
    Wd[:, :, :513] = torch.from_numpy(np.ascontiguousarray(W.T)).to(DEV)[None]
    Hd = torch.from_numpy(np.ascontiguousarray(H.T)).to(DEV).contiguous()
    gd = torch.from_numpy(g).to(DEV)
    Vbd = torch.zeros((N, ld), device=DEV)
    _lib.call("dvae_nmf_vb", _p(Wd), _p(Hd), _p(batch.frame_utt), N, 513, K, ld, _p(Vbd), _stream())
    fails, seg_frames, fstat, wp, utt_seg = [], None, None, None, None
    if wpart:
        seg_start, tile_seg, utt_seg, S, seg_frames = _segments_by_utterance(batch, C)
        wp = torch.full((int(_lib.load().dvae_vst_w_partial_floats(S, K, ld)) + 64,), float("nan"), device=DEV)
        _lib.call("dvae_vst_w_partials", w.dec.ref, _p(img), 16, 0, _p(vst), _p(idx), Rc, _p(Pd), _p(Vbd), _p(gd), _p(Hd), K, N, C, ld,
                  _p(seg_start), _p(tile_seg), _p(wp), _stream())
        torch.cuda.synchronize()
        body = wp[:-64].view(S, K, 2, ld)
        assert bool(torch.isnan(wp[-64:]).all()) and bool(torch.isnan(body[..., 513:]).all()), "partials written outside [S][K][2][0..F)"
        got = body[..., :513].cpu().numpy()
        us = utt_seg.cpu().numpy()
        for u in range(B):
            a, b = int(batch.fr_off_host[u]), int(batch.fr_off_host[u + 1])
            ref = mcem_port.m_step_f64(P[:, a:b], Vq[:, :, a:b], W, H[:, a:b], g[a:b], segments=seg_frames[u], chains=C)
            rel = np.array(ref["rel_Wsum"])[None, None, :, None]
            _check("vst_frame_stats<%d,wpart>" % (Rc if Rc in (10, 30) else 0), "Wpart", fam, got[us[u]:us[u + 1]], ref["Wpart"],
                   rel * ref["Wpart"], fails)
    else:
        fstat = torch.zeros(2 * N * ld, device=DEV)
        _lib.call("dvae_vst_frame_stats", w.dec.ref, _p(img), 16, 0, _p(vst), _p(idx), Rc, _p(Vbd), _p(gd), N, ld, _p(fstat),
                  _p(fstat[N * ld:]), _stream())
    cost = torch.full((B,), 7.0, dtype=torch.float64, device=DEV)
    st = torch.zeros(1, dtype=torch.int32, device=DEV)
    ws = torch.empty(int(_lib.load().dvae_nmf_workspace_floats(B, K, ld, batch.max_frames)), device=DEV)
    _lib.call("dvae_nmf_mstep_vst", w.dec.ref, _p(img), 16, 0, _p(Pd), _p(vst), _p(idx), Rc, _p(Wd), _p(Hd), _p(gd), _p(Vbd), _p(cost),
              _p(batch.fr_off), B, N, K, ld, batch.max_frames, _p(ws), _p(fstat), _p(wp), _p(utt_seg), C, _p(st), _stream())
    torch.cuda.synchronize()
    return dict(P=P, Vq=Vq, W=W, H=H, g=g, batch=batch, Wd=Wd, Hd=Hd, gd=gd, Vbd=Vbd, cost=cost, st=int(st.item()), fails=fails,
                seg_frames=seg_frames, route=vst_route(Rc, C, wpart))


@pytest.mark.parametrize("fam", EMISSION_FAMILIES)
@pytest.mark.parametrize("K,Rc,wpart", [(1, 10, False), (7, 30, False), (10, 10, False), (1, 30, True), (7, 10, True), (10, 30, True)])
def test_m_step_on_the_emission_against_f64(K, Rc, wpart, fam):
    r = _run_vst(fam, LENS_VST, K, Rc, 1, wpart, seed=K + Rc)
    assert r["route"][1] == "hg7<%d>" % Rc and r["st"] == 0
    fails = r["fails"]
    _compare_utterances("%s+%s" % r["route"], fam, r["P"], r["Vq"], r["W"], r["H"], r["g"], r["batch"], r["Wd"], r["Hd"], r["gd"],
                        r["Vbd"], r["cost"], fails, seg_frames=r["seg_frames"])
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("fam", EMISSION_FAMILIES)
@pytest.mark.parametrize("C,Rc", [(2, 30), (4, 10), (16, 10), (128, 10)])
def test_m_step_on_several_chains_per_frame_against_f64(C, Rc, fam):
    """``nmf_hg7w_kernel``: C chains x Rc kept samples per frame, walked in windows of 30; partial sums over chain rows."""
    r = _run_vst(fam, LENS_CHAINS[C], 10, Rc, C, True, seed=C + Rc)
    assert r["route"] == ("w_from_partials", "hg7w<%d>" % Rc) and r["st"] == 0
    fails = r["fails"]
    _compare_utterances("%s+%s" % r["route"], fam, r["P"], r["Vq"], r["W"], r["H"], r["g"], r["batch"], r["Wd"], r["Hd"], r["gd"],
                        r["Vbd"], r["cost"], fails, seg_frames=r["seg_frames"], chains=C)
    assert not fails, "\n".join(fails)


# --------------------------------------------------------------------------------------------- the stated range, both sides
def _scaled(kind, F, N, K, R, seed):
    """Inputs at one side of a range limit.  Scaling P, Vs and W by s scales every Vx of the M-step by s (the updates are
    scale-invariant), so the control family moves whole to the limit; 'spread' puts every sample but the first 2^34 above it."""
    P, Vs, W, H, g = family("control", F, N, K, R, seed)
    s = {"low_in": 2.0 ** -48, "low_out": 2.0 ** -70, "high_in": 2.0 ** 56, "high_out": 2.0 ** 75}.get(kind)
    if s is not None:
        return P * np.float32(s), Vs * np.float32(s), W * np.float32(s), H, g
    Vs[1:] = Vs[:1] * np.float32(2.0 ** 34)
    return P, Vs, W * np.float32(1e-12), H, g


# outside a limit: "nonfinite" = DVAE_STATUS_NONFINITE from the cost reduction (a pair product or its reciprocal flushed makes
# 0 / 0 or inf of the W / H sums; an overflowing product of four samples makes the cost infinite); "agree" = within the bound
# (the generic kernel has no per-bin scale: its cost takes one IEEE logarithm per sample)
OUTSIDE = {"low_out": "nonfinite", "high_out": "nonfinite", "spread_out": "nonfinite"}
OUTSIDE_GENERIC = dict(OUTSIDE, spread_out="agree")


@pytest.mark.parametrize("kind", ["low_in", "low_out", "high_in", "high_out", "spread_out"])
@pytest.mark.parametrize("F,K,R,hg", [(513, 10, 7, "hg_generic"), (513, 10, 10, "hg5<10>")])
def test_fp32_m_step_at_the_range_limits(F, K, R, hg, kind):
    lens = LENS_RAW
    P, Vs, W, H, g = _scaled(kind, F, sum(lens), K, R, seed=R)
    route, batch, Wd, Hd, gd, Vbd, cost, st = _run_raw(P, Vs, W, H, g, lens)
    assert route == ("nmf_w", hg)
    _expect_at_limit("%s+%s" % route, kind, P, Vs, W, H, g, batch, Wd, Hd, gd, Vbd, cost, st,
                     (OUTSIDE_GENERIC if hg == "hg_generic" else OUTSIDE).get(kind))


@pytest.mark.parametrize("kind", ["low_in", "low_out", "high_in", "high_out", "spread_out"])
def test_emission_m_step_at_the_range_limits(kind):
    lens, K, Rc = LENS_VST, 10, 10
    batch = RaggedBatch(lens, DEV)
    P, Vs, W, H, g = _scaled(kind, 513, batch.NT, K, Rc, seed=4)
    w = _weights("plain")
    vst, idx, Vq = _emission(w, Vs, 1)
    ld, B, N = 520, batch.B, batch.NT
    Pd, img = fm(P), tc.decoder_image(w)
    Wd = torch.zeros((B, K, ld), device=DEV)
    Wd[:, :, :513] = torch.from_numpy(np.ascontiguousarray(W.T)).to(DEV)[None]
    Hd = torch.from_numpy(np.ascontiguousarray(H.T)).to(DEV).contiguous()
    gd = torch.from_numpy(g).to(DEV)
    Vbd = torch.zeros((N, ld), device=DEV)
    _lib.call("dvae_nmf_vb", _p(Wd), _p(Hd), _p(batch.frame_utt), N, 513, K, ld, _p(Vbd), _stream())
    fstat = torch.zeros(2 * N * ld, device=DEV)
    _lib.call("dvae_vst_frame_stats", w.dec.ref, _p(img), 16, 0, _p(vst), _p(idx), Rc, _p(Vbd), _p(gd), N, ld, _p(fstat), _p(fstat[N * ld:]),
              _stream())
    cost = torch.zeros(B, dtype=torch.float64, device=DEV)
    st = torch.zeros(1, dtype=torch.int32, device=DEV)
    ws = torch.empty(int(_lib.load().dvae_nmf_workspace_floats(B, K, ld, batch.max_frames)), device=DEV)
    _lib.call("dvae_nmf_mstep_vst", w.dec.ref, _p(img), 16, 0, _p(Pd), _p(vst), _p(idx), Rc, _p(Wd), _p(Hd), _p(gd), _p(Vbd), _p(cost),
              _p(batch.fr_off), B, N, K, ld, batch.max_frames, _p(ws), _p(fstat), None, None, 1, _p(st), _stream())
    torch.cuda.synchronize()
    _expect_at_limit("%s+%s" % vst_route(Rc, 1, False), kind, P, Vq, W, H, g, batch, Wd, Hd, gd, Vbd, cost, int(st.item()),
                     OUTSIDE.get(kind))


def _expect_at_limit(route, kind, P, Vs, W, H, g, batch, Wd, Hd, gd, Vbd, cost, st, expected):
    inside = kind.endswith("_in")
    refs = [mcem_port.m_step_f64(P[:, a:b], Vs[:, :, a:b], W, H[:, a:b], g[a:b])
            for a, b in zip(batch.fr_off_host[:-1].tolist(), batch.fr_off_host[1:].tolist())]
    assert all(mcem_port.m_step_in_range(r) for r in refs) == inside, kind
    fails = []
    if inside or st == 0:
        _compare_utterances(route, kind, P, Vs, W, H, g, batch, Wd, Hd, gd, Vbd, cost, fails) if inside else \
            _compare_outside(route, kind, refs, P, batch, Wd, Hd, gd, Vbd, cost, fails)
    outcome = "nonfinite" if st == NONFINITE else ("agree" if st == 0 and not fails else "wrong")
    if inside:
        assert st == 0 and not fails, "\n".join(fails)
    else:
        assert outcome == expected, "outside the range: %s (status %d), expected %s\n%s" % (outcome, st, expected, "\n".join(fails))


def _compare_outside(route, kind, refs, P, batch, Wd, Hd, gd, Vbd, cost, fails):
    F = P.shape[0]
    off = batch.fr_off_host
    for u, ref in enumerate(refs):
        a, b = int(off[u]), int(off[u + 1])
        for k, got in (("W", Wd[u, :, :F].t().cpu().numpy()), ("H", Hd[a:b].t().cpu().numpy()), ("g", gd[a:b].cpu().numpy()),
                       ("Vb", unfm(Vbd[a:b], F))):
            ratio = _score(got, ref[k], ref["bound_" + k])
            if not ratio.max() <= 1.0:
                fails.append("%s %s [%s]: ratio %.3g" % (route, k, kind, ratio.max()))
        if not abs(cost[u].item() - ref["cost"]) <= ref["bound_cost"]:
            fails.append("%s cost [%s]: %r vs %r" % (route, kind, cost[u].item(), ref["cost"]))
