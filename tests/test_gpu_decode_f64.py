"""The tensor-core decode kernels and the final Wiener filter against float64, element by element.

* ``dvae_decode_tc`` and the Vs that ``dvae_decode_stats_tc`` / ``dvae_decode_stats_win_tc`` write: every element inside the
  interval of the float64 mirror (``oracle/decode_mirror.py``: the kernels' rounding points, tensor-core accumulation at one
  ulp per addition, ``tanh.approx.f32`` of the device on the FP32 ends of each pre-activation interval).
* A1 / A2 of the statistics kernels and the mask sums of ``dvae_decode_wiener_tc`` against float64 sums over the kernel's
  OWN written Vs (only FP32 arithmetic in the bound), or over the mirror's Vs interval for R = 25, which has no storing
  instance; ``WFn`` of the filter bit-identical to ``fl(Vb A1)`` of the storing instance on the same samples.
* ``dvae_wiener_accum`` (FP32 route), ``dvae_wiener_apply`` and ``McemEngine.wiener()`` end to end.

No max-normalised tolerance: ``|gpu - f64| <= bound`` for every element, so a collapsed gain or a spectral null is held to
the same relative bound as the loudest bin.  Sizes include steady-state ones: every CTA of the persistent kernels (148 of
them) works through at least three tiles (activation buffers reused, the W3 / accumulator ring wrapped, the next tile's Vb / g
prefetched) and the tile count is not a multiple of 148.

Input families (g, Vb and the decoder; nothing else reaches these kernels):
  benign   g ~ U(0.5, 1.5), Vb ~ Gamma around the speech level;
  late     g collapsed to 1e-22 .. 1e-12 on every third frame and Vb with a 120 dB null: g Vs << Vb, the masks ~ 1e-12;
  speech   Vb << g Vs: WFn small;
  bias     a decoder output bias spanning decades (``synth.speech_prior_bias``);
  edge     the sampler replay's edge decoder with v + b < -126 in every fifth bin: Vs flushes to zero there.
The largest error / bound ratio per (kernel, output, family) is printed at the end of the module.
"""
import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth, tc
from dvae_b200.engine import McemConfig, McemEngine, RaggedBatch, VaeWeights, _p, _stream, mcem_route
from oracle import decode_mirror as dm
from tests.gpu_util import DEV

pytestmark = pytest.mark.gpu
F, LD = 513, 520
NONFINITE = 2                                   # DVAE_STATUS_NONFINITE (include/dvae_b200.h)
SENT = -7.0
RATIOS = {}                                     # (kernel, output, family) -> largest |gpu - f64| / bound
LENS_SMALL = [1, 3, 4, 5, 12, 13, 37]           # crosses the 4- and 12-frame tiles of R = 30 / 25 and R = 10


@pytest.fixture(scope="module", autouse=True)
def _ratio_table():
    yield
    if RATIOS:
        print("\nlargest |gpu - f64| / bound")
        for (kern, out, fam), r in sorted(RATIOS.items()):
            print("  %-30s %-6s %-7s %9.3g" % (kern, out, fam, r))


def _check(kern, out, fam, got, ref, bound):
    got, ref, bound = (torch.as_tensor(a).to(DEV, torch.float64) for a in (got, ref, bound))
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


# --------------------------------------------------------------------------------------------- activation, decoders, families
def _act(x):
    y = torch.empty_like(x)
    _lib.call("dvae_tc_tanh_f32", _p(x), _p(y), x.numel(), _stream())
    return y


_DROP = []


def _tanh_drop():
    """The largest fall of tanh.approx.f32 over every finite FP32 input in [-10, 10] (chunks on the device):
    max over x1 < x2 of act(x1) - act(x2); 0 for a monotone activation.  The mirror widens its activation ends by it."""
    if not _DROP:
        top = int(np.array(10.0, np.float32).view(np.int32))
        chunk = 1 << 26
        worst = 0.0
        for sign in (1.0, -1.0):
            run = None
            for b0 in range(0, top + 1, chunk):
                x = torch.arange(b0, min(top + 1, b0 + chunk), device=DEV, dtype=torch.int32).view(torch.float32) * sign
                y = _act(x) * sign                              # |x| ascending; ascending too if monotone (odd function)
                if run is not None:
                    y = torch.cat([run, y])
                high = torch.cummax(y, 0).values
                worst = max(worst, float((high - y).max()))
                run = high[-1:].clone()
        _DROP.append(worst)
    return _DROP[0]


def test_tanh_approx_f32_is_monotone_up_to_a_small_measured_fall():
    """The mirror's interval step evaluates the activation at the ends of each interval.  tanh.approx.f32 is not exactly
    monotone (B200: it falls by 3.4e-6 in places); the mirror widens the ends by the measured fall, which must stay far
    below a BF16 step of the activation (2^-9 relative) for the interval to stay useful."""
    drop = _tanh_drop()
    print("\ntanh.approx.f32: largest fall over [-10, 10] = %.3g" % drop)
    assert drop <= 2.0 ** -16


def _decoder(kind, bias="plain"):
    """(state dict, variant, L, y_dim) of a decoder configuration."""
    if bias == "bias":
        _, s, _ = synth.synth_utterance(5, 1.0)
        out_bias = synth.speech_prior_bias(s)
    else:
        out_bias = (np.log(0.05) + np.linspace(-1.0, 1.0, F)).astype(np.float32)
    variant, L, h, y_dim = {"M1": ("M1", 16, [128, 128], 0), "M2": ("M2", 16, [128, 128], 1), "ibm": ("M2", 16, [128, 128], F),
                            "L32": ("M1", 32, [128], 0), "L32y3": ("M2", 32, [128], 3)}[kind]
    sd = synth.xavier_state_dict(variant, F, L, h, y_dim, seed=5, out_bias=out_bias)
    if bias == "edge":
        from tests.test_gpu_sampler_replay import _edge_decoder
        bins = _edge_decoder(sd)
        sd["decoder.reconstruction.bias"][bins] = np.float32(-10.0 / 1.4426950408889634)    # v + b = -129.5: flushed
    return sd, variant, L, y_dim


def _weights(kind, bias="plain"):
    sd, variant, L, y_dim = _decoder(kind, bias)
    w = VaeWeights(sd, variant, torch.device(DEV))
    return w, dm.DecodeMirror(sd, L, device=DEV, label_bias=w.tc_label_bias, act=_act, act_step=_tanh_drop())


def _family(fam, NT, seed):
    """g [NT], Vb [NT][LD] (pad columns SENT) of one input family."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    g = 0.5 + torch.rand(NT, device=DEV, generator=gen)
    Vb = torch.empty((NT, F), device=DEV).exponential_(generator=gen) * 0.05 + 1e-4
    if fam == "late":
        g[::3] = 10.0 ** (-22.0 + 10.0 * torch.rand(len(g[::3]), device=DEV, generator=gen))
        Vb[:, 100:143] *= 1e-12                                 # a 120 dB null
    elif fam == "speech":
        Vb *= 1e-6
    out = torch.full((NT, LD), SENT, device=DEV)
    out[:, :F] = Vb
    return g.contiguous(), out


def _labels(w, NT, seed):
    if w.y_dim == 0:
        return None, None, None
    gen = torch.Generator(device=DEV).manual_seed(seed + 1)
    y = (torch.rand((NT, w.y_dim), device=DEV, generator=gen) > 0.5).float()
    if w.tc_label_bias:
        from dvae_b200.engine import mlp_forward
        return y, None, mlp_forward(w.ybias_mlp, y, _lib.ACT_NONE).contiguous()
    return y, y, None


def _zs(NT, R, L, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn((NT, R, L), device=DEV, generator=gen)


def _status():
    return torch.zeros(1, dtype=torch.int32, device=DEV)


def _mirror_vs(mir, Zs, y_frame, ybias):
    """Mirror ``(Vs, bound)`` ``[NT][R][F]`` of the samples ``Zs [NT][R][L]``."""
    NT, R, L = Zs.shape
    y = None if y_frame is None else y_frame.repeat_interleave(R, 0)
    yb = None if ybias is None else ybias.repeat_interleave(R, 0)
    Vs, b = mir.vs(Zs.reshape(-1, L), y, yb)
    return Vs.view(NT, R, F), b.view(NT, R, F)


# --------------------------------------------------------------------------------------------- dvae_decode_tc
@pytest.mark.parametrize("kind,bias,rows", [("M1", "plain", 57_077), ("M2", "plain", 2_000), ("ibm", "plain", 1_000),
                                            ("L32", "plain", 1_000), ("L32y3", "plain", 1_000), ("M1", "bias", 3_000),
                                            ("M1", "edge", 3_000)])
def test_decode_tc_against_mirror(kind, bias, rows):
    w, mir = _weights(kind, bias)
    div = 25
    NT = (rows + div - 1) // div
    y, ylab, ybias = _labels(w, NT, rows)
    x = torch.randn((rows, w.z_dim), device=DEV, generator=torch.Generator(device=DEV).manual_seed(rows))
    out = torch.full((rows + 3, LD), SENT, device=DEV)
    st = _status()
    _lib.call("dvae_decode_tc", w.dec_tc.ref, _p(tc.decoder_image(w)), _p(x), rows, w.z_dim, _p(ylab), w.tc_y_dim, _p(ybias), div,
              _p(out), LD, _p(st), _stream())
    assert int(st.item()) == 0
    assert torch.all(out[rows:] == SENT) and torch.all(out[:rows, F:] == SENT)
    fr = torch.arange(rows, device=DEV) // div
    Vs, bound = mir.vs(x, None if ylab is None else ylab[fr], None if ybias is None else ybias[fr])
    _check("decode_tc", "Vs", bias if bias != "plain" else kind, out[:rows, :F], Vs, bound)
    if bias == "edge":
        assert bool((out[:rows, 0:F:5] == 0).all())             # flushed to zero, as the mirror expects


# --------------------------------------------------------------------------------------------- statistics kernels
def _stats(w, Zs, r0, R, ylab, ybias, g, Vb, Vs, A1, A2, acc, st):
    NT, R_total = Zs.shape[0], Zs.shape[1]
    _lib.call("dvae_decode_stats_win_tc", w.dec_tc.ref, _p(tc.decoder_image(w)), _p(Zs), R_total, r0, R, w.z_dim, _p(ylab), w.tc_y_dim,
              _p(ybias), _p(Vb), _p(g), NT, LD, _p(Vs), _p(A1), _p(A2), acc, _p(st), _stream())


@pytest.mark.parametrize("R_total,win,NT,fam,kind", [
    (10, 10, None, "benign", "M1"), (30, 30, None, "late", "M1"), (10, 10, 6_001, "late", "M1"), (30, 30, 2_001, "benign", "M1"),
    (30, 30, 2_001, "late", "M2"), (40, 10, None, "speech", "M1"), (60, 30, None, "late", "L32y3"), (160, 10, None, "benign", "ibm"),
    (30, 30, None, "bias", "M1"), (10, 10, None, "edge", "M1")])
def test_decode_stats_against_f64(R_total, win, NT, fam, kind):
    """dvae_decode_stats_tc (one window) / dvae_decode_stats_win_tc (windows accumulated): Vs against the mirror, A1 / A2
    against float64 over the kernel's own Vs; pad columns and rows beyond the batch untouched."""
    w, mir = _weights(kind, fam if fam in ("bias", "edge") else "plain")
    NT = NT or sum(LENS_SMALL)
    g, Vb = _family("benign" if fam in ("bias", "edge") else fam, NT, R_total + NT)
    y, ylab, ybias = _labels(w, NT, NT)
    Zs = _zs(NT, R_total, w.z_dim, R_total)
    Vs = torch.full((NT + 1, R_total, LD), SENT, device=DEV)
    A = torch.full((2, NT + 1, LD), SENT, device=DEV)
    st = _status()
    if R_total == win:
        _lib.call("dvae_decode_stats_tc", w.dec_tc.ref, _p(tc.decoder_image(w)), _p(Zs), win, w.z_dim, _p(ylab), w.tc_y_dim, _p(ybias),
                  _p(Vb), _p(g), NT, LD, _p(Vs), _p(A[0]), _p(A[1]), _p(st), _stream())
    else:
        for r0 in range(0, R_total, win):
            _stats(w, Zs, r0, win, ylab, ybias, g, Vb, Vs, A[0], A[1], int(r0 > 0), st)
    assert int(st.item()) == 0
    assert torch.all(Vs[NT] == SENT) and torch.all(A[:, NT] == SENT)
    assert torch.all(Vs[:, :, F:] == SENT) and torch.all(A[:, :, F:] == SENT)
    name = "decode_stats" if R_total == win else "decode_stats_win"
    famname = fam if NT < 1000 else fam + "*"                  # *: steady-state size
    ref, bound = _mirror_vs(mir, Zs, y if ylab is not None else None, ybias)
    _check("%s<%d>" % (name, win), "Vs", famname, Vs[:NT, :, :F], ref, bound)
    A1, A2, b1, b2 = dm.frame_stats_f64(Vs[:NT, :, :F], g, Vb[:, :F], win)
    _check("%s<%d>" % (name, win), "A1", famname, A[0, :NT, :F], A1, b1)
    _check("%s<%d>" % (name, win), "A2", famname, A[1, :NT, :F], A2, b2)


# --------------------------------------------------------------------------------------------- the fused filter
def _wiener(w, Zs, chunk, ylab, ybias, g, Vb, st, NT=None):
    NT = Zs.shape[0] if NT is None else NT
    WFs = torch.full((NT + 1, LD), SENT, device=DEV)
    WFn = torch.full((NT + 1, LD), SENT, device=DEV)
    for r0 in range(0, Zs.shape[1], chunk):
        _lib.call("dvae_decode_wiener_tc", w.dec_tc.ref, _p(tc.decoder_image(w)), _p(Zs), Zs.shape[1], r0, chunk, w.z_dim, _p(ylab),
                  w.tc_y_dim, _p(ybias), _p(Vb), _p(g), NT, LD, _p(WFs), _p(WFn), int(r0 > 0), _p(st), _stream())
    return WFs, WFn


@pytest.mark.parametrize("R_total,chunk,lens,fam", [
    (75, 25, [23, 9, 14], "benign"), (30, 30, [23, 9, 14], "benign"), (25, 25, [23, 9, 14], "benign"), (20, 10, [23, 9, 14], "benign"),
    (75, 25, LENS_SMALL, "late"), (30, 30, LENS_SMALL, "late"), (20, 10, LENS_SMALL, "late"), (30, 30, LENS_SMALL, "speech"),
    (30, 30, [2_001], "late"), (10, 10, [6_001], "late"), (75, 25, [2_001], "late")])
def test_decode_wiener_against_f64(R_total, chunk, lens, fam):
    """dvae_decode_wiener_tc: the mask sums against float64, both in [0, R]; R = 10 / 30: over the storing instance's Vs of
    the same samples, WFn bit-identical to fl(Vb A1) accumulated window by window; R = 25: over the mirror's Vs interval."""
    w, mir = _weights("M1")
    NT = sum(lens)
    g, Vb = _family(fam, NT, NT + R_total)
    Zs = _zs(NT, R_total, w.z_dim, 3 * R_total + NT)
    st = _status()
    WFs, WFn = _wiener(w, Zs, chunk, None, None, g, Vb, st)
    assert int(st.item()) == 0
    assert torch.all(WFs[NT] == SENT) and torch.all(WFn[NT] == SENT) and torch.all(WFs[:, F:] == SENT) and torch.all(WFn[:, F:] == SENT)
    famname = fam if NT < 1000 else fam + "*"
    kern = "decode_wiener<%d>" % chunk
    if chunk in (10, 30):
        Vs = torch.empty((NT, R_total, LD), device=DEV)
        A = torch.empty((2, NT, LD), device=DEV)
        wn = torch.zeros((NT, F), device=DEV)
        for r0 in range(0, R_total, chunk):
            _stats(w, Zs, r0, chunk, None, None, g, Vb, Vs, A[0], A[1], 0, st)
            t = Vb[:, :F] * A[0, :, :F]                         # FP32, IEEE: the kernel's fl(Vb A1), then its accumulation
            wn = t if r0 == 0 else wn + t
        assert int(st.item()) == 0
        assert torch.equal(WFn[:NT, :F], wn), "WFn differs from fl(Vb A1) of the storing instance"
        ref_s, ref_n, bs, bn = dm.mask_sums_f64(Vs[:, :, :F], g, Vb[:, :F], chunk)
    else:
        Vs, vb_err = _mirror_vs(mir, Zs, None, None)
        ref_s, ref_n, bs, bn = dm.mask_sums_f64(Vs, g, Vb[:, :F], chunk, vs_err=vb_err)
    _check(kern, "WFs", famname, WFs[:NT, :F], ref_s, bs)
    _check(kern, "WFn", famname, WFn[:NT, :F], ref_n, bn)
    assert bool((WFs[:NT, :F] >= 0).all()) and bool((WFn[:NT, :F] >= 0).all())
    assert bool((WFs[:NT, :F] <= R_total * (1 + 1e-5)).all()) and bool((WFn[:NT, :F] <= R_total * (1 + 1e-5)).all())


def test_wiener_accum_and_apply_against_f64():
    """The FP32 route of the filter (dvae_wiener_accum over materialised Vs) and the mask application (dvae_wiener_apply),
    late family."""
    w, _ = _weights("M1")
    NT, R = sum(LENS_SMALL), 7
    g, Vb = _family("late", NT, 9)
    Vs = torch.full((NT, R, LD), SENT, device=DEV)
    Vs[:, :, :F] = torch.exp(torch.randn((NT, R, F), device=DEV) * 3.0) * 0.05
    WFs, WFn = torch.empty((NT, LD), device=DEV), torch.empty((NT, LD), device=DEV)
    _lib.call("dvae_wiener_accum", _p(Vs), R, _p(Vb), _p(g), NT, F, LD, _p(WFs), _p(WFn), 1, _stream())
    ref_s, ref_n, bs, bn = dm.mask_sums_f64(Vs[:, :, :F], g, Vb[:, :F], R, route="accum")
    _check("wiener_accum", "WFs", "late", WFs[:, :F], ref_s, bs)
    _check("wiener_accum", "WFn", "late", WFn[:, :F], ref_n, bn)
    X = torch.complex(torch.randn((NT, LD), device=DEV), torch.randn((NT, LD), device=DEV)) * 10.0 ** torch.randint(-6, 3, (NT, 1), device=DEV)
    S = torch.empty((NT, LD), dtype=torch.complex64, device=DEV)
    Nn = torch.empty_like(S)
    _lib.call("dvae_wiener_apply", _p(X), _p(WFs), _p(WFn), R, NT, F, LD, _p(S), _p(Nn), _stream())
    rS, rN, bS, bN = dm.apply_f64(X[:, :F], WFs[:, :F], WFn[:, :F], R)
    for name, got, ref, b in (("S_hat", S, rS, bS), ("N_hat", Nn, rN, bN)):
        _check("wiener_apply", name + ".re", "late", got[:, :F].real, ref.real, b)
        _check("wiener_apply", name + ".im", "late", got[:, :F].imag, ref.imag, b)


# --------------------------------------------------------------------------------------------- range of the shared reciprocal
@pytest.mark.parametrize("side", ["low_in", "high_in", "low_out", "high_out"])
def test_decode_wiener_at_the_range_limits(side):
    """Inside [2^-60, 2^60] every Vx meets the bound; below 2^-63 the pair product underflows: DVAE_STATUS_NONFINITE; above
    2^63 it overflows: those samples drop out of the sums (finite, too small, no status bit), as include/dvae_b200.h states."""
    w, _ = _weights("M1")
    NT, R = 13, 30
    Zs = _zs(NT, R, w.z_dim, 77)
    st = _status()
    Vs = torch.empty((NT, R, LD), device=DEV)
    A = torch.empty((2, NT, LD), device=DEV)
    g0, Vb0 = _family("benign", NT, 5)
    _stats(w, Zs, 0, R, None, None, g0, Vb0, Vs, A[0], A[1], 0, st)
    vs = Vs[:, :, :F].double()
    scale = {"low_in": 2.0 ** -60, "high_in": 2.0 ** 60, "low_out": 2.0 ** -66, "high_out": 2.0 ** 66}[side]
    # g Vs + Vb = scale (1 + small): Vb carries the level, g Vs a tenth of it at most
    g = (0.1 * scale / vs.amax(dim=(1, 2))).float()
    Vb = torch.full((NT, LD), SENT, device=DEV)
    Vb[:, :F] = scale
    WFs, WFn = _wiener(w, Zs, R, None, None, g, Vb, st)
    ref_s, ref_n, bs, bn = dm.mask_sums_f64(Vs[:, :, :F], g, Vb[:, :F], R)
    status = int(st.item())
    if side.endswith("in"):
        assert status == 0
        _check("decode_wiener<30>", "WFs", side, WFs[:NT, :F], ref_s, bs)
        _check("decode_wiener<30>", "WFn", side, WFn[:NT, :F], ref_n, bn)
    elif side == "low_out":
        assert status & NONFINITE and not bool(torch.isfinite(WFn[:NT, :F]).all())
    else:
        # bins 0..511 pair their samples; bin 512 takes one reciprocal per sample and stays right
        assert status == 0 and bool(torch.isfinite(WFn[:NT, :F]).all()) and float(WFn[:NT, :512].max()) < 0.5 * R


# --------------------------------------------------------------------------------------------- the engine's final filter
ENGINE_CASES = {   # name: (decoder kind, keep_WF, n_chains, family, expected filter_chunk)
    "M1_75": ("M1", 75, 1, "late", 25), "M1_30": ("M1", 30, 1, "benign", 30), "M1_10": ("M1", 10, 1, "speech", 10),
    "M1_7": ("M1", 7, 1, "late", 0), "chains16x25": ("M1", 25, 16, "late", 25), "M2_y1": ("M2", 25, 1, "late", 25),
    "ibm": ("ibm", 25, 1, "benign", 25), "L32": ("L32", 30, 1, "late", 30), "L32y3": ("L32y3", 10, 1, "benign", 10),
}


@pytest.mark.parametrize("case", sorted(ENGINE_CASES))
def test_engine_wiener_against_f64(case):
    """McemEngine.wiener() on sampler="tc": the masks against float64 over the mirror's Vs of the filter samples
    (``eng._last_Zs``), S_hat / N_hat against float64 ``mask / R X``, and the lazily decoded ``eng.Vs`` against the mirror."""
    kind, keep, chains, fam, chunk = ENGINE_CASES[case]
    w, mir = _weights(kind)
    lens = LENS_SMALL
    NT = sum(lens)
    cfg = McemConfig(niter=1, keep_E=10, burn_E=2, keep_WF=keep, burn_WF=3, sampler="tc", seed=11, n_chains=chains)
    eng = McemEngine(w, cfg, DEV)
    assert eng.filter_chunk == chunk and mcem_route(cfg, F)[1] == chunk
    gen = torch.Generator(device=DEV).manual_seed(3)
    P = torch.zeros((NT, LD), device=DEV)
    P[:, :F] = torch.empty((NT, F), device=DEV).exponential_(generator=gen) * 0.05
    X = torch.zeros((NT, LD), dtype=torch.complex64, device=DEV)
    X[:, :F] = torch.complex(torch.randn((NT, F), device=DEV, generator=gen), torch.randn((NT, F), device=DEV, generator=gen))
    y = None if w.y_dim == 0 else (torch.rand((NT, w.y_dim), device=DEV, generator=gen) > 0.5).float()
    eng.init_parameters(X, P, RaggedBatch(lens, DEV), y)
    g, Vb = _family(fam, NT, 21)
    eng.g.copy_(g)
    eng.Vb[:, :F].copy_(Vb[:, :F])
    eng.wiener()
    tc.check_status(eng)
    Zs = eng._last_Zs
    R = Zs.shape[1]
    assert R == chains * keep
    ylab = eng.tc_y
    Vs, vs_err = _mirror_vs(mir, Zs, ylab, eng.ybias)
    route = "fused" if chunk else "accum"
    ref_s, ref_n, bs, bn = dm.mask_sums_f64(Vs, eng.g, eng.Vb[:, :F], chunk or R, vs_err=vs_err, route=route)
    _check("engine.wiener", "WFs", case, eng.WFs[:, :F], ref_s, bs)
    _check("engine.wiener", "WFn", case, eng.WFn[:, :F], ref_n, bn)
    rS, rN, bS, bN = dm.apply_f64(eng.X[:, :F], eng.WFs[:, :F], eng.WFn[:, :F], R)
    for name, got, ref, b in (("S_hat", eng.S_hat, rS, bS), ("N_hat", eng.N_hat, rN, bN)):
        _check("engine.wiener", name + ".re", case, got[:, :F].real, ref.real, b)
        _check("engine.wiener", name + ".im", case, got[:, :F].imag, ref.imag, b)
    _check("engine.Vs", "Vs", case, eng.Vs[:, :, :F], Vs, vs_err)
    tc.check_status(eng)
