"""Host glue of the tcgen05 (BF16 tensor-core) sampler and decode: packed operands and the C ABI calls.

``mh_chain_tc`` / ``decode_tc`` are what ``McemEngine`` runs when ``McemConfig.sampler == "tc"``.  Everything here is
bookkeeping: building the decoder's shared-memory image once per model, re-packing P / Vb once per ``sample_posterior``
call, sizing the sampler's emission buffers and checking the status word.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


POLY_EX2 = 1            # DVAE_TC_POLY_EX2
POLY_EX2_ALL = 2        # DVAE_TC_POLY_EX2_ALL
POLY_EX2_LIMIT = 120.0  # DVAE_TC_POLY_EX2_LIMIT
VST_MAX_KEEP = 31       # kept samples per chain the sampler's emission can index
VST_IDX_PITCH = 32


def decoder_image(weights):
    """The UMMA-ready image of ``weights.dec`` (cached on the weights object)."""
    img = getattr(weights, "_tc_image", None)
    if img is None:
        lib = _lib.load()
        n = lib.dvae_tc_image_bytes(weights.dec_tc.ref, weights.z_dim, weights.tc_y_dim)
        if n < 0:
            _lib.check(-1, "dvae_tc_image_bytes")
        img = torch.empty(int(n), dtype=torch.uint8, device=weights.device)
        _lib.call("dvae_tc_pack_decoder", weights.dec_tc.ref, weights.z_dim, weights.tc_y_dim, _p(img), _stream())
        weights._tc_image = img
        # one-off range query: may the sampler use the polynomial 2^x (see DVAE_TC_POLY_EX2 in include/dvae_b200.h)?
        bound = C.c_float(0.0)
        _lib.call("dvae_tc_decoder_exponent_bound", weights.dec_tc.ref, weights.z_dim, weights.tc_y_dim, C.byref(bound), _stream())
        mode = os.environ.get("DVAE_TC_POLY", "1")          # 0: MUFU only, 1: half of the exponentials, 2: all of them
        weights._tc_flags = ({"0": 0, "2": POLY_EX2 | POLY_EX2_ALL}.get(mode, POLY_EX2)) if bound.value < POLY_EX2_LIMIT else 0
    return img


def _status(eng):
    st = eng._buf.get("tc_status")
    if st is None:
        st = torch.zeros(1, dtype=torch.int32, device=eng.dev)
        eng._buf["tc_status"] = st
    return st


def check_status(eng):
    """Raise if a kernel of this engine reported a pipeline timeout or a non-finite likelihood / cost (synchronises).
    The status word is cleared when the error is raised, so the engine can be used again."""
    st = eng._buf.get("tc_status")
    if st is None:
        return
    v = int(st.item())
    if v == 0:
        return
    st.zero_()
    what = []
    if v & _lib.STATUS_TIMEOUT:
        what.append("a tcgen05 pipeline wait timed out")
    if v & _lib.STATUS_NONFINITE:
        what.append("a log-likelihood or cost was NaN / Inf")
    raise _lib.DvaeError("device status %d (%s): results are invalid" % (v, "; ".join(what) or "unknown"))


def row_scale(eng):
    """Per-frame quad scale of the sampler's likelihood arithmetic (dvae_tc_row_scale), once per batch: ``[NT]`` float32."""
    w, b = eng.w, eng.batch
    k = eng._get("kscale", (max(b.NT, 1),))
    _lib.call("dvae_tc_row_scale", w.dec_tc.ref, _p(decoder_image(w)), w.z_dim, w.tc_y_dim, _p(eng.P), b.NT, eng.F, eng.ld, _p(k), _stream())
    eng.kernel_launches += 1
    return k


def mh_chain_tc(eng, Zs, keep, burn, rng, a_trace, emit=False):
    """One ``sample_posterior`` call on the tcgen05 sampler.  ``emit``: also write the kept samples' variances
    (``eng.VsT`` / ``eng.vs_idx``, see dvae_mh_chain_tc2)."""
    w, b, cfg = eng.w, eng.batch, eng.cfg
    img = decoder_image(w)
    chains = b.NT * cfg.n_chains
    lib = _lib.load()
    pv = eng._get("PVpk", (max(int(lib.dvae_tc_packed_pv_bytes(chains)), 16),), torch.uint8)
    _lib.call("dvae_tc_pack_pv", w.dec_tc.ref, _p(img), w.z_dim, w.tc_y_dim, _p(eng.P), _p(eng.Vb), _p(eng.kscale), b.NT, cfg.n_chains,
              eng.F, eng.ld, _p(pv), _stream())
    eng.kernel_launches += 1
    vst = idx = None
    if emit:
        vst = eng._get("VsT", (max(int(lib.dvae_vst_bytes(chains, keep)), 16),), torch.uint8)
        idx = eng._get("vs_idx", (max(chains, 1) * VST_IDX_PITCH,), torch.uint8)
    with eng.stage("mh_kernel"):
        _lib.call("dvae_mh_chain_tc2", w.dec_tc.ref, _p(img), _p(pv), _p(eng.kscale), _p(eng.g), _p(eng.tc_y), w.tc_y_dim, _p(eng.ybias), _p(b.frame_gid), _p(b.frame_idx),
                  _p(eng.Z), _p(Zs), b.NT, w.z_dim, cfg.n_chains, burn, keep, float(cfg.var_rw), C.byref(rng), _p(eng.n_accept),
                  _p(a_trace), _p(vst), _p(idx), int(w._tc_flags), _p(_status(eng)), _stream())
    eng.kernel_launches += 1
    eng.VsT, eng.vs_idx = vst, idx


def vst_frame_stats(eng, R):
    """A1 | A2 (``[2][NT][ld]``) of the emitted samples with the E-step's g and Vb (dvae_vst_frame_stats)."""
    w, b = eng.w, eng.batch
    st = eng._get("fstat", (2 * b.NT * eng.ld,))
    A1, A2 = st[: b.NT * eng.ld], st[b.NT * eng.ld:]
    _lib.call("dvae_vst_frame_stats", w.dec_tc.ref, _p(decoder_image(w)), w.z_dim, w.tc_y_dim, _p(eng.VsT), _p(eng.vs_idx), R, _p(eng.Vb),
              _p(eng.g), b.NT, eng.ld, _p(A1), _p(A2), _stream())
    eng.kernel_launches += 1
    return st


def vst_w_partials(eng, R):
    """Per-segment partial sums of the W update, reduced inside the statistics pass (dvae_vst_w_partials); ``[S][K][2][ld]``."""
    w, b, K = eng.w, eng.batch, eng.cfg.nmf_rank
    seg_start, tile_seg, _, S = b.segments(n_chains=eng.cfg.n_chains)
    wp = eng._get("wpart", (max(int(_lib.load().dvae_vst_w_partial_floats(S, K, eng.ld)), 1),))
    _lib.call("dvae_vst_w_partials", w.dec_tc.ref, _p(decoder_image(w)), w.z_dim, w.tc_y_dim, _p(eng.VsT), _p(eng.vs_idx), R, _p(eng.P),
              _p(eng.Vb), _p(eng.g), _p(eng.H), K, b.NT, eng.cfg.n_chains, eng.ld, _p(seg_start), _p(tile_seg), _p(wp), _stream())
    eng.kernel_launches += 1
    return wp


def vst_unpack(eng, R, out=None):
    """Dense FP32 ``Vs [NT][n_chains * R][ld]`` of the emitted samples (dvae_vst_unpack, ``R`` kept samples per chain): the
    reference's ``self.Vs`` up to layout."""
    w, b, c = eng.w, eng.batch, eng.cfg.n_chains
    if out is None:
        out = torch.zeros((b.NT, c * R, eng.ld), dtype=torch.float32, device=eng.dev)
    _lib.call("dvae_vst_unpack", w.dec_tc.ref, _p(decoder_image(w)), w.z_dim, w.tc_y_dim, _p(eng.VsT), _p(eng.vs_idx), R, b.NT * c, eng.ld,
              _p(out), _stream())
    return out


def decode_tc(eng, x, x2, x2_row_div, out, ybias=None):
    """Vs rows for the kept samples ``x [rows][L]`` (+ labels ``x2`` or the per-frame label bias ``ybias``) through the
    tensor-core decoder."""
    w = eng.w
    img = decoder_image(w)
    if w.tc_label_bias:
        x2 = None                                   # the labels arrive as ybias (row r uses frame r / x2_row_div)
    _lib.call("dvae_decode_tc", w.dec_tc.ref, _p(img), _p(x), x.shape[0], w.z_dim, _p(x2), w.tc_y_dim, _p(ybias), max(1, x2_row_div),
              _p(out), out.stride(0), _p(_status(eng)), _stream())
    eng.kernel_launches += 1


def decode_stats_tc(eng, Zs, Vs):
    """Warp-specialised decode + per-frame reciprocal sums (dvae_decode_stats_tc); returns the [2][NT][ld] statistics.

    Frames with more than 30 samples (multi-chain runs) are decoded in sample windows of 30 or 10 that accumulate into the
    same statistics (dvae_decode_stats_win_tc)."""
    w, b = eng.w, eng.batch
    img = decoder_image(w)
    st = eng._get("fstat", (2 * b.NT * eng.ld,))
    A1, A2 = st[: b.NT * eng.ld], st[b.NT * eng.ld:]
    R = Zs.shape[1]
    if R in (10, 30):
        _lib.call("dvae_decode_stats_tc", w.dec_tc.ref, _p(img), _p(Zs), R, w.z_dim, _p(eng.tc_y), w.tc_y_dim, _p(eng.ybias), _p(eng.Vb),
                  _p(eng.g), b.NT, eng.ld, _p(Vs), _p(A1), _p(A2), _p(_status(eng)), _stream())
        eng.kernel_launches += 1
        return st
    win = 30 if R % 30 == 0 else 10
    for r0 in range(0, R, win):
        _lib.call("dvae_decode_stats_win_tc", w.dec_tc.ref, _p(img), _p(Zs), R, r0, win, w.z_dim, _p(eng.tc_y), w.tc_y_dim, _p(eng.ybias), _p(eng.Vb),
                  _p(eng.g), b.NT, eng.ld, _p(Vs), _p(A1), _p(A2), 0 if r0 == 0 else 1, _p(_status(eng)), _stream())
        eng.kernel_launches += 1
    return st


def decode_wiener_tc(eng, Zs, r0, R, WFs, WFn, accumulate):
    """Mask sums of the samples r0 .. r0+R of ``Zs`` without storing their variances (dvae_decode_wiener_tc):
    ``WFs (+)= g sum_r Vs / Vx``, ``WFn (+)= Vb sum_r 1 / Vx``, ``[NT][ld]``."""
    w, b = eng.w, eng.batch
    img = decoder_image(w)
    _lib.call("dvae_decode_wiener_tc", w.dec_tc.ref, _p(img), _p(Zs), Zs.shape[1], int(r0), int(R), w.z_dim, _p(eng.tc_y), w.tc_y_dim,
              _p(eng.ybias), _p(eng.Vb), _p(eng.g), b.NT, eng.ld, _p(WFs), _p(WFn), int(bool(accumulate)), _p(_status(eng)), _stream())
    eng.kernel_launches += 1
