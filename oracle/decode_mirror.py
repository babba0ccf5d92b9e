"""Float64 mirror of the tensor-core decode kernels, with an error interval per output.  Oracle: test infrastructure only.

The decode kernels (``decoder_tc_kernel``, csrc/tc_decode.cu; ``decode_stats_kernel``, csrc/decode_stats_tc.cu) share the
samplers' operands (``mh_replay.MirroredDecoder``: the layer-1 operand as BF16 hi + lo parts of z and of up to three labels,
b1 in BF16 on the constant-one column or a per-frame FP32 ``ybias``, W2 and ``W3 log2 e`` in BF16, ``b3 log2 e`` in FP32) but
round the hidden layers differently: the FP32 tensor-core pre-activation, plus ``ybias`` (layer 1) or ``b2`` (layer 2) in
FP32, goes through ``tanh.approx.f32`` and the result is rounded to BF16 (``cvt.rn.bf16x2``).  The output is
``ex2.approx.ftz(v + b)`` with ``v`` the layer-3 pre-activation in the log2 domain.

``DecodeMirror.v`` returns for every element a centre and a radius that contain what the kernels can compute:

* accumulation: a tensor-core sum of K exact BF16 x BF16 products is within ``K 2^-23 sum|terms|`` of its float64 value
  (nothing assumed about order or rounding mode beyond one ulp per addition; K is the MMA's K, zero columns included);
* activation: evaluated at the FP32 ends of ``[x - d - u|x|, x + d + u|x|]`` (``d``: accumulation bound plus the radii of
  the layer's inputs through ``sum|W| h_rad``; ``u|x|``: the FP32 bias add), both ends rounded to BF16.  The activation is
  assumed monotone up to ``act_step``, the largest fall ``max_{x1 < x2} act(x1) - act(x2)`` measured over its inputs, by
  which the ends are widened;
* output: ``vs_bound`` turns the interval of ``v + b`` into an absolute bound on ``Vs``: ``2^rad - 1`` relative, ex2.approx
  at 2^-22, the FP32 rounding of ``v + b``, and 2^-126 absolute where the interval reaches the flush-to-zero range.

``frame_stats_f64`` / ``mask_sums_f64`` are the float64 sums the statistics and filter kernels form from ``Vs``, with the
bound of their FP32 arithmetic named ingredient by ingredient.
"""
from __future__ import annotations

import numpy as np
import torch

from .mh_replay import F64, MirroredDecoder, bf16

U32 = 2.0 ** -24             # FP32 rounding
TC_ULP = 2.0 ** -23          # one ulp of an FP32 partial sum of the tensor core, relative to sum |terms|
EX2_REL = 2.0 ** -22         # ex2.approx.ftz.f32 (PTX ISA)
FLUSH = 2.0 ** -126          # ex2.approx.ftz: results below the normal range are flushed to zero
HID = 128

# 1 / Vx of the statistics / filter kernels (decode_stats_tc.cu), relative error of one reciprocal:
VX_FMA = U32                 # Vx = fmaf(g, Vs, Vb)
PAIR = U32                   # x0 x1 (or X Y lane by lane) of the shared reciprocal
RCP = 2 * U32                # rcp.approx.ftz.f32: 1 ulp
MUL = U32                    # x1 * rcp(x0 x1)
INV_PAIR = VX_FMA + PAIR + RCP + MUL     # samples in quads and pairs
INV_SINGLE = VX_FMA + RCP                # the last sample of R = 25, and bin 512 (no pair)

# 1 / Vx of the cast-off FP32 route (wiener_accum_kernel, nmf.cu): g Vs (u), + Vb (u), IEEE division (u)
ACC_SPEECH = 4 * U32         # g Vs / Vx: the product (u) in numerator and denominator, the sum (u), the division (u)
ACC_NOISE = 3 * U32          # Vb / Vx


class DecodeMirror:
    """``v(z, y, ybias) -> (centre, radius)`` of the layer-3 pre-activation (log2 domain, without the output bias) as the decode
    kernels compute it; ``b_log2`` the output bias as the image holds it.  ``act``: the hidden activation on FP32 inputs
    (``fn(float32 tensor) -> float32 tensor``; the device's ``tanh.approx.f32`` through ``dvae_tc_tanh_f32``); None:
    ``torch.tanh`` in FP32.  ``label_bias``: as ``MirroredDecoder``."""

    def __init__(self, sd, L, device="cpu", label_bias=False, act=None, act_step=0.0):
        m = MirroredDecoder(sd, L, device=device, label_bias=label_bias)
        self.L, self.label_bias = L, label_bias
        self.W1z, self.W1y, self.b1, self.hidden, self.W3, self.b_log2 = m.W1z, m.W1y, m.b1, m.hidden, m.W3, m.b_log2
        self.act = act if act is not None else (lambda x: torch.tanh(x))
        self.act_step = float(act_step)

    def layer1_k(self, y_dim):
        """The layer-1 MMA's K: the operand [hi(z) | lo(z) | labels hi, lo | 1] padded to 64-column blocks."""
        return 64 * ((2 * self.L + 2 * y_dim + 1 + 63) // 64)

    def activation(self, x, rad):
        """BF16(act(FP32 x')) for every FP32 x' in ``[x - rad, x + rad]``: ``(centre, radius)`` of the BF16 results."""
        lo, hi = x - rad, x + rad
        lo32, hi32 = lo.to(torch.float32), hi.to(torch.float32)
        lo32 = torch.where(lo32.to(F64) > lo, torch.nextafter(lo32, torch.full_like(lo32, -np.inf)), lo32)
        hi32 = torch.where(hi32.to(F64) < hi, torch.nextafter(hi32, torch.full_like(hi32, np.inf)), hi32)
        tlo, thi = self.act(lo32).to(F64), self.act(hi32).to(F64)
        if self.act_step:
            tlo, thi = tlo - self.act_step, thi + self.act_step
        blo, bhi = bf16(tlo), bf16(thi)
        return 0.5 * (blo + bhi), 0.5 * (bhi - blo)

    def layers(self, z, y=None, ybias=None):
        """Per hidden layer ``(pre, rad, h, h_rad)``: the float64 pre-activation with its bias, the half-width of the FP32
        interval the kernels' pre-activation lies in, and the centre / radius of the BF16 activations."""
        z32 = z.to(torch.float32)
        hi = z32.to(torch.bfloat16).to(torch.float32)
        a = torch.cat([hi.to(F64), bf16(z32 - hi)], 1)                        # hi | lo, both BF16-exact (z - hi exact in FP32)
        W = torch.cat([self.W1z, self.W1z], 1)
        y_dim = 0
        if ybias is None and y is not None and y.shape[1]:
            y32 = y.to(torch.float32)
            yh = y32.to(torch.bfloat16).to(torch.float32)
            a = torch.cat([a, yh.to(F64), bf16(y32 - yh)], 1)
            W = torch.cat([W, self.W1y, self.W1y], 1)
            y_dim = y.shape[1]
        pre = a @ W.T + self.b1
        if ybias is not None:
            pre = pre + ybias.to(F64)
        rad = self.layer1_k(y_dim) * TC_ULP * (a.abs() @ W.abs().T + self.b1.abs()) + U32 * pre.abs()
        out = [(pre, rad) + self.activation(pre, rad)]
        for w, b in self.hidden:
            h, hr = out[-1][2], out[-1][3]
            pre = h @ w.T + b
            rad = HID * TC_ULP * ((h.abs() + hr) @ w.abs().T) + hr @ w.abs().T + U32 * pre.abs()
            out.append((pre, rad) + self.activation(pre, rad))
        return out

    def v(self, z, y=None, ybias=None):
        h, hr = self.layers(z, y, ybias)[-1][2:]
        v = h @ self.W3.T
        vr = HID * TC_ULP * ((h.abs() + hr) @ self.W3.abs().T) + hr @ self.W3.abs().T
        return v, vr

    def vs(self, z, y=None, ybias=None):
        """``(Vs, bound)`` float64 ``[rows][F]``: ``vs_bound`` of ``v``."""
        return vs_bound(*self.v(z, y, ybias), self.b_log2)


def vs_bound(v, vr, b_log2):
    """``(Vs, bound)`` float64 from the interval ``v +- vr`` and the output bias: the centre ``2^(v + b)`` and an absolute
    bound on ``|ex2.approx.ftz(fl(v' + b)) - 2^(v + b)|`` for every ``v'`` in the interval."""
    e = v + b_log2
    er = vr + U32 * (e.abs() + vr)                                           # + the FP32 rounding of v' + b
    Vs = torch.exp2(e)
    bound = Vs * (torch.exp2(er) * (1 + EX2_REL) - 1)
    bound = bound + torch.where(e - er < -126.0, torch.full_like(e, FLUSH), torch.zeros_like(e))
    return Vs, bound


def _depths(R):
    """Longest chains of FP32 additions of ``decode_stats_kernel``'s sums for one sample window of R, bins 0..511:
    (A1, A2 / speech sum).  Quads feed packed lanes (A1: i0 + i1, then the lane; A2 and the speech sum: two FMAs per quad),
    then the pair or single sample, then the two lanes, then ``a1 +=``; bin 512 sums its R terms in one sequential loop."""
    nq = R // 4
    return nq + 3, 2 * nq + 3


def frame_stats_f64(Vs, g, Vb, R_win, vs_err=None):
    """``A1 = sum_r 1 / Vx``, ``A2 = sum_r 1 / Vx^2`` in float64 with ``Vx = g Vs + Vb`` and their bounds for the kernel's
    order: windows of ``R_win`` samples each accumulated onto the previous ones.  ``Vs [N][R][F]``, ``g [N]``, ``Vb [N][F]``
    (torch); ``vs_err``: an absolute bound of ``Vs`` (None: Vs is the kernels' own, exact)."""
    Vs, g, Vb = Vs.to(F64), g.to(F64)[:, None, None], Vb.to(F64)[:, None, :]
    N, R, F = Vs.shape
    Vx = g * Vs + Vb
    inv = 1.0 / Vx
    A1, A2 = inv.sum(1), (inv * inv).sum(1)
    n_win = R // R_win
    d1, d2 = _depths(R_win)
    i_rel = INV_PAIR                                                         # >= INV_SINGLE (R = 25's last sample, bin 512)
    dep1 = torch.full((F,), float(d1 + n_win - 1), dtype=F64, device=Vs.device)
    dep2 = torch.full((F,), float(d2 + n_win - 1), dtype=F64, device=Vs.device)
    if F > 512:
        dep1[512] = dep2[512] = R_win + n_win - 1
    b1 = (i_rel + dep1 * U32) * A1
    b2 = (2 * i_rel + U32 + dep2 * U32) * A2                                 # i^2 (2 i_rel) by FMA (u)
    if vs_err is not None:
        d_inv = g * vs_err.to(F64) * inv * inv                               # |d(1 / Vx)| <= g dVs / Vx^2
        b1 = b1 + d_inv.sum(1)
        b2 = b2 + (2 * inv * d_inv).sum(1)
    return A1, A2, b1, b2


def mask_sums_f64(Vs, g, Vb, R_win, vs_err=None, route="fused"):
    """The final filter's mask sums ``WFs = sum_r g Vs / Vx``, ``WFn = sum_r Vb / Vx`` in float64 and their bounds.
    ``route``: "fused" (``dvae_decode_wiener_tc``: windows of ``R_win`` samples, speech sum accumulated term by term, then
    ``g *``, ``Vb *``) or "accum" (``dvae_wiener_accum``: IEEE divisions, one chain over the R samples)."""
    Vs, g, Vb = Vs.to(F64), g.to(F64)[:, None, None], Vb.to(F64)[:, None, :]
    N, R, F = Vs.shape
    Vx = g * Vs + Vb
    ts, tn = g * Vs / Vx, Vb / Vx
    WFs, WFn = ts.sum(1), tn.sum(1)
    if route == "accum":
        bs = (ACC_SPEECH + R * U32) * WFs
        bn = (ACC_NOISE + R * U32) * WFn
    else:
        n_win = R // R_win
        d1, d2 = _depths(R_win)
        dep1 = torch.full((F,), float(d1 + n_win - 1), dtype=F64, device=Vs.device)
        dep2 = torch.full((F,), float(d2 + n_win - 1), dtype=F64, device=Vs.device)
        if F > 512:
            dep1[512] = dep2[512] = R_win + n_win - 1
        i_rel = INV_PAIR
        bn = (i_rel + MUL + dep1 * U32) * WFn                                # Vb * sum (u)
        bs = (i_rel + U32 + MUL + dep2 * U32) * WFs                          # Vs * (1 / Vx) inside the FMA (u), g * sum (u)
    if vs_err is not None:
        dv = vs_err.to(F64)
        bs = bs + (g * dv * Vb / (Vx * Vx)).sum(1)                           # |d(g Vs / Vx)| = g Vb dVs / Vx^2
        bn = bn + (Vb * g * dv / (Vx * Vx)).sum(1)                           # |d(Vb / Vx)| likewise
    return WFs, WFn, bs, bn


def apply_f64(X, WFs, WFn, R, bs=None, bn=None):
    """``S_hat = WFs / R X``, ``N_hat = WFn / R X`` (complex128) and per-component bounds of ``dvae_wiener_apply``: fl(1 / R),
    the mask product and the product with X (3u), plus the masks' own bounds carried through."""
    X = X.to(torch.complex128)
    ms, mn = WFs.to(F64) / R, WFn.to(F64) / R
    S, Nh = ms * X, mn * X
    ax = torch.maximum(X.real.abs(), X.imag.abs())
    bS = 3 * U32 * ms * ax + (0 if bs is None else bs.to(F64) / R * ax)
    bN = 3 * U32 * mn * ax + (0 if bn is None else bn.to(F64) / R * ax)
    return S, Nh, bS, bN
