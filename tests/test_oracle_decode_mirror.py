"""The float64 mirror of the decode kernels (oracle/decode_mirror.py) on the CPU, with ``bf16(tanh)`` in place of the device's
``tanh.approx.f32``: the intervals it returns are exact where nothing can round, contain the FP32-weight decoder up to the
BF16 rounding of weights and activations, and are wide exactly where a hidden unit straddles a BF16 rounding boundary."""
import numpy as np
import pytest
import torch

from dvae_b200 import synth
from oracle import decode_mirror as dm
from oracle.mh_replay import F64, PlainDecoder, bf16

F = 513
BF16_REL = 2.0 ** -8                     # BF16 rounding, relative (nearest: 2^-9; a margin of two)


def _sd(variant, L, h, y_dim, seed=3):
    return synth.xavier_state_dict(variant, F, L, h, y_dim, seed=seed, out_bias=-3.0)


def _bf16_exact(sd):
    """The state dict with every weight and bias a small BF16 number (and W3 log2(e) BF16 too: W3 multiples of 2^-6 / log2 e
    would not be; those stay as they are, layer 3 is not exercised here)."""
    out = dict(sd)
    for k, v in sd.items():
        if k.startswith("decoder.hidden"):
            out[k] = np.round(np.asarray(v) * 64.0).astype(np.float32) / np.float32(64.0)
    return out


def _bf16_np(x):
    """Round-to-nearest-even BF16 of float32 numbers, through their bit patterns (independent of torch's conversion)."""
    b = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000
    return b.astype(np.uint32).view(np.float32).astype(np.float64)


@pytest.mark.parametrize("variant,L,h,y_dim", [("M1", 16, [128, 128], 0), ("M2", 32, [128], 3)])
def test_bf16_exact_network_has_zero_hidden_radii_where_nothing_rounds(variant, L, h, y_dim):
    """BF16-exact weights and inputs (multiples of 2^-6 and 2^-4): every layer-1 product is exact and the sums of at most 71
    of them are exact in FP32, so a unit's interval is the accumulation bound alone; where both ends round to the same BF16
    activation the radius is zero and the centre is the activation of the exact float64 pre-activation."""
    sd = _bf16_exact(_sd(variant, L, h, y_dim))
    m = dm.DecodeMirror(sd, L)
    rows = 64
    gen = torch.Generator().manual_seed(1)
    z = torch.round(torch.randn((rows, L), generator=gen) * 16) / 16
    y = (torch.rand((rows, y_dim), generator=gen) > 0.5).float() if y_dim else None
    layers = m.layers(z, y)
    pre, rad, hc, hr = layers[0]
    w1 = torch.tensor(sd["decoder.hidden.0.weight"], dtype=F64)
    b1 = torch.tensor(sd["decoder.hidden.0.bias"], dtype=F64)
    exact = (z.to(F64) if y is None else torch.cat([z, y], 1).to(F64)) @ w1.T + b1
    assert torch.equal(pre, exact)
    direct = bf16(torch.tanh(exact.to(torch.float32)))
    zero = hr == 0
    assert float(zero.double().mean()) > 0.9
    assert torch.equal(hc[zero], direct[zero])
    # nothing but the accumulation bound and the bias add: K 2^-23 sum|terms| + u |x|
    K = m.layer1_k(y_dim)
    terms = (z.abs().to(F64) if y is None else torch.cat([z, y], 1).abs().to(F64)) @ w1.abs().T + b1.abs()
    assert torch.allclose(rad, K * dm.TC_ULP * terms + dm.U32 * exact.abs(), rtol=1e-12, atol=0)
    v, vr = m.v(z, y)
    assert bool((vr > 0).all()) and bool(torch.isfinite(v).all())


@pytest.mark.parametrize("variant,L,h,y_dim", [("M1", 16, [128, 128], 0), ("M2", 16, [128, 128], 1), ("M1", 32, [128], 0)])
def test_centre_is_the_fp32_weight_decoder_up_to_bf16_rounding(variant, L, h, y_dim):
    """|mirror centre - PlainDecoder| (log2 domain) <= mirror radius + the BF16 rounding of the weights and activations carried
    through the layers (first order, tanh' <= 1)."""
    sd = _sd(variant, L, h, y_dim)
    m = dm.DecodeMirror(sd, L)
    plain = PlainDecoder(sd)
    gen = torch.Generator().manual_seed(2)
    z = torch.randn((200, L), generator=gen)
    y = (torch.rand((200, y_dim), generator=gen) > 0.5).float() if y_dim else None
    v, vr = m.v(z, y)
    ref = plain.pre(z, y) * np.log2(np.e)
    x = (z.to(F64) if y is None else torch.cat([z, y], 1).to(F64))
    e, hx = None, x
    for i, (w, b) in enumerate(plain.layers[:-1]):
        pre = hx @ w.T + b
        e_pre = BF16_REL * (hx.abs() @ w.abs().T + (b.abs() if i == 0 else 0)) + (0 if e is None else e @ w.abs().T)
        hx = torch.tanh(pre)
        e = e_pre + BF16_REL * hx.abs() + 2.0 ** -20
    w3, b3 = plain.layers[-1]
    ev = (BF16_REL * (hx.abs() @ w3.abs().T) + e @ w3.abs().T) * np.log2(np.e)
    got = v + m.b_log2
    assert bool(((got - ref).abs() <= vr + ev + 1e-6).all()), float(((got - ref).abs() - vr - ev).max())
    assert float((got - ref).abs().max()) > 0                         # the rounding is there, the bound is not vacuous
    assert float(((got - ref).abs() / (vr + ev)).max()) > 0.005


def test_radius_is_nonzero_exactly_for_units_straddling_a_rounding_boundary():
    """Recomputed independently (BF16 rounding through bit patterns): a hidden unit has a non-zero radius
    exactly when the BF16 activations at the two FP32 ends of its interval differ, and then the radius is half their gap."""
    sd = _sd("M1", 16, [128, 128], 0, seed=8)
    m = dm.DecodeMirror(sd, 16)
    z = torch.randn((300, 16), generator=torch.Generator().manual_seed(4))
    for pre, rad, hc, hr in m.layers(z):
        p, r = pre.numpy(), rad.numpy()
        lo, hi = (p - r).astype(np.float32), (p + r).astype(np.float32)          # the FP32 ends, rounded outwards
        lo = np.where(lo.astype(np.float64) > p - r, np.nextafter(lo, np.float32(-np.inf)), lo)
        hi = np.where(hi.astype(np.float64) < p + r, np.nextafter(hi, np.float32(np.inf)), hi)
        blo, bhi = (_bf16_np(torch.tanh(torch.from_numpy(t)).numpy()) for t in (lo, hi))
        straddle = blo != bhi
        assert straddle.any() and not straddle.all()
        np.testing.assert_array_equal(hr.numpy() > 0, straddle)
        np.testing.assert_array_equal(hr.numpy(), 0.5 * (bhi - blo))
