"""Float64 replay of a Metropolis-Hastings run along the sampler's own decisions.  Oracle: test infrastructure only.

A sampler is run first; the replay then recomputes every proposal of every chain from the same draws and takes each
accept decision from the sampler (``decide``), so the two trajectories never diverge and every (iteration, chain) pair
can be compared, not only those before the first decision that differs.

* Proposal: ``z' = fl(z + fl(sd * eps))`` in float32 with ``sd = sqrtf(var_rw)``, as every sampler of the library (and the
  reference, mcem.py:243) writes it: the replayed states are bit-exact.
* Decoders, evaluated in float64 (torch, on the device of the inputs):
  ``PlainDecoder``    the FP32 weights as they are (models.py:119-122);
  ``MirroredDecoder`` the rounding points of the tensor-core sampler (csrc/tc_decode.cu, csrc/tc_common.cuh,
                      csrc/mh_tc2.cu): W1, W2, W3 log2(e) and b1 in BF16, the layer-1 operand as BF16 hi + lo parts, the
                      hidden pre-activations rounded to BF16 and passed through the samplers' activation (a table of
                      tanh.approx.bf16x2 over all BF16 inputs, ``dvae_tc_tanh_bf16_table``; without one: the correctly
                      rounded tanh), b2 and the per-frame label bias in FP32, the layer-3 bias left out (it is folded into
                      the P / Vb stream).
* Log-likelihood (mcem.py:251-253): ``l(z) = sum_f [ln Vx + P / Vx]``, ``a = l(z) - l(z') + 0.5 sum(z^2 - z'^2)``.
"""
from __future__ import annotations

import numpy as np
import torch

LOG2E_F32 = np.float32(1.4426950408889634)
F64 = torch.float64


def bf16(x):
    """Round to BF16 (nearest even, through FP32 as the kernels' FP32 accumulators are) and return float64."""
    return x.to(torch.float32).to(torch.bfloat16).to(F64)


def bf16_bits(x):
    """BF16 bit patterns (int64 in [0, 65536)) of ``x`` rounded to BF16."""
    return x.to(torch.float32).to(torch.bfloat16).view(torch.int16).to(torch.int64) & 0xFFFF


def bf16_from_bits(bits):
    """float64 values of BF16 bit patterns."""
    return ((bits.to(torch.int64) & 0xFFFF) << 16).to(torch.int32).view(torch.float32).to(F64)


def _layers(sd, device):
    out, i = [], 0
    while "decoder.hidden.%d.weight" % i in sd:
        out.append((torch.as_tensor(np.asarray(sd["decoder.hidden.%d.weight" % i]), device=device),
                    torch.as_tensor(np.asarray(sd["decoder.hidden.%d.bias" % i]), device=device)))
        i += 1
    out.append((torch.as_tensor(np.asarray(sd["decoder.reconstruction.weight"]), device=device),
                torch.as_tensor(np.asarray(sd["decoder.reconstruction.bias"]), device=device)))
    return out


class PlainDecoder:
    """The decoder with its FP32 weights, in float64: ``pre(z, y)`` is the output layer's pre-activation (ln Vs)."""

    def __init__(self, sd, device="cpu"):
        self.layers = [(w.to(F64), b.to(F64)) for w, b in _layers(sd, device)]

    def pre(self, z, y=None):
        h = z.to(F64) if y is None else torch.cat([z.to(F64), y.to(F64)], dim=1)
        for w, b in self.layers[:-1]:
            h = torch.tanh(h @ w.T + b)
        w, b = self.layers[-1]
        return h @ w.T + b


class MirroredDecoder:
    """The tensor-core sampler's decoder: ``v(z, y | ybias)`` is the layer-3 pre-activation in the log2 domain WITHOUT the
    output bias (``2^v`` is what the sampler emits); ``b_log2`` is the bias as the image holds it (FP32 ``b3 * log2 e``).

    ``label_bias``: the decoder is packed without its label columns and b1, which arrive as a per-frame FP32 layer-1 bias
    (``ybias``, more than three labels).  Otherwise up to three labels ride in the layer-1 operand as BF16 hi + lo parts and
    b1 (BF16) on its constant-one column.

    ``tanh_table``: the activation of each BF16 input, float64 ``[65536]`` indexed by bit pattern (``bf16_from_bits`` of what
    ``dvae_tc_tanh_bf16_table`` writes); None: ``bf16(tanh(x))``."""

    def __init__(self, sd, L, device="cpu", label_bias=False, tanh_table=None):
        lay = _layers(sd, device)
        (w1, b1), hidden, (w3, b3) = lay[0], lay[1:-1], lay[-1]
        self.L = L
        self.W1z = bf16(w1[:, :L])
        self.W1y = bf16(w1[:, L:])
        self.b1 = torch.zeros_like(b1, dtype=F64) if label_bias else bf16(b1)
        self.label_bias = label_bias
        self.hidden = [(bf16(w), b.to(F64)) for w, b in hidden]          # layer 2: BF16 weights, FP32 bias
        self.W3 = bf16(w3 * torch.tensor(LOG2E_F32, device=w3.device))     # FP32 product, then BF16
        self.b_log2 = (b3 * torch.tensor(LOG2E_F32, device=b3.device)).to(F64)
        self.tanh_table = tanh_table

    def act(self, pre):
        """The hidden activation of a pre-activation: rounded to BF16, then the samplers' tanh (BF16 result)."""
        if self.tanh_table is None:
            return bf16(torch.tanh(bf16(pre)))
        return self.tanh_table[bf16_bits(pre)]

    @staticmethod
    def _hi_lo(x):
        x = x.to(torch.float32)
        hi = x.to(torch.bfloat16).to(torch.float32)
        return hi.to(F64) + bf16(x - hi)                                # x - hi is exact in FP32

    def v(self, z, y=None, ybias=None):
        pre = self._hi_lo(z) @ self.W1z.T + self.b1
        if ybias is not None:
            pre = pre + ybias.to(F64)
        elif y is not None and y.shape[1]:
            pre = pre + self._hi_lo(y) @ self.W1y.T
        h = self.act(pre)
        for w, b in self.hidden:
            h = self.act(h @ w.T + b)
        return h @ self.W3.T


def loglik_plain(pre, g, Vb, P):
    """``(l, q)``: ``l = sum_f [ln Vx + P / Vx]`` and ``q = sum_f P / Vx`` with ``Vx = g exp(pre) + Vb`` (float64)."""
    Vx = g.to(F64)[:, None] * torch.exp(pre) + Vb.to(F64)
    r = P.to(F64) / Vx
    return (torch.log(Vx) + r).sum(1), r.sum(1)


def loglik_stream(v, g, Pp, Vbp):
    """The sampler's likelihood on the packed stream: ``sum_f [ln X + P' / X]``, ``X = g 2^v + Vb'``.  It differs from
    ``loglik_plain`` by a per-bin constant (the folded bias) that cancels in ``l(z) - l(z')``."""
    X = g.to(F64)[:, None] * torch.exp2(v) + Vbp
    return (torch.log(X) + Pp / X).sum(1)


def decode_stream(words, k, F=513):
    """``(P', Vb')`` float64 ``[rows][F]`` from the packed words ``[rows][>= F]`` (int32 bit patterns) and the rows' quad scale:
    word j of a quad is P' (divided by k for j >= 2) with bf16(Vb') (multiplied by k for j < 2) in its low half."""
    w = words[:, :F].to(torch.int64) & 0xFFFFFFFF
    whole = (w.to(torch.int32)).view(torch.float32).to(F64)
    low = ((w << 16) & 0xFFFFFFFF).to(torch.int32).view(torch.float32).to(F64)
    j = torch.arange(F, device=words.device) % 4
    k = k.to(F64)[:, None]
    Pp = torch.where(j >= 2, whole * k, whole)
    Vbp = torch.where(j < 2, low / k, low)
    return Pp, Vbp


def proposal(z, eps, sd):
    """``fl(z + fl(sd * eps))`` in float32, two separately rounded operations (no FMA)."""
    return z + eps * torch.tensor(np.float32(sd), device=z.device)


def replay(evaluators, z0, eps, var_rw, n_burn, decide):
    """Replay ``len(eps)`` iterations of ``rows`` chains.

    evaluators: ``{name: fn(z) -> (l [rows], q [rows] or None)}`` float64; the scale ``S = sum_f (2 + P/Vx + P/Vx')`` is
    built from the ``q`` of the evaluator named ``"plain"`` (``F`` from ``n_bins``).
    decide: ``fn(it, z, zp, a) -> bool [rows]``, the sampler's decision for iteration ``it`` (``a``: the replayed log ratios).
    Returns a dict: ``a`` {name: [n_iter][rows]}, ``S``, ``Z`` / ``Zp`` (state before, proposal) ``[n_iter][rows][L]``,
    ``acc`` ``[n_iter][rows]``, ``Zs [rows][n_keep][L]``, ``Z_end``, ``Z_burn`` (state at the end of the burn-in), ``n_acc``
    and ``slot [rows][n_keep]`` (the emission slot of kept sample r: 1 + r after an accept at kept iteration r, else the last
    accepted kept slot, else 0)."""
    sd = np.sqrt(np.float32(var_rw), dtype=np.float32)
    n_iter, rows = eps.shape[0], z0.shape[0]
    n_keep = n_iter - n_burn
    z = z0.clone()
    cur = {name: fn(z) for name, fn in evaluators.items()}
    n_bins = evaluators["plain"].n_bins
    out = dict(a={name: [] for name in evaluators}, S=[], Z=[], Zp=[], acc=[])
    dev = z0.device
    n_acc = torch.zeros(rows, dtype=torch.int64, device=dev)
    slot = torch.zeros((rows, max(n_keep, 0)), dtype=torch.int64, device=dev)
    state_slot = torch.zeros(rows, dtype=torch.int64, device=dev)
    Zs = torch.zeros((rows, max(n_keep, 0), z0.shape[1]), dtype=z0.dtype, device=dev)
    z_burn = z.clone()
    for it in range(n_iter):
        if it == n_burn:
            z_burn = z.clone()
        zp = proposal(z, eps[it], sd)
        prop = {name: fn(zp) for name, fn in evaluators.items()}
        prior = 0.5 * (z.to(F64) ** 2 - zp.to(F64) ** 2).sum(1)
        a = {name: cur[name][0] - prop[name][0] + prior for name in evaluators}
        S = 2.0 * n_bins + cur["plain"][1] + prop["plain"][1]
        acc = decide(it, z, zp, a).to(torch.bool)
        for name in evaluators:
            out["a"][name].append(a[name])
        out["S"].append(S)
        out["Z"].append(z.clone())
        out["Zp"].append(zp)
        out["acc"].append(acc)
        z = torch.where(acc[:, None], zp, z)
        for name in evaluators:
            cur[name] = tuple(None if c is None else torch.where(acc, p, c) for c, p in zip(cur[name], prop[name]))
        n_acc += acc.to(torch.int64)
        if it >= n_burn:
            r = it - n_burn
            state_slot = torch.where(acc, torch.full_like(state_slot, 1 + r), state_slot)
            slot[:, r] = state_slot
            Zs[:, r] = z
    if n_iter == n_burn:
        z_burn = z.clone()
    out["a"] = {name: torch.stack(v) for name, v in out["a"].items()}
    for key in ("S", "Z", "Zp", "acc"):
        out[key] = torch.stack(out[key])
    out.update(Zs=Zs, Z_end=z, Z_burn=z_burn, n_acc=n_acc, slot=slot)
    return out


class Evaluator:
    """``fn(z) -> (l, q)`` bound to the rows' labels / gains / spectra; ``n_bins`` = F."""

    def __init__(self, fn, n_bins):
        self.fn, self.n_bins = fn, n_bins

    def __call__(self, z):
        return self.fn(z)


def plain_evaluator(dec, P, Vb, g, y=None):
    """Rows' float64 likelihood with the FP32 weights (P, Vb ``[rows][F]``, g ``[rows]``, y ``[rows][y_dim]`` or None)."""
    return Evaluator(lambda z: loglik_plain(dec.pre(z, y), g, Vb, P), P.shape[1])


def mirrored_evaluator(dec, Pp, Vbp, g, y=None, ybias=None):
    """Rows' float64 likelihood with the sampler's rounding points, on the stream's own P' / Vb'."""
    return Evaluator(lambda z: (loglik_stream(dec.v(z, y, ybias), g, Pp, Vbp), None), Pp.shape[1])
