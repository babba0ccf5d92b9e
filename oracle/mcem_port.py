"""CPU restatement of the reference's Monte-Carlo EM enhancement algorithm.  Oracle: test infrastructure only.

Restates, with CPU torch float32 ops in the reference's arithmetic order (so that results are
bit-identical to the reference on the same inputs and draws; pinned by ``tests/golden/mcem_*.npz``,
see ``oracle/make_golden.py``):

* ``packages/models/models.py:8-38,91-122``  tanh-MLP encoder with Gaussian head / decoder with exp output;
* ``packages/models/mcem.py:36-58``          NMF / gain initialisation;
* ``packages/models/mcem.py:207-277`` (M1), ``372-448`` (M2), ``544-620`` (M2v2), ``716-792`` (M2v3)
                                             random-walk Metropolis-Hastings over the latents;
* ``packages/models/mcem.py:91-153``         multiplicative updates of W, H, g;
* ``packages/models/mcem.py:69-71,156-179``  cost, EM loop, Wiener estimates.

The four reference classes differ only in (a) whether a label ``y`` is concatenated to the decoder /
encoder inputs and (b) the M1 call-site quirk that shifts the Metropolis-Hastings schedule (SURVEY Q1).
Here they are one class with a ``variant`` switch and an explicit ``schedule()``.

Random numbers come from a *draw source* so tests can record the reference's draws and replay them
into both this port and the CUDA path (consumption order: SURVEY §3.3).
"""
from __future__ import annotations

import numpy as np
import torch

VARIANTS = ("M1", "M2", "M2v2", "M2v3")


# --------------------------------------------------------------------------- draw sources
class TorchDraws:
    """Draws from torch's global CPU generator, exactly like the reference on ``device='cpu'``."""

    def rand(self, *shape):
        return torch.rand(*shape)

    def randn(self, *shape):
        return torch.randn(*shape)


class RecordingDraws(TorchDraws):
    """Global-generator draws, remembered as ``[(kind, tensor), ...]``."""

    def __init__(self):
        self.log = []

    def rand(self, *shape):
        t = torch.rand(*shape)
        self.log.append(("rand", t.clone()))
        return t

    def randn(self, *shape):
        t = torch.randn(*shape)
        self.log.append(("randn", t.clone()))
        return t


class ReplayDraws:
    """Replays a recorded list of ``(kind, array)`` in order, checking kind and shape."""

    def __init__(self, log):
        self.log = [(k, torch.as_tensor(np.asarray(v), dtype=torch.float32)) for k, v in log]
        self.pos = 0

    def _next(self, kind, shape):
        if self.pos >= len(self.log):
            raise RuntimeError("replay exhausted after %d draws" % self.pos)
        k, t = self.log[self.pos]
        if len(shape) == 1 and isinstance(shape[0], (tuple, list, torch.Size)):
            shape = tuple(shape[0])
        if k != kind or tuple(t.shape) != tuple(shape):
            raise RuntimeError("draw %d: wanted %s%s, recorded %s%s" % (self.pos, kind, tuple(shape), k, tuple(t.shape)))
        self.pos += 1
        return t.clone()

    def rand(self, *shape):
        return self._next("rand", shape)

    def randn(self, *shape):
        return self._next("randn", shape)


# --------------------------------------------------------------------------- VAE MLPs (models.py)
def _t(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32) if not torch.is_tensor(a) else a


def _hidden_count(sd, prefix):
    n = 0
    while f"{prefix}hidden.{n}.weight" in sd:
        n += 1
    return n


def encoder_forward(sd, x, draws, prefix="encoder."):
    """``Encoder.forward`` + ``GaussianSample`` (models.py:24-38,102-105) -> ``(z, mu, log_var)``.

    The reparametrisation noise is ``randn(mu.size())`` drawn on the CPU generator (models.py:10).
    """
    h = x
    for i in range(_hidden_count(sd, prefix)):
        h = torch.tanh(torch.nn.functional.linear(h, _t(sd[f"{prefix}hidden.{i}.weight"]), _t(sd[f"{prefix}hidden.{i}.bias"])))
    mu = torch.nn.functional.linear(h, _t(sd[f"{prefix}sample.mu.weight"]), _t(sd[f"{prefix}sample.mu.bias"]))
    log_var = torch.nn.functional.linear(h, _t(sd[f"{prefix}sample.log_var.weight"]), _t(sd[f"{prefix}sample.log_var.bias"]))
    epsilon = draws.randn(mu.size())
    std = log_var.mul(0.5).exp_()
    z = mu.addcmul(std, epsilon)
    return z, mu, log_var


def decoder_forward(sd, z, prefix="decoder."):
    """``Decoder.forward`` (models.py:119-122): tanh hidden layers, ``exp`` of the output layer."""
    h = z
    for i in range(_hidden_count(sd, prefix)):
        h = torch.tanh(torch.nn.functional.linear(h, _t(sd[f"{prefix}hidden.{i}.weight"]), _t(sd[f"{prefix}hidden.{i}.bias"])))
    return torch.exp(torch.nn.functional.linear(h, _t(sd[f"{prefix}reconstruction.weight"]), _t(sd[f"{prefix}reconstruction.bias"])))


def vae_forward(sd, variant, x, y, draws):
    """Container ``forward`` (models.py:172-180 M1; 201-204 M2; 280-287 v3): ``(x_mu, z, z_mu, z_log_var)``."""
    enc_in = torch.cat([x, y], dim=1) if variant == "M2" else x
    z, mu, lv = encoder_forward(sd, enc_in, draws)
    dec_in = z if variant == "M1" else torch.cat([z, y], dim=1)
    return decoder_forward(sd, dec_in), z, mu, lv


# --------------------------------------------------------------------------- MCEM
class MCEMOracle:
    """One class for ``MCEM_M1`` / ``MCEM_M2`` / ``MCEM_M2v2`` / ``MCEM_M2v3`` (mcem.py:182-845)."""

    def __init__(self, variant, niter, nsamples_E_step=10, burnin_E_step=30, nsamples_WF=25, burnin_WF=75,
                 var_RW=0.01, draws=None):
        if variant not in VARIANTS:
            raise ValueError(variant)
        self.variant = variant
        self.niter = niter
        self.nsamples_E_step, self.burnin_E_step = nsamples_E_step, burnin_E_step
        self.nsamples_WF, self.burnin_WF = nsamples_WF, burnin_WF
        self.var_RW = var_RW
        self.draws = draws if draws is not None else TorchDraws()
        self.taps = None          # set to a list to record per-MH-iteration (Z', a, u, accepted)

    def schedule(self):
        """``((keep_E, burn_E), (keep_WF, burn_WF))`` actually executed.

        M1 calls ``sample_posterior(self.Z, nsamples, burnin)`` against the signature
        ``(Z, y, nsamples=10, burnin=30)`` (mcem.py:207 vs 297-298, 314-315), so the *burn-in argument*
        becomes the number of kept samples and the burn-in falls back to its default 30 (SURVEY Q1).
        """
        if self.variant == "M1":
            return (self.burnin_E_step, 30), (self.burnin_WF, 30)
        return (self.nsamples_E_step, self.burnin_E_step), (self.nsamples_WF, self.burnin_WF)

    # -- mcem.py:36-58 + 195-205 / 358-370 / 530-542 / 702-714
    def init_parameters(self, X, S, sd, nmf_rank, eps, y=None):
        if (self.variant == "M1") != (y is None):
            raise ValueError("y must be given exactly for the M2 variants")
        F, N = X.shape
        d = self.draws
        self.W = torch.max(d.rand(F, nmf_rank), eps * torch.ones(F, nmf_rank))
        self.H = torch.max(d.rand(nmf_rank, N), eps * torch.ones(nmf_rank, N))
        self.g = torch.ones(N)
        self.X = X
        self.P = torch.tensor(np.abs(X) ** 2)
        self.P_clean = torch.tensor(np.abs(S) ** 2)
        self.Vb = self.W @ self.H
        self.sd = sd
        self.y = None if y is None else _t(y)
        if self.variant == "M2":
            enc_x = torch.t(torch.cat([self.P, self.y], dim=0))
            enc_s = torch.t(torch.cat([self.P_clean, self.y], dim=0))
        else:
            enc_x, enc_s = torch.t(self.P), torch.t(self.P_clean)
        # `_, Z, _ = encoder(...)`: the reference keeps the posterior MEAN as the chain start;
        # the reparametrisation draw is consumed and discarded (mcem.py:200-203, models.py:38).
        _, mu_x, _ = encoder_forward(sd, enc_x, d)
        _, mu_s, _ = encoder_forward(sd, enc_s, d)
        self.Z = torch.t(mu_x)
        self.Zclean = torch.t(mu_s)
        self.L = self.Z.shape[0]
        self.Vs = self.Vs_scaled = self.Vx = None

    def _decode_cols(self, Z):
        """Decoder on latent columns ``Z`` (L, N) [+ labels] -> speech variance (F, N)."""
        inp = Z if self.y is None else torch.cat([Z, self.y], dim=0)
        return torch.t(decoder_forward(self.sd, torch.t(inp)))

    # -- mcem.py:207-277 (and the three M2 copies)
    def sample_posterior(self, Z, n_keep, n_burn):
        F, N = self.X.shape
        L = self.L
        var = torch.tensor(np.float32(self.var_RW))
        Zs = torch.zeros(N, n_keep, L)
        Zc = Z.clone()
        g, Vb, P = self.g.clone(), self.Vb.clone(), self.P
        Vx = g * self._decode_cols(Zc) + Vb
        kept = 0
        for m in range(n_keep + n_burn):
            Zp = Zc + torch.sqrt(var) * self.draws.randn(L, N)
            Vxp = g * self._decode_cols(Zp) + Vb
            a = (torch.sum(torch.log(Vx) - torch.log(Vxp) + (1 / Vx - 1 / Vxp) * P, 0)
                 + .5 * torch.sum(Zc.pow(2) - Zp.pow(2), 0))
            u = self.draws.rand(N)
            acc = torch.log(u) < a
            if self.taps is not None:
                self.taps.append(dict(Z=Zc.clone(), Zp=Zp.clone(), a=a.clone(), u=u.clone(), acc=acc.clone()))
            Zc[:, acc] = Zp[:, acc]
            Vx = g * self._decode_cols(Zc) + Vb
            if m > n_burn - 1:
                Zs[:, kept, :] = torch.t(Zc)
                kept += 1
        return Zs

    # -- mcem.py:280-290
    def compute_Vs(self, Zs):
        inp = Zs
        if self.y is not None:
            yy = torch.t(self.y)[:, None, :].expand(-1, Zs.shape[1], -1)
            inp = torch.cat([Zs, yy], dim=2)
        with torch.no_grad():
            V = decoder_forward(self.sd, inp)        # (N, R, F)
        self.Vs = V.permute(1, 2, 0)                 # (R, F, N) view, same strides as the reference's

    def _refresh(self):
        self.Vs_scaled = self.g * self.Vs
        self.Vx = self.Vs_scaled + self.Vb

    # -- mcem.py:292-308
    def E_step(self):
        (keep, burn), _ = self.schedule()
        Zs = self.sample_posterior(self.Z, keep, burn)
        self.Z = torch.t(torch.squeeze(Zs[:, -1, :]))
        self.compute_Vs(Zs)
        self._refresh()

    # -- mcem.py:91-153
    def M_step(self):
        P = self.P
        num = (P * torch.sum(self.Vx ** -2, axis=0)) @ self.H.T
        den = torch.sum(self.Vx ** -1, axis=0) @ self.H.T
        self.W = self.W * (num / den) ** .5
        self.Vb = self.W @ self.H
        self.Vx = self.Vs_scaled + self.Vb

        num = self.W.T @ (P * torch.sum(self.Vx ** -2, axis=0))
        den = self.W.T @ torch.sum(self.Vx ** -1, axis=0)
        self.H = self.H * (num / den) ** .5
        self.Vb = self.W @ self.H
        self.Vx = self.Vs_scaled + self.Vb

        # column-L1 normalisation of W, compensated in H; Vb is NOT recomputed afterwards (SURVEY Q4)
        norm = torch.sum(torch.abs(self.W), axis=0)
        self.W = self.W / norm.unsqueeze(0)
        self.H = self.H * norm.unsqueeze(1)

        num = torch.sum(P * torch.sum(self.Vs * (self.Vx ** -2), axis=0), axis=0)
        den = torch.sum(torch.sum(self.Vs * (self.Vx ** -1), axis=0), axis=0)
        self.g = self.g * (num / den) ** .5
        self._refresh()

    def cost_value(self):
        # mcem.py:69-71
        return torch.mean(torch.log(self.Vx) + self.P / self.Vx)

    # -- mcem.py:310-329
    def compute_WF(self):
        _, (keep, burn) = self.schedule()
        Zs = self.sample_posterior(self.Z, keep, burn)
        self.compute_Vs(Zs)
        self._refresh()
        return torch.mean(self.Vs_scaled / self.Vx, axis=0), torch.mean(self.Vb / self.Vx, axis=0)

    # -- mcem.py:156-179
    def run(self):
        cost = np.zeros(self.niter)
        for n in range(self.niter):
            self.E_step()
            self.M_step()
            cost[n] = self.cost_value()
        WFs, WFn = self.compute_WF()
        self.WFs, self.WFn = WFs, WFn
        self.S_hat = WFs.numpy() * self.X
        self.N_hat = WFn.numpy() * self.X
        return cost


# --------------------------------------------------------------------------- stage-level helpers for parity tests
def m_step_reference(P, Vs, W, H, g):
    """One M-step on explicit inputs (all torch, shapes as the reference: Vs (R,F,N)) -> dict of outputs."""
    o = MCEMOracle("M1", 1)
    o.P, o.Vs, o.W, o.H, o.g = P, Vs, W.clone(), H.clone(), g.clone()
    o.Vb = o.W @ o.H
    o._refresh()
    o.M_step()
    return dict(W=o.W, H=o.H, g=o.g, Vb=o.Vb, Vx=o.Vx, cost=o.cost_value())


# Error model of the CUDA M-step (nmf.cu, vst.cu, decode_stats_tc.cu) against float64.  Every sum of the M-step except the
# cost adds positive terms, so a relative error bound of the terms carries over to the sum plus u per addition along the
# longest chain of additions; products add their factors' bounds, sqrt halves its argument's.  u = 2^-24 (FP32 rounding).
U32 = 2.0 ** -24
RCP_REL = 4 * U32            # 1 / Vx through the pair trick: x0 x1 (u), rcp.approx (1 ulp <= 2u), x1 * rcp (u)
VX_IN_REL = 3 * U32          # g Vs: g E (u, emission), (g E) v (u), Vs = E v of the unpacked reference (u)
DEPTH_F = 17                 # additions of a sum over the bins: <= 3 bins per thread (2), 5 shuffle levels, 8 warps, bin 512's term
LG2_ABS = 2.0 ** -22         # lg2.approx.f32 absolute error (PTX ISA); one per product of up to four samples, counted per sample
QUAD_REL = 12 * U32          # P / Vx of the cost pass: three products of four y (3u), two sums (2u), rcp.approx (2u), scaling (5u)
# Vx = g Vs + Vb range the M-step's FP32 arithmetic handles: pair products x0 x1 stay normal (2^-126 .. 2^126 leaves the
# reciprocal normal under .ftz), with a margin of 2^4 for R <= 256 reciprocal squares summed and multiplied by P.
VX_MIN, VX_MAX = 2.0 ** -60, 2.0 ** 60
BIN_SPREAD_LOG2 = 31         # the cost passes' per-bin scale: samples of a bin within 2^+-31 of the bin's first sample


def m_step_f64(P, Vs, W, H, g, segments=None, chains=1, stats_rel=None):
    """One M-step (mcem.py:91-153, the order of ``MCEMOracle.M_step``) in float64, with its intermediates and error bounds.

    ``P`` (F,N), ``Vs`` (R,F,N), ``W`` (F,K), ``H`` (K,N), ``g`` (N,): one utterance, numpy or torch.  ``segments``: frame
    ranges ``[(a, b), ...]`` whose W-update sums are returned separately (the layout of ``Wpart``, [S][K][2][F]).  ``chains``:
    sample rows per frame in the W reduction (its additions run over ``N * chains`` rows).  ``stats_rel``: relative error of
    A1 / A2 when the caller hands them to the kernels itself (FP32 rounding of these float64 values: ``U32``).

    Returns float64 numpy arrays: ``W H g Vb cost`` as ``m_step_reference``, ``cost_terms`` = ln Vx + P / Vx (R,F,N), ``A1``
    ``A2`` (F,N) with the E-step's g and Vb, ``Wnum Wden`` (F,K) = sum_n P A2 H, sum_n A1 H (``Wpart`` with segments), the
    error-model bounds ``bound_W bound_H bound_g bound_Vb bound_A1 bound_A2 bound_Wsum`` (absolute, per element) and
    ``bound_cost``, and for range checks ``vx_min vx_max`` over every Vx the M-step forms and ``spread_log2``, the largest
    |log2(Vx_r / Vx_0)| of a bin in the cost pass.
    """
    f64 = lambda a: (a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)).astype(np.float64)
    P, Vs, W, H, g = f64(P), f64(Vs), f64(W), f64(H), f64(g)
    R, F, N = Vs.shape
    K = W.shape[1]
    u = U32
    out = {}
    Vx0 = g * Vs + W @ H
    A1, A2 = (1.0 / Vx0).sum(0), (1.0 / Vx0 ** 2).sum(0)
    numW, denW = (P * A2) @ H.T, A1 @ H.T
    Wt = W * np.sqrt(numW / denW)
    Vx1 = g * Vs + Wt @ H
    numH, denH = Wt.T @ (P * (Vx1 ** -2).sum(0)), Wt.T @ (Vx1 ** -1).sum(0)
    Ht = H * np.sqrt(numH / denH)
    Vb = Wt @ Ht
    Vx2 = g * Vs + Vb
    norm = np.abs(Wt).sum(0)
    ng, dg = (P * (Vs * Vx2 ** -2).sum(0)).sum(0), (Vs * Vx2 ** -1).sum(0).sum(0)
    gn = g * np.sqrt(ng / dg)
    Vx3 = gn * Vs + Vb
    terms = np.log(Vx3) + P / Vx3
    out.update(W=Wt / norm, H=Ht * norm[:, None], g=gn, Vb=Vb, cost=terms.mean() if terms.size else 0.0, cost_terms=terms,
               A1=A1, A2=A2, Wnum=numW, Wden=denW)
    if segments is not None:
        out["Wpart"] = np.stack([np.stack([(P * A2)[:, a:b] @ H[:, a:b].T, A1[:, a:b] @ H[:, a:b].T], 0).transpose(2, 0, 1)
                                 for a, b in segments]) if len(segments) else np.zeros((0, K, 2, F))
    # ---- relative bounds, pass by pass (all terms positive: one number per output)
    e_vx0 = VX_IN_REL + K * u + u                                        # Vb = W H by K FMAs, then + g Vs
    e_a1 = e_vx0 + RCP_REL + (R - 1) * u
    e_a2 = 2 * (e_vx0 + RCP_REL) + u + (R - 1) * u
    ea1w, ea2w = (stats_rel, stats_rel) if stats_rel is not None else (e_a1, e_a2)
    rows = N * chains + (len(segments) if segments else 0)               # W sums: every row, then the segments in order
    e_wsum_num, e_wsum_den = ea2w + 2 * u + rows * u, ea1w + u + rows * u
    e_wt = (e_wsum_num + e_wsum_den) / 2 + 3 * u                         # division, sqrt, product with W: u each
    e_norm = e_wt + DEPTH_F * u
    e_vx1 = max(VX_IN_REL, e_wt + K * u) + u
    e_a1h, e_a2h = e_vx1 + RCP_REL + (R - 1) * u, 2 * (e_vx1 + RCP_REL) + u + (R - 1) * u
    e_hs = ((e_wt + e_a2h + 2 * u) + (e_wt + e_a1h + u)) / 2 + DEPTH_F * u + 3 * u
    e_vb2 = e_wt + e_hs + K * u
    e_vx2 = max(VX_IN_REL, e_vb2) + u
    e_ng = 2 * (e_vx2 + RCP_REL) + 4 * u + (R + DEPTH_F) * u             # Vs / Vx (u), / Vx (u), E (u), P (u)
    e_dg = e_vx2 + RCP_REL + 2 * u + (R + DEPTH_F) * u
    e_g = (e_ng + e_dg) / 2 + 3 * u
    e_vx3 = max(e_g + VX_IN_REL, e_vb2) + 3 * u                           # + the bin scale folded into g E and Vb
    depth_c = 3 * R + DEPTH_F                                             # per-thread FP32 cost sum over <= 3 bins x R samples
    pv = P / Vx3
    per = (e_vx3 + QUAD_REL) * (1 + pv) + LG2_ABS * np.log(2.0) + depth_c * u * (1 + 2 * np.abs(np.log(Vx3)) + pv)
    out.update(bound_W=(e_wt + e_norm + u) * out["W"], bound_H=(e_hs + e_norm + u) * out["H"], bound_g=e_g * gn,
               bound_Vb=e_vb2 * Vb, bound_A1=e_a1 * A1, bound_A2=e_a2 * A2, rel_Wsum=(e_wsum_num, e_wsum_den),
               bound_cost=per.mean() if per.size else 0.0)
    vx = [Vx0, Vx1, Vx2, Vx3]
    out["vx_min"] = min(float(v.min()) for v in vx) if Vs.size else 1.0
    out["vx_max"] = max(float(v.max()) for v in vx) if Vs.size else 1.0
    out["spread_log2"] = float(np.abs(np.log2(Vx3 / Vx3[:1])).max()) if Vs.size else 0.0
    return out


def m_step_in_range(ref):
    """Whether the inputs of ``m_step_f64``'s result ``ref`` lie inside the range the M-step kernels handle (nmf.cu)."""
    return VX_MIN <= ref["vx_min"] and ref["vx_max"] <= VX_MAX and ref["spread_log2"] <= BIN_SPREAD_LOG2


def log_accept_reference(Vs_cur, Vs_prop, g, Vb, P, Z, Zp):
    """The log acceptance ratio of mcem.py:251-253 on explicit inputs ((F,N) variances, (L,N) latents)."""
    Vx, Vxp = g * Vs_cur + Vb, g * Vs_prop + Vb
    return (torch.sum(torch.log(Vx) - torch.log(Vxp) + (1 / Vx - 1 / Vxp) * P, 0)
            + .5 * torch.sum(Z.pow(2) - Zp.pow(2), 0))


def si_sdr(s_hat, s):
    """``si_sdr_leroux`` (packages/metrics.py:62-82) in float64."""
    s_hat = np.asarray(s_hat, np.float64)
    s = np.asarray(s, np.float64)
    alpha = np.dot(s_hat, s) / np.linalg.norm(s) ** 2
    tgt = alpha * s
    return 10 * np.log10(np.linalg.norm(tgt) ** 2 / np.linalg.norm(tgt - s_hat) ** 2)


def energy_ratios(s_hat, s, n):
    """``energy_ratios`` (packages/metrics.py:39-60) in float64 with the vectors of ``si_sdr_components`` (12-37) formed
    explicitly, exactly as the reference does."""
    s_hat, s, n = (np.asarray(a, np.float64) for a in (s_hat, s, n))
    s_target = np.dot(s_hat, s) / np.linalg.norm(s) ** 2 * s
    e_noise = np.dot(s_hat, n) / np.linalg.norm(n) ** 2 * n
    e_art = s_hat - s_target - e_noise
    st = np.linalg.norm(s_target) ** 2
    return (10 * np.log10(st / np.linalg.norm(e_noise + e_art) ** 2), 10 * np.log10(st / np.linalg.norm(e_noise) ** 2),
            10 * np.log10(st / np.linalg.norm(e_art) ** 2))

