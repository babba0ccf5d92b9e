"""The float64 replay of oracle/mh_replay.py against the oracle port's own Metropolis-Hastings taps (CPU only).

Given the port's decisions, the plain replay must walk the same chains bit for bit (proposals, states, kept samples) and
reproduce the port's float32 log ratios to float32 rounding: the replay is then a faithful reference for the GPU samplers
(tests/test_gpu_sampler_replay.py)."""
import pytest
import torch

from oracle import mcem_port, mh_replay
from tests.golden_io import Golden, case_names

# Error model of the port's float32 log ratio against float64: every bin term ln Vx - ln Vx' + (1/Vx - 1/Vx') P carries the
# float32 rounding of the decoder and of the sum, of the order of the unit roundoff 2^-24 relative to that term, and the
# terms add up to at most S = sum_f (2 + P/Vx + P/Vx') in magnitude (plus the prior term).  Measured over all golden cases
# (first E-step, every iteration): max |a_port - a_replay| / S = 6.5e-8 (cfg1_M1); bound 2^-23 = 1.2e-7.
A_REL = 2.0 ** -23


class _Recording:
    """Passes a draw source through and keeps the randn(L, N) / rand(N) pairs of the sampler."""

    def __init__(self, inner):
        self.inner, self.eps, self.u = inner, [], []

    def rand(self, *shape):
        t = self.inner.rand(*shape)
        self.u.append(t.clone())
        return t

    def randn(self, *shape):
        t = self.inner.randn(*shape)
        self.eps.append(t.clone())
        return t


@pytest.mark.parametrize("name", case_names())
def test_plain_replay_reproduces_the_oracle_taps(name):
    torch.set_num_threads(1)
    g = Golden(name)
    o = mcem_port.MCEMOracle(g.variant, g.niter, *g.sched, g.var_RW, draws=mcem_port.ReplayDraws(g.draws))
    o.init_parameters(g.X, g.S, g.sd, g.K, g.eps, y=g.y)
    (kE, bE), _ = o.schedule()
    rec = _Recording(o.draws)
    o.draws = rec
    o.taps = []
    z0 = o.Z.t().contiguous().clone()
    Zs_port = o.sample_posterior(o.Z, kE, bE)
    n_iter = kE + bE
    assert len(rec.eps) == n_iter and len(rec.u) == n_iter
    eps = torch.stack([e.t() for e in rec.eps]).contiguous()                    # randn(L, N) -> [it][N][L]
    y = None if o.y is None else o.y.t()
    dec = mh_replay.PlainDecoder(g.sd)
    ev = {"plain": mh_replay.plain_evaluator(dec, o.P.t(), o.Vb.t(), o.g, y)}
    acc = [t["acc"] for t in o.taps]
    rep = mh_replay.replay(ev, z0, eps, g.var_RW, bE, lambda it, z, zp, a: acc[it])
    N = g.X.shape[1]
    worst = 0.0
    for it, tap in enumerate(o.taps):
        assert torch.equal(rep["Z"][it], tap["Z"].t()), "state before iteration %d" % it
        assert torch.equal(rep["Zp"][it], tap["Zp"].t()), "proposal of iteration %d" % it
        err = (rep["a"]["plain"][it] - tap["a"].to(torch.float64)).abs()
        S = rep["S"][it]
        assert torch.all(err <= A_REL * S), "iteration %d: %s" % (it, (err / S).max().item())
        worst = max(worst, float((err / S).max()))
    assert torch.equal(rep["Zs"], Zs_port)
    assert torch.equal(rep["n_acc"], torch.stack(acc).sum(0))
    assert rep["Zs"].shape == (N, kE, g.L) and worst > 0.0
