"""``mcem_port.m_step_f64``: the float64 M-step the GPU M-step tests compare against, pinned to the reference's M-step
(``m_step_reference``) and to direct formulas of its intermediates."""
import numpy as np
import pytest
import torch

from oracle import mcem_port


def _inputs(F, N, K, R, seed):
    rng = np.random.default_rng(seed)
    P = rng.gamma(1.0, 1.0, size=(F, N)).astype(np.float32) * 0.1
    Vs = rng.gamma(2.0, 0.05, size=(R, F, N)).astype(np.float32)
    W = np.maximum(rng.uniform(size=(F, K)), 1e-8).astype(np.float32)
    H = np.maximum(rng.uniform(size=(K, N)), 1e-8).astype(np.float32)
    g = rng.uniform(0.5, 1.5, size=N).astype(np.float32)
    return P, Vs, W, H, g


@pytest.mark.parametrize("F,N,K,R", [(33, 9, 3, 7), (513, 12, 10, 10), (64, 1, 1, 1)])
def test_f64_equals_the_reference_m_step_to_float32_rounding(F, N, K, R):
    P, Vs, W, H, g = _inputs(F, N, K, R, seed=F + N)
    ref = mcem_port.m_step_reference(*(torch.tensor(a) for a in (P, Vs, W, H, g)))
    got = mcem_port.m_step_f64(P, Vs, W, H, g)
    assert mcem_port.m_step_in_range(got)
    for k in ("W", "H", "g", "Vb"):
        r = ref[k].numpy().astype(np.float64)
        assert np.all(np.abs(r - got[k]) <= 2e-6 * np.abs(got[k])), k
    assert abs(ref["cost"].item() - got["cost"]) <= 1e-6 * abs(got["cost"])


@pytest.mark.parametrize("F,N,K,R", [(33, 9, 3, 7), (513, 5, 10, 30)])
def test_f64_equals_the_reference_m_step_run_in_double(F, N, K, R):
    P, Vs, W, H, g = (a.astype(np.float64) for a in _inputs(F, N, K, R, seed=7 * F + N))
    ref = mcem_port.m_step_reference(*(torch.tensor(a) for a in (P, Vs, W, H, g)))
    got = mcem_port.m_step_f64(P, Vs, W, H, g)
    for k in ("W", "H", "g", "Vb"):
        np.testing.assert_allclose(got[k], ref[k].numpy(), rtol=1e-12, atol=0, err_msg=k)
    assert abs(ref["cost"].item() - got["cost"]) <= 1e-12 * abs(got["cost"])


def test_f64_intermediates_equal_direct_formulas():
    F, N, K, R = 40, 11, 4, 6
    P, Vs, W, H, g = (a.astype(np.float64) for a in _inputs(F, N, K, R, seed=3))
    segs = [(0, 1), (1, 8), (8, 11)]
    got = mcem_port.m_step_f64(P, Vs, W, H, g, segments=segs)
    Vx = g[None, None, :] * Vs + np.einsum("fk,kn->fn", W, H)[None]
    A1 = np.sum(1.0 / Vx, axis=0)
    A2 = np.sum(1.0 / Vx ** 2, axis=0)
    np.testing.assert_allclose(got["A1"], A1, rtol=1e-13)
    np.testing.assert_allclose(got["A2"], A2, rtol=1e-13)
    for s, (a, b) in enumerate(segs):
        for k in range(K):
            num = sum(P[:, n] * A2[:, n] * H[k, n] for n in range(a, b))
            den = sum(A1[:, n] * H[k, n] for n in range(a, b))
            np.testing.assert_allclose(got["Wpart"][s, k, 0], num, rtol=1e-13)
            np.testing.assert_allclose(got["Wpart"][s, k, 1], den, rtol=1e-13)
    np.testing.assert_allclose(got["Wpart"].sum(0)[:, 0].T, got["Wnum"], rtol=1e-13)
    np.testing.assert_allclose(got["Wpart"].sum(0)[:, 1].T, got["Wden"], rtol=1e-13)
    # the cost terms belong to the refreshed Vx = g_new Vs + Vb with the un-normalised Vb (SURVEY Q4)
    Vx3 = got["g"][None, None, :] * Vs + got["Vb"][None]
    np.testing.assert_allclose(got["cost_terms"], np.log(Vx3) + P[None] / Vx3, rtol=1e-13)
    assert got["cost"] == pytest.approx(got["cost_terms"].mean(), rel=1e-15)
    # Vb is W_new H_new before the column normalisation, whose factors cancel in the product
    np.testing.assert_allclose(got["Vb"], got["W"] @ got["H"], rtol=1e-12)


def test_f64_bounds_follow_the_error_model():
    """Relative bounds are positive, grow with the reduction lengths, and the float32 reference meets them on benign inputs."""
    F, N, K, R = 513, 20, 10, 10
    P, Vs, W, H, g = _inputs(F, N, K, R, seed=11)
    a = mcem_port.m_step_f64(P, Vs, W, H, g)
    b = mcem_port.m_step_f64(P, np.concatenate([Vs, Vs]), W, H, g)
    for k in ("W", "H", "g", "Vb", "A1", "A2"):
        assert np.all(a["bound_" + k] > 0)
        rel_a = np.max(a["bound_" + k] / np.abs(a[k]))
        assert 10 * mcem_port.U32 < rel_a < 1e-4, (k, rel_a)
        assert np.max(b["bound_" + k] / np.abs(b[k])) > rel_a                 # twice the samples: longer sums
    assert 0 < a["bound_cost"] < 1e-4 * abs(a["cost"])
    f32 = mcem_port.m_step_reference(*(torch.tensor(x) for x in (P, Vs, W, H, g)))
    for k in ("W", "H", "g", "Vb"):
        assert np.all(np.abs(f32[k].numpy() - a[k]) <= a["bound_" + k]), k
    assert abs(f32["cost"].item() - a["cost"]) <= a["bound_cost"]


def test_range_check_sees_every_pass():
    F, N, K, R = 16, 4, 2, 4
    P, Vs, W, H, g = (x.astype(np.float64) for x in _inputs(F, N, K, R, seed=5))
    assert mcem_port.m_step_in_range(mcem_port.m_step_f64(P, Vs, W, H, g))
    assert not mcem_port.m_step_in_range(mcem_port.m_step_f64(P, Vs * 2.0 ** 64, W * 2.0 ** 64, H, g))
    assert not mcem_port.m_step_in_range(mcem_port.m_step_f64(P * 2.0 ** -130, Vs * 2.0 ** -64, W * 2.0 ** -64, H, g))
    spread = Vs.copy()
    spread[1:] *= 2.0 ** 34                                                   # the bin's first sample far below the others
    assert not mcem_port.m_step_in_range(mcem_port.m_step_f64(P, spread, W * 1e-12, H, g))
