"""CPU-side checks of per-utterance EM stopping (McemConfig.stop_tol): a restatement of the stopping test on crafted cost rows,
and the argument errors raised before any device work."""
import math

import numpy as np
import pytest

from dvae_b200.engine import McemConfig, check_stop
from dvae_b200.packages.models import mcem


def stop_iterations(cost, tol, window, niter=None):
    """The stopping test restated with Python float sums in ascending order: ``cost [B][niter]`` (0-based iteration k) ->
    ``n_u``, the first ``n >= 2w`` (1-based count, ``n < niter``) with ``m_old - m_new <= tol |m_new|``, else ``niter``."""
    cost = np.asarray(cost, np.float64)
    niter = cost.shape[1] if niter is None else niter
    out = np.full(cost.shape[0], niter, np.int64)
    for u, row in enumerate(cost):
        for n in range(2 * window, niter):
            s_old = s_new = 0.0
            for k in range(n - 2 * window, n - window):
                s_old += float(row[k])
            for k in range(n - window, n):
                s_new += float(row[k])
            m_old, m_new = s_old / window, s_new / window
            if m_old - m_new <= tol * abs(m_new):
                out[u] = n
                break
    return out


def test_restatement_on_crafted_rows():
    # strictly decreasing by 1 per iteration: every improvement is positive, so tol = 0 never stops
    assert stop_iterations([100.0 - np.arange(12.0)], 0.0, 2)[0] == 12
    # the == boundary stops: after n = 4 (w = 2) m_old = 6, m_new = 4 and m_old - m_new = 2 = 0.5 * |4|, exactly
    edge = [6.0, 6.0, 4.0, 4.0, 4.0, 4.0]
    assert stop_iterations([edge], 0.5, 2)[0] == 4
    assert stop_iterations([edge], np.nextafter(0.5, 0.0), 2)[0] == 5
    # n < 2w never stops, even on a flat row
    flat = np.full(12, 3.0)
    assert stop_iterations([flat], 0.0, 3)[0] == 6
    assert stop_iterations([flat], 0.0, 6)[0] == 12                 # 2w = niter: no test before the cap
    # w = 1: compares single iterations
    assert stop_iterations([[5.0, 4.0, 4.0, 3.0]], 0.0, 1)[0] == 3
    # negative costs: |m_new| in the tolerance, a rise stops at once
    neg = -1000.0 - np.arange(10.0)
    assert stop_iterations([neg], 1.0 / 1000.0, 1)[0] == 2
    assert stop_iterations([neg], 0.5 / 1002.0, 1)[0] == 10
    assert stop_iterations([[-5.0, -4.0, -3.0, -2.0]], 0.0, 1)[0] == 2
    # NaN never passes the test
    nan_row = flat.copy()
    nan_row[3] = math.nan
    assert stop_iterations([nan_row], 1e9, 2)[0] == 8               # the first window pair without k = 3: n = 8 (k = 4..7)
    assert stop_iterations([np.full(8, math.nan)], 1e9, 1)[0] == 8


@pytest.mark.parametrize("kw", [dict(stop_tol=-1e-3), dict(stop_tol=math.nan), dict(stop_tol=math.inf), dict(stop_tol=True),
                                dict(stop_tol="0.1"), dict(stop_tol=1e-3, stop_window=0), dict(stop_tol=1e-3, stop_window=-2),
                                dict(stop_tol=1e-3, stop_window=2.0)])
def test_check_stop_rejects_bad_settings(kw):
    with pytest.raises(ValueError):
        check_stop(McemConfig(**kw))
    with pytest.raises(ValueError):
        mcem.MCEM_M1(100, **kw)


def test_check_stop_rejects_draws_and_checkpoints():
    cfg = McemConfig(stop_tol=1e-3)
    check_stop(cfg)
    check_stop(McemConfig(stop_window=0))                            # off: the window is not read
    with pytest.raises(ValueError):
        check_stop(cfg, draws=object())
    with pytest.raises(ValueError):
        check_stop(cfg, checkpoints=(2, 4))
    with pytest.raises(ValueError):
        mcem.MCEM_M1(100, stop_tol=1e-3, rng="torch")
    assert mcem.MCEM_M1(100, stop_tol=0, stop_window=3).stop_window == 3


def test_engine_and_enhancer_check_before_device_work():
    """McemEngine refuses a bad stopping setting before it looks for a device, Enhancer.enhance before it stages anything."""
    from dvae_b200.engine import Enhancer, McemEngine
    with pytest.raises(ValueError):
        McemEngine(None, McemConfig(stop_tol=-1.0), "cuda:0")
    enh = Enhancer.__new__(Enhancer)                                 # no weights, no device: only the argument checks run
    enh.engine = McemEngine.__new__(McemEngine)
    enh.engine.cfg = McemConfig(niter=6, stop_tol=1e-3, stop_window=2)
    enh.dev = None
    x = [np.zeros(4000, np.float32)]
    with pytest.raises(ValueError):
        Enhancer.enhance.__wrapped__(enh, x, ref_list=x, score_at=(2,))
    with pytest.raises(ValueError):
        Enhancer.enhance.__wrapped__(enh, x, draws=object())
