"""The host restatement of the random numbers (oracle/philox_np.py) pinned to published and hand-derived values, and the
engine's guard against chains that would share Philox counters.  No GPU."""
import numpy as np
import pytest

from dvae_b200.engine import check_counters
from oracle import philox_np as ph


@pytest.mark.parametrize("ctr,key,out", ph.KAT)
def test_philox_known_answers(ctr, key, out):
    got = ph.philox4x32_10(*ctr, *key)
    assert tuple(int(w) for w in got) == out


def test_philox_vectorises_and_wraps_its_inputs():
    """Arrays broadcast against scalars, negative ids are taken mod 2^32, and every element equals its scalar evaluation."""
    rng = np.random.default_rng(0)
    c0 = rng.integers(-2 ** 31, 2 ** 31, 64)
    c1 = rng.integers(0, 2 ** 32, 64, dtype=np.uint64).astype(np.uint32)
    vec = ph.philox4x32_10(c0, c1, 0xFFFFFFF0, 7, 0x12345678, 0x9ABCDEF0)
    for i in range(64):
        one = ph.philox4x32_10(int(c0[i]) % 2 ** 32, int(c1[i]), 0xFFFFFFF0, 7, 0x12345678, 0x9ABCDEF0)
        assert tuple(int(w[i]) for w in vec) == tuple(int(w) for w in one)
    a = ph.philox4x32_10(1, 2, 3, 4, 5, 6)
    b = ph.philox4x32_10(1, 2, 3, 4, 5 + 2 ** 32, 6)
    assert a == b


def _u01_exact(k):
    """(k + 1/2) 2^-24 rounded to the nearest float32, ties to even, with integer arithmetic only."""
    k = np.asarray(k, np.int64)
    # float32 has 24 significant bits: below 2^23 the sum k + 1/2 is exact; above it the spacing is 1 and the tie between k
    # and k + 1 goes to the even one
    out = np.where(k < 2 ** 23, (2 * k + 1).astype(np.float64) * 2.0 ** -25, np.where(k % 2 == 0, k, k + 1).astype(np.float64) * 2.0 ** -24)
    return out


def test_u01_is_ieee_round_to_nearest_and_reaches_one():
    k = np.concatenate([np.arange(0, 4096), np.arange(2 ** 23 - 4096, 2 ** 23 + 4096), np.arange(2 ** 24 - 4096, 2 ** 24)])
    words = (k.astype(np.uint64) << np.uint64(8)).astype(np.uint32) | np.uint32(0xA5)     # the low byte is ignored
    u = ph.u01(words)
    assert u.dtype == np.float32
    assert np.array_equal(u.astype(np.float64), _u01_exact(k))
    assert ph.u01(np.uint32(0))[()] == np.float32(2.0 ** -25)
    assert ph.u01(np.uint32(0xFFFFFFFF))[()] == np.float32(1.0)
    allk = np.arange(2 ** 24, dtype=np.uint32) << np.uint32(8)
    ua = ph.u01(allk)
    assert int((ua == 1.0).sum()) == 1 and int((ua <= 0).sum()) == 0
    assert np.all(np.diff(ua) >= 0)
    assert np.all(np.diff(ua[2 ** 23:].astype(np.float64)) % 2.0 ** -23 == 0)     # upper half: the 2^-23 grid


def test_u01_low_bytes_uses_the_low_bytes_of_three_words():
    x, y, z = np.uint32(0x123456FF), np.uint32(0xABCDEFFF), np.uint32(0x000000FF)
    assert ph.u01_low_bytes(x, y, z)[()] == np.float32(1.0)
    assert ph.u01_low_bytes(np.uint32(0xFFFFFF00), np.uint32(0xFFFFFF00), np.uint32(0xFFFFFF00))[()] == np.float32(2.0 ** -25)
    v = 0x01 | (0x02 << 8) | (0x03 << 16)
    assert ph.u01_low_bytes(np.uint32(0xAB01), np.uint32(0xCD02), np.uint32(0xEF03))[()] == np.float32((v + 0.5) * 2.0 ** -24)


def test_box_muller_bound_contains_float32_evaluations():
    """The bound is not vacuous and contains a plain float32 evaluation with correctly rounded log / sin / cos (an
    implementation inside the error model); it stays finite at u1 = 1 (r = 0) and at u2 = 1 (angle just past pi)."""
    rng = np.random.default_rng(1)
    a = np.concatenate([rng.integers(0, 2 ** 32, 20000, dtype=np.uint64), [0, 255, 0xFFFFFF00, 0xFFFFFEFF, 0xFFFFFFFF]]).astype(np.uint32)
    b = np.concatenate([rng.integers(0, 2 ** 32, 20000, dtype=np.uint64), [0, 0xFFFFFFFF, 0x80000000, 0x3FFFFF00, 0xBFFFFF00]]).astype(np.uint32)
    n0, n1, b0, b1 = ph.box_muller_f64(a, b)
    assert np.all(np.isfinite(b0)) and np.all(np.isfinite(b1))
    u1, u2 = ph.u01(a), ph.u01(b)
    r = np.sqrt(np.float32(-2.0) * np.log(u1).astype(np.float32)).astype(np.float32)
    t = (np.float32(ph.TWO_PI_F32) * u2 - np.float32(ph.PI_F32)).astype(np.float32)
    f0 = -r * np.cos(t.astype(np.float64)).astype(np.float32)
    f1 = -r * np.sin(t.astype(np.float64)).astype(np.float32)
    assert np.all(np.abs(f0 - n0) <= b0) and np.all(np.abs(f1 - n1) <= b1)
    r64 = np.sqrt(-2 * np.log(u1.astype(np.float64)))
    assert np.all(b0 <= 1e-5 * r64 + 1e-3) and np.all(b1 <= 1e-5 * r64 + 1e-3)
    assert n0[-1] == n1[-1] == n0[-3] == n1[-3] == 0.0 and n0[-5] > 5.88            # u1 = 1: r = 0; u1 = 2^-25: r = 5.89
    # moments of the centre: standard normals
    both = np.concatenate([n0[:-5], n1[:-5]])
    assert abs(both.mean()) < 0.03 and abs(both.std() - 1) < 0.03


def test_draws_layout_and_counters():
    """draws_f64: chain row m = frame * C + c, block b gives normals 4b..4b+3, the uniform is block 0's, iter0 + it wraps."""
    eps, bnd, u = ph.draws_f64(7, [5, -3], [0, 2 ** 20 - 1], 3, 6, 2, iter0=2 ** 32 - 1)
    assert eps.shape == (2, 6, 6) and u.shape == (2, 6) and u.dtype == np.float32
    m, it = 4, 1                                                                  # frame 1, chain 1; iteration 2^32 - 1 + 1 = 0
    fc = (2 ** 20 - 1) | (1 << 20)
    w0, w1 = ph.mh_words(7, -3, fc, 0, 0), ph.mh_words(7, -3, fc, 0, 1)
    assert u[it, m] == ph.u01_low_bytes(w0[0], w0[1], w0[2])
    assert eps[it, m, 2] == ph.box_muller_f64(w0[2], w0[3])[0] and eps[it, m, 3] == ph.box_muller_f64(w0[2], w0[3])[1]
    assert eps[it, m, 4] == ph.box_muller_f64(w1[0], w1[1])[0] and eps[it, m, 5] == ph.box_muller_f64(w1[0], w1[1])[1]
    assert bnd[it, m, 5] == ph.box_muller_f64(w1[0], w1[1])[3]
    w_first = ph.mh_words(7, 5, 0, 2 ** 32 - 1, 0)                                 # frame 0, chain 0, iteration 0: counter 2^32 - 1
    assert u[0, 0] == ph.u01_low_bytes(*w_first[:3])


def test_counter_guard():
    check_counters(2 ** 20, 4095)                                                 # frame indices < 2^20: distinct counters
    check_counters(2 ** 24, 1)                                                    # one chain: word 1 is the frame index
    with pytest.raises(ValueError, match="2\\^20"):
        check_counters(2 ** 20 + 1, 2)
