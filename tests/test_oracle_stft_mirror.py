"""The float64 STFT / ISTFT mirror (oracle/stft_mirror.py): its float64 core against three independent transforms, the
reference restatement's own float32 arithmetic inside its bounds, and bounds that are not vacuous."""
import numpy as np
import torch

from dvae_b200 import synth
from oracle import stft_mirror as sm
from oracle import stft_np

KW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
IKW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False)


def _speech(u, secs, snr=None):
    x, _, _ = synth.synth_utterance(u, secs, snr)
    return np.pad(x.astype(np.float32), (0, 256))                      # the end padding of stft.py:45-50


def _mirror(x, hop=256):
    N = 1 + (len(x) - 1024) // hop
    X, P, eb, fb, pb = sm.stft_f64(torch.from_numpy(x), [0], [len(x)], [0, N], hop)
    return N, X.numpy(), P.numpy(), eb.numpy(), fb.numpy(), pb.numpy()


def test_core_matches_independent_transforms():
    x = _speech(1, 1.0)
    N, X, P, _, _, _ = _mirror(x)
    ref = stft_np.stft(x[:-256], dtype="complex128", **KW).T
    T = torch.stft(torch.tensor(x, dtype=torch.float64), 1024, 256, window=torch.hann_window(1024, periodic=True, dtype=torch.float64),
                   center=False, return_complex=True).T.numpy()
    scale = np.abs(ref).max()
    assert X.shape == ref.shape == T.shape
    assert np.abs(X - ref).max() <= 1e-13 * scale and np.abs(X - T).max() <= 1e-13 * scale
    for i in (0, 17, N - 1):
        fr = x[i * 256:i * 256 + 1024].astype(np.float64) * stft_np.hann_periodic(1024)
        assert np.abs(X[i] - stft_np.dft_direct(fr)).max() <= 1e-11 * scale
    np.testing.assert_allclose(P, np.abs(X) ** 2, rtol=1e-14, atol=0)
    # the inverse: the mirror's float64 overlap-add against the restatement run on complex128 input, and the exact zeros
    y, b, wr = sm.istft_f64(torch.from_numpy(X.astype(np.complex64)), [0, N], [0], [len(x) + 100], len(x) + 100)
    ref_y = stft_np.istft(X.astype(np.complex64).T.astype(np.complex128), dtype="float64", max_len=len(x) + 100, **IKW)
    y, b = y.numpy(), b.numpy()
    assert bool(wr.all()) and np.all(np.abs(y - ref_y) <= 1e-6 * b)          # float64 rounding only, amplified at the edges
    assert y[0] == 0 and b[0] == 0 and np.all(y[len(x):] == 0) and np.all(b[len(x):] == 0)


def _ratio(err, bound):
    return float(np.max(np.where(err == 0, 0.0, err / np.where(bound > 0, bound, 1e-300))))


def test_restatement_and_float32_fft_stay_inside_the_bounds():
    """The reference's complex64 STFT and float32 overlap-add, and numpy's single-precision FFT (numpy 2.x computes
    ``rfft`` of float32 input in float32), inside the element, frame and sample bounds; on speech the float32 FFT reaches
    more than 1e-3 of the element bound, so the bounds are not vacuous."""
    worst = {}
    w32 = stft_np.hann_periodic(1024).astype(np.float32)
    for name, x in (("speech", _speech(2, 2.0, 5.0)), ("speech_hi_snr", _speech(3, 2.0, 20.0)),
                    ("noise", np.random.default_rng(0).uniform(-1, 1, 16384).astype(np.float32)),
                    ("tiny", (_speech(4, 1.0) * np.float32(1e-20)).astype(np.float32))):
        N, X, P, eb, fb, pb = _mirror(x)
        frames = np.lib.stride_tricks.sliding_window_view(x, 1024)[::256][:N]
        X32 = np.fft.rfft(frames * w32, axis=1)
        assert X32.dtype == np.complex64
        c64 = np.fft.rfft(frames.astype(np.float64) * stft_np.hann_periodic(1024), axis=1).astype(np.complex64)   # stft_np.stft
        for tag, got in (("f32 fft", X32), ("complex64", c64)):
            worst[(name, tag, "elem")] = _ratio(np.abs(got - X), eb)
            worst[(name, tag, "frame")] = _ratio(np.linalg.norm(got - X, axis=1), fb)
        P32 = (X32.real * X32.real + X32.imag * X32.imag).astype(np.float32)
        worst[(name, "f32 fft", "P")] = _ratio(np.abs(P32 - P), pb)
        # ISTFT: the restatement's float32 overlap-add of a Wiener-masked spectrum
        M = np.random.default_rng(1).uniform(0, 1, X.shape).astype(np.float32)
        Y = (M * c64).astype(np.complex64)
        y, b, _ = sm.istft_f64(torch.from_numpy(Y), [0, N], [0], [len(x)], len(x))
        yr = stft_np.istft(Y.T, max_len=len(x), **IKW)
        worst[(name, "restatement", "y")] = _ratio(np.abs(yr - y.numpy()), b.numpy())
    print("\nlargest |f32 - f64| / bound")
    for k, r in sorted(worst.items()):
        print("  %-14s %-12s %-6s %9.3g" % (k + (r,)))
    assert max(worst.values()) <= 1.0
    assert worst[("speech", "f32 fft", "elem")] > 1e-3 and worst[("speech", "f32 fft", "frame")] > 1e-3


def test_istft_bound_is_honest_at_the_edges():
    """Near sample 0 the division by the window sum-square amplifies the rounding: the bound there is many times the
    interior one, and the restatement's float32 result still lies inside it."""
    x = _speech(5, 1.0)
    N, X, _, _, _, _ = _mirror(x)
    y, b, _ = sm.istft_f64(torch.from_numpy(X.astype(np.complex64)), [0, N], [0], [len(x)], len(x))
    b = b.numpy()
    assert b[1] > 1e3 * np.median(b[2048:-2048])
    yr = stft_np.istft(X.astype(np.complex64).T, max_len=len(x), **IKW)
    assert np.all(np.abs(yr - y.numpy()) <= b)


def test_power_bound():
    rng = np.random.default_rng(2)
    X = (rng.standard_normal(4096) + 1j * rng.standard_normal(4096)).astype(np.complex64) * np.float32(1e-19)
    P, b = sm.power_f64(torch.from_numpy(X))
    P32 = (np.abs(X) ** 2).astype(np.float32)                         # np.abs of complex64, squared, as mcem.py:47
    assert np.all(np.abs(P32 - P.numpy()) <= b.numpy())
