"""STFT / ISTFT restatement: cross-checks against torch.stft, a direct DFT and scipy.signal (librosa itself is not installable and
the reference holds no vector at this boundary, see oracle/__init__.py)."""
import numpy as np
import pytest
import torch

from dvae_b200 import synth
from oracle import stft_np

KW = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)


def test_shape_and_padding_rule():
    x, _, _ = synth.synth_utterance(0)
    X = stft_np.stft(x, **KW)
    assert X.dtype == np.complex64 and X.shape == (513, 185)          # 3 s -> padded by one hop (SURVEY §8)
    assert synth.num_frames(48000) == 185
    x2 = np.zeros(16384 * 2, np.float32)                               # 2.048 s: 32 windows * 4 hops, integer -> no pad
    assert stft_np.stft(x2, **KW).shape == (513, 1 + (len(x2) - 1024) // 256)
    assert synth.padded_length(len(x2)) == len(x2)


def test_matches_torch_stft_float64():
    x, _, _ = synth.synth_utterance(1)
    X = stft_np.stft(x, **KW)
    xp = np.pad(x.astype(np.float64), (0, 256))
    T = torch.stft(torch.tensor(xp), 1024, 256, window=torch.hann_window(1024, periodic=True, dtype=torch.float64),
                   center=False, return_complex=True).numpy().astype(np.complex64)
    assert np.max(np.abs(T - X)) <= 1e-6 * np.max(np.abs(X))


def test_matches_direct_dft():
    x, _, _ = synth.synth_utterance(2)
    X = stft_np.stft(x, **KW)
    for i in (0, 77, 184):
        fr = np.pad(x.astype(np.float64), (0, 256))[i * 256:i * 256 + 1024] * stft_np.hann_periodic(1024)
        np.testing.assert_allclose(X[:, i], stft_np.dft_direct(fr), rtol=0, atol=1e-5 * np.abs(X[:, i]).max())


def _scipy_pair(xp):
    """scipy.signal's STFT / ISTFT with the reference's framing (no boundary extension, no padding, periodic Hann, hop 256):
    an implementation that shares no code with the restatement (scipy 1.x ShortTimeFFT machinery)."""
    import scipy.signal
    w = scipy.signal.get_window("hann", 1024)
    _, _, Z = scipy.signal.stft(xp, fs=16000, window="hann", nperseg=1024, noverlap=768, nfft=1024, boundary=None, padded=False,
                                return_onesided=True, scaling="spectrum")
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                                # NOLA warning: the first hop has no full window coverage
        _, y = scipy.signal.istft(Z, fs=16000, window="hann", nperseg=1024, noverlap=768, nfft=1024, boundary=False, scaling="spectrum")
    return Z * w.sum(), y


def test_stft_and_istft_match_scipy_signal():
    """Pins both halves of the restatement against an independent implementation: the STFT bit for bit after the cast to
    complex64, the ISTFT to float32 rounding wherever the two share semantics (away from the first / last window, where
    librosa divides by the window sum above float32 tiny and scipy above 1e-10)."""
    x, _, _ = synth.synth_utterance(3)
    xp = np.pad(x.astype(np.float64), (0, 256))
    Z, y = _scipy_pair(xp)
    X = stft_np.stft(x, **KW)
    assert Z.shape == X.shape and np.array_equal(Z.astype(np.complex64), X)
    yo = stft_np.istft(X, fs=16000, wlen_sec=64e-3, hop_percent=0.25, center=False, max_len=len(xp))
    n = min(len(y), len(yo))
    assert np.max(np.abs(y[1024:n - 1024] - yo[1024:n - 1024])) <= 3e-7
    # and on a spectrogram that is NOT the STFT of a signal (a Wiener-masked one): the inverse is a genuine least-squares
    # overlap-add, not just "undo the forward transform"
    rng = np.random.default_rng(0)
    M = rng.uniform(0.0, 1.0, size=X.shape).astype(np.float32)
    import scipy.signal
    import warnings
    w = scipy.signal.get_window("hann", 1024)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _, ym = scipy.signal.istft((M * X).astype(np.complex128) / w.sum(), fs=16000, window="hann", nperseg=1024, noverlap=768, nfft=1024,
                                   boundary=False, scaling="spectrum")
    yom = stft_np.istft((M * X).astype(np.complex64), fs=16000, wlen_sec=64e-3, hop_percent=0.25, center=False, max_len=len(xp))
    assert np.max(np.abs(ym[1024:n - 1024] - yom[1024:n - 1024])) <= 3e-7


def test_round_trip_interior():
    x, _, _ = synth.synth_utterance(3)
    X = stft_np.stft(x, **KW)
    y = stft_np.istft(X, fs=16000, wlen_sec=64e-3, hop_percent=0.25, center=False, max_len=len(x))
    assert y.dtype == np.float32 and y.shape == x.shape
    assert np.max(np.abs(y[800:-800] - x[800:-800])) < 1e-5
    assert y[0] == 0.0                                                  # sum of squared windows is 0 at sample 0


def test_istft_zero_pads_to_max_len():
    x, _, _ = synth.synth_utterance(4)
    X = stft_np.stft(x, **KW)[:, :100]                                 # frames truncated (video shorter than audio)
    y = stft_np.istft(X, fs=16000, wlen_sec=64e-3, hop_percent=0.25, center=False, max_len=len(x))
    assert len(y) == len(x) and np.all(y[1024 + 256 * 99:] == 0)


def test_errors():
    with pytest.raises(ValueError):
        stft_np.stft(np.zeros(4000), fs=16000, wlen_sec=50.01e-3)
    with pytest.raises(ValueError):
        stft_np.istft(np.zeros((513, 4), np.complex64), fs=16000, wlen_sec=50.01e-3)


def test_16bit_wav_vs_torch(tmp_path):
    """A 16-bit PCM wav as the evaluation reads it (integer samples / 2^15), of a length that is not a whole number of hops:
    the end-padding rule and the forward transform against torch.stft."""
    from scipy.io import wavfile
    from dvae_b200 import batch_io
    x0, _, _ = synth.synth_utterance(6, 2.9)
    batch_io.write_wav(str(tmp_path / "x.wav"), x0[:46397], 16000)
    fs, w = wavfile.read(str(tmp_path / "x.wav"))
    assert fs == 16000 and w.dtype == np.int16 and len(w) % 256 != 0
    x = w.astype(np.float64) / 32768.0
    X = stft_np.stft(x, **KW)
    xp = stft_np.end_pad(x, 16000, 64e-3, 0.25, 256)
    T = torch.stft(torch.tensor(xp), 1024, 256, window=torch.hann_window(1024, periodic=True, dtype=torch.float64),
                   center=False, return_complex=True).numpy().astype(np.complex64)
    assert X.shape == T.shape and np.max(np.abs(T - X)) <= 1e-6 * np.max(np.abs(X))


def test_label_port_matches_reference_golden():
    """packages/processing/target.py:5-105 on the seeded utterance of tests/golden/labels.npz (oracle/make_golden.py)."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "labels.npz"))
    S = stft_np.stft(g["s"], fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
    vad = stft_np.clean_speech_vad(g["s"])
    ibm = stft_np.clean_speech_ibm(S)
    assert np.array_equal(vad, g["vad"]) and np.array_equal(ibm, g["ibm"].astype(np.float32))
    assert np.array_equal(ibm * vad, g["nr"].astype(np.float32))
