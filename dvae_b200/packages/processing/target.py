"""``packages/processing/target.py`` (lines 5-105) on the device: time-domain VAD and ideal binary masks.

Same names, arguments and return values as the reference for the per-utterance functions; only the configuration the
evaluation scripts use is implemented (``center=False``; other values raise ``NotImplementedError``).  The ``*_batch``
functions are the ones the enhancement path uses: frame-major ragged device tensors in, labels out, nothing touches the
host.  CUDA only.
"""
from __future__ import annotations

import numpy as np
import torch

from ... import _lib
from ...engine import RaggedBatch, _ld_for, _p, _stream
from ...synth import num_frames


def _buffer(t, shape, dtype, device, what):
    if t is None:
        return torch.empty(shape, dtype=dtype, device=device)
    if t.dtype != dtype or not t.is_contiguous() or t.numel() < int(np.prod(shape)):
        raise ValueError("%s must be a contiguous %s tensor of at least %d elements" % (what, dtype, int(np.prod(shape))))
    return t


def vad_batch(x_flat, x_off, x_len, batch: RaggedBatch, n_fft=1024, hop=256, vad_threshold=1.70, out=None, ws=None):
    """``[NT]`` float32 labels for a concatenated float32 device signal (frames of ``RaggedBatch``).  ``out`` (float32,
    ``NT`` elements) and ``ws`` (float64, ``max(1, NT)`` elements): caller-owned buffers, allocated when not given."""
    vad = _buffer(out, (batch.NT,), torch.float32, x_flat.device, "out")[:batch.NT]
    ws = _buffer(ws, (max(1, batch.NT),), torch.float64, x_flat.device, "ws")
    with torch.cuda.device(x_flat.device):
        _lib.call("dvae_vad_labels", _p(x_flat), _p(x_off), _p(x_len), batch.B, _p(batch.frame_utt), _p(batch.fr_off), batch.NT,
                  n_fft, hop, float(vad_threshold), _p(vad), _p(ws), _stream())
    return vad


def ibm_batch(S, batch: RaggedBatch, F, eps=1e-8, ibm_threshold=50, vad=None, out=None, ws=None):
    """``[NT][ld]`` float32 mask of a frame-major complex64 spectrogram ``S [NT][ld]`` (optionally gated by ``vad [NT]``).
    ``out`` (float32 ``[NT][ld]``) and ``ws`` (int32, ``max(1, B)`` elements): caller-owned buffers, allocated when not
    given.  With ``ld = F`` the mask is the dense ``[NT][F]`` label matrix the M2 models read."""
    ld = S.shape[1]
    mask = _buffer(out, (batch.NT, ld), torch.float32, S.device, "out").view(-1)[:batch.NT * ld].view(batch.NT, ld)
    ws = _buffer(ws, (max(1, batch.B),), torch.int32, S.device, "ws")
    with torch.cuda.device(S.device):
        _lib.call("dvae_ibm_labels", _p(S), _p(batch.frame_utt), _p(batch.fr_off), batch.B, batch.NT, F, ld, float(eps),
                  float(ibm_threshold), _p(vad), _p(mask), _p(ws), _stream())
    return mask


def _check(fs, wlen_sec, center):
    if center:
        raise NotImplementedError("dvae_b200 implements center=False (the evaluation scripts' setting)")
    n_fft = wlen_sec * fs
    if n_fft != int(n_fft):
        raise ValueError("wlen_sample of STFT is not an integer.")
    return int(n_fft)


def _device(device):
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda" or not torch.cuda.is_available():
        raise _lib.DvaeError("dvae_b200 label front end runs on a CUDA device only")
    return dev


def clean_speech_VAD(speech_t, fs=16e3, wlen_sec=50e-3, hop_percent=0.25, center=True, pad_mode='reflect', pad_at_end=True,
                     vad_threshold=1.70, device=None):
    """``(1, N)`` float32 labels (target.py:5-56)."""
    n_fft = _check(fs, wlen_sec, center)
    if not pad_at_end:
        raise NotImplementedError("dvae_b200 implements pad_at_end=True")
    hop = int(hop_percent * n_fft)
    dev = _device(device)
    x = torch.from_numpy(np.ascontiguousarray(speech_t, dtype=np.float32)).to(dev)
    N = num_frames(len(speech_t), n_fft, hop, int(fs))
    batch = RaggedBatch([N], dev)
    off = torch.zeros(1, dtype=torch.int64, device=dev)
    lens = torch.full((1,), len(speech_t), dtype=torch.int32, device=dev)
    return vad_batch(x, off, lens, batch, n_fft, hop, vad_threshold).cpu().numpy()[None]


def clean_speech_IBM(speech_tf, eps=1e-8, ibm_threshold=50, device=None):
    """``(F, N)`` float32 mask of a ``(F, N)`` complex spectrogram (target.py:58-70)."""
    dev = _device(device)
    F, N = speech_tf.shape
    ld = _ld_for(F)
    S = torch.zeros((N, ld), dtype=torch.complex64, device=dev)
    S[:, :F] = torch.from_numpy(np.ascontiguousarray(np.asarray(speech_tf, np.complex64).T)).to(dev)
    return np.ascontiguousarray(ibm_batch(S, RaggedBatch([N], dev), F, eps, ibm_threshold)[:, :F].t().cpu().numpy())


def noise_robust_clean_speech_IBM(speech_t, speech_tf, fs=16e3, wlen_sec=50e-3, hop_percent=0.25, center=True, pad_mode='reflect',
                                  pad_at_end=True, vad_threshold=1.70, eps=1e-8, ibm_threshold=50, device=None):
    """IBM gated by the time-domain VAD (target.py:72-105)."""
    vad = clean_speech_VAD(speech_t, fs, wlen_sec, hop_percent, center, pad_mode, pad_at_end, vad_threshold, device)
    return clean_speech_IBM(speech_tf, eps, ibm_threshold, device) * vad
