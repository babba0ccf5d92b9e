"""``packages/metrics.py`` of the reference (packages/metrics.py:5-82) on the device.

Same names, arguments and return values as the reference for the per-utterance functions (numpy vectors in, Python floats /
numpy arrays out); the arithmetic runs in ``dvae_energy_ratios`` (six inner products in double, closed forms for the
energies) instead of forming ``s_target``, ``e_noise`` and ``e_art``.  ``energy_ratios_batch`` is the batched entry the
enhancement path uses: device tensors in the layout of ``Enhancer.run_device``, nothing leaves the GPU but 24 bytes per
utterance.  ``score_batch`` puts SI-SDR / SI-SIR / SI-SAR and STOI / ESTOI of a batch together (the scoring loop of the
reference's ``scripts/run_metrics.py``; ``score_reference`` + ``score_row`` are its two halves, for scoring several estimates
against one reference), ``pcm16`` quantises device signals as ``batch_io.write_wav`` does.  CUDA only: without
the library or a device the calls raise ``DvaeError``.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np
import torch

from .. import _lib
from ..engine import _p, _stream


def energy_ratios_batch(s_hat, s, n, off, lens):
    """SI-SDR, SI-SIR, SI-SAR of a ragged batch.

    ``s_hat``, ``s``, ``n``: 1-D float32 CUDA tensors (``n`` may be None); utterance ``u`` is ``[off[u], off[u]+lens[u])``.
    Returns a float64 CUDA tensor ``[B][3]`` (SI-SIR / SI-SAR are NaN without ``n``).
    """
    if not (s_hat.is_cuda and s.is_cuda and off.is_cuda and lens.is_cuda):
        raise _lib.DvaeError("energy_ratios_batch needs CUDA tensors")
    B = int(off.numel())
    out = torch.empty((B, 3), dtype=torch.float64, device=s_hat.device)
    with torch.cuda.device(s_hat.device):
        _lib.call("dvae_energy_ratios", _p(s_hat.contiguous()), _p(s.contiguous()), _p(n.contiguous()) if n is not None else None,
                  _p(off.to(torch.int64)), _p(lens.to(torch.int32)), B, _p(out), _stream())
    return out


def _one(s_hat, s, n, device):
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda" or not torch.cuda.is_available():
        raise _lib.DvaeError("dvae_b200 metrics run on a CUDA device only")
    T = len(s_hat)
    if len(s) != T or (n is not None and len(n) != T):
        raise ValueError("signals must have the same length")
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)      # noqa: E731
    off = torch.zeros(1, dtype=torch.int64, device=dev)
    lens = torch.full((1,), T, dtype=torch.int32, device=dev)
    return energy_ratios_batch(to(s_hat), to(s), None if n is None else to(n), off, lens)[0].cpu().numpy()


def energy_ratios(s_hat, s, n, device=None):
    """``(si_sdr, si_sir, si_sar)`` in dB (packages/metrics.py:39-60)."""
    r = _one(s_hat, s, n, device)
    return float(r[0]), float(r[1]), float(r[2])


def si_sdr_leroux(s_hat, s, device=None):
    """SI-SDR in dB (packages/metrics.py:62-82)."""
    return float(_one(s_hat, s, None, device)[0])


# ----------------------------------------------------------------------------------------------------------- STOI / ESTOI
_TAPS = {}          # (device, fs_sig) -> device copy of dvae_resample_taps(fs_sig)


def resample_taps(fs_sig):
    """Octave's anti-aliasing filter pystoi resamples ``fs_sig -> 10 kHz`` with (host numpy float32, unit sum)."""
    lib = _lib.load()
    n = lib.dvae_resample_taps(int(fs_sig), None, 0)
    _lib.check(min(n, 0), "dvae_resample_taps")
    taps = np.empty(n, np.float32)
    _lib.check(min(lib.dvae_resample_taps(int(fs_sig), taps.ctypes.data, n), 0), "dvae_resample_taps")
    return taps


def _device_taps(fs_sig, dev):
    key = (str(dev), int(fs_sig))
    t = _TAPS.get(key)
    if t is None:
        t = torch.from_numpy(resample_taps(fs_sig)).pin_memory().to(dev, non_blocking=True)
        _TAPS[key] = t
    return t


def _stoi_stage(x, y, off, lens, fs_sig):
    if not (x.is_cuda and y.is_cuda and off.is_cuda and lens.is_cuda):
        raise _lib.DvaeError("stoi_batch needs CUDA tensors")
    if x.dtype != torch.float32 or y.dtype != torch.float32 or x.shape != y.shape or x.dim() != 1:
        raise ValueError("x and y must be 1-D float32 tensors of the same length")
    B, total, dev = int(off.numel()), int(x.numel()), x.device
    lib = _lib.load()
    cap = lib.dvae_stoi_frame_capacity(B, total, int(fs_sig))
    wsb = lib.dvae_stoi_workspace_bytes(B, total, int(fs_sig))
    if cap < 0 or wsb < 0:
        raise ValueError("stoi_batch: bad sizes (B=%d, total=%d, fs_sig=%d)" % (B, total, fs_sig))
    st = dict(ws=torch.empty(wsb, dtype=torch.uint8, device=dev), env=torch.empty((cap, 2, 15), dtype=torch.float32, device=dev),
              keep=torch.empty(cap, dtype=torch.uint8, device=dev), frame_off=torch.empty(B, dtype=torch.int64, device=dev),
              counts=torch.empty((B, 2), dtype=torch.int32, device=dev))
    st["off"], st["lens"] = off.to(torch.int64).contiguous(), lens.to(torch.int32).contiguous()
    _lib.call("dvae_stoi_envelopes", _p(x.contiguous()), _p(y.contiguous()), _p(st["off"]), _p(st["lens"]), B, total, int(fs_sig),
              _p(_device_taps(fs_sig, dev)), _p(st["ws"]), _p(st["env"]), _p(st["keep"]), _p(st["frame_off"]), _p(st["counts"]),
              _stream())
    return st


def stoi_envelopes_batch(x, y, off, lens, fs_sig):
    """The front end of ``stoi_batch``: a dict of device tensors ``env [cap][2][15]`` (clean, processed third-octave
    envelopes of the STFT frames of the desilenced signals), ``keep [cap]`` (energy frame kept), ``frame_off [B]`` (first
    row of utterance u in both) and ``counts [B][2]`` (energy frames, STFT frames; -1 STFT frames where the score is NaN)."""
    with torch.cuda.device(x.device):
        return _stoi_stage(x, y, off, lens, fs_sig)


def stoi_batch(x, y, off, lens, fs_sig, out=None, frames_out=None):
    """STOI and ESTOI of a ragged batch: clean ``x`` and processed ``y`` (1-D float32 CUDA tensors in the layout of
    ``Enhancer.run_device``: utterance u is ``[off[u], off[u] + lens[u])``), sampled at ``fs_sig`` Hz.

    Returns a float64 CUDA tensor ``[B][2]`` = (STOI, ESTOI) (written into ``out`` when given); 1e-5 where fewer than 30
    STFT frames remain after silent-frame removal, NaN where the score is undefined (no complete 256-sample frame at 10 kHz,
    an all-zero or non-finite clean signal).  ``frames_out`` (int32 CUDA ``[B]``, optional) receives the STFT frame counts
    (-1 where NaN).  Enqueued on the current stream; nothing synchronises.
    """
    with torch.cuda.device(x.device):
        st = _stoi_stage(x, y, off, lens, fs_sig)
        B = int(off.numel())
        if out is None:
            out = torch.empty((B, 2), dtype=torch.float64, device=x.device)
        elif out.shape != (B, 2) or out.dtype != torch.float64 or not out.is_contiguous() or out.device != x.device:
            raise ValueError("out must be a contiguous float64 [B][2] tensor on the signals' device")
        _lib.call("dvae_stoi_scores", _p(st["env"]), _p(st["frame_off"]), _p(st["counts"]), B, _p(out), _stream())
        if frames_out is not None:
            frames_out.copy_(st["counts"][:, 1])
    return out


def stoi(x, y, fs_sig, extended=False, device=None):
    """pystoi's ``stoi(x, y, fs_sig, extended=False)`` on the device: clean ``x``, processed ``y`` (1-D arrays of the same
    length); returns STOI, or ESTOI when ``extended``, as a Python float.  Below 30 STFT frames after silent-frame removal:
    a ``RuntimeWarning`` and 1e-5, as pystoi.  ``ValueError`` when the lengths differ or the signal holds no complete frame."""
    import warnings
    if not torch.cuda.is_available() or (device is not None and torch.device(device).type != "cuda"):
        raise _lib.DvaeError("dvae_b200 metrics run on a CUDA device only")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    x = np.asarray(x)
    y = np.asarray(y)
    if x.shape != y.shape or x.ndim != 1:
        raise ValueError("x and y should be 1-D and have the same length, found %s and %s" % (x.shape, y.shape))
    if fs_sig <= 0 or (len(x) * 10000 + fs_sig - 1) // fs_sig <= 256:          # resampled length ceil(T 10000 / fs_sig)
        raise ValueError("the signal holds no complete 256-sample frame at 10 kHz")
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)      # noqa: E731
    frames = torch.empty(1, dtype=torch.int32, device=dev)
    r = stoi_batch(to(x), to(y), torch.zeros(1, dtype=torch.int64, device=dev),
                   torch.full((1,), len(x), dtype=torch.int32, device=dev), int(fs_sig), frames_out=frames)
    r, nfr = r[0].cpu().numpy(), int(frames.cpu()[0])
    if 0 <= nfr < 30:
        warnings.warn("Not enough STFT frames to compute intermediate intelligibility measure after removing silent "
                      "frames. Returning 1e-5. Please check you wav files", RuntimeWarning)
    return float(r[1 if extended else 0])


# --------------------------------------------------------------------------------------------- 16-bit PCM and batched scoring
SCORE_KEYS = ("si_sdr", "si_sir", "si_sar", "stoi", "estoi")


def pcm16(x, pcm=None, xq=None):
    """16-bit PCM quantisation of the float32 CUDA tensor ``x`` exactly as ``batch_io.write_wav`` does it
    (``clip(rint(x * 32768), -32768, 32767)``, round half to even; NaN maps to 0): writes the int16 samples into ``pcm`` and
    ``q / 32768`` (what ``read_wav`` returns for the written file) into ``xq``.  Either may be None, not both; given ones
    must be contiguous tensors of ``x``'s size.  Enqueued on the current stream."""
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("x must be a contiguous float32 CUDA tensor")
    for t, dt in ((pcm, torch.int16), (xq, torch.float32)):
        if t is not None and (t.dtype != dt or t.numel() != x.numel() or not t.is_contiguous() or t.device != x.device):
            raise ValueError("pcm / xq must be contiguous %s tensors of x's size on x's device" % dt)
    with torch.cuda.device(x.device):
        _lib.call("dvae_pcm16_f32", _p(x), x.numel(), _p(pcm), _p(xq), _stream())
    return pcm, xq


def score_batch(est, x, s, off, lens, fs, trim=None, out=None):
    """SI-SDR, SI-SIR, SI-SAR, STOI and ESTOI (``SCORE_KEYS``) of a ragged batch, for the estimate and for the mixture.

    ``est`` (speech estimate), ``x`` (noisy mixture), ``s`` (clean speech): 1-D float32 CUDA tensors in the layout of
    ``Enhancer.run_device`` (utterance u is ``[off[u], off[u] + lens[u])``), sampled at ``fs`` Hz.  Returns a float64 CUDA
    tensor ``[B][2][5]`` (written into ``out`` when given): row ``[u][0]`` scores ``est``, row ``[u][1]`` scores ``x``, so
    ``[u][0] - [u][1]`` is the improvement.  The noise reference of SI-SIR / SI-SAR is ``n = x - s`` (exact for additive
    mixtures).

    Every metric is computed on ``[off + trim, off + lens - trim)``: the reference's ``run_metrics.py`` drops 50 ms at both
    ends before scoring (default ``trim = round(0.05 fs)``, 800 samples at 16 kHz).  Whether it trims before ESTOI as well is
    not verified; here all five metrics see the same trimmed signal.  A row is NaN when ``lens <= 2 trim``; otherwise STOI's
    own rules apply (1e-5 below 30 frames, NaN where undefined).  Enqueued on the current stream; nothing synchronises.
    """
    if not est.is_cuda:
        raise _lib.DvaeError("score_batch needs CUDA tensors")
    if est.dtype != torch.float32 or est.dim() != 1 or est.shape != x.shape:
        raise ValueError("est, x and s must be 1-D float32 tensors of the same length")
    ref = score_reference(x, s, off, lens, fs, trim)
    B = int(off.numel())
    if out is None:
        out = torch.empty((B, 2, 5), dtype=torch.float64, device=x.device)
    elif out.shape != (B, 2, 5) or out.dtype != torch.float64 or not out.is_contiguous() or out.device != x.device:
        raise ValueError("out must be a contiguous float64 [B][2][5] tensor on the signals' device")
    for k, sig in enumerate((est, x)):
        score_row(sig, ref, out[:, k])
    return out


class ScoreReference(NamedTuple):
    """What every scored row of a batch shares (``score_reference``): clean speech ``s``, noise ``n = x - s``, the trimmed
    layout ``t_off`` / ``t_len``, the rows too short to score (``short``, bool ``[B]``) and the sample rate."""
    s: torch.Tensor
    n: torch.Tensor
    t_off: torch.Tensor
    t_len: torch.Tensor
    short: torch.Tensor
    fs: int


def score_reference(x, s, off, lens, fs, trim=None):
    """The clean side of ``score_batch`` for mixture ``x`` and clean speech ``s`` (arguments as there), computed once so that
    any number of estimates can be scored against it with ``score_row``.  Enqueued on the current stream."""
    if not all(t.is_cuda for t in (x, s, off, lens)):
        raise _lib.DvaeError("score_batch needs CUDA tensors")
    if not all(t.dtype == torch.float32 and t.dim() == 1 and t.shape == x.shape for t in (s, x)):
        raise ValueError("x and s must be 1-D float32 tensors of the same length")
    trim = int(round(0.05 * fs)) if trim is None else int(trim)
    if trim < 0 or fs <= 0:
        raise ValueError("fs must be positive and trim non-negative")
    with torch.cuda.device(x.device):
        s = s.contiguous()
        n = torch.sub(x.contiguous(), s)
        lens = lens.to(torch.int64)
        return ScoreReference(s, n, off.to(torch.int64) + trim, torch.clamp_min(lens - 2 * trim, 0).to(torch.int32),
                              lens <= 2 * trim, int(fs))


def score_row(est, ref, out):
    """One row of ``score_batch``: the five ``SCORE_KEYS`` of the 1-D float32 CUDA signal ``est`` against ``ref``
    (``score_reference``), written into the float64 ``[B][5]`` view ``out``; NaN where the utterance is too short for the
    trim.  Enqueued on the current stream; nothing synchronises."""
    if not est.is_cuda or est.dtype != torch.float32 or est.dim() != 1 or est.shape != ref.s.shape:
        raise ValueError("est must be a 1-D float32 CUDA tensor of the reference's length")
    with torch.cuda.device(est.device):
        est = est.contiguous()
        out[:, :3] = energy_ratios_batch(est, ref.s, ref.n, ref.t_off, ref.t_len)
        out[:, 3:] = stoi_batch(ref.s, est, ref.t_off, ref.t_len, ref.fs)
        out.masked_fill_(ref.short.view(-1, 1), float("nan"))
    return out


def si_sdr_components(s_hat, s, n):
    """``(s_target, e_noise, e_art)`` (packages/metrics.py:12-37); three axpy's on the host, kept for API completeness."""
    s_hat, s, n = (np.asarray(a) for a in (s_hat, s, n))
    s_target = (np.dot(s_hat, s) / np.dot(s, s)) * s
    e_noise = (np.dot(s_hat, n) / np.dot(n, n)) * n
    return s_target, e_noise, s_hat - s_target - e_noise


# ---------------------------------------------------------------------------------------------- statistics table (host)
def mean_confidence_interval(data, confidence=0.95, round=3):
    """Mean and half-width of the Student-t confidence interval, both rounded to 3 decimals (packages/metrics.py:5-10)."""
    import scipy.stats
    a = np.asarray(data, dtype=np.float64)
    half = scipy.stats.sem(a) * scipy.stats.t.ppf((1.0 + confidence) / 2.0, len(a) - 1)
    return np.round(np.mean(a), 3), np.round(half, 3)


def compute_stats(metrics_keys, all_metrics, model_data_dir, confidence, all_snr_db=None, all_noise_types=None, all_speakers=None,
                  all_noise_stationarities=None):
    """The evaluation table of the reference (packages/metrics.py:84-167): average and confidence interval of every metric
    over all utterances, then per input SNR / noise type / noise stationarity / speaker when those lists are given.  Prints
    the same tables (same headings and column format) and additionally RETURNS them:
    ``{"all": {key: {"avg", "+/-"}}, "snr": {value: {...}}, "noise_type": {...}, "noise_stationarity": {...}, "speaker": {...}}``.
    ``all_metrics`` is a list of per-utterance tuples in the order of ``metrics_keys`` (``scripts/run_metrics.py:117-129``)."""
    cols = {key: np.asarray([row[i] for row in all_metrics], dtype=np.float64) for i, key in enumerate(metrics_keys)}

    def table(select):
        print("{:<10} {:<10} {:<10}".format('METRIC', 'AVERAGE', 'CONF. INT.'))
        out = {}
        for key, col in cols.items():
            m, h = mean_confidence_interval(col[select], confidence=confidence)
            out[key] = {'avg': m, '+/-': h}
            print("{:<10} {:<10} {:<10}".format(key, m, h))
        print('\n')
        return out

    n = len(all_metrics)
    result = {"all": table(np.ones(n, dtype=bool))}
    groups = (("snr", all_snr_db, lambda v: 'Input SNR = {:.2f}'.format(v)),
              ("noise_type", all_noise_types, lambda v: 'Noise type = {}'.format(v)),
              ("noise_stationarity", all_noise_stationarities, lambda v: 'Noise type = {}'.format(v)),      # heading as in the reference
              ("speaker", all_speakers, lambda v: 'Speaker = {}'.format(v)))
    for name, labels, heading in groups:
        if labels is None:
            continue
        labels = np.asarray(labels)
        result[name] = {}
        for v in (np.unique(labels) if name == "snr" else sorted(set(labels.tolist()))):
            print(heading(v))
            result[name][v] = table(labels == v)
    return result
