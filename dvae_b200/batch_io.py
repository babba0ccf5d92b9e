"""Batched file front / back end of the enhancement path (SURVEY §8(f) N4).

The reference's ``process_utt`` (scripts/evaluate_ntcd_M1.py:81-188) reads one noisy wav, enhances it and writes
``*_s_est.wav`` / ``*_n_est.wav`` before touching the next file; ``process_sublist`` (190-214) loops over a file list in
one process per half GPU.  Here a sublist is cut into ragged batches for ``Enhancer.enhance``: wav decoding and encoding
run on a few host threads while the GPU works on the previous batch.

wav I/O is self-contained (RIFF PCM 8/16/24/32-bit and IEEE float 32/64, mono or first channel): ``soundfile`` and
``h5py``, which the reference uses, are not required.  ``sf.read`` semantics are kept: float64 samples in [-1, 1);
``write_wav`` writes 16-bit PCM like ``sf.write``'s default for ``.wav``.
"""
from __future__ import annotations

import os
import struct
from concurrent.futures import ThreadPoolExecutor

import numpy as np


def read_wav(path, channel=0):
    """``(samples float64 in [-1, 1), fs)`` of a RIFF/WAVE file (``sf.read`` for the formats listed in the module doc)."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:4] != b"RIFF" or data[8:12] != b"WAVE":
        raise ValueError("%s is not a RIFF/WAVE file" % path)
    pos, fmt, raw = 12, None, None
    while pos + 8 <= len(data):
        tag, size = data[pos:pos + 4], struct.unpack("<I", data[pos + 4:pos + 8])[0]
        body = data[pos + 8:pos + 8 + size]
        if tag == b"fmt ":
            code, nch, fs, _, _, bits = struct.unpack("<HHIIHH", body[:16])
            if code == 0xFFFE and size >= 26:                     # WAVE_FORMAT_EXTENSIBLE: the sub-format's first two bytes
                code = struct.unpack("<H", body[24:26])[0]
            fmt = (code, nch, fs, bits)
        elif tag == b"data":
            raw = body
        pos += 8 + size + (size & 1)
    if fmt is None or raw is None:
        raise ValueError("%s: missing fmt or data chunk" % path)
    code, nch, fs, bits = fmt
    if code == 1:                                                  # integer PCM
        if bits == 8:
            x = (np.frombuffer(raw, np.uint8).astype(np.float64) - 128.0) / 128.0
        elif bits == 16:
            x = np.frombuffer(raw, "<i2").astype(np.float64) / 32768.0
        elif bits == 24:
            b = np.frombuffer(raw[:len(raw) // 3 * 3], np.uint8).reshape(-1, 3).astype(np.int32)
            v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
            x = np.where(v >= 1 << 23, v - (1 << 24), v).astype(np.float64) / float(1 << 23)
        elif bits == 32:
            x = np.frombuffer(raw, "<i4").astype(np.float64) / 2147483648.0
        else:
            raise ValueError("%s: unsupported PCM width %d" % (path, bits))
    elif code == 3:                                                # IEEE float
        x = np.frombuffer(raw, "<f4" if bits == 32 else "<f8").astype(np.float64)
    else:
        raise ValueError("%s: unsupported wav format tag %d" % (path, code))
    if nch > 1:
        x = x[:len(x) // nch * nch].reshape(-1, nch)[:, channel]
    return np.ascontiguousarray(x), int(fs)


def write_wav(path, x, fs):
    """16-bit PCM mono wav (``sf.write(path, x, fs)`` for float input: scale by 2^15, round, clip).  An int16 array holds
    the PCM samples already (``Enhancer.enhance(..., pcm16=True)``) and is written as it is."""
    x = np.asarray(x)
    if x.dtype == np.int16:
        pcm = x.astype("<i2").tobytes()
    else:
        pcm = np.clip(np.rint(np.asarray(x, np.float64) * 32768.0), -32768, 32767).astype("<i2").tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(pcm)) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 1, 1, int(fs), int(fs) * 2, 2, 16) \
        + b"data" + struct.pack("<I", len(pcm))
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "wb") as f:
        f.write(hdr + pcm)


def output_stem(output_data_dir, proc_noisy_file_path):
    """``output_data_dir + proc_noisy_file_path`` without extension (scripts/evaluate_ntcd_M1.py:85-86, 172-173)."""
    return os.path.splitext(output_data_dir + proc_noisy_file_path)[0]


def utterance_id(path: str) -> int:
    """A stable 31-bit id of an utterance (CRC-32 of its path): word 0 of the Philox counters, so an utterance's random draws do
    not depend on the batch it lands in, its position in the batch or the rank that processes it."""
    import zlib
    return zlib.crc32(path.encode("utf-8")) & 0x7FFFFFFF


def _check_sublist(sublist, batch_size, fs, trim):
    if int(batch_size) < 1:
        raise ValueError("batch_size must be at least 1")
    if fs <= 0 or (trim is not None and int(trim) < 0):
        raise ValueError("fs must be positive and trim non-negative")
    if any(len(ab) != 2 for ab in sublist):
        raise ValueError("sublist must hold (proc_noisy_file_path, clean_file_path) pairs")


def _require_files(paths):
    for p in paths:
        if not os.path.isfile(p):
            raise FileNotFoundError("%s: no such file" % p)


def _read_checked(path, fs, length=None):
    x, f = read_wav(path)
    if f != fs:
        raise ValueError("%s: sampling rate %d, expected %d" % (path, f, fs))
    if length is not None and len(x) != length:
        raise ValueError("%s: %d samples, expected %d" % (path, len(x), length))
    return np.asarray(x, np.float32)


def process_sublist(sublist, enhancer, processed_wav_dir, output_data_dir, batch_size=512, max_frames=None, labels=None,
                    io_threads=8, fs=16000, utt_ids=None, score=False, score_at=(), oracle_labels=None):
    """Batched replacement of ``process_sublist`` / ``process_utt`` (scripts/evaluate_ntcd_M1.py:81-214).

    ``sublist``: ``(proc_noisy_file_path, clean_file_path)`` pairs as the reference builds them.  Files whose
    ``*_s_est.wav`` exists are skipped, like the reference.  ``max_frames(noisy_path, clean_path) -> int | None`` supplies the
    video-length frame cap the reference reads from HDF5; ``labels(noisy_path, clean_path) -> (y_dim, N) array`` supplies the
    labels of the M2 models.  ``utt_ids(noisy_path) -> int`` names the utterances for the random number generator
    (default: ``utterance_id``, a hash of the path), so every utterance gets its own draws whatever ``batch_size`` and
    sharding are - the reference draws fresh numbers per utterance too.  File I/O overlaps the GPU work: the next batch is read and
    the previous one written by ``io_threads`` workers while the current one is enhanced.  Returns the list of written stems.

    ``score=True`` also reads the clean file ``processed_wav_dir + clean_file_path`` of every pair, scores each estimate on
    the device while its batch is enhanced (``Enhancer.enhance(..., ref_list=..., pcm16=True)``: the score of exactly the
    16-bit samples written) and returns ``(written_stems, scores [n][2][5])`` (``metrics.SCORE_KEYS``; row 0 the estimate,
    row 1 the noisy input).  The files are the same bytes as without ``score``; ``score_sublist`` on them gives the same
    numbers.

    ``score_at`` (with ``score=True``): EM iteration counts as ``Enhancer.enhance(..., score_at=...)`` takes them; the call
    then returns ``(written_stems, scores, trace [n][len(score_at)][5])``, where ``trace[u][k]`` is the estimate's score row
    that a run with ``niter = score_at[k]`` would give, all from this one run.  The files do not change.

    ``oracle_labels``: ``"vad"``, ``"ibm"`` or ``"robust_ibm"``, the M2 models' labels derived from the clean speech on the
    device (``Enhancer.enhance(..., s_list=..., oracle_labels=...)``) instead of a ``labels`` callback.  The clean file of every
    pair is read by the same read-ahead workers; with ``score=True`` that one read (and one upload) serves both the labels
    and the scores.  Frame caps from ``max_frames`` cut the labels after they are computed on the whole clean signal.
    """
    score_at = tuple(score_at)
    if score_at and not score:
        raise ValueError("score_at needs score=True")
    if oracle_labels is not None:
        from .engine import ORACLE_LABELS
        if oracle_labels not in ORACLE_LABELS:
            raise ValueError("oracle_labels must be one of %s or None, got %r" % (ORACLE_LABELS, oracle_labels))
        if labels is not None:
            raise ValueError("oracle_labels and the labels callback are two sources of the same labels: pass one")
    clean = score or oracle_labels is not None               # the clean file of every pair is read
    if clean:
        _check_sublist(sublist, batch_size, fs, None)
    if score_at:
        from .engine import check_checkpoints
        score_at = check_checkpoints(score_at, enhancer.cfg.niter)
    utt_ids = utt_ids or utterance_id
    todo = [(a, b) for a, b in sublist if not os.path.exists(output_stem(output_data_dir, a) + "_s_est.wav")]
    if clean:
        _require_files([processed_wav_dir + p for ab in todo for p in ab])
    written, scores, traces = [], [], []
    with ThreadPoolExecutor(max(1, io_threads)) as pool:
        pending = None                                               # futures of the previous batch's wav writes

        def submit_reads(part):
            return [(pool.submit(_read_checked, processed_wav_dir + ab[0], fs),
                     pool.submit(_read_checked, processed_wav_dir + ab[1], fs) if clean else None) for ab in part]

        reads = submit_reads(todo[:batch_size])
        for lo in range(0, len(todo), batch_size):
            part = todo[lo:lo + batch_size]
            xs = [f.result() for f, _ in reads]
            cs = [g.result() for _, g in reads] if clean else None
            reads = submit_reads(todo[lo + batch_size:lo + 2 * batch_size])      # read ahead: the next batch loads while this one runs
            if clean:
                for x, c, ab in zip(xs, cs, part):
                    if len(c) != len(x):
                        raise ValueError("%s: %d samples, the noisy file has %d" % (processed_wav_dir + ab[1], len(c), len(x)))
            caps = [max_frames(*ab) for ab in part] if max_frames else None
            if caps is not None and any(c is None for c in caps):
                big = np.iinfo(np.int64).max
                caps = [big if c is None else c for c in caps]
            ys = [labels(*ab) for ab in part] if labels else None
            ids = [utt_ids(ab[0]) for ab in part]
            # the same list object for the labels and the scores: the enhancer then uploads the clean signals once
            lab = {} if oracle_labels is None else dict(s_list=cs, oracle_labels=oracle_labels)
            if score:
                s_hat, n_hat, _, sc, *tr = enhancer.enhance(xs, y_list=ys, max_frames_list=caps, utt_ids=ids, ref_list=cs, pcm16=True,
                                                            score_at=score_at, **lab)
                scores.append(sc)
                traces += tr
            else:
                s_hat, n_hat, _ = enhancer.enhance(xs, y_list=ys, max_frames_list=caps, utt_ids=ids, **lab)
            if pending:
                for fut in pending:
                    fut.result()
            pending = []
            for ab, s, n in zip(part, s_hat, n_hat):
                stem = output_stem(output_data_dir, ab[0])
                # the result arrays lease the enhancer's pinned buffers (Enhancer._pin_out): the writers hold them until done
                pending.append(pool.submit(write_wav, stem + "_s_est.wav", s, fs))
                pending.append(pool.submit(write_wav, stem + "_n_est.wav", n, fs))
                written.append(stem)
        if pending:
            for fut in pending:
                fut.result()
    if not score:
        return written
    scores = np.concatenate(scores) if scores else np.zeros((0, 2, 5))
    if not score_at:
        return written, scores
    return written, scores, (np.concatenate(traces) if traces else np.zeros((0, len(score_at), 5)))


def score_sublist(sublist, processed_wav_dir, output_data_dir, device=0, batch_size=512, io_threads=8, fs=16000, trim=None):
    """Batched replacement of the scoring loop of the reference's ``scripts/run_metrics.py``: SI-SDR, SI-SIR, SI-SAR, STOI and
    ESTOI (``metrics.SCORE_KEYS``) of every pair's ``*_s_est.wav`` on the GPU, in ragged batches of ``batch_size``.

    For each ``(proc_noisy_file_path, clean_file_path)`` pair it reads the estimate ``output_stem(output_data_dir, noisy) +
    "_s_est.wav"``, the noisy file ``processed_wav_dir + noisy`` and the clean file ``processed_wav_dir + clean``; the next
    batch is read by ``io_threads`` workers while the current one is scored (``metrics.score_batch``, trim as there).
    Returns ``(stems, scores [n][2][5])`` float64, row 0 the estimate and row 1 the noisy input; the rows feed
    ``metrics.compute_stats``.  A missing file raises ``FileNotFoundError`` before any device work.
    """
    _check_sublist(sublist, batch_size, fs, trim)
    stems = [output_stem(output_data_dir, a) for a, _ in sublist]
    triples = [(st + "_s_est.wav", processed_wav_dir + a, processed_wav_dir + b) for st, (a, b) in zip(stems, sublist)]
    _require_files([p for t in triples for p in t])
    import torch
    from .engine import _require_cuda
    from .packages import metrics
    dev = _require_cuda(device)
    out = []

    def read_triple(t):
        x = _read_checked(t[1], fs)
        return _read_checked(t[0], fs, len(x)), x, _read_checked(t[2], fs, len(x))

    with ThreadPoolExecutor(max(1, io_threads)) as pool, torch.cuda.device(dev):
        reads = [pool.submit(read_triple, t) for t in triples[:batch_size]]
        for lo in range(0, len(triples), batch_size):
            sigs = [f.result() for f in reads]
            reads = [pool.submit(read_triple, t) for t in triples[lo + batch_size:lo + 2 * batch_size]]
            lens = np.array([len(x) for _, x, _ in sigs], np.int32)
            off = np.zeros(len(sigs) + 1, np.int64)
            np.cumsum((lens.astype(np.int64) + 1) // 2 * 2, out=off[1:])            # even offsets, as Enhancer.enhance
            flat = np.zeros((3, int(off[-1])), np.float32)
            for u, trip in enumerate(sigs):
                for k in range(3):
                    flat[k, off[u]:off[u] + lens[u]] = trip[k]
            est, x, s = (torch.from_numpy(flat[k]).to(dev) for k in range(3))
            out.append(metrics.score_batch(est, x, s, torch.from_numpy(off[:-1].copy()).to(dev), torch.from_numpy(lens).to(dev), fs,
                                           trim=trim).cpu().numpy())
    return stems, (np.concatenate(out) if out else np.zeros((0, 2, 5)))
