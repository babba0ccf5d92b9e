"""CPU-side checks of the scoring path: int16 wav writing, argument errors of the batched scorers before any device work."""
import ctypes
import re

import numpy as np
import pytest

from dvae_b200 import _lib, batch_io


def _numpy_pcm16(x):
    return np.clip(np.rint(np.asarray(x, np.float64) * 32768.0), -32768, 32767).astype(np.int16)


def test_write_wav_int16_is_byte_identical_to_the_float_path(tmp_path):
    rng = np.random.default_rng(3)
    k = np.arange(-40, 40, dtype=np.float64)
    x = np.concatenate([rng.standard_normal(5001) * 0.3, [1.0, -1.0, 1.5, -1.5, 0.0, -0.0, 32767.5 / 32768, -32768.5 / 32768],
                        (k + 0.5) / 32768, [np.inf, -np.inf]]).astype(np.float32)
    a, b = str(tmp_path / "f.wav"), str(tmp_path / "i.wav")
    batch_io.write_wav(a, x, 16000)
    batch_io.write_wav(b, _numpy_pcm16(x), 16000)
    assert open(a, "rb").read() == open(b, "rb").read()
    y, fs = batch_io.read_wav(b)
    assert fs == 16000 and np.array_equal(y * 32768.0, _numpy_pcm16(x))


def test_pcm16_argument_errors_before_any_launch():
    lib = _lib.load()
    buf = (ctypes.c_float * 8)()
    p = lambda a: ctypes.cast(a, ctypes.c_void_p)      # noqa: E731
    assert lib.dvae_pcm16_f32(p(buf), 8, None, None, None) < 0 and b"dvae_pcm16_f32" in lib.dvae_last_error()
    assert lib.dvae_pcm16_f32(None, 8, p(buf), None, None) < 0
    assert lib.dvae_pcm16_f32(p(buf), -1, p(buf), None, None) < 0
    assert lib.dvae_pcm16_f32(p(buf), 0, p(buf), p(buf), None) == 0          # nothing to do, nothing launched


def _pairs(tmp_path, n=3):
    wav_dir = str(tmp_path / "in")
    sub = []
    for i in range(n):
        rel = "/spk/utt%d.wav" % i
        batch_io.write_wav(wav_dir + rel, np.zeros(4000, np.float32), 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, np.zeros(4000, np.float32), 16000)
        sub.append((rel, "/clean" + rel))
    return wav_dir, sub


def test_score_sublist_argument_errors_before_device_work(tmp_path):
    wav_dir, sub = _pairs(tmp_path)
    out_dir = str(tmp_path / "out")
    for rel, _ in sub[:2]:
        batch_io.write_wav(batch_io.output_stem(out_dir, rel) + "_s_est.wav", np.zeros(4000, np.float32), 16000)
    missing = batch_io.output_stem(out_dir, sub[2][0]) + "_s_est.wav"
    with pytest.raises(FileNotFoundError, match=re.escape(missing)):
        batch_io.score_sublist(sub, wav_dir, out_dir, device="cpu")
    with pytest.raises(ValueError):
        batch_io.score_sublist(sub[:2], wav_dir, out_dir, batch_size=0)
    with pytest.raises(ValueError):
        batch_io.score_sublist(sub[:2], wav_dir, out_dir, trim=-1)
    with pytest.raises(ValueError):
        batch_io.score_sublist([(sub[0][0],)], wav_dir, out_dir)


def test_process_sublist_score_argument_errors_before_device_work(tmp_path):
    wav_dir, sub = _pairs(tmp_path)
    import os
    os.remove(wav_dir + sub[1][1])

    class Stub:
        calls = 0

        def enhance(self, *a, **kw):
            Stub.calls += 1
            raise AssertionError("no enhancement expected")

    with pytest.raises(FileNotFoundError, match=re.escape(wav_dir + sub[1][1])):
        batch_io.process_sublist(sub, Stub(), wav_dir, str(tmp_path / "out"), score=True)
    with pytest.raises(ValueError):
        batch_io.process_sublist(sub, Stub(), wav_dir, str(tmp_path / "out"), batch_size=0, score=True)
    assert Stub.calls == 0
