"""CPU-side checks of the quality trace over EM iterations: checkpoint validation, and argument errors of
process_sublist(score_at=...) before any file or device work."""
import numpy as np
import pytest

from dvae_b200 import batch_io
from dvae_b200.engine import McemConfig, check_checkpoints


def test_check_checkpoints_accepts_sorted_unique_counts_in_range():
    assert check_checkpoints((), 6) == ()
    assert check_checkpoints([2, 4, 6], 6) == (2, 4, 6)
    assert check_checkpoints(np.array([1, 5]), 6) == (1, 5)
    assert all(type(n) is int for n in check_checkpoints(np.arange(1, 4), 3))
    assert check_checkpoints(range(1, 101), 100) == tuple(range(1, 101))


@pytest.mark.parametrize("bad", [(4, 2), (2, 2, 4), (0, 2), (-1,), (2, 7), (7,), (2.0, 4.0), (True,), ("2",)])
def test_check_checkpoints_rejects_unsorted_duplicate_and_out_of_range(bad):
    with pytest.raises(ValueError):
        check_checkpoints(bad, 6)


def _pairs(tmp_path, n=3):
    wav_dir = str(tmp_path / "in")
    sub = []
    for i in range(n):
        rel = "/spk/utt%d.wav" % i
        batch_io.write_wav(wav_dir + rel, np.zeros(4000, np.float32), 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, np.zeros(4000, np.float32), 16000)
        sub.append((rel, "/clean" + rel))
    return wav_dir, sub


class _Stub:
    """An enhancer that must not be reached."""
    cfg = McemConfig(niter=6)
    calls = 0

    def enhance(self, *a, **kw):
        _Stub.calls += 1
        raise AssertionError("no enhancement expected")


def test_process_sublist_score_at_argument_errors_before_any_work(tmp_path):
    wav_dir, sub = _pairs(tmp_path)
    out_dir = tmp_path / "out"
    with pytest.raises(ValueError, match="score=True"):
        batch_io.process_sublist(sub, _Stub(), wav_dir, str(out_dir), score_at=(2, 4))
    for bad in ((4, 2), (2, 2), (0, 3), (3, 7)):
        with pytest.raises(ValueError):
            batch_io.process_sublist(sub, _Stub(), wav_dir, str(out_dir), score=True, score_at=bad)
    # the check comes before the file checks: a missing clean file is not what is reported
    missing = tmp_path / "in" / "clean" / "spk" / "utt1.wav"
    missing.unlink()
    with pytest.raises(ValueError):
        batch_io.process_sublist(sub, _Stub(), wav_dir, str(out_dir), score=True, score_at=(7,))
    assert _Stub.calls == 0 and not out_dir.exists()
