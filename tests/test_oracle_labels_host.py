"""Host side of the oracle-label route (no GPU): process_sublist(..., oracle_labels=) reads each clean file once and hands the
enhancer one list as both s_list and ref_list; the argument checks of process_sublist and Enhancer.label_mode."""
import types

import numpy as np
import pytest

from dvae_b200 import batch_io
from dvae_b200.engine import ORACLE_LABELS, Enhancer


def _files(tmp_path, n=7):
    wav_dir = str(tmp_path / "in")
    rng = np.random.default_rng(0)
    sub = []
    for i in range(n):
        rel = "/spk%d/utt%d.wav" % (i % 2, i)
        T = 4000 + 100 * i
        batch_io.write_wav(wav_dir + rel, (0.1 * rng.standard_normal(T)).astype(np.float32), 16000)
        batch_io.write_wav(wav_dir + "/clean" + rel, (0.05 * rng.standard_normal(T)).astype(np.float32), 16000)
        sub.append((rel, "/clean" + rel))
    return wav_dir, sub


class Stub:
    """Records every enhance call's keyword arguments; returns scaled inputs and, with ref_list, zero scores."""

    def __init__(self):
        self.calls = []

    def enhance(self, xs, y_list=None, max_frames_list=None, utt_ids=None, ref_list=None, pcm16=False, score_at=(), s_list=None,
                oracle_labels=None):
        self.calls.append(dict(n=len(xs), y_list=y_list, ref_list=ref_list, s_list=s_list, oracle_labels=oracle_labels,
                               caps=max_frames_list))
        s = [(0.5 * x * 32768).astype(np.int16) if pcm16 else 0.5 * x for x in xs]
        out = (s, s, None)
        return out if ref_list is None else out + (np.zeros((len(xs), 2, 5)),)


def _count_reads(monkeypatch):
    reads = []
    real = batch_io._read_checked

    def counted(path, fs, length=None):
        reads.append(path)
        return real(path, fs, length)

    monkeypatch.setattr(batch_io, "_read_checked", counted)
    return reads


@pytest.mark.parametrize("score", [False, True])
@pytest.mark.parametrize("mode", ORACLE_LABELS)
def test_each_clean_file_is_read_once_and_passed_as_one_list(tmp_path, monkeypatch, score, mode):
    wav_dir, sub = _files(tmp_path)
    reads = _count_reads(monkeypatch)
    stub = Stub()
    out = batch_io.process_sublist(sub, stub, wav_dir, str(tmp_path / "out"), batch_size=3, oracle_labels=mode, score=score,
                                   max_frames=lambda a, b: 2)
    stems = out[0] if score else out
    assert len(stems) == len(sub)
    assert sorted(reads) == sorted(wav_dir + p for ab in sub for p in ab)          # every file once, clean ones included
    assert [c["n"] for c in stub.calls] == [3, 3, 1]
    lo = 0
    for c in stub.calls:
        assert c["oracle_labels"] == mode and c["y_list"] is None and c["caps"] == [2] * c["n"]
        assert c["ref_list"] is (c["s_list"] if score else None)
        for s, (_, clean) in zip(c["s_list"], sub[lo:lo + c["n"]]):
            assert np.array_equal(s, batch_io.read_wav(wav_dir + clean)[0].astype(np.float32))
        lo += c["n"]


def test_without_oracle_labels_nothing_changes(tmp_path, monkeypatch):
    wav_dir, sub = _files(tmp_path)
    reads = _count_reads(monkeypatch)
    stub = Stub()
    batch_io.process_sublist(sub, stub, wav_dir, str(tmp_path / "out"), batch_size=4)
    assert sorted(reads) == sorted(wav_dir + a for a, _ in sub)                       # no clean file is read
    assert all(c["s_list"] is None and c["oracle_labels"] is None for c in stub.calls)


def test_process_sublist_argument_errors_come_before_any_read(tmp_path, monkeypatch):
    wav_dir, sub = _files(tmp_path)
    reads = _count_reads(monkeypatch)
    stub = Stub()
    out = str(tmp_path / "out")
    with pytest.raises(ValueError, match="labels callback"):
        batch_io.process_sublist(sub, stub, wav_dir, out, oracle_labels="vad", labels=lambda a, b: np.ones((1, 3), np.float32))
    for bad in ("VAD", "ideal", 1, True):
        with pytest.raises(ValueError, match="oracle_labels must be"):
            batch_io.process_sublist(sub, stub, wav_dir, out, oracle_labels=bad)
    with pytest.raises(ValueError, match="pairs"):
        batch_io.process_sublist([(sub[0][0],)], stub, wav_dir, out, oracle_labels="ibm")
    assert reads == [] and stub.calls == []
    # a clean file of another length than its noisy file
    batch_io.write_wav(wav_dir + sub[2][1], np.zeros(10, np.float32), 16000)
    with pytest.raises(ValueError, match="samples, the noisy file has"):
        batch_io.process_sublist(sub, stub, wav_dir, out, oracle_labels="vad")
    assert stub.calls == []


def _model(y_dim):
    return types.SimpleNamespace(weights=types.SimpleNamespace(y_dim=y_dim), n_fft=1024)


def test_label_mode():
    s, y = [np.zeros(4)], [np.zeros((1, 1))]
    mode = Enhancer.label_mode
    assert mode(_model(0), None, None, None) is None
    assert mode(_model(0), None, s, None) is None                                     # M1: clean signals are only scored
    assert mode(_model(1), None, s, None) == "vad"                                    # today's meaning of s_list
    assert mode(_model(1), None, s, y) is None                                        # y_list wins, as before
    assert mode(_model(1), "vad", s, None) == "vad"
    for m in ("ibm", "robust_ibm"):
        assert mode(_model(513), m, s, None) == m
    assert mode(_model(513), None, None, y) is None


@pytest.mark.parametrize("y_dim, oracle, s, y, what", [
    (513, None, True, False, "oracle_labels='ibm'"),           # neither IBM kind is the default
    (3, None, True, False, "oracle_labels='ibm'"),
    (1, "ibm", True, False, "gives 513 labels"),
    (1, "robust_ibm", True, False, "gives 513 labels"),
    (513, "vad", True, False, "gives 1 labels"),
    (2, "vad", True, False, "gives 1 labels"),
    (0, "vad", True, False, "M1"),
    (0, "ibm", True, False, "M1"),
    (1, "vad", False, False, "s_list"),
    (513, "ibm", False, True, "s_list"),
    (1, "vad", True, True, "y_list"),
    (513, "robust_ibm", True, True, "y_list"),
    (1, "VAD", True, False, "must be one of"),
    (513, "nr_ibm", True, False, "must be one of"),
])
def test_label_mode_errors(y_dim, oracle, s, y, what):
    with pytest.raises(ValueError, match=what.replace("(", r"\(")):
        Enhancer.label_mode(_model(y_dim), oracle, [np.zeros(4)] if s else None, [np.zeros((1, 1))] if y else None)
