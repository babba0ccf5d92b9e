"""CPU-side checks: the C ABI library loads and exports what include/dvae_b200.h declares, host logic, sharding."""
import ctypes
import os
import pickle
import re

import numpy as np
import pytest
import torch

from dvae_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "dvae_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dvae_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from dvae_b200 import build
    build.build()                                   # nvcc cross-compiles sm_100a without a GPU
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "libdvae_b200.so does not export %s" % n
    assert set(names) == set(_lib.PROTOTYPES), "ctypes prototypes and header disagree"
    assert _lib.load().dvae_version() == _lib.ABI_VERSION


def test_library_is_sm100a_only():
    import subprocess
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_product_path_fails_loudly_without_gpu():
    from dvae_b200.engine import Enhancer, McemConfig
    from dvae_b200.packages.processing.stft import stft
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128])
    with pytest.raises(_lib.DvaeError):
        Enhancer(sd, "M1", McemConfig(), device=0)
    with pytest.raises(_lib.DvaeError):
        stft(np.zeros(16000, np.float32), fs=16000, wlen_sec=64e-3, center=False)
    from dvae_b200.packages.models.models import VariationalAutoencoder
    with pytest.raises(_lib.DvaeError):
        VariationalAutoencoder([513, 16, [128, 128]])(torch.zeros(2, 513))


def test_shim_signatures_and_schedules():
    from dvae_b200.packages.models import mcem
    m1 = mcem.MCEM_M1(niter=100, nsamples_E_step=10, burnin_E_step=30, nsamples_WF=25, burnin_WF=75, var_RW=0.01)
    assert m1.schedule() == ((30, 30), (75, 30))           # SURVEY Q1
    for cls in (mcem.MCEM_M2, mcem.MCEM_M2v2, mcem.MCEM_M2v3):
        assert cls(100, 10, 30, 25, 75, 0.01).schedule() == ((10, 30), (25, 75))
    m2 = pickle.loads(pickle.dumps(m1))                    # spawn pools pickle the algorithm object
    assert m2.schedule() == m1.schedule() and m2.niter == 100

    class RVAE:                                             # mcem.py:196-197
        pass
    with pytest.raises(NameError):
        m1.init_parameters(X=np.zeros((513, 4), np.complex64), S=np.zeros((513, 4), np.complex64), vae=RVAE(),
                           nmf_rank=10, eps=1e-8, device="cpu")


def test_state_dict_layout_matches_reference_keys():
    from dvae_b200.packages.models import models
    sd = synth.xavier_state_dict("M1", 513, 16, [128, 128])
    m = models.VariationalAutoencoder([513, 16, [128, 128]])
    assert set(m.state_dict()) == set(sd)
    m.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    sd2 = synth.xavier_state_dict("M2", 513, 16, [128, 128], 1)
    m2 = models.DeepGenerativeModel([513, 1, 16, [128, 128]], None)
    assert set(m2.state_dict()) == set(sd2)
    assert m2.encoder.hidden[0].weight.shape == (128, 514) and m2.decoder.hidden[0].weight.shape == (128, 17)
    v5 = models.DeepGenerativeModel_v5([513, 1, 16, [128, 128]])
    keys = set(v5.state_dict())
    assert {"enc_dec_clf.encoder.hidden.0.weight", "enc_dec_clf.decoder.reconstruction.bias",
            "enc_dec_clf.classifier.output_layer.weight", "auxiliary.hidden.0.weight"} <= keys
    # xavier-normal weights, zero biases (models.py:137-141)
    assert float(m.decoder.reconstruction.bias.abs().max()) == 0.0
    pickle.loads(pickle.dumps(m))


def test_ragged_batch_bookkeeping():
    from dvae_b200.engine import RaggedBatch
    b = RaggedBatch([3, 0, 2], "cpu", utt_ids=[10, 11, 12])
    assert b.NT == 5 and b.max_frames == 3
    assert b.fr_off.tolist() == [0, 3, 3, 5]
    assert b.frame_utt.tolist() == [0, 0, 0, 2, 2] and b.frame_gid.tolist() == [10, 10, 10, 12, 12]
    assert b.frame_idx.tolist() == [0, 1, 2, 0, 1]
    with pytest.raises(ValueError):
        RaggedBatch([], "cpu")


def test_synthetic_inputs_are_seeded_and_mixed_at_snr():
    x, s, n = synth.synth_utterance(5)
    x2, _, _ = synth.synth_utterance(5)
    assert np.array_equal(x, x2) and x.dtype == np.float32 and len(x) == 48000
    assert np.max(np.abs(x)) <= 1.0 + 1e-6
    np.testing.assert_allclose(s + n, x, atol=1e-6)
    snr = 10 * np.log10(np.sum(s.astype(np.float64) ** 2) / np.sum(n.astype(np.float64) ** 2))
    assert abs(snr - 0.0) < 1e-3                            # u % 4 == 1 -> 0 dB
    y = synth.energy_vad(s)
    assert y.shape == (1, 185) and set(np.unique(y)) <= {0.0, 1.0}


def test_wav_io_round_trip(tmp_path):
    """batch_io.read_wav / write_wav: 16-bit PCM like sf.write's default, sf.read scaling, other sample formats."""
    import struct
    from dvae_b200 import batch_io
    rng = np.random.default_rng(0)
    x = np.clip(rng.standard_normal(3000) * 0.2, -0.99, 0.99)
    p = str(tmp_path / "a" / "x.wav")
    batch_io.write_wav(p, x, 16000)
    y, fs = batch_io.read_wav(p)
    assert fs == 16000 and y.dtype == np.float64 and y.shape == x.shape
    assert np.max(np.abs(y - x)) <= 0.5 / 32768 + 1e-12
    assert np.array_equal(y * 32768.0, np.rint(x * 32768.0))
    # IEEE float32, two channels: first channel is returned
    st = np.stack([x, -x], 1).astype("<f4").tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(st)) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 3, 2, 8000, 8000 * 8, 8, 32) \
        + b"data" + struct.pack("<I", len(st))
    q = str(tmp_path / "f.wav")
    open(q, "wb").write(hdr + st)
    z, fs2 = batch_io.read_wav(q)
    assert fs2 == 8000 and np.allclose(z, x.astype(np.float32))
    with pytest.raises(ValueError):
        open(q, "wb").write(b"not a wav file")
        batch_io.read_wav(q)


def test_argument_errors_are_reported_before_any_launch():
    """Negative status + message for bad arguments (checked before the first CUDA call, so this runs without a GPU)."""
    lib = _lib.load()
    buf = (ctypes.c_float * 8)()
    off = (ctypes.c_int64 * 2)(0, 1)
    ln = (ctypes.c_int32 * 1)(8)
    p = lambda a: ctypes.cast(a, ctypes.c_void_p)
    # n_fft other than 1024
    rc = lib.dvae_stft_f32(p(buf), p(off), p(ln), 1, p(buf), None, p(off), 1, 512, 128, 520, None)
    assert rc < 0 and b"n_fft" in lib.dvae_last_error()
    # hop other than 256
    rc = lib.dvae_istft_f32(p(buf), p(off), 1, p(buf), p(off), p(ln), 8, 1024, 128, 520, None)
    assert rc < 0 and b"hop" in lib.dvae_last_error()
    # fused Wiener mask + ISTFT: the mask is mandatory, the row pitch must hold 513 bins
    rc = lib.dvae_istft_masked_f32(p(buf), None, 1.0, p(off), 1, p(buf), p(off), p(ln), 8, 1024, 256, 520, None)
    assert rc < 0 and b"mask" in lib.dvae_last_error()
    rc = lib.dvae_istft_masked_f32(p(buf), p(buf), 1.0, p(off), 1, p(buf), p(off), p(ln), 8, 1024, 256, 512, None)
    assert rc < 0 and b"bad sizes" in lib.dvae_last_error()
    with pytest.raises(ValueError):
        _lib.call("dvae_istft_masked_f32", p(buf), None, 1.0, p(off), 1, p(buf), p(off), p(ln), 8, 1024, 256, 520, None)


def test_compute_stats_prints_the_reference_tables():
    """``compute_stats`` of the metrics shim against what the reference's own function printed for the same rows
    (tests/golden/compute_stats.txt, written by oracle/make_golden.py).  The reference walks the noise types in ``set`` order,
    so the blocks are compared as a multiset of lines; the returned dictionary is checked against numpy / scipy directly."""
    import contextlib
    import io

    import scipy.stats
    from dvae_b200.packages.metrics import compute_stats, mean_confidence_interval
    from oracle.make_golden import stats_inputs
    keys, rows, snr, noise = stats_inputs()
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        out = compute_stats(keys, rows, "", 0.95, all_snr_db=snr, all_noise_types=noise)
    golden = open(os.path.join(os.path.dirname(__file__), "golden", "compute_stats.txt")).read()
    assert sorted(buf.getvalue().split("\n")) == sorted(golden.split("\n"))
    col = np.asarray([r[0] for r in rows])
    half = scipy.stats.sem(col) * scipy.stats.t.ppf(0.975, len(col) - 1)
    assert out["all"]["si_sdr"] == {"avg": np.round(col.mean(), 3), "+/-": np.round(half, 3)}
    assert set(out["snr"]) == {-5, 0, 5, 10} and set(out["noise_type"]) == {"Babble", "Cafe", "Car"}
    sel = col[snr == 5]
    assert out["snr"][5]["si_sdr"]["avg"] == np.round(sel.mean(), 3)
    assert mean_confidence_interval([1.0, 2.0, 4.0])[0] == np.round(7.0 / 3.0, 3)


def test_segment_tables_refine_tiles_and_utterances():
    """RaggedBatch.segments(): every segment lies in one 128-row tile and one utterance, the segments tile the row axis (frames, or
    frame x chain rows with several chains per frame), and an utterance's segments are consecutive (the fused W-update
    reduction relies on all three)."""
    from dvae_b200.engine import RaggedBatch
    for lens in ([3, 120, 5, 1, 128, 143], [185] * 7, [1], [0, 5, 0, 300, 0], [128, 128]):
        for c in (1, 4, 16, 128):
            b = RaggedBatch(lens, "cpu")
            seg, tile_seg, utt_seg, S = b.segments(n_chains=c)
            assert b.segments(n_chains=c)[0] is seg                      # cached per chain count
            seg, tile_seg, utt_seg = seg.numpy(), tile_seg.numpy(), utt_seg.numpy()
            rows = b.NT * c
            assert seg[0] == 0 and seg[-1] == rows and np.all(np.diff(seg) > 0) and len(seg) == S + 1
            off = b.fr_off_host * c
            for s in range(S):
                lo, hi = seg[s], seg[s + 1]
                assert lo // 128 == (hi - 1) // 128
                u = np.searchsorted(off, lo, side="right") - 1
                assert off[u] <= lo and hi <= off[u + 1] and utt_seg[u] <= s < utt_seg[u + 1]
                t = lo // 128
                assert tile_seg[t] <= s < tile_seg[t + 1]
            assert utt_seg[0] == 0 and utt_seg[-1] == S and tile_seg[-1] == S


@pytest.mark.parametrize("kw,F,route,chunk", [
    (dict(keep_E=30, keep_WF=75), 513, "emit", 25),                           # bench headline, M1
    (dict(keep_E=10, keep_WF=25), 513, "emit", 25),                           # M2 variants
    (dict(keep_E=10, keep_WF=25, n_chains=16), 513, "emit", 25),
    (dict(keep_E=10, keep_WF=25, w_partials=False), 513, "emit", 25),
    (dict(keep_E=10, keep_WF=25, n_chains=2, w_partials=False), 513, "stats", 25),
    (dict(keep_E=10, keep_WF=25, n_chains=3), 513, "stats", 25),
    (dict(keep_E=20, keep_WF=30), 513, "stats", 30),
    (dict(keep_E=5, keep_WF=5), 513, "decode", 0),
    (dict(keep_E=10, keep_WF=20, nmf_rank=12), 513, "decode", 10),
    (dict(keep_E=10, keep_WF=25, n_chains=256), 513, "stats", 25),
    (dict(keep_E=30, keep_WF=75, sampler="fp32"), 513, "decode", 0),
    (dict(keep_E=10, keep_WF=25, sampler="fp32"), 257, "decode", 0),
])
def test_mcem_route_table(kw, F, route, chunk):
    """mcem_route: which E-step route (sampler emission / FP32 decode + statistics / FP32 decode) and which final-filter chunk
    a configuration runs, without a device."""
    from dvae_b200.engine import McemConfig, mcem_route
    assert mcem_route(McemConfig(**dict(dict(sampler="tc"), **kw)), F) == (route, chunk)


def test_emission_consumers_validate_their_arguments_before_any_launch():
    """dvae_vst_w_partials / dvae_nmf_mstep_vst: chain counts that are not a power of two <= 128, several chains without the
    segment partial sums, both or neither of fstat / wpart, a wrong sample count - all refused with a negative status and a
    message before anything touches the device (runs without a GPU)."""
    lib = _lib.load()
    dec = _lib.DvaeMlp()
    dec.n_layers = 3
    for i, d in enumerate((16, 128, 128, 513)):
        dec.dims[i] = d
    buf = (ctypes.c_float * 64)()
    off = (ctypes.c_int64 * 2)(0, 1)
    seg = (ctypes.c_int32 * 2)(0, 1)
    p = lambda a: ctypes.cast(a, ctypes.c_void_p)
    D = ctypes.byref(dec)

    def w_partials(n_chains, R=10):
        return lib.dvae_vst_w_partials(D, p(buf), 16, 0, p(buf), ctypes.cast(buf, ctypes.POINTER(ctypes.c_uint8)), R, p(buf), p(buf), p(buf),
                                       p(buf), 10, 1, n_chains, 520, p(off), p(seg), p(buf), None)

    for bad in (0, 3, 12, 256):
        assert w_partials(bad) < 0 and b"power of two" in lib.dvae_last_error(), bad
    assert w_partials(1, R=40) < 0 and b"bad sizes" in lib.dvae_last_error()

    def mstep(n_chains, fstat, wpart, R=10, K=10):
        return lib.dvae_nmf_mstep_vst(D, p(buf), 16, 0, p(buf), p(buf), ctypes.cast(buf, ctypes.POINTER(ctypes.c_uint8)), R, p(buf), p(buf), p(buf),
                                      p(buf), p(buf), p(off), 1, 1, K, 520, 1, p(buf), fstat, wpart, p(seg), n_chains, None, None)

    assert mstep(1, None, None) < 0 and b"exactly one" in lib.dvae_last_error()
    assert mstep(1, p(buf), p(buf)) < 0 and b"exactly one" in lib.dvae_last_error()
    assert mstep(6, None, p(buf)) < 0 and b"power of two" in lib.dvae_last_error()
    assert mstep(4, p(buf), None) < 0 and b"segment partial sums" in lib.dvae_last_error()
    assert mstep(1, p(buf), None, R=20) < 0 and b"R in" in lib.dvae_last_error()
    assert mstep(1, p(buf), None, K=11) < 0 and b"K <=" in lib.dvae_last_error()
    dec.dims[3] = 257                                                   # not the 513-bin decoder the tensor-core path is built for
    assert mstep(1, p(buf), None) < 0 and b"F=513" in lib.dvae_last_error()


def test_process_sublist_batches_reads_and_writes_with_a_stub_enhancer(tmp_path):
    """File plumbing of batch_io.process_sublist without a GPU: every input is read exactly once and in order (the next batch is
    read ahead while the current one runs), both estimates are written per utterance, ids come from the paths, finished
    utterances are skipped on a second run."""
    from dvae_b200 import batch_io
    wav_dir, out_dir = str(tmp_path / "in"), str(tmp_path / "out")
    rng = np.random.default_rng(0)
    sub, sigs = [], {}
    for i in range(7):
        rel = "/spk%d/utt%d.wav" % (i % 2, i)
        x = (0.1 * rng.standard_normal(4000 + 100 * i)).astype(np.float32)
        batch_io.write_wav(wav_dir + rel, x, 16000)
        sigs[rel] = batch_io.read_wav(wav_dir + rel)[0]
        sub.append((rel, "/clean" + rel))

    class Stub:
        def __init__(self):
            self.calls = []

        def enhance(self, xs, y_list=None, max_frames_list=None, utt_ids=None):
            self.calls.append((len(xs), list(utt_ids)))
            return [0.5 * x for x in xs], [0.25 * x for x in xs], None

    for bs in (3, 7, 100):
        stub = Stub()
        out = out_dir + str(bs)
        done = batch_io.process_sublist(sub, stub, wav_dir, out, batch_size=bs)
        assert done == [batch_io.output_stem(out, rel) for rel, _ in sub]
        assert [n for n, _ in stub.calls] == [min(bs, 7 - lo) for lo in range(0, 7, bs)]
        assert [i for _, ids in stub.calls for i in ids] == [batch_io.utterance_id(rel) for rel, _ in sub]
        for rel, _ in sub:
            s, fs = batch_io.read_wav(batch_io.output_stem(out, rel) + "_s_est.wav")
            n, _ = batch_io.read_wav(batch_io.output_stem(out, rel) + "_n_est.wav")
            assert fs == 16000 and np.allclose(s, 0.5 * sigs[rel], atol=1e-4) and np.allclose(n, 0.25 * sigs[rel], atol=1e-4)
        assert batch_io.process_sublist(sub, stub, wav_dir, out, batch_size=bs) == []
