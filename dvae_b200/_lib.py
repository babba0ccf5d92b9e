"""ctypes binding of libdvae_b200.so (the C ABI declared in include/dvae_b200.h).

The library is opened lazily so that objects holding an engine stay picklable for the reference's
``torch.multiprocessing`` spawn pool (``scripts/evaluate_ntcd_M1.py:222,249-259``).  There is no CPU fallback: if the
shared library is missing or no CUDA device is present, the first call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdvae_b200.so")

MAX_LAYERS = 6
MAX_L = 64
MAX_K = 16
ACT_NONE, ACT_TANH, ACT_EXP = 0, 1, 2
ABI_VERSION = 4
STATUS_TIMEOUT, STATUS_NONFINITE = 1, 2

c_f32p = C.c_void_p      # device pointers are passed as integers
c_ptr = C.c_void_p


class DvaeMlp(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * (MAX_LAYERS + 1)),
                ("wt", C.c_void_p * MAX_LAYERS), ("bias", C.c_void_p * MAX_LAYERS)]


class DvaeRng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("iter0", C.c_uint32), ("reserved", C.c_uint32),
                ("eps", C.c_void_p), ("u", C.c_void_p), ("iter0_frame", C.c_void_p)]


PERMUTE_MAX_JOBS = 16


class DvaePermuteJob(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("map", C.c_void_p), ("n_rows", C.c_int64), ("row_bytes", C.c_int64),
                ("n_rep", C.c_int64), ("pitch", C.c_int64)]


# name -> (restype, argtypes); mirrors include/dvae_b200.h one to one
PROTOTYPES = {
    "dvae_version": (C.c_int, []),
    "dvae_last_error": (C.c_char_p, []),
    "dvae_stft_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int, C.c_int, C.c_int, c_ptr]),
    "dvae_istft_f32": (C.c_int, [c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr]),
    "dvae_istft_masked_f32": (C.c_int, [c_ptr, c_ptr, C.c_float, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int,
                                       C.c_int, c_ptr]),
    "dvae_mlp_workspace_floats": (C.c_int64, [C.POINTER(DvaeMlp), C.c_int64]),
    "dvae_mlp_fwd": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int64,
                               C.c_int, c_ptr, C.c_int, c_ptr, c_ptr]),
    "dvae_reparam": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "dvae_power": (C.c_int, [c_ptr, c_ptr, C.c_int64, c_ptr]),
    "dvae_nmf_vb": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "dvae_nmf_workspace_floats": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "dvae_nmf_mstep": (C.c_int, [c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64,
                                 C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "dvae_decode_stats_tc": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, c_ptr, C.c_int, C.c_int, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int64,
                                       C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "dvae_nmf_w_from_frame_stats": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "dvae_mh_workspace_floats": (C.c_int64, [C.POINTER(DvaeMlp), C.c_int64, C.c_int]),
    "dvae_mh_chain_f32": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr,
                                    C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                    C.POINTER(DvaeRng), c_ptr, c_ptr, c_ptr, c_ptr]),
    "dvae_rng_dump": (C.c_int, [C.POINTER(DvaeRng), c_ptr, c_ptr, C.c_int64, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr]),
    "dvae_wiener_accum": (C.c_int, [c_ptr, C.c_int, c_ptr, c_ptr, C.c_int64, C.c_int, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr]),
    "dvae_wiener_apply": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr]),
    "dvae_tc_image_bytes": (C.c_int64, [C.POINTER(DvaeMlp), C.c_int, C.c_int]),
    "dvae_tc_pack_decoder": (C.c_int, [C.POINTER(DvaeMlp), C.c_int, C.c_int, c_ptr, c_ptr]),
    "dvae_tc_packed_pv_bytes": (C.c_int64, [C.c_int64]),
    "dvae_tc_row_scale": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, C.c_int64, C.c_int, C.c_int, c_ptr, c_ptr]),
    "dvae_tc_pack_pv": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int64, C.c_int, C.c_int, C.c_int, c_ptr,
                                  c_ptr]),
    "dvae_vad_workspace_bytes": (C.c_int64, [C.c_int64]),
    "dvae_vad_labels": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, C.c_int64, C.c_int, C.c_int, C.c_float, c_ptr, c_ptr,
                                  c_ptr]),
    "dvae_ibm_labels": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_float, C.c_float, c_ptr, c_ptr,
                                  c_ptr, c_ptr]),
    "dvae_decode_stats_win_tc": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, C.c_int, c_ptr, c_ptr,
                                           c_ptr, C.c_int64, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr]),
    "dvae_decode_wiener_tc": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, C.c_int, c_ptr, c_ptr,
                                        c_ptr, C.c_int64, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr]),
    "dvae_energy_ratios": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr]),
    "dvae_pcm16_f32": (C.c_int, [c_ptr, C.c_int64, c_ptr, c_ptr, c_ptr]),
    "dvae_resample_taps": (C.c_int, [C.c_int, c_ptr, C.c_int]),
    "dvae_resample_poly_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "dvae_stoi_workspace_bytes": (C.c_int64, [C.c_int, C.c_int64, C.c_int]),
    "dvae_stoi_frame_capacity": (C.c_int64, [C.c_int, C.c_int64, C.c_int]),
    "dvae_stoi_envelopes": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                      c_ptr, c_ptr]),
    "dvae_stoi_scores": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr]),
    "dvae_tc_decoder_exponent_bound": (C.c_int, [C.POINTER(DvaeMlp), C.c_int, C.c_int, c_ptr, c_ptr]),
    "dvae_tc_image_bias_offset": (C.c_int64, [C.POINTER(DvaeMlp), C.c_int, C.c_int]),
    "dvae_tc_tanh_bf16_table": (C.c_int, [c_ptr, c_ptr]),
    "dvae_tc_tanh_f32": (C.c_int, [c_ptr, c_ptr, C.c_int64, c_ptr]),
    "dvae_box_muller_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64, c_ptr]),
    "dvae_decode_tc": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, c_ptr, C.c_int64, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int,
                                 c_ptr, c_ptr]),
    "dvae_vst_bytes": (C.c_int64, [C.c_int64, C.c_int]),
    "dvae_mh_chain_tc2": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int64,
                                    C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(DvaeRng), c_ptr, c_ptr, c_ptr, c_ptr,
                                    C.c_int, c_ptr, c_ptr]),
    "dvae_vst_frame_stats": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, C.c_int64,
                                       C.c_int, c_ptr, c_ptr, c_ptr]),
    "dvae_nmf_mstep_vst": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr,
                                     c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int,
                                     c_ptr, c_ptr]),
    "dvae_vst_w_partial_floats": (C.c_int64, [C.c_int64, C.c_int, C.c_int]),
    "dvae_vst_w_partials": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int,
                                      C.c_int64, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "dvae_nmf_w_from_partials": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "dvae_vst_unpack": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, c_ptr, c_ptr]),
    "dvae_vst_pack": (C.c_int, [C.POINTER(DvaeMlp), c_ptr, C.c_int, C.c_int, c_ptr, C.c_int, C.c_int64, C.c_int, c_ptr, c_ptr, c_ptr]),
    "dvae_em_stop_check": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, c_ptr, c_ptr]),
    "dvae_permute_rows": (C.c_int, [C.POINTER(DvaePermuteJob), C.c_int, c_ptr]),
    "dvae_nmf_init": (C.c_int, [C.c_uint64, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float,
                                c_ptr, c_ptr, c_ptr, c_ptr]),
}

_lock = threading.Lock()
_lib = None


class DvaeError(RuntimeError):
    pass


def load(path: str | None = None):
    """Open the shared library (once) and install the prototypes.  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        p = path or LIB_PATH
        if not os.path.exists(p):
            raise DvaeError("%s not found: run `python -m dvae_b200.build` (nvcc, sm_100a). "
                            "dvae_b200 has no CPU fallback." % p)
        lib = C.CDLL(p)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)          # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        if lib.dvae_version() != ABI_VERSION:
            raise DvaeError("libdvae_b200 ABI version %d, expected %d" % (lib.dvae_version(), ABI_VERSION))
        _lib = lib
        return lib


def check(rc: int, what: str):
    """Translate a status code: <0 -> ValueError (bad argument), >0 -> RuntimeError (CUDA error)."""
    if rc == 0:
        return
    msg = load().dvae_last_error().decode("utf-8", "replace")
    if rc < 0:
        raise ValueError("%s: %s" % (what, msg))
    raise DvaeError("%s: CUDA error %d: %s" % (what, rc, msg))


def call(name: str, *args):
    lib = load()
    check(getattr(lib, name)(*args), name)
