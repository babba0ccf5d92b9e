"""Oracle labels of the M2 models: per-utterance shims on the host against the device route of ``Enhancer.enhance``; prints
one JSON line.

    python tools/bench_labels.py [--batches 512,4096] [--niter 100] [--steps 3] [--warmup 1]
                                 [--out profiles/r07_bench_labels.json]

Workloads, each at every batch size (synthetic 3 s utterances, tensor-core sampler, bench.py's M2 schedule and seed):
- ``robust_ibm``: the IBM-conditioned M2 (``y_dim = 513``, scripts/evaluate_ntcd_M2.py:66-73), labels
  ``noise_robust_clean_speech_IBM(s, stft(s))``;
- ``vad``: the one-label M2, labels ``clean_speech_VAD(s)``.
Two arms, alternated in one process, ``--steps`` timed calls each after ``--warmup`` untimed ones:
- ``callback``: the labels of every utterance from the package's per-utterance shims (each call goes to the device and back),
  then ``enhance(y_list=...)``;
- ``device``: ``enhance(s_list=..., oracle_labels=...)``.
Per arm: the label stage alone (host clock around work that ends in a synchronise; for the device arm
``Enhancer.oracle_labels_device`` on the clean signals already on the device), the whole ``enhance`` call (host clock, the call
returns host arrays) and its H2D bytes.  Both arms must return the same estimates and cost bit for bit.  The GPU's name and
power limit are read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from bench_stoi import gpu_info  # noqa: E402
from dvae_b200 import synth  # noqa: E402
from dvae_b200.engine import Enhancer, McemConfig, RaggedBatch  # noqa: E402
from dvae_b200.packages.processing import stft as dstft  # noqa: E402
from dvae_b200.packages.processing import target as dtarget  # noqa: E402

KW = dict(fs=16000, wlen_sec=64e-3, hop_percent=0.25, center=False, pad_at_end=True)
WORKLOADS = {"robust_ibm": 513, "vad": 1}


def shim_labels(mode, s):
    if mode == "vad":
        return dtarget.clean_speech_VAD(s, **KW)
    S = dstft.stft(s, win="hann", **KW)
    if mode == "ibm":
        return dtarget.clean_speech_IBM(S)
    return dtarget.noise_robust_clean_speech_IBM(s, S, **KW)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def run_workload(mode, B, niter, steps, warmup, dev):
    T = int(bench.SECONDS * synth.FS)
    xs, ss = bench.synth_set(1000, B)
    sd = synth.xavier_state_dict("M2", 513, 16, [128, 128], WORKLOADS[mode], seed=1234, out_bias=bench.reference_power())
    cfg = McemConfig(var_rw=0.01, nmf_rank=10, eps=1e-8, seed=2024, sampler="tc", **bench.schedule("M2", niter))
    enh = Enhancer(sd, "M2", cfg, device=dev.index)
    ids = list(range(B))
    # the clean signals on the device in enhance's layout, for the device arm's label stage on its own
    off = np.arange(B + 1, dtype=np.int64) * ((T + 1) // 2 * 2)
    s_dev = torch.from_numpy(np.stack(ss)).to(dev).reshape(-1)
    x_off = torch.from_numpy(off[:-1].copy()).to(dev)
    x_len = torch.full((B,), T, dtype=torch.int32, device=dev)
    nfr = np.full(B, synth.num_frames(T), np.int64)
    batch = RaggedBatch(nfr, dev, ids)

    def callback_labels():
        return [shim_labels(mode, s) for s in ss]

    def device_labels():
        return enh.oracle_labels_device(mode, s_dev, x_off, x_len, nfr, batch)

    ys = callback_labels()
    arms = {
        "callback": (callback_labels, lambda: enh.enhance(xs, y_list=ys, utt_ids=ids)),
        "device": (device_labels, lambda: enh.enhance(xs, s_list=ss, oracle_labels=mode, utt_ids=ids)),
    }
    ms = {k: {"label_stage": [], "enhance": []} for k in arms}
    h2d, last = {}, {}
    for i in range(warmup + steps):
        for k, (label_fn, call) in arms.items():
            t_lab, _ = timed(label_fn)
            t_enh, res = timed(call)
            h2d[k] = int(enh.h2d_bytes)
            if i >= warmup:
                ms[k]["label_stage"].append(t_lab)
                ms[k]["enhance"].append(t_enh)
            last[k] = res
    a, b = last["callback"], last["device"]
    same = (all(np.array_equal(p, q) for p, q in zip(a[0], b[0])) and all(np.array_equal(p, q) for p, q in zip(a[1], b[1]))
            and np.array_equal(a[2], b[2]))
    assert same, "%s B=%d: the device labels do not reproduce the callback run" % (mode, B)
    med = {k: {s: float(np.median(v)) for s, v in d.items()} for k, d in ms.items()}
    out = {"mode": mode, "y_dim": WORKLOADS[mode], "batch": B, "niter": niter, "bit_identical_estimates_and_cost": bool(same)}
    for k in arms:
        out[k] = {"label_stage_ms": {"median": med[k]["label_stage"], "all": ms[k]["label_stage"]},
                  "enhance_ms": {"median": med[k]["enhance"], "all": ms[k]["enhance"]},
                  "h2d_bytes": h2d[k]}
    out["callback"]["labels_plus_enhance_ms"] = med["callback"]["label_stage"] + med["callback"]["enhance"]
    out["device"]["label_stage_share_of_enhance"] = med["device"]["label_stage"] / med["device"]["enhance"]
    out["speedup_labels_plus_enhance"] = out["callback"]["labels_plus_enhance_ms"] / med["device"]["enhance"]
    del enh, last, a, b, ys
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="512,4096")
    ap.add_argument("--modes", default=",".join(WORKLOADS))
    ap.add_argument("--niter", type=int, default=100)
    ap.add_argument("--steps", type=int, default=3, help="timed calls per arm (the arms alternate)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_bench_labels.json"), help="'' to print only")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_labels.py needs a CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    gpu = gpu_info()
    rows = [run_workload(m, int(B), a.niter, a.steps, a.warmup, dev) for m in a.modes.split(",") for B in a.batches.split(",")]
    line = {"tool": "bench_labels", "gpu": gpu,
            "workload": "M2 (tensor-core sampler, bench.py M2 schedule), synthetic %.0f s utterances; label stage and whole "
                        "enhance call on the host clock around work that ends in a synchronise" % bench.SECONDS,
            "rows": rows}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
