"""Cost of scoring inside the enhancement pass (Enhancer.enhance(ref_list=...)) on the headline workload; prints one JSON line.

    python tools/bench_score.py [--batch 512] [--niter 100] [--steps 3] [--pcm-batches 512,4096] [--iters 20] [--out FILE]

Workload: bench.py's headline (M1, 512 synthetic 3 s utterances, 100 EM iterations, tensor-core sampler), same weights,
schedule and seed.  Reported, with the GPU's name and power limit read in the same run:
- device time per step (CUDA events, device-resident inputs) of the enhancement alone and of the enhancement followed by
  what ``ref_list`` adds on the device (16-bit quantisation of the estimate + ``metrics.score_batch``), the two arms
  alternating in one process;
- the wall time of the public host call ``Enhancer.enhance`` with and without ``ref_list``, and its device-to-host bytes with
  and without ``pcm16``;
- CUDA-event times of ``dvae_pcm16_f32`` (both outputs) at each batch size of ``--pcm-batches`` and its share of the HBM
  peak, from the bytes the shapes imply (4 read + 2 + 4 written per sample), and of ``score_batch`` alone at ``--batch``.
Needs a CUDA device.
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
from bench_stoi import HBM_BPS, gpu_info, timed  # noqa: E402
from dvae_b200 import synth  # noqa: E402
from dvae_b200.engine import Enhancer, McemConfig, RaggedBatch  # noqa: E402
from dvae_b200.packages import metrics  # noqa: E402

FS = synth.FS


def pcm16_bench(B, T, iters, warmup):
    n = B * T
    x = torch.randn(n, device="cuda") * 0.3
    pcm = torch.empty(n, dtype=torch.int16, device="cuda")
    xq = torch.empty_like(x)
    t = timed(lambda: metrics.pcm16(x, pcm, xq), iters, warmup)
    nbytes = n * (4 + 2 + 4)
    del x, pcm, xq
    torch.cuda.empty_cache()
    return {"B": B, "samples": n, "bytes": nbytes, "ms_median_min_max": t, "bytes_per_s": nbytes / (t[0] * 1e-3),
            "share_of_hbm_peak": nbytes / HBM_BPS / (t[0] * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--niter", type=int, default=100)
    ap.add_argument("--steps", type=int, default=3, help="timed steps per arm (the arms alternate)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--pcm-batches", default="512,4096")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_score.py needs a CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    gpu = gpu_info()
    B, T = a.batch, int(bench.SECONDS * FS)
    x_host, s_host = bench.synth_set(1000, B)
    sd = bench.model_weights("M1", bench.reference_power())
    cfg = McemConfig(var_rw=0.01, nmf_rank=10, eps=1e-8, seed=2024, sampler="tc", **bench.schedule("M1", a.niter))
    enh = Enhancer(sd, "M1", cfg, device=0)
    ids = list(range(B))
    batch = RaggedBatch([synth.num_frames(T)] * B, dev, ids)
    x_dev = torch.from_numpy(np.stack(x_host)).to(dev).reshape(-1)
    s_dev = torch.from_numpy(np.stack(s_host)).to(dev).reshape(-1)
    off = (torch.arange(B, dtype=torch.int64) * T).to(dev)
    lens = torch.full((B,), T, dtype=torch.int32, device=dev)
    s_q = torch.empty(B * T, device=dev)
    scores = torch.empty((B, 2, 5), dtype=torch.float64, device=dev)

    def enhance_only():
        return enh.run_device(x_dev, off, lens, batch, None, B * T, T)

    def score(est):
        metrics.pcm16(est, None, s_q)
        metrics.score_batch(s_q, x_dev, s_dev, off, lens, FS, out=scores)

    def enhance_and_score():
        score(enhance_only()[0])

    arms = {"without_ref_list": enhance_only, "with_ref_list": enhance_and_score}
    for _ in range(a.warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(a.steps):
        for k, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    score(enhance_only()[0])
    t_score = timed(lambda: metrics.score_batch(s_q, x_dev, s_dev, off, lens, FS, out=scores), a.iters, 2)
    sc = scores.cpu().numpy()

    # the public host call: wall time with / without ref_list, device-to-host bytes with / without pcm16
    host = {}
    for name, kw in (("plain", {}), ("ref_list", dict(ref_list=s_host)), ("ref_list_pcm16", dict(ref_list=s_host, pcm16=True)),
                     ("pcm16", dict(pcm16=True))):
        res = enh.enhance(x_host, utt_ids=ids, **kw)                   # warm the pinned buffers of this shape
        del res
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = enh.enhance(x_host, utt_ids=ids, **kw)
        host[name] = {"wall_ms": (time.perf_counter() - t0) * 1e3, "d2h_bytes": int(enh.d2h_bytes), "h2d_bytes": int(enh.h2d_bytes)}
        del res
    del enh
    torch.cuda.empty_cache()
    pcm = [pcm16_bench(int(b), T, a.iters, 3) for b in a.pcm_batches.split(",")]

    line = {"tool": "bench_score", "gpu": gpu, "hbm_peak_bytes_per_s": HBM_BPS,
            "workload": "M1, %d synthetic %.0f s utterances, %d EM iterations, sampler tc (bench.py headline)" % (B, bench.SECONDS, a.niter),
            "device_ms_per_step": {k: {"median": med[k], "all": ms[k]} for k in arms},
            "scoring_overhead_ms": med["with_ref_list"] - med["without_ref_list"],
            "scoring_overhead_fraction": med["with_ref_list"] / med["without_ref_list"] - 1.0,
            "score_batch_ms_median_min_max": t_score,
            "host_enhance": host,
            "d2h_saving_pcm16_bytes": host["plain"]["d2h_bytes"] - host["pcm16"]["d2h_bytes"],
            "pcm16_kernel": pcm,
            "mean_scores": dict(zip(metrics.SCORE_KEYS, np.nanmean(sc[:, 0], axis=0).tolist())),
            "mean_scores_input": dict(zip(metrics.SCORE_KEYS, np.nanmean(sc[:, 1], axis=0).tolist()))}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
