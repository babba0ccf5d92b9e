"""Per-utterance stopping of the EM loop (McemConfig.stop_tol) on the headline workload; prints one JSON line.

    python tools/bench_stop.py [--batch 512] [--caps 100,500] [--tols 1e-3,1e-4] [--window 10] [--steps 3] [--warmup 1]
                               [--out profiles/r06_bench_stop.json]

Workload: bench.py's headline (M1, 512 synthetic 3 s utterances, tensor-core sampler), same weights, schedule and seed,
device-resident inputs, each step scored as ``enhance(ref_list=...)`` scores it.  For every cap ``niter`` one arm runs the
fixed count (``stop_tol=None``) and one arm per tolerance stops each utterance on its own cost.  The arms alternate in one
process, CUDA events around each step.  Reported with the GPU's name and power limit read in the same run, per arm:
- device time per step and audio seconds per second;
- the histogram of the utterances' EM iteration counts n_u, and the EM loop iterations executed against the cap;
- device time of the stages ``stop_check`` / ``stop_permute`` (from one extra step with stage timing on);
- step time per executed loop iteration next to the fixed arm's (the per-iteration synchronisation shows there);
- the mean score rows of the estimate next to the fixed-cap arm's.  The weights are synthetic: these numbers say nothing
  about the quality of stopping with trained models.
Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from bench_stoi import gpu_info  # noqa: E402
from dvae_b200 import synth  # noqa: E402
from dvae_b200.engine import Enhancer, McemConfig, RaggedBatch  # noqa: E402
from dvae_b200.packages import metrics  # noqa: E402

FS = synth.FS


class Step:
    """One scored enhancement step on device-resident inputs."""

    def __init__(self, sd, niter, tol, window, B, T, x_dev, s_dev, off, lens, batch):
        cfg = McemConfig(var_rw=0.01, nmf_rank=10, eps=1e-8, seed=2024, sampler="tc", stop_tol=tol, stop_window=window,
                         **bench.schedule("M1", niter))
        self.enh = Enhancer(sd, "M1", cfg, device=0)
        self.B, self.T = B, T
        self.x_dev, self.s_dev, self.off, self.lens, self.batch = x_dev, s_dev, off, lens, batch
        self.s_q = torch.empty(B * T, device=x_dev.device)
        self.scores = torch.empty((B, 2, 5), dtype=torch.float64, device=x_dev.device)

    def __call__(self):
        B, T = self.B, self.T
        s_dev, _, cost = self.enh.run_device(self.x_dev, self.off, self.lens, self.batch, None, B * T, T)
        metrics.pcm16(s_dev, None, self.s_q)
        metrics.score_batch(self.s_q, self.x_dev, self.s_dev, self.off, self.lens, FS, out=self.scores)
        return cost, self.scores


def event_time(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--caps", default="100,500")
    ap.add_argument("--tols", default="1e-3,1e-4")
    ap.add_argument("--window", type=int, default=10)
    ap.add_argument("--steps", type=int, default=3, help="timed steps per arm (the arms alternate)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_stop.json"), help="'' to print only")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stop.py needs a CUDA device")
    if a.steps < 3:
        raise SystemExit("--steps must be at least 3")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    gpu = gpu_info()
    B, T = a.batch, int(bench.SECONDS * FS)
    x_host, s_host = bench.synth_set(1000, B)
    sd = bench.model_weights("M1", bench.reference_power())
    batch = RaggedBatch([synth.num_frames(T)] * B, dev, list(range(B)))
    x_dev = torch.from_numpy(np.stack(x_host)).to(dev).reshape(-1)
    s_dev = torch.from_numpy(np.stack(s_host)).to(dev).reshape(-1)
    off = (torch.arange(B, dtype=torch.int64) * T).to(dev)
    lens = torch.full((B,), T, dtype=torch.int32, device=dev)
    caps = [int(c) for c in a.caps.split(",")]
    tols = [float(t) for t in a.tols.split(",")]
    arms = {}
    for cap in caps:
        for tol in [None] + tols:
            arms["niter%d_%s" % (cap, "fixed" if tol is None else "tol%g" % tol)] = (cap, tol)
    steps = {k: Step(sd, cap, tol, a.window, B, T, x_dev, s_dev, off, lens, batch) for k, (cap, tol) in arms.items()}

    for _ in range(a.warmup):
        for st in steps.values():
            st()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    last = {}
    for _ in range(a.steps):
        for k, st in steps.items():
            t, (cost, scores) = event_time(st)
            ms[k].append(t)
            last[k] = (cost.cpu().numpy(), scores.cpu().numpy(), st.enh.engine.n_iter.copy())
    stages = {}
    for k, st in steps.items():                    # one more step per arm with stage timing on (not in the timed steps)
        eng = st.enh.engine
        eng.timing = True
        st()
        stages[k] = {n: {"ms": v[0], "calls": v[1]} for n, v in eng.stage_times_ms().items()}
        eng.timing = False

    report = {}
    for k, (cap, tol) in arms.items():
        med = float(np.median(ms[k]))
        cost, scores, n_u = last[k]
        fixed = "niter%d_fixed" % cap
        loop = int(n_u.max())
        vals, counts = np.unique(n_u, return_counts=True)
        report[k] = {
            "niter_cap": cap, "stop_tol": tol, "stop_window": a.window if tol is not None else None,
            "device_ms_per_step": {"median": med, "all": ms[k]},
            "audio_s_per_s": B * bench.SECONDS / (med / 1e3),
            "n_u_histogram": {str(int(v)): int(c) for v, c in zip(vals, counts)},
            "n_u_mean": float(n_u.mean()),
            "em_loop_iterations": loop, "em_utterance_iterations": int(n_u.sum()), "em_utterance_iterations_cap": cap * B,
            "stage_ms": {n: stages[k][n] for n in ("stop_check", "stop_permute", "mh", "mstep") if n in stages[k]},
            "ms_per_loop_iteration": med / loop,
            "fixed_ms_per_iteration": float(np.median(ms[fixed])) / cap,
            "speedup_vs_fixed_cap": float(np.median(ms[fixed])) / med,
            "mean_scores_estimate_synthetic_weights": dict(zip(metrics.SCORE_KEYS, np.nanmean(scores[:, 0], axis=0).tolist())),
            "mean_scores_fixed_cap_synthetic_weights": dict(zip(metrics.SCORE_KEYS, np.nanmean(last[fixed][1][:, 0], axis=0).tolist())),
        }
    line = {"tool": "bench_stop", "gpu": gpu,
            "workload": "M1, %d synthetic %.0f s utterances, sampler tc (bench.py headline), scored as enhance(ref_list=...); "
                        "synthetic weights: score differences say nothing about trained models" % (B, bench.SECONDS),
            "arms": report}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
