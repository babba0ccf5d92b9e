"""Cost of the quality trace over EM iterations (Enhancer.enhance(..., score_at=...)) on the headline workload; prints one
JSON line.

    python tools/bench_trace.py [--batch 512] [--niter 100] [--steps 3] [--warmup 1] [--out profiles/r05_bench_trace.json]

Workload: bench.py's headline (M1, 512 synthetic 3 s utterances, 100 EM iterations, tensor-core sampler), same weights,
schedule and seed, device-resident inputs.  Every arm is one scored step as ``enhance(ref_list=...)`` runs it on the device
(``run_device``, 16-bit quantisation of the estimate, ``metrics.score_batch``), with the checkpoints of ``score_at`` scored on
the way.  Arms, alternating in one process, CUDA events around each step:
- ``no_trace``: ``score_at=()``;
- ``every_25``: ``score_at=(25, 50, 75, 100)``;
- ``every_10``: ``score_at=(10, 20, ..., 100)``.
Reported with the GPU's name and power limit read in the same run:
- device time per step of each arm, and per checkpoint: (arm - no_trace) / side runs (``niter`` itself needs none);
- what the trace replaces: separate scored runs with ``niter = 10`` and ``niter = 50``, timed the same way, plus the
  ``no_trace`` arm for ``niter = 100``; the other counts are extrapolated linearly through the 10 and 50 runs and labelled so;
- whether the traced steps returned the untraced cost and scores bit for bit, and whether the trace entries at 10 and 50
  equal the scores of those separate runs;
- the mean trace (the quality curve) over the batch.
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
SEPARATE = (10, 50)          # niter of the separate runs that are timed; others are extrapolated from these two


class ScoredStep:
    """One scored enhancement step of ``niter`` EM iterations on device-resident inputs, with an optional trace."""

    def __init__(self, sd, niter, B, T, x_dev, s_dev, off, lens, batch):
        cfg = McemConfig(var_rw=0.01, nmf_rank=10, eps=1e-8, seed=2024, sampler="tc", **bench.schedule("M1", niter))
        self.enh = Enhancer(sd, "M1", cfg, device=0)
        self.niter, self.B, self.T = niter, B, T
        self.x_dev, self.s_dev, self.off, self.lens, self.batch = x_dev, s_dev, off, lens, batch
        self.ref = metrics.score_reference(x_dev, s_dev, off, lens, FS)
        self.s_q = torch.empty(B * T, device=x_dev.device)
        self.scores = torch.empty((B, 2, 5), dtype=torch.float64, device=x_dev.device)

    def __call__(self, score_at=()):
        B, T, eng = self.B, self.T, self.enh.engine
        trace = eng._get("trace", (B, len(score_at), 5), torch.float64) if score_at else None
        on_checkpoint = None
        if score_at:
            on_checkpoint = self.enh.checkpoint_scorer(self.ref, self.off, self.lens, self.batch, B * T, T,
                                                       {n: trace[:, k] for k, n in enumerate(score_at)})
        side = tuple(n for n in score_at if n < self.niter)
        s_dev, _, cost = self.enh.run_device(self.x_dev, self.off, self.lens, self.batch, None, B * T, T, None, side, on_checkpoint)
        metrics.pcm16(s_dev, None, self.s_q)
        metrics.score_batch(self.s_q, self.x_dev, self.s_dev, self.off, self.lens, FS, out=self.scores)
        if score_at and score_at[-1] == self.niter:
            trace[:, -1].copy_(self.scores[:, 0])
        return cost, self.scores, trace


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
    ap.add_argument("--niter", type=int, default=100)
    ap.add_argument("--steps", type=int, default=3, help="timed steps per arm (the arms alternate)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_trace.json"), help="'' to print only")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_trace.py needs a CUDA device")
    if a.niter < max(SEPARATE) or a.steps < 3:
        raise SystemExit("--niter must be at least %d and --steps at least 3" % max(SEPARATE))
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
    step = ScoredStep(sd, a.niter, B, T, x_dev, s_dev, off, lens, batch)
    arms = {"no_trace": (), "every_25": tuple(range(25, a.niter + 1, 25)), "every_10": tuple(range(10, a.niter + 1, 10))}

    for _ in range(a.warmup):
        for cps in arms.values():
            step(cps)
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    res = {}
    for _ in range(a.steps):
        for k, cps in arms.items():
            t, (cost, scores, trace) = event_time(lambda: step(cps))
            ms[k].append(t)
            res[k] = (cost.clone(), scores.clone(), None if trace is None else trace.clone())
    med = {k: float(np.median(v)) for k, v in ms.items()}
    identical = {k: bool(torch.equal(res[k][0], res["no_trace"][0]) and
                         np.array_equal(res[k][1].cpu().numpy(), res["no_trace"][1].cpu().numpy(), equal_nan=True))
                 for k in arms if k != "no_trace"}

    # the separate scored runs the trace replaces (two timed; the no_trace arm is the niter run)
    sep_ms, sep_equal = {}, {}
    for n in SEPARATE:
        st = ScoredStep(sd, n, B, T, x_dev, s_dev, off, lens, batch)
        for _ in range(a.warmup):
            st()
        times = []
        for _ in range(a.steps):
            t, (_, scores, _) = event_time(st)
            times.append(t)
        sep_ms[n] = {"median": float(np.median(times)), "all": times}
        k = arms["every_10"].index(n)
        sep_equal[n] = bool(np.array_equal(res["every_10"][2][:, k].cpu().numpy(), scores[:, 0].cpu().numpy(), equal_nan=True))
        del st
        torch.cuda.empty_cache()
    (n0, n1), (t0, t1) = SEPARATE, (sep_ms[SEPARATE[0]]["median"], sep_ms[SEPARATE[1]]["median"])
    slope = (t1 - t0) / (n1 - n0)

    def separate_cost(cps):
        measured = {n: sep_ms[n]["median"] for n in cps if n in sep_ms}
        if a.niter in cps:
            measured[a.niter] = med["no_trace"]
        extrap = {n: t0 + slope * (n - n0) for n in cps if n not in measured}
        total = sum(measured.values()) + sum(extrap.values())
        return {"measured_ms": measured, "extrapolated_ms": extrap, "total_ms": total}

    report = {}
    for k, cps in arms.items():
        if not cps:
            continue
        side = len([n for n in cps if n < a.niter])
        sep = separate_cost(cps)
        report[k] = {"score_at": list(cps), "side_runs": side, "step_ms": med[k],
                     "ms_per_checkpoint": (med[k] - med["no_trace"]) / side,
                     "separate_runs": sep, "speedup_vs_separate_runs": sep["total_ms"] / med[k],
                     "outputs_identical_to_no_trace": identical[k]}
    curve = res["every_10"][2].cpu().numpy()
    line = {"tool": "bench_trace", "gpu": gpu,
            "workload": "M1, %d synthetic %.0f s utterances, %d EM iterations, sampler tc (bench.py headline), scored as "
                        "enhance(ref_list=...)" % (B, bench.SECONDS, a.niter),
            "device_ms_per_step": {k: {"median": med[k], "all": ms[k]} for k in arms},
            "trace": report,
            "separate_runs_ms": sep_ms,
            "separate_run_time_model": "t(n) = %.3f ms + %.4f ms x (n - %d), through the measured niter = %d and %d runs; "
                                       "entries under extrapolated_ms come from it" % (t0, slope, n0, n0, n1),
            "trace_equals_separate_runs": sep_equal,
            "mean_trace_every_10": {str(n): dict(zip(metrics.SCORE_KEYS, np.nanmean(curve[:, k], axis=0).tolist()))
                                    for k, n in enumerate(arms["every_10"])}}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
