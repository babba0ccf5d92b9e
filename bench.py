#!/usr/bin/env python
"""Benchmark of the MCEM VAE-NMF enhancement hot path (BASELINE.json metric: enhanced audio-seconds per second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One *step* = one pass of the hot path (STFT -> 100 EM iterations of MH E-step + NMF M-step -> Wiener -> ISTFT) over
one batch of synthetic 3 s utterances.  Headline workload at every N: BASELINE.json configs[1] per GPU ("M1 batch of 512
synthetic utterances on 1 B200"), i.e. weak scaling with 512 distinct utterances per rank and no data-path collective;
NCCL only gathers per-utterance metrics (SI-SDR, final cost) and the max-over-ranks time.  The same JSON line carries
``extra_configs``: BASELINE configs[2] (M2, 4 096 utterances in total split over the ranks: strong scaling) and, on 8 GPUs,
configs[3] (M2-info / MCEM_M2v3, 4 096 utterances x 16 chains), each with its own ms_per_step, roofline and e2e.

Printed JSON line (rank 0): `value` times the device-resident path with CUDA events; `e2e` times the public host API
(`dvae_b200.engine.Enhancer.enhance`: pinned host buffers in, host arrays out, copies inside the timed region);
`roofline` describes the dominant kernel (the Metropolis-Hastings sampler) from CUDA events recorded around it
inside the timed region; `cpu_baseline` is the CPU oracle port (the reference's algorithm, torch CPU ops) on the same
workload in two host layouts - one utterance on all threads, and one single-threaded process per core (the reference's
own layout) - with `value` the better of the two.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (rank 0's shard of the headline workload)
as `DIR/<name>.npy`, see `dump_outputs`.  Inputs, weights and the sampler's seed depend only on the arguments, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from dvae_b200 import synth  # noqa: E402

METRIC = "enhanced_audio_seconds_per_second"
UNIT = "audio-s/s"
SECONDS = 3.0
DEC_FLOP_PER_ROW = {("M1", 16): 168192, ("M2", 16): 168448, ("M2v3", 16): 168448}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="utterances per GPU")
    ap.add_argument("--niter", type=int, default=100)
    ap.add_argument("--variant", default="M1", choices=["M1", "M2", "M2v3"])
    ap.add_argument("--sampler", default=os.environ.get("DVAE_SAMPLER", "tc"), choices=["fp32", "tc"])
    ap.add_argument("--chains", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_configs blocks (BASELINE configs[2], configs[3])")
    ap.add_argument("--config3", action="store_true", help="run the configs[3] block at any GPU count (512 utterances x 16 chains per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline workload's outputs of the last timed step as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def measured_traffic(B, variant):
    """DRAM bytes of one sampler launch from the committed ncu capture, when one exists for this workload."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_tc_traffic.json")
    try:
        t = json.load(open(path))
    except (OSError, ValueError):
        return None
    if t.get("utterances_per_gpu") == B and t.get("variant") == variant:
        return t.get("dram_bytes_per_launch")
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tensor=1590.0, src="fallback")


def model_weights(variant, prior_bias):
    y_dim = 0 if variant == "M1" else 1
    return synth.xavier_state_dict(variant, 513, 16, [128, 128], y_dim, seed=1234, out_bias=prior_bias)


def schedule(variant, niter):
    from dvae_b200.engine import McemConfig
    if variant == "M1":      # the reference's effective M1 schedule (SURVEY Q1): 60 iterations keep 30; 105 keep 75
        return dict(niter=niter, keep_E=30, burn_E=30, keep_WF=75, burn_WF=30)
    return dict(niter=niter, keep_E=10, burn_E=30, keep_WF=25, burn_WF=75)


# ------------------------------------------------------------------------------------------------ reference arm / CPU baseline
def cpu_reference_run(variant, niter, u):
    """One utterance through the CPU oracle port exactly like ``process_utt`` (scripts/evaluate_ntcd_M1.py:81-188)."""
    from oracle import mcem_port, stft_np
    kw = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
    x, s, _ = synth.synth_utterance(u, SECONDS)
    t0 = time.perf_counter()
    X = stft_np.stft(x, **kw)
    S = stft_np.stft(s, **kw)
    sd = model_weights(variant, reference_power())
    y = synth.energy_vad(s) if variant != "M1" else None
    o = mcem_port.MCEMOracle(variant, niter, 10, 30, 25, 75, 0.01)
    o.init_parameters(X, S, sd, 10, 1e-8, y=y)
    o.run()
    ikw = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, max_len=len(x))
    stft_np.istft(o.S_hat, **ikw)
    stft_np.istft(o.N_hat, **ikw)
    return time.perf_counter() - t0


def _cpu_worker(variant, niter, u, barrier, queue):
    """One single-threaded worker of the process-per-core layout (the reference's own: scripts/evaluate_ntcd_M1.py:249-259
    spawns one process per slot and hands each a sublist of files)."""
    torch.set_num_threads(1)
    torch.manual_seed(u)
    cpu_reference_run(variant, max(1, niter // 20), u)                      # warm-up (imports, caches)
    barrier.wait(timeout=600)
    t0 = time.time()
    cpu_reference_run(variant, niter, u)
    queue.put((t0, time.time()))


def cpu_process_per_core(variant, niter, n_proc, u0=200):
    """``n_proc`` utterances at once, one single-threaded process each: ``(audio-s/s, wall seconds of the round)``."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    barrier, queue = ctx.Barrier(n_proc), ctx.Queue()
    procs = [ctx.Process(target=_cpu_worker, args=(variant, niter, u0 + i, barrier, queue)) for i in range(n_proc)]
    for pr in procs:
        pr.start()
    import queue as _queue
    spans, deadline = [], time.time() + 900
    try:
        while len(spans) < n_proc:
            try:
                spans.append(queue.get(timeout=2))
            except _queue.Empty:
                if any(pr.exitcode not in (None, 0) for pr in procs):
                    raise RuntimeError("a CPU worker exited with an error")
                if time.time() > deadline:
                    raise RuntimeError("CPU workers did not finish within 900 s")
    finally:
        for pr in procs:
            pr.join(timeout=5)
            if pr.is_alive():
                pr.terminate()
    wall = max(e for _, e in spans) - min(b for b, _ in spans)
    return n_proc * SECONDS / wall, wall


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_baseline_block(variant, niter, t_all_threads, cores, what):
    """The CPU side of the comparison in both layouts the host offers: one utterance on all threads (``t_all_threads`` seconds,
    measured by the caller) and one single-threaded process per core; ``value`` is the better of the two."""
    v_seq = SECONDS / t_all_threads
    layouts = {"one_utterance_all_threads": dict(value=v_seq, seconds_per_utterance=t_all_threads, threads=cores)}
    try:
        v_par, wall = cpu_process_per_core(variant, niter, cores)
    except Exception as e:                                              # a host that cannot spawn workers still gets a bench line
        sample = "%s; the process-per-core layout could not be measured here (%s: %s)" % (what, type(e).__name__, e)
        return dict(value=v_seq, unit=UNIT, cores=cores, kind="port", sample=sample, layouts=layouts, cpu_model=cpu_model())
    layouts["process_per_core"] = dict(value=v_par, processes=cores, threads_each=1, wall_seconds=wall)
    best = "process_per_core" if v_par >= v_seq else "one_utterance_all_threads"
    sample = ("%s; process-per-core layout (the reference's own, evaluate_ntcd_M1.py:249-259): %d utterances at once, one "
              "single-threaded process each, %.1f s; value = the better layout (%s)" % (what, cores, wall, best))
    return dict(value=max(v_seq, v_par), unit=UNIT, cores=cores, kind="port", sample=sample, layouts=layouts, cpu_model=cpu_model())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    for i in range(args.warmup):
        cpu_reference_run(args.variant, max(1, args.niter // 20), i)       # warm-up: short runs (thread pools, caches)
    times = [cpu_reference_run(args.variant, args.niter, 100 + i) for i in range(args.steps)]
    t = statistics.median(times)
    cpu = cpu_baseline_block(args.variant, args.niter, t, cores,
                             "%d steps of 1 utterance (3 s, %d EM iterations) on all %d host threads, median %.1f s" %
                             (args.steps, args.niter, cores, t))
    value = cpu["value"]
    out = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
               ms_per_step=SECONDS / value * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
               data="synthetic", impl="reference",
               config=dict(workload="%s MCEM enhancement, synthetic 3 s 16 kHz utterances, STFT 1024/256, NMF rank 10, "
                                    "%d EM iterations (BASELINE.json configs[1] workload; a step = one utterance; ms_per_step = "
                                    "host time per utterance in the better of the two CPU layouts)" % (args.variant, args.niter)),
               cpu_baseline=cpu,
               e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
               gpu_launches=0)
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [c.strip() for c in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=(statistics.median(sm) if sm else None), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------ B200 arm
# MUFU lane-operations the sampler needs per decoder row (SURVEY section 8d "MUFU ~ 1 795 / row" is the FP32 count; the
# tcgen05 sampler shares reciprocals / logarithms between four bins and takes half of the exponentials from a polynomial):
# 2 x 128 / 2 packed tanh + 528 x (0.5 ex2 + 0.25 rcp + 0.25 lg2)
MUFU_PER_ROW = 128 + 528
XU_LANES_PER_CLK_SM = 16


def synth_set(u0, count, seconds=SECONDS, threads=16):
    """``count`` distinct synthetic utterances with global ids u0 .. : ``(x, s)`` lists (threads: numpy releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max(1, min(threads, os.cpu_count() or 1))) as pool:
        trip = list(pool.map(lambda u: synth.synth_utterance(u, seconds), range(u0, u0 + count)))
    return [t[0] for t in trip], [t[1] for t in trip]


DUMP_BYTES = 64 << 20
DUMP_UTTERANCES = 128


def dump_outputs(path, s_dev, n_dev, cost, utt_ids, T):
    """Write what ``Enhancer.run_device`` returned: ``cost.npy`` the cost of every EM iteration and utterance ``[niter][B]``
    (float64, complete), ``s_hat.npy`` / ``n_hat.npy`` the speech / noise estimates ``[k][T]`` (float32) of a fixed sample of
    k <= 128 utterances (seed 0, in batch order) and ``utterance_ids.npy`` their global ids (float64): 64 MB at most."""
    B = len(utt_ids)
    cost_h = cost.to(torch.float64).cpu().numpy()
    k = int(min(B, DUMP_UTTERANCES, max(1, (DUMP_BYTES - cost_h.nbytes) // (2 * 4 * T + 8))))
    pick = np.sort(np.random.default_rng(0).choice(B, size=k, replace=False))
    idx = torch.from_numpy(pick).to(s_dev.device)
    out = dict(cost=cost_h,
               s_hat=s_dev.view(B, T).index_select(0, idx).cpu().numpy(),
               n_hat=n_dev.view(B, T).index_select(0, idx).cpu().numpy(),
               utterance_ids=np.asarray(utt_ids, np.float64)[pick])
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def measure(variant, n_total, chains, steps, warmup, want_e2e, scaling, niter, sampler, rank, world, dev, label, dump_dir=None):
    """One workload on this rank's shard; returns the JSON block (rank 0) or None.

    ``scaling`` "weak": ``n_total`` utterances PER RANK; "strong": ``n_total`` utterances split over the ranks with
    ``shard_range`` (the reference's np.array_split over processes, scripts/evaluate_ntcd_M2.py:298-327).
    """
    import torch.distributed as dist
    from dvae_b200.engine import Enhancer, McemConfig, RaggedBatch
    from dvae_b200.packages.metrics import energy_ratios_batch
    from dvae_b200.packages.processing.target import vad_batch
    from dvae_b200.shard import gather_metrics, max_over_ranks, shard_range

    if scaling == "weak":
        lo, hi, n_all = rank * n_total, (rank + 1) * n_total, world * n_total
    else:
        lo, hi = shard_range(n_total, rank, world)
        n_all = n_total
    B = hi - lo
    T = int(SECONDS * synth.FS)
    x_host, s_host = synth_set(1000 + lo, B)                     # every utterance distinct, global ids lo .. hi
    sd = model_weights(variant, reference_power())
    cfg = McemConfig(var_rw=0.01, nmf_rank=10, eps=1e-8, n_chains=chains, seed=2024, sampler=sampler, **schedule(variant, niter))
    enh = Enhancer(sd, variant, cfg, device=dev.index)
    eng = enh.engine
    utt_ids = list(range(lo, hi))
    nfr = [synth.num_frames(T)] * B
    batch = RaggedBatch(nfr, dev, utt_ids)
    x_dev = torch.from_numpy(np.stack(x_host)).to(dev).reshape(-1)
    s_clean = torch.from_numpy(np.stack(s_host)).to(dev).reshape(-1)
    x_off = (torch.arange(B, dtype=torch.int64) * T).to(dev)
    x_len = torch.full((B,), T, dtype=torch.int32, device=dev)
    y_dev = y_host = None
    if variant != "M1":                                         # speech-activity labels of the clean signal (target.py:5-56), on the device
        y_dev = vad_batch(s_clean, x_off, x_len, batch).view(batch.NT, 1)
        yh = y_dev.view(B, -1).cpu().numpy()
        y_host = [yh[u][None, :] for u in range(B)]

    def step_device():
        return enh.run_device(x_dev, x_off, x_len, batch, y_dev, B * T, T)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step_device()
    barrier()
    sampler_clk = ClockSampler(dev.index)
    if rank == 0:
        sampler_clk.start()
    eng.timing = True
    eng._events = []
    eng.kernel_launches = 0
    eng.mh_rows = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        s_dev, n_dev, cost = step_device()
    e1.record()
    barrier()
    clocks = sampler_clk.stop() if rank == 0 else None
    ms_total = max_over_ranks(e0.elapsed_time(e1), dev)
    stages = eng.stage_times_ms()
    launches = eng.kernel_launches
    mh_rows = eng.mh_rows
    eng.timing = False
    from dvae_b200 import tc
    tc.check_status(eng)
    value = n_all * SECONDS * steps / (ms_total * 1e-3)
    if dump_dir and rank == 0:                                  # before the e2e block reuses the output buffers
        dump_outputs(dump_dir, s_dev, n_dev, cost, utt_ids, T)

    # the path's only collective: per-utterance SI-SDR (packages/metrics.py:62-82, computed on the device) and final cost.
    # The first and last window of every utterance are left out: with center=False the overlap-add normalisation divides the
    # first samples by a window sum down to 1e-10 (stft.py:89-95, librosa's rule), which blows a filtered spectrogram up there;
    # the reference's evaluation only sees those samples after the 16-bit wav round trip has clipped them.
    m_off, m_len = x_off + 1024, x_len - 2048
    sdr_out = energy_ratios_batch(s_dev, s_clean, None, m_off, m_len)[:, 0]
    sdr_in = energy_ratios_batch(x_dev, s_clean, None, m_off, m_len)[:, 0]
    local = torch.stack([sdr_out, sdr_in, cost[-1].to(torch.float64)], dim=1)
    allm = gather_metrics(local, n_all)

    e2e = None
    if want_e2e:                                                # public host API: pinned host buffers in, host arrays out
        for _ in range(2 if steps > 1 else 1):                  # warm the pinned staging / result buffers
            res = enh.enhance(x_host, y_host, utt_ids=utt_ids)
        del res
        barrier()
        t0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        n_e2e = max(1, min(steps, 2))
        for _ in range(n_e2e):
            res = enh.enhance(x_host, y_host, utt_ids=utt_ids)
        g1.record()
        barrier()
        wall = max_over_ranks(max(time.perf_counter() - t0, g0.elapsed_time(g1) * 1e-3), dev)
        e2e = dict(value=n_all * SECONDS * n_e2e / wall, unit=UNIT, h2d_bytes_per_step=int(enh.h2d_bytes),
                   d2h_bytes_per_step=int(enh.d2h_bytes), steps=n_e2e)
        del res
    vs_bytes = (eng.VsT.numel() if getattr(eng, "VsT", None) is not None else eng.Vs_flat.numel() * 4)
    del enh, eng
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    pk = peaks()
    flop_row = DEC_FLOP_PER_ROW[(variant, 16)]
    # the sampler kernel itself (events around the dvae_mh_chain_tc2 launch); "mh" additionally holds the P / Vb packing
    mh_ms, mh_calls = stages.get("mh_kernel", stages.get("mh", (0.0, 0)))
    roof = None
    if mh_calls:
        flops_per_call = flop_row * mh_rows / mh_calls                       # algorithmic: one decoder row per proposal
        achieved = flops_per_call / (mh_ms / mh_calls * 1e-3) / 1e12
        sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        xu_peak = XU_LANES_PER_CLK_SM * 148 * sm_hz                          # MUFU lane-operations per second at the clocks seen
        xu_rate = MUFU_PER_ROW * mh_rows / (mh_ms * 1e-3)
        roof = dict(kernel="mh2_kernel (dvae_mh_chain_tc2)", bound="tensor", achieved=achieved, peak=pk["tensor"], unit="TFLOP/s",
                    frac=achieved / pk["tensor"], xu_frac=xu_rate / xu_peak, traffic=measured_traffic(B, variant), peak_source=pk["src"],
                    share_of_step=mh_ms / ms_total, launches_per_step=mh_calls / steps,
                    note="sampler time = CUDA events around dvae_mh_chain_tc2 inside the timed region; FLOPs = %d per decoder row x rows "
                         "(one row per proposal); xu_frac = %d MUFU lane-operations per row against 16 lanes per clock and SM at the SM "
                         "clock seen; traffic = dram read+write bytes of one E-step launch from ncu (profiles/r02_tc_traffic.json), null "
                         "if no capture matches this batch" % (flop_row, MUFU_PER_ROW))
    m = allm.cpu().numpy()
    return dict(workload=label, value=value, unit=UNIT, ms_per_step=ms_total / steps, steps=steps, warmup=warmup, scaling=scaling,
                utterances_total=n_all, utterances_this_rank=B, variant=variant, chains=chains, sampler=sampler,
                schedule=schedule(variant, niter), clocks=clocks, e2e=e2e, gpu_launches=int(launches), roofline=roof,
                stage_share={k: round(v[0] / ms_total, 4) for k, v in stages.items()},
                si_sdr_db=dict(mean_out=float(m[:, 0].mean()), mean_in=float(m[:, 1].mean()),
                               mean_improvement=float((m[:, 0] - m[:, 1]).mean()), n=int(m.shape[0])),
                mean_final_cost=float(m[:, 2].mean()), kept_sample_bytes=int(vs_bytes))


def oracle_si_sdr_delta(variant, niter, u=1000):
    """|SI-SDR(GPU, sampler="tc") - SI-SDR(CPU oracle)| in dB for one utterance of the workload, both fed the SAME random draws
    (torch's CPU generator in the reference's consumption order).  Returns (delta, oracle seconds)."""
    from dvae_b200.packages.models import mcem as shim_mcem
    from dvae_b200.packages.models import models as shim_models
    from dvae_b200.packages.processing.stft import istft
    from oracle import mcem_port, stft_np
    kw = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False, pad_at_end=True)
    ikw = dict(fs=16000, wlen_sec=64e-3, win="hann", hop_percent=0.25, center=False)
    x, s, _ = synth.synth_utterance(u, SECONDS)
    sd = model_weights(variant, reference_power())
    y = synth.energy_vad(s) if variant != "M1" else None
    t0 = time.perf_counter()
    X, S = stft_np.stft(x, **kw), stft_np.stft(s, **kw)
    torch.manual_seed(4321)
    o = mcem_port.MCEMOracle(variant, niter, 10, 30, 25, 75, 0.01)
    o.init_parameters(X, S, sd, 10, 1e-8, y=y)
    o.run()
    s_ref = stft_np.istft(o.S_hat, max_len=len(x), **ikw)
    stft_np.istft(o.N_hat, max_len=len(x), **ikw)
    t_cpu = time.perf_counter() - t0
    if variant == "M1":
        model = shim_models.VariationalAutoencoder([513, 16, [128, 128]])
        cls = shim_mcem.MCEM_M1
    else:
        model = shim_models.DeepGenerativeModel([513, 1, 16, [128, 128]], None) if variant == "M2" else shim_models.DeepGenerativeModel_v3([513, 1, 16, [128, 128]])
        cls = shim_mcem.MCEM_M2 if variant == "M2" else shim_mcem.MCEM_M2v3
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()}, strict=False)
    model.to("cuda:%d" % torch.cuda.current_device()).eval()
    algo = cls(niter, 10, 30, 25, 75, 0.01, rng="torch", sampler="tc")
    torch.manual_seed(4321)
    args = dict(X=X, S=S, vae=model, nmf_rank=10, eps=1e-8, device=torch.cuda.current_device())
    if variant != "M1":
        args["y"] = torch.tensor(y, device="cuda:%d" % torch.cuda.current_device())
    algo.init_parameters(**args)
    algo.run()
    s_gpu = istft(algo.S_hat, max_len=len(x), **ikw)
    a, b = mcem_port.si_sdr(s_gpu[800:-800], s[800:-800]), mcem_port.si_sdr(s_ref[800:-800], s[800:-800])
    return abs(a - b), b, t_cpu


def run_b200(args):
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its debug output (the version banner at NCCL_DEBUG=VERSION / WARN / INFO) to STDOUT by default: send it
        # to stderr so that stdout carries exactly the one JSON line
        # (NCCL honours NCCL_DEBUG_FILE only above the VERSION level, so VERSION / unset becomes WARN)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B = args.batch

    headline = (args.variant == "M1" and B == 512 and args.chains == 1)
    cfg_name = "BASELINE.json configs[1]" if headline else \
        "BASELINE.json configs[%d] shape (%s, %d utterances per GPU)" % (2 if args.variant == "M2" else (3 if args.variant == "M2v3" else 1), args.variant, B)
    label = cfg_name + ": %s batch of %d synthetic 3 s 16 kHz utterances per GPU (all distinct), STFT 1024/256, NMF rank 10, %d EM iterations" % (
        args.variant, B, args.niter)
    main = measure(args.variant, B, args.chains, args.steps, args.warmup, not args.no_e2e, "weak", args.niter, args.sampler, rank, world, dev, label,
                   dump_dir=args.dump_outputs)

    extra = []
    if headline and not args.no_extra:
        # configs[2]: M2, 4 096 utterances sharded over the ranks (strong scaling, scripts/evaluate_ntcd_M2.py:298-327)
        blk = measure("M2", 4096, 1, min(args.steps, 3), 1, not args.no_e2e, "strong", args.niter, args.sampler, rank, world, dev,
                      "BASELINE.json configs[2]: M2 speech-activity-conditioned VAE, 4 096 synthetic 3 s utterances in total, sharded over "
                      "%d GPU(s) with shard_range" % world)
        if blk:
            extra.append(blk)
        if world == 8 or args.config3:
            # configs[3]: M2-info weights layout (enc_dec_clf of DeepGenerativeModel_v5 = MCEM_M2v3), 4 096 utterances x 16 chains
            blk = measure("M2v3", 4096 if world == 8 else 512 * world, 16, 1, 1, False, "strong", args.niter, args.sampler, rank, world, dev,
                          "BASELINE.json configs[3]: M2-info (MCEM_M2v3) with visual-VAD-style label input, %d utterances x 16 MH chains "
                          "sharded over %d GPU(s)" % (4096 if world == 8 else 512 * world, world))
            if blk:
                extra.append(blk)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        cpu_reference_run(args.variant, max(1, args.niter // 20), 0)
        delta, sdr_ref, t_cpu = oracle_si_sdr_delta(args.variant, args.niter, 1000)
        cpu = cpu_baseline_block(args.variant, args.niter, t_cpu, cores,
                                 "1 of the %d utterances (3 s, %d EM iterations) through oracle.mcem_port on %d host threads: %.1f s" %
                                 (B, args.niter, cores, t_cpu))
        parity = dict(si_sdr_delta_db=delta, oracle_si_sdr_db=sdr_ref,
                      how="the CPU oracle run of cpu_baseline and the GPU path (sampler=tc, reference-signature MCEM shim) on the same "
                          "utterance and the same torch CPU draws (seed 4321); north star: within 0.05 dB")

    out = dict(metric=METRIC, value=main["value"], unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
               ms_per_step=main["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None,
               dtype="f32" if args.sampler == "fp32" else "bf16", data="synthetic",
               config=dict(workload=main["workload"] + ", MH schedule %s" % main["schedule"], utterances_per_gpu=B, sampler=args.sampler,
                           chains=args.chains,
                           l2="working set per EM iteration (kept-sample variances %.1f GB) exceeds the 126 MB L2; no explicit flush" %
                              (main["kept_sample_bytes"] / 1e9),
                           parallelism="utterance shards, %d rank(s), no data-path collective" % world),
               clocks=main["clocks"], e2e=main["e2e"], gpu_launches=main["gpu_launches"], roofline=main["roofline"], cpu_baseline=cpu,
               stage_share=main["stage_share"], mean_final_cost=main["mean_final_cost"], si_sdr_db=main["si_sdr_db"], parity=parity,
               extra_configs=extra)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def reference_power():
    """Decoder output bias shared by both arms: log of the mean clean-speech power spectrum of synthetic utterance 1000
    (random weights around it act as a crude speech prior, so the Wiener filter does real work).  The prior carries that
    utterance's harmonics: utterance 1000 is genuinely enhanced (the `parity` block compares its SI-SDR with the oracle's),
    the other utterances of the batch have other pitches, and with untrained weights their SI-SDR (gathered in `si_sdr_db`)
    is a payload for the metric path, not a quality claim (a pitch-independent envelope prior was tried: the rank-10 NMF
    then explains the stationary synthetic harmonics as noise for every utterance)."""
    _, s, _ = synth.synth_utterance(1000, SECONDS)
    return synth.speech_prior_bias(s)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
