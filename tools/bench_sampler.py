#!/usr/bin/env python
"""Time the tcgen05 sampler alone (one E-step call) with / without in-kernel Philox and with / without the emission of the kept
samples' variances; also the frame-statistics and M-step kernels on the emission.  python tools/bench_sampler.py [B] [variant]"""
import ctypes as C
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import bench  # noqa: E402
from dvae_b200 import _lib, synth, tc  # noqa: E402
from dvae_b200.engine import Enhancer, McemConfig, RaggedBatch, _p, _stream  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 512
variant = sys.argv[2] if len(sys.argv) > 2 else "M1"
dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
T = int(3.0 * synth.FS)
base_x, base_s = synth.synth_batch(1000, min(B, 32), 3.0)
x_host = [base_x[i % len(base_x)] for i in range(B)]
y_host = [synth.energy_vad(base_s[i % len(base_s)]) for i in range(B)] if variant != "M1" else None
sd = bench.model_weights(variant, bench.reference_power())
cfg = McemConfig(var_rw=0.01, nmf_rank=10, eps=1e-8, seed=2024, sampler="tc", **bench.schedule(variant, 3))
enh = Enhancer(sd, variant, cfg, device=0)
eng = enh.engine
nfr = [synth.num_frames(T)] * B
batch = RaggedBatch(nfr, dev, list(range(B)))
x_dev = torch.from_numpy(np.stack(x_host)).to(dev).reshape(-1)
x_off = (torch.arange(B, dtype=torch.int64) * T).to(dev)
x_len = torch.full((B,), T, dtype=torch.int32, device=dev)
y_dev = None if y_host is None else torch.from_numpy(np.ascontiguousarray(np.concatenate([y.T for y in y_host], 0))).to(dev)
enh.run_device(x_dev, x_off, x_len, batch, y_dev, B * T, T)          # warm: a short run leaves realistic W, H, g, Z
keep, burn = cfg.keep_E, cfg.burn_E
NT, L = batch.NT, eng.w.z_dim


def timed(fn, n=5):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


class Inj:
    def __init__(self):
        rng = _lib.DvaeRng()
        rng.seed, rng.iter0 = 1, 0
        self.eps = torch.empty((keep + burn, NT, L), device=dev)
        self.u = torch.empty((keep + burn, NT), device=dev)
        _lib.call("dvae_rng_dump", C.byref(rng), _p(batch.frame_gid), _p(batch.frame_idx), NT, 1, L, keep + burn, _p(self.eps), _p(self.u), _stream())

    def mh_draws(self, call, n_iter, chains, L_):
        return self.eps, self.u


inj = Inj()
out = {}
for name, draws, emit in (("philox+emit", None, True), ("philox", None, False), ("injected+emit", inj, True), ("injected", inj, False)):
    eng.timing = True
    eng._events = []
    timed(lambda: eng.sample_posterior(keep, burn, draws, emit=emit))
    st = eng.stage_times_ms()
    out[name] = st["mh_kernel"][0] / st["mh_kernel"][1]
# A/B against the round-1 sampler when it is compiled in (csrc/zz_ab_mh_r1.cu, not part of the repository)
lib = _lib.load()
if hasattr(lib, "dvae_mh_chain_tc2_r1"):
    fn = lib.dvae_mh_chain_tc2_r1
    fn.restype = C.c_int
    fn.argtypes = [C.POINTER(_lib.DvaeMlp)] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                   C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    w = eng.w
    img = tc.decoder_image(w)
    pv = eng._get("PVpk", (max(int(lib.dvae_tc_packed_pv_bytes(NT)), 16),), torch.uint8)
    Zs = eng._get("Zs%d" % keep, (NT, keep, L))
    st = tc._status(eng)

    def old():
        rc = fn(w.dec.ref, _p(img), _p(pv), _p(eng.g), _p(eng.y), w.y_dim, _p(eng.Z), _p(Zs), NT, L, 1, burn, keep, 0.01, _p(inj.eps), _p(inj.u),
                _p(eng.n_accept), None, int(w._tc_flags), _p(st), _stream())
        assert rc == 0
    out["round-1 kernel (injected)"] = timed(old)
# variants of the current sampler compiled under other names (csrc/zz_ab_v*.cu, not part of the repository)
eng.sample_posterior(keep, burn, None, emit=True)          # (re)creates the emission buffers the variants write to
for tag in "BCDEFG":
    name = "dvae_mh_chain_tc2_v" + tag
    if not hasattr(lib, name):
        continue
    fv = getattr(lib, name)
    fv.restype, fv.argtypes = _lib.PROTOTYPES["dvae_mh_chain_tc2"]
    w = eng.w
    img = tc.decoder_image(w)
    pv = eng._get("PVpk", (max(int(lib.dvae_tc_packed_pv_bytes(NT)), 16),), torch.uint8)
    Zs = eng._get("Zs%d" % keep, (NT, keep, L))
    st = tc._status(eng)
    for mode in ("philox", "philox+emit"):
        rng = _lib.DvaeRng()
        rng.seed, rng.iter0 = 1, 0
        if mode == "injected":
            rng.eps, rng.u = inj.eps.data_ptr(), inj.u.data_ptr()

        def var():
            rc = fv(w.dec.ref, _p(img), _p(pv), _p(eng.kscale), _p(eng.g), _p(eng.y), w.y_dim, None, _p(batch.frame_gid), _p(batch.frame_idx), _p(eng.Z), _p(Zs), NT, L,
                    1, burn, keep, 0.01, C.byref(rng), _p(eng.n_accept), None, _p(eng.VsT) if "emit" in mode else None,
                    _p(eng.vs_idx) if "emit" in mode else None, int(w._tc_flags), _p(st), _stream())
            assert rc == 0
        out["v%s %s" % (tag, mode)] = timed(var)
eng.timing = False
eng.sample_posterior(keep, burn, None, emit=True)
eng.R = keep
out["frame_stats"] = timed(lambda: tc.vst_frame_stats(eng, keep))
out["w_partials"] = timed(lambda: tc.vst_w_partials(eng, keep))
eng.wstat, eng.wpart = None, tc.vst_w_partials(eng, keep)
eng.timing = True
eng._events = []
timed(lambda: eng.m_step(0))
out["m_step"] = eng.stage_times_ms()["mstep"][0] / 6
tc.check_status(eng)
# the same kernels inside a realistic loop (E-step + M-step, 30 EM iterations back to back)
eng.timing = True
eng._events = []
for it in range(30):
    eng.e_step()
    eng.m_step(it % cfg.niter)
st = eng.stage_times_ms()
out["loop: sampler"] = st["mh_kernel"][0] / st["mh_kernel"][1]
out["loop: stats"] = st["decode"][0] / st["decode"][1]
out["loop: m_step"] = st["mstep"][0] / st["mstep"][1]
eng.timing = False
tc.check_status(eng)
rows = NT * (keep + burn + 1)
print({k: round(v, 3) for k, v in out.items()}, "ms;  sampler TFLOP/s (philox+emit): %.0f" % (168192.0 * rows / out["philox+emit"] / 1e9))
