"""Batched MCEM VAE-NMF enhancement engine: Python/PyTorch host code over libdvae_b200's C ABI.

PyTorch is plumbing here (device memory, streams); every arithmetic step of the path is a CUDA kernel of
``libdvae_b200.so`` reached through ``dvae_b200._lib``.  The engine processes a *ragged batch* of utterances at once
(the reference handles one utterance per process, ``scripts/evaluate_ntcd_M1.py:190-214``):

    STFT -> |X|^2 -> encoder mean (chain start) -> niter x [ MH E-step -> decode kept samples -> M-step (W,H,g,cost) ]
         -> long MH chain -> Wiener masks -> S_hat, N_hat -> ISTFT

Reference behaviour reproduced (SURVEY §3.2): chain start = encoder posterior MEAN (``_, Z, _ = encoder(..)``,
mcem.py:200); Vb kept un-normalised after the W/H renormalisation (Q4); per-variant MH schedules incl. the M1
argument shift (Q1, applied by the ``MCEM_M1`` shim, the engine takes explicit ``(keep, burn)`` pairs).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math
import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .synth import FS, HOP, N_FFT, num_frames

LD_ALIGN = 8
ORACLE_LABELS = ("vad", "ibm", "robust_ibm")       # labels Enhancer.enhance derives from the clean speech (oracle_labels=)


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _on_device(fn):
    """Run a method with the object's CUDA device current: the kernels of libdvae_b200 launch on the calling thread's current
    device and ``_stream()`` is that device's current stream, while the reference's scripts hand a device INDEX to every
    worker and never call ``set_device`` (scripts/evaluate_ntcd_M1.py:69,252)."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **kw):
        with torch.cuda.device(self.dev):
            return fn(self, *a, **kw)
    return wrapper


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise _lib.DvaeError("dvae_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    _lib.load()
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    if dev.type != "cuda":
        raise _lib.DvaeError("dvae_b200 runs on CUDA devices only (got %r)" % (device,))
    return dev


# --------------------------------------------------------------------------------------------- weights
class PackedMlp:
    """Transposed FP32 weights of a tanh MLP on the device + the host-side ``DvaeMlp`` struct that points at them."""

    def __init__(self, layers: Sequence[tuple], device):
        if not 1 <= len(layers) <= _lib.MAX_LAYERS:
            raise ValueError("an MLP needs 1..%d linear layers" % _lib.MAX_LAYERS)
        self.wt, self.bias, dims = [], [], []
        for w, b in layers:
            w = torch.as_tensor(np.asarray(w) if not torch.is_tensor(w) else w).detach().to(torch.float32)
            b = torch.as_tensor(np.asarray(b) if not torch.is_tensor(b) else b).detach().to(torch.float32)
            if dims and dims[-1] != w.shape[1]:
                raise ValueError("layer input %d does not match previous output %d" % (w.shape[1], dims[-1]))
            if not dims:
                dims.append(int(w.shape[1]))
            dims.append(int(w.shape[0]))
            self.wt.append(w.t().contiguous().to(device))
            self.bias.append(b.contiguous().to(device))
        self.dims = dims
        self.struct = _lib.DvaeMlp()
        self.struct.n_layers = len(layers)
        for i, d in enumerate(dims):
            self.struct.dims[i] = d
        for i in range(len(layers)):
            self.struct.wt[i] = self.wt[i].data_ptr()
            self.struct.bias[i] = self.bias[i].data_ptr()

    @property
    def ref(self):
        return C.byref(self.struct)

    @property
    def in_dim(self):
        return self.dims[0]

    @property
    def out_dim(self):
        return self.dims[-1]


def _sd_get(sd, key):
    v = sd[key]
    return v.detach().cpu() if torch.is_tensor(v) else torch.as_tensor(np.asarray(v))


class VaeWeights:
    """Device copies of one VAE's encoder / decoder in the layout the kernels want.

    ``sd`` uses the reference's state_dict keys (SURVEY §8a15): ``encoder.hidden.{i}``, ``encoder.sample.{mu,log_var}``,
    ``decoder.hidden.{i}``, ``decoder.reconstruction``.  ``variant``: "M1" | "M2" | "M2v2" | "M2v3".
    """

    def __init__(self, sd, variant: str, device, prefix: str = ""):
        if variant not in ("M1", "M2", "M2v2", "M2v3"):
            raise ValueError("unknown variant %r" % (variant,))
        self.variant = variant
        self.device = device

        def layers(stem):
            out, i = [], 0
            while f"{prefix}{stem}.hidden.{i}.weight" in sd:
                out.append((_sd_get(sd, f"{prefix}{stem}.hidden.{i}.weight"), _sd_get(sd, f"{prefix}{stem}.hidden.{i}.bias")))
                i += 1
            return out

        enc_h = layers("encoder")
        mu = (_sd_get(sd, f"{prefix}encoder.sample.mu.weight"), _sd_get(sd, f"{prefix}encoder.sample.mu.bias"))
        lv = (_sd_get(sd, f"{prefix}encoder.sample.log_var.weight"), _sd_get(sd, f"{prefix}encoder.sample.log_var.bias"))
        self.enc_mu = PackedMlp(enc_h + [mu], device)
        self.enc_lv = PackedMlp(enc_h + [lv], device)
        dec_h = layers("decoder")
        rec = (_sd_get(sd, f"{prefix}decoder.reconstruction.weight"), _sd_get(sd, f"{prefix}decoder.reconstruction.bias"))
        self.dec = PackedMlp(dec_h + [rec], device)
        self.z_dim = int(mu[0].shape[0])
        self.x_dim = self.dec.out_dim
        self.y_dim = self.dec.in_dim - self.z_dim
        # Tensor-core kernels carry at most three labels in their layer-1 operand.  Wider label vectors (the IBM-conditioned
        # M2 model: y_dim = 513, scripts/evaluate_ntcd_M2.py:66-73) are folded into a per-frame layer-1 bias: the decoder is
        # packed without its label columns and without b1, and W1[:, L:] y + b1 is evaluated once per batch (SURVEY 7.3.4).
        self.tc_label_bias = self.y_dim > 3
        if self.tc_label_bias:
            w1, b1 = dec_h[0]
            self.dec_tc = PackedMlp([(w1[:, :self.z_dim], torch.zeros_like(b1))] + dec_h[1:] + [rec], device)
            self.ybias_mlp = PackedMlp([(w1[:, self.z_dim:], b1)], device)
        else:
            self.dec_tc = self.dec
        self.tc_y_dim = 0 if self.tc_label_bias else self.y_dim
        self.enc_takes_y = self.enc_mu.in_dim == self.x_dim + self.y_dim and self.y_dim > 0
        if (variant == "M1") != (self.y_dim == 0):
            raise ValueError("variant %s does not match a decoder with %d label inputs" % (variant, self.y_dim))
        if variant == "M2" and not self.enc_takes_y:
            raise ValueError("M2 expects an encoder over [x; y]")
        if variant in ("M2v2", "M2v3") and self.enc_mu.in_dim != self.x_dim:
            raise ValueError("%s expects an encoder over x only" % variant)


# --------------------------------------------------------------------------------------------- ragged batch
class RaggedBatch:
    """Frame bookkeeping of a batch: prefix offsets and the per-frame index maps the kernels consume."""

    def __init__(self, n_frames: Sequence[int], device, utt_ids: Optional[Sequence[int]] = None):
        n = np.asarray(n_frames, dtype=np.int64)
        if n.ndim != 1 or len(n) == 0 or np.any(n < 0):
            raise ValueError("n_frames must be a non-empty list of non-negative counts")
        self.B = len(n)
        self.n_frames = n
        off = np.zeros(self.B + 1, np.int64)
        np.cumsum(n, out=off[1:])
        self.NT = int(off[-1])
        self.max_frames = int(n.max())
        ids = np.arange(self.B, dtype=np.int32) if utt_ids is None else np.asarray(utt_ids, np.int32)
        if len(ids) != self.B:
            raise ValueError("utt_ids length mismatch")
        self.fr_off_host = off
        self.utt_ids_host = ids
        self.fr_off = torch.from_numpy(off).to(device)
        self.utt_ids = torch.from_numpy(ids).to(device)
        local = np.repeat(np.arange(self.B, dtype=np.int32), n)
        self.frame_utt = torch.from_numpy(local).to(device)
        self.frame_gid = torch.from_numpy(ids[local] if self.NT else np.zeros(0, np.int32)).to(device)
        idx = (np.arange(self.NT, dtype=np.int64) - off[:-1][local]).astype(np.int32) if self.NT else np.zeros(0, np.int32)
        self.frame_idx = torch.from_numpy(idx).to(device)
        self._segments = None
        self._device = device

    def segments(self, tile: int = 128, n_chains: int = 1):
        """Segment tables of the fused W-update reduction (dvae_vst_w_partials): a segment is a maximal run of frames inside
        one ``tile``-frame tile AND one utterance.  Returns device tensors ``(seg_start [S+1] int64, tile_seg [n_tiles+1]
        int32, utt_seg [B+1] int32)`` and ``S``; utterance ``u`` owns the segments ``utt_seg[u] .. utt_seg[u+1]``.  With
        ``n_chains`` chains per frame the axis is the chain row ``frame * n_chains + chain`` (``tile`` rows per tile)."""
        key = (tile, n_chains)
        if self._segments is None or self._segments[0] != key:
            rows, off = self.NT * n_chains, self.fr_off_host * n_chains
            n_tiles = (rows + tile - 1) // tile
            cuts = np.unique(np.concatenate([np.arange(0, n_tiles + 1, dtype=np.int64) * tile, off]))
            cuts = cuts[cuts <= rows]
            if len(cuts) == 0 or cuts[-1] != rows:
                cuts = np.append(cuts, rows)
            S = len(cuts) - 1
            tile_seg = np.searchsorted(cuts[:-1], np.arange(0, n_tiles + 1, dtype=np.int64) * tile, side="left").astype(np.int32)
            utt_seg = np.searchsorted(cuts[:-1], off, side="left").astype(np.int32)
            dev = self._device
            self._segments = (key, (torch.from_numpy(cuts.astype(np.int64)).to(dev), torch.from_numpy(tile_seg).to(dev),
                                    torch.from_numpy(utt_seg).to(dev), S))
        return self._segments[1]


# --------------------------------------------------------------------------------------------- STFT / ISTFT
def _ld_for(F: int) -> int:
    return (F + LD_ALIGN - 1) // LD_ALIGN * LD_ALIGN


def stft_batch(x_flat: torch.Tensor, x_off: torch.Tensor, x_len: torch.Tensor, batch: RaggedBatch, n_fft=N_FFT, hop=HOP,
               want_power=True, ld=None, out=None):
    """STFT of a concatenated float32 device signal -> ``(X [NT][ld] complex64, P [NT][ld] float32 | None)``.  ``ld``: row
    stride in bins (default: ``n_fft / 2 + 1`` rounded up to a multiple of 8; at least ``n_fft / 2 + 1``); ``out``: a
    contiguous complex64 ``[NT][ld]`` tensor to write ``X`` into."""
    ld = _ld_for(n_fft // 2 + 1) if ld is None else int(ld)
    if out is not None and (tuple(out.shape) != (batch.NT, ld) or out.dtype != torch.complex64 or not out.is_contiguous()):
        raise ValueError("out must be a contiguous complex64 tensor [NT][ld=%d]" % ld)
    X = out if out is not None else torch.empty((batch.NT, ld), dtype=torch.complex64, device=x_flat.device)
    P = torch.empty((batch.NT, ld), dtype=torch.float32, device=x_flat.device) if want_power else None
    with torch.cuda.device(x_flat.device):
        _lib.call("dvae_stft_f32", _p(x_flat), _p(x_off), _p(x_len), batch.B, _p(X), _p(P), _p(batch.fr_off), batch.NT,
                  n_fft, hop, ld, _stream())
    return X, P


def istft_batch(X: torch.Tensor, batch: RaggedBatch, y_off: torch.Tensor, y_len: torch.Tensor, total_len: int,
                max_len: int, n_fft=N_FFT, hop=HOP, out: Optional[torch.Tensor] = None):
    """ISTFT of ``X [NT][ld]`` into a concatenated float32 signal of ``total_len`` samples."""
    y = out if out is not None else torch.empty(total_len, dtype=torch.float32, device=X.device)
    with torch.cuda.device(X.device):
        _lib.call("dvae_istft_f32", _p(X), _p(batch.fr_off), batch.B, _p(y), _p(y_off), _p(y_len), int(max_len), n_fft, hop,
                  X.shape[1], _stream())
    return y


def istft_masked_batch(X: torch.Tensor, mask: torch.Tensor, batch: RaggedBatch, y_off: torch.Tensor, y_len: torch.Tensor,
                       total_len: int, max_len: int, mask_scale: float = 1.0, n_fft=N_FFT, hop=HOP,
                       out: Optional[torch.Tensor] = None):
    """ISTFT of ``(mask * mask_scale) * X`` (real ``mask [NT][ld]``): the Wiener filter of mcem.py:176-177 applied while the
    frames are loaded, bit-identical to ``dvae_wiener_apply`` + ``istft_batch`` without materialising the product."""
    if mask.shape != X.shape or mask.dtype != torch.float32 or not mask.is_contiguous():
        raise ValueError("mask must be a contiguous float32 tensor of the spectrum's shape")
    y = out if out is not None else torch.empty(total_len, dtype=torch.float32, device=X.device)
    with torch.cuda.device(X.device):
        _lib.call("dvae_istft_masked_f32", _p(X), _p(mask), float(mask_scale), _p(batch.fr_off), batch.B, _p(y), _p(y_off), _p(y_len),
                  int(max_len), n_fft, hop, X.shape[1], _stream())
    return y


def mlp_forward(mlp: PackedMlp, x: torch.Tensor, act_last: int, x2: Optional[torch.Tensor] = None, x2_row_div: int = 1,
                out: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None):
    """Run a packed tanh MLP on the rows of ``x`` (2-D, last dim contiguous) [+ label columns ``x2``]."""
    rows, k1 = x.shape
    k2 = 0 if x2 is None else x2.shape[1]
    if out is None:
        out = torch.empty((rows, mlp.out_dim), dtype=torch.float32, device=x.device)
    need = _lib.load().dvae_mlp_workspace_floats(mlp.ref, rows)          # a host-side size formula, no device work
    if ws is None or ws.numel() < need:
        ws = torch.empty(max(need, 1), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.call("dvae_mlp_fwd", mlp.ref, _p(x), x.stride(0), k1, _p(x2), 0 if x2 is None else x2.stride(0), k2,
                  max(1, x2_row_div), rows, act_last, _p(out), out.stride(0), _p(ws), _stream())
    return out


# --------------------------------------------------------------------------------------------- MCEM
@dataclasses.dataclass
class McemConfig:
    niter: int = 100
    keep_E: int = 10
    burn_E: int = 30
    keep_WF: int = 25
    burn_WF: int = 75
    var_rw: float = 0.01
    nmf_rank: int = 10
    eps: float = 1e-8
    n_chains: int = 1
    seed: int = 0
    sampler: str = "fp32"        # "fp32": CUDA-core exact mode; "tc": tcgen05 BF16 kernels; "auto": tc when supported
    w_partials: bool = True      # emission route: reduce the W-update sums inside the statistics kernel (no A1 / A2 round trip)
    stop_tol: Optional[float] = None   # per-utterance stopping (check_stop, McemEngine.run); None: every utterance runs niter
    stop_window: int = 10              # EM iterations per window of the stopping test


class InjectedDraws:
    """Random numbers supplied by the caller (parity runs), in the batch layout.

    ``W0 [B][K][F]``, ``H0 [NT][K]`` and, per ``sample_posterior`` call c (0..niter-1 for the E-steps, niter for the
    final filter), ``eps[c]: [n_iter][NT*C][L]`` and ``u[c]: [n_iter][NT*C]``.
    """

    def __init__(self, W0, H0, eps, u):
        self.W0, self.H0, self.eps, self.u = W0, H0, eps, u

    def mh_draws(self, call, n_iter, chains, L):
        return self.eps[call], self.u[call]


class TorchCpuDraws(InjectedDraws):
    """Draws taken from torch's global CPU generator in the reference's consumption order (SURVEY §3.3), for ONE
    utterance: ``rand(F,K)``, ``rand(K,N)``, ``randn(N,L)`` x2 (the two encoder passes, unused), then per MH iteration
    ``randn(L,N)`` and ``rand(N)``.  With the same ``torch.manual_seed`` the reference on ``device='cpu'`` sees the
    very same numbers."""

    def __init__(self, F, K, N, L):
        W0 = torch.rand(F, K)
        H0 = torch.rand(K, N)
        torch.randn(N, L)
        torch.randn(N, L)
        super().__init__(W0.t().contiguous()[None], H0.t().contiguous(), None, None)

    def mh_draws(self, call, n_iter, chains, L):
        eps = torch.empty(n_iter, chains, L)
        u = torch.empty(n_iter, chains)
        for it in range(n_iter):
            eps[it] = torch.randn(L, chains).t()
            u[it] = torch.rand(chains)
        return eps, u


def tc_supported(w: "VaeWeights") -> bool:
    """True when the decoder fits the tcgen05 kernels: 513 bins, 1-2 hidden layers of 128 units, L in {16, 32}; any number of
    label inputs (more than three are folded into a per-frame bias, which needs a hidden layer to add it to)."""
    dims = w.dec.dims
    return dims[-1] == 513 and len(dims) in (3, 4) and all(d == 128 for d in dims[1:-1]) and w.z_dim in (16, 32)


def mcem_route(cfg: McemConfig, F: int) -> tuple:
    """``(e_route, filter_chunk)`` for a resolved ``cfg.sampler`` and ``F`` decoder outputs; no device work.  E-step routes: "emit"
    (the tcgen05 sampler writes the variances, BF16; a frame's chains share a 128-row tile of the M-step kernels), "stats" (FP32
    ``Vs`` + W-update statistics in one decode pass), "decode" (FP32 ``Vs``).  ``filter_chunk``: samples per fused decode of the
    final filter; 0: FP32 decode in frame chunks."""
    tc, c = cfg.sampler == "tc", cfg.n_chains
    if tc and cfg.nmf_rank <= 10 and cfg.keep_E in (10, 30) and F == 513 and (c == 1 or (c <= 128 and c & (c - 1) == 0 and cfg.w_partials)):
        route = "emit"
    elif tc and cfg.nmf_rank <= 10 and c * cfg.keep_E % 10 == 0:
        route = "stats"
    else:
        route = "decode"
    return route, next((k for k in (30, 25, 10) if c * cfg.keep_WF % k == 0), 0) if tc else 0


class McemEngine:
    """EM driver for one ragged batch (replaces ``EM.run`` + ``MCEM_*`` of packages/models/mcem.py).  ``route`` /
    ``filter_chunk`` (``mcem_route``) are plain attributes, not settings: tests override ``route`` to compare two routes."""

    def __init__(self, weights: VaeWeights, cfg: McemConfig, device):
        check_stop(cfg)
        self.dev = _require_cuda(device)
        self.w = weights
        self.cfg = cfg
        if cfg.sampler not in ("fp32", "tc", "auto"):
            raise ValueError("sampler must be 'fp32', 'tc' or 'auto'")
        if cfg.sampler == "auto":            # tensor cores whenever the decoder has the shape the tcgen05 kernels serve
            cfg = dataclasses.replace(cfg, sampler="tc" if tc_supported(weights) else "fp32")
            self.cfg = cfg
        if not 1 <= cfg.nmf_rank <= _lib.MAX_K:
            raise ValueError("nmf_rank must be in 1..%d" % _lib.MAX_K)
        if weights.z_dim > _lib.MAX_L:
            raise ValueError("latent dimension above %d" % _lib.MAX_L)
        self.F = weights.x_dim
        self.ld = _ld_for(self.F)
        self.route, self.filter_chunk = mcem_route(cfg, self.F)
        self._buf = {}
        self.mh_calls = 0
        self.mh_rows = 0             # decoder rows the sampler evaluated (one per chain and MH iteration), all calls
        self.kernel_launches = 0
        self.timing = False          # when True, CUDA events bracket every stage (read with stage_times_ms())
        self._events = []
        self._iter0_frame = None     # per-frame Philox iteration base of the next sample_posterior call (final filter of run)
        self.order = None            # after a run with stopping: slot -> caller's utterance index of the per-frame state
        self.n_iter = None           # after a run: EM iterations of every utterance, caller's order

    class _Stage:
        def __init__(self, eng, name):
            self.eng, self.name = eng, name

        def __enter__(self):
            if self.eng.timing:
                self.t0 = torch.cuda.Event(enable_timing=True)
                self.t1 = torch.cuda.Event(enable_timing=True)
                self.t0.record()

        def __exit__(self, *exc):
            if self.eng.timing:
                self.t1.record()
                self.eng._events.append((self.name, self.t0, self.t1))

    def stage(self, name):
        return McemEngine._Stage(self, name)

    def stage_times_ms(self, reset=True):
        """Sum of device time per stage (ms) and number of bracketed calls, from the recorded CUDA events."""
        torch.cuda.current_stream(self.dev).synchronize()
        out = {}
        for name, t0, t1 in self._events:
            ms, n = out.get(name, (0.0, 0))
            out[name] = (ms + t0.elapsed_time(t1), n + 1)
        if reset:
            self._events = []
        return out

    # -- buffers are cached by (name, shape) so repeated batches of the same geometry do not reallocate
    def _get(self, name, shape, dtype=torch.float32):
        key = (name, tuple(shape), dtype)
        t = self._buf.get(key)
        if t is None:
            for k in [k for k in self._buf if k[0] == name]:
                del self._buf[k]
            t = torch.empty(shape, dtype=dtype, device=self.dev)
            self._buf[key] = t
        return t

    @_on_device
    def init_parameters(self, X: torch.Tensor, P: torch.Tensor, batch: RaggedBatch, y: Optional[torch.Tensor] = None,
                        draws: Optional[InjectedDraws] = None):
        """``EM.init_parameters`` + ``MCEM_*.init_parameters`` (mcem.py:36-58, 195-205, 358-370) for the batch."""
        cfg, w = self.cfg, self.w
        if X.shape != (batch.NT, self.ld) or P.shape != (batch.NT, self.ld):
            raise ValueError("X / P must be [NT][ld=%d]" % self.ld)
        if (w.y_dim > 0) != (y is not None):
            raise ValueError("labels y are required exactly for the M2 variants")
        if y is not None and tuple(y.shape) != (batch.NT, w.y_dim):
            raise ValueError("y must be [NT][y_dim=%d]" % w.y_dim)
        check_counters(batch.max_frames, cfg.n_chains)
        self.batch, self.X, self.P, self.y = batch, X, P, (None if y is None else y.contiguous().float())
        # what the tensor-core kernels see of the labels: the labels themselves (<= 3) or a per-frame layer-1 bias
        self.tc_y, self.ybias, self.kscale = self.y, None, None
        if cfg.sampler == "tc":
            from . import tc
            self.kscale = tc.row_scale(self)
        if cfg.sampler == "tc" and w.tc_label_bias:
            self.tc_y = None
            self.ybias = mlp_forward(w.ybias_mlp, self.y, _lib.ACT_NONE, out=self._get("ybias", (batch.NT, 128)))
        B, NT, K, ld, C_ = batch.B, batch.NT, cfg.nmf_rank, self.ld, cfg.n_chains
        self.W = self._get("W", (B, K, ld))
        self.H = self._get("H", (NT, K))
        self.g = self._get("g", (NT,))
        self.Vb = self._get("Vb", (NT, ld))
        if draws is None:
            _lib.call("dvae_nmf_init", cfg.seed, _p(batch.utt_ids), _p(batch.fr_off), B, NT, self.F, K, ld, cfg.eps,
                      _p(self.W), _p(self.H), _p(self.g), _stream())
        else:
            self.W.zero_()
            self.W[:, :, :self.F] = torch.clamp_min(torch.as_tensor(draws.W0).to(self.dev, torch.float32), cfg.eps)
            self.H.copy_(torch.clamp_min(torch.as_tensor(draws.H0).to(self.dev, torch.float32), cfg.eps))
            self.g.fill_(1.0)
        _lib.call("dvae_nmf_vb", _p(self.W), _p(self.H), _p(batch.frame_utt), NT, self.F, K, ld, _p(self.Vb), _stream())
        # chain start = encoder posterior mean of the noisy power spectrogram (the clean-speech encoding of
        # mcem.py:201 is dead code whose only effect is consuming one randn draw)
        mu = mlp_forward(w.enc_mu, P[:, :self.F], _lib.ACT_NONE, x2=self.y if w.enc_takes_y else None)
        self.Z = self._get("Z", (NT * C_, w.z_dim))
        self.Z.copy_(mu.repeat_interleave(C_, dim=0) if C_ > 1 else mu)
        self.n_accept = self._get("n_accept", (NT * C_,), torch.int32)
        self.n_accept.zero_()
        self.mh_calls = 0
        self.mh_iter0 = 0
        self.VsT = self.vs_idx = self.wstat = self.wpart = None    # the last E-step's emission and W-update statistics
        self._Vs = None
        self._last_Zs = None              # the final filter's samples, from the filter until the next E-step
        self.cost = self._get("cost", (cfg.niter, B), torch.float64)
        self.kernel_launches = 0

    @property
    def Vs_flat(self):
        """Dense FP32 buffer for materialised speech variances: NT * R_E rows, and at least one frame's worth of Wiener
        samples.  Allocated on first use (the tensor-core path with one chain per frame never needs it)."""
        b, cfg = self.batch, self.cfg
        return self._get("Vs", (max(b.NT * cfg.n_chains * cfg.keep_E, cfg.n_chains * cfg.keep_WF), self.ld))

    @property
    @_on_device
    def Vs(self):
        """Speech variances of the last sampled set (the filter's until the next E-step), ``[NT][R][ld]`` FP32: the reference's
        ``self.Vs`` (R,F,N) up to layout.  The filter's samples and the "emit" route's BF16 emission are decoded on demand."""
        if self._Vs is None and self._last_Zs is not None:
            out = torch.zeros((self.batch.NT, self._last_Zs.shape[1], self.ld), dtype=torch.float32, device=self.dev)
            self.decode_samples(self._last_Zs, 0, self.batch.NT, out)
            self._Vs = out
        elif self._Vs is None and self.VsT is not None:      # only an E-step on the "emit" route leaves an emission behind
            from . import tc
            self._Vs = tc.vst_unpack(self, self.cfg.keep_E)
        return self._Vs

    # -- one sample_posterior call (mcem.py:207-277): returns kept samples [NT][C*keep][L]
    @_on_device
    def sample_posterior(self, keep: int, burn: int, draws: Optional[InjectedDraws] = None, a_trace=None, emit: bool = False):
        cfg, w, b = self.cfg, self.w, self.batch
        C_, L = cfg.n_chains, w.z_dim
        chains = b.NT * C_
        Zs = self._get("Zs%d" % keep, (b.NT, C_ * keep, L))
        rng = _lib.DvaeRng()
        rng.seed = cfg.seed & 0xFFFFFFFFFFFFFFFF
        rng.iter0 = self.mh_iter0
        rng.iter0_frame = None if self._iter0_frame is None else self._iter0_frame.data_ptr()
        eps = u = None
        if draws is not None:
            eps, u = draws.mh_draws(self.mh_calls, keep + burn, chains, L)
            eps = torch.as_tensor(eps).to(self.dev, torch.float32).contiguous()
            u = torch.as_tensor(u).to(self.dev, torch.float32).contiguous()
            if tuple(eps.shape) != (keep + burn, chains, L) or tuple(u.shape) != (keep + burn, chains):
                raise ValueError("injected draws for call %d have the wrong shape" % self.mh_calls)
            rng.eps, rng.u = eps.data_ptr(), u.data_ptr()
        with self.stage("mh"):
            if cfg.sampler == "tc":
                from . import tc
                tc.mh_chain_tc(self, Zs, keep, burn, rng, a_trace, emit)
            else:
                need = _lib.load().dvae_mh_workspace_floats(w.dec.ref, chains, self.F)
                ws = self._get("mh_ws", (max(int(need), 1),))
                _lib.call("dvae_mh_chain_f32", w.dec.ref, _p(self.P), _p(self.Vb), _p(self.g), _p(self.y), w.y_dim,
                          _p(b.frame_gid), _p(b.frame_idx), _p(self.Z), _p(Zs), b.NT, self.F, self.ld, L, C_, burn, keep,
                          float(cfg.var_rw), C.byref(rng), _p(self.n_accept), _p(a_trace), _p(ws), _stream())
                self.kernel_launches += (keep + burn + 1) * (len(w.dec.dims) - 1 + 1)
        self.mh_rows += chains * (keep + burn + 1)
        self.mh_calls += 1
        self.mh_iter0 += keep + burn
        return Zs

    @_on_device
    def decode_samples(self, Zs: torch.Tensor, n0: int, n1: int, Vs: torch.Tensor):
        """``compute_Vs`` (mcem.py:280-290) for frames [n0, n1): Vs[(n-n0)][r][ld] = decoder([Zs[n][r]; y[n]])."""
        R, L = Zs.shape[1], Zs.shape[2]
        rows = (n1 - n0) * R
        x = Zs[n0:n1].reshape(rows, L)
        x2 = None if self.y is None else self.y[n0:n1]
        out = Vs.view(-1, self.ld)[:rows]
        with self.stage("decode"):
            if self.cfg.sampler == "tc":
                from . import tc
                tc.decode_tc(self, x, x2, R, out, None if self.ybias is None else self.ybias[n0:n1])
            else:
                ws = self._get("mlp_ws", (max(int(_lib.load().dvae_mlp_workspace_floats(self.w.dec.ref, rows)), 1),))
                mlp_forward(self.w.dec, x, _lib.ACT_EXP, x2=x2, x2_row_div=R, out=out, ws=ws)
                self.kernel_launches += len(self.w.dec.dims) - 1

    @_on_device
    def e_step(self, draws=None):
        """E-step (mcem.py:292-308): sample, keep the last state, and hand the kept samples to the M-step along ``route``
        (``mcem_route``): the sampler's own BF16 emission + the W-update statistics, or FP32 ``Vs`` with or without them."""
        cfg = self.cfg
        self.wstat, self.wpart, self._Vs, self._last_Zs = None, None, None, None
        self.R = cfg.n_chains * cfg.keep_E                                  # samples per frame
        Zs = self.sample_posterior(cfg.keep_E, cfg.burn_E, draws, emit=self.route == "emit")
        if self.route != "emit":
            self._Vs = self.Vs_flat[: self.batch.NT * self.R].view(self.batch.NT, self.R, self.ld)
        if self.route == "decode":
            self.decode_samples(Zs, 0, self.batch.NT, self._Vs)
            return
        from . import tc
        with self.stage("decode"):
            if self.route == "stats":
                self.wstat = tc.decode_stats_tc(self, Zs, self._Vs)
            elif cfg.w_partials:
                self.wpart = tc.vst_w_partials(self, cfg.keep_E)
            else:
                self.wstat = tc.vst_frame_stats(self, cfg.keep_E)

    @_on_device
    def m_step(self, it: int):
        b, cfg = self.batch, self.cfg
        need = _lib.load().dvae_nmf_workspace_floats(b.B, cfg.nmf_rank, self.ld, b.max_frames)
        ws = self._get("nmf_ws", (int(need),))
        st = self._buf.get("tc_status")
        with self.stage("mstep"):
            if self.route == "emit":
                from . import tc
                w = self.w
                _lib.call("dvae_nmf_mstep_vst", w.dec_tc.ref, _p(tc.decoder_image(w)), w.z_dim, w.tc_y_dim, _p(self.P), _p(self.VsT),
                          _p(self.vs_idx), cfg.keep_E, _p(self.W), _p(self.H), _p(self.g), _p(self.Vb),
                          C.c_void_p(self.cost[it].data_ptr()), _p(b.fr_off), b.B, b.NT, cfg.nmf_rank, self.ld, b.max_frames,
                          _p(ws), _p(self.wstat), _p(self.wpart),
                          _p(b.segments(n_chains=cfg.n_chains)[2]) if self.wpart is not None else None, cfg.n_chains, _p(st), _stream())
            else:
                _lib.call("dvae_nmf_mstep", _p(self.P), _p(self._Vs), self.R, _p(self.W), _p(self.H), _p(self.g), _p(self.Vb),
                          C.c_void_p(self.cost[it].data_ptr()), _p(b.fr_off), _p(b.frame_utt), b.B, b.NT, self.F, cfg.nmf_rank,
                          self.ld, b.max_frames, _p(ws), _p(self.wstat), _p(st), _stream())
        self.kernel_launches += 4

    @_on_device
    def wiener(self, draws=None):
        """``compute_WF(sample=True)`` + the mask application of ``EM.run`` (mcem.py:310-329, 176-177)."""
        cfg, b = self.cfg, self.batch
        Zs = self.sample_posterior(cfg.keep_WF, cfg.burn_WF, draws)
        self._Vs, self._last_Zs = None, Zs
        R, chunk = Zs.shape[1], self.filter_chunk
        WFs = self._get("WFs", (b.NT, self.ld))
        WFn = self._get("WFn", (b.NT, self.ld))
        if chunk:
            # fused: the filter samples are decoded chunk by chunk straight into the mask sums, so none of the R x F x N
            # variances is written to memory
            from . import tc
            for r0 in range(0, R, chunk):
                tc.decode_wiener_tc(self, Zs, r0, chunk, WFs, WFn, accumulate=r0 > 0)
        else:
            # decode in frame chunks so the Vs buffer of the E-step (NT * R_E rows) is reused
            flat = self.Vs_flat
            step = max(1, min(b.NT, flat.shape[0] // R))
            for n0 in range(0, b.NT, step):
                n1 = min(b.NT, n0 + step)
                self.decode_samples(Zs, n0, n1, flat)
                _lib.call("dvae_wiener_accum", _p(flat), R, _p(self.Vb[n0:n1]), _p(self.g[n0:n1]), n1 - n0, self.F, self.ld,
                          _p(WFs[n0:n1]), _p(WFn[n0:n1]), 1, _stream())
                self.kernel_launches += 1
        self.S_hat = self._get("S_hat", (b.NT, self.ld), torch.complex64)
        self.N_hat = self._get("N_hat", (b.NT, self.ld), torch.complex64)
        _lib.call("dvae_wiener_apply", _p(self.X), _p(WFs), _p(WFn), R, b.NT, self.F, self.ld, _p(self.S_hat),
                  _p(self.N_hat), _stream())
        self.kernel_launches += 1
        self.WFs, self.WFn, self.R_wf = WFs, WFn, R

    @_on_device
    def run(self, draws: Optional[InjectedDraws] = None, checkpoints: Sequence[int] = (), on_checkpoint=None):
        """``EM.run`` (mcem.py:156-179): niter x (E-step, M-step, cost), then the Wiener estimates.

        Returns the device cost matrix ``[niter][B]`` (float64); nothing synchronises with the host.

        ``checkpoints``: EM iteration counts (``check_checkpoints``) at which ``on_checkpoint(n)`` is called while ``S_hat`` /
        ``N_hat`` hold the estimates that a run with ``niter = n`` returns, bit for bit: the MH draws are keyed by the global
        MH iteration, not by the call, so the final filter run on the side after M-step ``n`` draws what that run's own
        filter draws.  The side run's state is restored afterwards, so the main run does not change.  For ``n == niter`` the
        call follows the run's own filter.  Not with injected ``draws``: they are indexed by call and would be consumed out
        of order.
        """
        cps = check_checkpoints(checkpoints, self.cfg.niter)
        if cps and draws is not None:
            raise ValueError("checkpoints need the engine's own random numbers, not injected draws")
        check_stop(self.cfg, draws, cps)
        self.order, self.n_iter = None, np.full(self.batch.B, self.cfg.niter, np.int64)
        if self.cfg.stop_tol is not None:
            return self._run_stopping()
        for it in range(self.cfg.niter):
            self.e_step(draws)
            self.m_step(it)
            if it + 1 in cps and it + 1 < self.cfg.niter:
                self._side_filter(it + 1, on_checkpoint)
        self.wiener(draws)
        if on_checkpoint is not None and self.cfg.niter in cps:
            on_checkpoint(self.cfg.niter)
        return self.cost

    def _run_stopping(self):
        """``run`` with per-utterance stopping (``McemConfig.stop_tol``, test in ``dvae_em_stop_check``).

        The batch is kept as ``[active | parked]`` in the full-size buffers.  After each EM iteration ``n >= 2 stop_window``
        the device test flags the active utterances (one synchronisation); the active range is then stably partitioned into
        ``[continuing | just stopped]`` (``dvae_permute_rows`` through a scratch buffer) and the E- and M-steps run on the
        shorter prefix, whose ``RaggedBatch`` keeps the utterances' own ids, so their draws do not change.  A stopped
        utterance records the MH iteration counter at its stop; the one final filter over the whole batch starts every frame
        from its utterance's counter (``DvaeRng.iter0_frame``), which makes its output that of a run with ``niter = n_u``.
        Returns the cost ``[niter][B]`` in the caller's column order, NaN after each utterance's last iteration.  The
        per-frame state (``H``, ``g``, ``Z``, ``S_hat``, ...) stays in slot order: slot ``i`` is utterance ``order[i]`` and
        ``batch`` is the permuted batch."""
        cfg, full = self.cfg, self.batch
        B, w, niter = full.B, cfg.stop_window, cfg.niter
        self.cost.fill_(math.nan)
        order = np.arange(B)
        n_iter = np.full(B, niter, np.int64)
        iter0 = np.zeros(B, np.int64)                     # MH counter at each utterance's stop, caller's order
        flags = self._get("stop_flags", (B,), torch.uint8)
        self._stop_moved = set()                           # caller-owned inputs already replaced by engine buffers
        b_act = B
        for it in range(niter):
            self.e_step()
            self.m_step(it)
            n = it + 1
            if n < 2 * w or n == niter:
                continue
            with self.stage("stop_check"):
                _lib.call("dvae_em_stop_check", C.c_void_p(self.cost.data_ptr()), B, b_act, n, w, float(cfg.stop_tol), _p(flags),
                          _stream())
            stop = flags[:b_act].cpu().numpy().astype(bool)          # synchronises
            if not stop.any():
                continue
            n_iter[order[:b_act][stop]] = n
            iter0[order[:b_act][stop]] = self.mh_iter0
            keep = np.flatnonzero(~stop)
            if len(keep) == 0:
                b_act = 0
                break
            perm = np.concatenate([keep, np.flatnonzero(stop)])
            if np.any(perm != np.arange(b_act)):
                with self.stage("stop_permute"):
                    self._permute_active(perm, n)
                order[:b_act] = order[:b_act][perm]
            b_act = len(keep)
            self.batch = RaggedBatch(full.n_frames[order[:b_act]], self.dev, full.utt_ids_host[order[:b_act]])
        iter0[order[:b_act]] = self.mh_iter0
        self.batch = RaggedBatch(full.n_frames[order], self.dev, full.utt_ids_host[order])
        per_frame = np.repeat(iter0[order], full.n_frames[order]).astype(np.uint32)
        self._iter0_frame = torch.from_numpy(per_frame).to(self.dev)
        try:
            self.wiener()
        finally:
            self._iter0_frame = None
        out = self._get("cost_out", self.cost.shape, torch.float64)
        inv = np.empty(B, np.int32)
        inv[order] = np.arange(B, dtype=np.int32)
        inv_d = torch.from_numpy(inv).to(self.dev)
        with self.stage("stop_permute"):
            permute_rows([(self.cost, out, inv_d, B, 8, niter, 8 * B)])
        self.cost, self.order, self.n_iter = out, order, n_iter
        return out

    def _permute_active(self, perm, n):
        """Move the active utterances' state so that slot ``i`` holds what slot ``perm[i]`` held: per-frame, per-chain-row and
        per-utterance arrays and the ``n`` cost rows written so far, gathered into a scratch buffer sized for the full batch
        (one ``dvae_permute_rows`` launch) and copied back.  The inputs ``X`` / ``P`` / ``y`` belong to the caller: on their
        first move they are replaced by engine buffers instead of being overwritten."""
        b, C_ = self.batch, self.cfg.n_chains
        off = b.fr_off_host
        fmap = np.concatenate([np.arange(off[u], off[u + 1]) for u in perm])
        cmap = (fmap[:, None] * C_ + np.arange(C_)).reshape(-1)
        B_full = self.cost.shape[1]
        cost_map = np.concatenate([perm, np.arange(len(perm), B_full)])
        maps = torch.from_numpy(np.concatenate([fmap, cmap, perm, cost_map]).astype(np.int32)).to(self.dev)
        mf, mc, mu, mk = torch.split(maps, [len(fmap), len(cmap), len(perm), B_full])
        rows = {"f": (mf, b.NT), "c": (mc, b.NT * C_), "u": (mu, b.B)}
        arrays = [(k, kind) for k, kind in (("X", "f"), ("P", "f"), ("Vb", "f"), ("H", "f"), ("g", "f"), ("kscale", "f"),
                                            ("ybias", "f"), ("y", "f"), ("Z", "c"), ("n_accept", "c"), ("W", "u"))
                  if getattr(self, k) is not None]
        sizes = [getattr(self, k).numel() * getattr(self, k).element_size() for k, _ in arrays] + [self.cost.numel() * 8]
        offs = np.concatenate([[0], np.cumsum([(x + 15) // 16 * 16 for x in sizes])])
        scratch = self._get("stop_scratch", (int(offs[-1]),), torch.uint8)
        jobs = []
        for (k, kind), o in zip(arrays, offs):
            t = getattr(self, k)
            m, nr = rows[kind]
            jobs.append((t, scratch[o:], m, nr, t.numel() * t.element_size() // t.shape[0], 1, 0))
        jobs.append((self.cost, scratch[offs[-2]:], mk, B_full, 8, n, 8 * B_full))
        permute_rows(jobs)
        for k, (t, part, _, nr, rb, rep, pitch) in zip([k for k, _ in arrays] + ["cost"], jobs):
            nb = nr * rb if rep == 1 else rep * pitch
            target = t
            if k in ("X", "P", "y") and k not in self._stop_moved:
                target = self._get("stop_" + k, t.shape, t.dtype)
                _bytes(target)[nb:].copy_(_bytes(t)[nb:])          # the parked tail
                if k == "y" and self.tc_y is t:
                    self.tc_y = target
                setattr(self, k, target)
                self._stop_moved.add(k)
            _bytes(target)[:nb].copy_(part[:nb])
        self.kernel_launches += 1

    def _side_filter(self, n, on_checkpoint):
        """The final filter from the current state, ``on_checkpoint(n)``, then the state as it was before the filter.  The
        filter moves the chains (``Z``), the acceptance counts and the MH counters, and points the E-step's emission
        attributes elsewhere; Z and n_accept are snapshotted with device copies, the rest are host attributes.  The buffers
        it overwrites (filter samples, masks, spectra, the FP32 ``Vs`` scratch) are rewritten by the next E-step before any
        read.  Device time goes to the stage "trace" alone."""
        Z0 = self._get("Z_trace", self.Z.shape)
        acc0 = self._get("n_accept_trace", self.n_accept.shape, torch.int32)
        Z0.copy_(self.Z)
        acc0.copy_(self.n_accept)
        saved = {k: getattr(self, k) for k in ("mh_calls", "mh_iter0", "mh_rows", "_Vs", "_last_Zs", "VsT", "vs_idx")}
        with self.stage("trace"):
            timing, self.timing = self.timing, False
            try:
                self.wiener()
                if on_checkpoint is not None:
                    on_checkpoint(n)
            finally:
                self.timing = timing
        self.Z.copy_(Z0)
        self.n_accept.copy_(acc0)
        for k, v in saved.items():
            setattr(self, k, v)


def check_stop(cfg: McemConfig, draws=None, checkpoints: Sequence[int] = ()):
    """``ValueError`` when ``cfg.stop_tol`` is set together with something per-utterance stopping cannot serve: a negative or
    non-finite tolerance, ``stop_window < 1``, injected draws (they are indexed by call, and the final filter of a stopping
    run serves utterances stopped at different calls) or checkpoints.  No device work."""
    tol = cfg.stop_tol
    if tol is None:
        return
    if isinstance(tol, bool) or not isinstance(tol, (int, float, np.integer, np.floating)) or not math.isfinite(tol) or tol < 0:
        raise ValueError("stop_tol must be a finite number >= 0 or None, got %r" % (tol,))
    win = cfg.stop_window
    if isinstance(win, bool) or not isinstance(win, (int, np.integer)) or win < 1:
        raise ValueError("stop_window must be an integer >= 1, got %r" % (win,))
    if draws is not None:
        raise ValueError("stop_tol needs the engine's own random numbers, not injected draws")
    if tuple(checkpoints):
        raise ValueError("stop_tol cannot be combined with score_at / checkpoints")


def check_counters(max_frames: int, n_chains: int):
    """``ValueError`` when two chains of a batch would draw the same random numbers.  Word 1 of a draw's Philox counter is
    ``frame | chain << 20`` (csrc/common.cuh), so with several chains per frame an utterance of more than 2^20 frames (about
    4.7 hours at the 256-sample hop of 16 kHz audio) would give frame 2^20 of chain 0 the counters of frame 0 of chain 1.
    No device work."""
    if n_chains > 1 and max_frames > 1 << 20:
        raise ValueError("an utterance of %d frames exceeds the 2^20 frames per utterance that n_chains = %d leaves distinct "
                         "random numbers for" % (max_frames, n_chains))


def _bytes(t: torch.Tensor) -> torch.Tensor:
    return t.view(-1).view(torch.uint8)


def permute_rows(jobs):
    """One ``dvae_permute_rows`` launch over ``(src, dst, map, n_rows, row_bytes, n_rep, pitch)`` jobs (device tensors; ``map``
    int32): ``dst`` row ``i`` of every plane = ``src`` row ``map[i]``."""
    arr = (_lib.DvaePermuteJob * max(1, len(jobs)))()
    for j, (src, dst, m, n_rows, row_bytes, n_rep, pitch) in zip(arr, jobs):
        j.src, j.dst, j.map = src.data_ptr(), dst.data_ptr(), m.data_ptr()
        j.n_rows, j.row_bytes, j.n_rep, j.pitch = int(n_rows), int(row_bytes), int(n_rep), int(pitch)
    _lib.call("dvae_permute_rows", arr, len(jobs), _stream())


def check_checkpoints(checkpoints: Sequence[int], niter: int) -> tuple:
    """``checkpoints`` as a tuple of ints after checking they are sorted, unique integers in ``[1, niter]``; ``ValueError``
    otherwise.  No device work."""
    cps = tuple(checkpoints)
    if not all(isinstance(n, (int, np.integer)) and not isinstance(n, bool) for n in cps):
        raise ValueError("checkpoints must be integers, got %r" % (cps,))
    cps = tuple(int(n) for n in cps)
    if any(b <= a for a, b in zip(cps, cps[1:])):
        raise ValueError("checkpoints must be sorted and unique, got %r" % (cps,))
    if cps and (cps[0] < 1 or cps[-1] > niter):
        raise ValueError("checkpoints must lie in [1, niter=%d], got %r" % (niter, cps))
    return cps


# --------------------------------------------------------------------------------------------- end-to-end helper
class Enhancer:
    """``process_sublist`` replacement (scripts/evaluate_ntcd_M1.py:190-214): whole batches, host buffers in and out."""

    def __init__(self, sd, variant: str, cfg: McemConfig, device=0, fs=FS, n_fft=N_FFT, hop=HOP):
        self.dev = _require_cuda(device)
        self.weights = sd if isinstance(sd, VaeWeights) else VaeWeights(sd, variant, self.dev)
        self.cfg = cfg
        self.engine = McemEngine(self.weights, cfg, self.dev)
        self.fs, self.n_fft, self.hop = fs, n_fft, hop
        self._pinned = {}
        self._out_free = []              # pinned result buffers not leased to any caller (see _pin_out)
        self._h2d_done = None            # event after the last H2D copy out of the pinned staging buffers
        self._pool = None
        self._stage_threads = max(1, min(8, (os.cpu_count() or 1) // 2))

    def _pin(self, name, n, dtype):
        t = self._pinned.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(n, dtype=dtype).pin_memory()
            self._pinned[name] = t
        return t[:n]

    def _pin_out(self, n, dtype=torch.float32):
        """A pinned result buffer of ``dtype`` leased to the caller: ``(tensor, ndarray)``.

        Results are returned as views of pinned memory (no extra host copy).  Ownership is explicit: every lease gets a
        FRESH ndarray object over the pinned storage, the result views handed out keep that object alive through their
        ``.base``, and the storage goes back to the free list only when the object is collected (``weakref.finalize``),
        i.e. when the caller has dropped every array of that call.  Results never change under the caller, and no
        reference counts are inspected.
        """
        import weakref
        k = next((i for i, t in enumerate(self._out_free) if t.numel() >= n and t.dtype == dtype), None)
        t = self._out_free.pop(k) if k is not None else torch.empty(n, dtype=dtype).pin_memory()
        a = t.numpy()                                              # new ndarray object per lease
        free = self._out_free

        def give_back(tt=t):
            if len(free) < 4:                                      # keep a few buffers for reuse, let the rest go
                free.append(tt)

        weakref.finalize(a, give_back)
        return t, a

    def _stage(self, host_np, x_list, off, lens):
        """Copy the utterances into the pinned staging buffer (a few threads: numpy releases the GIL while copying)."""
        B = len(x_list)

        def work(lo, hi):
            for u in range(lo, hi):
                host_np[off[u]:off[u] + lens[u]] = x_list[u]

        nthr = min(self._stage_threads, max(1, B // 16))
        if nthr <= 1:
            work(0, B)
            return
        if self._pool is None:
            from concurrent.futures import ThreadPoolExecutor
            self._pool = ThreadPoolExecutor(self._stage_threads)
        step = (B + nthr - 1) // nthr
        futs = [self._pool.submit(work, lo, min(lo + step, B)) for lo in range(0, B, step)]
        for f in futs:
            f.result()

    @_on_device
    def run_device(self, x_dev, x_off, x_len, batch, y, total, max_len, draws=None, checkpoints=(), on_checkpoint=None):
        """The whole path on device-resident inputs: STFT -> MCEM -> Wiener -> ISTFT.  Nothing touches the host.

        ``x_dev``: concatenated float32 signals; ``x_off`` / ``x_len``: per-utterance offsets / lengths (device);
        returns ``(s_hat, n_hat)`` in the layout of ``x_dev`` and the cost matrix ``[niter][B]``.  ``checkpoints`` /
        ``on_checkpoint`` go to ``McemEngine.run`` (see ``checkpoint_scorer``).
        """
        eng = self.engine
        X, P = stft_batch(x_dev, x_off, x_len, batch, self.n_fft, self.hop)
        eng.init_parameters(X, P, batch, y, draws)
        cost = eng.run(draws, checkpoints, on_checkpoint)
        if eng.order is not None:            # stopping moved the frames: write every utterance through its slot's offset / length
            o = torch.from_numpy(eng.order.astype(np.int32)).to(self.dev)
            off_p, len_p = eng._get("x_off_perm", (batch.B,), torch.int64), eng._get("x_len_perm", (batch.B,), torch.int32)
            permute_rows([(x_off, off_p, o, batch.B, 8, 1, 0), (x_len, len_p, o, batch.B, 4, 1, 0)])
            batch, x_off, x_len = eng.batch, off_p, len_p
        s_dev = istft_batch(eng.S_hat, batch, x_off, x_len, total, max_len, self.n_fft, self.hop,
                            out=eng._get("s_out", (total,)))
        n_dev = istft_batch(eng.N_hat, batch, x_off, x_len, total, max_len, self.n_fft, self.hop,
                            out=eng._get("n_out", (total,)))
        eng.kernel_launches += 4          # stft, power-free init kernels are counted there; 2 istft + stft + vb
        return s_dev, n_dev, cost

    def checkpoint_scorer(self, ref, x_off, x_len, batch, total, max_len, rows):
        """An ``on_checkpoint`` for ``run_device`` that scores each checkpoint's speech estimate the way ``enhance`` scores
        ``scores[:, 0]``: ISTFT of ``S_hat`` as in ``run_device``, 16-bit PCM quantisation, then ``metrics.score_row``
        against ``ref`` (``metrics.score_reference``) into ``rows[n]``, a float64 ``[B][5]`` view.  Nothing synchronises."""
        from .packages import metrics
        eng = self.engine

        def score(n):
            est = istft_batch(eng.S_hat, batch, x_off, x_len, total, max_len, self.n_fft, self.hop,
                              out=eng._get("s_out", (total,)))
            s_q = eng._get("s_q", (total,))
            metrics.pcm16(est, None, s_q)
            metrics.score_row(s_q, ref, rows[n])
        return score

    def label_mode(self, oracle_labels, s_list, y_list):
        """The oracle label mode of an ``enhance`` call (``ORACLE_LABELS`` or ``None``: labels from ``y_list`` or none);
        ``ValueError`` when ``oracle_labels`` does not fit the model or the other arguments.  No device work."""
        y_dim, F = self.weights.y_dim, self.n_fft // 2 + 1
        if oracle_labels is None:
            if not y_dim or y_list is not None or s_list is None:
                return None
            if y_dim != 1:
                raise ValueError("a model with %d label inputs takes labels from s_list only with oracle_labels='ibm' or "
                                 "'robust_ibm' (%d inputs)" % (y_dim, F))
            return "vad"
        if oracle_labels not in ORACLE_LABELS:
            raise ValueError("oracle_labels must be one of %s or None, got %r" % (ORACLE_LABELS, oracle_labels))
        if not y_dim:
            raise ValueError("oracle_labels: an M1 model takes no labels")
        if s_list is None:
            raise ValueError("oracle_labels needs the clean signals s_list")
        if y_list is not None:
            raise ValueError("oracle_labels and y_list are two sources of the same labels: pass one")
        want = 1 if oracle_labels == "vad" else F
        if y_dim != want:
            raise ValueError("oracle_labels=%r gives %d labels per frame, the model takes %d" % (oracle_labels, want, y_dim))
        return oracle_labels

    def oracle_labels_device(self, mode, s_dev, x_off, x_len, n_clean, batch):
        """Oracle labels ``y [NT][y_dim]`` (engine buffers) of the clean signals ``s_dev`` (the layout of ``x_off`` / ``x_len``)
        for the frames of ``batch``.  They are computed over all ``n_clean[u]`` frames of each clean signal - the VAD's
        minimum frame power and the IBM's maximum magnitude are those of the whole utterance - and the first
        ``batch.n_frames[u]`` frames are kept (one ``dvae_permute_rows`` gather when a cap cuts), which is how the reference
        truncates ``y`` to the video length (scripts/evaluate_ntcd_M2.py:187-195).  The IBM's spectrogram and mask are laid
        out with a row stride of ``F = n_fft / 2 + 1`` bins, so the mask is the dense label matrix itself.  Nothing
        synchronises."""
        from .packages.processing.target import ibm_batch, vad_batch
        eng = self.engine
        n_clean = np.asarray(n_clean, np.int64)
        cut = bool(np.any(batch.n_frames != n_clean))
        full = RaggedBatch(n_clean, self.dev) if cut else batch
        NT = full.NT
        vad = None
        if mode in ("vad", "robust_ibm"):
            vad = vad_batch(s_dev, x_off, x_len, full, self.n_fft, self.hop, out=eng._get("oracle_vad", (NT,)),
                            ws=eng._get("oracle_vad_ws", (max(1, NT),), torch.float64))
        if mode == "vad":
            lab = vad.view(NT, 1)
        else:
            F = self.n_fft // 2 + 1
            S, _ = stft_batch(s_dev, x_off, x_len, full, self.n_fft, self.hop, want_power=False, ld=F,
                              out=eng._get("oracle_S", (NT, F), torch.complex64))
            lab = ibm_batch(S, full, F, vad=vad, out=eng._get("oracle_ibm", (NT, F)),
                            ws=eng._get("oracle_ibm_ws", (max(1, full.B),), torch.int32))
        if not cut:
            return lab
        y = eng._get("oracle_y", (batch.NT, lab.shape[1]))
        rows = np.repeat(full.fr_off_host[:-1] - batch.fr_off_host[:-1], batch.n_frames) + np.arange(batch.NT)
        permute_rows([(lab, y, torch.from_numpy(rows.astype(np.int32)).to(self.dev), batch.NT, lab.shape[1] * 4, 1, 0)])
        return y

    @_on_device
    def enhance(self, x_list, y_list=None, utt_ids=None, max_frames_list=None, draws=None, return_device=False, s_list=None,
                ref_list=None, pcm16=False, score_at=(), oracle_labels=None):
        """Enhance a list of 1-D float32 host signals.  Returns ``(s_hat_list, n_hat_list, cost [B][niter])``, and the scores
        ``[B][2][5]`` as a fourth element when ``ref_list`` is given, and the trace ``[B][len(score_at)][5]`` as a fifth when
        ``score_at`` is.

        ``y_list``: per-utterance label arrays ``(y_dim, N_u)`` as the reference passes them (M2 variants).
        ``max_frames_list``: optional per-utterance frame caps (the reference truncates to the video length).
        ``s_list``: clean signals, one per utterance and of its length, from which the device computes the oracle labels of
        scripts/evaluate_ntcd_M2.py (``oracle_labels_device``), so no label leaves or enters the host.
        ``oracle_labels`` (with ``s_list``, not with ``y_list``): ``"vad"`` (``clean_speech_VAD``, one label input), ``"ibm"``
        (``clean_speech_IBM`` of the clean STFT) or ``"robust_ibm"`` (``noise_robust_clean_speech_IBM``: the IBM times the
        VAD), both for ``n_fft / 2 + 1`` label inputs.  ``None`` means ``"vad"`` for a model with one label input and
        ``s_list``; a model with ``n_fft / 2 + 1`` label inputs needs the mode named.  Labels are computed over every frame of
        the clean signal and then cut to the first ``min(N_u, cap_u)`` frames, as the reference cuts ``y`` to the video
        length after computing it.
        ``utt_ids``: global utterance ids = Philox counter word 0; callers that enhance several batches must pass distinct
        ids per utterance (``batch_io.process_sublist`` does), or every batch replays the same random draws.
        ``ref_list``: clean signals, one per utterance and of its length, to score against on the device
        (``metrics.score_batch`` with its default trim, ``SCORE_KEYS`` order): row ``[u][0]`` scores the speech estimate
        after 16-bit PCM quantisation, i.e. exactly the samples ``batch_io.write_wav`` stores, row ``[u][1]`` the input.
        It may be the same list as ``s_list``; it then is copied to the device once.
        ``pcm16=True`` returns both estimates as int16 PCM (``write_wav``'s quantisation, done on the device), which halves
        their device-to-host bytes.  Neither option changes the estimates.
        ``score_at``: sorted, unique EM iteration counts in ``[1, niter]`` (needs ``ref_list``, not ``draws``).  Entry
        ``[u][k]`` of the trace (float64, ``SCORE_KEYS`` columns) is the score row ``[u][0]`` that this call with
        ``niter = score_at[k]`` would return, bit for bit; the input's row ``[u][1]`` does not change with ``niter``.  The
        whole curve comes from this one run (``McemEngine.run(checkpoints=...)``), and the estimates, cost and scores are
        those of the call without ``score_at``.
        ``return_device=True`` returns device tensors that alias the engine's output buffers: they are valid until the
        next call on this Enhancer (clone them to keep them).
        """
        eng, dev = self.engine, self.dev
        check_stop(eng.cfg, draws, score_at)
        B = len(x_list)
        lens = np.array([len(x) for x in x_list], np.int32)
        if np.any(lens < 1):
            raise ValueError("empty utterance")
        nfr = np.array([num_frames(int(t), self.n_fft, self.hop, self.fs) for t in lens], np.int64)
        if np.any(nfr < 1):
            raise ValueError("utterance shorter than one STFT frame")
        if ref_list is not None and (len(ref_list) != B or any(len(a) != t for a, t in zip(ref_list, lens))):
            raise ValueError("ref_list needs one clean signal per utterance, of the utterance's length")
        score_at = check_checkpoints(score_at, eng.cfg.niter)
        if score_at and (ref_list is None or draws is not None):
            raise ValueError("score_at needs ref_list and the engine's own random numbers (no injected draws)")
        mode = self.label_mode(oracle_labels, s_list, y_list)
        if mode is not None and (len(s_list) != B or any(len(a) != t for a, t in zip(s_list, lens))):
            raise ValueError("oracle labels need one clean signal per utterance, of the utterance's length")
        nfr_clean = nfr                            # the frames the oracle labels are computed over (truncation rule)
        if max_frames_list is not None:
            nfr = np.minimum(nfr, np.asarray(max_frames_list, np.int64))
        off = np.zeros(B + 1, np.int64)
        np.cumsum((lens + 1) // 2 * 2, out=off[1:])            # even offsets
        total = int(off[-1])
        if self._h2d_done is not None:          # the previous call's H2D copies must have left the staging buffers
            self._h2d_done.synchronize()
        host = self._pin("x", total, torch.float32)
        self._stage(host.numpy(), x_list, off, lens)
        x_dev = host.to(dev, non_blocking=True)
        x_off = torch.from_numpy(off[:-1].copy()).to(dev)
        x_len = torch.from_numpy(lens).to(dev)
        batch = RaggedBatch(nfr, dev, utt_ids)
        y = s_dev_in = None
        y_up = 0                                   # label bytes copied from the host
        if mode is not None:
            hs_in = self._pin("s_in", total, torch.float32)
            self._stage(hs_in.numpy(), s_list, off, lens)
            s_dev_in = hs_in.to(dev, non_blocking=True)
            y = self.oracle_labels_device(mode, s_dev_in, x_off, x_len, nfr_clean, batch)
        elif self.weights.y_dim:
            if y_list is None:
                raise ValueError("this model needs labels y")
            yc = np.concatenate([np.asarray(yy, np.float32)[:, :n].T for yy, n in zip(y_list, nfr)], axis=0)
            if yc.shape != (batch.NT, self.weights.y_dim):
                raise ValueError("labels do not cover the frames")
            y = torch.from_numpy(np.ascontiguousarray(yc)).to(dev)
            y_up = y.numel() * 4
        ref_dev = None
        if ref_list is not None:
            if ref_list is s_list and s_dev_in is not None:
                ref_dev = s_dev_in
            else:
                hr = self._pin("ref", total, torch.float32)
                self._stage(hr.numpy(), ref_list, off, lens)
                ref_dev = hr.to(dev, non_blocking=True)
        self._h2d_done = torch.cuda.Event()
        self._h2d_done.record()
        trace = on_checkpoint = None
        if score_at:
            from .packages import metrics
            trace = eng._get("trace", (B, len(score_at), 5), torch.float64)
            on_checkpoint = self.checkpoint_scorer(metrics.score_reference(x_dev, ref_dev, x_off, x_len, self.fs), x_off, x_len,
                                                   batch, total, int(lens.max()), {n: trace[:, k] for k, n in enumerate(score_at)})
        side = tuple(n for n in score_at if n < eng.cfg.niter)    # niter itself is the run's own filter, scored below
        s_dev, n_dev, cost = self.run_device(x_dev, x_off, x_len, batch, y, total, int(lens.max()), draws, side, on_checkpoint)
        clean_up = (s_dev_in is not None) + (ref_dev is not None and ref_dev is not s_dev_in)    # clean signals uploaded
        self.h2d_bytes = total * 4 * (1 + clean_up) + y_up
        scores = None
        if ref_list is not None or pcm16:
            from .packages import metrics
            s_pcm = eng._get("s_pcm", (total,), torch.int16) if pcm16 else None
            n_pcm = eng._get("n_pcm", (total,), torch.int16) if pcm16 else None
            s_q = eng._get("s_q", (total,)) if ref_list is not None else None
            metrics.pcm16(s_dev, s_pcm, s_q)
            if pcm16:
                metrics.pcm16(n_dev, n_pcm)
                s_dev, n_dev = s_pcm, n_pcm
            if ref_list is not None:
                scores = metrics.score_batch(s_q, x_dev, ref_dev, x_off, x_len, self.fs, out=eng._get("scores", (B, 2, 5), torch.float64))
            if score_at and score_at[-1] == eng.cfg.niter:
                trace[:, -1].copy_(scores[:, 0])
        esize = 2 if pcm16 else 4
        self.d2h_bytes = 2 * total * esize + cost.numel() * 8 + sum(0 if t is None else t.numel() * 8 for t in (scores, trace))
        extra = () if scores is None else (scores,) if trace is None else (scores, trace)
        from . import tc
        if return_device:
            tc.check_status(eng)                               # synchronises
            return (s_dev, n_dev, cost) + extra
        hs, s_np = self._pin_out(total, s_dev.dtype)
        hn, n_np = self._pin_out(total, n_dev.dtype)
        hs[:total].copy_(s_dev, non_blocking=True)
        hn[:total].copy_(n_dev, non_blocking=True)
        cost_h = cost.t().contiguous().cpu()                   # synchronises the stream
        extra = tuple(t.cpu().numpy() for t in extra)
        torch.cuda.current_stream().synchronize()
        tc.check_status(eng)
        s_list = [s_np[off[u]:off[u] + lens[u]] for u in range(B)]      # views of pinned memory, see _pin_out
        n_list = [n_np[off[u]:off[u] + lens[u]] for u in range(B)]
        return (s_list, n_list, cost_h.numpy()) + extra
