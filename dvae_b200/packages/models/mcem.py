"""``MCEM_M1`` / ``MCEM_M2`` / ``MCEM_M2v2`` / ``MCEM_M2v3`` with the reference's signatures, backed by the CUDA engine.

Drop-in for ``packages/models/mcem.py:182-845`` as the ``evaluate_ntcd_*`` scripts use it::

    mcem = MCEM_M1(niter=100, nsamples_E_step=10, burnin_E_step=30, nsamples_WF=25, burnin_WF=75, var_RW=0.01)
    mcem.init_parameters(X=x_tf, S=s_tf, vae=model, nmf_rank=10, eps=1e-8, device=device)   # X, S: (F,N) complex64
    cost = mcem.run()                                                                        # (niter,) float64
    S_hat, N_hat = mcem.S_hat, mcem.N_hat                                                    # (F,N) complex64

One object is reused across utterances (``scripts/evaluate_ntcd_M1.py:213-214,230``): ``init_parameters`` fully resets
the state.  Objects are picklable (spawn pools): device state is created lazily inside ``init_parameters``.

Behaviour carried over on purpose (SURVEY §3.2):
  Q1  ``MCEM_M1`` passes ``(Z, nsamples, burnin)`` into ``sample_posterior(Z, y, nsamples=10, burnin=30)``, so it runs
      ``burnin_arg + 30`` iterations keeping ``burnin_arg`` samples (60/30 per E-step, 105/75 for the filter with the
      shipped settings).  The M2 classes use their arguments as named.
  Q3  ``S`` is required but only consumes a random draw.
  Q5  ``device`` may be an int, a str or a ``torch.device``.

Extra keyword-only knobs (not in the reference): ``sampler`` ("auto": tcgen05 BF16 kernels when the decoder has the
shipped shape, else "fp32"; "fp32": exact CUDA-core decoder; "tc": force the tensor-core kernels),
``n_chains``, ``seed`` and ``rng`` ("philox": counter-based draws on the device; "torch": the reference's own draw
order taken from torch's CPU generator, for like-for-like comparisons), ``stop_tol`` / ``stop_window`` (stop the EM loop
once the cost has converged, ``McemConfig.stop_tol``; ``niter`` is then the cap, ``run()`` returns the cost NaN-padded to
``(niter,)`` and ``n_iter`` holds the iterations run; Philox draws only).
"""
from __future__ import annotations

import numpy as np
import torch

from ...engine import McemConfig, McemEngine, RaggedBatch, TorchCpuDraws, VaeWeights, _ld_for, _p, _stream, check_stop
from ... import _lib


def _find_prefix(sd):
    for pre in ("", "enc_dec_clf."):
        if f"{pre}decoder.reconstruction.weight" in sd:
            return pre
    raise ValueError("state_dict has no decoder.reconstruction.weight")


class _MCEM:
    _variant = None

    def __init__(self, niter, nsamples_E_step=10, burnin_E_step=30, nsamples_WF=25, burnin_WF=75, var_RW=0.01, *,
                 sampler="auto", n_chains=1, seed=0, rng="philox", stop_tol=None, stop_window=10):
        self.niter = niter
        self.nsamples_E_step, self.burnin_E_step = nsamples_E_step, burnin_E_step
        self.nsamples_WF, self.burnin_WF = nsamples_WF, burnin_WF
        self.var_RW = var_RW
        self.sampler, self.n_chains, self.seed, self.rng = sampler, n_chains, seed, rng
        if rng not in ("philox", "torch"):
            raise ValueError("rng must be 'philox' or 'torch'")
        self.stop_tol, self.stop_window = stop_tol, stop_window
        if stop_tol is not None and rng == "torch":
            raise ValueError("stop_tol needs rng='philox': the reference's draw order cannot serve utterances stopped early")
        check_stop(McemConfig(niter=niter, stop_tol=stop_tol, stop_window=stop_window))
        self._engine = None
        self._weights_key = None

    # schedule actually executed: ((keep_E, burn_E), (keep_WF, burn_WF))
    def schedule(self):
        return (self.nsamples_E_step, self.burnin_E_step), (self.nsamples_WF, self.burnin_WF)

    def __getstate__(self):
        d = self.__dict__.copy()
        for k in ("_engine", "_weights", "_draws", "vae", "y"):
            d.pop(k, None)
        d["_engine"] = None
        d["_weights_key"] = None
        return d

    def _setup(self, X, S, y, vae, nmf_rank, eps, device):
        if type(vae).__name__ == 'RVAE':
            raise NameError('MCEM algorithm only valid for FFNN VAE')
        X = np.asarray(X)
        S = np.asarray(S)
        if X.ndim != 2 or X.shape != S.shape:
            raise ValueError("X and S must be (F, N) spectrograms of the same shape")
        F, N = X.shape
        dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if dev.type != "cuda":
            raise _lib.DvaeError("dvae_b200 runs on CUDA devices only (got device=%r); there is no CPU fallback" % (device,))
        self.device = dev
        with torch.cuda.device(dev):               # the reference's workers never call set_device (evaluate_ntcd_M1.py:69,252)
            self._setup_on_device(X, S, y, vae, nmf_rank, eps, dev, F, N)

    def _setup_on_device(self, X, S, y, vae, nmf_rank, eps, dev, F, N):
        from ..processing import stft as _stft_shim
        _stft_shim.set_device(dev)                  # the numpy-facing stft / istft wrappers follow the MCEM device
        sd = vae.state_dict()
        key = (id(vae), str(dev), tuple(int(p._version) for p in vae.parameters()))
        if self._engine is None or self._weights_key != key or self._cfg_rank != (nmf_rank, eps):
            (kE, bE), (kW, bW) = self.schedule()
            cfg = McemConfig(niter=self.niter, keep_E=kE, burn_E=bE, keep_WF=kW, burn_WF=bW, var_rw=self.var_RW,
                             nmf_rank=nmf_rank, eps=eps, n_chains=self.n_chains, seed=self.seed, sampler=self.sampler,
                             stop_tol=self.stop_tol, stop_window=self.stop_window)
            self._weights = VaeWeights(sd, self._variant, dev, prefix=_find_prefix(sd))
            self._engine = McemEngine(self._weights, cfg, dev)
            self._weights_key, self._cfg_rank = key, (nmf_rank, eps)
        eng = self._engine
        if eng.F != F:
            raise ValueError("spectrogram has %d bins, the VAE models %d" % (F, eng.F))
        self.vae = vae
        self.X = X
        ld = _ld_for(F)
        Xd = torch.zeros((N, ld), dtype=torch.complex64, device=dev)
        Xd[:, :F] = torch.from_numpy(np.ascontiguousarray(X.T.astype(np.complex64))).to(dev)
        Pd = torch.zeros((N, ld), dtype=torch.float32, device=dev)
        _lib.call("dvae_power", _p(Xd), _p(Pd), N * ld, _stream())
        yd = None
        if self._variant != "M1":
            self.y = y
            yd = torch.as_tensor(y).detach().to(dev, torch.float32).t().contiguous()        # (y_dim,N) -> [N][y_dim]
        batch = RaggedBatch([N], dev)
        self._draws = None
        if self.rng == "torch":
            self._draws = TorchCpuDraws(F, nmf_rank, N, self._weights.z_dim)
        eng.init_parameters(Xd, Pd, batch, yd, self._draws)

    def run(self):
        eng = self._engine
        with torch.cuda.device(eng.dev):
            cost = eng.run(self._draws)
            F = eng.F
            from ... import tc
            tc.check_status(eng)
            self.S_hat = np.ascontiguousarray(eng.S_hat[:, :F].t().cpu().numpy())
            self.N_hat = np.ascontiguousarray(eng.N_hat[:, :F].t().cpu().numpy())
            return cost[:, 0].cpu().numpy().astype(np.float64)

    @property
    def n_iter(self):
        """EM iterations the last ``run()`` executed (``niter`` unless ``stop_tol`` stopped it earlier)."""
        return int(self._engine.n_iter[0])

    # ---- state exposed with the reference's shapes
    @property
    def W(self):
        return self._engine.W[0, :, :self._engine.F].t()                  # (F, K)

    @property
    def H(self):
        return self._engine.H.t()                                         # (K, N)

    @property
    def g(self):
        return self._engine.g                                             # (N,)

    @property
    def Z(self):
        C_ = self._engine.cfg.n_chains
        return self._engine.Z[::C_].t()                                   # (L, N), chain 0

    @property
    def Vb(self):
        return self._engine.Vb[:, :self._engine.F].t()                    # (F, N)

    # The variances of the last sampled set, with the reference's shapes (mcem.py:29-34, 76-80): (R, F, N).  After ``run()``
    # these are the filter's samples (mcem.py:316-320).  The engine keeps them in its own formats (BF16 emission of the
    # sampler / never materialised for the filter), so they are produced on first access.
    @property
    def Vs(self):
        v = self._engine.Vs
        return None if v is None else v[:, :, :self._engine.F].permute(1, 2, 0)

    @property
    def Vs_scaled(self):
        v = self.Vs
        return None if v is None else self._engine.g[None, None, :] * v

    @property
    def Vx(self):
        v = self.Vs_scaled
        return None if v is None else v + self.Vb[None]

    @property
    def X_abs_2(self):
        return self._engine.P[:, :self._engine.F].t()

    @property
    def acceptance_rate(self):
        """Fraction of accepted proposals so far (the reference computes and drops it, mcem.py:261-262)."""
        eng = self._engine
        return float(eng.n_accept.sum().item()) / max(1, eng.mh_iter0 * eng.n_accept.numel())


class MCEM_M1(_MCEM):
    """Audio-only VAE (``VariationalAutoencoder``); mcem.py:182-329."""
    _variant = "M1"

    def schedule(self):
        # mcem.py:297-298 / 314-315 call sample_posterior(self.Z, nsamples, burnin) against (Z, y, nsamples, burnin=30)
        return (self.burnin_E_step, 30), (self.burnin_WF, 30)

    def init_parameters(self, X, S, vae, nmf_rank, eps, device):
        self._setup(X, S, None, vae, nmf_rank, eps, device)


class MCEM_M2(_MCEM):
    """Label-conditioned VAE, encoder over ``[x; y]`` (``DeepGenerativeModel``); mcem.py:332-501."""
    _variant = "M2"

    def init_parameters(self, X, S, y, vae, nmf_rank, eps, device):
        self._setup(X, S, y, vae, nmf_rank, eps, device)


class MCEM_M2v2(_MCEM):
    """Label-conditioned decoder, encoder over ``x`` only; mcem.py:504-673."""
    _variant = "M2v2"

    def init_parameters(self, X, S, y, vae, nmf_rank, eps, device):
        self._setup(X, S, y, vae, nmf_rank, eps, device)


class MCEM_M2v3(MCEM_M2v2):
    """Line-for-line twin of ``MCEM_M2v2`` in the reference (mcem.py:676-845), used with ``DeepGenerativeModel_v5``."""
    _variant = "M2v3"
