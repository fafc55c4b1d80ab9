"""Candidate-side stages around recombination, on the device (SURVEY 8f rows 2-3).

Mirrors of the reference objects that produce ``pts_rec`` / ``pts_nys`` / ``init_weights``:

* ``PriorSampler``            - ``BASQ/_sampler.py:7-34`` (and SOBER ``Gaussian.sample``, ``SOBER/_prior.py:107-118``)
* ``calc_weights``            - ``UncertaintySampler.calc_weights``, ``BASQ/_sampler.py:190-217``
* ``lfi``                     - ``PI_BQ.lfi``, ``SOBER/_pi.py:121-139``
* ``cleansing_weights``       - ``WeightsStabiliser.cleansing_weights``, ``SOBER/_weights.py:21-38``
* ``mvn_logpdf``              - ``prior.log_prob`` / ``Gaussian.pdf``
* ``SIR`` / ``sir_indices``   - ``UncertaintySampler.SIR``, ``BASQ/_sampler.py:104-118`` (torch.multinomial)

Everything computes inside libbasq_b200.so (csrc/candidates.cu); torch only owns the buffers.
Random numbers are Philox4x32-10 keyed by (seed, global row), so N candidates sharded over ranks are
slices of one stream: rank r passes ``offset`` = its first global row.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib, ops

_F = {torch.float32: _lib.F32, torch.float64: _lib.F64}
SIR_DIGIT_BITS = 11    # BASQ_SIR_DIGIT_BITS


def _mvn_params(mean, cov=None, scale_tril=None):
    mean = torch.as_tensor(mean, dtype=torch.float64).detach().cpu().contiguous()
    if scale_tril is None:
        cov = torch.as_tensor(cov, dtype=torch.float64).detach().cpu()
        scale_tril = torch.linalg.cholesky(cov)
    L = torch.as_tensor(scale_tril, dtype=torch.float64).detach().cpu().contiguous()
    d = mean.numel()
    if L.shape != (d, d):
        raise ValueError(f"covariance factor has shape {tuple(L.shape)} for dimension {d}")
    return mean, L, d


def _prior_params(prior):
    """(mean, L) of a torch.distributions.MultivariateNormal-like object (.loc, .scale_tril)."""
    tril = getattr(prior, "scale_tril", None)
    if tril is None:
        return _mvn_params(prior.loc, cov=prior.covariance_matrix)
    return _mvn_params(prior.loc, scale_tril=tril)


def sample_mvn(mean, cov, n, seed=0, offset=0, device="cuda", dtype=torch.float32, scale_tril=None):
    """[n, d] draws of N(mean, cov): rows offset .. offset+n of the stream defined by `seed`."""
    mean, L, d = _mvn_params(mean, cov, scale_tril)
    device = torch.device(device)
    ctx = _lib.context_for(device)
    X = torch.empty(int(n), d, dtype=dtype, device=device)
    _lib.check(_lib.lib.basq_sample_mvn(ctx.handle, C.c_uint64(int(seed) & (2 ** 64 - 1)), int(offset), int(n), d,
                                        _F[dtype], mean.data_ptr(), L.data_ptr(), X.data_ptr()))
    return X


def mvn_logpdf(X, mean, cov=None, scale_tril=None):
    """log N(x_i; mean, cov) as fp64 [N] (prior.log_prob)."""
    mean, L, d = _mvn_params(mean, cov, scale_tril)
    if X.dtype not in _F:
        X = X.float()
    X = X.contiguous()
    ctx = _lib.context_for(X.device)
    out = torch.empty(len(X), dtype=torch.float64, device=X.device)
    _lib.check(_lib.lib.basq_mvn_logpdf(ctx.handle, X.data_ptr(), len(X), d, _F[X.dtype], mean.data_ptr(),
                                        L.data_ptr(), out.data_ptr()))
    return out


def _weights(kind, ratio, log, mean, var, normalise):
    mean = mean.to(torch.float64).contiguous()
    var = var.to(torch.float64).contiguous()
    ctx = _lib.context_for(mean.device)
    w = torch.empty_like(mean)
    _lib.check(_lib.lib.basq_candidate_weights(ctx.handle, kind, float(ratio), 1 if log else 0, mean.data_ptr(),
                                               var.data_ptr(), mean.numel(), 1 if normalise else 0, w.data_ptr()))
    return w


def calc_weights(kernel, pts_rec, ratio=0.5):
    """Importance weights w_IS = f / g of candidates drawn from the mixed proposal, normalised
    (UncertaintySampler.calc_weights, BASQ/_sampler.py:190-217): GP mean / variance over the
    candidates (basq_gp_predict) followed by one elementwise pass and a deterministic sum."""
    mean, var = ops.gp_predict(kernel, pts_rec, space=0, want_var=True)
    return _weights(0, ratio, False, mean, var, True)


def lfi(kernel, X_cand, log=False):
    """Phi((mu_g - 1) / sqrt(var_g)) from the model-space moments (PI_BQ.lfi, SOBER/_pi.py:121-139)."""
    mean, var = ops.gp_predict(kernel, X_cand, space=1, want_var=True)
    return _weights(1, 0.0, log, mean, var, False)


def cleansing_weights(weights, eps=torch.finfo(torch.float32).eps):
    """WeightsStabiliser.cleansing_weights (SOBER/_weights.py:21-38); returns a new tensor."""
    w = weights.detach().to(torch.float64).clone().contiguous()
    ctx = _lib.context_for(w.device)
    _lib.check(_lib.lib.basq_cleanse_weights(ctx.handle, w.data_ptr(), w.numel(), float(eps)))
    return w


def sir_indices(weights, n_return, seed=0):
    """Indices of `n_return` draws without replacement proportional to `weights`, in draw order
    (torch.multinomial(weights, n_return) of UncertaintySampler.SIR, BASQ/_sampler.py:104-118)."""
    w = weights.detach().to(torch.float64).contiguous()
    ctx = _lib.context_for(w.device)
    idx = torch.empty(int(n_return), dtype=torch.int64)
    got = C.c_int64(0)
    _lib.check(_lib.lib.basq_sir_resample(ctx.handle, w.data_ptr(), w.numel(), int(n_return),
                                          C.c_uint64(int(seed) & (2 ** 64 - 1)), idx.data_ptr(), C.byref(got)))
    return idx[: got.value].to(w.device)


def SIR(X, weights, n_return, seed=0):
    """UncertaintySampler.SIR (BASQ/_sampler.py:104-118): ``X[torch.multinomial(weights, n_return)]``."""
    return X[sir_indices(weights, n_return, seed=seed)]


class ShardEngine:
    """Rank-local steps of the candidate side over a row-sharded set (basq_weights_*, basq_sir_*), the engine of
    the functions in basq_b200.sharded, which sum the host results over the ranks between the calls.  Weights
    are fp64 device tensors; SIR keys are int64 tensors that hold the uint64 key bits."""

    def __init__(self, device):
        self.device = torch.device(device)
        self.ctx = _lib.context_for(self.device)

    def candidate_weights(self, kernel, X, ratio):
        """calc_weights before normalisation."""
        if len(X) == 0:
            return torch.empty(0, dtype=torch.float64, device=self.device)
        mean, var = ops.gp_predict(kernel, X, space=0, want_var=True)
        return _weights(0, ratio, False, mean, var, False)

    def weights_sum(self, w) -> float:
        out = C.c_double(0.0)
        _lib.check(_lib.lib.basq_weights_sum(self.ctx.handle, w.data_ptr(), w.numel(), C.byref(out)))
        return float(out.value)

    @property
    def reproducible(self) -> bool:
        return self.ctx.is_reproducible

    def weights_max(self, w) -> float:
        out = C.c_double(0.0)
        _lib.check(_lib.lib.basq_weights_max(self.ctx.handle, w.data_ptr(), w.numel(), C.byref(out)))
        return float(out.value)

    def weights_sum_grid(self, w, wmax, N_glob) -> np.ndarray:
        hilo = np.zeros(2, dtype=np.float64)
        _lib.check(_lib.lib.basq_weights_sum_grid(self.ctx.handle, w.data_ptr(), w.numel(), float(wmax), int(N_glob),
                                                  hilo.ctypes.data))
        return hilo

    def weights_normalise(self, w, total, N_glob):
        _lib.check(_lib.lib.basq_weights_normalise(self.ctx.handle, w.data_ptr(), w.numel(), float(total), int(N_glob)))

    def weights_cleanse(self, w, eps):
        _lib.check(_lib.lib.basq_weights_cleanse(self.ctx.handle, w.data_ptr(), w.numel(), float(eps)))

    def sir_keys(self, w, seed, idx_base):
        keys = torch.empty(w.numel(), dtype=torch.int64, device=self.device)
        _lib.check(_lib.lib.basq_sir_keys(self.ctx.handle, w.data_ptr(), w.numel(), C.c_uint64(int(seed) & (2 ** 64 - 1)),
                                          int(idx_base), keys.data_ptr()))
        return keys

    def sir_histogram(self, keys, mask, bits, shift):
        hist = np.zeros(1 << SIR_DIGIT_BITS, dtype=np.int64)
        _lib.check(_lib.lib.basq_sir_histogram(self.ctx.handle, keys.data_ptr(), keys.numel(), C.c_uint64(mask),
                                               C.c_uint64(bits), int(shift), hist.ctypes.data))
        return hist

    def sir_collect(self, keys, T, idx_base, cap):
        ks = torch.empty(cap, dtype=torch.int64, device=self.device)
        ids = torch.empty(cap, dtype=torch.int64, device=self.device)
        n = C.c_int64(0)
        _lib.check(_lib.lib.basq_sir_collect(self.ctx.handle, keys.data_ptr(), keys.numel(), C.c_uint64(T), int(idx_base),
                                             int(cap), ks.data_ptr(), ids.data_ptr(), C.byref(n)))
        return ks[: n.value], ids[: n.value]

    def sir_sort(self, keys, idx):
        """Stable sort of the pairs by key, in place (contiguous tensors); returns idx."""
        if not (keys.is_contiguous() and idx.is_contiguous() and keys.numel() == idx.numel()):
            raise ValueError("sir_sort: keys and idx must be contiguous and of the same length")
        _lib.check(_lib.lib.basq_sir_sort(self.ctx.handle, keys.data_ptr(), idx.data_ptr(), keys.numel()))
        return idx


class PriorSampler:
    """BASQ/_sampler.py:7-34 on the device: ``pts_nys, pts_rec, w = sampler(n_rec)``.

    `prior` is a torch.distributions.MultivariateNormal (only .loc and .scale_tril /
    .covariance_matrix are read).  Successive calls continue the stream (fresh candidates)."""

    def __init__(self, prior, n_rec, nys_ratio, device, seed=0, dtype=torch.float32, rank=0, world=1):
        self.mean, self.L, self.d = _prior_params(prior)
        self.n_rec, self.nys_ratio, self.device = n_rec, nys_ratio, torch.device(device)
        self.seed, self.dtype, self.rank, self.world = seed, dtype, rank, world
        self.drawn = 0

    def __call__(self, n_rec):
        from .sharded import shard_bounds
        lo, hi = shard_bounds(n_rec, self.world, self.rank)
        pts_rec = sample_mvn(self.mean, None, hi - lo, seed=self.seed, offset=self.drawn + lo, device=self.device,
                             dtype=self.dtype, scale_tril=self.L)
        n_nys = int(self.n_rec * self.nys_ratio)
        if self.world == 1:
            pts_nys = pts_rec[:n_nys]
        else:  # every rank regenerates the leading rows of the stream: identical landmarks, no broadcast
            pts_nys = sample_mvn(self.mean, None, n_nys, seed=self.seed, offset=self.drawn, device=self.device,
                                 dtype=self.dtype, scale_tril=self.L)
        self.drawn += n_rec
        w = torch.full((hi - lo,), 1.0 / n_rec, dtype=self.dtype, device=self.device)
        return pts_nys, pts_rec, w
