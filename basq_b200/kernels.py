"""Kernel descriptors: turn the reference's kernel objects into the POD the C ABI takes.

The reference hands ``recombination`` an opaque Python callable ``kernel(X, Y)`` (SURVEY 8b).  A
fused CUDA path cannot call back into Python, so the shim recognises the concrete objects the
reference constructs - by duck typing, gpytorch itself is not required - and extracts their
parameters.  Anything else raises: there is deliberately no generic (slow) fallback.

Recognised (reference file:line):
  * bound ``VanillaGP.predictive_kernel``                      BASQ/_vbq.py:119-128
  * bound ``WsabiGP.{predictive,wsabil,wsabim}_kernel``        BASQ/_wsabi.py:194-249
  * bound ``ScaleMmltGP.{hspace,gspace}_kernel``               SOBER/BASQ/_scale_mmlt.py:247-278
  * ``SOBER Kernel(model, mode)`` objects                      SOBER/_kernel.py:4-47
  * ``model.covar_module.forward`` / a ScaleKernel object      BASQ/_quadrature.py:101
  * ``KernelSpec`` instances built by the caller
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import torch

from . import _lib

_MODE_BY_METHOD = {
    "predictive_kernel": _lib.PRED_COV,
    "hspace_kernel": _lib.PRED_COV,
    "wsabil_kernel": _lib.WSABI_L,
    "wsabim_kernel": _lib.WSABI_M,
    "gspace_kernel": _lib.MMLT_G,
}
_MODE_BY_SOBER = {
    "predictive_covariance": _lib.PRED_COV,
    "weighted_predictive_covariance": _lib.WSABI_L,
    "kernel": _lib.PLAIN,
}


@dataclasses.dataclass
class KernelSpec:
    family: int                     # _lib.RBF / MATERN15 / MATERN25
    mode: int                       # _lib.PLAIN ... MMLT_G
    lengthscale: torch.Tensor       # 1 or d entries (host or device)
    outputscale: float
    noise: float = 0.0
    mean_const: float = 0.0
    diag_add: float = 0.0           # wsabi / mmlt jitter: added to the Gram diagonal after the warping
    noise_diag: bool = False        # BASQ/_gp.py:275-276 "+ lik_var" on the covariance diagonal, before warping
    Xobs: Optional[torch.Tensor] = None
    W: Optional[torch.Tensor] = None      # (K_XX + noise I)^-1
    alpha: Optional[torch.Tensor] = None  # mean cache
    offset: float = 0.0             # WSABI alpha (model-space mean offset)

    def to_desc(self, d: int, device, dtype):
        """(KernelDesc, keepalive) for inputs of dimension d / dtype on device."""
        if dtype not in (torch.float32, torch.float64):
            raise TypeError(f"basq_b200 evaluates kernels in float32 or float64, not {dtype}")
        if not (1 <= d <= _lib.BASQ_MAX_DIM):
            raise ValueError(f"input dimension {d} outside 1..{_lib.BASQ_MAX_DIM}")
        desc = _lib.KernelDesc()
        desc.family, desc.mode = int(self.family), int(self.mode)
        desc.dtype = _lib.F32 if dtype == torch.float32 else _lib.F64
        desc.d = d
        desc.outputscale = float(self.outputscale)
        ls = torch.as_tensor(self.lengthscale, dtype=torch.float64).detach().cpu().reshape(-1)
        if ls.numel() == 1:
            ls = ls.repeat(d)
        if ls.numel() != d:
            raise ValueError(f"lengthscale has {ls.numel()} entries for d={d}")
        for i in range(d):
            desc.lengthscale[i] = float(ls[i])
        desc.noise, desc.mean_const, desc.diag_add = float(self.noise), float(self.mean_const), float(self.diag_add)
        desc.noise_diag = 1 if self.noise_diag else 0
        keep = []
        if self.mode != _lib.PLAIN or self.Xobs is not None:
            if self.Xobs is None or self.W is None or self.alpha is None:
                raise ValueError("posterior kernels need Xobs, W and alpha")
            Xobs = self.Xobs.detach().to(device=device, dtype=dtype).contiguous()
            W = self.W.detach().to(device=device, dtype=torch.float64).contiguous()
            alpha = self.alpha.detach().to(device=device, dtype=torch.float64).contiguous()
            if Xobs.shape[1] != d or W.shape != (len(Xobs), len(Xobs)) or alpha.shape != (len(Xobs),):
                raise ValueError("inconsistent GP cache shapes")
            # fp64 observations beside the dtype copy: W belongs to these, and a call whose fp32 inputs are
            # promoted to the fp64 path (conditioning guard) must not evaluate k at their fp32 roundings
            Xobs_f64 = Xobs if dtype == torch.float64 else self.Xobs.detach().to(device=device, dtype=torch.float64).contiguous()
            keep += [Xobs, W, alpha, Xobs_f64]
            desc.n_obs = len(Xobs)
            desc.Xobs, desc.W, desc.alpha = Xobs.data_ptr(), W.data_ptr(), alpha.data_ptr()
            desc.Xobs_f64 = Xobs_f64.data_ptr()
        return desc, keep


def _family_of(base):
    name = type(base).__name__.lower()
    if "rbf" in name:
        return _lib.RBF
    if "matern" in name:
        nu = float(getattr(base, "nu", 2.5))
        if abs(nu - 1.5) < 1e-9:
            return _lib.MATERN15
        if abs(nu - 2.5) < 1e-9:
            return _lib.MATERN25
        raise NotImplementedError(f"Matern nu={nu}: only 1.5 and 2.5 are compiled")
    raise TypeError(f"unsupported base kernel {type(base).__name__} (RBFKernel / MaternKernel expected)")


def _scale_kernel_params(covar):
    if not (hasattr(covar, "base_kernel") and hasattr(covar, "outputscale")):
        raise TypeError("expected a ScaleKernel-like object with .base_kernel and .outputscale")
    base = covar.base_kernel
    return _family_of(base), base.lengthscale.detach().reshape(-1), float(covar.outputscale)


def _model_caches(model):
    """Xobs, W = (K + s2 I)^-1, alpha = W (y - c): BASQ/_gp.py:233-256 (get_cov_cache)."""
    Xobs = model.train_inputs[0]
    ps = getattr(model, "prediction_strategy", None)
    if ps is None:
        # gpytorch builds the strategy lazily on the first eval-mode call (BASQ/_gp.py:249-255)
        model.eval()
        model(Xobs[:1])
        ps = model.prediction_strategy
    S = ps.covar_cache
    return Xobs, _outer_gram(S), ps.mean_cache.double().reshape(-1)


def _outer_gram(S):
    """W = S S^T in fp64 (BASQ/_gp.py:251: woodbury_inv = S @ S.T).  For a CUDA tensor the product runs in
    the library's own DMMA GEMM (basq_dgemm), not in torch.matmul / cuBLAS: the caches are rebuilt on
    every recombination() call of a freshly updated GP, i.e. on the path this library replaces."""
    S64 = S.detach().double().contiguous()
    if not S64.is_cuda:
        return S64 @ S64.T
    import ctypes as C
    ctx = _lib.context_for(S64.device)
    n, r = S64.shape
    W = torch.empty(n, n, dtype=torch.float64, device=S64.device)
    _lib.check(_lib.lib.basq_dgemm(ctx.handle, 0, 1, n, n, r, C.c_double(1.0), S64.data_ptr(), r, S64.data_ptr(), r,
                                   C.c_double(0.0), W.data_ptr(), n))
    return W


def spec_from_model(model, mode, diag_add=0.0, offset=0.0) -> KernelSpec:
    fam, ls, os_ = _scale_kernel_params(model.covar_module)
    mean_const = 0.0
    mm = getattr(model, "mean_module", None)
    if mm is not None and hasattr(mm, "constant"):
        mean_const = float(mm.constant)
    noise = float(torch.as_tensor(model.likelihood.noise).reshape(-1)[0])
    Xobs, W, alpha = _model_caches(model)
    return KernelSpec(fam, mode, ls, os_, noise=noise, mean_const=mean_const, diag_add=diag_add,
                      Xobs=Xobs, W=W, alpha=alpha, offset=offset)


def describe_kernel(kernel) -> KernelSpec:
    """KernelSpec for one of the reference's kernel callables; TypeError otherwise (no fallback)."""
    if isinstance(kernel, KernelSpec):
        return kernel
    owner = getattr(kernel, "__self__", None)
    name = getattr(kernel, "__name__", "")
    if owner is not None and name in _MODE_BY_METHOD and hasattr(owner, "model"):
        mode = _MODE_BY_METHOD[name]
        diag = 0.0
        # BASQ's predictive_covariance adds lik_var to the leading diagonal (BASQ/_gp.py:275-276);
        # SOBER's does not (SOBER/_gp.py:297-304).  Oracle stand-ins carry the flag explicitly.
        flag = getattr(owner, "_diag", None)
        if flag is None:
            flag = type(owner).__module__.split(".")[0] == "BASQ"
        spec = spec_from_model(owner.model, mode, offset=float(getattr(owner, "alpha", 0.0) or 0.0))
        spec.noise_diag = bool(flag)
        if name in ("wsabil_kernel", "wsabim_kernel", "gspace_kernel"):
            diag += float(getattr(owner, "jitter", 0.0) or 0.0)
        spec.diag_add = diag
        return spec
    if owner is not None and name in ("forward", "__call__") and hasattr(owner, "base_kernel"):
        fam, ls, os_ = _scale_kernel_params(owner)
        return KernelSpec(fam, _lib.PLAIN, ls, os_)
    if hasattr(kernel, "model") and hasattr(kernel, "mode"):          # SOBER/_kernel.py
        if kernel.mode not in _MODE_BY_SOBER:
            raise ValueError('mode should be from ["predictive_covariance", '
                             '"weighted_predictive_covariance", "kernel"]')
        mode = _MODE_BY_SOBER[kernel.mode]
        if mode == _lib.PLAIN:
            fam, ls, os_ = _scale_kernel_params(kernel.model.covar_module)
            return KernelSpec(fam, _lib.PLAIN, ls, os_)
        return spec_from_model(kernel.model, mode)
    if hasattr(kernel, "base_kernel") and hasattr(kernel, "outputscale"):
        fam, ls, os_ = _scale_kernel_params(kernel)
        return KernelSpec(fam, _lib.PLAIN, ls, os_)
    raise TypeError(
        f"basq_b200 cannot fuse the kernel callable {kernel!r}: pass one of the reference's kernel objects "
        "(VanillaGP.predictive_kernel, WsabiGP.wsabi{l,m}_kernel, ScaleMmltGP.gspace_kernel, SOBER Kernel, "
        "covar_module.forward) or a basq_b200.KernelSpec.  There is no generic Python-callback fallback.")
