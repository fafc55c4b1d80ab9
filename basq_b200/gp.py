"""Device-side counterparts of the reference's GP helpers that sit on the candidate path.

``predict`` / ``predictive_covariance`` mirror ``BASQ/_gp.py:213-277`` (``SOBER/_gp.py:212-305``) and run
through libbasq_b200.so.  ``FixedGP`` is a minimal fixed-hyper-parameter GP exposing the gpytorch
attribute surface the reference introspects; hyper-parameter fitting is out of scope (SURVEY 2a), its
caches are a one-off n_obs^3 Cholesky done with torch on the device.
"""
from __future__ import annotations

import types

import torch

from . import _lib, ops
from .kernels import KernelSpec, spec_from_model


class _Base:
    def __init__(self, lengthscale, nu=None):
        self.lengthscale = torch.as_tensor(lengthscale, dtype=torch.float64).reshape(1, -1)
        if nu is not None:
            self.nu = nu


class RBFKernel(_Base):
    def __init__(self, lengthscale):
        super().__init__(lengthscale)


class MaternKernel(_Base):
    def __init__(self, lengthscale, nu=2.5):
        super().__init__(lengthscale, nu)


class ScaleKernel:
    def __init__(self, base_kernel, outputscale=1.0):
        self.base_kernel = base_kernel
        self.outputscale = torch.as_tensor(float(outputscale), dtype=torch.float64)

    def forward(self, x, y):
        return ops.gram(self, x, y).to(x.dtype)

    __call__ = forward


class FixedGP:
    """Exact GP with fixed hyper-parameters; K_XX comes from the library's own Gram kernel."""

    def __init__(self, train_x, train_y, covar_module, noise=1e-10, mean_const=0.0, jitter=0.0):
        self.train_inputs = (train_x,)
        self.train_targets = train_y
        self.covar_module = covar_module
        dev = train_x.device
        self.likelihood = types.SimpleNamespace(noise=torch.tensor([float(noise)], dtype=torch.float64, device=dev))
        self.mean_module = types.SimpleNamespace(constant=torch.tensor(float(mean_const), dtype=torch.float64, device=dev))
        K = ops.gram(covar_module, train_x, train_x)
        K = 0.5 * (K + K.T) + (float(noise) + float(jitter)) * torch.eye(len(train_x), dtype=torch.float64, device=dev)
        L = torch.linalg.cholesky(K)
        Linv = torch.linalg.solve_triangular(L, torch.eye(len(train_x), dtype=torch.float64, device=dev), upper=False)
        resid = (train_y.to(torch.float64) - float(mean_const)).unsqueeze(1)
        self.prediction_strategy = types.SimpleNamespace(
            covar_cache=Linv.T.contiguous(), mean_cache=torch.cholesky_solve(resid, L).squeeze(1))

    def eval(self):
        return self


def predict(test_x, model):
    """(mean, variance incl. likelihood noise) - BASQ/_gp.py:213-230 with the exact variance."""
    spec = spec_from_model(model, _lib.PRED_COV)
    mean, var = ops.gp_predict(spec, test_x, space=0, want_var=True)
    return mean.to(test_x.dtype), var.to(test_x.dtype)


def predict_mean(test_x, model):
    spec = spec_from_model(model, _lib.PRED_COV)
    mean, _ = ops.gp_predict(spec, test_x, space=0, want_var=False)
    return mean.to(test_x.dtype)


def predictive_covariance(x, y, model, add_noise_diag=False):
    """K_xy - K_xX W K_Xy - BASQ/_gp.py:259-277 (add_noise_diag=True adds its lik_var diagonal)."""
    spec = spec_from_model(model, _lib.PRED_COV)
    spec.noise_diag = bool(add_noise_diag)
    return ops.gram(spec, x, y).to(x.dtype)


def quadrature(X, w, kernel):
    """KernelQuadrature.quadrature tail (BASQ/_quadrature.py:60-62): EZy = w . m(X), VarZy = w^T K(X,X) w,
    with m the model-space mean of the kernel's mode."""
    mean, _ = ops.gp_predict(kernel, X, space=1, want_var=False)
    K = ops.gram(kernel, X, X)
    w64 = w.to(torch.float64)
    return float(w64 @ mean), float(w64 @ K @ w64)


def full_quadrature(X, w, kernel):
    """SOBER's full_quadrature (SOBER/BASQ/_basq.py:48-81) at candidate scale: the formulas of ``quadrature``,
    EZy = w . m(X) and VarZy = w^T K(X, X) w, with the variance streamed by ops.kernel_quadform instead of
    forming K (N = 1e6 would need 8 TB)."""
    mean, _ = ops.gp_predict(kernel, X, space=1, want_var=False)
    w64 = w.to(device=mean.device, dtype=torch.float64)
    return float(w64 @ mean), ops.kernel_quadform(kernel, X, w64)


def worst_case_error(kernel, X, idx, w, mu=None):
    """Squared worst-case error of the quadrature rule (idx, w) over the candidates X - the rule that
    ``recombination`` returns - in the kernel's RKHS: the squared MMD (mu - w~)^T K (mu - w~) between the rule
    and the candidate measure mu (None: uniform 1/N, as in recombination), where w~ is w scattered to idx.

    It is one quadratic form of a signed measure (ops.kernel_quadform), so the cancellation between the
    measure and the rule happens in the fp64 accumulators.  For fp32 inputs the kernel values are fp32
    (relative error ~2^-21): a rule at that resolution floor may come out as a tiny negative number."""
    device = X.device
    N = len(X)
    if mu is None:
        a = torch.full((N,), 1.0 / N, dtype=torch.float64, device=device)
    else:
        a = mu.to(device=device, dtype=torch.float64).clone()
    idx = torch.as_tensor(idx, device=device).long()
    if idx.numel() != torch.unique(idx).numel():
        raise ValueError("worst_case_error: the rule's indices must be distinct")
    a[idx] -= torch.as_tensor(w, device=device).to(torch.float64)
    return ops.kernel_quadform(kernel, X, a)
