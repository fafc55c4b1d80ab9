"""GPs beyond 4096 observations on the fp32 tensor-core posterior variance and the paths built on it.

A BASQ run appends every batch to the GP (n_obs = 2 + n k after k iterations), so it reaches 1e3 - 1e4
observations.  Up to 4096 L^-1 is prepared by two inversions; beyond, by one blocked Cholesky of the
reversed W (gpvar.cu).  The GPs here are built on the device (basq_b200.gp.FixedGP, noise 1e-2 as in the
other fp32 tests); the references are fp64 torch sums on the device, through the oracle's formulas with
the oracle's kernel function (oracle/gp_kernels.py), on the GP's own W and mean cache."""
import math
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import gp_kernels as ogp  # noqa: E402
from oracle import rchq as orchq  # noqa: E402
from oracle import sampler as osam  # noqa: E402

DEV = torch.device("cuda:0")
D = 10
LS = 2.5
TOL = 2e-4          # test_gpu_kernels.py::test_gp_predict, fp32: rel(mean) < TOL, |var - ref| < 1.2 TOL


def _obs(n_obs, seed, d=D):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return math.sqrt(2.0) * torch.randn(n_obs, d, generator=g, device=DEV, dtype=torch.float64)


def _build(X, family="rbf", nu=2.5, mean_const=0.1, log_targets=False):
    """(library GP, oracle twin): the same observations, W and mean cache; the twin evaluates k with the
    oracle's fp64 kernel function instead of the library's."""
    from basq_b200 import gp as bgp
    y = torch.exp(-0.25 * ((X - 0.5) ** 2).sum(-1)) / 3.0 + 0.1 * torch.sin(X[:, 0])
    if log_targets:
        y = torch.log(y + 1.0)
    if family == "rbf":
        base, obase = bgp.RBFKernel(LS), ogp.RBFKernel(LS)
    else:
        base, obase = bgp.MaternKernel(LS, nu), ogp.MaternKernel(LS, nu)
    model = bgp.FixedGP(X, y, bgp.ScaleKernel(base, 1.0), noise=1e-2, mean_const=mean_const)
    twin = types.SimpleNamespace(train_inputs=model.train_inputs, train_targets=y, likelihood=model.likelihood,
                                 mean_module=model.mean_module, prediction_strategy=model.prediction_strategy,
                                 covar_module=ogp.ScaleKernel(obase, 1.0))
    return model, twin


def _cands(n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (math.sqrt(2.0) * torch.randn(n, D, generator=g, device=DEV)).float()


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-300))


def _check_predict(model, twin, X):
    from basq_b200 import ops
    kern = ogp.VanillaGP(model).predictive_kernel
    mean, var = ops.gp_predict(kern, X)
    m_ref, v_ref = ogp.predict(X.double(), twin)
    assert _rel(mean, m_ref) < TOL
    assert float((var - v_ref).abs().max()) < TOL * 1.2
    return var


@pytest.mark.parametrize("n_obs", [1500, 4096, 4097, 9000, 16384])
def test_gp_predict_large(n_obs):
    model, twin = _build(_obs(n_obs, n_obs))
    _check_predict(model, twin, _cands(4096, 1))


@pytest.mark.parametrize("family,nu", [("matern", 1.5), ("matern", 2.5)])
def test_gp_predict_large_matern(family, nu):
    model, twin = _build(_obs(9000, 9000), family, nu)
    _check_predict(model, twin, _cands(4096, 2))


def test_route_continuity_4096_4097():
    """The 4097th observation lies far from every candidate, so the posterior variance there is the same
    for both GPs: the two L^-1 preparations (two inversions / reversed Cholesky) agree across the switch."""
    X = _obs(4096, 4096)
    far = torch.full((1, D), 60.0, dtype=torch.float64, device=DEV)
    Xc = _cands(4096, 4)
    v0 = _check_predict(*_build(X), Xc)
    v1 = _check_predict(*_build(torch.cat([X, far])), Xc)
    assert float((v0 - v1).abs().max()) < TOL * 1.2


def test_deterministic_large():
    from basq_b200 import ops
    model, _ = _build(_obs(9000, 9000))
    kern = ogp.VanillaGP(model).predictive_kernel
    Xc = _cands(20000, 5)
    m1, v1 = ops.gp_predict(kern, Xc)
    m2, v2 = ops.gp_predict(kern, Xc)
    assert torch.equal(m1, m2) and torch.equal(v1, v2)


@pytest.fixture(scope="module")
def gp6000():
    X = _obs(6000, 6000)
    return {"wsabim": _build(X, mean_const=0.1), "mmlt": _build(X, mean_const=0.0, log_targets=True)}


def test_model_space_moments_6000(gp6000):
    from basq_b200 import ops
    Xc = _cands(4096, 6)
    model, twin = gp6000["wsabim"]
    mean, var = ops.gp_predict(ogp.WsabiGP(model, alpha=0.05).wsabim_kernel, Xc, space=1)
    m_ref, v_ref = ogp.WsabiGP(twin, alpha=0.05).wsabim_predict(Xc.double())
    assert _rel(mean, m_ref) < TOL and _rel(var, v_ref) < TOL
    model, twin = gp6000["mmlt"]
    mean, var = ops.gp_predict(ogp.ScaleMmltGP(model).gspace_kernel, Xc, space=1)
    m_ref, v_ref = ogp.ScaleMmltGP(twin).gspace_predict(Xc.double())
    assert _rel(mean, m_ref) < TOL and _rel(var, v_ref) < TOL


def test_calc_weights_and_lfi_6000(gp6000):
    """The oracle formulas on the library's own moments (tight), and on the fp64 moments (to the fp32 moments'
    accuracy: the weights divide by (var + |mean|) / 2, lfi by sqrt(var))."""
    import basq_b200.sampler as bs
    from basq_b200 import ops
    Xc = _cands(5000, 7)
    model, twin = gp6000["wsabim"]
    kern = ogp.VanillaGP(model).predictive_kernel
    w = bs.calc_weights(kern, Xc, ratio=0.5).cpu().numpy()
    m, v = ops.gp_predict(kern, Xc)
    np.testing.assert_allclose(w, osam.calc_weights(m.cpu().numpy(), v.cpu().numpy(), np.zeros(len(Xc)), 0.5),
                               rtol=1e-9, atol=0)
    m, v = ogp.predict(Xc.double(), twin)
    ref = osam.calc_weights(m.cpu().numpy(), v.cpu().numpy(), np.zeros(len(Xc)), 0.5)
    np.testing.assert_allclose(w, ref, rtol=0, atol=5e-3 * ref.max())
    assert abs(w.sum() - 1.0) < 1e-12
    model, twin = gp6000["mmlt"]
    kern = ogp.ScaleMmltGP(model).gspace_kernel
    p = bs.lfi(kern, Xc).cpu().numpy()
    mg, vg = ops.gp_predict(kern, Xc, space=1)
    np.testing.assert_allclose(p, osam.lfi(mg.cpu().numpy(), vg.cpu().numpy()), rtol=1e-9, atol=1e-15)
    mg, vg = ogp.ScaleMmltGP(twin).gspace_predict(Xc.double())
    np.testing.assert_allclose(p, osam.lfi(mg.cpu().numpy(), vg.cpu().numpy()), rtol=0, atol=1e-3)


@pytest.mark.parametrize("name", ["wsabim", "mmlt"])
def test_recombination_6000(gp6000, name):
    """Non-linear recombination (N = 2e5, M = 2000, n = 200) on a 6000-observation GP: every candidate's
    warp factor goes through the large-GP variance."""
    import basq_b200
    from basq_b200 import ops
    model, _ = gp6000[name]
    kern = ogp.WsabiGP(model, alpha=0.05).wsabim_kernel if name == "wsabim" else ogp.ScaleMmltGP(model).gspace_kernel
    N, M, n = 200_000, 2000, 200
    X = _cands(N, 8)
    Z = X[:M].clone()
    torch.manual_seed(0)
    _, U = basq_b200.ker_svd_sparsify(Z, n - 1, kern, DEV)
    idx, w = ops.recombine(kern, X, Z, U)
    assert 1 <= len(idx) <= n and bool((w > 0).all())
    assert abs(float(w.double().sum()) - 1.0) < 1e-10
    Phi = ops.features(kern, X, Z, U).cpu()
    mu = torch.full((N,), 1.0 / N, dtype=torch.float64)
    assert orchq.moment_residual(Phi, mu, idx.cpu(), w.cpu()) < 1e-8


def test_kernel_quadform_mmlt_6000(gp6000):
    from basq_b200 import ops
    model, twin = gp6000["mmlt"]
    X = _cands(2500, 9)
    g = torch.Generator(device=DEV).manual_seed(10)
    a = torch.randn(len(X), generator=g, device=DEV, dtype=torch.float64)
    q = ops.kernel_quadform(ogp.ScaleMmltGP(model).gspace_kernel, X, a)
    K = ogp.ScaleMmltGP(twin).gspace_kernel(X.double(), X.double())
    S = float(a.abs() @ K.abs() @ a.abs())
    assert abs(q - float(a @ K @ a)) <= TOL * S


def test_limit_32769_observations():
    """One observation beyond the limit: refused as unsupported before anything is computed."""
    from basq_b200 import _lib, ops
    from basq_b200.kernels import KernelSpec
    n = 32769
    spec = KernelSpec(_lib.RBF, _lib.PRED_COV, torch.tensor([LS]), 1.0, noise=1e-2,
                      Xobs=torch.zeros(n, D, device=DEV), W=torch.zeros(n, n, dtype=torch.float64, device=DEV),
                      alpha=torch.zeros(n, dtype=torch.float64, device=DEV))
    with pytest.raises(_lib.BasqError) as e:
        ops.gp_predict(spec, _cands(256, 11))
    assert e.value.code == _lib.ERR_UNSUPPORTED and "32768" in str(e.value)
