"""Every compiled (kernel family, padded dimension) instance of the fp32 tensor-core kernels against fp64
references.

The fp32 hot path is instantiated once per kernel family and per padded dimension DP (``padded_dim`` in
csrc/common.cuh), and every instance is its own program: register allocation, shared-memory layout and
pipeline configuration differ by DP.
  * setsum_mma_kernel + build_lmA_kernel (linear set sums): KA = 3 DP + 6 rounded up to 16; NT = 128 points
    per tile at DP = 32 and 256 below; single-buffered landmark tiles at DP 20, 24 and 32.
  * gpvar_fused_kernel (posterior mean and variance): the observation staging stride, register pressure.
  * nlsum_kernel + kxgen_kernel (WSABI-M / MMLT set sums and features): the generator layout.
Each DP runs at d = DP (the bucket full) and at d = previous bucket + 1 (padding lanes live), for the three
families.  The references are the oracle's formulas (oracle/gp_kernels.py, oracle/rchq.py) evaluated in fp64
on the device, on the same inputs: every coordinate lies on a 2^-12 grid, so it is exact in fp32 and stays
exact under the translations of the edge cases.  Lengthscales grow like sqrt(d), and every case checks that
its fp64 kernel matrix is neither ~0 nor ~constant.

Set sums are compared entry by entry against the magnitude of the summed terms,
|A - ref| <= tau (|U'| T |mu|), T the pairwise magnitude of every quantity the library evaluates in fp32
(_magnitudes): a max-relative bound would let cancellation in U hide errors.

Tolerances, from the errors measured on one NVIDIA B200 (1000 W power limit) over every case of this file.
  * Posterior mean and variance keep the suite's fp32 bounds (test_gpu_kernels.py::test_gp_predict):
    relative mean error < 2e-4 (worst measured 8.9e-6), variance error < 2.4e-4 of the outputscale (worst 6.7e-6).
  * TAU_LIN = 5e-7 for the linear set sums: worst measured 1.6e-7 (3x margin).  A set-sum kernel that drops
    the lo half of the candidates' fp16 coordinates errs by 1.5e-6 .. 5e-5 here, at every DP.
  * TAU_NL = 5e-7 for the non-linear set sums and features: worst measured 8.1e-8 (6x margin)."""
import math
import os
import re

import pytest
import torch

from oracle import gp_kernels as ogp
from oracle import rchq as orchq

gpu = pytest.mark.gpu
DEV = torch.device("cuda:0")
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "basq_b200", "csrc")

DPS = [2, 4, 6, 8, 10, 12, 16, 20, 24, 32]
# (d = DP, d = previous bucket + 1) for every bucket
DIMS = [d for i, dp in enumerate(DPS) for d in (dp, (DPS[i - 1] if i else 0) + 1)]
FAMS = ["rbf", "matern15", "matern25"]

MEAN_TOL = 2e-4       # relative to max |mean|
VAR_TOL = 2.4e-4      # relative to the outputscale
TAU_LIN = 5e-7        # linear set sums, against the magnitude of the summed terms
TAU_NL = 5e-7         # non-linear set sums and features, likewise


# ------------------------------------------------------------------------------ the list of compiled instances
def _switch_cases(path, func):
    src = open(os.path.join(CSRC, path)).read()
    m = re.search(re.escape(func) + r"\([^)]*\)\s*\{[^{}]*?switch \([\w.]+\) \{(.*?)\}", src, re.S)
    assert m, f"{func} not found in {path}"
    return [int(c) for c in re.findall(r"case (\d+):", m.group(1))]


def test_instance_lists_match_the_tested_buckets():
    """Every padded dimension that has compiled kernels is one that the matrix below runs, and the other way
    round: a bucket added to padded_dim or to one launcher without tests fails here."""
    src = open(os.path.join(CSRC, "common.cuh")).read()
    m = re.search(r"padded_dim\(int d\)\s*\{\s*const int opts\[\] = \{([^}]*)\}", src)
    assert m
    assert [int(v) for v in m.group(1).split(",")] == DPS
    for path, func in [("setsum_mma.cuh", "launch_setsum_mma_family"), ("setsum_mma_prep.cu", "bool cfg"),
                       ("setsum_mma_prep.cu", "int build_lmA"), ("gpvar.cuh", "launch_gpvar_fused_family"),
                       ("nlsum.cuh", "launch_nlsum_family"), ("nlsum.cuh", "launch_kxgen_family")]:
        assert _switch_cases(path, func) == DPS, (path, func)


# ------------------------------------------------------------------------------ inputs
@pytest.fixture(scope="module")
def lib():
    import basq_b200  # noqa: F401
    from basq_b200 import _lib, ops
    return _lib, ops


def _grid(t):
    """Round to a multiple of 2^-12: exact in fp32 for |t| < 2^11, also after the translations below."""
    return torch.round(t * 4096.0) / 4096.0


def _points(n, d, seed, spread=math.sqrt(2.0)):
    g = torch.Generator().manual_seed(seed)
    return _grid(torch.as_tensor(spread, dtype=torch.float64) * torch.randn(n, d, generator=g, dtype=torch.float64))


def _ls(d):
    return 1.2 * math.sqrt(d)


def _gp(fam, Xobs, ls, os_=1.0, name="pred_cov"):
    """Oracle GP with fixed hyper-parameters on the device (noise 1e-2 of the outputscale, as in the other
    fp32 tests).  MMLT trains on log targets with a zero mean, the other modes on raw targets."""
    Xobs = Xobs.cpu()
    t = (Xobs - Xobs.mean(0)) / torch.as_tensor(ls, dtype=torch.float64)     # translation-invariant targets
    y = torch.exp(-0.5 * ((t - 0.3) ** 2).sum(-1)) / 3.0 + 0.1 * torch.sin(2.0 * t[:, 0])
    if name == "mmlt":
        y = torch.log(y + 1.0)
    base = ogp.RBFKernel(ls) if fam == "rbf" else ogp.MaternKernel(ls, 1.5 if fam == "matern15" else 2.5)
    return ogp.ExactGP(Xobs, math.sqrt(os_) * y, ogp.ScaleKernel(base, os_), noise=1e-2 * os_,
                       mean_const=0.0 if name == "mmlt" else 0.1 * math.sqrt(os_)).to(DEV)


def _kernel(model, name):
    return {"forward": model.covar_module.forward,
            "pred_cov": ogp.VanillaGP(model).predictive_kernel,
            "wsabim": ogp.WsabiGP(model, alpha=0.05).wsabim_kernel,
            "mmlt": ogp.ScaleMmltGP(model).gspace_kernel}[name]


def _basis(q, M, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.linalg.qr(torch.randn(M, q, generator=g, dtype=torch.float64)).Q.T.contiguous().to(DEV)


def _weights(N, seed):
    g = torch.Generator().manual_seed(seed)
    return ((0.25 + torch.rand(N, generator=g, dtype=torch.float64)) / N).to(DEV)


def _assert_nontrivial(K, os_):
    med = float(K.median()) / os_
    assert 0.05 < med < 0.9, f"degenerate test kernel: median k / outputscale = {med}"


# ------------------------------------------------------------------------------ references
def _per_set(V, S):
    """[rows, N] -> [rows, S]: column j sums the points p = j (mod S)."""
    out = torch.zeros(V.shape[0], S, dtype=V.dtype, device=V.device)
    return out.index_add_(1, torch.arange(V.shape[1], device=V.device) % S, V)


def _magnitudes(model, name, X, Z, U):
    """(U', T): the landmarks' projection and the [landmarks, N] magnitudes of the pairwise terms the library
    evaluates.  An error of relative size eps in every fp32 quantity moves a set sum by at most eps |U'| T |mu|.
      forward   k(z, x);
      pred_cov  k(z, x) on Z and k(xo, x) on the observations, which the projection U' = [U, -U Az] joins;
      wsabim    m_z m_x C + C^2 / 2 with C = k(z, x) - Az k(Xobs, x): |C| and the means m carry
                |k| + |Az| k(Xobs, x) and |c| + |alpha| k(Xobs, .);
      mmlt      g_z g_x (e^C - 1), g = exp(m + v / 2) - 1: as above, v carries the outputscale + noise."""
    cov = model.covar_module.forward
    Kzx = cov(Z, X)
    if name == "forward":
        return U, Kzx
    W, Xobs, noise = ogp.get_cov_cache(model)
    Kzo = cov(Z, Xobs)
    Az = Kzo @ W
    Kox = cov(Xobs, X)
    if name == "pred_cov":
        return torch.cat([U, -(U @ Az)], 1), torch.cat([Kzx, Kox], 0)
    C = Kzx - Az @ Kox
    Ca = (Kzx + Az.abs() @ Kox).abs()
    alpha = model.prediction_strategy.mean_cache.abs()
    c0 = abs(float(model.mean_module.constant))
    Mz, Mx = c0 + Kzo @ alpha, c0 + Kox.T @ alpha
    mz, vz = ogp.predict(Z, model)
    mx, vx = ogp.predict(X, model)
    if name == "wsabim":
        T = (mz.abs()[:, None] * mx.abs()[None] + C.abs()) * Ca \
            + C.abs() * (Mz[:, None] * mx.abs()[None] + mz.abs()[:, None] * Mx[None])
    else:
        base = float(model.covar_module.outputscale) + float(noise)
        gz, gx = torch.exp(mz + 0.5 * vz) - 1.0, torch.exp(mx + 0.5 * vx) - 1.0
        eC = torch.exp(C)
        T = (gz.abs()[:, None] * gx.abs()[None]) * eC * Ca \
            + (eC - 1.0).abs() * ((gz + 1.0)[:, None] * gx.abs()[None] * (Mz + base)[:, None]
                                  + gz.abs()[:, None] * (gx + 1.0)[None] * (Mx + base)[None])
    return U, T


def _session_sums(lib, kern, X, Z, U, mu):
    """A [n, S] of the reference's round (row 0 the set masses, rows 1.. the projected set sums), asserting
    that the conditioning guard kept the fp32 inputs on the fp32 kernels."""
    _lib, ops = lib
    promotions = _lib.context_for(DEV).conditioning()[1]
    sess = ops.Session(kern, X.float(), Z.float(), U, len(X), 0, mu_loc=mu)
    try:
        A = torch.zeros(sess.n, sess.S, dtype=torch.float64, device=DEV)
        sess.partial(len(X), 0, A)
    finally:
        sess.close()
    assert _lib.context_for(DEV).conditioning()[1] == promotions, "promoted to fp64: the fp32 kernels did not run"
    return A


def _check_set_sums(lib, model, name, X, Z, U, mu, tau):
    """Library set sums of `name` against the fp64 oracle sums sum_{p = j mod S} mu_p Phi_ref(x_p); returns
    (library A, worst error in units of the terms' magnitude)."""
    kern = _kernel(model, name)
    A = _session_sums(lib, kern, X, Z, U, mu)
    S = A.shape[1]
    assert bool(torch.isfinite(A).all())
    Phi = orchq.features(X, U, Z, kern)                               # [N, q]
    ref = _per_set((Phi * mu[:, None]).T, S)
    Up, T = _magnitudes(model, name, X, Z, U)
    scale = Up.abs() @ _per_set(T * mu.abs(), S)
    err = float(((A[1:] - ref).abs() / scale.clamp_min(1e-300)).max())
    assert err < tau, f"{name}: set sums off by {err:.3g} of the terms' magnitude"
    mass = _per_set(mu[None], S)[0]
    assert float((A[0] - mass).abs().max()) <= 1e-14 * float(mass.max())
    return A, err


def _check_features(lib, model, name, X, Z, U, tau):
    """GRAM mode of the non-linear kernels (one cell per candidate) against the oracle's features."""
    _lib, ops = lib
    kern = _kernel(model, name)
    promotions = _lib.context_for(DEV).conditioning()[1]
    Phi = ops.features(kern, X.float(), Z.float(), U)
    assert _lib.context_for(DEV).conditioning()[1] == promotions
    ref = orchq.features(X, U, Z, kern)
    Up, T = _magnitudes(model, name, X, Z, U)
    err = float(((Phi - ref).abs() / (Up.abs() @ T).T.clamp_min(1e-300)).max())
    assert err < tau, f"{name}: features off by {err:.3g} of the terms' magnitude"
    return err


def _check_predict(lib, model, X):
    """fp32 gp_predict (gpvar_fused_kernel) against the oracle's exact posterior; returns (mean, var, errors)."""
    _, ops = lib
    mean, var = ops.gp_predict(ogp.VanillaGP(model).predictive_kernel, X.float())
    m_ref, v_ref = ogp.predict(X, model)
    assert bool(torch.isfinite(mean).all()) and bool(torch.isfinite(var).all())
    os_ = float(model.covar_module.outputscale)
    e_mean = float((mean - m_ref).abs().max() / m_ref.abs().max())
    e_var = float((var - v_ref).abs().max()) / os_
    assert e_mean < MEAN_TOL, f"posterior mean off by {e_mean:.3g} (relative)"
    assert e_var < VAR_TOL, f"posterior variance off by {e_var:.3g} of the outputscale"
    return mean, var, e_mean, e_var


# sizes of the matrix: two 256-wide observation tiles (the second partial), a partial last candidate tile
N_PRED, NOBS_PRED = 1000, 300
# set sums: M = 300 landmarks (the second tile of a work item partly empty), n = 13 -> S = 26 sets (not a
# multiple of the 8 sets of a work item), 75 or 76 members per set (the last record tile partial for 32 and for
# 16 members per tile, i.e. NT = 256 and NT = 128), 37 observations (joined to the landmarks in pred_cov)
N_SET, M_SET, Q_SET, NOBS_SET = 26 * 75 + 11, 300, 12, 37


def _set_inputs(d, seed, spread=math.sqrt(2.0)):
    X = _points(N_SET, d, seed, spread).to(DEV)
    Z = _points(M_SET, d, seed + 1, spread).to(DEV)
    return X, Z, _basis(Q_SET, M_SET, seed + 2), _weights(N_SET, seed + 3)


# ------------------------------------------------------------------------------ 1. the instance matrix
@gpu
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam", FAMS)
def test_gp_predict_instance(lib, fam, d):
    """gpvar_fused_kernel<FAM, DP>: posterior mean and variance of 1000 candidates, 300 observations."""
    model = _gp(fam, _points(NOBS_PRED, d, 10 * d).to(DEV), _ls(d))
    X = _points(N_PRED, d, 10 * d + 1).to(DEV)
    _assert_nontrivial(model.covar_module.forward(X, model.train_inputs[0]), 1.0)
    _check_predict(lib, model, X)


@gpu
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam", FAMS)
def test_linear_set_sums_instance(lib, fam, d):
    """setsum_mma_kernel<FAM, DP> + build_lmA_kernel<DP>: the plain kernel, and the posterior covariance whose
    observations join the landmarks."""
    X, Z, U, mu = _set_inputs(d, 20 * d)
    model = _gp(fam, _points(NOBS_SET, d, 20 * d + 5).to(DEV), _ls(d))
    _assert_nontrivial(model.covar_module.forward(Z, X), 1.0)
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_LIN)


@gpu
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam", FAMS)
def test_nonlinear_set_sums_instance(lib, fam, d):
    """nlsum_kernel<FAM, DP, NL, SETSUM> + kxgen_kernel<FAM, DP> for WSABI-M and MMLT."""
    X, Z, U, mu = _set_inputs(d, 30 * d)
    Xobs = _points(NOBS_SET, d, 30 * d + 5).to(DEV)
    for name in ("wsabim", "mmlt"):
        model = _gp(fam, Xobs, _ls(d), name=name)
        _assert_nontrivial(model.covar_module.forward(Z, X), 1.0)
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_NL)


@gpu
@pytest.mark.parametrize("dp", [6, 8, 12, 16, 24, 32])     # test_gpu_nlsum.py runs GRAM mode at DP 2, 4, 10, 20
@pytest.mark.parametrize("fam", FAMS)
def test_nonlinear_features_instance(lib, fam, dp):
    """nlsum_kernel<FAM, DP, NL, GRAM>: features of 700 candidates against 257 landmarks, 70 observations."""
    X, Z, U = _points(700, dp, 40 * dp).to(DEV), _points(257, dp, 40 * dp + 1).to(DEV), _basis(11, 257, 40 * dp + 2)
    Xobs = _points(70, dp, 40 * dp + 3).to(DEV)
    for name in ("wsabim", "mmlt"):
        model = _gp(fam, Xobs, _ls(dp), name=name)
        _assert_nontrivial(model.covar_module.forward(Z, X), 1.0)
        _check_features(lib, model, name, X, Z, U, TAU_NL)


# ------------------------------------------------------------------------------ 2. edge inputs
@gpu
@pytest.mark.parametrize("d", [9, 32])
@pytest.mark.parametrize("fam", FAMS)
def test_landmarks_are_candidates(lib, fam, d):
    """Z = X[:M], as BASQ draws the landmarks: the self pairs have r^2 ~ 0 after cancellation (the Matern
    max(arg, 0) clamp).  The posterior at the observations themselves: the variance is the noise plus a small
    non-negative latent variance."""
    X, _, U, mu = _set_inputs(d, 50 * d)
    Z = X[:M_SET].clone()
    model = _gp(fam, _points(NOBS_SET, d, 50 * d + 5).to(DEV), _ls(d))
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_LIN)
    Xobs = model.train_inputs[0]
    _, var, _, _ = _check_predict(lib, model, Xobs)
    noise = float(model.likelihood.noise)
    assert float(var.min()) > noise - VAR_TOL and float(var.max()) < 2.0 * noise + VAR_TOL


@gpu
@pytest.mark.parametrize("fam", FAMS)
def test_translation(lib, fam):
    """A common offset of 40 lengthscales per coordinate (exact in fp32 on the inputs' grid) changes nothing:
    the fp32 expansions centre on the landmark mean (set sums) and on the observation mean (prediction)."""
    d = 13
    shift = _grid(torch.tensor(40.0 * _ls(d), dtype=torch.float64))
    X, Z, U, mu = _set_inputs(d, 60)
    Xobs = _points(NOBS_SET, d, 65).to(DEV)
    Xp = _points(N_PRED, d, 66).to(DEV)
    m0, m1 = _gp(fam, Xobs, _ls(d)), _gp(fam, Xobs + shift, _ls(d))
    for name in ("forward", "pred_cov"):
        A0, _ = _check_set_sums(lib, m0, name, X, Z, U, mu, TAU_LIN)
        A1, _ = _check_set_sums(lib, m1, name, X + shift, Z + shift, U, mu, TAU_LIN)
        Up, T = _magnitudes(m0, name, X, Z, U)
        scale = Up.abs() @ _per_set(T * mu, A0.shape[1])
        assert float(((A1[1:] - A0[1:]).abs() / scale).max()) < TAU_LIN
    mean0, var0, _, _ = _check_predict(lib, m0, Xp)
    mean1, var1, _, _ = _check_predict(lib, m1, Xp + shift)
    assert float((mean1 - mean0).abs().max() / mean0.abs().max()) < MEAN_TOL
    assert float((var1 - var0).abs().max()) < VAR_TOL


@gpu
@pytest.mark.parametrize("d", [9, 32])
@pytest.mark.parametrize("fam", FAMS)
def test_far_candidates(lib, fam, d):
    """Candidates 300 lengthscales from the cloud: |x'|^2 exceeds the +-6e4 fp16 range of the set-sum operands
    (split2h / clamp_h).  Their kernel values are 0, never NaN or inf, the other members of their sets are
    unaffected, and the posterior there is the prior: the constant mean and outputscale + noise."""
    X, Z, U, mu = _set_inputs(d, 70 + d)
    far = torch.tensor([3, 100, 101, 777, N_SET - 1], device=DEV)
    X[far] = _grid(torch.tensor(300.0 * _ls(d), dtype=torch.float64)) * torch.tensor(
        [1.0, -1.0, 1.0, 1.0, -1.0], dtype=torch.float64, device=DEV)[:, None]
    model = _gp(fam, _points(NOBS_SET, d, 75 + d).to(DEV), _ls(d))
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_LIN)
    mean, var, _, _ = _check_predict(lib, model, X[:N_PRED])
    prior = float(model.covar_module.outputscale) + float(model.likelihood.noise)
    c0 = float(model.mean_module.constant)
    assert float((var[far[:4]] - prior).abs().max()) < VAR_TOL
    assert float((mean[far[:4]] - c0).abs().max()) < MEAN_TOL * float(mean.abs().max())


@gpu
@pytest.mark.parametrize("os_", [1e-6, 1e4])
@pytest.mark.parametrize("fam", FAMS)
def test_outputscale_extremes(lib, fam, os_):
    """Outputscales 1e-6 and 1e4 (noise scaled along): kx_scale of the variance and non-linear operands,
    log2_os and os_f of the fp32 expansion; errors relative to the outputscale."""
    d = 9
    X, Z, U, mu = _set_inputs(d, 80)
    Xobs = _points(NOBS_SET, d, 85).to(DEV)
    model = _gp(fam, Xobs, _ls(d), os_=os_)
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_LIN)
    _check_set_sums(lib, _gp(fam, Xobs, _ls(d), os_=os_, name="wsabim"), "wsabim", X, Z, U, mu, TAU_NL)
    _check_predict(lib, _gp(fam, _points(NOBS_PRED, d, 86).to(DEV), _ls(d), os_=os_), X[:N_PRED])


@gpu
@pytest.mark.parametrize("fam", FAMS)
def test_ard_lengthscales(lib, fam):
    """Lengthscales from 0.3 to 30 across d = 13 (DP = 16); the points spread along each axis in proportion
    to its lengthscale, so that every dimension moves the kernel values."""
    d = 13
    ls = 0.3 * 100.0 ** (torch.arange(d, dtype=torch.float64) / (d - 1))
    spread = 0.35 * ls
    X, Z, U, mu = _set_inputs(d, 90, spread=spread)
    model = _gp(fam, _points(NOBS_SET, d, 95, spread).to(DEV), ls)
    _assert_nontrivial(model.covar_module.forward(Z, X), 1.0)
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_LIN)
    _check_predict(lib, _gp(fam, _points(NOBS_PRED, d, 96, spread).to(DEV), ls), _points(N_PRED, d, 97, spread).to(DEV))


@gpu
@pytest.mark.parametrize("N", [1, 127, 129, 257])
@pytest.mark.parametrize("fam", FAMS)
def test_ragged_candidates(lib, fam, N):
    """Candidate counts around the 128-row variance tile and the record tiles (d = 17, DP = 20: the
    single-buffered landmark pipeline)."""
    d = 17
    X, Z, U, mu = _set_inputs(d, 100 + N)
    model = _gp(fam, _points(NOBS_SET, d, 105 + N).to(DEV), _ls(d))
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X[:N], Z, U, mu[:N], TAU_LIN)
    _check_predict(lib, _gp(fam, _points(NOBS_PRED, d, 106 + N).to(DEV), _ls(d)), X[:N])


@gpu
@pytest.mark.parametrize("M", [1, 129, 257])
@pytest.mark.parametrize("fam", FAMS)
def test_ragged_landmarks(lib, fam, M):
    """Landmark counts around the 128-row landmark tile and the two-tile work item (d = 17, DP = 20)."""
    d = 17
    X, _, _, mu = _set_inputs(d, 110 + M)
    Z = _points(M, d, 111 + M).to(DEV)
    U = _basis(min(Q_SET, M), M, 112 + M)
    model = _gp(fam, _points(NOBS_SET, d, 115 + M).to(DEV), _ls(d))
    for name in ("forward", "pred_cov"):
        _check_set_sums(lib, model, name, X, Z, U, mu, TAU_LIN)


@gpu
@pytest.mark.parametrize("n_obs", [1, 31, 33, 255, 257, 513, 769])
@pytest.mark.parametrize("fam", FAMS)
def test_ragged_observations(lib, fam, n_obs):
    """Observation counts across the 32-observation K block and the 256-column tile, with odd numbers of
    column tiles: the fused kernel processes column tiles in pairs."""
    d = 17
    model = _gp(fam, _points(n_obs, d, 120 + n_obs).to(DEV), _ls(d))
    _check_predict(lib, model, _points(N_PRED, d, 121 + n_obs).to(DEV))
