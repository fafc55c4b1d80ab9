"""The tensor-core path of the pairwise non-linear kernels (csrc/nlsum.cuh: WSABI-M, MMLT on fp32
inputs) through the C ABI: features (GRAM mode) and set sums (SETSUM mode) against the fp64 oracle and
against the library's own chunked fp64-GEMM path (BASQ_NLSUM=0), recombination moments at moderate and
at BASELINE config 5's full size."""
import math
import os

import pytest
import torch

from oracle import gp_kernels as ogp
from oracle import rchq as orchq

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    import basq_b200
    from basq_b200 import _lib, gp, ops, sampler
    from basq_b200.kernels import spec_from_model
    return basq_b200, _lib, gp, ops, sampler, spec_from_model


def _kern(model, name):
    return ogp.WsabiGP(model, alpha=0.05).wsabim_kernel if name == "wsabim" else ogp.ScaleMmltGP(model).gspace_kernel


@pytest.mark.parametrize("name", ["wsabim", "mmlt"])
@pytest.mark.parametrize("family,nu", [("rbf", 2.5), ("matern", 1.5), ("matern", 2.5)])
@pytest.mark.parametrize("d,n_obs,M,N", [(4, 40, 60, 1500), (10, 130, 300, 5000), (2, 33, 129, 700), (20, 70, 257, 1111)])
def test_features_vs_oracle_and_pairwise_path(lib, monkeypatch, name, family, nu, d, n_obs, M, N):
    """Phi = (U K(Z, X))^T for the non-linear kernels: ragged sizes (n_obs and M not multiples of the
    tile sizes, several padded dimensions); the tensor-core path agrees with the fp64 oracle to the
    accuracy of fp32 kernel values and with the library's fp64-GEMM path to ~1e-6."""
    _, _lib, gp, ops, *_ = lib
    model = ogp.make_gp(d, n_obs, family=family, nu=nu, lengthscale=1.2 * math.sqrt(d), outputscale=1.3, noise=1e-2,
                        seed=7, log_targets=(name == "mmlt"), mean_const=0.1 if name == "wsabim" else 0.0)
    kern = _kern(model, name)
    g = torch.Generator().manual_seed(33 + d)
    X = (math.sqrt(2.0) * torch.randn(N, d, generator=g)).float()
    Z = (math.sqrt(2.0) * torch.randn(M, d, generator=g)).float()
    q = min(11, M - 1)
    U = torch.linalg.qr(torch.randn(M, q, generator=g, dtype=torch.float64)).Q.T.contiguous()
    monkeypatch.setenv("BASQ_NLSUM", "1")
    Phi = ops.features(kern, X.to(DEV), Z.to(DEV), U.to(DEV)).cpu()
    monkeypatch.setenv("BASQ_NLSUM", "0")
    Phi_old = ops.features(kern, X.to(DEV), Z.to(DEV), U.to(DEV)).cpu()
    ref = orchq.features(X.double(), U, Z.double(), kern)
    scale = float(ref.abs().max())
    assert float((Phi - ref).abs().max()) < 3e-4 * scale
    assert float((Phi - Phi_old).abs().max()) < 5e-6 * scale, float((Phi - Phi_old).abs().max()) / scale
    assert float((Phi_old - ref).abs().max()) < 3e-4 * scale


@pytest.mark.parametrize("name", ["wsabim", "mmlt"])
def test_set_sums_match_summed_features(lib, monkeypatch, name):
    """SETSUM mode (8 sets x 32 members per tile, several tiles per set, ragged tails) equals the sum of
    the GRAM-mode features of the same candidates to fp64 accumulation accuracy: both evaluate the same
    fp32 kernel values, so a rule built from the sweeps preserves the library's features to 1e-8."""
    _, _lib, gp, ops, *_ = lib
    monkeypatch.setenv("BASQ_NLSUM", "1")
    d, n_obs, M, N, n = 10, 130, 300, 40_000, 20
    model = ogp.make_gp(d, n_obs, lengthscale=2.5, noise=1e-3, seed=3, log_targets=(name == "mmlt"))
    kern = _kern(model, name)
    g = torch.Generator().manual_seed(5)
    X = (math.sqrt(2.0) * torch.randn(N, d, generator=g)).float().to(DEV)
    Z = X[:M].clone()
    U = torch.linalg.qr(torch.randn(M, n - 1, generator=g, dtype=torch.float64)).Q.T.contiguous().to(DEV)
    sess = ops.Session(kern, X, Z, U, N, 0)
    try:
        A = torch.zeros(sess.n, sess.S, dtype=torch.float64, device=DEV)
        sess.partial(N, 0, A)                    # the reference's round: S = 2 n sets, N / S = 1000 members each
    finally:
        sess.close()
    Phi = ops.features(kern, X, Z, U)            # [N, q]
    S = 2 * n
    sums = torch.zeros(n - 1, S, dtype=torch.float64, device=DEV)
    sums.index_add_(1, torch.arange(N, device=DEV) % S, Phi.T.contiguous())
    sums /= N
    assert float((A[1:] - sums).abs().max()) < 1e-11 * float(sums.abs().max()) + 1e-18
    assert float((A[0] - 1.0 / S).abs().max()) < 1e-15


@pytest.mark.parametrize("name", ["wsabim", "mmlt"])
@pytest.mark.parametrize("weighted", [False, True])
def test_recombination_moments_moderate(lib, monkeypatch, name, weighted):
    basq_b200, _lib, gp, ops, sampler, spec_from_model = lib
    monkeypatch.setenv("BASQ_NLSUM", "1")
    d, N, M, n = 10, 600_000, 2_000, 200
    omodel = ogp.make_gp(d, 202, lengthscale=2.5, noise=1e-4, seed=6, log_targets=(name == "mmlt"))
    kern = _kern(omodel, name)
    X = sampler.sample_mvn(torch.zeros(d), 2.0 * torch.eye(d), N, seed=24, device=DEV)
    Z = X[:M].clone()
    mu = None
    if weighted:
        mu = torch.rand(N, dtype=torch.float64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
        mu[::3] = 0.0
        mu /= mu.sum()
    torch.manual_seed(0)
    _, U = ops.nystrom_basis(kern, Z, n - 1, want_S=False)
    idx, w = ops.recombine(kern, X, Z, U, mu=mu)
    assert 1 <= len(idx) <= n and bool((w > 0).all()) and abs(float(w.sum()) - 1.0) < 1e-11
    rows = torch.randperm(n - 1, generator=torch.Generator().manual_seed(1))[:16].sort().values
    Us = U[rows.to(DEV)].contiguous()
    full = torch.zeros(16, dtype=torch.float64, device=DEV)
    for i in range(0, N, 200_000):
        Ph = ops.features(kern, X[i:i + 200_000], Z, Us)
        full += Ph.sum(0) / N if mu is None else Ph.T @ mu[i:i + 200_000]
    red = ops.features(kern, X[idx], Z, Us).T @ w
    res = float(torch.linalg.norm(full - red) / torch.linalg.norm(full))
    assert res < 1e-8, res
    # and in the ORACLE's features on a subsample: same functions up to fp32 kernel accuracy
    sub = torch.randperm(N, generator=torch.Generator().manual_seed(2))[:4000].to(DEV)
    ref = orchq.features(X[sub].cpu().double(), Us.cpu(), Z.cpu().double(), kern)
    lib_f = ops.features(kern, X[sub], Z, Us).cpu()
    assert float((lib_f - ref).abs().max()) < 1e-4 * float(ref.abs().max())


@pytest.mark.parametrize("name", ["wsabim", "mmlt"])
def test_config5_nonlinear_full_size(lib, monkeypatch, name):
    """BASELINE config 5 at full size for the pairwise kernels: N = 1e7 candidates, M = 1e4 landmarks,
    batch n = 1000, GP with 1002 observations (WSABI-M is the reference's default wsabi_type,
    BASQ/_parameters.py:25; MMLT is Tutorial 03's second model).  Moments of 12 Nystrom test functions
    over ALL candidates are preserved to 1e-8."""
    basq_b200, _lib, gp, ops, sampler, spec_from_model = lib
    monkeypatch.setenv("BASQ_NLSUM", "1")
    d, N, M, n = 10, 10_000_000, 10_000, 1000
    omodel = ogp.make_gp(d, 1002, lengthscale=2.5, noise=1e-10, seed=6 if name == "mmlt" else 5,
                         log_targets=(name == "mmlt"))
    if name == "wsabim":     # square-root warped targets, as WsabiGP trains on them (BASQ/_wsabi.py:60-80)
        omodel = ogp.ExactGP(omodel.train_inputs[0], torch.sqrt(2.0 * omodel.train_targets), omodel.covar_module,
                             noise=1e-10)
    kern = _kern(omodel, name)
    X = sampler.sample_mvn(torch.zeros(d), 2.0 * torch.eye(d), N, seed=23, device=DEV)
    Z = X[:M].clone()
    torch.manual_seed(0)
    _, U = ops.nystrom_basis(kern, Z, n - 1, want_S=False)
    torch.cuda.synchronize()
    import time
    t0 = time.perf_counter()
    idx, w = ops.recombine(kern, X, Z, U)
    torch.cuda.synchronize()
    print(f"[config 5 {name}] recombination of 1e7 candidates: {(time.perf_counter() - t0) * 1e3:.1f} ms")
    assert _lib.context_for(DEV).conditioning()[0] < 64.0
    assert 1 <= len(idx) <= n and bool((w > 0).all()) and abs(float(w.sum()) - 1.0) < 1e-11
    assert bool((idx[1:] > idx[:-1]).all()) and int(idx.max()) < N
    rows = torch.randperm(n - 1, generator=torch.Generator().manual_seed(1))[:12].sort().values
    Us = U[rows.to(DEV)].contiguous()
    full = torch.zeros(12, dtype=torch.float64, device=DEV)
    for i in range(0, N, 1_000_000):
        full += ops.features(kern, X[i:i + 1_000_000], Z, Us).sum(0)
    full /= N
    red = ops.features(kern, X[idx], Z, Us).T @ w
    res = float(torch.linalg.norm(full - red) / torch.linalg.norm(full))
    assert res < 1e-8, res


@pytest.mark.parametrize("name", ["wsabim", "mmlt"])
def test_sharded_sessions_match_one_session(lib, monkeypatch, name):
    """Three rank-local sessions on one GPU (uneven shards, so that the offsets cut through set groups and
    tiles) must produce partial systems whose sum is the single-session system, for the reference's round
    (F = 1) and for a refined pass (F = 4), with and without wrap-around of the cells (GRAM mode)."""
    _, _lib, gp, ops, *_ = lib
    from basq_b200 import sharded
    monkeypatch.setenv("BASQ_NLSUM", "1")
    d, n_obs, M, n = 6, 70, 200, 16
    model = ogp.make_gp(d, n_obs, lengthscale=2.0, noise=1e-3, seed=4, log_targets=(name == "mmlt"))
    kern = _kern(model, name)
    g = torch.Generator().manual_seed(9)
    S = 2 * n
    for N in (7001, 5 * S + 3, S - 5):           # many members per cell / few / fewer points than sets
        X = (math.sqrt(2.0) * torch.randn(N, d, generator=g)).float().to(DEV)
        Z = (math.sqrt(2.0) * torch.randn(M, d, generator=g)).float().to(DEV)
        U = torch.linalg.qr(torch.randn(M, n - 1, generator=g, dtype=torch.float64)).Q.T.contiguous().to(DEV)
        cuts = [0, N // 3 + 1, (2 * N) // 3 - 2, N]
        whole = ops.Session(kern, X, Z, U, N, 0)
        parts = [ops.Session(kern, X[cuts[i]:cuts[i + 1]], Z, U, N, cuts[i]) for i in range(3)]
        try:
            for F in ((1, 4) if N >= 4 * 4 * S else (1,)):
                tree = sharded.LevelTree(S, F, N)
                whole.pass_begin(N, 0, F)
                for i, sp in enumerate(parts):
                    sp.pass_begin(N, cuts[i], F)
                A = torch.zeros(n, S, dtype=torch.float64, device=DEV)
                whole.level(0, tree.node, tree.ppos, tree.fpar, A)
                Asum = torch.zeros_like(A)
                for sp in parts:
                    Ap = torch.zeros_like(A)
                    sp.level(0, tree.node, tree.ppos, tree.fpar, Ap)
                    Asum += Ap
                scale = float(A.abs().max())
                assert float((A - Asum).abs().max()) < 1e-12 * scale, (N, F)
                assert abs(float(A[0].sum()) - 1.0) < 1e-12
        finally:
            whole.close()
            for sp in parts:
                sp.close()
