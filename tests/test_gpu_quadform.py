"""Weighted kernel double sums (basq_kernel_quadform / basq_kernel_bilinear) against dense fp64 sums of the oracle's
kernels, and the Python layer on top of them (gp.full_quadrature, gp.worst_case_error,
sharded.kernel_quadform_sharded).  Tolerances are relative to S = sum_ij |a_i| |b_j| |kernel_ij|, the scale of
the sum, with the per-mode tolerances of test_gpu_kernels.py (test_gram_plain / test_gram_modes)."""
import ctypes
import math
import os
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import gp_kernels as ogp

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
D = 10
LS = 1.5 * math.sqrt(D / 2.0)


def _tol(name, dtype):
    if dtype == torch.float64:
        return 1e-11
    return 1e-5 if name == "forward" else 2e-4


def _model(dtype, family="rbf", nu=2.5, n_obs=40, d=D, log_targets=False):
    # fp32 kernel values carry ~1e-7 relative noise that W amplifies: a well-conditioned GP for fp32 inputs
    return ogp.make_gp(d, n_obs, family=family, nu=nu, lengthscale=LS, outputscale=1.2,
                       noise=1e-2 if dtype == torch.float32 else 1e-6, mean_const=0.1, seed=7,
                       log_targets=log_targets)


def _kernel(name, model, diag=False):
    if name == "forward":
        return model.covar_module.forward
    if name == "pred_cov":
        return ogp.VanillaGP(model, add_noise_diag=diag).predictive_kernel
    if name == "wsabil":
        return ogp.WsabiGP(model, alpha=0.05, jitter=1e-3 if diag else 0.0, add_noise_diag=diag).wsabil_kernel
    if name == "wsabim":
        return ogp.WsabiGP(model, alpha=0.05, jitter=1e-3 if diag else 0.0, add_noise_diag=diag).wsabim_kernel
    return ogp.ScaleMmltGP(model, jitter=1e-3 if diag else 0.0).gspace_kernel


def _points(n, seed, d=D):
    g = torch.Generator().manual_seed(seed)
    return math.sqrt(2.0) * torch.randn(n, d, generator=g, dtype=torch.float64)


def _weights(n, seed, zeros=0.3):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(n, generator=g, dtype=torch.float64)
    w[torch.rand(n, generator=g) < zeros] = 0.0
    return w


MODES = ("forward", "pred_cov", "wsabil", "wsabim", "mmlt")
CASES = ([("rbf", 2.5, name) for name in MODES] +
         [(fam, nu, name) for fam, nu in (("matern", 1.5), ("matern", 2.5)) for name in ("forward", "pred_cov")])


@pytest.mark.parametrize("family,nu,name", CASES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("N", [1, 2, 130, 2500])
def test_dense_agreement(family, nu, name, dtype, N):
    from basq_b200 import ops
    kern = _kernel(name, _model(dtype, family, nu, log_targets=(name == "mmlt")))
    X, Y = _points(N, 1), _points(N // 2 + 3, 2)
    a, b = _weights(N, 3), _weights(len(Y), 4)
    if not bool((a != 0).any()):
        a[0] = 0.7
    Xr, Yr = X.to(dtype).double(), Y.to(dtype).double()
    tol = _tol(name, dtype)
    K = kern(Xr, Xr)
    q = ops.kernel_quadform(kern, X.to(DEV, dtype), a.to(DEV))
    S = float(a.abs() @ K.abs() @ a.abs())
    assert abs(q - float(a @ K @ a)) <= tol * S, (q, float(a @ K @ a), S)
    Kxy = kern(Xr, Yr)
    bl = ops.kernel_bilinear(kern, X.to(DEV, dtype), a.to(DEV), Y.to(DEV, dtype), b.to(DEV))
    S = float(a.abs() @ Kxy.abs() @ b.abs())
    assert abs(bl - float(a @ Kxy @ b)) <= tol * S, (bl, float(a @ Kxy @ b), S)


@pytest.mark.parametrize("name", MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_diagonal_terms(name, dtype):
    """noise_diag (before the warping) and diag_add (after it) are part of Q, as in the square basq_gram; with both
    off, Q(X, a) is B(X, a; X, a)."""
    from basq_b200 import ops
    from basq_b200.kernels import describe_kernel
    model = _model(dtype, log_targets=(name == "mmlt"))
    spec = describe_kernel(_kernel(name, model, diag=True))
    spec.noise_diag, spec.diag_add = True, 1e-3
    X, a = _points(700, 5).to(DEV, dtype), _weights(700, 6).to(DEV)
    K = ops.gram(spec, X, X)
    ref = float(a @ K @ a)
    S = float(a.abs() @ K.abs() @ a.abs())
    assert abs(ops.kernel_quadform(spec, X, a) - ref) <= _tol(name, dtype) * S
    spec.noise_diag, spec.diag_add = False, 0.0
    q, bl = ops.kernel_quadform(spec, X, a), ops.kernel_bilinear(spec, X, a, X, a)
    assert abs(q - bl) <= _tol(name, dtype) * S
    assert abs(q - ref) > 1e-6 * S                    # the diagonal terms were not negligible


@pytest.mark.parametrize("name,dtype,N", [("forward", torch.float32, 100_003), ("pred_cov", torch.float32, 100_003),
                                          ("wsabim", torch.float32, 100_003), ("pred_cov", torch.float64, 40_000)])
def test_many_blocks_and_split_identity(name, dtype, N):
    """N = 100 003 spans three landmark blocks of the sweep (148 x 256 rows on a B200), N = 40 000 two: the
    'later rows' sums and blocks that start inside the records, on the tensor-core, the non-linear and the fp64
    set-sum kernels."""
    from basq_b200 import ops
    kern = _kernel(name, _model(dtype))
    X, a = _points(N, 8).to(DEV, dtype), _weights(N, 9).to(DEV)
    ref, S = 0.0, 0.0
    for r0 in range(0, N, 4096):
        Kc = ops.gram(kern, X[r0:r0 + 4096], X)
        ref += float(a[r0:r0 + 4096] @ (Kc @ a))
        S += float(a[r0:r0 + 4096].abs() @ (Kc.abs() @ a.abs()))
        del Kc
    tol = _tol(name, dtype)
    q = ops.kernel_quadform(kern, X, a)
    assert abs(q - ref) <= tol * S, (q, ref, S)
    k = 37_891                                        # odd split row
    q1 = ops.kernel_quadform(kern, X[:k], a[:k])
    q2 = ops.kernel_quadform(kern, X[k:], a[k:])
    b12 = ops.kernel_bilinear(kern, X[:k], a[:k], X[k:], a[k:])
    assert abs(q - (q1 + q2 + 2.0 * b12)) <= tol * S
    assert q == ops.kernel_quadform(kern, X, a)      # bit-reproducible


@pytest.mark.parametrize("name", MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_deterministic(name, dtype):
    from basq_b200 import ops
    kern = _kernel(name, _model(dtype, log_targets=(name == "mmlt")))
    X, Y = _points(5000, 10).to(DEV, dtype), _points(3001, 11).to(DEV, dtype)
    a, b = _weights(5000, 12).to(DEV), _weights(3001, 13).to(DEV)
    assert ops.kernel_quadform(kern, X, a) == ops.kernel_quadform(kern, X, a)
    assert ops.kernel_bilinear(kern, X, a, Y, b) == ops.kernel_bilinear(kern, X, a, Y, b)


def test_f32_eval_of_f64_inputs():
    """basq_ctx_allow_f32_eval: fp64 inputs evaluated on the fp32 path give the fp32-input result."""
    from basq_b200 import _lib, ops
    kern = _kernel("pred_cov", _model(torch.float32))
    X, a = _points(3000, 14), _weights(3000, 15).to(DEV)
    ctx = _lib.context_for(DEV)
    q32 = ops.kernel_quadform(kern, X.float().double().to(DEV).float(), a)
    try:
        ctx.allow_f32_eval(True)
        q = ops.kernel_quadform(kern, X.float().double().to(DEV), a)
    finally:
        ctx.allow_f32_eval(False)
    assert q == q32


def test_f32_eval_counts_a_demotion():
    from basq_b200 import _lib, ops
    kern = _kernel("forward", _model(torch.float64))
    X, a = _points(500, 26).to(DEV), _weights(500, 27).to(DEV)
    ctx = _lib.context_for(DEV)
    try:
        n0 = ctx.allow_f32_eval(True)
        ops.kernel_quadform(kern, X, a)
        assert ctx.allow_f32_eval() == n0 + 1
    finally:
        ctx.allow_f32_eval(False)


def test_stiff_gp_is_promoted():
    """A stiff 2-D GP (40 clustered observations, noise 1e-10: kappa ~ 1e3 > 64, as in test_gpu_parity_gaps): the
    fp32 WSABI-M quadratic form is promoted to the fp64 path and agrees with the fp64 inputs."""
    from basq_b200 import _lib, ops
    model = ogp.make_gp(2, 40, lengthscale=1.0, noise=1e-10, seed=5)
    kern = ogp.WsabiGP(model, alpha=0.05).wsabim_kernel
    X = (math.sqrt(2.0) * torch.randn(3000, 2, generator=torch.Generator().manual_seed(28))).float()
    a = _weights(3000, 29)
    ctx = _lib.context_for(DEV)
    _, n0 = ctx.conditioning()
    q32 = ops.kernel_quadform(kern, X.to(DEV), a.to(DEV))
    kappa, n1 = ctx.conditioning()
    assert kappa > 64.0 and n1 == n0 + 1, (kappa, n0, n1)
    q64 = ops.kernel_quadform(kern, X.double().to(DEV), a.to(DEV))
    Xr = X.double()
    S = float(a.abs() @ kern(Xr, Xr).abs() @ a.abs())
    assert abs(q32 - q64) <= 1e-9 * S, (q32, q64, S)


def test_input_checks():
    from basq_b200 import _lib, ops
    from basq_b200.kernels import describe_kernel
    kern = _kernel("pred_cov", _model(torch.float64))
    X, a = _points(64, 18).to(DEV), _weights(64, 19).to(DEV)
    ctx = _lib.context_for(DEV)
    desc, keep = describe_kernel(kern).to_desc(D, DEV, torch.float64)
    out = ctypes.c_double(0.0)
    assert _lib.lib.basq_kernel_quadform(ctx.handle, ctypes.byref(desc), None, 64, a.data_ptr(),
                                         ctypes.byref(out)) == _lib.ERR_INVALID
    assert _lib.lib.basq_kernel_quadform(ctx.handle, ctypes.byref(desc), X.data_ptr(), 0, a.data_ptr(),
                                         ctypes.byref(out)) == _lib.ERR_INVALID
    assert _lib.lib.basq_kernel_bilinear(ctx.handle, ctypes.byref(desc), X.data_ptr(), 64, a.data_ptr(), None, 64,
                                         a.data_ptr(), ctypes.byref(out)) == _lib.ERR_INVALID
    bad = a.clone()
    bad[17] = float("nan")
    with pytest.raises(_lib.BasqError) as e:
        ops.kernel_quadform(kern, X, bad)
    assert e.value.code == _lib.ERR_NUMERIC
    with pytest.raises(_lib.BasqError) as e:
        ops.kernel_bilinear(kern, X, a, X, bad)
    assert e.value.code == _lib.ERR_NUMERIC


# ------------------------------------------------------------------------------------------- Python layer
@pytest.mark.parametrize("name", ["pred_cov", "wsabil"])
def test_full_quadrature_matches_dense_quadrature(name):
    from basq_b200 import gp
    dtype = torch.float32
    model = _model(dtype)
    kern = ogp.VanillaGP(model).predictive_kernel if name == "pred_cov" else ogp.WsabiGP(model, alpha=0.05).wsabil_kernel
    X = _points(2000, 20).to(DEV, dtype)
    w = torch.rand(2000, generator=torch.Generator().manual_seed(21), dtype=torch.float64).to(DEV)
    w /= w.sum()
    e0, v0 = gp.quadrature(X, w, kern)
    e1, v1 = gp.full_quadrature(X, w, kern)
    assert abs(e1 - e0) <= 1e-12 * abs(e0)
    K = ogp.VanillaGP(model).predictive_kernel(X.double().cpu(), X.double().cpu()) if name == "pred_cov" else \
        kern(X.double().cpu(), X.double().cpu())
    S = float(w.cpu() @ K.abs() @ w.cpu())
    assert abs(v1 - v0) <= 2e-4 * S, (v1, v0, S)


def test_worst_case_error():
    from basq_b200 import gp
    model = _model(torch.float64)
    kern = ogp.VanillaGP(model).predictive_kernel
    N = 3000
    X = _points(N, 22)
    g = torch.Generator().manual_seed(23)
    idx = torch.randperm(N, generator=g)[:60]
    w = torch.rand(60, generator=g, dtype=torch.float64)
    w /= w.sum()
    r = torch.full((N,), 1.0 / N, dtype=torch.float64)
    r[idx] -= w
    K = kern(X, X)
    S = float(r.abs() @ K.abs() @ r.abs())
    e64 = gp.worst_case_error(kern, X.to(DEV), idx.to(DEV), w.to(DEV))
    assert abs(e64 - float(r @ K @ r)) <= 1e-11 * S
    e32 = gp.worst_case_error(kern, X.to(DEV, torch.float32), idx.to(DEV), w.to(DEV))
    assert abs(e32 - e64) <= 2e-4 * S


def test_recombination_rule_beats_uniform_subsample():
    """Config-1 shapes (N = 2e4, M = 200, n = 100, VBQ kernel): the recombination rule has a smaller worst-case
    error than 100 uniformly drawn candidates at weight 1/100."""
    import basq_b200
    from basq_b200 import gp
    g = torch.Generator().manual_seed(0)
    N, d, M, n = 20000, 10, 200, 100
    X = (math.sqrt(2.0) * torch.randn(N, d, generator=g)).to(DEV)
    model = ogp.make_gp(d, 102, lengthscale=2.5, outputscale=1.0, noise=1e-4, seed=1)
    kern = ogp.VanillaGP(model).predictive_kernel
    torch.manual_seed(0)
    idx, w = basq_b200.recombination(X, X[:M].clone(), n, kern, DEV)
    e_rule = gp.worst_case_error(kern, X, idx, w)
    pick = torch.randperm(N, generator=g)[:n].to(DEV)
    e_unif = gp.worst_case_error(kern, X, pick, torch.full((n,), 1.0 / n, dtype=torch.float64, device=DEV))
    print(f"worst-case error^2: recombination rule {e_rule:.4e}, 100 uniform candidates {e_unif:.4e}")
    assert e_rule < e_unif


# ------------------------------------------------------------------------------------------- sharded
def _shard_case():
    kern = _kernel("pred_cov", _model(torch.float32))
    N = 10_001
    return kern, _points(N, 24).float(), _weights(N, 25), 4000


def _worker(rank, world, rdzv, out_path):
    from basq_b200 import sharded
    dist.init_process_group("gloo", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        kern, X, a, cut = _shard_case()
        lo, hi = (0, cut) if rank == 0 else (cut, len(X))
        q = sharded.kernel_quadform_sharded(kern, X[lo:hi].to(DEV), a[lo:hi].to(DEV))
        chk = torch.tensor([q], dtype=torch.float64)
        ref = chk.clone()
        dist.broadcast(ref, 0)
        assert torch.equal(chk, ref)
        if rank == 0:
            torch.save({"q": q}, out_path)
    finally:
        dist.destroy_process_group()


def test_sharded_two_ranks():
    from basq_b200 import ops
    kern, X, a, _ = _shard_case()
    q0 = ops.kernel_quadform(kern, X.to(DEV), a.to(DEV))
    Xr = X.double()
    S = float(a.abs() @ kern(Xr, Xr).abs() @ a.abs())
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "q.pt")
        mp.spawn(_worker, args=(2, os.path.join(tmp, "rdzv"), out), nprocs=2, join=True)
        q = torch.load(out)["q"]
    assert abs(q - q0) <= 2e-4 * S, (q, q0, S)
