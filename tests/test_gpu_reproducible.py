"""Reproducible mode (basq_ctx_reproducible / ops.reproducible): the rule of basq_recombine on one GPU and of the
sharded loop over 2-4 ranks with uneven splits and an empty shard are the same bits, for every mode and both
dtypes; the grid-exact fold columns of shard sessions sum to the single session's columns for every compiled
(family, padded dimension) instance; the grid rounding stays within its accuracy bound of the default sums."""
import math
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import gp_kernels as ogp
from oracle import rchq as orchq

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")

# (mode, dtype, weighted mu with zeros, objective row, allow_f32_eval)
CASES = [("plain", torch.float32, False, False, False), ("plain", torch.float64, True, False, False),
         ("pred_cov", torch.float32, True, True, False), ("pred_cov", torch.float64, False, False, False),
         ("wsabil", torch.float32, False, False, False), ("wsabil", torch.float64, True, False, False),
         ("wsabim", torch.float32, True, False, False), ("wsabim", torch.float64, False, True, False),
         ("mmlt", torch.float32, False, False, False), ("mmlt", torch.float64, True, False, False),
         ("pred_cov", torch.float64, True, False, True),
         # 300 observations: the chunked fp64 correction GEMM would split its k-sum by chunk size on small shards
         ("mmlt", torch.float64, True, False, False, 300), ("wsabim", torch.float64, False, False, False, 300)]


def _kernel(mode, dtype, d=4, family="rbf", nu=2.5, n_obs=40):
    if mode == "plain":
        base = ogp.RBFKernel(1.7) if family == "rbf" else ogp.MaternKernel(1.7, nu)
        return ogp.ScaleKernel(base, 1.2).forward
    model = ogp.make_gp(d, n_obs, family=family, nu=nu, lengthscale=1.7, outputscale=1.2,
                        noise=1e-2 if dtype == torch.float32 else 1e-6, seed=7, log_targets=(mode == "mmlt"),
                        mean_const=0.1 if mode.startswith("wsabi") else 0.0)
    return {"pred_cov": ogp.VanillaGP(model).predictive_kernel,
            "wsabil": ogp.WsabiGP(model, alpha=0.05).wsabil_kernel,
            "wsabim": ogp.WsabiGP(model, alpha=0.05).wsabim_kernel,
            "mmlt": ogp.ScaleMmltGP(model).gspace_kernel}[mode]


def _n_obs(case):
    return case[5] if len(case) > 5 else 40


def _problem(case, N=20011, d=4, n=14, seed=44):
    mode, dtype, weighted, with_obj = case[:4]
    M = 600 if _n_obs(case) > 40 else 70
    g = torch.Generator().manual_seed(seed)
    X = (math.sqrt(2.0) * torch.randn(N, d, generator=g, dtype=torch.float64)).to(dtype)
    Z = (math.sqrt(2.0) * torch.randn(M, d, generator=g, dtype=torch.float64)).to(dtype)
    U = torch.linalg.qr(torch.randn(M, n - 1, generator=g, dtype=torch.float64)).Q.T.contiguous()
    mu = obj = None
    if weighted:
        mu = torch.rand(N, generator=g, dtype=torch.float64) ** 2
        mu[torch.rand(N, generator=g) < 0.2] = 0.0
        mu = mu / mu.sum()
    if with_obj:
        obj = -torch.rand(N, generator=g, dtype=torch.float64)
    return X, Z, U, mu, obj


def _bounds(N, world):
    """Uneven shards, the second one empty when world > 2 (as in test_gpu_sharded_sampling.py)."""
    cuts = sorted({0, N} | {int(N * f) for f in (0.15, 0.15, 0.6)[: world - 1]})
    while len(cuts) < world + 1:
        cuts.insert(1, cuts[1])
    return cuts


def _set_mode(_ops, on, f32_eval=False):
    from basq_b200 import _lib
    ctx = _lib.context_for(DEV)
    ctx.reproducible(on)
    ctx.allow_f32_eval(f32_eval)


def _worker(rank, world, rdzv, out_path):
    from basq_b200 import ops, sharded
    dist.init_process_group("gloo", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        rules = []
        for case in CASES:
            _set_mode(ops, True, case[4])
            X, Z, U, mu, obj = _problem(case)
            N = len(X)
            b = _bounds(N, world)
            lo, hi = b[rank], b[rank + 1]
            sess = ops.Session(_kernel(case[0], case[1], n_obs=_n_obs(case)), X[lo:hi].to(DEV), Z.to(DEV), U.to(DEV), N, lo,
                               mu_loc=None if mu is None else mu[lo:hi].to(DEV),
                               obj_loc=None if obj is None else obj[lo:hi].to(DEV))
            try:
                assert sess.reproducible
                idx, w = sharded.recombine_sharded(sess, sess.n, sess.S, device=sess.device)
                rules.append(sharded.gather_result(idx.cpu(), w.cpu(), sess.n))
            finally:
                sess.close()
        # the candidate side: weights, cleansing and SIR on the shards
        _set_mode(ops, True)
        N = 120_001
        lo, hi = _bounds(N, world)[rank], _bounds(N, world)[rank + 1]
        X, raw, kern = _candidates(N)
        cw = sharded.calc_weights_sharded(kern, X[lo:hi].to(DEV), 0.5, N).cpu()
        cl = sharded.cleansing_weights_sharded(raw[lo:hi].to(DEV), N).cpu()
        cws = torch.cat([p.cpu() for p in sharded._all_gather_var(cw, None, False)])
        draws = sharded.sir_indices_sharded(cws[lo:hi].to(DEV), 5000, seed=5, idx_base=lo).cpu()
        _set_mode(ops, False)
        if rank == 0:
            torch.save(rules, out_path)
        torch.save({"cw": cw, "cl": cl, "draws": draws}, f"{out_path}.w{rank}")
    finally:
        dist.destroy_process_group()


def _candidates(N):
    g = torch.Generator().manual_seed(4)
    X = math.sqrt(2.0) * torch.randn(N, 3, generator=g, dtype=torch.float64)
    raw = torch.rand(N, generator=g, dtype=torch.float64) ** 2 * 1e-3
    raw[torch.rand(N, generator=g) < 0.2] = 0.0
    raw[::7] = float("inf")
    model = ogp.make_gp(3, 40, lengthscale=1.6, outputscale=1.2, noise=1e-4, seed=8)
    return X, raw, ogp.VanillaGP(model).predictive_kernel


def _single_gpu_rules():
    from basq_b200 import ops
    rules = []
    for case in CASES:
        _set_mode(ops, True, case[4])
        X, Z, U, mu, obj = _problem(case)
        idx, w = ops.recombine(_kernel(case[0], case[1], n_obs=_n_obs(case)), X.to(DEV), Z.to(DEV), U.to(DEV),
                               mu=None if mu is None else mu.to(DEV), obj=None if obj is None else obj.to(DEV))
        rules.append((idx.cpu(), w.cpu()))
    _set_mode(ops, False)
    return rules


@pytest.fixture(scope="module")
def single_rules():
    return _single_gpu_rules()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_spawned_ranks_recombine_what_one_gpu_recombines(single_rules, world):
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "r.pt")
        mp.spawn(_worker, args=(world, os.path.join(tmp, "rdzv"), out), nprocs=world, join=True)
        rules = torch.load(out)
        parts = [torch.load(f"{out}.w{r}") for r in range(world)]
    for case, (idx, w), (ridx, rw) in zip(CASES, rules, single_rules):
        assert torch.equal(idx, ridx) and torch.equal(w, rw), case
    # weights, cleansing and SIR: the bits of one GPU (sampler's single-call entries in reproducible mode)
    from basq_b200 import sampler
    N = 120_001
    X, raw, kern = _candidates(N)
    _set_mode(None, True)
    try:
        cw = sampler.calc_weights(kern, X.to(DEV), ratio=0.5).cpu()
        cl = sampler.cleansing_weights(raw.to(DEV)).cpu()
        draws = sampler.sir_indices(cw.to(DEV), 5000, seed=5).cpu()
    finally:
        _set_mode(None, False)
    assert torch.equal(torch.cat([p["cw"] for p in parts]), cw)
    assert torch.equal(torch.cat([p["cl"] for p in parts]), cl)
    for p in parts:
        assert torch.equal(p["draws"], draws)
    assert abs(float(cw.sum()) - 1.0) < 1e-12 and abs(float(cl.sum()) - 1.0) < 1e-12


def test_reproducible_rules_keep_the_parity_bars(single_rules):
    """The rule of the reproducible mode keeps the moments (features of the default path) and the total mass."""
    from basq_b200 import ops
    for case, (idx, w) in zip(CASES, single_rules):
        X, Z, U, mu, obj = _problem(case)
        N = len(X)
        full = torch.full((N,), 1.0 / N, dtype=torch.float64) if mu is None else mu
        assert 1 <= len(idx) <= U.shape[0] + 1 and bool((w > 0).all()) and bool((idx[1:] > idx[:-1]).all())
        assert abs(float(w.sum()) - 1.0) < 1e-12, case
        Phi = ops.features(_kernel(case[0], case[1], n_obs=_n_obs(case)), X.to(DEV), Z.to(DEV), U.to(DEV)).cpu()
        # allow_f32_eval: the rule was built from fp32 kernel values, the features are fp64 (test_gpu_recombination.py's
        # bar for fp32 evaluation against fp64 features)
        assert orchq.moment_residual(Phi, full, idx, w) <= (2e-5 if case[4] else 1e-8), case


def test_quadrature_estimate_matches_oracle_in_reproducible_mode():
    """gp.quadrature on the reproducible rule against the oracle's formulas, and the rule's estimate of the
    integral of the GP mean against the full measure's (test_gpu_recombination.py's bars)."""
    from basq_b200 import gp as bgp, ops
    model = ogp.make_gp(4, 40, lengthscale=1.7, outputscale=1.2, noise=1e-6, seed=7)
    vbq = ogp.VanillaGP(model)
    g = torch.Generator().manual_seed(50)
    N, M, n = 5000, 80, 20
    X = math.sqrt(2.0) * torch.randn(N, 4, generator=g, dtype=torch.float64)
    Z = X[:M].clone()
    torch.manual_seed(3)
    _, U = orchq.nystrom_basis(Z, n - 1, vbq.predictive_kernel)
    _set_mode(ops, True)
    try:
        idx, w = ops.recombine(vbq.predictive_kernel, X.to(DEV), Z.to(DEV), U.to(DEV))
    finally:
        _set_mode(ops, False)
    Xs = X[idx.cpu()]
    ez, vz = bgp.quadrature(Xs.to(DEV), w, vbq.predictive_kernel)
    ez_o, vz_o = orchq.quadrature(Xs, w.cpu().double(), vbq.predict_mean, vbq.predictive_kernel)
    assert abs(ez - ez_o) <= 1e-9 * abs(ez_o) and abs(vz - vz_o) <= 1e-7 * abs(vz_o) + 1e-14
    idx_o, w_o = orchq.recombination(X, Z, n, vbq.predictive_kernel, U=U)
    ez_ref = float(w_o @ vbq.predict_mean(X[idx_o]))
    full = float(vbq.predict_mean(X).mean())
    assert abs(ez - full) <= 10.0 * abs(ez_ref - full) + 0.02 * abs(full)


# ---- one process: shard sessions against the single session, every compiled instance ---------------------------
DPS = [2, 4, 6, 8, 10, 12, 16, 20, 24, 32]
FAMILIES = [("rbf", 2.5), ("matern", 1.5), ("matern", 2.5)]


def _sessions(ops, kern, X, Z, U, mu, bounds):
    N = len(X)
    return [ops.Session(kern, X[lo:hi].to(DEV), Z.to(DEV), U.to(DEV), N, lo, mu_loc=mu[lo:hi].to(DEV))
            for lo, hi in zip(bounds[:-1], bounds[1:])]


def s_mass(G):
    """Row of the masses (hi parts) in the [2 (Mtot + 2), K] exact columns."""
    return G.shape[0] // 2 - 2


def _fold(sessions, R, F, counts):
    """Level 0 of a pass over F cells per set on every session: the grid-exact columns of each."""
    mx = np.max(np.stack([s.grid_maxima() for s in sessions]), 0)
    outs = []
    off = 0
    for s, c in zip(sessions, counts):
        s.set_grid(R, mx)
        s.pass_begin(R, off, F)
        off += c
        node = np.arange(s.S, dtype=np.int32)
        Gf = torch.zeros(2 * (s.landmarks() + 2) * s.S, dtype=torch.float64, device=DEV)
        s.level_fold_exact(0, node, Gf)
        outs.append(Gf.view(-1, s.S).cpu())
    return outs


@pytest.mark.parametrize("mode", ["plain", "wsabim", "mmlt"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_shard_folds_sum_to_the_single_session_fold(mode, dtype):
    """Every compiled reproducible (family, padded dimension) instance: fp32 linear modes run the tcgen05 set sums,
    fp32 WSABI-M / MMLT the kind::f16 pairwise kernels, fp64 inputs the CUDA-core kernels (linear and chunked)."""
    from basq_b200 import ops
    _set_mode(ops, True)
    try:
        for fam, nu in FAMILIES:
            for dp in DPS:
                g = torch.Generator().manual_seed(dp)
                N, M, n = 3001, 40, 6
                X = (math.sqrt(2.0) * torch.randn(N, dp, generator=g, dtype=torch.float64)).to(dtype)
                Z = (math.sqrt(2.0) * torch.randn(M, dp, generator=g, dtype=torch.float64)).to(dtype)
                U = torch.linalg.qr(torch.randn(M, n - 1, generator=g, dtype=torch.float64)).Q.T.contiguous()
                mu = torch.rand(N, generator=g, dtype=torch.float64)
                mu[::5] = 0.0
                mu = mu / mu.sum()
                kern = _kernel(mode, dtype, d=dp, family=fam, nu=nu)
                single = _sessions(ops, kern, X, Z, U, mu, [0, N])
                shards = _sessions(ops, kern, X, Z, U, mu, [0, 700, 700, 2400, N])
                try:
                    R = single[0].count()
                    counts = [s.count() for s in shards]
                    assert sum(counts) == R
                    ref = _fold(single, R, 2, [R])[0]
                    parts = _fold(shards, R, 2, counts)
                    tot = torch.zeros_like(ref)
                    for p in parts[::-1]:                   # any order: the sums are exact
                        tot += p
                    assert torch.equal(tot, ref), (fam, nu, dp)
                    assert bool((ref[s_mass(ref)] > 0).all())   # masses
                finally:
                    for s in single + shards:
                        s.close()
    finally:
        _set_mode(ops, False)


def _grids(B, R):
    """(Q, Q2) of session_set_grid for a bound B on sums of at most R terms: Q = 2^(ceil(log2 B) - 51), Q2 the grid
    of the remainders, whose sum is below R Q / 2."""
    Q = math.ldexp(1.0, math.frexp(B)[1] - 51)
    return Q, math.ldexp(1.0, math.frexp(R * Q / 2)[1] - 51)


@pytest.mark.parametrize("mode", ["plain", "pred_cov"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_grid_rounding_meets_the_accuracy_bar(mode, dtype):
    """Reproducible against default columns on the same inputs (the same per-pair kernel values), entry by entry:
    |difference| <= 2^-24 (fp32 inputs: one grid) or 2^-45 (fp64 inputs: hi and lo grids) of the entry's own
    sum_p |w_p k(z_m, x_p)|, plus the grid floor (members) Q_last / 2 - an entry whose terms all lie below the
    finest grid is resolved to that grid and no better, whatever the bar."""
    from basq_b200 import ops
    g = torch.Generator().manual_seed(9)
    N, M, n, d = 20011, 70, 14, 4
    X = (math.sqrt(2.0) * torch.randn(N, d, generator=g, dtype=torch.float64)).to(dtype)
    Z = (math.sqrt(2.0) * torch.randn(M, d, generator=g, dtype=torch.float64)).to(dtype)
    U = torch.linalg.qr(torch.randn(M, n - 1, generator=g, dtype=torch.float64)).Q.T.contiguous()
    mu = torch.rand(N, generator=g, dtype=torch.float64)
    mu = mu / mu.sum()
    kern = _kernel(mode, dtype)
    cols = {}
    for on in (False, True):
        _set_mode(ops, on)
        s = ops.Session(kern, X.to(DEV), Z.to(DEV), U.to(DEV), N, 0, mu_loc=mu.to(DEV))
        try:
            Mtot = s.landmarks()
            F = s.cell_factor(N, N)
            node = np.arange(s.S, dtype=np.int32)
            Gf = torch.zeros(2 * (Mtot + 2) * s.S, dtype=torch.float64, device=DEV)
            if on:
                s.set_grid(N, s.grid_maxima())
                s.pass_begin(N, 0, F)
                s.level_fold_exact(0, node, Gf)
                G = Gf.view(2, Mtot + 2, s.S).cpu()
                cols[on] = G[0, :Mtot] + G[1, :Mtot]
                mass = G[0, Mtot] + G[1, Mtot]
                assert abs(float(mass.sum()) - 1.0) < 1e-13
            else:
                s.pass_begin(N, 0, F)
                s.level_fold(0, node, Gf)
                cols[on] = Gf.view(-1, s.S)[:Mtot].cpu()
        finally:
            s.close()
    _set_mode(ops, False)
    members = torch.zeros(s.S, dtype=torch.float64)
    members.index_add_(0, torch.arange(N) % s.S, torch.ones(N, dtype=torch.float64))
    absum = cols[False].abs()          # w > 0 and k > 0 (RBF): the entry's sum of |w k| (to its own rounding)
    Q, Q2 = _grids(N * float(mu.max()) * 1.2, N)   # B = R max|w| sigma_f^2
    if dtype == torch.float32:
        bar, floor = 2.0 ** -24, members * Q / 2
    else:
        bar, floor = 2.0 ** -45, members * Q2 / 2
    diff = (cols[True] - cols[False]).abs()
    excess = diff - (bar * absum + floor.unsqueeze(0))
    assert float(excess.max()) <= 0.0, (mode, float(excess.max()))
    # the bar is met without the floor wherever an entry's terms reach the grid
    big = absum > 2.0 ** 30 * floor.unsqueeze(0)
    assert bool(big.any()) and bool((diff[big] <= bar * absum[big]).all())


def test_masses_keep_the_total_where_one_grid_would_not():
    """N = 2e6 uniform weights 1 / N: rounded to one grid the masses alone would drift by ~7e-10; the hi / lo grids
    keep sum(w) of the rule to 1e-12."""
    from basq_b200 import ops
    N, M, n, d = 2_000_000, 200, 50, 4
    Q, _ = _grids(N * (1.0 / N), N)
    one_grid = abs(N * (round((1.0 / N) / Q) * Q) - 1.0)
    assert one_grid > 1e-10
    g = torch.Generator(device=DEV).manual_seed(12)
    X = math.sqrt(2.0) * torch.randn(N, d, generator=g, device=DEV, dtype=torch.float32)
    Z = X[:M].clone()
    kern = _kernel("plain", torch.float32)
    _, U = ops.nystrom_basis(kern, Z, n - 1, want_S=False, seed=3)
    _set_mode(ops, True)
    try:
        idx, w = ops.recombine(kern, X, Z, U)
    finally:
        _set_mode(ops, False)
    assert 1 <= len(idx) <= n and abs(float(w.sum()) - 1.0) < 1e-12


def test_non_finite_weight_fails_the_grid():
    from basq_b200 import _lib, ops
    g = torch.Generator().manual_seed(2)
    X = torch.randn(500, 3, generator=g, dtype=torch.float64)
    U = torch.linalg.qr(torch.randn(30, 5, generator=g, dtype=torch.float64)).Q.T.contiguous()
    mu = torch.rand(500, generator=g, dtype=torch.float64)
    mu[17] = float("nan")
    _set_mode(ops, True)
    try:
        s = ops.Session(_kernel("plain", torch.float64), X.to(DEV), X[:30].to(DEV), U.to(DEV), 500, 0, mu_loc=mu.to(DEV))
        try:
            assert math.isnan(s.grid_maxima()[1])
            with pytest.raises(_lib.BasqError):
                s.set_grid(500, s.grid_maxima())
        finally:
            s.close()
    finally:
        _set_mode(ops, False)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_nccl_recombines_what_one_gpu_recombines(single_rules):
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "r.pt")
        mp.spawn(_nccl_worker, args=(2, os.path.join(tmp, "rdzv"), out), nprocs=2, join=True)
        rules = torch.load(out)
    for case, (idx, w), (ridx, rw) in zip(CASES, rules, single_rules):
        assert torch.equal(idx, ridx) and torch.equal(w, rw), case


def _nccl_worker(rank, world, rdzv, out_path):
    from basq_b200 import ops, sharded
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        rules = []
        for case in CASES:
            ops.reproducible(True, dev)
            ops._lib.context_for(dev).allow_f32_eval(case[4])
            X, Z, U, mu, obj = _problem(case)
            N = len(X)
            lo, hi = _bounds(N, world)[rank], _bounds(N, world)[rank + 1]
            sess = ops.Session(_kernel(case[0], case[1], n_obs=_n_obs(case)), X[lo:hi].to(dev), Z.to(dev), U.to(dev), N, lo,
                               mu_loc=None if mu is None else mu[lo:hi].to(dev),
                               obj_loc=None if obj is None else obj[lo:hi].to(dev))
            try:
                idx, w = sharded.recombine_sharded(sess, sess.n, sess.S, device=dev)
                rules.append(tuple(t.cpu() for t in sharded.gather_result(idx, w, sess.n)))
            finally:
                sess.close()
        if rank == 0:
            torch.save(rules, out_path)
    finally:
        dist.destroy_process_group()
