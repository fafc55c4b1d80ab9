"""The reproducible branch of basq_b200.sharded.recombine_sharded on CPU with gloo: worlds 1 to 4, uneven
splits and an empty shard give the same rule bit for bit.  The CUDA session is replaced by an oracle engine with
the same stage interface whose sums are exact: every term is rounded to the pass's power-of-two grid, fixed from
maxima over every rank, as the library's reproducible kernels do.  This exercises the host protocol of the exact
branch - the grid all-reduce (MAX), the cell factor from R_glob alone, the all-reduce of the grid-exact columns
and the full projection on every rank."""
import math
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from basq_b200 import sharded
from oracle import gp_kernels as ogp
from oracle import rchq as orchq


def _grid(B):
    """Q = 2^(ceil(log2 B) - 51) for a bound B on the sum of |terms| (the library's session_set_grid)."""
    return math.ldexp(1.0, (math.frexp(B)[1] if B > 0 else -1000) - 51)


class ExactOracleEngine:
    """count / cell_factor / grid_maxima / set_grid / pass_begin / level_fold_exact / level_project_exact / car /
    apply / result with torch CPU ops (tests only)."""

    reproducible = True

    def __init__(self, X_loc, Z, U, kernel, N_glob, idx_base, mu_loc=None, obj_loc=None):
        self.X, self.Z, self.U, self.kernel = X_loc.double(), Z.double(), U.double(), kernel
        self.mu = torch.full((len(X_loc),), 1.0 / N_glob, dtype=torch.float64) if mu_loc is None else mu_loc.double()
        self.obj = obj_loc.double() if obj_loc is not None else None
        self.idx = torch.arange(len(X_loc)) + idx_base
        live = self.mu != 0
        self.X, self.mu, self.idx = self.X[live], self.mu[live], self.idx[live]
        if self.obj is not None:
            self.obj = self.obj[live]
        self.n = U.shape[0] + 1
        self.S = 2 * self.n
        self.rows = self.n + (1 if obj_loc is not None else 0)
        self.device = "cpu"

    def count(self):
        return len(self.mu)

    def landmarks(self):
        return len(self.Z)                      # level_fold_exact writes 2 (landmarks + 2) rows

    def cell_factor(self, R, R_loc_max):
        F = 1                                    # R_glob only: the cells must not depend on the split
        while F < 4 and R >= 4 * (2 * F) * self.S:
            F *= 2
        return F

    def grid_maxima(self):
        if len(self.mu) == 0:
            return np.zeros(3)
        o = (self.mu * self.obj).abs().max().item() if self.obj is not None else 0.0
        return np.array([self.mu.abs().max().item(), self.mu.abs().max().item(), o])

    def set_grid(self, R, mx):
        # |k| <= 1 for the unit-outputscale RBF kernel
        self.Q = [_grid(R * mx[0]), _grid(R * mx[1]), _grid(R * mx[2])]

    def pass_begin(self, R, off, F):
        self.F = F
        M = len(self.Z)
        self.cellG = torch.zeros(M + 2, F * self.S, dtype=torch.float64)
        if len(self.mu) == 0:
            return
        cells = (off + torch.arange(len(self.mu))) % (F * self.S)
        on_grid = lambda t, Q: torch.round(t / Q) * Q
        self.cellG[:M].index_add_(1, cells, on_grid(self.kernel(self.Z, self.X) * self.mu.unsqueeze(0), self.Q[0]))
        self.cellG[M].index_add_(0, cells, on_grid(self.mu, self.Q[1]))
        if self.obj is not None:
            self.cellG[M + 1].index_add_(0, cells, on_grid(self.mu * self.obj, self.Q[2]))

    def level_fold_exact(self, lvl, node, Gf):
        stride, cnt, K = self.S << lvl, self.F >> lvl, len(node)
        cols = torch.as_tensor(np.asarray(node, dtype=np.int64))
        out = sum(self.cellG[:, cols + k * stride] for k in range(cnt))
        Gf.view(-1, K).zero_()
        Gf.view(-1, K)[:len(out)].copy_(out)       # hi parts; the remainders' rows stay zero (grid-exact terms)

    def level_project_exact(self, lvl, node, ppos, fpar, Gf, A):
        K, M = len(node), len(self.Z)
        G = Gf.view(2, -1, K)
        G = G[0] + G[1]
        raw = torch.cat([G[M:M + 1], self.U @ G[:M]] + ([G[M + 1:M + 2]] if self.rows > self.n else []))
        if lvl > 0:
            raw = torch.cat([raw, self.prev[:, torch.as_tensor(np.asarray(ppos, dtype=np.int64))] - raw], 1)
        self.prev = raw
        A.zero_()
        f = torch.as_tensor(np.asarray(fpar, dtype=np.float64))
        A[:, :raw.shape[1]] = raw * (torch.cat([f, f]) if lvl > 0 else f).unsqueeze(0)

    def car(self, A, C, omega):
        mass = A[0, :C]
        bary = (A[1:self.n, :C] / mass.unsqueeze(0)).T
        w, keep = orchq.caratheodory(bary, mass.clone())
        omega.zero_()
        omega[keep] = w / mass[keep]

    def apply(self, R, off, F, factor):
        scale = factor[(off + torch.arange(len(self.mu))) % (F * self.S)]
        live = scale > 0
        self.X, self.mu, self.idx = self.X[live], (self.mu * scale)[live], self.idx[live]
        if self.obj is not None:
            self.obj = self.obj[live]
        return len(self.mu)

    def result(self):
        return self.idx.clone(), self.mu.clone()


def uneven_bounds(N, world, rank):
    """Contiguous shards of unequal sizes; rank 1 of a world of 3 or more holds nothing."""
    if world == 1:
        return 0, N
    sizes = [N * (r + 1) for r in range(world)]
    if world >= 3:
        sizes[1] = 0
    cuts = np.concatenate([[0], np.cumsum(sizes)]) * N // sum(sizes)
    return int(cuts[rank]), int(cuts[rank + 1])


def _problem(N, weighted, with_obj):
    g = torch.Generator().manual_seed(321)
    d, M, n = 3, 30, 7
    X = math.sqrt(2.0) * torch.randn(N, d, generator=g, dtype=torch.float64)
    Z = math.sqrt(2.0) * torch.randn(M, d, generator=g, dtype=torch.float64)
    U = torch.linalg.qr(torch.randn(M, n - 1, generator=g, dtype=torch.float64)).Q.T.contiguous()
    mu = None
    if weighted:
        mu = torch.rand(N, generator=g, dtype=torch.float64)
        mu[torch.rand(N, generator=g) < 0.3] = 0.0
        mu = mu / mu.sum()
    obj = -torch.rand(N, generator=g, dtype=torch.float64) if with_obj else None
    return X, Z, U, mu, obj


def _run(rank, world, N, weighted, with_obj):
    X, Z, U, mu, obj = _problem(N, weighted, with_obj)
    kern = lambda a, b: ogp.base_kernel(a, b, "rbf", 1.4, 1.0)
    lo, hi = uneven_bounds(N, world, rank)
    eng = ExactOracleEngine(X[lo:hi], Z, U, kern, N, lo, None if mu is None else mu[lo:hi],
                            None if obj is None else obj[lo:hi])
    idx, w = sharded.recombine_sharded(eng, eng.n, eng.S)
    return sharded.gather_result(idx, w, eng.n)


def _worker(rank, world, N, weighted, with_obj, out_path):
    os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")
    dist.init_process_group("gloo", init_method=f"file://{out_path}.rdzv", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        idx, w = _run(rank, world, N, weighted, with_obj)
        if rank == 0:
            torch.save({"idx": idx, "w": w}, out_path)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("N,weighted,with_obj", [(2000, False, False), (1537, True, False), (1200, True, True),
                                                 (20, False, False)])
def test_worlds_return_the_same_rule(tmp_path, N, weighted, with_obj):
    torch.set_num_threads(1)
    ref_idx, ref_w = _run(0, 1, N, weighted, with_obj)
    X, Z, U, mu, obj = _problem(N, weighted, with_obj)
    full_mu = torch.full((N,), 1.0 / N, dtype=torch.float64) if mu is None else mu
    Phi = orchq.features(X, U, Z, lambda a, b: ogp.base_kernel(a, b, "rbf", 1.4, 1.0))
    assert orchq.moment_residual(Phi, full_mu, ref_idx, ref_w) < 1e-10
    assert abs(float(ref_w.sum()) - 1.0) < 1e-12
    for world in (2, 3, 4):
        out = str(tmp_path / f"rule{world}.pt")
        mp.spawn(_worker, args=(world, N, weighted, with_obj, out), nprocs=world, join=True)
        r = torch.load(out)
        assert torch.equal(r["idx"], ref_idx) and torch.equal(r["w"], ref_w), world


def test_uneven_bounds_cover_the_set_with_an_empty_shard():
    for world in (1, 2, 3, 4):
        b = [uneven_bounds(1537, world, r) for r in range(world)]
        assert b[0][0] == 0 and b[-1][1] == 1537 and all(b[r][1] == b[r + 1][0] for r in range(world - 1))
        if world >= 3:
            assert b[1][0] == b[1][1]
