"""Recombination of a candidate set sharded over ranks (one process per GPU).

Per Tchernychova-Lyons pass every rank forms the barycentre numerators of ITS points
(cell = global position mod F*S) in one sweep of kernel evaluations; for each of the pass's
Caratheodory levels one all-reduce sums the small [n, S] system over NVLink, every rank runs the
same deterministic Caratheodory kernel on the identical reduced system, and at the end of the pass
rescales / compacts its own shard.  Counts and offsets after a round follow analytically from the kept sets,
so the collectives on the data path are that all-reduce (SURVEY 8e) and, under NCCL, a
reduce-scatter of the level's folded set-sum columns by landmark rows in front of it, which lets
every rank project 1/G of the rows instead of repeating the whole fp64 projection.

The loop is written against a tiny engine interface so the host logic can be exercised on CPU with
gloo and an oracle-backed engine (tests/test_sharded_gloo.py); the product engine is ops.Session.
"""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(N, world, rank):
    """Contiguous shard [lo, hi) of N candidates for `rank`."""
    base, rem = divmod(N, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def kept_before(g, S, keep_prefix, K):
    """Number of kept points among global positions < g when the kept sets have exclusive prefix
    counts keep_prefix[0..S] (keep_prefix[S] = K)."""
    e, j = divmod(int(g), S)
    return e * K + int(keep_prefix[j])


class LevelTree:
    """Host bookkeeping of one pass (mirror of LevelTree in csrc/api.cu): which nodes of the cell
    hierarchy are presented to the next Caratheodory level.  Node u of level l = cells
    u + k * S * 2^l; its children are u (low half) and u + S * 2^l (high half).  numpy arrays
    throughout (int32 node ids / parent columns, fp64 factors): they go to the C ABI as they are."""

    def __init__(self, S, F, R_glob):
        self.S, self.F, self.L, self.lvl = S, F, F.bit_length() - 1, 0
        S0 = min(S, R_glob)
        self.node = np.arange(S0, dtype=np.int32)
        self.ppos = np.zeros(S0, dtype=np.int32)
        self.fpar = np.ones(S0, dtype=np.float64)
        self.act, self.fac = self.node, self.fpar

    def columns(self):
        return len(self.act)

    def advance(self, om, factor):
        """Consume the level's factors om (1 = untouched).  Returns (more_levels, kept); after the
        last level `factor` [F*S] holds the product of the factors along every surviving path."""
        om = np.asarray(om, dtype=np.float64)
        f = self.fac * om
        keep = np.nonzero((om > 0.0) & (f > 0.0))[0]
        kept = len(keep)
        if self.lvl == self.L:
            factor[torch.from_numpy(self.act[keep].astype(np.int64))] = torch.from_numpy(f[keep])
            return False, kept
        stride = self.S << self.lvl
        self.node = np.ascontiguousarray(self.act[keep], dtype=np.int32)
        self.ppos = keep.astype(np.int32)
        self.fpar = np.ascontiguousarray(f[keep])
        self.act = np.concatenate([self.node, self.node + np.int32(stride)])
        self.fac = np.concatenate([self.fpar, self.fpar])
        self.lvl += 1
        return True, kept


def recombine_sharded(engine, n, S, group=None, device=None, max_rounds=256):
    """Run the pass loop on `engine` (count/cell_factor/pass_begin/level/car/apply/result).
    Returns this rank's surviving (idx, w); concatenate over ranks (gather_result) for the full rule.

    A pass over F*S cells (cell = global position mod F*S, set j = cells j, j+S, ...) costs ONE
    sweep of kernel evaluations; each of its log2(F)+1 Caratheodory levels all-reduces one small
    [n, S] system, and the candidates shrink by 2F."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    device = device if device is not None else getattr(engine, "device", "cpu")
    counts = torch.zeros(world, dtype=torch.int64, device=device)
    counts[rank] = engine.count()
    if world > 1:
        dist.all_reduce(counts, group=group)
    counts = counts.cpu().tolist()
    # With NCCL the ranks also share the projection (level_fold -> reduce-scatter -> level_project):
    # BASQ_SHARE_PROJECTION=0 keeps every rank projecting its own cell sums.
    share_projection = (world > 1 and hasattr(engine, "level_fold") and dist.get_backend(group) == "nccl"
                        and os.environ.get("BASQ_SHARE_PROJECTION", "1") != "0")
    A = torch.zeros(getattr(engine, "rows", n), S, dtype=torch.float64, device=device)   # n + 1 rows with an objective
    omega = torch.zeros(S, dtype=torch.float64, device=device)
    rounds = 0
    while sum(counts) > n:
        rounds += 1
        if rounds > max_rounds:
            raise RuntimeError("recombine_sharded: no convergence")
        R = sum(counts)
        off = sum(counts[:rank])
        F = engine.cell_factor(R, max(counts))          # same inputs on every rank -> same F
        cells = F * S
        engine.pass_begin(R, off, F)
        factor = torch.zeros(cells, dtype=torch.float64)
        tree = LevelTree(S, F, R)
        while True:
            C = tree.columns()
            if C > n or tree.lvl < tree.L:
                if share_projection:
                    # fold locally, reduce-scatter the folded columns by landmark rows, project 1/world
                    # of the rows here; the all-reduce of A below completes the sum over row blocks
                    K = len(tree.node)
                    Mtot, rows_blk, Gf, blk = engine.shared_buffers(world)
                    Gv, bv = Gf[: rows_blk * world * K].view(rows_blk * world, K), blk[: rows_blk * K].view(rows_blk, K)
                    engine.level_fold(tree.lvl, tree.node, Gv)
                    dist.reduce_scatter_tensor(bv, Gv, group=group)
                    row0 = min(rank * rows_blk, Mtot)
                    engine.level_project(tree.lvl, tree.node, tree.ppos, tree.fpar, bv, row0,
                                         min(rows_blk, Mtot - row0), A)
                else:
                    engine.level(tree.lvl, tree.node, tree.ppos, tree.fpar, A)
            if C > n:
                if world > 1:
                    dist.all_reduce(A, group=group)
                engine.car(A, C, omega)                   # identical system -> identical factors on every rank
                om = omega[:C].cpu().numpy()
            else:
                om = np.ones(C)
            more, kept = tree.advance(om, factor)
            if kept < 1:
                raise RuntimeError("recombine_sharded: the Caratheodory step kept no set")
            if not more:
                break
        new_local = engine.apply(R, off, F, factor)
        # every rank derives every rank's new count from the kept cells: no extra collective
        c_eff = min(cells, R)
        keep = (factor[:c_eff] > 0).to(torch.int64)
        prefix = torch.zeros(cells + 1, dtype=torch.int64)
        prefix[1:c_eff + 1] = torch.cumsum(keep, 0)
        prefix[c_eff + 1:] = prefix[c_eff]
        K = int(prefix[cells])
        new_counts, o = [], 0
        for c in counts:
            new_counts.append(kept_before(o + c, cells, prefix, K) - kept_before(o, cells, prefix, K))
            o += c
        if new_counts[rank] != new_local:
            raise RuntimeError(f"rank {rank}: survivor count mismatch {new_counts[rank]} != {new_local}")
        if sum(new_counts) >= R:
            raise RuntimeError("recombine_sharded: pass made no progress")
        counts = new_counts
    return engine.result()


def gather_result(idx, w, n, group=None):
    """All-gather the per-rank survivors into one ascending (idx, w) on every rank."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return idx, w
    world = dist.get_world_size(group)
    dev = idx.device
    pad_i = torch.full((n,), -1, dtype=torch.int64, device=dev)
    pad_w = torch.zeros(n, dtype=torch.float64, device=dev)
    pad_i[: len(idx)] = idx
    pad_w[: len(w)] = w
    all_i = [torch.empty_like(pad_i) for _ in range(world)]
    all_w = [torch.empty_like(pad_w) for _ in range(world)]
    dist.all_gather(all_i, pad_i, group=group)
    dist.all_gather(all_w, pad_w, group=group)
    I, W = torch.cat(all_i), torch.cat(all_w)
    m = I >= 0
    I, W = I[m], W[m]
    order = torch.argsort(I)
    return I[order], W[order]


def recombination_sharded(pts_rec_local, pts_nys, num_pts, kernel, N_glob, idx_base, U, init_weights_local=None,
                          group=None, obj_local=None, staged=None):
    """Sharded counterpart of recombination(): this rank holds pts_rec_local = rows
    [idx_base, idx_base + len) of the global candidate set; pts_nys, U and the GP caches are
    replicated.  Returns the full (idx, w) on every rank.  staged = ops.stage_candidates(X_host_local, ...):
    the shard comes from host memory through the C ABI (pts_rec_local / init_weights_local are ignored)."""
    from . import ops

    sess = ops.Session(kernel, pts_rec_local, pts_nys, U, N_glob, idx_base, mu_loc=init_weights_local,
                       obj_loc=obj_local, staged=staged, device=pts_nys.device if staged is not None else None)
    try:
        idx, w = recombine_sharded(sess, sess.n, sess.S, group=group, device=sess.device)
        return gather_result(idx, w, sess.n, group=group)
    finally:
        sess.close()


_XCHG_BUFFERS = {}


def nystrom_basis_sharded(kernel, Z, q, omega=None, niter=2, group=None, seed=None, device=None):
    """U [q, M], the Nystrom basis of ops.nystrom_basis, with the rows of K(Z, Z) sharded over the ranks
    (basq_nystrom_basis_sharded): every rank evaluates and multiplies M / world rows; per product the ranks
    all-reduce a q x q Gram matrix and all-gather the orthonormalised rows.  Z (and omega, or the seed) must
    be the same on every rank; every rank returns the same U.  The collectives are torch.distributed's on the
    current stream (NCCL); with a gloo group they are staged through the host (tests).  Without a process
    group the call degenerates to one shard."""
    import ctypes as C

    from . import _lib, ops

    spec, ctx, device, dtype = ops._common(kernel, Z, device)
    Zd = ops._prep(Z, device, dtype)
    M = len(Zd)
    on = dist.is_initialized() and dist.get_world_size(group) > 1
    world = dist.get_world_size(group) if on else 1
    rank = dist.get_rank(group) if on else 0
    chunk = -(-M // world)
    # exchange buffers live across calls: allocating 130 MB of them per call made torch's caching allocator
    # re-carve its blocks every few steps (sporadic 40-130 ms stalls in the 2-GPU bench)
    key = (device.index, world, chunk, q)
    bufs = _XCHG_BUFFERS.get(key)
    if bufs is None:
        _XCHG_BUFFERS.clear()       # one shape at a time is enough; do not hoard memory for old ones
        bufs = _XCHG_BUFFERS[key] = (torch.empty(q * q, dtype=torch.float64, device=device),
                                     torch.zeros(world * chunk * q, dtype=torch.float64, device=device),
                                     torch.empty(chunk * q, dtype=torch.float64, device=device))
    gram_buf, rows_buf, mine = bufs
    staged = on and dist.get_backend(group) != "nccl"
    failure = []

    def exchange(_user, op, count):
        try:
            if not on:
                return 0
            if op == 0:
                if staged:
                    h = gram_buf.cpu()
                    dist.all_reduce(h, group=group)
                    gram_buf.copy_(h)
                else:
                    dist.all_reduce(gram_buf, group=group)
            else:
                mine.copy_(rows_buf[rank * count:(rank + 1) * count])
                if staged:
                    parts = [torch.empty(count, dtype=torch.float64) for _ in range(world)]
                    dist.all_gather(parts, mine.cpu(), group=group)
                    rows_buf.copy_(torch.cat(parts))
                else:
                    dist.all_gather_into_tensor(rows_buf, mine, group=group)
            return 0
        except Exception as e:      # never let an exception cross the C frame
            failure.append(e)
            return 1

    cb = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int64)(exchange)
    if omega is not None:
        omega = ops._prep(omega, device, torch.float64)
    else:
        ops._seed_context(ctx, seed if seed is not None else _shared_seed(group, on, device))
    desc, keep = spec.to_desc(Zd.shape[1], device, dtype)
    U = torch.empty(q, M, dtype=torch.float64, device=device)
    rc = _lib.lib.basq_nystrom_basis_sharded(ctx.handle, C.byref(desc), Zd.data_ptr(), M, int(q),
                                             omega.data_ptr() if omega is not None else None, int(niter), rank, world,
                                             gram_buf.data_ptr(), rows_buf.data_ptr(), C.cast(cb, C.c_void_p), None, U.data_ptr())
    if failure:
        raise failure[0]
    _lib.check(rc)
    return U


def _shared_seed(group, on, device):
    """One draw of rank 0's torch generator, shared with the other ranks: the test matrix must be the same
    everywhere (torch.manual_seed on rank 0 reproduces the run)."""
    s = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64)
    if on:
        s = s.to(device) if dist.get_backend(group) == "nccl" else s
        dist.broadcast(s, dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return int(s.item())


def quadform_pair_assignment(world):
    """Cross terms of a sharded quadratic form, assigned to ranks: tasks[r] lists (i, j, half) for rank r,
    meaning 2 B(X_i, a_i; X_j, a_j) restricted to the rows of shard i given by `half` (None: all rows, 0: the
    first len_i // 2 rows, 1: the rest).  Every unordered pair i < j of shards is covered exactly once: rank r
    takes the pairs (r, r + k mod G) for k = 1 .. (G - 1) // 2, and for even G the antipodal pair
    (r, r + G / 2) is split by rows between its two ranks (B is linear in a).  Every rank gets (G - 1) / 2
    pair-equivalents."""
    tasks = [[] for _ in range(world)]
    for r in range(world):
        for k in range(1, (world - 1) // 2 + 1):
            s = (r + k) % world
            tasks[r].append((min(r, s), max(r, s), None))
        if world % 2 == 0 and world > 1:
            h = world // 2
            tasks[r].append((r, r + h, 0) if r < h else (r - h, r, 1))
    return tasks


def _all_gather_var(t, group, nccl):
    """All-gather tensors whose first dimension differs between ranks (padded to the largest)."""
    world = dist.get_world_size(group)
    dev = t.device
    n = torch.tensor([len(t)], dtype=torch.int64, device=dev if nccl else "cpu")
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n, group=group)
    sizes = [int(s) for s in sizes]
    pad = torch.zeros((max(sizes),) + tuple(t.shape[1:]), dtype=t.dtype, device=dev if nccl else "cpu")
    pad[: len(t)] = t
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    return [p[:s].to(dev) for p, s in zip(parts, sizes)]


def kernel_quadform_sharded(kernel, X_local, a_local, group=None) -> float:
    """a^T kernel(X, X) a (ops.kernel_quadform) for X, a sharded by rows over the ranks, one process per GPU:
    the shards are all-gathered, rank r adds its own Q(X_r, a_r) and the cross terms 2 B(X_i, a_i; X_j, a_j)
    that quadform_pair_assignment gives it, and one all-reduce of a scalar sums the ranks.  Every rank
    returns the total.  With a gloo group the collectives are staged through the host."""
    from . import ops

    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return ops.kernel_quadform(kernel, X_local, a_local)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    nccl = dist.get_backend(group) == "nccl"
    a_local = a_local.to(device=X_local.device, dtype=torch.float64)
    Xs = _all_gather_var(X_local.contiguous(), group, nccl)
    As = _all_gather_var(a_local.contiguous(), group, nccl)
    total = ops.kernel_quadform(kernel, X_local, a_local) if len(X_local) else 0.0
    for i, j, half in quadform_pair_assignment(world)[rank]:
        lo, hi = 0, len(Xs[i])
        if half is not None:
            lo, hi = (0, hi // 2) if half == 0 else (hi // 2, hi)
        if hi > lo and len(Xs[j]):
            total += 2.0 * ops.kernel_bilinear(kernel, Xs[i][lo:hi], As[i][lo:hi], Xs[j], As[j])
    s = torch.tensor([total], dtype=torch.float64, device=X_local.device if nccl else "cpu")
    dist.all_reduce(s, group=group)
    return float(s.item())
