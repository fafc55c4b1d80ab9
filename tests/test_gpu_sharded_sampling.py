"""The candidate side over a sharded set on the device (basq_weights_*, basq_sir_* through basq_b200.sharded): one
shard must reproduce the single-GPU calls (basq_sir_resample, basq_candidate_weights, basq_cleanse_weights), and
2-4 ranks (processes sharing one GPU, gloo) must draw exactly what one GPU draws."""
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
from oracle import sampler as osam

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _sir_cases():
    """The weight vectors of test_gpu_candidates.py::test_sir_matches_oracle_race_and_weights."""
    g = torch.Generator().manual_seed(3)
    w = torch.rand(200_000, generator=g, dtype=torch.float64) ** 3
    w[::5] = 0.0
    w2 = torch.zeros(5000, dtype=torch.float64)
    w2[torch.arange(0, 5000, 50)] = 1.0
    w3 = torch.ones(4000, dtype=torch.float64)
    w3[:2000] = 3.0
    return [(w, 1000, 99), (w2, 500, 1), (w3, 40, 0), (w3, 40, 7), (w, 1, 5), (w, 200_000, 2)]


def test_one_shard_equals_sir_resample_and_oracle():
    from basq_b200 import sampler, sharded
    for w, n, seed in _sir_cases():
        got = sharded.sir_indices_sharded(w.to(DEV), n, seed=seed)
        assert got.device == DEV
        assert torch.equal(got.cpu(), sampler.sir_indices(w.to(DEV), n, seed=seed).cpu())
        assert np.array_equal(got.cpu().numpy(), osam.sir_indices(w.numpy(), n, seed=seed))
    # no positive weight: no draw
    assert len(sharded.sir_indices_sharded(torch.zeros(10, dtype=torch.float64, device=DEV), 3)) == 0


def test_one_shard_equals_sir_resample_large():
    from basq_b200 import sampler, sharded
    g = torch.Generator(device=DEV).manual_seed(11)
    w = torch.rand(10_000_000, generator=g, dtype=torch.float64, device=DEV)
    w[torch.rand(10_000_000, generator=g, device=DEV) < 0.2] = 0.0
    got = sharded.sir_indices_sharded(w, 1_000_000, seed=123)
    ref = sampler.sir_indices(w, 1_000_000, seed=123)
    assert len(got) == 1_000_000 and torch.equal(got, ref)


def test_sort_is_stable_on_equal_keys():
    """basq_sir_sort keeps the input order among equal keys (the race's ties go to the lower index)."""
    from basq_b200.sampler import ShardEngine
    eng = ShardEngine(DEV)
    g = torch.Generator().manual_seed(2)
    keys = torch.randint(0, 40, (300_000,), generator=g, dtype=torch.int64) << 50
    keys[::3] += torch.randint(0, 2 ** 40, (100_000,), generator=g, dtype=torch.int64)
    idx = torch.arange(len(keys), dtype=torch.int64)
    got = eng.sir_sort(keys.to(DEV), idx.to(DEV)).cpu()
    ref = torch.from_numpy(np.argsort(keys.numpy(), kind="stable"))
    assert torch.equal(got, ref)


def _bounds(N, world):
    """Uneven shards, the second one empty when world > 2."""
    cuts = sorted({0, N} | {int(N * f) for f in (0.15, 0.15, 0.6)[: world - 1]})
    while len(cuts) < world + 1:
        cuts.insert(1, cuts[1])
    return cuts


def _weights(N):
    g = torch.Generator().manual_seed(17)
    w = torch.rand(N, generator=g, dtype=torch.float64) ** 2
    w[torch.rand(N, generator=g) < 0.2] = 0.0
    return w


def _gp(d=3):
    model = ogp.make_gp(d, 40, lengthscale=1.6, outputscale=1.2, noise=1e-4, seed=8)
    return ogp.VanillaGP(model).predictive_kernel


def _worker(rank, world, rdzv, bounds, out_path):
    from basq_b200 import ops, sharded
    dist.init_process_group("gloo", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        lo, hi = bounds[rank], bounds[rank + 1]
        N = bounds[-1]
        w = _weights(N).to(DEV)
        n_pos = int((w > 0).sum())
        draws = [sharded.sir_indices_sharded(w[lo:hi], n, seed=77, idx_base=lo).cpu() for n in (1, 1000, n_pos + 5)]
        # every rank holds the same draws
        for d in draws:
            ref = d.clone()
            dist.broadcast(ref, 0)
            assert torch.equal(d, ref)
        kern = _gp()
        X = math.sqrt(2.0) * torch.randn(N, 3, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
        cw = sharded.calc_weights_sharded(kern, X[lo:hi].to(DEV), 0.5, N).cpu()
        raw = _weights(N) * 1e-3
        raw[::7] = float("inf")
        cl = sharded.cleansing_weights_sharded(raw[lo:hi].to(DEV), N).cpu()
        # SIR_sharded straight into the sharded recombination (the session and round loop of recombination_sharded;
        # the gather goes through the host because gloo gathers no CUDA tensors)
        Xd, N_new, base, src = sharded.SIR_sharded(X[lo:hi].to(DEV), cw.to(DEV), 3000, seed=5, idx_base=lo)
        Z = X[:200].to(DEV)
        q = 19
        _, U = ops.nystrom_basis(kern, Z, q, want_S=False, seed=6)
        sess = ops.Session(kern, Xd, Z, U, N_new, base)
        try:
            idx, wq = sharded.recombine_sharded(sess, sess.n, sess.S, device=sess.device)
            idx, wq = sharded.gather_result(idx.cpu(), wq.cpu(), sess.n)
        finally:
            sess.close()
        srcs = [s.cpu() for s in sharded._all_gather_var(src.cpu(), None, False)]
        if rank == 0:
            torch.save({"draws": draws, "cw": cw, "cl": cl, "idx": idx, "wq": wq, "src": torch.cat(srcs),
                        "N_new": N_new, "U": U.cpu()}, out_path)
        else:
            torch.save({"cw": cw, "cl": cl}, f"{out_path}.{rank}")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_spawned_ranks_draw_what_one_gpu_draws(world):
    from basq_b200 import ops, sampler
    N = 120_001
    bounds = _bounds(N, world)
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "r.pt")
        mp.spawn(_worker, args=(world, os.path.join(tmp, "rdzv"), bounds, out), nprocs=world, join=True)
        r = torch.load(out)
        parts = [r] + [torch.load(f"{out}.{k}") for k in range(1, world)]
    w = _weights(N).to(DEV)
    n_pos = int((w > 0).sum())
    for d, n in zip(r["draws"], (1, 1000, n_pos + 5)):
        assert torch.equal(d, sampler.sir_indices(w, n, seed=77).cpu())
    kern = _gp()
    X = math.sqrt(2.0) * torch.randn(N, 3, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    cw = torch.cat([p["cw"] for p in parts])
    ref = sampler.calc_weights(kern, X.to(DEV), ratio=0.5).cpu()
    torch.testing.assert_close(cw, ref, rtol=1e-14, atol=0)
    assert abs(float(cw.sum()) - 1.0) < 1e-12
    raw = _weights(N) * 1e-3
    raw[::7] = float("inf")
    cl = torch.cat([p["cl"] for p in parts])
    torch.testing.assert_close(cl, sampler.cleansing_weights(raw.to(DEV)).cpu(), rtol=1e-14, atol=0)
    assert abs(float(cl.sum()) - 1.0) < 1e-12
    # the end-to-end rule: the drawn set in rank-major order, recombined with the invariants of the recombination tests
    src, idx, wq = r["src"], r["idx"], r["wq"]
    assert r["N_new"] == 3000 and len(src) == 3000
    assert torch.equal(src.sort().values, sampler.sir_indices(cw.to(DEV), 3000, seed=5).cpu().sort().values)
    assert 1 <= len(idx) <= 20 and bool((wq > 0).all()) and abs(float(wq.sum()) - 1.0) < 1e-12
    Xn = X[src]
    Phi = ops.features(kern, Xn.to(DEV), X[:200].to(DEV), r["U"].to(DEV)).cpu()
    mu = torch.full((3000,), 1.0 / 3000, dtype=torch.float64)
    assert orchq.moment_residual(Phi, mu, idx, wq) <= 1e-8


def test_full_quadrature_one_shard_equals_gp():
    from basq_b200 import gp, sharded
    kern = _gp()
    X = math.sqrt(2.0) * torch.randn(5000, 3, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    w = torch.rand(5000, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    e0, v0 = gp.full_quadrature(X.to(DEV), w, kern)
    e1, v1 = sharded.full_quadrature_sharded(X.to(DEV), w.to(DEV), kern)
    assert e1 == e0 and v1 == v0
