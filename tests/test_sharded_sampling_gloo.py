"""Host protocol of the sharded candidate side (basq_b200.sharded: calc_weights_sharded, cleansing_weights_sharded,
sir_indices_sharded, SIR_sharded) on CPU with gloo.  The device engine (sampler.ShardEngine) is replaced by numpy
restatements of its steps over the oracle's race keys, so this checks the radix select, the per-rank counts, the
rank-ordered gather and the folded totals: the draws must be the oracle's race on the concatenated weights."""
import math
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from basq_b200 import sharded
from oracle import gp_kernels as ogp
from oracle import sampler as osam

NO_KEY = np.uint64(2 ** 64 - 1)


def race_keys(w, seed, idx_base):
    """The keys of oracle.sampler.sir_indices for rows idx_base.. of a larger set: -log(u) / w with u from
    Philox(seed; counter (global row, 0, 0x53495200)), inf where w is not > 0."""
    rows = np.arange(len(w), dtype=np.uint64) + np.uint64(idx_base)
    ctr = np.zeros((len(w), 4), dtype=np.uint32)
    ctr[:, 0] = (rows & osam.MASK).astype(np.uint32)
    ctr[:, 1] = (rows >> np.uint64(32)).astype(np.uint32)
    ctr[:, 3] = 0x53495200
    key = np.empty((len(w), 2), dtype=np.uint32)
    key[:, 0] = np.uint32(seed & 0xFFFFFFFF)
    key[:, 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    r = osam.philox4x32_10(ctr, key)
    u = ((r[:, 0] >> np.uint32(5)).astype(np.float64) * 2.0 ** 26
         + (r[:, 1] >> np.uint32(6)).astype(np.float64) + 0.5) * 2.0 ** -53
    with np.errstate(divide="ignore"):
        return np.where(w > 0, -np.log(u) / np.where(w > 0, w, 1.0), np.inf)


def test_race_keys_order_like_the_oracle_race():
    """race_keys at idx_base = 0 ranks rows as oracle.sampler.sir_indices does; a shard's keys are a slice."""
    w = _weights(5000).numpy()
    k = race_keys(w, 9, 0)
    n = int((w > 0).sum())
    assert np.array_equal(np.lexsort((np.arange(len(w)), k))[:n], osam.sir_indices(w, n, seed=9))
    assert np.array_equal(race_keys(w[1234:], 9, 1234), k[1234:])


class OracleShardEngine:
    """The steps of sampler.ShardEngine on CPU tensors (tests only).  `kernel` of candidate_weights is a callable
    X -> (GP mean, GP variance)."""

    device = torch.device("cpu")

    def candidate_weights(self, kernel, X, ratio):
        mean, var = (np.asarray(a, dtype=np.float64) for a in kernel(X))
        am = np.abs(mean)
        g = ratio * var + (1.0 - ratio) * am if ratio < 1.0 else ratio * var
        with np.errstate(divide="ignore", invalid="ignore"):
            w = am / g
        w[~(g > 0) & (am == 0)] = 0.0
        return torch.from_numpy(w)

    def weights_sum(self, w):
        return float(np.sum(w.numpy()))

    def weights_normalise(self, w, total, N_glob):
        if total != 0.0 and math.isfinite(total):
            w /= total
        else:
            w.fill_(1.0 / N_glob)

    def weights_cleanse(self, w, eps):
        v = w.numpy()
        v[v < eps] = 0.0
        v[~np.isfinite(v)] = eps

    def sir_keys(self, w, seed, idx_base):
        k = race_keys(w.numpy(), seed, idx_base)
        bits = k.view(np.uint64).copy()
        bits[~np.isfinite(k)] = NO_KEY
        return torch.from_numpy(bits.view(np.int64))

    def sir_histogram(self, keys, mask, bits, shift):
        k = keys.numpy().view(np.uint64)
        k = k[(k & np.uint64(mask)) == np.uint64(bits)]
        return np.bincount(((k >> np.uint64(shift)) & np.uint64(2047)).astype(np.int64), minlength=2048)

    def sir_collect(self, keys, T, idx_base, cap):
        k = keys.numpy().view(np.uint64)
        i = np.nonzero(k <= np.uint64(T))[0]
        assert len(i) <= cap
        return torch.from_numpy(k[i].view(np.int64).copy()), torch.from_numpy(i.astype(np.int64) + idx_base)

    def sir_sort(self, keys, idx):
        return idx[torch.from_numpy(np.argsort(keys.numpy().view(np.uint64), kind="stable"))]


def _weights(N, seed=3):
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(N, generator=g, dtype=torch.float64) ** 3
    w[torch.rand(N, generator=g) < 0.2] = 0.0
    return w


def _gp_case(N):
    model = ogp.make_gp(3, 30, lengthscale=1.5, outputscale=1.1, noise=1e-4, seed=2)
    X = math.sqrt(2.0) * torch.randn(N, 3, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    return X, (lambda Xs: tuple(t.numpy() for t in ogp.predict(Xs, model)))


def _check_all(bounds, group_on):
    """Runs every sharded function on this rank's shard [bounds[rank], bounds[rank + 1]) and checks it."""
    rank = dist.get_rank() if group_on else 0
    lo, hi = bounds[rank], bounds[rank + 1]
    N = bounds[-1]
    eng = OracleShardEngine()
    w = _weights(N)
    n_pos = int((w > 0).sum())
    for n in (1, 1000, n_pos + 17):
        for seed in (0, 0xFEEDFACE12345):
            idx = sharded.sir_indices_sharded(w[lo:hi], n, seed=seed, idx_base=lo, engine=eng)
            ref = osam.sir_indices(w.numpy(), n, seed=seed)
            assert np.array_equal(idx.numpy(), ref), (n, seed)
    # SIR_sharded: this rank keeps its drawn rows, numbered rank-major
    X = torch.arange(N, dtype=torch.float64).unsqueeze(1)
    Xd, N_new, base, src = sharded.SIR_sharded(X[lo:hi], w[lo:hi], 500, seed=4, idx_base=lo, engine=eng)
    ref = osam.sir_indices(w.numpy(), 500, seed=4)
    assert N_new == 500 and base == int((ref < lo).sum())
    assert np.array_equal(src.numpy(), ref[(ref >= lo) & (ref < hi)])
    assert torch.equal(Xd[:, 0], src.double())
    # cleansing: replacements per weight, one global normalisation
    raw = w * 1e-3
    raw[::7] = float("inf")
    raw[1::11] = float("nan")
    out = sharded.cleansing_weights_sharded(raw[lo:hi], N, engine=eng)
    np.testing.assert_allclose(out.numpy(), osam.cleansing_weights(raw.numpy())[lo:hi], rtol=1e-14, atol=0)
    zero = sharded.cleansing_weights_sharded(torch.zeros(hi - lo, dtype=torch.float64), N, engine=eng)
    assert bool((zero == 1.0 / N).all())
    # calc_weights
    Xg, kern = _gp_case(N)
    mean, var = kern(Xg)
    for ratio in (0.5, 1.0):
        cw = sharded.calc_weights_sharded(kern, Xg[lo:hi], ratio, N, engine=eng)
        np.testing.assert_allclose(cw.numpy(), osam.calc_weights(mean, var, np.zeros(N), ratio)[lo:hi],
                                   rtol=1e-14, atol=0)
    zero_gp = lambda Xs: (np.zeros(len(Xs)), np.ones(len(Xs)))
    cz = sharded.calc_weights_sharded(zero_gp, Xg[lo:hi], 0.5, N, engine=eng)
    assert bool((cz == 1.0 / N).all())


def _worker(rank, world, bounds, rdzv):
    dist.init_process_group("gloo", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        _check_all(bounds, True)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("bounds", [[0, 1000, 3001], [0, 1700, 1700, 3001], [0, 0, 2500, 3001]],
                         ids=["world2", "world3-empty-middle", "world3-empty-first"])
def test_sharded_sampling_equals_the_race_on_the_concatenation(tmp_path, bounds):
    world = len(bounds) - 1
    mp.spawn(_worker, args=(world, bounds, str(tmp_path / "rdzv")), nprocs=world, join=True)


def test_one_shard_without_a_process_group():
    _check_all([0, 3001], False)
