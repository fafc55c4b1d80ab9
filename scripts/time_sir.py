"""Time SIR resampling over N = 1e7 candidates: the single-GPU call (basq_sir_resample: host-bracketed cut, host
sort) against the device radix select of sharded.sir_indices_sharded on one shard, per n in {1e3, 1e5, 1e6, 1e7},
and the steps of the new path.  With two or more GPUs the sharded call is also timed on 2 NCCL ranks.

    python scripts/time_sir.py [--reps 5] [--out DIR]

Device events around each call (every call ends in a host synchronise: both paths return host-known results);
median of --reps after one warm-up.  20 % of the weights are zero.  The draws of the two paths are compared."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

N = 10_000_000
NS = (1_000, 100_000, 1_000_000, 10_000_000)


def _weights(device):
    g = torch.Generator(device=device).manual_seed(1)
    w = torch.rand(N, generator=g, dtype=torch.float64, device=device)
    w[torch.rand(N, generator=g, device=device) < 0.2] = 0.0
    return w


def _time(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return statistics.median(out)


def _steps(w, n, reps):
    """Median ms of the new path's steps on one shard (keys, the 6 histogram passes, collect, sort)."""
    from basq_b200 import sharded
    from basq_b200.sampler import ShardEngine

    eng = ShardEngine(w.device)
    keys = eng.sir_keys(w, 3, 0)
    t = {"keys": _time(lambda: eng.sir_keys(w, 3, 0), reps)}
    sel = {}

    def select():
        mask = bits = below = mine = 0
        m = None
        for shift in sharded.SIR_SHIFTS:
            h = eng.sir_histogram(keys, mask, bits, shift)
            if m is None:
                h[-1] = 0
                m = min(n, int(h.sum()))
            cum = h.cumsum()
            d = int(cum.searchsorted(m - below))
            below += int(cum[d - 1]) if d else 0
            mine += int(h[:d].sum())
            mask |= (2047 << shift) & (2 ** 64 - 1)
            bits |= d << shift
        sel.update(T=bits, count=mine + int(h[d]), m=m)

    t["histograms"] = _time(select, reps)
    t["collect"] = _time(lambda: eng.sir_collect(keys, sel["T"], 0, sel["count"]), reps)
    ks, ids = eng.sir_collect(keys, sel["T"], 0, sel["count"])
    t["sort"] = _time(lambda: eng.sir_sort(ks.clone(), ids.clone()), reps)
    t["sort_copy_only"] = _time(lambda: (ks.clone(), ids.clone()), reps)
    t["pairs_sorted"] = sel["count"]
    return t


def _nccl_worker(rank, world, rdzv, reps, out):
    import torch.distributed as dist

    from basq_b200 import sharded
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        dev = torch.device("cuda", rank)
        w = _weights(dev)
        lo, hi = sharded.shard_bounds(N, world, rank)
        res = {}
        for n in NS:
            def call():
                dist.barrier()
                sharded.sir_indices_sharded(w[lo:hi], n, seed=3, idx_base=lo)
            res[str(n)] = _time(call, reps)
        if rank == 0:
            with open(out, "w") as f:
                json.dump(res, f)
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_sir.py needs a CUDA device")
    from basq_b200 import sampler, sharded
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rep = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "N": N, "zero_fraction": 0.2, "reps": a.reps,
           "single_gpu": {}}
    w = _weights(dev)
    for n in NS:
        old = _time(lambda: sampler.sir_indices(w, n, seed=3), a.reps)
        new = _time(lambda: sharded.sir_indices_sharded(w, n, seed=3), a.reps)
        same = torch.equal(sampler.sir_indices(w, n, seed=3), sharded.sir_indices_sharded(w, n, seed=3))
        rep["single_gpu"][str(n)] = {"old_ms": old, "new_ms": new, "identical": same, "new_steps_ms": _steps(w, n, a.reps)}
        print(f"n={n:>9}: basq_sir_resample {old:9.2f} ms   device select {new:8.2f} ms   identical={same}", flush=True)
    del w
    torch.cuda.empty_cache()
    if torch.cuda.device_count() >= 2:
        import torch.multiprocessing as mp
        with tempfile.TemporaryDirectory() as tmp:
            out = os.path.join(tmp, "t.json")
            mp.spawn(_nccl_worker, args=(2, os.path.join(tmp, "rdzv"), a.reps, out), nprocs=2, join=True)
            rep["two_gpu_nccl_ms"] = json.load(open(out))
    else:
        rep["two_gpu_nccl_ms"] = "not measured: one GPU"
    print(json.dumps(rep, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_sir.json"), "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
