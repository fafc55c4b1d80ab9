"""Cost of the reproducible mode (ops.reproducible): basq_recombine in the default and the reproducible mode,
alternating in one process, on BASELINE config 3 (VBQ predictive covariance, N = 1e7, d = 10, M = 1e4, n = 1000)
and the config-5 non-linear modes (WSABI-M, MMLT).  Prints one JSON line per config with the card name and power
limit.  Single GPU; the sharded loop adds one all-reduce of [Mtot + 2, K] columns per level (not timed here).

    python scripts/time_reproducible.py [--N 10000000] [--reps 3]
"""
import argparse
import json
import math
import subprocess
import sys
import os

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from basq_b200 import _lib, ops  # noqa: E402
from oracle import gp_kernels as ogp  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    d, M, n, n_obs = 10, 10_000, 1000, 1002
    g = torch.Generator(device=dev).manual_seed(1)
    X = math.sqrt(2.0) * torch.randn(args.N, d, generator=g, device=dev, dtype=torch.float32)
    Z = X[:M].clone()
    ctx = _lib.context_for(dev)
    for name in ("config3_vbq", "config5_wsabim", "config5_mmlt"):
        model = ogp.make_gp(d, n_obs, lengthscale=2.5, outputscale=1.0, noise=1e-4 if name != "config3_vbq" else 1e-10,
                            seed=3, log_targets=(name == "config5_mmlt"), mean_const=0.1 if "wsabi" in name else 0.0)
        kern = {"config3_vbq": ogp.VanillaGP(model).predictive_kernel,
                "config5_wsabim": ogp.WsabiGP(model, alpha=0.05).wsabim_kernel,
                "config5_mmlt": ogp.ScaleMmltGP(model).gspace_kernel}[name]
        _, U = ops.nystrom_basis(kern, Z, n - 1, want_S=False, seed=7)
        times = {False: [], True: []}
        rules = {}
        for rep in range(args.reps + 1):            # the first round warms up both modes
            for on in (False, True):
                ctx.reproducible(on)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                rules[on] = ops.recombine(kern, X, Z, U)
                e1.record()
                torch.cuda.synchronize()
                if rep:
                    times[on].append(e0.elapsed_time(e1))
        ctx.reproducible(False)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        print(json.dumps({"config": name, "N": args.N, "gpu": card(), "default_ms": med[False],
                          "reproducible_ms": med[True], "ratio": med[True] / med[False],
                          "all_ms": {"default": times[False], "reproducible": times[True]},
                          "points_default": len(rules[False][0]), "points_reproducible": len(rules[True][0]),
                          "w_sum": float(rules[True][1].sum())}), flush=True)


if __name__ == "__main__":
    main()
