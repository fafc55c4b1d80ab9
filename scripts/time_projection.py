"""The projection GEMM of the level columns, raw[1..q, :K] = U'[q, Mtot] Gf[Mtot, K], on the fp64 DMMA path
(ops.dgemm) against the int8 Ozaki GEMM (ops.igemm, igemm.cu), at the shapes of the bench's sessions.

    python scripts/time_projection.py [--reps 20] [--out DIR]

CUDA events time whole calls after warm-up; a torch.profiler run of its own splits the int8 call into its
kernels (the GEMM, and the slicing of each operand - a session slices U' once and the level columns per level).
Operands total 100-400 MB per shape, so they do not stay in the 126 MB L2 across the fp64 calls; the digit
operands of the int8 GEMM do partly.  Prints the card's name, power limit and SM clocks first."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from basq_b200 import ops

INT8_PEAK = 4.5e15     # dense int8 ops/s of one B200 (NVIDIA data sheet, 1000 W card)
PAIRS = 36             # digit products of igemm.cu


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "nvidia-smi unavailable"


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_ms(fn, reps):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for name in ("igemm_kernel", "ig_split_kernel<true>", "ig_split_kernel<false>", "ig_rowmax"):
            if name in ev.key:
                out[name] = out.get(name, 0.0) + ev.device_time_total / 1e3 / reps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    print(card(), flush=True)
    shapes = [(999, 2000, 11002), (999, 1000, 11002), (999, 2000, 10000), (499, 1000, 5000), (255, 500, 10000)]
    rows = []
    for q, K, mtot in shapes:
        g = torch.Generator(device=dev).manual_seed(q + K)
        U = torch.randn(q, mtot, generator=g, device=dev, dtype=torch.float64)
        G = torch.rand(mtot, K, generator=g, device=dev, dtype=torch.float64)
        C = torch.empty(q, K, device=dev, dtype=torch.float64)
        t_d = timed(lambda: ops.dgemm(U, G), a.reps)
        t_i = timed(lambda: ops.igemm(U, G, out=C), a.reps)
        ks = kernel_ms(lambda: ops.igemm(U, G, out=C), a.reps)
        t_k = ks.get("igemm_kernel", float("nan"))
        flop = 2.0 * q * K * mtot
        r = {"shape": [q, K, mtot], "dgemm_ms": t_d, "igemm_call_ms": t_i, "igemm_kernels_ms": ks,
             "dgemm_tflops": flop / t_d / 1e9, "igemm_equiv_fp64_tflops": flop / t_k / 1e9,
             "int8_ops_per_s": PAIRS * flop / (t_k * 1e-3), "int8_peak_share": PAIRS * flop / (t_k * 1e-3) / INT8_PEAK,
             "speedup_kernel": t_d / t_k, "speedup_call": t_d / t_i}
        rows.append(r)
        print(f"{q} x {K} x {mtot}: dgemm {t_d:.3f} ms ({r['dgemm_tflops']:.1f} TF/s) | igemm call {t_i:.3f} ms, "
              f"GEMM kernel {t_k:.3f} ms ({r['igemm_equiv_fp64_tflops']:.1f} fp64-equivalent TF/s, "
              f"{r['int8_ops_per_s'] / 1e15:.2f} int8 POPS = {100 * r['int8_peak_share']:.1f} % of 4.5) | "
              f"x{r['speedup_kernel']:.2f} kernel, x{r['speedup_call']:.2f} call | {ks}", flush=True)
        del U, G, C
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "time_projection.json"), "w") as f:
            json.dump({"card": card(), "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
