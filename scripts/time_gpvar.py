"""The posterior-variance kernels on one box, same process: fused (kernel values generated on the SM) vs
the round-1 fp64 GEMM path; SM clock sampled."""
import math, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from basq_b200 import _lib, gp, ops, sampler
from basq_b200.kernels import spec_from_model
import bench
dev = torch.device("cuda:0")
Xo, yo = bench.make_observations(10, 1002, seed=5)
model = gp.FixedGP(Xo.to(dev, torch.float32), yo.to(dev), gp.ScaleKernel(gp.RBFKernel(2.5), 1.0), noise=1e-10)
kern = spec_from_model(model, _lib.PRED_COV)
N = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
X = sampler.sample_mvn(torch.zeros(10), 2.0 * torch.eye(10), N, seed=9, device=dev)
def clock():
    return subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
def run(tag, env, reps=4):
    os.environ.update(env)
    ops.gp_predict(kern, X, space=0, want_var=True)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); mean, var = ops.gp_predict(kern, X, space=0, want_var=True); e1.record()
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); ops.gp_predict(kern, X, space=0, want_var=False); e1.record(); torch.cuda.synchronize()
    print(f"{tag:28s} mean+var {min(ts):7.2f} ms (median {sorted(ts)[len(ts)//2]:7.2f}); mean only {e0.elapsed_time(e1):6.2f} ms; {clock()}", flush=True)
    return var
for rnd in range(2):
    v1 = run("fused", {"BASQ_GPVAR": "1"})
v3 = run("fp64 GEMM (round 1)", {"BASQ_GPVAR": "0"}, reps=2)
print("max |fused - fp64| %.3e" % float((v1 - v3).abs().max()))

# where calc_weights spends its time (UncertaintySampler.calc_weights = moments + one elementwise pass)
os.environ.update({"BASQ_GPVAR": "1"})
from basq_b200 import sampler as bs
bs.calc_weights(kern, X, ratio=0.5); torch.cuda.synchronize()
for rep in range(2):
    t0 = time.perf_counter(); mean, var = ops.gp_predict(kern, X, space=0, want_var=True); torch.cuda.synchronize()
    t1 = time.perf_counter(); w = bs._weights(0, 0.5, False, mean, var, True); torch.cuda.synchronize()
    t2 = time.perf_counter(); w2 = bs.calc_weights(kern, X, ratio=0.5); torch.cuda.synchronize()
    t3 = time.perf_counter()
    print(f"gp_predict {1e3*(t1-t0):.1f} ms, weights kernel + normalise {1e3*(t2-t1):.1f} ms, calc_weights (both) {1e3*(t3-t2):.1f} ms")
