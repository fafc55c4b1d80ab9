"""GP posterior mean over 1e7 candidates (n_obs = 1002) on the tensor-core path of fp32 inputs, and its
agreement with the fp64 path."""
import math, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from basq_b200 import _lib, gp, ops, sampler
from basq_b200.kernels import spec_from_model
dev = torch.device("cuda:0")
N = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
g = torch.Generator().manual_seed(5)
Xo = math.sqrt(2.0) * torch.randn(1002, 10, generator=g, dtype=torch.float64)
c = 1.5 * torch.randn(3, 10, generator=g, dtype=torch.float64)
yo = sum(torch.exp(-0.25 * ((Xo - ci) ** 2).sum(-1)) for ci in c) / 3.0
m = gp.FixedGP(Xo.to(dev, torch.float32), torch.sqrt(2.0 * yo).to(dev), gp.ScaleKernel(gp.RBFKernel(2.5), 1.0), noise=1e-4)
kern = spec_from_model(m, _lib.WSABI_L)
X = sampler.sample_mvn(torch.zeros(10), 2.0 * torch.eye(10), N, seed=9, device=dev)
def t(fn, reps=5):
    fn(); fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): out = fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out
ms, (mean, _) = t(lambda: ops.gp_predict(kern, X, space=0, want_var=False))
ref = (ops.gp_predict(kern, X[:200000].double(), space=0, want_var=False)[0])
err = float((mean[:200000] - ref).abs().max() / ref.abs().max())
print(f"fp32 tensor-core mean over {N:.0e} candidates {ms:.2f} ms; max rel. difference to the fp64 path {err:.2e}")
