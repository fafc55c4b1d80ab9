"""One-off probes: (1) cuBLAS fp64 GEMM rate on the projection shape vs basq_dgemm; (2) orthonormality
and captured trace of the Nystrom basis."""
import math, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from basq_b200 import _lib, ops, gp as bgp
from basq_b200.kernels import spec_from_model
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)

def timeit(fn, reps=5):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps

if "gemm" in sys.argv:
    q, K, N = 999, 11002, 2000
    A = torch.randn(q, K, generator=g, device=dev, dtype=torch.float64)
    B = torch.randn(K, N, generator=g, device=dev, dtype=torch.float64)
    fl = 2.0 * q * K * N
    t = timeit(lambda: torch.matmul(A, B)); print(f"cuBLAS dgemm {q}x{K}x{N}: {t:.3f} ms  {fl/t/1e9:.1f} TF/s")
    t = timeit(lambda: ops.dgemm(A, B)); print(f"basq  dgemm {q}x{K}x{N}: {t:.3f} ms  {fl/t/1e9:.1f} TF/s")
    Y = torch.randn(10000, 999, generator=g, device=dev, dtype=torch.float64)
    fl = 2.0 * 999 * 999 * 10000
    t = timeit(lambda: torch.matmul(Y.T, Y)); print(f"cuBLAS Y^T Y: {t:.3f} ms  {fl/t/1e9:.1f} TF/s")
    t = timeit(lambda: ops.dgemm(Y, Y, transA=True)); print(f"basq  Y^T Y: {t:.3f} ms  {fl/t/1e9:.1f} TF/s")

if "nys" in sys.argv:
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    d, M, q, n_obs = 10, 10000, 999, 1002
    Xo, yo = bench.make_observations(d, n_obs)
    model = bgp.FixedGP(Xo.to(dev, torch.float32), yo.to(dev), bgp.ScaleKernel(bgp.RBFKernel(2.5), 1.0), noise=1e-10)
    kern = spec_from_model(model, _lib.PRED_COV)
    X = math.sqrt(2.0) * torch.randn(M, d, generator=g, device=dev)
    Om = torch.randn(M, q, generator=g, device=dev, dtype=torch.float64)
    t = timeit(lambda: ops.nystrom_basis(kern, X, q, omega=Om, want_S=False), reps=3)
    _, U = ops.nystrom_basis(kern, X, q, omega=Om, want_S=False)
    E = U @ U.T - torch.eye(q, device=dev, dtype=torch.float64)
    Kp = ops.gram(kern, X, X)
    # captured energy of the posterior-covariance Gram in span(U), relative to the exact top-q eigenspace
    ev = torch.linalg.eigvalsh(Kp)
    cap = torch.trace(U @ Kp @ U.T)
    print(f"nystrom: {t:.2f} ms  |UU^T-I|_max={float(E.abs().max()):.2e}  "
          f"captured trace {float(cap):.6f} vs top-q eigenvalues {float(ev[-q:].sum()):.6f} (total {float(ev.sum()):.6f})")
