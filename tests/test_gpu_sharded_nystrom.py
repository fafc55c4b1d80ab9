"""Row-sharded Nystrom basis (basq_nystrom_basis_sharded): one shard must reproduce basq_nystrom_basis, two ranks
(two processes on the one GPU of the test box, gloo with host staging standing in for NCCL) must agree with it
up to the summation order of the Gram matrices."""
import math
import os
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import gp_kernels as ogp

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _case(kind):
    g = torch.Generator().manual_seed(31)
    M, d, q = 301, 5, 40
    Z = math.sqrt(2.0) * torch.randn(M, d, generator=g)
    omega = torch.randn(M, q, generator=g, dtype=torch.float64)
    if kind == "plain":
        kern = ogp.ScaleKernel(ogp.RBFKernel(1.8), 1.2).forward
    else:   # posterior covariance with the BASQ noise-diagonal quirk: the diagonal sits at (i, row0 + i) of a row block
        model = ogp.make_gp(d, 25, lengthscale=1.8, outputscale=1.2, noise=1e-2, seed=4)
        kern = ogp.VanillaGP(model, add_noise_diag=True).predictive_kernel
    return Z, omega, q, kern


@pytest.mark.parametrize("kind,dtype,niter", [
    pytest.param(kind, dtype, niter, id=kind + suffix)
    for dtype, niter, suffix in [(torch.float32, 2, ""), (torch.float64, 2, "-fp64"), (torch.float32, 0, "-niter0")]
    for kind in ("plain", "pred_cov_noise_diag")])
def test_one_shard_equals_the_plain_entry(kind, dtype, niter):
    from basq_b200 import ops, sharded
    Z, omega, q, kern = _case(kind)
    Z = Z.to(DEV, dtype)
    _, U0 = ops.nystrom_basis(kern, Z, q, omega=omega.to(DEV), niter=niter, want_S=False)
    U1 = sharded.nystrom_basis_sharded(kern, Z, q, omega=omega.to(DEV), niter=niter)
    assert torch.equal(U0, U1)


def _worker(rank, world, rdzv, kind, out_path):
    from basq_b200 import sharded
    dist.init_process_group("gloo", init_method=f"file://{rdzv}", rank=rank, world_size=world)
    try:
        Z, omega, q, kern = _case(kind)
        U = sharded.nystrom_basis_sharded(kern, Z.to(DEV), q, omega=omega.to(DEV))
        # the library-drawn test matrix: rank 0's torch generator decides, every rank must end with the same basis
        torch.manual_seed(100 + rank)
        U2 = sharded.nystrom_basis_sharded(kern, Z.to(DEV), q)
        chk = torch.stack([U.sum(), U.abs().sum(), U2.sum(), U2.abs().sum()]).cpu()
        ref = chk.clone()
        dist.broadcast(ref, 0)
        assert torch.equal(chk, ref)
        if rank == 0:
            torch.save({"U": U.cpu(), "U2": U2.cpu()}, out_path)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("kind", ["plain", "pred_cov_noise_diag"])
def test_two_ranks_agree_with_the_plain_entry(kind):
    from basq_b200 import ops
    Z, omega, q, kern = _case(kind)
    _, U0 = ops.nystrom_basis(kern, Z.to(DEV), q, omega=omega.to(DEV), want_S=False)
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "u.pt")
        mp.spawn(_worker, args=(2, os.path.join(tmp, "rdzv"), kind, out), nprocs=2, join=True)
        got = torch.load(out)
    U, U2 = got["U"].to(DEV), got["U2"].to(DEV)
    eye = torch.eye(q, dtype=torch.float64, device=DEV)
    assert float((U @ U.T - eye).abs().max()) < 1e-12 and float((U2 @ U2.T - eye).abs().max()) < 1e-12
    # same algorithm; a row block centres its coordinates on its own rows and sums the Gram matrices in another
    # order, so the fp32 kernel values differ in their last bits (observed 7e-7 on the basis)
    assert float((U - U0).abs().max()) < 5e-6
    # another test matrix, (nearly) the same dominant subspace: captured energy of K agrees
    K = ops.gram(kern, Z.to(DEV), Z.to(DEV)).double()
    e0, e2 = float(torch.trace(U0 @ K @ U0.T)), float(torch.trace(U2 @ K @ U2.T))
    assert abs(e0 - e2) < 5e-3 * abs(e0)        # observed 5.5e-4: q = 40 of 301 directions, two random test matrices
