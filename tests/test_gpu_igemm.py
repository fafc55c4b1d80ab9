"""The fp64 GEMM on the int8 tensor cores (Ozaki slicing, igemm.cu) against correctly rounded references of
sampled entries, and against the fp64 DMMA GEMM on the same entries.  Run on the B200 box: pytest -m gpu."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def ops():
    from basq_b200 import ops
    return ops


def _two_prod(a, b):
    """a * b = p + e exactly (Dekker / Veltkamp splitting; no overflow or underflow at these magnitudes)."""
    p = a * b
    c = 134217729.0   # 2^27 + 1
    t = c * a; ah = t - (t - a); al = a - ah
    t = c * b; bh = t - (t - b); bl = b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact(a_row, b_col):
    """Correctly rounded sum_k a[k] b[k]."""
    p, e = _two_prod(np.asarray(a_row, dtype=np.float64), np.asarray(b_col, dtype=np.float64))
    return math.fsum(np.concatenate([p, e]).tolist())


def sample(m, n, count, seed):
    rng = np.random.default_rng(seed)
    return list(zip(rng.integers(0, m, count).tolist(), rng.integers(0, n, count).tolist()))


def errors(C, A, B, pts):
    """|C - exact| and (|A||B|)_ij at the sampled entries (A [m, k], B [k, n], CPU fp64)."""
    err, absab = [], []
    for i, j in pts:
        ref = exact(A[i], B[:, j])
        err.append(abs(float(C[i, j]) - ref))
        absab.append(float(np.abs(A[i]) @ np.abs(B[:, j])))
    return np.array(err), np.array(absab)


def bound(A, B, C, pts):
    """igemm.cu's error bound: 2^-50.8 K max|A_i.| max|B_.j| + 7 ulp-units of |C|, per sampled entry."""
    k = A.shape[1]
    return np.array([2.0 ** -50.8 * k * np.abs(A[i]).max() * np.abs(B[:, j]).max() + 7 * 2.0 ** -53 * abs(float(C[i, j]))
                     for i, j in pts])


def projection_operands(q, K, mtot, seed):
    """Operands drawn like the projection's: U' rows signed with per-row scales, folded set sums non-negative
    with columns spanning four decades."""
    g = torch.Generator().manual_seed(seed)
    U = torch.randn(q, mtot, generator=g, dtype=torch.float64) * torch.exp(torch.randn(q, 1, generator=g, dtype=torch.float64))
    G = 10.0 ** (-4.0 * torch.rand(mtot, K, generator=g, dtype=torch.float64))
    G *= 10.0 ** (3.0 * torch.rand(1, K, generator=g, dtype=torch.float64) - 1.0)
    return U, G


@pytest.mark.parametrize("K", [2000, 1000])
def test_projection_shapes(ops, K):
    q, mtot = 999, 11002
    U, G = projection_operands(q, K, mtot, seed=K)
    Ud, Gd = U.to(DEV), G.to(DEV)
    Ci = ops.igemm(Ud, Gd).cpu().numpy()
    Cd = ops.dgemm(Ud, Gd).cpu().numpy()
    A, B = U.numpy(), G.numpy()
    pts = sample(q, K, 48, seed=K + 1) + [(0, 0), (q - 1, K - 1)]
    ei, absab = errors(Ci, A, B, pts)
    ed, _ = errors(Cd, A, B, pts)
    assert (ei <= 2.0 ** -50 * absab).all(), f"worst {float((ei / absab).max()):.3g} of |A||B|"
    # no larger than the fp64 GEMM's error on the same entries, taken over the sample
    assert ei.max() <= ed.max() and ei.sum() <= ed.sum(), (ei.max(), ed.max(), ei.sum(), ed.sum())


def test_adversarial_rows(ops):
    """Rows whose entries span 2^-40 .. 2^40: the error stays within the bound relative to the row maximum."""
    m, n, k = 200, 130, 3000
    g = torch.Generator().manual_seed(5)
    sign = torch.where(torch.rand(m, k, generator=g) < 0.5, -1.0, 1.0).double()
    A = sign * torch.exp2(80.0 * torch.rand(m, k, generator=g, dtype=torch.float64) - 40.0)
    B = torch.randn(k, n, generator=g, dtype=torch.float64)
    C = ops.igemm(A.to(DEV), B.to(DEV)).cpu().numpy()
    An, Bn = A.numpy(), B.numpy()
    pts = sample(m, n, 64, seed=6)
    e, _ = errors(C, An, Bn, pts)
    assert (e <= bound(An, Bn, C, pts)).all()
    assert np.isfinite(C).all()


def test_zero_rows_and_columns(ops):
    m, n, k = 260, 150, 700
    g = torch.Generator().manual_seed(7)
    A = torch.randn(m, k, generator=g, dtype=torch.float64)
    B = torch.rand(k, n, generator=g, dtype=torch.float64)
    A[[0, 17, 259]] = 0.0
    B[:, [0, 63, 64, 149]] = 0.0
    C = ops.igemm(A.to(DEV), B.to(DEV)).cpu().numpy()
    assert (C[[0, 17, 259]] == 0.0).all() and (C[:, [0, 63, 64, 149]] == 0.0).all()
    An, Bn = A.numpy(), B.numpy()
    pts = sample(m, n, 40, seed=8)
    e, absab = errors(C, An, Bn, pts)
    assert (e <= 2.0 ** -50 * absab + 1e-300).all()


@pytest.mark.parametrize("m,n,k", [(130, 70, 1001), (1, 1, 1), (129, 65, 33)])
def test_ragged_shapes(ops, m, n, k):
    """I, J and K that are not multiples of the tiles (128, 64) or the K block (32)."""
    g = torch.Generator().manual_seed(m + n + k)
    A = torch.randn(m, k, generator=g, dtype=torch.float64)
    B = torch.randn(k, n, generator=g, dtype=torch.float64)
    C = ops.igemm(A.to(DEV), B.to(DEV)).cpu().numpy()
    An, Bn = A.numpy(), B.numpy()
    pts = [(i, j) for i in range(m) for j in range(n)] if m * n <= 64 else sample(m, n, 48, seed=k)
    e, _ = errors(C, An, Bn, pts)
    assert (e <= bound(An, Bn, C, pts)).all()
    ref = (A @ B).numpy()
    assert np.abs(C - ref).max() <= 1e-12 * np.abs(An).max() * np.abs(Bn).max() * k


@pytest.mark.parametrize("row0,nrows", [(37, 3001), (4999 - 17, 17), (0, 5000)])
def test_row_offset(ops, row0, nrows):
    """B multiplies the columns [row0, row0 + nrows) of A, as in the row-sharded projection."""
    m, n, k = 150, 90, 5000
    g = torch.Generator().manual_seed(row0)
    A = torch.randn(m, k, generator=g, dtype=torch.float64)
    B = torch.rand(nrows, n, generator=g, dtype=torch.float64)
    C = ops.igemm(A.to(DEV), B.to(DEV), row0=row0).cpu().numpy()
    As = A[:, row0:row0 + nrows].numpy()
    pts = sample(m, n, 40, seed=9)
    e, absab = errors(C, As, B.numpy(), pts)
    assert (e <= 2.0 ** -50 * absab).all()


def test_long_k_and_accumulate(ops):
    """K beyond one exact s32 launch (65504): the launches add in fp64; `out` is accumulated into."""
    m, n, k = 8, 16, 70000
    g = torch.Generator().manual_seed(11)
    A = torch.randn(m, k, generator=g, dtype=torch.float64)
    B = torch.rand(k, n, generator=g, dtype=torch.float64)
    C = ops.igemm(A.to(DEV), B.to(DEV)).cpu().numpy()
    An, Bn = A.numpy(), B.numpy()
    pts = [(i, j) for i in range(m) for j in range(n)]
    e, _ = errors(C, An, Bn, pts)
    assert (e <= bound(An, Bn, C, pts)).all()
    base = torch.full((m, n), 3.0, dtype=torch.float64, device=DEV)
    C2 = ops.igemm(A.to(DEV), B.to(DEV), out=base).cpu().numpy()
    assert np.abs(C2 - 3.0 - C).max() <= 4 * 2.0 ** -52 * (np.abs(C).max() + 3.0)
