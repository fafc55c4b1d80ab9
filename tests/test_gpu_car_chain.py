"""Caratheodory step on the register-resident pivot-chain kernel (car2.cu) at shapes that exercise every
compiled block size B, ragged last owner blocks, dependent rows (skipped in stage 1) and non-basic
sets that eliminate themselves (no basic set leaves, or a ratio >= 1).

`caratheodory_fast` picks B from S: the smallest of 1, 2, 4, 8 with ceil(S / B) <= #SMs (148 on a
B200), so S = 2n with n = 50, 100, 250, 1000 gives B = 1, 2, 4, 8.
"""
import pytest
import torch

from basq_b200 import ops

pytestmark = pytest.mark.gpu


def _system(n, S, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(n, S, generator=g, device="cuda", dtype=torch.float64)
    A[0] = torch.rand(S, generator=g, device="cuda", dtype=torch.float64) + 0.1  # set masses
    return A


def _check(A, om):
    n, S = A.shape
    assert om.shape == (S,)
    assert bool(torch.isfinite(om).all())
    assert float(om.min()) >= 0.0
    assert int((om > 0).sum()) <= n
    # A omega = A 1: row 0 is the mass, the other rows are moments
    res = (A @ om - A.sum(1)).abs() / A.abs().sum(1)
    assert float(res[0]) <= 1e-12, f"mass residual {float(res[0]):.2e}"
    assert float(res.max()) <= 1e-12, f"moment residual {float(res.max()):.2e}"


def _check_repeatable(A, om):
    # a second run of the same system must give the same bits (the pivot chain has no races)
    om2 = ops.caratheodory(A)
    assert torch.equal(om.view(torch.int64), om2.view(torch.int64))


@pytest.mark.parametrize("n", [50, 100, 250, 1000])
def test_car_chain_every_block_size(n):
    A = _system(n, 2 * n, seed=n)
    om = ops.caratheodory(A)
    _check(A, om)
    _check_repeatable(A, om)


@pytest.mark.parametrize("n,S", [(997, 1994), (251, 502), (101, 203)])
def test_car_chain_ragged_last_block(n, S):
    # n and S - n not multiples of B (8, 4, 2): the last owner block of both stages is partial
    A = _system(n, S, seed=n + S)
    om = ops.caratheodory(A)
    _check(A, om)
    _check_repeatable(A, om)


def test_car_chain_dependent_rows():
    n, S = 300, 600
    A = _system(n, S, seed=7)
    g = torch.Generator(device="cuda").manual_seed(8)
    C = torch.randn(12, 12, generator=g, device="cuda", dtype=torch.float64)
    A[20:32] = C @ A[1:13]          # rows 20..31 depend on rows 1..12: stage 1 skips 12 rows
    A[150] = 2.0 * A[3] - A[4]
    om = ops.caratheodory(A)
    _check(A, om)
    assert int((om > 0).sum()) <= n - 13
    _check_repeatable(A, om)


def test_car_chain_self_eliminating_sets():
    n, S = 250, 500
    A = _system(n, S, seed=11)
    # duplicates of other sets: their null vector has no negative entry, so no basic set can leave;
    # 2 a - b combinations: one negative entry with a ratio of about 1
    A[:, 300:340] = A[:, 0:40]
    A[:, 340:380] = 2.0 * A[:, 40:80] - A[:, 80:120]
    A[0, 340:380] = A[0, 40:80]     # keep the masses positive
    om = ops.caratheodory(A)
    _check(A, om)
    _check_repeatable(A, om)
