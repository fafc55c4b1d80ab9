"""The precision sessions and weighted double sums evaluate the kernel in: fp64 inputs narrowed to fp32 at the
caller's request (basq_ctx_allow_f32_eval), fp32 evaluation restarted in fp64 when the conditioning guard trips
(kappa > 64).  Each route gives bit for bit the result of a call that hands the library the arrays the route
evaluates on, and counts one demotion / promotion per call.  Sessions are exercised through ops.features and
ops.recombine (VBQ kernel), the double sums through WSABI-M, the mode family their guard covers."""
import ctypes as C
import dataclasses
import math

import pytest
import torch

from oracle import gp_kernels as ogp

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
KINDS = ["session", "double_sums"]


def _stiff():
    # 40 clustered observations at noise 1e-10: kappa ~ 1e3 over Z and over X
    return ogp.make_gp(2, 40, lengthscale=1.0, noise=1e-10, seed=5)


def _tame():
    # the same observations at noise 1e-2: kappa ~ 8
    return ogp.make_gp(2, 40, lengthscale=1.0, noise=1e-2, seed=5)


def _spec(kind, model):
    # one spec per test: every call then sees the same W
    from basq_b200.kernels import describe_kernel
    gp = ogp.VanillaGP(model).predictive_kernel if kind == "session" else ogp.WsabiGP(model, alpha=0.05).wsabim_kernel
    return describe_kernel(gp)


@pytest.fixture(scope="module")
def pts():
    """fp64 X [3000, 2], Z = X[:200], U [20, 200], weights a, and a second operand Y [1700, 2] with weights b."""
    g = torch.Generator().manual_seed(31)
    X = math.sqrt(2.0) * torch.randn(3000, 2, generator=g, dtype=torch.float64)
    Y = math.sqrt(2.0) * torch.randn(1700, 2, generator=g, dtype=torch.float64)
    U = torch.linalg.qr(torch.randn(200, 20, generator=g, dtype=torch.float64)).Q.T.contiguous()
    a = torch.randn(3000, generator=g, dtype=torch.float64)
    b = torch.randn(1700, generator=g, dtype=torch.float64)
    return X, X[:200].clone(), U, a, Y, b


def _counts():
    from basq_b200 import _lib
    ctx = _lib.context_for(DEV)
    return ctx.allow_f32_eval(), ctx.conditioning()[1]


def _calls(kind, spec, X, Z, U, a, Y, b, counts):
    """Outputs of the kind's calls: features and recombine of a session on (X, Z, U), or the quadratic form Q(X, a)
    and the bilinear form B(X, a; Y, b).  Each call must count `counts` = (demotions, promotions)."""
    from basq_b200 import ops
    X, Z, Y = X.to(DEV), Z.to(DEV), Y.to(DEV)
    U, a, b = U.to(DEV), a.to(DEV), b.to(DEV)
    if kind == "session":
        calls = [lambda: ops.features(spec, X, Z, U), lambda: ops.recombine(spec, X, Z, U)]
    else:
        calls = [lambda: ops.kernel_quadform(spec, X, a), lambda: ops.kernel_bilinear(spec, X, a, Y, b)]
    out = []
    for call in calls:
        d0, p0 = _counts()
        out.append(call())
        d1, p1 = _counts()
        assert (d1 - d0, p1 - p0) == counts, (kind, d1 - d0, p1 - p0, counts)
    return out


def _assert_identical(got, want):
    for g, w in zip(got, want):
        if isinstance(g, float):
            assert g == w, (g, w)
        else:
            for gt, wt in zip(g if isinstance(g, tuple) else (g,), w if isinstance(w, tuple) else (w,)):
                assert torch.equal(gt, wt)


@pytest.mark.parametrize("kind", KINDS)
def test_promotion_evaluates_the_widened_inputs(kind, pts):
    """fp32 inputs of a stiff GP: the fp64 restart evaluates the inputs widened and the caller's fp64 observations."""
    X, Z, U, a, Y, b = pts
    spec = _spec(kind, _stiff())
    X32, Z32, Y32 = X.float(), Z.float(), Y.float()
    got = _calls(kind, spec, X32, Z32, U, a, Y32, b, (0, 1))
    want = _calls(kind, spec, X32.double(), Z32.double(), U, a, Y32.double(), b, (0, 0))
    _assert_identical(got, want)


@pytest.mark.parametrize("kind", KINDS)
def test_demotion_evaluates_the_narrowed_inputs(kind, pts):
    """fp64 inputs with the fp32 opt-in: the result of the fp32 inputs X.float(), Z.float() (Y.float())."""
    from basq_b200 import _lib
    X, Z, U, a, Y, b = pts
    spec = _spec(kind, _tame())
    want = _calls(kind, spec, X.float(), Z.float(), U, a, Y.float(), b, (0, 0))
    ctx = _lib.context_for(DEV)
    try:
        ctx.allow_f32_eval(True)
        got = _calls(kind, spec, X, Z, U, a, Y, b, (1, 0))
    finally:
        ctx.allow_f32_eval(False)
    _assert_identical(got, want)


@pytest.mark.parametrize("kind", KINDS)
def test_demotion_then_promotion_evaluates_the_callers_inputs(kind, pts):
    """fp64 inputs of a stiff GP with the fp32 opt-in: the guard sends the call back to the caller's own arrays."""
    from basq_b200 import _lib
    X, Z, U, a, Y, b = pts
    spec = _spec(kind, _stiff())
    want = _calls(kind, spec, X, Z, U, a, Y, b, (0, 0))
    ctx = _lib.context_for(DEV)
    try:
        ctx.allow_f32_eval(True)
        got = _calls(kind, spec, X, Z, U, a, Y, b, (1, 1))
    finally:
        ctx.allow_f32_eval(False)
    _assert_identical(got, want)


def test_promotion_without_fp64_observations_widens_them(pts):
    """A descriptor without Xobs_f64 (C callers may leave it NULL): the fp64 restart widens the fp32 observations."""
    from basq_b200 import _lib, ops
    X, Z, U, *_ = pts
    spec = _spec("session", _stiff())
    X32, Z32, Ud = X.float().to(DEV), Z.float().to(DEV), U.to(DEV)
    ctx = _lib.context_for(DEV)
    desc, keep = spec.to_desc(2, DEV, torch.float32)
    desc.Xobs_f64 = None
    Phi = torch.empty(len(X32), len(Ud), dtype=torch.float64, device=DEV)
    d0, p0 = _counts()
    _lib.check(_lib.lib.basq_features(ctx.handle, C.byref(desc), X32.data_ptr(), len(X32), Z32.data_ptr(), len(Z32),
                                      Ud.data_ptr(), len(Ud), Phi.data_ptr()))
    d1, p1 = _counts()
    assert (d1 - d0, p1 - p0) == (0, 1)
    widened = dataclasses.replace(spec, Xobs=spec.Xobs.float().double())
    d0, p0 = _counts()
    want = ops.features(widened, X32.double(), Z32.double(), Ud)
    assert _counts() == (d0, p0)
    assert torch.equal(Phi, want)
