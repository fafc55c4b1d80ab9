"""Thin torch-tensor wrappers over the C ABI (device pointers in, torch tensors out).

torch is used for device memory and streams only; all arithmetic happens inside libbasq_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .kernels import KernelSpec, describe_kernel


def _prep(x: torch.Tensor, device, dtype):
    return x.detach().to(device=device, dtype=dtype).contiguous()


def _common(kernel, X, device=None):
    spec = describe_kernel(kernel)
    device = torch.device(device) if device is not None else X.device
    dtype = X.dtype if X.dtype in (torch.float32, torch.float64) else torch.float32
    ctx = _lib.context_for(device)
    return spec, ctx, device, dtype


def gram(kernel, X, Y, device=None) -> torch.Tensor:
    """kernel(X, Y) as an fp64 [a, b] tensor - replaces the reference's kernel callable."""
    spec, ctx, device, dtype = _common(kernel, X, device)
    Xd, Yd = _prep(X, device, dtype), _prep(Y, device, dtype)
    desc, keep = spec.to_desc(Xd.shape[1], device, dtype)
    out = torch.empty(len(Xd), len(Yd), dtype=torch.float64, device=device)
    _lib.check(_lib.lib.basq_gram(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), Yd.data_ptr(), len(Yd),
                                  out.data_ptr()))
    return out


def gp_predict(kernel, X, space=0, want_var=True, device=None):
    """GP posterior mean / variance over candidates (BASQ/_gp.py:213-230, exact variance).
    space=1 returns the model-space moments of the kernel's mode (wsabi*_predict / gspace_predict).
    For float32 inputs the variance (also needed by the WSABI-M / MMLT model space) takes GPs of at most 32768
    observations; more raises BasqError with ERR_UNSUPPORTED."""
    spec, ctx, device, dtype = _common(kernel, X, device)
    Xd = _prep(X, device, dtype)
    desc, keep = spec.to_desc(Xd.shape[1], device, dtype)
    mean = torch.empty(len(Xd), dtype=torch.float64, device=device)
    var = torch.empty(len(Xd), dtype=torch.float64, device=device) if want_var else None
    _lib.check(_lib.lib.basq_gp_predict(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), int(space),
                                        float(spec.offset), mean.data_ptr(), var.data_ptr() if want_var else None))
    return mean, var


def _weights(w, n, device, what):
    wd = _prep(torch.as_tensor(w), device, torch.float64)
    if wd.shape != (n,):
        raise ValueError(f"{what} must have one entry per point ({n}), not shape {tuple(wd.shape)}")
    return wd


def kernel_quadform(kernel, X, a, device=None) -> float:
    """a^T kernel(X, X) a for fp64 weights a [N] (any sign) without forming the N x N matrix
    (basq_kernel_quadform): the square Gram matrix of ``gram``, diagonal terms included, summed in fp64 in a
    fixed order.  Every mode of ``describe_kernel``."""
    spec, ctx, device, dtype = _common(kernel, X, device)
    Xd = _prep(X, device, dtype)
    ad = _weights(a, len(Xd), device, "a")
    desc, keep = spec.to_desc(Xd.shape[1], device, dtype)
    out = C.c_double(0.0)
    _lib.check(_lib.lib.basq_kernel_quadform(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), ad.data_ptr(),
                                             C.byref(out)))
    return float(out.value)


def kernel_bilinear(kernel, X, a, Y, b, device=None) -> float:
    """sum_ij a_i b_j kernel(x_i, y_j) (basq_kernel_bilinear): the kernel function alone, without the diagonal
    terms of the square Gram matrix even when Y is X."""
    spec, ctx, device, dtype = _common(kernel, X, device)
    Xd, Yd = _prep(X, device, dtype), _prep(Y, device, dtype)
    ad, bd = _weights(a, len(Xd), device, "a"), _weights(b, len(Yd), device, "b")
    desc, keep = spec.to_desc(Xd.shape[1], device, dtype)
    out = C.c_double(0.0)
    _lib.check(_lib.lib.basq_kernel_bilinear(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), ad.data_ptr(),
                                             Yd.data_ptr(), len(Yd), bd.data_ptr(), C.byref(out)))
    return float(out.value)


def _seed_context(ctx, seed):
    """Key of the library's next Gaussian draw: the caller's, or - like every torch routine the reference
    calls - the next value of torch's global generator, so that torch.manual_seed reproduces a run."""
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64))
    ctx.set_seed(seed)


def nystrom_basis(kernel, Z, q, omega=None, niter=2, device=None, want_S=True, seed=None):
    """(S, U): U [q, M] is an orthonormal basis of the randomised range of K(Z, Z) (ker_svd_sparsify,
    BASQ/_rchq.py:28-31) - an arbitrary basis of that span, not the singular vectors (recombination
    only depends on the span); S [q] holds the Rayleigh quotients u_i^T K u_i of its rows, unordered.
    omega [M, q] = None lets the library draw the Gaussian test matrix on the device, as torch.svd_lowrank
    does inside the reference; its Philox key is `seed`, by default the next value of torch's global generator
    (torch.manual_seed reproduces the basis, as it does in the reference).  want_S=False skips S (the
    reference discards it, BASQ/_rchq.py:36)."""
    spec, ctx, device, dtype = _common(kernel, Z, device)
    Zd = _prep(Z, device, dtype)
    M = len(Zd)
    if omega is not None:
        omega = _prep(omega, device, torch.float64)
    else:
        _seed_context(ctx, seed)
    desc, keep = spec.to_desc(Zd.shape[1], device, dtype)
    U = torch.empty(q, M, dtype=torch.float64, device=device)
    S = torch.empty(q, dtype=torch.float64, device=device) if want_S else None
    _lib.check(_lib.lib.basq_nystrom_basis(ctx.handle, C.byref(desc), Zd.data_ptr(), M, int(q),
                                           omega.data_ptr() if omega is not None else None,
                                           int(niter), U.data_ptr(), S.data_ptr() if want_S else None))
    return S, U


def features(kernel, X, Z, U, device=None) -> torch.Tensor:
    """Phi [N, q] = (U @ kernel(Z, X))^T in fp64 - the test functions recombination preserves."""
    spec, ctx, device, dtype = _common(kernel, X, device)
    Xd, Zd = _prep(X, device, dtype), _prep(Z, device, dtype)
    Ud = _prep(U, device, torch.float64)
    desc, keep = spec.to_desc(Xd.shape[1], device, dtype)
    q = Ud.shape[0]
    Phi = torch.empty(len(Xd), q, dtype=torch.float64, device=device)
    _lib.check(_lib.lib.basq_features(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), Zd.data_ptr(), len(Zd),
                                      Ud.data_ptr(), q, Phi.data_ptr()))
    return Phi


def caratheodory(A: torch.Tensor) -> torch.Tensor:
    """omega [S] >= 0 with <= n non-zeros and A omega = A 1 for A [n, S] (row 0 = set masses)."""
    ctx = _lib.context_for(A.device)
    Ad = A.detach().to(torch.float64).contiguous().clone()
    n, S = Ad.shape
    omega = torch.zeros(S, dtype=torch.float64, device=A.device)
    _lib.check(_lib.lib.basq_car(ctx.handle, Ad.data_ptr(), n, S, S, omega.data_ptr(), None))
    return omega


def dgemm(A, B, transA=False, transB=False):
    ctx = _lib.context_for(A.device)
    A = A.contiguous(); B = B.contiguous()
    m = A.shape[1] if transA else A.shape[0]
    k = A.shape[0] if transA else A.shape[1]
    n = B.shape[0] if transB else B.shape[1]
    Cm = torch.empty(m, n, dtype=torch.float64, device=A.device)
    _lib.check(_lib.lib.basq_dgemm(ctx.handle, int(transA), int(transB), m, n, k, 1.0, A.data_ptr(), A.shape[1],
                                   B.data_ptr(), B.shape[1], 0.0, Cm.data_ptr(), n))
    return Cm


def tgemm(A, B):
    """A @ B.T on the tensor cores with fp32 accuracy (fp16 hi/lo split, three products); fp64 tensors in and out."""
    ctx = _lib.context_for(A.device)
    A = A.to(torch.float64).contiguous(); B = B.to(torch.float64).contiguous()
    m, k = A.shape
    n = B.shape[0]
    assert B.shape[1] == k
    Cm = torch.empty(m, n, dtype=torch.float64, device=A.device)
    _lib.check(_lib.lib.basq_tgemm(ctx.handle, m, n, k, A.data_ptr(), k, B.data_ptr(), k, Cm.data_ptr(), n))
    return Cm


def igemm(A, B, row0=0, out=None):
    """A[:, row0:row0 + len(B)] @ B with fp64 accuracy on the int8 tensor cores (Ozaki slicing, the projection's
    GEMM); fp64 tensors in and out.  With ``out`` the product is added to it."""
    ctx = _lib.context_for(A.device)
    A = A.to(torch.float64).contiguous(); B = B.to(torch.float64).contiguous()
    m, k = A.shape
    nrows, n = B.shape
    if row0 < 0 or row0 + nrows > k:
        raise ValueError(f"rows [{row0}, {row0 + nrows}) of B lie outside A's {k} columns")
    accumulate = out is not None
    if out is None:
        out = torch.empty(m, n, dtype=torch.float64, device=A.device)
    assert out.shape == (m, n) and out.dtype == torch.float64 and out.is_contiguous()
    _lib.check(_lib.lib.basq_igemm(ctx.handle, m, n, k, A.data_ptr(), k, row0, nrows, B.data_ptr(), n,
                                   out.data_ptr(), n, int(accumulate)))
    return out


def recombine(kernel, pts_rec, pts_nys, U, mu=None, device=None, obj=None):
    """Tchernychova-Lyons recombination with a given basis U [q, M]: (idx int64, w fp64) on device.
    obj [N]: the reference's ``-calc_obj(samp)`` for the objective-aware variant (SOBER/_rchq.py:67-69)."""
    spec, ctx, device, dtype = _common(kernel, pts_rec, device)
    Xd, Zd = _prep(pts_rec, device, dtype), _prep(pts_nys, device, dtype)
    Ud = _prep(U, device, torch.float64)
    q = Ud.shape[0]
    if Ud.shape[1] != len(Zd):
        raise ValueError(f"U has {Ud.shape[1]} columns for {len(Zd)} Nystrom points")
    mud = None
    if mu is not None:
        mud = _prep(mu, device, torch.float64)
        if mud.shape != (len(Xd),):
            raise ValueError("init_weights must have one entry per candidate")
    desc, keep = spec.to_desc(Xd.shape[1], device, dtype)
    idx = torch.empty(q + 1, dtype=torch.int64, device=device)
    w = torch.empty(q + 1, dtype=torch.float64, device=device)
    n_out = C.c_int(0)
    if obj is not None:
        objd = _prep(obj, device, torch.float64)
        if objd.shape != (len(Xd),):
            raise ValueError("obj must have one entry per candidate")
        _lib.check(_lib.lib.basq_recombine_objective(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), Zd.data_ptr(),
                                                     len(Zd), Ud.data_ptr(), q,
                                                     mud.data_ptr() if mud is not None else None, objd.data_ptr(),
                                                     idx.data_ptr(), w.data_ptr(), C.byref(n_out)))
        return idx[: n_out.value], w[: n_out.value]
    _lib.check(_lib.lib.basq_recombine(ctx.handle, C.byref(desc), Xd.data_ptr(), len(Xd), Zd.data_ptr(), len(Zd),
                                       Ud.data_ptr(), q, mud.data_ptr() if mud is not None else None,
                                       idx.data_ptr(), w.data_ptr(), C.byref(n_out)))
    return idx[: n_out.value], w[: n_out.value]


def recombine_host(kernel, X_host, Z_host, q, U_host=None, omega_host=None, mu_host=None, niter=2, device="cuda",
                   seed=None):
    """The same through basq_recombine_host: HOST (ideally pinned) buffers in, host tensors out;
    all host<->device copies happen inside the call (bench.py's end-to-end leg).  With neither U_host
    nor omega_host the library draws the Nystrom test matrix on the device (the reference's call shape:
    torch.svd_lowrank draws its own, BASQ/_rchq.py:28-31) with the Philox key `seed` (see nystrom_basis)."""
    spec = describe_kernel(kernel)
    device = torch.device(device)
    ctx = _lib.context_for(device)
    dtype = X_host.dtype
    if dtype not in (torch.float32, torch.float64):
        raise TypeError(f"recombine_host: candidates must be float32 or float64, not {dtype}")
    if X_host.device.type != "cpu" or Z_host.device.type != "cpu":
        raise ValueError("recombine_host takes HOST tensors (use recombine for device tensors)")
    if X_host.dim() != 2 or Z_host.dim() != 2 or Z_host.shape[1] != X_host.shape[1]:
        raise ValueError(f"recombine_host: X {tuple(X_host.shape)} and Z {tuple(Z_host.shape)} must be [N, d] and [M, d]")
    # the C call copies raw bytes with the descriptor's element size: every buffer must have it
    X_host, Z_host = X_host.contiguous(), Z_host.to(dtype).contiguous()
    N, M = len(X_host), len(Z_host)
    if U_host is not None and tuple(U_host.shape) != (q, M):
        raise ValueError(f"U_host has shape {tuple(U_host.shape)}, expected {(q, M)}")
    if omega_host is not None and tuple(omega_host.shape) != (M, q):
        raise ValueError(f"omega_host has shape {tuple(omega_host.shape)}, expected {(M, q)}")
    if mu_host is not None and tuple(mu_host.shape) != (N,):
        raise ValueError(f"mu_host has shape {tuple(mu_host.shape)}, expected {(N,)}")
    for name, t in (("U_host", U_host), ("omega_host", omega_host), ("mu_host", mu_host)):
        if t is not None and t.device.type != "cpu":
            raise ValueError(f"{name} must be a host tensor")
    desc, keep = spec.to_desc(X_host.shape[1], device, dtype)
    idx = torch.empty(q + 1, dtype=torch.int64)
    w = torch.empty(q + 1, dtype=torch.float64)
    n_out = C.c_int(0)
    ptr = lambda t: (t.contiguous().data_ptr() if t is not None else None)
    if U_host is not None:
        U_host = U_host.to(torch.float64).contiguous()
    if omega_host is not None:
        omega_host = omega_host.to(torch.float64).contiguous()
    if mu_host is not None:
        mu_host = mu_host.to(torch.float64).contiguous()
    if U_host is None and omega_host is None:
        _seed_context(ctx, seed)
    _lib.check(_lib.lib.basq_recombine_host(ctx.handle, C.byref(desc), X_host.data_ptr(), len(X_host),
                                            Z_host.data_ptr(), len(Z_host), ptr(U_host), int(q), ptr(omega_host),
                                            int(niter), ptr(mu_host), idx.data_ptr(), w.data_ptr(),
                                            C.byref(n_out)))
    return idx[: n_out.value], w[: n_out.value]


_F = {torch.float32: _lib.F32, torch.float64: _lib.F64}


def stage_candidates(X_host, mu_host=None, device="cuda"):
    """Start copying a rank's shard of candidates (and weights) from HOST (ideally pinned) memory into the
    context's device buffer (basq_ctx_stage_candidates); returns (N_loc, dtype) for Session(staged=...).
    The copy runs on a side stream: build the basis meanwhile."""
    if X_host.device.type != "cpu" or X_host.dim() != 2 or X_host.dtype not in _F:
        raise ValueError("stage_candidates takes a host tensor [N_loc, d] in float32 or float64")
    X_host = X_host.contiguous()
    if mu_host is not None:
        if mu_host.device.type != "cpu" or tuple(mu_host.shape) != (len(X_host),):
            raise ValueError(f"mu_host must be a host tensor of shape {(len(X_host),)}")
        mu_host = mu_host.to(torch.float64).contiguous()
    ctx = _lib.context_for(torch.device(device))
    _lib.check(_lib.lib.basq_ctx_stage_candidates(ctx.handle, X_host.data_ptr(), len(X_host), X_host.shape[1],
                                                  _F[X_host.dtype], mu_host.data_ptr() if mu_host is not None else None))
    ctx._staged_keep = (X_host, mu_host)      # the host buffers must outlive the copy
    return len(X_host), X_host.dtype


class Session:
    """Staged recombination over a rank-local shard (basq_session_* in the C ABI)."""

    def __init__(self, kernel, X_loc, Z, U, N_glob, idx_base, mu_loc=None, device=None, obj_loc=None, staged=None):
        """staged = (N_loc, dtype): the shard was handed over with stage_candidates (host buffers); X_loc and
        mu_loc are then ignored."""
        if staged is not None:
            n_loc, dtype = int(staged[0]), staged[1]
            spec = describe_kernel(kernel)
            device = torch.device(device if device is not None else Z.device)
            ctx = _lib.context_for(device)
        else:
            spec, ctx, device, dtype = _common(kernel, X_loc, device)
        self.ctx, self.device = ctx, device
        Zd = _prep(Z, device, dtype)
        Ud = _prep(U, device, torch.float64)
        self.q = Ud.shape[0]
        self.n = self.q + 1
        self.S = 2 * self.n
        desc, keep = spec.to_desc(Zd.shape[1], device, dtype)
        h = C.c_void_p()
        if staged is not None:
            self._keep = keep + [Zd, Ud]
            _lib.check(_lib.lib.basq_session_create_staged(ctx.handle, C.byref(desc), n_loc, int(N_glob), int(idx_base),
                                                           Zd.data_ptr(), len(Zd), Ud.data_ptr(), self.q, C.byref(h)))
        else:
            Xd = _prep(X_loc, device, dtype)
            n_loc = len(Xd)
            mud = _prep(mu_loc, device, torch.float64) if mu_loc is not None else None
            self._keep = keep + [Xd, Zd, Ud, mud]
            _lib.check(_lib.lib.basq_session_create(ctx.handle, C.byref(desc), Xd.data_ptr() if len(Xd) else None,
                                                    len(Xd), int(N_glob), int(idx_base), Zd.data_ptr(), len(Zd),
                                                    Ud.data_ptr(), self.q,
                                                    mud.data_ptr() if mud is not None else None, C.byref(h)))
        self.handle = h
        self.rows = self.n
        if obj_loc is not None:
            objd = _prep(obj_loc, device, torch.float64)
            assert objd.shape == (n_loc,)
            self._keep.append(objd)
            _lib.check(_lib.lib.basq_session_set_objective(h, objd.data_ptr()))
            self.rows = self.n + 1
        self.has_obj = obj_loc is not None

    def close(self):
        h, self.handle = getattr(self, "handle", None), None
        if h and _lib is not None and _lib.lib is not None:
            _lib.lib.basq_session_destroy(h)

    __del__ = close

    def count(self) -> int:
        c = C.c_int64(0)
        _lib.check(_lib.lib.basq_session_count(self.handle, C.byref(c)))
        return int(c.value)

    def cell_factor(self, R_glob, R_loc_max) -> int:
        """Cells per set (1, 2, 4, 8) the library picks for a pass over R_glob live points."""
        f = C.c_int(1)
        _lib.check(_lib.lib.basq_session_cell_factor(self.handle, int(R_glob), int(R_loc_max), C.byref(f)))
        return int(f.value)

    def partial(self, R_glob, off_glob, A: torch.Tensor):
        """The reference's round: local part of the [n, S] barycentre system (pass with F = 1)."""
        assert A.dtype == torch.float64 and A.is_contiguous() and A.shape == (self.n, self.S)
        _lib.check(_lib.lib.basq_session_partial(self.handle, int(R_glob), int(off_glob), A.data_ptr()))

    def pass_begin(self, R_glob, off_glob, F):
        """The sweep of a pass: cell sums of this rank's live points over F*S cells."""
        _lib.check(_lib.lib.basq_session_pass_begin(self.handle, int(R_glob), int(off_glob), int(F)))

    def level(self, lvl, node, ppos, fpar, A: torch.Tensor):
        """Local part of level `lvl` of the current pass into A [n, S] (see basq_session_level)."""
        assert A.dtype == torch.float64 and A.is_contiguous() and A.shape == (self.rows, self.S)
        K = len(node)
        nd = np.ascontiguousarray(node, dtype=np.int32)
        pp = np.ascontiguousarray(ppos if lvl > 0 else np.zeros(K), dtype=np.int32)
        fp = np.ascontiguousarray(fpar, dtype=np.float64)
        _lib.check(_lib.lib.basq_session_level(self.handle, int(lvl), K, nd.ctypes.data, pp.ctypes.data,
                                               fp.ctypes.data, A.data_ptr()))

    # --- the same level in two halves, with a reduce-scatter of the folded columns in between ---------
    def landmarks(self) -> int:
        m = C.c_int(0)
        _lib.check(_lib.lib.basq_session_landmarks(self.handle, C.byref(m)))
        return int(m.value)

    def shared_buffers(self, world):
        """(Gf flat buffer for [Mtot_pad, K] views, block buffer for [Mtot_pad / world, K]); rows padded
        to a multiple of `world` (padding rows never enter a projection)."""
        if getattr(self, "_shared", None) is None or self._shared[0] != world:
            Mtot = self.landmarks()
            rows_blk = -(-Mtot // world)
            Gf = torch.zeros(rows_blk * world * self.S, dtype=torch.float64, device=self.device)
            blk = torch.zeros(rows_blk * self.S, dtype=torch.float64, device=self.device)
            self._shared = (world, Mtot, rows_blk, Gf, blk)
        return self._shared[1:]

    def level_fold(self, lvl, node, Gf: torch.Tensor):
        K = len(node)
        nd = np.ascontiguousarray(node, dtype=np.int32)
        _lib.check(_lib.lib.basq_session_level_fold(self.handle, int(lvl), K, nd.ctypes.data, Gf.data_ptr(), K))

    def level_project(self, lvl, node, ppos, fpar, Gf_rows: torch.Tensor, row0, nrows, A: torch.Tensor):
        assert A.dtype == torch.float64 and A.is_contiguous() and A.shape == (self.rows, self.S)
        K = len(node)
        nd = np.ascontiguousarray(node, dtype=np.int32)
        pp = np.ascontiguousarray(ppos if lvl > 0 else np.zeros(K), dtype=np.int32)
        fp = np.ascontiguousarray(fpar, dtype=np.float64)
        _lib.check(_lib.lib.basq_session_level_project(self.handle, int(lvl), K, nd.ctypes.data, pp.ctypes.data,
                                                       fp.ctypes.data, Gf_rows.data_ptr(), K, int(row0), int(nrows),
                                                       A.data_ptr()))

    def car(self, A: torch.Tensor, C_cols: int, omega: torch.Tensor):
        if self.has_obj:
            _lib.check(_lib.lib.basq_car_objective(self.ctx.handle, A.data_ptr(), self.n, int(C_cols), self.S,
                                                   omega.data_ptr()))
        else:
            _lib.check(_lib.lib.basq_car(self.ctx.handle, A.data_ptr(), self.n, int(C_cols), self.S, omega.data_ptr(), None))

    def apply(self, R_glob, off_glob, F, factor: torch.Tensor) -> int:
        c = C.c_int64(0)
        assert factor.device.type == "cpu" and factor.dtype == torch.float64 and factor.numel() == F * self.S
        factor = factor.contiguous()
        _lib.check(_lib.lib.basq_session_apply_cells(self.handle, int(R_glob), int(off_glob), int(F),
                                                     factor.data_ptr(), C.byref(c)))
        return int(c.value)

    def result(self):
        idx = torch.empty(self.n, dtype=torch.int64, device=self.device)
        w = torch.empty(self.n, dtype=torch.float64, device=self.device)
        k = C.c_int(0)
        _lib.check(_lib.lib.basq_session_result(self.handle, idx.data_ptr(), w.data_ptr(), self.n, C.byref(k)))
        return idx[: k.value], w[: k.value]


def standard_normals(rows, cols, seed=0, offset=0, device="cuda") -> torch.Tensor:
    """[rows, cols] fp64 N(0, 1) draws of the Philox stream `seed` (basq_standard_normals)."""
    device = torch.device(device)
    ctx = _lib.context_for(device)
    out = torch.empty(int(rows), int(cols), dtype=torch.float64, device=device)
    _lib.check(_lib.lib.basq_standard_normals(ctx.handle, int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset), int(rows),
                                              int(cols), out.data_ptr()))
    return out


def release_memory(device=None, keep_bytes: int = 0):
    """Hand the scratch memory cached by the library (block cache, host-call buffer) back to the driver (all
    contexts of `device`, or of every device)."""
    for (index, _stream), ctx in list(_lib._contexts.items()):
        if device is None or torch.device(device).index in (None, index):
            ctx.trim(keep_bytes)
