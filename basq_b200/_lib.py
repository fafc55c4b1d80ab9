"""ctypes binding of libbasq_b200.so (the C ABI in include/basq_b200.h).

There is no CPU fallback: if the shared library is missing the import of this module fails, and
every compute entry point fails with BasqError when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BASQ_B200_LIB") or os.path.join(_HERE, "libbasq_b200.so")  # override: A/B builds

BASQ_MAX_DIM = 32
OK, ERR_INVALID, ERR_CUDA, ERR_NUMERIC, ERR_UNSUPPORTED = range(5)
RBF, MATERN15, MATERN25 = 0, 1, 2
PLAIN, PRED_COV, WSABI_L, WSABI_M, MMLT_G = 0, 1, 2, 3, 4
F32, F64 = 0, 1
PHASES = ("prepare", "set_sum", "projection", "caratheodory", "apply", "nystrom", "gp_predict", "other")


class BasqError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"basq_b200 error {code}: {msg}")
        self.code = code


class KernelDesc(C.Structure):
    _fields_ = [
        ("family", C.c_int32), ("mode", C.c_int32), ("dtype", C.c_int32), ("d", C.c_int32),
        ("outputscale", C.c_double),
        ("lengthscale", C.c_double * BASQ_MAX_DIM),
        ("noise", C.c_double), ("mean_const", C.c_double), ("diag_add", C.c_double),
        ("n_obs", C.c_int32), ("noise_diag", C.c_int32),
        ("Xobs", C.c_void_p), ("W", C.c_void_p), ("alpha", C.c_void_p), ("Xobs_f64", C.c_void_p),
    ]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA extension first (python buildlib.py). "
            "basq_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    P, I, L, D = C.c_void_p, C.c_int, C.c_int64, C.c_double
    KD = C.POINTER(KernelDesc)
    sig = {
        "basq_abi_version": (I, []),
        "basq_last_error": (C.c_char_p, []),
        "basq_ctx_create": (I, [I, P, C.POINTER(P)]),
        "basq_ctx_destroy": (None, [P]),
        "basq_ctx_trim": (I, [P, L]),
        "basq_ctx_conditioning": (I, [P, D, C.POINTER(D), C.POINTER(L)]),
        "basq_ctx_launch_count": (L, [P]),
        "basq_ctx_pair_evals": (L, [P]),
        "basq_ctx_profile": (I, [P, I]),
        "basq_ctx_profile_read": (I, [P, C.POINTER(D), C.POINTER(L), I]),
        "basq_gram": (I, [P, KD, P, L, P, L, P]),
        "basq_gp_predict": (I, [P, KD, P, L, I, D, P, P]),
        "basq_kernel_quadform": (I, [P, KD, P, L, P, C.POINTER(D)]),
        "basq_kernel_bilinear": (I, [P, KD, P, L, P, P, L, P, C.POINTER(D)]),
        "basq_ctx_stage_candidates": (I, [P, P, L, I, I, P]),
        "basq_session_create_staged": (I, [P, KD, L, L, L, P, L, P, I, C.POINTER(P)]),
        "basq_nystrom_basis_sharded": (I, [P, KD, P, L, I, P, I, I, I, P, P, P, P, P]),
        "basq_nystrom_basis": (I, [P, KD, P, L, I, P, I, P, P]),
        "basq_features": (I, [P, KD, P, L, P, L, P, I, P]),
        "basq_car": (I, [P, P, I, I, I, P, C.POINTER(I)]),
        "basq_recombine": (I, [P, KD, P, L, P, L, P, I, P, P, P, C.POINTER(I)]),
        "basq_recombine_objective": (I, [P, KD, P, L, P, L, P, I, P, P, P, P, C.POINTER(I)]),
        "basq_car_objective": (I, [P, P, I, I, I, P]),
        "basq_session_set_objective": (I, [P, P]),
        "basq_recombine_host": (I, [P, KD, P, L, P, L, P, I, P, I, P, P, P, C.POINTER(I)]),
        "basq_session_create": (I, [P, KD, P, L, L, L, P, L, P, I, P, C.POINTER(P)]),
        "basq_session_destroy": (None, [P]),
        "basq_session_count": (I, [P, C.POINTER(L)]),
        "basq_session_partial": (I, [P, L, L, P]),
        "basq_session_apply": (I, [P, L, L, P, C.POINTER(L)]),
        "basq_session_result": (I, [P, P, P, I, C.POINTER(I)]),
        "basq_session_cell_factor": (I, [P, L, L, C.POINTER(I)]),
        "basq_session_pass_begin": (I, [P, L, L, I]),
        "basq_session_level": (I, [P, I, I, P, P, P, P]),
        "basq_session_landmarks": (I, [P, C.POINTER(I)]),
        "basq_session_level_fold": (I, [P, I, I, P, P, L]),
        "basq_session_level_project": (I, [P, I, I, P, P, P, P, L, I, I, P]),
        "basq_session_apply_cells": (I, [P, L, L, I, P, C.POINTER(L)]),
        "basq_sample_mvn": (I, [P, C.c_uint64, L, L, I, I, P, P, P]),
        "basq_standard_normals": (I, [P, C.c_uint64, L, L, I, P]),
        "basq_ctx_set_seed": (I, [P, C.c_uint64]),
        "basq_ctx_memory": (I, [P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(L)]),
        "basq_ctx_allow_f32_eval": (I, [P, I, C.POINTER(L)]),
        "basq_mvn_logpdf": (I, [P, P, L, I, I, P, P, P]),
        "basq_candidate_weights": (I, [P, I, D, I, P, P, L, I, P]),
        "basq_cleanse_weights": (I, [P, P, L, D]),
        "basq_sir_resample": (I, [P, P, L, L, C.c_uint64, P, C.POINTER(L)]),
        "basq_dgemm": (I, [P, I, I, I, I, I, D, P, I, P, I, D, P, I]),
        "basq_tgemm": (I, [P, I, I, I, P, I, P, I, P, I]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib, tuple(sig)


lib, SYMBOLS = _load()


def check(code):
    if code != OK:
        raise BasqError(code, lib.basq_last_error().decode("utf-8", "replace"))


class Context:
    """One basq_ctx per (device, stream)."""

    def __init__(self, device_index: int, stream_ptr: int = 0):
        h = C.c_void_p()
        check(lib.basq_ctx_create(int(device_index), C.c_void_p(stream_ptr or None), C.byref(h)))
        self.handle = h
        self.device_index = device_index
        self.stream_ptr = stream_ptr

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h and lib is not None:          # lib is None while the interpreter shuts down
            lib.basq_ctx_destroy(h)

    @property
    def launches(self) -> int:
        return int(lib.basq_ctx_launch_count(self.handle))

    @property
    def pair_evals(self) -> int:
        return int(lib.basq_ctx_pair_evals(self.handle))

    def memory(self):
        """(bytes cached for reuse, bytes handed out to live sessions, driver allocations so far)."""
        c, l, n = C.c_uint64(0), C.c_uint64(0), C.c_int64(0)
        check(lib.basq_ctx_memory(self.handle, C.byref(c), C.byref(l), C.byref(n)))
        return int(c.value), int(l.value), int(n.value)

    def trim(self, keep_bytes: int = 0):
        """Hand the context's cached scratch memory back to the driver (down to keep_bytes)."""
        check(lib.basq_ctx_trim(self.handle, int(keep_bytes)))

    def allow_f32_eval(self, on=None) -> int:
        """fp64 inputs may be evaluated on the fp32 tensor-core path (basq_ctx_allow_f32_eval); returns the
        number of sessions demoted so far.  on=None only reads the counter."""
        n = C.c_int64(0)
        check(lib.basq_ctx_allow_f32_eval(self.handle, -1 if on is None else int(bool(on)), C.byref(n)))
        return int(n.value)

    def set_seed(self, seed: int):
        """Key of the library's own Gaussian draws (basq_ctx_set_seed)."""
        check(lib.basq_ctx_set_seed(self.handle, int(seed) & 0xFFFFFFFFFFFFFFFF))

    def conditioning(self, kappa_max: float = -1.0):
        """(last kappa = max_m |(K_ZX W)_m|_1, number of fp32 -> fp64 promotions so far); a non-negative
        kappa_max sets the promotion threshold (0 = never promote)."""
        k, n = C.c_double(0.0), C.c_int64(0)
        check(lib.basq_ctx_conditioning(self.handle, float(kappa_max), C.byref(k), C.byref(n)))
        return float(k.value), int(n.value)

    def profile(self, enable: bool):
        check(lib.basq_ctx_profile(self.handle, 1 if enable else 0))

    def profile_read(self, reset=True):
        ms = (C.c_double * 8)()
        calls = (C.c_int64 * 8)()
        check(lib.basq_ctx_profile_read(self.handle, ms, calls, 1 if reset else 0))
        return {PHASES[i]: (float(ms[i]), int(calls[i])) for i in range(8)}


_contexts = {}


def context_for(device) -> Context:
    """Context bound to torch's current stream on `device` (a torch.device with type cuda)."""
    import torch

    if not torch.cuda.is_available():
        raise BasqError(ERR_CUDA, "no CUDA device available; basq_b200 has no CPU fallback")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise BasqError(ERR_CUDA, f"device {dev} is not a CUDA device; basq_b200 has no CPU fallback")
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    stream = torch.cuda.current_stream(index).cuda_stream
    key = (index, stream)
    ctx = _contexts.get(key)
    if ctx is None:
        ctx = _contexts[key] = Context(index, stream)
    return ctx
