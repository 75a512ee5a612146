"""ctypes binding of ``libldeq.so`` -- the only door from Python into the CUDA product path.

There is NO CPU fallback: if the library is missing or no CUDA device is present, every entry
point raises.  Signatures mirror ``include/ldeq.h`` one to one.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LDEQ_LIB") or os.path.join(_HERE, "lib", "libldeq.so")  # LDEQ_LIB: tuning builds

# enums of include/ldeq.h
F32, F64 = 0, 1
RHS_PENDULUM, RHS_PENDULUM_FRICTION = 0, 1
RET_SUCCESS, RET_MAXITERS, RET_DTLESSTHANMIN, RET_UNSTABLE = 0, 1, 2, 3
NORM_GLOBAL, NORM_PER_TRAJ = 0, 1
MLP_MATH_FP32, MLP_MATH_BF16X3 = 0, 1
OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM, ERR_COMPILE, ERR_TAPE_OVERFLOW = 0, -1, -2, -3, -4, -5, -6
SOLVER_TSIT5, SOLVER_DP5, SOLVER_BS3, SOLVER_RK4 = 0, 1, 2, 3

# every symbol include/ldeq.h declares (tests check the library exports exactly these)
SYMBOLS = [
    "ldeq_version", "ldeq_opts_default", "ldeq_opts_default_solver", "ldeq_create", "ldeq_destroy", "ldeq_last_error", "ldeq_launch_count",
    "ldeq_rhs_builtin", "ldeq_rhs_from_source", "ldeq_rhs_dims", "ldeq_rhs_free",
    "ldeq_solve_fwd", "ldeq_solve_bwd", "ldeq_tape_overflow", "ldeq_tape_free",
    "ldeq_solve_fwd_host", "ldeq_solve_bwd_host", "ldeq_solve_fwd_bwd_host", "ldeq_debug_trig",
    "ldeq_mlp_solve_fwd", "ldeq_mlp_solve_bwd", "ldeq_mlp_tape_free", "ldeq_mlp_bwd_stats", "ldeq_debug_cadj_trace",
    "ldeq_pattern_extractor_param_count", "ldeq_pattern_extractor_fwd", "ldeq_pattern_extractor_bwd", "ldeq_pe_tape_free",
    "ldeq_sample", "ldeq_elbo_fwd_bwd", "ldeq_elbo_logits_fwd_bwd", "ldeq_adamw_step", "ldeq_allreduce_adamw_step",
    "ldeq_sample_dev", "ldeq_elbo_fwd_bwd_dev", "ldeq_elbo_logits_fwd_bwd_dev", "ldeq_adamw_step_dev",
    "ldeq_comm_unique_id", "ldeq_comm_init", "ldeq_allreduce_grads", "ldeq_comm_destroy",
]
COMM_ID_BYTES = 128
SENSE_DISCRETE_ADJOINT, SENSE_FORWARD_DUAL, SENSE_INTERPOLATING_ADJOINT = 0, 1, 2


class Opts(C.Structure):
    """``ldeq_opts``: the ``solve`` keyword arguments a diffeq struct forwards through ``kwargs``
    (reference ``src/models/GOKU.jl:108,121``)."""
    _fields_ = [
        ("abstol", C.c_double), ("reltol", C.c_double), ("adaptive", C.c_int32), ("controller_pow", C.c_int32),
        ("dt", C.c_double), ("dtmax", C.c_double), ("dtmin", C.c_double), ("maxiters", C.c_int64),
        ("gamma", C.c_double), ("qmin", C.c_double), ("qmax", C.c_double), ("beta1", C.c_double),
        ("beta2", C.c_double), ("qoldinit", C.c_double), ("qsteady_min", C.c_double), ("qsteady_max", C.c_double),
        ("tape_steps", C.c_int32), ("norm_mode", C.c_int32), ("mlp_math", C.c_int32), ("sensealg", C.c_int32),
        ("solver", C.c_int32), ("reserved_", C.c_int32),
    ]


class LdeqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libldeq error {code}: {msg}")
        self.code = code


_lib = None


def load() -> C.CDLL:
    """Load ``libldeq.so`` (built in-tree by ``build.py``).  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python latentdiffeq.jl_b200/build.py` "
            "(there is no CPU fallback for the hot path)")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl, flt = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_float
    pvp = C.POINTER(C.c_void_p)
    lib.ldeq_version.restype = i32
    lib.ldeq_opts_default.argtypes = [C.POINTER(Opts)]
    lib.ldeq_opts_default.restype = None
    lib.ldeq_opts_default_solver.argtypes = [C.POINTER(Opts), i32]
    lib.ldeq_create.argtypes = [pvp, i32]
    lib.ldeq_destroy.argtypes = [vp]
    lib.ldeq_destroy.restype = None
    lib.ldeq_last_error.argtypes = [vp]
    lib.ldeq_last_error.restype = C.c_char_p
    lib.ldeq_launch_count.argtypes = [vp]
    lib.ldeq_launch_count.restype = i64
    lib.ldeq_rhs_builtin.argtypes = [vp, i32, pvp]
    lib.ldeq_rhs_from_source.argtypes = [vp, C.c_char_p, i32, i32, pvp]
    lib.ldeq_rhs_dims.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    lib.ldeq_rhs_free.argtypes = [vp, vp]
    lib.ldeq_rhs_free.restype = None
    lib.ldeq_solve_fwd.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, C.POINTER(Opts), vp, vp, vp, vp, pvp, vp]
    lib.ldeq_solve_bwd.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.ldeq_tape_overflow.argtypes = [vp, vp, C.POINTER(C.c_int32), vp]
    lib.ldeq_tape_free.argtypes = [vp, vp, vp]
    lib.ldeq_tape_free.restype = None
    lib.ldeq_solve_fwd_host.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, C.POINTER(Opts), vp, vp, vp, vp, pvp, vp]
    lib.ldeq_solve_bwd_host.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.ldeq_solve_fwd_bwd_host.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, C.POINTER(Opts), vp, vp, vp, vp, vp, vp, vp, vp]
    lib.ldeq_debug_trig.argtypes = [vp, i32, vp, vp, vp, i64, vp]
    lib.ldeq_mlp_solve_fwd.argtypes = [vp, i32, vp, vp, vp, i32, vp, i32, i32, C.POINTER(Opts), vp, vp, vp, vp, pvp, vp]
    lib.ldeq_mlp_solve_bwd.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.ldeq_mlp_bwd_stats.argtypes = [vp, vp, vp, vp]
    lib.ldeq_debug_cadj_trace.argtypes = [vp, vp, vp, C.c_int]
    lib.ldeq_mlp_tape_free.argtypes = [vp, vp, vp]
    lib.ldeq_mlp_tape_free.restype = None
    lib.ldeq_pattern_extractor_param_count.argtypes = [i32, i32, i32]
    lib.ldeq_pattern_extractor_fwd.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, pvp, vp]
    lib.ldeq_pattern_extractor_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.ldeq_pe_tape_free.argtypes = [vp, vp, vp]
    lib.ldeq_pe_tape_free.restype = None
    lib.ldeq_sample.argtypes = [vp, vp, vp, vp, vp, i64, C.c_uint64, C.c_uint64, vp]
    lib.ldeq_elbo_fwd_bwd.argtypes = [vp, vp, vp, vp, vp, vp, i32, flt, i32, i32, i32, flt, vp, vp, vp, vp, vp]
    lib.ldeq_elbo_logits_fwd_bwd.argtypes = lib.ldeq_elbo_fwd_bwd.argtypes
    lib.ldeq_adamw_step.argtypes = [vp, vp, vp, vp, vp, i64, dbl, dbl, dbl, dbl, flt, i64, flt, vp]
    lib.ldeq_sample_dev.argtypes = [vp, vp, vp, vp, vp, i64, C.c_uint64, vp, vp]
    lib.ldeq_elbo_fwd_bwd_dev.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, i32, i32, i32, flt, vp, vp, vp, vp, vp]
    lib.ldeq_elbo_logits_fwd_bwd_dev.argtypes = lib.ldeq_elbo_fwd_bwd_dev.argtypes
    lib.ldeq_adamw_step_dev.argtypes = [vp, vp, vp, vp, vp, i64, dbl, dbl, dbl, dbl, flt, vp, flt, vp]
    lib.ldeq_allreduce_adamw_step.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, i64, dbl, dbl, dbl, dbl, flt, i64, flt, vp]
    lib.ldeq_comm_unique_id.argtypes = [vp, vp]
    lib.ldeq_comm_init.argtypes = [vp, vp, i32, i32]
    lib.ldeq_allreduce_grads.argtypes = [vp, vp, i64, vp]
    lib.ldeq_comm_destroy.argtypes = [vp]
    _lib = lib
    return lib


def default_opts(**kw) -> Opts:
    """OrdinaryDiffEq's defaults for ``solver`` (Tsit5 unless given: the controller exponents depend on the algorithm),
    overridden by keyword (same names as ``solve`` kwargs)."""
    o = Opts()
    rc = load().ldeq_opts_default_solver(C.byref(o), int(kw.get("solver", SOLVER_TSIT5)))
    if rc != OK:
        raise LdeqError(rc, f"unknown solver code {kw.get('solver')!r}")
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown solver option {k!r}")
        setattr(o, k, int(v) if isinstance(v, bool) else v)
    return o


class Handle:
    """One ``ldeq_handle`` (one per GPU and host thread)."""

    def __init__(self, device: int = 0):
        self._lib = load()
        self._h = C.c_void_p()
        rc = self._lib.ldeq_create(C.byref(self._h), int(device))
        if rc != 0:
            raise LdeqError(rc, f"ldeq_create(device={device}) failed: no usable CUDA device "
                                "(the hot path has no CPU fallback)")
        self.device = int(device)
        self._rhs = {}

    @property
    def ptr(self):
        return self._h

    def check(self, rc: int):
        if rc != 0:
            raise LdeqError(rc, (self._lib.ldeq_last_error(self._h) or b"").decode())

    def launch_count(self) -> int:
        return int(self._lib.ldeq_launch_count(self._h))

    def rhs_builtin(self, kind: int) -> C.c_void_p:
        if kind not in self._rhs:
            r = C.c_void_p()
            self.check(self._lib.ldeq_rhs_builtin(self._h, int(kind), C.byref(r)))
            self._rhs[kind] = r
        return self._rhs[kind]

    def rhs_from_source(self, src: str, z_dim: int, p_dim: int) -> C.c_void_p:
        key = (src, z_dim, p_dim)
        if key not in self._rhs:
            r = C.c_void_p()
            self.check(self._lib.ldeq_rhs_from_source(self._h, src.encode(), int(z_dim), int(p_dim), C.byref(r)))
            self._rhs[key] = r
        return self._rhs[key]

    # ---- NCCL route of the gradient all-reduce (ldeq_comm.cu) ----
    def comm_unique_id(self) -> bytes:
        """Rank 0: a fresh 128-byte NCCL id; distribute it to the other ranks (file, socket, MPI ...)."""
        buf = C.create_string_buffer(COMM_ID_BYTES)
        self.check(self._lib.ldeq_comm_unique_id(self._h, buf))
        return buf.raw

    def comm_init(self, unique_id: bytes, rank: int, nranks: int):
        if len(unique_id) != COMM_ID_BYTES:
            raise ValueError("unique_id must be the 128 bytes of comm_unique_id()")
        self.check(self._lib.ldeq_comm_init(self._h, C.c_char_p(unique_id), int(rank), int(nranks)))

    def allreduce_grads(self, flat_grad, stream=None):
        """In-place sum of a flat Float32 CUDA tensor over the ranks of ``comm_init``."""
        import torch
        if flat_grad.dtype != torch.float32 or not flat_grad.is_cuda or not flat_grad.is_contiguous():
            raise TypeError("allreduce_grads: a contiguous Float32 CUDA tensor is required")
        st = stream if stream is not None else torch.cuda.current_stream(flat_grad.device).cuda_stream
        self.check(self._lib.ldeq_allreduce_grads(self._h, C.c_void_p(flat_grad.data_ptr()), flat_grad.numel(), C.c_void_p(st)))

    def comm_destroy(self):
        self.check(self._lib.ldeq_comm_destroy(self._h))

    def close(self):
        if self._h:
            for r in self._rhs.values():
                self._lib.ldeq_rhs_free(self._h, r)
            self._rhs.clear()
            self._lib.ldeq_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_handles: dict[int, Handle] = {}


def handle(device: int = 0) -> Handle:
    """Process-wide handle of a device (created on first use)."""
    if device not in _handles:
        _handles[device] = Handle(device)
    return _handles[device]
