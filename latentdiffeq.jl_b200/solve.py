"""Torch-facing wrappers of the C-ABI solve entry points.

Tensors are contiguous torch tensors whose bytes equal the reference's column-major Julia arrays:
``z0`` is ``[B, z]`` (Julia ``(z,B)``), ``theta`` is ``[B, p]``, trajectories are ``[T, B, z]``
(Julia ``(z,B,T)``, what ``permutedims(z, [1,3,2])`` yields at reference ``src/models/GOKU.jl:125``).

PyTorch is plumbing here (device memory, streams, autograd glue); all arithmetic runs in
``libldeq.so``.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np
import torch

from . import _cabi


def _dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return _cabi.F32
    if dt == torch.float64:
        return _cabi.F64
    raise TypeError(f"state dtype must be float32 or float64, got {dt}")


def _tgrid(t) -> np.ndarray:
    """The save grid as host Float64 (the reference's ``t`` is a Float64 range; SURVEY.md 7.2)."""
    if isinstance(t, torch.Tensor):
        t = t.detach().cpu().numpy()
    t = np.ascontiguousarray(np.asarray(t, dtype=np.float64))
    if t.ndim != 1 or t.size < 1:
        raise ValueError("t must be a non-empty 1-D grid")
    return t


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _aligned16(x: torch.Tensor) -> torch.Tensor:
    """A contiguous view may start anywhere inside its storage (``time_loader`` slices); the vectorised kernels want
    16-byte aligned bases."""
    return x if x.data_ptr() % 16 == 0 else x.clone(memory_format=torch.contiguous_format)


def _p(x: torch.Tensor | None) -> C.c_void_p:
    return C.c_void_p(0 if x is None else x.data_ptr())


class _Tape:
    """Owns an ``ldeq_tape`` (or ``ldeq_mlp_tape``); frees it stream-ordered when dropped."""

    def __init__(self, h: _cabi.Handle, ptr: C.c_void_p, mlp: bool = False):
        self.h, self.ptr, self.mlp = h, ptr, mlp

    def overflow(self) -> int:
        if self.mlp:
            raise TypeError("overflow() is a GOKU-tape query; an MLP tape reports overflow from mlp_bwd_raw (LdeqError -6)")
        if not self.ptr:
            raise RuntimeError("tape already freed")
        n = C.c_int32(0)
        self.h.check(self.h._lib.ldeq_tape_overflow(self.h.ptr, self.ptr, C.byref(n), _stream()))
        return int(n.value)

    def free(self):
        if self.ptr:
            try:
                with torch.cuda.device(self.h.device):
                    if self.mlp:
                        self.h._lib.ldeq_mlp_tape_free(self.h.ptr, self.ptr, _stream())
                    else:
                        self.h._lib.ldeq_tape_free(self.h.ptr, self.ptr, _stream())
            finally:
                self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class SolveStats:
    """Per-trajectory ``retcode`` / ``naccept`` / ``nreject`` (device int32 tensors)."""

    def __init__(self, retcode, naccept, nreject):
        self.retcode, self.naccept, self.nreject = retcode, naccept, nreject


def goku_solve_raw(z0: torch.Tensor, theta: torch.Tensor, t, rhs, opts: _cabi.Opts | None = None,
                   want_tape: bool = False, want_stats: bool = True):
    """One call of ``ldeq_solve_fwd``: B independent Tsit5 solves (reference GOKU.jl:111-125).

    ``rhs`` is a built-in kind (``_cabi.RHS_PENDULUM`` ...) or an ``ldeq_rhs`` pointer from
    ``Handle.rhs_from_source``.  Returns ``(traj[T,B,z], stats, tape_or_None)``.
    """
    if not z0.is_cuda:
        raise RuntimeError("goku_solve_raw needs CUDA tensors; use goku_solve_host for host buffers "
                           "(there is no CPU implementation of the hot path)")
    h = _cabi.handle(z0.device.index or 0)
    opts = opts or _cabi.default_opts()
    z0 = z0.contiguous()
    theta = theta.to(z0.dtype).contiguous()
    tg = _tgrid(t)
    B, Z = z0.shape
    T = tg.shape[0]
    rhs_ptr = h.rhs_builtin(rhs) if isinstance(rhs, int) else rhs
    traj = torch.empty((T, B, Z), dtype=z0.dtype, device=z0.device)
    ret = na = nr = None
    if want_stats:
        ret = torch.empty(B, dtype=torch.int32, device=z0.device)
        na = torch.empty(B, dtype=torch.int32, device=z0.device)
        nr = torch.empty(B, dtype=torch.int32, device=z0.device)
    tape = C.c_void_p()
    with torch.cuda.device(z0.device):
        h.check(h._lib.ldeq_solve_fwd(h.ptr, rhs_ptr, _dtype_code(z0.dtype), _p(z0), _p(theta),
                                      tg.ctypes.data_as(C.c_void_p), B, T, C.byref(opts), _p(traj), _p(ret), _p(na),
                                      _p(nr), C.byref(tape) if want_tape else None, _stream()))
    tp = None
    if want_tape:
        tp = _Tape(h, tape)
        tp.p_dim = theta.shape[1]
    return traj, SolveStats(ret, na, nr), tp


def goku_bwd_raw(tape: _Tape, dtraj: torch.Tensor):
    """One call of ``ldeq_solve_bwd``: the pullback by the tape's sensealg (dual re-solves or discrete adjoint)."""
    h = tape.h
    if not tape.ptr:
        raise RuntimeError("the tape of this solve was already consumed and freed (backward twice? the tape is released "
                           "after the first pullback; re-run the forward solve)")
    dtraj = dtraj.contiguous()
    T, B, Z = dtraj.shape
    dz0 = torch.empty((B, Z), dtype=dtraj.dtype, device=dtraj.device)
    # p_dim is a property of the rhs; ask the tape's rhs through the handle-independent call
    dth = torch.empty((B, tape.p_dim), dtype=dtraj.dtype, device=dtraj.device)
    with torch.cuda.device(dtraj.device):
        h.check(h._lib.ldeq_solve_bwd(h.ptr, tape.ptr, _p(dtraj), _p(dz0), _p(dth), _stream()))
    return dz0, dth


class _GokuSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z0, theta, tg, rhs, opts, stats_out):
        need = z0.requires_grad or theta.requires_grad
        traj, stats, tape = goku_solve_raw(z0, theta, tg, rhs, opts, want_tape=need, want_stats=True)
        if tape is not None:
            tape.p_dim = theta.shape[1]
        ctx.tape = tape
        if stats_out is not None:
            stats_out.append(stats)
        return traj

    @staticmethod
    def backward(ctx, dtraj):
        tape = ctx.tape
        if tape is None:
            if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                raise RuntimeError("goku_solve: backward called twice; the tape is released after the first pullback")
            return None, None, None, None, None, None
        dz0, dth = goku_bwd_raw(tape, dtraj)
        tape.free()
        ctx.tape = None
        return dz0, dth, None, None, None, None


def goku_solve(z0: torch.Tensor, theta: torch.Tensor, t, rhs=_cabi.RHS_PENDULUM, opts: _cabi.Opts | None = None,
               stats_out: list | None = None) -> torch.Tensor:
    """Differentiable batched solve: the body of ``diffeq_layer(::Decoder{<:GOKU}, (z0, theta), t)``
    (reference ``src/models/GOKU.jl:98-130``).  Gradients flow to ``z0`` and ``theta`` by ``opts.sensealg``: the
    reference's dual-number re-solves (default) or the discrete adjoint of the accepted steps."""
    return _GokuSolve.apply(z0, theta, _tgrid(t), rhs, opts, stats_out)


# ---- host-buffer entry points (what a CPU-resident Flux model passes, GOKU.jl:102-103,128) --------
def goku_solve_host(z0: torch.Tensor, theta: torch.Tensor, t, rhs=_cabi.RHS_PENDULUM,
                    opts: _cabi.Opts | None = None, device: int = 0, want_tape: bool = False,
                    out: torch.Tensor | None = None, handle: _cabi.Handle | None = None):
    """``ldeq_solve_fwd_host``: host tensors in, host tensor out; copies are inside the call (which returns when the
    result is on the host).  ``handle``: a private ``Handle`` for a second host thread (one handle per host thread)."""
    assert not z0.is_cuda and not theta.is_cuda
    h = handle or _cabi.handle(device)
    device = h.device
    opts = opts or _cabi.default_opts()
    z0 = z0.contiguous()
    theta = theta.to(z0.dtype).contiguous()
    tg = _tgrid(t)
    B, Z = z0.shape
    T = tg.shape[0]
    rhs_ptr = h.rhs_builtin(rhs) if isinstance(rhs, int) else rhs
    if out is None:
        out = torch.empty((T, B, Z), dtype=z0.dtype, pin_memory=True)
    tape = C.c_void_p()
    with torch.cuda.device(device):
        h.check(h._lib.ldeq_solve_fwd_host(h.ptr, rhs_ptr, _dtype_code(z0.dtype), _p(z0), _p(theta),
                                           tg.ctypes.data_as(C.c_void_p), B, T, C.byref(opts), _p(out), None, None,
                                           None, C.byref(tape) if want_tape else None, _stream()))
    tp = None
    if want_tape:
        tp = _Tape(h, tape)
        tp.p_dim = theta.shape[1]
    return out, tp


def goku_bwd_host(tape: _Tape, dtraj: torch.Tensor, dz0: torch.Tensor | None = None,
                  dtheta: torch.Tensor | None = None):
    """``ldeq_solve_bwd_host``: host cotangent in, host gradients out."""
    assert not dtraj.is_cuda
    h = tape.h
    dtraj = dtraj.contiguous()
    T, B, Z = dtraj.shape
    if dz0 is None:
        dz0 = torch.empty((B, Z), dtype=dtraj.dtype, pin_memory=True)
    if dtheta is None:
        dtheta = torch.empty((B, tape.p_dim), dtype=dtraj.dtype, pin_memory=True)
    with torch.cuda.device(h.device):
        h.check(h._lib.ldeq_solve_bwd_host(h.ptr, tape.ptr, _p(dtraj), _p(dz0), _p(dtheta), _stream()))
    return dz0, dtheta


def goku_fwd_bwd_host(z0: torch.Tensor, theta: torch.Tensor, t, dtraj: torch.Tensor, rhs=_cabi.RHS_PENDULUM,
                      opts: _cabi.Opts | None = None, device: int = 0, out: torch.Tensor | None = None,
                      dz0: torch.Tensor | None = None, dtheta: torch.Tensor | None = None, handle: _cabi.Handle | None = None):
    """``ldeq_solve_fwd_bwd_host``: forward solve and pullback of a known cotangent, host tensors in and out, one call;
    the cotangent slabs go up while the trajectory slabs come down."""
    assert not z0.is_cuda and not theta.is_cuda and not dtraj.is_cuda
    h = handle or _cabi.handle(device)
    opts = opts or _cabi.default_opts()
    z0 = z0.contiguous()
    theta = theta.to(z0.dtype).contiguous()
    dtraj = dtraj.to(z0.dtype).contiguous()
    tg = _tgrid(t)
    B, Z = z0.shape
    T = tg.shape[0]
    assert tuple(dtraj.shape) == (T, B, Z)
    rhs_ptr = h.rhs_builtin(rhs) if isinstance(rhs, int) else rhs
    if out is None:
        out = torch.empty((T, B, Z), dtype=z0.dtype, pin_memory=True)
    if dz0 is None:
        dz0 = torch.empty((B, Z), dtype=z0.dtype, pin_memory=True)
    if dtheta is None:
        dtheta = torch.empty((B, theta.shape[1]), dtype=z0.dtype, pin_memory=True)
    with torch.cuda.device(h.device):
        h.check(h._lib.ldeq_solve_fwd_bwd_host(h.ptr, rhs_ptr, _dtype_code(z0.dtype), _p(z0), _p(theta),
                                               tg.ctypes.data_as(C.c_void_p), B, T, C.byref(opts), _p(dtraj), _p(out), _p(dz0),
                                               _p(dtheta), None, None, None, _stream()))
    return out, dz0, dtheta


def debug_trig(x: torch.Tensor, which: int = 0):
    """``ldeq_debug_trig``: the kernels' Float32 sine / cosine on a CUDA tensor (0 fast pair, 1 Julia's, 2 fast sine)."""
    h = _cabi.handle(x.device.index or 0)
    x = x.contiguous().float()
    s, c = torch.empty_like(x), torch.empty_like(x)
    with torch.cuda.device(x.device):
        h.check(h._lib.ldeq_debug_trig(h.ptr, int(which), _p(x), _p(s), _p(c), x.numel(), _stream()))
    return s, c


# ---- LatentODE path: one solve on the (D,B) matrix state with an MLP right-hand side ---------------
def mlp_solve_raw(z0: torch.Tensor, params_flat: torch.Tensor, dims: Sequence[int], t, opts: _cabi.Opts | None = None,
                  want_tape: bool = False):
    """One call of ``ldeq_mlp_solve_fwd`` (reference ``src/models/LatentODE.jl:61-78``).

    ``z0`` is ``[B, D]``; ``params_flat`` is ``Flux.destructure`` order; ``dims = [D, H1, ..., D]``.
    Returns ``(traj[T,B,D], stats, tape_or_None)``."""
    if not z0.is_cuda:
        raise RuntimeError("mlp_solve_raw needs CUDA tensors (there is no CPU implementation of the hot path)")
    h = _cabi.handle(z0.device.index or 0)
    opts = opts or _cabi.default_opts()
    z0 = z0.contiguous()
    params_flat = params_flat.to(z0.dtype).contiguous()
    tg = _tgrid(t)
    B, D = z0.shape
    T = tg.shape[0]
    dims_a = np.ascontiguousarray(np.asarray(dims, dtype=np.int32))
    assert dims_a[0] == D and dims_a[-1] == D
    traj = torch.empty((T, B, D), dtype=z0.dtype, device=z0.device)
    ret = torch.empty(B, dtype=torch.int32, device=z0.device)
    na = torch.empty(B, dtype=torch.int32, device=z0.device)
    nr = torch.empty(B, dtype=torch.int32, device=z0.device)
    tape = C.c_void_p()
    with torch.cuda.device(z0.device):
        h.check(h._lib.ldeq_mlp_solve_fwd(h.ptr, _dtype_code(z0.dtype), _p(z0), _p(params_flat),
                                          dims_a.ctypes.data_as(C.c_void_p), len(dims_a) - 1,
                                          tg.ctypes.data_as(C.c_void_p), B, T, C.byref(opts), _p(traj), _p(ret), _p(na),
                                          _p(nr), C.byref(tape) if want_tape else None, _stream()))
    tp = None
    if want_tape:
        tp = _Tape(h, tape, mlp=True)
        tp.n_params = int(params_flat.numel())
    return traj, SolveStats(ret, na, nr), tp


def mlp_bwd_raw(tape: _Tape, dtraj: torch.Tensor):
    """One call of ``ldeq_mlp_solve_bwd``: ``dtraj[T,B,D] -> (dz0[B,D], dparams_flat)``."""
    h = tape.h
    dtraj = dtraj.contiguous()
    T, B, D = dtraj.shape
    dz0 = torch.empty((B, D), dtype=dtraj.dtype, device=dtraj.device)
    dp = torch.empty(tape.n_params, dtype=dtraj.dtype, device=dtraj.device)
    with torch.cuda.device(dtraj.device):
        h.check(h._lib.ldeq_mlp_solve_bwd(h.ptr, tape.ptr, _p(dtraj), _p(dz0), _p(dp), _stream()))
    return dz0, dp


def mlp_bwd_stats(tape: _Tape):
    """``(naccept, nreject, retcode)`` of the backward solve ``LDEQ_SENSE_INTERPOLATING_ADJOINT`` ran for this tape."""
    import ctypes
    out = (ctypes.c_int32 * 3)()
    h = tape.h
    h.check(h._lib.ldeq_mlp_bwd_stats(h.ptr, tape.ptr, out, _stream()))
    return int(out[0]), int(out[1]), int(out[2])


class _MlpSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z0, params_flat, tg, dims, opts, stats_out):
        need = z0.requires_grad or params_flat.requires_grad
        traj, stats, tape = mlp_solve_raw(z0, params_flat, dims, tg, opts, want_tape=need)
        ctx.tape = tape
        if stats_out is not None:
            stats_out.append(stats)
        return traj

    @staticmethod
    def backward(ctx, dtraj):
        tape = ctx.tape
        if tape is None:
            if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                raise RuntimeError("mlp_solve: backward called twice; the tape is released after the first pullback")
            return None, None, None, None, None, None
        dz0, dp = mlp_bwd_raw(tape, dtraj)
        tape.free()
        ctx.tape = None
        return dz0, dp, None, None, None, None


def mlp_solve(z0, params_flat, dims, t, opts: _cabi.Opts | None = None, stats_out: list | None = None):
    """Differentiable LatentODE solve: the body of ``diffeq_layer(::Decoder{LatentODE}, z0, t)``."""
    return _MlpSolve.apply(z0, params_flat, _tgrid(t), list(dims), opts, stats_out)


# ---- recurrent pattern extractor (SURVEY.md 8(f)2) ----------------------------------------------------------------
PE_HIDDEN = 16            # GOKU's stacks (GOKU.jl:201): relu-RNN + two LSTM stacks
PE_HIDDEN_RNN_ONLY = 32   # LatentODE's relu-RNN stack (LatentODE.jl:102)
PE_INPUTS = (16, 32, 64)


def pe_flat_params(layers, lstm: bool) -> torch.Tensor:
    """One stack's parameters as the flat vector ``ldeq_pattern_extractor_*`` read -- ``Flux.destructure`` order: per layer
    ``Wi`` (rows x in, column-major = the row-major ``[in, rows]`` of ``W.t()``), ``Wh``, ``b``, ``state0`` (LSTM: ``h0``,
    ``c0``).  Built with differentiable torch ops, so autograd routes the flat gradient back to the layers' own tensors."""
    parts = []
    for l in layers:
        parts += [l.Wi.t().reshape(-1), l.Wh.t().reshape(-1), l.b]
        parts += [l.h0, l.c0] if lstm else [l.state0]
    return torch.cat(parts).float()


class _PeTape:
    """Owns an ``ldeq_pe_tape``; frees it stream-ordered when dropped."""

    def __init__(self, h: _cabi.Handle, ptr: C.c_void_p):
        self.h, self.ptr = h, ptr

    def free(self):
        if self.ptr:
            try:
                with torch.cuda.device(self.h.device):
                    self.h._lib.ldeq_pe_tape_free(self.h.ptr, self.ptr, _stream())
            finally:
                self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _PatternExtractor(torch.autograd.Function):
    """``apply_pattern_extractor`` (GOKU.jl:30-49 / LatentODE.jl:20-34) through the persistent recurrent kernels."""

    @staticmethod
    def forward(ctx, x, rnn, lstm_f, lstm_b):
        h = _cabi.handle(x.device.index or 0)
        T, B, F = x.shape
        x = _aligned16(x.contiguous().float())
        rnn = rnn.contiguous()
        has_lstm = lstm_f is not None
        lstm_f = lstm_f.contiguous() if has_lstm else None
        lstm_b = lstm_b.contiguous() if has_lstm else None
        lib = h._lib
        H = next((hh for hh in ((PE_HIDDEN,) if has_lstm else (PE_HIDDEN, PE_HIDDEN_RNN_ONLY))
                  if rnn.numel() == lib.ldeq_pattern_extractor_param_count(0, F, hh)), None)
        if H is None or (has_lstm and lstm_f.numel() != lib.ldeq_pattern_extractor_param_count(1, F, H)):
            raise _cabi.LdeqError(_cabi.ERR_UNSUPPORTED, "pattern extractor: the parameter vectors match no built size (H = 16, or H = 32 for the RNN stack alone)")
        z0 = torch.empty(B, H, device=x.device, dtype=torch.float32)
        th = torch.empty(B, 2 * H, device=x.device, dtype=torch.float32) if has_lstm else None
        need = any(ctx.needs_input_grad)
        tape = C.c_void_p()
        with torch.cuda.device(x.device):
            h.check(lib.ldeq_pattern_extractor_fwd(h.ptr, _p(x), B, T, F, H, _p(rnn), _p(lstm_f), _p(lstm_b), _p(z0), _p(th),
                                                   C.byref(tape) if need else None, _stream()))
        ctx.h, ctx.tape, ctx.has_lstm = h, (tape if need else None), has_lstm
        ctx.save_for_backward(x, rnn, *( [lstm_f, lstm_b] if has_lstm else []))
        if need:
            ctx.freer = _PeTape(h, tape)
        return (z0, th) if has_lstm else (z0, torch.empty(0, device=x.device))

    @staticmethod
    def backward(ctx, dz0, dth):
        if ctx.tape is None:
            raise RuntimeError("the tape of this pattern-extractor call was already consumed and freed (backward twice?)")
        saved = ctx.saved_tensors
        x, rnn = saved[0], saved[1]
        lf, lb = (saved[2], saved[3]) if ctx.has_lstm else (None, None)
        h = ctx.h
        dz0 = dz0.contiguous().float()
        dth = dth.contiguous().float() if ctx.has_lstm else None
        dx = torch.empty_like(x)
        drnn = torch.empty_like(rnn)
        dlf = torch.empty_like(lf) if ctx.has_lstm else None
        dlb = torch.empty_like(lb) if ctx.has_lstm else None
        with torch.cuda.device(x.device):
            h.check(h._lib.ldeq_pattern_extractor_bwd(h.ptr, ctx.tape, _p(x), _p(rnn), _p(lf), _p(lb), _p(dz0), _p(dth), _p(dx), _p(drnn),
                                                      _p(dlf), _p(dlb), _stream()))
        ctx.freer.free()
        ctx.tape = None
        return dx, drnn, dlf, dlb


def pattern_extractor(x: torch.Tensor, rnn_layers, lstm_f_layers=None, lstm_b_layers=None):
    """Final hidden states of the pattern extractor's recurrent stacks over the frame sequence ``x [T, B, F]``:
    ``(z0_out [B, 16], theta_out [B, 32])`` for GOKU, ``z0_out`` alone for LatentODE (no LSTM stacks).  Differentiable."""
    if not x.is_cuda:
        raise RuntimeError("pattern_extractor needs CUDA tensors (no CPU fallback)")
    rnn = pe_flat_params(rnn_layers, False)
    if lstm_f_layers is None:
        return _PatternExtractor.apply(x, rnn, None, None)[0]
    return _PatternExtractor.apply(x, rnn, pe_flat_params(lstm_f_layers, True), pe_flat_params(lstm_b_layers, True))


# ---- reparameterised sample, ELBO, AdamW ------------------------------------------------------------
def sample_raw(mu: torch.Tensor, logvar: torch.Tensor, seed: int, offset: int = 0, want_eps: bool = True,
               calls: torch.Tensor | None = None):
    """``ldeq_sample``: ``z = mu + eps * exp(logvar/2)``, ``eps ~ N(0,1)`` drawn on the device (Philox4x32-10).
    ``calls`` (a one-element int64 CUDA tensor): ``ldeq_sample_dev`` instead, which increments the counter on the device and
    draws at offset ``calls << 32`` (``offset`` is ignored) -- what a CUDA graph replays with new noise every time."""
    h = _cabi.handle(mu.device.index or 0)
    mu = mu.contiguous().float()
    logvar = logvar.contiguous().float()
    z = torch.empty_like(mu)
    eps = torch.empty_like(mu) if want_eps else None
    with torch.cuda.device(mu.device):
        if calls is not None:
            h.check(h._lib.ldeq_sample_dev(h.ptr, _p(mu), _p(logvar), _p(z), _p(eps), mu.numel(), C.c_uint64(seed & (2**64 - 1)),
                                           _p(calls), _stream()))
        else:
            h.check(h._lib.ldeq_sample(h.ptr, _p(mu), _p(logvar), _p(z), _p(eps), mu.numel(), C.c_uint64(seed & (2**64 - 1)),
                                       C.c_uint64(offset & (2**64 - 1)), _stream()))
    return z, eps


class _Sample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, logvar, seed, offset, calls):
        z, eps = sample_raw(mu, logvar, seed, offset, calls=calls)
        ctx.save_for_backward(eps, logvar)
        return z

    @staticmethod
    def backward(ctx, dz):
        eps, logvar = ctx.saved_tensors
        return dz, dz * eps * torch.exp(logvar * 0.5) * 0.5, None, None, None


def sample_reparam(mu, logvar, seed: int, offset: int = 0, calls: torch.Tensor | None = None):
    """Differentiable reparameterised sample (reference ``src/models/GOKU.jl:155-173``); ``calls``: see ``sample_raw``."""
    return _Sample.apply(mu, logvar, int(seed), int(offset), calls)


def elbo_raw(x: torch.Tensor, xhat: torch.Tensor, mus, logvars, beta, want_grad: bool = True,
             grad_scale: float = 1.0, logits: bool = False):
    """``ldeq_elbo_fwd_bwd``: ``x, xhat`` are ``[T, B, P]``; ``mus/logvars`` lists of ``[B, d_h]`` heads.
    Returns ``(loss3 = [total, reconstruction, kl], dxhat, dmus, dlogvars)``.  ``logits=True``
    (``ldeq_elbo_logits_fwd_bwd``): ``xhat`` holds the pre-activations of a sigmoid output layer; the gradient returned in
    ``dxhat``'s place is with respect to them.  ``beta`` is a Python float, or a 0-d Float32 CUDA tensor that the kernels
    read on the device (the ``_dev`` entry points: a CUDA graph replays it with its current value)."""
    h = _cabi.handle(x.device.index or 0)
    x = _aligned16(x.contiguous().float())
    xhat = _aligned16(xhat.contiguous().float())
    T, B, P = x.shape
    mus = [m.contiguous().float() for m in mus]
    logvars = [l.contiguous().float() for l in logvars]
    nh = len(mus)
    loss = torch.empty(3, dtype=torch.float32, device=x.device)
    dxhat = torch.empty_like(xhat) if want_grad else None
    dmus = [torch.empty_like(m) for m in mus] if want_grad else None
    dlvs = [torch.empty_like(l) for l in logvars] if want_grad else None
    PA = C.c_void_p * max(nh, 1)
    mu_a = PA(*[m.data_ptr() for m in mus])
    lv_a = PA(*[l.data_ptr() for l in logvars])
    dmu_a = PA(*[m.data_ptr() for m in dmus]) if want_grad else None
    dlv_a = PA(*[l.data_ptr() for l in dlvs]) if want_grad else None
    hd = (C.c_int32 * max(nh, 1))(*[m.shape[1] for m in mus])
    with torch.cuda.device(x.device):
        if isinstance(beta, torch.Tensor):
            if not (beta.is_cuda and beta.dtype == torch.float32 and beta.numel() == 1):
                raise TypeError("elbo: a tensor beta must be one Float32 element on the CUDA device")
            fn = h._lib.ldeq_elbo_logits_fwd_bwd_dev if logits else h._lib.ldeq_elbo_fwd_bwd_dev
            beta_arg = _p(beta)
        else:
            fn = h._lib.ldeq_elbo_logits_fwd_bwd if logits else h._lib.ldeq_elbo_fwd_bwd
            beta_arg = C.c_float(beta)
        h.check(fn(h.ptr, _p(x), _p(xhat), mu_a, lv_a, hd, nh, beta_arg, B, T, P,
                   C.c_float(grad_scale), _p(loss), _p(dxhat), dmu_a, dlv_a, _stream()))
    return loss, dxhat, dmus, dlvs


class _Elbo(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, xhat, beta, nh, logits, unit_cotangent, grad_scale, *heads):
        mus, lvs = list(heads[:nh]), list(heads[nh:])
        loss, dxhat, dmus, dlvs = elbo_raw(x, xhat, mus, lvs, beta, want_grad=True, logits=logits, grad_scale=grad_scale)
        ctx.save_for_backward(dxhat, *dmus, *dlvs)
        ctx.nh = nh
        ctx.unit = unit_cotangent
        ctx.parts = loss
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        dxhat, rest = saved[0], saved[1:]
        if ctx.unit:
            # the caller differentiates the loss itself (`loss.backward()`): the cotangent is 1 and the (P,B,T) gradient
            # the kernel already wrote is handed on as it is (scaling it would be one more pass over 1.3 GB at B = 8192)
            return (None, dxhat, None, None, None, None, None, *rest)
        return (None, g * dxhat, None, None, None, None, None, *[g * r for r in rest])


def elbo_loss(x, xhat, mu, logvar, beta, logits: bool = False, unit_cotangent: bool = False, grad_scale: float = 1.0):
    """``loss_batch``'s reduction (reference ``examples/pendulum_friction-less/model_train.jl:225-238``):
    ``sum(mean((x - xhat)^2, dims=(2,3))) + beta * vector_kl(mu, logvar)`` as one fused forward+gradient pass.
    ``logits=True``: ``xhat`` are the pre-activations of the reconstructor's sigmoid output layer (folded into the kernel).
    ``unit_cotangent=True``: the result is differentiated directly (``loss.backward()``), never scaled further; a constant
    factor on the gradients (the data-parallel ``B_local / B_global``) then goes in as ``grad_scale`` -- the kernel writes the
    gradients already multiplied by it, the returned loss value stays unscaled.  ``beta``: a float or a 0-d CUDA tensor
    (``elbo_raw``)."""
    mus = list(mu) if isinstance(mu, (tuple, list)) else [mu]
    lvs = list(logvar) if isinstance(logvar, (tuple, list)) else [logvar]
    return _Elbo.apply(x, xhat, beta if isinstance(beta, torch.Tensor) else float(beta), len(mus), bool(logits), bool(unit_cotangent), float(grad_scale), *mus, *lvs)


def adamw_step(params: torch.Tensor, grads: torch.Tensor, m: torch.Tensor, v: torch.Tensor, step: int, lr=1e-3,
               betas=(0.9, 0.999), eps=1e-8, decay=1e-3, grad_scale: float = 1.0):
    """``ldeq_adamw_step`` on flat fp32 buffers: Flux ``ADAMW(eta, beta, decay)`` semantics (model_train.jl:138)."""
    h = _cabi.handle(params.device.index or 0)
    assert params.is_contiguous() and grads.is_contiguous() and m.is_contiguous() and v.is_contiguous()
    with torch.cuda.device(params.device):
        h.check(h._lib.ldeq_adamw_step(h.ptr, _p(params), _p(grads), _p(m), _p(v), params.numel(), float(lr),
                                       float(betas[0]), float(betas[1]), float(eps), C.c_float(decay), int(step),
                                       C.c_float(grad_scale), _stream()))


def adamw_step_dev(params: torch.Tensor, grads: torch.Tensor, m: torch.Tensor, v: torch.Tensor, state: torch.Tensor, lr=1e-3,
                   betas=(0.9, 0.999), eps=1e-8, decay=1e-3, grad_scale: float = 1.0):
    """``ldeq_adamw_step_dev``: ``adamw_step`` with the step count and the beta powers in ``state``, a 3-element Float64 CUDA
    tensor holding ``ldeq_adamw_state`` (``int64 step`` bit-cast, ``beta1^step``, ``beta2^step``), advanced on the device."""
    h = _cabi.handle(params.device.index or 0)
    assert params.is_contiguous() and grads.is_contiguous() and m.is_contiguous() and v.is_contiguous()
    if not (state.is_cuda and state.dtype == torch.float64 and state.numel() == 3 and state.is_contiguous()):
        raise TypeError("adamw_step_dev: state must be a contiguous 3-element Float64 CUDA tensor (ldeq_adamw_state)")
    with torch.cuda.device(params.device):
        h.check(h._lib.ldeq_adamw_step_dev(h.ptr, _p(params), _p(grads), _p(m), _p(v), params.numel(), float(lr),
                                           float(betas[0]), float(betas[1]), float(eps), C.c_float(decay), _p(state),
                                           C.c_float(grad_scale), _stream()))


def adamw_state(step: int, betas=(0.9, 0.999), device=None) -> torch.Tensor:
    """The ``ldeq_adamw_state`` after ``step`` steps, as ``adamw_step_dev`` keeps it: the beta powers are the running Float64
    products of ``ldeq_adamw_step`` (Python floats are IEEE doubles: same multiplications, same bits)."""
    p1 = p2 = 1.0
    for _ in range(step):
        p1 *= float(betas[0])
        p2 *= float(betas[1])
    st = torch.tensor([0.0, p1, p2], dtype=torch.float64)
    st.view(torch.int64)[0] = int(step)
    return st.to(device) if device is not None else st


def allreduce_adamw_step(params, peer_grad_ptrs, m, v, step: int, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, decay=1e-3,
                         grad_scale: float = 1.0, peer_param_ptrs=None, rank: int = 0):
    """``ldeq_allreduce_adamw_step``: sum the flat gradient buckets of all ranks straight over NVLink peer memory
    (``peer_grad_ptrs[r]`` = rank r's bucket mapped into this process) and apply AdamW in the same kernel.  With
    ``peer_param_ptrs`` (every rank's parameter replica, peer-mapped) the kernel is two-shot: this rank reduces and
    updates only its slice and writes the new parameters into every replica.  The caller provides the cross-GPU
    barriers around the call."""
    h = _cabi.handle(params.device.index or 0)
    W = len(peer_grad_ptrs)
    PA = C.c_void_p * W
    garr = PA(*[int(p) for p in peer_grad_ptrs])
    parr = PA(*[int(p) for p in peer_param_ptrs]) if peer_param_ptrs is not None else None
    with torch.cuda.device(params.device):
        h.check(h._lib.ldeq_allreduce_adamw_step(h.ptr, _p(params), parr, garr, W, int(rank), _p(m), _p(v), params.numel(),
                                                 float(lr), float(betas[0]), float(betas[1]), float(eps), C.c_float(decay),
                                                 int(step), C.c_float(grad_scale), _stream()))
