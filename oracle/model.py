"""Float64 restatement of whole ``GOKU_basic`` and ``LatentODE`` training steps -- TEST INFRASTRUCTURE (see
``oracle/__init__.py``).

Plain torch functions on the CPU over a ``{name: tensor}`` parameter dict whose names are those of
``LatentDiffEqModel.named_parameters()`` (``default_layers``' structure), so a model's parameters map onto it one to
one and torch autograd through these functions is the reference gradient.  The formulas are restated from the
reference, not taken from the product:

  * feature extractor / reconstructor  ``Chain(Dense, SkipConnection(Dense, +) x 2, Dense)`` (``GOKU.jl:199-274``)
  * pattern extractor  per-step Flux 0.13 cells with trainable initial states: ``RNN(relu)``: ``h' = relu(Wi x + Wh h + b)``;
    ``LSTM``: gates input, forget, cell, output; the z0 stack runs over the reversed sequence, theta is
    ``[fwd-stack(x)[end]; bwd-stack(reverse(x))[end]]`` (``GOKU.jl:30-49``, ``LatentODE.jl:20-34``)
  * heads  ``latent_in`` (``GOKU.jl:61-72``), ``sample`` with an injected eps (``GOKU.jl:155-173``), ``latent_out`` with
    the identity on z0 and softplus on theta (``GOKU.jl:83-91``)
  * solve  a ``torch.autograd.Function`` over ``oracle.goku`` (GOKU) or ``oracle.mlp`` (LatentODE, zero-padded by
    ``augment_dim``, ``LatentODE.jl:71``), the pullback chosen by the diffeq's sensitivity algorithm
  * loss  ``sum(mean((x - sigmoid(a))^2, dims=(T,B))) + beta * vector_kl(mu, logvar)`` (``model_train.jl:225-238``)

Arrays are in the product's order: frames ``[T, B, P]``, heads ``[B, d]``, trajectories ``[T, B, z]``.
"""
from __future__ import annotations

from dataclasses import dataclass, field, fields

import numpy as np
import torch
import torch.nn.functional as F

from . import goku as og
from . import mlp as om

GOKU, LATENTODE = "GOKU", "LatentODE"


# ---- the solve node ---------------------------------------------------------------------------------------------------
@dataclass
class SolveSpec:
    """What the solve node integrates and how it differentiates.

    ``kind``: ``GOKU`` or ``LATENTODE``.  ``rhs``: ``oracle.goku.PENDULUM`` / ``PENDULUM_FRICTION`` (GOKU).
    ``sensealg``: ``"forward_dual"`` (ForwardDiffSensitivity: partials in the error norm), ``"discrete"`` (the exact
    derivative of the taped primal steps) or ``"interpolating"`` (LatentODE's continuous adjoint).
    ``dtype``: state precision of the oracle solve (``np.float32`` is the reference's own Float32 arithmetic).
    ``dims`` / ``augment_dim``: the LatentODE right-hand side ``[D, H, H, D]`` and its zero padding."""
    kind: str
    opts: og.Opts
    sensealg: str
    dtype: type = np.float64
    rhs: int = og.PENDULUM
    dims: list = field(default_factory=list)
    augment_dim: int = 0


_SENSEALG = {"ForwardDiffSensitivity": "forward_dual", "DiscreteAdjoint": "discrete", "InterpolatingAdjoint": "interpolating"}


def spec_from_diffeq(diffeq, dtype=np.float64) -> SolveSpec:
    """The ``SolveSpec`` of a diffeq struct (``Pendulum`` / ``Pendulum_friction`` / ``NODE``), read from the struct's own
    fields the way ``diffeq_layer`` reads them: ``prob.f`` or ``dims``, ``kwargs``, ``sensealg`` (GOKU structs take it as
    the ``sensalg`` keyword), ``augment_dim``.  Only Tsit5 is restated."""
    if type(diffeq.solver).__name__ != "Tsit5":
        raise NotImplementedError(f"oracle.model restates Tsit5 only, not {diffeq.solver!r}")
    known = {f.name for f in fields(og.Opts)}
    unknown = set(diffeq.kwargs) - known
    if unknown:
        raise NotImplementedError(f"solve options {sorted(unknown)} are not restated by the oracle")
    opts = og.Opts(**diffeq.kwargs)
    sensealg = _SENSEALG[type(diffeq.sensealg).__name__]
    if hasattr(diffeq, "dims"):
        return SolveSpec(LATENTODE, opts, sensealg, dtype, dims=list(diffeq.dims), augment_dim=int(diffeq.augment_dim))
    return SolveSpec(GOKU, opts, sensealg, dtype, rhs=int(diffeq.prob.f))


def _np(x, dtype):
    return np.ascontiguousarray(x.detach().cpu().numpy().astype(dtype))


class _GokuSolve(torch.autograd.Function):
    """``oracle.goku.solve`` / ``grad`` as an autograd node.  ``pin``: ``(z0, theta)`` values to solve from instead of the
    inputs' own; the gradient is still routed to the inputs."""

    @staticmethod
    def forward(ctx, z0, theta, t, spec, pin, record):
        z0v, thv = pin if pin is not None else (z0, theta)
        ctx.z0, ctx.th = _np(torch.as_tensor(z0v), spec.dtype), _np(torch.as_tensor(thv), spec.dtype)
        ctx.t, ctx.spec = t, spec
        traj, ret, na, nr = og.solve(spec.rhs, ctx.z0, ctx.th, t, spec.opts)
        record.update(retcode=ret, naccept=na, nreject=nr)
        return torch.from_numpy(traj.astype(np.float64))

    @staticmethod
    def backward(ctx, dtraj):
        s = ctx.spec
        if s.sensealg not in ("forward_dual", "discrete"):
            raise NotImplementedError(f"GOKU pullback {s.sensealg!r}")
        dz0, dth = og.grad(s.rhs, ctx.z0, ctx.th, ctx.t, _np(dtraj, s.dtype), s.opts, norm_partials=s.sensealg == "forward_dual")
        return torch.from_numpy(dz0.astype(np.float64)), torch.from_numpy(dth.astype(np.float64)), None, None, None, None


class _MlpSolve(torch.autograd.Function):
    """``oracle.mlp.solve(record=True)`` with ``interpolating_adjoint`` or ``discrete_adjoint`` on its tape."""

    @staticmethod
    def forward(ctx, z0, p_flat, t, spec, pin, record):
        ctx.z0 = _np(torch.as_tensor(pin if pin is not None else z0), spec.dtype)
        ctx.p = _np(p_flat, spec.dtype)
        ctx.t, ctx.spec = t, spec
        traj, na, nr, ctx.tape = om.solve(ctx.z0, ctx.p, spec.dims, t, spec.opts, record=True)
        record.update(naccept=na, nreject=nr)
        return torch.from_numpy(traj.astype(np.float64))

    @staticmethod
    def backward(ctx, dtraj):
        s = ctx.spec
        d = dtraj.detach().numpy().astype(np.float64)
        if s.sensealg == "interpolating":
            dz0, dp = om.interpolating_adjoint(ctx.z0, ctx.p, s.dims, ctx.t, d, s.opts, tape=ctx.tape)
        elif s.sensealg == "discrete":
            dz0, dp = om.discrete_adjoint(ctx.p, s.dims, ctx.t, ctx.tape, d)
        else:
            raise NotImplementedError(f"LatentODE pullback {s.sensealg!r}")
        return torch.from_numpy(np.asarray(dz0, np.float64)), torch.from_numpy(np.asarray(dp, np.float64)), None, None, None, None


# ---- layers -----------------------------------------------------------------------------------------------------------
def dense(P, name, x, act=None):
    y = F.linear(x, P[name + ".weight"], P[name + ".bias"])
    return act(y) if act is not None else y


def resnet(P, prefix, x, out_act=None):
    """``Chain(Dense(relu), SkipConnection(Dense(relu), +), SkipConnection(Dense(relu), +), Dense(out_act))``."""
    h = dense(P, prefix + ".0", x, torch.relu)
    h = h + dense(P, prefix + ".1.layer", h, torch.relu)
    h = h + dense(P, prefix + ".2.layer", h, torch.relu)
    return dense(P, prefix + ".3", h, out_act)


def recurrent_final(P, prefix, xs, reverse):
    """Last hidden state ``[B, H]`` of a two-layer ``Chain`` of Flux ``RNN(relu)`` or ``LSTM`` cells over ``xs [T, B, F]``,
    hidden states restarting from the trainable initial states."""
    T, B, _ = xs.shape
    layers = [f"{prefix}.0", f"{prefix}.1"]
    lstm = (layers[0] + ".h0") in P
    hs = [P[l + (".h0" if lstm else ".state0")].expand(B, -1) for l in layers]
    cs = [P[l + ".c0"].expand(B, -1) for l in layers] if lstm else None
    for k in (range(T - 1, -1, -1) if reverse else range(T)):
        inp = xs[k]
        for i, l in enumerate(layers):
            g = inp @ P[l + ".Wi"].t() + hs[i] @ P[l + ".Wh"].t() + P[l + ".b"]
            if lstm:
                o = hs[i].shape[1]
                gi, gf = torch.sigmoid(g[:, :o]), torch.sigmoid(g[:, o:2 * o])
                gc, go = torch.tanh(g[:, 2 * o:3 * o]), torch.sigmoid(g[:, 3 * o:])
                cs[i] = gf * cs[i] + gi * gc
                hs[i] = go * torch.tanh(cs[i])
            else:
                hs[i] = torch.relu(g)
            inp = hs[i]
    return hs[-1]


def encoder(P, kind, x):
    """``(mu, logvar)``: tuples ``(z0 head, theta head)`` for GOKU, single ``[B, d]`` tensors for LatentODE."""
    fe = resnet(P, "encoder.feature_extractor", x, torch.relu)
    if kind == GOKU:
        pre = "encoder.pattern_extractor.layers"
        z0_out = recurrent_final(P, pre + ".0", fe, reverse=True)
        th_out = torch.cat([recurrent_final(P, pre + ".1", fe, reverse=False), recurrent_final(P, pre + ".2", fe, reverse=True)], 1)
        li = "encoder.latent_in.layers"
        return ((dense(P, li + ".0", z0_out), dense(P, li + ".2", th_out)),
                (dense(P, li + ".1", z0_out), dense(P, li + ".3", th_out)))
    pe = recurrent_final(P, "encoder.pattern_extractor", fe, reverse=True)
    return dense(P, "encoder.latent_in.layers.0", pe), dense(P, "encoder.latent_in.layers.1", pe)


def sample(mu, logvar, eps):
    """``mu + eps * exp(logvar / 2)`` per head, ``eps`` given."""
    if isinstance(mu, tuple):
        return tuple(m + e * torch.exp(lv / 2) for m, lv, e in zip(mu, logvar, eps))
    return mu + eps * torch.exp(logvar / 2)


def latent_out(P, kind, l_tilde):
    if kind == GOKU:
        lo = "decoder.latent_out.layers"
        z0 = dense(P, lo + ".0.1", dense(P, lo + ".0.0", l_tilde[0], torch.relu))
        th = dense(P, lo + ".1.1", dense(P, lo + ".1.0", l_tilde[1], torch.relu), F.softplus)
        return z0, th
    return l_tilde


def diffeq_layer(P, spec: SolveSpec, l_hat, t, pin=None, record=None):
    """``z_hat [T, B, z]``.  ``pin``: the values the solve starts from (GOKU: ``(z0, theta)``; LatentODE: ``z0`` before the
    padding); gradients still flow into ``l_hat``."""
    t = np.ascontiguousarray(np.asarray(t, dtype=np.float64))
    record = {} if record is None else record
    if spec.kind == GOKU:
        return _GokuSolve.apply(l_hat[0], l_hat[1], t, spec, pin, record)
    z0 = l_hat
    if spec.augment_dim:
        z0 = torch.cat([z0, z0.new_zeros(z0.shape[0], spec.augment_dim)], 1)
        if pin is not None:
            pin = torch.cat([torch.as_tensor(pin), torch.zeros(z0.shape[0], spec.augment_dim, dtype=torch.as_tensor(pin).dtype)], 1)
    # Flux.destructure order of dudt: per layer vec(W) (column-major) then b
    p_flat = torch.cat([torch.cat([P[f"decoder.diffeq.weights.{i}"].t().reshape(-1), P[f"decoder.diffeq.biases.{i}"]])
                        for i in range(len(spec.dims) - 1)])
    return _MlpSolve.apply(z0, p_flat, t, spec, pin, record)


def reconstructor_logits(P, z_hat):
    """The reconstructor up to the pre-activations of its sigmoid output layer."""
    return resnet(P, "decoder.reconstructor", z_hat)


def vector_kl(mu, logvar):
    """``utils.jl:18-44``: per head ``sum(kl) / batch``, summed over heads."""
    mus = mu if isinstance(mu, tuple) else (mu,)
    lvs = logvar if isinstance(logvar, tuple) else (logvar,)
    return sum(((torch.exp(lv) + m ** 2 - lv - 1) / 2).sum() / m.shape[0] for m, lv in zip(mus, lvs))


def loss_batch(P, spec: SolveSpec, x, t, beta, eps=None, pin=None, record=None):
    """One ``loss_batch`` (``model_train.jl:225-238``) of the model ``P`` on frames ``x [T, B, P]``.  ``eps``: the noise of
    ``sample`` (``None``: not variational, ``l_tilde = mu``).  Returns ``(loss, extras)``; ``extras`` holds the
    intermediate ``mu``, ``logvar``, ``l_hat``, ``z_hat`` and the solve's statistics (``extras['solve']``)."""
    x = torch.as_tensor(x, dtype=torch.float64)
    mu, logvar = encoder(P, spec.kind, x)
    l_tilde = sample(mu, logvar, eps) if eps is not None else mu
    l_hat = latent_out(P, spec.kind, l_tilde)
    stats = {} if record is None else record
    z_hat = diffeq_layer(P, spec, l_hat, t, pin, stats)
    a = reconstructor_logits(P, z_hat)
    loss = ((x - torch.sigmoid(a)) ** 2).mean(dim=(0, 1)).sum() + beta * vector_kl(mu, logvar)
    return loss, {"mu": mu, "logvar": logvar, "l_hat": l_hat, "z_hat": z_hat, "solve": stats}


def params_from(named_parameters, requires_grad: bool = True) -> dict:
    """Float64 CPU copies ``{name: tensor}`` of a model's ``named_parameters()``, leaves of the reference graph."""
    return {n: p.detach().to("cpu", torch.float64).clone().requires_grad_(requires_grad) for n, p in named_parameters}
