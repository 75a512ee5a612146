"""The training step of the reference's example script on the CUDA path.

``loss_batch`` (``examples/pendulum_friction-less/model_train.jl:225-238``), the gradient step
``Flux.pullback`` + ``update!(ADAMW(...))`` (``model_train.jl:138,195-201``) and, for several GPUs of
one box, the data-parallel layout the north star asks for: every rank integrates its own slice of
the batch, the parameter gradient lives in ONE flat fp32 bucket that is all-reduced once per step
over NCCL, then every rank applies the same fused AdamW.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _cabi
from . import model as _model
from .solve import _tgrid, adamw_state, adamw_step, adamw_step_dev, allreduce_adamw_step, elbo_loss


def loss_batch(model, x, t, beta, variational, fused_output: bool = True, unit_cotangent: bool = False, grad_scale: float = 1.0):
    """model_train.jl:225-238.  ``x`` is ``[T, B, P]``.  With ``fused_output`` (default) the sigmoid of the reconstructor's
    output layer (GOKU.jl:265-268) is evaluated inside the loss kernel (``ldeq_elbo_logits_fwd_bwd``): same loss, same
    gradients, no x-hat array.  ``unit_cotangent``: the caller differentiates the returned loss directly (``grad_scale``: constant
    factor the kernel applies to the gradients, see ``elbo_loss``)."""
    if not x.is_cuda:
        raise RuntimeError("loss_batch runs in libldeq.so on a CUDA device (no CPU fallback)")
    out = model.forward_logits(x, t, variational) if fused_output and hasattr(model, "forward_logits") else None
    if out is not None:
        (logits, z_hat, l_hat), mu, logvar = out
        return elbo_loss(x, logits, mu, logvar, beta, logits=True, unit_cotangent=unit_cotangent, grad_scale=grad_scale)
    X_hat, mu, logvar = model(x, t, variational)
    x_hat, z_hat, l_hat = X_hat
    return elbo_loss(x, x_hat, mu, logvar, beta, unit_cotangent=unit_cotangent, grad_scale=grad_scale)


def shard_bounds(n: int, rank: int, world: int):
    """Contiguous batch slice of ``rank``: trajectories are independent (GOKU.jl:111), so the batch is
    simply cut into ``world`` pieces; remainders go to the first ranks."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class FlatParams:
    """All trainable parameters of a model viewed through ONE contiguous fp32 buffer (and one gradient
    buffer): a single all-reduce and a single fused AdamW launch per step."""

    def __init__(self, module: torch.nn.Module, symmetric: bool = False):
        """``symmetric=True`` (several CUDA ranks of one box): the gradient bucket is NVLink symmetric memory, every
        rank can read every other rank's bucket, and the optimiser step fuses the all-reduce (``ADAMW.step``)."""
        self.params = [p for p in module.parameters() if p.requires_grad]
        n = sum(p.numel() for p in self.params)
        n_pad = (n + 3) // 4 * 4
        dev = self.params[0].device
        self.n = n
        self.symm = self.symm_p = None
        if symmetric and dev.type == "cuda" and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            import torch.distributed._symmetric_memory as symm_mem
            self.grad = symm_mem.empty(n_pad, dtype=torch.float32, device=dev)
            self.grad.zero_()
            self.symm = symm_mem.rendezvous(self.grad, dist.group.WORLD)
            self.flat = symm_mem.empty(n_pad, dtype=torch.float32, device=dev)   # replicas are peer-writable (two-shot step)
            self.flat.zero_()
            self.symm_p = symm_mem.rendezvous(self.flat, dist.group.WORLD)
        else:
            self.flat = torch.zeros(n_pad, dtype=torch.float32, device=dev)
            self.grad = torch.zeros(n_pad, dtype=torch.float32, device=dev)
        self.m = torch.zeros(n_pad, dtype=torch.float32, device=dev)
        self.v = torch.zeros(n_pad, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:
            k = p.numel()
            self.flat[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off:off + k].view_as(p)
            p.grad = self.grad[off:off + k].view_as(p)
            off += k

    def zero_grad(self):
        self.grad.zero_()
        off = 0
        for p in self.params:  # autograd may have replaced .grad
            k = p.numel()
            p.grad = self.grad[off:off + k].view_as(p)
            off += k


class ADAMW:
    """``ADAMW(eta, (b1, b2), decay)`` of the reference (model_train.jl:138) on a :class:`FlatParams`."""

    def __init__(self, flat: FlatParams, eta=1e-3, beta=(0.9, 0.999), decay=1e-3, eps=1e-8):
        self.flat, self.eta, self.beta, self.decay, self.eps = flat, eta, beta, decay, eps
        self.step_count = 0

    def step(self, grad_scale: float = 1.0):
        """Local AdamW on the (already all-reduced) flat gradient."""
        self.step_count += 1
        f = self.flat
        if f.flat.is_cuda:
            adamw_step(f.flat, f.grad, f.m, f.v, self.step_count, self.eta, self.beta, self.eps, self.decay, grad_scale)
        else:
            raise RuntimeError("the optimiser step runs in libldeq.so on a CUDA device (no CPU fallback)")

    def step_dev(self, state: torch.Tensor, grad_scale: float = 1.0):
        """``step`` with the step count and the beta powers in the device tensor ``state`` (``adamw_step_dev``), which the
        kernel advances; ``step_count`` is left to the caller (``GraphedTrainStep`` keeps it as the host mirror)."""
        f = self.flat
        adamw_step_dev(f.flat, f.grad, f.m, f.v, state, self.eta, self.beta, self.eps, self.decay, grad_scale)

    def fused_allreduce_step(self, grad_scale: float = 1.0):
        """All-reduce + AdamW in ONE kernel over NVLink peer memory (needs ``FlatParams(..., symmetric=True)``):
        barrier (all buckets written) -> sum in rank order + AdamW -> barrier (every rank has read every bucket / written
        every replica before the next pass).  Two ranks: one-shot (each rank reduces everything).  More: two-shot (each
        rank reduces and updates its 1/N slice and stores the new parameters into every replica)."""
        f = self.flat
        assert f.symm is not None, "FlatParams was not built with symmetric=True"
        self.step_count += 1
        two_shot = f.symm.world_size > 2 and f.symm_p is not None
        f.symm.barrier(channel=0)
        allreduce_adamw_step(f.flat, list(f.symm.buffer_ptrs), f.m, f.v, self.step_count, self.eta, self.beta, self.eps,
                             self.decay, grad_scale, peer_param_ptrs=list(f.symm_p.buffer_ptrs) if two_shot else None,
                             rank=f.symm.rank)
        f.symm.barrier(channel=1)


def allreduce_grads(flat: FlatParams):
    """One sum all-reduce of the flat gradient bucket (NCCL over NVLink on the GPU box, gloo in the CPU tests)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(flat.grad, op=dist.ReduceOp.SUM)


def train_step(model, flat: FlatParams, opt: ADAMW, x_local, t, beta, variational=True, global_batch=None, timers=None):
    """One data-parallel training step on this rank's slice ``x_local`` ``[T, B_local, P]``.

    The loss is a mean over the GLOBAL batch: the local loss is scaled by ``B_local / B_global`` before the
    backward pass, gradients are summed across ranks, and every rank applies the same AdamW update.
    ``timers`` (a dict) receives CUDA events at the phase boundaries: start, loss, backward, update."""
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    B_local = x_local.shape[1]
    B_global = global_batch or B_local * world
    def mark(name):
        if timers is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            timers[name] = ev
    mark("start")
    flat.zero_grad()
    # the loss is a mean over the GLOBAL batch: the factor B_local / B_global rides inside the loss kernel's gradients
    # (grad_scale), the loss itself is differentiated with a unit cotangent -- no extra pass over the (P,B,T) gradient
    loss = loss_batch(model, x_local, t, beta, variational, unit_cotangent=True, grad_scale=B_local / B_global)
    mark("loss")
    loss.backward()
    mark("backward")
    if flat.symm is not None:
        opt.fused_allreduce_step()
    else:
        allreduce_grads(flat)
        opt.step()
    mark("update")
    return loss.detach()


class GraphedTrainStep:
    """``train_step`` captured once as a CUDA graph and replayed: ``loss = step(x, beta)``.

    At the reference's batch of 64 every kernel of a step runs for microseconds and the eager step is bound by launches and
    host work; a replay is one launch.  The per-step values live in device memory: the AdamW step state, the sample counter
    (``ldeq_sample_dev``) and beta (the ELBO's ``_dev`` entry points), so replay k computes what eager step k computes, bit
    for bit.  ``opt.step_count`` and the module's sample counter stay the host mirrors: each call advances them, and eager
    calls in between (a validation ``loss_batch``) keep working on the same handle and stream; when the mirrors moved
    without the graph (an eager ``train_step``), the device state is refreshed from them before the replay.

    Built for single-GPU GOKU training on its default path: Pendulum / Pendulum_friction / NVRTC right-hand sides with
    ``ForwardDiffSensitivity()``, the pattern-extractor kernels, the fused logits ELBO and AdamW.  Everything else is refused
    before any capture: LatentODE (its reverse passes need the host), ``DiscreteAdjoint()``, world size > 1 and a
    reconstructor without the sigmoid output layer the fused loss needs.  ``x`` must keep ``x_example``'s shape, ``t`` is
    fixed, and the noise seed is ``torch.initial_seed()`` at construction.  Construction warms the exact shapes up on a side
    stream (modules, the device grid, the workspaces) and leaves parameters, gradients, ``m``, ``v``, ``opt.step_count`` and
    the sample counter as it found them."""

    def __init__(self, model, flat: FlatParams, opt: ADAMW, x_example: torch.Tensor, t, variational: bool = True, warmup: int = 2):
        if not x_example.is_cuda:
            raise RuntimeError("GraphedTrainStep: the batch must be a CUDA tensor")
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            raise NotImplementedError("GraphedTrainStep: single GPU only (the gradient all-reduce is not captured)")
        if flat.symm is not None:
            raise NotImplementedError("GraphedTrainStep: FlatParams(symmetric=True) belongs to the fused multi-GPU step")
        if not isinstance(model.model_type, _model.GOKU):
            raise NotImplementedError("GraphedTrainStep: GOKU models only; LatentODE's reverse passes need the host (the MLP tape "
                                      "check and the continuous adjoint)")
        diffeq = model.decoder.diffeq
        opts = _model._opts_from_kwargs(diffeq.kwargs, getattr(diffeq, "sensealg", None), getattr(diffeq, "solver", None))
        if opts.sensealg != _cabi.SENSE_FORWARD_DUAL:
            raise NotImplementedError("GraphedTrainStep: ForwardDiffSensitivity() only; the discrete adjoint checks its tape on the host")
        if _model._logits_layers(model.decoder) is None:
            raise NotImplementedError("GraphedTrainStep: the reconstructor must end in a Dense layer with the sigmoid output "
                                      "activation (the fused logits ELBO)")
        self.model, self.flat, self.opt, self.variational = model, flat, opt, variational
        dev = x_example.device
        self._t = _tgrid(t)
        self._x = x_example.detach().clone(memory_format=torch.contiguous_format)
        self._beta = torch.zeros((), dtype=torch.float32, device=dev)
        self._state = torch.zeros(3, dtype=torch.float64, device=dev)   # ldeq_adamw_state
        self._calls = torch.zeros(1, dtype=torch.int64, device=dev)
        saved = [b.clone() for b in (flat.flat, flat.grad, flat.m, flat.v)]
        step0, calls0 = opt.step_count, _model._sample_calls
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._body()
        cur.wait_stream(side)
        for b, v in zip((flat.flat, flat.grad, flat.m, flat.v), saved):
            b.copy_(v)
        opt.step_count = step0
        _model._sample_calls = calls0
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._loss = self._body()
        self._draws = _model._sample_calls - calls0   # samples per step
        _model._sample_calls = calls0
        self._synced = None   # (step_count, sample counter) the device state holds

    def _body(self):
        self.flat.zero_grad()
        with _model.device_sample_counter(self._calls):
            loss = loss_batch(self.model, self._x, self._t, self._beta, self.variational, unit_cotangent=True)
        loss.backward()
        self.opt.step_dev(self._state)
        return loss.detach()

    def __call__(self, x: torch.Tensor, beta) -> torch.Tensor:
        """One training step on ``x`` (``x_example``'s shape) with KL weight ``beta`` (float or 0-d CUDA tensor); returns the
        loss as a device tensor, without synchronising."""
        if (self.opt.step_count, _model._sample_calls) != self._synced:
            self._state.copy_(adamw_state(self.opt.step_count, self.opt.beta))
            self._calls.fill_(_model._sample_calls)
        self._x.copy_(x)
        if isinstance(beta, torch.Tensor):
            self._beta.copy_(beta)
        else:
            self._beta.fill_(beta)
        self._graph.replay()
        self.opt.step_count += 1
        _model._sample_calls += self._draws
        self._synced = (self.opt.step_count, _model._sample_calls)
        return self._loss.clone()
