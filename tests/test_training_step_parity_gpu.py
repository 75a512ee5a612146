"""Whole training steps on the CUDA path against the float64 reference of ``oracle/model.py``.

Each kernel has its own parity test; these check the composition a user trains with: the autograd functions of
``solve.py`` (flat-parameter order of the pattern extractor, the sample's logvar derivative, the ELBO's cotangent and
``grad_scale``, the solve tapes), the routing of ``model.py`` (logits route, head order, augment padding) and the one
flat gradient bucket that ``ADAMW.step`` reads.

The default initialisation gives nearly constant pendulum lengths (|z0| <~ 0.005, L ~ 0.695 for every sample), where the
solve and its pullback barely reach the loss.  ``_condition`` puts the model into the data's regime first
(``create_data.jl:19-22``: angle ~ +-pi/6, velocity ~ +-pi/3, L in [1, 2]) and every test asserts that it did.

Comparison rule, per parameter tensor: ``|g - g_ref| <= tol |g_ref| + 1e-7 |g_ref,all|`` (2-norms; the second term is a
floor for tensors whose gradient is legitimately ~0), whole model ``|g - g_ref|_all <= tol |g_ref|_all``, loss 1e-5
relative."""
import copy
import math
import time
from importlib import import_module

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import loss as ol
from oracle import model as rm

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, T, P_IN = 64, 50, 784
T_GRID = 0.05 * np.arange(T)
BETA = 0.5
Z0_STD = (0.3, 0.6)                       # ~U(+-0.5 rad), ~U(+-1 rad/s)
L_RANGE = (1.0, 2.0)                      # create_data.jl:19-22


@pytest.fixture
def exact_fp32():
    """fp32 matmuls and cuDNN without TF32 for the test; both settings restored afterwards."""
    saved = (torch.get_float32_matmul_precision(), torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.set_float32_matmul_precision("highest")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.set_float32_matmul_precision(saved[0])
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved[1], saved[2]


def _frames(seed=0):
    return torch.rand(T, B, P_IN, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _softplus_inv(y):
    return math.log(math.expm1(y))


def _condition(ldeq, model, x, variational, seed):
    """Non-trivial biases and initial states (+0.05 N(0,1) on every 1-D parameter); for GOKU the final ``Dense`` of each
    ``latent_out`` head rescaled so that, over the batch, z0 has the spreads ``Z0_STD`` and L = softplus(.) spreads over
    ``L_RANGE``.  With ``variational`` the spreads are set on a sample of the encoder's distribution."""
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for p in model.parameters():
            if p.dim() == 1:
                p.add_(0.05 * torch.randn(p.shape, generator=gen).to(p.device))
        if not isinstance(model.model_type, ldeq.GOKU):
            return
        mu, lv = model.encoder(x)
        l_tilde = mu
        if variational:
            l_tilde = tuple(m + torch.randn(m.shape, generator=gen).to(m.device) * torch.exp(v / 2) for m, v in zip(mu, lv))
        lo, hi = _softplus_inv(L_RANGE[0]), _softplus_inv(L_RANGE[1])
        targets = ((torch.zeros(2), torch.tensor(Z0_STD)), (torch.tensor([(lo + hi) / 2]), torch.tensor([(hi - lo) / (2 * math.sqrt(3))])))
        for head, lt, (center, std) in zip(model.decoder.latent_out, l_tilde, targets):
            last = head[1]
            o = F.linear(head[0](lt), last.weight, last.bias)
            a = std.to(o.device) / o.std(0)
            last.weight.mul_(a[:, None])
            last.bias.mul_(a).add_(center.to(o.device) - a * o.mean(0))


def _assert_conditioned(l_hat):
    z0, L = l_hat[0].double().cpu(), l_hat[1].double().cpu()
    s = z0.std(0)
    print(f"conditioning: z0 std {s[0]:.3f} rad, {s[1]:.3f} rad/s; L in [{L.min():.3f}, {L.max():.3f}]")
    assert 0.15 <= s[0] <= 0.6 and 0.3 <= s[1] <= 1.2, s
    assert L.min() >= 0.5 and L.max() <= 3.0 and L.max() - L.min() >= 0.5, (L.min(), L.max())


def _model(ldeq, model_type, diffeq, x, variational, seed=333):
    torch.manual_seed(seed)
    enc, dec = ldeq.default_layers(model_type, P_IN, diffeq, device=DEV)
    model = ldeq.LatentDiffEqModel(model_type, enc, dec)
    _condition(ldeq, model, x, variational, seed)
    return model


class _Capture:
    """What the CUDA forward saw: every ``sample_reparam`` call (inputs, counter, output) and ``diffeq_layer``'s ``l_hat``
    and solve statistics."""

    def __init__(self, monkeypatch):
        mod = import_module("latentdiffeq_jl_b200.model")
        self.samples, self.l_hat, self.stats = [], None, []
        sample_reparam, diffeq_layer = mod.sample_reparam, mod.diffeq_layer

        def sample_rec(mu, logvar, seed, offset=0):
            z = sample_reparam(mu, logvar, seed, offset)
            self.samples.append((mu.detach().clone(), logvar.detach().clone(), seed, offset, z.detach().clone()))
            return z

        def diffeq_layer_rec(decoder, l_hat, t, stats_out=None):
            self.l_hat = tuple(v.detach().clone() for v in l_hat) if isinstance(l_hat, tuple) else l_hat.detach().clone()
            return diffeq_layer(decoder, l_hat, t, self.stats)

        monkeypatch.setattr(mod, "sample_reparam", sample_rec)
        monkeypatch.setattr(mod, "diffeq_layer", diffeq_layer_rec)
        # the noise offset of `sample` counts calls process-wide: from 0, a test draws the same noise whichever tests ran
        # before it, so its measured errors are reproducible
        monkeypatch.setattr(mod, "_sample_calls", 0)

    def eps(self, ldeq, n_heads):
        """The noise of every recorded sample, drawn again from its (seed, offset) -- and checked to be that noise."""
        assert len(self.samples) == n_heads
        out = []
        for mu, lv, seed, offset, z in self.samples:
            z2, e = ldeq.sample_raw(mu, lv, seed, offset)
            assert torch.equal(z2, z)
            want = mu.double() + e.double() * torch.exp(lv.double() / 2)
            assert (z.double() - want).abs().max() <= 2e-6 * want.abs().max()
            out.append(e.double().cpu())
        return tuple(out) if n_heads > 1 else out[0]

    def pin(self):
        return tuple(v.cpu() for v in self.l_hat) if isinstance(self.l_hat, tuple) else self.l_hat.cpu()


def _cuda_step(ldeq, model, x, variational, fused_output=True):
    model.zero_grad(set_to_none=True)
    loss = ldeq.loss_batch(model, x, T_GRID, BETA, variational, fused_output=fused_output)
    loss.backward()
    torch.cuda.synchronize()
    grads = {}
    for n, p in model.named_parameters():
        assert p.grad is not None, f"{n} received no gradient"
        grads[n] = p.grad.detach().double().cpu()
    return float(loss), grads


def _reference_step(model, spec, x, eps, pin=None):
    P = rm.params_from(model.named_parameters())
    stats = {}
    loss, extras = rm.loss_batch(P, spec, x.double().cpu(), T_GRID, BETA, eps, pin, stats)
    loss.backward()
    return float(loss.detach()), {n: p.grad for n, p in P.items()}, extras


def _assert_l_hat_agrees(l_hat, l_hat_ref):
    for got, want in zip(*((l_hat, l_hat_ref) if isinstance(l_hat, tuple) else ((l_hat,), (l_hat_ref,)))):
        got, want = got.double().cpu(), want.detach()
        assert (got - want).abs().max() <= 1e-5 * want.abs().max(), float((got - want).abs().max() / want.abs().max())


def _compare(label, loss, grads, loss_ref, grads_ref, tol):
    """The comparison rule of the module docstring; prints every tensor's error.  Returns the largest ``|err| / |g_ref|``
    over the tensors above the floor, and the whole-model relative error."""
    g_all = math.sqrt(sum(float(g.square().sum()) for g in grads_ref.values()))
    d_all, worst, bad = 0.0, 0.0, []
    for n, g_ref in grads_ref.items():
        e, r = float((grads[n] - g_ref).norm()), float(g_ref.norm())
        d_all += e * e
        ok = e <= tol * r + 1e-7 * g_all
        if r > 1e-7 * g_all:
            worst = max(worst, e / r)
        print(f"{label} {n:52s} |g_ref| {r:.3e}  |err| {e:.3e}  rel {e / max(r, 1e-300):.2e}{'' if ok else '  <-- over ' + str(tol)}")
        if not ok:
            bad.append(n)
    d_all = math.sqrt(d_all)
    loss_err = abs(loss - loss_ref) / abs(loss_ref)
    print(f"{label} whole model |g_ref| {g_all:.3e} rel err {d_all / g_all:.2e}; worst tensor {worst:.2e}; "
          f"loss {loss:.8e} vs {loss_ref:.8e} rel {loss_err:.2e}")
    assert not bad, f"{label}: gradients over tolerance {tol}: {bad}"
    assert d_all <= tol * g_all
    assert loss_err <= 1e-5
    return worst, d_all / g_all


@pytest.mark.parametrize("rhs", ["Pendulum", "Pendulum_friction"])
def test_goku_fixed_step_gradients(ldeq, exact_fp32, monkeypatch, rhs):
    # fixed step: the CUDA pullback is the exact derivative of the primal discretisation, so the whole reference runs in
    # float64 (solve included) from its own l_hat, without pinning
    t0 = time.perf_counter()
    diffeq = getattr(ldeq, rhs)(adaptive=False, dt=0.01)
    x = _frames()
    model = _model(ldeq, ldeq.GOKU_basic(), diffeq, x, variational=True)
    cap = _Capture(monkeypatch)
    loss, grads = _cuda_step(ldeq, model, x, variational=True)
    _assert_conditioned(cap.l_hat)
    loss_ref, grads_ref, ex = _reference_step(model, rm.spec_from_diffeq(diffeq), x, cap.eps(ldeq, 2))
    _assert_l_hat_agrees(cap.l_hat, ex["l_hat"])
    assert (cap.stats[0].naccept.cpu().numpy() == ex["solve"]["naccept"]).all()
    _compare(f"[{rhs} fixed]", loss, grads, loss_ref, grads_ref, 1e-4)
    print(f"[{rhs} fixed] wall {time.perf_counter() - t0:.1f} s")


@pytest.mark.parametrize("fused_output", [True, False])
@pytest.mark.parametrize("sensalg,tol", [("ForwardDiffSensitivity", 5e-6), ("DiscreteAdjoint", 2.7e-5)])
def test_goku_c1_default_gradients(ldeq, exact_fp32, monkeypatch, sensalg, tol, fused_output):
    # C1 with the default adaptive Tsit5: the reference's solve node is the oracle's Float32 arithmetic (the kernels'
    # precision) started from the l_hat the kernel saw; the layers around it are float64.  The kernels keep the stage
    # arithmetic in fp32 where Julia promotes it to Float64, so a few trajectories take another accept/reject path
    # (naccept equal on 63 of 64 here).  tol is twice the worst tensor's error measured on a B200 (1000 W power limit):
    # 2.3e-6 with ForwardDiffSensitivity, 1.31e-5 with DiscreteAdjoint (whole model 6.2e-7 / 1.5e-6).
    t0 = time.perf_counter()
    diffeq = ldeq.Pendulum(sensalg=getattr(ldeq, sensalg)())
    x = _frames()
    model = _model(ldeq, ldeq.GOKU_basic(), diffeq, x, variational=True)
    cap = _Capture(monkeypatch)
    loss, grads = _cuda_step(ldeq, model, x, variational=True, fused_output=fused_output)
    _assert_conditioned(cap.l_hat)
    loss_ref, grads_ref, ex = _reference_step(model, rm.spec_from_diffeq(diffeq, np.float32), x, cap.eps(ldeq, 2), cap.pin())
    _assert_l_hat_agrees(cap.l_hat, ex["l_hat"])
    agree = (cap.stats[0].naccept.cpu().numpy() == ex["solve"]["naccept"]).mean()
    label = f"[C1 {sensalg} fused={fused_output}]"
    worst, whole = _compare(label, loss, grads, loss_ref, grads_ref, tol)
    print(f"{label} naccept equal on {agree:.3f} of the trajectories; worst tensor {worst:.2e}, whole {whole:.2e}; "
          f"wall {time.perf_counter() - t0:.1f} s")
    assert agree >= 0.9


@pytest.mark.parametrize("config,tol", [("interpolating", 5e-3), ("discrete_fixed", 2e-4)])
def test_latentode_gradients(ldeq, exact_fp32, monkeypatch, config, tol):
    # the reference solves from the kernel's z0 (pinned) in the oracle's mixed Float32 arithmetic; the interpolating adjoint
    # agrees with the fp32 kernel to its documented 5e-3 (test_mlp_gpu.py), the fixed-step discrete adjoint is exact
    t0 = time.perf_counter()
    if config == "interpolating":
        diffeq = ldeq.NODE(16)
    else:
        diffeq = ldeq.NODE(16, augment_dim=2, sensealg=ldeq.DiscreteAdjoint(), adaptive=False, dt=0.02)
    x = _frames()
    model = _model(ldeq, ldeq.LatentODE(), diffeq, x, variational=True)
    cap = _Capture(monkeypatch)
    loss, grads = _cuda_step(ldeq, model, x, variational=True)
    spec = rm.spec_from_diffeq(diffeq, np.float32)
    assert spec.sensealg == ("interpolating" if config == "interpolating" else "discrete")
    loss_ref, grads_ref, ex = _reference_step(model, spec, x, cap.eps(ldeq, 1), cap.pin())
    _assert_l_hat_agrees(cap.l_hat, ex["l_hat"])
    assert ex["z_hat"].shape == (T, B, 16 + diffeq.augment_dim)
    _compare(f"[LatentODE {config}]", loss, grads, loss_ref, grads_ref, tol)
    print(f"[LatentODE {config}] wall {time.perf_counter() - t0:.1f} s")


def test_train_step_applies_flux_adamw_to_the_bucket(ldeq, exact_fp32):
    x = _frames()
    model = _model(ldeq, ldeq.GOKU_basic(), ldeq.Pendulum(), x, variational=False)
    twin = copy.deepcopy(model)
    flat = ldeq.FlatParams(model)
    opt = ldeq.ADAMW(flat, 1e-3, (0.9, 0.999), 1e-3)
    flat.zero_grad()
    ldeq.loss_batch(model, x, T_GRID, BETA, False, unit_cotangent=True).backward()
    # every gradient autograd wrote is a view of the one bucket the optimiser reads
    lo, hi = flat.grad.data_ptr(), flat.grad.data_ptr() + flat.grad.numel() * flat.grad.element_size()
    for n, p in model.named_parameters():
        assert p.grad is not None and p.grad.untyped_storage().data_ptr() == flat.grad.untyped_storage().data_ptr(), n
        assert lo <= p.grad.data_ptr() and p.grad.data_ptr() + p.grad.numel() * 4 <= hi, n
    names = [n for n, _ in model.named_parameters()]
    before = [p.detach().cpu().numpy().copy() for p in flat.params]
    grads = [p.grad.detach().cpu().numpy().copy() for p in flat.params]
    opt.step()
    ref = ol.ADAMW(1e-3, (0.9, 0.999), np.float32(1e-3))
    for n, p, x0, g in zip(names, flat.params, before, grads):
        want = ref.update(n, x0.copy(), g)
        got = p.detach().cpu().numpy()
        assert np.abs(got - want).max() <= 2e-7 * np.abs(want).max(), n
        assert not np.array_equal(got, x0), n
    # train_step on an identical model: the same update, bit for bit
    flat2 = ldeq.FlatParams(twin)
    ldeq.train_step(twin, flat2, ldeq.ADAMW(flat2, 1e-3, (0.9, 0.999), 1e-3), x, T_GRID, BETA, variational=False)
    assert torch.equal(flat2.flat, flat.flat)


def test_sharded_batch_equals_full_batch(ldeq, exact_fp32):
    # the data-parallel layout on one GPU: ragged shards, each differentiated with grad_scale = B_r / B into one bucket,
    # against the full batch
    x = _frames()
    model = _model(ldeq, ldeq.GOKU_basic(), ldeq.Pendulum(), x, variational=False)
    flat = ldeq.FlatParams(model)
    flat.zero_grad()
    loss_sh = 0.0
    for r in range(3):
        lo, hi = ldeq.shard_bounds(B, r, 3)
        gs = (hi - lo) / B
        loss = ldeq.loss_batch(model, x[:, lo:hi], T_GRID, BETA, False, unit_cotangent=True, grad_scale=gs)
        loss.backward()
        loss_sh += gs * float(loss)
    sharded = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
    flat.zero_grad()
    loss_full = ldeq.loss_batch(model, x, T_GRID, BETA, False, unit_cotangent=True)
    loss_full.backward()
    print(f"sharded loss {loss_sh:.8e} full {float(loss_full):.8e}")
    assert abs(loss_sh - float(loss_full)) <= 1e-6 * abs(float(loss_full))
    for n, p in model.named_parameters():
        err = float((sharded[n] - p.grad).abs().max())
        print(f"[sharded] {n:52s} max|g| {float(p.grad.abs().max()):.3e}  max err {err:.3e}")
        assert err <= 2e-5 * float(p.grad.abs().max()), n
