"""Pins of the float64 whole-model reference (``oracle/model.py``) on the CPU: its gradient is the derivative of its loss.

Directional derivatives by central differences against ``g . v`` for three seeded random directions through every
parameter at once, in fixed-step mode where the solve's pullback is exact (ForwardDiffSensitivity and the discrete adjoint
are then both the derivative of the primal discretisation).  Tiny dimensions keep each loss evaluation in milliseconds.
No CUDA and no ``libldeq.so``: the models are built on the CPU only for their parameter names and initial values."""
import numpy as np
import pytest
import torch

from oracle import model as rm

T, B, P_IN = 5, 3, 12
TINY = dict(hidden_dim_resnet=8, rnn_input_dim=6)


def _reference(ldeq, model_type, diffeq, seed):
    torch.manual_seed(seed)
    if isinstance(model_type, ldeq.GOKU):
        enc, dec = ldeq.default_layers(model_type, P_IN, diffeq, rnn_output_dim=4, latent_dim_z0=3, latent_dim_theta=3,
                                       latent_to_diffeq_dim=8, **TINY)
    else:
        enc, dec = ldeq.default_layers(model_type, P_IN, diffeq, rnn_output_dim=5, **TINY)
    model = ldeq.LatentDiffEqModel(model_type, enc, dec)
    P = rm.params_from(model.named_parameters())
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():      # non-trivial biases and initial states, so that every parameter has a gradient
        for p in P.values():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, generator=gen, dtype=torch.float64))
    x = torch.rand(T, B, P_IN, generator=gen, dtype=torch.float64)
    return P, x, rm.spec_from_diffeq(diffeq)


def _check_directional_derivatives(P, spec, x, eps, beta=0.5, h=1e-5):
    t = 0.05 * np.arange(T)
    loss, _ = rm.loss_batch(P, spec, x, t, beta, eps)
    loss.backward()
    missing = [n for n, p in P.items() if p.grad is None or not p.grad.abs().sum() > 0]
    assert not missing, f"the reference leaves these parameters without a gradient: {missing}"
    rng = torch.Generator().manual_seed(7)
    for k in range(3):
        v = {n: torch.randn(p.shape, generator=rng, dtype=torch.float64) for n, p in P.items()}
        gv = sum(float((P[n].grad * v[n]).sum()) for n in P)
        with torch.no_grad():
            lp = float(rm.loss_batch({n: P[n] + h * v[n] for n in P}, spec, x, t, beta, eps)[0])
            lm = float(rm.loss_batch({n: P[n] - h * v[n] for n in P}, spec, x, t, beta, eps)[0])
        fd = (lp - lm) / (2 * h)
        print(f"direction {k}: g.v {gv:.12e}  central difference {fd:.12e}  rel {abs(fd - gv) / abs(gv):.2e}")
        assert abs(fd - gv) <= 1e-6 * abs(gv)


@pytest.mark.parametrize("rhs,sensalg", [("Pendulum", "ForwardDiffSensitivity"), ("Pendulum_friction", "DiscreteAdjoint")])
def test_goku_reference_gradient_is_the_derivative_of_its_loss(ldeq, rhs, sensalg):
    diffeq = getattr(ldeq, rhs)(sensalg=getattr(ldeq, sensalg)(), adaptive=False, dt=0.01)
    P, x, spec = _reference(ldeq, ldeq.GOKU_basic(), diffeq, seed=11)
    assert spec.kind == rm.GOKU and spec.sensealg == {"ForwardDiffSensitivity": "forward_dual", "DiscreteAdjoint": "discrete"}[sensalg]
    eps = tuple(torch.randn(B, 3, generator=torch.Generator().manual_seed(3 + i), dtype=torch.float64) for i in range(2))
    _check_directional_derivatives(P, spec, x, eps)


@pytest.mark.parametrize("augment_dim", [0, 2])
def test_latentode_reference_gradient_is_the_derivative_of_its_loss(ldeq, augment_dim):
    diffeq = ldeq.NODE(4, hidden_dim=8, augment_dim=augment_dim, sensealg=ldeq.DiscreteAdjoint(), adaptive=False, dt=0.02)
    P, x, spec = _reference(ldeq, ldeq.LatentODE(), diffeq, seed=12)
    assert spec.kind == rm.LATENTODE and spec.dims == [4 + augment_dim, 8, 8, 4 + augment_dim]
    eps = torch.randn(B, 4, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    _check_directional_derivatives(P, spec, x, eps)


def test_reference_pattern_extractor_equals_the_recurrent_oracle(ldeq):
    # the whole-model reference and oracle/recurrent.py restate the same stacks independently (named tensors here, the
    # flat Flux.destructure vectors there): same final states, so the z0 / theta halves and the stack order agree
    from oracle import recurrent as orc
    P, x, _ = _reference(ldeq, ldeq.GOKU_basic(), ldeq.Pendulum(), seed=13)
    fe = rm.resnet(P, "encoder.feature_extractor", x, torch.relu)
    pre = "encoder.pattern_extractor.layers"

    def flat(i, lstm):
        parts = []
        for l in (f"{pre}.{i}.0", f"{pre}.{i}.1"):
            parts += [P[l + ".Wi"].t().reshape(-1), P[l + ".Wh"].t().reshape(-1), P[l + ".b"]]
            parts += [P[l + ".h0"], P[l + ".c0"]] if lstm else [P[l + ".state0"]]
        return torch.cat(parts).detach()
    with torch.no_grad():
        z0 = rm.recurrent_final(P, pre + ".0", fe, reverse=True)
        th = torch.cat([rm.recurrent_final(P, pre + ".1", fe, False), rm.recurrent_final(P, pre + ".2", fe, True)], 1)
        oz, oth = orc.pattern_extractor(fe.numpy(), flat(0, False).numpy(), flat(1, True).numpy(), flat(2, True).numpy(), H=4)
    assert np.allclose(z0.numpy(), oz, rtol=1e-12, atol=1e-14) and np.allclose(th.numpy(), oth, rtol=1e-12, atol=1e-14)
