"""The reference's public API on the CUDA path: LatentDiffEqModel / default_layers / diffeq structs / loss_batch /
one ADAMW step (examples/pendulum_friction-less/model_train.jl)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _frames(T, B, seed=0):
    return torch.rand(T, B, 784, generator=torch.Generator().manual_seed(seed)).to(DEV)


def test_goku_tutorial_step(ldeq):
    # C1: GOKU-net friction-less pendulum tutorial shape, batch 64, 50-step series
    torch.manual_seed(333)
    mt = ldeq.GOKU_basic()
    enc, dec = ldeq.default_layers(mt, 784, ldeq.Pendulum(), device=DEV)
    model = ldeq.LatentDiffEqModel(mt, enc, dec)
    assert sum(p.numel() for p in model.parameters()) == 503387
    x = _frames(50, 64)
    t = np.arange(50) * 0.05
    (xh, zh, lh), mu, lv = model(x, t, True)
    assert xh.shape == (50, 64, 784) and zh.shape == (50, 64, 2) and lh[0].shape == (64, 2) and lh[1].shape == (64, 1)
    assert torch.isfinite(xh).all() and (lh[1] > 0).all()   # softplus keeps the pendulum length positive
    flat = ldeq.FlatParams(model)
    opt = ldeq.ADAMW(flat, 1e-3, (0.9, 0.999), 1e-3)
    losses = [float(ldeq.train_step(model, flat, opt, x, t, beta=0.5, variational=True)) for _ in range(5)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    # the fused ELBO equals the reference expression evaluated with torch ops
    with torch.no_grad():
        (xh, zh, lh), mu, lv = model(x, t, False)
        ref = ((x - xh) ** 2).mean(dim=(0, 1)).sum() + 0.5 * ldeq.vector_kl(mu, lv)
        got = ldeq.elbo_loss(x, xh, mu, lv, 0.5)
        assert abs(float(ref) - float(got)) <= 1e-5 * abs(float(ref))


def test_goku_gradients_flow_through_the_solve(ldeq):
    torch.manual_seed(1)
    mt = ldeq.GOKU_basic()
    enc, dec = ldeq.default_layers(mt, 784, ldeq.Pendulum_friction(abstol=1e-8, reltol=1e-8), device=DEV)
    model = ldeq.LatentDiffEqModel(mt, enc, dec).double()
    x = _frames(20, 8).double()
    t = np.arange(20) * 0.05
    (xh, zh, lh), mu, lv = model(x, t, False)
    zh.sum().backward()
    g = [p.grad for p in model.decoder.latent_out.parameters()]
    assert all(gi is not None and torch.isfinite(gi).all() and gi.abs().sum() > 0 for gi in g)


def test_latentode_step(ldeq):
    torch.manual_seed(1)
    mt = ldeq.LatentODE()
    node = ldeq.NODE(16)
    enc, dec = ldeq.default_layers(mt, 784, node, device=DEV)
    model = ldeq.LatentDiffEqModel(mt, enc, dec)
    x = _frames(50, 32)
    t = np.arange(50) * 0.05
    (xh, zh, z0), mu, lv = model(x, t, True)
    assert xh.shape == (50, 32, 784) and zh.shape == (50, 32, 16)
    loss = ldeq.loss_batch(model, x, t, 1.0, True)
    loss.backward()
    assert all(w.grad is not None and torch.isfinite(w.grad).all() and w.grad.abs().sum() > 0 for w in node.weights)
    # augmented neural ODE: zero-padded extra state rows (LatentODE.jl:71)
    node2 = ldeq.NODE(16, augment_dim=2)
    enc, dec = ldeq.default_layers(mt, 784, node2, device=DEV)
    model2 = ldeq.LatentDiffEqModel(mt, enc, dec)
    (xh, zh, z0), mu, lv = model2(x, t, False)
    assert zh.shape == (50, 32, 18) and torch.isfinite(xh).all()


def test_cpu_tensors_are_refused(ldeq):
    with pytest.raises(RuntimeError):
        ldeq.goku_solve(torch.zeros(4, 2), torch.ones(4, 1), np.arange(5) * 0.05)


def test_fused_recurrent_layers_equal_the_per_step_flux_loops(ldeq, monkeypatch):
    # the cuDNN route of the pattern extractor must be the same function (values and gradients) as the Flux-style loops
    from importlib import import_module
    model_mod = import_module("latentdiffeq_jl_b200.model")
    torch.manual_seed(3)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)   # restored when the test ends
    mt = ldeq.GOKU_basic()
    enc, dec = ldeq.default_layers(mt, 784, ldeq.Pendulum(), device=DEV)
    encoder = ldeq.Encoder(mt, enc)
    for p in encoder.parameters():           # non-trivial biases / initial states
        if p.dim() == 1:
            p.data.add_(0.05 * torch.randn_like(p))
    x = torch.rand(30, 16, 784, device=DEV)
    outs = {}
    for fuse in (True, False):
        monkeypatch.setattr(model_mod, "FUSE_RECURRENT", fuse)
        encoder.zero_grad()
        mu, lv = encoder(x)
        (mu[0].square().sum() + mu[1].sum() + lv[0].sum() + lv[1].square().sum()).backward()
        outs[fuse] = ([m.detach().clone() for m in mu + lv], [p.grad.detach().clone() for p in encoder.parameters()])
    for a, b in zip(outs[True][0], outs[False][0]):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6)
    for a, b in zip(outs[True][1], outs[False][1]):
        assert torch.allclose(a, b, rtol=2e-3, atol=1e-5)
