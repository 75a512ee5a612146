"""CUDA graph capture of the GOKU training step (``GraphedTrainStep``) and of the capture-safe library entry points.

The device-state entry points (``ldeq_adamw_step_dev``, ``ldeq_sample_dev``, ``ldeq_elbo*_dev``) must equal the host-value
ones bit for bit; every capture-safe entry point replayed from a graph with new inputs must equal its eager call; a graph
keeps integrating on the grid it captured after an eager call on another grid; a graphed training step must equal the
eager ``train_step`` bit for bit; and everything that needs the host is refused under capture without breaking it."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, T, P_IN = 64, 50, 784
T_GRID = 0.05 * np.arange(T)
T_VAL = 0.05 * np.arange(100)
PENDULUM_SRC = r"""
template <class S> __device__ void ldeq_user_rhs(S* du, const S* u, const S* p, S t) {
    du[0] = u[1];
    du[1] = -S(10.0f) / p[0] * sin(u[0]);
}
"""


def _bits_equal(a, b):
    """Bitwise equality (NaN payloads included) of two tensors of the same dtype."""
    if a.dtype.is_floating_point:
        view = {torch.float32: torch.int32, torch.float64: torch.int64}[a.dtype]
        a, b = a.contiguous().view(view), b.contiguous().view(view)
    return a.shape == b.shape and torch.equal(a, b)


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _pendulum_inputs(seed, n=B):
    g = _gen(seed)
    z0 = torch.stack([(torch.rand(n, generator=g, device=DEV) - 0.5) * (np.pi / 3),
                      (torch.rand(n, generator=g, device=DEV) - 0.5) * (2 * np.pi / 3)], 1)
    th = 1.0 + torch.rand(n, 1, generator=g, device=DEV)
    return z0, th


def _capture(fn):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def _model(ldeq, seed, diffeq=None, **layer_kw):
    torch.manual_seed(seed)
    diffeq = diffeq or ldeq.Pendulum()
    mt = ldeq.LatentODE() if isinstance(diffeq, ldeq.NODE) else ldeq.GOKU_basic()
    enc, dec = ldeq.default_layers(mt, P_IN, diffeq, device=DEV, **layer_kw)
    model = ldeq.LatentDiffEqModel(mt, enc, dec)
    flat = ldeq.FlatParams(model)
    return model, flat, ldeq.ADAMW(flat, 1e-3, (0.9, 0.999), 1e-3)


def _frames(seed, b=B, t=T):
    return torch.rand(t, b, P_IN, generator=_gen(seed), device=DEV)


# ---- 1. device-state entry points equal the host-value ones ----------------------------------------------------------
def test_adamw_step_dev_equals_host_step(ldeq):
    n = 1_000_003                       # not a multiple of 4: the tail path too
    g = _gen(1)
    x = torch.randn(n, generator=g, device=DEV)
    bufs_h = [x.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)]
    bufs_d = [x.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)]
    state = ldeq.adamw_state(0, device=DEV)
    for k in range(1, 7):
        grad = torch.randn(n, generator=g, device=DEV)
        ldeq.adamw_step(bufs_h[0], grad, bufs_h[1], bufs_h[2], k, 1e-3, (0.9, 0.999), 1e-8, 1e-3, 0.5)
        ldeq.adamw_step_dev(bufs_d[0], grad, bufs_d[1], bufs_d[2], state, 1e-3, (0.9, 0.999), 1e-8, 1e-3, 0.5)
        for a, b in zip(bufs_h, bufs_d):
            assert _bits_equal(a, b), k
    assert _bits_equal(state.cpu(), ldeq.adamw_state(6))
    assert int(state.cpu().view(torch.int64)[0]) == 6


@pytest.mark.parametrize("n", [1024, 1003])
def test_sample_dev_equals_sample_at_the_same_offset(ldeq, n):
    g = _gen(2)
    mu, lv = torch.randn(n, generator=g, device=DEV), torch.randn(n, generator=g, device=DEV) * 0.3
    for c0 in (0, 7, 2**31 + 5):
        calls = torch.tensor([c0], dtype=torch.int64, device=DEV)
        z_d, e_d = ldeq.sample_raw(mu, lv, 1234, calls=calls)
        z_h, e_h = ldeq.sample_raw(mu, lv, 1234, (c0 + 1) << 32)
        assert _bits_equal(z_d, z_h) and _bits_equal(e_d, e_h)
        assert int(calls.item()) == c0 + 1


def test_model_sample_with_a_device_counter_draws_the_eager_noise_for_both_heads(ldeq):
    from importlib import import_module
    M = import_module("latentdiffeq_jl_b200.model")
    g = _gen(3)
    mu = (torch.randn(B, 16, generator=g, device=DEV), torch.randn(B, 16, generator=g, device=DEV))
    lv = (torch.randn(B, 16, generator=g, device=DEV) * 0.2, torch.randn(B, 16, generator=g, device=DEV) * 0.2)
    c0 = M._sample_calls
    eager = ldeq.sample(mu, lv, None, seed=99)
    M._sample_calls = c0
    calls = torch.tensor([c0], dtype=torch.int64, device=DEV)
    with ldeq.device_sample_counter(calls):
        dev = ldeq.sample(mu, lv, None, seed=99)
    assert M._sample_calls == c0 + 2 and int(calls.item()) == c0 + 2
    for a, b in zip(eager, dev):
        assert _bits_equal(a, b)


@pytest.mark.parametrize("logits", [False, True])
def test_elbo_dev_equals_host_beta(ldeq, logits):
    g = _gen(4)
    x = torch.rand(T, B, P_IN, generator=g, device=DEV)
    xh = torch.randn(T, B, P_IN, generator=g, device=DEV)
    mus = [torch.randn(B, 2, generator=g, device=DEV), torch.randn(B, 1, generator=g, device=DEV)]
    lvs = [torch.randn(B, 2, generator=g, device=DEV) * 0.1, torch.randn(B, 1, generator=g, device=DEV) * 0.1]
    for beta in (0.0, 0.37, 1.0, 3.3e-3, 0.7123456789):
        ref = ldeq.elbo_raw(x, xh, mus, lvs, beta, grad_scale=0.25, logits=logits)
        dev = ldeq.elbo_raw(x, xh, mus, lvs, torch.tensor(beta, dtype=torch.float32, device=DEV), grad_scale=0.25, logits=logits)
        assert _bits_equal(ref[0], dev[0]) and _bits_equal(ref[1], dev[1]), beta
        for a, b in zip(ref[2] + ref[3], dev[2] + dev[3]):
            assert _bits_equal(a, b), beta


# ---- 2. capture-safe entry points replayed from a graph -----------------------------------------------------------------
@pytest.mark.parametrize("rhs_kind", ["builtin", "nvrtc"])
@pytest.mark.parametrize("adaptive", [True, False])
def test_goku_solve_and_forward_dual_pullback_replay(ldeq, rhs_kind, adaptive):
    rhs = ldeq.RHS_PENDULUM if rhs_kind == "builtin" else ldeq.handle(0).rhs_from_source(PENDULUM_SRC, 2, 1)
    opts = ldeq.default_opts() if adaptive else ldeq.default_opts(adaptive=False, dt=0.01)
    z0, th = _pendulum_inputs(10)
    dtraj = torch.randn(T, B, 2, generator=_gen(11), device=DEV)

    def run():
        traj, st, tape = ldeq.goku_solve_raw(z0, th, T_GRID, rhs, opts, want_tape=True)
        dz0, dth = ldeq.goku_bwd_raw(tape, dtraj)
        tape.free()
        return traj, st.naccept, st.retcode, dz0, dth

    run()                                     # eager: the grid reaches the device
    graph, outs = _capture(run)
    for k in range(3):
        z, p = _pendulum_inputs(20 + k)
        z0.copy_(z); th.copy_(p)
        dtraj.copy_(torch.randn(T, B, 2, generator=_gen(30 + k), device=DEV))
        graph.replay()
        ref = run()
        for a, b in zip(outs, ref):
            assert _bits_equal(a, b), k
    assert (outs[2] == 0).all()


def test_pattern_extractor_forward_and_reverse_replay(ldeq):
    model, _, _ = _model(ldeq, 5)
    pe = model.encoder.pattern_extractor
    params = [p for p in pe.parameters()]
    x = torch.randn(T, B, 32, generator=_gen(6), device=DEV)
    w0, w1 = torch.randn(B, 16, generator=_gen(7), device=DEV), torch.randn(B, 32, generator=_gen(8), device=DEV)

    def run():
        xs = x.detach().requires_grad_(True)
        z0, th = ldeq.pattern_extractor(xs, list(pe[0]), list(pe[1]), list(pe[2]))
        grads = torch.autograd.grad((z0 * w0).sum() + (th * w1).sum(), [xs, *params])
        return (z0.detach(), th.detach(), *grads)

    run()
    graph, outs = _capture(run)
    for k in range(3):
        x.copy_(torch.randn(T, B, 32, generator=_gen(40 + k), device=DEV))
        graph.replay()
        ref = run()
        for a, b in zip(outs, ref):
            assert _bits_equal(a, b), k


def test_sample_elbo_and_adamw_replay_with_new_values(ldeq):
    """sample_dev -> ELBO with a device beta -> AdamW with a device step, captured once; every replay equals the host-value
    calls of the next step at the next sample offsets."""
    g = _gen(9)
    mu = torch.randn(B, 16, generator=g, device=DEV)
    lv = torch.randn(B, 16, generator=g, device=DEV) * 0.2
    x = torch.rand(T, B, P_IN, generator=g, device=DEV)
    logits = torch.randn(T, B, P_IN, generator=g, device=DEV)
    n = 4099
    p0 = torch.randn(n, generator=g, device=DEV)
    grads = torch.randn(n, generator=g, device=DEV)
    calls = torch.zeros(1, dtype=torch.int64, device=DEV)
    beta = torch.zeros((), dtype=torch.float32, device=DEV)
    state = ldeq.adamw_state(0, device=DEV)
    pd, md, vd = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    ph, mh, vh = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)

    def body():
        z, _ = ldeq.sample_raw(mu, lv, 77, calls=calls)
        loss, dlog, dmu, dlv = ldeq.elbo_raw(x, logits, [z], [lv], beta, logits=True)
        ldeq.adamw_step_dev(pd, grads, md, vd, state)
        return z, loss, dlog, dmu[0], dlv[0]

    body()                                   # eager: workspaces exist before the capture
    ldeq.adamw_step(ph, grads, mh, vh, 1)
    graph, outs = _capture(body)
    for k in range(3):
        b = 0.1 + 0.3 * k
        beta.fill_(b)
        mu.add_(0.01)
        graph.replay()
        z, _ = ldeq.sample_raw(mu, lv, 77, (k + 2) << 32)
        ref = ldeq.elbo_raw(x, logits, [z], [lv], b, logits=True)
        ldeq.adamw_step(ph, grads, mh, vh, k + 2)
        assert _bits_equal(outs[0], z) and _bits_equal(outs[1], ref[0]) and _bits_equal(outs[2], ref[1]), k
        assert _bits_equal(outs[3], ref[2][0]) and _bits_equal(outs[4], ref[3][0]), k
        for a, c in ((pd, ph), (md, mh), (vd, vh)):
            assert _bits_equal(a, c), k
    assert int(calls.item()) == 4


# ---- 3. the grid a graph captured survives eager calls on another grid ----------------------------------------------------
def test_replay_keeps_the_captured_grid_after_an_eager_solve_on_another(ldeq):
    z0, th = _pendulum_inputs(12)
    run = lambda t: ldeq.goku_solve_raw(z0, th, t, ldeq.RHS_PENDULUM)[0]
    run(T_GRID)
    graph, out = _capture(lambda: run(T_GRID))
    graph.replay()
    first = out.clone()
    other = run(0.037 * np.arange(T))             # same length, other values: the eager grid buffer is overwritten
    run(T_VAL)
    graph.replay()
    assert _bits_equal(out, first)
    assert _bits_equal(out, run(T_GRID))
    assert not torch.equal(other, first)


# ---- 4. whole training steps ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("interleave_validation", [False, True])
@pytest.mark.parametrize("diffeq", ["Pendulum", "Pendulum_friction"])
def test_graphed_train_step_equals_eager_train_step(ldeq, diffeq, interleave_validation):
    from importlib import import_module
    M = import_module("latentdiffeq_jl_b200.model")
    K = 6
    xs = [_frames(100 + k) for k in range(K)]
    betas = [0.05 + 0.15 * k for k in range(K)]
    x_val = _frames(200, b=45, t=100)
    c0 = M._sample_calls
    runs = []
    for graphed in (False, True):
        M._sample_calls = c0
        model, flat, opt = _model(ldeq, 21, getattr(ldeq, diffeq)())
        step = ldeq.GraphedTrainStep(model, flat, opt, xs[0], T_GRID) if graphed else None
        losses, vals = [], []
        for k in range(K):
            if graphed:
                losses.append(step(xs[k], betas[k]))
            else:
                losses.append(ldeq.train_step(model, flat, opt, xs[k], T_GRID, betas[k]))
            if interleave_validation:
                with torch.no_grad():
                    vals.append(ldeq.loss_batch(model, x_val, T_VAL, betas[k], False))
        torch.cuda.synchronize()
        runs.append(dict(flat=flat.flat.clone(), m=flat.m.clone(), v=flat.v.clone(), losses=torch.stack(losses), vals=vals,
                         step=opt.step_count, calls=M._sample_calls))
    e, g = runs
    assert g["step"] == e["step"] == K and g["calls"] == e["calls"] == c0 + 2 * K
    assert _bits_equal(e["losses"], g["losses"])
    for key in ("flat", "m", "v"):
        assert _bits_equal(e[key], g[key]), key
    for a, b in zip(e["vals"], g["vals"]):
        assert _bits_equal(a, b)
    assert torch.isfinite(g["losses"]).all() and not torch.equal(runs[1]["flat"], _model(ldeq, 21)[1].flat)


def test_graphed_step_after_eager_steps_continues_the_optimiser_state(ldeq):
    """An eager train_step between replays moves the host mirrors; the next replay starts from them."""
    from importlib import import_module
    M = import_module("latentdiffeq_jl_b200.model")
    xs = [_frames(300 + k) for k in range(4)]
    c0 = M._sample_calls
    out = []
    for graphed in (False, True):
        M._sample_calls = c0
        model, flat, opt = _model(ldeq, 22)
        step = ldeq.GraphedTrainStep(model, flat, opt, xs[0], T_GRID) if graphed else None
        for k, x in enumerate(xs):
            if graphed and k != 1:
                step(x, 0.3)
            else:
                ldeq.train_step(model, flat, opt, x, T_GRID, 0.3)
        out.append((flat.flat.clone(), flat.m.clone(), flat.v.clone(), opt.step_count))
    assert out[0][3] == out[1][3] == 4
    for a, b in zip(out[0][:3], out[1][:3]):
        assert _bits_equal(a, b)


# ---- 5. construction leaves the training state alone --------------------------------------------------------------------
def test_construction_leaves_training_state_untouched(ldeq):
    from importlib import import_module
    M = import_module("latentdiffeq_jl_b200.model")
    model, flat, opt = _model(ldeq, 23)
    ldeq.train_step(model, flat, opt, _frames(400), T_GRID, 0.5)     # non-trivial m, v, grad, step_count
    before = [b.clone() for b in (flat.flat, flat.grad, flat.m, flat.v)]
    step0, calls0 = opt.step_count, M._sample_calls
    ldeq.GraphedTrainStep(model, flat, opt, _frames(401), T_GRID)
    torch.cuda.synchronize()
    for a, b in zip(before, (flat.flat, flat.grad, flat.m, flat.v)):
        assert _bits_equal(a, b)
    assert opt.step_count == step0 and M._sample_calls == calls0


# ---- 6. refusals --------------------------------------------------------------------------------------------------------
def test_graphed_train_step_refuses_what_it_cannot_capture(ldeq):
    x = _frames(500)
    cases = [
        (_model(ldeq, 24, ldeq.NODE(16)), "LatentODE"),
        (_model(ldeq, 24, ldeq.Pendulum(sensalg=ldeq.DiscreteAdjoint())), "ForwardDiffSensitivity"),
        (_model(ldeq, 24, output_activation="identity"), "sigmoid"),
    ]
    for (model, flat, opt), word in cases:
        with pytest.raises(NotImplementedError, match=word):
            ldeq.GraphedTrainStep(model, flat, opt, x, T_GRID)
        assert opt.step_count == 0
    with pytest.raises(RuntimeError, match="CUDA"):
        model, flat, opt = _model(ldeq, 24)
        ldeq.GraphedTrainStep(model, flat, opt, x.cpu(), T_GRID)
    model, flat, opt = _model(ldeq, 24)
    assert torch.isfinite(ldeq.train_step(model, flat, opt, x, T_GRID, 0.5))


def test_host_dependent_entry_points_are_refused_under_capture(ldeq):
    h = ldeq.handle(0)
    z0, th = _pendulum_inputs(13)
    dtraj = torch.randn(T, B, 2, generator=_gen(14), device=DEV)
    ref = ldeq.goku_solve_raw(z0, th, T_GRID, ldeq.RHS_PENDULUM)[0]
    da = ldeq.default_opts(sensealg=ldeq.SENSE_DISCRETE_ADJOINT)
    _, _, da_tape = ldeq.goku_solve_raw(z0, th, T_GRID, ldeq.RHS_PENDULUM, da, want_tape=True)
    _, _, fd_tape = ldeq.goku_solve_raw(z0, th, T_GRID, ldeq.RHS_PENDULUM, want_tape=True)
    dims = [4, 8, 8, 4]
    mz = torch.randn(B, 4, generator=_gen(15), device=DEV) * 0.1
    mp = torch.randn(148, generator=_gen(16), device=DEV) * 0.1
    _, _, mlp_tape = ldeq.mlp_solve_raw(mz, mp, dims, T_GRID, want_tape=True)
    mdtraj = torch.randn(T, B, 4, generator=_gen(17), device=DEV)
    pin = lambda *s: torch.empty(*s, pin_memory=True)
    z_cpu, th_cpu, dtraj_cpu = z0.cpu(), th.cpu(), dtraj.cpu()
    out, dz0, dth = pin(T, B, 2), pin(B, 2), pin(B, 1)
    grad = torch.zeros(1024, device=DEV)
    params, m, v = torch.zeros(1024, device=DEV), torch.zeros(1024, device=DEV), torch.zeros(1024, device=DEV)
    torch.cuda.synchronize()
    refused = {}
    calls = {
        "discrete-adjoint tape": lambda: ldeq.goku_solve_raw(z0, th, T_GRID, ldeq.RHS_PENDULUM, da, want_tape=True),
        "discrete-adjoint pullback": lambda: ldeq.goku_bwd_raw(da_tape, dtraj),
        "tape_overflow": lambda: fd_tape.overflow(),
        "mlp_solve_fwd": lambda: ldeq.mlp_solve_raw(mz, mp, dims, T_GRID),
        "mlp_solve_bwd": lambda: ldeq.mlp_bwd_raw(mlp_tape, mdtraj),
        "solve_fwd_host": lambda: ldeq.goku_solve_host(z_cpu, th_cpu, T_GRID, out=out),
        "solve_bwd_host": lambda: ldeq.goku_bwd_host(fd_tape, dtraj_cpu, dz0=dz0, dtheta=dth),
        "solve_fwd_bwd_host": lambda: ldeq.goku_fwd_bwd_host(z_cpu, th_cpu, T_GRID, dtraj_cpu, out=out, dz0=dz0, dtheta=dth),
        "allreduce_grads": lambda: h.allreduce_grads(grad),
        "allreduce_adamw_step": lambda: ldeq.allreduce_adamw_step(params, [grad.data_ptr()], m, v, 1),
        "new grid": lambda: ldeq.goku_solve_raw(z0, th, 0.011 * np.arange(T), ldeq.RHS_PENDULUM),
    }
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for name, fn in calls.items():
            try:
                fn()
            except ldeq.LdeqError as e:
                refused[name] = (e.code, str(e))
    assert set(refused) == set(calls), set(calls) - set(refused)
    for name, (code, msg) in refused.items():
        assert code == ldeq._cabi.ERR_UNSUPPORTED and "capture" in msg, (name, msg)
    # the capture ended cleanly, eager work is still right, and the tapes made before it still work
    assert _bits_equal(ldeq.goku_solve_raw(z0, th, T_GRID, ldeq.RHS_PENDULUM)[0], ref)
    assert fd_tape.overflow() == 0 and da_tape.overflow() >= 0
    dz, dp = ldeq.goku_bwd_raw(da_tape, dtraj)
    assert torch.isfinite(dz).all() and torch.isfinite(dp).all()
    assert torch.isfinite(ldeq.mlp_bwd_raw(mlp_tape, mdtraj)[0]).all()
    for tp in (da_tape, fd_tape, mlp_tape):
        tp.free()
