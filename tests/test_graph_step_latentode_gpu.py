"""CUDA graph capture of the LatentODE training step: ``ldeq_mlp_solve_fwd_dev`` and its device-checked tape.

The ``_dev`` forward plus pullback must equal ``ldeq_mlp_solve_fwd`` plus pullback bit for bit on every kernel path; a graph
of them replayed with new inputs must equal the eager calls and keep integrating on its own grid; a tape that overflows
must give NaN gradients and a sticky overflow word instead of an error; a graphed LatentODE training step must equal the
eager ``train_step`` bit for bit; and what still needs the host is refused under capture without breaking it."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, T, P_IN = 64, 50, 784
DIMS = [16, 200, 200, 16]
T_GRID = 0.05 * np.arange(T)
T_VAL = 0.05 * np.arange(100)
T_OTHER = 0.037 * np.arange(T)       # same length, other values: overwrites the handle's eager grid buffer


def _bits_equal(a, b):
    """Bitwise equality (NaN payloads included) of two tensors of the same dtype."""
    if a.dtype.is_floating_point:
        view = {torch.float32: torch.int32, torch.float64: torch.int64}[a.dtype]
        a, b = a.contiguous().view(view), b.contiguous().view(view)
    return a.shape == b.shape and torch.equal(a, b)


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _capture(fn):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def _flag():
    return torch.zeros(1, dtype=torch.int32, device=DEV)


# ---- solve-level inputs ------------------------------------------------------------------------------------------------
PATHS = {
    # name: (opts kwargs, dtype, LDEQ_MLP_NO_RESIDENT, batch)
    "resident_global": (dict(), torch.float32, False, B),
    "exact_global": (dict(), torch.float32, True, B),        # the general kernels, cooperative mlp_fwd_kernel<..., true>
    "per_traj": (dict(norm_mode=1), torch.float32, False, B),
    "fixed_step": (dict(adaptive=0, dt=0.01), torch.float32, False, B),
    # two tiles of 128 trajectories: the reverse pass's step records of the second tile start one stride after the first's
    "bf16x3": (dict(mlp_math=1), torch.float32, False, 256),
    "fp64": (dict(), torch.float64, False, B),
}


def _opts(ldeq, **kw):
    return ldeq.default_opts(sensealg=ldeq.SENSE_DISCRETE_ADJOINT, **kw)


def _params(ldeq, seed, dtype=torch.float32, scale=1.0):
    torch.manual_seed(seed)
    node = ldeq.NODE(16)
    with torch.no_grad():
        p = node.flat_params().to(DEV, dtype)
    return p * scale


def _inputs(seed, dtype=torch.float32, n=B):
    g = _gen(seed)
    z0 = (torch.randn(n, 16, generator=g, device=DEV) * 0.5).to(dtype)
    dtraj = torch.randn(T, n, 16, generator=g, device=DEV).to(dtype)
    return z0, dtraj


def _path(ldeq, monkeypatch, name):
    kw, dtype, no_res, n = PATHS[name]
    if no_res:
        monkeypatch.setenv("LDEQ_MLP_NO_RESIDENT", "1")
    return _opts(ldeq, **kw), dtype, n


def _eager(ldeq, z0, p, dtraj, opts, t=T_GRID):
    traj, st, tape = ldeq.mlp_solve_raw(z0, p, DIMS, t, opts, want_tape=True)
    dz0, dp = ldeq.mlp_bwd_raw(tape, dtraj)
    tape.free()
    return traj, st.retcode, st.naccept, st.nreject, dz0, dp


def _dev(ldeq, z0, p, dtraj, opts, flag, t=T_GRID):
    traj, st, tape = ldeq.mlp_solve_raw(z0, p, DIMS, t, opts, want_tape=True, overflow=flag)
    dz0, dp = ldeq.mlp_bwd_raw(tape, dtraj)
    tape.free()
    return traj, st.retcode, st.naccept, st.nreject, dz0, dp


# ---- a. the _dev twin equals the eager entry point ---------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS))
def test_dev_solve_and_pullback_equal_the_eager_tape(ldeq, monkeypatch, path):
    opts, dtype, n = _path(ldeq, monkeypatch, path)
    p = _params(ldeq, 1, dtype)
    z0, dtraj = _inputs(2, dtype, n)
    flag = _flag()
    ref = _eager(ldeq, z0, p, dtraj, opts)
    out = _dev(ldeq, z0, p, dtraj, opts, flag)
    names = ("traj", "retcode", "naccept", "nreject", "dz0", "dparams")
    for name, a, b in zip(names, ref, out):
        assert _bits_equal(a, b), (path, name)
    assert (out[1] == 0).all() and torch.isfinite(out[5]).all() and int(flag.item()) == 0
    assert int(out[2].max()) > 3


# ---- b. a captured _dev solve + pullback replays like the eager calls, on its own grid ------------------------------------------
@pytest.mark.parametrize("path", ["resident_global", "exact_global", "per_traj", "bf16x3"])
def test_dev_solve_and_pullback_replay_on_the_captured_grid(ldeq, monkeypatch, path):
    opts, dtype, n = _path(ldeq, monkeypatch, path)
    p = _params(ldeq, 3, dtype)
    z0, dtraj = _inputs(4, dtype, n)
    flag = _flag()
    run = lambda: _dev(ldeq, z0, p, dtraj, opts, flag)
    run()                                      # eager: the grid reaches the device, the scratch is sized
    graph, outs = _capture(run)
    for k in range(2):
        z, d = _inputs(10 + k, dtype, n)
        z0.copy_(z)
        dtraj.copy_(d)
        p.copy_(_params(ldeq, 20 + k, dtype, scale=1.0 + 0.25 * k))
        graph.replay()
        ref = _eager(ldeq, z0, p, dtraj, opts)
        for i, (a, b) in enumerate(zip(outs, ref)):
            assert _bits_equal(a, b), (path, k, i)
        other = ldeq.mlp_solve_raw(z0, p, DIMS, T_OTHER, opts)[0]
        assert not torch.equal(other, ref[0])
    assert int(flag.item()) == 0


# ---- c. overflow: NaN gradients and a sticky overflow word ----------------------------------------------------------------------
@pytest.mark.parametrize("path", ["resident_global", "exact_global", "per_traj", "bf16x3"])
def test_overflowing_device_checked_tape(ldeq, monkeypatch, path):
    opts, dtype, n = _path(ldeq, monkeypatch, path)
    z0, dtraj = _inputs(5, dtype, n)
    p_small, p_big = _params(ldeq, 6, dtype), _params(ldeq, 6, dtype, scale=3.0)
    na_small = int(ldeq.mlp_solve_raw(z0, p_small, DIMS, T_GRID, opts)[1].naccept.max())
    st_big = ldeq.mlp_solve_raw(z0, p_big, DIMS, T_GRID, opts)[1]
    n_big = int(st_big.naccept[st_big.retcode == 0].max())
    assert n_big > na_small, (n_big, na_small)
    opts.tape_steps = na_small                 # the small parameters fit, the big ones overflow
    over_rows = (st_big.retcode == 0) & (st_big.naccept > na_small)

    # the eager tape refuses the pullback and names the count
    _, _, tape = ldeq.mlp_solve_raw(z0, p_big, DIMS, T_GRID, opts, want_tape=True)
    with pytest.raises(ldeq.LdeqError) as err:
        ldeq.mlp_bwd_raw(tape, dtraj)
    assert err.value.code == ldeq._cabi.ERR_TAPE_OVERFLOW and str(n_big) in str(err.value)
    tape.free()

    def check(out, flag):
        dz0, dp = out[4], out[5]
        assert torch.isnan(dp).all()
        nan_rows = torch.isnan(dz0).any(1)
        assert torch.equal(nan_rows, over_rows) and torch.equal(torch.isnan(dz0).all(1), over_rows)
        assert torch.isfinite(dz0[~over_rows]).all()
        assert int(flag.item()) == n_big

    flag = _flag()
    check(_dev(ldeq, z0, p_big, dtraj, opts, flag), flag)
    # replayed: overflowing, then within the tape (the word stays), then cleared
    p = p_small.clone()
    flag.fill_(0)
    _dev(ldeq, z0, p, dtraj, opts, flag)       # eager warm-up within the tape
    graph, outs = _capture(lambda: _dev(ldeq, z0, p, dtraj, opts, flag))
    p.copy_(p_big)
    graph.replay()
    check(outs, flag)
    p.copy_(p_small)
    graph.replay()
    ref = _eager(ldeq, z0, p_small, dtraj, opts)
    for a, b in zip(outs, ref):
        assert _bits_equal(a, b)
    assert int(flag.item()) == n_big           # sticky
    flag.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert int(flag.item()) == 0 and torch.isfinite(outs[5]).all()


# ---- d. whole training steps ------------------------------------------------------------------------------------------------------
def _model(ldeq, seed, make_node):
    torch.manual_seed(seed)             # the NODE's weights too: it is built after the seed
    mt = ldeq.LatentODE()
    enc, dec = ldeq.default_layers(mt, P_IN, make_node(ldeq), device=DEV)
    model = ldeq.LatentDiffEqModel(mt, enc, dec)
    flat = ldeq.FlatParams(model)
    return model, flat, ldeq.ADAMW(flat, 1e-3, (0.9, 0.999), 1e-3)


def _frames(seed, b=B, t=T):
    return torch.rand(t, b, P_IN, generator=_gen(seed), device=DEV)


NODES = {
    "discrete_adjoint": lambda ldeq: ldeq.NODE(16, sensealg=ldeq.DiscreteAdjoint()),
    "augmented": lambda ldeq: ldeq.NODE(16, augment_dim=2, sensealg=ldeq.DiscreteAdjoint()),
    "per_traj_norm": lambda ldeq: ldeq.NODE(16, norm_mode=1),
    "bf16x3": lambda ldeq: ldeq.NODE(16, mlp_math=1),
    "fixed_step": lambda ldeq: ldeq.NODE(16, sensealg=ldeq.DiscreteAdjoint(), adaptive=False, dt=0.05),
}


@pytest.mark.parametrize("node", list(NODES))
def test_graphed_latentode_step_equals_eager_train_step(ldeq, node):
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
        model, flat, opt = _model(ldeq, 21, NODES[node])
        step = ldeq.GraphedTrainStep(model, flat, opt, xs[0], T_GRID) if graphed else None
        losses, vals = [], []
        for k in range(K):
            if graphed:
                losses.append(step(xs[k], betas[k]))
            else:
                losses.append(ldeq.train_step(model, flat, opt, xs[k], T_GRID, betas[k]))
            with torch.no_grad():
                vals.append(ldeq.loss_batch(model, x_val, T_VAL, betas[k], False))
        torch.cuda.synchronize()
        runs.append(dict(flat=flat.flat.clone(), grad=flat.grad.clone(), m=flat.m.clone(), v=flat.v.clone(),
                         losses=torch.stack(losses), vals=vals, step=opt.step_count, calls=M._sample_calls,
                         overflow=step.tape_overflow() if graphed else 0))
    e, g = runs
    assert g["step"] == e["step"] == K and g["calls"] == e["calls"]
    assert g["overflow"] == 0
    assert _bits_equal(e["losses"], g["losses"])
    for key in ("flat", "grad", "m", "v"):
        assert _bits_equal(e[key], g[key]), key
    for a, b in zip(e["vals"], g["vals"]):
        assert _bits_equal(a, b)
    assert torch.isfinite(g["losses"]).all() and torch.isfinite(g["flat"]).all()
    assert not torch.equal(g["flat"], _model(ldeq, 21, NODES[node])[1].flat)


# ---- e. construction leaves the training state alone --------------------------------------------------------------------------------
def test_latentode_construction_leaves_training_state_untouched(ldeq):
    from importlib import import_module
    M = import_module("latentdiffeq_jl_b200.model")
    model, flat, opt = _model(ldeq, 23, NODES["discrete_adjoint"])
    ldeq.train_step(model, flat, opt, _frames(400), T_GRID, 0.5)     # non-trivial m, v, grad, step_count
    before = [b.clone() for b in (flat.flat, flat.grad, flat.m, flat.v)]
    step0, calls0 = opt.step_count, M._sample_calls
    step = ldeq.GraphedTrainStep(model, flat, opt, _frames(401), T_GRID)
    torch.cuda.synchronize()
    for a, b in zip(before, (flat.flat, flat.grad, flat.m, flat.v)):
        assert _bits_equal(a, b)
    assert opt.step_count == step0 and M._sample_calls == calls0 and step.tape_overflow() == 0


# ---- f. refusals ----------------------------------------------------------------------------------------------------------------------
def test_latentode_refusals(ldeq):
    model, flat, opt = _model(ldeq, 24, lambda ldeq: ldeq.NODE(16))
    with pytest.raises(NotImplementedError, match="InterpolatingAdjoint") as err:
        ldeq.GraphedTrainStep(model, flat, opt, _frames(500), T_GRID)
    assert "LatentODE" in str(err.value) and "DiscreteAdjoint()" in str(err.value) and opt.step_count == 0

    p = _params(ldeq, 7)
    z0, dtraj = _inputs(8)
    flag = _flag()
    da = _opts(ldeq)
    ref = _dev(ldeq, z0, p, dtraj, da, flag)
    ia = ldeq.default_opts(sensealg=ldeq.SENSE_INTERPOLATING_ADJOINT)
    calls = {
        "interpolating-adjoint tape": lambda: ldeq.mlp_solve_raw(z0, p, DIMS, T_GRID, ia, want_tape=True, overflow=flag),
        "new grid": lambda: ldeq.mlp_solve_raw(z0, p, DIMS, 0.013 * np.arange(T), da, overflow=flag),
    }
    refused = {}
    torch.cuda.synchronize()
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
    with pytest.raises(ldeq.LdeqError, match="null|overflow"):
        h = ldeq.handle(0)
        import ctypes as C
        tape = C.c_void_p()
        dims = np.asarray(DIMS, dtype=np.int32)
        tg = np.ascontiguousarray(T_GRID)
        traj = torch.empty(T, B, 16, device=DEV)
        h.check(h._lib.ldeq_mlp_solve_fwd_dev(h.ptr, ldeq.F32, z0.data_ptr(), p.data_ptr(), dims.ctypes.data_as(C.c_void_p), 3,
                                              tg.ctypes.data_as(C.c_void_p), B, T, C.byref(da), traj.data_ptr(), None, None, None,
                                              None, C.byref(tape), torch.cuda.current_stream().cuda_stream))
    # the capture ended cleanly and eager work is still right
    out = _dev(ldeq, z0, p, dtraj, da, flag)
    for a, b in zip(ref, out):
        assert _bits_equal(a, b)
    assert int(flag.item()) == 0
