"""Host-side mirror of the reference's model / layer API above the C ABI.

Same names, argument meaning and composition as the reference:
``LatentDiffEqModel(model_type, encoder_layers, decoder_layers)`` with
``model(x, t, variational=False) -> ((x_hat, z_hat, l_hat), mu, logvar)``
(``src/models/LatentDiffEqModel.jl:16-37``), ``Encoder`` / ``Decoder`` (``:41-113``), the model
types ``GOKU_basic`` / ``LatentODE`` and ``default_layers`` (``src/models/GOKU.jl:199-274``,
``src/models/LatentODE.jl:100-152``), and the overloadable steps ``apply_feature_extractor``,
``apply_pattern_extractor``, ``apply_latent_in``, ``sample``, ``apply_latent_out``,
``diffeq_layer``, ``transform_after_diffeq``, ``apply_reconstructor``.

Only ``diffeq_layer`` and ``sample`` are on the hot path and run in ``libldeq.so``; the dense /
recurrent layers around them are stock PyTorch (out of scope as kernels, SURVEY.md section 8).

Array convention: torch tensors carry the reference's arrays with the dimension order reversed so
the bytes are identical: Julia ``(features, batch, time)`` is torch ``[time, batch, features]``.
"""
from __future__ import annotations

import contextlib
import math

import torch
import torch.nn.functional as F
from torch import nn

from . import _cabi
from .diffeqs import NODE, CudaRHS
from .solve import goku_solve, mlp_solve, sample_reparam, pattern_extractor


# ---- model types (src/models/GOKU.jl:6-7, src/models/LatentODE.jl:7) ------------------------------
class LatentDE:
    pass


class GOKU(LatentDE):
    pass


class GOKU_basic(GOKU):
    pass


class LatentODE(LatentDE):
    pass


# ---- Flux layers the default architecture is made of ---------------------------------------------
def kaiming_uniform_(w: torch.Tensor, gain: float = 1.0 / math.sqrt(3.0)):
    """``Flux.kaiming_uniform(gain = 1/sqrt(3))``: U(+-gain*sqrt(3/fan_in)) (GOKU.jl:204)."""
    fan_in = w.shape[1]
    bound = gain * math.sqrt(3.0 / fan_in)
    with torch.no_grad():
        w.uniform_(-bound, bound)
    return w


_ACT = {"relu": F.relu, "identity": lambda x: x, "softplus": F.softplus, "sigmoid": torch.sigmoid,
        "tanh": torch.tanh}


def _act(a):
    return _ACT[a] if isinstance(a, str) else a


class Dense(nn.Module):
    """``Flux.Dense(in, out, act; init)``: ``act.(W x .+ b)``, zero bias."""

    def __init__(self, fan_in, fan_out, act="identity", init=kaiming_uniform_):
        super().__init__()
        self.weight = nn.Parameter(init(torch.empty(fan_out, fan_in)))
        self.bias = nn.Parameter(torch.zeros(fan_out))
        self.act = _act(act)

    def forward(self, x):
        return self.act(F.linear(x, self.weight, self.bias))


class SkipConnection(nn.Module):
    """``Flux.SkipConnection(layer, +)``."""

    def __init__(self, layer):
        super().__init__()
        self.layer = layer

    def forward(self, x):
        return self.layer(x) + x


class Chain(nn.Sequential):
    """``Flux.Chain``."""


class RNN(nn.Module):
    """``Flux.RNN(in, out, act; init)``: ``h' = act(Wi x + Wh h + b)`` with a trainable ``state0``.
    Applied to a whole sequence ``[T, B, in]``; returns all hidden states ``[T, B, out]``."""

    def __init__(self, fan_in, fan_out, act="relu", init=kaiming_uniform_):
        super().__init__()
        self.Wi = nn.Parameter(init(torch.empty(fan_out, fan_in)))
        self.Wh = nn.Parameter(init(torch.empty(fan_out, fan_out)))
        self.b = nn.Parameter(torch.zeros(fan_out))
        self.state0 = nn.Parameter(torch.zeros(fan_out))
        self.act = _act(act)

    def forward(self, xs):
        pre = F.linear(xs, self.Wi, self.b)  # input projection of every time step at once
        h = self.state0.expand(xs.shape[1], -1)
        out = []
        for k in range(xs.shape[0]):
            h = self.act(pre[k] + F.linear(h, self.Wh))
            out.append(h)
        return torch.stack(out, 0)


class LSTM(nn.Module):
    """``Flux.LSTM(in, out; init)``: gate order input, forget, cell, output; forget-gate bias 1;
    trainable ``state0 = (h, c)``."""

    def __init__(self, fan_in, fan_out, init=kaiming_uniform_):
        super().__init__()
        self.out = fan_out
        self.Wi = nn.Parameter(init(torch.empty(4 * fan_out, fan_in)))
        self.Wh = nn.Parameter(init(torch.empty(4 * fan_out, fan_out)))
        b = torch.zeros(4 * fan_out)
        b[fan_out:2 * fan_out] = 1.0
        self.b = nn.Parameter(b)
        self.h0 = nn.Parameter(torch.zeros(fan_out))
        self.c0 = nn.Parameter(torch.zeros(fan_out))

    def forward(self, xs):
        pre = F.linear(xs, self.Wi, self.b)
        B, o = xs.shape[1], self.out
        h, c = self.h0.expand(B, -1), self.c0.expand(B, -1)
        out = []
        for k in range(xs.shape[0]):
            g = pre[k] + F.linear(h, self.Wh)
            i, f, cell, og = torch.sigmoid(g[:, :o]), torch.sigmoid(g[:, o:2 * o]), torch.tanh(g[:, 2 * o:3 * o]), \
                torch.sigmoid(g[:, 3 * o:])
            c = f * c + i * cell
            h = og * torch.tanh(c)
            out.append(h)
        return torch.stack(out, 0)


def _fused_recurrent(chain, xs):
    """A ``Chain`` of same-width Flux ``RNN(relu)`` or ``LSTM`` layers applied to a CUDA sequence through cuDNN's fused
    multi-layer kernels (one launch per stack instead of ~10 per time step and layer).  Same parameters and arithmetic as
    the per-step loops above: Flux cells have ONE bias, so cuDNN's second bias is a constant zero; the trainable initial
    state ``state0`` is broadcast over the batch.  Returns all hidden states of the last layer ``[T, B, H]``."""
    layers = list(chain)
    B = xs.shape[1]
    flat = []
    for l in layers:
        flat += [l.Wi, l.Wh, l.b, torch.zeros_like(l.b)]
    if isinstance(layers[0], LSTM):
        h0 = torch.stack([l.h0.expand(B, -1) for l in layers]).contiguous()
        c0 = torch.stack([l.c0.expand(B, -1) for l in layers]).contiguous()
        out, _, _ = torch._VF.lstm(xs, (h0, c0), flat, True, len(layers), 0.0, chain.training, False, False)
    else:
        h0 = torch.stack([l.state0.expand(B, -1) for l in layers]).contiguous()
        out, _ = torch._VF.rnn_relu(xs, h0, flat, True, len(layers), 0.0, chain.training, False, False)
    return out


def _can_fuse(chain, xs):
    if not (xs.is_cuda and isinstance(chain, nn.Sequential) and len(chain) > 0 and torch.backends.cudnn.is_available()):
        return False
    layers = list(chain)
    if all(isinstance(l, LSTM) for l in layers):
        return len({l.out for l in layers}) == 1
    if all(isinstance(l, RNN) and l.act is F.relu for l in layers):
        return len({l.Wh.shape[0] for l in layers}) == 1
    return False


def run_recurrent(chain, xs):
    """Apply a recurrent stack to a whole sequence ``[T, B, in]`` (fused on CUDA, per-step loops otherwise)."""
    if FUSE_RECURRENT and _can_fuse(chain, xs):
        return _fused_recurrent(chain, xs)
    return chain(xs)


FUSE_RECURRENT = True


class _Tuple(nn.Module):
    """A tuple of layers (``pattern_extractor``, ``latent_in``, ``latent_out`` are tuples in GOKU.jl:234,243,258)."""

    def __init__(self, *layers):
        super().__init__()
        self.layers = nn.ModuleList(layers)

    def __iter__(self):
        return iter(self.layers)

    def __len__(self):
        return len(self.layers)

    def __getitem__(self, i):
        return self.layers[i]


class Identity(nn.Module):
    def forward(self, x):
        return x


# ---- the per-model-type steps (multiple dispatch in the reference; isinstance here) ---------------
def apply_feature_extractor(encoder, x):
    """GOKU.jl:19, LatentODE.jl:9: every time frame independently through the feature extractor."""
    return encoder.feature_extractor(x)


def _pe_kernel_ok(fe_out, rnn_chain, lstm_chains=()):
    """The default architecture's stacks (two layers, 16 hidden units, relu RNN / LSTM; GOKU.jl:224-234) on a CUDA
    sequence: the shapes ``ldeq_pattern_extractor_fwd`` is built for."""
    from .solve import PE_HIDDEN, PE_HIDDEN_RNN_ONLY, PE_INPUTS
    if not (PERSISTENT_RECURRENT and fe_out.is_cuda and fe_out.dtype == torch.float32 and fe_out.dim() == 3 and fe_out.shape[-1] in PE_INPUTS):
        return False

    def stack_ok(chain, cls, hidden):
        layers = list(chain) if isinstance(chain, nn.Sequential) else []
        if len(layers) != 2 or not all(isinstance(l, cls) for l in layers):
            return False
        rows = hidden * (4 if cls is LSTM else 1)
        return (all(l.Wi.dtype == torch.float32 for l in layers) and tuple(layers[0].Wi.shape) == (rows, fe_out.shape[-1]) and tuple(layers[1].Wi.shape) == (rows, hidden)
                and (cls is LSTM or all(l.act is F.relu for l in layers)))
    if lstm_chains:     # GOKU: all three stacks with 16 hidden units
        return stack_ok(rnn_chain, RNN, PE_HIDDEN) and all(stack_ok(c, LSTM, PE_HIDDEN) for c in lstm_chains)
    # LatentODE: the RNN stack alone, 16 or 32 hidden units (LatentODE.jl:102 defaults to 32, input 32 or 64)
    return stack_ok(rnn_chain, RNN, PE_HIDDEN) or (fe_out.shape[-1] in (32, 64) and stack_ok(rnn_chain, RNN, PE_HIDDEN_RNN_ONLY))


PERSISTENT_RECURRENT = True   # False: the cuDNN / per-step route below (kept for other layer shapes and as a cross-check)


def apply_pattern_extractor(encoder, fe_out):
    """GOKU.jl:30-49 / LatentODE.jl:20-34: recurrent layers over the (reversed) sequence; only the
    final hidden state is used; hidden states start from ``state0`` on every call (``Flux.reset!``).
    The default architecture runs through the persistent kernels of ``csrc/ldeq_recurrent.cu`` (SURVEY.md 8(f)2)."""
    if isinstance(encoder.model_type, GOKU):
        pe_z0, pe_th_f, pe_th_b = encoder.pattern_extractor
        if _pe_kernel_ok(fe_out, pe_z0, (pe_th_f, pe_th_b)):
            return pattern_extractor(fe_out, list(pe_z0), list(pe_th_f), list(pe_th_b))
    elif _pe_kernel_ok(fe_out, encoder.pattern_extractor):
        return pattern_extractor(fe_out, list(encoder.pattern_extractor))
    rev = torch.flip(fe_out, dims=[0])
    if isinstance(encoder.model_type, GOKU):
        pe_z0, pe_th_f, pe_th_b = encoder.pattern_extractor
        z0_out = run_recurrent(pe_z0, rev)[-1]
        th_out = torch.cat([run_recurrent(pe_th_f, fe_out)[-1], run_recurrent(pe_th_b, rev)[-1]], dim=-1)
        return z0_out, th_out
    return run_recurrent(encoder.pattern_extractor, rev)[-1]


def apply_latent_in(encoder, pe_out):
    """GOKU.jl:61-72 / LatentODE.jl:36-43."""
    if isinstance(encoder.model_type, GOKU):
        pe_z0_out, pe_th_out = pe_out
        li_mu_z0, li_lv_z0, li_mu_th, li_lv_th = encoder.latent_in
        return (li_mu_z0(pe_z0_out), li_mu_th(pe_th_out)), (li_lv_z0(pe_z0_out), li_lv_th(pe_th_out))
    li_mu, li_lv = encoder.latent_in
    return li_mu(pe_out), li_lv(pe_out)


_sample_calls = 0
_sample_counter = None


@contextlib.contextmanager
def device_sample_counter(calls: torch.Tensor):
    """Inside the block ``sample`` draws through ``ldeq_sample_dev`` with the device counter ``calls`` (one int64 element that
    mirrors ``_sample_calls``): a captured CUDA graph then draws new noise on every replay.  The host counter still advances
    once per draw, as it does outside the block."""
    global _sample_counter
    prev, _sample_counter = _sample_counter, calls
    try:
        yield
    finally:
        _sample_counter = prev


def sample(mu, logvar, model, seed: int | None = None):
    """Reparameterised sample ``mu + eps * exp(logvar/2)`` (GOKU.jl:155-173, LatentODE.jl:82-98).
    The noise is drawn on the device by ``ldeq_sample`` (the reference draws it on the host and
    uploads it, GOKU.jl:169-170)."""
    if seed is None:
        seed = int(torch.initial_seed() & 0x7FFFFFFFFFFFFFFF)

    def draw(m, lv):
        global _sample_calls
        _sample_calls += 1
        if _sample_counter is None:
            return sample_reparam(m, lv, seed, _sample_calls << 32)
        return sample_reparam(m, lv, seed, _sample_calls << 32, _sample_counter)
    if isinstance(mu, tuple):
        return tuple(draw(m, lv) for m, lv in zip(mu, logvar))
    return draw(mu, logvar)


def apply_latent_out(decoder, l_tilde):
    """GOKU.jl:83-91 / LatentODE.jl:54."""
    if isinstance(decoder.model_type, GOKU):
        z0_t, th_t = l_tilde
        lo_z0, lo_th = decoder.latent_out
        return lo_z0(z0_t), lo_th(th_t)
    return decoder.latent_out(l_tilde)


def transform_after_diffeq(x, diffeq):
    """Identity by default (GOKU.jl:136); a diffeq struct may define its own ``transform_after_diffeq``."""
    f = getattr(diffeq, "transform_after_diffeq", None)
    return f(x) if f is not None else x


def _opts_from_kwargs(kwargs: dict, sensealg=None, solver=None) -> _cabi.Opts:
    """The diffeq struct's ``kwargs`` / ``sensealg`` / ``solver`` fields (GOKU.jl:105-108) as ``ldeq_opts``."""
    kw = dict(kwargs)
    kw.pop("saveat", None)
    if sensealg is not None:
        code = getattr(sensealg, "code", None)
        if code is None:
            raise TypeError(f"sensealg {sensealg!r}: ForwardDiffSensitivity() / InterpolatingAdjoint() (the reference's) or DiscreteAdjoint()")
        kw["sensealg"] = code
    if solver is not None:
        code = getattr(solver, "code", None)
        if code is None:
            raise NotImplementedError(f"solver {solver!r}: Tsit5() (pendulum.jl:11,58), DP5(), BS3() and RK4() are built")
        kw["solver"] = code
    return _cabi.default_opts(**kw)


def diffeq_layer(decoder, l_hat, t, stats_out=None):
    """THE HOT PATH.  GOKU: B independent solves of the diffeq struct's problem with initial
    conditions / parameters ``l_hat = (z0_hat, theta_hat)``, saved at ``t`` (GOKU.jl:98-130).
    LatentODE: one solve on the matrix state with the MLP right-hand side (LatentODE.jl:61-78).
    Returns ``z_hat`` as ``[T, B, z]`` (Julia ``(z, B, T)``)."""
    diffeq = decoder.diffeq
    if isinstance(decoder.model_type, GOKU):
        z0_hat, th_hat = l_hat
        f = diffeq.prob.f
        if isinstance(f, CudaRHS):
            f = f.resolve(_cabi.handle(z0_hat.device.index or 0))
        z = goku_solve(z0_hat, th_hat, t, f, _opts_from_kwargs(diffeq.kwargs, getattr(diffeq, 'sensealg', None),
                                                               getattr(diffeq, 'solver', None)), stats_out)
        return transform_after_diffeq(z, diffeq)
    z0 = l_hat
    if diffeq.augment_dim:
        # AugmentedNDELayer (LatentODE.jl:71): zero-pad augment_dim extra state rows
        z0 = torch.cat([z0, z0.new_zeros(z0.shape[0], diffeq.augment_dim)], dim=1)
    z = mlp_solve(z0, diffeq.flat_params(), diffeq.dims, t, _opts_from_kwargs(diffeq.kwargs, getattr(diffeq, 'sensealg', None),
                                                                          getattr(diffeq, 'solver', None)), stats_out)
    return transform_after_diffeq(z, diffeq)


def apply_reconstructor(decoder, z_hat):
    """GOKU.jl:148 / LatentODE.jl:80."""
    return decoder.reconstructor(z_hat)


def _logits_layers(decoder):
    """The reconstructor's layers when its last one is a ``Dense`` with the sigmoid output activation, else ``None``."""
    rec = decoder.reconstructor
    layers = list(rec) if isinstance(rec, nn.Sequential) else []
    if not layers or not isinstance(layers[-1], Dense) or layers[-1].act is not torch.sigmoid:
        return None
    return layers


def reconstructor_logits(decoder, z_hat):
    """The reconstructor up to the pre-activations of its last layer, when that layer is a ``Dense`` with the sigmoid output
    activation of ``default_layers`` (GOKU.jl:265-268); ``None`` otherwise.  ``ldeq_elbo_logits_fwd_bwd`` applies the sigmoid
    inside the loss kernel."""
    layers = _logits_layers(decoder)
    if layers is None:
        return None
    h = z_hat
    for l in layers[:-1]:
        h = l(h)
    return F.linear(h, layers[-1].weight, layers[-1].bias)


# ---- containers (src/models/LatentDiffEqModel.jl) --------------------------------------------------
class Encoder(nn.Module):
    def __init__(self, model_type, encoder_layers):
        super().__init__()
        self.model_type = model_type
        self.feature_extractor, self.pattern_extractor, self.latent_in = encoder_layers

    def forward(self, x):
        fe_out = apply_feature_extractor(self, x)
        pe_out = apply_pattern_extractor(self, fe_out)
        return apply_latent_in(self, pe_out)


class Decoder(nn.Module):
    def __init__(self, model_type, decoder_layers):
        super().__init__()
        self.model_type = model_type
        self.latent_out, self.diffeq, self.reconstructor = decoder_layers

    def forward(self, l_tilde, t):
        l_hat = apply_latent_out(self, l_tilde)
        z_hat = diffeq_layer(self, l_hat, t)
        x_hat = apply_reconstructor(self, z_hat)
        return x_hat, z_hat, l_hat


class LatentDiffEqModel(nn.Module):
    """``LatentDiffEqModel(model_type, encoder_layers, decoder_layers)`` (LatentDiffEqModel.jl:16-22)."""

    def __init__(self, model_type, encoder_layers, decoder_layers):
        super().__init__()
        self.model_type = model_type
        self.encoder = Encoder(model_type, encoder_layers)
        self.decoder = Decoder(model_type, decoder_layers)

    def forward(self, x, t, variational=False):
        mu, logvar = self.encoder(x)
        l_tilde = sample(mu, logvar, self) if variational else mu
        X_hat = self.decoder(l_tilde, t)
        return X_hat, mu, logvar

    def forward_logits(self, x, t, variational=False):
        """``forward`` with the reconstruction left as the pre-activations of the sigmoid output layer: returns
        ``((logits, z_hat, l_hat), mu, logvar)``, or ``None`` when the reconstructor does not end in such a layer."""
        mu, logvar = self.encoder(x)
        l_tilde = sample(mu, logvar, self) if variational else mu
        l_hat = apply_latent_out(self.decoder, l_tilde)
        z_hat = diffeq_layer(self.decoder, l_hat, t)
        logits = reconstructor_logits(self.decoder, z_hat)
        if logits is None:
            return None
        return (logits, z_hat, l_hat), mu, logvar


def _resnet(d_in, hidden, d_out, act, out_act, init):
    return Chain(Dense(d_in, hidden, act, init), SkipConnection(Dense(hidden, hidden, act, init)),
                 SkipConnection(Dense(hidden, hidden, act, init)), Dense(hidden, d_out, out_act, init))


def default_layers(model_type, input_dim, diffeq, device="cpu", hidden_dim_resnet=200, rnn_input_dim=32,
                   rnn_output_dim=None, latent_dim_z0=16, latent_dim_theta=16, latent_to_diffeq_dim=200,
                   general_activation="relu", z0_activation="identity", theta_activation="softplus",
                   output_activation="sigmoid", init=kaiming_uniform_):
    """Default encoder / decoder layers (GOKU.jl:199-274 for ``GOKU_basic``, LatentODE.jl:100-152 for
    ``LatentODE``).  Returns ``(encoder_layers, decoder_layers)`` to feed ``LatentDiffEqModel``."""
    if isinstance(model_type, GOKU):
        rnn_output_dim = rnn_output_dim or 16
        z_dim, th_dim = len(diffeq.prob.u0), len(diffeq.prob.p)
        fe = _resnet(input_dim, hidden_dim_resnet, rnn_input_dim, general_activation, general_activation, init)
        pe_z0 = Chain(RNN(rnn_input_dim, rnn_output_dim, "relu", init), RNN(rnn_output_dim, rnn_output_dim, "relu", init))
        pe_f = Chain(LSTM(rnn_input_dim, rnn_output_dim, init), LSTM(rnn_output_dim, rnn_output_dim, init))
        pe_b = Chain(LSTM(rnn_input_dim, rnn_output_dim, init), LSTM(rnn_output_dim, rnn_output_dim, init))
        latent_in = _Tuple(Dense(rnn_output_dim, latent_dim_z0, init=init), Dense(rnn_output_dim, latent_dim_z0, init=init),
                           Dense(2 * rnn_output_dim, latent_dim_theta, init=init),
                           Dense(2 * rnn_output_dim, latent_dim_theta, init=init))
        lo_z0 = Chain(Dense(latent_dim_z0, latent_to_diffeq_dim, general_activation, init),
                      Dense(latent_to_diffeq_dim, z_dim, z0_activation, init))
        lo_th = Chain(Dense(latent_dim_theta, latent_to_diffeq_dim, general_activation, init),
                      Dense(latent_to_diffeq_dim, th_dim, theta_activation, init))
        rec = _resnet(z_dim, hidden_dim_resnet, input_dim, general_activation, output_activation, init)
        enc = (fe.to(device), _Tuple(pe_z0, pe_f, pe_b).to(device), latent_in.to(device))
        dec = (_Tuple(lo_z0, lo_th).to(device), diffeq, rec.to(device))
        return enc, dec
    if isinstance(model_type, LatentODE):
        rnn_output_dim = rnn_output_dim or 32
        fe = _resnet(input_dim, hidden_dim_resnet, rnn_input_dim, "relu", "relu", init)
        pe = Chain(RNN(rnn_input_dim, rnn_output_dim, "relu", init), RNN(rnn_output_dim, rnn_output_dim, "relu", init))
        latent_in = _Tuple(Dense(rnn_output_dim, diffeq.latent_dim_in, init=init),
                           Dense(rnn_output_dim, diffeq.latent_dim_in, init=init))
        rec = _resnet(diffeq.latent_dim_out, hidden_dim_resnet, input_dim, "relu", output_activation, init)
        if isinstance(diffeq, nn.Module):
            diffeq = diffeq.to(device)
        return (fe.to(device), pe.to(device), latent_in.to(device)), (Identity(), diffeq, rec.to(device))
    raise TypeError(f"unknown model type {model_type!r}")
