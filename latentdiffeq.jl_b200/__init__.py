"""latentdiffeq.jl_b200 -- B200 (sm_100a) drop-in for the hot path of gabrevaya/LatentDiffEq.jl.

The hot path is the batched latent ODE solve inside ``diffeq_layer`` of the GOKU-net and LatentODE
models (reference ``src/models/GOKU.jl:98-130``, ``src/models/LatentODE.jl:61-78``), its reverse
pass, the ELBO reduction and the optimiser step.  It runs in hand-written CUDA behind the C ABI of
``include/ldeq.h`` (``lib/libldeq.so``); this package is the host-side mirror of the reference's
model / layer / diffeq-struct API above that ABI.  The directory name contains a dot, so import it
through the repo-root shim: ``import latentdiffeq_jl_b200 as ldeq``.
"""
from . import _cabi
from . import bson_io
from ._cabi import (F32, F64, RHS_PENDULUM, RHS_PENDULUM_FRICTION, RET_SUCCESS, RET_MAXITERS, RET_DTLESSTHANMIN,
                    RET_UNSTABLE, NORM_GLOBAL, NORM_PER_TRAJ, MLP_MATH_FP32, MLP_MATH_BF16X3, LdeqError, default_opts,
                    handle, Handle, SOLVER_TSIT5, SOLVER_DP5, SOLVER_BS3, SOLVER_RK4, SENSE_DISCRETE_ADJOINT, SENSE_FORWARD_DUAL, SENSE_INTERPOLATING_ADJOINT)
from .solve import (goku_solve, goku_solve_raw, goku_bwd_raw, goku_solve_host, goku_bwd_host, goku_fwd_bwd_host, debug_trig, mlp_solve, mlp_solve_raw,
                    mlp_bwd_raw, device_tape_check, mlp_bwd_stats, pattern_extractor, pe_flat_params, sample_raw, sample_reparam, elbo_raw, elbo_loss, adamw_step, adamw_step_dev, adamw_state,
                    allreduce_adamw_step)
from .diffeqs import (Tsit5, DP5, BS3, RK4, ForwardDiffSensitivity, DiscreteAdjoint, InterpolatingAdjoint, ODEProblem, CudaRHS, Pendulum, Pendulum_friction,
                      UserDiffEq, NODE)
from .model import (LatentDE, GOKU, GOKU_basic, LatentODE, Dense, SkipConnection, Chain, RNN, LSTM, Encoder, Decoder,
                    LatentDiffEqModel, default_layers, diffeq_layer, transform_after_diffeq, apply_feature_extractor,
                    apply_pattern_extractor, apply_latent_in, apply_latent_out, apply_reconstructor, sample, device_sample_counter)
from .utils import (vector_mse, kl, vector_kl, frange_cycle_linear, normalize_to_unit_segment, denormalize_unit_segment,
                    time_loader, rand_time)
from .train import loss_batch, shard_bounds, FlatParams, ADAMW, allreduce_grads, train_step, GraphedTrainStep

__all__ = [n for n in dir() if not n.startswith("_")]
