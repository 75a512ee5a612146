/* ldeq.h -- C ABI of libldeq.so: the B200 (sm_100a) drop-in for LatentDiffEq.jl's hot path.
 *
 * Every entry point replaces work that the reference does below one of its own interfaces
 * (citations are relative to the reference tree, gabrevaya/LatentDiffEq.jl):
 *
 *   ldeq_solve_fwd / ldeq_solve_bwd      diffeq_layer(::Decoder{<:GOKU}, l, t)   src/models/GOKU.jl:98-130
 *                                        (EnsembleProblem + Tsit5 per column, GOKU.jl:111-121; NaN block on
 *                                        failure, GOKU.jl:114; (z,B,T) layout, GOKU.jl:125) and its pullback
 *                                        (sensealg, examples/pendulum_friction-less/pendulum.jl:11)
 *   ldeq_rhs_builtin / _from_source      the user-defined diffeq struct's f!        pendulum.jl:19-26, 65-74
 *   ldeq_mlp_solve_fwd / _bwd            diffeq_layer(::Decoder{LatentODE}, z0, t) src/models/LatentODE.jl:61-78
 *                                        with dudt = Chain(Dense,Dense,Dense)      examples/.../nODE.jl:14-16
 *   ldeq_pattern_extractor_fwd / _bwd    apply_pattern_extractor(encoder, fe_out)  src/models/GOKU.jl:30-49, 224-234
 *   ldeq_sample                          sample(mu, logvar, model)                src/models/GOKU.jl:155-173,
 *                                                                                  src/models/LatentODE.jl:82-98
 *   ldeq_elbo_fwd_bwd                    loss_batch + vector_kl                   examples/.../model_train.jl:225-238,
 *                                                                                  src/utils/utils.jl:16-49
 *   ldeq_adamw_step                      Flux.Optimise.update!(ADAMW(...))        examples/.../model_train.jl:138,201
 *
 * Conventions
 *   - All array arguments are DEVICE pointers owned by the caller unless the name ends in _host.
 *     The library never keeps a caller pointer after the call returns; a tape holds its own copies.
 *   - Layout is the reference's column-major layout: z0 is (z,B) => element (d,b) at b*z+d;
 *     trajectories are (z,B,T) => element (d,b,k) at (k*B+b)*z+d  (what permutedims(.,[1,3,2])
 *     produces, GOKU.jl:125).  A contiguous torch tensor of shape [T,B,z] has the same bytes.
 *   - Calls are asynchronous on the given CUDA stream (cudaStream_t passed as void*); functions
 *     whose name ends in _host synchronise that stream before returning.
 *   - Return value: 0 on success, negative ldeq_status on error (ldeq_last_error gives text).
 *     A solver failure of one trajectory is NOT an error: its (z,T) block is filled with NaN
 *     (GOKU.jl:114), retcode[b] says why, and its gradient contribution is zero.
 *   - One handle per GPU and host thread; a handle is not thread-safe.
 *
 * CUDA graph capture
 *   Every entry point that takes a stream checks whether that stream is being captured (cudaStreamIsCapturing).  A
 *   captured call records the same kernels and copies it would run eagerly; values the host passes are frozen into the
 *   graph, so per-step values go through the _dev entry points below, which read them from device memory.
 *   Capture-safe: ldeq_solve_fwd (no tape, or a FORWARD_DUAL tape) and ldeq_solve_bwd of such a tape, ldeq_tape_free,
 *   ldeq_pattern_extractor_fwd / _bwd / ldeq_pe_tape_free, ldeq_sample / _dev, ldeq_elbo_* / _dev, ldeq_adamw_step /
 *   _dev, ldeq_mlp_solve_fwd_dev (no tape, or a device-checked tape other than INTERPOLATING_ADJOINT), ldeq_mlp_solve_bwd of
 *   such a tape and ldeq_mlp_tape_free.  Rules:
 *   - A tape recorded under capture has no host mirror and no event: its allocation and release become graph nodes.
 *   - A captured solve reads an immutable device copy of its time grid, kept by the handle until ldeq_destroy (the grid
 *     an eager call uses is overwritten when another grid arrives).  The copy is made by an eager solve on the same grid:
 *     a capture whose grid has not been solved eagerly before is refused, since a copy from pageable host memory cannot
 *     be captured.  Likewise the ELBO workspace, device scratch and the NVRTC variant of a user right-hand side for a
 *     non-Tsit5 solver are created by a first eager call; under capture their absence is refused.
 *   - Refused with LDEQ_ERR_UNSUPPORTED, before anything is enqueued (the capture stays valid and can be ended), because
 *     they need the host while the work runs: a DISCRETE_ADJOINT tape and its reverse pass (the tape's overflow check,
 *     tape_heal), ldeq_tape_overflow, ldeq_mlp_solve_fwd, ldeq_mlp_solve_bwd of its tape and ldeq_mlp_bwd_stats (the MLP
 *     tape check on the host and the continuous adjoint), every _host entry point (staging and stream synchronisation), ldeq_allreduce_grads and
 *     ldeq_allreduce_adamw_step (multi-GPU capture is not built).  ldeq_comm_unique_id / _init / _destroy take no stream:
 *     they are set-up calls that synchronise the device and must not be made while a capture is open.
 */
#ifndef LDEQ_H
#define LDEQ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LDEQ_VERSION 210

typedef struct ldeq_handle ldeq_handle;
typedef struct ldeq_rhs ldeq_rhs;
typedef struct ldeq_tape ldeq_tape;
typedef struct ldeq_mlp_tape ldeq_mlp_tape;
typedef void* ldeq_stream; /* cudaStream_t */

/* Device-resident AdamW step state for ldeq_adamw_step_dev: the 1-based step count and the running Float64 products
 * beta1^step, beta2^step that Flux keeps.  Zero-initialised step with beta1_pow = beta2_pow = 1 is the state before step 1. */
typedef struct ldeq_adamw_state {
    int64_t step;
    double beta1_pow;
    double beta2_pow;
} ldeq_adamw_state;

enum ldeq_status {
    LDEQ_OK = 0,
    LDEQ_ERR_INVALID = -1,     /* bad argument */
    LDEQ_ERR_CUDA = -2,        /* CUDA runtime error; text in ldeq_last_error */
    LDEQ_ERR_UNSUPPORTED = -3, /* combination not built (e.g. z_dim of a compiled RHS too large) */
    LDEQ_ERR_NOMEM = -4,
    LDEQ_ERR_COMPILE = -5,     /* NVRTC could not compile a user RHS; log in ldeq_last_error */
    LDEQ_ERR_TAPE_OVERFLOW = -6 /* ldeq_mlp_solve_bwd: the solve took more accepted steps than the tape holds; the
                                   message names the count -- repeat the forward solve with opts.tape_steps >= it */
};

enum ldeq_dtype { LDEQ_F32 = 0, LDEQ_F64 = 1 };

/* built-in right-hand sides: the reference's example diffeq structs */
enum ldeq_rhs_kind {
    LDEQ_RHS_PENDULUM = 0,         /* du = [y, -G/L sin x], G = 10            pendulum.jl:19-26 */
    LDEQ_RHS_PENDULUM_FRICTION = 1 /* du = [y, -G/L sin x - (b/m) y], b=.7,m=1 pendulum.jl:65-74 */
};

/* per-trajectory return codes (SciMLBase retcodes the reference tests for at GOKU.jl:114) */
enum ldeq_retcode {
    LDEQ_RET_SUCCESS = 0,
    LDEQ_RET_MAXITERS = 1,
    LDEQ_RET_DTLESSTHANMIN = 2,
    LDEQ_RET_UNSTABLE = 3
};

/* error-norm scope of the MLP (LatentODE) solve */
enum ldeq_norm_mode {
    LDEQ_NORM_GLOBAL = 0,  /* one dt for the whole (D,B) matrix state: reference semantics (LatentODE.jl:70-72) */
    LDEQ_NORM_PER_TRAJ = 1 /* per-trajectory error control: documented deviation, no cross-CTA reduction */
};

/* arithmetic of the MLP right-hand side */
enum ldeq_mlp_math {
    LDEQ_MLP_MATH_FP32 = 0,    /* CUDA-core fp32 (fp64 when dtype is F64): exact-parity path */
    LDEQ_MLP_MATH_BF16X3 = 1   /* tcgen05 tensor cores, 3-term bf16 split of fp32 operands, fp32 accumulate */
};

/* The diffeq struct's `sensealg` field (pendulum.jl:11,58: ForwardDiffSensitivity()).
 *   LDEQ_SENSE_FORWARD_DUAL      the reference's algorithm itself (SciMLSensitivity `ForwardDiffSensitivity`): two
 *        dual-number re-solves per trajectory (seeded on theta, then on u0) whose error norm includes the partials, so
 *        each takes its own step sequence.  DEFAULT (ldeq_opts_default): it is what the reference's structs request,
 *        and the only mode whose gradients equal the reference's to 1e-4 at the default tolerances.
 *   LDEQ_SENSE_DISCRETE_ADJOINT  reverse sweep over the taped accepted steps of the primal solve: the exact derivative of
 *        the primal discretisation (step sizes frozen), one kernel, ~the cost of the forward solve, ~3x cheaper than
 *        the dual solves.  An explicit opt-in (Python: `sensealg = DiscreteAdjoint()`): it agrees with the reference's
 *        gradient only within the solver tolerance (2e-2 at reltol 1e-3), exactly in fixed-step mode.
 *   LDEQ_SENSE_INTERPOLATING_ADJOINT  (ldeq_mlp_* only) the reference's algorithm for the LatentODE path: DiffEqFlux's
 *        NeuralODE default `InterpolatingAdjoint(autojacvec = ZygoteVJP())` (LatentODE.jl:70 under Zygote) -- the continuous
 *        adjoint ODE on [lambda; mu] solved backwards by adaptive Tsit5 with the forward dense output and a callback at
 *        every save time (csrc/ldeq_mlp_cadj.cuh).  Needs the batch-global norm and the exact arithmetic path; any other
 *        value makes ldeq_mlp_solve_bwd run the discrete adjoint of the taped steps.  The GOKU entry points refuse it. */
typedef enum { LDEQ_SENSE_DISCRETE_ADJOINT = 0, LDEQ_SENSE_FORWARD_DUAL = 1, LDEQ_SENSE_INTERPOLATING_ADJOINT = 2 } ldeq_sensealg;

/* The diffeq struct's `solver` field, handed to `solve` at GOKU.jl:121.  The reference's structs use Tsit5()
 * (pendulum.jl:11,58); the field is the user's to set, so OrdinaryDiffEq's DP5(), BS3() and RK4() are built as well
 * (SURVEY.md 8(f)4; csrc/ldeq_erk.cuh: the same integrator kernels with a table-driven method, dense output as
 * OrdinaryDiffEq defines it -- dopri5's contd5 for DP5, cubic Hermite for BS3 / RK4).  GOKU entry points only: the
 * LatentODE kernels are Tsit5.  RK4 is accepted with adaptive = 0 only (OrdinaryDiffEq's adaptive RK4 is a defect-control
 * estimate that is not restated).  Anything unsupported is refused with LDEQ_ERR_UNSUPPORTED, never silently replaced. */
typedef enum { LDEQ_SOLVER_TSIT5 = 0, LDEQ_SOLVER_DP5 = 1, LDEQ_SOLVER_BS3 = 2, LDEQ_SOLVER_RK4 = 3 } ldeq_solver;

/* The keyword arguments the diffeq struct's `kwargs` field forwards to `solve` (pendulum.jl:11,43;
 * GOKU.jl:108,121).  ldeq_opts_default fills OrdinaryDiffEq's defaults for Tsit5. */
typedef struct ldeq_opts {
    double abstol;       /* 1e-6 */
    double reltol;       /* 1e-3 */
    int32_t adaptive;    /* 1; 0 = fixed step `dt` */
    int32_t controller_pow; /* 0 = DiffEqBase.fastpow (reference), 1 = exact pow */
    double dt;           /* 0 = automatic initial step (adaptive); required when adaptive = 0 */
    double dtmax;        /* 0 = t[T-1] - t[0] */
    double dtmin;        /* 0 = max(eps, eps(t[0])) */
    int64_t maxiters;    /* 1000000 */
    double gamma;        /* 0.9 */
    double qmin;         /* 0.2 */
    double qmax;         /* 10 */
    double beta1;        /* 7/50 */
    double beta2;        /* 2/25 */
    double qoldinit;     /* 1e-4 */
    double qsteady_min;  /* 1 */
    double qsteady_max;  /* 1 */
    int32_t tape_steps;  /* accepted-step capacity per trajectory of a tape; 0 = automatic: max(64, T) and
                            what earlier solves on this handle needed (a too-small tape heals itself) */
    int32_t norm_mode;   /* ldeq_norm_mode, MLP solve only */
    int32_t mlp_math;    /* ldeq_mlp_math, MLP solve only */
    int32_t sensealg;    /* ldeq_sensealg: how ldeq_solve_bwd differentiates a GOKU solve (default FORWARD_DUAL) */
    int32_t solver;      /* ldeq_solver (default TSIT5) */
    int32_t reserved_;   /* keeps the struct a multiple of 8 bytes */
} ldeq_opts;

int ldeq_version(void);
void ldeq_opts_default(ldeq_opts* opts);
/* The same with `solver` set and the PI-controller exponents OrdinaryDiffEq gives that algorithm (beta2 = 2/(5 order),
 * beta1 = 7/(10 order); DP5: beta2 = 4/100, beta1 = 1/5 - 3 beta2/4).  Returns LDEQ_ERR_INVALID for an unknown solver. */
int ldeq_opts_default_solver(ldeq_opts* opts, int solver);

/* ---- handle ------------------------------------------------------------------------------------ */
int ldeq_create(ldeq_handle** out, int device);
void ldeq_destroy(ldeq_handle* h);
const char* ldeq_last_error(const ldeq_handle* h);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches) */
int64_t ldeq_launch_count(const ldeq_handle* h);

/* ---- right-hand sides -------------------------------------------------------------------------- */
int ldeq_rhs_builtin(ldeq_handle* h, int kind, ldeq_rhs** out);
/* User-defined RHS compiled with NVRTC for sm_100a.  `cuda_src` must define
 *   template <class S> __device__ void ldeq_user_rhs(S* du, const S* u, const S* p, S t);
 * It is instantiated with float, double and a forward-mode dual type (for the reverse pass). */
int ldeq_rhs_from_source(ldeq_handle* h, const char* cuda_src, int z_dim, int p_dim, ldeq_rhs** out);
int ldeq_rhs_dims(const ldeq_rhs* rhs, int* z_dim, int* p_dim);
void ldeq_rhs_free(ldeq_handle* h, ldeq_rhs* rhs);

/* ---- GOKU path: B independent solves ----------------------------------------------------------- */
/* z0 (z,B), theta (p,B), t_host[T] (host, Float64 grid; t_host[0], t_host[T-1] are the tspan),
 * traj_out (z,B,T), or NULL when only the tape / statistics are wanted.  retcode/naccept/nreject are
 * optional device int32[B] outputs.
 * If tape_out != NULL a tape of the accepted steps is recorded for ldeq_solve_bwd. */
int ldeq_solve_fwd(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0, const void* theta,
                   const double* t_host, int B, int T, const ldeq_opts* opts, void* traj_out,
                   int32_t* retcode, int32_t* naccept, int32_t* nreject, ldeq_tape** tape_out,
                   ldeq_stream stream);
/* Pullback dtraj (z,B,T) -> dz0 (z,B), dtheta (p,B) by the tape's sensealg (dual re-solves or discrete adjoint). */
int ldeq_solve_bwd(ldeq_handle* h, ldeq_tape* tape, const void* dtraj, void* dz0, void* dtheta,
                   ldeq_stream stream);
/* Trajectories whose accepted steps exceeded the tape capacity.  ldeq_solve_bwd heals such a tape by
 * replaying the forward solve into a larger one (it waits for the forward kernel to learn this), so
 * gradients are always exact; this call only reports how many trajectories needed that.  Waits for the
 * forward kernel. */
int ldeq_tape_overflow(ldeq_handle* h, ldeq_tape* tape, int32_t* count_host, ldeq_stream stream);
void ldeq_tape_free(ldeq_handle* h, ldeq_tape* tape, ldeq_stream stream);

/* Same calls with HOST buffers (what a CPU-resident Flux model passes, GOKU.jl:102-103,128): the library stages
 * through its own device scratch; copies are inside the call; returns after sync.  The batch is cut into column
 * slabs (trajectories are independent): transfers of one slab run on the library's copy streams under the kernels
 * of the next, so one caller thread keeps the PCIe link and the SMs busy together.  Pinned host buffers make the
 * copies asynchronous; pageable ones work (the runtime stages them). */
int ldeq_solve_fwd_host(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0_host,
                        const void* theta_host, const double* t_host, int B, int T, const ldeq_opts* opts,
                        void* traj_out_host, int32_t* retcode_host, int32_t* naccept_host,
                        int32_t* nreject_host, ldeq_tape** tape_out, ldeq_stream stream);
int ldeq_solve_bwd_host(ldeq_handle* h, ldeq_tape* tape, const void* dtraj_host, void* dz0_host,
                        void* dtheta_host, ldeq_stream stream);
/* Forward solve and pullback of a KNOWN cotangent in one call (replaying a stored batch, gradient checks, the
 * throughput benchmark): the cotangent slabs go up while the trajectory slabs come down -- both directions of the
 * link at once, from a single caller thread.  No tape is returned. */
int ldeq_solve_fwd_bwd_host(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0_host,
                            const void* theta_host, const double* t_host, int B, int T, const ldeq_opts* opts,
                            const void* dtraj_host, void* traj_out_host, void* dz0_host, void* dtheta_host,
                            int32_t* retcode_host, int32_t* naccept_host, int32_t* nreject_host,
                            ldeq_stream stream);

/* ---- LatentODE path: one solve on the (D,B) matrix state with an MLP right-hand side ------------ */
/* params_flat is Flux.destructure order: per layer vec(W) with W (out,in) column-major, then b.
 * layer_dims[n_layers+1] = {D, H1, ..., D}; relu on every layer but the last (nODE.jl:14-16). */
int ldeq_mlp_solve_fwd(ldeq_handle* h, int dtype, const void* z0, const void* params_flat,
                       const int32_t* layer_dims_host, int n_layers, const double* t_host, int B, int T,
                       const ldeq_opts* opts, void* traj_out, int32_t* retcode, int32_t* naccept,
                       int32_t* nreject, ldeq_mlp_tape** tape_out, ldeq_stream stream);
/* The same solve with a DEVICE-CHECKED tape, for CUDA graphs (a training step of LatentODE.jl:61-78 captured once and
 * replayed): same checks, same kernels, the same traj / retcode / naccept / nreject and tape contents bit for bit, eagerly
 * and under capture.  The tape takes no pinned host mirror or event and its pullback never waits for the host: where the
 * tape of ldeq_mlp_solve_fwd makes ldeq_mlp_solve_bwd return LDEQ_ERR_TAPE_OVERFLOW (more accepted steps N than
 * opts->tape_steps), this one's pullback writes NaN into the overflowed rows of dz0 (as both do) and into EVERY element of
 * dparams_flat, and raises the caller-owned device word *overflow to max(*overflow, N) -- the tape_steps to ask for.  The
 * word is sticky: only the caller clears it.  The pullback of a tape whose steps all fit writes exactly what the pullback
 * of the ldeq_mlp_solve_fwd tape writes.  A tape needs a non-null `overflow` (LDEQ_ERR_INVALID otherwise).
 * Refused with LDEQ_ERR_UNSUPPORTED before anything is enqueued: a tape for LDEQ_SENSE_INTERPOLATING_ADJOINT (the continuous
 * adjoint sizes its dense output from the host count), and under capture a grid no eager solve has brought to the device or
 * device scratch that would have to grow.  A BF16X3 tape's reverse pass keeps tape_steps step records per 128 trajectories
 * (about 3 MB each for the reference's 16-200-200-16 network): this call allocates them, or refuses with their size. */
int ldeq_mlp_solve_fwd_dev(ldeq_handle* h, int dtype, const void* z0, const void* params_flat,
                           const int32_t* layer_dims_host, int n_layers, const double* t_host, int B, int T,
                           const ldeq_opts* opts, void* traj_out, int32_t* retcode, int32_t* naccept,
                           int32_t* nreject, int32_t* overflow /* device word, caller-owned */,
                           ldeq_mlp_tape** tape_out, ldeq_stream stream);
/* The pullback of either tape.  An ldeq_mlp_solve_fwd tape: waits for its forward kernel, returns LDEQ_ERR_TAPE_OVERFLOW
 * when the tape was too short, and is refused under capture.  A device-checked tape: capture-safe, never waits. */
int ldeq_mlp_solve_bwd(ldeq_handle* h, ldeq_mlp_tape* tape, const void* dtraj, void* dz0,
                       void* dparams_flat, ldeq_stream stream);
/* {accepted steps, rejected steps, retcode} of the backward solve that LDEQ_SENSE_INTERPOLATING_ADJOINT ran for this
 * tape (zeros before ldeq_mlp_solve_bwd or in the discrete-adjoint mode); synchronises `stream`. */
int ldeq_mlp_bwd_stats(ldeq_handle* h, ldeq_mlp_tape* tape, int32_t* out3_host, ldeq_stream stream);
/* debugging aid: with LDEQ_CADJ_TRACE=1 in the environment, the first n attempted steps of that backward solve as
 * (t, dt, EEst, accepted) quadruples of doubles; synchronises the device. */
int ldeq_debug_cadj_trace(ldeq_handle* h, ldeq_mlp_tape* tape, double* out_host, int n);
void ldeq_mlp_tape_free(ldeq_handle* h, ldeq_mlp_tape* tape, ldeq_stream stream);

/* ---- recurrent pattern extractor (SURVEY.md 8(f)2) ----------------------------------------------------------------
 * Replaces the body of apply_pattern_extractor (src/models/GOKU.jl:30-49; src/models/LatentODE.jl:20-34): the two-layer
 * relu-RNN stack on the REVERSED frame sequence and, for GOKU, the two two-layer LSTM stacks (forward and reversed
 * sequence) of default_layers (GOKU.jl:224-234), each one persistent kernel over all T frames (csrc/ldeq_recurrent.cu);
 * only the final hidden states leave, and every call starts from the trainable initial states (`Flux.reset!`).
 *   x            (F,B,T) Float32 device array, the feature extractor's output per frame: element (f,b,k) at (k*B+b)*F+f
 *   *_params     one flat Float32 vector per stack in `Flux.destructure` order: per layer Wi (rows x in, column-major),
 *                Wh (rows x H), b (rows), state0 (H) [LSTM: h0 (H), c0 (H)]; rows = H (RNN) or 4H (LSTM, gate order input,
 *                forget, cell, output); layer 1 has in = F, layer 2 in = H.  ldeq_pattern_extractor_param_count(cell = 0
 *                RNN / 1 LSTM, F, H) gives the length.  lstm_f_params / lstm_b_params / theta_out may all be NULL (LatentODE).
 *   z0_out       (H,B): final state of the RNN stack;  theta_out (2H,B): [LSTM forward; LSTM reversed] (GOKU.jl:42)
 *   tape_out     non-NULL: keep the hidden / cell states of every step for ldeq_pattern_extractor_bwd
 * Built for H = 16 with F in {16, 32, 64} (defaults F = 32, H = 16, GOKU.jl:200-201) and, for the RNN stack alone, H = 32
 * with F in {32, 64} (LatentODE's defaults F = 32, H = 32, LatentODE.jl:101-102); anything else LDEQ_ERR_UNSUPPORTED.
 * The reverse pass is back-propagation through time: dx (F,B,T) and the three flat parameter gradients are OUTPUTS
 * (overwritten), x and the parameters must be those of the forward call. */
typedef struct ldeq_pe_tape ldeq_pe_tape;
int ldeq_pattern_extractor_param_count(int cell, int F, int H);
int ldeq_pattern_extractor_fwd(ldeq_handle* h, const float* x, int B, int T, int F, int H, const float* rnn_params,
                               const float* lstm_f_params, const float* lstm_b_params, float* z0_out, float* theta_out,
                               ldeq_pe_tape** tape_out, ldeq_stream stream);
int ldeq_pattern_extractor_bwd(ldeq_handle* h, ldeq_pe_tape* tape, const float* x, const float* rnn_params,
                               const float* lstm_f_params, const float* lstm_b_params, const float* dz0_out,
                               const float* dtheta_out, float* dx, float* d_rnn_params, float* d_lstm_f_params,
                               float* d_lstm_b_params, ldeq_stream stream);
void ldeq_pe_tape_free(ldeq_handle* h, ldeq_pe_tape* tape, ldeq_stream stream);

/* ---- reparameterised sample: z = mu + eps * exp(logvar/2), eps ~ N(0,1) drawn on the device ---- */
int ldeq_sample(ldeq_handle* h, const float* mu, const float* logvar, float* z_out, float* eps_out /*opt*/,
                int64_t n, uint64_t seed, uint64_t offset, ldeq_stream stream);
/* The same with the offset taken from a device counter: increments *calls (device uint64) and draws at
 * offset = *calls << 32, the value after the increment -- bit-identical to ldeq_sample at that offset.  For CUDA graphs:
 * every replay draws new noise. */
int ldeq_sample_dev(ldeq_handle* h, const float* mu, const float* logvar, float* z_out, float* eps_out /*opt*/,
                    int64_t n, uint64_t seed, uint64_t* calls, ldeq_stream stream);

/* ---- ELBO: L = sum_pixels mean_{B,T}(x-xhat)^2 + beta * sum_heads (1/B) sum 0.5(e^lv + mu^2 - lv - 1)
 * x, xhat (P,B,T); mu[h], logvar[h] (d_h,B) for n_heads heads (host arrays of device pointers).
 * Writes loss (device float[3]: total, reconstruction, kl) and, if non-NULL, the gradients
 * dxhat (P,B,T), dmu[h], dlogvar[h] of the TOTAL loss scaled by grad_scale. */
int ldeq_elbo_fwd_bwd(ldeq_handle* h, const float* x, const float* xhat, const float* const* mu_host,
                      const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, float beta,
                      int B, int T, int P, float grad_scale, float* loss, float* dxhat, float* const* dmu_host,
                      float* const* dlogvar_host, ldeq_stream stream);
/* The same with the reconstructor's sigmoid output activation folded in (GOKU.jl:265-268: the last Dense layer has
 * output_activation = sigma): `logits` (P,B,T) are that layer's pre-activations a, xhat = 1/(1+exp(-a)) is formed inside and
 * `dlogits` is the gradient with respect to a -- no xhat array, no separate activation passes. */
int ldeq_elbo_logits_fwd_bwd(ldeq_handle* h, const float* x, const float* logits, const float* const* mu_host,
                      const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, float beta,
                      int B, int T, int P, float grad_scale, float* loss, float* dlogits, float* const* dmu_host,
                      float* const* dlogvar_host, ldeq_stream stream);
/* Both with beta read from a device float (CUDA graphs: a replay uses the current value); results are bit-identical to
 * the host-value calls with that beta. */
int ldeq_elbo_fwd_bwd_dev(ldeq_handle* h, const float* x, const float* xhat, const float* const* mu_host,
                          const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, const float* beta,
                          int B, int T, int P, float grad_scale, float* loss, float* dxhat, float* const* dmu_host,
                          float* const* dlogvar_host, ldeq_stream stream);
int ldeq_elbo_logits_fwd_bwd_dev(ldeq_handle* h, const float* x, const float* logits, const float* const* mu_host,
                                 const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, const float* beta,
                                 int B, int T, int P, float grad_scale, float* loss, float* dlogits, float* const* dmu_host,
                                 float* const* dlogvar_host, ldeq_stream stream);

/* ---- fused multi-tensor AdamW with Flux semantics:
 * m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; x -= lr * m/(1-b1^t) / (sqrt(v/(1-b2^t)) + eps) + decay * x
 * (Flux 0.13 ADAMW = Optimiser(ADAM, WeightDecay): the decay is NOT scaled by lr).  lr, betas and eps are
 * Float64 in Flux (the example passes eta = 1e-3), decay is the example's Float32 0.001f0; `step` is 1-based;
 * gradients are multiplied by grad_scale first (1/world_size after a sum all-reduce). */
int ldeq_adamw_step(ldeq_handle* h, float* params, const float* grads, float* m, float* v, int64_t n, double lr,
                    double beta1, double beta2, double eps, float decay, int64_t step, float grad_scale,
                    ldeq_stream stream);
/* The same with the step taken from device memory: one single-thread kernel advances *state (step + 1, beta powers times
 * beta1 / beta2, the multiplications of ldeq_adamw_step in the same order), then the update reads it.  Step k gives
 * parameters, m and v bit-identical to ldeq_adamw_step(..., step = k).  For CUDA graphs: every replay is the next step. */
int ldeq_adamw_step_dev(ldeq_handle* h, float* params, const float* grads, float* m, float* v, int64_t n, double lr,
                        double beta1, double beta2, double eps, float decay, ldeq_adamw_state* state, float grad_scale,
                        ldeq_stream stream);

/* ---- gradient all-reduce FUSED with AdamW over NVLink peer memory (data-parallel training, model_train.jl:195-201
 * on several GPUs).  peer_grads_host[r] is rank r's flat gradient bucket mapped into this process (symmetric memory /
 * CUDA IPC; the caller owns the mappings and the cross-GPU barriers before and after the call).  ONE kernel:
 *   peer_params_host == NULL  (one-shot):  every rank reads all nranks buckets over NVLink, sums them in rank order,
 *        scales by grad_scale and applies the AdamW update of ldeq_adamw_step to its whole replica;
 *   peer_params_host != NULL  (two-shot):  rank `rank` reduces and updates only its 1/nranks slice (its slice of m, v is
 *        the only optimiser state it ever touches) and stores the updated parameters into every rank's replica
 *        (peer_params_host[r] = rank r's flat parameter buffer): nranks times less NVLink traffic.
 * Either way all replicas end up bit-identical. */
int ldeq_allreduce_adamw_step(ldeq_handle* h, float* params, float* const* peer_params_host,
                              const float* const* peer_grads_host, int nranks, int rank, float* m, float* v, int64_t n,
                              double lr, double beta1, double beta2, double eps, float decay, int64_t step,
                              float grad_scale, ldeq_stream stream);

/* ---- NCCL route for the same exchange (SURVEY.md 8(b)/(e): the flat fp32 parameter gradient is summed over the ranks once
 * per training step, model_train.jl:195-201 run data-parallel; the ODE state itself never crosses GPUs).  For hosts that
 * cannot map peer memory themselves (the Julia glue: one process per GPU, no torch).  libnccl.so.2 is loaded at run
 * time (LDEQ_NCCL_LIB overrides the name); the library has no link-time NCCL dependency.
 *   ldeq_comm_unique_id  rank 0 fills a 128-byte id (ncclGetUniqueId) that the host distributes to the other ranks;
 *   ldeq_comm_init       collective over the nranks processes (ncclCommInitRank) on the handle's device;
 *   ldeq_allreduce_grads in-place sum of n floats on `stream` (ncclAllReduce, ncclFloat32, ncclSum);
 *   ldeq_comm_destroy    also called by ldeq_destroy. */
#define LDEQ_COMM_ID_BYTES 128
int ldeq_comm_unique_id(ldeq_handle* h, void* id_out);
int ldeq_comm_init(ldeq_handle* h, const void* unique_id, int rank, int nranks);
int ldeq_allreduce_grads(ldeq_handle* h, float* grads_flat, int64_t n, ldeq_stream stream);
int ldeq_comm_destroy(ldeq_handle* h);

/* ---- diagnostics: the Float32 sine / cosine the integrator kernels evaluate, on device arrays of n arguments.
 * which = 0: the 13/19-instruction pair of the primal / adjoint kernels (csrc/ldeq_common.cuh);
 * which = 1: Base.sin / Base.cos(::Float32) as Julia computes them, used by the forward-dual pullback
 *            (csrc/ldeq_julia_trig.cuh; bit-equal to the oracle's restatement);
 * which = 2: the sine of the forward kernel alone (cos_out is zeroed). */
int ldeq_debug_trig(ldeq_handle* h, int which, const float* x, float* sin_out, float* cos_out, int64_t n,
                    ldeq_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* LDEQ_H */
