// ldeq_api.cu -- handle, right-hand-side objects and the GOKU solve entry points of libldeq.so.
//
// ldeq_solve_fwd / ldeq_solve_bwd are the drop-in for the body of
// diffeq_layer(::Decoder{<:GOKU}, l, t) (reference src/models/GOKU.jl:98-130) and its pullback.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "ldeq_internal.h"
#include "ldeq_rhs.cuh"
#include "ldeq_tsit5.cuh"
#include "ldeq_julia_trig.cuh"

namespace ldeq {

// ldeq_erk.cu: the forward kernel for solver = DP5 / BS3 / RK4 (built-in right-hand sides)
cudaError_t launch_erk_fwd(int solver, int dtype, bool friction, bool with_tape, const void* z0, const void* theta, const double* tg, int B,
                           int T, const KOpts& ko, void* traj, int32_t* ret, int32_t* na, int32_t* nr, const TapeView<float>& tv,
                           const GridInfo& gi, cudaStream_t s);

int set_err(ldeq_handle* h, int code, const char* what, cudaError_t ce) {
    if (h) {
        h->err = what ? what : "";
        if (ce != cudaSuccess) {
            h->err += ": ";
            h->err += cudaGetErrorString(ce);
        }
    }
    return code;
}

bool capturing(cudaStream_t s) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone;
}

int refuse_capture(ldeq_handle* h, cudaStream_t s, const char* what, const char* why) {
    if (!capturing(s)) return LDEQ_OK;
    std::string msg = std::string(what) + ": not available under CUDA graph capture (" + why + ")";
    return set_err(h, LDEQ_ERR_UNSUPPORTED, msg.c_str());
}

static bool same_grid(const std::vector<double>& a, const double* t, int T) {
    return a.size() == (size_t)T && std::memcmp(a.data(), t, (size_t)T * sizeof(double)) == 0;
}

// An immutable device copy of the grid upload_tgrid has just put into d_tgrid (ldeq_handle::grid_cache).  Eager solves
// never read these copies, so an unpinned one can be freed at any time.
static int cache_grid(ldeq_handle* h, int T, cudaStream_t s) {
    size_t lru = h->grid_cache.size();
    int unpinned = 0;
    for (size_t i = 0; i < h->grid_cache.size(); ++i) {
        ldeq_handle::GridEntry& g = h->grid_cache[i];
        if (same_grid(g.t, h->h_tgrid.data(), T)) { g.last_use = ++h->grid_clock; return LDEQ_OK; }
        if (!g.pinned) {
            ++unpinned;
            if (lru == h->grid_cache.size() || g.last_use < h->grid_cache[lru].last_use) lru = i;
        }
    }
    if (unpinned >= LDEQ_GRID_CACHE) {
        LDEQ_CUDA(cudaFreeAsync(h->grid_cache[lru].d, s));
        h->grid_cache.erase(h->grid_cache.begin() + lru);
    }
    ldeq_handle::GridEntry g;
    LDEQ_CUDA(cudaMallocAsync((void**)&g.d, (size_t)T * sizeof(double), s));
    LDEQ_CUDA(cudaMemcpyAsync(g.d, h->d_tgrid, (size_t)T * sizeof(double), cudaMemcpyDeviceToDevice, s));
    g.t = h->h_tgrid;
    g.t0 = h->grid_t0; g.h = h->grid_h; g.uniform = h->grid_uniform;
    g.last_use = ++h->grid_clock;
    h->grid_cache.push_back(std::move(g));
    return LDEQ_OK;
}

int upload_tgrid(ldeq_handle* h, const double* t_host, int T, cudaStream_t s) {
    if ((size_t)T > h->d_tgrid_cap) {
        // stream-ordered free so that kernels still reading the old grid finish first
        if (h->d_tgrid) LDEQ_CUDA(cudaFreeAsync(h->d_tgrid, s));
        h->d_tgrid = nullptr;
        h->d_tgrid_cap = 0;
        size_t cap = (size_t)T < 256 ? 256 : (size_t)T;
        LDEQ_CUDA(cudaMallocAsync((void**)&h->d_tgrid, cap * sizeof(double), s));
        h->d_tgrid_cap = cap;
        h->h_tgrid.clear();
    }
    if (!same_grid(h->h_tgrid, t_host, T)) {
        h->h_tgrid.assign(t_host, t_host + T);
        h->grid_t0 = t_host[0];
        h->grid_h = T > 1 ? t_host[1] - t_host[0] : 0.0;
        h->grid_uniform = T > 1;
#ifdef LDEQ_NO_UNIFORM_GRID
        h->grid_uniform = 0;
#endif
        for (int k = 0; k < T && h->grid_uniform; ++k)
            if (std::fma((double)k, h->grid_h, h->grid_t0) != t_host[k]) h->grid_uniform = 0;
        // source is pageable host memory: the runtime stages it before returning
        LDEQ_CUDA(cudaMemcpyAsync(h->d_tgrid, t_host, (size_t)T * sizeof(double), cudaMemcpyHostToDevice, s));
        return cache_grid(h, T, s);
    }
    return LDEQ_OK;
}

int ensure_scratch(ldeq_handle* h, int slot, size_t bytes, cudaStream_t s) {
    const bool graph = capturing(s);
    if (bytes <= h->scratch_cap[slot]) {
        h->scratch_captured[slot] |= graph;
        return LDEQ_OK;
    }
    if (graph) return set_err(h, LDEQ_ERR_UNSUPPORTED, "device scratch must grow, which cannot happen under CUDA graph capture: run the "
                                                       "same call once outside the capture first");
    if (h->scratch[slot]) {
        if (h->scratch_captured[slot]) {
            h->retired_scratch.push_back(h->scratch[slot]);  // a captured graph may still read it
        } else {
            LDEQ_CUDA(cudaDeviceSynchronize());
            LDEQ_CUDA(cudaFree(h->scratch[slot]));
        }
        h->scratch[slot] = nullptr;
        h->scratch_cap[slot] = 0;
        h->scratch_captured[slot] = false;
    }
    size_t cap = bytes + bytes / 8 + 4096;
    cudaError_t e = cudaMalloc(&h->scratch[slot], cap);
    if (e != cudaSuccess) return set_err(h, LDEQ_ERR_NOMEM, "cudaMalloc(scratch)", e);
    h->scratch_cap[slot] = cap;
    return LDEQ_OK;
}

KOpts to_kopts(const ldeq_opts* o) {
    KOpts k;
    k.abstol = o->abstol; k.reltol = o->reltol; k.dt = o->dt; k.dtmax = o->dtmax; k.dtmin = o->dtmin;
    k.gamma = o->gamma; k.qmin = o->qmin; k.qmax = o->qmax; k.beta1 = o->beta1; k.beta2 = o->beta2;
    k.qoldinit = o->qoldinit; k.qsteady_min = o->qsteady_min; k.qsteady_max = o->qsteady_max;
    k.maxiters = o->maxiters; k.adaptive = o->adaptive; k.controller_pow = o->controller_pow;
    return k;
}

// The forward kernel fills the tape's own copies (theta, grid, statistics) itself; a replay into a fresh tape (tape_heal)
// reads theta / the grid FROM the tape, where they already are.
template <class S>
static TapeView<S> fwd_tape_view(const ldeq_tape* tape, const void* theta, const double* tg) {
    return TapeView<S>{tape->t, (S*)tape->u, tape->info, tape->cap,
                       theta == tape->theta ? nullptr : (S*)tape->theta, tg == tape->tgrid ? nullptr : tape->tgrid,
                       tape->retcode, tape->naccept, tape->nreject};
}

template <class S, bool FRICTION, bool TAPE>
static cudaError_t launch_fwd(const void* z0, const void* theta, const double* tg, int B, int T, const KOpts& ko,
                              void* traj, int32_t* ret, int32_t* na, int32_t* nr, const ldeq_tape* tape,
                              const GridInfo& gi, cudaStream_t s) {
    TapeView<S> tv{nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (TAPE) tv = fwd_tape_view<S>(tape, theta, tg);
    const int grid = (B + LDEQ_FWD_THREADS - 1) / LDEQ_FWD_THREADS;
    const size_t smem = Ring<S, 2>::bytes(LDEQ_FWD_THREADS) + (T <= LDEQ_TGRID_SMEM_MAX ? (size_t)T * sizeof(double) : 0);
    tsit5_fwd_kernel<PendulumRHS<S, FRICTION>, S, TAPE><<<grid, LDEQ_FWD_THREADS, smem, s>>>(
        (const S*)z0, (const S*)theta, tg, B, T, ko, (S*)traj, ret, na, nr, tv, gi);
    return cudaGetLastError();
}

// The discrete-adjoint kernels re-deal the trajectories of a CTA to lanes by their accepted-step count (measured at
// 2^20 x 200: 1.135 -> 1.095 ms); LDEQ_BWD_SORT=0 keeps the batch order (A/B switch; the results are identical bit for bit).
int bwd_sort_lanes() {
    static const int on = [] { const char* e = getenv("LDEQ_BWD_SORT"); return (e && e[0] == '0') ? 0 : 1; }();
    return on;
}

template <class S, bool FRICTION>
static cudaError_t launch_bwd(const ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s) {
    TapeView<S> tv{tape->t, (S*)tape->u, tape->info, tape->cap, nullptr, nullptr, nullptr, nullptr, nullptr};
    const int grid = (tape->B + LDEQ_BWD_THREADS - 1) / LDEQ_BWD_THREADS;
    const size_t smem =
        Ring<S, 2>::bytes(LDEQ_BWD_THREADS) + (tape->T <= LDEQ_TGRID_SMEM_MAX ? (size_t)tape->T * sizeof(double) : 0);
    tsit5_bwd_kernel<PendulumRHS<S, FRICTION>, S><<<grid, LDEQ_BWD_THREADS, smem, s>>>(
        (const S*)tape->theta, tape->tgrid, tape->B, tape->T, (const S*)dtraj, tv, tape->retcode, tape->naccept,
        (S*)dz0, (S*)dtheta, GridInfo{tape->grid_t0, tape->grid_h, tape->grid_uniform, ld, bwd_sort_lanes()});
    return cudaGetLastError();
}

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

// shared memory of one CTA for a state of z_dim elements of `es` bytes: per-lane ring + staged time grid
static size_t ring_smem(int z_dim, size_t es, int threads, int T) {
    int rows = LDEQ_RING_BYTES / (z_dim * (int)es);
    rows = rows >= 64 ? 64 : rows >= 32 ? 32 : rows >= 16 ? 16 : rows >= 8 ? 8 : 4;
    return (size_t)rows * threads * z_dim * es + (T <= LDEQ_TGRID_SMEM_MAX ? (size_t)T * sizeof(double) : 0);
}

// kernels of an NVRTC-compiled user right-hand side (ldeq_user_rhs.cu): fn[] = {fwd f32, fwd f32 tape, fwd f64,
// fwd f64 tape, bwd f32, bwd f64}; same signatures as the built-in instantiations
static cudaError_t launch_user_fwd(void* const* fn, const ldeq_rhs* rhs, int dtype, const void* z0, const void* theta, const double* tg,
                                   int B, int T, const KOpts& ko, void* traj, int32_t* ret, int32_t* na, int32_t* nr,
                                   const ldeq_tape* tape, const GridInfo& gi, cudaStream_t s) {
    TapeView<float> tv{nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr};  // identical layout for float and double
    if (tape) tv = fwd_tape_view<float>(tape, theta, tg);
    KOpts kov = ko;
    GridInfo giv = gi;
    void* args[] = {&z0, &theta, &tg, &B, &T, &kov, &traj, &ret, &na, &nr, &tv, &giv};
    const int grid = (B + LDEQ_FWD_THREADS - 1) / LDEQ_FWD_THREADS;
    const size_t es = dtype == LDEQ_F32 ? 4 : 8;
    void* kfn = fn[(dtype == LDEQ_F32 ? 0 : 2) + (tape ? 1 : 0)];
    return cudaLaunchKernel(kfn, dim3(grid), dim3(LDEQ_FWD_THREADS), args, ring_smem(rhs->z_dim, es, LDEQ_FWD_THREADS, T), s);
}
static cudaError_t launch_user_bwd(void* const* fn, const ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s) {
    TapeView<float> tv{tape->t, (float*)tape->u, tape->info, tape->cap, nullptr, nullptr, nullptr, nullptr, nullptr};
    const void* theta = tape->theta;
    const double* tg = tape->tgrid;
    int B = tape->B, T = tape->T;
    const int32_t* ret = tape->retcode;
    const int32_t* na = tape->naccept;
    GridInfo giv{tape->grid_t0, tape->grid_h, tape->grid_uniform, ld, bwd_sort_lanes()};
    void* args[] = {&theta, &tg, &B, &T, &dtraj, &tv, &ret, &na, &dz0, &dtheta, &giv};
    const int grid = (B + LDEQ_BWD_THREADS - 1) / LDEQ_BWD_THREADS;
    const size_t es = tape->dtype == LDEQ_F32 ? 4 : 8;
    void* kfn = fn[tape->dtype == LDEQ_F32 ? 4 : 5];
    return cudaLaunchKernel(kfn, dim3(grid), dim3(LDEQ_BWD_THREADS), args, ring_smem(tape->z_dim, es, LDEQ_BWD_THREADS, T), s);
}

// fn[6..9] = forward-dual pullback {theta-seeded f32, u0-seeded f32, theta-seeded f64, u0-seeded f64}
static cudaError_t launch_user_fwdsens(void* const* fn, const ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s) {
    const void* z0 = tape->u;
    const void* theta = tape->theta;
    const double* tg = tape->tgrid;
    int B = tape->B, T = tape->T, np = 1;
    GridInfo gi{tape->grid_t0, tape->grid_h, tape->grid_uniform, ld};
    KOpts kov = tape->kopts;
    const int32_t* ret = tape->retcode;
    const int32_t* key = tape->naccept;  // lanes re-dealt by the primal step count (ldeq_fwdsens.cuh)
    const int grid = (B + 127) / 128;
    const int base = tape->dtype == LDEQ_F32 ? 6 : 8;
    void* args_p[] = {&z0, &theta, &tg, &B, &gi, &T, &kov, &np, &key, &dtraj, &ret, &dtheta};
    cudaError_t e = cudaLaunchKernel(fn[base], dim3(grid), dim3(128), args_p, 0, s);
    if (e != cudaSuccess) return e;
    void* args_u[] = {&z0, &theta, &tg, &B, &gi, &T, &kov, &np, &key, &dtraj, &ret, &dz0};
    return cudaLaunchKernel(fn[base + 1], dim3(grid), dim3(128), args_u, 0, s);
}

// Pinned two-int mirrors + events come from a per-handle pool: cudaMallocHost / cudaFreeHost cost milliseconds of host time
// (and the free synchronises the device), far more than a small solve.
bool slot_acquire(ldeq_handle* h, int32_t** h_info, cudaEvent_t* ev) {
    for (const ldeq_handle::Slot& sl : h->deferred_slots) slot_release(h, sl.h_info, sl.ev);
    h->deferred_slots.clear();
    if (h->free_slots.empty()) {
        const int n = 64;
        int32_t* blk = nullptr;
        if (cudaMallocHost((void**)&blk, n * 2 * sizeof(int32_t)) != cudaSuccess) return false;
        h->pinned_blocks.push_back(blk);
        for (int i = 0; i < n; ++i) {
            cudaEvent_t e;
            if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return false;
            h->free_slots.push_back({blk + 2 * i, e});
        }
    }
    ldeq_handle::Slot sl = h->free_slots.back();
    h->free_slots.pop_back();
    *h_info = sl.h_info;
    *ev = sl.ev;
    return true;
}
void slot_release(ldeq_handle* h, int32_t* h_info, cudaEvent_t ev) {
    if (h_info && ev) {
        cudaEventSynchronize(ev);  // the async copy into the slot must have landed before reuse
        if (h) h->free_slots.push_back({h_info, ev});
    }
}
static bool slot_get(ldeq_handle* h, ldeq_tape* tape) { return slot_acquire(h, &tape->h_info, &tape->ready); }
// Under capture the wait for the slot's copy is not allowed: the slot is handed back by the next slot_acquire instead.
static void slot_put(ldeq_handle* h, ldeq_tape* tape, cudaStream_t s) {
    if (tape->ready && capturing(s))
        h->deferred_slots.push_back({tape->h_info, tape->ready});
    else
        slot_release(h, tape->h_info, tape->ready);
    tape->h_info = nullptr;
    tape->ready = nullptr;
}

// Carve the step arrays of a tape with capacity `cap` out of one stream-ordered allocation.
static int tape_alloc(ldeq_handle* h, ldeq_tape* tape, int cap, cudaStream_t s) {
    const size_t es = tape->dtype == LDEQ_F32 ? 4 : 8;
    const size_t nB = (size_t)tape->B, c = (size_t)cap, ZD = tape->z_dim, PD = tape->p_dim;
    size_t off = 0;
    const size_t o_t = off;   off += align_up(c * nB * 8);
    const size_t o_u = off;   off += align_up(c * nB * ZD * es);
    const size_t o_th = off;  off += align_up(nB * PD * es);
    const size_t o_tg = off;  off += align_up((size_t)tape->T * 8);
    const size_t o_ret = off; off += align_up(nB * 4);
    const size_t o_na = off;  off += align_up(nB * 4);
    const size_t o_nr = off;  off += align_up(nB * 4);
    const size_t o_info = off; off += 256;
    void* base = nullptr;
    cudaError_t e = cudaMallocAsync(&base, off, s);
    if (e != cudaSuccess) return set_err(h, LDEQ_ERR_NOMEM, "cudaMallocAsync(tape)", e);
    char* bp = (char*)base;
    tape->base = base; tape->cap = cap;
    tape->t = (double*)(bp + o_t); tape->u = bp + o_u;
    tape->theta = bp + o_th; tape->tgrid = (double*)(bp + o_tg); tape->retcode = (int32_t*)(bp + o_ret);
    tape->naccept = (int32_t*)(bp + o_na); tape->nreject = (int32_t*)(bp + o_nr);
    tape->info = (int32_t*)(bp + o_info);
    cudaMemsetAsync(tape->info, 0, 8, s);
    return LDEQ_OK;
}

static cudaError_t dispatch_fwd(ldeq_handle* h, int solver, const ldeq_rhs* rhs, int dtype, const void* z0, const void* theta,
                                const double* tg, int B, int T, const KOpts& ko, void* traj, int32_t* ret, int32_t* na, int32_t* nr,
                                const ldeq_tape* tape, const GridInfo& gi, cudaStream_t s) {
    if (rhs->kind < 0) {
        void* const* fn = user_rhs_kernels(h, rhs, solver);
        if (!fn) return cudaErrorLaunchFailure;  // h->err holds the NVRTC log
        return launch_user_fwd(fn, rhs, dtype, z0, theta, tg, B, T, ko, traj, ret, na, nr, tape, gi, s);
    }
    const bool friction = rhs->kind == LDEQ_RHS_PENDULUM_FRICTION;
    if (solver != LDEQ_SOLVER_TSIT5) {
        TapeView<float> tv{nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr};
        if (tape) tv = fwd_tape_view<float>(tape, theta, tg);
        return launch_erk_fwd(solver, dtype, friction, tape != nullptr, z0, theta, tg, B, T, ko, traj, ret, na, nr, tv, gi, s);
    }
#define LDEQ_DISPATCH_FWD(S)                                                                              \
    (tape ? (friction ? launch_fwd<S, true, true>(z0, theta, tg, B, T, ko, traj, ret, na, nr, tape, gi, s)    \
                      : launch_fwd<S, false, true>(z0, theta, tg, B, T, ko, traj, ret, na, nr, tape, gi, s))  \
          : (friction ? launch_fwd<S, true, false>(z0, theta, tg, B, T, ko, traj, ret, na, nr, tape, gi, s)   \
                      : launch_fwd<S, false, false>(z0, theta, tg, B, T, ko, traj, ret, na, nr, tape, gi, s)))
    return dtype == LDEQ_F32 ? LDEQ_DISPATCH_FWD(float) : LDEQ_DISPATCH_FWD(double);
#undef LDEQ_DISPATCH_FWD
}

// A tape whose capacity turned out too small heals itself before the backward pass: the forward
// solve is replayed (same inputs, same arithmetic, hence the same steps) into a tape sized by the
// largest accepted-step count the first pass reported.  Costs one extra forward kernel, only then.
static int tape_heal(ldeq_handle* h, ldeq_tape* tape, cudaStream_t s) {
    if (tape->checked) return LDEQ_OK;
    LDEQ_CUDA(cudaEventSynchronize(tape->ready));
    tape->checked = true;
    if (tape->h_info[1] > h->tape_hint) h->tape_hint = tape->h_info[1];
    if (tape->h_info[0] == 0) return LDEQ_OK;
    ldeq_tape old = *tape;
    int rc = tape_alloc(h, tape, old.h_info[1], s);
    if (rc) { *tape = old; return rc; }
    const size_t es = tape->dtype == LDEQ_F32 ? 4 : 8;
    cudaMemcpyAsync(tape->theta, old.theta, (size_t)tape->B * tape->p_dim * es, cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(tape->tgrid, old.tgrid, (size_t)tape->T * 8, cudaMemcpyDeviceToDevice, s);
    // step 0 of the old tape holds u0 for every trajectory (capacity is always >= 1)
    cudaError_t e = dispatch_fwd(h, tape->solver, tape->rhs, tape->dtype, old.u, tape->theta,
                                 tape->tgrid, tape->B, tape->T, tape->kopts, nullptr, nullptr, nullptr,
                                 nullptr, tape, GridInfo{tape->grid_t0, tape->grid_h, tape->grid_uniform, tape->B}, s);
    h->launches += 1;
    cudaFreeAsync(old.base, s);
    if (e != cudaSuccess) return set_err(h, LDEQ_ERR_CUDA, "tsit5_fwd_kernel (tape replay) launch", e);
    return LDEQ_OK;
}

}  // namespace ldeq

using namespace ldeq;

extern "C" {

int ldeq_version(void) { return LDEQ_VERSION; }

void ldeq_opts_default(ldeq_opts* o) {
    std::memset(o, 0, sizeof(*o));
    o->abstol = 1e-6; o->reltol = 1e-3; o->adaptive = 1; o->controller_pow = 0; o->dt = 0.0; o->dtmax = 0.0;
    o->dtmin = 0.0; o->maxiters = 1000000; o->gamma = 0.9; o->qmin = 0.2; o->qmax = 10.0; o->beta1 = 7.0 / 50.0;
    o->beta2 = 2.0 / 25.0; o->qoldinit = 1e-4; o->qsteady_min = 1.0; o->qsteady_max = 1.0; o->tape_steps = 0;
    o->norm_mode = LDEQ_NORM_GLOBAL; o->mlp_math = LDEQ_MLP_MATH_FP32;
    o->sensealg = LDEQ_SENSE_FORWARD_DUAL;  // what the reference's diffeq structs ask for (pendulum.jl:11,58)
    o->solver = LDEQ_SOLVER_TSIT5;
}

int ldeq_opts_default_solver(ldeq_opts* o, int solver) {
    if (!o || solver < LDEQ_SOLVER_TSIT5 || solver > LDEQ_SOLVER_RK4) return LDEQ_ERR_INVALID;
    ldeq_opts_default(o);
    o->solver = solver;
    // OrdinaryDiffEq alg_utils.jl [3P]: beta2_default = 2/(5 order), beta1_default = 7/(10 order); DP5 has its own pair
    const double order = solver == LDEQ_SOLVER_BS3 ? 3.0 : solver == LDEQ_SOLVER_RK4 ? 4.0 : 5.0;
    o->beta2 = 2.0 / (5.0 * order);
    o->beta1 = 7.0 / (10.0 * order);
    if (solver == LDEQ_SOLVER_DP5) {
        o->beta2 = 4.0 / 100.0;
        o->beta1 = 1.0 / 5.0 - 3.0 * o->beta2 / 4.0;
    }
    return LDEQ_OK;
}

int ldeq_create(ldeq_handle** out, int device) {
    if (!out) return LDEQ_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return LDEQ_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return LDEQ_ERR_CUDA;
    ldeq_handle* h = new ldeq_handle();
    h->device = device;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    // keep stream-ordered allocations (tapes) in the pool instead of returning them to the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = h;
    return LDEQ_OK;
}

void ldeq_destroy(ldeq_handle* h) {
    if (!h) return;
    ldeq_comm_destroy(h);
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    if (h->d_tgrid) cudaFree(h->d_tgrid);
    for (int i = 0; i < 4; ++i)
        if (h->scratch[i]) cudaFree(h->scratch[i]);
    if (h->d_partials) cudaFree(h->d_partials);
    if (h->d_counter) cudaFree(h->d_counter);
    if (h->up) {
        cudaStreamDestroy(h->up);
        cudaStreamDestroy(h->down);
        for (int i = 0; i < LDEQ_MAX_SLABS; ++i) { cudaEventDestroy(h->ev_fwd[i]); cudaEventDestroy(h->ev_up[i]); }
        cudaEventDestroy(h->ev_join);
    }
    for (auto& g : h->grid_cache) cudaFree(g.d);
    for (void* p : h->retired_scratch) cudaFree(p);
    for (auto& sl : h->free_slots) cudaEventDestroy(sl.ev);
    for (auto& sl : h->deferred_slots) cudaEventDestroy(sl.ev);
    for (auto* blk : h->pinned_blocks) cudaFreeHost(blk);
    delete h;
}

const char* ldeq_last_error(const ldeq_handle* h) { return h ? h->err.c_str() : "null handle"; }
int64_t ldeq_launch_count(const ldeq_handle* h) { return h ? h->launches : 0; }

int ldeq_rhs_builtin(ldeq_handle* h, int kind, ldeq_rhs** out) {
    if (!h || !out) return LDEQ_ERR_INVALID;
    if (kind != LDEQ_RHS_PENDULUM && kind != LDEQ_RHS_PENDULUM_FRICTION)
        return set_err(h, LDEQ_ERR_INVALID, "unknown built-in rhs kind");
    ldeq_rhs* r = new ldeq_rhs();
    r->kind = kind;
    r->z_dim = 2;
    r->p_dim = 1;
    *out = r;
    return LDEQ_OK;
}

int ldeq_rhs_dims(const ldeq_rhs* rhs, int* z_dim, int* p_dim) {
    if (!rhs) return LDEQ_ERR_INVALID;
    if (z_dim) *z_dim = rhs->z_dim;
    if (p_dim) *p_dim = rhs->p_dim;
    return LDEQ_OK;
}

}  // extern "C"

namespace ldeq {

// The device grid a solve reads: d_tgrid for eager calls, an immutable cache entry under capture.
struct GridRef {
    const double* d;
    double t0, h;
    int uniform;
};
static GridRef eager_grid(const ldeq_handle* h) { return GridRef{h->d_tgrid, h->grid_t0, h->grid_h, h->grid_uniform}; }

// ---- one column slab of a solve -----------------------------------------------------------------------
// All pointers are already offset to the slab's first trajectory; `ld` is the row stride of traj (trajectories of
// the whole batch).  The grid is on the device (upload_tgrid or the grid cache).  `graph`: the stream is capturing, so
// a tape gets no host mirror of its statistics and no event.
static int solve_fwd_slab(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0, const void* theta, const double* t_host,
                          const GridRef& grid, bool graph, int B, int ld, int T, const ldeq_opts* opts, void* traj_out,
                          int32_t* retcode, int32_t* naccept, int32_t* nreject, ldeq_tape** tape_out, cudaStream_t s) {
    KOpts ko = to_kopts(opts);
    const int ZD = rhs->z_dim, PD = rhs->p_dim;
    const bool fwd_dual = tape_out && opts->sensealg == LDEQ_SENSE_FORWARD_DUAL;
    ldeq_tape* tape = nullptr;
    int rc;
    if (tape_out) {
        *tape_out = nullptr;
        tape = new ldeq_tape();
        tape->dtype = dtype; tape->rhs_kind = rhs->kind; tape->rhs = rhs; tape->B = B; tape->T = T;
        tape->z_dim = ZD; tape->p_dim = PD; tape->kopts = ko;
        tape->grid_t0 = grid.t0; tape->grid_h = grid.h; tape->grid_uniform = grid.uniform;
        long long cap = opts->tape_steps;
        tape->sense = opts->sensealg;
        tape->solver = opts->solver;
        if (fwd_dual) {
            cap = 1;  // the dual re-solves need only u0 (record 0), theta, the grid and the options
        } else if (cap <= 0) {
            if (opts->adaptive) {
                cap = T > 64 ? T : 64;
                if (cap < (long long)h->tape_hint + h->tape_hint / 4) cap = (long long)h->tape_hint + h->tape_hint / 4;
            } else {
                cap = (long long)((t_host[T - 1] - t_host[0]) / opts->dt) + 3;
            }
        }
        if (cap > opts->maxiters) cap = opts->maxiters;
        if (cap > (1 << 24)) cap = 1 << 24;
        if (cap < 1) cap = 1;
        rc = tape_alloc(h, tape, (int)cap, s);
        if (rc) { delete tape; return rc; }
        if (!graph && !slot_get(h, tape)) {
            cudaFreeAsync(tape->base, s);
            delete tape;
            return set_err(h, LDEQ_ERR_NOMEM, "tape host mirror");
        }
        // theta, the grid, the statistics and u0 (record 0) reach the tape through the forward kernel itself (TapeView)
    }
    cudaError_t e = dispatch_fwd(h, opts->solver, rhs, dtype, z0, theta, grid.d, B, T, ko, traj_out, retcode, naccept, nreject, tape,
                                 GridInfo{grid.t0, grid.h, grid.uniform, ld}, s);
    h->launches += 1;
    if (e != cudaSuccess) {
        if (tape) {
            cudaFreeAsync(tape->base, s);
            if (tape->ready) cudaEventRecord(tape->ready, s);
            slot_put(h, tape, s);
            delete tape;
        }
        if (rhs->kind < 0 && e == cudaErrorLaunchFailure && !h->err.empty() && h->err.compare(0, 5, "NVRTC") == 0) return LDEQ_ERR_COMPILE;
        return set_err(h, LDEQ_ERR_CUDA, "tsit5_fwd_kernel launch", e);
    }
    if (tape) {
        if (tape->ready) {
            cudaMemcpyAsync(tape->h_info, tape->info, 8, cudaMemcpyDeviceToHost, s);
            cudaEventRecord(tape->ready, s);
        }
        *tape_out = tape;
    }
    return LDEQ_OK;
}

// reverse pass of one slab (a single-part tape); dtraj / dz0 / dtheta already offset, ld = row stride of dtraj
static int solve_bwd_slab(ldeq_handle* h, ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s) {
    void* const* ufn = nullptr;
    if (tape->rhs_kind < 0 && !(ufn = user_rhs_kernels(h, tape->rhs, tape->solver))) return LDEQ_ERR_COMPILE;
    if (tape->sense == LDEQ_SENSE_FORWARD_DUAL) {
        const cudaError_t e2 = tape->rhs_kind < 0 ? launch_user_fwdsens(ufn, tape, dtraj, ld, dz0, dtheta, s)
                                                  : launch_fwdsens(tape, dtraj, ld, dz0, dtheta, s);
        h->launches += 2;
        if (e2 != cudaSuccess) return set_err(h, LDEQ_ERR_CUDA, "tsit5_fwdsens_kernel launch", e2);
        return LDEQ_OK;
    }
    int rc = tape_heal(h, tape, s);
    if (rc) return rc;
    const bool fr = tape->rhs_kind == LDEQ_RHS_PENDULUM_FRICTION;
    cudaError_t e;
    if (tape->rhs_kind < 0)
        e = launch_user_bwd(ufn, tape, dtraj, ld, dz0, dtheta, s);
    else if (tape->solver != LDEQ_SOLVER_TSIT5)
        e = launch_erk_bwd(tape, dtraj, ld, dz0, dtheta, s);
    else if (tape->dtype == LDEQ_F32)
        e = fr ? launch_bwd<float, true>(tape, dtraj, ld, dz0, dtheta, s) : launch_bwd<float, false>(tape, dtraj, ld, dz0, dtheta, s);
    else
        e = fr ? launch_bwd<double, true>(tape, dtraj, ld, dz0, dtheta, s) : launch_bwd<double, false>(tape, dtraj, ld, dz0, dtheta, s);
    h->launches += 1;
    if (e != cudaSuccess) return set_err(h, LDEQ_ERR_CUDA, "tsit5_bwd_kernel launch", e);
    return LDEQ_OK;
}

static int check_solve_args(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0, const void* theta, const double* t_host,
                            int B, int T, const ldeq_opts* opts) {
    if (!rhs || !z0 || !theta || !t_host || !opts) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    if (B < 0 || T < 1) return set_err(h, LDEQ_ERR_INVALID, "B must be >= 0 and T >= 1");
    if (dtype != LDEQ_F32 && dtype != LDEQ_F64) return set_err(h, LDEQ_ERR_INVALID, "dtype");
    if (!opts->adaptive && !(opts->dt > 0.0)) return set_err(h, LDEQ_ERR_INVALID, "adaptive = 0 needs dt > 0");
    for (int k = 1; k < T; ++k)
        if (!(t_host[k] > t_host[k - 1])) return set_err(h, LDEQ_ERR_INVALID, "t must be strictly increasing");
    if (opts->sensealg != LDEQ_SENSE_DISCRETE_ADJOINT && opts->sensealg != LDEQ_SENSE_FORWARD_DUAL)
        return set_err(h, LDEQ_ERR_INVALID, "sensealg");
    if (opts->solver < LDEQ_SOLVER_TSIT5 || opts->solver > LDEQ_SOLVER_RK4)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "solver: LDEQ_SOLVER_TSIT5 / DP5 / BS3 / RK4 are built");
    if (opts->solver == LDEQ_SOLVER_RK4 && opts->adaptive)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "solver RK4: fixed step only (adaptive = 0, dt > 0); OrdinaryDiffEq's defect-control estimate of adaptive RK4 is not built");
    return LDEQ_OK;
}

static void free_parts(ldeq_handle* h, ldeq_tape* tape, cudaStream_t s) {
    for (ldeq_tape* p : tape->parts) {
        if (p->base) cudaFreeAsync(p->base, s);
        slot_put(h, p, s);
        delete p;
    }
    tape->parts.clear();
}

// ---- host-buffer pipeline ---------------------------------------------------------------------------------
// Trajectories are independent, so a host-resident batch is cut into column slabs: the download of slab i's
// trajectories (copy stream "down") runs under the kernel of slab i+1 (the caller's stream), and the upload of slab
// i+1's cotangent (copy stream "up") under the reverse pass of slab i.  B200 has separate copy engines per direction:
// in the combined call the PCIe link is busy in both directions at once.
static int host_streams(ldeq_handle* h) {
    if (h->up) return LDEQ_OK;
    LDEQ_CUDA(cudaStreamCreateWithFlags(&h->up, cudaStreamNonBlocking));
    LDEQ_CUDA(cudaStreamCreateWithFlags(&h->down, cudaStreamNonBlocking));
    for (int i = 0; i < LDEQ_MAX_SLABS; ++i) {
        LDEQ_CUDA(cudaEventCreateWithFlags(&h->ev_fwd[i], cudaEventDisableTiming));
        LDEQ_CUDA(cudaEventCreateWithFlags(&h->ev_up[i], cudaEventDisableTiming));
    }
    LDEQ_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    return LDEQ_OK;
}
static int slab_count(int B) {
    // slabs of at least 32 Ki trajectories (a slab must still fill the GPU: 148 SMs x 640 resident threads), at most 8
    int n = B / 32768;
    return n < 1 ? 1 : n > LDEQ_MAX_SLABS ? LDEQ_MAX_SLABS : n;
}
static void slab_bounds(int B, int n, int i, int* b0, int* nb) {
    // multiples of 128 trajectories (CTA size), remainder to the last slab
    int per = ((B / n) + 127) / 128 * 128;
    *b0 = i * per < B ? i * per : B;
    int e = (i == n - 1) ? B : ((i + 1) * per < B ? (i + 1) * per : B);
    *nb = e - *b0;
}

struct HostBufs {
    char *z0, *th, *traj, *dtraj, *dz0, *dth;
    int32_t *ret, *na, *nr;
};
static int host_bufs(ldeq_handle* h, size_t nz, size_t np, size_t nt, int B, bool fwd, bool bwd, HostBufs* hb, cudaStream_t s) {
    int rc;
    if ((rc = ensure_scratch(h, 0, 2 * align_up(nz) + 2 * align_up(np) + 3 * align_up((size_t)B * 4), s))) return rc;
    char* in = (char*)h->scratch[0];
    hb->z0 = in; in += align_up(nz);
    hb->th = in; in += align_up(np);
    hb->dz0 = in; in += align_up(nz);
    hb->dth = in; in += align_up(np);
    hb->ret = (int32_t*)in; in += align_up((size_t)B * 4);
    hb->na = (int32_t*)in; in += align_up((size_t)B * 4);
    hb->nr = (int32_t*)in;
    hb->traj = hb->dtraj = nullptr;
    if (fwd) { if ((rc = ensure_scratch(h, 1, nt, s))) return rc; hb->traj = (char*)h->scratch[1]; }
    if (bwd) { if ((rc = ensure_scratch(h, 2, nt, s))) return rc; hb->dtraj = (char*)h->scratch[2]; }
    return LDEQ_OK;
}

}  // namespace ldeq

using namespace ldeq;

extern "C" {

int ldeq_solve_fwd(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0, const void* theta,
                   const double* t_host, int B, int T, const ldeq_opts* opts, void* traj_out, int32_t* retcode,
                   int32_t* naccept, int32_t* nreject, ldeq_tape** tape_out, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (tape_out) *tape_out = nullptr;
    int rc = check_solve_args(h, rhs, dtype, z0, theta, t_host, B, T, opts);
    if (rc) return rc;
    if (!traj_out && !tape_out && !naccept) return set_err(h, LDEQ_ERR_INVALID, "nothing to compute: traj_out, tape_out and naccept are all null");
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    if (B == 0) return LDEQ_OK;
    if (!capturing(s)) {
        if ((rc = upload_tgrid(h, t_host, T, s))) return rc;
        return solve_fwd_slab(h, rhs, dtype, z0, theta, t_host, eager_grid(h), false, B, B, T, opts, traj_out, retcode, naccept, nreject,
                              tape_out, s);
    }
    // Under capture nothing may be enqueued before every check has passed, so that a refusal leaves the capture intact.
    if (tape_out && opts->sensealg != LDEQ_SENSE_FORWARD_DUAL)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "ldeq_solve_fwd: a discrete-adjoint tape is not available under CUDA graph capture (its "
                                                "reverse pass reads the tape's overflow count on the host)");
    if (rhs->kind < 0 && opts->solver != LDEQ_SOLVER_TSIT5 && !rhs->alt[opts->solver].module)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "ldeq_solve_fwd: the right-hand side has not been compiled for this solver yet, and NVRTC "
                                                "cannot run under CUDA graph capture: solve once outside the capture first");
    ldeq_handle::GridEntry* g = nullptr;
    for (auto& e : h->grid_cache)
        if (same_grid(e.t, t_host, T)) { g = &e; break; }
    if (!g)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "ldeq_solve_fwd: the time grid is not on the device, and a copy from host memory cannot be "
                                                "captured: solve once on this grid outside the capture first");
    g->pinned = true;  // the graph reads g->d for as long as the handle lives
    return solve_fwd_slab(h, rhs, dtype, z0, theta, t_host, GridRef{g->d, g->t0, g->h, g->uniform}, true, B, B, T, opts, traj_out, retcode,
                          naccept, nreject, tape_out, s);
}

int ldeq_solve_bwd(ldeq_handle* h, ldeq_tape* tape, const void* dtraj, void* dz0, void* dtheta, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!tape || !dtraj || !dz0 || !dtheta) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    if (capturing(s)) {
        if (!tape->parts.empty() || tape->sense != LDEQ_SENSE_FORWARD_DUAL)
            return set_err(h, LDEQ_ERR_UNSUPPORTED, "ldeq_solve_bwd: only the forward-dual pullback of a device solve is available under CUDA "
                                                    "graph capture (the discrete adjoint reads the tape's overflow count on the host)");
        if (tape->rhs_kind < 0 && tape->solver != LDEQ_SOLVER_TSIT5 && !tape->rhs->alt[tape->solver].module)
            return set_err(h, LDEQ_ERR_UNSUPPORTED, "ldeq_solve_bwd: the right-hand side has not been compiled for this solver yet, and "
                                                    "NVRTC cannot run under CUDA graph capture");
    }
    if (tape->parts.empty()) return solve_bwd_slab(h, tape, dtraj, tape->B, dz0, dtheta, s);
    // a tape recorded slab by slab (ldeq_solve_fwd_host): same column slabs of the device arrays
    const size_t es = tape->dtype == LDEQ_F32 ? 4 : 8;
    for (size_t i = 0; i < tape->parts.size(); ++i) {
        ldeq_tape* p = tape->parts[i];
        const size_t b0 = (size_t)tape->part_b0[i];
        int rc = solve_bwd_slab(h, p, (const char*)dtraj + b0 * tape->z_dim * es, tape->B, (char*)dz0 + b0 * tape->z_dim * es,
                                (char*)dtheta + b0 * tape->p_dim * es, s);
        if (rc) return rc;
    }
    return LDEQ_OK;
}

int ldeq_tape_overflow(ldeq_handle* h, ldeq_tape* tape, int32_t* count_host, ldeq_stream stream) {
    if (!h || !tape || !count_host) return LDEQ_ERR_INVALID;
    int rc = refuse_capture(h, (cudaStream_t)stream, "ldeq_tape_overflow", "it waits for the forward kernel and reads its result on the host");
    if (rc) return rc;
    *count_host = 0;
    auto one = [&](ldeq_tape* t) -> int {
        if (!t->ready) return LDEQ_OK;  // recorded under capture: a forward-dual tape, which cannot overflow
        LDEQ_CUDA(cudaEventSynchronize(t->ready));
        if (t->sense == LDEQ_SENSE_FORWARD_DUAL) return LDEQ_OK;  // the dual re-solves keep no step records: nothing can overflow
        *count_host += t->checked && t->h_info[0] > 0 && t->cap >= t->h_info[1] ? 0 : t->h_info[0];
        return LDEQ_OK;
    };
    if (tape->parts.empty()) return one(tape);
    for (ldeq_tape* p : tape->parts) { int rc = one(p); if (rc) return rc; }
    return LDEQ_OK;
}

void ldeq_tape_free(ldeq_handle* h, ldeq_tape* tape, ldeq_stream stream) {
    if (!tape) return;
    if (h) cudaSetDevice(h->device);
    free_parts(h, tape, (cudaStream_t)stream);
    if (tape->base) cudaFreeAsync(tape->base, (cudaStream_t)stream);
    slot_put(h, tape, (cudaStream_t)stream);
    delete tape;
}

int ldeq_solve_fwd_host(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0_host, const void* theta_host,
                        const double* t_host, int B, int T, const ldeq_opts* opts, void* traj_out_host,
                        int32_t* retcode_host, int32_t* naccept_host, int32_t* nreject_host, ldeq_tape** tape_out,
                        ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (tape_out) *tape_out = nullptr;
    int rc = check_solve_args(h, rhs, dtype, z0_host, theta_host, t_host, B, T, opts);
    if (rc) return rc;
    if (!traj_out_host) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    if (B <= 0) return set_err(h, LDEQ_ERR_INVALID, "B must be > 0");
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = refuse_capture(h, s, "ldeq_solve_fwd_host", "it stages through host memory and synchronises the stream"))) return rc;
    LDEQ_CUDA(cudaSetDevice(h->device));
    if ((rc = host_streams(h))) return rc;
    const size_t es = dtype == LDEQ_F32 ? 4 : 8, zb = (size_t)rhs->z_dim * es, pb = (size_t)rhs->p_dim * es;
    const size_t nz = (size_t)B * zb, np = (size_t)B * pb, nt = nz * (size_t)T;
    HostBufs hb;
    if ((rc = host_bufs(h, nz, np, nt, B, true, false, &hb, s))) return rc;
    if ((rc = upload_tgrid(h, t_host, T, s))) return rc;
    LDEQ_CUDA(cudaMemcpyAsync(hb.z0, z0_host, nz, cudaMemcpyHostToDevice, s));
    LDEQ_CUDA(cudaMemcpyAsync(hb.th, theta_host, np, cudaMemcpyHostToDevice, s));
    ldeq_tape* parent = nullptr;
    if (tape_out) {
        parent = new ldeq_tape();
        parent->dtype = dtype; parent->rhs_kind = rhs->kind; parent->rhs = rhs; parent->B = B; parent->T = T;
        parent->z_dim = rhs->z_dim; parent->p_dim = rhs->p_dim; parent->sense = opts->sensealg; parent->solver = opts->solver;
    }
    const int ns = slab_count(B);
    for (int i = 0; i < ns; ++i) {
        int b0, nb;
        slab_bounds(B, ns, i, &b0, &nb);
        if (nb <= 0) continue;
        ldeq_tape* part = nullptr;
        rc = solve_fwd_slab(h, rhs, dtype, hb.z0 + b0 * zb, hb.th + b0 * pb, t_host, eager_grid(h), false, nb, B, T, opts, hb.traj + b0 * zb, hb.ret + b0,
                            hb.na + b0, hb.nr + b0, parent ? &part : nullptr, s);
        if (rc) { if (parent) { free_parts(h, parent, s); delete parent; } return rc; }
        if (parent) { parent->parts.push_back(part); parent->part_b0.push_back(b0); }
        // this slab's columns of every row: a strided (2-D) download behind the kernel that produced them
        LDEQ_CUDA(cudaEventRecord(h->ev_fwd[i], s));
        LDEQ_CUDA(cudaStreamWaitEvent(h->down, h->ev_fwd[i], 0));
        LDEQ_CUDA(cudaMemcpy2DAsync((char*)traj_out_host + b0 * zb, (size_t)B * zb, hb.traj + b0 * zb, (size_t)B * zb, (size_t)nb * zb,
                                    (size_t)T, cudaMemcpyDeviceToHost, h->down));
    }
    if (retcode_host) LDEQ_CUDA(cudaMemcpyAsync(retcode_host, hb.ret, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    if (naccept_host) LDEQ_CUDA(cudaMemcpyAsync(naccept_host, hb.na, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    if (nreject_host) LDEQ_CUDA(cudaMemcpyAsync(nreject_host, hb.nr, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    LDEQ_CUDA(cudaStreamSynchronize(s));
    LDEQ_CUDA(cudaStreamSynchronize(h->down));
    if (tape_out) *tape_out = parent;
    return LDEQ_OK;
}

int ldeq_solve_bwd_host(ldeq_handle* h, ldeq_tape* tape, const void* dtraj_host, void* dz0_host, void* dtheta_host,
                        ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!tape || !dtraj_host || !dz0_host || !dtheta_host) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    if ((rc = refuse_capture(h, s, "ldeq_solve_bwd_host", "it stages through host memory and synchronises the stream"))) return rc;
    LDEQ_CUDA(cudaSetDevice(h->device));
    if ((rc = host_streams(h))) return rc;
    const size_t es = tape->dtype == LDEQ_F32 ? 4 : 8, zb = (size_t)tape->z_dim * es, pb = (size_t)tape->p_dim * es;
    const int B = tape->B, T = tape->T;
    const size_t nz = (size_t)B * zb, np = (size_t)B * pb, nt = nz * (size_t)T;
    HostBufs hb;
    if ((rc = host_bufs(h, nz, np, nt, B, false, true, &hb, s))) return rc;
    // every part's cotangent slab goes up on the copy stream; its reverse pass follows on the caller's stream
    const size_t nparts = tape->parts.empty() ? 1 : tape->parts.size();
    LDEQ_CUDA(cudaEventRecord(h->ev_join, s));   // uploads must not overtake earlier work of the caller on this scratch
    LDEQ_CUDA(cudaStreamWaitEvent(h->up, h->ev_join, 0));
    for (size_t i = 0; i < nparts; ++i) {
        ldeq_tape* p = tape->parts.empty() ? tape : tape->parts[i];
        const size_t b0 = tape->parts.empty() ? 0 : (size_t)tape->part_b0[i];
        LDEQ_CUDA(cudaMemcpy2DAsync(hb.dtraj + b0 * zb, (size_t)B * zb, (const char*)dtraj_host + b0 * zb, (size_t)B * zb,
                                    (size_t)p->B * zb, (size_t)T, cudaMemcpyHostToDevice, h->up));
        LDEQ_CUDA(cudaEventRecord(h->ev_up[i % LDEQ_MAX_SLABS], h->up));
        LDEQ_CUDA(cudaStreamWaitEvent(s, h->ev_up[i % LDEQ_MAX_SLABS], 0));
        rc = solve_bwd_slab(h, p, hb.dtraj + b0 * zb, B, hb.dz0 + b0 * zb, hb.dth + b0 * pb, s);
        if (rc) return rc;
    }
    LDEQ_CUDA(cudaMemcpyAsync(dz0_host, hb.dz0, nz, cudaMemcpyDeviceToHost, s));
    LDEQ_CUDA(cudaMemcpyAsync(dtheta_host, hb.dth, np, cudaMemcpyDeviceToHost, s));
    LDEQ_CUDA(cudaStreamSynchronize(s));
    return LDEQ_OK;
}

int ldeq_solve_fwd_bwd_host(ldeq_handle* h, const ldeq_rhs* rhs, int dtype, const void* z0_host, const void* theta_host,
                            const double* t_host, int B, int T, const ldeq_opts* opts, const void* dtraj_host,
                            void* traj_out_host, void* dz0_host, void* dtheta_host, int32_t* retcode_host,
                            int32_t* naccept_host, int32_t* nreject_host, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    int rc = check_solve_args(h, rhs, dtype, z0_host, theta_host, t_host, B, T, opts);
    if (rc) return rc;
    if (!dtraj_host || !traj_out_host || !dz0_host || !dtheta_host) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    if (B <= 0) return set_err(h, LDEQ_ERR_INVALID, "B must be > 0");
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = refuse_capture(h, s, "ldeq_solve_fwd_bwd_host", "it stages through host memory and synchronises the stream"))) return rc;
    LDEQ_CUDA(cudaSetDevice(h->device));
    if ((rc = host_streams(h))) return rc;
    const size_t es = dtype == LDEQ_F32 ? 4 : 8, zb = (size_t)rhs->z_dim * es, pb = (size_t)rhs->p_dim * es;
    const size_t nz = (size_t)B * zb, np = (size_t)B * pb, nt = nz * (size_t)T;
    HostBufs hb;
    if ((rc = host_bufs(h, nz, np, nt, B, true, true, &hb, s))) return rc;
    if ((rc = upload_tgrid(h, t_host, T, s))) return rc;
    LDEQ_CUDA(cudaMemcpyAsync(hb.z0, z0_host, nz, cudaMemcpyHostToDevice, s));
    LDEQ_CUDA(cudaMemcpyAsync(hb.th, theta_host, np, cudaMemcpyHostToDevice, s));
    LDEQ_CUDA(cudaEventRecord(h->ev_join, s));
    LDEQ_CUDA(cudaStreamWaitEvent(h->up, h->ev_join, 0));
    const int ns = slab_count(B);
    // the whole cotangent streams up slab by slab while the forward slabs stream down
    for (int i = 0; i < ns; ++i) {
        int b0, nb;
        slab_bounds(B, ns, i, &b0, &nb);
        if (nb <= 0) continue;
        LDEQ_CUDA(cudaMemcpy2DAsync(hb.dtraj + b0 * zb, (size_t)B * zb, (const char*)dtraj_host + b0 * zb, (size_t)B * zb,
                                    (size_t)nb * zb, (size_t)T, cudaMemcpyHostToDevice, h->up));
        LDEQ_CUDA(cudaEventRecord(h->ev_up[i], h->up));
    }
    for (int i = 0; i < ns; ++i) {
        int b0, nb;
        slab_bounds(B, ns, i, &b0, &nb);
        if (nb <= 0) continue;
        ldeq_tape* part = nullptr;
        rc = solve_fwd_slab(h, rhs, dtype, hb.z0 + b0 * zb, hb.th + b0 * pb, t_host, eager_grid(h), false, nb, B, T, opts, hb.traj + b0 * zb, hb.ret + b0,
                            hb.na + b0, hb.nr + b0, &part, s);
        if (rc) return rc;
        LDEQ_CUDA(cudaEventRecord(h->ev_fwd[i], s));
        LDEQ_CUDA(cudaStreamWaitEvent(h->down, h->ev_fwd[i], 0));
        LDEQ_CUDA(cudaMemcpy2DAsync((char*)traj_out_host + b0 * zb, (size_t)B * zb, hb.traj + b0 * zb, (size_t)B * zb, (size_t)nb * zb,
                                    (size_t)T, cudaMemcpyDeviceToHost, h->down));
        LDEQ_CUDA(cudaStreamWaitEvent(s, h->ev_up[i], 0));
        rc = solve_bwd_slab(h, part, hb.dtraj + b0 * zb, B, hb.dz0 + b0 * zb, hb.dth + b0 * pb, s);
        cudaFreeAsync(part->base, s);
        slot_put(h, part, s);
        delete part;
        if (rc) return rc;
    }
    LDEQ_CUDA(cudaMemcpyAsync(dz0_host, hb.dz0, nz, cudaMemcpyDeviceToHost, s));
    LDEQ_CUDA(cudaMemcpyAsync(dtheta_host, hb.dth, np, cudaMemcpyDeviceToHost, s));
    if (retcode_host) LDEQ_CUDA(cudaMemcpyAsync(retcode_host, hb.ret, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    if (naccept_host) LDEQ_CUDA(cudaMemcpyAsync(naccept_host, hb.na, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    if (nreject_host) LDEQ_CUDA(cudaMemcpyAsync(nreject_host, hb.nr, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    LDEQ_CUDA(cudaStreamSynchronize(s));
    LDEQ_CUDA(cudaStreamSynchronize(h->down));
    return LDEQ_OK;
}

// ---- diagnostics ------------------------------------------------------------------------------------------
__global__ void debug_trig_kernel(int which, const float* __restrict__ x, float* __restrict__ sn, float* __restrict__ cs, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float a, b;
    if (which == 0) fast_sincosf(x[i], &a, &b);
    else if (which == 1) jl_sincosf(x[i], &a, &b);
    else { a = fast_sinf(x[i]); b = 0.0f; }
    sn[i] = a;
    cs[i] = b;
}

int ldeq_debug_trig(ldeq_handle* h, int which, const float* x, float* sin_out, float* cos_out, int64_t n, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!x || !sin_out || !cos_out || n < 0 || which < 0 || which > 2) return set_err(h, LDEQ_ERR_INVALID, "bad argument");
    LDEQ_CUDA(cudaSetDevice(h->device));
    if (n == 0) return LDEQ_OK;
    debug_trig_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(which, x, sin_out, cos_out, n);
    h->launches += 1;
    LDEQ_CUDA(cudaGetLastError());
    return LDEQ_OK;
}

}  // extern "C"
