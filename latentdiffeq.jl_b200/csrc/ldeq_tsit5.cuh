// ldeq_tsit5.cuh -- fused Tsit5 integrator kernels for B independent small ODE systems (sm_100a).
//
// Replaces everything below `solve(ens_prob, solver, EnsembleThreads(); ...)` at reference
// src/models/GOKU.jl:111-125: one THREAD per trajectory holds the state, the seven stage slopes,
// its own step size and PI-controller memory in registers for the whole time span, emits the
// saveat points through the Tsit5 dense interpolant straight into the (z,B,T) output layout
// (so the reference's Array + permutedims passes, GOKU.jl:124-125, never exist), and applies the
// NaN-block failure rule of GOKU.jl:114.  The backward kernel is the discrete adjoint of exactly
// the accepted steps the forward kernel recorded on its tape.
//
// Time (t, dt, Theta, the controller) is Float64 even when the state is Float32: the reference's
// time grid is a Float64 range while its state is Float32 (SURVEY.md 7.2), and fixed-step
// accepted-step counts must be identical.
#pragma once

#include "ldeq_common.cuh"
#include "ldeq_erk.cuh"

namespace ldeq {

#define LDEQ_FWD_THREADS 128
#define LDEQ_BWD_THREADS 128
#ifndef LDEQ_FWD_MINBLOCKS
#define LDEQ_FWD_MINBLOCKS 5  // measured: 1.50 ms -> 1.41 ms at 2^20 x 200 (6 CTAs/SM spills and is slower)
#endif
#ifndef LDEQ_BWD_MINBLOCKS
#define LDEQ_BWD_MINBLOCKS 4
#endif

// Accepted-step tape, step-major so that a warp reading/writing step n touches contiguous memory:
//   t[n*B + b], u[(n*B + b)*ZD + d]   -- the start time and the state of accepted step n.
// The step size is not stored: the reverse pass takes dt_n = t_{n+1} - t_n (t_{na} = tend), which equals the forward
// pass' dt_n to a few ulp of t (1e-15 relative; the adjoint of the Float64 build agrees with the oracle to 1e-9 either
// way) and keeps the tape at 8 + ZD sizeof(S) bytes per accepted step (16 B for the Float32 pendulum, was 24).
template <class S> struct TapeView {
    double* t;
    S* u;
    int* info;  // info[0]: trajectories that ran past `cap`; info[1]: largest accepted-step count
    int cap;
    // the tape's own copies of what the reverse pass needs, written by the forward kernel itself (no extra copy
    // launches around a solve: at small batches they cost as much as the kernel); null = skip
    S* theta;        // (p,B)
    double* tgrid;   // T
    int* ret;        // B
    int* na;         // B
    int* nr;         // B
};

// ---- the seven stages --------------------------------------------------------------------------
// k[0] holds f(u) on entry (FSAL).  Fills k[1..6] and un.  With KEEP (reverse pass), also returns the stage inputs
// g[0..5] (g[0] = u) and the RHS' auxiliaries aux[0..5] for the reverse sweep; k[6] = f(u_{n+1}) is then NOT
// evaluated -- its value is not needed by the adjoint and its auxiliaries are those of the NEXT step's k1, which the
// reverse sweep has just used (the caller carries them over).
template <class RHS, class S, bool KEEP, bool SAFE, bool PACK = KEEP>
__device__ __forceinline__ void tsit5_stages(const S* u, const S* p, double t, double dts, S (*k)[RHS::ZD], S* un,
                                             S (*g)[RHS::ZD], typename RHS::Aux* aux) {
    constexpr int ZD = RHS::ZD;
    using Tb = Tab<S>;
    using V = VecOps<S, ZD, PACK>;
    const S h = (S)dts;
    S gi[ZD], acc[ZD];
#define LDEQ_EVAL(J, TJ)                                   \
    if constexpr (KEEP) {                                  \
        _Pragma("unroll") for (int i = 0; i < ZD; ++i) g[J][i] = gi[i]; \
        RHS::template f<SAFE>(k[J], gi, p, (TJ), aux[J]);  \
    } else {                                               \
        RHS::template f<SAFE>(k[J], gi, p, (TJ));          \
    }
    if constexpr (KEEP) {
#pragma unroll
        for (int i = 0; i < ZD; ++i) gi[i] = u[i];
        LDEQ_EVAL(0, t)  // recompute k1 = f(u_n) together with its auxiliaries
    }
    V::fma(gi, h * Tb::a21, k[0], u);
    LDEQ_EVAL(1, t + Tb::c2 * dts)
    V::scale(acc, Tb::a31, k[0]);
    V::axpy(acc, Tb::a32, k[1]);
    V::fma(gi, h, acc, u);
    LDEQ_EVAL(2, t + Tb::c3 * dts)
    V::scale(acc, Tb::a41, k[0]);
    V::axpy(acc, Tb::a42, k[1]);
    V::axpy(acc, Tb::a43, k[2]);
    V::fma(gi, h, acc, u);
    LDEQ_EVAL(3, t + Tb::c4 * dts)
    V::scale(acc, Tb::a51, k[0]);
    V::axpy(acc, Tb::a52, k[1]);
    V::axpy(acc, Tb::a53, k[2]);
    V::axpy(acc, Tb::a54, k[3]);
    V::fma(gi, h, acc, u);
    LDEQ_EVAL(4, t + Tb::c5 * dts)
    V::scale(acc, Tb::a61, k[0]);
    V::axpy(acc, Tb::a62, k[1]);
    V::axpy(acc, Tb::a63, k[2]);
    V::axpy(acc, Tb::a64, k[3]);
    V::axpy(acc, Tb::a65, k[4]);
    V::fma(gi, h, acc, u);
    LDEQ_EVAL(5, t + dts)
    V::scale(acc, Tb::a71, k[0]);
    V::axpy(acc, Tb::a72, k[1]);
    V::axpy(acc, Tb::a73, k[2]);
    V::axpy(acc, Tb::a74, k[3]);
    V::axpy(acc, Tb::a75, k[4]);
    V::axpy(acc, Tb::a76, k[5]);
    V::fma(un, h, acc, u);
    if constexpr (!KEEP) RHS::template f<SAFE>(k[6], un, p, t + dts);
#undef LDEQ_EVAL
}

// out of line: the redo of a step whose end points left the fast sine's range (keeps the hot loop's code small)
template <class M, class RHS, class S, bool KEEP>
__device__ __forceinline__ void erk_stages_safe(const S* u, const S* p, double t, double dts, S (*k)[RHS::ZD], S* un,
                                                S (*g)[RHS::ZD], typename RHS::Aux* aux) {
    M::template stages<RHS, S, KEEP, true, KEEP>(u, p, t, dts, k, un, g, aux);
}

// scaled RMS error estimate (SURVEY.md A.2)
template <class S, int ZD>
__device__ __forceinline__ double tsit5_eest(const S* u, const S* un, S (*k)[ZD], double dts, S abstol, S reltol) {
    using Tb = Tab<S>;
    using V = VecOps<S, ZD, false>;
    const S h = (S)dts;
    S s[ZD];
    V::scale(s, Tb::bt1, k[0]);
    V::axpy(s, Tb::bt2, k[1]);
    V::axpy(s, Tb::bt3, k[2]);
    V::axpy(s, Tb::bt4, k[3]);
    V::axpy(s, Tb::bt5, k[4]);
    V::axpy(s, Tb::bt6, k[5]);
    V::axpy(s, Tb::bt7, k[6]);
    S e2 = (S)0;
#pragma unroll
    for (int i = 0; i < ZD; ++i) {
        const S utilde = h * s[i];
        const S sk = s_fma<S>(s_max<S>(s_abs<S>(u[i]), s_abs<S>(un[i])), reltol, abstol);
        const S a = s_div_fast<S>(utilde, sk);
        e2 = s_fma<S>(a, a, e2);
    }
    return (double)s_sqrt<S>(e2 / (S)ZD);
}

// Hairer initial step (OrdinaryDiffEq ode_determine_initdt; SURVEY.md A.4)
template <class RHS, class S, int ORDER = 5>
__device__ double tsit5_initdt(const S* u0, const S* p, const S* f0, double t0, double dtmax, double dtmin,
                               const KOpts& o) {
    constexpr int ZD = RHS::ZD;
    const S abstol = (S)o.abstol, reltol = (S)o.reltol;
    S sk[ZD], s0 = (S)0, s1 = (S)0;
#pragma unroll
    for (int i = 0; i < ZD; ++i) {
        sk[i] = s_fma<S>(s_abs<S>(u0[i]), reltol, abstol);
        const S a = u0[i] / sk[i], b = f0[i] / sk[i];
        s0 = s_fma<S>(a, a, s0);
        s1 = s_fma<S>(b, b, s1);
    }
    const double d0 = (double)s_sqrt<S>(s0 / (S)ZD), d1 = (double)s_sqrt<S>(s1 / (S)ZD);
    double dt0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * (d0 / d1);
    dt0 = fmin(dt0, dtmax);
    if (dt0 < 10.0 * 2.220446049250313e-16) return fmax(1e-6, dtmin);
    S u1[ZD], f1[ZD];
    const S h0 = (S)dt0;
#pragma unroll
    for (int i = 0; i < ZD; ++i) u1[i] = s_fma<S>(h0, f0[i], u0[i]);
    RHS::f(f1, u1, p, t0 + dt0);
    S s2 = (S)0;
#pragma unroll
    for (int i = 0; i < ZD; ++i) {
        const S a = (f1[i] - f0[i]) / sk[i];
        s2 = s_fma<S>(a, a, s2);
    }
    const double d2 = (double)s_sqrt<S>(s2 / (S)ZD) / dt0;
    const double m = fmax(d1, d2);
    const double dt1 = (m <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : pow(10.0, -(2.0 + log10(m)) / (double)ORDER);
    return fmax(dtmin, fmin(100.0 * dt0, fmin(dt1, dtmax)));
}

// ---- dense output in Horner form -------------------------------------------------------------------
// sum_j b_j(Theta) k_j = Theta (c1 + Theta (c2 + Theta (c3 + Theta c4))) with c_m = sum_j r_jm k_j, so a step
// pays 21 vector FMAs once and every save point inside it only 4.
template <class S, int ZD>
__device__ __forceinline__ void interp_coeffs(S (*k)[ZD], S (*c)[ZD]) {
    using Tb = Tab<S>;
    using V = VecOps<S, ZD, false>;
#pragma unroll
    for (int i = 0; i < ZD; ++i) c[0][i] = k[0][i];  // r11 = 1
    V::scale(c[1], Tb::r12, k[0]); V::scale(c[2], Tb::r13, k[0]); V::scale(c[3], Tb::r14, k[0]);
    V::axpy(c[1], Tb::r22, k[1]);  V::axpy(c[2], Tb::r23, k[1]);  V::axpy(c[3], Tb::r24, k[1]);
    V::axpy(c[1], Tb::r32, k[2]);  V::axpy(c[2], Tb::r33, k[2]);  V::axpy(c[3], Tb::r34, k[2]);
    V::axpy(c[1], Tb::r42, k[3]);  V::axpy(c[2], Tb::r43, k[3]);  V::axpy(c[3], Tb::r44, k[3]);
    V::axpy(c[1], Tb::r52, k[4]);  V::axpy(c[2], Tb::r53, k[4]);  V::axpy(c[3], Tb::r54, k[4]);
    V::axpy(c[1], Tb::r62, k[5]);  V::axpy(c[2], Tb::r63, k[5]);  V::axpy(c[3], Tb::r64, k[5]);
    V::axpy(c[1], Tb::r72, k[6]);  V::axpy(c[2], Tb::r73, k[6]);  V::axpy(c[3], Tb::r74, k[6]);
}
// adjoint of interp_coeffs: kbar_j += sum_m r_jm cbar_m
template <class S, int ZD>
__device__ __forceinline__ void interp_coeffs_adj(S (*cb)[ZD], S (*kbar)[ZD]) {
    using Tb = Tab<S>;
    using V = VecOps<S, ZD>;
    V::add(kbar[0], cb[0]);
    V::axpy(kbar[0], Tb::r12, cb[1]); V::axpy(kbar[0], Tb::r13, cb[2]); V::axpy(kbar[0], Tb::r14, cb[3]);
    V::axpy(kbar[1], Tb::r22, cb[1]); V::axpy(kbar[1], Tb::r23, cb[2]); V::axpy(kbar[1], Tb::r24, cb[3]);
    V::axpy(kbar[2], Tb::r32, cb[1]); V::axpy(kbar[2], Tb::r33, cb[2]); V::axpy(kbar[2], Tb::r34, cb[3]);
    V::axpy(kbar[3], Tb::r42, cb[1]); V::axpy(kbar[3], Tb::r43, cb[2]); V::axpy(kbar[3], Tb::r44, cb[3]);
    V::axpy(kbar[4], Tb::r52, cb[1]); V::axpy(kbar[4], Tb::r53, cb[2]); V::axpy(kbar[4], Tb::r54, cb[3]);
    V::axpy(kbar[5], Tb::r62, cb[1]); V::axpy(kbar[5], Tb::r63, cb[2]); V::axpy(kbar[5], Tb::r64, cb[3]);
    V::axpy(kbar[6], Tb::r72, cb[1]); V::axpy(kbar[6], Tb::r73, cb[2]); V::axpy(kbar[6], Tb::r74, cb[3]);
}

// reverse sweep through the seven stages of one taped step (see ErkM::reverse_sweep for the contract)
template <class RHS, class S>
__device__ __forceinline__ void tsit5_reverse_sweep(const S* p, double tn, double dtn, S (*g)[RHS::ZD], const S* un,
                                                    typename RHS::Aux* aux, const typename RHS::Aux& aux_next,
                                                    S (*kbar)[RHS::ZD], S* ubn, S* ub, S* pbar) {
    constexpr int ZD = RHS::ZD;
    using Tb = Tab<S>;
    using V = VecOps<S, ZD>;
    const S h = (S)dtn;
    // k7 = f(u_{n+1}) (it is also next step's k1, whose adjoint was already folded into ubn)
    RHS::vjp(ubn, pbar, un, p, tn + dtn, kbar[6], aux_next);
    // u_{n+1} = u_n + h sum_j a7j k_j
    S v[ZD];
    V::scale(v, h, ubn);
    V::add(ub, ubn);
    V::axpy(kbar[0], Tb::a71, v); V::axpy(kbar[1], Tb::a72, v); V::axpy(kbar[2], Tb::a73, v);
    V::axpy(kbar[3], Tb::a74, v); V::axpy(kbar[4], Tb::a75, v); V::axpy(kbar[5], Tb::a76, v);
    S gb[ZD];
    // stage 6: g6 = u + h (a61 k1 + ... + a65 k5)
#pragma unroll
    for (int i = 0; i < ZD; ++i) gb[i] = (S)0;
    RHS::vjp(gb, pbar, g[5], p, tn + dtn, kbar[5], aux[5]);
    V::scale(v, h, gb);
    V::add(ub, gb);
    V::axpy(kbar[0], Tb::a61, v); V::axpy(kbar[1], Tb::a62, v); V::axpy(kbar[2], Tb::a63, v);
    V::axpy(kbar[3], Tb::a64, v); V::axpy(kbar[4], Tb::a65, v);
    // stage 5
#pragma unroll
    for (int i = 0; i < ZD; ++i) gb[i] = (S)0;
    RHS::vjp(gb, pbar, g[4], p, tn + Tb::c5 * dtn, kbar[4], aux[4]);
    V::scale(v, h, gb);
    V::add(ub, gb);
    V::axpy(kbar[0], Tb::a51, v); V::axpy(kbar[1], Tb::a52, v); V::axpy(kbar[2], Tb::a53, v);
    V::axpy(kbar[3], Tb::a54, v);
    // stage 4
#pragma unroll
    for (int i = 0; i < ZD; ++i) gb[i] = (S)0;
    RHS::vjp(gb, pbar, g[3], p, tn + Tb::c4 * dtn, kbar[3], aux[3]);
    V::scale(v, h, gb);
    V::add(ub, gb);
    V::axpy(kbar[0], Tb::a41, v); V::axpy(kbar[1], Tb::a42, v); V::axpy(kbar[2], Tb::a43, v);
    // stage 3
#pragma unroll
    for (int i = 0; i < ZD; ++i) gb[i] = (S)0;
    RHS::vjp(gb, pbar, g[2], p, tn + Tb::c3 * dtn, kbar[2], aux[2]);
    V::scale(v, h, gb);
    V::add(ub, gb);
    V::axpy(kbar[0], Tb::a31, v); V::axpy(kbar[1], Tb::a32, v);
    // stage 2
#pragma unroll
    for (int i = 0; i < ZD; ++i) gb[i] = (S)0;
    RHS::vjp(gb, pbar, g[1], p, tn + Tb::c2 * dtn, kbar[1], aux[1]);
    V::add(ub, gb);
    V::axpy(kbar[0], h * Tb::a21, gb);
    // stage 1: k1 = f(u_n)
    RHS::vjp(ub, pbar, g[0], p, tn, kbar[0], aux[0]);
}

// The method interface of the integrator bodies: the hand-unrolled Tsit5 (the reference's solver, pendulum.jl:11,58).
// ErkM<...> (ldeq_erk.cuh) supplies the same members for the table-driven DP5 / BS3 / RK4.
struct Tsit5M {
    static constexpr int NS = 7, ORDER = 5;
    template <class RHS, class S, bool KEEP, bool SAFE, bool PACK>
    __device__ __forceinline__ static void stages(const S* u, const S* p, double t, double dts, S (*k)[RHS::ZD], S* un,
                                                  S (*g)[RHS::ZD], typename RHS::Aux* aux) {
        tsit5_stages<RHS, S, KEEP, SAFE, PACK>(u, p, t, dts, k, un, g, aux);
    }
    template <class S, int ZD>
    __device__ __forceinline__ static double eest(const S* u, const S* un, S (*k)[ZD], double dts, S abstol, S reltol) {
        return tsit5_eest<S, ZD>(u, un, k, dts, abstol, reltol);
    }
    template <class S, int ZD> __device__ __forceinline__ static void interp_coeffs(S (*k)[ZD], S (*c)[ZD]) { ldeq::interp_coeffs<S, ZD>(k, c); }
    template <class S, int ZD> __device__ __forceinline__ static void interp_coeffs_adj(S (*cb)[ZD], S (*kbar)[ZD]) { ldeq::interp_coeffs_adj<S, ZD>(cb, kbar); }
    template <class RHS, class S>
    __device__ __forceinline__ static void reverse_sweep(const S* p, double tn, double dtn, S (*g)[RHS::ZD], const S* un,
                                                         typename RHS::Aux* aux, const typename RHS::Aux& aux_next,
                                                         S (*kbar)[RHS::ZD], S* ubn, S* ub, S* pbar) {
        tsit5_reverse_sweep<RHS, S>(p, tn, dtn, g, un, aux, aux_next, kbar, ubn, ub, pbar);
    }
};

// The save grid is staged in shared memory (explicit LDS, not a generic load); grids too long for
// that are read through the global pointer.
#define LDEQ_TGRID_SMEM_MAX 2048
// A grid the host has verified to be t0 + k*h bit for bit (GridInfo::uniform) is not looked up at all: a save time
// is one DFMA, and the save points that fall into a step are found by ONE division per step (count_le) instead of one
// Float64 comparison per save point.
struct TGrid {
    const double* __restrict__ g;
    const double* s;
    double t0, h, inv_h;
    int T;
    bool in_smem, uniform;
    __device__ __forceinline__ double operator[](int i) const {
        if (uniform) return fma((double)i, h, t0);
        return in_smem ? s[i] : g[i];
    }
    // number of grid points t_k <= x (k in [0, T)), i.e. the first index whose save time lies beyond x.  `from` is a
    // lower bound the caller knows (t_k <= x for all k < from); a table grid is scanned upwards from there.
    __device__ __forceinline__ int count_le(double x, int from) const {
        if (uniform) {
            // floor((x - t0) / h) is off by at most one; the DFMA comparisons make the answer exact
            double q = (x - t0) * inv_h;
            q = fmin(fmax(q, -1.0), (double)(T - 1));
            int k = __double2int_rd(q);
            if (k + 1 < T && fma((double)(k + 1), h, t0) <= x) ++k;
            else if (k >= 0 && fma((double)k, h, t0) > x) --k;
            return k + 1;
        }
        int k = from;
        while (k < T && (in_smem ? s[k] : g[k]) <= x) ++k;
        return k;
    }
    // the same, for the reverse pass: t_k > x is known for all k >= from; a table grid is scanned downwards
    __device__ __forceinline__ int count_le_down(double x, int from) const {
        if (uniform) return count_le(x, 0);
        int k = from;
        while (k > 0 && (in_smem ? s[k - 1] : g[k - 1]) > x) --k;
        return k;
    }
};
__device__ __forceinline__ TGrid stage_tgrid(const double* __restrict__ tg, int T, double* s_tg, const GridInfo& gi) {
    TGrid r{tg, s_tg, gi.t0, gi.h, gi.uniform ? 1.0 / gi.h : 0.0, T, T <= LDEQ_TGRID_SMEM_MAX, gi.uniform != 0};
    if (r.in_smem && !r.uniform) {
        for (int i = threadIdx.x; i < T; i += blockDim.x) s_tg[i] = tg[i];
        __syncthreads();
    }
    return r;
}
#define LDEQ_TINF __longlong_as_double(0x7ff0000000000000LL)

// ---- per-lane save-point ring ----------------------------------------------------------------------
// With adaptive steps the lanes of a warp reach a given save index k at different times, so a
// thread-per-trajectory kernel that stores straight to the (z,B,T) array issues 8-byte stores to 32
// different rows per instruction (ncu: 8.7 of 32 bytes per sector used, the store queue backs up and
// the kernel runs 1.7x slower than with the stores removed).  Instead every lane owns one COLUMN of a
// shared-memory ring of LDEQ_RING_BYTES per lane; it parks its save points there, and the warp moves
// complete ROWS (all 32 lanes, same k) to global memory together: full 32-byte sectors, one
// 256-byte coalesced store per row.  A lane that gets LDEQ ring rows ahead of the slowest lane of
// its warp waits for it; the warp's iteration count is set by its slowest lane either way.
// The backward kernel uses the same ring the other way round (rows of the cotangent are fetched
// with cp.async, coalesced, ahead of use).
#ifndef LDEQ_RING_BYTES
#define LDEQ_RING_BYTES 256
#endif
template <class S, int ZD> struct Ring {
    static constexpr int floor_pow2(int x) { return x >= 64 ? 64 : x >= 32 ? 32 : x >= 16 ? 16 : x >= 8 ? 8 : 4; }
    static constexpr int R = floor_pow2(LDEQ_RING_BYTES / (ZD * (int)sizeof(S)));
    S* col;      // this lane's column
    int stride;  // elements between consecutive rows
    __device__ __forceinline__ S* at(int k) const { return col + (size_t)(k & (R - 1)) * stride; }
    __host__ __device__ static constexpr size_t bytes(int threads) { return (size_t)R * threads * ZD * sizeof(S); }
};

__device__ __forceinline__ int warp_min_i(int v) { return __reduce_min_sync(0xffffffffu, v); }
__device__ __forceinline__ int warp_max_i(int v) { return __reduce_max_sync(0xffffffffu, v); }

template <int BYTES> __device__ __forceinline__ void cp_async_vec(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(d), "l"(gsrc), "n"(BYTES));
}
// one ZD-vector row: a single 8/16-byte copy when the row has that size, element-wise otherwise
template <class S, int ZD> __device__ __forceinline__ void cp_async_row(S* smem_dst, const S* gsrc) {
    if constexpr (ZD * sizeof(S) == 8 || ZD * sizeof(S) == 16) {
        cp_async_vec<ZD * (int)sizeof(S)>(smem_dst, gsrc);
    } else {
#pragma unroll
        for (int i = 0; i < ZD; ++i) cp_async_vec<(int)sizeof(S)>(smem_dst + i, gsrc + i);
    }
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// ---- forward ------------------------------------------------------------------------------------
template <class M, class RHS, class S, bool TAPE>
__device__ __forceinline__ void
erk_fwd_body(const S* __restrict__ z0, const S* __restrict__ theta, const double* __restrict__ tg_global, int B,
                 int T, KOpts o, S* __restrict__ traj, int* __restrict__ retcode, int* __restrict__ naccept,
                 int* __restrict__ nreject, TapeView<S> tape, GridInfo ginfo) {
    constexpr int ZD = RHS::ZD, PD = RHS::PD;
    using RingT = Ring<S, ZD>;
    using V = VecOps<S, ZD, false>;  // forward kernel: scalar FFMAs (see VecOps)
    constexpr int R = RingT::R;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RingT ring{reinterpret_cast<S*>(smem_raw) + threadIdx.x * ZD, (int)blockDim.x * ZD};
    const TGrid tg = stage_tgrid(tg_global, T, reinterpret_cast<double*>(smem_raw + RingT::bytes(blockDim.x)), ginfo);
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = b < B;
    const int bb = live ? b : B - 1;  // dead lanes of the last warp shadow a valid trajectory and store nothing

    constexpr int NS = M::NS;  // stages, the FSAL stage included
    S u[ZD], un[ZD], p[PD], k[NS][ZD];
    load_vec<S, ZD>(z0 + (size_t)bb * ZD, u);
#pragma unroll
    for (int i = 0; i < PD; ++i) p[i] = theta[(size_t)bb * PD + i];
    if (TAPE) {
        if (tape.theta && live) {
#pragma unroll
            for (int i = 0; i < PD; ++i) tape.theta[(size_t)b * PD + i] = p[i];
        }
        if (tape.tgrid && blockIdx.x == 0)
            for (int kk = threadIdx.x; kk < T; kk += blockDim.x) tape.tgrid[kk] = tg_global[kk];
        // record 0 always holds u0 (a trajectory that fails before its first accepted step leaves nothing else there;
        // a replay into a larger tape and the forward-dual pullback start from this record)
        if (live && tape.u) store_vec<S, ZD>(tape.u + (size_t)b * ZD, u);
    }

    const double t0 = tg[0], tend = tg[T - 1];
    const double dtmax = o.dtmax > 0.0 ? o.dtmax : (tend - t0);
    const double dtmin = o.dtmin > 0.0 ? o.dtmin : fmax(2.220446049250313e-16, ulp_of(t0));
    const S abstol = (S)o.abstol, reltol = (S)o.reltol;
    const double abs_tend = fabs(tend);
    const double snap_end = 100.0 * ulp_of(abs_tend);  // 100 ulp(max(|t|, |tend|)) whenever |t| <= |tend|

    RHS::f(k[0], u, p, t0);  // fsalfirst
    double t = t0;
    double dt = (o.adaptive && !(o.dt > 0.0)) ? tsit5_initdt<RHS, S, M::ORDER>(u, p, k[0], t0, dtmax, dtmin, o) : o.dt;
    PiState pist = pi_init(o);
    int na = 0, nr = 0, ret = RET_SUCCESS;
    int iters_left = (int)(o.maxiters < 0x7fffffffLL ? o.maxiters : 0x7fffffffLL);

    const size_t ld = (size_t)ginfo.ld;
    if (traj && live) store_vec<S, ZD>(traj + (size_t)b * ZD, u);  // t[1] == tspan[1]: stored exactly
    if (!(dt > 0.0) || !isfinite(dt)) ret = RET_DTLESSTHANMIN;

    int ks = live ? 1 : T;  // next save index this lane emits
    int kflush = 1;         // warp-uniform: rows below it are in global memory
    bool active = live && T > 1 && ret == RET_SUCCESS;  // still has steps to take
    bool pending = false;   // an accepted step whose save points are not all parked yet
    int kend = 1;           // save points ks .. kend-1 fall into the pending step
    int kanchor = 1;        // ... the first of them: Theta of the step's points is anchored there
    bool hit = false;       // ... and the last of them coincides with the step end (stored as u_{n+1} itself)
    double dts = 0.0, tnew = t0;

    while (kflush < T) {
        if (active && !pending) {
            if (iters_left <= 0) {
                ret = RET_MAXITERS;
                active = false;
            } else {
                --iters_left;
                // tstop handling: never step past tend; snap onto it within 100 ulp
                dts = fmin(dt, tend - t);
                tnew = t + dts;
                if (fabs(tnew - tend) < (fabs(t) > abs_tend ? 100.0 * ulp_of(fabs(t)) : snap_end)) tnew = tend;

                M::template stages<RHS, S, false, false, false>(u, p, t, dts, k, un, nullptr, nullptr);
                if (!(RHS::fast_ok(u) && RHS::fast_ok(un)))  // an end point outside the fast sine's range: libdevice (never for a pendulum)
                    erk_stages_safe<M, RHS, S, false>(u, p, t, dts, k, un, nullptr, nullptr);

                bool finite = true;
#pragma unroll
                for (int i = 0; i < ZD; ++i) finite = finite && s_finite<S>(un[i]);
                bool accept = true;
                double dt_next = dt;
                if (o.adaptive) {
                    const double EEst = M::template eest<S, ZD>(u, un, k, dts, abstol, reltol);
                    if (EEst != EEst) finite = false;
                    accept = pi_controller(o, EEst, dts, dtmax, pist, dt_next);
                }
                if (!finite) {
                    ret = RET_UNSTABLE;
                    active = false;
                } else {
                    if (accept) {
                        if (TAPE) {
                            if (na < tape.cap) {
                                const size_t r = (size_t)na * B + b;
                                tape.t[r] = t;
                                if (na) store_vec<S, ZD>(tape.u + r * ZD, u);
                            }
                        }
                        ++na;
                        pending = true;
                        // saveat: every pending grid time <= tnew belongs to this step
                        kend = tg.count_le(tnew, ks);
                        kanchor = ks;
                        hit = kend > ks && tg[kend - 1] == tnew;
                    } else {
                        ++nr;
                    }
                    dt = dt_next;
                    if (o.adaptive && !(accept && tnew == tend) && (!(fabs(dt) > dtmin) || !isfinite(dt))) {
                        ret = RET_DTLESSTHANMIN;
                        active = false;
                        pending = false;
                    }
                }
            }
        }
        if (pending) {
            // interior points through the dense interpolant of this step (Horner form); a grid time that coincides
            // with the step end stores u_{n+1} itself.  At most R rows beyond the warp's flush mark fit the ring.
            const int kint = kend - (hit ? 1 : 0);
            const int klim = kflush + R;
            const int kstop = kint < klim ? kint : klim;
            if (ks < kstop) {
                S c[4][ZD];
                M::template interp_coeffs<S, ZD>(k, c);
                const S h = (S)dts;
                const double inv = 1.0 / dts;
                // Theta of consecutive points of a uniform grid advances by h_grid / dt: one FMA per point, anchored at
                // the first save point of the STEP (|Theta| <= 1, so the anchor's rounding is the only error that matters).
                // Anchoring at the step, not at this visit, keeps the arithmetic of a trajectory independent of how the
                // ring splits its save points into visits, i.e. of the other lanes of its warp: a solve commutes bit for
                // bit with any split or permutation of the batch (tests/test_properties_gpu.py).
                const S th0 = (S)((tg[kanchor] - t) * inv);
                const S dth = (S)(tg.h * inv);
                S fk = (S)(ks - kanchor);
                do {
                    const S th = tg.uniform ? s_fma<S>(fk, dth, th0) : (S)((tg[ks] - t) * inv);
                    S pl[ZD], out[ZD];
                    V::fma(pl, th, c[3], c[2]);
                    V::fma(pl, th, pl, c[1]);
                    V::fma(pl, th, pl, c[0]);
                    V::fma(out, h * th, pl, u);
                    store_vec<S, ZD>(ring.at(ks), out);
                    ++ks;
                    fk += (S)1;
                } while (ks < kstop);
            }
            if (hit && ks == kint && ks < klim) {
                store_vec<S, ZD>(ring.at(ks), un);
                ++ks;
            }
            if (ks >= kend) {  // all save points of this step are parked: commit it
                t = tnew;
#pragma unroll
                for (int i = 0; i < ZD; ++i) { u[i] = un[i]; k[0][i] = k[NS - 1][i]; }  // FSAL
                pending = false;
                if (ks >= T) active = false;
            }
        }
        // move the rows every lane of the warp has passed to global memory, coalesced
        const int kmin = warp_min_i((active || pending) ? ks : T);
        if (traj && live) {
            int r = kflush;
            for (; r + 1 < kmin; r += 2) {
                S v0[ZD], v1[ZD];
                load_vec<S, ZD>(ring.at(r), v0);
                load_vec<S, ZD>(ring.at(r + 1), v1);
                store_vec<S, ZD>(traj + ((size_t)r * ld + b) * ZD, v0);
                store_vec<S, ZD>(traj + ((size_t)(r + 1) * ld + b) * ZD, v1);
            }
            if (r < kmin) {
                S v0[ZD];
                load_vec<S, ZD>(ring.at(r), v0);
                store_vec<S, ZD>(traj + ((size_t)r * ld + b) * ZD, v0);
            }
        }
        kflush = kmin;
    }

    if (!live) return;
    if (ret != RET_SUCCESS && traj) {  // GOKU.jl:114: the whole (z,T) block of a failed solve is NaN
        S nanv[ZD];
#pragma unroll
        for (int i = 0; i < ZD; ++i) nanv[i] = s_nan<S>();
        for (int kk = 0; kk < T; ++kk) store_vec<S, ZD>(traj + ((size_t)kk * ld + b) * ZD, nanv);
    }
    if (retcode) retcode[b] = ret;
    if (naccept) naccept[b] = na;
    if (nreject) nreject[b] = nr;
    if (TAPE) {
        if (tape.ret) tape.ret[b] = ret;
        if (tape.na) tape.na[b] = na;
        if (tape.nr) tape.nr[b] = nr;
        // tape.info = {trajectories that ran past the capacity, largest accepted-step count}; one atomic per warp
        const unsigned am = __activemask();
        const int wmax = __reduce_max_sync(am, ret == RET_SUCCESS ? na : 0);
        const int wover = __reduce_add_sync(am, (ret == RET_SUCCESS && na > tape.cap) ? 1 : 0);
        if ((threadIdx.x & 31) == (__ffs(am) - 1)) {
            if (wover) atomicAdd(tape.info, wover);
            atomicMax(tape.info + 1, wmax);
        }
    }
}

// ---- backward: discrete adjoint of the taped steps ----------------------------------------------
// dtraj (z,B,T) -> dz0 (z,B), dtheta (p,B).  Step sizes are constants of the differentiation, as in
// the reference's ForwardDiffSensitivity where tspan/dt stay plain Float64 (SURVEY.md A.6).
template <class M, class RHS, class S>
__device__ __forceinline__ void
erk_bwd_body(const S* __restrict__ theta, const double* __restrict__ tg_global, int B, int T,
                 const S* __restrict__ dtraj, TapeView<S> tape, const int* __restrict__ retcode,
                 const int* __restrict__ naccept, S* __restrict__ dz0, S* __restrict__ dtheta, GridInfo ginfo) {
    constexpr int ZD = RHS::ZD, PD = RHS::PD;
    using Tb = Tab<S>;
    using RingT = Ring<S, ZD>;
    using V = VecOps<S, ZD>;
    constexpr int R = RingT::R;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RingT ring{reinterpret_cast<S*>(smem_raw) + threadIdx.x * ZD, (int)blockDim.x * ZD};
    const TGrid tg = stage_tgrid(tg_global, T, reinterpret_cast<double*>(smem_raw + RingT::bytes(blockDim.x)), ginfo);
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    // Lanes of a warp run until the trajectory with the most taped steps is done.  The forward pass has counted every
    // trajectory's accepted steps: the CTA ranks its trajectories by that count and re-deals them, so a warp holds 32
    // neighbours in step count (the same re-deal as the forward-dual kernels, ldeq_fwdsens.cuh).  Only the assignment of
    // trajectories to lanes changes -- every trajectory's arithmetic and its output slots are the same.
    if (ginfo.sort) {
        __shared__ int s_key[LDEQ_BWD_THREADS];
        __shared__ short s_order[LDEQ_BWD_THREADS];
        const int tid = threadIdx.x, nt = blockDim.x;
        const int key = b < B ? naccept[b] : 0x7fffffff;  // dead lanes go last
        s_key[tid] = key;
        __syncthreads();
        int rank = 0;
        for (int j = 0; j < nt; ++j) {
            const int kj = s_key[j];
            rank += (kj < key || (kj == key && j < tid)) ? 1 : 0;
        }
        s_order[rank] = (short)tid;
        __syncthreads();
        b = blockIdx.x * blockDim.x + s_order[tid];
    }
    const bool live = b < B;
    const int bb = live ? b : B - 1;  // dead lanes of the last warp read a valid column and write nothing

    S p[PD], pbar[PD], ubn[ZD];
#pragma unroll
    for (int i = 0; i < PD; ++i) pbar[i] = (S)0;
#pragma unroll
    for (int i = 0; i < ZD; ++i) ubn[i] = (S)0;
    int na = naccept[bb];
    const int ret = retcode[bb];
#pragma unroll
    for (int i = 0; i < PD; ++i) p[i] = theta[(size_t)bb * PD + i];
    const bool overflow = ret == RET_SUCCESS && na > tape.cap;  // a failed solve has a zero gradient whatever it recorded
    if (!live || ret != RET_SUCCESS || overflow) na = 0;

    // rows 1..T-1 of the cotangent travel through the ring: [kload, T) has been fetched so far
    const size_t ld = (size_t)ginfo.ld;
    int kload = T;
    auto refill = [&](int ks_max) {
        if (ks_max < 1) return;  // no lane of the warp has a row left to consume (finished, failed or overflowed)
        int klo = ks_max - R + 1;
        klo = klo < 1 ? 1 : klo;
        for (int r = kload - 1; r >= klo; --r)
            cp_async_row<S, ZD>(ring.at(r), dtraj + ((size_t)r * ld + bb) * ZD);
        kload = klo < kload ? klo : kload;
    };

    int n = na - 1;        // next taped step of this lane
    int ks = T - 1;        // next save point of this lane (descending); row 0 is handled at the end
    bool holding = false;  // a step whose stages are recomputed and whose save points are being consumed
    int klo_step = T;      // save points klo_step .. ks fall into the step being held
    int kanchor = T;       // ... the topmost interior one: Theta of the step's points is anchored there
    bool hit = false;      // ... and the topmost of them coincides with the step end t_{n+1}
    double tnext = tg[T - 1];  // time after step n; the forward pass ended exactly on tend
    double tn = 0.0, dtn = 0.0;
    constexpr int NS = M::NS;
    S g[NS - 1][ZD], un[ZD], kbar[NS][ZD], cb[4][ZD], ub[ZD];
    typename RHS::Aux aux[NS - 1], aux_next;  // aux_next: f's auxiliaries at u_{n+1} (= those of step n+1's k1)

    refill(warp_max_i(n >= 0 ? ks : 0));
    // the record of the step a lane will need next is fetched one step ahead (its latency hides behind
    // the stage recomputation of the current step)
    double tn_pre = 0.0;
    S u_pre[ZD];
#pragma unroll
    for (int i = 0; i < ZD; ++i) u_pre[i] = (S)0;
    if (n >= 0) {
        const size_t r = (size_t)n * B + b;
        tn_pre = tape.t[r];
        load_vec<S, ZD>(tape.u + r * ZD, u_pre);
    }
    bool first = true;
    // runs until every lane of the warp has swept its step 0 (early steps may hold no save point at all)
    while (__any_sync(0xffffffffu, holding || n >= 0)) {
        if (!holding && n >= 0) {
            tn = tn_pre;
            dtn = tnext - tn;
            S u[ZD], k[NS][ZD];
#pragma unroll
            for (int i = 0; i < ZD; ++i) u[i] = u_pre[i];
            if (n >= 1) {
                const size_t r = (size_t)(n - 1) * B + b;
                tn_pre = tape.t[r];
                load_vec<S, ZD>(tape.u + r * ZD, u_pre);
            }
            M::template stages<RHS, S, true, false, true>(u, p, tn, dtn, k, un, g, aux);
            if (!(RHS::fast_ok(u) && RHS::fast_ok(un))) erk_stages_safe<M, RHS, S, true>(u, p, tn, dtn, k, un, g, aux);
            if (first) {  // the last step of the solve: nothing follows it, evaluate f's auxiliaries at u(tend) here
                S ktmp[ZD];
                RHS::f(ktmp, un, p, tn + dtn, aux_next);
                first = false;
            }
#pragma unroll
            for (int j = 0; j < NS; ++j)
#pragma unroll
                for (int i = 0; i < ZD; ++i) kbar[j][i] = (S)0;
#pragma unroll
            for (int m = 0; m < 4; ++m)
#pragma unroll
                for (int i = 0; i < ZD; ++i) cb[m][i] = (S)0;
#pragma unroll
            for (int i = 0; i < ZD; ++i) ub[i] = (S)0;
            // save points with t_n < t_k <= t_{n+1}: indices klo_step .. ks
            klo_step = tg.count_le_down(tn, ks + 1);
            klo_step = klo_step < 1 ? 1 : klo_step;
            hit = ks >= klo_step && tg[ks] == tnext;
            kanchor = hit ? ks - 1 : ks;
            holding = true;
        }
        cp_async_wait_all();  // rows fetched at the end of the previous iteration have landed by now
        if (holding) {
            const S h = (S)dtn;
            if (hit && ks >= kload) {  // the cotangent of a save point at the step end belongs to u_{n+1}
                S d[ZD];
                load_vec<S, ZD>(ring.at(ks), d);
                V::add(ubn, d);
                --ks;
                hit = false;
            }
            if (!hit) {
                int kstop = klo_step > kload ? klo_step : kload;  // consume ks, ks-1, ..., kstop
                if (ks >= kstop) {
                    const double inv = 1.0 / dtn;
                    // anchored at the step's topmost interior save point, not at this visit (see the forward kernel)
                    const S th0 = (S)((tg[kanchor] - tn) * inv);
                    const S dth = (S)(tg.h * inv);
                    S fk = (S)(kanchor - ks);
                    do {
                        S d[ZD];
                        load_vec<S, ZD>(ring.at(ks), d);
                        const S th = tg.uniform ? s_fma<S>(fk, -dth, th0) : (S)((tg[ks] - tn) * inv);
                        const S w1 = h * th, w2 = w1 * th, w3 = w2 * th, w4 = w3 * th;
                        V::axpy(cb[0], w1, d);
                        V::axpy(cb[1], w2, d);
                        V::axpy(cb[2], w3, d);
                        V::axpy(cb[3], w4, d);
                        V::add(ub, d);
                        --ks;
                        fk += (S)1;
                    } while (ks >= kstop);
                }
            }
            if (ks < klo_step) {
                // every save point of this step has been consumed: reverse sweep through the stages
                M::template interp_coeffs_adj<S, ZD>(cb, kbar);
                M::template reverse_sweep<RHS, S>(p, tn, dtn, g, un, aux, aux_next, kbar, ubn, ub, pbar);
#pragma unroll
                for (int i = 0; i < ZD; ++i) ubn[i] = ub[i];
                aux_next = aux[0];  // u_n is the end point of step n-1
                tnext = tn;
                --n;
                holding = false;
            }
        }
        // fetch the rows the slowest lane of the warp will need next, coalesced, ahead of use
        refill(warp_max_i((holding || n >= 0) ? ks : 0));
    }
    cp_async_wait_all();

    if (!live) return;
    if (ret == RET_SUCCESS && !overflow) {
        S d[ZD];
        load_vec<S, ZD>(dtraj + (size_t)b * ZD, d);  // traj[:, b, 1] is u0 itself
#pragma unroll
        for (int i = 0; i < ZD; ++i) ubn[i] += d[i];
    } else {
        // failed solve: NaN block is a constant, zero gradient; tape overflow: gradient unavailable -> NaN
#pragma unroll
        for (int i = 0; i < ZD; ++i) ubn[i] = overflow ? s_nan<S>() : (S)0;
#pragma unroll
        for (int i = 0; i < PD; ++i) pbar[i] = overflow ? s_nan<S>() : (S)0;
    }
    store_vec<S, ZD>(dz0 + (size_t)b * ZD, ubn);
#pragma unroll
    for (int i = 0; i < PD; ++i) dtheta[(size_t)b * PD + i] = pbar[i];
}

// ---- kernel entry points ---------------------------------------------------------------------------------
// M: the method, Tsit5M or the table-driven DP5M / BS3M / RK4M (ldeq_erk.cuh)
template <class M, class RHS, class S, bool TAPE>
__global__ void __launch_bounds__(LDEQ_FWD_THREADS, LDEQ_FWD_MINBLOCKS)
erk_fwd_kernel(const S* __restrict__ z0, const S* __restrict__ theta, const double* __restrict__ tg_global, int B,
               int T, KOpts o, S* __restrict__ traj, int* __restrict__ retcode, int* __restrict__ naccept,
               int* __restrict__ nreject, TapeView<S> tape, GridInfo ginfo) {
    erk_fwd_body<M, RHS, S, TAPE>(z0, theta, tg_global, B, T, o, traj, retcode, naccept, nreject, tape, ginfo);
}

template <class M, class RHS, class S>
__global__ void __launch_bounds__(LDEQ_BWD_THREADS, LDEQ_BWD_MINBLOCKS)
erk_bwd_kernel(const S* __restrict__ theta, const double* __restrict__ tg_global, int B, int T,
               const S* __restrict__ dtraj, TapeView<S> tape, const int* __restrict__ retcode,
               const int* __restrict__ naccept, S* __restrict__ dz0, S* __restrict__ dtheta, GridInfo ginfo) {
    erk_bwd_body<M, RHS, S>(theta, tg_global, B, T, dtraj, tape, retcode, naccept, dz0, dtheta, ginfo);
}

}  // namespace ldeq
