// ldeq_fwdsens.cuh -- the reference's OWN gradient algorithm for the GOKU solve: sensealg = ForwardDiffSensitivity()
// (examples/pendulum_friction-less/pendulum.jl:11,58; SciMLSensitivity 7.10 `_concrete_solve_adjoint`, SURVEY.md A.6).
//
// Pullback per trajectory: seed theta with Dual partials and re-solve, dtheta = sum_k (du_k/dtheta)^T Delta_k; seed u0
// and re-solve, dz0 likewise.  The error norm of a Dual state includes the partials (sse(value) + sum sse(partials),
// partials counted as entries), so each dual solve takes its OWN accepted-step sequence -- this is what makes the
// reference's gradient differ from the discrete adjoint of the primal steps (erk_bwd_kernel) by up to the solver
// tolerance.  The body restates that algorithm literally, including Julia's arithmetic promotion (a Float32 state
// meets the Float64 dt: `uprev + dt*(...)` is evaluated in Float64 and rounded on the store; the dense-output
// polynomials are evaluated in Float64), so that its step sequences are the oracle's (oracle/ldeq_oracle.cpp::solve_one
// with NP > 0).  One thread per trajectory, two launches (theta-seeded NP = p_dim, u0-seeded NP = z_dim); the
// cotangent is consumed on the fly, nothing is stored.  RHS: ZD, PD, NPRE + prepare(D* p) (per-trajectory constants kept
// in p[PD..PD+NPRE)) and  template <class D> f(D* du, const D* u, const D* p, double t)  on duals -- the built-in pendulums (ldeq_fwdsens.cu) or a user's NVRTC function.
#pragma once

#include "ldeq_dual.cuh"
#include "ldeq_erk.cuh"

namespace ldeq {

#define LDEQ_DL _Pragma("unroll") for (int i_ = 0; i_ < N; ++i_)
template <class S, int N> __device__ __forceinline__ Dual<S, N> dual_fma(S s, Dual<S, N> k, Dual<S, N> acc) {
    acc.v = s_fma<S>(s, k.v, acc.v);
    LDEQ_DL acc.d[i_] = s_fma<S>(s, k.d[i_], acc.d[i_]);
    return acc;
}
template <class S, int N> __device__ __forceinline__ Dual<S, N> dual_scale(S a, Dual<S, N> b) {
    b.v *= a;
    LDEQ_DL b.d[i_] *= a;
    return b;
}
// uprev + dt*sum with dt in Float64: promoted, fused, rounded back to S on the store
template <class S, int N> __device__ __forceinline__ Dual<S, N> dual_axpy_time(Dual<S, N> uprev, double dt, Dual<S, N> sum) {
    Dual<S, N> r;
    r.v = (S)fma(dt, (double)sum.v, (double)uprev.v);
    LDEQ_DL r.d[i_] = (S)fma(dt, (double)sum.d[i_], (double)uprev.d[i_]);
    return r;
}
template <class S, int N> __device__ __forceinline__ Dual<S, N> dual_scale_time(double dt, Dual<S, N> sum) {
    Dual<S, N> r;
    r.v = (S)(dt * (double)sum.v);
    LDEQ_DL r.d[i_] = (S)(dt * (double)sum.d[i_]);
    return r;
}
template <class S, int N> __device__ __forceinline__ S dual_sse(Dual<S, N> a, bool wp) {
    S s = a.v * a.v;
    if (wp) { LDEQ_DL s += a.d[i_] * a.d[i_]; }
    return s;
}
template <class S, int N> __device__ __forceinline__ S dual_absnorm(Dual<S, N> a, bool wp) { return wp ? s_sqrt<S>(dual_sse(a, true)) : s_abs<S>(a.v); }
template <class S, int N> __device__ __forceinline__ Dual<S, N> dual_div_s(Dual<S, N> a, S s) {
    a.v /= s;
    LDEQ_DL a.d[i_] /= s;
    return a;
}
template <class S, int N> __device__ __forceinline__ S dual_rms(const Dual<S, N>* a, int n, bool wp) {
    S s = (S)0;
    for (int i = 0; i < n; ++i) s += dual_sse(a[i], wp);
    const int len = wp ? n * (1 + N) : n;
    return s_sqrt<S>(s / (S)len);
}
#undef LDEQ_DL

#ifndef LDEQ_FWDSENS_PREFETCH_ROWS
#define LDEQ_FWDSENS_PREFETCH_ROWS 24
#endif
#ifndef LDEQ_FWDSENS_THREADS
#define LDEQ_FWDSENS_THREADS 128
#endif

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// ---- one step on duals, per method ---------------------------------------------------------------------------
// Tsit5: written out (the arithmetic order is the oracle's tsit5_step, bit for bit); DP5 / BS3 / RK4: the table-driven
// form of the oracle's erk_step (zero coefficients skipped, first term a product, the rest FMAs).
struct Tsit5Dual {
    static constexpr int NS = 7, ORDER = 5;
    template <class RHS, class S, int NP>
    __device__ __forceinline__ static void step(const Dual<S, NP>* u, const Dual<S, NP>* L, double t, double dts,
                                                Dual<S, NP> (*k)[RHS::ZD], Dual<S, NP>* unew) {
        constexpr int Z = RHS::ZD;
        using D = Dual<S, NP>;
        using Tb = Tab<S>;
        D tmp[Z], sum;
        for (int i = 0; i < Z; ++i) { sum = dual_scale(Tb::a21, k[0][i]); tmp[i] = dual_axpy_time(u[i], dts, sum); }
        RHS::f(k[1], tmp, L, t + Tb::c2 * dts);
        for (int i = 0; i < Z; ++i) {
            sum = dual_scale(Tb::a31, k[0][i]); sum = dual_fma(Tb::a32, k[1][i], sum);
            tmp[i] = dual_axpy_time(u[i], dts, sum);
        }
        RHS::f(k[2], tmp, L, t + Tb::c3 * dts);
        for (int i = 0; i < Z; ++i) {
            sum = dual_scale(Tb::a41, k[0][i]); sum = dual_fma(Tb::a42, k[1][i], sum); sum = dual_fma(Tb::a43, k[2][i], sum);
            tmp[i] = dual_axpy_time(u[i], dts, sum);
        }
        RHS::f(k[3], tmp, L, t + Tb::c4 * dts);
        for (int i = 0; i < Z; ++i) {
            sum = dual_scale(Tb::a51, k[0][i]); sum = dual_fma(Tb::a52, k[1][i], sum); sum = dual_fma(Tb::a53, k[2][i], sum);
            sum = dual_fma(Tb::a54, k[3][i], sum);
            tmp[i] = dual_axpy_time(u[i], dts, sum);
        }
        RHS::f(k[4], tmp, L, t + Tb::c5 * dts);
        for (int i = 0; i < Z; ++i) {
            sum = dual_scale(Tb::a61, k[0][i]); sum = dual_fma(Tb::a62, k[1][i], sum); sum = dual_fma(Tb::a63, k[2][i], sum);
            sum = dual_fma(Tb::a64, k[3][i], sum); sum = dual_fma(Tb::a65, k[4][i], sum);
            tmp[i] = dual_axpy_time(u[i], dts, sum);
        }
        RHS::f(k[5], tmp, L, t + dts);
        for (int i = 0; i < Z; ++i) {
            sum = dual_scale(Tb::a71, k[0][i]); sum = dual_fma(Tb::a72, k[1][i], sum); sum = dual_fma(Tb::a73, k[2][i], sum);
            sum = dual_fma(Tb::a74, k[3][i], sum); sum = dual_fma(Tb::a75, k[4][i], sum); sum = dual_fma(Tb::a76, k[5][i], sum);
            unew[i] = dual_axpy_time(u[i], dts, sum);
        }
        RHS::f(k[6], unew, L, t + dts);
    }
    // sum_j btilde_j k_j of one state component
    template <class S, int NP, int Z>
    __device__ __forceinline__ static Dual<S, NP> err_sum(Dual<S, NP> (*k)[Z], int i) {
        using Tb = Tab<S>;
        Dual<S, NP> sum = dual_scale(Tb::bt1, k[0][i]);
        sum = dual_fma(Tb::bt2, k[1][i], sum); sum = dual_fma(Tb::bt3, k[2][i], sum);
        sum = dual_fma(Tb::bt4, k[3][i], sum); sum = dual_fma(Tb::bt5, k[4][i], sum); sum = dual_fma(Tb::bt6, k[5][i], sum);
        sum = dual_fma(Tb::bt7, k[6][i], sum);
        return sum;
    }
    // the Horner coefficients c_2..c_4 of one partial (c_1 = k_1), contracted in Float64: sum_j r_jm = 0 for m >= 2
    __device__ __forceinline__ static void dense_c(const double* kk, double* c2, double* c3, double* c4) {
        using Td = Tab<double>;
        *c2 = fma(Td::r72, kk[6], fma(Td::r62, kk[5], fma(Td::r52, kk[4], fma(Td::r42, kk[3], fma(Td::r32, kk[2], fma(Td::r22, kk[1], Td::r12 * kk[0]))))));
        *c3 = fma(Td::r73, kk[6], fma(Td::r63, kk[5], fma(Td::r53, kk[4], fma(Td::r43, kk[3], fma(Td::r33, kk[2], fma(Td::r23, kk[1], Td::r13 * kk[0]))))));
        *c4 = fma(Td::r74, kk[6], fma(Td::r64, kk[5], fma(Td::r54, kk[4], fma(Td::r44, kk[3], fma(Td::r34, kk[2], fma(Td::r24, kk[1], Td::r14 * kk[0]))))));
    }
};

template <class TB> struct ErkDual {
    static constexpr int NS = TB::NS, ORDER = TB::ORDER;
    template <class RHS, class S, int NP>
    __device__ __forceinline__ static void step(const Dual<S, NP>* u, const Dual<S, NP>* L, double t, double dts,
                                                Dual<S, NP> (*k)[RHS::ZD], Dual<S, NP>* unew) {
        constexpr int Z = RHS::ZD;
        using D = Dual<S, NP>;
        D tmp[Z];
#pragma unroll
        for (int j = 1; j < NS; ++j) {
            for (int i = 0; i < Z; ++i) {
                D sum = D((S)0);
                bool first = true;
#pragma unroll
                for (int l = 0; l < j; ++l) {
                    if (TB::a(j, l) == 0.0) continue;
                    sum = first ? dual_scale((S)TB::a(j, l), k[l][i]) : dual_fma((S)TB::a(j, l), k[l][i], sum);
                    first = false;
                }
                if (j < NS - 1) tmp[i] = dual_axpy_time(u[i], dts, sum);
                else unew[i] = dual_axpy_time(u[i], dts, sum);
            }
            if (j < NS - 1) RHS::f(k[j], tmp, L, t + TB::c(j) * dts);
            else RHS::f(k[j], unew, L, t + dts);
        }
    }
    template <class S, int NP, int Z>
    __device__ __forceinline__ static Dual<S, NP> err_sum(Dual<S, NP> (*k)[Z], int i) {
        Dual<S, NP> sum = Dual<S, NP>((S)0);
        bool first = true;
#pragma unroll
        for (int j = 0; j < NS; ++j) {
            if (TB::bt(j) == 0.0) continue;
            sum = first ? dual_scale((S)TB::bt(j), k[j][i]) : dual_fma((S)TB::bt(j), k[j][i], sum);
            first = false;
        }
        return sum;
    }
    __device__ __forceinline__ static void dense_c(const double* kk, double* c2, double* c3, double* c4) {
        double c[3] = {0.0, 0.0, 0.0};
#pragma unroll
        for (int m = 1; m < 4; ++m)
#pragma unroll
            for (int j = 0; j < NS; ++j)
                if (erk_r<TB>(j, m) != 0.0) c[m - 1] = fma(erk_r<TB>(j, m), kk[j], c[m - 1]);
        *c2 = c[0]; *c3 = c[1]; *c4 = c[2];
    }
};

// SEED_P: partials seeded on theta (NP = PD) -> dout = dtheta (p,B);  else on u0 (NP = ZD) -> dout = dz0 (z,B)
template <class M, class RHS, class S, int NP, bool SEED_P>
__device__ __forceinline__ void
erk_fwdsens_body(const S* __restrict__ z0, const S* __restrict__ theta, const double* __restrict__ tg, int B, GridInfo gi, int T,
                   KOpts o, int norm_partials, const int* __restrict__ sort_key, const S* __restrict__ dtraj, const int* __restrict__ primal_ret,
                   S* __restrict__ dout) {
    constexpr int Z = RHS::ZD, PD = RHS::PD;
    using D = Dual<S, NP>;
    constexpr int NS = M::NS;
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int ld = gi.ld;
    // save times of a verified-uniform grid are one DFMA (bit-identical to the table, ldeq_api.cu::upload_tgrid), not a load
    auto tgrid = [&](int k) -> double { return gi.uniform ? fma((double)k, gi.h, gi.t0) : tg[k]; };
    const bool wp = norm_partials != 0;
    // Lanes of a warp run until the slowest trajectory finishes.  The primal solve has already counted every trajectory's
    // accepted steps (sort_key = the tape's naccept): the CTA ranks its trajectories by that count and re-deals them, so a
    // warp holds 32 neighbours in step count.  Only the assignment of trajectories to lanes changes -- every trajectory's
    // arithmetic and its output slot are the same.
    if (sort_key) {
        __shared__ int s_key[LDEQ_FWDSENS_THREADS];
        __shared__ short s_order[LDEQ_FWDSENS_THREADS];
        const int tid = threadIdx.x, nt = blockDim.x;
        const int key = b < B ? sort_key[b] : 0x7fffffff;  // dead lanes go last
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
    if (b >= B) return;
    D u[Z], k[NS][Z], unew[Z], tmp[Z], sum, L[PD + RHS::NPRE];   // NPRE: slots for per-trajectory constants of the right-hand side
    const double t0 = tg[0], tend = tg[T - 1];
    const double dtmax = o.dtmax > 0.0 ? o.dtmax : (tend - t0);
    const double dtmin = o.dtmin > 0.0 ? o.dtmin : fmax(2.220446049250313e-16, ulp_of(t0));
    const S abstol = (S)o.abstol, reltol = (S)o.reltol;
    double acc[NP];
    double t = t0, dt = o.dt;
    {
        {
            for (int i = 0; i < Z; ++i) {
                u[i] = D(z0[(size_t)b * Z + i]);
                if (!SEED_P) u[i].d[i] = (S)1;
            }
            for (int i = 0; i < PD; ++i) {
                L[i] = D(theta[(size_t)b * PD + i]);
                if (SEED_P) L[i].d[i] = (S)1;
            }
            RHS::prepare(L);
            RHS::f(k[0], u, L, t0);  // fsalfirst
            if (o.adaptive && !(o.dt > 0.0)) {
                // Hairer initial step on the dual state
                S sk[Z];
                for (int i = 0; i < Z; ++i) {
                    sk[i] = abstol + dual_absnorm(u[i], wp) * reltol;
                    tmp[i] = dual_div_s(u[i], sk[i]);
                }
                const double d0 = (double)dual_rms(tmp, Z, wp);
                for (int i = 0; i < Z; ++i) tmp[i] = dual_div_s(k[0][i], sk[i]);
                const double d1 = (double)dual_rms(tmp, Z, wp);
                double dt0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * (d0 / d1);
                dt0 = fmin(dt0, dtmax);
                if (dt0 < 10.0 * 2.220446049250313e-16) {
                    dt = fmax(1e-6, dtmin);
                } else {
                    D u1[Z], f1[Z];
                    for (int i = 0; i < Z; ++i) u1[i] = dual_axpy_time(u[i], dt0, k[0][i]);
                    RHS::f(f1, u1, L, t0 + dt0);
                    for (int i = 0; i < Z; ++i) tmp[i] = dual_div_s(f1[i] - k[0][i], sk[i]);
                    const double d2 = (double)dual_rms(tmp, Z, wp) / dt0;
                    const double m = fmax(d1, d2);
                    const double dt1 = (m <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : ::pow(10.0, -(2.0 + log10(m)) / (double)M::ORDER);
                    dt = fmax(dtmin, fmin(100.0 * dt0, fmin(dt1, dtmax)));
                }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < NP; ++q) acc[q] = 0.0;
    // save point 0 is u0 itself
    for (int i = 0; i < Z; ++i)
#pragma unroll
        for (int q = 0; q < NP; ++q) acc[q] += (double)u[i].d[q] * (double)dtraj[(size_t)b * Z + i];
    PiState pst = pi_init(o);
    int ks = 1, ret = RET_SUCCESS;
    long long iters = 0;
    if (!(dt > 0.0) || !isfinite(dt)) ret = RET_DTLESSTHANMIN;
    // The cotangent rows this lane will consume are requested into L1 a few steps ahead (one prefetch per row, 8 sectors
    // per warp instruction): without it the save loop below waits ~600 cycles on every row (ncu: 45 % of all stall samples).
    int kpf = 1;
    // dvn always holds the cotangent row of the next pending save point: its load is in flight during the stages
    S dvn[Z];
#pragma unroll
    for (int i = 0; i < Z; ++i) dvn[i] = T > 1 ? dtraj[((size_t)ld + b) * Z + i] : (S)0;
    while (ks < T && ret == RET_SUCCESS) {
        if (iters >= o.maxiters) { ret = RET_MAXITERS; break; }
        ++iters;
        {
            const int hi = ks + LDEQ_FWDSENS_PREFETCH_ROWS < T ? ks + LDEQ_FWDSENS_PREFETCH_ROWS : T;
            for (; kpf < hi; ++kpf) prefetch_l1(dtraj + ((size_t)kpf * ld + b) * Z);
        }
        const double dts = fmin(dt, tend - t);
        double tnew = t + dts;
        if (::fabs(tnew - tend) < 100.0 * ulp_of(fmax(::fabs(t), ::fabs(tend)))) tnew = tend;
        M::template step<RHS, S, NP>(u, L, t, dts, k, unew);  // one step on duals
        double EEst = 0.0;
        if (o.adaptive) {
            for (int i = 0; i < Z; ++i) {
                sum = M::template err_sum<S, NP, Z>(k, i);
                const D ut = dual_scale_time(dts, sum);
                const S a0 = dual_absnorm(u[i], wp), a1 = dual_absnorm(unew[i], wp);
                const S sk = abstol + (a0 > a1 ? a0 : a1) * reltol;
                tmp[i] = dual_div_s(ut, sk);
            }
            EEst = (double)dual_rms(tmp, Z, wp);
        }
        bool finite = true;
        for (int i = 0; i < Z; ++i) finite = finite && s_finite<S>(unew[i].v);
        if (!finite || EEst != EEst) { ret = RET_UNSTABLE; break; }
        bool accept = true;
        double dt_next = dt;
        if (o.adaptive) accept = pi_controller(o, EEst, dts, dtmax, pst, dt_next);
        if (accept) {
            // saveat: every pending time <= tnew.  Only  sum_k <d u(t_k)/d seed, Delta_k>  is wanted, and the dense output is
            // linear in the partials of (u_n, k_1..k_7): with Horner coefficients c_m = sum_j r_jm k_j,
            //   d u(t_k) = d u_n + dt Theta (d c_1 + Theta (d c_2 + Theta (d c_3 + Theta d c_4))),
            // so every save point only accumulates the 4 weights dt Theta^m Delta_k (and Delta_k itself) per state
            // component -- independent of the number of partials -- and the step pays the contraction with the d c_m once.
            // (The dense output does not feed back into the step-size control, so this regrouping of the reference's
            // per-point evaluation leaves the step sequence untouched; the result agrees to rounding.)
            S wsum[Z], w1[Z], w2[Z], w3[Z], w4[Z];
#pragma unroll
            for (int i = 0; i < Z; ++i) wsum[i] = w1[i] = w2[i] = w3[i] = w4[i] = (S)0;
            bool interior = false;
            const double inv = 1.0 / dts;
            double tsv = ks < T ? tgrid(ks) : 0.0;
            while (ks < T && tsv <= tnew) {
                S dv[Z];
#pragma unroll
                for (int i = 0; i < Z; ++i) dv[i] = dvn[i];
                if (ks + 1 < T) {
#pragma unroll
                    for (int i = 0; i < Z; ++i) dvn[i] = dtraj[((size_t)(ks + 1) * ld + b) * Z + i];
                }
                if (tsv == tnew) {
#pragma unroll
                    for (int i = 0; i < Z; ++i)
#pragma unroll
                        for (int q = 0; q < NP; ++q) acc[q] += (double)unew[i].d[q] * (double)dv[i];
                } else {
                    const S th = (S)((tsv - t) * inv);
                    const S a1 = (S)dts * th, a2 = a1 * th, a3 = a2 * th, a4 = a3 * th;
#pragma unroll
                    for (int i = 0; i < Z; ++i) {
                        wsum[i] += dv[i];
                        w1[i] = s_fma<S>(a1, dv[i], w1[i]);
                        w2[i] = s_fma<S>(a2, dv[i], w2[i]);
                        w3[i] = s_fma<S>(a3, dv[i], w3[i]);
                        w4[i] = s_fma<S>(a4, dv[i], w4[i]);
                    }
                    interior = true;
                }
                ++ks;
                tsv = ks < T ? tgrid(ks) : 0.0;
            }
            if (interior) {
#pragma unroll
                for (int i = 0; i < Z; ++i)
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        // c_m = sum_j r_jm k_j cancels heavily (sum_j r_jm = 0 for m >= 2): contract in Float64
                        double kk[NS], c2, c3, c4;
#pragma unroll
                        for (int j = 0; j < NS; ++j) kk[j] = (double)k[j][i].d[q];
                        const double k1 = kk[0];
                        M::dense_c(kk, &c2, &c3, &c4);
                        acc[q] += (double)u[i].d[q] * (double)wsum[i] +
                                  (k1 * (double)w1[i] + c2 * (double)w2[i] + c3 * (double)w3[i] + c4 * (double)w4[i]);
                    }
            }
            t = tnew;
            for (int i = 0; i < Z; ++i) { u[i] = unew[i]; k[0][i] = k[NS - 1][i]; }
        }
        if (o.adaptive) dt = dt_next;
        if (ks < T && o.adaptive && (!(::fabs(dt) > dtmin) || !isfinite(dt))) { ret = RET_DTLESSTHANMIN; break; }
    }
    // a failed solve (dual or primal) contributes nothing: its NaN block is a constant of the differentiation (GOKU.jl:114)
    const bool ok = ret == RET_SUCCESS && primal_ret[b] == RET_SUCCESS;
#pragma unroll
    for (int q = 0; q < NP; ++q) dout[(size_t)b * NP + q] = ok ? (S)acc[q] : (S)0;
}

}  // namespace ldeq
