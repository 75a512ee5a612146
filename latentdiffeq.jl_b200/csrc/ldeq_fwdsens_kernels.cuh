// ldeq_fwdsens_kernels.cuh -- kernel entry points of the forward-dual pullback for the built-in right-hand sides, shared by
// ldeq_fwdsens.cu (Tsit5) and ldeq_erk_fwdsens.cu (DP5 / BS3 / RK4).  Both are compiled with -fmad=false (build.py).
#pragma once
#include "ldeq_internal.h"
#include "ldeq_fwdsens.cuh"

#ifndef LDEQ_FWDSENS_MINBLOCKS
// 5 CTAs of 128 threads per SM (<= 102 registers; the u0-seeded Float32 kernel spills 80 bytes): measured 6.20 -> 5.93 ms for
// the pair of pullback launches at 2^20 x 200 against 4 CTAs / 128 registers (6 CTAs: 5.90 ms with 3x the spills)
#define LDEQ_FWDSENS_MINBLOCKS 5
#endif

namespace ldeq {

// pendulum.jl:19-26 / :65-74 on duals (G, b, m are Float32 literals of the reference, rounded to S)
template <bool FRICTION> struct PendulumDualRHS {
    static constexpr int ZD = 2, PD = 1;
    // -G/L is a constant of the trajectory: the dual quotient (1 + NP IEEE divisions) is taken ONCE and kept in an extra
    // parameter slot instead of in each of the ~7 right-hand-side evaluations of every step -- the same bits, 21 divisions
    // per attempted step fewer
    static constexpr int NPRE = 1;
    template <class D> __device__ __forceinline__ static void prepare(D* p) {
        typedef typename D::value_type S;
        const D G((S)10.0f);
        p[PD] = -G / p[0];
    }
    template <class D> __device__ __forceinline__ static void f(D* du, const D* u, const D* p, double) {
        typedef typename D::value_type S;
        du[0] = u[1];
        const D a = p[PD] * sin(u[0]);
        if (FRICTION) {
            const S bm = (S)0.7f / (S)1.0f;
            du[1] = a - bm * u[1];
        } else {
            du[1] = a;
        }
    }
};

// MD: the method on duals, Tsit5Dual or ErkDual<TabDP5> ...
template <class MD, class S, int NP, bool FRICTION, bool SEED_P>
__global__ void __launch_bounds__(LDEQ_FWDSENS_THREADS, LDEQ_FWDSENS_MINBLOCKS)
erk_fwdsens_kernel(const S* __restrict__ z0, const S* __restrict__ theta, const double* __restrict__ tg, int B, GridInfo gi, int T,
                   KOpts o, int norm_partials, const int* __restrict__ sort_key, const S* __restrict__ dtraj, const int* __restrict__ primal_ret,
                   S* __restrict__ dout) {
    erk_fwdsens_body<MD, PendulumDualRHS<FRICTION>, S, NP, SEED_P>(z0, theta, tg, B, gi, T, o, norm_partials, sort_key, dtraj, primal_ret, dout);
}

// the pullback entries of the kernel table of method MD
template <class MD, bool FRICTION>
void fill_fwdsens(GokuKernels& k) {
    k.fwdsens[LDEQ_F32][0] = (void*)erk_fwdsens_kernel<MD, float, 1, FRICTION, true>;
    k.fwdsens[LDEQ_F32][1] = (void*)erk_fwdsens_kernel<MD, float, 2, FRICTION, false>;
    k.fwdsens[LDEQ_F64][0] = (void*)erk_fwdsens_kernel<MD, double, 1, FRICTION, true>;
    k.fwdsens[LDEQ_F64][1] = (void*)erk_fwdsens_kernel<MD, double, 2, FRICTION, false>;
}
template <class MD>
void fill_fwdsens(int kind, GokuKernels& k) {
    if (kind == LDEQ_RHS_PENDULUM_FRICTION) fill_fwdsens<MD, true>(k);
    else fill_fwdsens<MD, false>(k);
}

}  // namespace ldeq
