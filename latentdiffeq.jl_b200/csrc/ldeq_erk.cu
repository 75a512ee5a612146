// ldeq_erk.cu -- the forward and discrete-adjoint kernels of the built-in right-hand sides (ldeq_tsit5.cuh), one set per
// value of the diffeq struct's `solver` field: Tsit5 (the reference's structs, pendulum.jl:11,58) and the table-driven
// methods of ldeq_erk.cuh, DP5(), BS3() and RK4() (SURVEY.md 8(f)4).  Same thread-per-trajectory kernels, ring, tape and
// discrete adjoint.
#include "ldeq_internal.h"
#include "ldeq_rhs.cuh"
#include "ldeq_tsit5.cuh"

namespace ldeq {

template <class M, class S, bool FRICTION>
static void fill(GokuKernels& k, int dtype) {
    k.fwd[dtype][0] = (void*)erk_fwd_kernel<M, PendulumRHS<S, FRICTION>, S, false>;
    k.fwd[dtype][1] = (void*)erk_fwd_kernel<M, PendulumRHS<S, FRICTION>, S, true>;
    k.bwd[dtype] = (void*)erk_bwd_kernel<M, PendulumRHS<S, FRICTION>, S>;
}

template <bool FRICTION>
static void fill_solvers(GokuKernels* k) {
    fill<Tsit5M, float, FRICTION>(k[LDEQ_SOLVER_TSIT5], LDEQ_F32);
    fill<Tsit5M, double, FRICTION>(k[LDEQ_SOLVER_TSIT5], LDEQ_F64);
    fill<DP5M, float, FRICTION>(k[LDEQ_SOLVER_DP5], LDEQ_F32);
    fill<DP5M, double, FRICTION>(k[LDEQ_SOLVER_DP5], LDEQ_F64);
    fill<BS3M, float, FRICTION>(k[LDEQ_SOLVER_BS3], LDEQ_F32);
    fill<BS3M, double, FRICTION>(k[LDEQ_SOLVER_BS3], LDEQ_F64);
    fill<RK4M, float, FRICTION>(k[LDEQ_SOLVER_RK4], LDEQ_F32);
    fill<RK4M, double, FRICTION>(k[LDEQ_SOLVER_RK4], LDEQ_F64);
}

void builtin_solve_kernels(int kind, GokuKernels* k) {
    if (kind == LDEQ_RHS_PENDULUM_FRICTION) fill_solvers<true>(k);
    else fill_solvers<false>(k);
}

}  // namespace ldeq
