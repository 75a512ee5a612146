// ldeq_erk_fwdsens.cu -- LDEQ_SENSE_FORWARD_DUAL (the reference's dual-number re-solves, ldeq_fwdsens.cuh) for the other
// values of the diffeq struct's `solver` field: DP5, BS3, RK4 (SURVEY.md 8(f)4).  Compiled with -fmad=false like
// ldeq_fwdsens.cu.
#include "ldeq_fwdsens_kernels.cuh"

namespace ldeq {

void builtin_fwdsens_erk(int kind, GokuKernels* k) {
    fill_fwdsens<ErkDual<TabDP5>>(kind, k[LDEQ_SOLVER_DP5]);
    fill_fwdsens<ErkDual<TabBS3>>(kind, k[LDEQ_SOLVER_BS3]);
    fill_fwdsens<ErkDual<TabRK4>>(kind, k[LDEQ_SOLVER_RK4]);
}

}  // namespace ldeq
