// ldeq_fwdsens.cu -- LDEQ_SENSE_FORWARD_DUAL for the built-in right-hand sides: instantiations of ldeq_fwdsens.cuh (the
// reference's ForwardDiffSensitivity pullback restated literally).  Compiled with -fmad=false (build.py) like the oracle's
// -ffp-contract=off: only the explicit fma() calls fuse.  This IS the library's default reverse pass since round 2 (what the
// reference's diffeq structs request, pendulum.jl:11); the discrete adjoint (~3x cheaper, equal to this within the solver
// tolerance) is the explicit opt-in LDEQ_SENSE_DISCRETE_ADJOINT.
#include "ldeq_fwdsens_kernels.cuh"

namespace ldeq {

void builtin_fwdsens_tsit5(int kind, GokuKernels* k) { fill_fwdsens<Tsit5Dual>(kind, k[LDEQ_SOLVER_TSIT5]); }

}  // namespace ldeq
