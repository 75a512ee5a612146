// ldeq_internal.h -- host-side objects behind the opaque C-ABI types of include/ldeq.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/ldeq.h"
#include "ldeq_common.cuh"

#define LDEQ_MAX_SLABS 8  // column slabs a host-resident batch is cut into (ldeq_api.cu)
#define LDEQ_GRID_CACHE 16  // unpinned immutable grid copies a handle keeps (ldeq_handle::grid_cache)

struct ldeq_handle {
    int device = 0;
    std::string err;
    int64_t launches = 0;
    // device copy of the most recent time grid (re-uploaded only when the host grid changes)
    double* d_tgrid = nullptr;
    size_t d_tgrid_cap = 0;
    std::vector<double> h_tgrid;
    // the cached grid is t0 + k*h bit for bit (checked on upload): kernels then compute save times instead of looking them up
    double grid_t0 = 0.0, grid_h = 0.0;
    int grid_uniform = 0;
    // Grids a captured CUDA graph may read: d_tgrid above is overwritten in place when a call brings another grid, so a
    // solve under stream capture reads an immutable device copy from this cache instead.  Every eager upload of a new grid
    // adds one (the most recent LDEQ_GRID_CACHE unpinned ones are kept); a capture pins the entry it reads, and pinned
    // entries live until ldeq_destroy.
    struct GridEntry {
        std::vector<double> t;
        double* d = nullptr;
        double t0 = 0.0, h = 0.0;
        int uniform = 0;
        bool pinned = false;
        uint64_t last_use = 0;
    };
    std::vector<GridEntry> grid_cache;
    uint64_t grid_clock = 0;
    // grow-only device scratch for the *_host entry points and reductions
    void* scratch[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t scratch_cap[4] = {0, 0, 0, 0};
    // a scratch slot that a capture has referenced is retired (kept until ldeq_destroy) instead of freed when it grows
    bool scratch_captured[4] = {false, false, false, false};
    std::vector<void*> retired_scratch;
    // ELBO reduction workspace
    double* d_partials = nullptr;
    unsigned int* d_counter = nullptr;
    int n_partials = 0;
    int sm_count = 148;
    int tape_hint = 0;  // largest accepted-step count seen so far: sizes the next automatic tape
    // recycled {pinned info slot, event} pairs for tapes (cudaMallocHost / cudaEventCreate are slow)
    struct Slot { int32_t* h_info; cudaEvent_t ev; };
    std::vector<Slot> free_slots;
    std::vector<Slot> deferred_slots;  // released under capture: returned to free_slots by the next slot_acquire
    std::vector<int32_t*> pinned_blocks;
    // NCCL communicator of the gradient all-reduce (ldeq_comm.cu; libnccl is dlopen'ed on first use)
    void* nccl_lib = nullptr;
    void* nccl_comm = nullptr;
    void* nccl_fn[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    int nccl_rank = 0, nccl_nranks = 0;
    // copy streams + events of the pipelined *_host entry points (created on first use)
    cudaStream_t up = nullptr, down = nullptr;
    cudaEvent_t ev_fwd[LDEQ_MAX_SLABS] = {}, ev_up[LDEQ_MAX_SLABS] = {}, ev_join = nullptr;
};

struct ldeq_rhs {
    int kind = 0;  // ldeq_rhs_kind, or -1 for an NVRTC-compiled user RHS
    int z_dim = 2, p_dim = 1;
    void* module = nullptr;  // CUmodule of a user RHS
    void* fn[12] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // a user RHS under another `solver`: its own NVRTC module, compiled on first use from the kept source
    struct PerSolver { void* module = nullptr; void* fn[12] = {}; };
    PerSolver alt[4];
    std::string user_src;
};

struct ldeq_tape {
    int dtype = 0, rhs_kind = 0, B = 0, T = 0, z_dim = 2, p_dim = 1, cap = 0;
    const ldeq_rhs* rhs = nullptr;
    void* base = nullptr;  // one stream-ordered allocation, carved into the arrays below
    double* t = nullptr;
    void* u = nullptr;
    void* theta = nullptr;
    double* tgrid = nullptr;
    int32_t* retcode = nullptr;
    int32_t* naccept = nullptr;
    int32_t* nreject = nullptr;
    int32_t* info = nullptr;     // device {overflow count, max naccept}
    int32_t* h_info = nullptr;   // pinned host mirror of info, valid once `ready` has completed
    cudaEvent_t ready = nullptr;
    bool checked = false;
    ldeq::KOpts kopts;
    double grid_t0 = 0.0, grid_h = 0.0;
    int grid_uniform = 0;
    int sense = 0;  // ldeq_sensealg of the solve that made this tape
    int solver = 0; // ldeq_solver of that solve
    // a tape recorded slab by slab (ldeq_solve_fwd_host) is a list of single-slab tapes: parts[i] covers trajectories
    // part_b0[i] .. part_b0[i] + parts[i]->B - 1 and owns its own arrays; the parent then owns nothing else
    std::vector<ldeq_tape*> parts;
    std::vector<int> part_b0;
};

namespace ldeq {

int set_err(ldeq_handle* h, int code, const char* what, cudaError_t ce = cudaSuccess);
// True while `s` is being captured into a CUDA graph (or its capture was invalidated): work enqueued now is recorded, not
// run, so the host can neither wait for it nor read its results, and every pointer it reads is frozen into the graph.
bool capturing(cudaStream_t s);
// LDEQ_ERR_UNSUPPORTED with "<what>: not available under CUDA graph capture (<why>)" when `s` is capturing, else LDEQ_OK.
int refuse_capture(ldeq_handle* h, cudaStream_t s, const char* what, const char* why);
int upload_tgrid(ldeq_handle* h, const double* t_host, int T, cudaStream_t s);
// grows scratch[slot] to `bytes` on `s`; under capture it refuses to grow (LDEQ_ERR_UNSUPPORTED) and marks the slot captured
int ensure_scratch(ldeq_handle* h, int slot, size_t bytes, cudaStream_t s);
KOpts to_kopts(const ldeq_opts* o);
int bwd_sort_lanes();  // ldeq_api.cu: lane re-deal of the discrete-adjoint kernels (LDEQ_BWD_SORT)
// pooled pinned {int32 x 2} mirror + event (ldeq_api.cu)
bool slot_acquire(ldeq_handle* h, int32_t** h_info, cudaEvent_t* ev);
void slot_release(ldeq_handle* h, int32_t* h_info, cudaEvent_t ev);
// ldeq_fwdsens.cu: the reference's ForwardDiffSensitivity pullback (two dual-number re-solves per trajectory)
cudaError_t launch_fwdsens(const ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s);
// ldeq_erk_fwdsens.cu / ldeq_erk.cu: the same kernels for solver = DP5 / BS3 / RK4 (built-in right-hand sides)
cudaError_t launch_erk_fwdsens(const ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s);
cudaError_t launch_erk_bwd(const ldeq_tape* tape, const void* dtraj, int ld, void* dz0, void* dtheta, cudaStream_t s);
// ldeq_user_rhs.cu: kernel table of a user RHS for `solver` (compiles the variant on first use); null + error text on failure
void* const* user_rhs_kernels(ldeq_handle* h, const ldeq_rhs* rhs, int solver);

#define LDEQ_CUDA(call)                                                    \
    do {                                                                   \
        cudaError_t _e = (call);                                           \
        if (_e != cudaSuccess) return ldeq::set_err(h, LDEQ_ERR_CUDA, #call, _e); \
    } while (0)

}  // namespace ldeq
