// ldeq_comm.cu -- NCCL route of the one exchange step of the path: the sum of the flat parameter gradient over the
// data-parallel ranks (SURVEY.md 8(e); the reference's training step, examples/pendulum_friction-less/model_train.jl:195-201,
// is single-process).  NCCL is resolved at run time so that the library loads on machines without it.
#include <dlfcn.h>

#include <cstdlib>
#include <cstring>

#include "ldeq_internal.h"

namespace {

struct NcclId { char internal[LDEQ_COMM_ID_BYTES]; };  // ncclUniqueId
typedef int (*fn_get_id)(NcclId*);
typedef int (*fn_init_rank)(void**, int, NcclId, int);
typedef int (*fn_allreduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*fn_destroy)(void*);
typedef const char* (*fn_errstr)(int);
enum { F_ID = 0, F_INIT, F_ALLREDUCE, F_DESTROY, F_ERRSTR };
const int kNcclFloat32 = 7, kNcclSum = 0;

int load_nccl(ldeq_handle* h) {
    if (h->nccl_lib) return LDEQ_OK;
    const char* name = getenv("LDEQ_NCCL_LIB");
    void* lib = dlopen(name && *name ? name : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return ldeq::set_err(h, LDEQ_ERR_UNSUPPORTED, "libnccl.so.2 not found (set LDEQ_NCCL_LIB)");
    const char* syms[5] = {"ncclGetUniqueId", "ncclCommInitRank", "ncclAllReduce", "ncclCommDestroy", "ncclGetErrorString"};
    for (int i = 0; i < 5; ++i) {
        h->nccl_fn[i] = dlsym(lib, syms[i]);
        if (!h->nccl_fn[i]) {
            dlclose(lib);
            return ldeq::set_err(h, LDEQ_ERR_UNSUPPORTED, "libnccl: missing symbol");
        }
    }
    h->nccl_lib = lib;
    return LDEQ_OK;
}

int nccl_err(ldeq_handle* h, const char* what, int rc) {
    std::string msg = std::string(what) + ": " + ((fn_errstr)h->nccl_fn[F_ERRSTR])(rc);
    return ldeq::set_err(h, LDEQ_ERR_CUDA, msg.c_str());
}

}  // namespace

extern "C" {

int ldeq_comm_unique_id(ldeq_handle* h, void* id_out) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!id_out) return ldeq::set_err(h, LDEQ_ERR_INVALID, "null argument");
    int rc = load_nccl(h);
    if (rc) return rc;
    NcclId id;
    const int nrc = ((fn_get_id)h->nccl_fn[F_ID])(&id);
    if (nrc) return nccl_err(h, "ncclGetUniqueId", nrc);
    memcpy(id_out, &id, sizeof(id));
    return LDEQ_OK;
}

int ldeq_comm_init(ldeq_handle* h, const void* unique_id, int rank, int nranks) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!unique_id || nranks < 1 || rank < 0 || rank >= nranks) return ldeq::set_err(h, LDEQ_ERR_INVALID, "comm_init: bad rank / nranks / id");
    if (h->nccl_comm) return ldeq::set_err(h, LDEQ_ERR_INVALID, "comm_init: the handle already has a communicator");
    int rc = load_nccl(h);
    if (rc) return rc;
    LDEQ_CUDA(cudaSetDevice(h->device));
    NcclId id;
    memcpy(&id, unique_id, sizeof(id));
    void* comm = nullptr;
    const int nrc = ((fn_init_rank)h->nccl_fn[F_INIT])(&comm, nranks, id, rank);
    if (nrc) return nccl_err(h, "ncclCommInitRank", nrc);
    h->nccl_comm = comm;
    h->nccl_rank = rank;
    h->nccl_nranks = nranks;
    return LDEQ_OK;
}

int ldeq_allreduce_grads(ldeq_handle* h, float* grads_flat, int64_t n, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (int rc = ldeq::refuse_capture(h, (cudaStream_t)stream, "ldeq_allreduce_grads", "multi-GPU capture is not supported")) return rc;
    if (!h->nccl_comm) return ldeq::set_err(h, LDEQ_ERR_INVALID, "allreduce_grads: call ldeq_comm_init first");
    if (!grads_flat || n < 0) return ldeq::set_err(h, LDEQ_ERR_INVALID, "allreduce_grads: bad buffer");
    if (n == 0) return LDEQ_OK;
    LDEQ_CUDA(cudaSetDevice(h->device));
    const int nrc = ((fn_allreduce)h->nccl_fn[F_ALLREDUCE])(grads_flat, grads_flat, (size_t)n, kNcclFloat32, kNcclSum, h->nccl_comm,
                                                           (cudaStream_t)stream);
    if (nrc) return nccl_err(h, "ncclAllReduce", nrc);
    return LDEQ_OK;
}

int ldeq_comm_destroy(ldeq_handle* h) {
    if (!h) return LDEQ_ERR_INVALID;
    if (h->nccl_comm) {
        cudaSetDevice(h->device);
        cudaDeviceSynchronize();
        ((fn_destroy)h->nccl_fn[F_DESTROY])(h->nccl_comm);
        h->nccl_comm = nullptr;
        h->nccl_nranks = 0;
    }
    return LDEQ_OK;
}

}  // extern "C"
