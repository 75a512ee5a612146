// ldeq_loss.cu -- ELBO reduction (forward + gradient), fused AdamW and the reparameterised sample.
//
//   ldeq_elbo_fwd_bwd   loss_batch (reference examples/pendulum_friction-less/model_train.jl:225-238) with
//                       kl / vector_kl (src/utils/utils.jl:16-49)
//   ldeq_adamw_step     Flux.Optimise.update!(ADAMW(eta,(b1,b2),decay), ps, grad)  (model_train.jl:138,201)
//   ldeq_sample         sample(mu, logvar, model)  (src/models/GOKU.jl:155-173, src/models/LatentODE.jl:82-98);
//                       the reference draws the noise on the host and uploads it (GOKU.jl:169-170), here it
//                       is drawn on the device with a counter-based Philox4x32-10 generator.
//
// All three are HBM-bound streaming kernels: 128-bit loads, grid sized to the SM count, one pass.
#include "ldeq_internal.h"

namespace ldeq {

// ---- ELBO ----------------------------------------------------------------------------------------
// Reconstruction term: sum_pixels mean_{B,T}(x - xhat)^2 = (1/(B T)) sum_all (x - xhat)^2.
// One streaming pass computes the sum of squares and (optionally) writes
// dxhat = grad_scale * 2 (xhat - x) / (B T).  Block partials are combined in a fixed order by the
// last block to finish, so the result is run-to-run deterministic.
#define ELBO_THREADS 256

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// KL of all heads: one block, grid-stride; writes loss[2] = sum_h (1/B) sum 0.5 (e^lv + mu^2 - lv - 1)
struct KlHeads {
    const float* mu[4];
    const float* lv[4];
    float* dmu[4];
    float* dlv[4];
    int n[4];  // elements per head = d_h * B
    int n_heads;
};

// KL term and its gradients, grid-strided over the heads' elements; block b leaves its partial sum in kl_partials[b]
// (summed in index order by the last block of elbo_mse_kernel: deterministic).  One block used to do all of it: 0.53 ms
// at B = 8192 (ncu, profiles/r2_loss_kernels_summary.txt) -- as long as the 1.3 GB reconstruction term next to it.
#define ELBO_KL_BLOCKS 64
// DEV: beta is read from beta_dev (a CUDA graph replays it with new values) and gscale_beta = gscale * beta is formed here,
// in the same Float32 rounding as the host forms it for DEV = false
template <bool DEV>
__global__ void __launch_bounds__(ELBO_THREADS) elbo_kl_kernel(KlHeads hd, int B, float gscale_beta, const float* __restrict__ beta_dev,
                                                               double* __restrict__ kl_partials) {
    __shared__ double sh[ELBO_THREADS / 32];
    if (DEV) gscale_beta = __fmul_rn(gscale_beta, *beta_dev);
    double acc = 0.0;
    const float invB = 1.0f / (float)B;
    for (int hI = 0; hI < hd.n_heads; ++hI) {
        const float* __restrict__ mu = hd.mu[hI];
        const float* __restrict__ lv = hd.lv[hI];
        float part = 0.f;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hd.n[hI]; i += gridDim.x * blockDim.x) {
            const float m = mu[i], l = lv[i];
            const float e = expf(l);
            part += (e + m * m - l - 1.0f) * 0.5f;
            if (hd.dmu[hI]) hd.dmu[hI][i] = gscale_beta * m * invB;
            if (hd.dlv[hI]) hd.dlv[hI][i] = gscale_beta * 0.5f * (e - 1.0f) * invB;
        }
        acc += (double)part * (double)invB;
    }
    acc = warp_sum_d(acc);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < ELBO_THREADS / 32; ++w) t += sh[w];
        kl_partials[blockIdx.x] = t;
    }
}

// LOGITS: `xhat` holds the pre-activations a of a sigmoid output layer (the reconstructor's last layer, GOKU.jl:265-268):
// xhat = 1 / (1 + exp(-a)) is formed here and the gradient is taken with respect to a -- the activation's forward pass,
// its backward pass and the x-hat round trip through HBM between them and the loss never exist.
__device__ __forceinline__ float elbo_sigmoid(float a) { return 1.0f / (1.0f + expf(-a)); }

template <bool GRAD, bool LOGITS, bool DEV>
__global__ void __launch_bounds__(ELBO_THREADS)
elbo_mse_kernel(const float* __restrict__ x, const float* __restrict__ xhat, float* __restrict__ dxhat, size_t n,
                float inv_bt, float gscale, float beta, const float* __restrict__ beta_dev, double* __restrict__ partials,
                unsigned int* __restrict__ counter, const double* __restrict__ kl_partials, int n_kl, float* __restrict__ loss) {
    __shared__ float shw[ELBO_THREADS / 32];
    __shared__ bool is_last;
    const size_t n4 = n >> 2;
    const float g2 = 2.0f * inv_bt * gscale;
    float acc = 0.f;
    const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
    const float4* __restrict__ h4 = reinterpret_cast<const float4*>(xhat);
    float4* __restrict__ d4 = reinterpret_cast<float4*>(dxhat);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 a = __ldcs(x4 + i);
        float4 b = __ldcs(h4 + i);
        if (LOGITS) { b.x = elbo_sigmoid(b.x); b.y = elbo_sigmoid(b.y); b.z = elbo_sigmoid(b.z); b.w = elbo_sigmoid(b.w); }
        const float e0 = b.x - a.x, e1 = b.y - a.y, e2 = b.z - a.z, e3 = b.w - a.w;
        acc = fmaf(e0, e0, acc); acc = fmaf(e1, e1, acc); acc = fmaf(e2, e2, acc); acc = fmaf(e3, e3, acc);
        if (GRAD) {
            if (LOGITS) __stcs(d4 + i, make_float4(g2 * e0 * b.x * (1.0f - b.x), g2 * e1 * b.y * (1.0f - b.y), g2 * e2 * b.z * (1.0f - b.z),
                                                   g2 * e3 * b.w * (1.0f - b.w)));
            else __stcs(d4 + i, make_float4(g2 * e0, g2 * e1, g2 * e2, g2 * e3));
        }
    }
    // tail (n not a multiple of 4)
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const size_t i = (n4 << 2) + threadIdx.x;
        const float bh = LOGITS ? elbo_sigmoid(xhat[i]) : xhat[i];
        const float e = bh - x[i];
        acc = fmaf(e, e, acc);
        if (GRAD) dxhat[i] = LOGITS ? g2 * e * bh * (1.0f - bh) : g2 * e;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) shw[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < ELBO_THREADS / 32; ++w) t += (double)shw[w];
        partials[blockIdx.x] = t;
        __threadfence();
        const unsigned int done = atomicAdd(counter, 1u);
        is_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double t = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) t += __ldcg(partials + i);
        t = warp_sum_d(t);
        __shared__ double shd[ELBO_THREADS / 32];
        if ((threadIdx.x & 31) == 0) shd[threadIdx.x >> 5] = t;
        __syncthreads();
        if (threadIdx.x == 0) {
            double r = 0.0;
            for (int w = 0; w < ELBO_THREADS / 32; ++w) r += shd[w];
            const float rec = (float)(r * (double)inv_bt);
            double klsum = 0.0;
            for (int i = 0; i < n_kl; ++i) klsum += __ldcg(kl_partials + i);   // written by the preceding elbo_kl_kernel
            const float klf = (float)klsum;
            if (DEV) beta = *beta_dev;
            loss[1] = rec;
            loss[2] = klf;
            loss[0] = rec + beta * klf;
            *counter = 0u;  // ready for the next call
        }
    }
}

// ---- AdamW (Flux 0.13: Optimiser(ADAM, WeightDecay)) ---------------------------------------------
// Flux keeps (b1, b2) and their running powers in Float64, so the moment updates and the step are
// evaluated in Float64 and rounded to Float32 on the store; the weight decay term is Float32.
__device__ __forceinline__ void adamw_one(float& x, float g, float& m, float& v, double b1, double b2, double c1,
                                          double c2, double eps, double lr, float decay) {
    const double gd = (double)g;
    m = (float)(b1 * (double)m + (1.0 - b1) * gd);
    v = (float)(b2 * (double)v + (1.0 - b2) * gd * gd);
    float d = (float)((double)m / c1 / (sqrt((double)v / c2) + eps) * lr);
    d = __fadd_rn(d, __fmul_rn(decay, x));
    x = x - d;
}

// DEV: the bias corrections come from the device state that adamw_advance_kernel has just advanced
template <bool DEV>
__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ x, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t n,
             double b1, double b2, double c1, double c2, double eps, double lr, float decay, float gscale,
             const ldeq_adamw_state* __restrict__ state) {
    if (DEV) {
        c1 = 1.0 - state->beta1_pow;
        c2 = 1.0 - state->beta2_pow;
    }
    const size_t n4 = n >> 2;
    float4* x4 = reinterpret_cast<float4*>(x);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 xx = x4[i], gg = g4[i], mm = m4[i], vv = v4[i];
        adamw_one(xx.x, gg.x * gscale, mm.x, vv.x, b1, b2, c1, c2, eps, lr, decay);
        adamw_one(xx.y, gg.y * gscale, mm.y, vv.y, b1, b2, c1, c2, eps, lr, decay);
        adamw_one(xx.z, gg.z * gscale, mm.z, vv.z, b1, b2, c1, c2, eps, lr, decay);
        adamw_one(xx.w, gg.w * gscale, mm.w, vv.w, b1, b2, c1, c2, eps, lr, decay);
        x4[i] = xx; m4[i] = mm; v4[i] = vv;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const size_t i = (n4 << 2) + threadIdx.x;
        float xx = x[i], mm = m[i], vv = v[i];
        adamw_one(xx, g[i] * gscale, mm, vv, b1, b2, c1, c2, eps, lr, decay);
        x[i] = xx; m[i] = mm; v[i] = vv;
    }
}

// One thread: the next step of the running Float64 beta powers, the same multiplications in the same order as the host loop
// of ldeq_adamw_step.  A launch of its own, so that every CTA of the update reads the state after it has advanced.
__global__ void adamw_advance_kernel(ldeq_adamw_state* state, double b1, double b2) {
    state->step += 1;
    state->beta1_pow *= b1;
    state->beta2_pow *= b2;
}

// ---- all-reduce fused with AdamW over peer memory ----------------------------------------------------------------
#define LDEQ_MAX_PEERS 16
struct PeerBufs {
    const float* g[LDEQ_MAX_PEERS];  // gradient bucket of every rank (peer-mapped)
    float* x[LDEQ_MAX_PEERS];        // parameter replica of every rank (two-shot mode), else null
    int n;
};
// Plain 128-bit loads / stores on peer-mapped pointers travel over NVLink (peer data is not cached in the local L2).
// One-shot: every rank sums all buckets (rank order) and updates its whole replica.  Two-shot: every rank sums and
// updates its own slice [lo4, hi4) only and writes the new parameters into every replica.  2 MB per bucket for the
// default GOKU: latency-bound either way, so ONE launch instead of an NCCL all-reduce plus an optimiser kernel.
template <bool TWO_SHOT>
__global__ void __launch_bounds__(256)
allreduce_adamw_kernel(float* __restrict__ x, PeerBufs pb, float* __restrict__ m, float* __restrict__ v, size_t lo4, size_t hi4,
                       double b1, double b2, double c1, double c2, double eps, double lr, float decay, float gscale) {
    float4* x4 = reinterpret_cast<float4*>(x);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = lo4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi4; i += stride) {
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = 0; r < pb.n; ++r) {
            const float4 t = __ldcg(reinterpret_cast<const float4*>(pb.g[r]) + i);
            g.x += t.x; g.y += t.y; g.z += t.z; g.w += t.w;
        }
        float4 xx = x4[i], mm = m4[i], vv = v4[i];
        adamw_one(xx.x, g.x * gscale, mm.x, vv.x, b1, b2, c1, c2, eps, lr, decay);
        adamw_one(xx.y, g.y * gscale, mm.y, vv.y, b1, b2, c1, c2, eps, lr, decay);
        adamw_one(xx.z, g.z * gscale, mm.z, vv.z, b1, b2, c1, c2, eps, lr, decay);
        adamw_one(xx.w, g.w * gscale, mm.w, vv.w, b1, b2, c1, c2, eps, lr, decay);
        m4[i] = mm; v4[i] = vv;
        if (TWO_SHOT) {
            for (int r = 0; r < pb.n; ++r) reinterpret_cast<float4*>(pb.x[r])[i] = xx;  // includes this rank's own replica
        } else {
            x4[i] = xx;
        }
    }
}

// ---- Philox4x32-10 + Box-Muller -------------------------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0,
                                             uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
}
__device__ __forceinline__ void philox4x32_10(uint64_t ctr, uint64_t seed, uint32_t* out) {
    uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0u, c3 = 0u;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float* n0, float* n1) {
    // u in (0,1], v in [0,1)
    const float u = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);
    const float v = (float)(b >> 8) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * logf(u));
    float s, c;
    sincospif(2.0f * v, &s, &c);
    *n0 = r * c;
    *n1 = r * s;
}

// each thread produces 4 normals (one Philox block) for elements 4i..4i+3
// DEV: offset = *calls << 32, from the counter sample_advance_kernel has just incremented
template <bool DEV>
__global__ void __launch_bounds__(256)
sample_kernel(const float* __restrict__ mu, const float* __restrict__ lv, float* __restrict__ z, float* __restrict__ eps,
              size_t n, uint64_t seed, uint64_t offset, const uint64_t* __restrict__ calls) {
    if (DEV) offset = *calls << 32;
    const size_t nb = (n + 3) >> 2;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += stride) {
        uint32_t r[4];
        philox4x32_10(offset + i, seed, r);
        float e[4];
        box_muller(r[0], r[1], &e[0], &e[1]);
        box_muller(r[2], r[3], &e[2], &e[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const size_t idx = (i << 2) + j;
            if (idx < n) {
                // z = mu + eps * exp(logvar / 2)
                z[idx] = __fadd_rn(mu[idx], __fmul_rn(e[j], expf(lv[idx] * 0.5f)));
                if (eps) eps[idx] = e[j];
            }
        }
    }
}

__global__ void sample_advance_kernel(uint64_t* calls) { *calls += 1; }

}  // namespace ldeq

using namespace ldeq;

extern "C" {

// beta_dev != null: the _dev variants, beta is read on the device
static int elbo_impl(bool logits, ldeq_handle* h, const float* x, const float* xhat, const float* const* mu_host,
                     const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, float beta, const float* beta_dev,
                     int B, int T, int P, float grad_scale, float* loss, float* dxhat, float* const* dmu_host,
                     float* const* dlogvar_host, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!x || !xhat || !loss || n_heads < 0 || n_heads > 4 || B <= 0 || T <= 0 || P <= 0)
        return set_err(h, LDEQ_ERR_INVALID, "elbo: bad argument (n_heads <= 4)");
    if (n_heads > 0 && (!mu_host || !logvar_host || !head_dims_host)) return set_err(h, LDEQ_ERR_INVALID, "elbo: null heads");
    if ((((uintptr_t)x) | ((uintptr_t)xhat) | ((uintptr_t)dxhat)) & 15) return set_err(h, LDEQ_ERR_INVALID, "elbo: x, xhat, dxhat must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    const int max_blocks = h->sm_count * 8;
    if (!h->d_partials) {
        if (capturing(s))
            return set_err(h, LDEQ_ERR_UNSUPPORTED, "elbo: the reduction workspace is allocated by the first call, which cannot happen under "
                                                    "CUDA graph capture: call the loss once outside the capture first");
        LDEQ_CUDA(cudaMalloc((void**)&h->d_partials, sizeof(double) * (max_blocks + ELBO_KL_BLOCKS)));
        LDEQ_CUDA(cudaMalloc((void**)&h->d_counter, sizeof(unsigned int)));
        LDEQ_CUDA(cudaMemset(h->d_counter, 0, sizeof(unsigned int)));
        h->n_partials = max_blocks;
    }
    KlHeads hd;
    hd.n_heads = n_heads;
    for (int i = 0; i < 4; ++i) {
        hd.mu[i] = hd.lv[i] = nullptr; hd.dmu[i] = hd.dlv[i] = nullptr; hd.n[i] = 0;
    }
    for (int i = 0; i < n_heads; ++i) {
        hd.mu[i] = mu_host[i]; hd.lv[i] = logvar_host[i];
        hd.dmu[i] = dmu_host ? dmu_host[i] : nullptr;
        hd.dlv[i] = dlogvar_host ? dlogvar_host[i] : nullptr;
        hd.n[i] = head_dims_host[i] * B;
    }
    double* kl_partials = h->d_partials + max_blocks;
    int kl_grid = 1;
    for (int i = 0; i < n_heads; ++i) { const int w = (hd.n[i] + 4 * ELBO_THREADS - 1) / (4 * ELBO_THREADS); if (w > kl_grid) kl_grid = w; }
    if (kl_grid > ELBO_KL_BLOCKS) kl_grid = ELBO_KL_BLOCKS;
    if (beta_dev) elbo_kl_kernel<true><<<kl_grid, ELBO_THREADS, 0, s>>>(hd, B, grad_scale, beta_dev, kl_partials);
    else elbo_kl_kernel<false><<<kl_grid, ELBO_THREADS, 0, s>>>(hd, B, grad_scale * beta, nullptr, kl_partials);
    LDEQ_CUDA(cudaGetLastError());
    const size_t n = (size_t)P * B * T;
    size_t want = ((n >> 2) + ELBO_THREADS - 1) / ELBO_THREADS;
    int grid = (int)(want < (size_t)max_blocks ? (want ? want : 1) : (size_t)max_blocks);
    const float inv_bt = 1.0f / ((float)B * (float)T);
#define LDEQ_ELBO_LAUNCH(G, L, D) elbo_mse_kernel<G, L, D><<<grid, ELBO_THREADS, 0, s>>>(x, xhat, dxhat, n, inv_bt, grad_scale, beta, beta_dev, h->d_partials, h->d_counter, kl_partials, kl_grid, loss)
#define LDEQ_ELBO_LAUNCH_D(G, L) do { if (beta_dev) LDEQ_ELBO_LAUNCH(G, L, true); else LDEQ_ELBO_LAUNCH(G, L, false); } while (0)
    if (dxhat) { if (logits) LDEQ_ELBO_LAUNCH_D(true, true); else LDEQ_ELBO_LAUNCH_D(true, false); }
    else { if (logits) LDEQ_ELBO_LAUNCH_D(false, true); else LDEQ_ELBO_LAUNCH_D(false, false); }
#undef LDEQ_ELBO_LAUNCH_D
#undef LDEQ_ELBO_LAUNCH
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 2;
    return LDEQ_OK;
}

int ldeq_elbo_fwd_bwd(ldeq_handle* h, const float* x, const float* xhat, const float* const* mu_host,
                      const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, float beta, int B,
                      int T, int P, float grad_scale, float* loss, float* dxhat, float* const* dmu_host,
                      float* const* dlogvar_host, ldeq_stream stream) {
    return elbo_impl(false, h, x, xhat, mu_host, logvar_host, head_dims_host, n_heads, beta, nullptr, B, T, P, grad_scale, loss, dxhat, dmu_host,
                     dlogvar_host, stream);
}

int ldeq_elbo_fwd_bwd_dev(ldeq_handle* h, const float* x, const float* xhat, const float* const* mu_host,
                          const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, const float* beta, int B,
                          int T, int P, float grad_scale, float* loss, float* dxhat, float* const* dmu_host,
                          float* const* dlogvar_host, ldeq_stream stream) {
    if (h && !beta) return set_err(h, LDEQ_ERR_INVALID, "elbo: null beta");
    return elbo_impl(false, h, x, xhat, mu_host, logvar_host, head_dims_host, n_heads, 0.0f, beta, B, T, P, grad_scale, loss, dxhat, dmu_host,
                     dlogvar_host, stream);
}

int ldeq_elbo_logits_fwd_bwd(ldeq_handle* h, const float* x, const float* logits, const float* const* mu_host,
                             const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, float beta, int B,
                             int T, int P, float grad_scale, float* loss, float* dlogits, float* const* dmu_host,
                             float* const* dlogvar_host, ldeq_stream stream) {
    return elbo_impl(true, h, x, logits, mu_host, logvar_host, head_dims_host, n_heads, beta, nullptr, B, T, P, grad_scale, loss, dlogits, dmu_host,
                     dlogvar_host, stream);
}

int ldeq_elbo_logits_fwd_bwd_dev(ldeq_handle* h, const float* x, const float* logits, const float* const* mu_host,
                                 const float* const* logvar_host, const int32_t* head_dims_host, int n_heads, const float* beta, int B,
                                 int T, int P, float grad_scale, float* loss, float* dlogits, float* const* dmu_host,
                                 float* const* dlogvar_host, ldeq_stream stream) {
    if (h && !beta) return set_err(h, LDEQ_ERR_INVALID, "elbo: null beta");
    return elbo_impl(true, h, x, logits, mu_host, logvar_host, head_dims_host, n_heads, 0.0f, beta, B, T, P, grad_scale, loss, dlogits, dmu_host,
                     dlogvar_host, stream);
}

int ldeq_adamw_step(ldeq_handle* h, float* params, const float* grads, float* m, float* v, int64_t n, double lr,
                    double beta1, double beta2, double eps, float decay, int64_t step, float grad_scale,
                    ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!params || !grads || !m || !v || n < 0 || step < 1) return set_err(h, LDEQ_ERR_INVALID, "adamw: bad argument");
    if ((((uintptr_t)params) | ((uintptr_t)grads) | ((uintptr_t)m) | ((uintptr_t)v)) & 15)
        return set_err(h, LDEQ_ERR_INVALID, "adamw: buffers must be 16-byte aligned");
    if (n == 0) return LDEQ_OK;
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    // Flux: beta powers are running Float64 products of the Float64 betas
    const double b1 = beta1, b2 = beta2, lrd = lr, epsd = eps;
    double p1 = 1.0, p2 = 1.0;
    for (int64_t i = 0; i < step; ++i) { p1 *= b1; p2 *= b2; }
    size_t want = (((size_t)n >> 2) + 255) / 256;
    int grid = (int)(want < (size_t)h->sm_count * 8 ? (want ? want : 1) : (size_t)h->sm_count * 8);
    adamw_kernel<false><<<grid, 256, 0, s>>>(params, grads, m, v, (size_t)n, b1, b2, 1.0 - p1, 1.0 - p2, epsd, lrd, decay, grad_scale, nullptr);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    return LDEQ_OK;
}

int ldeq_adamw_step_dev(ldeq_handle* h, float* params, const float* grads, float* m, float* v, int64_t n, double lr,
                        double beta1, double beta2, double eps, float decay, ldeq_adamw_state* state, float grad_scale,
                        ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!params || !grads || !m || !v || !state || n < 0) return set_err(h, LDEQ_ERR_INVALID, "adamw: bad argument");
    if ((((uintptr_t)params) | ((uintptr_t)grads) | ((uintptr_t)m) | ((uintptr_t)v)) & 15)
        return set_err(h, LDEQ_ERR_INVALID, "adamw: buffers must be 16-byte aligned");
    if ((uintptr_t)state & 7) return set_err(h, LDEQ_ERR_INVALID, "adamw: state must be 8-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    adamw_advance_kernel<<<1, 1, 0, s>>>(state, beta1, beta2);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    if (n == 0) return LDEQ_OK;
    size_t want = (((size_t)n >> 2) + 255) / 256;
    int grid = (int)(want < (size_t)h->sm_count * 8 ? (want ? want : 1) : (size_t)h->sm_count * 8);
    adamw_kernel<true><<<grid, 256, 0, s>>>(params, grads, m, v, (size_t)n, beta1, beta2, 0.0, 0.0, eps, lr, decay, grad_scale, state);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    return LDEQ_OK;
}

int ldeq_allreduce_adamw_step(ldeq_handle* h, float* params, float* const* peer_params_host,
                              const float* const* peer_grads_host, int nranks, int rank, float* m, float* v, int64_t n,
                              double lr, double beta1, double beta2, double eps, float decay, int64_t step,
                              float grad_scale, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!params || !peer_grads_host || !m || !v || n < 0 || step < 1 || nranks < 1 || nranks > LDEQ_MAX_PEERS || rank < 0 ||
        rank >= nranks)
        return set_err(h, LDEQ_ERR_INVALID, "allreduce_adamw: bad argument (1 <= nranks <= 16)");
    if (n & 3) return set_err(h, LDEQ_ERR_INVALID, "allreduce_adamw: n must be a multiple of 4 (pad the flat buffers)");
    uintptr_t al = ((uintptr_t)params) | ((uintptr_t)m) | ((uintptr_t)v);
    PeerBufs pb;
    pb.n = nranks;
    for (int r = 0; r < LDEQ_MAX_PEERS; ++r) {
        pb.g[r] = r < nranks ? peer_grads_host[r] : nullptr;
        pb.x[r] = (r < nranks && peer_params_host) ? peer_params_host[r] : nullptr;
    }
    for (int r = 0; r < nranks; ++r) {
        if (!pb.g[r] || (peer_params_host && !pb.x[r])) return set_err(h, LDEQ_ERR_INVALID, "allreduce_adamw: null peer pointer");
        al |= (uintptr_t)pb.g[r] | (uintptr_t)pb.x[r];
    }
    if (al & 15) return set_err(h, LDEQ_ERR_INVALID, "allreduce_adamw: buffers must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    if (int rc = refuse_capture(h, s, "ldeq_allreduce_adamw_step", "multi-GPU capture is not supported")) return rc;
    if (n == 0) return LDEQ_OK;
    LDEQ_CUDA(cudaSetDevice(h->device));
    double p1 = 1.0, p2 = 1.0;
    for (int64_t i = 0; i < step; ++i) { p1 *= beta1; p2 *= beta2; }
    const size_t n4 = (size_t)n >> 2;
    size_t lo4 = 0, hi4 = n4;
    if (peer_params_host) {  // contiguous slice of this rank (remainder to the first ranks)
        const size_t base = n4 / nranks, rem = n4 % nranks;
        lo4 = rank * base + ((size_t)rank < rem ? rank : rem);
        hi4 = lo4 + base + ((size_t)rank < rem ? 1 : 0);
    }
    const size_t want = (hi4 - lo4 + 255) / 256;
    const int grid = (int)(want < (size_t)h->sm_count * 4 ? (want ? want : 1) : (size_t)h->sm_count * 4);
    if (peer_params_host)
        allreduce_adamw_kernel<true><<<grid, 256, 0, s>>>(params, pb, m, v, lo4, hi4, beta1, beta2, 1.0 - p1, 1.0 - p2, eps, lr, decay, grad_scale);
    else
        allreduce_adamw_kernel<false><<<grid, 256, 0, s>>>(params, pb, m, v, lo4, hi4, beta1, beta2, 1.0 - p1, 1.0 - p2, eps, lr, decay, grad_scale);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    return LDEQ_OK;
}

int ldeq_sample(ldeq_handle* h, const float* mu, const float* logvar, float* z_out, float* eps_out, int64_t n,
                uint64_t seed, uint64_t offset, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!mu || !logvar || !z_out || n < 0) return set_err(h, LDEQ_ERR_INVALID, "sample: bad argument");
    if (n == 0) return LDEQ_OK;
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    size_t want = ((((size_t)n + 3) >> 2) + 255) / 256;
    int grid = (int)(want < (size_t)h->sm_count * 8 ? want : (size_t)h->sm_count * 8);
    sample_kernel<false><<<grid, 256, 0, s>>>(mu, logvar, z_out, eps_out, (size_t)n, seed, offset, nullptr);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    return LDEQ_OK;
}

int ldeq_sample_dev(ldeq_handle* h, const float* mu, const float* logvar, float* z_out, float* eps_out, int64_t n,
                    uint64_t seed, uint64_t* calls, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!mu || !logvar || !z_out || !calls || n < 0) return set_err(h, LDEQ_ERR_INVALID, "sample: bad argument");
    if ((uintptr_t)calls & 7) return set_err(h, LDEQ_ERR_INVALID, "sample: calls must be 8-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    sample_advance_kernel<<<1, 1, 0, s>>>(calls);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    if (n == 0) return LDEQ_OK;
    size_t want = ((((size_t)n + 3) >> 2) + 255) / 256;
    int grid = (int)(want < (size_t)h->sm_count * 8 ? want : (size_t)h->sm_count * 8);
    sample_kernel<true><<<grid, 256, 0, s>>>(mu, logvar, z_out, eps_out, (size_t)n, seed, 0, calls);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 1;
    return LDEQ_OK;
}

}  // extern "C"
