// ldeq_mlp_res.cu -- LatentODE exact path with the Float32 weights RESIDENT in shared memory.
//
// Same arithmetic and the same entry points as ldeq_mlp.cu (drop-in for diffeq_layer(::Decoder{LatentODE}, z0, t),
// reference src/models/LatentODE.jl:61-78, and for its reverse pass), for networks whose padded weight image fits one
// SM's shared memory next to the tile state (the reference's 16-200-200-16 dudt, examples/pendulum_friction-less/
// nODE.jl:14-16, takes 189 kB of the 227 kB).  The general kernels read the 187 kB of weights through L1/L2 for every
// right-hand side of every tile and are bound by that latency (1 % of the FP32 peak at B = 256); here a CTA stages the
// weights once and every dense layer is a shared-memory matrix-vector product:
//   forward   mlp_fwd_kernel<float, TB, GLOBAL, RES = true, 512 threads> (ldeq_mlp_common.cuh);
//   backward  mlp_bwd_res_kernel below: discrete adjoint of the taped steps, restructured so that one step costs
//             6 forward passes + 6 VJPs (instead of 13 + 7):
//             * the hidden activations of the recomputed stages are kept (7 slots) and reused by the VJPs;
//             * k7 of step n and k1 of step n+1 are the same function evaluation (FSAL), so their cotangents are added
//               and pulled back once;
//             * the gradient of the large interior layer is a rank-(6 TB) update applied once per step from the kept
//               activations (x) and pre-activation cotangents (stored over the slot's own output), instead of a
//               read-modify-write of all 40 000 accumulators per stage; the small first/last layers update per stage.
#include "ldeq_mlp_common.cuh"

namespace ldeq {

// gW[k*N + n] += sum_b dy[n][b] x[k][b];  gb[n] += sum_b dy[n][b]   (small layers: per stage)
template <int TB, int NT>
__device__ void grad_immediate(float* __restrict__ gW, float* __restrict__ gb, const float* dy, const float* x, int K, int N,
                               int SL, bool sync) {
    const int kper = (K + SL - 1) / SL;
    const int w = threadIdx.x;
    if (w < N * SL) {
        const int s = w / N, n = w - s * N;
        const int k0 = s * kper, k1 = min(K, k0 + kper);
        float d[TB];
#pragma unroll
        for (int b = 0; b < TB; ++b) d[b] = dy[n * TB + b];
#pragma unroll 8
        for (int k = k0; k < k1; ++k) {
            float a = 0.f;
#pragma unroll
            for (int b = 0; b < TB; ++b) a = fmaf(d[b], x[k * TB + b], a);
            atomicAdd(gW + (size_t)k * N + n, a);  // RED: no round trip (the slice is private to the CTA, one add per address per pass)
        }
        if (s == 0) {
            float a = 0.f;
#pragma unroll
            for (int b = 0; b < TB; ++b) a += d[b];
            atomicAdd(gb + n, a);
        }
    }
    if (sync) __syncthreads();
}

// rank-(NSLOT*TB) update of the batched layer from the activation slots [slot_lo, 7):
// x = slot's output of layer lb-1, dy = slot's (overwritten) output of layer lb
template <int TB, int NT>
__device__ void grad_batched(float* __restrict__ gW, float* __restrict__ gb, const float* acts, int slot_stride, int x_off,
                             int dy_off, int slot_lo, int K, int N, int SL) {
    const int kper = (K + SL - 1) / SL;
    for (int w = threadIdx.x; w < N * SL; w += NT) {
        const int s = w / N, n = w - s * N;
        const int k0 = s * kper, k1 = min(K, k0 + kper);
        float d[7][TB];
#pragma unroll
        for (int j = 0; j < 7; ++j)
#pragma unroll
            for (int b = 0; b < TB; ++b) d[j][b] = j >= slot_lo ? acts[j * slot_stride + dy_off + n * TB + b] : 0.f;
        if (slot_lo <= 1) {
#pragma unroll 8
            for (int k = k0; k < k1; ++k) {
                float a = 0.f;
#pragma unroll
                for (int j = 1; j < 7; ++j)
#pragma unroll
                    for (int b = 0; b < TB; ++b) a = fmaf(d[j][b], acts[j * slot_stride + x_off + k * TB + b], a);
                atomicAdd(gW + (size_t)k * N + n, a);  // RED: no round trip (the slice is private to the CTA, one add per address per pass)
            }
        } else {
            // only the merged stage (slot 6) carries a cotangent in this iteration
#pragma unroll 4
            for (int k = k0; k < k1; ++k) {
                float a = 0.f;
#pragma unroll
                for (int b = 0; b < TB; ++b) a = fmaf(d[6][b], acts[6 * slot_stride + x_off + k * TB + b], a);
                atomicAdd(gW + (size_t)k * N + n, a);  // RED: no round trip (the slice is private to the CTA, one add per address per pass)
            }
        }
        if (s == 0) {
            float a = 0.f;
#pragma unroll
            for (int j = 1; j < 7; ++j)
#pragma unroll
                for (int b = 0; b < TB; ++b) a += d[j][b];
            atomicAdd(gb + n, a);
        }
    }
    __syncthreads();
}

// Pull kbar (D x TB) back through the MLP linearised at the activations kept in `slot`; x is the stage input.
// Parameter gradients of every layer but net.lb are accumulated here; layer lb's cotangent is left in the slot.
template <int TB, int NT>
__device__ void mlp_vjp_res(const MlpNet& net, const float* img, float* __restrict__ gP, const float* x, const float* kbar,
                            float* gbar, float* slot, float* dbuf0, float* dbuf1) {
    const float* dy = kbar;
    for (int l = net.n_layers - 1; l >= 0; --l) {
        const int K = net.dims[l], N = net.dims[l + 1];
        const float* xin = l == 0 ? x : slot + net.act_off[l - 1] * TB;
        // the update only reads dy / xin and writes global memory: it needs a barrier before the dense layer below only
        // when that layer overwrites xin in place
        if (l != net.lb)
            grad_immediate<TB, NT>(gP + net.w_off[l], gP + net.b_off[l], dy, xin, K, N, net.g_sl[l], l >= 1 && l - 1 == net.lb);
        float* dx;
        const float* mask = nullptr;
        if (l == 0) {
            dx = gbar;
        } else {
            float* a_prev = slot + net.act_off[l - 1] * TB;  // output of layer l-1 = input of layer l
            mask = a_prev;
            dx = (l - 1 == net.lb) ? a_prev : ((l & 1) ? dbuf1 : dbuf0);
        }
        dense_res<TB>(net, img, l, 1, dy, dx, false, mask);
        dy = dx;
    }
}

template <int TB>
__global__ void __launch_bounds__(RES_THREADS)
mlp_bwd_res_kernel(MlpNet net, const float* __restrict__ P, const double* tg, int B, int T,
                   const float* __restrict__ dtraj, MlpTapeView<float> tape, const int* __restrict__ retcode,
                   const int* __restrict__ naccept, float* __restrict__ dz0, float* __restrict__ gscratch) {
    constexpr int NT = RES_THREADS;
    using S = float;
    const int D = net.dims[0];
    const int HW = net.max_width;
    const int DT = D * TB;
    const int ACT = net.act_rows * TB;  // one activation slot
    extern __shared__ __align__(16) unsigned char smem_raw[];
    S* Wimg = reinterpret_cast<S*>(smem_raw);
    S* Gst = Wimg + net.n_img;   // [7][DT] stage inputs (Gst[0] = u_n, Gst[6] = u_{n+1})
    S* Kst = Gst + 7 * DT;       // [6][DT] k1..k6
    S* Kbar = Kst + 6 * DT;      // [7][DT]
    S* K1c = Kbar + 7 * DT;      // cotangent of k1 of the step processed before (= k7 of this one)
    S* XM = K1c + DT;            // input of the merged stage, u_{n+1}
    S* UB = XM + DT;             // adjoint of u_n
    S* UBN = UB + DT;            // adjoint of u_{n+1}
    S* GB = UBN + DT;            // stage-input adjoint
    S* ytmp = GB + DT;
    S* acts = ytmp + DT;         // [7][ACT]: slots 0..5 = stages 1..6 of this step, slot 6 = the merged stage
    S* dbuf0 = acts + 7 * ACT;
    S* dbuf1 = dbuf0 + HW * TB;
    const size_t s_bytes = (((size_t)net.n_img + (size_t)26 * DT + 7 * (size_t)ACT + (size_t)(2 * HW) * TB) * sizeof(S) + 15) & ~(size_t)15;
    double* tn_s = reinterpret_cast<double*>(smem_raw + s_bytes);  // [TB]
    double* dtn_s = tn_s + TB;
    double* tnext_s = dtn_s + TB;
    int* n_s = reinterpret_cast<int*>(tnext_s + TB);  // [TB] step index; -1: pull back k1 of step 0 and finish; -2: done
    int* ks_s = n_s + TB;
    int* flag_s = ks_s + TB;
    __shared__ int s_any, s_live;
    __shared__ double tg_s[RES_TGRID_MAX];
    if (T <= RES_TGRID_MAX) {
        for (int i = threadIdx.x; i < T; i += NT) tg_s[i] = tg[i];
        tg = tg_s;  // every save-time lookup below is a shared-memory read
    }

    stage_weight_image<NT>(net, P, Wimg);
    float* gP = gscratch + (size_t)blockIdx.x * net.n_params;  // this CTA's private gradient accumulator (L2 resident)
    for (int i = threadIdx.x; i < net.n_params; i += NT) gP[i] = 0.f;
    const int lb = net.lb;
    const int ntiles = (B + TB - 1) / TB;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b0 = tile * TB;
        if (threadIdx.x < TB) {
            const int b = threadIdx.x;
            const bool ok = b0 + b < B && retcode[b0 + b] == RET_SUCCESS && naccept[b0 + b] <= tape.cap;
            n_s[b] = ok ? naccept[b0 + b] - 1 : -2;
            ks_s[b] = T - 1;
            tnext_s[b] = tg[T - 1];
        }
        for (int i = threadIdx.x; i < DT; i += NT) { UBN[i] = 0.f; K1c[i] = 0.f; XM[i] = 0.f; }
        bool first = true;
        __syncthreads();
        for (;;) {
            if (threadIdx.x == 0) { s_any = 0; s_live = 0; }
            __syncthreads();
            if (threadIdx.x < TB) {
                if (n_s[threadIdx.x] >= -1) s_live = 1;
                if (n_s[threadIdx.x] >= 0) s_any = 1;
            }
            __syncthreads();
            if (!s_live) break;
            const bool any_active = s_any != 0;  // uniform over the CTA
            // ---- step records, stage recomputation (activations kept) ----------------------------------------
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                if (n_s[b] >= 0) {
                    tn_s[b] = tape.t[(size_t)n_s[b] * B + b0 + b];
                    dtn_s[b] = tape.dt[(size_t)n_s[b] * B + b0 + b];
                } else {
                    tn_s[b] = 0.0; dtn_s[b] = 0.0;
                }
            }
            for (int i = threadIdx.x; i < DT; i += NT) {
                const int d = i / TB, b = i - d * TB;
                Gst[i] = n_s[b] >= 0 ? tape.u[((size_t)n_s[b] * B + b0 + b) * D + d] : 0.f;
            }
            for (int i = threadIdx.x; i < 7 * DT; i += NT) Kbar[i] = 0.f;
            for (int i = threadIdx.x; i < DT; i += NT) UB[i] = 0.f;
            __syncthreads();
            if (any_active || first) {
                for (int j = 0; j < 6; ++j) {
                    mlp_fwd_res<TB>(net, Wimg, Gst + j * DT, Kst + j * DT, dbuf0, dbuf1, acts + j * ACT);
                    for (int i = threadIdx.x; i < DT; i += NT) {
                        S acc = tab_a<S>(j + 1, 0) * Kst[i];
                        for (int q = 1; q <= j; ++q) acc = fmaf(tab_a<S>(j + 1, q), Kst[q * DT + i], acc);
                        Gst[(j + 1) * DT + i] = fmaf((S)dtn_s[i % TB], acc, Gst[i]);
                    }
                    __syncthreads();
                }
                if (first) {
                    // the last step of every trajectory: activations at u_end are not carried from a later step
                    mlp_fwd_res<TB>(net, Wimg, Gst + 6 * DT, ytmp, dbuf0, dbuf1, acts + 6 * ACT);
                    for (int i = threadIdx.x; i < DT; i += NT) XM[i] = Gst[6 * DT + i];
                    __syncthreads();
                }
            }
            // ---- cotangents of the save points in (t_n, t_{n+1}] -----------------------------------------------
            for (;;) {
                if (threadIdx.x == 0) s_any = 0;
                __syncthreads();
                if (threadIdx.x < TB) {
                    const int b = threadIdx.x;
                    const int pend = n_s[b] >= 0 && ks_s[b] >= 1 && tg[ks_s[b]] > tn_s[b];
                    flag_s[b] = pend;
                    if (pend) s_any = 1;
                }
                __syncthreads();
                if (!s_any) break;
                for (int i = threadIdx.x; i < DT; i += NT) {
                    const int d = i / TB, b = i - d * TB;
                    if (flag_s[b]) {
                        const int ks = ks_s[b];
                        const double tsv = tg[ks];
                        const S dv = dtraj[((size_t)ks * B + b0 + b) * D + d];
                        if (tsv == tnext_s[b]) {
                            UBN[i] += dv;
                        } else {
                            S bw[7];
                            interp_weights<S>((S)((tsv - tn_s[b]) / dtn_s[b]), bw);
                            const S hd = (S)dtn_s[b] * dv;
#pragma unroll
                            for (int q = 0; q < 7; ++q) Kbar[q * DT + i] = fmaf(bw[q], hd, Kbar[q * DT + i]);
                            UB[i] += dv;
                        }
                    }
                }
                __syncthreads();
                if (threadIdx.x < TB && flag_s[threadIdx.x]) ks_s[threadIdx.x]--;
            }
            // ---- merged stage: k7 of this step and k1 of the step after it share f(u_{n+1}) -------------------
            for (int i = threadIdx.x; i < DT; i += NT) Kbar[6 * DT + i] += K1c[i];
            __syncthreads();
            mlp_vjp_res<TB, NT>(net, Wimg, gP, XM, Kbar + 6 * DT, GB, acts + 6 * ACT, dbuf0, dbuf1);
            for (int i = threadIdx.x; i < DT; i += NT) {
                const int d = i / TB, b = i - d * TB;
                const S v = UBN[i] + GB[i];
                UBN[i] = v;
                if (n_s[b] == -1) {
                    // save point 0 is u0 itself
                    dz0[(size_t)(b0 + b) * D + d] = v + dtraj[(size_t)(b0 + b) * D + d];
                } else if (n_s[b] >= 0) {
                    UB[i] += v;
                    const S hv = (S)dtn_s[b] * v;
                    for (int q = 0; q < 6; ++q) Kbar[q * DT + i] = fmaf(tab_a<S>(6, q), hv, Kbar[q * DT + i]);
                }
            }
            __syncthreads();
            if (any_active) {
                for (int j = 5; j >= 1; --j) {
                    mlp_vjp_res<TB, NT>(net, Wimg, gP, Gst + j * DT, Kbar + j * DT, GB, acts + j * ACT, dbuf0, dbuf1);
                    for (int i = threadIdx.x; i < DT; i += NT) {
                        const S v = GB[i];
                        UB[i] += v;
                        const S hv = (S)dtn_s[i % TB] * v;
                        for (int q = 0; q < j; ++q) Kbar[q * DT + i] = fmaf(tab_a<S>(j, q), hv, Kbar[q * DT + i]);
                    }
                    __syncthreads();
                }
            }
            // layer lb: one rank-(6 TB) update for the whole step
            if (lb >= 0)
                grad_batched<TB, NT>(gP + net.w_off[lb], gP + net.b_off[lb], acts, ACT, net.act_off[lb - 1] * TB,
                                     net.act_off[lb] * TB, any_active ? 1 : 6, net.dims[lb], net.dims[lb + 1], net.g_sl[lb]);
            // stage 1 is deferred: its cotangent and its activations (slot 0) travel to the next iteration
            for (int i = threadIdx.x; i < DT; i += NT) {
                const int b = i % TB;
                const bool act = n_s[b] >= 0;
                K1c[i] = act ? Kbar[i] : 0.f;
                if (act) { UBN[i] = UB[i]; XM[i] = Gst[i]; }
            }
            if (any_active)
                for (int i = threadIdx.x; i < ACT; i += NT) acts[6 * ACT + i] = acts[i];
            __syncthreads();
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                if (n_s[b] >= 0) { tnext_s[b] = tn_s[b]; n_s[b]--; }
                else if (n_s[b] == -1) n_s[b] = -2;
            }
            first = false;
            __syncthreads();
        }
        // failed trajectories get a zero gradient (their NaN block is a constant), tape overflow NaN
        for (int i = threadIdx.x; i < DT; i += NT) {
            const int d = i / TB, b = i - d * TB;
            if (b0 + b < B) {
                const bool ok = retcode[b0 + b] == RET_SUCCESS;
                const bool over = ok && naccept[b0 + b] > tape.cap;
                if (!ok || over) dz0[(size_t)(b0 + b) * D + d] = over ? s_nan<S>() : 0.f;
            }
        }
        __syncthreads();
    }
}

template <int TB> static size_t bwd_res_smem(const MlpNet& net) {
    const size_t D = net.dims[0], HW = net.max_width, DT = D * TB, ACT = (size_t)net.act_rows * TB;
    size_t n = ((size_t)net.n_img + 26 * DT + 7 * ACT + (2 * HW) * TB) * sizeof(float);
    n = (n + 15) & ~(size_t)15;
    return n + 3 * TB * sizeof(double) + 3 * TB * sizeof(int) + 64;
}

template <class S> __global__ void mlp_res_reduce_grads_kernel(const S* __restrict__ gscratch, int n_cta, int n_params,
                                                               S* __restrict__ dparams) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_params; i += gridDim.x * blockDim.x) {
        double a = 0.0;
        for (int c = 0; c < n_cta; ++c) a += (double)gscratch[(size_t)c * n_params + i];
        dparams[i] = (S)a;
    }
}

static constexpr size_t kSmemMax = 227 * 1024 - RES_TGRID_MAX * sizeof(double) - 64;  // dynamic part

template <int TB, bool GLOBAL, int NT>
static int launch_res_fwd(ldeq_handle* h, const MlpNet& net, const float* P, const float* z0, const double* tg, int B, int T,
                          const KOpts& ko, float* traj, int32_t* ret, int32_t* na, int32_t* nr, MlpTapeView<float> tv,
                          double* partials, int grid, cudaStream_t s) {
    const size_t smem = fwd_smem<float, TB, true, NT>(net);
    auto kern = mlp_fwd_kernel<float, TB, GLOBAL, true, NT>;
    LDEQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MlpNet netv = net;
    res_plan(netv, NT);
    KOpts kov = ko;
    void* args[] = {&netv, &P, &z0, &tg, &B, &T, &kov, &traj, &ret, &na, &nr, &tv, &partials};
    if (GLOBAL) {
        LDEQ_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(NT), args, smem, s));
    } else {
        LDEQ_CUDA(cudaLaunchKernel((void*)kern, dim3(grid), dim3(NT), args, smem, s));
    }
    h->launches += 1;
    return LDEQ_OK;
}

}  // namespace ldeq

using namespace ldeq;

int ldeq_mlp_res_forward(ldeq_handle* h, const MlpNet& net, const float* P, const float* z0, const double* tg, int B, int T,
                         const KOpts& ko, int norm_mode, float* traj, int32_t* ret, int32_t* na, int32_t* nr,
                         MlpTapeView<float> tv, double* partials, cudaStream_t s) {
    const int sms = h->sm_count;
    const bool global = norm_mode == LDEQ_NORM_GLOBAL && ko.adaptive;
    // smallest tile that gives every SM at most one tile (one CTA per SM: the image takes most of its shared memory).
    // A resident CTA is bound by the latency of its own dependent chain, so batches that need several rounds of tiles
    // are better served by the general kernels, which keep 2-4 CTAs per SM in flight.
    auto ok = [&](int tb, size_t smem) { return res_layout_ok(net, tb) && smem <= kSmemMax; };
    const bool ok2 = ok(2, fwd_smem<float, 2, true, RES_THREADS>(net));
    const bool ok4 = ok(4, fwd_smem<float, 4, true, RES_THREADS>(net));
    const bool ok8 = ok(8, fwd_smem<float, 8, true, RES_THREADS>(net));
    int tb = 0;
    if (ok2 && (B + 1) / 2 <= sms) tb = 2;
    else if (ok4 && (B + 3) / 4 <= sms) tb = 4;
    else if (ok8 && (B + 7) / 8 <= sms) tb = 8;
    if (!tb) return LDEQ_ERR_UNSUPPORTED;
    const int tiles = (B + tb - 1) / tb;
    const int grid = tiles < sms ? tiles : sms;
#define LDEQ_RES_FWD(TBV, NTV)                                                                                              \
    return global ? launch_res_fwd<TBV, true, NTV>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, grid, s) \
                  : launch_res_fwd<TBV, false, NTV>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, grid, s)
    if (tb == 2) { LDEQ_RES_FWD(2, RES_THREADS); }
    if (tb == 4) { LDEQ_RES_FWD(4, RES_THREADS); }
    LDEQ_RES_FWD(8, RES_THREADS);
#undef LDEQ_RES_FWD
}

int ldeq_mlp_res_backward(ldeq_handle* h, const MlpNet& net, const float* P, const double* tg, int B, int T, const float* dtraj,
                          MlpTapeView<float> tv, const int32_t* ret, const int32_t* na, float* dz0, float* dparams,
                          cudaStream_t s) {
    constexpr int TB = 2;
    const size_t smem = bwd_res_smem<TB>(net);
    if (!res_layout_ok(net, TB) || smem > kSmemMax) return LDEQ_ERR_UNSUPPORTED;
    const int tiles = (B + TB - 1) / TB;
    if (tiles > 4 * h->sm_count) return LDEQ_ERR_UNSUPPORTED;  // many rounds of tiles: the general kernel's 2 CTAs per SM win
    const int grid = tiles < h->sm_count ? tiles : h->sm_count;
    int rc = ensure_scratch(h, 1, (size_t)grid * net.n_params * sizeof(float), s);
    if (rc) return rc;
    LDEQ_CUDA(cudaFuncSetAttribute(mlp_bwd_res_kernel<TB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MlpNet netv = net;
    res_plan(netv, RES_THREADS);
    mlp_bwd_res_kernel<TB><<<grid, RES_THREADS, smem, s>>>(netv, P, tg, B, T, dtraj, tv, ret, na, dz0, (float*)h->scratch[1]);
    LDEQ_CUDA(cudaGetLastError());
    mlp_res_reduce_grads_kernel<float><<<(net.n_params + 255) / 256, 256, 0, s>>>((const float*)h->scratch[1], grid, net.n_params, dparams);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 2;
    return LDEQ_OK;
}
