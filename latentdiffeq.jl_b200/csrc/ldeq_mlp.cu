// ldeq_mlp.cu -- LatentODE hot path: Tsit5 on the (D,B) matrix state with an MLP right-hand side.
//
// Drop-in for the body of diffeq_layer(::Decoder{LatentODE}, z0, t) (reference src/models/LatentODE.jl:61-78):
//   nODE = NeuralODE(dudt, (t[1], t[end]), Tsit5(); saveat = t, kwargs...);  z = Array(nODE(z0))
// with dudt = Chain(Dense(D,H,relu), Dense(H,H,relu), Dense(H,D)) (examples/pendulum_friction-less/nODE.jl:14-16)
// and parameters in Flux.destructure order (per layer vec(W) column-major with W (out,in), then b).
//
// This file holds the exact-arithmetic path (CUDA cores, fp32 or fp64): one persistent CTA integrates a
// tile of TB trajectories for the whole time span.  Stage vectors, hidden activations and the
// per-trajectory controller state live in shared memory; the weights are read through L1 (187 kB for the
// default 16-200-200-16 network).  Two error-norm scopes:
//   LDEQ_NORM_GLOBAL    one dt for the whole batch, RMS over all D*B entries (reference semantics); the CTAs
//                       meet at a cooperative grid barrier once per attempted step to sum the error norm;
//   LDEQ_NORM_PER_TRAJ  every trajectory has its own dt / accept-reject sequence (documented deviation).
// The backward kernel is the discrete adjoint of the accepted steps (the reference's InterpolatingAdjoint is a
// continuous adjoint that agrees with it to the solver tolerance, SURVEY.md A.7).
#include <cstdio>
#include <cstdlib>

#include "ldeq_mlp_common.cuh"

namespace ldeq {


// ---- backward -----------------------------------------------------------------------------------------
// y = relu?(W x + b) on a tile, keeping the output; used to recompute hidden activations.
// Input gradient: dx[k][b] = sum_n Wt[n*K + k] dy[n][b]  (Wt = W transposed once per call: coalesced over k)
template <class S, int TB>
__device__ void dense_bwd_input(const S* __restrict__ Wt, const S* __restrict__ dy, S* __restrict__ dx, S* __restrict__ red,
                                int K, int N) {
    // same mapping as dense_fwd with the roles of K and N swapped
    int SL = 1;
    while (SL * 2 * K <= MLP_THREADS && SL < 16 && SL * 2 <= N) SL *= 2;
    const int nper = (N + SL - 1) / SL;
    for (int w = threadIdx.x; w < K * SL; w += MLP_THREADS) {
        const int s = w / K, k = w - s * K;
        const int n0 = s * nper, n1 = min(N, n0 + nper);
        S acc[TB];
#pragma unroll
        for (int b = 0; b < TB; ++b) acc[b] = (S)0;
#pragma unroll 8
        for (int n = n0; n < n1; ++n) {
            const S wv = Wt[(size_t)n * K + k];
#pragma unroll
            for (int b = 0; b < TB; ++b) acc[b] = s_fma<S>(wv, dy[n * TB + b], acc[b]);
        }
        if (SL == 1) {
#pragma unroll
            for (int b = 0; b < TB; ++b) dx[k * TB + b] = acc[b];
        } else {
#pragma unroll
            for (int b = 0; b < TB; ++b) red[(s * K + k) * TB + b] = acc[b];
        }
    }
    if (SL > 1) {
        __syncthreads();
        for (int i = threadIdx.x; i < K * TB; i += MLP_THREADS) {
            S a = (S)0;
            for (int s = 0; s < SL; ++s) a += red[s * K * TB + i];
            dx[i] = a;
        }
    }
    __syncthreads();
}

// Parameter gradient of one layer accumulated into this CTA's private slice of the scratch buffer:
// gW[k*N + n] += sum_b dy[n][b] x[k][b];  gb[n] += sum_b dy[n][b]
// RED: the accumulator is global memory -> reduction atomics (no read round trip; the slice is private to the CTA and
// every address gets one add per pass, so the result does not depend on timing)
template <class S, int TB, bool RED>
__device__ void dense_bwd_params(S* __restrict__ gW, S* __restrict__ gb, const S* __restrict__ dy, const S* __restrict__ x,
                                 int K, int N) {
    // thread = output neuron n x k-slice: dy[n][:] stays in registers, x[k][:] is a shared-memory broadcast, the
    // accumulator is updated with consecutive threads on consecutive addresses (no integer division in the loop)
    int SL = 1;
    while (SL * 2 * N <= MLP_THREADS && SL < 16 && SL * 2 <= K) SL *= 2;
    const int kper = (K + SL - 1) / SL;
    for (int w = threadIdx.x; w < N * SL; w += MLP_THREADS) {
        const int s = w / N, n = w - s * N;
        const int k0 = s * kper, k1 = min(K, k0 + kper);
        S d[TB];
#pragma unroll
        for (int b = 0; b < TB; ++b) d[b] = dy[n * TB + b];
#pragma unroll 8
        for (int k = k0; k < k1; ++k) {
            S a = (S)0;
#pragma unroll
            for (int b = 0; b < TB; ++b) a = s_fma<S>(d[b], x[k * TB + b], a);
            if (RED) atomicAdd(gW + (size_t)k * N + n, a); else gW[(size_t)k * N + n] += a;
        }
        if (s == 0) {
            S a = (S)0;
#pragma unroll
            for (int b = 0; b < TB; ++b) a += d[b];
            if (RED) atomicAdd(gb + n, a); else gb[n] += a;
        }
    }
    __syncthreads();
}

// VJP of the MLP at stage input x: recompute the hidden activations (kept in `acts`), then sweep back.
// kbar (D x TB) in, gbar (D x TB) out (overwritten), parameter gradients accumulated into gP.
template <class S, int TB, bool RED>
__device__ void mlp_vjp(const MlpNet& net, const S* __restrict__ P, const S* __restrict__ Pt, S* __restrict__ gP, const S* x,
                        const S* kbar, S* gbar, S* acts /*[n_layers-1][HW*TB]*/, S* dbuf0, S* dbuf1, S* ytmp, S* red,
                        int HW) {
    // forward, keeping every hidden activation
    const S* in = x;
    for (int l = 0; l < net.n_layers; ++l) {
        const bool last = l + 1 == net.n_layers;
        S* out = last ? ytmp : acts + (size_t)l * HW * TB;
        dense_fwd<S, TB>(P + net.w_off[l], P + net.b_off[l], in, out, red, net.dims[l], net.dims[l + 1], !last);
        in = out;
    }
    // backward
    const S* dy = kbar;
    for (int l = net.n_layers - 1; l >= 0; --l) {
        const int K = net.dims[l], N = net.dims[l + 1];
        const S* xin = l == 0 ? x : acts + (size_t)(l - 1) * HW * TB;
        dense_bwd_params<S, TB, RED>(gP + net.w_off[l], gP + net.b_off[l], dy, xin, K, N);
        S* dx = l == 0 ? gbar : ((l & 1) ? dbuf1 : dbuf0);
        dense_bwd_input<S, TB>(Pt + net.w_off[l], dy, dx, red, K, N);
        if (l > 0) {
            // through the relu of layer l-1: its output is xin
            for (int i = threadIdx.x; i < K * TB; i += MLP_THREADS) dx[i] = xin[i] > (S)0 ? dx[i] : (S)0;
            __syncthreads();
        }
        dy = dx;
    }
}

// SMEM_GRAD: the CTA's private parameter-gradient accumulator lives in shared memory (187 kB for 16-200-200-16 in fp32)
// instead of its slice of the global scratch: the accumulation is a read-modify-write of every parameter per stage.
template <class S, int TB, bool SMEM_GRAD>
__global__ void __launch_bounds__(MLP_THREADS)
mlp_bwd_kernel(MlpNet net, const S* __restrict__ P, const S* __restrict__ Pt, const double* __restrict__ tg, int B, int T,
               const S* __restrict__ dtraj, MlpTapeView<S> tape, const int* __restrict__ retcode,
               const int* __restrict__ naccept, S* __restrict__ dz0, S* __restrict__ gscratch) {
    const int D = net.dims[0];
    const int HW = net.max_width;
    const int DT = D * TB;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    S* Gst = reinterpret_cast<S*>(smem_raw);   // [7][D][TB] stage inputs (Gst[0] = u_n, Gst[6] = u_{n+1})
    S* Kst = Gst + 7 * DT;                      // [7][D][TB]
    S* Kbar = Kst + 7 * DT;                     // [7][D][TB]
    S* UB = Kbar + 7 * DT;                      // adjoint of u_n
    S* UBN = UB + DT;                           // adjoint of u_{n+1}
    S* GB = UBN + DT;                           // stage-input adjoint
    S* ytmp = GB + DT;
    S* acts = ytmp + DT;                        // [(L-1)][HW][TB]
    S* dbuf0 = acts + (size_t)(net.n_layers - 1) * HW * TB;
    S* dbuf1 = dbuf0 + HW * TB;
    S* red = dbuf1 + HW * TB;                   // [MLP_THREADS][TB]
    const size_t s_bytes =
        (((size_t)(25 * D + (net.n_layers - 1) * HW + 2 * HW + MLP_THREADS) * TB * sizeof(S)) + 15) & ~(size_t)15;
    double* tn_s = reinterpret_cast<double*>(smem_raw + s_bytes);  // [TB]
    double* dtn_s = tn_s + TB;
    double* tnext_s = dtn_s + TB;
    int* n_s = reinterpret_cast<int*>(tnext_s + TB);  // [TB] current step index (-1: done)
    int* ks_s = n_s + TB;
    int* flag_s = ks_s + TB;
    __shared__ int s_any;

    // this CTA's private gradient accumulator
    S* gP = SMEM_GRAD ? reinterpret_cast<S*>(smem_raw + ((s_bytes + 3 * TB * sizeof(double) + 3 * TB * sizeof(int) + 15) & ~(size_t)15))
                      : gscratch + (size_t)blockIdx.x * net.n_params;
    for (int i = threadIdx.x; i < net.n_params; i += MLP_THREADS) gP[i] = (S)0;
    const int ntiles = (B + TB - 1) / TB;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b0 = tile * TB;
        if (threadIdx.x < TB) {
            const int b = threadIdx.x;
            const bool ok = b0 + b < B && retcode[b0 + b] == RET_SUCCESS && naccept[b0 + b] <= tape.cap;
            n_s[b] = ok ? naccept[b0 + b] - 1 : -1;
            ks_s[b] = T - 1;
            tnext_s[b] = tg[T - 1];
        }
        for (int i = threadIdx.x; i < DT; i += MLP_THREADS) UBN[i] = (S)0;
        __syncthreads();
        for (;;) {
            if (threadIdx.x == 0) s_any = 0;
            __syncthreads();
            if (threadIdx.x < TB && n_s[threadIdx.x] >= 0) s_any = 1;
            __syncthreads();
            if (!s_any) break;
            // load the step record of every live trajectory and recompute its stages
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                if (n_s[b] >= 0) {
                    tn_s[b] = tape.t[(size_t)n_s[b] * B + b0 + b];
                    dtn_s[b] = tape.dt[(size_t)n_s[b] * B + b0 + b];
                } else {
                    tn_s[b] = 0.0; dtn_s[b] = 0.0;
                }
            }
            for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
                const int d = i / TB, b = i - d * TB;
                Gst[i] = n_s[b] >= 0 ? tape.u[((size_t)n_s[b] * B + b0 + b) * D + d] : (S)0;
            }
            for (int i = threadIdx.x; i < 7 * DT; i += MLP_THREADS) Kbar[i] = (S)0;
            for (int i = threadIdx.x; i < DT; i += MLP_THREADS) UB[i] = (S)0;
            __syncthreads();
            mlp_fwd<S, TB>(net, P, Gst, Kst, dbuf0, dbuf1, red);
            for (int j = 1; j < 7; ++j) {
                for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
                    S acc = tab_a<S>(j, 0) * Kst[i];
                    for (int q = 1; q < j; ++q) acc = s_fma<S>(tab_a<S>(j, q), Kst[q * DT + i], acc);
                    Gst[j * DT + i] = s_fma<S>((S)dtn_s[i % TB], acc, Gst[i]);
                }
                __syncthreads();
                mlp_fwd<S, TB>(net, P, Gst + j * DT, Kst + j * DT, dbuf0, dbuf1, red);
            }
            // cotangents of the save points in (t_n, t_{n+1}]
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
                for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
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
                            for (int q = 0; q < 7; ++q) Kbar[q * DT + i] = s_fma<S>(bw[q], hd, Kbar[q * DT + i]);
                            UB[i] += dv;
                        }
                    }
                }
                __syncthreads();
                if (threadIdx.x < TB && flag_s[threadIdx.x]) ks_s[threadIdx.x]--;
            }
            // k7 = f(u_{n+1}): UBN += J^T kbar7
            mlp_vjp<S, TB, !SMEM_GRAD>(net, P, Pt, gP, Gst + 6 * DT, Kbar + 6 * DT, GB, acts, dbuf0, dbuf1, ytmp, red, HW);
            for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
                const S v = UBN[i] + GB[i];
                UBN[i] = v;
                UB[i] += v;
                const S hv = (S)dtn_s[i % TB] * v;
                for (int q = 0; q < 6; ++q) Kbar[q * DT + i] = s_fma<S>(tab_a<S>(6, q), hv, Kbar[q * DT + i]);
            }
            __syncthreads();
            for (int j = 5; j >= 1; --j) {
                mlp_vjp<S, TB, !SMEM_GRAD>(net, P, Pt, gP, Gst + j * DT, Kbar + j * DT, GB, acts, dbuf0, dbuf1, ytmp, red, HW);
                for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
                    const S v = GB[i];
                    UB[i] += v;
                    const S hv = (S)dtn_s[i % TB] * v;
                    for (int q = 0; q < j; ++q) Kbar[q * DT + i] = s_fma<S>(tab_a<S>(j, q), hv, Kbar[q * DT + i]);
                }
                __syncthreads();
            }
            mlp_vjp<S, TB, !SMEM_GRAD>(net, P, Pt, gP, Gst, Kbar, GB, acts, dbuf0, dbuf1, ytmp, red, HW);
            for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
                const int b = i % TB;
                if (n_s[b] >= 0) UBN[i] = UB[i] + GB[i];  // adjoint of u_n becomes "u_{n+1}" of step n-1
            }
            __syncthreads();
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                if (n_s[b] >= 0) { tnext_s[b] = tn_s[b]; n_s[b]--; }
            }
            __syncthreads();
        }
        // save point 0 is u0 itself; failed trajectories get a zero gradient, tape overflow NaN
        for (int i = threadIdx.x; i < DT; i += MLP_THREADS) {
            const int d = i / TB, b = i - d * TB;
            if (b0 + b < B) {
                const bool ok = retcode[b0 + b] == RET_SUCCESS;
                const bool over = ok && naccept[b0 + b] > tape.cap;
                S v = ok ? UBN[i] + dtraj[(size_t)(b0 + b) * D + d] : (S)0;
                if (over) v = s_nan<S>();
                dz0[(size_t)(b0 + b) * D + d] = v;
            }
        }
        __syncthreads();
    }
    if (SMEM_GRAD) {
        S* out = gscratch + (size_t)blockIdx.x * net.n_params;
        for (int i = threadIdx.x; i < net.n_params; i += MLP_THREADS) out[i] = gP[i];
    }
}

// transpose every layer's W (N,K col-major: W[k*N+n]) into Wt[n*K + k]; biases are copied
template <class S> __global__ void mlp_transpose_kernel(MlpNet net, const S* __restrict__ P, S* __restrict__ Pt) {
    for (int l = 0; l < net.n_layers; ++l) {
        const int K = net.dims[l], N = net.dims[l + 1];
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < K * N; i += gridDim.x * blockDim.x) {
            const int n = i / K, k = i - n * K;
            Pt[net.w_off[l] + i] = P[net.w_off[l] + (size_t)k * N + n];
        }
    }
}

// dparams[i] = sum over CTAs of their private accumulators, in a fixed order (deterministic)
template <class S> __global__ void mlp_reduce_grads_kernel(const S* __restrict__ gscratch, int n_cta, int n_params,
                                                            S* __restrict__ dparams) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_params; i += gridDim.x * blockDim.x) {
        double a = 0.0;
        for (int c = 0; c < n_cta; ++c) a += (double)gscratch[(size_t)c * n_params + i];
        dparams[i] = (S)a;
    }
}

}  // namespace ldeq
#include "ldeq_mlp_cadj.cuh"
namespace ldeq {

template <class S, int TB> static size_t bwd_smem(const MlpNet& net) {
    const size_t D = net.dims[0], HW = net.max_width;
    size_t n = (21 * D + 4 * D + (net.n_layers - 1) * HW + 2 * HW + MLP_THREADS) * TB * sizeof(S);
    n = (n + 15) & ~(size_t)15;
    return n + 3 * TB * sizeof(double) + 3 * TB * sizeof(int) + 64;
}

}  // namespace ldeq

using namespace ldeq;

// ldeq_mlp_tc.cu: the tcgen05 / TMEM forward kernel (LDEQ_MLP_MATH_BF16X3)
int ldeq_mlp_tc_backward(ldeq_handle* h, const int32_t* dims, int n_layers, const float* params, const double* d_tgrid, int B, int T,
                         const float* dtraj, double* tape_t, double* tape_dt, float* tape_u, int tape_cap, const int32_t* ret,
                         const int32_t* na, int max_na, float* dz0, float* dparams, cudaStream_t s);
int ldeq_mlp_tc_forward(ldeq_handle* h, const int32_t* dims, int n_layers, const float* params, const float* z0,
                        const double* d_tgrid, int B, int T, const KOpts& ko, int norm_mode, float* traj, int32_t* ret,
                        int32_t* na, int32_t* nr, double* tape_t, double* tape_dt, float* tape_u, int tape_cap,
                        cudaStream_t s);

struct ldeq_mlp_tape {
    int dtype = 0, B = 0, T = 0, cap = 0, tb = 0;
    int math = 0;  // ldeq_mlp_math of the forward solve: its reverse pass runs on the same arithmetic
    int sense = 0, norm_mode = 0;  // ldeq_sensealg / ldeq_norm_mode of the forward solve
    ldeq::KOpts kopts;             // the solve's options: the continuous adjoint integrates with the same tolerances
    MlpNet net;
    void* base = nullptr;
    double* t = nullptr;
    double* dt = nullptr;
    void* u = nullptr;
    void* params = nullptr;  // copy of the flat parameters
    void* params_t = nullptr;
    double* tgrid = nullptr;
    int32_t* retcode = nullptr;
    int32_t* naccept = nullptr;
    int32_t* nreject = nullptr;
    int32_t* info = nullptr;     // device: largest accepted-step count of a successful trajectory
    int32_t* h_info = nullptr;   // pinned host mirror, valid once `ready` has completed
    cudaEvent_t ready = nullptr;
};

// largest naccept among the trajectories that succeeded: what the reverse pass will want to find on the tape
__global__ void mlp_max_naccept_kernel(const int32_t* __restrict__ na, const int32_t* __restrict__ ret, int B, int32_t* out) {
    int m = 0;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
        if (ret[b] == RET_SUCCESS && na[b] > m) m = na[b];
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

static int make_net(ldeq_handle* h, const int32_t* dims, int n_layers, MlpNet* net) {
    if (n_layers < 1 || n_layers > MLP_MAX_LAYERS) return set_err(h, LDEQ_ERR_UNSUPPORTED, "mlp: 1..8 layers supported");
    if (dims[0] != dims[n_layers]) return set_err(h, LDEQ_ERR_INVALID, "mlp: first and last layer width must be equal");
    net->n_layers = n_layers;
    int off = 0, mw = 0;
    for (int l = 0; l <= n_layers; ++l) {
        if (dims[l] < 1 || dims[l] > 1024) return set_err(h, LDEQ_ERR_UNSUPPORTED, "mlp: layer widths 1..1024 supported");
        net->dims[l] = dims[l];
        if (dims[l] > mw) mw = dims[l];
    }
    for (int l = 0; l < n_layers; ++l) {
        net->w_off[l] = off; off += dims[l] * dims[l + 1];
        net->b_off[l] = off; off += dims[l + 1];
    }
    net->n_params = off;
    net->max_width = mw;
    // padded shared-memory image (resident path), activation slot layout, the layer with the batched gradient pass
    int io = 0, ao = 0, lb = -1;
    for (int l = 0; l < n_layers; ++l) {
        net->i_ld[l] = dims[l + 1] | 1;
        net->i_w[l] = io; io += (dims[l] * net->i_ld[l] + 3) & ~3;
        net->i_b[l] = io; io += (dims[l + 1] + 3) & ~3;
        net->act_off[l] = ao;
        if (l + 1 < n_layers) ao += dims[l + 1];
        if (l >= 1 && l + 1 < n_layers && (lb < 0 || dims[l] * dims[l + 1] > dims[lb] * dims[lb + 1])) lb = l;
    }
    net->n_img = io;
    net->act_rows = ao;
    net->lb = lb;
    return LDEQ_OK;
}

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

template <class S, int TB, bool GLOBAL>
static int launch_mlp_fwd(ldeq_handle* h, const MlpNet& net, const void* P, const void* z0, const double* tg, int B, int T,
                          const KOpts& ko, void* traj, int32_t* ret, int32_t* na, int32_t* nr, MlpTapeView<S> tv,
                          double* partials, int grid, cudaStream_t s) {
    const size_t smem = fwd_smem<S, TB>(net);
    auto kern = mlp_fwd_kernel<S, TB, GLOBAL>;
    LDEQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MlpNet netv = net;
    const S* Pp = (const S*)P;
    const S* zp = (const S*)z0;
    S* tp = (S*)traj;
    KOpts kov = ko;
    void* args[] = {&netv, &Pp, &zp, &tg, &B, &T, &kov, &tp, &ret, &na, &nr, &tv, &partials};
    if (GLOBAL) {
        LDEQ_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(MLP_THREADS), args, smem, s));
    } else {
        LDEQ_CUDA(cudaLaunchKernel((void*)kern, dim3(grid), dim3(MLP_THREADS), args, smem, s));
    }
    h->launches += 1;
    return LDEQ_OK;
}

template <class S>
static int mlp_fwd_dispatch(ldeq_handle* h, const MlpNet& net, const void* P, const void* z0, const double* tg, int B, int T,
                            const KOpts& ko, int norm_mode, void* traj, int32_t* ret, int32_t* na, int32_t* nr,
                            ldeq_mlp_tape* tape, cudaStream_t s) {
    MlpTapeView<S> tv{nullptr, nullptr, nullptr, 0};
    if (tape) tv = MlpTapeView<S>{tape->t, tape->dt, (S*)tape->u, tape->cap};
    // reduction scratch for the grid sums
    int rc = ensure_scratch(h, 0, sizeof(double) * 4096, s);
    if (rc) return rc;
    double* partials = (double*)h->scratch[0];
    const int sms = h->sm_count;
    if constexpr (sizeof(S) == 4) {
        // Float32 networks that fit one SM's shared memory run on the resident-weights kernels (ldeq_mlp_res.cu)
        if (!getenv("LDEQ_MLP_NO_RESIDENT")) {
            rc = ldeq_mlp_res_forward(h, net, (const float*)P, (const float*)z0, tg, B, T, ko, norm_mode, (float*)traj, ret, na, nr,
                                      tv, partials, s);
            if (rc != LDEQ_ERR_UNSUPPORTED) return rc;
        }
    }
    if (norm_mode == LDEQ_NORM_GLOBAL && ko.adaptive) {   // fixed-step mode computes no error norm: no grid barrier
        // one tile per CTA, all CTAs co-resident (cooperative launch): pick the smallest tile that fits the chip
        auto fits = [&](int tb, size_t smem, const void* fn) -> int {
            int per_sm = 0;
            cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, MLP_THREADS, smem);
            return per_sm * sms >= (B + tb - 1) / tb;
        };
        if (fits(2, fwd_smem<S, 2>(net), (const void*)mlp_fwd_kernel<S, 2, true>))
            return launch_mlp_fwd<S, 2, true>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, (B + 1) / 2, s);
        if (fits(8, fwd_smem<S, 8>(net), (const void*)mlp_fwd_kernel<S, 8, true>))
            return launch_mlp_fwd<S, 8, true>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, (B + 7) / 8, s);
        if (fits(32, fwd_smem<S, 32>(net), (const void*)mlp_fwd_kernel<S, 32, true>))
            return launch_mlp_fwd<S, 32, true>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, (B + 31) / 32, s);
        return set_err(h, LDEQ_ERR_UNSUPPORTED,
                       "mlp: batch too large for the global-norm mode of the exact path (all tiles must be co-resident); "
                       "use LDEQ_NORM_PER_TRAJ");
    }
    if (B <= 2 * sms * 2) {
        const int tiles = (B + 1) / 2;
        return launch_mlp_fwd<S, 2, false>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, tiles, s);
    }
    const int tiles = (B + 7) / 8;
    const int grid = tiles < 4 * sms ? tiles : 4 * sms;
    return launch_mlp_fwd<S, 8, false>(h, net, P, z0, tg, B, T, ko, traj, ret, na, nr, tv, partials, grid, s);
}

extern "C" {

int ldeq_mlp_solve_fwd(ldeq_handle* h, int dtype, const void* z0, const void* params_flat, const int32_t* layer_dims_host,
                       int n_layers, const double* t_host, int B, int T, const ldeq_opts* opts, void* traj_out,
                       int32_t* retcode, int32_t* naccept, int32_t* nreject, ldeq_mlp_tape** tape_out,
                       ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (tape_out) *tape_out = nullptr;
    if (int rc0 = refuse_capture(h, (cudaStream_t)stream, "ldeq_mlp_solve_fwd", "its tape records the accepted-step count for a host-side check")) return rc0;
    if (!z0 || !params_flat || !layer_dims_host || !t_host || !opts || !traj_out) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    if (B < 1 || T < 1) return set_err(h, LDEQ_ERR_INVALID, "B and T must be >= 1");
    if (dtype != LDEQ_F32 && dtype != LDEQ_F64) return set_err(h, LDEQ_ERR_INVALID, "dtype");
    if (!opts->adaptive && !(opts->dt > 0.0)) return set_err(h, LDEQ_ERR_INVALID, "adaptive = 0 needs dt > 0");
    for (int k = 1; k < T; ++k)
        if (!(t_host[k] > t_host[k - 1])) return set_err(h, LDEQ_ERR_INVALID, "t must be strictly increasing");
    if (opts->solver != LDEQ_SOLVER_TSIT5)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "solver: the LatentODE kernels are Tsit5 (nODE.jl:17); DP5 / BS3 / RK4 exist for the GOKU entry points only");
    if (opts->mlp_math != LDEQ_MLP_MATH_FP32 && opts->mlp_math != LDEQ_MLP_MATH_BF16X3) return set_err(h, LDEQ_ERR_INVALID, "mlp_math");
    if (opts->mlp_math == LDEQ_MLP_MATH_BF16X3 && dtype != LDEQ_F32)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "mlp_math BF16X3 (tensor cores) needs a Float32 state; Float64 runs on the exact path");
    MlpNet net;
    int rc = make_net(h, layer_dims_host, n_layers, &net);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    LDEQ_CUDA(cudaSetDevice(h->device));
    if ((rc = upload_tgrid(h, t_host, T, s))) return rc;
    KOpts ko = to_kopts(opts);
    const size_t es = dtype == LDEQ_F32 ? 4 : 8;
    const int D = net.dims[0];
    ldeq_mlp_tape* tape = nullptr;
    if (tape_out) {
        tape = new ldeq_mlp_tape();
        tape->dtype = dtype; tape->B = B; tape->T = T; tape->net = net; tape->math = opts->mlp_math;
        tape->sense = opts->sensealg; tape->norm_mode = opts->norm_mode; tape->kopts = ko;
        long long cap = opts->tape_steps;
        if (cap <= 0) cap = opts->adaptive ? (4LL * T > 256 ? 4LL * T : 256) : (long long)((t_host[T - 1] - t_host[0]) / opts->dt) + 3;
        if (cap > opts->maxiters) cap = opts->maxiters;
        tape->cap = (int)cap;
        const size_t nB = B, c = (size_t)cap;
        size_t off = 0;
        const size_t o_t = off; off += al256(c * nB * 8);
        const size_t o_dt = off; off += al256(c * nB * 8);
        const size_t o_u = off; off += al256(c * nB * D * es);
        const size_t o_p = off; off += al256((size_t)net.n_params * es);
        const size_t o_pt = off; off += al256((size_t)net.n_params * es);
        const size_t o_tg = off; off += al256((size_t)T * 8);
        const size_t o_r = off; off += al256(nB * 4);
        const size_t o_na = off; off += al256(nB * 4);
        const size_t o_nr = off; off += al256(nB * 4);
        const size_t o_info = off; off += 256;
        cudaError_t e = cudaMallocAsync(&tape->base, off, s);
        if (e != cudaSuccess) { delete tape; return set_err(h, LDEQ_ERR_NOMEM, "cudaMallocAsync(mlp tape)", e); }
        char* bp = (char*)tape->base;
        tape->t = (double*)(bp + o_t); tape->dt = (double*)(bp + o_dt); tape->u = bp + o_u; tape->params = bp + o_p;
        tape->params_t = bp + o_pt; tape->tgrid = (double*)(bp + o_tg); tape->retcode = (int32_t*)(bp + o_r);
        tape->naccept = (int32_t*)(bp + o_na); tape->nreject = (int32_t*)(bp + o_nr);
        tape->info = (int32_t*)(bp + o_info);
        cudaMemsetAsync(tape->info, 0, 32, s);
        if (!slot_acquire(h, &tape->h_info, &tape->ready)) {
            cudaFreeAsync(tape->base, s);
            delete tape;
            return set_err(h, LDEQ_ERR_NOMEM, "mlp tape host mirror");
        }
        cudaMemcpyAsync(tape->params, params_flat, (size_t)net.n_params * es, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(tape->tgrid, h->d_tgrid, (size_t)T * 8, cudaMemcpyDeviceToDevice, s);
    }
    int32_t* d_ret = tape ? tape->retcode : retcode;
    int32_t* d_na = tape ? tape->naccept : naccept;
    int32_t* d_nr = tape ? tape->nreject : nreject;
    if (opts->mlp_math == LDEQ_MLP_MATH_BF16X3)
        rc = ldeq_mlp_tc_forward(h, layer_dims_host, n_layers, (const float*)params_flat, (const float*)z0, h->d_tgrid, B, T, ko,
                                 opts->norm_mode, (float*)traj_out, d_ret, d_na, d_nr, tape ? tape->t : nullptr,
                                 tape ? tape->dt : nullptr, tape ? (float*)tape->u : nullptr, tape ? tape->cap : 0, s);
    else if (dtype == LDEQ_F32)
        rc = mlp_fwd_dispatch<float>(h, net, params_flat, z0, h->d_tgrid, B, T, ko, opts->norm_mode, traj_out, d_ret, d_na, d_nr, tape, s);
    else
        rc = mlp_fwd_dispatch<double>(h, net, params_flat, z0, h->d_tgrid, B, T, ko, opts->norm_mode, traj_out, d_ret, d_na, d_nr, tape, s);
    if (rc) {
        if (tape) { cudaFreeAsync(tape->base, s); cudaEventRecord(tape->ready, s); slot_release(h, tape->h_info, tape->ready); delete tape; }
        return rc;
    }
    if (tape) {
        // the reverse pass must know whether every accepted step found room on the tape (ldeq_mlp_solve_bwd checks)
        mlp_max_naccept_kernel<<<64, 256, 0, s>>>(tape->naccept, tape->retcode, B, tape->info);
        h->launches += 1;
        cudaMemcpyAsync(tape->h_info, tape->info, 4, cudaMemcpyDeviceToHost, s);
        cudaEventRecord(tape->ready, s);
        if (retcode) cudaMemcpyAsync(retcode, tape->retcode, (size_t)B * 4, cudaMemcpyDeviceToDevice, s);
        if (naccept) cudaMemcpyAsync(naccept, tape->naccept, (size_t)B * 4, cudaMemcpyDeviceToDevice, s);
        if (nreject) cudaMemcpyAsync(nreject, tape->nreject, (size_t)B * 4, cudaMemcpyDeviceToDevice, s);
        *tape_out = tape;
    }
    return LDEQ_OK;
}

}  // extern "C"

template <class S, int TB>
static int launch_mlp_bwd(ldeq_handle* h, ldeq_mlp_tape* tape, const void* dtraj, void* dz0, void* dparams, cudaStream_t s) {
    const MlpNet& net = tape->net;
    const int B = tape->B;
    const int tiles = (B + TB - 1) / TB;
    const size_t smem_g = ((bwd_smem<S, TB>(net) + 15) & ~(size_t)15) + (size_t)net.n_params * sizeof(S);
    // on-chip accumulator only when there is at most one tile per SM anyway (it costs the second resident CTA and the L1
    // that otherwise holds the weights)
    const bool smem_grad = smem_g <= 225 * 1024 && tiles <= h->sm_count;
    const int per_sm = smem_grad ? 1 : 2;
    const int grid = tiles < per_sm * h->sm_count ? tiles : per_sm * h->sm_count;
    int rc = ensure_scratch(h, 1, (size_t)grid * net.n_params * sizeof(S), s);
    if (rc) return rc;
    mlp_transpose_kernel<S><<<64, 256, 0, s>>>(net, (const S*)tape->params, (S*)tape->params_t);
    // biases are not used from the transposed copy
    MlpTapeView<S> tv{tape->t, tape->dt, (S*)tape->u, tape->cap};
    if (smem_grad) {
        LDEQ_CUDA(cudaFuncSetAttribute(mlp_bwd_kernel<S, TB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g));
        mlp_bwd_kernel<S, TB, true><<<grid, MLP_THREADS, smem_g, s>>>(net, (const S*)tape->params, (const S*)tape->params_t,
                                                                      tape->tgrid, B, tape->T, (const S*)dtraj, tv, tape->retcode,
                                                                      tape->naccept, (S*)dz0, (S*)h->scratch[1]);
    } else {
        const size_t smem = bwd_smem<S, TB>(net);
        LDEQ_CUDA(cudaFuncSetAttribute(mlp_bwd_kernel<S, TB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_bwd_kernel<S, TB, false><<<grid, MLP_THREADS, smem, s>>>(net, (const S*)tape->params, (const S*)tape->params_t,
                                                                     tape->tgrid, B, tape->T, (const S*)dtraj, tv, tape->retcode,
                                                                     tape->naccept, (S*)dz0, (S*)h->scratch[1]);
    }
    LDEQ_CUDA(cudaGetLastError());
    mlp_reduce_grads_kernel<S><<<(net.n_params + 255) / 256, 256, 0, s>>>((const S*)h->scratch[1], grid, net.n_params, (S*)dparams);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 3;
    return LDEQ_OK;
}

// LDEQ_SENSE_INTERPOLATING_ADJOINT (ldeq_mlp_cadj.cuh): one cooperative launch, a tile of TB trajectories per CTA.
// Returns LDEQ_ERR_UNSUPPORTED (quietly) when the tiles of this TB cannot all be resident.
template <class S, int TB>
static int launch_mlp_cadj(ldeq_handle* h, ldeq_mlp_tape* tape, const void* dtraj, void* dz0, void* dparams, cudaStream_t s) {
    const MlpNet& net = tape->net;
    const int B = tape->B, grid = (B + TB - 1) / TB;
    // BATCH (stage records in shared memory, one weight-gradient pass per attempt) whenever the records fit;
    // LDEQ_CADJ_BATCH=0 keeps the per-stage reduction atomics (A/B switch)
    static const bool allow_batch = [] { const char* e = getenv("LDEQ_CADJ_BATCH"); return !(e && e[0] == '0'); }();
    static const bool allow_res = [] { const char* e = getenv("LDEQ_CADJ_RES"); return !(e && e[0] == '0'); }();
    // (stage records are instantiated for the smallest tile only: seven records of a wider tile do not fit next to the tile
    // state for the reference's network, and the unrolled 7 x TB pass would dominate the build time)
    bool batch = TB == 2 && allow_batch && cadj_smem<S, TB>(net, true) <= 227 * 1024;
    // RES: Float32, the smallest tile, the padded weight image + one working record fit next to the tile state
    bool res = false;
    if constexpr (sizeof(S) == 4 && TB == 2)
        res = allow_res && allow_batch && !getenv("LDEQ_MLP_NO_RESIDENT") && res_layout_ok(net, TB) && net.n_img > 0 &&
              cadj_smem<S, TB>(net, true, true) <= 227 * 1024 - 1024 && grid <= h->sm_count;
    if (res) batch = true;
    const size_t smem = cadj_smem<S, TB>(net, batch, res);
    const int nthreads = res ? RES_THREADS : MLP_THREADS;
    void* kern = (void*)mlp_cadj_kernel<S, TB, false, false>;
    if constexpr (TB == 2) { if (batch) kern = (void*)mlp_cadj_kernel<S, TB, true, false>; }
    if constexpr (sizeof(S) == 4 && TB == 2) { if (res) kern = (void*)mlp_cadj_kernel<S, TB, true, true>; }
    if (smem > 227 * 1024 || grid > GRID_SUM_HALF) return LDEQ_ERR_UNSUPPORTED;
    LDEQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    LDEQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nthreads, smem));
    if (per_sm * h->sm_count < grid) return LDEQ_ERR_UNSUPPORTED;
    const size_t NP = net.n_params, D = net.dims[0];
    const int na = tape->h_info[0] > 0 ? tape->h_info[0] : 1;
    int rc;
    if ((rc = ensure_scratch(h, 0, sizeof(double) * 4096, s))) return rc;
    if ((rc = ensure_scratch(h, 1, (size_t)grid * 2 * NP * sizeof(S), s))) return rc;
    const size_t dense_bytes = ((size_t)na * 7 * D * grid * TB * sizeof(S) + 255) & ~(size_t)255;
    const size_t grec_bytes = res ? (size_t)grid * 7 * CadjRec<S, TB>::floats(net.dims[0], net.max_width, net.n_layers) * sizeof(S) : 0;
    if ((rc = ensure_scratch(h, 3, dense_bytes + grec_bytes, s))) return rc;
    const size_t mu_bytes = (3 * NP * sizeof(S) + 255) & ~(size_t)255;
    const int trace_cap = getenv("LDEQ_CADJ_TRACE") ? 4096 : 0;  // debugging aid: (t, dt, EEst, accept) of every attempt
    if ((rc = ensure_scratch(h, 2, mu_bytes + (size_t)trace_cap * 32 + 256, s))) return rc;
    mlp_transpose_kernel<S><<<64, 256, 0, s>>>(net, (const S*)tape->params, (S*)tape->params_t);
    LDEQ_CUDA(cudaGetLastError());
    MlpNet netv = net;
    if (res) res_plan(netv, RES_THREADS);
    S* grec = res ? (S*)((char*)h->scratch[3] + dense_bytes) : nullptr;
    const S* Pp = (const S*)tape->params;
    const S* Pt = (const S*)tape->params_t;
    const double* tg = tape->tgrid;
    int Bv = B, Tv = tape->T;
    KOpts kov = tape->kopts;
    const S* dt_ = (const S*)dtraj;
    MlpTapeView<S> tv{tape->t, tape->dt, (S*)tape->u, tape->cap};
    const int* ret = tape->retcode;
    const int* nacc = tape->naccept;
    S* dense = (S*)h->scratch[3];
    S* gscr = (S*)h->scratch[1];
    S* mubuf = (S*)h->scratch[2];
    double* partials = (double*)h->scratch[0];
    S* dz = (S*)dz0;
    S* dp = (S*)dparams;
    int* status = tape->info + 4;
    double* trace = trace_cap ? (double*)((char*)h->scratch[2] + mu_bytes) : nullptr;
    int tcap = trace_cap;
    void* args[] = {&netv, &Pp, &Pt, &tg, &Bv, &Tv, &kov, &dt_, &tv, &ret, &nacc, &dense, &gscr, &mubuf, &partials, &dz, &dp, &status, &trace, &tcap, &grec};
    LDEQ_CUDA(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(nthreads), args, smem, s));
    h->launches += 2;
    return LDEQ_OK;
}

template <class S>
static int mlp_cadj_dispatch(ldeq_handle* h, ldeq_mlp_tape* tape, const void* dtraj, void* dz0, void* dparams, cudaStream_t s) {
    const char* force = getenv("LDEQ_CADJ_TB");  // tuning aid: 2, 8 or 32 rows per CTA
    const int ftb = force ? atoi(force) : 0;
    int rc = LDEQ_ERR_UNSUPPORTED;
    if (ftb == 0 || ftb == 2) rc = launch_mlp_cadj<S, 2>(h, tape, dtraj, dz0, dparams, s);
    if (rc == LDEQ_ERR_UNSUPPORTED && (ftb == 0 || ftb == 8)) rc = launch_mlp_cadj<S, 8>(h, tape, dtraj, dz0, dparams, s);
    if (ftb == 2 || ftb == 8) { if (rc == LDEQ_ERR_UNSUPPORTED) return set_err(h, rc, "LDEQ_CADJ_TB: does not fit"); return rc; }
    if (rc == LDEQ_ERR_UNSUPPORTED) rc = launch_mlp_cadj<S, 32>(h, tape, dtraj, dz0, dparams, s);
    if (rc == LDEQ_ERR_UNSUPPORTED)
        return set_err(h, LDEQ_ERR_UNSUPPORTED, "interpolating adjoint: batch too large (all tiles must be co-resident for the "
                                                "error norm over the augmented state); use LDEQ_SENSE_DISCRETE_ADJOINT");
    return rc;
}

extern "C" {

int ldeq_mlp_solve_bwd(ldeq_handle* h, ldeq_mlp_tape* tape, const void* dtraj, void* dz0, void* dparams_flat,
                       ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!tape || !dtraj || !dz0 || !dparams_flat) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (int rc0 = refuse_capture(h, s, "ldeq_mlp_solve_bwd", "it waits for the forward kernel to check the tape for overflow on the host")) return rc0;
    LDEQ_CUDA(cudaSetDevice(h->device));
    // a solve that took more accepted steps than the tape holds has no exact gradient: say so instead of returning
    // NaN / partial sums (waits for the forward kernel, as the GOKU path's tape check does)
    LDEQ_CUDA(cudaEventSynchronize(tape->ready));
    if (tape->h_info[0] > tape->cap) {
        char msg[200];
        snprintf(msg, sizeof msg, "mlp tape overflow: the solve accepted %d steps, the tape holds %d; repeat ldeq_mlp_solve_fwd "
                 "with opts.tape_steps >= %d", tape->h_info[0], tape->cap, tape->h_info[0]);
        return set_err(h, LDEQ_ERR_TAPE_OVERFLOW, msg);
    }
    if (tape->sense == LDEQ_SENSE_INTERPOLATING_ADJOINT) {
        if (tape->norm_mode != LDEQ_NORM_GLOBAL)
            return set_err(h, LDEQ_ERR_UNSUPPORTED, "interpolating adjoint: the reference's backward solve has one step size for the "
                                                    "whole batch; it needs norm_mode = LDEQ_NORM_GLOBAL");
        if (tape->math != LDEQ_MLP_MATH_FP32)
            return set_err(h, LDEQ_ERR_UNSUPPORTED, "interpolating adjoint: exact arithmetic path only (mlp_math = LDEQ_MLP_MATH_FP32)");
        return tape->dtype == LDEQ_F32 ? mlp_cadj_dispatch<float>(h, tape, dtraj, dz0, dparams_flat, s)
                                       : mlp_cadj_dispatch<double>(h, tape, dtraj, dz0, dparams_flat, s);
    }
    if (tape->math == LDEQ_MLP_MATH_BF16X3 && !getenv("LDEQ_MLP_TC_BWD_OFF")) {
        // the tensor-core tape: adjoint sweep + weight-gradient GEMM on tcgen05 (ldeq_mlp_tc_bwd.cu)
        int32_t dims[MLP_MAX_LAYERS + 1];
        for (int l = 0; l <= tape->net.n_layers; ++l) dims[l] = tape->net.dims[l];
        return ldeq_mlp_tc_backward(h, dims, tape->net.n_layers, (const float*)tape->params, tape->tgrid, tape->B, tape->T,
                                    (const float*)dtraj, tape->t, tape->dt, (float*)tape->u, tape->cap, tape->retcode, tape->naccept,
                                    tape->h_info[0], (float*)dz0, (float*)dparams_flat, s);
    }
    const bool small = tape->B <= 4 * h->sm_count;
    if (tape->dtype == LDEQ_F32 && !getenv("LDEQ_MLP_NO_RESIDENT")) {
        MlpTapeView<float> tv{tape->t, tape->dt, (float*)tape->u, tape->cap};
        const int rc = ldeq_mlp_res_backward(h, tape->net, (const float*)tape->params, tape->tgrid, tape->B, tape->T,
                                             (const float*)dtraj, tv, tape->retcode, tape->naccept, (float*)dz0,
                                             (float*)dparams_flat, s);
        if (rc != LDEQ_ERR_UNSUPPORTED) return rc;
    }
    if (tape->dtype == LDEQ_F32)
        return small ? launch_mlp_bwd<float, 2>(h, tape, dtraj, dz0, dparams_flat, s)
                     : launch_mlp_bwd<float, 8>(h, tape, dtraj, dz0, dparams_flat, s);
    return small ? launch_mlp_bwd<double, 2>(h, tape, dtraj, dz0, dparams_flat, s)
                 : launch_mlp_bwd<double, 8>(h, tape, dtraj, dz0, dparams_flat, s);
}

// debugging aid (LDEQ_CADJ_TRACE=1): the first n attempts of the last interpolating-adjoint solve as (t, dt, EEst, accept)
int ldeq_debug_cadj_trace(ldeq_handle* h, ldeq_mlp_tape* tape, double* out_host, int n) {
    if (!h || !tape || !out_host) return LDEQ_ERR_INVALID;
    if (!getenv("LDEQ_CADJ_TRACE")) return set_err(h, LDEQ_ERR_INVALID, "set LDEQ_CADJ_TRACE=1 before the backward call");
    const size_t es = tape->dtype == LDEQ_F32 ? 4 : 8;
    const size_t mu_bytes = (3 * (size_t)tape->net.n_params * es + 255) & ~(size_t)255;
    LDEQ_CUDA(cudaSetDevice(h->device));
    LDEQ_CUDA(cudaDeviceSynchronize());
    LDEQ_CUDA(cudaMemcpy(out_host, (char*)h->scratch[2] + mu_bytes, (size_t)(n < 4096 ? n : 4096) * 32, cudaMemcpyDeviceToHost));
    return LDEQ_OK;
}

int ldeq_mlp_bwd_stats(ldeq_handle* h, ldeq_mlp_tape* tape, int32_t* out3_host, ldeq_stream stream) {
    if (!h) return LDEQ_ERR_INVALID;
    if (!tape || !out3_host) return set_err(h, LDEQ_ERR_INVALID, "null argument");
    if (int rc0 = refuse_capture(h, (cudaStream_t)stream, "ldeq_mlp_bwd_stats", "it synchronises the stream")) return rc0;
    LDEQ_CUDA(cudaSetDevice(h->device));
    LDEQ_CUDA(cudaMemcpyAsync(out3_host, tape->info + 4, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    LDEQ_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return LDEQ_OK;
}

void ldeq_mlp_tape_free(ldeq_handle* h, ldeq_mlp_tape* tape, ldeq_stream stream) {
    if (!tape) return;
    if (h) cudaSetDevice(h->device);
    if (tape->base) cudaFreeAsync(tape->base, (cudaStream_t)stream);
    slot_release(h, tape->h_info, tape->ready);
    delete tape;
}

}  // extern "C"
