// ldeq_mlp_common.cuh -- pieces shared by the exact-arithmetic LatentODE kernels (ldeq_mlp.cu: weights read through
// L1/L2, any dtype/size; ldeq_mlp_res.cu: Float32 weights resident in shared memory).
#pragma once
#include <cooperative_groups.h>

#include "ldeq_internal.h"
#include "ldeq_gridsum.cuh"

namespace ldeq {

#define MLP_THREADS 256
#define MLP_MAX_LAYERS 8

struct MlpNet {
    int n_layers;
    int dims[MLP_MAX_LAYERS + 1];
    int w_off[MLP_MAX_LAYERS];  // offset of vec(W_l) in the flat parameter vector
    int b_off[MLP_MAX_LAYERS];
    int n_params;
    int max_width;  // widest layer input/output
    // shared-memory weight image of the resident path: W_l at i_w[l] with leading dimension i_ld[l] (odd, so that both
    // W[k*ld + n] over n and over k are bank-conflict free), b_l at i_b[l]; n_img floats in all
    int i_w[MLP_MAX_LAYERS];
    int i_b[MLP_MAX_LAYERS];
    int i_ld[MLP_MAX_LAYERS];
    int n_img;
    int act_off[MLP_MAX_LAYERS];  // offset (in rows) of hidden layer l's output inside one activation slot
    int act_rows;                 // sum of the hidden widths
    int lb;                       // the layer whose parameter gradient is accumulated once per step (largest interior layer), or -1
    // thread mapping of the resident dense layers, fixed on the host for the launch's thread count (res_plan):
    // [0][l] forward (outputs = dims[l+1]), [1][l] transposed (outputs = dims[l]); a warp covers 2^lgG output groups x
    // 32 >> lgG contraction slices of cper rows each
    int m_lgG[2][MLP_MAX_LAYERS], m_cper[2][MLP_MAX_LAYERS];
    int g_sl[MLP_MAX_LAYERS];  // k-slices of the gradient update of layer l (thread = output neuron x slice)
};
#define RES_THREADS 512
#define RES_TGRID_MAX 256

template <class S> struct MlpTapeView {
    double* t;   // [cap][B]
    double* dt;  // [cap][B]
    S* u;        // [cap][B][D]
    int cap;
};

// ---- dense layers on a tile ------------------------------------------------------------------------
// Activations are stored feature-major per tile: x[k*TB + b].  W is (N,K) column-major: W[k*N + n].
// Thread w handles output neuron n = w % N over the k-slice s = w / N; slices are summed through `red`.
template <class S, int TB>
__device__ void dense_fwd(const S* __restrict__ W, const S* __restrict__ bias, const S* __restrict__ x, S* __restrict__ y,
                          S* __restrict__ red, int K, int N, bool relu) {
    int SL = 1;
    while (SL * 2 * N <= MLP_THREADS && SL < 16 && SL * 2 <= K) SL *= 2;
    const int kper = (K + SL - 1) / SL;
    for (int w = threadIdx.x; w < N * SL; w += MLP_THREADS) {
        const int s = w / N, n = w - s * N;
        const int k0 = s * kper, k1 = min(K, k0 + kper);
        S acc[TB];
        const S b0 = s == 0 ? bias[n] : (S)0;
#pragma unroll
        for (int b = 0; b < TB; ++b) acc[b] = b0;
#pragma unroll 8
        for (int k = k0; k < k1; ++k) {
            const S wv = W[(size_t)k * N + n];
#pragma unroll
            for (int b = 0; b < TB; ++b) acc[b] = s_fma<S>(wv, x[k * TB + b], acc[b]);
        }
        if (SL == 1) {
#pragma unroll
            for (int b = 0; b < TB; ++b) y[n * TB + b] = relu ? s_max<S>(acc[b], (S)0) : acc[b];
        } else {
#pragma unroll
            for (int b = 0; b < TB; ++b) red[(s * N + n) * TB + b] = acc[b];
        }
    }
    if (SL > 1) {
        __syncthreads();
        for (int i = threadIdx.x; i < N * TB; i += MLP_THREADS) {
            S a = (S)0;
            for (int s = 0; s < SL; ++s) a += red[s * N * TB + i];
            y[i] = relu ? s_max<S>(a, (S)0) : a;
        }
    }
    __syncthreads();
}


// ---- dense layers from the resident weight image (Float32) -------------------------------------------
// y[i][b] = epi( sum_{c<NC} W[i*sa + c*sc] x[c][b] ), i < NI.  Forward: i = output neuron (sa = 1, sc = ld);
// transposed (input gradient): i = input index (sa = ld, sc = 1).  Each thread owns NPT outputs (m, m+NS, ..) over a
// slice of the contraction; x is read four rows at a time as 16-byte broadcasts.  Epilogue: + bias, relu, or the relu
// mask of `mask` (which may alias y: an element is read and written by the same thread).
template <int TB> __device__ __forceinline__ void load_rows4(const float* x, float (&v)[4][TB]) {
    const float4* p = reinterpret_cast<const float4*>(x);
#pragma unroll
    for (int q = 0; q < TB; ++q) {  // 4 rows x TB floats = TB float4
        const float4 f = p[q];
        const int e = q * 4;
        v[(e + 0) / TB][(e + 0) % TB] = f.x;
        v[(e + 1) / TB][(e + 1) % TB] = f.y;
        v[(e + 2) / TB][(e + 2) % TB] = f.z;
        v[(e + 3) / TB][(e + 3) % TB] = f.w;
    }
}
template <int TB>
__device__ __forceinline__ void res_epilogue(float a, int o, int b, float* y, const float* bias, bool relu, const float* mask) {
    if (bias) a += bias[o];
    if (relu) a = fmaxf(a, 0.f);
    if (mask) a = mask[o * TB + b] > 0.f ? a : 0.f;
    y[o * TB + b] = a;
}
template <int TB, int NPT>
__device__ __forceinline__ void dense_res_impl(const float* W, int sa, int sc, int NI, int NC, int lgG, int cper,
                                               const float* x, float* y, const float* bias, bool relu, const float* mask) {
    // A warp owns G = 2^lgG consecutive output groups and splits the contraction into 32/G slices of cper rows, one per
    // group of G lanes; the slices meet through warp shuffles (no shared-memory reduction, one barrier per layer).
    // cper = G * odd and an odd leading dimension keep the 32 weight addresses of every load in 32 different banks,
    // forward (stride 1 between outputs) and transposed (stride ld) alike.
    const int NS = (NI + NPT - 1) / NPT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if ((warp << lgG) < NS) {  // warp-uniform
        const int G = 1 << lgG;
        const int s = lane >> lgG, m = (warp << lgG) + (lane & (G - 1));
        const bool on = m < NS;
        const int c0 = s * cper, c1 = on ? min(NC, c0 + cper) : c0;
        float acc[NPT][TB];
        const float* pw[NPT];
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const int i = min(m + j * NS, NI - 1);  // an output past the end shadows the last one and is dropped below
            pw[j] = W + i * sa + c0 * sc;
#pragma unroll
            for (int b = 0; b < TB; ++b) acc[j][b] = 0.f;
        }
        const int sc2 = 2 * sc, sc3 = 3 * sc, sc4 = 4 * sc;
        int c = c0;
#pragma unroll 2
        for (; c + 4 <= c1; c += 4) {
            float xv[4][TB];
            load_rows4<TB>(x + c * TB, xv);
#pragma unroll
            for (int j = 0; j < NPT; ++j) {
                const float w0 = pw[j][0], w1 = pw[j][sc], w2 = pw[j][sc2], w3 = pw[j][sc3];
                pw[j] += sc4;
#pragma unroll
                for (int b = 0; b < TB; ++b) {
                    acc[j][b] = fmaf(w0, xv[0][b], acc[j][b]);
                    acc[j][b] = fmaf(w1, xv[1][b], acc[j][b]);
                    acc[j][b] = fmaf(w2, xv[2][b], acc[j][b]);
                    acc[j][b] = fmaf(w3, xv[3][b], acc[j][b]);
                }
            }
        }
        for (; c < c1; ++c) {
#pragma unroll
            for (int j = 0; j < NPT; ++j) {
                const float w0 = pw[j][0];
                pw[j] += sc;
#pragma unroll
                for (int b = 0; b < TB; ++b) acc[j][b] = fmaf(w0, x[c * TB + b], acc[j][b]);
            }
        }
        for (int off = G; off < 32; off <<= 1) {
#pragma unroll
            for (int j = 0; j < NPT; ++j)
#pragma unroll
                for (int b = 0; b < TB; ++b) acc[j][b] += __shfl_xor_sync(0xffffffffu, acc[j][b], off);
        }
        if (on && s == 0) {
#pragma unroll
            for (int j = 0; j < NPT; ++j) {
                const int o = m + j * NS;
                if (o < NI) {
#pragma unroll
                    for (int b = 0; b < TB; ++b) res_epilogue<TB>(acc[j][b], o, b, y, bias, relu, mask);
                }
            }
        }
    }
    __syncthreads();
}
// dir 0: forward (y = act(W x + b)), dir 1: transposed (dx = W^T dy, relu mask of `mask`)
template <int TB>
__device__ __forceinline__ void dense_res(const MlpNet& net, const float* img, int l, int dir, const float* x, float* y,
                                          bool relu, const float* mask) {
    const int K = net.dims[l], N = net.dims[l + 1], ld = net.i_ld[l];
    const float* W = img + net.i_w[l];
    const float* bias = dir ? nullptr : img + net.i_b[l];
    const int NI = dir ? K : N, NC = dir ? N : K, sa = dir ? ld : 1, sc = dir ? 1 : ld;
    const int lgG = net.m_lgG[dir][l], cper = net.m_cper[dir][l];
    if (NI >= 128)
        dense_res_impl<TB, 2>(W, sa, sc, NI, NC, lgG, cper, x, y, bias, relu, mask);
    else
        dense_res_impl<TB, 1>(W, sa, sc, NI, NC, lgG, cper, x, y, bias, relu, mask);
}
// host: fix the thread mapping of every resident dense layer for a launch with NT threads -- the split with the
// shortest per-thread contraction whose output groups fit the CTA's warps
static inline void res_plan(MlpNet& net, int NT) {
    const int warps = NT / 32;
    for (int l = 0; l < net.n_layers; ++l) {
        const int K = net.dims[l], N = net.dims[l + 1];
        int SL = 1;
        while (SL * 2 * N <= NT && SL < 32 && SL * 2 <= K) SL *= 2;
        net.g_sl[l] = SL;
    }
    for (int dir = 0; dir < 2; ++dir)
        for (int l = 0; l < net.n_layers; ++l) {
            const int NI = dir ? net.dims[l] : net.dims[l + 1], NC = dir ? net.dims[l + 1] : net.dims[l];
            const int NPT = NI >= 128 ? 2 : 1, NS = (NI + NPT - 1) / NPT;
            int best_lg = 5, best_cper = (NC + 3) & ~3;  // no split: a lane per output group
            for (int lgG = 4; lgG >= 2; --lgG) {
                const int G = 1 << lgG, SL = 32 / G;
                if ((NS + G - 1) / G > warps) continue;
                int odd = ((NC + SL - 1) / SL + G - 1) / G;
                if (!(odd & 1)) ++odd;
                const int cper = G * odd;
                if (cper < best_cper) { best_cper = cper; best_lg = lgG; }
            }
            if ((NS + 31) / 32 > warps && best_lg == 5) best_lg = 5;  // checked by res_layout_ok
            net.m_lgG[dir][l] = best_lg;
            net.m_cper[dir][l] = best_cper;
        }
}
// stage the padded weight image: img[i_w + k*ld + n] = W[k*N + n]
template <int NT> __device__ void stage_weight_image(const MlpNet& net, const float* __restrict__ P, float* img) {
    for (int l = 0; l < net.n_layers; ++l) {
        const int K = net.dims[l], N = net.dims[l + 1], ld = net.i_ld[l];
        const float* Wg = P + net.w_off[l];
        float* Ws = img + net.i_w[l];
        for (int idx = threadIdx.x; idx < K * N; idx += NT) {
            const int k = idx / N, n = idx - k * N;
            Ws[k * ld + n] = Wg[idx];
        }
        for (int n = threadIdx.x; n < N; n += NT) img[net.i_b[l] + n] = P[net.b_off[l] + n];
    }
    __syncthreads();
}
// forward through the resident image; with `acts` the hidden activations of every layer are kept there
template <int TB>
__device__ __forceinline__ void mlp_fwd_res(const MlpNet& net, const float* img, const float* x, float* y, float* hid0,
                                            float* hid1, float* acts) {
    const float* in = x;
    for (int l = 0; l < net.n_layers; ++l) {
        const bool last = l + 1 == net.n_layers;
        float* out = last ? y : (acts ? acts + net.act_off[l] * TB : ((l & 1) ? hid1 : hid0));
        dense_res<TB>(net, img, l, 0, in, out, !last, nullptr);
        in = out;
    }
}

// MLP forward on a tile: x (dims[0] x TB) -> y (dims[L] x TB).  hid: two ping-pong buffers of max_width*TB.
// With KEEP the post-activation outputs of every hidden layer are left in act[l] (for the VJP).
template <class S, int TB>
__device__ void mlp_fwd(const MlpNet& net, const S* __restrict__ P, const S* x, S* y, S* hid0, S* hid1, S* red) {
    const S* in = x;
    for (int l = 0; l < net.n_layers; ++l) {
        const bool last = l + 1 == net.n_layers;
        S* out = last ? y : ((l & 1) ? hid1 : hid0);
        dense_fwd<S, TB>(P + net.w_off[l], P + net.b_off[l], in, out, red, net.dims[l], net.dims[l + 1], !last);
        in = out;
    }
}

template <class S> __device__ __forceinline__ S tab_a(int j, int i) {
    using Tb = Tab<S>;
    switch (j * 8 + i) {
        case 1 * 8 + 0: return Tb::a21;
        case 2 * 8 + 0: return Tb::a31; case 2 * 8 + 1: return Tb::a32;
        case 3 * 8 + 0: return Tb::a41; case 3 * 8 + 1: return Tb::a42; case 3 * 8 + 2: return Tb::a43;
        case 4 * 8 + 0: return Tb::a51; case 4 * 8 + 1: return Tb::a52; case 4 * 8 + 2: return Tb::a53; case 4 * 8 + 3: return Tb::a54;
        case 5 * 8 + 0: return Tb::a61; case 5 * 8 + 1: return Tb::a62; case 5 * 8 + 2: return Tb::a63; case 5 * 8 + 3: return Tb::a64;
        case 5 * 8 + 4: return Tb::a65;
        case 6 * 8 + 0: return Tb::a71; case 6 * 8 + 1: return Tb::a72; case 6 * 8 + 2: return Tb::a73; case 6 * 8 + 3: return Tb::a74;
        case 6 * 8 + 4: return Tb::a75; case 6 * 8 + 5: return Tb::a76;
    }
    return (S)0;
}
template <class S> __device__ __forceinline__ S tab_bt(int i) {
    using Tb = Tab<S>;
    switch (i) {
        case 0: return Tb::bt1; case 1: return Tb::bt2; case 2: return Tb::bt3; case 3: return Tb::bt4;
        case 4: return Tb::bt5; case 5: return Tb::bt6; case 6: return Tb::bt7;
    }
    return (S)0;
}

// Per-trajectory controller / bookkeeping state of a tile (shared memory)
template <int TB> struct TileState {
    double t[TB], dt[TB], dts[TB], tnew[TB], qold[TB], esum[TB], dt_next[TB];
    long long iters[TB];
    int ks[TB], na[TB], nr[TB], ret[TB];
    int accept[TB], active[TB], nsave[TB];
};

// ---- forward ------------------------------------------------------------------------------------------
// RES: Float32 weights staged once into shared memory (padded image) and read from there by NT threads
template <class S, int TB, bool GLOBAL, bool RES = false, int NT = MLP_THREADS>
__global__ void __launch_bounds__(NT)
mlp_fwd_kernel(MlpNet net, const S* __restrict__ P, const S* __restrict__ z0, const double* __restrict__ tg_in, int B, int T,
               KOpts o, S* __restrict__ traj, int* __restrict__ retcode, int* __restrict__ naccept,
               int* __restrict__ nreject, MlpTapeView<S> tape, double* __restrict__ partials) {
    cg::grid_group grid = cg::this_grid();
    int gs_parity = 0;
    const int D = net.dims[0];
    const int HW = net.max_width;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    S* Wimg = reinterpret_cast<S*>(smem_raw);
    S* U = Wimg + (RES ? net.n_img : 0);  // [D][TB]
    S* G = U + D * TB;                      // stage input
    S* UN = G + D * TB;                     // u_{n+1}
    S* Kst = UN + D * TB;                   // [7][D][TB]
    S* hid0 = Kst + 7 * D * TB;
    S* hid1 = hid0 + HW * TB;
    S* red = hid1 + HW * TB;                // [NT][TB] (not on the resident path: its slices meet through shuffles)
    const size_t s_bytes =
        (((size_t)(RES ? net.n_img : 0) * sizeof(S) + (size_t)(10 * D + 2 * HW + (RES ? 0 : NT)) * TB * sizeof(S)) + 15) & ~(size_t)15;
    TileState<TB>* ts = reinterpret_cast<TileState<TB>*>(smem_raw + s_bytes);
    __shared__ int s_any;
    const double* tg = tg_in;
    if constexpr (RES) {
        // the save-time lookups of the step loop are on the critical path of a latency-bound CTA: keep the grid on chip
        __shared__ double tg_s[RES_TGRID_MAX];
        if (T <= RES_TGRID_MAX) {
            for (int i = threadIdx.x; i < T; i += NT) tg_s[i] = tg_in[i];
            __syncthreads();
            tg = tg_s;
        }
    }

    const double t0 = tg[0], tend = tg[T - 1];
    const double dtmax = o.dtmax > 0.0 ? o.dtmax : (tend - t0);
    const double dtmin = o.dtmin > 0.0 ? o.dtmin : fmax(2.220446049250313e-16, ulp_of(t0));
    const S abstol = (S)o.abstol, reltol = (S)o.reltol;
    const int ntiles = (B + TB - 1) / TB;
    const int DT = D * TB;
    auto rhs = [&](const S* x, S* y) {
        if constexpr (RES)
            mlp_fwd_res<TB>(net, Wimg, x, y, hid0, hid1, nullptr);
        else
            mlp_fwd<S, TB>(net, P, x, y, hid0, hid1, red);
    };
    if constexpr (RES) stage_weight_image<NT>(net, P, Wimg);

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // GLOBAL mode runs exactly one tile per CTA (the host sizes the grid so): all CTAs then take the same
        // steps (one dt for the batch) and meet at the same grid reductions
        const int b0 = tile * TB;
        // ---- load the tile, k1 = f(u0), initial step ---------------------------------------------------
        for (int i = threadIdx.x; i < DT; i += NT) {
            const int d = i / TB, b = i - d * TB;
            const int gb = b0 + b;
            U[i] = gb < B ? z0[(size_t)gb * D + d] : (S)0;
        }
        if (threadIdx.x < TB) {
            const int b = threadIdx.x;
            ts->t[b] = t0; ts->qold[b] = (double)pi_init(o).qold_pow;  /* controller memory: fastpow(qold, beta2) */ ts->iters[b] = 0; ts->ks[b] = 1; ts->na[b] = 0; ts->nr[b] = 0;
            ts->ret[b] = RET_SUCCESS; ts->active[b] = (b0 + b < B) && T > 1; ts->dt[b] = o.dt;
        }
        __syncthreads();
        rhs(U, Kst);  // fsalfirst
        // save point 0 is u0 itself
        for (int i = threadIdx.x; i < DT; i += NT) {
            const int d = i / TB, b = i - d * TB;
            if (b0 + b < B) traj[(size_t)(b0 + b) * D + d] = U[i];
        }
        if (o.adaptive && !(o.dt > 0.0)) {
            // Hairer initial step (SURVEY.md A.4); norms per trajectory or over the whole batch.
            // column sums: thread b adds the D entries of its trajectory (D is small)
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                double a0 = 0.0, a1 = 0.0;
                if (b0 + b < B)
                    for (int d = 0; d < D; ++d) {
                        const S sk = s_fma<S>(s_abs<S>(U[d * TB + b]), reltol, abstol);
                        const S a = U[d * TB + b] / sk, c = Kst[d * TB + b] / sk;
                        a0 += (double)(a * a);
                        a1 += (double)(c * c);
                    }
                ts->esum[b] = a0;
                ts->dt_next[b] = a1;
            }
            __syncthreads();
            double d0[TB], d1[TB];
            if (GLOBAL) {
                double s0 = 0.0, s1 = 0.0;
                for (int b = 0; b < TB; ++b) { s0 += ts->esum[b]; s1 += ts->dt_next[b]; }
                const double n = (double)D * (double)B;
                s0 = grid_sum(s0, partials, grid, gs_parity);
                s1 = grid_sum(s1, partials, grid, gs_parity);
                for (int b = 0; b < TB; ++b) { d0[b] = (double)s_sqrt<S>((S)(s0 / n)); d1[b] = (double)s_sqrt<S>((S)(s1 / n)); }
            } else {
                for (int b = 0; b < TB; ++b) {
                    d0[b] = (double)s_sqrt<S>((S)(ts->esum[b] / D));
                    d1[b] = (double)s_sqrt<S>((S)(ts->dt_next[b] / D));
                }
            }
            __syncthreads();
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                const double dt0 = (d0[b] < 1e-5 || d1[b] < 1e-5) ? 1e-6 : 0.01 * (d0[b] / d1[b]);
                ts->dts[b] = fmin(dt0, dtmax);
            }
            __syncthreads();
            // u1 = u0 + dt0 f0, f1 = f(u1)
            for (int i = threadIdx.x; i < DT; i += NT) G[i] = s_fma<S>((S)ts->dts[i % TB], Kst[i], U[i]);
            __syncthreads();
            rhs(G, UN);  // f1 in UN
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                double a2 = 0.0;
                if (b0 + b < B)
                    for (int d = 0; d < D; ++d) {
                        const S sk = s_fma<S>(s_abs<S>(U[d * TB + b]), reltol, abstol);
                        const S a = (UN[d * TB + b] - Kst[d * TB + b]) / sk;
                        a2 += (double)(a * a);
                    }
                ts->esum[b] = a2;
            }
            __syncthreads();
            double s2 = 0.0;
            if (GLOBAL) {
                for (int b = 0; b < TB; ++b) s2 += ts->esum[b];
                s2 = grid_sum(s2, partials, grid, gs_parity);
            }
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                const double dt0 = ts->dts[b];
                const double d2 = (double)s_sqrt<S>((S)(GLOBAL ? s2 / ((double)D * (double)B) : ts->esum[b] / D)) / dt0;
                double dtv;
                if (dt0 < 10.0 * 2.220446049250313e-16) {
                    dtv = fmax(1e-6, dtmin);
                } else {
                    const double m = fmax(d1[b], d2);
                    const double dt1 = (m <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : pow(10.0, -(2.0 + log10(m)) / 5.0);
                    dtv = fmax(dtmin, fmin(100.0 * dt0, fmin(dt1, dtmax)));
                }
                ts->dt[b] = dtv;
            }
            __syncthreads();
        }
        if (threadIdx.x < TB) {
            const int b = threadIdx.x;
            if (ts->active[b] && (!(ts->dt[b] > 0.0) || !isfinite(ts->dt[b]))) { ts->ret[b] = RET_DTLESSTHANMIN; ts->active[b] = 0; }
        }
        __syncthreads();

        // ---- step loop ----------------------------------------------------------------------------------
        for (;;) {
            if (threadIdx.x == 0) s_any = 0;
            __syncthreads();
            if (threadIdx.x < TB && ts->active[threadIdx.x]) s_any = 1;
            __syncthreads();
            // GLOBAL: all trajectories share the step sequence and every tile holds at least one of them, so
            // every CTA leaves this loop in the same iteration (no CTA is left waiting at a grid barrier)
            if (!s_any) break;
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                if (ts->active[b]) {
                    if (ts->iters[b] >= o.maxiters) {
                        ts->ret[b] = RET_MAXITERS; ts->active[b] = 0;
                    } else {
                        ts->iters[b]++;
                        const double t = ts->t[b];
                        const double dts = fmin(ts->dt[b], tend - t);
                        double tnew = t + dts;
                        if (fabs(tnew - tend) < 100.0 * ulp_of(fmax(fabs(t), fabs(tend)))) tnew = tend;
                        ts->dts[b] = dts; ts->tnew[b] = tnew;
                    }
                }
                ts->esum[b] = 0.0;
            }
            __syncthreads();
            // stages 2..7 (k1 is Kst[0] by FSAL)
            for (int j = 1; j < 7; ++j) {
                for (int i = threadIdx.x; i < DT; i += NT) {
                    S acc = tab_a<S>(j, 0) * Kst[i];
                    for (int q = 1; q < j; ++q) acc = s_fma<S>(tab_a<S>(j, q), Kst[q * DT + i], acc);
                    const S v = s_fma<S>((S)ts->dts[i % TB], acc, U[i]);
                    G[i] = v;
                    if (j == 6) UN[i] = v;
                }
                __syncthreads();
                rhs(G, Kst + j * DT);
            }
            // error estimate: squared scaled residuals into G (free after the stages), then column sums
            double part = 0.0;
            if (o.adaptive) {
                for (int i = threadIdx.x; i < DT; i += NT) {
                    const int b = i % TB;
                    S acc = tab_bt<S>(0) * Kst[i];
                    for (int q = 1; q < 7; ++q) acc = s_fma<S>(tab_bt<S>(q), Kst[q * DT + i], acc);
                    const S ut = (S)ts->dts[b] * acc;
                    const S sk = s_fma<S>(s_max<S>(s_abs<S>(U[i]), s_abs<S>(UN[i])), reltol, abstol);
                    const S a = ut / sk;
                    G[i] = a * a;
                }
                __syncthreads();
                if (threadIdx.x < TB) {
                    const int b = threadIdx.x;
                    double e = 0.0;
                    if (ts->active[b]) {
                        for (int d = 0; d < D; ++d) e += (double)G[d * TB + b];
                        if (GLOBAL) {
                            // one integrator for the whole matrix state (LatentODE.jl:70-72): a non-finite entry anywhere fails
                            // the WHOLE solve.  The flag travels inside the grid-wide sum (NaN), so every CTA takes the same
                            // decision in the same iteration and none is left waiting at a grid barrier.
                            bool fin = true;
                            for (int d = 0; d < D; ++d) fin = fin && s_finite<S>(UN[d * TB + b]);
                            if (!fin) e = __longlong_as_double(0x7ff8000000000000LL);
                        }
                    }
                    ts->esum[b] = e;
                }
                __syncthreads();
                if (GLOBAL) {
                    for (int b = 0; b < TB; ++b) part += ts->esum[b];
                    part = grid_sum(part, partials, grid, gs_parity);
                }
            }
            // controller, one thread per trajectory
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                ts->accept[b] = 0;
                if (ts->active[b]) {
                    bool finite = true;
                    for (int d = 0; d < D; ++d) finite = finite && s_finite<S>(UN[d * TB + b]);
                    bool accept = true;
                    double dt_next = ts->dt[b];
                    if (o.adaptive) {
                        const double e2 = GLOBAL ? part / ((double)D * (double)B) : ts->esum[b] / (double)D;
                        const double EEst = (double)s_sqrt<S>((S)e2);
                        if (EEst != EEst) finite = false;
                        PiState pst = pi_init(o);  // loop invariants; the controller memory lives in shared memory per row
                        pst.qold_pow = (float)ts->qold[b];
                        accept = pi_controller(o, EEst, ts->dts[b], dtmax, pst, dt_next);
                        ts->qold[b] = (double)pst.qold_pow;
                    }
                    if (!finite) {
                        ts->ret[b] = RET_UNSTABLE; ts->active[b] = 0;
                    } else {
                        if (accept) {
                            const int n = ts->na[b];
                            if (tape.cap > 0 && n < tape.cap) {
                                tape.t[(size_t)n * B + b0 + b] = ts->t[b];
                                tape.dt[(size_t)n * B + b0 + b] = ts->dts[b];
                            }
                            ts->accept[b] = 1;
                        } else {
                            ts->nr[b]++;
                        }
                        ts->dt[b] = dt_next;
                        if (o.adaptive && !(accept && ts->tnew[b] == tend) && (!(fabs(dt_next) > dtmin) || !isfinite(dt_next))) {
                            ts->ret[b] = RET_DTLESSTHANMIN; ts->active[b] = 0; ts->accept[b] = 0;
                        }
                    }
                }
            }
            __syncthreads();
            // tape: state at the start of the accepted step
            if (tape.cap > 0) {
                for (int i = threadIdx.x; i < DT; i += NT) {
                    const int d = i / TB, b = i - d * TB;
                    if (ts->accept[b] && ts->na[b] < tape.cap)
                        tape.u[((size_t)ts->na[b] * B + b0 + b) * D + d] = U[i];
                }
            }
            // saveat through the dense interpolant; a trajectory may have several pending save points
            for (;;) {
                if (threadIdx.x == 0) s_any = 0;
                __syncthreads();
                if (threadIdx.x < TB) {
                    const int b = threadIdx.x;
                    const int pend = ts->accept[b] && ts->ks[b] < T && tg[ts->ks[b]] <= ts->tnew[b];
                    ts->nsave[b] = pend;
                    if (pend) s_any = 1;
                }
                __syncthreads();
                if (!s_any) break;
                for (int i = threadIdx.x; i < DT; i += NT) {
                    const int d = i / TB, b = i - d * TB;
                    if (ts->nsave[b]) {
                        const int ks = ts->ks[b];
                        const double tsv = tg[ks];
                        S out;
                        if (tsv == ts->tnew[b]) {
                            out = UN[i];
                        } else {
                            S bw[7];
                            interp_weights<S>((S)((tsv - ts->t[b]) / ts->dts[b]), bw);
                            S acc = bw[0] * Kst[i];
#pragma unroll
                            for (int q = 1; q < 7; ++q) acc = s_fma<S>(bw[q], Kst[q * DT + i], acc);
                            out = s_fma<S>((S)ts->dts[b], acc, U[i]);
                        }
                        traj[((size_t)ks * B + b0 + b) * D + d] = out;
                    }
                }
                __syncthreads();
                if (threadIdx.x < TB && ts->nsave[threadIdx.x]) ts->ks[threadIdx.x]++;
            }
            // commit accepted steps
            for (int i = threadIdx.x; i < DT; i += NT) {
                if (ts->accept[i % TB]) { U[i] = UN[i]; Kst[i] = Kst[6 * DT + i]; }
            }
            __syncthreads();
            if (threadIdx.x < TB) {
                const int b = threadIdx.x;
                if (ts->accept[b]) {
                    ts->t[b] = ts->tnew[b];
                    ts->na[b]++;
                    if (ts->ks[b] >= T) ts->active[b] = 0;
                }
            }
            __syncthreads();
        }
        // ---- epilogue of the tile: NaN block on failure (GOKU.jl:114 convention), statistics -----------
        for (int i = threadIdx.x; i < DT; i += NT) {
            const int d = i / TB, b = i - d * TB;
            if (b0 + b < B && ts->ret[b] != RET_SUCCESS)
                for (int k = 0; k < T; ++k) traj[((size_t)k * B + b0 + b) * D + d] = s_nan<S>();
        }
        if (threadIdx.x < TB && b0 + threadIdx.x < B) {
            const int b = threadIdx.x;
            if (retcode) retcode[b0 + b] = ts->ret[b];
            if (naccept) naccept[b0 + b] = ts->na[b];
            if (nreject) nreject[b0 + b] = ts->nr[b];
        }
        __syncthreads();
        if (GLOBAL) break;
    }
}


template <class S, int TB, bool RES = false, int NT = MLP_THREADS> static size_t fwd_smem(const MlpNet& net) {
    const size_t D = net.dims[0], HW = net.max_width;
    size_t n = (RES ? (size_t)net.n_img : 0) * sizeof(S) + (3 * D + 7 * D + 2 * HW + (RES ? 0 : NT)) * TB * sizeof(S);
    n = (n + 15) & ~(size_t)15;
    return n + sizeof(TileState<TB>) + 64;
}

// the resident path reads activations as 16-byte vectors: every buffer of a tile must start 16-byte aligned
static inline bool res_layout_ok(const MlpNet& net, int TB, int NT = RES_THREADS) {
    for (int l = 0; l <= net.n_layers; ++l) {
        if ((net.dims[l] * TB) % 4) return false;
        if (net.dims[l] > 2 * NT) return false;  // two outputs per thread at most
    }
    return true;
}

}  // namespace ldeq

// ldeq_mlp_res.cu: Float32 weights resident in shared memory.  Both return LDEQ_ERR_UNSUPPORTED (without touching the
// handle's error text) when the network / batch does not fit that path; the caller then uses the general kernels.
// info / overflow: the tape's largest accepted-step count and, for a device-checked tape, its overflow word (null for an
// eager tape), read by the gradient reduction (mlp_tape_overflowed).
struct ldeq_mlp_tape;
int ldeq_mlp_res_forward(ldeq_handle* h, const ldeq::MlpNet& net, const float* params, const float* z0, const double* d_tgrid,
                         int B, int T, const ldeq::KOpts& ko, int norm_mode, float* traj, int32_t* ret, int32_t* na, int32_t* nr,
                         ldeq::MlpTapeView<float> tv, double* partials, cudaStream_t s);
int ldeq_mlp_res_backward(ldeq_handle* h, const ldeq::MlpNet& net, const float* params, const double* d_tgrid, int B, int T,
                          const float* dtraj, ldeq::MlpTapeView<float> tv, const int32_t* ret, const int32_t* na, float* dz0,
                          float* dparams, const int32_t* info, int32_t* overflow, cudaStream_t s);
