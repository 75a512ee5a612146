// ldeq_mlp_tc.cu -- LatentODE forward solve with the MLP right-hand side on the 5th-generation tensor cores
// (tcgen05 + TMEM), `LDEQ_MLP_MATH_BF16X3`.
//
// Same semantics as mlp_fwd_kernel (ldeq_mlp.cu; reference src/models/LatentODE.jl:61-78 with the NODE struct's
// Chain(Dense(D,H,relu), Dense(H,H,relu), Dense(H,D)), examples/pendulum_friction-less/nODE.jl:14-16), for
// batches where batch x hidden is a genuine dense contraction.
//
// One CTA integrates a tile of 128 trajectories for the whole time span; thread r owns trajectory (row) r:
// its state, step size and controller memory stay in registers, exactly as in the GOKU kernel.  One RHS
// evaluation is three dependent GEMMs with M = 128 (the tile), issued by one thread as tcgen05.mma:
//   * B operand = weights, staged ONCE per CTA in shared memory as bf16 "hi" and "lo" images in the UMMA
//     canonical K-major (no swizzle) layout (195 kB for 16-200-200-16, widths padded to multiples of 16);
//   * A operand = activations, read by the MMA straight from TMEM: the epilogue of layer l (tcgen05.ld the
//     fp32 accumulators, + bias, relu, split into bf16 hi/lo, tcgen05.st) writes the A operand of layer l+1,
//     so activations never touch shared memory;
//   * fp32 parity: x*w ~ x_hi*w_hi + x_hi*w_lo + x_lo*w_hi (three MMAs per K-step, fp32 accumulate in TMEM),
//     relative error 2^-16 per product instead of bf16's 2^-8;
//   * the stage slopes k1..k6 live in the 96 TMEM columns left over (512 = 208 accumulator + 2*104 operand + 96).
// TMEM column map: see the TC_COL_* constants below.
#include "ldeq_mlp_tc.cuh"

namespace ldeq {

// ---- forward ---------------------------------------------------------------------------------------------------
// Phases of the single-call-site state machine (the RHS evaluation is inlined exactly once).
enum { PH_F0 = 0, PH_INITDT = 1, PH_STAGE = 2 };

// epilogue of a hidden layer on the chunks [c_lo, c_hi) of a region: accumulators -> relu(acc + bias) -> bf16 hi/lo
// written back IN PLACE (8 hi columns + 8 lo columns per 16-column chunk) as the A operand of the next layer
__device__ __forceinline__ void tc_epilogue_inplace(uint32_t region_addr, const float* __restrict__ bias, int c_lo, int c_hi) {
    for (int c = c_lo; c < c_hi; c += 16) {
        float v[16];
        uint32_t hi[8], lo[8];
        tc_ld16(region_addr + c, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i] + bias[c + i], 0.f);
        split_pack16(v, hi, lo);
        tc_st8(region_addr + c, hi);
        tc_st8(region_addr + c + 8, lo);
    }
}

template <bool GLOBAL>
__global__ void __launch_bounds__(TC_THREADS, 1)
mlp_tc_fwd_kernel(TcNet net, const unsigned char* __restrict__ img_global, const float* __restrict__ z0,
                  const double* __restrict__ tg, int B, int T, KOpts o, float* __restrict__ traj, int* __restrict__ retcode,
                  int* __restrict__ naccept, int* __restrict__ nreject, MlpTapeViewTc<float> tape, double* __restrict__ partials) {
    cg::grid_group grid = cg::this_grid();
    int gs_parity = 0;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t mbar[4];  // [0] first column half, [1] second column half, [2] output layer, [3] weight images (TMA)
    __shared__ uint32_t tmem_base_s;
    __shared__ double red_s[TC_ROWS / 32];

    const int tid = threadIdx.x, warp = tid >> 5;
    const int quad = warp & 3, hf = warp >> 2;     // TMEM lane quadrant / column half of this warp
    const int row = quad * 32 + (tid & 31);           // trajectory (row of the tile) this thread works on
    const int D = net.d;
    // the weight images (and biases) are staged ONCE per CTA by the TMA unit: one thread issues bulk copies of the 195 kB
    // image (cp.async.bulk, UBLKCP in SASS) that complete on mbar[3]; everybody else goes on with the set-up meanwhile
    const float* bias1 = reinterpret_cast<const float*>(smem + net.bias_off);
    const float* bias2 = bias1 + net.n1;
    const float* bias3 = bias2 + net.n2;
    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        mbar_init(&mbar[2], 1);
        mbar_init(&mbar[3], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        stage_image_tma(smem, img_global, (uint32_t)net.smem_bytes, &mbar[3]);
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TC_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    mbar_wait(&mbar[3], 0);  // the images have landed (written by the async proxy, read by the tensor cores' async proxy)
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);  // this warp's 32-lane quadrant
    const uint32_t R0 = lane_addr + TC_COL_R0, R1 = lane_addr + TC_COL_R1, KS = lane_addr + TC_COL_K;
    uint32_t par_half = 0, par_out = 0;  // phase parity of the barrier this warp waits on for its half / the output layer

    const uint32_t lbo1 = (net.n1 / 8) * 128, lbo2 = (net.n2 / 8) * 128, lbo3 = (16 / 8) * 128;
    const uint32_t sbase = smem_u32(smem);
    // column halves of the two hidden layers (multiples of 16)
    const int n1a = ((net.n1 / 16 + 1) / 2) * 16, n2a = ((net.n2 / 16 + 1) / 2) * 16;

    const double t0 = tg[0], tend = tg[T - 1];
    const double dtmax = o.dtmax > 0.0 ? o.dtmax : (tend - t0);
    const double dtmin = o.dtmin > 0.0 ? o.dtmin : fmax(2.220446049250313e-16, ulp_of(t0));
    const float abstol = (float)o.abstol, reltol = (float)o.reltol;
    const int ntiles = (B + TC_ROWS - 1) / TC_ROWS;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b = tile * TC_ROWS + row;
        const bool live = b < B;
        const bool writer = hf == 0;  // both column halves carry the row's state redundantly (identical arithmetic, hence
        // identical values: TMEM stores of state are issued by both); only one half writes to global memory
        float u[16], g[16], kout[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) u[i] = (live && i < D) ? z0[(size_t)b * D + i] : 0.f;
        if (live && writer) {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < D) traj[(size_t)b * D + i] = u[i];  // save point 0 is u0 itself
        }
        PiState pist = pi_init(o);
        double t = t0, dt = o.dt, dts = 0.0, tnew = t0, dt0 = 0.0, d1n = 0.0;
        int na = 0, nr = 0, ks = 1, ret = RET_SUCCESS, stage = 0;
        long long iters = 0;
        bool active = live && T > 1;
        int phase = PH_F0;

        for (;;) {
            // ---- input of this RHS evaluation -------------------------------------------------------------------
            if (phase == PH_F0) {
#pragma unroll
                for (int i = 0; i < 16; ++i) g[i] = u[i];
            } else if (phase == PH_INITDT) {
                float k1[16];
                tc_ld16(KS, k1);  // f0 = k1
#pragma unroll
                for (int i = 0; i < 16; ++i) g[i] = fmaf((float)dt0, k1[i], u[i]);
            } else {
                if (stage == 1 && active) {
                    if (iters >= o.maxiters) { ret = RET_MAXITERS; active = false; }
                    else {
                        ++iters;
                        dts = fmin(dt, tend - t);
                        tnew = t + dts;
                        if (fabs(tnew - tend) < 100.0 * ulp_of(fmax(fabs(t), fabs(tend)))) tnew = tend;
                    }
                }
                float acc[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[i] = 0.f;
                for (int q = 0; q < stage; ++q) {
                    float kq[16];
                    tc_ld16(KS + 16 * q, kq);
                    const float a = c_a[stage][q];
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[i] = fmaf(a, kq[i], acc[i]);
                }
                const float h = (float)dts;
#pragma unroll
                for (int i = 0; i < 16; ++i) g[i] = fmaf(h, acc[i], u[i]);
            }
            // ---- RHS: three GEMMs on the tensor cores, activations TMEM -> TMEM ------------------------------------
            {
                {  // g -> R1[0:16) as bf16 hi (8 columns) + lo (8 columns)
                    uint32_t hi[8], lo[8];
                    split_pack16(g, hi, lo);
                    tc_st8(R1, hi);
                    tc_st8(R1 + 8, lo);
                    tc_wait_st();
                }
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {
                    tc_fence_after();
                    const uint32_t wh = sbase + net.img_off[0], wl = sbase + net.img_off[1];
                    tc_issue_layer(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, wh, wl, lbo1, 0, n1a, 1);
                    tc_commit(&mbar[0]);
                    tc_issue_layer(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, wh, wl, lbo1, n1a, net.n1 - n1a, 1);
                    tc_commit(&mbar[1]);
                }
                mbar_wait(&mbar[hf], par_half);
                par_half ^= 1;
                tc_fence_after();
                // epilogue 1 (this warp's column half), in place in R0 -> A operand of layer 2
                tc_epilogue_inplace(R0, bias1, hf ? n1a : 0, hf ? net.n1 : n1a);
                tc_wait_st();
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {
                    tc_fence_after();
                    const uint32_t wh = sbase + net.img_off[2], wl = sbase + net.img_off[3];
                    tc_issue_layer(tmem_base + TC_COL_R1, tmem_base + TC_COL_R0, wh, wl, lbo2, 0, n2a, net.n1 / 16);
                    tc_commit(&mbar[0]);
                    tc_issue_layer(tmem_base + TC_COL_R1, tmem_base + TC_COL_R0, wh, wl, lbo2, n2a, net.n2 - n2a, net.n1 / 16);
                    tc_commit(&mbar[1]);
                }
                mbar_wait(&mbar[hf], par_half);
                par_half ^= 1;
                tc_fence_after();
                // epilogue 2, in place in R1 -> A operand of layer 3
                tc_epilogue_inplace(R1, bias2, hf ? n2a : 0, hf ? net.n2 : n2a);
                tc_wait_st();
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {
                    tc_fence_after();
                    tc_issue_layer(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, sbase + net.img_off[4], sbase + net.img_off[5], lbo3, 0, 16,
                                   net.n2 / 16);
                    tc_commit(&mbar[2]);
                }
                mbar_wait(&mbar[2], par_out);
                par_out ^= 1;
                tc_fence_after();
                tc_ld16(R0, kout);
#pragma unroll
                for (int i = 0; i < 16; ++i) kout[i] = i < D ? kout[i] + bias3[i] : 0.f;
            }
            // ---- what the evaluation was for ---------------------------------------------------------------------
            bool all_done = false;
            if (phase == PH_F0) {
                tc_st16(KS, kout);  // k1 = f(u0)  (fsalfirst)
                tc_wait_st();
                if (o.adaptive && !(o.dt > 0.0)) {
                    // Hairer initial step, first half (SURVEY.md A.4)
                    float s0 = 0.f, s1 = 0.f;
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (i < D) {
                            const float sk = fmaf(fabsf(u[i]), reltol, abstol);
                            const float a = u[i] / sk, c = kout[i] / sk;
                            s0 = fmaf(a, a, s0);
                            s1 = fmaf(c, c, s1);
                        }
                    double e0 = s0, e1 = s1, n = D;
                    if (GLOBAL) {
                        // one dt for the batch: RMS over all D*B entries (summed by the `writer` half only)
                        double v0 = (live && writer) ? e0 : 0.0, v1 = (live && writer) ? e1 : 0.0;
                        for (int off = 16; off > 0; off >>= 1) { v0 += __shfl_xor_sync(0xffffffffu, v0, off); v1 += __shfl_xor_sync(0xffffffffu, v1, off); }
                        if (writer && (tid & 31) == 0) red_s[quad] = v0;
                        __syncthreads();
                        double b0 = 0.0;
                        for (int w = 0; w < TC_ROWS / 32; ++w) b0 += red_s[w];
                        __syncthreads();
                        if (writer && (tid & 31) == 0) red_s[quad] = v1;
                        __syncthreads();
                        double b1 = 0.0;
                        for (int w = 0; w < TC_ROWS / 32; ++w) b1 += red_s[w];
                        __syncthreads();
                        e0 = grid_sum(b0, partials, grid, gs_parity);
                        e1 = grid_sum(b1, partials, grid, gs_parity);
                        n = (double)D * (double)B;
                    }
                    const double d0 = (double)sqrtf((float)(e0 / n));
                    d1n = (double)sqrtf((float)(e1 / n));
                    dt0 = (d0 < 1e-5 || d1n < 1e-5) ? 1e-6 : 0.01 * (d0 / d1n);
                    dt0 = fmin(dt0, dtmax);
                    phase = PH_INITDT;
                } else {
                    phase = PH_STAGE;
                    stage = 1;
                    if (active && (!(dt > 0.0) || !isfinite(dt))) { ret = RET_DTLESSTHANMIN; active = false; }
                }
            } else if (phase == PH_INITDT) {
                float k1[16];
                tc_ld16(KS, k1);
                float s2 = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (i < D) {
                        const float sk = fmaf(fabsf(u[i]), reltol, abstol);
                        const float a = (kout[i] - k1[i]) / sk;
                        s2 = fmaf(a, a, s2);
                    }
                double e2 = s2, n = D;
                if (GLOBAL) {
                    double v = (live && writer) ? e2 : 0.0;
                    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                    if (writer && (tid & 31) == 0) red_s[quad] = v;
                    __syncthreads();
                    double bsum = 0.0;
                    for (int w = 0; w < TC_ROWS / 32; ++w) bsum += red_s[w];
                    __syncthreads();
                    e2 = grid_sum(bsum, partials, grid, gs_parity);
                    n = (double)D * (double)B;
                }
                const double d2 = (double)sqrtf((float)(e2 / n)) / dt0;
                if (dt0 < 10.0 * 2.220446049250313e-16) {
                    dt = fmax(1e-6, dtmin);
                } else {
                    const double m = fmax(d1n, d2);
                    const double dt1 = (m <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : pow(10.0, -(2.0 + log10(m)) / 5.0);
                    dt = fmax(dtmin, fmin(100.0 * dt0, fmin(dt1, dtmax)));
                }
                phase = PH_STAGE;
                stage = 1;
                if (active && (!(dt > 0.0) || !isfinite(dt))) { ret = RET_DTLESSTHANMIN; active = false; }
            } else if (stage < 6) {
                tc_st16(KS + 16 * stage, kout);  // k_{stage+1}
                tc_wait_st();
                ++stage;
            } else {
                // ---- end of an attempted step: g = u_{n+1}, kout = k7 -------------------------------------------------
                // dense-output coefficients and the error estimate from k1..k7 in one pass over the TMEM slots
                float c2[16], c3[16], c4[16], et[16], k1v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    c2[i] = c_r[6][1] * kout[i]; c3[i] = c_r[6][2] * kout[i]; c4[i] = c_r[6][3] * kout[i];
                    et[i] = c_bt[6] * kout[i];
                }
                for (int q = 0; q < 6; ++q) {
                    float kq[16];
                    tc_ld16(KS + 16 * q, kq);
                    const float r2 = c_r[q][1], r3 = c_r[q][2], r4 = c_r[q][3], bt = c_bt[q];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        c2[i] = fmaf(r2, kq[i], c2[i]); c3[i] = fmaf(r3, kq[i], c3[i]); c4[i] = fmaf(r4, kq[i], c4[i]);
                        et[i] = fmaf(bt, kq[i], et[i]);
                        if (q == 0) k1v[i] = kq[i];
                    }
                }
                const float h = (float)dts;
                bool finite = true;
                float e2f = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (i < D) {
                        finite = finite && isfinite(g[i]);
                        const float sk = fmaf(fmaxf(fabsf(u[i]), fabsf(g[i])), reltol, abstol);
                        const float a = h * et[i] / sk;
                        e2f = fmaf(a, a, e2f);
                    }
                bool accept = true;
                double dt_next = dt;
                if (o.adaptive) {
                    double e2 = e2f, n = D;
                    if (GLOBAL) {
                        // a non-finite row fails the WHOLE matrix solve (one integrator, LatentODE.jl:70-72): the NaN rides in the
                        // grid-wide sum, so every CTA decides the same in the same iteration (no CTA left at a grid barrier)
                        if (active && !finite) e2 = __longlong_as_double(0x7ff8000000000000LL);
                        double v = (active && writer) ? e2 : 0.0;
                        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                        if (writer && (tid & 31) == 0) red_s[quad] = v;
                        __syncthreads();
                        double bsum = 0.0;
                        for (int w = 0; w < TC_ROWS / 32; ++w) bsum += red_s[w];
                        __syncthreads();
                        e2 = grid_sum(bsum, partials, grid, gs_parity);
                        n = (double)D * (double)B;
                    }
                    const double EEst = (double)sqrtf((float)(e2 / n));
                    if (EEst != EEst) finite = false;
                    accept = pi_controller(o, EEst, dts, dtmax, pist, dt_next);
                }
                // every thread of the warp has read k1..k6 by now; the FSAL store below may overwrite slot 0 only
                // after the other half has read it as well
                tc_fence_before();
                __syncthreads();
                tc_fence_after();
                if (active) {
                    if (!finite) {
                        ret = RET_UNSTABLE;
                        active = false;
                    } else {
                        if (accept) {
                            if (writer && tape.cap > 0 && na < tape.cap) {
                                tape.t[(size_t)na * B + b] = t;
                                tape.dt[(size_t)na * B + b] = dts;
#pragma unroll
                                for (int i = 0; i < 16; ++i)
                                    if (i < D) tape.u[((size_t)na * B + b) * D + i] = u[i];
                            }
                            ++na;
                            // saveat through the dense interpolant (Horner form)
                            const double inv = 1.0 / dts;
                            while (ks < T && tg[ks] <= tnew) {
                                if (writer) {
                                    const double tsv = tg[ks];
                                    float* dst = traj + ((size_t)ks * B + b) * D;
                                    if (tsv == tnew) {
#pragma unroll
                                        for (int i = 0; i < 16; ++i)
                                            if (i < D) dst[i] = g[i];
                                    } else {
                                        const float th = (float)((tsv - t) * inv);
                                        const float hth = h * th;
#pragma unroll
                                        for (int i = 0; i < 16; ++i)
                                            if (i < D) dst[i] = fmaf(hth, fmaf(th, fmaf(th, fmaf(th, c4[i], c3[i]), c2[i]), k1v[i]), u[i]);
                                    }
                                }
                                ++ks;
                            }
                            t = tnew;
#pragma unroll
                            for (int i = 0; i < 16; ++i) u[i] = g[i];
                            if (ks >= T) active = false;
                        } else {
                            ++nr;
                        }
                        dt = dt_next;
                        if (active && o.adaptive && (!(fabs(dt) > dtmin) || !isfinite(dt))) { ret = RET_DTLESSTHANMIN; active = false; }
                    }
                }
                // FSAL: k7 becomes k1 of the next step for the rows that accepted, the others keep their k1
                // (tcgen05.st is warp-aligned: every thread executes it, the DATA is selected per row)
                {
                    const bool take = accept && finite;
#pragma unroll
                    for (int i = 0; i < 16; ++i) k1v[i] = take ? kout[i] : k1v[i];
                    tc_st16(KS, k1v);
                    tc_wait_st();
                }
                stage = 1;
                tc_fence_before();
                all_done = __syncthreads_or(active ? 1 : 0) == 0;
                tc_fence_after();
            }
            if (all_done) break;
            if (phase != PH_STAGE && T <= 1) break;
        }
        if (live && writer) {
            if (ret != RET_SUCCESS) {
                for (int k = 0; k < T; ++k)
                    for (int i = 0; i < D; ++i) traj[((size_t)k * B + b) * D + i] = __int_as_float(0x7fc00000);
            }
            if (retcode) retcode[b] = ret;
            if (naccept) naccept[b] = na;
            if (nreject) nreject[b] = nr;
        }
        __syncthreads();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC_TMEM_COLS));
}

}  // namespace ldeq

using namespace ldeq;

// Host side: called from ldeq_mlp_solve_fwd when opts->mlp_math == LDEQ_MLP_MATH_BF16X3.
// Returns LDEQ_ERR_UNSUPPORTED for shapes this kernel is not built for (the caller reports it; no silent fallback).
int ldeq_mlp_tc_forward(ldeq_handle* h, const int32_t* dims, int n_layers, const float* params, const float* z0,
                        const double* d_tgrid, int B, int T, const KOpts& ko, int norm_mode, float* traj, int32_t* ret,
                        int32_t* na, int32_t* nr, double* tape_t, double* tape_dt, float* tape_u, int tape_cap,
                        cudaStream_t s) {
    TcNet net;
    int rc = ldeq_tc_make_net(h, dims, n_layers, &net);
    if (rc) return rc;
    const int D = dims[0], H1 = dims[1], H2 = dims[2];
    rc = ensure_scratch(h, 2, (size_t)net.smem_bytes, s);
    if (rc) return rc;
    rc = ensure_scratch(h, 0, sizeof(double) * 4096, s);
    if (rc) return rc;
    unsigned char* img = (unsigned char*)h->scratch[2];
    mlp_tc_prep_kernel<<<64, 256, 0, s>>>(net, params, D, H1, H2, img);
    LDEQ_CUDA(cudaGetLastError());
    const int tiles = (B + TC_ROWS - 1) / TC_ROWS;
    MlpTapeViewTc<float> tv{tape_t, tape_dt, tape_u, tape_cap};
    double* partials = (double*)h->scratch[0];
    KOpts kov = ko;
    const unsigned char* imgc = img;
    void* args[] = {&net, &imgc, &z0, &d_tgrid, &B, &T, &kov, &traj, &ret, &na, &nr, &tv, &partials};
    // fixed-step mode computes no error norm: no grid barrier, no co-residency limit
    if (norm_mode == LDEQ_NORM_GLOBAL && ko.adaptive) {
        if (tiles > h->sm_count)
            return set_err(h, LDEQ_ERR_UNSUPPORTED, "bf16x3 tensor-core path, global norm: B <= 128 * SM count (all tiles co-resident)");
        LDEQ_CUDA(cudaFuncSetAttribute(mlp_tc_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, net.smem_bytes));
        LDEQ_CUDA(cudaLaunchCooperativeKernel((void*)mlp_tc_fwd_kernel<true>, dim3(tiles), dim3(TC_THREADS), args, net.smem_bytes, s));
    } else {
        const int grid = tiles < h->sm_count ? tiles : h->sm_count;
        LDEQ_CUDA(cudaFuncSetAttribute(mlp_tc_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, net.smem_bytes));
        LDEQ_CUDA(cudaLaunchKernel((void*)mlp_tc_fwd_kernel<false>, dim3(grid), dim3(TC_THREADS), args, net.smem_bytes, s));
    }
    h->launches += 2;
    return LDEQ_OK;
}
