// ldeq_mlp_tc_bwd.cu -- reverse pass of the LatentODE solve on the 5th-generation tensor cores (tcgen05 + TMEM):
// the discrete adjoint of the taped Tsit5 steps (what ldeq_mlp_solve_bwd computes, reference src/models/LatentODE.jl:70-72
// under Zygote) for tapes recorded by the tensor-core forward kernel (ldeq_mlp_tc.cu, LDEQ_MLP_MATH_BF16X3).
//
// Two kernels:
//
//  mlp_tc_adj_kernel   one CTA per tile of 128 trajectories, thread pair (row, half) per trajectory, steps in reverse.
//      Per step: (F) the seven stage inputs are recomputed exactly as the forward kernel computed them (same images,
//      same bf16x3 products, activations TMEM -> TMEM), and (R) the reverse sweep through the stages runs the three
//      TRANSPOSED products per stage  dz2 = (kbar W3) .* [h2 > 0],  dz1 = (dz2 W2) .* [h1 > 0],  gbar = dz1 W1  on the
//      same shared-memory weight images read through MN-major descriptors (no second image set).  The Tsit5 adjoint
//      bookkeeping (7 x 16 stage cotangents, dense-output cotangents) stays in the registers of the two threads of a row.
//      What the parameter gradient needs -- per (tile, step, stage) the operands g, h1, h2, kbar, dz1, dz2 -- leaves the
//      SM as bf16 hi/lo records, 16-byte chunks written straight into the MN-major canonical layout.
//  mlp_tc_wgrad_kernel a split-K GEMM over those records:  dW2 += dz2^T h1,  dW1 += dz1^T [g 1],  dW3^T += h2^T kbar  with the
//      record slices (16 rows, one bulk TMA copy each) streamed through a four-stage shared-memory ring as BOTH operands (MN-major A and B), fp32
//      accumulators for all three products resident in TMEM (416 + 64 + 32 = 512 columns), bf16x3 products.  The bias
//      gradients are the constant-1 column of h1 / h2 / [g 1] (ldeq_mlp_tc.cuh: the padded bias entry is 1).
//  mlp_tc_wgrad_reduce_kernel sums the per-CTA partials into Flux.destructure order.
#include "ldeq_mlp_tc.cuh"

namespace ldeq {

// ---- record geometry ------------------------------------------------------------------------------------------------
// One block = the operands of one (tile, step, stage): 128 rows (the reduction dimension of the weight gradient), stored as
// 8 SLICES of 16 rows; a slice is one pipeline stage of the weight-gradient kernel and is contiguous in memory, so that a
// stage is ONE bulk copy.  Inside a slice every operand ("part") of F features holds its two 8-row groups as
//   [2 row groups][F/8 chunks][8 rows] x 16 bytes: element (feature f, row r) at ((r/8)%2) * (F/8)*128 + (f/8)*128 + (r%8)*16 + (f%8)*2
// -- the MN-major no-swizzle canonical layout (LBO = (F/8)*128 between row groups, SBO = 128 between feature chunks).
struct TcRec {
    int nch1, nch2;                     // 16-byte chunks per row of an n1- / n2-wide part
    // byte offsets of the parts inside a slice (A operands whose second M-tile reads past their own part come first)
    unsigned o_z2h, o_z2l, o_z1h, o_z1l, o_h2h, o_h2l, o_h1h, o_h1l, o_gh, o_gl, o_dh, o_dl;
    unsigned slice_bytes, block_bytes;
    int nsteps;                         // step slots per tile (largest accepted-step count of the batch)
};
#define TC_G_FEATS 32
#define TC_D_FEATS 16
#define TC_SLICE_ROWS 16

// 16 bytes (8 features) of `row` into chunk `chunk` of the part at offset `part_off` of its slice
__device__ __forceinline__ void st_chunk(unsigned char* blk, const TcRec& rec, unsigned part_off, int nch, int row, int chunk, uint32_t a,
                                         uint32_t b, uint32_t c, uint32_t d) {
    *reinterpret_cast<uint4*>(blk + (size_t)(row >> 4) * rec.slice_bytes + part_off + ((size_t)((row >> 3) & 1) * nch + chunk) * 128 +
                              (row & 7) * 16) = make_uint4(a, b, c, d);
}
__device__ __forceinline__ void tc_st4(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tc_ld8(uint32_t taddr, float* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    tc_wait_ld();
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// forward epilogue of a hidden layer + record + relu mask: acc -> h = relu(acc + bias) -> bf16 hi/lo in place, the same
// 16-byte chunks to the record, bit (c - c_lo + i) of `mask` = [h > 0]
__device__ __forceinline__ void adj_epilogue_fwd(uint32_t region, const float* __restrict__ bias, int c_lo, int c_hi, int row,
                                                 unsigned char* blk, const TcRec& rec, unsigned o_hi, unsigned o_lo, int nch, uint32_t* mask) {
#pragma unroll 1
    for (int c = c_lo; c < c_hi; c += 16) {
        float v[16];
        uint32_t hi[8], lo[8];
        tc_ld16(region + c, v);
        uint32_t m = 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            v[i] = fmaxf(v[i] + bias[c + i], 0.f);
            m |= (v[i] > 0.f ? 1u : 0u) << i;
        }
        const int w = (c - c_lo) >> 4;
        mask[w >> 1] = (w & 1) ? (mask[w >> 1] | (m << 16)) : m;
        split_pack16(v, hi, lo);
        tc_st8(region + c, hi);
        tc_st8(region + c + 8, lo);
        st_chunk(blk, rec, o_hi, nch, row, c >> 3, hi[0], hi[1], hi[2], hi[3]);
        st_chunk(blk, rec, o_hi, nch, row, (c >> 3) + 1, hi[4], hi[5], hi[6], hi[7]);
        st_chunk(blk, rec, o_lo, nch, row, c >> 3, lo[0], lo[1], lo[2], lo[3]);
        st_chunk(blk, rec, o_lo, nch, row, (c >> 3) + 1, lo[4], lo[5], lo[6], lo[7]);
    }
}
// reverse epilogue: acc -> dz = acc .* mask -> bf16 hi/lo in place + record
__device__ __forceinline__ void adj_epilogue_bwd(uint32_t region, int c_lo, int c_hi, int row, unsigned char* blk, const TcRec& rec,
                                                 unsigned o_hi, unsigned o_lo, int nch, const uint32_t* mask) {
#pragma unroll 1
    for (int c = c_lo; c < c_hi; c += 16) {
        float v[16];
        uint32_t hi[8], lo[8];
        tc_ld16(region + c, v);
        const int w = (c - c_lo) >> 4;
        const uint32_t m = (w & 1) ? (mask[w >> 1] >> 16) : (mask[w >> 1] & 0xFFFFu);
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = ((m >> i) & 1u) ? v[i] : 0.f;
        split_pack16(v, hi, lo);
        tc_st8(region + c, hi);
        tc_st8(region + c + 8, lo);
        st_chunk(blk, rec, o_hi, nch, row, c >> 3, hi[0], hi[1], hi[2], hi[3]);
        st_chunk(blk, rec, o_hi, nch, row, (c >> 3) + 1, hi[4], hi[5], hi[6], hi[7]);
        st_chunk(blk, rec, o_lo, nch, row, c >> 3, lo[0], lo[1], lo[2], lo[3]);
        st_chunk(blk, rec, o_lo, nch, row, (c >> 3) + 1, lo[4], lo[5], lo[6], lo[7]);
    }
}

// ---- the adjoint sweep -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TC_THREADS, 1)
mlp_tc_adj_kernel(TcNet net, const unsigned char* __restrict__ img_global, const double* __restrict__ tg, int B, int T,
                  const float* __restrict__ dtraj, MlpTapeViewTc<float> tape, const int* __restrict__ retcode,
                  const int* __restrict__ naccept, float* __restrict__ dz0, TcRec rec, unsigned char* __restrict__ records,
                  int* __restrict__ tile_nsteps) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t mbar[4];  // [0] first column half, [1] second column half, [2] narrow output, [3] weight images (TMA)
    __shared__ uint32_t tmem_base_s;
    __shared__ int nmax_s;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int quad = warp & 3, hf = warp >> 2;
    const int row = quad * 32 + (tid & 31);
    const int D = net.d;
    const int c0 = hf * 8;  // the state components this thread keeps the adjoint bookkeeping of
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
    mbar_wait(&mbar[3], 0);
    const float* bias1 = reinterpret_cast<const float*>(smem + net.bias_off);
    const float* bias2 = bias1 + net.n1;
    const float* bias3 = bias2 + net.n2;
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    const uint32_t R0 = lane_addr + TC_COL_R0, R1 = lane_addr + TC_COL_R1, KS = lane_addr + TC_COL_K;
    uint32_t par_half = 0, par_out = 0;
    const uint32_t lbo1 = (net.n1 / 8) * 128, lbo2 = (net.n2 / 8) * 128, lbo3 = (16 / 8) * 128;
    const uint32_t sbase = smem_u32(smem);
    const int n1a = ((net.n1 / 16 + 1) / 2) * 16, n2a = ((net.n2 / 16 + 1) / 2) * 16;
    const int c1_lo = hf ? n1a : 0, c1_hi = hf ? net.n1 : n1a, c2_lo = hf ? n2a : 0, c2_hi = hf ? net.n2 : n2a;
    const double tend = tg[T - 1];
    const int ntiles = (B + TC_ROWS - 1) / TC_ROWS;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b = tile * TC_ROWS + row;
        const bool live = b < B;
        const int bb = live ? b : B - 1;
        const int na_row = (live && retcode[bb] == RET_SUCCESS && naccept[bb] <= tape.cap) ? naccept[bb] : 0;
        if (tid == 0) nmax_s = 0;
        __syncthreads();
        if (na_row > 0) atomicMax(&nmax_s, na_row);
        __syncthreads();
        const int nmax = nmax_s;
        if (tid == 0) tile_nsteps[tile] = nmax;
        float ubn[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) ubn[i] = 0.f;
        int ks = T - 1;
        double tnext = tend;
        uint32_t m1[7][4], m2[7][4];  // relu masks of this thread's column half, per stage (local memory: indexed by stage)

        for (int n = nmax - 1; n >= 0; --n) {
            const bool valid = n < na_row;
            unsigned char* blk0 = records + ((size_t)tile * rec.nsteps + n) * 7 * rec.block_bytes;
            double tn = 0.0, dtn = 1.0;
            float u[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) u[i] = 0.f;
            if (valid) {
                const size_t r = (size_t)n * B + b;
                tn = tape.t[r];
                dtn = tape.dt[r];
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (i < D) u[i] = tape.u[r * D + i];
            }
            const float h = (float)dtn;
            // ---- cotangents of the save points in (t_n, t_{n+1}] (this thread's 8 components) ----
            float kbar[7][8], ub[8];
            {
                float cb[4][8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { cb[0][i] = cb[1][i] = cb[2][i] = cb[3][i] = 0.f; ub[i] = 0.f; }
                if (valid) {
                    const double inv = 1.0 / dtn;
                    while (ks >= 1 && tg[ks] > tn) {
                        const double ts = tg[ks];
                        float d[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) d[i] = (c0 + i < D) ? dtraj[((size_t)ks * B + b) * D + c0 + i] : 0.f;
                        if (ts == tnext) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) ubn[i] += d[i];
                        } else {
                            const float th = (float)((ts - tn) * inv);
                            const float w1 = h * th, w2 = w1 * th, w3 = w2 * th, w4 = w3 * th;
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                cb[0][i] = fmaf(w1, d[i], cb[0][i]);
                                cb[1][i] = fmaf(w2, d[i], cb[1][i]);
                                cb[2][i] = fmaf(w3, d[i], cb[2][i]);
                                cb[3][i] = fmaf(w4, d[i], cb[3][i]);
                                ub[i] += d[i];
                            }
                        }
                        --ks;
                    }
                }
                // adjoint of the Horner coefficients c_m = sum_j r_jm k_j
#pragma unroll
                for (int j = 0; j < 7; ++j)
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        kbar[j][i] = fmaf(c_r[j][3], cb[3][i], fmaf(c_r[j][2], cb[2][i], fmaf(c_r[j][1], cb[1][i], j == 0 ? cb[0][i] : 0.f)));
            }

            // ---- (F) recompute the stage inputs, hidden activations and slopes of this step -------------------------------
#pragma unroll 1
            for (int st = 0; st < 7; ++st) {
                unsigned char* blk = blk0 + (size_t)st * rec.block_bytes;
                float g[16];
                if (st == 0) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) g[i] = u[i];
                } else {
                    float acc[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
                    for (int q = 0; q < st; ++q) {
                        float kq[16];
                        tc_ld16(KS + 16 * q, kq);
                        const float a = c_a[st][q];
#pragma unroll
                        for (int i = 0; i < 16; ++i) acc[i] = fmaf(a, kq[i], acc[i]);
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) g[i] = valid ? fmaf(h, acc[i], u[i]) : 0.f;
                }
                {
                    uint32_t hi[8], lo[8];
                    split_pack16(g, hi, lo);
                    tc_st8(R1, hi);
                    tc_st8(R1 + 8, lo);
                    tc_wait_st();
                    if (hf == 0) {  // [g 1]: 16 state features, the constant 1, zero padding
                        st_chunk(blk, rec, rec.o_gh, TC_G_FEATS / 8, row, 0, hi[0], hi[1], hi[2], hi[3]);
                        st_chunk(blk, rec, rec.o_gh, TC_G_FEATS / 8, row, 1, hi[4], hi[5], hi[6], hi[7]);
                        st_chunk(blk, rec, rec.o_gh, TC_G_FEATS / 8, row, 2, 0x00003F80u, 0u, 0u, 0u);  // bf16(1.0) in feature 16
                        st_chunk(blk, rec, rec.o_gh, TC_G_FEATS / 8, row, 3, 0u, 0u, 0u, 0u);
                        st_chunk(blk, rec, rec.o_gl, TC_G_FEATS / 8, row, 0, lo[0], lo[1], lo[2], lo[3]);
                        st_chunk(blk, rec, rec.o_gl, TC_G_FEATS / 8, row, 1, lo[4], lo[5], lo[6], lo[7]);
                        st_chunk(blk, rec, rec.o_gl, TC_G_FEATS / 8, row, 2, 0u, 0u, 0u, 0u);
                        st_chunk(blk, rec, rec.o_gl, TC_G_FEATS / 8, row, 3, 0u, 0u, 0u, 0u);
                    }
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
                adj_epilogue_fwd(R0, bias1, c1_lo, c1_hi, row, blk, rec, rec.o_h1h, rec.o_h1l, rec.nch1, m1[st]);
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
                adj_epilogue_fwd(R1, bias2, c2_lo, c2_hi, row, blk, rec, rec.o_h2h, rec.o_h2l, rec.nch2, m2[st]);
                tc_wait_st();
                tc_fence_before();
                __syncthreads();
                if (st < 6) {  // the slope k_{st+1}; k7 = f(u_{n+1}) itself is not needed by the adjoint
                    if (tid == 0) {
                        tc_fence_after();
                        tc_issue_layer(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, sbase + net.img_off[4], sbase + net.img_off[5], lbo3, 0, 16,
                                       net.n2 / 16);
                        tc_commit(&mbar[2]);
                    }
                    mbar_wait(&mbar[2], par_out);
                    par_out ^= 1;
                    tc_fence_after();
                    float kout[16];
                    tc_ld16(R0, kout);
#pragma unroll
                    for (int i = 0; i < 16; ++i) kout[i] = i < D ? kout[i] + bias3[i] : 0.f;
                    tc_st16(KS + 16 * st, kout);
                    tc_wait_st();
                }
            }

            // ---- (R) reverse sweep through the stages: three transposed products per stage -----------------------------------
#pragma unroll 1
            for (int st = 6; st >= 0; --st) {
                unsigned char* blk = blk0 + (size_t)st * rec.block_bytes;
                {   // kbar_{st+1} (this thread's 8 components) -> A operand R1[0:16) (hi: columns 0-7, lo: 8-15) + record
                    float d3[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) d3[i] = valid ? kbar[st][i] : 0.f;
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t hh = pack_bf16x2(d3[2 * j], d3[2 * j + 1]);
                        hi[j] = hh;
                        lo[j] = pack_bf16x2(d3[2 * j] - __uint_as_float(hh << 16), d3[2 * j + 1] - __uint_as_float(hh & 0xFFFF0000u));
                    }
                    tc_st4(R1 + hf * 4, hi);
                    tc_st4(R1 + 8 + hf * 4, lo);
                    tc_wait_st();
                    st_chunk(blk, rec, rec.o_dh, TC_D_FEATS / 8, row, hf, hi[0], hi[1], hi[2], hi[3]);
                    st_chunk(blk, rec, rec.o_dl, TC_D_FEATS / 8, row, hf, lo[0], lo[1], lo[2], lo[3]);
                }
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {  // dz2_pre = kbar W3 : N' = n2, K' = 16, image of layer 3 transposed
                    tc_fence_after();
                    const uint32_t wh = sbase + net.img_off[4], wl = sbase + net.img_off[5];
                    tc_issue_layer_T(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, wh, wl, lbo3, 0, n2a, 1);
                    tc_commit(&mbar[0]);
                    tc_issue_layer_T(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, wh, wl, lbo3, n2a, net.n2 - n2a, 1);
                    tc_commit(&mbar[1]);
                }
                mbar_wait(&mbar[hf], par_half);
                par_half ^= 1;
                tc_fence_after();
                adj_epilogue_bwd(R0, c2_lo, c2_hi, row, blk, rec, rec.o_z2h, rec.o_z2l, rec.nch2, m2[st]);
                tc_wait_st();
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {  // dz1_pre = dz2 W2 : N' = n1, K' = n2
                    tc_fence_after();
                    const uint32_t wh = sbase + net.img_off[2], wl = sbase + net.img_off[3];
                    tc_issue_layer_T(tmem_base + TC_COL_R1, tmem_base + TC_COL_R0, wh, wl, lbo2, 0, n1a, net.n2 / 16);
                    tc_commit(&mbar[0]);
                    tc_issue_layer_T(tmem_base + TC_COL_R1, tmem_base + TC_COL_R0, wh, wl, lbo2, n1a, net.n1 - n1a, net.n2 / 16);
                    tc_commit(&mbar[1]);
                }
                mbar_wait(&mbar[hf], par_half);
                par_half ^= 1;
                tc_fence_after();
                adj_epilogue_bwd(R1, c1_lo, c1_hi, row, blk, rec, rec.o_z1h, rec.o_z1l, rec.nch1, m1[st]);
                tc_wait_st();
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {  // gbar = dz1 W1 : N' = 16, K' = n1
                    tc_fence_after();
                    tc_issue_layer_T(tmem_base + TC_COL_R0, tmem_base + TC_COL_R1, sbase + net.img_off[0], sbase + net.img_off[1], lbo1, 0, 16,
                                     net.n1 / 16);
                    tc_commit(&mbar[2]);
                }
                mbar_wait(&mbar[2], par_out);
                par_out ^= 1;
                tc_fence_after();
                float gb[8];
                tc_ld8(R0 + c0, gb);
#pragma unroll
                for (int i = 0; i < 8; ++i) gb[i] = (valid && c0 + i < D) ? gb[i] : 0.f;
                // Tsit5 adjoint bookkeeping (stage st+1; mirrors tsit5_bwd_body of ldeq_tsit5.cuh)
                if (st == 6) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        ubn[i] += gb[i];
                        const float v = h * ubn[i];
                        ub[i] += ubn[i];
#pragma unroll
                        for (int q = 0; q < 6; ++q) kbar[q][i] = fmaf(c_a[6][q], v, kbar[q][i]);
                    }
                } else if (st > 0) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float v = h * gb[i];
                        ub[i] += gb[i];
#pragma unroll
                        for (int q = 0; q < 5; ++q)
                            if (q < st) kbar[q][i] = fmaf(c_a[st][q], v, kbar[q][i]);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) ub[i] += gb[i];
                }
                // the next stage overwrites R1[0:16) and reads R0: everybody must be done with this stage's TMEM reads
                tc_fence_before();
                __syncthreads();
                tc_fence_after();
            }
            if (valid) {
#pragma unroll
                for (int i = 0; i < 8; ++i) ubn[i] = ub[i];
                tnext = tn;
            }
        }
        if (live) {
            const bool ok = retcode[b] == RET_SUCCESS;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (c0 + i < D) dz0[(size_t)b * D + c0 + i] = ok ? ubn[i] + dtraj[(size_t)b * D + c0 + i] : 0.f;
        }
        __syncthreads();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC_TMEM_COLS));
}

// ---- the weight-gradient GEMM over the records ------------------------------------------------------------------------
#define WG_THREADS 192       // warp 0: TMA producer, warp 1: MMA issuer, warps 2-5: epilogue (TMEM lane quadrants 2,3,0,1)
#define WG_ROWS 16           // rows (K of the GEMM) per pipeline stage: one MMA K-step, an eighth of a record block
#define WG_STAGES 4          // 4 x 56 kB: deep enough to keep the TMA loads ahead of the MMAs (2 x 112 kB ran at 2 TB/s)
// TMEM columns: dW2 [0, 416): M-tile 0 -> [0, n1), M-tile 1 -> [208, 208 + n1);  dW1 [416, 480): 2 x 32;  dW3^T [480, 512): 2 x 16

__device__ __forceinline__ void tc_mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[128 x N] (+)= A^T B over WG_ROWS rows, A = features [m0, m0+128) of an MN-major part, B = N features of another, bf16x3
__device__ __forceinline__ void wg_issue(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t ga, int m0, uint32_t b_hi, uint32_t b_lo,
                                         uint32_t gb, int n, bool first) {
    const uint32_t idesc = make_idesc_mn(n, 1, 1);
    const uint32_t aoff = (uint32_t)(m0 / 8) * 128;
#pragma unroll
    for (int kk = 0; kk < WG_ROWS / 16; ++kk) {
        const uint64_t ah = make_smem_desc(a_hi + aoff + kk * 2 * ga, ga, 128), al = make_smem_desc(a_lo + aoff + kk * 2 * ga, ga, 128);
        const uint64_t bh = make_smem_desc(b_hi + kk * 2 * gb, gb, 128), bl = make_smem_desc(b_lo + kk * 2 * gb, gb, 128);
        tc_mma_ss(d_tmem, ah, bh, idesc, (first && kk == 0) ? 0u : 1u);
        tc_mma_ss(d_tmem, ah, bl, idesc, 1u);
        tc_mma_ss(d_tmem, al, bh, idesc, 1u);
    }
}

__global__ void __launch_bounds__(WG_THREADS, 1)
mlp_tc_wgrad_kernel(TcNet net, TcRec rec, const unsigned char* __restrict__ records, const int* __restrict__ tile_nsteps,
                    int ntiles, float* __restrict__ partials /* [grid][n2*n1 + n1*32 + n2*16] */) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full_bar[WG_STAGES], empty_bar[WG_STAGES], done_bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < WG_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(&done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TC_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    // the tail a second M-tile reads past the last part of the last stage must be finite: zero the slack once
    for (int i = tid; i < 1024 / 16; i += WG_THREADS) reinterpret_cast<uint4*>(smem + (size_t)WG_STAGES * rec.slice_bytes)[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t g1 = (uint32_t)rec.nch1 * 128, g2 = (uint32_t)rec.nch2 * 128, gg = (TC_G_FEATS / 8) * 128, gd = (TC_D_FEATS / 8) * 128;
    const int quarters = TC_ROWS / WG_ROWS;

    // items of this CTA: (tile, step, stage, quarter), blocks dealt round-robin over the grid
    if (warp == 0) {
        // ===== TMA producer: the whole warp.  One bulk copy is served as a single stream (a 56 kB copy per stage ran at
        // 2.1 TB/s, twelve smaller ones at 2.6 TB/s): every lane issues 1/32 of the slice, 32 copies in flight per stage =====
        int it = 0;
        unsigned base = 0;  // linear index of this tile's first block, modulo the grid
        const uint32_t piece = rec.slice_bytes / 32;   // the slice size is a multiple of 512 bytes
        for (int tile = 0; tile < ntiles; ++tile) {
            const unsigned nb = (unsigned)tile_nsteps[tile] * 7u;   // blocks of this tile: (step, stage) pairs
            // blocks are dealt round-robin over the grid: this CTA owns those with (base + j) % grid == blockIdx.x
            for (unsigned j = (blockIdx.x + gridDim.x - base) % gridDim.x; j < nb; j += gridDim.x) {
                const unsigned char* blk = records + ((size_t)tile * rec.nsteps * 7 + j) * rec.block_bytes;
                for (int q = 0; q < quarters; ++q, ++it) {
                    const int s = it % WG_STAGES;
                    const uint32_t ph = (uint32_t)((it / WG_STAGES) & 1);
                    if (lane == 0) {
                        mbar_wait(&empty_bar[s], ph ^ 1);
                        mbar_expect_tx(&full_bar[s], rec.slice_bytes);
                    }
                    __syncwarp();
                    bulk_g2s(smem + (size_t)s * rec.slice_bytes + lane * piece, blk + (size_t)q * rec.slice_bytes + lane * piece, piece,
                             &full_bar[s]);
                }
            }
            base = (base + nb) % gridDim.x;
        }
    } else if (warp == 1 && lane == 0) {
        // ===== MMA issuer =====
        int it = 0;
        unsigned base = 0;
        for (int tile = 0; tile < ntiles; ++tile) {
            const unsigned nb = (unsigned)tile_nsteps[tile] * 7u;
            for (unsigned j = (blockIdx.x + gridDim.x - base) % gridDim.x; j < nb; j += gridDim.x) {
                for (int q = 0; q < quarters; ++q, ++it) {
                    const int s = it % WG_STAGES;
                    const uint32_t ph = (uint32_t)((it / WG_STAGES) & 1);
                    mbar_wait(&full_bar[s], ph);
                    tc_fence_after();
                    const uint32_t base_s = smem_u32(smem + (size_t)s * rec.slice_bytes);
                    const bool first = it == 0;
                    for (int mt = 0; mt < 2; ++mt) {
                        // dW2[n2 feature, n1 feature] += dz2^T h1
                        wg_issue(tmem_base + mt * TC_MAXW, base_s + rec.o_z2h, base_s + rec.o_z2l, g2, mt * 128, base_s + rec.o_h1h, base_s + rec.o_h1l, g1, net.n1, first);
                        // dW1[n1 feature, g feature | 1] += dz1^T [g 1]
                        wg_issue(tmem_base + 416 + mt * TC_G_FEATS, base_s + rec.o_z1h, base_s + rec.o_z1l, g1, mt * 128, base_s + rec.o_gh, base_s + rec.o_gl, gg, TC_G_FEATS, first);
                        // dW3^T[n2 feature | 1, state component] += h2^T kbar
                        wg_issue(tmem_base + 480 + mt * TC_D_FEATS, base_s + rec.o_h2h, base_s + rec.o_h2l, g2, mt * 128, base_s + rec.o_dh, base_s + rec.o_dl, gd, TC_D_FEATS, first);
                    }
                    tc_commit(&empty_bar[s]);  // frees the stage once these MMAs have read it
                }
            }
            base = (base + nb) % gridDim.x;
        }
        tc_commit(&done_bar);
        if (it == 0) {  // no work for this CTA: nothing was accumulated
            // (the epilogue below writes zeros in that case)
        }
    }
    // ===== epilogue: accumulators -> this CTA's partial gradient =====
    // does this CTA own any block at all?  (same enumeration, cheap)
    unsigned nblocks = 0;
    for (int tile = 0; tile < ntiles && nblocks <= blockIdx.x; ++tile) nblocks += (unsigned)tile_nsteps[tile] * 7u;
    const bool has_work = nblocks > blockIdx.x;
    if (warp >= 2) {
        if (has_work) {
            mbar_wait(&done_bar, 0);
            tc_fence_after();
        }
        const int quad = warp & 3;  // TMEM lane quadrant this warp may access
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
        float* P2 = partials + (size_t)blockIdx.x * ((size_t)net.n2 * net.n1 + (size_t)net.n1 * TC_G_FEATS + (size_t)net.n2 * TC_D_FEATS);
        float* P1 = P2 + (size_t)net.n2 * net.n1;
        float* P3 = P1 + (size_t)net.n1 * TC_G_FEATS;
        for (int mt = 0; mt < 2; ++mt) {
            const int m = mt * 128 + quad * 32 + lane;  // feature index = TMEM lane
            for (int c = 0; c < net.n1; c += 16) {
                float v[16];
                if (has_work) tc_ld16(lane_addr + mt * TC_MAXW + c, v);
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (m < net.n2) P2[(size_t)m * net.n1 + c + i] = has_work ? v[i] : 0.f;
            }
            for (int c = 0; c < TC_G_FEATS; c += 16) {
                float v[16];
                if (has_work) tc_ld16(lane_addr + 416 + mt * TC_G_FEATS + c, v);
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (m < net.n1) P1[(size_t)m * TC_G_FEATS + c + i] = has_work ? v[i] : 0.f;
            }
            {
                float v[16];
                if (has_work) tc_ld16(lane_addr + 480 + mt * TC_D_FEATS, v);
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (m < net.n2) P3[(size_t)m * TC_D_FEATS + i] = has_work ? v[i] : 0.f;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC_TMEM_COLS));
}

// partials [grid][P2 | P1 | P3] -> dparams in Flux.destructure order (per layer vec(W) column-major with W (out, in), then b)
__global__ void mlp_tc_wgrad_reduce_kernel(TcNet net, int D, int H1, int H2, const float* __restrict__ partials, int nparts,
                                           float* __restrict__ dparams) {
    const size_t stride = (size_t)net.n2 * net.n1 + (size_t)net.n1 * TC_G_FEATS + (size_t)net.n2 * TC_D_FEATS;
    const int o1 = 0, ob1 = H1 * D, o2 = ob1 + H1, ob2 = o2 + H2 * H1, o3 = ob2 + H2, ob3 = o3 + D * H2, total = ob3 + D;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        size_t src;
        if (i < ob1) { const int k = (i - o1) / H1, n = (i - o1) % H1; src = (size_t)net.n2 * net.n1 + (size_t)n * TC_G_FEATS + k; }              // dW1[n, k]
        else if (i < o2) { const int n = i - ob1; src = (size_t)net.n2 * net.n1 + (size_t)n * TC_G_FEATS + 16; }                                  // db1[n]: the 1 of [g 1]
        else if (i < ob2) { const int k = (i - o2) / H2, n = (i - o2) % H2; src = (size_t)n * net.n1 + k; }                                       // dW2[n, k]
        else if (i < o3) { const int n = i - ob2; src = (size_t)n * net.n1 + H1; }                                                                // db2[n]: h1's constant-1 column
        else if (i < ob3) { const int k = (i - o3) / D, d = (i - o3) % D; src = (size_t)net.n2 * net.n1 + (size_t)net.n1 * TC_G_FEATS + (size_t)k * TC_D_FEATS + d; }  // dW3[d, k]
        else { const int d = i - ob3; src = (size_t)net.n2 * net.n1 + (size_t)net.n1 * TC_G_FEATS + (size_t)H2 * TC_D_FEATS + d; }                // db3[d]: h2's constant-1 row
        float s = 0.f;
        for (int p = 0; p < nparts; ++p) s += partials[(size_t)p * stride + src];
        dparams[i] = s;
    }
}

}  // namespace ldeq

using namespace ldeq;

// Host side: called from ldeq_mlp_solve_bwd for a tape recorded with LDEQ_MLP_MATH_BF16X3.  `max_na` = largest accepted-step
// count of a successful trajectory (known to the caller from the forward pass).
int ldeq_mlp_tc_backward(ldeq_handle* h, const int32_t* dims, int n_layers, const float* params, const double* d_tgrid, int B, int T,
                         const float* dtraj, double* tape_t, double* tape_dt, float* tape_u, int tape_cap, const int32_t* ret,
                         const int32_t* na, int max_na, float* dz0, float* dparams, cudaStream_t s) {
    TcNet net;
    int rc = ldeq_tc_make_net(h, dims, n_layers, &net);
    if (rc) return rc;
    const int D = dims[0], H1 = dims[1], H2 = dims[2];
    const int tiles = (B + TC_ROWS - 1) / TC_ROWS;
    TcRec rec;
    rec.nch1 = net.n1 / 8; rec.nch2 = net.n2 / 8;
    {
        const unsigned q1 = 2u * rec.nch1 * 128, q2 = 2u * rec.nch2 * 128, qg = 2u * (TC_G_FEATS / 8) * 128, qd = 2u * (TC_D_FEATS / 8) * 128;
        unsigned o = 0;
        rec.o_z2h = o; o += q2; rec.o_z2l = o; o += q2; rec.o_z1h = o; o += q1; rec.o_z1l = o; o += q1; rec.o_h2h = o; o += q2; rec.o_h2l = o; o += q2;
        rec.o_h1h = o; o += q1; rec.o_h1l = o; o += q1; rec.o_gh = o; o += qg; rec.o_gl = o; o += qg; rec.o_dh = o; o += qd; rec.o_dl = o; o += qd;
        rec.slice_bytes = o;
    }
    rec.block_bytes = (TC_ROWS / TC_SLICE_ROWS) * rec.slice_bytes;
    rec.nsteps = max_na > 0 ? max_na : 1;
    const size_t wg_smem = (size_t)WG_STAGES * rec.slice_bytes + 1024;
    if (wg_smem > 227 * 1024) return set_err(h, LDEQ_ERR_UNSUPPORTED, "bf16x3 tensor-core reverse pass: record tiles do not fit in shared memory");
    const size_t rec_bytes = (size_t)tiles * rec.nsteps * 7 * rec.block_bytes;
    const int wg_grid = h->sm_count;
    const size_t part_floats = (size_t)net.n2 * net.n1 + (size_t)net.n1 * TC_G_FEATS + (size_t)net.n2 * TC_D_FEATS;
    // scratch: [2] weight images, [1] records + tile step counts, [3] per-CTA partial gradients
    if ((rc = ensure_scratch(h, 2, (size_t)net.smem_bytes, s))) return rc;
    if ((rc = ensure_scratch(h, 1, rec_bytes + (size_t)tiles * sizeof(int) + 256, s))) return rc;
    if ((rc = ensure_scratch(h, 3, (size_t)wg_grid * part_floats * sizeof(float), s))) return rc;
    unsigned char* img = (unsigned char*)h->scratch[2];
    unsigned char* records = (unsigned char*)h->scratch[1];
    int* tile_nsteps = (int*)(records + ((rec_bytes + 255) & ~(size_t)255));
    float* partials = (float*)h->scratch[3];
    mlp_tc_prep_kernel<<<64, 256, 0, s>>>(net, params, D, H1, H2, img);
    LDEQ_CUDA(cudaGetLastError());
    MlpTapeViewTc<float> tv{tape_t, tape_dt, tape_u, tape_cap};
    const int grid = tiles < h->sm_count ? tiles : h->sm_count;
    LDEQ_CUDA(cudaFuncSetAttribute(mlp_tc_adj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, net.smem_bytes));
    mlp_tc_adj_kernel<<<grid, TC_THREADS, net.smem_bytes, s>>>(net, img, d_tgrid, B, T, dtraj, tv, ret, na, dz0, rec, records, tile_nsteps);
    LDEQ_CUDA(cudaGetLastError());
    LDEQ_CUDA(cudaFuncSetAttribute(mlp_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wg_smem));
    mlp_tc_wgrad_kernel<<<wg_grid, WG_THREADS, wg_smem, s>>>(net, rec, records, tile_nsteps, tiles, partials);
    LDEQ_CUDA(cudaGetLastError());
    const int total = H1 * D + H1 + H2 * H1 + H2 + D * H2 + D;
    mlp_tc_wgrad_reduce_kernel<<<(total + 255) / 256, 256, 0, s>>>(net, D, H1, H2, partials, wg_grid, dparams);
    LDEQ_CUDA(cudaGetLastError());
    h->launches += 4;
    return LDEQ_OK;
}
