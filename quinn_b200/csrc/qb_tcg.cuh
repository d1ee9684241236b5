// Tensor-core evaluation of the log-posterior AND its gradient (kernel 2 on tcgen05) for fp32 MLPs
//   in (d <= 7) -> H0 -> H1 -> 1,   H0 == H1 in {32, 64}, tanh or relu on both hidden layers, linear output.
// Reverse mode of nnwrap.py:128-150 (autograd over NegLogPost, losses.py:186-206), restated in oracle/quinn_oracle.py.
//
// One tile = 128 data points = the 128 lanes of tensor memory.  A thread owns one point and one chunk of 16 units
// (G = H/16 thread groups share the points), exactly as in the value path (qb_tc.cuh).  All products are "3xTF32":
// both operands split hi/lo, three MMA passes (lo*hi, hi*lo, hi*hi), fp32 accumulation in tensor memory.
//
// Per tile (P = points on lanes):
//   L0    CUDA cores   a0 = act(W0 x + b0)                       -> tensor memory (A operand) + shared memory (MN-major)
//   FWD   tcgen05      D1[p][j] = sum_i a0[p][i] W1[j][i]         A = a0 (tensor memory), B = W1   (K-major smem)
//   EPI1  CUDA cores   a1 = act(D1 + b1); y = Wl.a1 + bl (partial sums of the G groups meet in shared memory);
//                      dy = (ydata - y)/sigma^2; z1 = dy Wl act'(a1); dWl += dy a1 (registers, reduced once per evaluation)
//                                                                 -> tensor memory (A operand) + shared memory (MN-major)
//   BWD   tcgen05      D0[p][i] = sum_j z1[p][j] W1[j][i]         A = z1 (tensor memory), B = W1^T (K-major smem)
//   DW1   tcgen05      G1[j][i] += sum_p z1[p][j] a0[p][i]        A = z1, B = a0, both MN-major smem, M = 64, K = points;
//   DB1   tcgen05      g1[j][c] += sum_p z1[p][j] X[p][c]         B = X = [x | 1 | 0] K-major smem (column d: db1)
//   EPI0  CUDA cores   z0 = D0 act'(a0)                           -> shared memory (MN-major, over z1)
//   DW0   tcgen05      G0[i][c] += sum_p z0[p][i] X[p][c]         columns < d: dW0, column d: db0
// G1, g1, G0 stay in tensor memory for the whole evaluation and are read once at the end.
//
// Shared-memory operand layouts (established with scripts/tc_probe3.cu, profiles/r2_tc_probe3_layouts.log):
//   * K-major, no swizzle (weights): 128-byte core matrices of 8 rows x 4 k; LBO = 128 (k chunks), SBO = 128*K/4;
//   * MN-major fp32 operands must use SWIZZLE_128B_BASE32B (layout type 1): atom = 4 k-rows (points) x 128 bytes
//     (32 units); inside a row the 32-byte piece index is XORed with the row index; LBO = stride between 32-unit
//     atoms (512), SBO = stride between 4-point atoms.  A point's 16-unit chunk is 64 contiguous bytes up to a swap
//     of its two 32-byte halves: the thread-per-point writer uses 128-bit stores;
//   * X^T (8 rows x 128 points, K-major): written transposed with scalar stores; chunk stride 144 instead of 128 so
//     that the 8 point groups of a warp hit different banks.
//   * an M = 64 accumulator keeps row m in lane (m % 16) + 32 * (m / 16).
#pragma once
#include <stdint.h>
#include "qb_plan.h"
#include "qb_tc.cuh"
#include "qb_tcgen05.cuh"

struct QbTcgPlan {
    int in_dim, ni, n_params;
    int h0, h1, act;
    int G, nthreads;
    int w0_off, b0_off, w1_off, b1_off, wl_off, bl_off;   // offsets in theta (b*_off < 0: no bias)
    int w1hi, w1lo, w1thi, w1tlo;                         // byte offsets: W1 (N=j,K=i) and W1^T (N=i,K=j), K-major
    int a0hi, a0lo, zhi, zlo;                             // byte offsets: MN-major point buffers
    int a0_sbo, z_sbo;                                    // 512 * atoms
    int xt;                                               // byte offset: 2 tiles x (hi 4608 | lo 4608)
    int fl_base, w0, b1, wl, bl;                          // float area (byte offset) and float indices in it
    int ybuf;                                             // byte offset: [G][128] partial outputs
    int c_a0hi, c_a0lo, c_zhi, c_zlo, c_d1, c_d0, c_dw1, c_db1, c_dw0, tmem_cols;
    int smem_bytes;
};

#ifdef __CUDACC__
enum { QB_TCG_BARF = 320, QB_TCG_SLOT = 328, QB_TCG_ABAR = 336, QB_TCG_BARB = 344, QB_TCG_BARW = 352, QB_TCG_BARZ = 360,
       QB_TCG_HDR = 512, QB_TCG_XT_HALF = 4608, QB_TCG_XT_TILE = 9216 };

struct QbTcgCtx { uint32_t tmem, abar, barf, barb, barw, barz, ph; };   // ph: parity bits (0 abar, 1 f, 2 b, 3 w, 4 z)

__device__ __forceinline__ void qb_tcg_init(const QbTcgPlan& tp, unsigned char* smem, QbTcgCtx& cx) {
    const uint32_t bars[5] = {QB_TCG_ABAR, QB_TCG_BARF, QB_TCG_BARB, QB_TCG_BARW, QB_TCG_BARZ};
    const uint32_t counts[5] = {QB_MBAR_BLOCK, 1u, 1u, 1u, 1u};
    cx.tmem = qb_tc_start(smem, QB_TCG_SLOT, (uint32_t)tp.tmem_cols, bars, counts);
    cx.abar = qb_smem_u32(smem + QB_TCG_ABAR);
    cx.barf = qb_smem_u32(smem + QB_TCG_BARF);
    cx.barb = qb_smem_u32(smem + QB_TCG_BARB);
    cx.barw = qb_smem_u32(smem + QB_TCG_BARW);
    cx.barz = qb_smem_u32(smem + QB_TCG_BARZ);
    cx.ph = 0;
}

// flat theta (global) -> shared: layer-0 rows (paired units, bias in slot in_dim), W1 (scaled for tanh) and W1^T (unscaled),
// both split hi/lo in the K-major canonical layout, biases, output layer.  Also clears the X^T buffers once per call.
__device__ __forceinline__ void qb_tcg_stage(const QbTcgPlan& tp, unsigned char* smem, const float* __restrict__ theta) {
    float* F = reinterpret_cast<float*>(smem + tp.fl_base);
    const int tid = threadIdx.x, nt = blockDim.x;
    const float sc = tp.act == QB_ACT_TANH ? 2.8853900817779268f : 1.0f;
    for (int e = tid; e < tp.h0 * tp.ni; e += nt) {
        const int u = e & 1, q = (e >> 1) % tp.ni, j = ((e >> 1) / tp.ni) * 2 + u;
        float v = 0.0f;
        if (q < tp.in_dim) v = theta[tp.w0_off + j * tp.in_dim + q] * sc;
        else if (q == tp.in_dim && tp.b0_off >= 0) v = theta[tp.b0_off + j] * sc;
        F[tp.w0 + e] = v;
    }
    {
        // forward B operand: W1[j][i], rows n = j, k = i
        const int K = tp.h0, N = tp.h1, kc4 = K >> 2;
        float* hi = reinterpret_cast<float*>(smem + tp.w1hi);
        float* lo = reinterpret_cast<float*>(smem + tp.w1lo);
        for (int e = tid; e < N * K; e += nt) {
            const int q = e & 3, r = (e >> 2) & 7, g = e >> 5;
            const int n8 = g / kc4, kc = g - n8 * kc4;
            const float w = theta[tp.w1_off + (n8 * 8 + r) * K + kc * 4 + q] * sc;
            const float h = qb_tf32_hi(w);
            hi[e] = h;
            lo[e] = w - h;
        }
    }
    {
        // backward B operand: W1^T, rows n = i, k = j (unscaled: the chain rule uses the true weights)
        const int K = tp.h1, N = tp.h0, kc4 = K >> 2;
        float* hi = reinterpret_cast<float*>(smem + tp.w1thi);
        float* lo = reinterpret_cast<float*>(smem + tp.w1tlo);
        for (int e = tid; e < N * K; e += nt) {
            const int q = e & 3, r = (e >> 2) & 7, g = e >> 5;
            const int n8 = g / kc4, kc = g - n8 * kc4;
            const int i = n8 * 8 + r, j = kc * 4 + q;
            const float w = theta[tp.w1_off + j * tp.h0 + i];
            const float h = qb_tf32_hi(w);
            hi[e] = h;
            lo[e] = w - h;
        }
    }
    for (int j = tid; j < tp.h1; j += nt) {
        F[tp.b1 + j] = tp.b1_off >= 0 ? theta[tp.b1_off + j] * sc : 0.0f;
        F[tp.wl + j] = theta[tp.wl_off + j];
    }
    if (tid == 0) F[tp.bl] = tp.bl_off >= 0 ? theta[tp.bl_off] : 0.0f;
    qb_fence_proxy_async();
}

template <int ACT> __device__ __forceinline__ float qb_tcg_dact(float a) {
    if (ACT == QB_ACT_TANH) return fmaf(-a, a, 1.0f);
    return a > 0.0f ? 1.0f : 0.0f;
}

// byte offset (inside an MN-major point buffer) of the 32-byte piece `q` (units 8q .. 8q+7 of the 32-unit atom `atom`) of
// point pt; sbo = 512 * atoms
__device__ __forceinline__ uint32_t qb_tcg_piece(uint32_t pt, uint32_t atom, uint32_t q, uint32_t sbo) {
    const uint32_t r = pt & 3u;
    return (pt >> 2) * sbo + atom * 512u + r * 128u + ((q ^ r) << 5);
}
// split 16 values (units c .. c+15 of this thread's point) and store them into the MN-major buffers
__device__ __forceinline__ void qb_tcg_store_mn(unsigned char* bhi, unsigned char* blo, uint32_t pt, int c, uint32_t sbo,
                                                const float (&h)[16]) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int u0 = c + 8 * half;
        const uint32_t off = qb_tcg_piece(pt, (uint32_t)u0 >> 5, ((uint32_t)u0 >> 3) & 3u, sbo);
        float hh[8], ll[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { hh[i] = qb_tf32_hi(h[8 * half + i]); ll[i] = h[8 * half + i] - hh[i]; }
        float4* ph = reinterpret_cast<float4*>(bhi + off);
        float4* pl = reinterpret_cast<float4*>(blo + off);
        ph[0] = make_float4(hh[0], hh[1], hh[2], hh[3]);
        ph[1] = make_float4(hh[4], hh[5], hh[6], hh[7]);
        pl[0] = make_float4(ll[0], ll[1], ll[2], ll[3]);
        pl[1] = make_float4(ll[4], ll[5], ll[6], ll[7]);
    }
}

// ---- MMA issue (one elected lane of warp 0).  Descriptors are {lo, hi} 32-bit halves; k-steps add a constant to lo.
// A (tensor memory, hi at column ahi_col, lo at alo_col) x B (K-major weights): 3 passes x KS k-steps, then commit
template <int KS>
__device__ __forceinline__ void qb_tcg_issue_ts(uint32_t d, uint32_t ahi_col, uint32_t alo_col, uint32_t bhi_lo, uint32_t blo_lo,
                                                uint32_t b_hi, uint32_t idesc, uint32_t bar) {
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const uint32_t a = (pass == 0 ? alo_col : ahi_col) + 8u * s;
            const uint32_t b = (pass == 1 ? blo_lo : bhi_lo) + 16u * s;
            qb_mma_ts<false>(d, a, b, b_hi, idesc, (pass == 0 && s == 0) ? 0u : 1u);
        }
    }
    qb_commit(bar);
}
// A (smem, MN-major point buffer) x B (smem): 3 passes x 16 k-steps (128 points); `acc0`: accumulate into D from the start
__device__ __forceinline__ void qb_tcg_issue_ss(uint32_t d, uint32_t ahi_lo, uint32_t alo_lo, uint32_t a_hi, uint32_t a_step,
                                                uint32_t bhi_lo, uint32_t blo_lo, uint32_t b_hi, uint32_t b_step, uint32_t idesc,
                                                uint32_t acc0) {
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
        for (int s = 0; s < 16; ++s) {
            const uint32_t a = (pass == 0 ? alo_lo : ahi_lo) + a_step * s;
            const uint32_t b = (pass == 1 ? blo_lo : bhi_lo) + b_step * s;
            qb_mma_ss<false>(d, a, a_hi, b, b_hi, idesc, (pass == 0 && s == 0) ? acc0 : 1u);
        }
    }
}

// everybody: my stores (tensor memory and shared memory) are visible to the tensor core; returns after arriving
__device__ __forceinline__ void qb_tcg_publish(QbTcgCtx& cx) {
    qb_tmem_st_wait();
    qb_fence_proxy_async();
    qb_tc_fence_before();
    qb_mbar_arrive(cx.abar);
}
__device__ __forceinline__ void qb_tcg_wait(uint32_t bar, QbTcgCtx& cx, int bit) {
    qb_mbar_wait_timed(bar, (cx.ph >> bit) & 1u);
    cx.ph ^= 1u << bit;
    qb_tc_fence_after();
}

// Value + gradient of the data term over points [n0, n1) for the staged parameter vector.  Returns the block-wide sum of
// squared residuals; g[0..P) (global, this block's row) receives d/dtheta of -0.5*ssq/sigma^2.
template <int H, int NI, int ACT>
__device__ __forceinline__ double qb_tcg_eval(const QbTcgPlan& tp, QbTcgCtx& cx, unsigned char* smem, const float* __restrict__ x,
                                              const float* __restrict__ y, int64_t n0, int64_t n1, float is2, float* __restrict__ g) {
    constexpr int G = H / 16, KS = H / 8;
    const float* F = reinterpret_cast<const float*>(smem + tp.fl_base);
    float* ybuf = reinterpret_cast<float*>(smem + tp.ybuf);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = warp >> 2, quarter = warp & 3;
    const uint32_t pt = (uint32_t)(quarter * 32 + lane);               // this thread's point of the tile = tensor-memory lane
    const int c = grp * 16;                                            // this thread's chunk of units
    const uint32_t tl = cx.tmem + ((uint32_t)(quarter * 32) << 16);
    const int ntiles = (int)((n1 - n0 + 127) / 128);
    unsigned char* a0hi = smem + tp.a0hi; unsigned char* a0lo = smem + tp.a0lo;
    unsigned char* zhi = smem + tp.zhi;   unsigned char* zlo = smem + tp.zlo;

    // descriptors (warp 0 uses them; cheap to compute everywhere)
    const uint32_t id_base = (1u << 4) | (2u << 7) | (2u << 10);
    const uint32_t id_fwd = id_base | ((uint32_t)(H >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t id_dw1 = id_base | (1u << 15) | (1u << 16) | ((uint32_t)(H >> 3) << 17) | ((64u >> 4) << 24);
    const uint32_t id_dx = id_base | (1u << 15) | (1u << 17) | ((64u >> 4) << 24);            // A MN-major, B = X^T K-major, N = 8
    const uint32_t w_hi = qb_desc_hi(128u * (H / 4), 0u);
    const uint32_t w1hi_lo = qb_desc_lo(qb_smem_u32(smem + tp.w1hi), 128u), w1lo_lo = qb_desc_lo(qb_smem_u32(smem + tp.w1lo), 128u);
    const uint32_t w1thi_lo = qb_desc_lo(qb_smem_u32(smem + tp.w1thi), 128u), w1tlo_lo = qb_desc_lo(qb_smem_u32(smem + tp.w1tlo), 128u);
    const uint32_t a0_hi = qb_desc_hi((uint32_t)tp.a0_sbo, 1u), z_hi = qb_desc_hi((uint32_t)tp.z_sbo, 1u);
    const uint32_t a0hi_lo = qb_desc_lo(qb_smem_u32(a0hi), 512u), a0lo_lo = qb_desc_lo(qb_smem_u32(a0lo), 512u);
    const uint32_t zhi_lo = qb_desc_lo(qb_smem_u32(zhi), 512u), zlo_lo = qb_desc_lo(qb_smem_u32(zlo), 512u);
    const uint32_t a0_step = (2u * (uint32_t)tp.a0_sbo) >> 4, z_step = (2u * (uint32_t)tp.z_sbo) >> 4;
    const uint32_t x_hi = qb_desc_hi(4608u, 0u);

    float dwl[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) dwl[i] = 0.0f;
    float ssq = 0.0f, dbl = 0.0f;
    __syncthreads();               // staged weights visible; the previous evaluation's readers are done

    // Pipeline (two block-wide hand-overs per tile):
    //   phase B(t): wait FWD(t) -> EPI1(t) -> [wait DW0(t-1)] store z1            -> issue BWD(t), DW1(t), DB1(t)
    //   phase A(t): wait BWD(t) -> EPI0(t) and L0(t+1), results parked in tensor memory (the z and a0 OPERAND columns are
    //               free once BWD(t) / FWD(t) are done) while DW1(t) / DB1(t) still read the shared-memory operands
    //               -> wait DW1(t) -> copy z0(t) and a0(t+1) from tensor memory to shared memory -> issue FWD(t+1), DW0(t)
    // so layer 0 of the next tile and the back-propagation epilogue overlap the weight-gradient MMAs.
    // Inputs and target of a point are fetched one tile ahead (one block per SM in lock step: nothing else hides L2 latency).
    float xn[NI], yn = 0.0f;
    auto fetch = [&](int tt) {
        const int64_t pp = n0 + (int64_t)tt * 128 + pt;
#pragma unroll
        for (int q = 0; q < NI; ++q) xn[q] = (q < tp.in_dim && pp < n1) ? __ldg(x + pp * tp.in_dim + q) : 0.0f;
        yn = pp < n1 ? __ldg(y + pp) : 0.0f;
    };
    // layer 0 of tile tt from the prefetched inputs: X^T rows (group 0) to shared memory, a0 to tensor memory
    auto layer0 = [&](int tt) {
        unsigned char* xt = smem + tp.xt + (tt & 1) * QB_TCG_XT_TILE;
        float xr[NI];
#pragma unroll
        for (int q = 0; q < NI; ++q) xr[q] = (q == tp.in_dim) ? 1.0f : xn[q];
        if (grp == 0) {
            // X^T rows q = 0..7 (inputs, then the constant 1, then zeros), element (q, pt): chunk stride 144
            float* xh = reinterpret_cast<float*>(xt + (pt >> 2) * 144u + (pt & 3u) * 4u);
            float* xl = reinterpret_cast<float*>(xt + QB_TCG_XT_HALF + (pt >> 2) * 144u + (pt & 3u) * 4u);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float v = q < NI ? xr[q < NI ? q : 0] : 0.0f;
                const float h = qb_tf32_hi(v);
                xh[q * 4] = h;
                xl[q * 4] = v - h;
            }
        }
        float h[16];
        const float4* W = reinterpret_cast<const float4*>(F + tp.w0 + c * NI);
#pragma unroll
        for (int gq = 0; gq < 4; ++gq) {
            float2 z0 = make_float2(0.0f, 0.0f), z1 = make_float2(0.0f, 0.0f);
#pragma unroll
            for (int q = 0; q < NI; q += 2) {
                const float4 wa = W[(2 * gq) * (NI / 2) + q / 2], wb = W[(2 * gq + 1) * (NI / 2) + q / 2];
                z0 = __ffma2_rn(make_float2(wa.x, wa.y), make_float2(xr[q], xr[q]), z0);
                z0 = __ffma2_rn(make_float2(wa.z, wa.w), make_float2(xr[q + 1], xr[q + 1]), z0);
                z1 = __ffma2_rn(make_float2(wb.x, wb.y), make_float2(xr[q], xr[q]), z1);
                z1 = __ffma2_rn(make_float2(wb.z, wb.w), make_float2(xr[q + 1], xr[q + 1]), z1);
            }
            qb_tc_act4<ACT>(z0, z1);
            h[4 * gq + 0] = z0.x; h[4 * gq + 1] = z0.y; h[4 * gq + 2] = z1.x; h[4 * gq + 3] = z1.y;
        }
        qb_tc_split_store(tl + tp.c_a0hi + c, tl + tp.c_a0lo + c, h);
    };
    // this thread's 16-unit chunk, already split, from tensor memory columns (hi_col, lo_col) to an MN-major point buffer
    auto park_to_smem = [&](uint32_t hi_col, uint32_t lo_col, unsigned char* bhi, unsigned char* blo, uint32_t sbo) {
        uint32_t vh[16], vl[16];
        qb_tmem_ld16(tl + hi_col + c, vh);
        qb_tmem_ld16(tl + lo_col + c, vl);
        qb_tmem_ld_wait16(vh);
        qb_tmem_ld_wait16(vl);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int u0 = c + 8 * half;
            const uint32_t off = qb_tcg_piece(pt, (uint32_t)u0 >> 5, ((uint32_t)u0 >> 3) & 3u, sbo);
            uint4* ph = reinterpret_cast<uint4*>(bhi + off);
            uint4* pl = reinterpret_cast<uint4*>(blo + off);
            ph[0] = make_uint4(vh[8 * half + 0], vh[8 * half + 1], vh[8 * half + 2], vh[8 * half + 3]);
            ph[1] = make_uint4(vh[8 * half + 4], vh[8 * half + 5], vh[8 * half + 6], vh[8 * half + 7]);
            pl[0] = make_uint4(vl[8 * half + 0], vl[8 * half + 1], vl[8 * half + 2], vl[8 * half + 3]);
            pl[1] = make_uint4(vl[8 * half + 4], vl[8 * half + 5], vl[8 * half + 6], vl[8 * half + 7]);
        }
    };

    if (ntiles > 0) {
        fetch(0);
        layer0(0);
        fetch(1);
        qb_tmem_st_wait();
        park_to_smem(tp.c_a0hi, tp.c_a0lo, a0hi, a0lo, (uint32_t)tp.a0_sbo);
        qb_tcg_publish(cx);
        if (warp == 0) {
            qb_mbar_wait_timed(cx.abar, cx.ph & 1u);
            qb_tc_fence_after();
            if (qb_elect())
                qb_tcg_issue_ts<KS>(cx.tmem + tp.c_d1, cx.tmem + tp.c_a0hi, cx.tmem + tp.c_a0lo, w1hi_lo, w1lo_lo, w_hi, id_fwd, cx.barf);
            __syncwarp();
        }
        cx.ph ^= 1u;
    }
    float yv = 0.0f;                                             // target of this thread's point of the current tile
    {
        const int64_t p0 = n0 + pt;
        if (p0 < n1) yv = __ldg(y + p0);
    }
    for (int t = 0; t < ntiles; ++t) {
        const int64_t p = n0 + (int64_t)t * 128 + pt;
        const bool live = p < n1;
        const bool more = t + 1 < ntiles;
        // ---------------- phase B: EPI1(t)
        qb_tcg_wait(cx.barf, cx, 1);
        {
            float a1[16];
            float dy;
            uint32_t v[16];
            qb_tmem_ld16(tl + tp.c_d1 + c, v);
            qb_tmem_ld_wait16(v);
            qb_tc_epi_chunk<ACT>(F + tp.b1, c, v, a1);
            float2 acc = make_float2(0.0f, 0.0f);
            const float4* w4 = reinterpret_cast<const float4*>(F + tp.wl + c);
#pragma unroll
            for (int gq = 0; gq < 4; ++gq) {
                const float4 w = w4[gq];
                acc = __ffma2_rn(make_float2(w.x, w.y), make_float2(a1[4 * gq + 0], a1[4 * gq + 1]), acc);
                acc = __ffma2_rn(make_float2(w.z, w.w), make_float2(a1[4 * gq + 2], a1[4 * gq + 3]), acc);
            }
            ybuf[grp * 128 + pt] = acc.x + acc.y;
            asm volatile("bar.sync %0, %1;" :: "r"(1 + quarter), "r"(32 * G) : "memory");
            float yo = F[tp.bl];
#pragma unroll
            for (int gg = 0; gg < G; ++gg) yo += ybuf[gg * 128 + pt];
            const float r = live ? yv - yo : 0.0f;
            dy = r * is2;
            if (grp == 0) { ssq = fmaf(r, r, ssq); dbl += dy; }
            float z[16];
#pragma unroll
            for (int gq = 0; gq < 4; ++gq) {
                const float4 w = w4[gq];
                const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float a = a1[4 * gq + e];
                    z[4 * gq + e] = dy * wv[e] * qb_tcg_dact<ACT>(a);
                    dwl[4 * gq + e] = fmaf(dy, a, dwl[4 * gq + e]);
                }
            }
            if (t > 0) qb_tcg_wait(cx.barz, cx, 4);            // DW0(t-1) has finished reading the z buffer
            qb_tc_split_store(tl + tp.c_zhi + c, tl + tp.c_zlo + c, z);
            qb_tcg_store_mn(zhi, zlo, pt, c, (uint32_t)tp.z_sbo, z);
        }
        qb_tcg_publish(cx);
        if (warp == 0) {
            qb_mbar_wait_timed(cx.abar, cx.ph & 1u);
            qb_tc_fence_after();
            if (qb_elect()) {
                qb_tcg_issue_ts<KS>(cx.tmem + tp.c_d0, cx.tmem + tp.c_zhi, cx.tmem + tp.c_zlo, w1thi_lo, w1tlo_lo, w_hi, id_fwd, cx.barb);
                const uint32_t acc0 = t > 0 ? 1u : 0u;
                qb_tcg_issue_ss(cx.tmem + tp.c_dw1, zhi_lo, zlo_lo, z_hi, z_step, a0hi_lo, a0lo_lo, a0_hi, a0_step, id_dw1, acc0);
                const uint32_t xs = qb_smem_u32(smem + tp.xt + (t & 1) * QB_TCG_XT_TILE);
                qb_tcg_issue_ss(cx.tmem + tp.c_db1, zhi_lo, zlo_lo, z_hi, z_step, qb_desc_lo(xs, 144u),
                                qb_desc_lo(xs + QB_TCG_XT_HALF, 144u), x_hi, 18u, id_dx, acc0);
                qb_commit(cx.barw);
            }
            __syncwarp();
        }
        cx.ph ^= 1u;
        // ---------------- phase A: EPI0(t) and L0(t+1), parked in tensor memory while DW1(t) / DB1(t) run
        qb_tcg_wait(cx.barb, cx, 2);
        {
            float z[16];
            uint32_t v[16], ah[16], al[16];
            qb_tmem_ld16(tl + tp.c_d0 + c, v);
            qb_tmem_ld16(tl + tp.c_a0hi + c, ah);
            qb_tmem_ld16(tl + tp.c_a0lo + c, al);
            qb_tmem_ld_wait16(v);
            qb_tmem_ld_wait16(ah);
            qb_tmem_ld_wait16(al);
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const float a = __uint_as_float(ah[e]) + __uint_as_float(al[e]);
                z[e] = __uint_as_float(v[e]) * qb_tcg_dact<ACT>(a);
            }
            qb_tc_split_store(tl + tp.c_zhi + c, tl + tp.c_zlo + c, z);      // BWD(t) is done: the z operand columns are free
        }
        if (more) {
            yv = yn;
            layer0(t + 1);                                       // FWD(t) is done and a0(t) was consumed above
            fetch(t + 2);
        }
        qb_tmem_st_wait();
        qb_tcg_wait(cx.barw, cx, 3);                             // DW1 / DB1 have finished reading the z and a0 buffers
        park_to_smem(tp.c_zhi, tp.c_zlo, zhi, zlo, (uint32_t)tp.z_sbo);
        if (more) park_to_smem(tp.c_a0hi, tp.c_a0lo, a0hi, a0lo, (uint32_t)tp.a0_sbo);
        qb_tcg_publish(cx);
        if (warp == 0) {
            qb_mbar_wait_timed(cx.abar, cx.ph & 1u);
            qb_tc_fence_after();
            if (qb_elect()) {
                if (more)
                    qb_tcg_issue_ts<KS>(cx.tmem + tp.c_d1, cx.tmem + tp.c_a0hi, cx.tmem + tp.c_a0lo, w1hi_lo, w1lo_lo, w_hi, id_fwd, cx.barf);
                const uint32_t xs = qb_smem_u32(smem + tp.xt + (t & 1) * QB_TCG_XT_TILE);
                qb_tcg_issue_ss(cx.tmem + tp.c_dw0, zhi_lo, zlo_lo, z_hi, z_step, qb_desc_lo(xs, 144u),
                                qb_desc_lo(xs + QB_TCG_XT_HALF, 144u), x_hi, 18u, id_dx, t > 0 ? 1u : 0u);
                qb_commit(cx.barz);
            }
            __syncwarp();
        }
        cx.ph ^= 1u;
    }
    if (ntiles > 0) qb_tcg_wait(cx.barz, cx, 4);

    // ---------------- gradient out.  Rows of the M = 64 accumulators: lane (m % 16) + 32 * (m / 16).
    const int d = tp.in_dim;
    if (ntiles > 0) {
        const int row = quarter * 16 + lane;                   // valid when lane < 16
        const bool rv = lane < 16 && row < H;
        {
            uint32_t v[16];
            qb_tmem_ld16(tl + tp.c_dw1 + c, v);
            qb_tmem_ld_wait16(v);
            if (rv) {
                float4* dst = reinterpret_cast<float4*>(g + tp.w1_off + row * H + c);
                if ((reinterpret_cast<uintptr_t>(g + tp.w1_off) & 15) == 0) {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        dst[q] = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                                             __uint_as_float(v[4 * q + 3]));
                } else {
#pragma unroll
                    for (int q = 0; q < 16; ++q) g[tp.w1_off + row * H + c + q] = __uint_as_float(v[q]);
                }
            }
        }
        if (grp == 0) {
            uint32_t v[16];
            qb_tmem_ld16(tl + tp.c_db1, v);                    // columns c_db1 .. +8 = DB1, +8 .. +16 = DW0 (adjacent)
            qb_tmem_ld_wait16(v);
            if (rv) {
                if (tp.b1_off >= 0) {
                    float s = 0.0f;
#pragma unroll
                    for (int q = 0; q < 8; ++q) if (q == d) s = __uint_as_float(v[q]);
                    g[tp.b1_off + row] = s;
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (q < d) g[tp.w0_off + row * d + q] = __uint_as_float(v[8 + q]);
                    else if (q == d && tp.b0_off >= 0) g[tp.b0_off + row] = __uint_as_float(v[8 + q]);
                }
            }
        }
    } else {
        for (int i = threadIdx.x; i < tp.n_params; i += blockDim.x) g[i] = 0.0f;
    }
    // dWl[j] = sum over the 128 point slots of the per-thread partial sums (fixed order); the z buffer is free now
    __syncthreads();
    {
        float* scr = reinterpret_cast<float*>(zhi);            // [H][129]
#pragma unroll
        for (int e = 0; e < 16; ++e) scr[(c + e) * 129 + pt] = dwl[e];
        __syncthreads();
        if (threadIdx.x < H) {
            float s = 0.0f;
            for (int q = 0; q < 128; ++q) s += scr[threadIdx.x * 129 + q];
            g[tp.wl_off + threadIdx.x] = s;
        }
    }
    const double sb = qb_block_sum((double)dbl, reinterpret_cast<double*>(smem));
    if (threadIdx.x == 0 && tp.bl_off >= 0) g[tp.bl_off] = (float)sb;
    return qb_block_sum((double)ssq, reinterpret_cast<double*>(smem));
}
#endif  // __CUDACC__
