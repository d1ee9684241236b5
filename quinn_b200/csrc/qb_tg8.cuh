// Tensor-core evaluation of the log-posterior AND its gradient (kernel 2 on tcgen05) for the 128-wide fp32 MLPs
//   in (d <= 15) -> H -> H -> 1, H in {64, 128}, tanh on both hidden layers, linear output
//   (BASELINE configs 3 and 4: 10-128-128-1; config 5 / north_star's HMC target: 3-64-64-1)
// Reverse mode of nnwrap.py:128-150 (autograd over NegLogPost, losses.py:186-206), restated in oracle/quinn_oracle.py.
// qb_tcg.cuh (widths 32 / 64, kind::tf32) does not scale to this width: its four fp32 copies of W1 alone are 256 KB.
//
// Everything here is "3 x FP16": kind::f16 MMAs (K = 16 per instruction) on operands split into fp16 hi + lo
// (a_lo*b_hi + a_hi*b_lo + a_hi*b_hi, fp32 accumulation in tensor memory), with exact power-of-two scaling so that the
// 5-bit exponent never costs accuracy (qb_tc3.cuh uses the same arithmetic for the value path).  kind::f16 does not
// accept an fp16 operand next to a bf16 one (scripts/tc_probe5.cu: illegal instruction), so the back-propagated
// quantities are fp16 as well, scaled by a bound that is known BEFORE the tile loop (see qb_tg8_stage).
//
// One tile = 128 data points = the 128 lanes of tensor memory.  H/8 compute warps: thread = (point, 32 of the H units);
// the warp behind them only issues MMAs.  (H = 64, config 5's net, runs the same code with two blocks per SM.)  Per tile (p = point, i = layer-0 unit, j = layer-1 unit):
//   L0    tcgen05      DL[p][i] = sum_c X[p][c] W0'[i][c]            A = X image = [x | 1 | 0] (K-major view), B = W0 image = [W0 | b0 | 0]
//   EPIL  CUDA cores   a0 = tanh(DL)                                 -> a0 image
//   FWD   tcgen05      D1[p][j] = sum_i a0[p][i] W1[j][i]            A = a0 image (K-major view), B = W image (K-major view)
//   EPI1  CUDA cores   a1 = tanh(D1 + b1); y = wl.a1 + bl; dy = (ydata - y)/sigma^2; z1 = dy wl (1 - a1^2); dwl += dy a1
//                                                                    -> z image
//   BWD   tcgen05      D0[p][i] = sum_j z1[p][j] W1[j][i]            A = z image (K-major view), B = W image (MN-major view)
//   DW1   tcgen05      G1[j][i] += sum_p z1[p][j] a0[p][i]           A = z image, B = a0 image (+ a block of ones: db1), MN-major views
//   EPI0  CUDA cores   z0 = D0 (1 - a0^2)                            -> z image (over z1, once DW1 has read it)
//   DW0   tcgen05      G0[i][c] += sum_p z0[p][i] X[p][c]            A = z image, B = X image = [x | 1 | 0] (column d: db0)
// G1 (128 x 144) and G0 (128 x 16) stay in tensor memory for the whole evaluation.
//
// Shared-memory operands: ONE image per matrix serves both of its uses (scripts/tc_probe5.cu, no swizzle):
//   point image P (a0, z, X):  element (point p, unit u) at (u/8)*2048 + (p/8)*128 + (p%8)*16 + (u%8)*2
//       K-major view  (rows = points, k = units):  LBO 2048 (8-unit chunks),  SBO 128 (8-point groups), k-step +4096
//       MN-major view (rows = units,  k = points): LBO 128 (8-point groups),  SBO 2048 (8-unit chunks), k-step +256
//   weight image W (W1[j][i]): element (j, i) at (j/8)*2048 + (i/8)*128 + (j%8)*16 + (i%8)*2
//       K-major view  (rows = j, k = i):           LBO 128,  SBO 2048, k-step +256
//       MN-major view (rows = i, k = j):           LBO 2048, SBO 128,  k-step +4096
// A thread writes its point's 8-unit chunk with one 16-byte store; the 32 lanes of a warp cover 512 contiguous bytes.
//
// Pipeline (two block-wide hand-overs per tile, as in qb_tcg.cuh); tensor memory: R1 = columns [0,128), R0 = [128,256),
// G1 = [256,400), G0 = [400,416):
//   phase B(t): wait FWD(t) -> EPI1(t), first pass from R1 (a1 waits in R0 across the reduction of y over the thread groups)
//               -> [wait DW0(t-1)] X(t+1) -> X image                                     => issue L0(t+1) -> R1
//               -> second pass: z1 -> z image                                            => issue BWD(t) -> R0, DW1(t)
//   phase A(t): wait L0(t+1) -> EPIL(t+1): R1 -> a0(t+1), packed, back into R1 (under BWD(t)); wait BWD(t) -> EPI0(t): R0 -> z0,
//               packed, back into R0 (under DW1(t), which still reads both images) -> wait DW1(t) -> R1 -> a0 image  => issue FWD(t+1)
//               -> R0 -> z image                                                                                     => issue DW0(t)
//   DW0(t) runs under EPI1(t+1).
#pragma once
#include <stdint.h>
#include "qb_plan.h"
#include "qb_tc.cuh"
#include "qb_tcgen05.cuh"
#include "qb_tg8_plan.h"


#ifdef __CUDACC__
enum { QB_TG8_BAR_F = 400, QB_TG8_BAR_B = 408, QB_TG8_BAR_W = 416, QB_TG8_BAR_Z = 424, QB_TG8_BAR_RDY = 432, QB_TG8_SLOT = 440, QB_TG8_BAR_L = 448, QB_TG8_BAR_RDY2 = 456, QB_TG8_BAR_RDY3 = 464,
       QB_TG8_HDR = 512, QB_TG8_XIMG = 4096 };
// Hidden width H (128: configs 3 / 4, one block per SM; 64: config 5, two blocks per SM): G = H/32 thread groups of 128 compute
// threads (thread = point x 32 units), the issue warp comes after them.  Images of 128 points x H units; tensor-memory
// columns R1 | R0 | G1 (H + 16: the ones block yields db1) | G0 (16)
template <int H> struct QbTg8Dim {
    static constexpr int G = H / 32, NCOMP = 128 * G, ISSUER = 4 * G;
    static constexpr int IMG = 256 * H, AIMG = IMG + 4096, W0IMG = 32 * H, WIMG = 2 * H * H, WSBO = 16 * H;
    static constexpr int C_D1 = 0, C_D0 = H, C_DW1 = 2 * H, C_DW0 = 3 * H + 16;
    static constexpr int CPG = 16 / G;                    // X image columns laid out by one thread group
};
// float slots behind tp.sc
enum { QB_TG8_S_C1 = 0, QB_TG8_S_SZ1 = 1, QB_TG8_S_K0 = 2, QB_TG8_S_UW1 = 3, QB_TG8_S_UW0 = 4, QB_TG8_S_SX = 5, QB_TG8_S_C0 = 6 };

// Development aid (-DQB_TG8_TRACE, scripts/tg8_trace.py): SM-clock stamps of the phases of every warp of the first blocks.
#ifdef QB_TG8_TRACE
enum { QB_TG8_TR_BLOCKS = 8, QB_TG8_TR_WARPS = 17, QB_TG8_TR_TILES = 48, QB_TG8_TR_EV = 12 };
__device__ unsigned int qb_tg8_trace_buf[QB_TG8_TR_BLOCKS * QB_TG8_TR_WARPS * QB_TG8_TR_TILES * QB_TG8_TR_EV];
#define QB_TG8_STAMP(tile, ev) do { if ((threadIdx.x & 31) == 0 && blockIdx.x < QB_TG8_TR_BLOCKS && blockIdx.y == 0 && (tile) < QB_TG8_TR_TILES) \
    qb_tg8_trace_buf[((blockIdx.x * QB_TG8_TR_WARPS + (threadIdx.x >> 5)) * QB_TG8_TR_TILES + (tile)) * QB_TG8_TR_EV + (ev)] = (unsigned int)clock64(); } while (0)
#else
#define QB_TG8_STAMP(tile, ev) do { } while (0)
#endif

__device__ __forceinline__ float qb_tg8_pow2(int e) { return __uint_as_float((uint32_t)(127 + max(-126, min(127, e))) << 23); }

// all threads: tensor-memory allocation and the mbarriers
template <int H>
__device__ __forceinline__ uint32_t qb_tg8_init(const QbTg8Plan& tp, unsigned char* smem) {
    using D = QbTg8Dim<H>;
    const uint32_t bars[8] = {QB_TG8_BAR_F, QB_TG8_BAR_B, QB_TG8_BAR_W, QB_TG8_BAR_Z, QB_TG8_BAR_RDY, QB_TG8_BAR_L, QB_TG8_BAR_RDY2, QB_TG8_BAR_RDY3};
    const uint32_t counts[8] = {1u, 1u, 1u, 1u, (uint32_t)D::NCOMP, 1u, (uint32_t)D::NCOMP, (uint32_t)D::NCOMP};
    return qb_tc_start(smem, QB_TG8_SLOT, (uint32_t)tp.tmem_cols, bars, counts);
}
// between evaluations (thread 0): every barrier starts again at parity 0
template <int H>
__device__ __forceinline__ void qb_tg8_reset_barriers(unsigned char* smem) {
    using D = QbTg8Dim<H>;
    const uint32_t bars[8] = {QB_TG8_BAR_F, QB_TG8_BAR_B, QB_TG8_BAR_W, QB_TG8_BAR_Z, QB_TG8_BAR_RDY, QB_TG8_BAR_L, QB_TG8_BAR_RDY2, QB_TG8_BAR_RDY3};
    const uint32_t counts[8] = {1u, 1u, 1u, 1u, (uint32_t)D::NCOMP, 1u, (uint32_t)D::NCOMP, (uint32_t)D::NCOMP};
    qb_mbar_reset(smem, bars, counts);
}
// fp16 pair -> two floats
__device__ __forceinline__ float2 qb_tg8_unpack(uint32_t w) {
    float a, b;
    asm("{ .reg .b16 l, h; mov.b32 {l, h}, %2; cvt.f32.f16 %0, l; cvt.f32.f16 %1, h; }" : "=f"(a), "=f"(b) : "r"(w));
    return make_float2(a, b);
}
// S * tanh of four pre-activations that were already multiplied by 2 log2 e (one reciprocal for the four, as
// qb_tanh4_prescaled)
__device__ __forceinline__ void qb_tg8_tanh4(float2& a, float2& b, float S) {
    const float2 one = make_float2(1.0f, 1.0f), s2 = make_float2(S, S), m2 = make_float2(-2.0f * S, -2.0f * S);
    float2 ea, eb;
    ea.x = qb_ex2(qb_min_nan(a.x, 30.0f)); ea.y = qb_ex2(qb_min_nan(a.y, 30.0f));
    eb.x = qb_ex2(qb_min_nan(b.x, 30.0f)); eb.y = qb_ex2(qb_min_nan(b.y, 30.0f));
    const float2 da = __fadd2_rn(ea, one), db = __fadd2_rn(eb, one);
    const float2 m = __fmul2_rn(da, db);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(m.x * m.y));
    float2 rr;
    rr.x = r * m.y; rr.y = r * m.x;
    const float2 ia = __fmul2_rn(rr, db), ib = __fmul2_rn(rr, da);
    a = __ffma2_rn(ia, m2, s2);
    b = __ffma2_rn(ib, m2, s2);
}

// flat theta (global) -> shared.  All threads of the block; ends with the async-proxy fence.
//   W0 image  : fp16 hi / lo of 2^s0 * 2 log2 e * [W0 | b0 | 0] (128 x 16, K-major: LBO 128, SBO 256), max in [2^13, 2^14)
//   W image   : fp16 hi / lo of 2^sW * W1, max |2^sW W1| in [2^13, 2^14)
//   F[b1 + j] = 2 log2 e * b1_j;  F[wl + j] = wl_j;  F[bl]
//   ones block of the a0 image (units 128 .. 143 of every point: 2^14, 0, 0, ..): column 128 of G1 becomes db1
//   scales (all powers of two, exact):
//     a0 image = 2^14 a0;  X image = 2^sX x (max |x| from absmax[0], ones column 2^sX);
//     z1 image = sz1 z1 with sz1 * B1 <= 60000 where |z1| <= B1 = (max|y| + |bl| + sum|wl|) / sigma^2 * max|wl|   (|a1| <= 1)
//     z0 image = sz0 z0 with sz0 * B0 <= 60000 where |z0| <= B0 = B1 * max_i sum_j |W1[j][i]|
//   A value far below its bound loses nothing until it is ~2^17 below it (fp16 keeps 2^16 .. 2^-24; hi and lo need 22 bits);
//   further down the lo part runs out of bits one by one (absolute error 2^-25 in image units) - only gradients that are
//   tiny against these bounds in EVERY entry (saturated units AND residuals far below sigma) see it, at the 1e-5 level.
template <int H>
__device__ __forceinline__ void qb_tg8_stage(const QbTg8Plan& tp, unsigned char* smem, const float* __restrict__ theta,
                                             const float* __restrict__ absmax, float is2) {
    using D = QbTg8Dim<H>;
    float* F = reinterpret_cast<float*>(smem + tp.fl_base);
    float* sred = reinterpret_cast<float*>(smem);                      // [17][4] + [17]
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
    const int hr = tp.hr;                      // the net's own width (32-wide nets run zero-padded on the 64-wide kernel)
    const float fold = 2.8853900817779268f;
    float mx = 0.0f, cs = 0.0f, wa = 0.0f, m0 = 0.0f;
    {
        // one coalesced sweep over W1: warps take rows, lanes take columns lane + 32 q; maximum and per-warp column sums of |W1|
        // (the z image is free during staging: scratch [warps][H])
        const int nw = nt >> 5;
        float csum[H / 32];
#pragma unroll
        for (int q = 0; q < H / 32; ++q) csum[q] = 0.0f;
        for (int j = wid; j < hr; j += nw) {
#pragma unroll
            for (int q = 0; q < H / 32; ++q) {
                const float w = lane + 32 * q < hr ? fabsf(theta[tp.w1_off + j * hr + lane + 32 * q]) : 0.0f;
                mx = fmaxf(mx, w);
                csum[q] += w;
            }
        }
        float* cscr = reinterpret_cast<float*>(smem + tp.z_img);
#pragma unroll
        for (int q = 0; q < H / 32; ++q) cscr[wid * H + lane + 32 * q] = csum[q];
        __syncthreads();
        if (tid < H)
            for (int w = 0; w < nw; ++w) cs += cscr[w * H + tid];
    }
    for (int e = tid; e < hr * tp.in_dim; e += nt) m0 = fmaxf(m0, fabsf(theta[tp.w0_off + e]));
    if (tid < hr && tp.b0_off >= 0) m0 = fmaxf(m0, fabsf(theta[tp.b0_off + tid]));
    if (tid < hr) wa = fabsf(theta[tp.wl_off + tid]);
    float ws = wa;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        cs = fmaxf(cs, __shfl_xor_sync(0xffffffffu, cs, off));
        wa = fmaxf(wa, __shfl_xor_sync(0xffffffffu, wa, off));
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, off));
        ws += __shfl_xor_sync(0xffffffffu, ws, off);
    }
    __syncthreads();                       // the previous evaluation's readers of the header / float area are done
    if (lane == 0) { sred[4 * wid + 0] = mx; sred[4 * wid + 1] = cs; sred[4 * wid + 2] = wa; sred[4 * wid + 3] = ws; sred[68 + wid] = m0; }
    __syncthreads();
    mx = cs = wa = ws = m0 = 0.0f;
    for (int w = 0; w < (nt + 31) >> 5; ++w) {
        mx = fmaxf(mx, sred[4 * w + 0]); cs = fmaxf(cs, sred[4 * w + 1]); wa = fmaxf(wa, sred[4 * w + 2]); ws += sred[4 * w + 3];
        m0 = fmaxf(m0, sred[68 + w]);
    }
    auto ilog = [](float v, int dflt) { return (v > 0.0f && v < 3.0e38f) ? ilogbf(v) : dflt; };
    const int sW = max(-40, min(40, 13 - ilog(mx, 13)));
    const int sX = max(-24, min(14, 13 - ilog(absmax[0], 13)));
    const int s0 = max(-40, min(40, 13 - ilog(m0 * fold, 13)));
    const float blv = tp.bl_off >= 0 ? theta[tp.bl_off] : 0.0f;
    const float B1 = (absmax[1] + fabsf(blv) + ws) * is2 * wa;
    // 2^(14 - e) * B <= 60000 (fp16 holds 65504): e = 14 - floor(log2(60000 / B))
    const int e1 = max(-50, min(50, 14 - ilog(60000.0f / B1, 14)));
    const int e0 = max(-50, min(50, 14 - ilog(60000.0f / (B1 * cs), 14)));
    const float wscale = qb_tg8_pow2(sW);
    // ---- W0 image: element (unit i, column q) at halfword (i/8)*128 + (q/8)*64 + (i%8)*8 + q%8
    {
        uint32_t* hi = reinterpret_cast<uint32_t*>(smem + tp.w0_img);
        uint32_t* lo = hi + D::W0IMG / 4;
        const float sc0 = fold * qb_tg8_pow2(s0);
        for (int e = tid; e < H * 8; e += nt) {
            const int i = e >> 3, q = (e & 7) * 2;
            float v[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                v[u] = 0.0f;
                if (i >= hr) continue;
                if (q + u < tp.in_dim) v[u] = theta[tp.w0_off + i * tp.in_dim + q + u] * sc0;
                else if (q + u == tp.in_dim && tp.b0_off >= 0) v[u] = theta[tp.b0_off + i] * sc0;
            }
            uint32_t h2, l2;
            qb_split_f16(v[0], v[1], h2, l2);
            const int idx = ((i >> 3) * 128 + (q >> 3) * 64 + (i & 7) * 8 + (q & 7)) >> 1;
            hi[idx] = h2; lo[idx] = l2;
        }
    }
    // ---- W image: one 128-byte core matrix (8 rows j x 8 columns i) per warp and step, lane = (row, column pair): the 32 words
    // of a core matrix are contiguous, so the stores are conflict-free
    {
        uint32_t* hi = reinterpret_cast<uint32_t*>(smem + tp.w_img);
        uint32_t* lo = hi + D::WIMG / 4;
        const int nw = nt >> 5;
        for (int cm = wid; cm < (H / 8) * (H / 8); cm += nw) {
            const int j = (cm / (H / 8)) * 8 + (lane >> 2), i = (cm % (H / 8)) * 8 + 2 * (lane & 3);
            const bool real = j < hr && i < hr;
            const float w0 = real ? theta[tp.w1_off + j * hr + i] : 0.0f, w1 = real ? theta[tp.w1_off + j * hr + i + 1] : 0.0f;
            uint32_t h2, l2;
            qb_split_f16(w0 * wscale, w1 * wscale, h2, l2);
            hi[cm * 32 + lane] = h2; lo[cm * 32 + lane] = l2;
        }
    }
    // ---- ones block of the a0 hi image (the lo image has none: its pass of DW1 runs with N = 128)
    {
        uint32_t* hi = reinterpret_cast<uint32_t*>(smem + tp.a_img + D::IMG);            // units H .. H + 15
        for (int e = tid; e < 2 * 2048 / 4; e += nt)
            hi[e] = (e < 512 && (e & 3) == 0) ? 0x00007400u : 0u;      // chunk 16: word 0 of every point's 16-byte row = (2^14, 0)
    }
    for (int j = tid; j < H; j += nt) {
        F[tp.b1 + j] = (tp.b1_off >= 0 && j < hr) ? theta[tp.b1_off + j] * fold : 0.0f;
        F[tp.wl + j] = j < hr ? theta[tp.wl_off + j] : 0.0f;
    }
    if (tid == 0) {
        F[tp.bl] = blv;
        F[tp.sc + QB_TG8_S_C1] = fold * qb_tg8_pow2(-14 - sW);
        F[tp.sc + QB_TG8_S_SZ1] = qb_tg8_pow2(14 - e1);
        F[tp.sc + QB_TG8_S_K0] = qb_tg8_pow2(-sW + e1 - e0);            // D0 / (sz1 2^sW) * sz0
        F[tp.sc + QB_TG8_S_UW1] = qb_tg8_pow2(-14 - (14 - e1));
        F[tp.sc + QB_TG8_S_UW0] = qb_tg8_pow2(-sX - (14 - e0));
        F[tp.sc + QB_TG8_S_SX] = qb_tg8_pow2(sX);
        F[tp.sc + QB_TG8_S_C0] = qb_tg8_pow2(-sX - s0);                // DL -> 2 log2 e * (W0 x + b0)
    }
    qb_fence_proxy_async();
}

// three passes (a_lo*b_hi, a_hi*b_lo, a_hi*b_hi) x KS k-steps of 16; *_img are descriptor low words of the hi / lo images;
// idesc1: instruction descriptor of the pass that reads b_lo (DW1: the lo image of a0 has no ones block, N = 128 there)
template <int KS>
__device__ __forceinline__ void qb_tg8_issue3(uint32_t d, uint32_t a_hi_img, uint32_t a_lo_img, uint32_t a_dhi, uint32_t a_step,
                                              uint32_t b_hi_img, uint32_t b_lo_img, uint32_t b_dhi, uint32_t b_step, uint32_t idesc,
                                              uint32_t idesc1, uint32_t acc0) {
    // the bases are laundered so that ptxas forms the descriptor pairs here, next to their MMAs: hoisted out of the tile
    // loop, the ~120 pairs of the GEMMs overflow the uniform register file and come back from local memory
    asm volatile("" : "+r"(a_hi_img), "+r"(a_lo_img), "+r"(b_hi_img), "+r"(b_lo_img));
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const uint32_t a = (pass == 0 ? a_lo_img : a_hi_img) + a_step * s;
            const uint32_t b = (pass == 1 ? b_lo_img : b_hi_img) + b_step * s;
            qb_mma_ss<true>(d, a, a_dhi, b, b_dhi, pass == 1 ? idesc1 : idesc, (pass == 0 && s == 0) ? acc0 : 1u);
        }
    }
}

// Value + gradient of the data term over points [n0, n1) for the staged parameter vector.  Every thread of the block
// (512 compute threads + the issue warp) calls it.  Returns the block-wide sum of squared residuals; g[0..P) (global, this
// block's row) receives d/dtheta of -0.5*ssq/sigma^2.
template <int H>
__device__ __forceinline__ double qb_tg8_eval(const QbTg8Plan& tp, uint32_t tmem, unsigned char* smem, const float* __restrict__ x,
                                              const float* __restrict__ y, int64_t n0, int64_t n1, float is2, float* __restrict__ g) {
    using D = QbTg8Dim<H>;
    constexpr int G = D::G, KS = H / 16;
    const float* F = reinterpret_cast<const float*>(smem + tp.fl_base);
    const uint32_t sb = qb_smem_u32(smem);
    const uint32_t bar_f = sb + QB_TG8_BAR_F, bar_b = sb + QB_TG8_BAR_B, bar_w = sb + QB_TG8_BAR_W, bar_z = sb + QB_TG8_BAR_Z,
                   bar_rdy = sb + QB_TG8_BAR_RDY, bar_l = sb + QB_TG8_BAR_L, bar_rdy2 = sb + QB_TG8_BAR_RDY2, bar_rdy3 = sb + QB_TG8_BAR_RDY3;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = (int)((n1 - n0 + 127) / 128);
    __syncthreads();                               // staging complete; nobody is still inside the previous evaluation
    if (threadIdx.x == 0) qb_tg8_reset_barriers<H>(smem);
    __syncthreads();
    float ssq = 0.0f, dbl = 0.0f;
    float2 dwl2[16];                               // output-layer weight gradient of this thread's 32 units, over its points
#pragma unroll
    for (int i = 0; i < 16; ++i) dwl2[i] = make_float2(0.0f, 0.0f);

    if (wid == D::ISSUER) {
        // ================================ issue warp ================================
        // D = f32; M = 128 (points) for L0 / FWD / BWD, M = H (units) for the weight gradients
        const uint32_t id_pts = (1u << 4) | ((128u >> 4) << 24), id_unt = (1u << 4) | ((uint32_t)(H >> 4) << 24) | (1u << 15) | (1u << 16);
        const uint32_t id_fwd = id_pts | ((uint32_t)(H >> 3) << 17);
        const uint32_t id_bwd = id_fwd | (1u << 16);
        const uint32_t id_dw1 = id_unt | ((uint32_t)((H + 16) >> 3) << 17);
        const uint32_t id_dw1n = id_unt | ((uint32_t)(H >> 3) << 17);
        const uint32_t id_dw0 = id_unt | ((16u >> 3) << 17);
        const uint32_t dh_a = qb_desc_hi(128u, 0u), dh_b = qb_desc_hi(2048u, 0u), dh_w = qb_desc_hi((uint32_t)D::WSBO, 0u);   // SBO 128 / 2048 / 16 H
        const uint32_t a_img = sb + (uint32_t)tp.a_img, z_img = sb + (uint32_t)tp.z_img, w_img = sb + (uint32_t)tp.w_img,
                       w0_img = sb + (uint32_t)tp.w0_img;
        // K-major views of the point images and the MN-major view of W: LBO 2048; the other views: LBO 128
        const uint32_t aK_hi = qb_desc_lo(a_img, 2048u), aK_lo = qb_desc_lo(a_img + D::AIMG, 2048u);
        const uint32_t aM_hi = qb_desc_lo(a_img, 128u), aM_lo = qb_desc_lo(a_img + D::AIMG, 128u);
        const uint32_t zK_hi = qb_desc_lo(z_img, 2048u), zK_lo = qb_desc_lo(z_img + D::IMG, 2048u);
        const uint32_t zM_hi = qb_desc_lo(z_img, 128u), zM_lo = qb_desc_lo(z_img + D::IMG, 128u);
        const uint32_t wK_hi = qb_desc_lo(w_img, 128u), wK_lo = qb_desc_lo(w_img + D::WIMG, 128u);
        const uint32_t wM_hi = qb_desc_lo(w_img, (uint32_t)D::WSBO), wM_lo = qb_desc_lo(w_img + D::WIMG, (uint32_t)D::WSBO);
        const uint32_t w0_hi = qb_desc_lo(w0_img, 128u), w0_lo = qb_desc_lo(w0_img + D::W0IMG, 128u), dh_w0 = qb_desc_hi(256u, 0u);
        // Hand-overs from the compute threads.  Two arrivals of one thread on the same mbarrier must be separated by a wait that
        // depends on the issue warp having seen the first one (else a fast thread's second arrival completes the phase while a slow
        // thread has not arrived once): the second hand-over of phase A follows the first without such a wait and has its own barrier.
        // The issue warp polls without a suspend hint: every hand-over is on the critical path of the tile loop.
        uint32_t n = 0, n2 = 0, n3 = 0;
        auto wait_rdy = [&]() {
            qb_mbar_spin(bar_rdy, n & 1u);
            ++n;
            qb_tc_fence_after();
            __syncwarp();
        };
        auto wait_rdy3 = [&]() {
            qb_mbar_spin(bar_rdy3, n3 & 1u);
            ++n3;
            qb_tc_fence_after();
            __syncwarp();
        };
        auto wait_rdy2 = [&]() {
            qb_mbar_spin(bar_rdy2, n2 & 1u);
            ++n2;
            qb_tc_fence_after();
            __syncwarp();
        };
        // layer 0 of tile u: X image (K-major view, K = 16: one k-step) x W0 image -> R1
        auto issue_l0 = [&](int u) {
            const uint32_t x_img = sb + (uint32_t)tp.x_img + (uint32_t)(u & 1) * 2u * QB_TG8_XIMG;
            qb_tg8_issue3<1>(tmem + D::C_D1, qb_desc_lo(x_img, 2048u), qb_desc_lo(x_img + QB_TG8_XIMG, 2048u), dh_a, 0u,
                             w0_hi, w0_lo, dh_w0, 0u, id_fwd, id_fwd, 0u);
        };
        if (T > 0) {
            wait_rdy();                                                   // X(0) is in the X image
            if (qb_elect()) { issue_l0(0); qb_commit(bar_l); }
            __syncwarp();
            wait_rdy();                                                   // a0(0) is in the a0 image
            if (qb_elect()) {
                qb_tg8_issue3<KS>(tmem + D::C_D1, aK_hi, aK_lo, dh_a, 256u, wK_hi, wK_lo, dh_w, 16u, id_fwd, id_fwd, 0u);
                qb_commit(bar_f);
            }
            __syncwarp();
        }
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
            const uint32_t acc0 = t > 0 ? 1u : 0u;
            if (t + 1 < T) {
                wait_rdy3();                                              // X(t+1) is in the X image, R1 has been read (EPI1(t), first pass)
                if (qb_elect()) { issue_l0(t + 1); qb_commit(bar_l); }
                __syncwarp();
            }
            wait_rdy();                                                   // z1(t) is in the z image; R0 is free
            QB_TG8_STAMP(t, 0);
            if (qb_elect()) {
                qb_tg8_issue3<KS>(tmem + D::C_D0, zK_hi, zK_lo, dh_a, 256u, wM_hi, wM_lo, dh_a, (uint32_t)(2 * D::WSBO) >> 4, id_bwd, id_bwd, 0u);
                qb_commit(bar_b);
                qb_tg8_issue3<8>(tmem + D::C_DW1, zM_hi, zM_lo, dh_b, 16u, aM_hi, aM_lo, dh_b, 16u, id_dw1, id_dw1n, acc0);
                qb_commit(bar_w);
            }
            __syncwarp();
            QB_TG8_STAMP(t, 1);
            if (t + 1 < T) {
                wait_rdy();                                               // a0(t+1) is in the a0 image, R1 is free
                if (qb_elect()) {
                    qb_tg8_issue3<KS>(tmem + D::C_D1, aK_hi, aK_lo, dh_a, 256u, wK_hi, wK_lo, dh_w, 16u, id_fwd, id_fwd, 0u);
                    qb_commit(bar_f);
                }
                __syncwarp();
            }
            wait_rdy2();                                                  // z0(t) is in the z image
            QB_TG8_STAMP(t, 2);
            if (qb_elect()) {
                const uint32_t x_img = sb + (uint32_t)tp.x_img + (uint32_t)(t & 1) * 2u * QB_TG8_XIMG;
                qb_tg8_issue3<8>(tmem + D::C_DW0, zM_hi, zM_lo, dh_b, 16u, qb_desc_lo(x_img, 128u), qb_desc_lo(x_img + QB_TG8_XIMG, 128u),
                                 dh_b, 16u, id_dw0, id_dw0, acc0);
                qb_commit(bar_z);
            }
            __syncwarp();
            QB_TG8_STAMP(t, 3);
        }
    } else {
        // ================================ compute warps ================================
        const int quarter = wid & 3, grp = wid >> 2;
        const uint32_t pt = (uint32_t)(quarter * 32 + lane);               // this thread's point of the tile = tensor-memory lane
        const int c = grp * 32;                                            // this thread's units
        const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16);
        const uint32_t prow = (pt >> 3) * 128u + (pt & 7u) * 16u;           // this point's 16-byte row inside an 8-unit chunk
        const uint32_t poff = prow + (uint32_t)(c >> 3) * 2048u;            // chunk j of this thread: + 2048 j
        unsigned char* a_hi = smem + tp.a_img + poff; unsigned char* a_lo = a_hi + D::AIMG;
        unsigned char* z_hi = smem + tp.z_img + poff; unsigned char* z_lo = z_hi + D::IMG;
        // X image: thread group g lays out columns CPG g .. CPG g + CPG - 1 of its point (a 16-byte row, or half of one)
        unsigned char* x_row = smem + tp.x_img + ((grp * D::CPG) >> 3) * 2048 + prow + ((grp * D::CPG) & 7) * 2;
        float* ybuf = reinterpret_cast<float*>(smem + tp.ybuf);
        const float c1 = F[tp.sc + QB_TG8_S_C1], sz1 = F[tp.sc + QB_TG8_S_SZ1], k0 = F[tp.sc + QB_TG8_S_K0], sx = F[tp.sc + QB_TG8_S_SX],
                    c0 = F[tp.sc + QB_TG8_S_C0];
        const float4* B4 = reinterpret_cast<const float4*>(F + tp.b1 + c);
        const float4* W4 = reinterpret_cast<const float4*>(F + tp.wl + c);

        auto publish = [&](uint32_t bar) {
            qb_fence_proxy_async();
            qb_tc_fence_before();
            qb_mbar_arrive(bar);
        };
        // this thread's 32 columns of region `col` hold packed results: per half of 16 columns, 8 hi words then 8 lo words
        // (units 16 hf .. 16 hf + 15).  Copy them into the images.
        auto unpark = [&](uint32_t col, unsigned char* hi, unsigned char* lo) {
            uint32_t v[2][16];
            qb_tmem_ld16(tl + col + c, v[0]);                  // both halves in flight before the first store
            qb_tmem_ld16(tl + col + c + 16, v[1]);
            qb_tmem_ld_wait16(v[0]);
            qb_tmem_ld_wait16(v[1]);
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
#pragma unroll
                for (int jj = 0; jj < 2; ++jj) {
                    *reinterpret_cast<uint4*>(hi + 2048 * (2 * hf + jj)) = make_uint4(v[hf][4 * jj], v[hf][4 * jj + 1], v[hf][4 * jj + 2], v[hf][4 * jj + 3]);
                    *reinterpret_cast<uint4*>(lo + 2048 * (2 * hf + jj)) = make_uint4(v[hf][8 + 4 * jj], v[hf][9 + 4 * jj], v[hf][10 + 4 * jj], v[hf][11 + 4 * jj]);
                }
            }
        };
        // inputs of tile tt: this thread's four columns of its point (x, then the constant 1, then zeros) and the target
        float xq[D::CPG], yn = 0.0f;
        auto fetch = [&](int tt) {
            const int64_t pp = n0 + (int64_t)tt * 128 + pt;
#pragma unroll
            for (int j = 0; j < D::CPG; ++j) {
                const int q = D::CPG * grp + j;
                float v = 0.0f;
                if (q < tp.in_dim && pp < n1) v = __ldg(x + pp * tp.in_dim + q);
                xq[j] = (q == tp.in_dim) ? 1.0f : v;
            }
            yn = pp < n1 ? __ldg(y + pp) : 0.0f;
        };
        auto xstore = [&](int tt) {
            uint32_t h[D::CPG / 2], l[D::CPG / 2];
#pragma unroll
            for (int j = 0; j < D::CPG / 2; ++j) qb_split_f16(xq[2 * j] * sx, xq[2 * j + 1] * sx, h[j], l[j]);
            unsigned char* xi = x_row + (tt & 1) * 2 * QB_TG8_XIMG;
            if constexpr (D::CPG == 4) {
                *reinterpret_cast<uint2*>(xi) = make_uint2(h[0], h[1]);
                *reinterpret_cast<uint2*>(xi + QB_TG8_XIMG) = make_uint2(l[0], l[1]);
            } else {
                *reinterpret_cast<uint4*>(xi) = make_uint4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<uint4*>(xi + QB_TG8_XIMG) = make_uint4(l[0], l[1], l[2], l[3]);
            }
        };
        // EPIL: R1 holds layer 0 of a tile (this thread's 32 columns) -> 2^14 tanh, packed, back into the same columns
        auto epil = [&]() {
            const float2 c2 = make_float2(c0, c0);
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                uint32_t v[16], o[16];
                qb_tmem_ld16(tl + D::C_D1 + c + 16 * hf, v);
                qb_tmem_ld_wait16(v);
#pragma unroll
                for (int gq = 0; gq < 4; ++gq) {
                    float2 z0 = __fmul2_rn(make_float2(__uint_as_float(v[4 * gq]), __uint_as_float(v[4 * gq + 1])), c2);
                    float2 z1 = __fmul2_rn(make_float2(__uint_as_float(v[4 * gq + 2]), __uint_as_float(v[4 * gq + 3])), c2);
                    qb_tg8_tanh4(z0, z1, 16384.0f);
                    qb_split_f16(z0.x, z0.y, o[2 * gq], o[8 + 2 * gq]);
                    qb_split_f16(z1.x, z1.y, o[2 * gq + 1], o[8 + 2 * gq + 1]);
                }
                qb_tmem_st16(tl + D::C_D1 + c + 16 * hf, o);
            }
        };

        float yv = 0.0f;                                             // target of this thread's point of the current tile
        if (T > 0) {
            fetch(0);
            yv = yn;
            xstore(0);
            publish(bar_rdy);
            qb_mbar_wait_counted(bar_l, 0u);
            qb_tc_fence_after();
            epil();
            qb_tmem_st_wait();
            unpark(D::C_D1, a_hi, a_lo);
            publish(bar_rdy);
        }
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
            const int64_t p = n0 + (int64_t)t * 128 + pt;
            const bool live = p < n1;
            const bool more = t + 1 < T;
            // ---------------- phase B: EPI1(t)
            QB_TG8_STAMP(t, 0);
            if (more) fetch(t + 1);
            qb_mbar_wait_counted(bar_f, (uint32_t)t & 1u);
            qb_tc_fence_after();
            QB_TG8_STAMP(t, 1);
            {
                float2 acc = make_float2(0.0f, 0.0f);
                const float2 c2 = make_float2(c1, c1);
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[16];
                    qb_tmem_ld16(tl + D::C_D1 + c + 16 * hf, v);
                    qb_tmem_ld_wait16(v);
#pragma unroll
                    for (int gq = 0; gq < 4; ++gq) {
                        const float4 b = B4[4 * hf + gq], w = W4[4 * hf + gq];
                        float2 z0 = __ffma2_rn(make_float2(__uint_as_float(v[4 * gq]), __uint_as_float(v[4 * gq + 1])), c2, make_float2(b.x, b.y));
                        float2 z1 = __ffma2_rn(make_float2(__uint_as_float(v[4 * gq + 2]), __uint_as_float(v[4 * gq + 3])), c2, make_float2(b.z, b.w));
                        qb_tg8_tanh4(z0, z1, 1.0f);
                        acc = __ffma2_rn(make_float2(w.x, w.y), z0, acc);
                        acc = __ffma2_rn(make_float2(w.z, w.w), z1, acc);
                        v[4 * gq] = __float_as_uint(z0.x); v[4 * gq + 1] = __float_as_uint(z0.y);
                        v[4 * gq + 2] = __float_as_uint(z1.x); v[4 * gq + 3] = __float_as_uint(z1.y);
                    }
                    qb_tmem_st16(tl + D::C_D0 + c + 16 * hf, v);           // a1 waits in R0 (free until BWD(t)); R1 is released below
                }
                ybuf[grp * 128 + pt] = acc.x + acc.y;
                QB_TG8_STAMP(t, 2);
                asm volatile("bar.sync %0, %1;" :: "r"(1 + quarter), "n"(32 * G) : "memory");
                qb_tmem_st_wait();                                     // the stash is read back below
                float yo = F[tp.bl];
#pragma unroll
                for (int gg = 0; gg < G; ++gg) yo += ybuf[gg * 128 + pt];
                const float r = live ? yv - yo : 0.0f;
                const float dy = r * is2, dyz = dy * sz1;
                const float2 dy2 = make_float2(dy, dy), dyz2 = make_float2(dyz, dyz), one2 = make_float2(1.0f, 1.0f);
                if (grp == 0) { ssq = fmaf(r, r, ssq); dbl += dy; }
                if (t > 0) { qb_mbar_wait_counted(bar_z, (uint32_t)(t - 1) & 1u); qb_tc_fence_after(); }     // DW0(t-1) has read the z and X images
                QB_TG8_STAMP(t, 3);
                if (more) {
                    xstore(t + 1);
                    publish(bar_rdy3);                                 // => L0(t+1) into R1, under the second pass
                }
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[16];
                    qb_tmem_ld16(tl + D::C_D0 + c + 16 * hf, v);
                    qb_tmem_ld_wait16(v);
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        uint32_t h[4], l[4];
#pragma unroll
                        for (int g2 = 0; g2 < 2; ++g2) {
                            const int gq = 2 * jj + g2;
                            const float4 w = W4[4 * hf + gq];
                            const float2 a01 = make_float2(__uint_as_float(v[4 * gq]), __uint_as_float(v[4 * gq + 1]));
                            const float2 a23 = make_float2(__uint_as_float(v[4 * gq + 2]), __uint_as_float(v[4 * gq + 3]));
                            const float2 z01 = __fmul2_rn(__fmul2_rn(make_float2(w.x, w.y), dyz2), __ffma2_rn(make_float2(-a01.x, -a01.y), a01, one2));
                            const float2 z23 = __fmul2_rn(__fmul2_rn(make_float2(w.z, w.w), dyz2), __ffma2_rn(make_float2(-a23.x, -a23.y), a23, one2));
                            dwl2[8 * hf + 2 * gq] = __ffma2_rn(dy2, a01, dwl2[8 * hf + 2 * gq]);
                            dwl2[8 * hf + 2 * gq + 1] = __ffma2_rn(dy2, a23, dwl2[8 * hf + 2 * gq + 1]);
                            qb_split_f16(z01.x, z01.y, h[2 * g2], l[2 * g2]);
                            qb_split_f16(z23.x, z23.y, h[2 * g2 + 1], l[2 * g2 + 1]);
                        }
                        *reinterpret_cast<uint4*>(z_hi + 2048 * (2 * hf + jj)) = make_uint4(h[0], h[1], h[2], h[3]);
                        *reinterpret_cast<uint4*>(z_lo + 2048 * (2 * hf + jj)) = make_uint4(l[0], l[1], l[2], l[3]);
                    }
                }
            }
            QB_TG8_STAMP(t, 4);
            publish(bar_rdy);
            // ---------------- phase A: EPIL(t+1) while BWD(t) runs, EPI0(t) while DW1(t) runs; results stay in tensor memory until
            // DW1(t) has read the images
            if (more) {
                qb_mbar_wait_counted(bar_l, (uint32_t)(t + 1) & 1u);               // layer 0 of tile t+1 is in R1 (issued ahead of BWD(t))
                qb_tc_fence_after();
                QB_TG8_STAMP(t, 10);
                epil();
                yv = yn;
            }
            QB_TG8_STAMP(t, 5);
            qb_mbar_wait_counted(bar_b, (uint32_t)t & 1u);
            qb_tc_fence_after();
            QB_TG8_STAMP(t, 6);
            {
                const float2 k2 = make_float2(k0, k0), sa = make_float2(6.103515625e-05f, 6.103515625e-05f), one = make_float2(1.0f, 1.0f);
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[16], o[16];
                    qb_tmem_ld16(tl + D::C_D0 + c + 16 * hf, v);
                    qb_tmem_ld_wait16(v);
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        const uint4 h4 = *reinterpret_cast<const uint4*>(a_hi + 2048 * (2 * hf + jj));
                        const uint4 l4 = *reinterpret_cast<const uint4*>(a_lo + 2048 * (2 * hf + jj));
                        const uint32_t hw[4] = {h4.x, h4.y, h4.z, h4.w}, lw[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
                        for (int w = 0; w < 4; ++w) {
                            float2 a = __fadd2_rn(qb_tg8_unpack(hw[w]), qb_tg8_unpack(lw[w]));
                            a = __fmul2_rn(a, sa);
                            const float2 da = __ffma2_rn(make_float2(-a.x, -a.y), a, one);
                            const float2 d = make_float2(__uint_as_float(v[8 * jj + 2 * w]), __uint_as_float(v[8 * jj + 2 * w + 1]));
                            const float2 z = __fmul2_rn(__fmul2_rn(d, k2), da);
                            qb_split_f16(z.x, z.y, o[4 * jj + w], o[8 + 4 * jj + w]);
                        }
                    }
                    qb_tmem_st16(tl + D::C_D0 + c + 16 * hf, o);      // the z image is still an operand of DW1(t)
                }
            }
            qb_tmem_st_wait();
            QB_TG8_STAMP(t, 7);
            qb_mbar_wait_counted(bar_w, (uint32_t)t & 1u);                      // DW1(t) has read the z and a0 images
            qb_tc_fence_after();
            QB_TG8_STAMP(t, 8);
            if (more) {
                unpark(D::C_D1, a_hi, a_lo);
                publish(bar_rdy);                                    // => FWD(t+1)
            }
            unpark(D::C_D0, z_hi, z_lo);
            publish(bar_rdy2);                                       // => DW0(t)
            QB_TG8_STAMP(t, 9);
        }
        if (T > 0) { qb_mbar_wait_counted(bar_z, (uint32_t)(T - 1) & 1u); qb_tc_fence_after(); }

        // ---------------- gradient out: row j (G1) / i (G0).  An M = 128 accumulator keeps row m in lane m; an M = 64 one in
        // lane (m % 16) + 32 (m / 16): the first 16 lanes of every warp quarter
        const int d = tp.in_dim;
        if (T > 0) {
            const float uw1 = F[tp.sc + QB_TG8_S_UW1], uw0 = F[tp.sc + QB_TG8_S_UW0];
            const int hr = tp.hr;
            const int row = H == 128 ? (int)pt : quarter * 16 + lane;
            const bool rv = (H == 128 || lane < 16) && row < hr;
            const bool al16 = (reinterpret_cast<uintptr_t>(g + tp.w1_off) & 15) == 0;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                uint32_t v[16];
                qb_tmem_ld16(tl + D::C_DW1 + c + 16 * hf, v);
                qb_tmem_ld_wait16(v);
                float* dst = g + tp.w1_off + row * hr + c + 16 * hf;
                if (!rv || c + 16 * hf >= hr) continue;
                if (al16) {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        reinterpret_cast<float4*>(dst)[q] = make_float4(__uint_as_float(v[4 * q]) * uw1, __uint_as_float(v[4 * q + 1]) * uw1,
                                                                        __uint_as_float(v[4 * q + 2]) * uw1, __uint_as_float(v[4 * q + 3]) * uw1);
                } else {
#pragma unroll
                    for (int q = 0; q < 16; ++q) dst[q] = __uint_as_float(v[q]) * uw1;
                }
            }
            if (grp == 0) {
                uint32_t v[16];
                qb_tmem_ld16(tl + D::C_DW1 + H, v);                    // column H: db1
                qb_tmem_ld_wait16(v);
                if (rv && tp.b1_off >= 0) g[tp.b1_off + row] = __uint_as_float(v[0]) * uw1;
                qb_tmem_ld16(tl + D::C_DW0, v);                        // columns < d: dW0, column d: db0
                qb_tmem_ld_wait16(v);
                if (rv) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        if (q < d) g[tp.w0_off + row * d + q] = __uint_as_float(v[q]) * uw0;
                        else if (q == d && tp.b0_off >= 0) g[tp.b0_off + row] = __uint_as_float(v[q]) * uw0;
                    }
                }
            }
        }
    }
    if (T <= 0)
        for (int i = threadIdx.x; i < tp.n_params; i += blockDim.x) g[i] = 0.0f;
    // dWl[j] = sum over the 128 point slots of the per-thread partial sums (fixed order); the images are free now
    qb_tc_fence_before();
    __syncthreads();
    if (T > 0) {
        float* scr = reinterpret_cast<float*>(smem + tp.a_img);            // [H][132] floats over the a0 / z / X images
        if (wid < D::ISSUER) {
            const int pt = (wid & 3) * 32 + lane, c = (wid >> 2) * 32;
#pragma unroll
            for (int e = 0; e < 16; ++e) { scr[(c + 2 * e) * 132 + pt] = dwl2[e].x; scr[(c + 2 * e + 1) * 132 + pt] = dwl2[e].y; }
        }
        __syncthreads();
        // four threads per unit, each sums every fourth point slot (row stride 132: the 32 lanes of a warp hit 32 banks), then the
        // four meet through shuffles
        if (threadIdx.x < 4 * H) {
            const int u = threadIdx.x >> 2, part = threadIdx.x & 3;
            float s = 0.0f;
#pragma unroll 8
            for (int q = 0; q < 32; ++q) s += scr[u * 132 + 4 * q + part];
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if (part == 0 && u < tp.hr) g[tp.wl_off + u] = s;
        }
    }
    // block-wide sums of the squared residuals and of dy (= the output bias gradient) in one pass
    double* red = reinterpret_cast<double*>(smem);                         // 2 x 17 doubles + 2
    double v0 = (double)ssq, v1 = (double)dbl;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { v0 += __shfl_xor_sync(0xffffffffu, v0, off); v1 += __shfl_xor_sync(0xffffffffu, v1, off); }
    __syncthreads();
    if (lane == 0) { red[2 * wid] = v0; red[2 * wid + 1] = v1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s0 = 0.0, s1 = 0.0;
        for (int w = 0; w < (int)(blockDim.x + 31) >> 5; ++w) { s0 += red[2 * w]; s1 += red[2 * w + 1]; }
        red[34] = s0;
        if (tp.bl_off >= 0) g[tp.bl_off] = (float)s1;
    }
    __syncthreads();
    return red[34];
}
#endif  // __CUDACC__
