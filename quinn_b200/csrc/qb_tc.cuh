// Tensor-core evaluation of the data term for fp32 MLPs: tcgen05.mma kind::tf32 with the operands split in two
// ("3xTF32": a*b ~= a_hi*b_hi + a_lo*b_hi + a_hi*b_lo, products accumulated in fp32 in tensor memory), which keeps
// fp32-level accuracy (relative error of a product ~2^-21) while the 64x64 hidden-layer GEMMs leave the CUDA cores.
//
// One tile = 128 data points = the 128 lanes of tensor memory; a thread works on one point (lane) and, in the pipelined
// variants, on a subset of the units / accumulator columns:
//   layer 0 (n_in <= 15):  CUDA cores; tanh; the result is split into hi/lo and written with tcgen05.st to tensor
//                          memory as the A operand (lane = point, column = unit);
//   hidden layers 1..L-2:  D[128 x n_out] = A[128 x n_in] * W^T, A from tensor memory, W (hi and lo) staged once per
//                          parameter vector in shared memory in the K-major no-swizzle canonical layout (W is stored
//                          (n_out, n_in) row-major in theta = already K-major).  One elected lane of a convergent warp
//                          issues the 3 * n_in/8 MMAs back to back and a tcgen05.commit to an mbarrier; everybody waits
//                          on the mbarrier, reads D back with tcgen05.ld, adds the bias, applies the activation and
//                          either writes the next A operand or, for the last hidden layer, feeds
//   last layer (n_out<=4): a per-thread dot product with weights broadcast from shared memory, then the residual
//                          (kernels 1, 3) or the store of the network output (kernel 4).
// Tensor-memory columns: [0,Kmax) A_hi, [Kmax,2Kmax) A_lo, [2Kmax, 2Kmax+Nmax) D (pipelined path: a second D buffer
// follows).  Two code paths: qb_tc_pipe_run (one hidden GEMM, 256 or 512 threads, mbarrier pipeline) and
// qb_tc_forward_tile (any eligible depth, 128 threads, one block barrier per layer).
// The tensor pipe of one block overlaps with the CUDA-core phases of the other block resident on the SM.
#pragma once
#include <stdint.h>
#include "qb_plan.h"
#include "qb_tcgen05.cuh"

struct QbTcLayer {
    int n_in, n_out, w_off, b_off, act;
    int bhi, blo;        // byte offsets in dynamic shared memory of the split weight tiles (canonical layout)
    int bias;            // float index (in the float area) of the n_out biases
};
struct QbTcPlan {
    int n_layers;                       // layers 1 .. n_layers-2 run on the tensor cores
    int in_dim, ni, out_dim, n_params;  // ni: padded input width (4, 12 or 16; slot in_dim carries the bias)
    int h0, kl;                         // width after layer 0; n_in of the last layer
    int act0, act_last, final_exp;
    int pipe;                           // one tensor-core layer: software-pipelined tile loop with 2 (widths <= 64) or 4
                                        // (<= 128) column groups; 0: simple 128-thread loop
    int w0, wl, bl;                     // float indices: layer-0 rows [h0][ni], last-layer W [out][kl], last bias
    int w0_off, b0_off, wl_off, bl_off; // offsets in theta (b*_off < 0: no bias)
    int fl_base, ybuf;                  // byte offsets of the float area and of the partial-output exchange buffer
    int nthreads;                       // 256 (pipelined) or 128
    int a_lo_col, d_col, tmem_cols;
    int smem_bytes;
    int v3;                             // warp-specialised path (qb_tc3.cuh): 1 = hidden width 64 (288 threads), 2 = 128 (544); layouts below
    int v3_w0, v3_w1, v3_x;             // byte offsets: W0 tf32 hi|lo, W1 fp16 hi|lo, x tiles [2][hi|lo]
    int v3_c1;                          // float index of the accumulator scale of the hidden GEMM
    int v3_xbar;                        // byte offset of the three x_full mbarriers
    int v3_state;                       // byte offset of the chain state kept in shared memory (chain kernel): cur | prop | scale
    QbTcLayer L[QB_MAX_LAYERS];
};

#ifdef __CUDACC__
// shared-memory header: [0,320) reduction scratch, three mbarriers, tensor-memory base
enum { QB_TC_RED_BYTES = 320, QB_TC_BAR_OFF = 320, QB_TC_SLOT_OFF = 328, QB_TC_ABAR_OFF = 336,
       QB_TC_HBAR_OFF = 344, QB_TC_HDR_BYTES = 384 };

struct QbTcCtx { uint32_t tmem, bar, phase, abar, aphase, hbar, hphase; };

// all threads; allocates tensor memory and initialises the mbarriers
__device__ __forceinline__ void qb_tc_init(const QbTcPlan& tp, unsigned char* smem, QbTcCtx& cx) {
    const uint32_t bars[3] = {QB_TC_BAR_OFF, QB_TC_ABAR_OFF, QB_TC_HBAR_OFF}, counts[3] = {1u, QB_MBAR_BLOCK, 1u};
    cx.tmem = qb_tc_start(smem, QB_TC_SLOT_OFF, (uint32_t)tp.tmem_cols, bars, counts);
    cx.bar = qb_smem_u32(smem + QB_TC_BAR_OFF);
    cx.abar = qb_smem_u32(smem + QB_TC_ABAR_OFF);
    cx.hbar = qb_smem_u32(smem + QB_TC_HBAR_OFF);
    cx.phase = 0; cx.aphase = 0; cx.hphase = 0;
}

__device__ __forceinline__ float qb_tf32_hi(float w) { return __uint_as_float(__float_as_uint(w) & 0xFFFFE000u); }

// flat theta (global) -> shared: layer-0 rows, split hidden weights in the canonical K-major layout, biases, last layer.
// Canonical layout (no swizzle): core matrix = 8 rows (n) x 16 bytes (4 k), stored as 128 contiguous bytes; core
// matrices adjacent along k (LBO = 128 B), groups of 8 rows SBO = 128*(K/4) B apart => float index
// e = ((n/8)*(K/4) + k/4)*32 + (n%8)*4 + k%4.
__device__ __forceinline__ void qb_tc_stage(const QbTcPlan& tp, unsigned char* smem, const float* __restrict__ theta) {
    float* F = reinterpret_cast<float*>(smem + tp.fl_base);
    const int tid = threadIdx.x, nt = blockDim.x;
    const float fold = 2.8853900817779268f;
    {
        // layer 0, units in pairs: float index ((j/2)*ni + q)*2 + (j&1); slot q == in_dim carries the bias
        const float s0 = tp.act0 == QB_ACT_TANH ? fold : 1.0f;
        for (int e = tid; e < tp.h0 * tp.ni; e += nt) {
            const int u = e & 1, q = (e >> 1) % tp.ni, j = ((e >> 1) / tp.ni) * 2 + u;
            float v = 0.0f;
            if (q < tp.in_dim) v = theta[tp.w0_off + j * tp.in_dim + q] * s0;
            else if (q == tp.in_dim && tp.b0_off >= 0) v = theta[tp.b0_off + j] * s0;
            F[tp.w0 + e] = v;
        }
    }
    for (int l = 1; l < tp.n_layers - 1; ++l) {
        const QbTcLayer& L = tp.L[l];
        const int K = L.n_in, N = L.n_out, kc4 = K >> 2;
        const float sc = L.act == QB_ACT_TANH ? fold : 1.0f;
        float* hi = reinterpret_cast<float*>(smem + L.bhi);
        float* lo = reinterpret_cast<float*>(smem + L.blo);
        for (int e = tid; e < N * K; e += nt) {
            const int q = e & 3, r = (e >> 2) & 7, g = e >> 5;
            const int n8 = g / kc4, kc = g - n8 * kc4;
            const float w = theta[L.w_off + (n8 * 8 + r) * K + kc * 4 + q] * sc;
            const float h = qb_tf32_hi(w);
            hi[e] = h;
            lo[e] = w - h;
        }
        for (int j = tid; j < N; j += nt) F[L.bias + j] = L.b_off >= 0 ? theta[L.b_off + j] * sc : 0.0f;
    }
    {
        const float sl = tp.act_last == QB_ACT_TANH ? fold : 1.0f;
        for (int e = tid; e < tp.out_dim * tp.kl; e += nt) F[tp.wl + e] = theta[tp.wl_off + e] * sl;
        for (int j = tid; j < tp.out_dim; j += nt) F[tp.bl + j] = tp.bl_off >= 0 ? theta[tp.bl_off + j] * sl : 0.0f;
    }
    qb_fence_proxy_async();
}

// tanh of four pre-activations that were already multiplied by 2*log2(e): tanh = 1 - 2/(1 + 2^z'), with ONE
// reciprocal for the four denominators (the MUFU pipe, 16 results/clk/SM, is what bounds this kernel):
// m = (da*db), r = 1/(m.x*m.y), 1/da = (r*m.y, r*m.x)*db ... .  z' is clamped at 30 (tanh(10.4) == 1.0f) so that the
// product of four denominators stays finite; min.NaN keeps NaN pre-activations NaN.
__device__ __forceinline__ float qb_min_nan(float a, float b) {
    float r;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float qb_ex2(float z) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z));
    return e;
}
__device__ __forceinline__ void qb_tanh4_prescaled(float2& a, float2& b) {
    const float2 one = make_float2(1.0f, 1.0f), m2 = make_float2(-2.0f, -2.0f);
    float2 ea, eb;
    ea.x = qb_ex2(qb_min_nan(a.x, 30.0f)); ea.y = qb_ex2(qb_min_nan(a.y, 30.0f));
    eb.x = qb_ex2(qb_min_nan(b.x, 30.0f)); eb.y = qb_ex2(qb_min_nan(b.y, 30.0f));
    const float2 da = __fadd2_rn(ea, one), db = __fadd2_rn(eb, one);
    const float2 m = __fmul2_rn(da, db);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(m.x * m.y));
    float2 rr;
    rr.x = r * m.y; rr.y = r * m.x;                 // (1/m.x, 1/m.y)
    const float2 ia = __fmul2_rn(rr, db), ib = __fmul2_rn(rr, da);
    a = __ffma2_rn(ia, m2, one);
    b = __ffma2_rn(ib, m2, one);
}
// D = A_lo*Bhi^T + A_hi*Blo^T + A_hi*Bhi^T, then commit to the mbarrier.
// Issue by a whole (convergent) warp with one elected lane, K/8 known at compile time: every descriptor is
// base + constant, so the 3*K/8 MMAs go out back to back (a single thread doing address arithmetic between the
// MMAs was the critical path of the tile loop: ~80 cycles per MMA).
// HALF: the MMAs of the first half of K (all three passes) are committed to `hbar` on their own, so that the A columns
// of that half can be refilled while the second half is still running.
template <int KS, bool HALF = false>
__device__ __forceinline__ void qb_tc_issue_ks(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t bhi, uint32_t blo,
                                               uint32_t dhi, uint32_t idesc, uint32_t bar, uint32_t hbar = 0) {
    if (qb_elect()) {
#pragma unroll
        for (int half = 0; half < (HALF ? 2 : 1); ++half) {
            constexpr int S0 = 0, SN = HALF ? KS / 2 : KS;
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                for (int ss = S0; ss < SN; ++ss) {
                    const int s = ss + half * SN;
                    const uint32_t a = (pass == 0 ? a_lo : a_hi) + (uint32_t)s * 8u;
                    const uint32_t bl = (pass == 1 ? blo : bhi) + (uint32_t)s * 16u;   // +256 bytes, in 16-byte units
                    if (half == 0 && pass == 0 && ss == 0) qb_mma_ts<false, false>(d, a, bl, dhi, idesc);
                    else qb_mma_ts<false, true>(d, a, bl, dhi, idesc);
                }
            }
            if (HALF && half == 0) qb_commit(hbar);
        }
        qb_commit(bar);
    }
    __syncwarp();
}
// called by all lanes of warp 0
template <bool HALF = false, int KSH = 8>
__device__ __forceinline__ void qb_tc_issue_warp(const QbTcPlan& tp, const QbTcLayer& L, const QbTcCtx& cx, unsigned char* smem,
                                                 uint32_t d_off) {
    const uint32_t K = L.n_in, N = L.n_out;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((N >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t dhi = qb_desc_hi(128u * (K >> 2), 0u);
    const uint32_t bhi = qb_desc_lo(qb_smem_u32(smem + L.bhi), 128u);
    const uint32_t blo = qb_desc_lo(qb_smem_u32(smem + L.blo), 128u);
    const uint32_t d = cx.tmem + tp.d_col + d_off, a_hi = cx.tmem, a_lo = cx.tmem + tp.a_lo_col;
    if constexpr (HALF) {        // K == 8*KSH: 64 (two column groups) or 128 (four)
        qb_tc_issue_ks<KSH, true>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar, cx.hbar);
        return;
    }
    switch (K >> 3) {
        case 2: qb_tc_issue_ks<2>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        case 4: qb_tc_issue_ks<4>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        case 6: qb_tc_issue_ks<6>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        case 8: qb_tc_issue_ks<8>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        case 10: qb_tc_issue_ks<10>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        case 12: qb_tc_issue_ks<12>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        case 14: qb_tc_issue_ks<14>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
        default: qb_tc_issue_ks<16>(d, a_hi, a_lo, bhi, blo, dhi, idesc, cx.bar); break;
    }
}

template <int ACT> __device__ __forceinline__ void qb_tc_act4(float2& a, float2& b) {
    if (ACT == QB_ACT_TANH) qb_tanh4_prescaled(a, b);
    else if (ACT == QB_ACT_RELU) { a.x = fmaxf(a.x, 0.0f); a.y = fmaxf(a.y, 0.0f); b.x = fmaxf(b.x, 0.0f); b.y = fmaxf(b.y, 0.0f); }
}

// split 16 fp32 values into tf32 hi + remainder lo and write them to tensor memory (this thread's lane)
__device__ __forceinline__ void qb_tc_split_store(uint32_t t_hi, uint32_t t_lo, const float (&h)[16]) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
        const float2 hh = make_float2(qb_tf32_hi(h[i]), qb_tf32_hi(h[i + 1]));
        const float2 ll = __fadd2_rn(make_float2(h[i], h[i + 1]), make_float2(-hh.x, -hh.y));
        hi[i] = __float_as_uint(hh.x); hi[i + 1] = __float_as_uint(hh.y);
        lo[i] = __float_as_uint(ll.x); lo[i + 1] = __float_as_uint(ll.y);
    }
    qb_tmem_st16(t_hi, hi);
    qb_tmem_st16(t_lo, lo);
}

// layer 0 on the CUDA cores for units c .. c+15 of this thread's point: h = act(W0 x + b0) (packed FFMA2, two units
// per instruction; the bias rides in slot in_dim of the padded input, xr[in_dim] == 1)
template <int NI, int ACT>
__device__ __forceinline__ void qb_tc_l0_chunk(const QbTcPlan& tp, const float* F, int c, const float (&xr)[NI], float (&h)[16]) {
    const float4* W = reinterpret_cast<const float4*>(F + tp.w0 + c * NI);     // pair p of the chunk: W[p*NI/2 + q/2]
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        float2 z0 = make_float2(0.0f, 0.0f), z1 = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int q = 0; q < NI; q += 2) {
            const float4 wa = W[(2 * g) * (NI / 2) + q / 2], wb = W[(2 * g + 1) * (NI / 2) + q / 2];
            z0 = __ffma2_rn(make_float2(wa.x, wa.y), make_float2(xr[q], xr[q]), z0);
            z0 = __ffma2_rn(make_float2(wa.z, wa.w), make_float2(xr[q + 1], xr[q + 1]), z0);
            z1 = __ffma2_rn(make_float2(wb.x, wb.y), make_float2(xr[q], xr[q]), z1);
            z1 = __ffma2_rn(make_float2(wb.z, wb.w), make_float2(xr[q + 1], xr[q + 1]), z1);
        }
        qb_tc_act4<ACT>(z0, z1);
        h[4 * g + 0] = z0.x; h[4 * g + 1] = z0.y; h[4 * g + 2] = z1.x; h[4 * g + 3] = z1.y;
    }
}

// accumulator columns c .. c+15 of this thread's point -> h = act(D + bias)
template <int ACT>
__device__ __forceinline__ void qb_tc_epi_chunk(const float* bias, int c, const uint32_t (&v)[16], float (&h)[16]) {
    const float4* B4 = reinterpret_cast<const float4*>(bias + c);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const float4 b = B4[g];
        float2 z0 = __fadd2_rn(make_float2(__uint_as_float(v[4 * g + 0]), __uint_as_float(v[4 * g + 1])), make_float2(b.x, b.y));
        float2 z1 = __fadd2_rn(make_float2(__uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3])), make_float2(b.z, b.w));
        qb_tc_act4<ACT>(z0, z1);
        h[4 * g + 0] = z0.x; h[4 * g + 1] = z0.y; h[4 * g + 2] = z1.x; h[4 * g + 3] = z1.y;
    }
}

// narrow output layer: yacc[o] (two partial sums each) += W_last[o][c .. c+15] . h
template <int OD>
__device__ __forceinline__ void qb_tc_dot_chunk(const QbTcPlan& tp, const float* F, int c, const float (&h)[16], float2 (&yacc)[OD]) {
#pragma unroll
    for (int o = 0; o < OD; ++o) {
        if (o < tp.out_dim) {
            const float4* w4 = reinterpret_cast<const float4*>(F + tp.wl + o * tp.kl + c);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const float4 w = w4[g];
                yacc[o] = __ffma2_rn(make_float2(w.x, w.y), make_float2(h[4 * g + 0], h[4 * g + 1]), yacc[o]);
                yacc[o] = __ffma2_rn(make_float2(w.z, w.w), make_float2(h[4 * g + 2], h[4 * g + 3]), yacc[o]);
            }
        }
    }
}

template <int NI, int ACT>
__device__ __forceinline__ void qb_tc_layer0(const QbTcPlan& tp, const float* F, uint32_t tl, const float (&xr)[NI]) {
#pragma unroll 1
    for (int c = 0; c < tp.h0; c += 16) {
        float h[16];
        qb_tc_l0_chunk<NI, ACT>(tp, F, c, xr, h);
        qb_tc_split_store(tl + c, tl + tp.a_lo_col + c, h);
    }
}

// hidden-layer epilogue: D -> +bias -> act -> next A operand
template <int ACT>
__device__ __forceinline__ void qb_tc_epi_mid(const QbTcPlan& tp, const QbTcLayer& L, const float* F, uint32_t tl) {
#pragma unroll 1
    for (int c = 0; c < L.n_out; c += 16) {
        uint32_t v[16];
        qb_tmem_ld16(tl + tp.d_col + c, v);
        qb_tmem_ld_wait16(v);
        float h[16];
        qb_tc_epi_chunk<ACT>(F + L.bias, c, v, h);
        qb_tc_split_store(tl + c, tl + tp.a_lo_col + c, h);
    }
}

// last hidden layer's epilogue fused with the narrow output layer
template <int ACT>
__device__ __forceinline__ void qb_tc_epi_last(const QbTcPlan& tp, const QbTcLayer& L, const float* F, uint32_t tl,
                                               float2 (&yacc)[4]) {
#pragma unroll 1
    for (int c = 0; c < L.n_out; c += 16) {
        uint32_t v[16];
        qb_tmem_ld16(tl + tp.d_col + c, v);
        qb_tmem_ld_wait16(v);
        float h[16];
        qb_tc_epi_chunk<ACT>(F + L.bias, c, v, h);
        qb_tc_dot_chunk<4>(tp, F, c, h, yacc);
    }
}

// network output o from the finished dot product (bias, last activation, optional exp)
__device__ __forceinline__ float qb_tc_out(const QbTcPlan& tp, const float* F, int o, float acc) {
    float v = acc + F[tp.bl + o];
    if (tp.act_last == QB_ACT_TANH) v = qb_tanh_prescaled(v);
    else if (tp.act_last == QB_ACT_RELU) v = fmaxf(v, 0.0f);
    if (tp.final_exp) v = expf(v);
    return v;
}
__device__ __forceinline__ void qb_tc_finish_out(const QbTcPlan& tp, const float* F, const float2 (&yacc)[4], float (&yout)[4]) {
#pragma unroll
    for (int o = 0; o < 4; ++o) yout[o] = o < tp.out_dim ? qb_tc_out(tp, F, o, yacc[o].x + yacc[o].y) : 0.0f;
}

template <int NI>
__device__ __forceinline__ void qb_tc_load_x(const QbTcPlan& tp, const float* __restrict__ x, int64_t p, bool live, float (&xr)[NI]) {
#pragma unroll
    for (int q = 0; q < NI; ++q) {
        float v = 0.0f;
        if (q < tp.in_dim && live) v = __ldg(x + p * tp.in_dim + q);
        xr[q] = (q == tp.in_dim) ? 1.0f : v;                       // slot in_dim: bias (selects, no indexed stores)
    }
}

// forward pass of the tile of 128 points starting at p0 (thread t = point p0+t); leaves the network output of this
// thread's point in yout[0..out_dim)
template <int NI>
__device__ __forceinline__ void qb_tc_forward_tile(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                                   const float* __restrict__ x, int64_t p, bool live, float (&yout)[4]) {
    const float* F = reinterpret_cast<const float*>(smem + tp.fl_base);
    const uint32_t tl = cx.tmem + ((uint32_t)((threadIdx.x >> 5) * 32) << 16);
    float xr[NI];
    qb_tc_load_x<NI>(tp, x, p, live, xr);
    switch (tp.act0) {
        case QB_ACT_TANH: qb_tc_layer0<NI, QB_ACT_TANH>(tp, F, tl, xr); break;
        case QB_ACT_RELU: qb_tc_layer0<NI, QB_ACT_RELU>(tp, F, tl, xr); break;
        default: qb_tc_layer0<NI, QB_ACT_IDENTITY>(tp, F, tl, xr); break;
    }
    float2 yacc[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) yacc[o] = make_float2(0.0f, 0.0f);
    const int last_tc = tp.n_layers - 2;
    for (int l = 1; l <= last_tc; ++l) {
        const QbTcLayer& L = tp.L[l];
        // A (and the reads of D by the previous tile / layer) are complete in every thread before the MMAs start
        qb_tmem_st_wait();
        qb_tc_fence_before();
        __syncthreads();
        if (threadIdx.x < 32) {
            qb_tc_fence_after();
            qb_tc_issue_warp(tp, L, cx, smem, 0u);
        }
        qb_mbar_wait_timed(cx.bar, cx.phase);
        cx.phase ^= 1u;
        qb_tc_fence_after();
        if (l < last_tc) {
            switch (L.act) {
                case QB_ACT_TANH: qb_tc_epi_mid<QB_ACT_TANH>(tp, L, F, tl); break;
                case QB_ACT_RELU: qb_tc_epi_mid<QB_ACT_RELU>(tp, L, F, tl); break;
                default: qb_tc_epi_mid<QB_ACT_IDENTITY>(tp, L, F, tl); break;
            }
        } else {
            switch (L.act) {
                case QB_ACT_TANH: qb_tc_epi_last<QB_ACT_TANH>(tp, L, F, tl, yacc); break;
                case QB_ACT_RELU: qb_tc_epi_last<QB_ACT_RELU>(tp, L, F, tl, yacc); break;
                default: qb_tc_epi_last<QB_ACT_IDENTITY>(tp, L, F, tl, yacc); break;
            }
        }
    }
    qb_tc_finish_out(tp, F, yacc, yout);
}

// sum of squared residuals over points [n0, n1) for the staged parameter vector (block-wide result)
template <int NI>
__device__ __forceinline__ double qb_tc_eval_ni(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                                const float* __restrict__ x, const float* __restrict__ y,
                                                int64_t n0, int64_t n1) {
    float ssq = 0.0f;
    for (int64_t p0 = n0; p0 < n1; p0 += 128) {
        const int64_t p = p0 + threadIdx.x;
        const bool live = p < n1;
        float yv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int o = 0; o < 4; ++o) if (o < tp.out_dim && live) yv[o] = __ldg(y + p * tp.out_dim + o);
        float yo[4];
        qb_tc_forward_tile<NI>(tp, cx, smem, x, p, live, yo);
        if (live) {
#pragma unroll
            for (int o = 0; o < 4; ++o) if (o < tp.out_dim) { const float r = yv[o] - yo[o]; ssq = fmaf(r, r, ssq); }
        }
    }
    return qb_block_sum((double)ssq, reinterpret_cast<double*>(smem));
}

// Software-pipelined tile loop for networks with ONE tensor-core layer (in -> H -> H' -> out, same activation on both
// hidden layers).  G = 2 (H, H' <= 64, 256 threads, two blocks per SM) or 4 (<= 128, 512 threads, one block per SM)
// warps share each quarter of the tile's 128 points (tensor-memory lanes) and split the units / accumulator columns
// in chunks of 16 (thread group g owns chunks g and G+g), so G times as many warps hide the MUFU / tcgen05.ld latencies
// for the same tensor-memory footprint.
// Per tile: wait for the MMAs of tile t, compute layer 0 of tile t+1 straight into tensor memory, start the MMAs of
// tile t+1 into the OTHER accumulator buffer (D is double-buffered), and only then read D(t) and do the tanh /
// dot-product epilogue of tile t, which overlaps those MMAs; no register array lives across a wait.
// The G partial dot products of a point meet through shared memory one tile later (ybuf, double-buffered, named
// producer / consumer barriers); group 0 finishes the point and hands the network output to the sink.
// FULL: both hidden widths are 32*G, so every thread owns two full chunks and the chunk guards vanish (no branches
// between the chunks: the compiler interleaves their independent dependency chains).
struct QbSinkSsq {              // squared residuals against y (kernels 1 and 3)
    const float* __restrict__ y; int od; float ssq;
    template <int OD> __device__ __forceinline__ void prefetch(int64_t p, bool live, float (&s)[OD]) const {
#pragma unroll
        for (int o = 0; o < OD; ++o) { s[o] = 0.0f; if (o < od && live) s[o] = __ldg(y + p * od + o); }
    }
    template <int OD> __device__ __forceinline__ void consume(int64_t, bool live, const float (&s)[OD], const float (&yo)[OD]) {
        if (live) {
#pragma unroll
            for (int o = 0; o < OD; ++o) if (o < od) { const float r = s[o] - yo[o]; ssq = fmaf(r, r, ssq); }
        }
    }
};
struct QbSinkStore {            // network outputs to out[p, o] (kernel 4)
    float* __restrict__ out; int od;
    template <int OD> __device__ __forceinline__ void prefetch(int64_t, bool, float (&s)[OD]) const {
#pragma unroll
        for (int o = 0; o < OD; ++o) s[o] = 0.0f;
    }
    template <int OD> __device__ __forceinline__ void consume(int64_t p, bool live, const float (&)[OD], const float (&yo)[OD]) {
        if (live) {
#pragma unroll
            for (int o = 0; o < OD; ++o) if (o < od) out[p * od + o] = yo[o];
        }
    }
};

template <int NI, int ACT, int OD, bool FULL, int G, typename Sink, bool HALFK_REQ = false>
__device__ __forceinline__ Sink qb_tc_pipe_run(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                               const float* __restrict__ x, int64_t n0, int64_t n1, Sink sink) {
    const float* F = reinterpret_cast<const float*>(smem + tp.fl_base);
    float* ybuf = reinterpret_cast<float*>(smem + tp.ybuf);          // [2][3][4][128]
    const int grp = threadIdx.x >> 7, pt = threadIdx.x & 127;
    // named barriers of the G warps of a quarter: id 1+w for even tiles, 5+w for odd tiles (a producer may run one tile
    // ahead of the consumer, never two: see the a_ready / mma_done chain below)
    const int pair_id = 1 + ((threadIdx.x >> 5) & 3);
    const uint32_t tl = cx.tmem + ((uint32_t)(((threadIdx.x >> 5) & 3) * 32) << 16);
    const QbTcLayer& L = tp.L[1];
    const int K = tp.h0, N = L.n_out, od = tp.out_dim;
    // HALFK (K = N = 64, two column groups): the MMAs of the first half of K are committed separately, so the first
    // layer-0 chunk of tile t+1 (columns < 32) is written while the second half of tile t's MMAs is still running
    constexpr bool HALFK = (FULL && G == 2) || HALFK_REQ;          // HALFK_REQ: the caller checked K == 32*G
    const int ntiles = (int)((n1 - n0 + 127) / 128);   // tile counters are 32-bit: this loop is register-bound
    const int64_t pbase = n0 + pt;                     // this thread's point of tile 0
    float xn[NI];
    float yprev[OD], sp[OD];
#pragma unroll
    for (int o = 0; o < OD; ++o) { yprev[o] = 0.0f; sp[o] = 0.0f; }
    __syncthreads();           // the previous evaluation's readers of ybuf / F are done (weights were restaged)
    if (ntiles > 0) {
        qb_tc_load_x<NI>(tp, x, pbase, pbase < n1, xn);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int c = (G * j + grp) * 16;
            if (FULL || c < K) {
                float h[16];
                qb_tc_l0_chunk<NI, ACT>(tp, F, c, xn, h);
                qb_tc_split_store(tl + c, tl + tp.a_lo_col + c, h);
            }
        }
        qb_tmem_st_wait();
        qb_tc_fence_before();
        qb_mbar_arrive(cx.abar);
        if (threadIdx.x < 32) {
            qb_mbar_wait_timed(cx.abar, cx.aphase);
            qb_tc_fence_after();
            qb_tc_issue_warp<HALFK, 4 * G>(tp, L, cx, smem, 0u);
        }
        cx.aphase ^= 1u;
    }
    for (int t = 0; t < ntiles; ++t) {
        const bool more = t + 1 < ntiles;
        const int64_t pc = pbase + (int64_t)t * 128;                 // this thread's point of tile t
        float sv[OD];
        if (grp == 0) sink.template prefetch<OD>(pc, pc < n1, sv);
        if constexpr (HALFK) {
            qb_mbar_wait_timed(cx.hbar, cx.hphase);                        // first K-half of tile t done: A columns [0,32) are free
            cx.hphase ^= 1u;
            qb_tc_fence_after();
            if (more) {
                qb_tc_load_x<NI>(tp, x, pc + 128, pc + 128 < n1, xn);
                float h[16];
                qb_tc_l0_chunk<NI, ACT>(tp, F, grp * 16, xn, h);
                qb_tc_split_store(tl + grp * 16, tl + tp.a_lo_col + grp * 16, h);
            }
        }
        qb_mbar_wait_timed(cx.bar, cx.phase);                              // MMAs of tile t complete: A is free, D[t&1] is ready
        cx.phase ^= 1u;
        qb_tc_fence_after();
        // finish tile t-1 (the partner warps published their partial sums one epilogue ago); these reads come before
        // this thread's arrival below, which is what lets the partners reuse the slot two tiles later
        if (grp == 0 && t > 0) {
            asm volatile("bar.sync %0, %1;" :: "r"(pair_id + (int)((t - 1) & 1) * 4), "r"(32 * G) : "memory");
            const float* yb = ybuf + ((t - 1) & 1) * 1536 + pt;
            float yo[OD];
#pragma unroll
            for (int o = 0; o < OD; ++o) {
                float acc = yprev[o];
#pragma unroll
                for (int g = 1; g < G; ++g) acc += yb[((g - 1) * 4 + o) * 128];
                yo[o] = o < od ? qb_tc_out(tp, F, o, acc) : 0.0f;
            }
            sink.template consume<OD>(pc - 128, pc - 128 < n1, sp, yo);
        }
        if (more) {
            // layer 0 of tile t+1 straight into tensor memory, then let warp 0 start the MMAs of tile t+1 into the other
            // accumulator buffer (x is L1/L2-resident and shared by every chain: no prefetch registers are spent on it)
            if constexpr (!HALFK) qb_tc_load_x<NI>(tp, x, pc + 128, pc + 128 < n1, xn);
#pragma unroll
            for (int j = HALFK ? 1 : 0; j < 2; ++j) {
                const int c = (G * j + grp) * 16;
                if (FULL || c < K) {
                    float h[16];
                    qb_tc_l0_chunk<NI, ACT>(tp, F, c, xn, h);
                    qb_tc_split_store(tl + c, tl + tp.a_lo_col + c, h);
                }
            }
            qb_tmem_st_wait();
            qb_tc_fence_before();
            qb_mbar_arrive(cx.abar);
            if (threadIdx.x < 32) {
                qb_mbar_wait_timed(cx.abar, cx.aphase);
                qb_tc_fence_after();
                qb_tc_issue_warp<HALFK, 4 * G>(tp, L, cx, smem, (uint32_t)((t + 1) & 1) * (uint32_t)N);
            }
            cx.aphase ^= 1u;
        }
        // epilogue of tile t from D[t&1] (overlaps the MMAs of tile t+1, which write the other buffer)
        float2 yacc[OD];
#pragma unroll
        for (int o = 0; o < OD; ++o) yacc[o] = make_float2(0.0f, 0.0f);
        const uint32_t dcol = tp.d_col + (uint32_t)(t & 1) * (uint32_t)N;
        if constexpr (FULL) {
            // both accumulator chunks are requested before either is processed (the hot instantiation has the registers)
            uint32_t v[2][16];
#pragma unroll
            for (int j = 0; j < 2; ++j) qb_tmem_ld16(tl + dcol + (G * j + grp) * 16, v[j]);
#pragma unroll
            for (int j = 0; j < 2; ++j) qb_tmem_ld_wait16(v[j]);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int c = (G * j + grp) * 16;
                float hh[16];
                qb_tc_epi_chunk<ACT>(F + L.bias, c, v[j], hh);
                qb_tc_dot_chunk<OD>(tp, F, c, hh, yacc);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int c = (G * j + grp) * 16;
                if (c < N) {
                    uint32_t v[16];
                    qb_tmem_ld16(tl + dcol + c, v);
                    qb_tmem_ld_wait16(v);
                    float hh[16];
                    qb_tc_epi_chunk<ACT>(F + L.bias, c, v, hh);
                    qb_tc_dot_chunk<OD>(tp, F, c, hh, yacc);
                }
            }
        }
        if (grp != 0) {
            float* yb = ybuf + (t & 1) * 1536 + ((grp - 1) * 4) * 128 + pt;
#pragma unroll
            for (int o = 0; o < OD; ++o) if (o < od) yb[o * 128] = yacc[o].x + yacc[o].y;
            asm volatile("bar.arrive %0, %1;" :: "r"(pair_id + (int)(t & 1) * 4), "r"(32 * G) : "memory");
        } else {
#pragma unroll
            for (int o = 0; o < OD; ++o) { yprev[o] = yacc[o].x + yacc[o].y; sp[o] = sv[o]; }
        }
    }
    if (grp == 0 && ntiles > 0) {
        asm volatile("bar.sync %0, %1;" :: "r"(pair_id + (int)((ntiles - 1) & 1) * 4), "r"(32 * G) : "memory");
        const float* yb = ybuf + ((ntiles - 1) & 1) * 1536 + pt;
        float yo[OD];
#pragma unroll
        for (int o = 0; o < OD; ++o) {
            float acc = yprev[o];
#pragma unroll
            for (int g = 1; g < G; ++g) acc += yb[((g - 1) * 4 + o) * 128];
            yo[o] = o < od ? qb_tc_out(tp, F, o, acc) : 0.0f;
        }
        const int64_t pl = pbase + (int64_t)(ntiles - 1) * 128;
        sink.template consume<OD>(pl, pl < n1, sp, yo);
    }
    return sink;
}

template <int NI, int ACT, int OD, bool FULL, int G>
__device__ __forceinline__ double qb_tc_eval_pipe(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                                  const float* __restrict__ x, const float* __restrict__ y,
                                                  int64_t n0, int64_t n1) {
    QbSinkSsq sink;
    sink.y = y; sink.od = tp.out_dim; sink.ssq = 0.0f;
    const QbSinkSsq done = qb_tc_pipe_run<NI, ACT, OD, FULL, G>(tp, cx, smem, x, n0, n1, sink);
    return qb_block_sum((double)done.ssq, reinterpret_cast<double*>(smem));
}

// Everything but the most common shape (<= 3 inputs, tanh, one 64x64 tensor-core layer, one output) is compiled out of line: inlining
// all variants into the chain kernels made them so large that the compiler stopped unrolling the chunk loops and put
// the register arrays in local memory.
static __device__ __noinline__ double qb_tc_eval_other(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                                const float* __restrict__ x, const float* __restrict__ y,
                                                int64_t n0, int64_t n1) {
    if (tp.pipe == 4) {
        if (tp.act0 == QB_ACT_TANH) {
            if (tp.ni == 12) return qb_tc_eval_pipe<12, QB_ACT_TANH, 4, false, 4>(tp, cx, smem, x, y, n0, n1);
            return qb_tc_eval_pipe<16, QB_ACT_TANH, 4, false, 4>(tp, cx, smem, x, y, n0, n1);
        }
        return qb_tc_eval_pipe<16, QB_ACT_RELU, 4, false, 4>(tp, cx, smem, x, y, n0, n1);
    }
    if (tp.pipe) {
        if (tp.ni == 4 && tp.act0 == QB_ACT_TANH) return qb_tc_eval_pipe<4, QB_ACT_TANH, 4, false, 2>(tp, cx, smem, x, y, n0, n1);
        if (tp.ni == 4) return qb_tc_eval_pipe<4, QB_ACT_RELU, 4, false, 2>(tp, cx, smem, x, y, n0, n1);
        if (tp.act0 == QB_ACT_TANH) return qb_tc_eval_pipe<16, QB_ACT_TANH, 4, false, 2>(tp, cx, smem, x, y, n0, n1);
        return qb_tc_eval_pipe<16, QB_ACT_RELU, 4, false, 2>(tp, cx, smem, x, y, n0, n1);
    }
    if (tp.ni == 4) return qb_tc_eval_ni<4>(tp, cx, smem, x, y, n0, n1);
    return qb_tc_eval_ni<16>(tp, cx, smem, x, y, n0, n1);
}

// The chain kernel and kernel 1 exist in two instantiations: HOT contains only the config-5 shape (<= 3 inputs, tanh,
// one 64x64 tensor-core layer, one output), fully inlined; the general one calls qb_tc_eval_other.  Keeping them apart
// stops unrelated variants from disturbing the register allocation of the hot loop (it sits exactly at 128 registers:
// every perturbation showed up as spills and -3..10 %).
__host__ __device__ __forceinline__ bool qb_tc_is_hot(const QbTcPlan& tp) {
    return tp.pipe == 2 && tp.ni == 4 && tp.act0 == QB_ACT_TANH && tp.out_dim == 1 && tp.h0 == 64 && tp.kl == 64 &&
           tp.L[1].n_out == 64;
}
// the shapes the warp-specialised path (qb_tc3.cuh) covers: in -> H -> H -> 1 with tanh, H = 64 (in <= 7) or 128 (in <= 15);
// returns H or 0
__host__ __device__ __forceinline__ int qb_tc_v3_shape(const QbTcPlan& tp) {
    if (!tp.pipe || tp.act0 != QB_ACT_TANH || tp.out_dim != 1 || tp.h0 != tp.kl || tp.L[1].n_out != tp.h0) return 0;
    if (tp.h0 == 64 && tp.in_dim <= 7) return 64;
    if (tp.h0 == 128 && tp.in_dim <= 15) return 128;
    return 0;
}
template <bool HOT>
__device__ __forceinline__ double qb_tc_eval(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                             const float* __restrict__ x, const float* __restrict__ y,
                                             int64_t n0, int64_t n1) {
    if constexpr (HOT) {
        return qb_tc_eval_pipe<4, QB_ACT_TANH, 1, true, 2>(tp, cx, smem, x, y, n0, n1);
    } else {
        QbTcCtx c2 = cx;            // only this copy has its address taken (keeps cx itself in registers)
        const double r = qb_tc_eval_other(tp, c2, smem, x, y, n0, n1);
        cx = c2;
        return r;
    }
}

// kernel 4 on the tensor cores: network outputs of points [n0, n1) for the staged parameter vector -> out[p, o]
__device__ __forceinline__ void qb_tc_predict(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                              const float* __restrict__ x, float* __restrict__ out, int64_t n0, int64_t n1) {
    QbSinkStore sink;
    sink.out = out; sink.od = tp.out_dim;
    if (tp.pipe == 4) {
        if (tp.act0 == QB_ACT_TANH && tp.ni == 12 && tp.h0 == 128)      // config-3 shape: half-K commits
            qb_tc_pipe_run<12, QB_ACT_TANH, 4, false, 4, QbSinkStore, true>(tp, cx, smem, x, n0, n1, sink);
        else if (tp.act0 == QB_ACT_TANH && tp.ni == 12) qb_tc_pipe_run<12, QB_ACT_TANH, 4, false, 4>(tp, cx, smem, x, n0, n1, sink);
        else if (tp.act0 == QB_ACT_TANH) qb_tc_pipe_run<16, QB_ACT_TANH, 4, false, 4>(tp, cx, smem, x, n0, n1, sink);
        else qb_tc_pipe_run<16, QB_ACT_RELU, 4, false, 4>(tp, cx, smem, x, n0, n1, sink);
    } else if (tp.pipe) {
        if (tp.ni == 4 && tp.act0 == QB_ACT_TANH) qb_tc_pipe_run<4, QB_ACT_TANH, 4, false, 2>(tp, cx, smem, x, n0, n1, sink);
        else if (tp.ni == 4) qb_tc_pipe_run<4, QB_ACT_RELU, 4, false, 2>(tp, cx, smem, x, n0, n1, sink);
        else if (tp.act0 == QB_ACT_TANH) qb_tc_pipe_run<16, QB_ACT_TANH, 4, false, 2>(tp, cx, smem, x, n0, n1, sink);
        else qb_tc_pipe_run<16, QB_ACT_RELU, 4, false, 2>(tp, cx, smem, x, n0, n1, sink);
    } else {
        for (int64_t p0 = n0; p0 < n1; p0 += 128) {
            const int64_t p = p0 + threadIdx.x;
            float yo[4];
            if (tp.ni == 4) qb_tc_forward_tile<4>(tp, cx, smem, x, p, p < n1, yo);
            else qb_tc_forward_tile<16>(tp, cx, smem, x, p, p < n1, yo);
            if (p < n1) for (int o = 0; o < tp.out_dim; ++o) out[p * tp.out_dim + o] = yo[o];
        }
    }
}
#endif  // __CUDACC__
