// Warp-specialised tensor-core value path for the hot shape (in <= 7 -> 64 -> 64 -> 1, tanh): kernels 1 and 3 at the
// config-5 shape.  Same arithmetic contract as qb_tc.cuh (fp32-level accuracy through split operands), different
// machine mapping:
//   * 8 compute warps (256 threads: thread = one of the tile's 128 points x one half of the 64 columns) and ONE issue
//     warp (warp 8) that never computes: it stages the x tile, issues every tcgen05.mma and commits them to mbarriers.
//     No compute warp ever issues an MMA or waits for the other warps to arrive (the old loop spent 20 % of its stall
//     samples there and ~1100 cycles per tile of warp 0 on the issue itself).
//   * layer 0 runs on the tensor cores as well: D0[128 x 64] = X[128 x 8] * W0^T, kind::tf32, 3 passes, both operands in
//     shared memory.  X = (x_0 .. x_{in-1}, 1, 0 ..): the bias rides in the K slot that holds 1.0.  The issue warp
//     loads x two tiles ahead, splits it into tf32 hi + lo and writes the canonical K-major tile; the compute warps
//     never touch x.
//   * the hidden 64x64 GEMM runs as kind::f16 with fp16 hi + lo splits ("3 x FP16": a_hi*b_hi + a_lo*b_hi + a_hi*b_lo,
//     fp32 accumulation): K = 16 per MMA instead of 8 (12 MMAs per tile instead of 24) and the A operand takes 64
//     tensor-memory columns instead of 128.  fp16 has 11 significant bits like tf32; its narrow exponent is handled
//     by exact power-of-two scaling: activations are produced as 2^14 * sigmoid (in (2^-16, 2^14]) and the weights
//     are scaled per parameter vector so that max |w| lies in [2^13, 2^14): every lo part within 2^16 of the largest
//     is a normal fp16 number, smaller ones carry an absolute error of 2^-25 in units of the scaled maximum.
//   * tanh = 1 - 2 s with s = 1 / (1 + 2^z'): the affine part is folded into the NEXT layer's weights and bias at
//     staging (W' = -2 W, b' = b + sum_k W_k), so the epilogues produce s only (2 packed FMAs per 4 activations less).
// Tensor memory (256 columns per block, two blocks per SM): D0 x 2 [0,128) | A_hi [128,160) | -A_lo [160,192) | D1 [192,256).
// Per tile t:   issue warp:     wait a_ready(t) -> MMA0(t+2) into D0[t&1] -> commit d0_full -> wait d1_free(t-1) -> MMA1(t)
//                               -> commit d1_full -> stage X(t+3)
//               compute warps:  EPI1(t-1) [D1 -> registers -> arrive d1_free -> s -> dot with the output row]  then
//                               EPI0(t+1) [D0[(t+1)&1] -> 2^14 s -> fp16 hi/lo; wait d1_full(t) = "A is free" -> A]
//                               -> arrive a_ready(t+1)
// Layer 0 runs two tiles ahead (D0 is double-buffered), so d0_full is never waited for in steady state; between a
// warp's arrival on a_ready(t) and its need for d1_full(t) lies almost a whole tile of its own work (EPI1(t-1) and the
// arithmetic of EPI0(t+1)), which is the slack that absorbs the skew between the eight compute warps and the
// ~800 cycles from the last arrival to the commit of MMA1(t).  D1 needs no second buffer: its reader copies it to
// registers first thing and releases it at once.
#pragma once
#include "qb_tc.cuh"
#include "qb_tcgen05.cuh"

#ifdef __CUDACC__
// Development aid (-DQB3_TRACE, scripts/tc3_trace.py): SM-clock stamps of the phases of every compute warp.
#ifdef QB3_TRACE
enum { QB3_TR_BLOCKS = 296, QB3_TR_WARPS = 17, QB3_TR_TILES = 82, QB3_TR_EV = 8 };
__device__ unsigned int qb3_trace_buf[QB3_TR_BLOCKS * QB3_TR_WARPS * QB3_TR_TILES * QB3_TR_EV];
__device__ unsigned int qb3_trace_sm[QB3_TR_BLOCKS];
#define QB3_STAMP(tile, ev) do { if ((threadIdx.x & 31) == 0 && blockIdx.x < QB3_TR_BLOCKS && blockIdx.y == 0 && (tile) < QB3_TR_TILES) \
    qb3_trace_buf[((blockIdx.x * QB3_TR_WARPS + (threadIdx.x >> 5)) * QB3_TR_TILES + (tile)) * QB3_TR_EV + (ev)] = (unsigned int)clock64(); } while (0)
#else
#define QB3_STAMP(tile, ev) do { } while (0)
#endif
enum { QB3_D0F = 320, QB3_ARDY = 336, QB3_D1F = 344, QB3_D1FREE = 352, QB3_D0F1 = 360 };   // mbarriers in the shared-memory header
       // (d0_full exists once per D0 buffer: layer 0 runs two tiles ahead and a parity wait must never fall two phases behind)
// Hidden width H (64: config 5, two blocks per SM; 128: config 3, one block per SM): G = H/32 column groups of 128 compute
// threads each, the issue warp comes after them; tensor-memory columns D0 x 2 | A_hi | -A_lo | D1
template <int H> struct Qb3Dim {
    static constexpr int G = H / 32, NCOMP = 128 * G, ISSUER = 4 * G;
    static constexpr int COL_AHI = 2 * H, COL_ALO = 2 * H + H / 2, COL_D1 = 3 * H;
};

// all threads; tensor-memory allocation (the mbarriers are (re)initialised by every evaluation)
template <int H>
__device__ __forceinline__ void qb_tc3_init(const QbTcPlan& tp, unsigned char* smem, QbTcCtx& cx) {
    constexpr uint32_t QB3_NCOMPUTE = Qb3Dim<H>::NCOMP;
    const uint32_t x = (uint32_t)tp.v3_xbar;
    const uint32_t bars[8] = {QB3_D0F, QB3_ARDY, QB3_D1F, QB3_D1FREE, QB3_D0F1, x, x + 8u, x + 16u};
    const uint32_t counts[8] = {1u, QB3_NCOMPUTE, 1u, QB3_NCOMPUTE, 1u, 1u, 1u, 1u};   // x_full[3]: their phases run across evaluations
    cx.tmem = qb_tc_start(smem, QB_TC_SLOT_OFF, (uint32_t)tp.tmem_cols, bars, counts);
    cx.bar = cx.abar = cx.hbar = 0; cx.phase = cx.aphase = cx.hphase = 0;
}
// between evaluations (thread 0): the five barriers of the tile loop start again at parity 0
template <int H>
__device__ __forceinline__ void qb_tc3_reset_barriers(unsigned char* smem) {
    const uint32_t bars[5] = {QB3_D0F, QB3_ARDY, QB3_D1F, QB3_D1FREE, QB3_D0F1};
    const uint32_t counts[5] = {1u, (uint32_t)Qb3Dim<H>::NCOMP, 1u, (uint32_t)Qb3Dim<H>::NCOMP, 1u};
    qb_mbar_reset(smem, bars, counts);
}

// flat theta (global) -> shared operands of the three layers.  All threads of the block; ends with the async-proxy fence.
//   W0  : tf32 hi / lo, [64 x 8] canonical K-major (k < in: weight, k == in: bias, else 0), times 2 log2 e
//   W1  : fp16 hi / lo / -hi of -2 * 2 log2 e * 2^sW * W1 (the -2: tanh = 1 - 2 s), [64 x 64] canonical K-major
//         (core matrix = 8 rows x 8 halves; LBO 128 B, SBO 1024 B); -hi multiplies the negated lo parts of A
//   F[bias1 + j] = 2 log2 e * (b1_j + sum_k W1_jk);  F[c1] = 2^(-14 - sW)  (D1 is in units of 2^14 * 2^sW)
//   F[wl + k] = -2 * 2^-14 * sl * wl_k (the epilogue produces 2^14 s);  F[bl] = sl * (bl + sum_k wl_k)
// wmax: this thread's share of max |W1| when the caller has already looked at every W1 entry (all threads pass >= 0,
// block-uniformly), else < 0 and the entries are scanned here
template <int H, int K0>
__device__ __forceinline__ void qb_tc3_stage(const QbTcPlan& tp, unsigned char* smem, const float* __restrict__ theta, float wmax) {
    constexpr int NCW = Qb3Dim<H>::ISSUER;          // compute warps
    float* F = reinterpret_cast<float*>(smem + tp.fl_base);
    double* red = reinterpret_cast<double*>(smem);
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
    const float fold = 2.8853900817779268f;
    const QbTcLayer& L = tp.L[1];
    // ---- scale of W1: largest magnitude -> [2^13, 2^14)
    float mx = fmaxf(wmax, 0.0f);
    if (wmax < 0.0f)
        for (int e = tid; e < H * H; e += nt) mx = fmaxf(mx, fabsf(theta[L.w_off + e]));
    uint32_t mb = __reduce_max_sync(0xffffffffu, __float_as_uint(mx));
    __syncthreads();                       // the previous evaluation's readers of F / red are done
    if (lane == 0) reinterpret_cast<uint32_t*>(red)[wid] = mb;
    __syncthreads();
    mb = 0;
    for (int w = 0; w < (nt + 31) >> 5; ++w) mb = max(mb, reinterpret_cast<const uint32_t*>(red)[w]);
    int sW = 0;
    {
        const float m = __uint_as_float(mb) * fold;
        if (m > 0.0f && m < 3.0e38f) sW = 13 - ilogbf(m);
        sW = max(-60, min(60, sW));
    }
    const float wscale = -2.0f * fold * __uint_as_float((uint32_t)(127 + sW) << 23);
    // ---- W0 (tf32 hi / lo): element (n, k) at float index ((n/8)*(K0/4) + k/4)*32 + (n%8)*4 + k%4
    {
        float* hi = reinterpret_cast<float*>(smem + tp.v3_w0);
        float* lo = hi + H * K0;
        for (int e = tid; e < H * K0; e += nt) {
            const int n = e / K0, k = e % K0;
            float v = 0.0f;
            if (k < tp.in_dim) v = theta[tp.w0_off + n * tp.in_dim + k] * fold;
            else if (k == tp.in_dim && tp.b0_off >= 0) v = theta[tp.b0_off + n] * fold;
            const float h = qb_tf32_hi(v);
            const int idx = ((n >> 3) * (K0 / 4) + (k >> 2)) * 32 + (n & 7) * 4 + (k & 3);
            hi[idx] = h; lo[idx] = v - h;
        }
    }
    // ---- W1 (fp16 hi / lo) and its row sums: warp w of the first eight takes rows w, w+8, ..; lane = a pair of columns
    if (wid < NCW) {
        uint32_t* hi = reinterpret_cast<uint32_t*>(smem + tp.v3_w1);
        uint32_t* lo = hi + H * H / 2;
        uint32_t* nhi = lo + H * H / 2;
        for (int n = wid; n < H; n += NCW) {
            float s = 0.0f;                        // pairwise tree: the error stays below that of the GEMM's own fp32 sums
#pragma unroll
            for (int jj = 0; jj < H / 64; ++jj) {
                const int k = (lane + 32 * jj) * 2;
                const float w0 = theta[L.w_off + n * H + k], w1 = theta[L.w_off + n * H + k + 1];
                uint32_t h2, l2;
                qb_split_f16_nlo(w0 * wscale, w1 * wscale, h2, l2);
                const int idx = (((n >> 3) * (H / 8) + (k >> 3)) * 64 + (n & 7) * 8 + (k & 7)) >> 1;      // 32-bit word index
                hi[idx] = h2; lo[idx] = l2 ^ 0x80008000u; nhi[idx] = h2 ^ 0x80008000u;
                s += w0 + w1;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
            if (lane == 0) F[L.bias + n] = fold * ((L.b_off >= 0 ? theta[L.b_off + n] : 0.0f) + s);
        }
    } else if (wid == NCW) {
        // ---- output row: -2 sl wl, bias sl (bl + sum wl)
        const float sl = tp.act_last == QB_ACT_TANH ? fold : 1.0f;
        double s = 0.0;
#pragma unroll
        for (int jj = 0; jj < H / 32; ++jj) {
            const float a = theta[tp.wl_off + lane + 32 * jj];
            F[tp.wl + lane + 32 * jj] = -1.220703125e-04f * sl * a;     // -2 * 2^-14
            s += (double)a;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0) {
            F[tp.bl] = (float)((double)sl * ((tp.bl_off >= 0 ? (double)theta[tp.bl_off] : 0.0) + s));
            F[tp.v3_c1] = __uint_as_float((uint32_t)(127 - 14 - sW) << 23);
        }
    }
    qb_fence_proxy_async();
}

// 2^14 / (1 + 2^z) for EIGHT pre-activations with ONE reciprocal (the MUFU pipe, 16 results/clk/SM, is the first
// bound of this kernel: 9 MUFU operations per 8 activations).  d_i = 2^-14 (1 + 2^min(z_i, 26)) lies in [2^-14, 2^12], so
// the product of eight stays inside the fp32 range; 1/d_i comes out of a product tree of the other seven times the
// reciprocal of the whole product: 12 multiplies (8 of them packed) for 8 values, the same count as two groups of four.
// The clamp at 26 is exact for tanh: 1 - 2/(1 + 2^26) rounds to 1.0f.  min.NaN keeps NaN pre-activations NaN.
__device__ __forceinline__ void qb3_sig8(float2 (&v)[4]) {
    const float2 c = make_float2(6.103515625e-05f, 6.103515625e-05f);        // 2^-14
    float2 d[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 e;
        e.x = qb_ex2(qb_min_nan(v[i].x, 26.0f)); e.y = qb_ex2(qb_min_nan(v[i].y, 26.0f));
        d[i] = __ffma2_rn(e, c, c);
    }
    const float2 p01 = __fmul2_rn(d[0], d[1]), p23 = __fmul2_rn(d[2], d[3]);
    const float2 q = __fmul2_rn(p01, p23);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(q.x * q.y));
    float2 rq;
    rq.x = r * q.y; rq.y = r * q.x;                       // (1/q.x, 1/q.y)
    const float2 i01 = __fmul2_rn(rq, p23), i23 = __fmul2_rn(rq, p01);      // 1/p01, 1/p23
    v[0] = __fmul2_rn(i01, d[1]); v[1] = __fmul2_rn(i01, d[0]);
    v[2] = __fmul2_rn(i23, d[3]); v[3] = __fmul2_rn(i23, d[2]);
}

// The issue warp's view of an x tile: lane l owns points 4l .. 4l+3
template <int IN, int K0>          // IN: upper bound of the input width (3, 7 or 15), K0: padded K of layer 0 (8 or 16)
struct Qb3X {
    float v[4][IN];
    int in_dim;
    __device__ __forceinline__ void load(const float* __restrict__ x, int64_t p0, int64_t n1, int lane) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t p = p0 + lane * 4 + i;
#pragma unroll
            for (int q = 0; q < IN; ++q) v[i][q] = (p < n1 && q < in_dim) ? __ldg(x + p * in_dim + q) : 0.0f;
        }
    }
    // canonical K-major tile [128 x K0]: element (m, k) at float index ((m/8)*(K0/4) + k/4)*32 + (m%8)*4 + k%4
    __device__ __forceinline__ void store(float* hi, float* lo, int lane) const {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = lane * 4 + i;
            float w[K0], h[K0], l[K0];
#pragma unroll
            for (int q = 0; q < K0; ++q) {
                const float xv = q < IN ? v[i][q < IN ? q : 0] : 0.0f;
                w[q] = (q == in_dim) ? 1.0f : xv;                // the bias slot (a select: no indexed store)
                h[q] = qb_tf32_hi(w[q]); l[q] = w[q] - h[q];
            }
            const int idx = ((m >> 3) * (K0 / 4)) * 32 + (m & 7) * 4;
#pragma unroll
            for (int c4 = 0; c4 < K0 / 4; ++c4) {
                *reinterpret_cast<float4*>(hi + idx + 32 * c4) = make_float4(h[4 * c4], h[4 * c4 + 1], h[4 * c4 + 2], h[4 * c4 + 3]);
                *reinterpret_cast<float4*>(lo + idx + 32 * c4) = make_float4(l[4 * c4], l[4 * c4 + 1], l[4 * c4 + 2], l[4 * c4 + 3]);
            }
        }
    }
};

// What happens to the network output of a point: squared residual against y (kernels 1, 3) or store (kernel 4)
struct Qb3SinkSsq {
    const float* __restrict__ y; float ssq;
    __device__ __forceinline__ float prefetch(int64_t p, bool live) const { return live ? __ldg(y + p) : 0.0f; }
    __device__ __forceinline__ void consume(int64_t, bool live, float yt, float yo) { if (live) { const float r = yt - yo; ssq = fmaf(r, r, ssq); } }
};
struct Qb3SinkStore {
    float* __restrict__ out;
    __device__ __forceinline__ float prefetch(int64_t, bool) const { return 0.0f; }
    __device__ __forceinline__ void consume(int64_t p, bool live, float, float yo) { if (live) out[p] = yo; }
};

// The tile loop over points [n0, n1) for the staged parameter vector; every thread of the block (128 G compute threads + the
// issue warp) calls it; returns the sink (its state is meaningful in group-0 threads).  PRESTAGE (chain kernel: same x, n0, n1
// in every call): the issue warp leaves the first three x tiles of the NEXT evaluation in the ring when it is done, so an
// evaluation does not start with global loads.
template <int H, int K0, int IN, bool PRESTAGE, typename Sink>
__device__ __forceinline__ Sink qb_tc3_run(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem, const float* __restrict__ x,
                                           int64_t n0, int64_t n1, const float* __restrict__ xs, Sink sink) {
    using D = Qb3Dim<H>;
    constexpr int G = D::G;
    constexpr uint32_t XT = 128u * K0 * 4u;                  // bytes of one half (hi or lo) of an x tile
    const float* F = reinterpret_cast<const float*>(smem + tp.fl_base);
    const uint32_t sb = qb_smem_u32(smem);
    const uint32_t bar_d0f = sb + QB3_D0F, bar_ardy = sb + QB3_ARDY, bar_d1f = sb + QB3_D1F, bar_d1free = sb + QB3_D1FREE;
    const int T = (int)((n1 - n0 + 127) / 128);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();                               // staging complete; nobody is still inside the previous evaluation
    if (threadIdx.x == 0) qb_tc3_reset_barriers<H>(smem);
    // Without ready-made x tiles (xs == nullptr) the COMPUTE threads lay the x tiles out: thread (point, group g) owns the four K
    // slots 4g .. 4g+3 of its point = one 16-byte row of a core matrix of the hi and of the lo tile.  Tile u+2 is written
    // inside EPI0(u), ahead of the arrival on a_ready(u) that lets the issue warp start layer 0 of tile u+2; tiles 0 and 1
    // here, ahead of the block barrier.  (An issue warp that stages x itself needs ~4000 cycles per 128 x 16 tile and
    // becomes the critical path of the 128-wide kernel: profiles/r2_tc3_trace_predict_*.log.)
    const bool bulk = xs != nullptr;
    auto xstage = [&](int u, const float (&xv)[4]) {
        const int g = threadIdx.x >> 7, pt = threadIdx.x & 127;
        float* hi = reinterpret_cast<float*>(smem + tp.v3_x) + (u % 3) * (2 * 128 * K0) + ((pt >> 3) * (K0 / 4) + g) * 32 + (pt & 7) * 4;
        float h[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) h[j] = qb_tf32_hi(xv[j]);
        *reinterpret_cast<float4*>(hi) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(hi + 128 * K0) = make_float4(xv[0] - h[0], xv[1] - h[1], xv[2] - h[2], xv[3] - h[3]);
    };
    auto xfetch = [&](int u, float (&xv)[4]) {
        const int g = threadIdx.x >> 7, pt = threadIdx.x & 127;
        const int64_t p = n0 + (int64_t)u * 128 + pt;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = 4 * g + j;
            float v = 0.0f;
            if (k < tp.in_dim && p < n1) v = __ldg(x + p * tp.in_dim + k);
            xv[j] = (k == tp.in_dim) ? 1.0f : v;
        }
    };
    if (!bulk && wid < D::ISSUER && 4 * (int)(threadIdx.x >> 7) < K0) {
        float xv[4];
        for (int u = 0; u < 2 && u < T; ++u) { xfetch(u, xv); xstage(u, xv); }
        qb_fence_proxy_async();
    }
    __syncthreads();
    if (T > 0 && wid == D::ISSUER) {
        // ================================ issue warp ================================
        float* xb = reinterpret_cast<float*>(smem + tp.v3_x);         // [3][hi | lo], 128 x K0 floats each
        const uint32_t dhi0 = qb_desc_hi(128u * (K0 / 4), 0u);        // tf32 operands with K = K0: SBO 128 K0/4 bytes
        const uint32_t dhi1 = qb_desc_hi(16u * H, 0u);                // fp16 W1, K = H: SBO 16 H bytes
        const uint32_t w0hi = qb_desc_lo(qb_smem_u32(smem + tp.v3_w0), 128u), w0lo = w0hi + ((uint32_t)(H * K0 * 4) >> 4);
        const uint32_t w1hi = qb_desc_lo(qb_smem_u32(smem + tp.v3_w1), 128u), w1lo = w1hi + ((uint32_t)(H * H * 2) >> 4),
                       w1nhi = w1lo + ((uint32_t)(H * H * 2) >> 4);
        const uint32_t xd = qb_desc_lo(qb_smem_u32(xb), 128u);        // + 2 XT / 16 per ring slot, + XT / 16 for lo
        const uint32_t id_tf32 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(H >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t id_f16 = (1u << 4) | ((uint32_t)(H >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t d0 = cx.tmem, a_hi = cx.tmem + D::COL_AHI, a_lo = cx.tmem + D::COL_ALO;
        // x tiles come either as ready-made operand images from global memory (xs: tile u = tf32 hi | lo in the canonical
        // layout, written once per launch by k_tc3_xsplit; one bulk copy per tile, completion on x_full[u % 3]) or,
        // without such a buffer, from the compute threads (see above)
        const uint32_t bar_x = sb + (uint32_t)tp.v3_xbar;
        uint32_t xpar = cx.hphase;                 // parities of x_full[0..2] (they are never re-initialised)
        auto xcopy = [&](int u) {                  // one lane: start the bulk copy of tile u into ring slot u % 3
            const uint32_t bar = bar_x + (uint32_t)(u % 3) * 8u, dst = qb_smem_u32(xb) + (uint32_t)(u % 3) * 2u * XT;
            const float* src = xs + (int64_t)u * (2 * 128 * K0);
            asm volatile("{ .reg .b64 st; mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1; }" :: "r"(bar), "r"(2u * XT) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(dst), "l"(src), "r"(2u * XT), "r"(bar) : "memory");
        };
        auto xwait = [&](int u) {                  // all lanes: tile u has landed
            const int sl = u % 3;
            qb_mbar_wait_counted(bar_x + (uint32_t)sl * 8u, (xpar >> sl) & 1u);
            xpar ^= 1u << sl;
        };
        auto mma0 = [&](int u) {           // layer 0 of tile u: x ring slot u % 3 -> D0[u & 1]
            const uint32_t xa = xd + (uint32_t)(u % 3) * (2u * XT >> 4), d = d0 + (uint32_t)(u & 1) * (uint32_t)H;
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                for (int ks = 0; ks < K0 / 8; ++ks) {
                    const uint32_t a = xa + (pass == 0 ? (XT >> 4) : 0u) + 16u * ks, b = (pass == 1 ? w0lo : w0hi) + 16u * ks;
                    if (pass == 0 && ks == 0) qb_mma_ss<false, false>(d, a, dhi0, b, dhi0, id_tf32);
                    else qb_mma_ss<false, true>(d, a, dhi0, b, dhi0, id_tf32);
                }
            }
            qb_commit((u & 1) ? sb + QB3_D0F1 : bar_d0f);
        };
        // x tiles 0 .. 2 staged up front (unless the previous evaluation left them), layer 0 of tiles 0 and 1 started
        if (bulk && !(PRESTAGE && cx.phase) && lane == 0)
            for (int u = 0; u < 3 && u < T; ++u) xcopy(u);
        if (bulk) { xwait(0); if (T > 1) xwait(1); }
        __syncwarp();
        if (qb_elect()) {
            mma0(0);
            if (T > 1) mma0(1);
        }
        __syncwarp();
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
            if (bulk && t + 2 < T) xwait(t + 2);                                      // long since landed
            qb_mbar_wait_counted(bar_ardy, (uint32_t)t & 1u);                                     // A(t) written, D0[t&1] read
            QB3_STAMP(t, 0);
            qb_tc_fence_after();
            __syncwarp();
            if (t + 2 < T && qb_elect()) mma0(t + 2);
            __syncwarp();
            QB3_STAMP(t, 1);
            if (t >= 1) { qb_mbar_wait_counted(bar_d1free, (uint32_t)(t - 1) & 1u); qb_tc_fence_after(); }   // EPI1(t-1) holds D1 in registers
            __syncwarp();
            QB3_STAMP(t, 2);
            if (qb_elect()) {
                const uint32_t d1 = cx.tmem + D::COL_D1;
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                    for (int ks = 0; ks < H / 16; ++ks) {
                        const uint32_t a = (pass == 0 ? a_lo : a_hi) + 8u * ks;
                        const uint32_t b = (pass == 0 ? w1nhi : pass == 1 ? w1lo : w1hi) + 16u * ks;
                        if (pass == 0 && ks == 0) qb_mma_ts<true, false>(d1, a, b, dhi1, id_f16);
                        else qb_mma_ts<true, true>(d1, a, b, dhi1, id_f16);
                    }
                }
                qb_commit(bar_d1f);
            }
            __syncwarp();
            QB3_STAMP(t, 3);
            if (t + 3 < T) {
                // ring slot t % 3 was read by MMA0(t), which completed before the compute warps arrived on a_ready(t)
                if (bulk && lane == 0) xcopy(t + 3);
            }
        }
        if (PRESTAGE && bulk) {
            // every MMA0 has completed (a_ready(T-1) was waited for): the ring is free
            if (lane == 0) for (int u = 0; u < 3 && u < T; ++u) xcopy(u);
            cx.phase = 1u;
        }
        cx.hphase = xpar;
    } else if (T > 0) {
        // ================================ compute warps ================================
        const int g = threadIdx.x >> 7, pt = threadIdx.x & 127;
        const uint32_t tl = cx.tmem + ((uint32_t)((wid & 3) * 32) << 16);
        float* ybuf = reinterpret_cast<float*>(smem + tp.ybuf);           // [4][G-1][128] partial outputs of groups 1 .. G-1
        const float c1 = F[tp.v3_c1];
        const float4* B4 = reinterpret_cast<const float4*>(F + tp.L[1].bias + 32 * g);
        const float4* W4 = reinterpret_cast<const float4*>(F + tp.wl + 32 * g);
        const int64_t pbase = n0 + pt;
        float own0 = 0.0f, own1 = 0.0f, yt0 = 0.0f, yt1 = 0.0f;          // group 0: own partial sum / target of tiles t-1, t-2

        // EPI0(u): D0 -> 2^14 * s -> fp16 hi / lo -> A; the stores wait for d1_full(u - 1) = "A is free"
        const bool xmine = !bulk && 4 * g < K0;                       // this thread lays out a row of the x tiles
        auto epi0 = [&](int u) {
            QB3_STAMP(u, 0);
            float xv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            if (xmine && u + 2 < T) xfetch(u + 2, xv);                // consumed at the end of this epilogue
            // layer 0 of tiles u >= 2 was issued BEFORE MMA1(u-2), whose commit (d1_full(u-2), waited for in EPI0(u-1))
            // covers every earlier tcgen05 operation of the issuing thread: only the first two tiles wait on d0_full
            if (u < 2) {
                qb_mbar_wait_counted((u & 1) ? sb + QB3_D0F1 : bar_d0f, 0u);
                qb_tc_fence_after();
            }
            uint32_t v[2][16];
            qb_tmem_ld16(tl + H * (u & 1) + 32 * g, v[0]);
            qb_tmem_ld16(tl + H * (u & 1) + 32 * g + 16, v[1]);
            qb_tmem_ld_wait16(v[0]);
            qb_tmem_ld_wait16(v[1]);
            QB3_STAMP(u, 1);
            uint32_t hi[2][8], lo[2][8];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    float2 a[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) a[i] = make_float2(__uint_as_float(v[j][8 * q + 2 * i]), __uint_as_float(v[j][8 * q + 2 * i + 1]));
                    qb3_sig8(a);
#pragma unroll
                    for (int i = 0; i < 4; ++i) qb_split_f16_nlo(a[i].x, a[i].y, hi[j][4 * q + i], lo[j][4 * q + i]);
                }
            }
            QB3_STAMP(u, 2);
            if (u > 0) {
                qb_mbar_wait_counted(bar_d1f, (uint32_t)(u - 1) & 1u);           // MMA1(u-1) complete: A is free, D1 is ready
                qb_tc_fence_after();
            }
            QB3_STAMP(u, 3);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                qb_tmem_st8(tl + D::COL_AHI + 16 * g + 8 * j, hi[j]);
                qb_tmem_st8(tl + D::COL_ALO + 16 * g + 8 * j, lo[j]);
            }
            if (xmine && u + 2 < T) {
                xstage(u + 2, xv);        // slot (u+2) % 3 was last read by MMA0(u-1), whose D0 this thread consumed a tile ago
                qb_fence_proxy_async();
            }
            qb_tmem_st_wait();
            qb_tc_fence_before();
            qb_mbar_arrive(bar_ardy);
            QB3_STAMP(u, 4);
        };
        // EPI1(u): D1 -> s -> partial dot product with the output row
        auto epi1 = [&](int u) -> float {
            QB3_STAMP(u, 5);
            uint32_t v[2][16];
            const uint32_t dcol = D::COL_D1 + 32u * g;
            qb_tmem_ld16(tl + dcol, v[0]);
            qb_tmem_ld16(tl + dcol + 16, v[1]);
            qb_tmem_ld_wait16(v[0]);
            qb_tmem_ld_wait16(v[1]);
            qb_tc_fence_before();
            qb_mbar_arrive(bar_d1free);                                  // the accumulator is in registers
            QB3_STAMP(u, 6);
            float2 acc = make_float2(0.0f, 0.0f);
            const float2 c2 = make_float2(c1, c1);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    float2 a[4];
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const float4 bb = B4[4 * j + 2 * q + i];
                        a[2 * i] = __ffma2_rn(make_float2(__uint_as_float(v[j][8 * q + 4 * i]), __uint_as_float(v[j][8 * q + 4 * i + 1])), c2, make_float2(bb.x, bb.y));
                        a[2 * i + 1] = __ffma2_rn(make_float2(__uint_as_float(v[j][8 * q + 4 * i + 2]), __uint_as_float(v[j][8 * q + 4 * i + 3])), c2, make_float2(bb.z, bb.w));
                    }
                    qb3_sig8(a);
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const float4 ww = W4[4 * j + 2 * q + i];
                        acc = __ffma2_rn(a[2 * i], make_float2(ww.x, ww.y), acc);
                        acc = __ffma2_rn(a[2 * i + 1], make_float2(ww.z, ww.w), acc);
                    }
                }
            }
            QB3_STAMP(u, 7);
            return acc.x + acc.y;
        };
        // group 0: output of tile u (own partial sum + the partners' from ybuf) to the sink
        auto finish = [&](int u, float own, float yt) {
            const int64_t p = pbase + (int64_t)u * 128;
            float acc = own;
#pragma unroll
            for (int gg = 0; gg < G - 1; ++gg) acc += ybuf[((u & 3) * (G - 1) + gg) * 128 + pt];
            sink.consume(p, p < n1, yt, qb_tc_out(tp, F, 0, acc));
        };

        epi0(0);
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
            if (t >= 1) {
                // tile t-1 (d1_full(t-1) was waited for in EPI0(t)); the partners' partial sums of tile t-3 became visible
                // with d1_full(t-1) at the latest (they arrived on a_ready(t-1) after writing them)
                const int u = t - 1;
                float ytn = 0.0f;
                if (g == 0) { const int64_t p = pbase + (int64_t)u * 128; ytn = sink.prefetch(p, p < n1); }
                const float part = epi1(u);
                if (g == 0) {
                    if (u >= 2) finish(u - 2, own1, yt1);
                    own1 = own0; yt1 = yt0; own0 = part; yt0 = ytn;
                } else {
                    ybuf[((u & 3) * (G - 1) + g - 1) * 128 + pt] = part;
                }
            }
            if (t + 1 < T) epi0(t + 1);
            else { qb_mbar_wait_counted(bar_d1f, (uint32_t)t & 1u); qb_tc_fence_after(); }
        }
        {
            const int u = T - 1;
            float ytn = 0.0f;
            if (g == 0) { const int64_t p = pbase + (int64_t)u * 128; ytn = sink.prefetch(p, p < n1); }
            const float part = epi1(u);
            if (g != 0) ybuf[((u & 3) * (G - 1) + g - 1) * 128 + pt] = part;
            asm volatile("bar.sync 1, %0;" :: "n"(D::NCOMP) : "memory");               // the compute warps only
            if (g == 0) {
                if (u >= 2) finish(u - 2, own1, yt1);
                if (u >= 1) finish(u - 1, own0, yt0);
                finish(u, part, ytn);
            }
        }
    }
    return sink;
}

// shape dispatch: hidden width 64 -> K0 = 8 (in <= 7), 128 -> K0 = 16 (in <= 15)
template <int H, bool PRESTAGE, typename Sink>
__device__ __forceinline__ Sink qb_tc3_dispatch(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem, const float* __restrict__ x,
                                                int64_t n0, int64_t n1, const float* __restrict__ xs, Sink sink) {
    if constexpr (H == 64) {
        if (tp.in_dim <= 3) return qb_tc3_run<64, 8, 3, PRESTAGE>(tp, cx, smem, x, n0, n1, xs, sink);
        return qb_tc3_run<64, 8, 7, PRESTAGE>(tp, cx, smem, x, n0, n1, xs, sink);
    } else {
        return qb_tc3_run<128, 16, 15, PRESTAGE>(tp, cx, smem, x, n0, n1, xs, sink);
    }
}
template <int H> struct Qb3K0 { static constexpr int value = H == 64 ? 8 : 16; };

// sum of squared residuals over points [n0, n1) (block-wide result): kernels 1 and 3
template <int H, bool PRESTAGE>
__device__ __forceinline__ double qb_tc3_eval_any(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem,
                                                  const float* __restrict__ x, const float* __restrict__ y,
                                                  int64_t n0, int64_t n1, const float* __restrict__ xs) {
    Qb3SinkSsq sink;
    sink.y = y; sink.ssq = 0.0f;
    sink = qb_tc3_dispatch<H, PRESTAGE>(tp, cx, smem, x, n0, n1, xs, sink);
    return qb_block_sum((double)sink.ssq, reinterpret_cast<double*>(smem));
}
#endif  // __CUDACC__
