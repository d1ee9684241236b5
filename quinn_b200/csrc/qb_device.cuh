// Device code of the fused MLP log-posterior / gradient evaluation (kernels 1 and 2) that the
// chain-step, predictive and VI kernels all call.  sm_100a, CUDA cores (FP32 / FP64 FMA pipes).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "qb_plan.h"

#ifndef QB_UNROLL
#define QB_UNROLL 2
#endif
#ifndef QB_TAIL_UNROLL
#define QB_TAIL_UNROLL 2
#endif
#define QB_STR_(x) #x
#define QB_PRAGMA_UNROLL(n) _Pragma(QB_STR_(unroll n))

__device__ __forceinline__ float qb_mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double qb_mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float qb_add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double qb_add_rn(double a, double b) { return __dadd_rn(a, b); }

// --------------------------------------------------------------------------------------------
// per-dtype tile constants and 128-bit vector access
// --------------------------------------------------------------------------------------------
template <typename T> struct VT;
template <> struct VT<float>  { static constexpr int TP = 8, TU = 8, LDPAD = 4, PV = 4, VW = 4; };
template <> struct VT<double> { static constexpr int TP = 4, TU = 4, LDPAD = 2, PV = 2, VW = 2; };

template <int N> __device__ __forceinline__ void ldv(float* d, const float* s) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
        float4 v = *reinterpret_cast<const float4*>(s + 4 * q);
        d[4 * q] = v.x; d[4 * q + 1] = v.y; d[4 * q + 2] = v.z; d[4 * q + 3] = v.w;
    }
}
template <int N> __device__ __forceinline__ void ldv(double* d, const double* s) {
#pragma unroll
    for (int q = 0; q < N / 2; ++q) {
        double2 v = *reinterpret_cast<const double2*>(s + 2 * q);
        d[2 * q] = v.x; d[2 * q + 1] = v.y;
    }
}
template <int N> __device__ __forceinline__ void stv(float* d, const float* s) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q)
        *reinterpret_cast<float4*>(d + 4 * q) = make_float4(s[4 * q], s[4 * q + 1], s[4 * q + 2], s[4 * q + 3]);
}
template <int N> __device__ __forceinline__ void stv(double* d, const double* s) {
#pragma unroll
    for (int q = 0; q < N / 2; ++q)
        *reinterpret_cast<double2*>(d + 2 * q) = make_double2(s[2 * q], s[2 * q + 1]);
}

// Column permutation of the staged weight rows.  Thread tile `g` (of G) owns units g + G*u, u = 0..TU-1; its TU
// weights are fetched with TU/VW 128-bit loads.  Load number h of all G tiles is laid out contiguously
// (col = h*G*VW + g*VW + q, u = h*VW + q) so that the lanes of a quarter warp (consecutive g) read 128
// contiguous bytes: one conflict-free wavefront (the first layout, col = g*TU + u, strided the lanes by
// 32 B and measured 8 wavefronts per LDS.128 in ncu, profiles/r1_amcmc_v0.md).
template <typename T> __device__ __forceinline__ int qb_col_to_unit(int col, int G) {
    constexpr int VW = VT<T>::VW;
    const int h = col / (G * VW), rem = col - h * (G * VW);
    const int g = rem / VW, q = rem - g * VW;
    return g + G * (h * VW + q);
}
// load the TU weights of tile g from a staged row
template <typename T> __device__ __forceinline__ void qb_ld_wrow(T (&w)[VT<T>::TU], const T* row, int g, int G) {
    constexpr int VW = VT<T>::VW, TU = VT<T>::TU;
#pragma unroll
    for (int h = 0; h < TU / VW; ++h) ldv<VW>(&w[h * VW], row + h * G * VW + g * VW);
}


// --------------------------------------------------------------------------------------------
// activations
// --------------------------------------------------------------------------------------------
// fp32 tanh = 1 - 2/(exp(2z)+1) with one MUFU.EX2 and one MUFU.RCP (abs. error ~2e-7; MUFU.TANH's
// 2^-11 relative error does not keep the 1e-4 log-posterior tolerance, SURVEY.md section 7 item 3).
__device__ __forceinline__ float qb_tanh(float z) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * 2.8853900817779268f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}
__device__ __forceinline__ double qb_tanh(double z) { return tanh(z); }
__device__ __forceinline__ float qb_exp(float z) { return expf(z); }
__device__ __forceinline__ double qb_exp(double z) { return exp(z); }

// tanh of a pre-activation that was already multiplied by 2*log2(e) (folded into the staged fp32 weights)
__device__ __forceinline__ float qb_tanh_prescaled(float z2) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z2));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}
__device__ __forceinline__ double qb_tanh_prescaled(double z) { return tanh(z); }   // never folded in fp64
template <typename T> __device__ __forceinline__ T qb_tanh_fold() { return T(1); }
template <> __device__ __forceinline__ float qb_tanh_fold<float>() { return 2.8853900817779268f; }

// Who cooperates on a tile: the whole block (p_base = 0, p_count = TM) or, in warp-synchronous mode, one warp
// that owns WP consecutive points of the tile for ALL layers (no block barrier inside the tile loop).
struct QbScope {
    int nthr, tid, p_base, p_count;
    bool warp;
    __device__ __forceinline__ void sync() const { if (warp) __syncwarp(); else __syncthreads(); }
};
__device__ __forceinline__ QbScope qb_block_scope(int TM) {
    QbScope s; s.nthr = blockDim.x; s.tid = threadIdx.x; s.p_base = 0; s.p_count = TM; s.warp = false; return s;
}
__device__ __forceinline__ QbScope qb_warp_scope(int WP) {
    QbScope s; s.nthr = 32; s.tid = threadIdx.x & 31; s.p_base = (threadIdx.x >> 5) * WP; s.p_count = WP; s.warp = true; return s;
}

template <int ACT, typename T> __device__ __forceinline__ T qb_act(T z) {
    if (ACT == QB_ACT_TANH) return qb_tanh_prescaled(z);
    if (ACT == QB_ACT_RELU) return z > T(0) ? z : T(0);
    return z;
}
// derivative of the activation expressed through its VALUE a = act(z)
template <int ACT, typename T> __device__ __forceinline__ T qb_dact_c(T a) {
    if (ACT == QB_ACT_TANH) return T(1) - a * a;
    if (ACT == QB_ACT_RELU) return a > T(0) ? T(1) : T(0);
    return T(1);
}
template <typename T> __device__ __forceinline__ T qb_dact(int act, T a) {
    if (act == QB_ACT_TANH) return T(1) - a * a;
    if (act == QB_ACT_RELU) return a > T(0) ? T(1) : T(0);
    return T(1);
}

// --------------------------------------------------------------------------------------------
// deterministic block reduction (fixed order: lane tree, then warps in order)
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ double qb_block_sum(double v, double* red /* >= 33 doubles */) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        const int nw = (blockDim.x + 31) >> 5;
        for (int w = 0; w < nw; ++w) s += red[w];
        red[32] = s;
    }
    __syncthreads();
    return red[32];
}

// --------------------------------------------------------------------------------------------
// weight staging: flat theta (global) -> Wt / Wr / bias (shared), once per parameter vector
// --------------------------------------------------------------------------------------------
// One weight / bias entry of a layer.  Polynomial-in-depth layers (rnet.py:344-347) sum their terms in the reference's
// order, val = 0; val += pars[m] * t^m, with separate multiply and add (no FMA contraction) so that fp64 reproduces it.
template <typename T>
__device__ __forceinline__ T qb_layer_param(const QbLayerPlan& L, const T* __restrict__ theta, int off, int stride) {
    if (L.n_terms <= 1) return theta[off];
    T v = T(0);
    for (int m = 0; m < L.n_terms; ++m) v = qb_add_rn(v, qb_mul_rn(theta[off + m * stride], (T)L.coef[m]));
    return v;
}

template <typename T>
__device__ void qb_stage_weights(const QbPlan& P, T* sW, const T* theta) {
    constexpr int TU = VT<T>::TU;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int l = 0; l < P.n_layers; ++l) {
        const QbLayerPlan& L = P.L[l];
        // skip layers that alias an earlier layer's staged copy (shared weights, rnet.py:344-347)
        bool dup = false;
        for (int m = 0; m < l; ++m) dup = dup || (P.L[m].wt_off == L.wt_off);
        if (dup) continue;
        const int UG = L.n_out_pad / TU;
        const bool gemm = (L.mode == QB_MODE_GEMM);
        T* Wt = sW + L.wt_off;
        const int nwt = L.n_in * L.n_out_pad;
        const T fold = (L.act == QB_ACT_TANH) ? qb_tanh_fold<T>() : T(1);      // 2*log2(e) for fp32 tanh layers
        for (int idx = tid; idx < nwt; idx += nt) {
            const int i = idx / L.n_out_pad, col = idx - i * L.n_out_pad;
            const int j = gemm ? qb_col_to_unit<T>(col, UG) : col;
            Wt[idx] = (j < L.n_out) ? qb_layer_param<T>(L, theta, L.w_off + j * L.n_in + i, L.w_stride) * fold : T(0);
        }
        T* bs = sW + L.bias_off;
        for (int col = tid; col < L.n_out_pad; col += nt) {
            const int j = gemm ? qb_col_to_unit<T>(col, UG) : col;
            bs[col] = (j < L.n_out && L.b_off >= 0) ? qb_layer_param<T>(L, theta, L.b_off + j, L.b_stride) * fold : T(0);
        }
        if (L.wr_off >= 0) {
            const int UGI = L.n_in_pad / TU;
            T* Wr = sW + L.wr_off;
            const int nwr = L.n_out * L.n_in_pad;
            for (int idx = tid; idx < nwr; idx += nt) {
                const int j = idx / L.n_in_pad, col = idx - j * L.n_in_pad;
                const int i = qb_col_to_unit<T>(col, UGI);
                Wr[idx] = (i < L.n_in) ? qb_layer_param<T>(L, theta, L.w_off + j * L.n_in + i, L.w_stride) : T(0);
            }
        }
    }
}

// --------------------------------------------------------------------------------------------
// forward layers
// --------------------------------------------------------------------------------------------
// GEMM mode: each thread owns a TU x TP register tile (units x points); per input unit i it issues TU/VW
// 128-bit loads of weights and TP/VW 128-bit loads of activations for TU*TP FMAs.  Operands of step i+1 are
// fetched before the FMAs of step i (register double buffering).  Accumulators start from the bias.
//
// Fused tail (tail != nullptr): the NEXT layer is a narrow linear output layer (n_out <= 4, identity): instead of
// storing this layer's activations, every thread dots its TU x TP activations with the tail weights, the UG lanes
// that share the same points combine with an xor-shuffle tree (UG is a power of two in this mode) and the lane
// with ug == 0 receives tail_out[q][p] = sum_j Wtail[q][j] h[j][p] (bias not yet added).
template <typename T> struct QbTailCtx {   // what the fused tail needs to turn outputs into squared residuals
    const QbLayerPlan* tail;
    const T* y;
    int64_t p0, n1;
    int o, final_exp;
};

// ---- the hot loop of the library:  acc[u][p] = bias[u] + sum_i W[i][unit u of tile ug] * A[i][pcol + p] ----------
// Thread tile = TU units x TP points (TP = 8 in the value / predictive kernels, 4 in the gradient kernel, whose
// blocks need twice the threads per tile to reach 4 warps per scheduler).  Three running pointers (activation
// row, two halves of the weight row) advance by constant strides; the operands of step i+1 are fetched before
// the FMAs of step i (register double buffering; after the last pair one row past the end is read, the plan pads
// for it).
//
// fp32: the accumulators live as float2 values (aligned register pairs along the point axis) and every FMA is
// Blackwell's packed FFMA2 (two FMAs per lane per issued instruction, weight broadcast by the hardware:
// SASS `FFMA2 Rd, Ra.F32x2.HI_LO, Rb.F32, Rc.F32x2.HI_LO`).  The kernels are issue-bound, so halving the FMA
// instruction count is what lets the FMA pipe, not the scheduler, set the pace.
template <int TP> __device__ __forceinline__ void qb_ldp(float2 (&d)[TP / 2], const float* s) {
#pragma unroll
    for (int q = 0; q < TP / 4; ++q) {
        const float4 v = *reinterpret_cast<const float4*>(s + 4 * q);
        d[2 * q] = make_float2(v.x, v.y);
        d[2 * q + 1] = make_float2(v.z, v.w);
    }
}
__device__ __forceinline__ void qb_ldw8(float (&w)[8], const float* w0p, const float* w1p) {
    const float4 lo = *reinterpret_cast<const float4*>(w0p), hi = *reinterpret_cast<const float4*>(w1p);
    w[0] = lo.x; w[1] = lo.y; w[2] = lo.z; w[3] = lo.w; w[4] = hi.x; w[5] = hi.y; w[6] = hi.z; w[7] = hi.w;
}
template <int TP> __device__ __forceinline__ void qb_fma2_tile(float2 (&c)[8][TP / 2], const float (&w)[8], const float2 (&a)[TP / 2]) {
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int q = 0; q < TP / 2; ++q) c[u][q] = __ffma2_rn(a[q], make_float2(w[u], w[u]), c[u][q]);
}
template <int TP>
__device__ __forceinline__ void qb_gemm_accumulate(float (&acc)[8][TP], const float* __restrict__ Wt,
                                                   const float* __restrict__ bias, const float* __restrict__ ap,
                                                   int n_in, int lda, int ldw, int ug, int UG) {
    float2 c[8][TP / 2];
    {
        float b[8];
        if (bias) qb_ldw8(b, bias + ug * 4, bias + UG * 4 + ug * 4);
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int q = 0; q < TP / 2; ++q) c[u][q] = bias ? make_float2(b[u], b[u]) : make_float2(0.f, 0.f);
    }
    const float* w0p = Wt + ug * 4;
    const float* w1p = Wt + UG * 4 + ug * 4;
    const int lda2 = 2 * lda, ldw2 = 2 * ldw;
    float2 a0[TP / 2], a1[TP / 2];
    float w0[8], w1[8];
    qb_ldp<TP>(a0, ap);
    qb_ldw8(w0, w0p, w1p);
    int pairs = n_in >> 1;
#pragma unroll 1
    while (pairs > 0) {
        qb_ldp<TP>(a1, ap + lda);
        qb_ldw8(w1, w0p + ldw, w1p + ldw);
        qb_fma2_tile<TP>(c, w0, a0);
        ap += lda2;
        w0p += ldw2;
        w1p += ldw2;
        --pairs;
        qb_ldp<TP>(a0, ap);          // after the last pair this reads one row past the end: the plan pads for it
        qb_ldw8(w0, w0p, w1p);
        qb_fma2_tile<TP>(c, w1, a1);
    }
    if (n_in & 1) qb_fma2_tile<TP>(c, w0, a0);
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int q = 0; q < TP / 2; ++q) { acc[u][2 * q] = c[u][q].x; acc[u][2 * q + 1] = c[u][q].y; }
}

// fp64: 4 x 4 tile, scalar DFMA
template <int TP>
__device__ __forceinline__ void qb_gemm_accumulate(double (&acc)[4][TP], const double* __restrict__ Wt,
                                                   const double* __restrict__ bias, const double* __restrict__ ap,
                                                   int n_in, int lda, int ldw, int ug, int UG) {
    static_assert(TP == 4, "fp64 tiles are 4 x 4");
    {
        double b[4];
        if (bias) { ldv<2>(&b[0], bias + ug * 2); ldv<2>(&b[2], bias + UG * 2 + ug * 2); }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = bias ? b[u] : 0.0;
    }
    const double* w0p = Wt + ug * 2;
    const double* w1p = Wt + UG * 2 + ug * 2;
    double a0[4], w0[4], a1[4], w1[4];
    ldv<4>(a0, ap);
    ldv<2>(&w0[0], w0p);
    ldv<2>(&w0[2], w1p);
    int pairs = n_in >> 1;
#pragma unroll 1
    while (pairs > 0) {
        ldv<4>(a1, ap + lda);
        ldv<2>(&w1[0], w0p + ldw);
        ldv<2>(&w1[2], w1p + ldw);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = fma(w0[u], a0[p], acc[u][p]);
        ap += 2 * lda;
        w0p += 2 * ldw;
        w1p += 2 * ldw;
        --pairs;
        ldv<4>(a0, ap);
        ldv<2>(&w0[0], w0p);
        ldv<2>(&w0[2], w1p);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = fma(w1[u], a1[p], acc[u][p]);
    }
    if (n_in & 1) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = fma(w0[u], a0[p], acc[u][p]);
    }
}

// activation (+ residual) of one accumulator row
template <typename T, int ACT, int TP>
__device__ __forceinline__ void qb_act_row(T (&h)[TP], const T (&accrow)[TP], bool res, T step,
                                           const T* ain_row) {
#pragma unroll
    for (int p = 0; p < TP; ++p) h[p] = qb_act<ACT>(accrow[p]);
    if (res) {
        T r[TP];
        ldv<TP>(r, ain_row);
#pragma unroll
        for (int p = 0; p < TP; ++p) h[p] = fma(step, h[p], r[p]);
    }
}

template <typename T, int ACT, int TP>
__device__ __forceinline__ void qb_epilogue_store(const T (&acc)[VT<T>::TU][TP], const T* Ain, T* Aout, int lda,
                                                  int pcol, int ug, int UG, bool res, T step) {
    constexpr int TU = VT<T>::TU;
#pragma unroll
    for (int u = 0; u < TU; ++u) {
        const int j = ug + UG * u;
        T h[TP];
        qb_act_row<T, ACT, TP>(h, acc[u], res, step, Ain + j * lda + pcol);
        stv<TP>(Aout + j * lda + pcol, h);
    }
}

template <typename T, int ACT, int NT, int TP>
__device__ __forceinline__ void qb_epilogue_tail(const T (&acc)[VT<T>::TU][TP], const T* Ain, int lda, int pcol,
                                                 int ug, int UG, bool res, T step, int n_out, const T* Wl, int ldl,
                                                 int n_tail, T (&part)[NT][TP]) {
    constexpr int TU = VT<T>::TU;
#pragma unroll
    for (int u = 0; u < TU; ++u) {
        const int j = ug + UG * u;
        T h[TP];
        qb_act_row<T, ACT, TP>(h, acc[u], res, step, Ain + j * lda + pcol);
        if (j < n_out) {
#pragma unroll
            for (int q = 0; q < NT; ++q) {
                if (q < n_tail) {                      // uniform
                    const T wq = Wl[j * ldl + q];
#pragma unroll
                    for (int p = 0; p < TP; ++p) part[q][p] = fma(wq, h[p], part[q][p]);
                }
            }
        }
    }
}

// tc == nullptr: store the activations; else fused tail with up to 4 outputs.  ONE instance of the hot loop serves
// both (separate template instances of the tail made ptxas spill the accumulators inside the loop).
template <typename T, int TP>
__device__ __forceinline__ T qb_fwd_gemm(const QbLayerPlan& L, const T* sW, const T* Ain, T* Aout,
                                         int lda, const QbScope& sc, bool sync_before_store,
                                         const QbTailCtx<T>* tc) {
    constexpr int TU = VT<T>::TU;
    const int UG = L.n_out_pad / TU, PG = sc.p_count / TP, items = UG * PG;
    const T* Wt = sW + L.wt_off;
    const T* bias = sW + L.bias_off;
    const int n_in = L.n_in, ldw = L.n_out_pad, act = L.act;
    const bool res = L.has_res != 0;
    const T step = T(L.res_step);
    T ssq = T(0);
    const QbLayerPlan* tail = tc ? tc->tail : nullptr;
    for (int base = 0; base < items; base += sc.nthr) {
        const int item = base + sc.tid;
        const bool valid = item < items;
        int pg, ug;
        if (L.ug_shift >= 0) { pg = item >> L.ug_shift; ug = item & (UG - 1); }
        else { pg = item / UG; ug = item - pg * UG; }
        const int pcol = sc.p_base + pg * TP;
        T acc[TU][TP];
        if (valid) qb_gemm_accumulate<TP>(acc, Wt, bias, Ain + pcol, n_in, lda, ldw, ug, UG);
        if (sync_before_store) sc.sync();       // every lane has finished READING the input rows
        if (tc) {
            constexpr int NTA = 4;
            T part[NTA][TP];
#pragma unroll
            for (int q = 0; q < NTA; ++q)
#pragma unroll
                for (int p = 0; p < TP; ++p) part[q][p] = T(0);
            if (valid) {
                const T* Wl = sW + tail->wt_off;
                const int ldl = tail->n_out_pad, nt = tail->n_out;
                if (act == QB_ACT_TANH) qb_epilogue_tail<T, QB_ACT_TANH, NTA, TP>(acc, Ain, lda, pcol, ug, UG, res, step, L.n_out, Wl, ldl, nt, part);
                else if (act == QB_ACT_RELU) qb_epilogue_tail<T, QB_ACT_RELU, NTA, TP>(acc, Ain, lda, pcol, ug, UG, res, step, L.n_out, Wl, ldl, nt, part);
                else qb_epilogue_tail<T, QB_ACT_IDENTITY, NTA, TP>(acc, Ain, lda, pcol, ug, UG, res, step, L.n_out, Wl, ldl, nt, part);
            }
            // combine the UG lanes that hold the same points (consecutive lanes; fixed order => deterministic)
            for (int off = UG >> 1; off > 0; off >>= 1) {
#pragma unroll
                for (int q = 0; q < NTA; ++q) {
                    if (q < tail->n_out) {
#pragma unroll
                        for (int p = 0; p < TP; ++p) part[q][p] += __shfl_xor_sync(0xffffffffu, part[q][p], off);
                    }
                }
            }
            if (valid && ug == 0) {
                const T* bo = sW + tail->bias_off;
#pragma unroll
                for (int q = 0; q < NTA; ++q) {
                    if (q < tc->o) {
#pragma unroll
                        for (int p = 0; p < TP; ++p) {
                            const int64_t gp = tc->p0 + pcol + p;
                            if (gp < tc->n1) {
                                T out = part[q][p] + bo[q];
                                if (tc->final_exp) out = qb_exp(out);
                                const T r = __ldg(tc->y + gp * tc->o + q) - out;
                                ssq = fma(r, r, ssq);
                            }
                        }
                    }
                }
            }
        } else if (valid) {
            if (act == QB_ACT_TANH) qb_epilogue_store<T, QB_ACT_TANH, TP>(acc, Ain, Aout, lda, pcol, ug, UG, res, step);
            else if (act == QB_ACT_RELU) qb_epilogue_store<T, QB_ACT_RELU, TP>(acc, Ain, Aout, lda, pcol, ug, UG, res, step);
            else qb_epilogue_store<T, QB_ACT_IDENTITY, TP>(acc, Ain, Aout, lda, pcol, ug, UG, res, step);
        }
    }
    return ssq;
}

// DOT mode (narrow outputs): one thread per point column, NJ outputs at a time.  A thread only ever
// touches its own column, so this is in-place safe whenever n_out <= NJ.
template <typename T, int NJ, int ACT>
__device__ __forceinline__ void qb_fwd_dot(const QbLayerPlan& L, const T* sW, const T* Ain, T* Aout,
                                           int lda, const QbScope& sc) {
    const T* Wt = sW + L.wt_off;
    const T* bias = sW + L.bias_off;
    const int n_in = L.n_in, ldw = L.n_out_pad, n_out = L.n_out;
    const bool res = L.has_res != 0;
    const T step = T(L.res_step);
    for (int pl = sc.tid; pl < sc.p_count; pl += sc.nthr) {
        const int p = sc.p_base + pl;
        for (int j0 = 0; j0 < n_out; j0 += NJ) {
            T acc[NJ];
#pragma unroll
            for (int q = 0; q < NJ; ++q) acc[q] = bias[j0 + q];
#pragma unroll 4
            for (int i = 0; i < n_in; ++i) {
                const T a = Ain[i * lda + p];
#pragma unroll
                for (int q = 0; q < NJ; ++q) acc[q] = fma(Wt[i * ldw + j0 + q], a, acc[q]);
            }
#pragma unroll
            for (int q = 0; q < NJ; ++q) {
                T v = qb_act<ACT>(acc[q]);
                if (res && j0 + q < n_out) v = fma(step, v, Ain[(j0 + q) * lda + p]);
                acc[q] = v;
            }
#pragma unroll
            for (int q = 0; q < NJ; ++q)
                if (j0 + q < n_out) Aout[(j0 + q) * lda + p] = acc[q];
        }
    }
}

template <typename T, int TP = VT<T>::TP>
__device__ T qb_layer_forward(const QbLayerPlan& L, const T* sW, const T* Ain, T* Aout, int lda, const QbScope& sc,
                              bool inplace, const QbTailCtx<T>* tc = nullptr) {
    T ssq = T(0);
    if (L.mode == QB_MODE_GEMM) {
        ssq = qb_fwd_gemm<T, TP>(L, sW, Ain, Aout, lda, sc, inplace, tc);
    } else {
#define QB_DOT(NJ)                                                                            \
    switch (L.act) {                                                                          \
        case QB_ACT_TANH: qb_fwd_dot<T, NJ, QB_ACT_TANH>(L, sW, Ain, Aout, lda, sc); break;     \
        case QB_ACT_RELU: qb_fwd_dot<T, NJ, QB_ACT_RELU>(L, sW, Ain, Aout, lda, sc); break;     \
        default: qb_fwd_dot<T, NJ, QB_ACT_IDENTITY>(L, sW, Ain, Aout, lda, sc); break;          \
    }
        if (L.nj == 1) { QB_DOT(1) } else if (L.nj == 2) { QB_DOT(2) } else { QB_DOT(4) }
#undef QB_DOT
    }
    sc.sync();
    return ssq;
}

// x[p0 + p_base .. + p_count) -> rows 0..d-1 of A (zero for points beyond pend)
template <typename T>
__device__ __forceinline__ void qb_load_x_tile(const T* __restrict__ x, int d, int64_t p0, int64_t pend,
                                               T* A, int lda, const QbScope& sc) {
    const int n = sc.p_count * d;
    const int64_t g0 = p0 + sc.p_base;
    for (int idx = sc.tid; idx < n; idx += sc.nthr) {
        const int p = idx / d, i = idx - p * d;
        const int64_t gp = g0 + p;
        A[i * lda + sc.p_base + p] = (gp < pend) ? __ldg(x + gp * d + i) : T(0);
    }
}

// --------------------------------------------------------------------------------------------
// kernel 1 body: sum of squared residuals of one parameter vector over points [n0, n1)
// --------------------------------------------------------------------------------------------
struct QbSmem {
    double* red;     // 40 doubles
    void* w;         // staged weights
    void* act;       // activation rows
};
template <typename T> __device__ __forceinline__ QbSmem qb_carve(const QbPlan& P, unsigned char* raw) {
    QbSmem s;
    s.red = reinterpret_cast<double*>(raw);
    s.w = raw + 40 * sizeof(double);
    s.act = reinterpret_cast<T*>(s.w) + P.w_elems;
    return s;
}

template <typename T>
__device__ __forceinline__ double qb_eval_value(const QbPlan& P, const QbSmem& S, const T* theta, const T* __restrict__ x,
                                const T* __restrict__ y, int64_t n0, int64_t n1, bool restage) {
    T* sW = reinterpret_cast<T*>(S.w);
    T* A0 = reinterpret_cast<T*>(S.act);
    const int lda = P.lda, TM = P.TM, o = P.out_dim;
    T* A1 = P.inplace ? A0 : A0 + (size_t)P.buf_rows * lda;
    __syncthreads();
    if (restage) {
        qb_stage_weights<T>(P, sW, theta);
        __syncthreads();
    }
    T ssq = T(0);
    const QbScope sc = P.ws ? qb_warp_scope(P.WP) : qb_block_scope(TM);
    for (int64_t p0 = n0; p0 < n1; p0 += TM) {
        qb_load_x_tile<T>(x, P.in_dim, p0, n1, A0, lda, sc);
        sc.sync();
        T* cur = A0;
        T* oth = A1;
        const int nfull = P.fuse_tail ? P.n_layers - 1 : P.n_layers;
        QbTailCtx<T> tc;
        tc.tail = &P.L[P.n_layers - 1]; tc.y = y; tc.p0 = p0; tc.n1 = n1; tc.o = o; tc.final_exp = P.final_exp;
        for (int l = 0; l < nfull; ++l) {
            // with fuse_tail the last hidden layer also applies the narrow linear output layer and the residuals
            const QbTailCtx<T>* tcp = (P.fuse_tail && l == nfull - 1) ? &tc : nullptr;
            ssq += qb_layer_forward<T>(P.L[l], sW, cur, oth, lda, sc, P.inplace != 0, tcp);
            T* t = cur; cur = oth; oth = t;
        }
        if (!P.fuse_tail) {
            // residuals (losses.py:197: sum over all points and outputs)
            const int n = sc.p_count * o;
            for (int idx = sc.tid; idx < n; idx += sc.nthr) {
                const int j = idx / sc.p_count, p = sc.p_base + (idx - j * sc.p_count);
                const int64_t gp = p0 + p;
                if (gp < n1) {
                    T out = cur[j * lda + p];
                    if (P.final_exp) out = qb_exp(out);
                    const T r = __ldg(y + gp * o + j) - out;
                    ssq = fma(r, r, ssq);
                }
            }
        }
        sc.sync();
    }
    return qb_block_sum((double)ssq, S.red);
}

// --------------------------------------------------------------------------------------------
// kernel 2 body: value + gradient (reverse mode) of the data term
// --------------------------------------------------------------------------------------------
// write delta_z of layer Lm for (unit j, TP consecutive points) given delta_a (gradient wrt the layer output)
template <typename T, int TP, int ACT>
__device__ __forceinline__ void qb_finish_delta_vec(const QbLayerPlan& Lm, T* R, T* D, int lda, int j, int pcol,
                                                    T (&da)[TP]) {
    T aout[TP], dz[TP];
    T* po = R + (size_t)(Lm.row_out + j) * lda + pcol;
    ldv<TP>(aout, po);
    if (Lm.has_res) {
        T ain[TP];
        ldv<TP>(ain, R + (size_t)(Lm.row_in + j) * lda + pcol);
        const T step = T(Lm.res_step), inv = T(1) / step;
#pragma unroll
        for (int p = 0; p < TP; ++p) {
            const T t = (aout[p] - ain[p]) * inv;
            dz[p] = step * da[p] * qb_dact_c<ACT, T>(t);
        }
        stv<TP>(D + (size_t)j * lda + pcol, da);
    } else {
#pragma unroll
        for (int p = 0; p < TP; ++p) dz[p] = da[p] * qb_dact_c<ACT, T>(aout[p]);
    }
    stv<TP>(po, dz);
}
template <typename T>
__device__ __forceinline__ void qb_finish_delta(const QbLayerPlan& Lm, T* R, T* D, int lda, int j, int p, T da) {
    T* po = R + (size_t)(Lm.row_out + j) * lda + p;
    const T aout = *po;
    T dz;
    if (Lm.has_res) {
        const T ain = R[(size_t)(Lm.row_in + j) * lda + p];
        const T step = T(Lm.res_step);
        const T t = (aout - ain) / step;
        dz = step * da * qb_dact<T>(Lm.act, t);
        D[(size_t)j * lda + p] = da;
    } else {
        dz = da * qb_dact<T>(Lm.act, aout);
    }
    *po = dz;
}

// one PV-point step of the dW patch: acc[a][b] += sum_q dz[a][q]*av[b][q].  fp32: the (q, q+1) pairs that come out of
// the 128-bit loads feed FFMA2 directly; even and odd q accumulate separately (acc / acc2) and are folded at the end.
template <typename T>
__device__ __forceinline__ void qb_dw_fma(T (&acc)[4][4], T (&acc2)[4][4], const T (&dz)[4][VT<T>::PV],
                                          const T (&av)[4][VT<T>::PV]) {
    constexpr int PV = VT<T>::PV;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int q = 0; q < PV; ++q) acc[a][b] = fma(dz[a][q], av[b][q], acc[a][b]);
    }
}
#ifndef QB_NO_FFMA2
template <>
__device__ __forceinline__ void qb_dw_fma<float>(float (&acc)[4][4], float (&acc2)[4][4],
                                                 const float (&dz)[4][4], const float (&av)[4][4]) {
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            float2 c = make_float2(acc[a][b], acc2[a][b]);
            c = __ffma2_rn(make_float2(dz[a][0], dz[a][1]), make_float2(av[b][0], av[b][1]), c);
            c = __ffma2_rn(make_float2(dz[a][2], dz[a][3]), make_float2(av[b][2], av[b][3]), c);
            acc[a][b] = c.x;
            acc2[a][b] = c.y;
        }
    }
}
#endif
template <typename T> __device__ __forceinline__ void qb_dw_fold(T (&acc)[4][4], const T (&acc2)[4][4]) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] += acc2[a][b];
}

// dW_l += delta_z_l (rows) x a_in (rows) over the tile's points; db_l += row sums of delta_z_l.
// Each thread owns a 4x4 patch of dW (rows interleaved by JG / IG so that the 8 lanes of a quarter
// warp hit distinct banks) and, for narrow layers, one of `dw_chunks` slices of the points; slices are
// combined with a fixed-order xor-shuffle tree, so the result is deterministic.
template <typename T>
__device__ void qb_dw_accumulate(const QbLayerPlan& L, const T* R, int lda, int TM, T* g) {
    constexpr int PV = VT<T>::PV;
    const int JG = (L.n_out + 3) >> 2, IG = (L.n_in + 3) >> 2;
    const int C = L.dw_chunks, patches = JG * IG, items = patches * C;
    const int clen = TM / C;
    const T* Rz = R + (size_t)L.row_out * lda;
    const T* Ra = R + (size_t)L.row_in * lda;
    for (int base = 0; base < items; base += blockDim.x) {
        const int item = base + threadIdx.x;
        const bool valid = item < items;
        const int it = valid ? item : 0;
        const int patch = it >> L.c_shift, chunk = it & (C - 1);          // C is a power of two
        int jg, ig;
        if (L.ig_shift >= 0) { jg = patch >> L.ig_shift; ig = patch & (IG - 1); }
        else { jg = patch / IG; ig = patch - jg * IG; }
        T acc[4][4], acc2[4][4];      // acc2: odd-q partial sums of the packed fp32 path
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) { acc[a][b] = T(0); acc2[a][b] = T(0); }
        const bool writer = valid && chunk == 0;
        // the running gradient entries this thread owns: fetched BEFORE the point loop so the global-memory
        // latency hides behind it (they were 30 % of the kernel's stall samples as a load-add-store at the end)
        T gold[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int j = jg + JG * a;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int i = ig + IG * b;
                gold[a][b] = (writer && j < L.n_out && i < L.n_in) ? g[L.w_off + j * L.n_in + i] : T(0);
            }
        }
        const T* zr = Rz + (size_t)jg * lda + chunk * clen;
        const T* ar = Ra + (size_t)ig * lda + chunk * clen;
        const size_t zs = (size_t)JG * lda, as = (size_t)IG * lda;
        for (int p = 0; p < clen; p += PV) {
            T dz[4][PV], av[4][PV];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                ldv<PV>(dz[c], zr + c * zs + p);
                ldv<PV>(av[c], ar + c * as + p);
            }
            qb_dw_fma<T>(acc, acc2, dz, av);
        }
        qb_dw_fold<T>(acc, acc2);
        for (int off = C >> 1; off > 0; off >>= 1) {
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] += __shfl_xor_sync(0xffffffffu, acc[a][b], off);
        }
        if (writer) {
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const int j = jg + JG * a;
                if (j < L.n_out) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int i = ig + IG * b;
                        if (i < L.n_in) {
                            const int e = L.w_off + j * L.n_in + i;
                            if (L.n_terms <= 1) g[e] = gold[a][b] + acc[a][b];
                            else {
                                // chain rule through W = sum_m coef[m] * ww_m: every term receives coef[m] * dW
                                g[e] = gold[a][b] + (T)L.coef[0] * acc[a][b];
                                for (int m = 1; m < L.n_terms; ++m) g[e + m * L.w_stride] += (T)L.coef[m] * acc[a][b];
                            }
                        }
                    }
                }
            }
        }
    }
    // db[j] += sum_p delta_z[j][p]: one warp per row, lanes stride the points, fixed-order shuffle tree.  (Kept out
    // of the patch loop: a per-lane "this patch also owns the bias" test made every warp run the loop twice.)
    if (L.b_off >= 0) {
        // 8 rows per warp at a time, 4 lanes per row, each lane sums every 4th vector of the row
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
        const int rloc = lane >> 2, q = lane & 3;
        for (int jb = warp * 8; jb < L.n_out; jb += nw * 8) {
            const int j = jb + rloc;
            T sacc = T(0);
            if (j < L.n_out) {
                const T* zr = Rz + (size_t)j * lda;
                for (int p = q * PV; p < TM; p += 4 * PV) {
                    T v[PV];
                    ldv<PV>(v, zr + p);
#pragma unroll
                    for (int e = 0; e < PV; ++e) sacc += v[e];
                }
            }
            sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
            sacc += __shfl_xor_sync(0xffffffffu, sacc, 2);
            if (q == 0 && j < L.n_out) {
                if (L.n_terms <= 1) g[L.b_off + j] += sacc;
                else for (int m = 0; m < L.n_terms; ++m) g[L.b_off + j + m * L.b_stride] += (T)L.coef[m] * sacc;
            }
        }
    }
}

// delta_a of layer l's INPUT (= output of layer l-1): W_l^T delta_z_l (+ pass-through if layer l is
// residual), immediately converted to delta_z of layer l-1 and stored in place over that layer's
// activations.
// GLOBALW: the (rare) fallback when Wt and Wr do not both fit in shared memory: W is read straight from
// the flat parameter vector in global memory / L1 with contiguous (un-permuted) units.
template <typename T, bool GLOBALW, int TP, int ACTM>
__device__ void qb_bwd_gemm_a(const QbLayerPlan& L, const QbLayerPlan& Lm, const T* sW, const T* theta, T* R, T* D,
                              int lda, int TM) {
    constexpr int TU = VT<T>::TU;
    const int UGI = L.n_in_pad / TU, PG = TM / TP, items = UGI * PG;
    const T* Wr = GLOBALW ? theta + L.w_off : sW + L.wr_off;
    const T* Rz = R + (size_t)L.row_out * lda;
    const int n_out = L.n_out, ldw = GLOBALW ? L.n_in : L.n_in_pad;
    for (int base = 0; base < items; base += blockDim.x) {
        const int item = base + threadIdx.x;
        if (item >= items) continue;
        int pg, ig;
        if (L.ugi_shift >= 0) { pg = item >> L.ugi_shift; ig = item & (UGI - 1); }
        else { pg = item / UGI; ig = item - pg * UGI; }
        T acc[TU][TP];
        if (!GLOBALW) {
            // same hot loop as the forward pass: rows = output units j, "weights" = staged Wr, no bias
            qb_gemm_accumulate<TP>(acc, Wr, (const T*)nullptr, Rz + pg * TP, n_out, lda, ldw, ig, UGI);
        } else {
#pragma unroll
            for (int u = 0; u < TU; ++u)
#pragma unroll
                for (int p = 0; p < TP; ++p) acc[u][p] = T(0);
            const T* zp = Rz + pg * TP;
            const T* wp = Wr + ig * TU;
            for (int j = 0; j < n_out; ++j) {
                T d[TP], w[TU];
                ldv<TP>(d, zp);
#pragma unroll
                for (int u = 0; u < TU; ++u) w[u] = (ig * TU + u < L.n_in) ? wp[u] : T(0);
                zp += lda;
                wp += ldw;
#pragma unroll
                for (int u = 0; u < TU; ++u)
#pragma unroll
                    for (int p = 0; p < TP; ++p) acc[u][p] = fma(w[u], d[p], acc[u][p]);
            }
        }
#pragma unroll
        for (int u = 0; u < TU; ++u) {
            const int i = GLOBALW ? ig * TU + u : ig + UGI * u;
            if (i < L.n_in) {
                if (L.has_res) {
                    T pass[TP];
                    ldv<TP>(pass, D + (size_t)i * lda + pg * TP);
#pragma unroll
                    for (int p = 0; p < TP; ++p) acc[u][p] += pass[p];
                }
                qb_finish_delta_vec<T, TP, ACTM>(Lm, R, D, lda, i, pg * TP, acc[u]);
            }
        }
    }
}

template <typename T, bool GLOBALW, int TP>
__device__ __forceinline__ void qb_bwd_gemm(const QbLayerPlan& L, const QbLayerPlan& Lm, const T* sW, const T* theta,
                                            T* R, T* D, int lda, int TM) {
    if (Lm.act == QB_ACT_TANH) qb_bwd_gemm_a<T, GLOBALW, TP, QB_ACT_TANH>(L, Lm, sW, theta, R, D, lda, TM);
    else if (Lm.act == QB_ACT_RELU) qb_bwd_gemm_a<T, GLOBALW, TP, QB_ACT_RELU>(L, Lm, sW, theta, R, D, lda, TM);
    else qb_bwd_gemm_a<T, GLOBALW, TP, QB_ACT_IDENTITY>(L, Lm, sW, theta, R, D, lda, TM);
}

// The tile of qb_backprop_tiles as its hooks see it: activation rows R (leading dimension lda) of TM points from p0 on,
// the first `valid` of them below n1, o outputs from the top layer Ltop, and the pass over the tile.
template <typename T>
struct QbTile {
    T* R;
    const QbLayerPlan& Ltop;
    int lda, TM, o;
    int64_t p0;
    int valid, pass;
    // output j at tile point p
    __device__ __forceinline__ T& top(int j, int p) const { return R[(size_t)(Ltop.row_out + j) * lda + p]; }
};

// The back-propagation tile loop of kernels 2, 6 and 7, for one parameter vector over points [n0, n1): stage the
// weights, then per tile run the forward pass, set the top delta and walk the layers top-down.  At layer l's dW point
// its input rows a_in are intact and delta_z has been written in place over its output rows; the backward GEMM then
// overwrites layer l-1's output rows with its delta_z, so every activation above the input is gone after a pass.
// What differs between the kernels is in the hooks H (all __forceinline__):
//   zero()                          clears the block's output row before the first tile
//   passes(o)                       forward + backward passes per tile
//   after_forward(t)                after each forward pass; a hook that writes the tile adds its own barrier
//   top_delta(t, j, p, ssq)         delta of output j at tile point p; also called for the padded points of a partial
//                                   tile (p >= t.valid)
//   at_dw(t, l)                     layer l's dW point
//   sums_squares                    the loop returns the block sum of ssq (otherwise 0)
// TPG = points per thread tile in the gradient kernel: 4 (twice the threads per tile, for layers >= 64 wide) or 8
template <typename T, int TPG, typename H>
__device__ double qb_backprop_tiles_t(const QbPlan& P, const QbSmem& S, const T* theta, const T* __restrict__ x,
                                      int64_t n0, int64_t n1, H& h) {
    T* sW = reinterpret_cast<T*>(S.w);
    T* R = reinterpret_cast<T*>(S.act);
    const int lda = P.lda, TM = P.TM, o = P.out_dim, nl = P.n_layers;
    T* D = P.d_row >= 0 ? R + (size_t)P.d_row * lda : nullptr;
    __syncthreads();
    qb_stage_weights<T>(P, sW, theta);
    h.zero();
    __syncthreads();
    T ssq = T(0);
    const QbLayerPlan& Ltop = P.L[nl - 1];
    const QbScope bsc = qb_block_scope(TM);
    for (int64_t p0 = n0; p0 < n1; p0 += TM) {
        const int valid = (int)min((int64_t)TM, n1 - p0);
        qb_load_x_tile<T>(x, P.in_dim, p0, n1, R, lda, bsc);
        __syncthreads();
        for (int pass = 0; pass < h.passes(o); ++pass) {
            const QbTile<T> t{R, Ltop, lda, TM, o, p0, valid, pass};
            for (int l = 0; l < nl; ++l) {
                const QbLayerPlan& L = P.L[l];
                qb_layer_forward<T, TPG>(L, sW, R + (size_t)L.row_in * lda, R + (size_t)L.row_out * lda, lda, bsc, false);
            }
            h.after_forward(t);
            const int n = TM * o;
            for (int idx = threadIdx.x; idx < n; idx += blockDim.x) {
                const int j = idx / TM, p = idx - j * TM;
                const T da = h.top_delta(t, j, p, ssq);
                qb_finish_delta<T>(Ltop, R, D, lda, j, p, da);
            }
            __syncthreads();
            for (int l = nl - 1; l >= 0; --l) {
                const QbLayerPlan& L = P.L[l];
                h.at_dw(t, l);
                __syncthreads();
                if (l > 0) {
                    if (L.wr_off >= 0) qb_bwd_gemm<T, false, TPG>(L, P.L[l - 1], sW, theta, R, D, lda, TM);
                    else qb_bwd_gemm<T, true, TPG>(L, P.L[l - 1], sW, theta, R, D, lda, TM);
                    __syncthreads();
                }
            }
        }
    }
    if (H::sums_squares) return qb_block_sum((double)ssq, S.red);
    return 0.0;
}

template <typename T, typename H>
__device__ double qb_backprop_tiles(const QbPlan& P, const QbSmem& S, const T* theta, const T* __restrict__ x,
                                    int64_t n0, int64_t n1, H& h) {
    if (sizeof(T) == 4 && P.tpg == 8) return qb_backprop_tiles_t<T, VT<T>::TP>(P, S, theta, x, n0, n1, h);
    return qb_backprop_tiles_t<T, 4>(P, S, theta, x, n0, n1, h);
}

// kernel 2's hooks: g[0..n_params) receives d/dtheta of -0.5*ssq/sigma^2; delta at the top is r / sigma^2 (final_exp:
// times e^u) and zero at padded points
template <typename T>
struct QbGradHooks {
    static constexpr bool sums_squares = true;
    const QbPlan& P;
    const T* __restrict__ y;
    int64_t n1;
    double inv_sigma2;
    T* g;
    __device__ __forceinline__ void zero() const {
        for (int idx = threadIdx.x; idx < P.n_params; idx += blockDim.x) g[idx] = T(0);
    }
    __device__ __forceinline__ int passes(int) const { return 1; }
    __device__ __forceinline__ void after_forward(const QbTile<T>&) const {}
    __device__ __forceinline__ T top_delta(const QbTile<T>& t, int j, int p, T& ssq) const {
        const int64_t gp = t.p0 + p;
        T da = T(0);
        if (gp < n1) {
            T out = t.top(j, p);
            if (P.final_exp) out = qb_exp(out);
            const T r = __ldg(y + gp * t.o + j) - out;
            ssq = fma(r, r, ssq);
            da = r * T(inv_sigma2);
            if (P.final_exp) da *= out;
        }
        return da;
    }
    __device__ __forceinline__ void at_dw(const QbTile<T>& t, int l) const {
        qb_dw_accumulate<T>(P.L[l], t.R, t.lda, t.TM, g);
    }
};

// value + gradient of the data term for one parameter vector over points [n0, n1):
// returns sum of squared residuals; g[0..P) receives d/dtheta of  -0.5*ssq/sigma^2  (i.e. of lp's data term).
// g must be addressable by this block only (one row per (chain, split)).
template <typename T>
__device__ double qb_eval_value_grad(const QbPlan& P, const QbSmem& S, const T* theta, const T* __restrict__ x,
                                     const T* __restrict__ y, int64_t n0, int64_t n1, double inv_sigma2, T* g) {
    QbGradHooks<T> h{P, y, n1, inv_sigma2, g};
    return qb_backprop_tiles<T>(P, S, theta, x, n0, n1, h);
}

// --------------------------------------------------------------------------------------------
// likelihood / prior scalars
// --------------------------------------------------------------------------------------------
struct QbLikDev {
    double sigma, inv_sigma2, prior_sigma, prior_scale;
    const void* anchor;
    int anchor_per_chain;
    int has_prior;
};

// sum_p (theta_p - anchor_p)^2, block-uniform
template <typename T>
__device__ double qb_prior_ss(const QbLikDev& lk, const T* theta, int64_t k, int P, double* red) {
    const T* a = reinterpret_cast<const T*>(lk.anchor);
    if (a && lk.anchor_per_chain) a += k * (int64_t)P;
    double s = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const double d = (double)theta[i] - (a ? (double)a[i] : 0.0);
        s += d * d;
    }
    return qb_block_sum(s, red);
}

__device__ __forceinline__ double qb_lp_from(const QbLikDev& lk, double ssq, int64_t N, double prior_ss, int P) {
    const double LOG_2PI = 1.8378770664093454835606594728112;
    double nlp = 0.5 * ssq * lk.inv_sigma2 + 0.5 * (double)N * LOG_2PI + (double)N * log(lk.sigma);
    if (lk.has_prior) {
        const double sp2 = lk.prior_sigma * lk.prior_sigma;
        nlp += lk.prior_scale * (prior_ss / (2.0 * sp2) + 0.5 * (double)P * log(2.0 * 3.14159265358979323846 * sp2));
    }
    return -nlp;
}

// g += d/dtheta of the prior term of lp
template <typename T>
__device__ void qb_prior_grad_add(const QbLikDev& lk, const T* theta, int64_t k, int P, T* g) {
    if (!lk.has_prior) return;
    const T* a = reinterpret_cast<const T*>(lk.anchor);
    if (a && lk.anchor_per_chain) a += k * (int64_t)P;
    const double c = lk.prior_scale / (lk.prior_sigma * lk.prior_sigma);
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const double d = (double)theta[i] - (a ? (double)a[i] : 0.0);
        g[i] = (T)((double)g[i] - c * d);
    }
}

// --------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG + Box-Muller
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 qb_philox(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
enum { QB_STREAM_INCR = 0, QB_STREAM_Z0 = 1, QB_STREAM_UNIF = 2, QB_STREAM_VI = 3, QB_STREAM_SWAG = 4, QB_STREAM_NUTS = 5 };

__device__ __forceinline__ uint4 qb_rand4(uint64_t seed, int64_t chain, int64_t step, int stream, uint32_t idx4) {
    // seed and chain live in DIFFERENT words (key = seed, counter = chain/step/index): two (seed, chain) pairs never share
    // a stream, whatever their bits.  Injective for chain < 2^48, step < 2^40, stream < 256.
    const uint64_t ch = (uint64_t)chain, sp = (uint64_t)step;
    uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x5851F42Du);
    uint4 ctr = make_uint4(idx4, (uint32_t)sp, (uint32_t)ch,
                           ((uint32_t)stream & 0xFFu) | (((uint32_t)(sp >> 32) & 0xFFu) << 8) | (((uint32_t)(ch >> 32) & 0xFFFFu) << 16));
    return qb_philox(ctr, key);
}
__device__ __forceinline__ double qb_u01(uint32_t a) { return ((double)a + 0.5) * 2.3283064365386963e-10; }
__device__ __forceinline__ void qb_normal4(uint4 r, double (&z)[4]) {
    const double r1 = sqrt(-2.0 * log(qb_u01(r.x))), r2 = sqrt(-2.0 * log(qb_u01(r.z)));
    double s1, c1, s2, c2;
    sincospi(2.0 * qb_u01(r.y), &s1, &c1);
    sincospi(2.0 * qb_u01(r.w), &s2, &c2);
    z[0] = r1 * c1; z[1] = r1 * s1; z[2] = r2 * c2; z[3] = r2 * s2;
}
// fp32 Box-Muller on the special-function unit: lg2 / sqrt / sin / cos approximations (absolute error of sin and cos
// 2^-20.9 on (-pi, pi), which is where the angle is kept: cos(2 pi u) = -cos(2 pi u - pi)).  The fp64 version above is
// the one the numpy Philox oracle replays; the fp32 draws only have to be the same in every fp32 kernel.
__device__ __forceinline__ void qb_normal4(uint4 r, float (&z)[4]) {
    const float u1 = ((float)(r.x >> 8) + 0.5f) * 5.9604644775390625e-8f;
    const float u2 = ((float)(r.z >> 8) + 0.5f) * 5.9604644775390625e-8f;
    float r1, r2;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(-2.0f * __logf(u1)));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r2) : "f"(-2.0f * __logf(u2)));
    const float a1 = ((float)(r.y >> 8) + 0.5f) * 3.7450702829239286e-7f - 3.14159265358979f;     // 2 pi 2^-24
    const float a2 = ((float)(r.w >> 8) + 0.5f) * 3.7450702829239286e-7f - 3.14159265358979f;
    z[0] = -r1 * __cosf(a1); z[1] = -r1 * __sinf(a1); z[2] = -r2 * __cosf(a2); z[3] = -r2 * __sinf(a2);
}
