// Layer-streamed evaluation: networks whose parameter vector does not fit in shared memory next to one tile of
// activations.  Only activations stay resident; every layer's weights pass through a ring of NST shared-memory slots in
// chunks of consecutive OUTPUT rows (contiguous in theta: a Linear weight is (n_out, n_in) row-major).  Each slot is
// filled with per-thread cp.async of one element (theta rows start at k*P, which is not 16-byte aligned for odd P) and
// completes on its own mbarrier, so chunk c+1 and c+2 land while chunk c is multiplied.  sm_100a, CUDA cores: FFMA2 for
// fp32, DFMA for fp64.
//
// Per tile of TM points and per layer (DESIGN.md "Layer-streamed path"):
//   forward        out[j0+r][p] = act(sum_i W[j0+r][i] * in[i][p] + b[j0+r]) for the R rows of a chunk;
//   back-prop      dIn[i][p] += sum_r W[j0+r][i] * dz[j0+r][p] for the same chunks, in chunk order;
//   weight grads   dW = dz a_in^T over the whole layer (qb_dw_accumulate of the resident kernel: it needs no weights).
// The reduction axis of a chunk is split over KS lanes of one warp (KS a power of two) and combined with a fixed
// xor-shuffle tree, so fp64 results are the same bits run to run.
#pragma once
#include "qb_device.cuh"

#define QS_THREADS 256
#define QS_STAGES 3

struct QbStreamLayer {
    int R, nch;             // output rows per chunk (a multiple of TU), chunks per layer
    int ldw;                // shared row stride of a staged chunk: rup(n_in, TU)
    int lg_ks, kl;          // forward: log2 of the lanes splitting the n_in reduction, inputs per lane
    int lg_bks, bkl;        // back-propagation: log2 of the lanes splitting the R-row reduction, rows per lane
    int fwd_c0, bwd_c0;     // first chunk of this layer in the per-tile chunk schedule (bwd_c0 < 0: none)
    int cp_dr, cp_di;       // copy loop: QS_THREADS = cp_dr * n_in + cp_di
};

struct QbStreamPlan {
    int n_layers, in_dim, out_dim, n_params, final_exp, want_grad;
    int TM, lda, lg_pg;     // tile points, activation row stride, log2(TM / TP)
    int slot_elems;         // elements of one ring slot
    int n_chunks;           // chunks per tile (forward + back-propagation)
    int buf_rows;           // value path: rows of each of the two activation buffers
    int total_rows;         // gradient path: rows of all kept activations
    int da_rows;            // gradient path: rows of the back-propagated delta accumulator
    int ring_off, act_off, da_off;   // byte offsets in dynamic shared memory
    int act_elems;          // elements of the activation area (scratch of the chain kernels' proposal pass)
    long long smem_bytes;
    QbLayerPlan L[QB_MAX_LAYERS];    // n_in, n_out, offsets, activation, residual, polynomial terms; row_in / row_out and
                                     // the dW split of the gradient path (qb_dw_accumulate)
    QbStreamLayer SL[QB_MAX_LAYERS];
};

// thread tile: TU output rows x TP points; VW = elements per 128-bit load
template <typename T> struct QsT;
template <> struct QsT<float>  { static constexpr int TU = 8, TP = 4, VW = 4; };
template <> struct QsT<double> { static constexpr int TU = 4, TP = 4, VW = 2; };

// --------------------------------------------------------------------------------------------
// weight ring: NST slots, one mbarrier each (NST arrivals per fill: every thread's cp.async group)
// --------------------------------------------------------------------------------------------
struct QsRing {
    unsigned char* slots;
    uint64_t* bar;
    long long used;         // chunks consumed by earlier evaluations of this block (slot / parity bookkeeping)
};

__device__ __forceinline__ uint32_t qs_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void qs_ring_init(const QbStreamPlan& P, unsigned char* smem, QsRing& rg) {
    rg.slots = smem + P.ring_off;
    rg.bar = reinterpret_cast<uint64_t*>(smem + 40 * sizeof(double));
    rg.used = 0;
    if (threadIdx.x < QS_STAGES)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(qs_smem(rg.bar + threadIdx.x)), "r"(QS_THREADS) : "memory");
    __syncthreads();
}

template <typename T> __device__ __forceinline__ void qs_cp(T* dst, const T* src);
template <> __device__ __forceinline__ void qs_cp<float>(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(qs_smem(dst)), "l"(src) : "memory");
}
template <> __device__ __forceinline__ void qs_cp<double>(double* dst, const double* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(qs_smem(dst)), "l"(src) : "memory");
}

// bounded like qb_mbar_wait (qb_tc.cuh): a protocol bug ends the kernel with an error instead of hanging the GPU
__device__ __forceinline__ void qs_wait(uint64_t* bar, uint32_t parity) {
    unsigned long long t0 = 0;
    for (uint32_t it = 0;; ++it) {
        uint32_t ok;
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.b32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(qs_smem(bar)), "r"(parity) : "memory");
        if (ok) return;
        if ((it & 1023u) == 1023u) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 20000000000ULL) __trap();
        }
    }
}

// chunk c of the per-tile schedule -> layer, first row, direction
__device__ __forceinline__ void qs_decode(const QbStreamPlan& P, int c, int& l, int& j0) {
    for (l = 0; l < P.n_layers; ++l) {
        const QbStreamLayer& S = P.SL[l];
        if (c >= S.fwd_c0 && c < S.fwd_c0 + S.nch) { j0 = (c - S.fwd_c0) * S.R; return; }
        if (S.bwd_c0 >= 0 && c >= S.bwd_c0 && c < S.bwd_c0 + S.nch) { j0 = (c - S.bwd_c0) * S.R; return; }
    }
    l = 0; j0 = 0;
}

// issue the copies of chunk c (schedule position c % n_chunks) into its slot; every thread arrives once on the slot's
// mbarrier when its own copies have landed.  Polynomial layers stage each term in its own part of the slot.
template <typename T>
__device__ __forceinline__ void qs_fetch(const QbStreamPlan& P, const QsRing& rg, const T* __restrict__ theta, long long g) {
    const int slot = (int)(g % QS_STAGES);
    T* dst0 = reinterpret_cast<T*>(rg.slots) + (size_t)slot * P.slot_elems;
    int l, j0;
    qs_decode(P, (int)(g - rg.used) % P.n_chunks, l, j0);
    const QbLayerPlan& L = P.L[l];
    const QbStreamLayer& S = P.SL[l];
    const int n_in = L.n_in, rv = min(S.R, L.n_out - j0), n = rv * n_in, ldw = S.ldw;
    const int nterm = L.n_terms > 1 ? L.n_terms : 1;
    for (int m = 0; m < nterm; ++m) {
        const T* src = theta + L.w_off + (size_t)m * L.w_stride + (size_t)j0 * n_in;
        T* dst = dst0 + (size_t)m * S.R * ldw;
        int r = threadIdx.x / n_in, i = threadIdx.x - r * n_in;
        for (int e = threadIdx.x; e < n; e += QS_THREADS) {
            qs_cp<T>(dst + r * ldw + i, src + e);
            i += S.cp_di; r += S.cp_dr;
            if (i >= n_in) { i -= n_in; ++r; }
        }
    }
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" :: "r"(qs_smem(rg.bar + slot)) : "memory");
}

// wait for chunk g; on return every thread has finished with chunk g-1, so its slot is refilled with chunk g+NST-1
template <typename T>
__device__ __forceinline__ T* qs_acquire(const QbStreamPlan& P, const QsRing& rg, const T* theta, long long g, long long g_end) {
    const int slot = (int)(g % QS_STAGES);
    qs_wait(rg.bar + slot, (uint32_t)((g / QS_STAGES) & 1));
    __syncthreads();
    if (g + QS_STAGES - 1 < g_end) qs_fetch<T>(P, rg, theta, g + QS_STAGES - 1);
    T* w = reinterpret_cast<T*>(rg.slots) + (size_t)slot * P.slot_elems;
    // polynomial-in-depth layer: W = sum_m coef[m] * W_m, summed in the reference's order (qb_layer_param)
    int l, j0;
    qs_decode(P, (int)(g - rg.used) % P.n_chunks, l, j0);
    const QbLayerPlan& L = P.L[l];
    if (L.n_terms > 1) {
        const QbStreamLayer& S = P.SL[l];
        const int n = S.R * S.ldw;
        for (int e = threadIdx.x; e < n; e += QS_THREADS) {
            T v = T(0);
            for (int m = 0; m < L.n_terms; ++m) v = qb_add_rn(v, qb_mul_rn(w[e + m * n], (T)L.coef[m]));
            w[e] = v;
        }
        __syncthreads();
    }
    return w;
}

// --------------------------------------------------------------------------------------------
// chunk products
// --------------------------------------------------------------------------------------------
// acc[u][p] += sum_{i in [i0, i1)} W[u][i] * A[i][p]   (W: TU rows of stride ldw, A: rows of stride lda at the tile's points)
__device__ __forceinline__ void qs_fwd_acc(float (&acc)[8][4], const float* W, int ldw, const float* A, int lda, int i0, int i1) {
    float2 c[8][2];
#pragma unroll
    for (int u = 0; u < 8; ++u) { c[u][0] = make_float2(0.f, 0.f); c[u][1] = make_float2(0.f, 0.f); }
    int i = i0;
#pragma unroll 1
    for (; i + 4 <= i1; i += 4) {
        float4 w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) w[u] = *reinterpret_cast<const float4*>(W + u * ldw + i);
        float2 a[4][2];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 v = *reinterpret_cast<const float4*>(A + (i + q) * lda);
            a[q][0] = make_float2(v.x, v.y); a[q][1] = make_float2(v.z, v.w);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float ws[4] = {w[u].x, w[u].y, w[u].z, w[u].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float2 wb = make_float2(ws[q], ws[q]);
                c[u][0] = __ffma2_rn(a[q][0], wb, c[u][0]);
                c[u][1] = __ffma2_rn(a[q][1], wb, c[u][1]);
            }
        }
    }
#pragma unroll 1
    for (; i < i1; ++i) {
        const float4 v = *reinterpret_cast<const float4*>(A + i * lda);
        const float2 a0 = make_float2(v.x, v.y), a1 = make_float2(v.z, v.w);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float ws = W[u * ldw + i];
            c[u][0] = __ffma2_rn(a0, make_float2(ws, ws), c[u][0]);
            c[u][1] = __ffma2_rn(a1, make_float2(ws, ws), c[u][1]);
        }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) { acc[u][0] = c[u][0].x; acc[u][1] = c[u][0].y; acc[u][2] = c[u][1].x; acc[u][3] = c[u][1].y; }
}
__device__ __forceinline__ void qs_fwd_acc(double (&acc)[4][4], const double* W, int ldw, const double* A, int lda, int i0, int i1) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[u][p] = 0.0;
    int i = i0;
#pragma unroll 1
    for (; i + 2 <= i1; i += 2) {
        double2 w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) w[u] = *reinterpret_cast<const double2*>(W + u * ldw + i);
        double a[2][4];
#pragma unroll
        for (int q = 0; q < 2; ++q) ldv<4>(a[q], A + (i + q) * lda);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = fma(w[u].y, a[1][p], fma(w[u].x, a[0][p], acc[u][p]));
    }
    if (i < i1) {
        double a[4];
        ldv<4>(a, A + i * lda);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double ws = W[u * ldw + i];
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = fma(ws, a[p], acc[u][p]);
        }
    }
}

// acc[t][p] += sum_{r in [r0, r1)} W[r][t] * D[r][p]   (back-propagation: TU consecutive inputs t, W rows of stride ldw)
__device__ __forceinline__ void qs_bwd_acc(float (&acc)[8][4], const float* W, int ldw, const float* D, int lda, int r0, int r1) {
    float2 c[8][2];
#pragma unroll
    for (int u = 0; u < 8; ++u) { c[u][0] = make_float2(0.f, 0.f); c[u][1] = make_float2(0.f, 0.f); }
#pragma unroll 2
    for (int r = r0; r < r1; ++r) {
        const float4 w0 = *reinterpret_cast<const float4*>(W + r * ldw), w1 = *reinterpret_cast<const float4*>(W + r * ldw + 4);
        const float4 v = *reinterpret_cast<const float4*>(D + r * lda);
        const float2 d0 = make_float2(v.x, v.y), d1 = make_float2(v.z, v.w);
        const float ws[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float2 wb = make_float2(ws[u], ws[u]);
            c[u][0] = __ffma2_rn(d0, wb, c[u][0]);
            c[u][1] = __ffma2_rn(d1, wb, c[u][1]);
        }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) { acc[u][0] = c[u][0].x; acc[u][1] = c[u][0].y; acc[u][2] = c[u][1].x; acc[u][3] = c[u][1].y; }
}
__device__ __forceinline__ void qs_bwd_acc(double (&acc)[4][4], const double* W, int ldw, const double* D, int lda, int r0, int r1) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[u][p] = 0.0;
#pragma unroll 2
    for (int r = r0; r < r1; ++r) {
        double w[4], d[4];
        ldv<4>(w, W + r * ldw);
        ldv<4>(d, D + r * lda);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[u][p] = fma(w[u], d[p], acc[u][p]);
    }
}

// Work items of a chunk: `nsub` thread tiles x KS = 2^lg_ks reduction slices.  The KS slices of a tile sit in lanes
// lane, lane + 32/KS, .. of one warp (tiles vary fastest within a warp: the points of one weight row are neighbours),
// and are combined with a fixed xor-shuffle tree.  Every thread runs the same number of passes (the shuffles need
// whole warps).
struct QsItem { int sub, ks; bool valid; };
__device__ __forceinline__ QsItem qs_item(int item, int lg_ks, int nsub) {
    const int lg = 5 - lg_ks, lane = item & 31;
    QsItem it;
    it.ks = lane >> lg;
    it.sub = ((item >> 5) << lg) | (lane & ((1 << lg) - 1));
    it.valid = it.sub < nsub;
    return it;
}
__host__ __device__ __forceinline__ int qs_items(int nsub, int lg_ks) {
    const int g = 1 << (5 - lg_ks);
    return ((nsub + g - 1) / g * g) << lg_ks;
}
template <typename T, int A, int B>
__device__ __forceinline__ void qs_reduce(T (&acc)[A][B], int lg_ks) {
    for (int off = 16; off >= (1 << (5 - lg_ks)); off >>= 1) {
#pragma unroll
        for (int a = 0; a < A; ++a)
#pragma unroll
            for (int b = 0; b < B; ++b) acc[a][b] += __shfl_xor_sync(0xffffffffu, acc[a][b], off);
    }
}

// forward chunk: rows j0 .. j0+R of layer L from the staged W (rows of stride ldw)
template <typename T>
__device__ __forceinline__ void qs_fwd_chunk(const QbStreamPlan& P, int l, const T* W, const T* __restrict__ theta,
                                             const T* Ain, T* Aout, int j0) {
    constexpr int TU = QsT<T>::TU, TP = QsT<T>::TP;
    const QbLayerPlan& L = P.L[l];
    const QbStreamLayer& S = P.SL[l];
    const int lda = P.lda, rv = min(S.R, L.n_out - j0), PGm = (1 << P.lg_pg) - 1;
    const int nsub = (S.R / TU) << P.lg_pg, items = qs_items(nsub, S.lg_ks);
    const bool res = L.has_res != 0;
    const T step = T(L.res_step);
    for (int base = 0; base < items; base += QS_THREADS) {
        const QsItem it = qs_item(base + threadIdx.x, S.lg_ks, nsub);
        const int pg = it.sub & PGm, ug = it.sub >> P.lg_pg, pcol = pg * TP;
        const int i0 = it.ks * S.kl, i1 = min(L.n_in, i0 + S.kl);
        T acc[TU][TP];
        if (it.valid && i0 < i1) qs_fwd_acc(acc, W + ug * TU * S.ldw, S.ldw, Ain + pcol, lda, i0, i1);
        else {
#pragma unroll
            for (int u = 0; u < TU; ++u)
#pragma unroll
                for (int p = 0; p < TP; ++p) acc[u][p] = T(0);
        }
        qs_reduce(acc, S.lg_ks);
        if (it.valid && it.ks == 0) {
#pragma unroll
            for (int u = 0; u < TU; ++u) {
                const int r = ug * TU + u;
                if (r < rv) {
                    const int j = j0 + r;
                    const T b = L.b_off >= 0 ? qb_layer_param<T>(L, theta, L.b_off + j, L.b_stride) : T(0);
                    T h[TP];
#pragma unroll
                    for (int p = 0; p < TP; ++p) {
                        const T z = acc[u][p] + b;
                        // fp32 tanh: qb_tanh applies the 2*log2(e) scale that the resident path folds into its staged W
                        h[p] = L.act == QB_ACT_TANH ? qb_tanh(z) : (L.act == QB_ACT_RELU ? (z > T(0) ? z : T(0)) : z);
                    }
                    if (res) {
                        T rin[TP];
                        ldv<TP>(rin, Ain + (size_t)j * lda + pcol);
#pragma unroll
                        for (int p = 0; p < TP; ++p) h[p] = fma(step, h[p], rin[p]);
                    }
                    stv<TP>(Aout + (size_t)j * lda + pcol, h);
                }
            }
        }
    }
}

// back-propagation chunk: DA[i][p] (+)= sum_{r < R} W[r][i] * dz[j0+r][p]; `first`: the chunk overwrites DA
template <typename T>
__device__ __forceinline__ void qs_bwd_chunk(const QbStreamPlan& P, int l, const T* W, const T* Dz, T* DA, int j0, bool first) {
    constexpr int TU = QsT<T>::TU, TP = QsT<T>::TP;
    const QbLayerPlan& L = P.L[l];
    const QbStreamLayer& S = P.SL[l];
    const int lda = P.lda, rv = min(S.R, L.n_out - j0), PGm = (1 << P.lg_pg) - 1;
    const int nsub = ((L.n_in + TU - 1) / TU) << P.lg_pg, items = qs_items(nsub, S.lg_bks);
    const T* D = Dz + (size_t)j0 * lda;
    for (int base = 0; base < items; base += QS_THREADS) {
        const QsItem it = qs_item(base + threadIdx.x, S.lg_bks, nsub);
        const int pg = it.sub & PGm, ig = it.sub >> P.lg_pg, pcol = pg * TP;
        const int r0 = it.ks * S.bkl, r1 = min(rv, r0 + S.bkl);
        T acc[TU][TP];
        if (it.valid && r0 < r1) qs_bwd_acc(acc, W + ig * TU, S.ldw, D + pcol, lda, r0, r1);
        else {
#pragma unroll
            for (int u = 0; u < TU; ++u)
#pragma unroll
                for (int p = 0; p < TP; ++p) acc[u][p] = T(0);
        }
        qs_reduce(acc, S.lg_bks);
        if (it.valid && it.ks == 0) {
#pragma unroll
            for (int u = 0; u < TU; ++u) {
                const int i = ig * TU + u;
                if (i < L.n_in) {
                    T* da = DA + (size_t)i * lda + pcol;
                    T v[TP];
                    if (first) {
#pragma unroll
                        for (int p = 0; p < TP; ++p) v[p] = acc[u][p];
                    } else {
                        ldv<TP>(v, da);
#pragma unroll
                        for (int p = 0; p < TP; ++p) v[p] += acc[u][p];
                    }
                    stv<TP>(da, v);
                }
            }
        }
    }
}

// --------------------------------------------------------------------------------------------
// one parameter vector over points [n0, n1)
// --------------------------------------------------------------------------------------------
// GRAD = false: returns the sum of squared residuals, or (out != nullptr, predictive) writes out[p*o + j] instead.
// GRAD = true: also g[0..P) = d/dtheta of -0.5*ssq*inv_sigma2 (g is owned by this block, as in qb_eval_value_grad).
template <typename T, bool GRAD>
__device__ double qs_eval(const QbStreamPlan& P, unsigned char* smem, QsRing& rg, const T* __restrict__ theta,
                          const T* __restrict__ x, const T* __restrict__ y, int64_t n0, int64_t n1, double inv_sigma2,
                          T* g, T* out) {
    const int lda = P.lda, TM = P.TM, o = P.out_dim, nl = P.n_layers;
    T* act = reinterpret_cast<T*>(smem + P.act_off);
    T* DA = reinterpret_cast<T*>(smem + P.da_off);
    double* red = reinterpret_cast<double*>(smem);
    const int64_t ntiles = (n1 - n0 + TM - 1) / TM;
    const long long g_beg = rg.used, g_end = rg.used + ntiles * P.n_chunks;
    __syncthreads();                  // earlier users of the ring and of the activation area are done
    if (GRAD) {
        for (int idx = threadIdx.x; idx < P.n_params; idx += blockDim.x) g[idx] = T(0);
    }
    for (long long q = g_beg; q < g_beg + QS_STAGES - 1 && q < g_end; ++q) qs_fetch<T>(P, rg, theta, q);
    long long gc = g_beg;
    T ssq = T(0);
    const T is2 = T(inv_sigma2);
    const QbScope bsc = qb_block_scope(TM);
    const QbLayerPlan& Ltop = P.L[nl - 1];
    for (int64_t p0 = n0; p0 < n1; p0 += TM) {
        __syncthreads();              // the previous tile no longer reads the input rows
        qb_load_x_tile<T>(x, P.in_dim, p0, n1, act, lda, bsc);
        T* cur = act;
        T* oth = act + (size_t)P.buf_rows * lda;
        for (int l = 0; l < nl; ++l) {
            const QbLayerPlan& L = P.L[l];
            const T* Ain = GRAD ? act + (size_t)L.row_in * lda : cur;
            T* Aout = GRAD ? act + (size_t)L.row_out * lda : oth;
            for (int ch = 0; ch < P.SL[l].nch; ++ch, ++gc) {
                const T* W = qs_acquire<T>(P, rg, theta, gc, g_end);
                qs_fwd_chunk<T>(P, l, W, theta, Ain, Aout, ch * P.SL[l].R);
            }
            T* t = cur; cur = oth; oth = t;
        }
        __syncthreads();
        const T* top = GRAD ? act + (size_t)Ltop.row_out * lda : cur;
        for (int idx = threadIdx.x; idx < TM * o; idx += blockDim.x) {
            const int j = idx / TM, p = idx - j * TM;
            const int64_t gp = p0 + p;
            if (!GRAD && out) {
                if (gp < n1) {
                    T v = top[(size_t)j * lda + p];
                    if (P.final_exp) v = qb_exp(v);
                    out[gp * o + j] = v;
                }
                continue;
            }
            T da = T(0);
            T v = top[(size_t)j * lda + p];
            if (gp < n1) {
                T f = v;
                if (P.final_exp) f = qb_exp(f);
                const T r = __ldg(y + gp * o + j) - f;
                ssq = fma(r, r, ssq);
                da = r * is2;
                if (P.final_exp) da *= f;
            }
            if (GRAD) {
                // delta_z of the top layer, in place over its outputs; a residual top layer passes da on through DA
                T* po = act + (size_t)(Ltop.row_out + j) * lda + p;
                if (Ltop.has_res) {
                    const T ain = act[(size_t)(Ltop.row_in + j) * lda + p];
                    const T step = T(Ltop.res_step);
                    *po = step * da * qb_dact<T>(Ltop.act, (v - ain) / step);
                    DA[(size_t)j * lda + p] = da;
                } else {
                    *po = da * qb_dact<T>(Ltop.act, v);
                }
            }
        }
        if (GRAD) {
            __syncthreads();
            for (int l = nl - 1; l >= 0; --l) {
                const QbLayerPlan& L = P.L[l];
                qb_dw_accumulate<T>(L, act, lda, TM, g);
                if (l == 0) break;
                const T* Dz = act + (size_t)L.row_out * lda;
                for (int ch = 0; ch < P.SL[l].nch; ++ch, ++gc) {
                    const T* W = qs_acquire<T>(P, rg, theta, gc, g_end);
                    qs_bwd_chunk<T>(P, l, W, Dz, DA, ch * P.SL[l].R, ch == 0 && !L.has_res);
                }
                __syncthreads();
                // DA = delta of layer l-1's output -> its delta_z, in place over its activations (qb_finish_delta);
                // a residual layer l-1 keeps DA as the pass-through of its own back-propagation
                const QbLayerPlan& Lm = P.L[l - 1];
                const int n = Lm.n_out * TM;
                for (int idx = threadIdx.x; idx < n; idx += blockDim.x) {
                    const int i = idx / TM, p = idx - i * TM;
                    const T da = DA[(size_t)i * lda + p];
                    T* po = act + (size_t)(Lm.row_out + i) * lda + p;
                    const T aout = *po;
                    if (Lm.has_res) {
                        const T ain = act[(size_t)(Lm.row_in + i) * lda + p];
                        const T step = T(Lm.res_step);
                        *po = step * da * qb_dact<T>(Lm.act, (aout - ain) / step);
                    } else {
                        *po = da * qb_dact<T>(Lm.act, aout);
                    }
                }
                __syncthreads();
            }
        }
    }
    rg.used = g_end;
    if (!GRAD && out) { __syncthreads(); return 0.0; }
    return qb_block_sum((double)ssq, red);
}
