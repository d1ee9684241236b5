// Kernel 7: per-point output Jacobians of the network with respect to theta, as per-layer pairs (a_l, d_l), through
// kernel 2's resident body.  sm_100a, CUDA cores (FFMA2 in fp32, DFMA in fp64).
//
// For output j of point i, layer l's part of d f_j(x_i) / d [W_l | b_l] is the outer product d_l[j] (x) [a_l; 1] of the
// layer's pre-activation gradient d_l[j] = d f_j / d z_l [n_out] and its input a_l [n_in].  Kernel 2 back-propagates
// delta = (y - f) / sigma^2 from the top; with delta = e_j (times e^u for final_exp) its delta_z rows are d_l[j].  At the
// point where kernel 2 calls qb_dw_accumulate for layer l, a_l is intact in shared memory and delta_z is written in
// place over the layer's output: both are copied to global memory there.  Polynomial terms (coef) and shared weights are
// applied by the caller when it assembles J from the pairs.
//
// Back-propagation overwrites the activations of every layer above the input, so each output j > 0 runs the forward
// pass again (the x rows are not overwritten).  Padded points of a partial last tile are never stored.
#pragma once
#include "qb_device.cuh"

struct QbJacPlan {
    QbPlan P;                        // kernel 2's resident plan (no tensor cores, not streamed)
    int row0[QB_MAX_LAYERS];         // first row of layer l in the factor buffer: n_in rows of a_l, then o*n_out of d_l
    int n_rows;                      // F = sum_l (n_in_l + o * n_out_l): rows of N elements
    int pad_;
};

// rows [r0, r0 + nr) of the tile (shared, leading dimension lda) -> rows of fac (leading dimension N) at column p0,
// the first `valid` points only
template <typename T>
__device__ __forceinline__ void qb_jac_store_rows(const T* R, int lda, int nr, int valid, T* dst, int64_t N) {
    for (int idx = threadIdx.x; idx < nr * valid; idx += blockDim.x) {
        const int r = idx / valid, p = idx - r * valid;
        dst[(int64_t)r * N + p] = R[(size_t)r * lda + p];
    }
}

// f(x) for the points [n0, n1) to out[N, o], and their pairs to fac (layout in quinn_b200.h)
template <typename T, int TPG>
__device__ void qb_jac_eval_t(const QbJacPlan& J, const QbSmem& S, const T* theta, const T* __restrict__ x,
                              int64_t N, int64_t n0, int64_t n1, T* out, T* fac) {
    const QbPlan& P = J.P;
    T* sW = reinterpret_cast<T*>(S.w);
    T* R = reinterpret_cast<T*>(S.act);
    const int lda = P.lda, TM = P.TM, o = P.out_dim, nl = P.n_layers;
    T* D = P.d_row >= 0 ? R + (size_t)P.d_row * lda : nullptr;
    __syncthreads();
    qb_stage_weights<T>(P, sW, theta);
    __syncthreads();
    const QbLayerPlan& Ltop = P.L[nl - 1];
    const QbScope bsc = qb_block_scope(TM);
    for (int64_t p0 = n0; p0 < n1; p0 += TM) {
        const int valid = (int)min((int64_t)TM, n1 - p0);
        qb_load_x_tile<T>(x, P.in_dim, p0, n1, R, lda, bsc);
        __syncthreads();
        for (int j = 0; j < o; ++j) {
            for (int l = 0; l < nl; ++l) {
                const QbLayerPlan& L = P.L[l];
                qb_layer_forward<T, TPG>(L, sW, R + (size_t)L.row_in * lda, R + (size_t)L.row_out * lda, lda, bsc, false);
            }
            // f (first pass) and the top delta e_j (final_exp: times e^u); each thread reads and writes its own entries
            for (int idx = threadIdx.x; idx < TM * o; idx += blockDim.x) {
                const int q = idx / TM, p = idx - q * TM;
                T f = R[(size_t)(Ltop.row_out + q) * lda + p];
                if (P.final_exp) f = qb_exp(f);
                if (j == 0 && p < valid) out[(p0 + p) * o + q] = f;
                const T da = q == j ? (P.final_exp ? f : T(1)) : T(0);
                qb_finish_delta<T>(Ltop, R, D, lda, q, p, da);
            }
            __syncthreads();
            for (int l = nl - 1; l >= 0; --l) {
                const QbLayerPlan& L = P.L[l];
                T* base = fac + (int64_t)J.row0[l] * N + p0;
                if (j == 0) qb_jac_store_rows<T>(R + (size_t)L.row_in * lda, lda, L.n_in, valid, base, N);
                qb_jac_store_rows<T>(R + (size_t)L.row_out * lda, lda, L.n_out, valid,
                                     base + (int64_t)(L.n_in + j * L.n_out) * N, N);
                __syncthreads();
                if (l > 0) {
                    if (L.wr_off >= 0) qb_bwd_gemm<T, false, TPG>(L, P.L[l - 1], sW, theta, R, D, lda, TM);
                    else qb_bwd_gemm<T, true, TPG>(L, P.L[l - 1], sW, theta, R, D, lda, TM);
                    __syncthreads();
                }
            }
        }
    }
}

template <typename T>
__device__ void qb_jac_eval(const QbJacPlan& J, const QbSmem& S, const T* theta, const T* __restrict__ x, int64_t N,
                            int64_t n0, int64_t n1, T* out, T* fac) {
    if (sizeof(T) == 4 && J.P.tpg == 8) qb_jac_eval_t<T, VT<T>::TP>(J, S, theta, x, N, n0, n1, out, fac);
    else qb_jac_eval_t<T, 4>(J, S, theta, x, N, n0, n1, out, fac);
}
