// Kernel 6: Kronecker factors of the per-point empirical Fisher of every Linear layer, accumulated through kernel 2's
// resident body.  sm_100a, CUDA cores (FFMA2 in fp32, DFMA in fp64).
//
// For layer l with input activations a_i and pre-activation gradients delta_i = d log p_i / d z_l of point i:
//   A_l = sum_i a_i a_i^T [n_in, n_in],   s_l = sum_i a_i [n_in] (layers with a bias),   G_l = sum_i delta_i delta_i^T
// [n_out, n_out].  Kernel 2 forms dW_l = delta_z a_in^T with qb_dw_accumulate at the point where both operands are in
// shared memory: a_in intact, delta_z written in place over the layer's output.  The factors are the same accumulation
// on the operand pairs (a_in, a_in) and (delta_z, delta_z), so each layer runs qb_dw_accumulate twice on re-pointed
// plans built by the host (LA: rows and "dz" = the input rows, bias pass = s_l; LG: both operands the delta rows, no
// bias) in place of the dW call.  The block's output row g holds the factors of all layers (layout in quinn_b200.h).
//
// Padded points of the last, partial tile carry delta = 0, but their activation columns do not (act(b) etc.): those
// columns are zeroed after the forward pass, before any factor pass reads them.
#pragma once
#include "qb_device.cuh"

struct QbKfacPlan {
    QbPlan P;                        // kernel 2's resident plan (no tensor cores, not streamed)
    QbLayerPlan LA[QB_MAX_LAYERS];   // A_l and s_l:  n_out = n_in, row_out = row_in, w_off -> A_l, b_off -> s_l or -1
    QbLayerPlan LG[QB_MAX_LAYERS];   // G_l:          n_in = n_out, row_in = row_out, w_off -> G_l, b_off = -1
    int n_factors;                   // elements of the factor row
    int pad_;
};

// Factors of the points [n0, n1) added to g[0..n_factors) (zeroed first).  g must be addressable by this block only.
template <typename T, int TPG>
__device__ void qb_kfac_eval_t(const QbKfacPlan& K, const QbSmem& S, const T* theta, const T* __restrict__ x,
                               const T* __restrict__ y, int64_t n0, int64_t n1, double inv_sigma2, T* g) {
    const QbPlan& P = K.P;
    T* sW = reinterpret_cast<T*>(S.w);
    T* R = reinterpret_cast<T*>(S.act);
    const int lda = P.lda, TM = P.TM, o = P.out_dim, nl = P.n_layers;
    T* D = P.d_row >= 0 ? R + (size_t)P.d_row * lda : nullptr;
    __syncthreads();
    qb_stage_weights<T>(P, sW, theta);
    for (int idx = threadIdx.x; idx < K.n_factors; idx += blockDim.x) g[idx] = T(0);
    __syncthreads();
    const T is2 = T(inv_sigma2);
    const QbLayerPlan& Ltop = P.L[nl - 1];
    const QbScope bsc = qb_block_scope(TM);
    for (int64_t p0 = n0; p0 < n1; p0 += TM) {
        qb_load_x_tile<T>(x, P.in_dim, p0, n1, R, lda, bsc);
        __syncthreads();
        for (int l = 0; l < nl; ++l) {
            const QbLayerPlan& L = P.L[l];
            qb_layer_forward<T, TPG>(L, sW, R + (size_t)L.row_in * lda, R + (size_t)L.row_out * lda, lda, bsc, false);
        }
        const int valid = (int)min((int64_t)TM, n1 - p0);
        if (valid < TM) {
            // padded points: every activation column zero (their delta is zero; their activations would enter A and s)
            const int w = TM - valid;
            for (int idx = threadIdx.x; idx < P.total_rows * w; idx += blockDim.x) {
                const int r = idx / w, p = valid + (idx - r * w);
                R[(size_t)r * lda + p] = T(0);
            }
            __syncthreads();
        }
        // delta at the top: d lp_i / d out = r / sigma^2 (final_exp: times e^u), as in kernel 2
        for (int idx = threadIdx.x; idx < TM * o; idx += blockDim.x) {
            const int j = idx / TM, p = idx - j * TM;
            const int64_t gp = p0 + p;
            T da = T(0);
            if (gp < n1) {
                T out = R[(size_t)(Ltop.row_out + j) * lda + p];
                if (P.final_exp) out = qb_exp(out);
                da = (__ldg(y + gp * o + j) - out) * is2;
                if (P.final_exp) da *= out;
            }
            qb_finish_delta<T>(Ltop, R, D, lda, j, p, da);
        }
        __syncthreads();
        for (int l = nl - 1; l >= 0; --l) {
            const QbLayerPlan& L = P.L[l];
            qb_dw_accumulate<T>(K.LA[l], R, lda, TM, g);
            qb_dw_accumulate<T>(K.LG[l], R, lda, TM, g);
            __syncthreads();
            if (l > 0) {
                if (L.wr_off >= 0) qb_bwd_gemm<T, false, TPG>(L, P.L[l - 1], sW, theta, R, D, lda, TM);
                else qb_bwd_gemm<T, true, TPG>(L, P.L[l - 1], sW, theta, R, D, lda, TM);
                __syncthreads();
            }
        }
    }
}

template <typename T>
__device__ void qb_kfac_eval(const QbKfacPlan& K, const QbSmem& S, const T* theta, const T* __restrict__ x,
                             const T* __restrict__ y, int64_t n0, int64_t n1, double inv_sigma2, T* g) {
    if (sizeof(T) == 4 && K.P.tpg == 8) qb_kfac_eval_t<T, VT<T>::TP>(K, S, theta, x, y, n0, n1, inv_sigma2, g);
    else qb_kfac_eval_t<T, 4>(K, S, theta, x, y, n0, n1, inv_sigma2, g);
}
