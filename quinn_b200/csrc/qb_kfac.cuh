// Kernel 6: Kronecker factors of the per-point empirical Fisher of every Linear layer, accumulated in kernel 2's
// back-propagation tile loop (qb_backprop_tiles) with the hooks below.  sm_100a, CUDA cores (FFMA2 in fp32, DFMA in fp64).
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

// Kernel 2's top delta (its sum of squares is not returned); the factor row g[0..n_factors) is zeroed first, padded
// activation columns are zeroed after each forward pass, and layer l's dW point accumulates its factors.
// Inherited from QbGradHooks on purpose: top_delta and passes (one pass per tile).  Every other hook is defined here,
// so a hook added to QbGradHooks must be checked for kernel 6 as well.
template <typename T>
struct QbKfacHooks : QbGradHooks<T> {
    static constexpr bool sums_squares = false;
    const QbKfacPlan& K;
    __device__ __forceinline__ void zero() const {
        for (int idx = threadIdx.x; idx < K.n_factors; idx += blockDim.x) this->g[idx] = T(0);
    }
    __device__ __forceinline__ void after_forward(const QbTile<T>& t) const {
        // the value of t.valid, formed again here: reading t.valid instead costs the fp64 kernel 8 SASS instructions
        const int valid = (int)min((int64_t)t.TM, this->n1 - t.p0);
        if (valid < t.TM) {
            // padded points: every activation column zero (their delta is zero; their activations would enter A and s)
            const int w = t.TM - valid;
            for (int idx = threadIdx.x; idx < K.P.total_rows * w; idx += blockDim.x) {
                const int r = idx / w, p = valid + (idx - r * w);
                t.R[(size_t)r * t.lda + p] = T(0);
            }
            __syncthreads();
        }
    }
    __device__ __forceinline__ void at_dw(const QbTile<T>& t, int l) const {
        qb_dw_accumulate<T>(K.LA[l], t.R, t.lda, t.TM, this->g);
        qb_dw_accumulate<T>(K.LG[l], t.R, t.lda, t.TM, this->g);
    }
};
