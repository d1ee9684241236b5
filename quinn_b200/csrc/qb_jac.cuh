// Kernel 7: per-point output Jacobians of the network with respect to theta, as per-layer pairs (a_l, d_l), from kernel
// 2's back-propagation tile loop (qb_backprop_tiles) with the hooks below.  sm_100a, CUDA cores (FFMA2 in fp32, DFMA in
// fp64).
//
// For output j of point i, layer l's part of d f_j(x_i) / d [W_l | b_l] is the outer product d_l[j] (x) [a_l; 1] of the
// layer's pre-activation gradient d_l[j] = d f_j / d z_l [n_out] and its input a_l [n_in].  Kernel 2 back-propagates
// delta = (y - f) / sigma^2 from the top; with delta = e_j (times e^u for final_exp) its delta_z rows are d_l[j].  At the
// point where kernel 2 calls qb_dw_accumulate for layer l, a_l is intact in shared memory and delta_z is written in
// place over the layer's output: both are copied to global memory there.  Polynomial terms (coef) and shared weights are
// applied by the caller when it assembles J from the pairs.
//
// Back-propagation overwrites the activations of every layer above the input, so each output j is a pass of its own
// that runs the forward pass again (the x rows are not overwritten).  Padded points of a partial last tile are never
// stored.
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

// Pass j back-propagates e_j (final_exp: times e^u) and stores the d_l rows of output j; pass 0 also writes f(x) to
// out[N, o] and stores the a_l rows (layout of fac in quinn_b200.h).
template <typename T>
struct QbJacHooks {
    static constexpr bool sums_squares = false;
    const QbJacPlan& J;
    int64_t N;
    T* out;
    T* fac;
    __device__ __forceinline__ void zero() const {}
    __device__ __forceinline__ int passes(int o) const { return o; }
    __device__ __forceinline__ void after_forward(const QbTile<T>&) const {}
    __device__ __forceinline__ T top_delta(const QbTile<T>& t, int q, int p, T&) const {
        T f = t.top(q, p);
        if (J.P.final_exp) f = qb_exp(f);
        if (t.pass == 0 && p < t.valid) out[(t.p0 + p) * t.o + q] = f;
        return q == t.pass ? (J.P.final_exp ? f : T(1)) : T(0);
    }
    __device__ __forceinline__ void at_dw(const QbTile<T>& t, int l) const {
        const QbLayerPlan& L = J.P.L[l];
        T* base = fac + (int64_t)J.row0[l] * N + t.p0;
        if (t.pass == 0) qb_jac_store_rows<T>(t.R + (size_t)L.row_in * t.lda, t.lda, L.n_in, t.valid, base, N);
        qb_jac_store_rows<T>(t.R + (size_t)L.row_out * t.lda, t.lda, L.n_out, t.valid,
                             base + (int64_t)(L.n_in + t.pass * L.n_out) * N, N);
    }
};
