// Kernel 5: exact Hessian-vector products of the log-posterior, hv = (d^2 lp / d theta^2) v, by forward-over-reverse
// differentiation (Pearlmutter's R-operator) of kernel 2's body.  sm_100a, CUDA cores (FFMA2 in fp32, DFMA in fp64).
//
// One block evaluates one direction v_k over one N-split at a single theta.  Shared memory holds, per layer,
//   forward block   [W^T (n_in_pad rows, rows >= n_in zero) ; V^T (n_in rows)]      (columns permuted as in kernel 2)
//   biases          [b (n_out_pad) ; v_b (n_out_pad)]
//   backward block  [W (n_out_pad rows, rows >= n_out zero) ; V (n_out rows)]       (layers > 0)
// and, per layer boundary, the tangent rows directly followed by the activation rows of one tile: [a_dot ; a].  Because
// the weight blocks are stacked the same way, one pass of the shared GEMM helper computes
//   z_dot       = W a_dot_in + V a_in + v_b               over [a_dot_in ; a_in]      with [W^T ; V^T]
//   dda_in      = W^T dz_dot + V^T dz                    over [dz_dot ; dz]          with [W ; V]
// fp32 tanh layers stage W, b, V and v_b times 2 log2(e) (DESIGN.md section 3), so z_dot comes out with the same fold and
// is divided by it in the epilogue.
//
// Ordering: as in kernel 2, delta_z and its tangent overwrite the activation and tangent rows of a layer's output in
// place.  Each element is converted by the thread that computed delta_a for it, after it has read a_out, a_dot_out and,
// for residual layers, a_in and a_dot_in of that element; rows of the layer's input are converted only when the layer
// below is back-propagated, after both weight-gradient passes of this layer have read them.
#pragma once
#include "qb_device.cuh"

struct QbHvpPlan {
    QbPlan P;                        // forward layers (all GEMM mode), weight offsets, activation rows
    QbLayerPlan LA[QB_MAX_LAYERS];   // weight pass 1: dz_dot x a_in^T and sum dz_dot (bias)
    QbLayerPlan LB[QB_MAX_LAYERS];   // weight pass 2: dz x a_dot_in^T (no bias)
    int dd_row;                      // first row of the tangent residual pass-through buffer, or -1 (P.d_row: primal)
    int pad_;
};

// One entry of V (or v_b) of a layer: from the direction vector, or from the unit vector e_unit when v is NULL.  The unit
// case gives exactly what qb_layer_param gives for an explicit e_unit (one non-zero term, the others add zeros).
template <typename T>
__device__ __forceinline__ T qb_hvp_dir(const QbLayerPlan& L, const T* v, int unit, int off, int stride) {
    if (v) return qb_layer_param<T>(L, v, off, stride);
    if (L.n_terms <= 1) return off == unit ? T(1) : T(0);
    T r = T(0);
    for (int m = 0; m < L.n_terms; ++m)
        if (off + m * stride == unit) r = (T)L.coef[m];
    return r;
}

template <typename T>
__device__ void qb_hvp_stage(const QbPlan& P, T* sW, const T* theta, const T* v, int unit) {
    constexpr int TU = VT<T>::TU;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int l = 0; l < P.n_layers; ++l) {
        const QbLayerPlan& L = P.L[l];
        const int UG = L.n_out_pad / TU;
        const T fold = (L.act == QB_ACT_TANH) ? qb_tanh_fold<T>() : T(1);
        T* Wt = sW + L.wt_off;
        const int nwt = (L.n_in_pad + L.n_in) * L.n_out_pad;
        for (int idx = tid; idx < nwt; idx += nt) {
            const int r = idx / L.n_out_pad, col = idx - r * L.n_out_pad;
            const int j = qb_col_to_unit<T>(col, UG);
            const bool dir = r >= L.n_in_pad;
            const int i = dir ? r - L.n_in_pad : r;
            T val = T(0);
            if (j < L.n_out && i < L.n_in) {
                const int off = L.w_off + j * L.n_in + i;
                val = dir ? qb_hvp_dir<T>(L, v, unit, off, L.w_stride) : qb_layer_param<T>(L, theta, off, L.w_stride);
            }
            Wt[idx] = val * fold;
        }
        T* bs = sW + L.bias_off;
        for (int idx = tid; idx < 2 * L.n_out_pad; idx += nt) {
            const bool dir = idx >= L.n_out_pad;
            const int j = qb_col_to_unit<T>(dir ? idx - L.n_out_pad : idx, UG);
            T val = T(0);
            if (j < L.n_out && L.b_off >= 0)
                val = dir ? qb_hvp_dir<T>(L, v, unit, L.b_off + j, L.b_stride) : qb_layer_param<T>(L, theta, L.b_off + j, L.b_stride);
            bs[idx] = val * fold;
        }
        if (L.wr_off >= 0) {
            const int UGI = L.n_in_pad / TU;
            T* Wr = sW + L.wr_off;
            const int nwr = (L.n_out_pad + L.n_out) * L.n_in_pad;
            for (int idx = tid; idx < nwr; idx += nt) {
                const int r = idx / L.n_in_pad, col = idx - r * L.n_in_pad;
                const int i = qb_col_to_unit<T>(col, UGI);
                const bool dir = r >= L.n_out_pad;
                const int j = dir ? r - L.n_out_pad : r;
                T val = T(0);
                if (j < L.n_out && i < L.n_in) {
                    const int off = L.w_off + j * L.n_in + i;
                    val = dir ? qb_hvp_dir<T>(L, v, unit, off, L.w_stride) : qb_layer_param<T>(L, theta, off, L.w_stride);
                }
                Wr[idx] = val;
            }
        }
    }
}

template <int TP, typename T> __device__ __forceinline__ void qb_hvp_ld(T (&d)[TP], const T* s) {
    if constexpr (TP == 1) d[0] = *s; else ldv<TP>(d, s);
}
template <int TP, typename T> __device__ __forceinline__ void qb_hvp_st(T* d, const T (&s)[TP]) {
    if constexpr (TP == 1) *d = s[0]; else stv<TP>(d, s);
}

// Tangent forward of layer L: a_dot_out = s_dot (or a_dot_in + step * s_dot), s_dot = act'(z) z_dot.  Needs the primal
// forward of the layer to be complete (s is read back from a_out).
template <typename T, int TP, int ACT>
__device__ void qb_hvp_tangent_fwd_a(const QbLayerPlan& L, const T* sW, T* R, int lda, int TM) {
    constexpr int TU = VT<T>::TU;
    const int UG = L.n_out_pad / TU, PG = TM / TP, items = UG * PG;
    const T* Wt = sW + L.wt_off;
    const T* vb = sW + L.bias_off + L.n_out_pad;
    const T* Tin = R + (size_t)(L.row_in - L.n_in_pad) * lda;
    const T* Ain = R + (size_t)L.row_in * lda;
    const T* Aout = R + (size_t)L.row_out * lda;
    T* Tout = R + (size_t)(L.row_out - L.n_out_pad) * lda;
    const T inv_fold = T(1) / (ACT == QB_ACT_TANH ? qb_tanh_fold<T>() : T(1));
    const bool res = L.has_res != 0;
    const T step = T(L.res_step), inv_step = res ? T(1) / step : T(1);
    for (int item = threadIdx.x; item < items; item += blockDim.x) {
        int pg, ug;
        if (L.ug_shift >= 0) { pg = item >> L.ug_shift; ug = item & (UG - 1); }
        else { pg = item / UG; ug = item - pg * UG; }
        const int pcol = pg * TP;
        T acc[TU][TP];
        qb_gemm_accumulate<TP>(acc, Wt, vb, Tin + pcol, L.n_in_pad + L.n_in, lda, L.n_out_pad, ug, UG);
#pragma unroll
        for (int u = 0; u < TU; ++u) {
            const int j = ug + UG * u;
            T s[TP], ta[TP];
            ldv<TP>(s, Aout + (size_t)j * lda + pcol);
            if (res) {
                T ai[TP], ti[TP];
                ldv<TP>(ai, Ain + (size_t)j * lda + pcol);
                ldv<TP>(ti, Tin + (size_t)j * lda + pcol);
#pragma unroll
                for (int p = 0; p < TP; ++p) {
                    const T sd = qb_dact_c<ACT, T>((s[p] - ai[p]) * inv_step) * (acc[u][p] * inv_fold);
                    ta[p] = fma(step, sd, ti[p]);
                }
            } else {
#pragma unroll
                for (int p = 0; p < TP; ++p) ta[p] = qb_dact_c<ACT, T>(s[p]) * (acc[u][p] * inv_fold);
            }
            stv<TP>(Tout + (size_t)j * lda + pcol, ta);
        }
    }
}

template <typename T, int TP>
__device__ __forceinline__ void qb_hvp_tangent_fwd(const QbLayerPlan& L, const T* sW, T* R, int lda, int TM) {
    if (L.act == QB_ACT_TANH) qb_hvp_tangent_fwd_a<T, TP, QB_ACT_TANH>(L, sW, R, lda, TM);
    else if (L.act == QB_ACT_RELU) qb_hvp_tangent_fwd_a<T, TP, QB_ACT_RELU>(L, sW, R, lda, TM);
    else qb_hvp_tangent_fwd_a<T, TP, QB_ACT_IDENTITY>(L, sW, R, lda, TM);
}

// delta_z = step act'(z) delta_a and its tangent step (act'(z) dda + act''(z) z_dot delta_a) of layer Lm for unit j and
// TP points, written in place over a_out / a_dot_out.  act''(z) z_dot = -2 s s_dot for tanh, 0 for relu and identity.
// Residual layers keep delta_a and dda in D / DD for the pass-through to their input.
template <typename T, int TP>
__device__ __forceinline__ void qb_hvp_finish(const QbLayerPlan& Lm, T* R, T* D, T* DD, int lda, int j, int pcol,
                                              const T (&da)[TP], const T (&dda)[TP]) {
    T* pa = R + (size_t)(Lm.row_out + j) * lda + pcol;
    T* pt = R + (size_t)(Lm.row_out - Lm.n_out_pad + j) * lda + pcol;
    T s[TP], sd[TP], dz[TP], ddz[TP];
    qb_hvp_ld<TP>(s, pa);
    qb_hvp_ld<TP>(sd, pt);
    T step = T(1);
    if (Lm.has_res) {
        T ai[TP], ti[TP];
        qb_hvp_ld<TP>(ai, R + (size_t)(Lm.row_in + j) * lda + pcol);
        qb_hvp_ld<TP>(ti, R + (size_t)(Lm.row_in - Lm.n_in_pad + j) * lda + pcol);
        step = T(Lm.res_step);
        const T inv = T(1) / step;
#pragma unroll
        for (int p = 0; p < TP; ++p) { s[p] = (s[p] - ai[p]) * inv; sd[p] = (sd[p] - ti[p]) * inv; }
        qb_hvp_st<TP>(D + (size_t)j * lda + pcol, da);
        qb_hvp_st<TP>(DD + (size_t)j * lda + pcol, dda);
    }
    const bool tanh_act = Lm.act == QB_ACT_TANH;
#pragma unroll
    for (int p = 0; p < TP; ++p) {
        const T d1 = qb_dact<T>(Lm.act, s[p]);
        const T d2 = tanh_act ? T(-2) * s[p] * sd[p] : T(0);
        dz[p] = step * d1 * da[p];
        ddz[p] = step * (d1 * dda[p] + d2 * da[p]);
    }
    qb_hvp_st<TP>(pa, dz);
    qb_hvp_st<TP>(pt, ddz);
}

// delta_a and dda of layer L's input (W^T dz, W^T dz_dot + V^T dz, plus the pass-through of residual layers), converted
// at once to delta_z and its tangent of the layer below (Lm)
template <typename T, int TP>
__device__ void qb_hvp_bwd(const QbLayerPlan& L, const QbLayerPlan& Lm, const T* sW, T* R, T* D, T* DD, int lda, int TM) {
    constexpr int TU = VT<T>::TU;
    const int UGI = L.n_in_pad / TU, PG = TM / TP, items = UGI * PG;
    const T* Wr = sW + L.wr_off;
    const T* Z = R + (size_t)L.row_out * lda;
    const T* Zt = R + (size_t)(L.row_out - L.n_out_pad) * lda;
    for (int item = threadIdx.x; item < items; item += blockDim.x) {
        int pg, ig;
        if (L.ugi_shift >= 0) { pg = item >> L.ugi_shift; ig = item & (UGI - 1); }
        else { pg = item / UGI; ig = item - pg * UGI; }
        const int pcol = pg * TP;
        T acc[TU][TP], acct[TU][TP];
        qb_gemm_accumulate<TP>(acc, Wr, (const T*)nullptr, Z + pcol, L.n_out, lda, L.n_in_pad, ig, UGI);
        qb_gemm_accumulate<TP>(acct, Wr, (const T*)nullptr, Zt + pcol, L.n_out_pad + L.n_out, lda, L.n_in_pad, ig, UGI);
#pragma unroll
        for (int u = 0; u < TU; ++u) {
            const int i = ig + UGI * u;
            if (i < L.n_in) {
                if (L.has_res) {
                    T pass[TP], passt[TP];
                    ldv<TP>(pass, D + (size_t)i * lda + pcol);
                    ldv<TP>(passt, DD + (size_t)i * lda + pcol);
#pragma unroll
                    for (int p = 0; p < TP; ++p) { acc[u][p] += pass[p]; acct[u][p] += passt[p]; }
                }
                qb_hvp_finish<T, TP>(Lm, R, D, DD, lda, i, pcol, acc[u], acct[u]);
            }
        }
    }
}

// g[0..P) = (d^2 lp_data / d theta^2) v over the points [n0, n1) (the data term only; the prior is added by the caller).
// v == NULL: v = e_unit.  g must be addressable by this block only.
template <typename T>
__device__ void qb_hvp_eval(const QbHvpPlan& H, unsigned char* smem, const T* theta, const T* v, int unit,
                            const T* __restrict__ x, const T* __restrict__ y, int64_t n0, int64_t n1, double inv_sigma2,
                            T* g) {
    constexpr int TP = 4;
    const QbPlan& P = H.P;
    T* sW = reinterpret_cast<T*>(smem);
    T* R = sW + P.w_elems;
    const int lda = P.lda, TM = P.TM, o = P.out_dim, nl = P.n_layers;
    T* D = P.d_row >= 0 ? R + (size_t)P.d_row * lda : nullptr;
    T* DD = H.dd_row >= 0 ? R + (size_t)H.dd_row * lda : nullptr;
    qb_hvp_stage<T>(P, sW, theta, v, unit);
    // every row starts finite: padding rows and the (zero) tangent of the input are read by the stacked GEMMs
    for (int idx = threadIdx.x; idx < (P.total_rows + 1) * lda; idx += blockDim.x) R[idx] = T(0);
    for (int idx = threadIdx.x; idx < P.n_params; idx += blockDim.x) g[idx] = T(0);
    __syncthreads();
    const T is2 = T(inv_sigma2);
    const QbLayerPlan& Ltop = P.L[nl - 1];
    const QbScope bsc = qb_block_scope(TM);
    for (int64_t p0 = n0; p0 < n1; p0 += TM) {
        qb_load_x_tile<T>(x, P.in_dim, p0, n1, R + (size_t)P.L[0].row_in * lda, lda, bsc);
        __syncthreads();
        for (int l = 0; l < nl; ++l) {
            const QbLayerPlan& L = P.L[l];
            qb_layer_forward<T, TP>(L, sW, R + (size_t)L.row_in * lda, R + (size_t)L.row_out * lda, lda, bsc, false);
        }
        for (int l = 0; l < nl; ++l) {
            qb_hvp_tangent_fwd<T, TP>(P.L[l], sW, R, lda, TM);
            __syncthreads();
        }
        // top: delta = d lp / d out = r / sigma^2 and its tangent (final_exp: d/du of r e^u / sigma^2)
        const T* U = R + (size_t)Ltop.row_out * lda;
        const T* Ud = R + (size_t)(Ltop.row_out - Ltop.n_out_pad) * lda;
        for (int idx = threadIdx.x; idx < TM * o; idx += blockDim.x) {
            const int j = idx / TM, p = idx - j * TM;
            const int64_t gp = p0 + p;
            T da[1] = {T(0)}, dda[1] = {T(0)};
            if (gp < n1) {
                const T u = U[(size_t)j * lda + p], ud = Ud[(size_t)j * lda + p];
                const T yv = __ldg(y + gp * o + j);
                if (P.final_exp) {
                    const T e = qb_exp(u), r = yv - e;
                    da[0] = r * e * is2;
                    dda[0] = e * ud * (r - e) * is2;
                } else {
                    da[0] = (yv - u) * is2;
                    dda[0] = -ud * is2;
                }
            }
            qb_hvp_finish<T, 1>(Ltop, R, D, DD, lda, j, p, da, dda);
        }
        __syncthreads();
        for (int l = nl - 1; l >= 0; --l) {
            qb_dw_accumulate<T>(H.LA[l], R, lda, TM, g);
            if (l > 0) qb_dw_accumulate<T>(H.LB[l], R, lda, TM, g);      // the input's tangent is zero for l == 0
            __syncthreads();
            if (l > 0) {
                qb_hvp_bwd<T, TP>(P.L[l], P.L[l - 1], sW, R, D, DD, lda, TM);
                __syncthreads();
            }
        }
    }
}
