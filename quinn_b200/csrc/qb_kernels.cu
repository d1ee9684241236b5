// quinn_b200: kernels + C ABI (include/quinn_b200.h).  Build: see quinn_b200/build.py
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <atomic>

#include "quinn_b200.h"
#include "qb_device.cuh"
#include "qb_chain.cuh"
#include "qb_nuts.cuh"
#include "qb_pt.cuh"
#include "qb_launch.h"
#include "qb_value_tc3.h"
#include "qb_grad_tc.h"
#include "qb_grad_tc128.h"

#ifndef QB_LB_T
#define QB_LB_T 256
#define QB_LB_B 2
#endif

// =================================================================================================
// error plumbing
// =================================================================================================
thread_local char g_err[512] = "";          // error text of the calling thread (qb_fail, qb_launch.cu)
static std::atomic<long long> g_launches{0};

#define QB_CUDA(call)                                                                                    \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            snprintf(g_err, sizeof(g_err), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return -2;                                                                                   \
        }                                                                                                \
    } while (0)

extern "C" const char* qb_last_error(void) { return g_err; }
// used by the other translation units of the library (qb_post.cu)
void qb_internal_set_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg); }
void qb_internal_count_launches(int n) { g_launches += n; }
extern "C" int qb_version(void) { return QB_ABI_VERSION; }
extern "C" int qb_struct_sizes(int64_t* out, int n) {
    const int64_t sz[] = {(int64_t)sizeof(qb_layer_t), (int64_t)sizeof(qb_net_t), (int64_t)sizeof(qb_lik_t), (int64_t)sizeof(qb_data_t),
                          (int64_t)sizeof(qb_chain_t), (int64_t)sizeof(qb_rng_t), (int64_t)sizeof(qb_record_t),
                          (int64_t)sizeof(qb_amcmc_t), (int64_t)sizeof(qb_hmc_t)};
    const int m = (int)(sizeof(sz) / sizeof(sz[0]));
    for (int i = 0; i < n && i < m; ++i) out[i] = sz[i];
    return m;
}
extern "C" int64_t qb_launch_count(void) { return (int64_t)g_launches.load(); }

static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

template <typename K>
static int set_smem(K kernel, long long bytes) {
    QB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

static QbLikDev lik_dev(const qb_lik_t* lik) {
    QbLikDev d;
    d.sigma = lik->sigma; d.inv_sigma2 = 1.0 / (lik->sigma * lik->sigma);
    d.prior_sigma = lik->prior_sigma; d.prior_scale = lik->prior_scale;
    d.anchor = lik->prior_anchor; d.anchor_per_chain = lik->anchor_per_chain;
    d.has_prior = lik->prior_sigma > 0.0;
    return d;
}

// =================================================================================================
// kernels 1 and 2 (stand-alone entry points)
// =================================================================================================
template <typename T>
__global__ void __launch_bounds__(512, 1) k_logpost(const __grid_constant__ QbPlan P, const EvalArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(P, smem_raw);
    const long long k = blockIdx.x, s = blockIdx.y;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    const double ssq = qb_eval_value<T>(P, S, a.theta + k * P.n_params, a.x + k * a.xs, a.y + k * a.ys, n0, n1, true);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
}

template <typename T>
__global__ void __launch_bounds__(256, 2) k_logpost_grad(const __grid_constant__ QbPlan P, const EvalArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(P, smem_raw);
    const long long k = blockIdx.x, s = blockIdx.y;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    T* g = (a.S == 1) ? a.grad + k * P.n_params : a.gpart + (k * a.S + s) * P.n_params;
    const double ssq = qb_eval_value_grad<T>(P, S, a.theta + k * P.n_params, a.x + k * a.xs, a.y + k * a.ys, n0, n1, a.lk.inv_sigma2, g);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
}


// kernels 1 and 2, layer-streamed (qb_stream.cuh): block b = chain b / S, split b % S, so the N-splits of one chain are
// neighbours in launch order and read each weight chunk from L2 after the first of them brought it from HBM
template <typename T, bool GRAD>
__global__ void __launch_bounds__(QS_THREADS, 1) k_logpost_stream(const __grid_constant__ QbStreamPlan P, const EvalArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QsRing rg;
    qs_ring_init(P, smem_raw, rg);
    const long long b = blockIdx.x, k = b / a.S, s = b - k * a.S;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    T* g = nullptr;
    if (GRAD) g = (a.S == 1) ? a.grad + k * P.n_params : a.gpart + (k * a.S + s) * P.n_params;
    const double ssq = qs_eval<T, GRAD>(P, smem_raw, rg, a.theta + k * P.n_params, a.x + k * a.xs, a.y + k * a.ys, n0, n1,
                                        a.lk.inv_sigma2, g, nullptr);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
}

// kernel 1 on the tensor cores (fp32 eligible networks, see qb_tc.cuh)
__global__ void __launch_bounds__(512, 1) k_logpost_tc(const __grid_constant__ QbTcPlan tp, const EvalArgs<float> a) {
    extern __shared__ __align__(128) unsigned char smem_tc[];
    QbTcCtx cx;
    qb_tc_init(tp, smem_tc, cx);
    const long long k = blockIdx.x, s = blockIdx.y;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    qb_tc_stage(tp, smem_tc, a.theta + k * tp.n_params);
    __syncthreads();
    const double ssq = qb_tc_eval<false>(tp, cx, smem_tc, a.x + k * a.xs, a.y + k * a.ys, n0, n1);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

template <typename T> static int launch_logpost_tc(const QbTcPlan&, const EvalArgs<T>&, dim3, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_logpost_tc<float>(const QbTcPlan& tp, const EvalArgs<float>& a, dim3 grid, cudaStream_t st) {
    if (tp.v3) {                  // hot shape: warp-specialised kernel (qb_value_tc3.cu)
        QB_CUDA(qb_tc3_launch_logpost(tp, a, grid, st));
    } else {
        if (set_smem(k_logpost_tc, tp.smem_bytes)) return -2;
        k_logpost_tc<<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, a);
    }
    return 0;
}

// kernel 2 on the tensor cores (qb_grad_tc.cu)
template <typename T> static int launch_grad_tc(const QbTcgPlan&, const EvalArgs<T>&, dim3, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_grad_tc<float>(const QbTcgPlan& tg, const EvalArgs<float>& a, dim3 grid, cudaStream_t st) {
    QB_CUDA(qb_tcg_launch_eval(tg, a, grid, st));
    return 0;
}
// kernel 2 on the tensor cores, 128-wide nets (qb_grad_tc128.cu)
template <typename T> static int launch_grad_tc128(const QbTg8Plan&, const EvalArgs<T>&, void*, dim3, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_grad_tc128<float>(const QbTg8Plan& tg, const EvalArgs<float>& a, void* scratch, dim3 grid, cudaStream_t st) {
    QB_CUDA(qb_tg8_launch_eval(tg, a, scratch, grid, st));
    return 0;
}
template <typename T> static int launch_hmc_tc128(const QbTg8Plan&, const ChainArgs<T>&, const HmcArgs<T>&, long long, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_hmc_tc128<float>(const QbTg8Plan& tg, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st) {
    QB_CUDA(qb_tg8_launch_hmc(tg, c, h, K, st));
    return 0;
}
template <typename T> static int launch_hmc_tc(const QbTcgPlan&, const ChainArgs<T>&, const HmcArgs<T>&, long long, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_hmc_tc<float>(const QbTcgPlan& tg, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st) {
    QB_CUDA(qb_tcg_launch_hmc(tg, c, h, K, st));
    return 0;
}
template <typename T> static int launch_nuts_tc128(const QbTg8Plan&, const ChainArgs<T>&, const NutsArgs<T>&, long long, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_nuts_tc128<float>(const QbTg8Plan& tg, const ChainArgs<float>& c, const NutsArgs<float>& a, long long K, cudaStream_t st) {
    QB_CUDA(qb_tg8_launch_nuts(tg, c, a, K, st));
    return 0;
}
template <typename T> static int launch_nuts_tc(const QbTcgPlan&, const ChainArgs<T>&, const NutsArgs<T>&, long long, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_nuts_tc<float>(const QbTcgPlan& tg, const ChainArgs<float>& c, const NutsArgs<float>& a, long long K, cudaStream_t st) {
    QB_CUDA(qb_tcg_launch_nuts(tg, c, a, K, st));
    return 0;
}

// gradient rows of the N-splits added in fixed order, one thread per element (k_finalize alone, one block per chain, is
// latency-bound on this: 224 us for 256 x 5 x 18049 floats; this kernel moves them at memory speed)
template <typename T>
__global__ void __launch_bounds__(256) k_sum_gparts(const EvalArgs<T> a, int P) {
    const long long k = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const T* src = a.gpart + k * a.S * (long long)P + i;
    T v = T(0);
    for (int s = 0; s < a.S; ++s) v += src[(long long)s * P];
    a.grad[k * P + i] = v;
}

// combine the N-splits (fixed order), add constants and the prior; want_grad == 2: the gradient rows are already summed
template <typename T>
__global__ void __launch_bounds__(128) k_finalize(const EvalArgs<T> a, int P, int want_grad) {
    __shared__ double red[40];
    const long long k = blockIdx.x;
    double ssq = 0.0;
    for (int s = 0; s < a.S; ++s) ssq += a.part[k * a.S + s];
    const T* th = a.theta + k * P;
    double pss = 0.0;
    if (a.lk.has_prior) pss = qb_prior_ss<T>(a.lk, th, k, P, red);
    if (threadIdx.x == 0) a.lp[k] = qb_lp_from(a.lk, ssq, a.N, pss, P);
    if (want_grad) {
        T* g = a.grad + k * P;
        if (a.S > 1 && want_grad != 2) {
            for (int i = threadIdx.x; i < P; i += blockDim.x) {
                T v = T(0);
                for (int s = 0; s < a.S; ++s) v += a.gpart[(k * a.S + s) * P + i];
                g[i] = v;
            }
            __syncthreads();
        }
        qb_prior_grad_add<T>(a.lk, th, k, P, g);
    }
}

template <typename T>
static int run_eval(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
                    const qb_lik_t* lik, double* lp, void* grad, void* ws, size_t ws_bytes, cudaStream_t st,
                    int64_t x_stride = 0, int64_t y_stride = 0) {
    const bool want_grad = grad != nullptr;
    QbLaunch L;
    if (plan_eval(net, dtype, want_grad, K, data->n, false, &L)) return -1;
    if (ws_bytes < L.ws_bytes || (L.ws_bytes && !ws)) return qb_fail("workspace too small%s (need %lld bytes)", "", (long long)L.ws_bytes);
    EvalArgs<T> a;
    a.theta = (const T*)theta; a.x = (const T*)data->x; a.y = (const T*)data->y;
    a.xs = x_stride; a.ys = y_stride;
    a.K = K; a.N = data->n; a.S = L.S; a.pps = L.pts_per_split;
    a.part = (double*)ws;
    a.grad = (T*)grad;
    a.gpart = (L.S > 1 && want_grad) ? (T*)((char*)ws + L.gpart_off) : nullptr;
    a.lp = lp; a.lk = lik_dev(lik);
    a.xsplit = nullptr;
    dim3 grid((unsigned)K, (unsigned)L.S);
    if (L.path == QB_PATH_STREAM) {
        const dim3 sgrid((unsigned)(K * L.S));
        if (want_grad) {
            if (set_smem(k_logpost_stream<T, true>, L.sp.smem_bytes)) return -2;
            k_logpost_stream<T, true><<<sgrid, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, a);
        } else {
            if (set_smem(k_logpost_stream<T, false>, L.sp.smem_bytes)) return -2;
            k_logpost_stream<T, false><<<sgrid, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, a);
        }
    } else if (L.path == QB_PATH_TG8) {
        // tanh nets of width 64 / 128: fp16-split operands, scaled with max |x|, max |y| (the workspace's tail scratch)
        if (launch_grad_tc128<T>(L.t8, a, (char*)ws + L.tail_off, grid, st)) return -2;
        g_launches += 1;
    } else if (L.path == QB_PATH_TCG) {
        if (launch_grad_tc<T>(L.tg, a, grid, st)) return -2;
    } else if (L.path != QB_PATH_CUDA) {
        // hot shape with shared data: x goes to the kernel as ready-made operand tiles in the workspace's tail scratch
        if (L.tp.v3 && x_stride == 0) a.xsplit = (const T*)((char*)ws + L.tail_off);
        if (launch_logpost_tc<T>(L.tp, a, grid, st)) return -2;
    } else if (want_grad) {
        if (set_smem(k_logpost_grad<T>, L.plan.smem_bytes)) return -2;
        k_logpost_grad<T><<<grid, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, a);
    } else {
        if (set_smem(k_logpost<T>, L.plan.smem_bytes)) return -2;
        k_logpost<T><<<grid, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, a);
    }
    QB_CUDA(cudaGetLastError());
    int fin_mode = want_grad ? 1 : 0;
    if (want_grad && L.S > 1 && K <= 65535) {
        k_sum_gparts<T><<<dim3((unsigned)cdiv(net->n_params, 256), (unsigned)K), 256, 0, st>>>(a, net->n_params);
        QB_CUDA(cudaGetLastError());
        fin_mode = 2;
        g_launches += 1;
    }
    k_finalize<T><<<(unsigned)K, 128, 0, st>>>(a, net->n_params, fin_mode);
    QB_CUDA(cudaGetLastError());
    g_launches += 2;
    return 0;
}

extern "C" int qb_logpost(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
                          const qb_lik_t* lik, double* lp, void* ws, size_t ws_bytes, void* stream) {
    if (!theta || !data || !lik || !lp) return qb_fail("NULL argument to qb_logpost");
    if (dtype == QB_F64) return run_eval<double>(net, dtype, theta, K, data, lik, lp, nullptr, ws, ws_bytes, (cudaStream_t)stream);
    return run_eval<float>(net, dtype, theta, K, data, lik, lp, nullptr, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int qb_logpost_grad(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
                               const qb_lik_t* lik, double* lp, void* grad, void* ws, size_t ws_bytes, void* stream) {
    if (!theta || !data || !lik || !lp || !grad) return qb_fail("NULL argument to qb_logpost_grad");
    if (dtype == QB_F64) return run_eval<double>(net, dtype, theta, K, data, lik, lp, grad, ws, ws_bytes, (cudaStream_t)stream);
    return run_eval<float>(net, dtype, theta, K, data, lik, lp, grad, ws, ws_bytes, (cudaStream_t)stream);
}

/* Kernels 1 / 2 with per-member data (batched ensemble training: every member sees its own subset / minibatch). */
extern "C" int qb_logpost_members(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
                                  int64_t x_stride, int64_t y_stride, const qb_lik_t* lik, double* lp, void* grad,
                                  void* ws, size_t ws_bytes, void* stream) {
    if (!theta || !data || !lik || !lp) return qb_fail("NULL argument to qb_logpost_members");
    if (x_stride < 0 || y_stride < 0) return qb_fail("negative data stride");
    if (dtype == QB_F64) return run_eval<double>(net, dtype, theta, K, data, lik, lp, grad, ws, ws_bytes, (cudaStream_t)stream, x_stride, y_stride);
    return run_eval<float>(net, dtype, theta, K, data, lik, lp, grad, ws, ws_bytes, (cudaStream_t)stream, x_stride, y_stride);
}

// =================================================================================================
// kernel 5: Hessian-vector products (qb_hvp.cuh)
// =================================================================================================
template <typename T> struct HvpArgs {
    const T* theta; const T* v; long long col0;
    const T* x; const T* y;
    long long N; int S; long long pps;
    T* hv;          // [K,P]
    T* gpart;       // [K,S,P] (S > 1)
    double inv_sigma2, prior_c;      // prior_c = prior_scale / prior_sigma^2, or 0
};

template <typename T>
__global__ void __launch_bounds__(256, 1) k_logpost_hvp(const __grid_constant__ QbHvpPlan H, const HvpArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const long long k = blockIdx.x, s = blockIdx.y;
    const int P = H.P.n_params;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    T* g = (a.S == 1) ? a.hv + k * P : a.gpart + (k * a.S + s) * P;
    qb_hvp_eval<T>(H, smem_raw, a.theta, a.v ? a.v + k * P : nullptr, (int)(a.col0 + k), a.x, a.y, n0, n1, a.inv_sigma2, g);
}

// hv[k,:] = sum of the N-split rows in fixed order - prior_c * v_k
template <typename T>
__global__ void __launch_bounds__(256) k_hvp_finalize(const HvpArgs<T> a, long long K, int P) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= K * P) return;
    const long long k = e / P;
    const int i = (int)(e - k * P);
    T h;
    if (a.S > 1) {
        const T* src = a.gpart + k * a.S * (long long)P + i;
        h = T(0);
        for (int s = 0; s < a.S; ++s) h += src[(long long)s * P];
    } else {
        h = a.hv[e];
    }
    if (a.prior_c != 0.0) {
        const double vi = a.v ? (double)a.v[e] : (i == a.col0 + k ? 1.0 : 0.0);
        h = (T)((double)h - a.prior_c * vi);
    }
    a.hv[e] = h;
}

template <typename T>
static int run_hvp(const qb_net_t* net, int dtype, const void* theta, const void* v, int64_t col0, int64_t K,
                   const qb_data_t* data, const qb_lik_t* lik, void* hv, void* ws, size_t ws_bytes, cudaStream_t st) {
    QbHvpLaunch L;
    if (make_hvp_launch(net, dtype, K, data->n, &L)) return -1;
    if (ws_bytes < L.ws_bytes || (L.ws_bytes && !ws)) return qb_fail("workspace too small%s (need %lld bytes)", "", (long long)L.ws_bytes);
    HvpArgs<T> a;
    a.theta = (const T*)theta; a.v = (const T*)v; a.col0 = col0;
    a.x = (const T*)data->x; a.y = (const T*)data->y;
    a.N = data->n; a.S = L.S; a.pps = L.pps;
    a.hv = (T*)hv; a.gpart = L.S > 1 ? (T*)ws : nullptr;
    a.inv_sigma2 = 1.0 / (lik->sigma * lik->sigma);
    a.prior_c = lik->prior_sigma > 0.0 ? lik->prior_scale / (lik->prior_sigma * lik->prior_sigma) : 0.0;
    if (set_smem(k_logpost_hvp<T>, L.H.P.smem_bytes)) return -2;
    k_logpost_hvp<T><<<dim3((unsigned)K, (unsigned)L.S), L.H.P.nthreads, L.H.P.smem_bytes, st>>>(L.H, a);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    if (L.S > 1 || a.prior_c != 0.0) {
        const long long n = K * (long long)net->n_params;
        k_hvp_finalize<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>(a, K, net->n_params);
        QB_CUDA(cudaGetLastError());
        g_launches += 1;
    }
    return 0;
}

extern "C" int qb_logpost_hvp(const qb_net_t* net, int dtype, const void* theta, const void* v, int64_t col0, int64_t K,
                              const qb_data_t* data, const qb_lik_t* lik, void* hv, void* ws, size_t ws_bytes, void* stream) {
    if (!theta || !data || !lik || (K > 0 && !hv)) return qb_fail("NULL argument to qb_logpost_hvp");
    if (K < 0) return qb_fail("K must not be negative");
    if (lik->anchor_per_chain) return qb_fail("qb_logpost_hvp evaluates one theta: anchor_per_chain must be 0");
    if (!net) return qb_fail("net is NULL");
    if (!v && (col0 < 0 || col0 + K > net->n_params)) return qb_fail("unit directions col0 .. col0+K-1 out of range");
    if (K == 0) return 0;
    if (dtype == QB_F64) return run_hvp<double>(net, dtype, theta, v, col0, K, data, lik, hv, ws, ws_bytes, (cudaStream_t)stream);
    return run_hvp<float>(net, dtype, theta, v, col0, K, data, lik, hv, ws, ws_bytes, (cudaStream_t)stream);
}

// =================================================================================================
// kernel 6: Kronecker factors of the per-point empirical Fisher (qb_kfac.cuh)
// =================================================================================================
template <typename T> struct KfacArgs {
    const T* theta; const T* x; const T* y;
    long long N; int S; long long pps;
    T* part;            // [S, F]
    double* factors;    // [F]
    double inv_sigma2;
};

// fp32: one block per SM in the register budget (163 registers; at two, 128 registers spill the fp32 factor passes)
template <typename T>
__global__ void __launch_bounds__(256, sizeof(T) == 8 ? 2 : 1) k_logpost_kfac(const __grid_constant__ QbKfacPlan K, const KfacArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(K.P, smem_raw);
    const long long s = blockIdx.x;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    QbKfacHooks<T> h{{K.P, a.y, n1, a.inv_sigma2, a.part + s * K.n_factors}, K};
    qb_backprop_tiles<T>(K.P, S, a.theta, a.x, n0, n1, h);
}

// factors[e] = sum of the N-split rows in fixed order, in double
template <typename T>
__global__ void __launch_bounds__(256) k_kfac_finalize(const KfacArgs<T> a, int F) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= F) return;
    double v = 0.0;
    for (int s = 0; s < a.S; ++s) v += (double)a.part[(long long)s * F + e];
    a.factors[e] = v;
}

template <typename T>
static int run_kfac(const qb_net_t* net, int dtype, const void* theta, const qb_data_t* data, const qb_lik_t* lik,
                    double* factors, void* ws, size_t ws_bytes, cudaStream_t st) {
    QbKfacLaunch L;
    if (make_kfac_launch(net, dtype, std::max<int64_t>(data->n, 1), &L)) return -1;
    if (data->n == 0) {               // no points: zero factors, no kernel
        QB_CUDA(cudaMemsetAsync(factors, 0, (size_t)L.K.n_factors * sizeof(double), st));
        return 0;
    }
    if (ws_bytes < L.ws_bytes || !ws) return qb_fail("workspace too small%s (need %lld bytes)", "", (long long)L.ws_bytes);
    KfacArgs<T> a;
    a.theta = (const T*)theta; a.x = (const T*)data->x; a.y = (const T*)data->y;
    a.N = data->n; a.S = L.S; a.pps = L.pps;
    a.part = (T*)ws; a.factors = factors;
    a.inv_sigma2 = 1.0 / (lik->sigma * lik->sigma);
    if (set_smem(k_logpost_kfac<T>, L.K.P.smem_bytes)) return -2;
    k_logpost_kfac<T><<<(unsigned)L.S, L.K.P.nthreads, L.K.P.smem_bytes, st>>>(L.K, a);
    QB_CUDA(cudaGetLastError());
    k_kfac_finalize<T><<<(unsigned)cdiv(L.K.n_factors, 256), 256, 0, st>>>(a, L.K.n_factors);
    QB_CUDA(cudaGetLastError());
    g_launches += 2;
    return 0;
}

extern "C" int qb_logpost_kfac(const qb_net_t* net, int dtype, const void* theta, const qb_data_t* data,
                               const qb_lik_t* lik, double* factors, void* ws, size_t ws_bytes, void* stream) {
    if (!theta || !data || !lik || !factors) return qb_fail("NULL argument to qb_logpost_kfac");
    if (data->n < 0) return qb_fail("N must not be negative");
    if (lik->anchor_per_chain) return qb_fail("qb_logpost_kfac evaluates one theta: anchor_per_chain must be 0");
    if (dtype == QB_F64) return run_kfac<double>(net, dtype, theta, data, lik, factors, ws, ws_bytes, (cudaStream_t)stream);
    return run_kfac<float>(net, dtype, theta, data, lik, factors, ws, ws_bytes, (cudaStream_t)stream);
}

// =================================================================================================
// kernel 7: per-point output Jacobians as per-layer pairs (qb_jac.cuh)
// =================================================================================================
template <typename T> struct JacArgs {
    const T* theta; const T* x;
    long long N; long long pps;
    T* out;             // [N, o]
    T* fac;             // [F, N]
};

template <typename T>
__global__ void __launch_bounds__(256, 2) k_predict_jac(const __grid_constant__ QbJacPlan J, const JacArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(J.P, smem_raw);
    const long long s = blockIdx.x;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    QbJacHooks<T> h{J, a.N, a.out, a.fac};
    qb_backprop_tiles<T>(J.P, S, a.theta, a.x, n0, n1, h);
}

template <typename T>
static int run_jac(const qb_net_t* net, int dtype, const void* theta, const void* x, int64_t N, void* out, void* fac,
                   cudaStream_t st) {
    QbJacLaunch L;
    if (make_jac_launch(net, dtype, std::max<int64_t>(N, 1), &L)) return -1;
    if (N == 0) return 0;             // no points: no kernel
    JacArgs<T> a;
    a.theta = (const T*)theta; a.x = (const T*)x;
    a.N = N; a.pps = L.pps;
    a.out = (T*)out; a.fac = (T*)fac;
    if (set_smem(k_predict_jac<T>, L.J.P.smem_bytes)) return -2;
    k_predict_jac<T><<<(unsigned)L.S, L.J.P.nthreads, L.J.P.smem_bytes, st>>>(L.J, a);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

extern "C" int qb_predict_jac(const qb_net_t* net, int dtype, const void* theta, const void* x, int64_t N, void* out,
                              void* fac, void* stream) {
    if (!theta || (N > 0 && (!x || !out || !fac))) return qb_fail("NULL argument to qb_predict_jac");
    if (N < 0) return qb_fail("N must not be negative");
    if (dtype == QB_F64) return run_jac<double>(net, dtype, theta, x, N, out, fac, (cudaStream_t)stream);
    return run_jac<float>(net, dtype, theta, x, N, out, fac, (cudaStream_t)stream);
}

// Adam (torch.optim.Adam semantics, quinn/nns/nnfit.py:92-93) on a flat array: g = grad*grad_scale + wd*theta
template <typename T>
__global__ void k_adam(T* th, const T* g, T* m, T* v, long long n, double lr, double b1, double b2, double eps, double wd,
                       double bc1, double bc2s, double gscale) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double t = (double)th[i];
    const double gi = (double)g[i] * gscale + wd * t;
    const double mi = b1 * (double)m[i] + (1.0 - b1) * gi;
    const double vi = b2 * (double)v[i] + (1.0 - b2) * gi * gi;
    m[i] = (T)mi; v[i] = (T)vi;
    th[i] = (T)(t - (lr / bc1) * mi / (sqrt(vi) / bc2s + eps));
}
extern "C" int qb_adam_step(int dtype, void* theta, const void* grad, void* m, void* v, int64_t n, double lr, double beta1,
                            double beta2, double eps, double wd, int64_t step, double grad_scale, void* stream) {
    if (!theta || !grad || !m || !v || n < 1 || step < 1) return qb_fail("bad argument to qb_adam_step");
    const double bc1 = 1.0 - pow(beta1, (double)step), bc2s = sqrt(1.0 - pow(beta2, (double)step));
    const unsigned blocks = (unsigned)cdiv(n, 256);
    if (dtype == QB_F64) k_adam<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((double*)theta, (const double*)grad, (double*)m, (double*)v, n, lr, beta1, beta2, eps, wd, bc1, bc2s, grad_scale);
    else k_adam<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((float*)theta, (const float*)grad, (float*)m, (float*)v, n, lr, beta1, beta2, eps, wd, bc1, bc2s, grad_scale);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

// best-model tracking: dst[k,:] = src[k,:] where mask[k] != 0
template <typename T>
__global__ void k_copy_rows_where(T* dst, const T* src, const unsigned char* mask, long long P) {
    const long long k = blockIdx.x;          // rows on grid.x (2^31-1 blocks): K is not limited to 65535
    if (!mask[k]) return;
    const long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x;
    if (i < P) dst[k * P + i] = src[k * P + i];
}
extern "C" int qb_copy_rows_where(int dtype, void* dst, const void* src, const unsigned char* mask, int64_t K, int64_t P,
                                  void* stream) {
    if (!dst || !src || !mask || K < 1 || P < 1 || cdiv(P, 256) > 65535) return qb_fail("bad argument to qb_copy_rows_where");
    dim3 grid((unsigned)K, (unsigned)cdiv(P, 256));
    if (dtype == QB_F64) k_copy_rows_where<double><<<grid, 256, 0, (cudaStream_t)stream>>>((double*)dst, (const double*)src, mask, P);
    else k_copy_rows_where<float><<<grid, 256, 0, (cudaStream_t)stream>>>((float*)dst, (const float*)src, mask, P);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

// =================================================================================================
// kernel 3: fused chain steps
// =================================================================================================
// in-block Cholesky of fac*(cov + jitter*I) -> lower factor Lf (global, [P,P])
template <typename T>
__device__ void qb_cholesky(const T* cov, T* Lf, int P, double fac, double jitter) {
    for (int idx = threadIdx.x; idx < P * P; idx += blockDim.x) Lf[idx] = T(0);
    __syncthreads();
    for (int j = 0; j < P; ++j) {
        for (int i = j + threadIdx.x; i < P; i += blockDim.x) {
            double s = fac * ((double)cov[i * P + j] + (i == j ? jitter : 0.0));
            for (int q = 0; q < j; ++q) s -= (double)Lf[i * P + q] * (double)Lf[j * P + q];
            Lf[i * P + j] = (T)s;
        }
        __syncthreads();
        // In exact arithmetic the pivot is >= fac*jitter (the matrix is PSD + jitter*I); in floating point a rank-deficient
        // covariance (fewer samples than parameters at the first adaptation) can round it to <= 0.  Such a direction has no
        // variance beyond the jitter: clamp the pivot and zero the column instead of producing NaN proposals.
        const double piv = (double)Lf[j * P + j], floor_ = fac * jitter;
        const bool ok = piv > floor_;              // false for NaN too
        const double d = sqrt(ok ? piv : floor_);
        __syncthreads();
        for (int i = j + threadIdx.x; i < P; i += blockDim.x)
            Lf[i * P + j] = (i == j) ? (T)d : (ok ? (T)((double)Lf[i * P + j] / d) : T(0));
        __syncthreads();
    }
}

// per-chain scalars that live across the evaluation (kept in a struct so that the cold step logic can be compiled
// out of line for the tensor-core kernel, whose hot loop needs every register)
struct QbAmcmcLocal { double lp_cur, map_lp; long long na; int kind; };

// one AMCMC step up to the proposal (admcmc.py:52-70): moments, proposal covariance, proposal -> a.prop
template <typename T>
__device__ __forceinline__ void qb_amcmc_pre(const ChainArgs<T>& c, const AmcmcArgs<T>& a, int P, long long k, long long s,
                                             int& kind, T* zbuf) {
    const int tid = threadIdx.x, nt = blockDim.x;
    T* cur = c.theta + k * P;
    T* prop = a.prop + k * P;
    T* xm = a.xm ? a.xm + k * P : nullptr;
    T* pscale = a.pscale + k * P;
    const bool full = a.track == 2;               // shape of cov: [P,P] (2) or [P] (1)
    T* cov = a.cov ? a.cov + k * (full ? (long long)P * P : (long long)P) : nullptr;
    T* chol = a.chol ? a.chol + k * (long long)P * P : nullptr;
    const long long t = c.t_start + s;
        // ---- running mean / covariance (admcmc.py:52-59)
        if (a.track && xm) {
            if (t == 0) {
                for (int i = tid; i < P; i += nt) xm[i] = cur[i];
                if (cov) { const long long n = full ? (long long)P * P : P; for (long long i = tid; i < n; i += nt) cov[i] = T(0); }
            } else {
                const double td = (double)t;
                const T rt = (T)((td - 1.0) / td), st = (T)((td + 1.0) / (td * td));
                for (int i = tid; i < P; i += nt)
                    xm[i] = qb_add<T>(qb_mul<T>((T)td, xm[i]), cur[i]) / (T)(td + 1.0);
                __syncthreads();
                if (cov && full) {
                    for (int idx = tid; idx < P * P; idx += nt) {
                        const int r = idx / P, q = idx - r * P;
                        const T dr = cur[r] - xm[r], dq = cur[q] - xm[q];
                        cov[idx] = qb_add<T>(qb_mul<T>(rt, cov[idx]), qb_mul<T>(st, qb_mul<T>(dr, dq)));
                    }
                } else if (cov) {
                    for (int i = tid; i < P; i += nt) {
                        const T d = cur[i] - xm[i];
                        cov[i] = qb_add<T>(qb_mul<T>(rt, cov[i]), qb_mul<T>(st, qb_mul<T>(d, d)));
                    }
                }
            }
            __syncthreads();
        }
        // ---- proposal covariance (admcmc.py:61-67)
        if (t == 0) {
            if (a.chol_ini) kind = 3;
            else {
                kind = 0;
                for (int i = tid; i < P; i += nt) pscale[i] = (T)sqrt(0.09 * fabs((double)cur[i]));
            }
            __syncthreads();
        } else if (a.adapt != QB_ADAPT_NONE && t > a.t0 && (t % a.tadapt) == 0) {
            const double fac = a.gamma * 2.4 * 2.4 / (double)P;
            if (full) { qb_cholesky<T>(cov, chol, P, fac, 1e-8); kind = 2; }
            else {
                for (int i = tid; i < P; i += nt) pscale[i] = (T)sqrt(fac * ((double)cov[i] + 1e-8));
                kind = 1;
            }
            __syncthreads();
        }
        // ---- proposal (admcmc.py:70)
        if (c.rng_mode == QB_RNG_REPLAY) {
            const T* xi = c.incr + (s * c.K + k) * P;
            for (int i = tid; i < P; i += nt) prop[i] = qb_add<T>(cur[i], xi[i]);
        } else {
            const long long chain = c.chain_offset + k;
            if (kind == 0 || kind == 1) {
                T z0 = T(0);
                if (kind == 0) { T zz[4]; qb_normal4(qb_rand4(c.seed, chain, t, QB_STREAM_Z0, 0), zz); z0 = T(0.1) * zz[0]; }
                for (int i4 = tid; i4 * 4 < P; i4 += nt) {
                    T z[4];
                    qb_normal4(qb_rand4(c.seed, chain, t, QB_STREAM_INCR, (uint32_t)i4), z);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < P) prop[i] = cur[i] + (z0 + pscale[i] * z[q]);
                    }
                }
            } else {
                for (int i4 = tid; i4 * 4 < P; i4 += nt) {
                    T z[4];
                    qb_normal4(qb_rand4(c.seed, chain, t, QB_STREAM_INCR, (uint32_t)i4), z);
#pragma unroll
                    for (int q = 0; q < 4; ++q) if (i4 * 4 + q < P) zbuf[i4 * 4 + q] = z[q];
                }
                __syncthreads();
                const T* Lf = (kind == 3) ? a.chol_ini : chol;
                for (int i = tid; i < P; i += nt) {
                    T acc = T(0);
                    for (int q = 0; q <= i; ++q) acc = fma(Lf[(long long)i * P + q], zbuf[q], acc);
                    prop[i] = cur[i] + acc;
                }
            }
        }
    __syncthreads();
}
template <typename T>
__device__ __noinline__ void qb_amcmc_pre_cold(const ChainArgs<T>& c, const AmcmcArgs<T>& a, int P, long long k, long long s,
                                               int& kind, T* zbuf) {
    qb_amcmc_pre<T>(c, a, P, k, s, kind, zbuf);
}

// accept / reject and bookkeeping after the evaluation (mcmc.py:55-61 for the initial state, 69-85 per step)
template <typename T>
__device__ __forceinline__ void qb_amcmc_post(const ChainArgs<T>& c, const AmcmcArgs<T>& a, int P, long long k, long long s,
                                              double ssq, double* red, QbAmcmcLocal& st) {
    T* cur = c.theta + k * P;
    T* prop = a.prop + k * P;
    T* mapth = c.map_theta + k * P;
    double pss = 0.0;
    if (c.lk.has_prior) pss = qb_prior_ss<T>(c.lk, s < 0 ? cur : prop, k, P, red);
    const double lp_prop = qb_lp_from(c.lk, ssq, c.N, pss, P);
    if (s < 0) {
        st.lp_cur = lp_prop; st.map_lp = lp_prop; st.na = 0;
        if (threadIdx.x == 0 && c.rec_lp0) c.rec_lp0[k] = lp_prop;
        for (int i = threadIdx.x; i < P; i += blockDim.x) mapth[i] = cur[i];
    } else {
        qb_mh_step<T>(c, k, s, P, lp_prop, 0.0, 0.0, cur, prop, mapth, st.lp_cur, st.map_lp, st.na);
    }
    __syncthreads();
}
template <typename T>
__device__ __noinline__ void qb_amcmc_post_cold(const ChainArgs<T>& c, const AmcmcArgs<T>& a, int P, long long k, long long s,
                                                double ssq, double* red, QbAmcmcLocal& st) {
    qb_amcmc_post<T>(c, a, P, k, s, ssq, red, st);
}

// TC = 2 (fp32 only): the evaluation runs on the tensor cores (qb_tc.cuh); the config-5 shape has its own kernel
// (qb_value_tc3.cu).
template <typename T, int TC>
__global__ void __launch_bounds__(512, 1)
k_amcmc(const __grid_constant__ QbPlan plan, const __grid_constant__ QbTcPlan tp, const __grid_constant__ ChainArgs<T> c,
        const __grid_constant__ AmcmcArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QbSmem S;
    QbTcCtx cx;
    if constexpr (TC) {
        S.red = reinterpret_cast<double*>(smem_raw); S.w = nullptr;
        S.act = smem_raw + tp.fl_base;       // never used as scratch: full-covariance proposals take the SIMT kernel
        qb_tc_init(tp, smem_raw, cx);
    } else {
        S = qb_carve<T>(plan, smem_raw);
    }
    const long long k = blockIdx.x;
    const int P = plan.n_params;
    T* zbuf = reinterpret_cast<T*>(S.act);       // scratch between evaluations

    // One evaluation call site: step s == -1 (only when init_lp) evaluates the incoming state itself
    // (mcmc.py:55-56) and initialises the MAP bookkeeping.
    QbAmcmcLocal st;
    st.lp_cur = 0.0; st.map_lp = 0.0; st.na = 0;
    if (!c.init_lp) { st.lp_cur = c.lp[k]; st.map_lp = c.map_lp[k]; st.na = c.naccept[k]; }
    st.kind = a.prop_kind[k];
    __syncthreads();

    for (long long s = c.init_lp ? -1 : 0; s < c.nsteps; ++s) {
        const T* evalp = (s < 0 ? c.theta : a.prop) + k * P;
        if (s >= 0) {
            if constexpr (TC) qb_amcmc_pre_cold<T>(c, a, P, k, s, st.kind, zbuf);
            else qb_amcmc_pre<T>(c, a, P, k, s, st.kind, zbuf);
        } else {
            __syncthreads();
        }
        // ---- evaluate + accept
        double ssq;
        if constexpr (TC == 2) {
            qb_tc_stage(tp, smem_raw, evalp);
            __syncthreads();
            ssq = qb_tc_eval<false>(tp, cx, smem_raw, c.x, c.y, 0, c.N);
        } else {
            ssq = qb_eval_value<T>(plan, S, evalp, c.x, c.y, 0, c.N, true);
        }
        if constexpr (TC) qb_amcmc_post_cold<T>(c, a, P, k, s, ssq, S.red, st);
        else qb_amcmc_post<T>(c, a, P, k, s, ssq, S.red, st);
    }
    if (threadIdx.x == 0) { c.lp[k] = st.lp_cur; c.map_lp[k] = st.map_lp; c.naccept[k] = st.na; a.prop_kind[k] = st.kind; }
    if constexpr (TC) qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

// kernel 3 (AMCMC), layer-streamed: one block per chain, the proposal pass uses the activation area as scratch
template <typename T>
__global__ void __launch_bounds__(QS_THREADS, 1)
k_amcmc_stream(const __grid_constant__ QbStreamPlan P, const __grid_constant__ ChainArgs<T> c, const __grid_constant__ AmcmcArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QsRing rg;
    qs_ring_init(P, smem_raw, rg);
    double* red = reinterpret_cast<double*>(smem_raw);
    T* zbuf = reinterpret_cast<T*>(smem_raw + P.act_off);
    const long long k = blockIdx.x;
    const int np = P.n_params;
    QbAmcmcLocal st;
    st.lp_cur = 0.0; st.map_lp = 0.0; st.na = 0;
    if (!c.init_lp) { st.lp_cur = c.lp[k]; st.map_lp = c.map_lp[k]; st.na = c.naccept[k]; }
    st.kind = a.prop_kind[k];
    __syncthreads();
    for (long long s = c.init_lp ? -1 : 0; s < c.nsteps; ++s) {
        const T* evalp = (s < 0 ? c.theta : a.prop) + k * np;
        if (s >= 0) qb_amcmc_pre<T>(c, a, np, k, s, st.kind, zbuf);
        else __syncthreads();
        const double ssq = qs_eval<T, false>(P, smem_raw, rg, evalp, c.x, c.y, 0, c.N, 0.0, nullptr, nullptr);
        qb_amcmc_post<T>(c, a, np, k, s, ssq, red, st);
    }
    if (threadIdx.x == 0) { c.lp[k] = st.lp_cur; c.map_lp[k] = st.map_lp; c.naccept[k] = st.na; a.prop_kind[k] = st.kind; }
}

template <typename T> static int launch_amcmc_tc(const QbPlan&, const QbTcPlan&, const ChainArgs<T>&, const AmcmcArgs<T>&, long long, cudaStream_t) {
    return qb_fail("tensor-core path is fp32 only");
}
template <> int launch_amcmc_tc<float>(const QbPlan& plan, const QbTcPlan& tp, const ChainArgs<float>& c, const AmcmcArgs<float>& a,
                                       long long K, cudaStream_t st) {
    if (tp.v3) {                  // hot shape: warp-specialised kernel with the chain state in shared memory (qb_value_tc3.cu)
        QB_CUDA(qb_tc3_launch_amcmc(tp, c, a, K, st));
    } else {
        if (set_smem(k_amcmc<float, 2>, tp.smem_bytes)) return -2;
        k_amcmc<float, 2><<<(unsigned)K, tp.nthreads, tp.smem_bytes, st>>>(plan, tp, c, a);
    }
    return 0;
}

template <typename T> struct QbGradSimt {
    const QbPlan& plan; const QbSmem& S; const ChainArgs<T>& c; long long k;
    __device__ __forceinline__ double operator()(const T* th, T* g) const {
        double lp;
        qb_full_grad<T>(plan, S, c, k, th, g, &lp);
        return lp;
    }
};

template <typename T>
__global__ void __launch_bounds__(256, 2) k_hmc(const __grid_constant__ QbPlan plan, const ChainArgs<T> c, const HmcArgs<T> h) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(plan, smem_raw);
    QbGradSimt<T> eval{plan, S, c, (long long)blockIdx.x};
    qb_hmc_body<T>(c, h, plan.n_params, S.red, eval);
}

// HMC / MALA, layer-streamed: the evaluation functor of qb_hmc_body (value + gradient + prior, as qb_full_grad)
template <typename T> struct QbGradStream {
    const QbStreamPlan& P; unsigned char* smem; QsRing& rg; const ChainArgs<T>& c; long long k;
    __device__ __forceinline__ double operator()(const T* th, T* g) const {
        const double ssq = qs_eval<T, true>(P, smem, rg, th, c.x, c.y, 0, c.N, c.lk.inv_sigma2, g, nullptr);
        double* red = reinterpret_cast<double*>(smem);
        double pss = 0.0;
        if (c.lk.has_prior) {
            pss = qb_prior_ss<T>(c.lk, th, k, P.n_params, red);
            qb_prior_grad_add<T>(c.lk, th, k, P.n_params, g);
        }
        __syncthreads();
        return qb_lp_from(c.lk, ssq, c.N, pss, P.n_params);
    }
};

template <typename T>
__global__ void __launch_bounds__(QS_THREADS, 1) k_hmc_stream(const __grid_constant__ QbStreamPlan P, const ChainArgs<T> c, const HmcArgs<T> h) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QsRing rg;
    qs_ring_init(P, smem_raw, rg);
    QbGradStream<T> eval{P, smem_raw, rg, c, (long long)blockIdx.x};
    qb_hmc_body<T>(c, h, P.n_params, reinterpret_cast<double*>(smem_raw), eval);
}

// NUTS (qb_nuts.cuh) on the same evaluation functors as k_hmc / k_hmc_stream
template <typename T>
__global__ void __launch_bounds__(256, 1) k_nuts(const __grid_constant__ QbPlan plan, const ChainArgs<T> c, const NutsArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(plan, smem_raw);
    QbGradSimt<T> eval{plan, S, c, (long long)blockIdx.x};
    qb_nuts_body<T>(c, a, plan.n_params, S.red, eval);
}

template <typename T>
__global__ void __launch_bounds__(QS_THREADS, 1) k_nuts_stream(const __grid_constant__ QbStreamPlan P, const ChainArgs<T> c, const NutsArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QsRing rg;
    qs_ring_init(P, smem_raw, rg);
    QbGradStream<T> eval{P, smem_raw, rg, c, (long long)blockIdx.x};
    qb_nuts_body<T>(c, a, P.n_params, reinterpret_cast<double*>(smem_raw), eval);
}

// parallel-tempering twins of k_hmc / k_hmc_stream (qb_pt.cuh): same evaluation functors, tempered
template <typename T>
__global__ void __launch_bounds__(256, 2) k_pt_hmc(const __grid_constant__ QbPlan plan, const ChainArgs<T> c, const HmcArgs<T> h,
                                                   const PtArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(plan, smem_raw);
    QbGradSimt<T> inner{plan, S, c, (long long)blockIdx.x};
    qb_pt_hmc_body<T>(c, h, a, plan.n_params, S.red, inner);
}

template <typename T>
__global__ void __launch_bounds__(QS_THREADS, 1) k_pt_hmc_stream(const __grid_constant__ QbStreamPlan P, const ChainArgs<T> c,
                                                                 const HmcArgs<T> h, const PtArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QsRing rg;
    qs_ring_init(P, smem_raw, rg);
    QbGradStream<T> inner{P, smem_raw, rg, c, (long long)blockIdx.x};
    qb_pt_hmc_body<T>(c, h, a, P.n_params, reinterpret_cast<double*>(smem_raw), inner);
}

template <typename T>
static void fill_chain_args(ChainArgs<T>& c, const qb_data_t* data, const qb_lik_t* lik, const qb_chain_t* ch,
                            const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start, int64_t nsteps, int init_lp) {
    c.K = ch->K; c.N = data->n; c.x = (const T*)data->x; c.y = (const T*)data->y; c.lk = lik_dev(lik);
    c.theta = (T*)ch->theta; c.lp = ch->lp; c.naccept = (long long*)ch->naccept; c.map_theta = (T*)ch->map_theta; c.map_lp = ch->map_lp;
    c.rng_mode = rng->mode; c.seed = rng->seed; c.chain_offset = rng->chain_offset; c.incr = (const T*)rng->incr; c.unif = rng->unif;
    c.rec_lp = rec ? rec->logpost : nullptr; c.rec_alpha = rec ? rec->alpha : nullptr; c.rec_acc = rec ? rec->accepted : nullptr;
    c.rec_ld = rec ? rec->ld : 0; c.samples = rec ? (T*)rec->samples : nullptr; c.rec_lp0 = rec ? rec->logpost0 : nullptr;
    c.store_every = rec ? rec->store_every : 0; c.n_slots = rec ? rec->n_slots : 0;
    c.t_start = t_start; c.nsteps = nsteps; c.init_lp = init_lp;
}

static int check_chain_common(const qb_data_t* data, const qb_lik_t* lik, const qb_chain_t* ch, const qb_rng_t* rng) {
    if (!data || !lik || !ch || !rng) return qb_fail("NULL argument to chain run");
    if (!ch->theta || !ch->lp || !ch->naccept || !ch->map_theta || !ch->map_lp) return qb_fail("chain state has NULL arrays");
    if (rng->mode == QB_RNG_REPLAY && (!rng->incr || !rng->unif)) return qb_fail("replay mode needs incr and unif");
    if (ch->K < 1) return qb_fail("K must be positive");
    return 0;
}

template <typename T>
static int run_amcmc(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik, qb_chain_t* ch,
                     qb_amcmc_t* am, const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start, int64_t nsteps,
                     int init_lp, void* scratch, cudaStream_t st) {
    QbLaunch L;
    if (make_launch(net, dtype, false, ch->K, data->n, true, &L)) return -1;
    const int P = net->n_params;
    if (am->adapt == QB_ADAPT_FULL || am->chol_ini) {
        const long long act_elems = L.streamed ? L.sp.act_elems : (L.plan.smem_bytes - 40 * 8) / L.plan.elem_size - L.plan.w_elems;
        if (P > act_elems) return qb_fail("full-covariance proposals need P <= tile scratch%s (P=%lld)", "", P);
    }
    ChainArgs<T> c; fill_chain_args<T>(c, data, lik, ch, rng, rec, t_start, nsteps, init_lp);
    AmcmcArgs<T> a;
    a.gamma = am->gamma; a.t0 = am->t0; a.tadapt = am->tadapt; a.adapt = am->adapt;
    a.track = am->track_moments;
    if (am->adapt == QB_ADAPT_DIAG) a.track = 1;
    if (am->adapt == QB_ADAPT_FULL) a.track = 2;
    if (a.track < 0 || a.track > 2) return qb_fail("track_moments must be 0, 1 (diagonal cov) or 2 (full cov)");
    if (a.track && !am->cov) return qb_fail("moment tracking needs cov");
    a.xm = (T*)am->xm; a.cov = (T*)am->cov; a.pscale = (T*)am->pscale; a.chol = (T*)am->chol;
    a.chol_ini = (const T*)am->chol_ini; a.prop_kind = am->prop_kind; a.prop = (T*)scratch;
    if (a.track && (!a.xm)) return qb_fail("moment tracking needs xm");
    if (am->adapt != QB_ADAPT_NONE && !a.cov) return qb_fail("adaptation needs cov");
    if (am->adapt == QB_ADAPT_FULL && !a.chol) return qb_fail("full adaptation needs chol");
    if (!a.pscale || !a.prop_kind || !a.prop) return qb_fail("amcmc needs pscale, prop_kind and scratch");
    QbTcPlan tp;
    const bool tc = !L.streamed && am->adapt != QB_ADAPT_FULL && !am->chol_ini && make_tc_plan(net, dtype, &tp, 2);
    if (L.streamed) {
        if (set_smem(k_amcmc_stream<T>, L.sp.smem_bytes)) return -2;
        k_amcmc_stream<T><<<(unsigned)ch->K, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, c, a);
    } else if (tc) {
        if (launch_amcmc_tc<T>(L.plan, tp, c, a, ch->K, st)) return -2;
    } else {
        memset(&tp, 0, sizeof(tp));
        if (set_smem(k_amcmc<T, 0>, L.plan.smem_bytes)) return -2;
        k_amcmc<T, 0><<<(unsigned)ch->K, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, tp, c, a);
    }
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

extern "C" int qb_amcmc_run(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik,
                            qb_chain_t* chain, qb_amcmc_t* am, const qb_rng_t* rng, const qb_record_t* rec,
                            int64_t t_start, int64_t nsteps, int init_lp, void* scratch, void* stream) {
    if (check_chain_common(data, lik, chain, rng) || !am) return g_err[0] ? -1 : qb_fail("NULL amcmc state");
    if (dtype == QB_F64) return run_amcmc<double>(net, dtype, data, lik, chain, am, rng, rec, t_start, nsteps, init_lp, scratch, (cudaStream_t)stream);
    return run_amcmc<float>(net, dtype, data, lik, chain, am, rng, rec, t_start, nsteps, init_lp, scratch, (cudaStream_t)stream);
}

template <typename T>
static int run_hmc(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik, qb_chain_t* ch,
                   qb_hmc_t* hm, const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start, int64_t nsteps,
                   int init_lp, cudaStream_t st) {
    QbLaunch L;
    if (plan_eval(net, dtype, true, ch->K, data->n, true, &L)) return -1;
    if (!hm->grad_cur || !hm->mom || !hm->prop || !hm->grad_prop) return qb_fail("hmc state has NULL arrays");
    if (hm->method == 0 && hm->L < 1) return qb_fail("HMC needs L >= 1");
    ChainArgs<T> c; fill_chain_args<T>(c, data, lik, ch, rng, rec, t_start, nsteps, init_lp);
    HmcArgs<T> h;
    h.method = hm->method; h.L = hm->L; h.eps = hm->epsilon;
    h.gcur = (T*)hm->grad_cur; h.mom = (T*)hm->mom; h.prop = (T*)hm->prop; h.gprop = (T*)hm->grad_prop;
    if (L.path == QB_PATH_STREAM) {
        if (set_smem(k_hmc_stream<T>, L.sp.smem_bytes)) return -2;
        k_hmc_stream<T><<<(unsigned)ch->K, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, c, h);
    } else if (L.path == QB_PATH_TG8) {
        if (launch_hmc_tc128<T>(L.t8, c, h, ch->K, st)) return -2;
        g_launches += 1;
    } else if (L.path == QB_PATH_TCG) {
        if (launch_hmc_tc<T>(L.tg, c, h, ch->K, st)) return -2;
    } else {
        if (set_smem(k_hmc<T>, L.plan.smem_bytes)) return -2;
        k_hmc<T><<<(unsigned)ch->K, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, c, h);
    }
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

extern "C" int qb_hmc_run(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik,
                          qb_chain_t* chain, qb_hmc_t* hm, const qb_rng_t* rng, const qb_record_t* rec,
                          int64_t t_start, int64_t nsteps, int init_lp, void* stream) {
    if (check_chain_common(data, lik, chain, rng) || !hm) return g_err[0] ? -1 : qb_fail("NULL hmc state");
    if (dtype == QB_F64) return run_hmc<double>(net, dtype, data, lik, chain, hm, rng, rec, t_start, nsteps, init_lp, (cudaStream_t)stream);
    return run_hmc<float>(net, dtype, data, lik, chain, hm, rng, rec, t_start, nsteps, init_lp, (cudaStream_t)stream);
}

template <typename T> static int launch_pt_tc128(const QbTg8Plan&, const ChainArgs<T>&, const HmcArgs<T>&, const PtArgs&, long long,
                                                 const float*, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_pt_tc128<float>(const QbTg8Plan& tg, const ChainArgs<float>& c, const HmcArgs<float>& h, const PtArgs& a,
                                       long long K, const float* absmax, cudaStream_t st) {
    QB_CUDA(qb_tg8_launch_pt(tg, c, h, a, K, absmax, st));
    return 0;
}
template <typename T> static int pt_absmax(const QbTg8Plan&, const ChainArgs<T>&, cudaStream_t, const float**) {
    return qb_fail("tensor-core path is fp32 only");
}
template <> int pt_absmax<float>(const QbTg8Plan& tg, const ChainArgs<float>& c, cudaStream_t st, const float** absmax) {
    QB_CUDA(qb_tg8_pt_absmax(tg, c, st, absmax));
    return 0;
}
template <typename T> static int launch_pt_tc(const QbTcgPlan&, const ChainArgs<T>&, const HmcArgs<T>&, const PtArgs&, long long,
                                              cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_pt_tc<float>(const QbTcgPlan& tg, const ChainArgs<float>& c, const HmcArgs<float>& h, const PtArgs& a,
                                    long long K, cudaStream_t st) {
    QB_CUDA(qb_tcg_launch_pt(tg, c, h, a, K, st));
    return 0;
}

// The local ChainArgs of the sub-launch [s, s + n) of a call: its t_start, step count and record positions.  Stored
// draws keep the slots qb_hmc_run gives the whole call: slot (s + j + 1) / store_every - 1 after call step s + j.
template <typename T>
static void pt_sub_args(ChainArgs<T>& cs, const ChainArgs<T>& c, long long s, long long n, int P) {
    cs = c;
    cs.t_start = c.t_start + s; cs.nsteps = n; cs.init_lp = c.init_lp && s == 0;
    if (c.rec_lp) cs.rec_lp = c.rec_lp + s;
    if (c.rec_alpha) cs.rec_alpha = c.rec_alpha + s;
    if (c.rec_acc) cs.rec_acc = c.rec_acc + s;
    cs.samples = nullptr;
    const long long se = c.store_every;
    if (!c.samples || se <= 0) return;
    long long slot0, every;
    if (s % se == 0) { slot0 = s / se; every = se; }                  // stores at local steps j with (j + 1) % se == 0
    else if ((s + n) % se == 0) { slot0 = (s + n) / se - 1; every = n; }   // one store, after the last step
    else return;
    if (slot0 >= c.n_slots) return;
    cs.samples = c.samples + slot0 * P;          // row k stays at k * n_slots (the kernel's stride)
    cs.store_every = every;
}

template <typename T>
static int run_pt(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik, qb_chain_t* ch, qb_hmc_t* hm,
                  const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start, int64_t nsteps, int init_lp, int64_t G,
                  const double* beta, const double* eps, int64_t swap_every, int32_t* replica, int8_t* last_end,
                  int64_t* round_trips, int64_t* attempts, int64_t* accepts, cudaStream_t st) {
    QbLaunch L;
    if (plan_eval(net, dtype, true, ch->K, data->n, true, &L)) return -1;
    if (!hm->grad_cur || !hm->mom || !hm->prop || !hm->grad_prop) return qb_fail("hmc state has NULL arrays");
    if (hm->method == 0 && hm->L < 1) return qb_fail("HMC needs L >= 1");
    const int P = net->n_params;
    const long long K = ch->K, nT = K / G;
    ChainArgs<T> c; fill_chain_args<T>(c, data, lik, ch, rng, rec, t_start, nsteps, init_lp);
    HmcArgs<T> h;
    h.method = hm->method; h.L = hm->L; h.eps = hm->epsilon;
    h.gcur = (T*)hm->grad_cur; h.mom = (T*)hm->mom; h.prop = (T*)hm->prop; h.gprop = (T*)hm->grad_prop;
    const PtArgs a{beta, eps, (long long)G};
    PtSwapArgs sw{beta, (long long)G, (int)nT, rng->seed, rng->chain_offset, 0, ch->lp, replica, (signed char*)last_end,
                  (long long*)round_trips, (long long*)attempts, (long long*)accepts};
    const float* absmax = nullptr;
    if (L.path == QB_PATH_TG8 && pt_absmax<T>(L.t8, c, st, &absmax)) return -2;      // once per call, not per launch
    if (L.path == QB_PATH_STREAM && set_smem(k_pt_hmc_stream<T>, L.sp.smem_bytes)) return -2;
    const bool simt = L.path != QB_PATH_STREAM && L.path != QB_PATH_TG8 && L.path != QB_PATH_TCG;
    if (simt && set_smem(k_pt_hmc<T>, L.plan.smem_bytes)) return -2;
    // sub-launches end at swap boundaries and, so that no store passes the last slot, at n_slots * store_every
    const long long cut = (c.samples && c.store_every > 0) ? c.n_slots * c.store_every : -1;
    for (long long s = 0; s < nsteps;) {
        const long long t = t_start + s;
        long long n = std::min<long long>(swap_every - t % swap_every, nsteps - s);
        if (s < cut) n = std::min(n, cut - s);
        ChainArgs<T> cs; pt_sub_args<T>(cs, c, s, n, P);
        if (L.path == QB_PATH_STREAM) {
            k_pt_hmc_stream<T><<<(unsigned)K, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, cs, h, a);
        } else if (L.path == QB_PATH_TG8) {
            if (launch_pt_tc128<T>(L.t8, cs, h, a, K, absmax, st)) return -2;
        } else if (L.path == QB_PATH_TCG) {
            if (launch_pt_tc<T>(L.tg, cs, h, a, K, st)) return -2;
        } else {
            k_pt_hmc<T><<<(unsigned)K, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, cs, h, a);
        }
        QB_CUDA(cudaGetLastError());
        g_launches += 1;
        s += n;
        if ((t_start + s) % swap_every == 0 && nT > 1) {
            sw.r = (t_start + s) / swap_every - 1;
            const int npairs = (int)(nT / 2);
            k_pt_swap<T><<<(unsigned)G, 256, std::max(npairs, 1) * (int)sizeof(int), st>>>(sw, (T*)ch->theta, h.gcur, P);
            QB_CUDA(cudaGetLastError());
            g_launches += 1;
        }
    }
    if (L.path == QB_PATH_TG8) g_launches += 1;
    return 0;
}

extern "C" int qb_pt_run(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik, qb_chain_t* chain,
                         qb_hmc_t* hm, const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start, int64_t nsteps,
                         int init_lp, int64_t n_groups, const double* beta, const double* eps, int64_t swap_every,
                         int32_t* replica, int8_t* last_end, int64_t* round_trips, int64_t* swap_attempts,
                         int64_t* swap_accepts, void* stream) {
    if (!net || !data || !lik || !chain || !rng || !hm) return qb_fail("NULL argument to chain run");
    if (rng->mode == QB_RNG_REPLAY) return qb_fail("parallel tempering has no replay mode: its draws come from Philox");
    if (!beta || !eps || !replica || !last_end || !round_trips || !swap_attempts || !swap_accepts)
        return qb_fail("parallel-tempering state has NULL arrays");
    if (n_groups < 1) return qb_fail("parallel tempering needs n_groups >= 1");
    if (chain->K % n_groups != 0) return qb_fail("K must be a multiple of n_groups%s (K=%lld)", "", chain->K);
    if (swap_every < 1) return qb_fail("parallel tempering needs swap_every >= 1");
    if (nsteps < 0 || t_start < 0) return qb_fail("nsteps and t_start must be >= 0");
    if (t_start % swap_every != 0) return qb_fail("t_start must be a multiple of swap_every%s (t_start=%lld)", "", t_start);
    if (rec && rec->samples && rec->store_every > 0 && rec->store_every % swap_every != 0 && swap_every % rec->store_every != 0)
        return qb_fail("store_every and swap_every must divide one another%s (store_every=%lld)", "", rec->store_every);
    if (chain->K == 0 || nsteps == 0) return 0;
    if (check_chain_common(data, lik, chain, rng)) return -1;
    if (dtype == QB_F64)
        return run_pt<double>(net, dtype, data, lik, chain, hm, rng, rec, t_start, nsteps, init_lp, n_groups, beta, eps,
                              swap_every, replica, last_end, round_trips, swap_attempts, swap_accepts, (cudaStream_t)stream);
    return run_pt<float>(net, dtype, data, lik, chain, hm, rng, rec, t_start, nsteps, init_lp, n_groups, beta, eps, swap_every,
                         replica, last_end, round_trips, swap_attempts, swap_accepts, (cudaStream_t)stream);
}

template <typename T>
static void fill_nuts_args(NutsArgs<T>& a, double epsilon, int max_depth, int64_t n_adapt, double target_accept, double* log_eps,
                           double* log_eps_bar, double* h_bar, void* grad_cur, void* scratch, int32_t* rec_depth,
                           int32_t* rec_n_leapfrog, uint8_t* rec_diverging, double* rec_step_size) {
    a.eps0 = epsilon; a.target = target_accept; a.max_depth = max_depth; a.n_adapt = n_adapt;
    a.log_eps = log_eps; a.log_eps_bar = log_eps_bar; a.h_bar = h_bar;
    a.gcur = (T*)grad_cur; a.scratch = (T*)scratch;
    a.rec_depth = rec_depth; a.rec_nleap = rec_n_leapfrog; a.rec_div = rec_diverging; a.rec_eps = rec_step_size;
}

template <typename T>
static int run_nuts(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik, qb_chain_t* ch,
                    const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start, int64_t nsteps, int init_lp,
                    const NutsArgs<T>& a, cudaStream_t st) {
    QbLaunch L;
    if (plan_eval(net, dtype, true, ch->K, data->n, true, &L)) return -1;
    ChainArgs<T> c; fill_chain_args<T>(c, data, lik, ch, rng, rec, t_start, nsteps, init_lp);
    if (L.path == QB_PATH_STREAM) {
        if (set_smem(k_nuts_stream<T>, L.sp.smem_bytes)) return -2;
        k_nuts_stream<T><<<(unsigned)ch->K, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, c, a);
    } else if (L.path == QB_PATH_TG8) {
        if (launch_nuts_tc128<T>(L.t8, c, a, ch->K, st)) return -2;
        g_launches += 1;
    } else if (L.path == QB_PATH_TCG) {
        if (launch_nuts_tc<T>(L.tg, c, a, ch->K, st)) return -2;
    } else {
        if (set_smem(k_nuts<T>, L.plan.smem_bytes)) return -2;
        k_nuts<T><<<(unsigned)ch->K, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, c, a);
    }
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

extern "C" int qb_nuts_run(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik,
                           qb_chain_t* chain, const qb_rng_t* rng, const qb_record_t* rec, int64_t t_start,
                           int64_t nsteps, int init_lp, double epsilon, int max_depth, int64_t n_adapt,
                           double target_accept, double* log_eps, double* log_eps_bar, double* h_bar, void* grad_cur,
                           void* scratch, int32_t* rec_depth, int32_t* rec_n_leapfrog, uint8_t* rec_diverging,
                           double* rec_step_size, void* stream) {
    if (!net || !data || !lik || !chain || !rng) return qb_fail("NULL argument to chain run");
    if (rng->mode == QB_RNG_REPLAY) return qb_fail("NUTS has no replay mode: its draws come from Philox");
    if (!(epsilon > 0.0 && epsilon < INFINITY)) return qb_fail("NUTS needs a finite epsilon > 0");
    if (max_depth < 1 || max_depth > QB_NUTS_MAX_DEPTH)
        return qb_fail("NUTS needs 1 <= max_depth <= 12%s (max_depth=%lld)", "", max_depth);
    if (!(target_accept > 0.0 && target_accept < 1.0)) return qb_fail("NUTS needs 0 < target_accept < 1");
    if (n_adapt < 0 || nsteps < 0 || t_start < 0) return qb_fail("n_adapt, nsteps and t_start must be >= 0");
    if (!log_eps || !log_eps_bar || !h_bar || !grad_cur || !scratch) return qb_fail("NUTS state has NULL arrays");
    if (!rec && (rec_depth || rec_n_leapfrog || rec_diverging || rec_step_size))
        return qb_fail("NUTS records need rec: they share its leading dimension");
    if (chain->K == 0 || nsteps == 0) return 0;
    if (check_chain_common(data, lik, chain, rng)) return -1;
    if (dtype == QB_F64) {
        NutsArgs<double> a;
        fill_nuts_args<double>(a, epsilon, max_depth, n_adapt, target_accept, log_eps, log_eps_bar, h_bar, grad_cur, scratch,
                               rec_depth, rec_n_leapfrog, rec_diverging, rec_step_size);
        return run_nuts<double>(net, dtype, data, lik, chain, rng, rec, t_start, nsteps, init_lp, a, (cudaStream_t)stream);
    }
    NutsArgs<float> a;
    fill_nuts_args<float>(a, epsilon, max_depth, n_adapt, target_accept, log_eps, log_eps_bar, h_bar, grad_cur, scratch,
                          rec_depth, rec_n_leapfrog, rec_diverging, rec_step_size);
    return run_nuts<float>(net, dtype, data, lik, chain, rng, rec, t_start, nsteps, init_lp, a, (cudaStream_t)stream);
}

// =================================================================================================
// kernel 4: posterior predictive
// =================================================================================================
template <typename T> struct PredArgs {
    const T* theta; const T* x; long long M, N;
    T* out; T* mean; T* var;
    int fused;     // 1: block = point tile, loops over all members, Welford in registers
    long long tiles_per_block;   // member-parallel mode
};

template <typename T>
__global__ void __launch_bounds__(512, 1) k_predict(const __grid_constant__ QbPlan P, const PredArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(P, smem_raw);
    T* sW = reinterpret_cast<T*>(S.w);
    T* A0 = reinterpret_cast<T*>(S.act);
    const int lda = P.lda, TM = P.TM, o = P.out_dim;
    T* A1 = P.inplace ? A0 : A0 + (size_t)P.buf_rows * lda;
    const int n = TM * o;
    const QbScope sc = P.ws ? qb_warp_scope(P.WP) : qb_block_scope(TM);
    if (!a.fused) {
        // member-parallel: this block owns member blockIdx.y and a chunk of consecutive tiles; the weights are
        // staged once and every warp (warp-synchronous plans) copies out its own points without a block barrier
        const long long m = blockIdx.x;          // members on grid.x: M is not limited to 65535
        const long long ntiles = (a.N + TM - 1) / TM;
        const long long t0 = (long long)blockIdx.y * a.tiles_per_block, t1 = min(ntiles, t0 + a.tiles_per_block);
        qb_stage_weights<T>(P, sW, a.theta + m * P.n_params);
        __syncthreads();
        for (long long t = t0; t < t1; ++t) {
            const long long p0 = t * TM;
            qb_load_x_tile<T>(a.x, P.in_dim, p0, a.N, A0, lda, sc);
            sc.sync();
            T* cur = A0; T* oth = A1;
            for (int l = 0; l < P.n_layers; ++l) {
                qb_layer_forward<T>(P.L[l], sW, cur, oth, lda, sc, P.inplace != 0);
                T* tt = cur; cur = oth; oth = tt;
            }
            const int nn = sc.p_count * o;
            for (int idx = sc.tid; idx < nn; idx += sc.nthr) {
                const int pl = idx / o, j = idx - pl * o, p = sc.p_base + pl;
                const long long gp = p0 + p;
                if (gp < a.N) {
                    T v = cur[j * lda + p];
                    if (P.final_exp) v = qb_exp(v);
                    a.out[(m * a.N + gp) * o + j] = v;
                }
            }
            sc.sync();
        }
        return;
    }
    const long long p0 = (long long)blockIdx.x * TM;
    constexpr int QMAX = 4;
    T wmean[QMAX], wm2[QMAX];
#pragma unroll
    for (int q = 0; q < QMAX; ++q) { wmean[q] = T(0); wm2[q] = T(0); }
    for (long long m = 0; m < a.M; ++m) {
        __syncthreads();
        qb_stage_weights<T>(P, sW, a.theta + m * P.n_params);
        __syncthreads();
        qb_load_x_tile<T>(a.x, P.in_dim, p0, a.N, A0, lda, sc);
        sc.sync();
        T* cur = A0; T* oth = A1;
        for (int l = 0; l < P.n_layers; ++l) {
            qb_layer_forward<T>(P.L[l], sW, cur, oth, lda, sc, P.inplace != 0);
            T* t = cur; cur = oth; oth = t;
        }
        __syncthreads();          // the accumulation below reads points of every warp
        const T inv_n = T(1) / (T)(m + 1);
#pragma unroll
        for (int q = 0; q < QMAX; ++q) {
            const int idx = threadIdx.x + q * blockDim.x;
            if (idx < n) {
                // idx = p * o + j : consecutive threads write consecutive addresses of out[m, p0+p, j]
                const int p = idx / o, j = idx - p * o;
                const long long gp = p0 + p;
                if (gp < a.N) {
                    T v = cur[j * lda + p];
                    if (P.final_exp) v = qb_exp(v);
                    if (a.out) a.out[(m * a.N + gp) * o + j] = v;
                    const T d = v - wmean[q];
                    wmean[q] += d * inv_n;
                    wm2[q] = fma(d, v - wmean[q], wm2[q]);
                }
            }
        }
    }
    if (a.fused) {
#pragma unroll
        for (int q = 0; q < QMAX; ++q) {
            const int idx = threadIdx.x + q * blockDim.x;
            if (idx < n) {
                const int p = idx / o, j = idx - p * o;
                const long long gp = p0 + p;
                if (gp < a.N) {
                    if (a.mean) a.mean[gp * o + j] = wmean[q];
                    if (a.var) a.var[gp * o + j] = a.M > 1 ? wm2[q] / (T)(a.M - 1) : T(NAN);
                }
            }
        }
    }
}

// kernel 4, layer-streamed: block b = member b / chunks, tile chunk b % chunks (a member's chunks are neighbours)
template <typename T>
__global__ void __launch_bounds__(QS_THREADS, 1) k_predict_stream(const __grid_constant__ QbStreamPlan P, const PredArgs<T> a,
                                                                 long long chunks) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    QsRing rg;
    qs_ring_init(P, smem_raw, rg);
    const long long b = blockIdx.x, m = b / chunks, ch = b - m * chunks;
    const long long n0 = ch * a.tiles_per_block * P.TM, n1 = min(a.N, n0 + a.tiles_per_block * P.TM);
    qs_eval<T, false>(P, smem_raw, rg, a.theta + m * P.n_params, a.x, nullptr, n0, n1, 0.0, nullptr,
                      a.out + m * a.N * P.out_dim);
}

// mean / var(ddof=1) over the leading axis of out[M, n]  (HBM-bound, coalesced over n)
template <typename T>
__global__ void k_moments(const T* out, long long M, long long n, T* mean, T* var) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T mu = T(0), m2 = T(0);
    for (long long m = 0; m < M; ++m) {
        const T v = out[m * n + i];
        const T d = v - mu;
        mu += d / (T)(m + 1);
        m2 = fma(d, v - mu, m2);
    }
    if (mean) mean[i] = mu;
    if (var) var[i] = M > 1 ? m2 / (T)(M - 1) : T(NAN);
}

// kernel 4 on the tensor cores (member-parallel: block = member blockIdx.y x a chunk of consecutive tiles)
__global__ void __launch_bounds__(512, 1) k_predict_tc(const __grid_constant__ QbTcPlan tp, const PredArgs<float> a) {
    extern __shared__ __align__(128) unsigned char smem_tc[];
    QbTcCtx cx;
    qb_tc_init(tp, smem_tc, cx);
    const long long m = blockIdx.x;
    const long long n0 = (long long)blockIdx.y * a.tiles_per_block * 128, n1 = min(a.N, n0 + a.tiles_per_block * 128);
    qb_tc_stage(tp, smem_tc, a.theta + m * tp.n_params);
    __syncthreads();
    qb_tc_predict(tp, cx, smem_tc, a.x, a.out + m * a.N * tp.out_dim, n0, n1);
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}
template <typename T> static int launch_predict_tc(const QbTcPlan&, const PredArgs<T>&, dim3, cudaStream_t) { return qb_fail("tensor-core path is fp32 only"); }
template <> int launch_predict_tc<float>(const QbTcPlan& tp, const PredArgs<float>& a, dim3 grid, cudaStream_t st) {
    if (tp.v3) {                  // 64- / 128-wide tanh nets with one output: warp-specialised kernel (qb_value_tc3.cu)
        QB_CUDA(qb_tc3_launch_predict(tp, a.theta, a.x, a.N, a.out, a.tiles_per_block, grid, st));
        return 0;
    }
    if (set_smem(k_predict_tc, tp.smem_bytes)) return -2;
    k_predict_tc<<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, a);
    return 0;
}

template <typename T>
static int run_predict(const qb_net_t* net, int dtype, const void* theta, int64_t M, const void* x, int64_t N,
                       void* out, void* mean, void* var, cudaStream_t st) {
    QbLaunch L;
    if (make_launch(net, dtype, false, M, N, true, &L)) return -1;
    if (L.streamed) {
        const QbStreamPlan& SP = L.sp;
        if (!out) return qb_fail("moments without `out` need TM*out_dim <= 4*threads; pass an `out` buffer");
        PredArgs<T> a;
        a.theta = (const T*)theta; a.x = (const T*)x; a.M = M; a.N = N;
        a.out = (T*)out; a.mean = (T*)mean; a.var = (T*)var; a.fused = 0;
        const long long chunks = qb_tile_chunks(cdiv(N, SP.TM), (long long)qb_num_sms() * 2, M, &a.tiles_per_block);
        if (set_smem(k_predict_stream<T>, SP.smem_bytes)) return -2;
        k_predict_stream<T><<<(unsigned)(M * chunks), QS_THREADS, SP.smem_bytes, st>>>(SP, a, chunks);
        QB_CUDA(cudaGetLastError());
        g_launches += 1;
        if (mean || var) {
            const long long n = N * SP.out_dim;
            k_moments<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>((const T*)out, M, n, (T*)mean, (T*)var);
            QB_CUDA(cudaGetLastError());
            g_launches += 1;
        }
        return 0;
    }
    const QbPlan& P = L.plan;
    const long long tiles = cdiv(N, P.TM);
    const bool want_mom = mean || var;
    const bool can_fuse = (long long)P.TM * P.out_dim <= 4LL * P.nthreads;
    bool fused = want_mom && can_fuse && !out;     // with an `out` buffer: member-parallel + k_moments (weights staged once)
    if (want_mom && !fused && !out) return qb_fail("moments without `out` need TM*out_dim <= 4*threads; pass an `out` buffer");
    PredArgs<T> a;
    a.theta = (const T*)theta; a.x = (const T*)x; a.M = M; a.N = N;
    a.out = (T*)out; a.mean = (T*)mean; a.var = (T*)var; a.fused = fused ? 1 : 0;
    QbTcPlan tp;
    if (!fused && out && make_tc_plan(net, dtype, &tp, 3)) {
        // tensor-core forward (qb_tc.cuh / qb_tc3.cuh): 128-point tiles, weights staged once per block, >= 8 waves of blocks
        const long long ch = qb_tile_chunks(cdiv(N, 128), (long long)qb_num_sms() * 2 * 8, M, &a.tiles_per_block);
        if (launch_predict_tc<T>(tp, a, dim3((unsigned)M, (unsigned)ch), st)) return -2;
        QB_CUDA(cudaGetLastError());
        g_launches += 1;
        if (want_mom) {
            const long long n = N * P.out_dim;
            k_moments<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>((const T*)out, M, n, (T*)mean, (T*)var);
            QB_CUDA(cudaGetLastError());
            g_launches += 1;
        }
        return 0;
    }
    if (set_smem(k_predict<T>, P.smem_bytes)) return -2;
    long long chunks = tiles;
    a.tiles_per_block = 1;
    if (!fused) chunks = qb_tile_chunks(tiles, (long long)qb_num_sms() * 8, M, &a.tiles_per_block);
    dim3 grid(fused ? (unsigned)chunks : (unsigned)M, fused ? 1u : (unsigned)chunks);
    k_predict<T><<<grid, P.nthreads, P.smem_bytes, st>>>(P, a);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    if (want_mom && !fused) {
        const long long n = N * P.out_dim;
        k_moments<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>((const T*)out, M, n, (T*)mean, (T*)var);
        QB_CUDA(cudaGetLastError());
        g_launches += 1;
    }
    return 0;
}

extern "C" int qb_predict(const qb_net_t* net, int dtype, const void* theta, int64_t M, const void* x, int64_t N,
                          void* out, void* mean, void* var, void* stream) {
    if (!theta || !x) return qb_fail("NULL argument to qb_predict");
    if (!out && !mean && !var) return qb_fail("qb_predict: nothing to compute");
    if (dtype == QB_F64) return run_predict<double>(net, dtype, theta, M, x, N, out, mean, var, (cudaStream_t)stream);
    return run_predict<float>(net, dtype, theta, M, x, N, out, mean, var, (cudaStream_t)stream);
}

// =================================================================================================
// variational inference element-wise kernels
// =================================================================================================
template <typename T>
__global__ void __launch_bounds__(256, 2) k_vi_sample(const T* mu, const T* rho, T* eps, long long nsam, long long P, double pi,
                                                   double s1, double s2, unsigned long long seed, unsigned long long step,
                                                   T* w, double* logq, double* logp) {
    __shared__ double red[40];
    const long long s = blockIdx.x;
    const double LOG_SQRT_2PI = 0.91893853320467274178;
    double lq = 0.0, lpr = 0.0;
    if (seed) {
        for (long long i4 = threadIdx.x; i4 * 4 < P; i4 += blockDim.x) {
            T z[4];
            qb_normal4(qb_rand4(seed, s, (long long)step, QB_STREAM_VI, (uint32_t)i4), z);
            for (int q = 0; q < 4; ++q) if (i4 * 4 + q < P) eps[s * P + i4 * 4 + q] = z[q];
        }
        __syncthreads();
    }
    for (long long i = threadIdx.x; i < P; i += blockDim.x) {
        const double m = (double)mu[i], r = (double)rho[i], e = (double)eps[s * P + i];
        const double sig = exp(r);
        const T wv = (T)(m + sig * e);
        w[s * P + i] = wv;
        const double wd = (double)wv;
        // Gaussian_1d.log_prob (rvs.py:124-126)
        const double dq = wd - m;
        lq += -LOG_SQRT_2PI - log(sig) - dq * dq / (2.0 * sig * sig);
        // GMM2_1d.log_prob (rvs.py:169-171): exp-then-log, not log-sum-exp
        const double p1 = exp(-wd * wd / (2.0 * s1 * s1) - log(s1) - LOG_SQRT_2PI);
        const double p2 = exp(-wd * wd / (2.0 * s2 * s2) - log(s2) - LOG_SQRT_2PI);
        lpr += log(pi * p1 + (1.0 - pi) * p2);
    }
    lq = qb_block_sum(lq, red);
    lpr = qb_block_sum(lpr, red);
    if (threadIdx.x == 0) { logq[s] = lq; logp[s] = lpr; }
}

template <typename T>
__global__ void __launch_bounds__(256) k_vi_backward(const T* mu, const T* rho, const T* eps, const T* w, const T* glp, long long nsam, long long P,
                                                     double pi, double s1, double s2, double c_ssq, double c_logp, double c_logq, T* gmu, T* grho) {
    // block = 32 parameters x 8 sample lanes: lane y takes samples y, y + 8, ..; the eight partial sums meet in shared memory in
    // fixed order (one thread per parameter looping over all samples was latency-bound: 198 us for 128 x 18049)
    __shared__ double sm_[8][32], sr_[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const long long i = (long long)blockIdx.x * 32 + tx;
    const double LOG_SQRT_2PI = 0.91893853320467274178;
    const double c1 = -log(s1) - LOG_SQRT_2PI, c2 = -log(s2) - LOG_SQRT_2PI, h1 = 1.0 / (2.0 * s1 * s1), h2 = 1.0 / (2.0 * s2 * s2);
    double am = 0.0, ar = 0.0;
    if (i < P) {
        const double sig = exp((double)rho[i]);
        for (long long s = ty; s < nsam; s += 8) {
            const double wd = (double)w[s * P + i], e = (double)eps[s * P + i];
            const double p1 = pi * exp(-wd * wd * h1 + c1);
            const double p2 = (1.0 - pi) * exp(-wd * wd * h2 + c2);
            const double dlogp = (p1 * (-wd / (s1 * s1)) + p2 * (-wd / (s2 * s2))) / (p1 + p2);
            const double dw = c_ssq * (-2.0 * (double)glp[s * P + i]) + c_logp * dlogp;
            am += dw;
            ar += dw * sig * e - c_logq;      // log q: total derivative wrt mu is 0, wrt rho is -1 per sample
        }
    }
    sm_[ty][tx] = am; sr_[ty][tx] = ar;
    __syncthreads();
    if (ty == 0 && i < P) {
        double m = 0.0, r = 0.0;
#pragma unroll
        for (int y = 0; y < 8; ++y) { m += sm_[y][tx]; r += sr_[y][tx]; }
        gmu[i] = (T)m;
        grho[i] = (T)r;
    }
}

extern "C" int qb_vi_sample(int dtype, const void* mu, const void* rho, void* eps, int64_t nsam, int64_t P, double pi,
                            double sigma1, double sigma2, uint64_t seed, uint64_t step, void* w, double* logq,
                            double* logp, void* stream) {
    if (!mu || !rho || !eps || !w || !logq || !logp) return qb_fail("NULL argument to qb_vi_sample");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == QB_F64)
        k_vi_sample<double><<<(unsigned)nsam, 256, 0, st>>>((const double*)mu, (const double*)rho, (double*)eps, nsam, P, pi, sigma1, sigma2, seed, step, (double*)w, logq, logp);
    else
        k_vi_sample<float><<<(unsigned)nsam, 256, 0, st>>>((const float*)mu, (const float*)rho, (float*)eps, nsam, P, pi, sigma1, sigma2, seed, step, (float*)w, logq, logp);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

extern "C" int qb_vi_backward(int dtype, const void* mu, const void* rho, const void* eps, const void* w, const void* glp,
                              int64_t nsam, int64_t P, double pi, double sigma1, double sigma2, double c_ssq,
                              double c_logp, double c_logq, void* gmu, void* grho, void* stream) {
    if (!mu || !rho || !eps || !w || !glp || !gmu || !grho) return qb_fail("NULL argument to qb_vi_backward");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)cdiv(P, 32);
    if (dtype == QB_F64)
        k_vi_backward<double><<<blocks, 256, 0, st>>>((const double*)mu, (const double*)rho, (const double*)eps, (const double*)w, (const double*)glp, nsam, P, pi, sigma1, sigma2, c_ssq, c_logp, c_logq, (double*)gmu, (double*)grho);
    else
        k_vi_backward<float><<<blocks, 256, 0, st>>>((const float*)mu, (const float*)rho, (const float*)eps, (const float*)w, (const float*)glp, nsam, P, pi, sigma1, sigma2, c_ssq, c_logp, c_logq, (float*)gmu, (float*)grho);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

// =================================================================================================
// SWAG: SGD step with snapshot moments, and the posterior draws (qb_swag.cuh)
// =================================================================================================
#include "qb_swag.cuh"

extern "C" int qb_swag_step(int dtype, void* theta, const void* grad, int64_t K, int64_t P, double lr, double grad_scale,
                            int64_t n_snap, double* mean, double* m2, void* dev, int64_t k, void* stream) {
    if (!theta || !grad) return qb_fail("NULL argument to qb_swag_step");
    if (K < 1 || P < 1) return qb_fail("qb_swag_step needs K >= 1 and P >= 1");
    if (n_snap < 0) return qb_fail("n_snap must not be negative");
    if (n_snap > 0 && (!mean || !m2 || !dev)) return qb_fail("NULL argument to qb_swag_step (a snapshot needs mean, m2 and dev)");
    if (n_snap > 0 && k < 1) return qb_fail("a snapshot needs k >= 1 deviation columns");
    const long long n = (long long)K * P;
    const unsigned blocks = (unsigned)cdiv(n, 256);
    const double lrs = lr * grad_scale;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == QB_F64)
        k_swag_step<double><<<blocks, 256, 0, st>>>((double*)theta, (const double*)grad, n, P, lrs, n_snap, mean, m2, (double*)dev, k);
    else
        k_swag_step<float><<<blocks, 256, 0, st>>>((float*)theta, (const float*)grad, n, P, lrs, n_snap, mean, m2, (float*)dev, k);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

extern "C" int qb_swag_sample(int dtype, const double* mean, const double* m2, const void* dev, int64_t K, int64_t P,
                              int64_t k, int64_t n_snap, int lowrank, const int32_t* members, int64_t nsam, uint64_t seed,
                              int64_t sample_offset, double cov_scale, void* theta_out, void* stream) {
    if (!mean || !m2 || !members || !theta_out || (lowrank && !dev)) return qb_fail("NULL argument to qb_swag_sample");
    if (K < 1 || P < 1) return qb_fail("qb_swag_sample needs K >= 1 and P >= 1");
    if (nsam < 0 || sample_offset < 0) return qb_fail("nsam and sample_offset must not be negative");
    if (n_snap < 2) return qb_fail("qb_swag_sample needs n_snap >= 2 snapshots (got %s%lld)", "", (long long)n_snap);
    if (lowrank && k < 1) return qb_fail("the low-rank draw needs k >= 1 deviation columns");
    if (!(cov_scale >= 0.0)) return qb_fail("cov_scale must not be negative");
    const long long R = lowrank ? std::min<long long>(k, n_snap) : 0;
    if (lowrank && R < 2) return qb_fail("the low-rank draw needs R = min(k, n_snap) >= 2 (got %s%lld)", "", R);
    if (R > QB_SWAG_MAX_R) return qb_fail("the low-rank draw takes at most %s%lld deviation columns", "", (long long)QB_SWAG_MAX_R);
    if (nsam == 0) return 0;                  // no draws: no kernel
    if (nsam > 0x7FFFFFFFLL) return qb_fail("nsam exceeds the grid (%s%lld)", "", (long long)nsam);
    const double sc = sqrt(cov_scale);
    const double c1 = lowrank ? sc / sqrt(2.0) : sc;
    const double c2 = lowrank ? sc / sqrt(2.0 * (double)(R - 1)) : 0.0;
    const size_t smem = (size_t)R * sizeof(double);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == QB_F64)
        k_swag_sample<double><<<(unsigned)nsam, 256, smem, st>>>(mean, m2, (const double*)dev, P, k, n_snap, (int)R, members, seed, sample_offset, c1, c2, (double*)theta_out);
    else
        k_swag_sample<float><<<(unsigned)nsam, 256, smem, st>>>(mean, m2, (const float*)dev, P, k, n_snap, (int)R, members, seed, sample_offset, c1, c2, (float*)theta_out);
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    return 0;
}

// =================================================================================================
// FMA peak micro-benchmark (roofline denominator for the CUDA-core kernels)
// =================================================================================================
template <typename T, int CH>
__global__ void __launch_bounds__(256, 2) k_fma_peak(long long iters, T* sink) {
    T a[CH];
    const T b = T(1.0000001) + T(threadIdx.x) * T(1e-9), c = T(1e-7);
#pragma unroll
    for (int q = 0; q < CH; ++q) a[q] = T(q) * T(0.01) + T(threadIdx.x) * T(1e-6);
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int q = 0; q < CH; ++q) a[q] = fma(a[q], b, c);
    }
    T s = T(0);
#pragma unroll
    for (int q = 0; q < CH; ++q) s += a[q];
    if (s == T(123.456)) sink[0] = s;
}

// variant 2 (fp32 only): packed FFMA2 chains -- the Blackwell-specific way to issue FP32 FMAs
__global__ void __launch_bounds__(256, 2) k_fma2_peak(long long iters, float* sink) {
    float2 a[8];
    const float2 b = make_float2(1.0000001f + threadIdx.x * 1e-9f, 1.0000002f), c = make_float2(1e-7f, 2e-7f);
#pragma unroll
    for (int q = 0; q < 8; ++q) a[q] = make_float2(q * 0.01f + threadIdx.x * 1e-6f, q * 0.02f);
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int q = 0; q < 8; ++q) a[q] = __ffma2_rn(a[q], b, c);
    }
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += a[q].x + a[q].y;
    if (s == 123.456f) sink[0] = s;
}

extern "C" int qb_fma_peak(int dtype, int variant, int64_t iters, double* flops_out_host, void* sink, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = qb_num_sms() * 8, threads = 256;
    if (dtype == QB_F32 && variant == 2) {
        k_fma2_peak<<<blocks, threads, 0, st>>>(iters, (float*)sink);
        QB_CUDA(cudaGetLastError());
        g_launches += 1;
        if (flops_out_host) *flops_out_host = 2.0 * (double)blocks * threads * (double)iters * 8.0 * 8 * 2;
        return 0;
    }
    const int CH = variant == 1 ? 16 : 8;
    if (dtype == QB_F64) {
        if (variant == 1) k_fma_peak<double, 16><<<blocks, threads, 0, st>>>(iters, (double*)sink);
        else k_fma_peak<double, 8><<<blocks, threads, 0, st>>>(iters, (double*)sink);
    } else {
        if (variant == 1) k_fma_peak<float, 16><<<blocks, threads, 0, st>>>(iters, (float*)sink);
        else k_fma_peak<float, 8><<<blocks, threads, 0, st>>>(iters, (float*)sink);
    }
    QB_CUDA(cudaGetLastError());
    g_launches += 1;
    if (flops_out_host) *flops_out_host = 2.0 * (double)blocks * threads * (double)iters * 8.0 * CH;
    return 0;
}
