// quinn_b200: kernel 2 (log-posterior + gradient) and the HMC / MALA chain kernel on the tensor cores with fp16-split
// operands (widths 64 and 128: configs 3 / 4 / 5).  Device code: qb_tg8.cuh.  Separate translation unit so that it compiles
// in parallel with the others.
#include <cuda_runtime.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <utility>

#include "quinn_b200.h"
#include "qb_plan.h"
#include "qb_device.cuh"
#include "qb_chain.cuh"
#include "qb_nuts.cuh"
#include "qb_pt.cuh"
#include "qb_tc.cuh"
#include "qb_tg8.cuh"
#include "qb_grad_tc128.h"
#include "qb_launch.h"

bool qb_tg8_make_plan(const qb_net_t* net, int dtype, QbTg8Plan* tp) {
    memset(tp, 0, sizeof(*tp));
    if (dtype != QB_F32 || qb_env_int("QB_NO_TC", 0) || qb_env_int("QB_NO_TCG", 0) || qb_env_int("QB_NO_TG8", 0)) return false;
    if (net->n_layers != 3 || net->in_dim > 15 || net->out_dim != 1 || net->final_exp) return false;
    const qb_layer_t& L0 = net->layers[0];
    const qb_layer_t& L1 = net->layers[1];
    const qb_layer_t& L2 = net->layers[2];
    if (L0.res_step != 0.0 || L1.res_step != 0.0 || L2.res_step != 0.0) return false;
    if (L0.n_terms > 1 || L1.n_terms > 1 || L2.n_terms > 1) return false;
    const int HR = L0.n_out;
    if ((HR != 128 && HR != 64 && HR != 32) || L1.n_out != HR) return false;
    if (HR <= 64 && !qb_env_int("QB_TG8_64", 1)) return false;
    const int H = HR == 32 ? 64 : HR;                        // 32-wide nets: zero-padded units on the 64-wide instance
    if (L0.act != QB_ACT_TANH || L1.act != QB_ACT_TANH || L2.act != QB_ACT_IDENTITY) return false;
    tp->in_dim = net->in_dim; tp->n_params = net->n_params; tp->h = H; tp->hr = HR;
    tp->w0_off = L0.w_off; tp->b0_off = L0.b_off; tp->w1_off = L1.w_off; tp->b1_off = L1.b_off;
    tp->wl_off = L2.w_off; tp->bl_off = L2.b_off;
    const int img = 256 * H;
    int off = QB_TG8_HDR;
    tp->w_img = off; off += 2 * (2 * H * H);
    tp->w0_img = off; off += 2 * (32 * H);
    tp->a_img = off; off += (img + 4096) + img;             // hi image + ones block | lo image
    tp->z_img = off; off += 2 * img;
    tp->x_img = off; off += 4 * QB_TG8_XIMG;                // a0, z, X images are contiguous (scratch of the final reduction)
    tp->fl_base = off;
    int f = 0;
    tp->b1 = f; f += H;
    tp->wl = f; f += H;
    tp->bl = f; f += 4;
    tp->sc = f; f += 8;
    off += f * 4;
    off = (off + 15) / 16 * 16;
    tp->ybuf = off; off += (H / 32) * 128 * 4;
    const int cols = 3 * H + 32;
    tp->tmem_cols = cols <= 256 ? 256 : 512;
    tp->nthreads = 4 * H + 32;
    if (off > QB_SMEM_MAX) return false;
    tp->smem_bytes = (int)std::min<long long>(QB_SMEM_MAX, std::max<long long>(off, qb_tmem_smem_floor(tp->tmem_cols)));
    return true;
}

// max |x|, max |y| as float bit patterns (non-negative floats order like unsigned integers)
__global__ void __launch_bounds__(256) k_tg8_absmax(const float* __restrict__ x, long long nx, const float* __restrict__ y, long long ny,
                                                    unsigned int* out) {
    float mx = 0.0f, my = 0.0f;
    const long long stride = (long long)gridDim.x * blockDim.x, i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long i = i0; i < nx; i += stride) mx = fmaxf(mx, fabsf(__ldg(x + i)));
    for (long long i = i0; i < ny; i += stride) my = fmaxf(my, fabsf(__ldg(y + i)));
    unsigned int ux = __reduce_max_sync(0xffffffffu, __float_as_uint(mx)), uy = __reduce_max_sync(0xffffffffu, __float_as_uint(my));
    if ((threadIdx.x & 31) == 0) {
        if (ux) atomicMax(out, ux);
        if (uy) atomicMax(out + 1, uy);
    }
}
static cudaError_t tg8_absmax(const float* x, long long nx, const float* y, long long ny, void* scratch, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(scratch, 0, 8, st);
    if (e != cudaSuccess) return e;
    const int blocks = (int)std::max<long long>(1, std::min<long long>(1184, (std::max(nx, ny) + 255) / 256));
    k_tg8_absmax<<<blocks, 256, 0, st>>>(x, nx, y, ny, (unsigned int*)scratch);
    return cudaGetLastError();
}

template <int H>
__global__ void __launch_bounds__(4 * H + 32, H == 64 ? 2 : 1) k_logpost_grad_tc128(const __grid_constant__ QbTg8Plan tp, const EvalArgs<float> a,
                                                                                    const float* __restrict__ absmax) {
    extern __shared__ __align__(1024) unsigned char smem_g[];
    const uint32_t tmem = qb_tg8_init<H>(tp, smem_g);
    const long long k = blockIdx.x, s = blockIdx.y;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    float* g = (a.S == 1) ? a.grad + k * tp.n_params : a.gpart + (k * a.S + s) * tp.n_params;
    const float is2 = (float)a.lk.inv_sigma2;
    qb_tg8_stage<H>(tp, smem_g, a.theta + k * tp.n_params, absmax, is2);
    const double ssq = qb_tg8_eval<H>(tp, tmem, smem_g, a.x + k * a.xs, a.y + k * a.ys, n0, n1, is2, g);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
    qb_tc_stop(tmem, (uint32_t)tp.tmem_cols);
}

template <int H> struct QbGradTg8 {
    const QbTg8Plan& tp; uint32_t tmem; unsigned char* smem; const ChainArgs<float>& c; const float* absmax; long long k;
    __device__ __forceinline__ double operator()(const float* th, float* g) const {
        const int P = tp.n_params;
        double* red = reinterpret_cast<double*>(smem);
        const float is2 = (float)c.lk.inv_sigma2;
        __syncthreads();
        qb_tg8_stage<H>(tp, smem, th, absmax, is2);
        const double ssq = qb_tg8_eval<H>(tp, tmem, smem, c.x, c.y, 0, c.N, is2, g);
        double pss = 0.0;
        if (c.lk.has_prior) {
            pss = qb_prior_ss<float>(c.lk, th, k, P, red);
            qb_prior_grad_add<float>(c.lk, th, k, P, g);
        }
        __syncthreads();
        return qb_lp_from(c.lk, ssq, c.N, pss, P);
    }
};

template <int H>
__global__ void __launch_bounds__(4 * H + 32, H == 64 ? 2 : 1) k_hmc_tc128(const __grid_constant__ QbTg8Plan tp, const __grid_constant__ ChainArgs<float> c,
                                                                           const __grid_constant__ HmcArgs<float> h, const float* __restrict__ absmax) {
    extern __shared__ __align__(1024) unsigned char smem_g[];
    const uint32_t tmem = qb_tg8_init<H>(tp, smem_g);
    QbGradTg8<H> eval{tp, tmem, smem_g, c, absmax, (long long)blockIdx.x};
    qb_hmc_body<float>(c, h, tp.n_params, reinterpret_cast<double*>(smem_g), eval);
    qb_tc_stop(tmem, (uint32_t)tp.tmem_cols);
}

template <int H>
__global__ void __launch_bounds__(4 * H + 32, 1) k_nuts_tc128(const __grid_constant__ QbTg8Plan tp, const __grid_constant__ ChainArgs<float> c,
                                                                            const __grid_constant__ NutsArgs<float> a, const float* __restrict__ absmax) {
    extern __shared__ __align__(1024) unsigned char smem_g[];
    const uint32_t tmem = qb_tg8_init<H>(tp, smem_g);
    QbGradTg8<H> eval{tp, tmem, smem_g, c, absmax, (long long)blockIdx.x};
    qb_nuts_body<float>(c, a, tp.n_params, reinterpret_cast<double*>(smem_g), eval);
    qb_tc_stop(tmem, (uint32_t)tp.tmem_cols);
}

// parallel-tempering twin of k_hmc_tc128 (qb_pt.cuh)
template <int H>
__global__ void __launch_bounds__(4 * H + 32, H == 64 ? 2 : 1) k_pt_hmc_tc128(const __grid_constant__ QbTg8Plan tp, const __grid_constant__ ChainArgs<float> c,
                                                                              const __grid_constant__ HmcArgs<float> h, const __grid_constant__ PtArgs a,
                                                                              const float* __restrict__ absmax) {
    extern __shared__ __align__(1024) unsigned char smem_g[];
    const uint32_t tmem = qb_tg8_init<H>(tp, smem_g);
    QbGradTg8<H> inner{tp, tmem, smem_g, c, absmax, (long long)blockIdx.x};
    qb_pt_hmc_body<float>(c, h, a, tp.n_params, reinterpret_cast<double*>(smem_g), inner);
    qb_tc_stop(tmem, (uint32_t)tp.tmem_cols);
}

template <int H>
static cudaError_t launch_eval_t(const QbTg8Plan& tp, const EvalArgs<float>& a, const float* absmax, dim3 grid, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_logpost_grad_tc128<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    k_logpost_grad_tc128<H><<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, a, absmax);
    return cudaGetLastError();
}
template <int H>
static cudaError_t launch_hmc_t(const QbTg8Plan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, const float* absmax,
                                cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_hmc_tc128<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    k_hmc_tc128<H><<<(unsigned)K, tp.nthreads, tp.smem_bytes, st>>>(tp, c, h, absmax);
    return cudaGetLastError();
}

template <int H>
static cudaError_t launch_nuts_t(const QbTg8Plan& tp, const ChainArgs<float>& c, const NutsArgs<float>& a, long long K, const float* absmax,
                                 cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_nuts_tc128<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    k_nuts_tc128<H><<<(unsigned)K, tp.nthreads, tp.smem_bytes, st>>>(tp, c, a, absmax);
    return cudaGetLastError();
}

template <int H>
static cudaError_t launch_pt_t(const QbTg8Plan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, const PtArgs& a, long long K,
                               const float* absmax, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_pt_hmc_tc128<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    k_pt_hmc_tc128<H><<<(unsigned)K, tp.nthreads, tp.smem_bytes, st>>>(tp, c, h, a, absmax);
    return cudaGetLastError();
}

cudaError_t qb_tg8_launch_eval(const QbTg8Plan& tp, const EvalArgs<float>& a, void* scratch, dim3 grid, cudaStream_t st) {
    // scales of the fp16 operand images need max |x| and max |y| of everything this launch reads
    const long long nx = (a.xs > 0 ? (a.K - 1) * a.xs : 0) + a.N * tp.in_dim, ny = (a.ys > 0 ? (a.K - 1) * a.ys : 0) + a.N;
    cudaError_t e = tg8_absmax(a.x, nx, a.y, ny, scratch, st);
    if (e != cudaSuccess) return e;
    if (tp.h == 64) return launch_eval_t<64>(tp, a, (const float*)scratch, grid, st);
    return launch_eval_t<128>(tp, a, (const float*)scratch, grid, st);
}

// 256 bytes of device memory per (device, stream) for max |x|, max |y| of a chain launch: allocated on first use and kept (a
// stream-ordered allocation per launch went back to the OS at every synchronisation and cost more than a 1024-chain step)
static void* tg8_stream_scratch(cudaStream_t st) {
    static std::mutex mu;
    static std::map<std::pair<int, cudaStream_t>, void*> pool;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    void*& p = pool[std::make_pair(dev, st)];
    if (!p && cudaMalloc(&p, QB_TG8_SCRATCH_BYTES) != cudaSuccess) p = nullptr;
    return p;
}

cudaError_t qb_tg8_launch_hmc(const QbTg8Plan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st) {
    void* scratch = tg8_stream_scratch(st);
    if (!scratch) return cudaErrorMemoryAllocation;
    cudaError_t e = tg8_absmax(c.x, c.N * tp.in_dim, c.y, c.N, scratch, st);
    if (e != cudaSuccess) return e;
    return tp.h == 64 ? launch_hmc_t<64>(tp, c, h, K, (const float*)scratch, st) : launch_hmc_t<128>(tp, c, h, K, (const float*)scratch, st);
}

cudaError_t qb_tg8_launch_nuts(const QbTg8Plan& tp, const ChainArgs<float>& c, const NutsArgs<float>& a, long long K, cudaStream_t st) {
    void* scratch = tg8_stream_scratch(st);
    if (!scratch) return cudaErrorMemoryAllocation;
    cudaError_t e = tg8_absmax(c.x, c.N * tp.in_dim, c.y, c.N, scratch, st);
    if (e != cudaSuccess) return e;
    return tp.h == 64 ? launch_nuts_t<64>(tp, c, a, K, (const float*)scratch, st) : launch_nuts_t<128>(tp, c, a, K, (const float*)scratch, st);
}

cudaError_t qb_tg8_pt_absmax(const QbTg8Plan& tp, const ChainArgs<float>& c, cudaStream_t st, const float** absmax) {
    void* scratch = tg8_stream_scratch(st);
    if (!scratch) return cudaErrorMemoryAllocation;
    *absmax = (const float*)scratch;
    return tg8_absmax(c.x, c.N * tp.in_dim, c.y, c.N, scratch, st);
}

cudaError_t qb_tg8_launch_pt(const QbTg8Plan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, const PtArgs& a, long long K,
                             const float* absmax, cudaStream_t st) {
    return tp.h == 64 ? launch_pt_t<64>(tp, c, h, a, K, absmax, st) : launch_pt_t<128>(tp, c, h, a, K, absmax, st);
}

#ifdef QB_TG8_TRACE
// development aid: copy the phase stamps of the last launch to the host
extern "C" int qb_tg8_trace_dump(unsigned int* buf) {
    return cudaMemcpyFromSymbol(buf, qb_tg8_trace_buf, sizeof(unsigned int) * QB_TG8_TR_BLOCKS * QB_TG8_TR_WARPS * QB_TG8_TR_TILES * QB_TG8_TR_EV) == cudaSuccess ? 0 : -1;
}
#endif
