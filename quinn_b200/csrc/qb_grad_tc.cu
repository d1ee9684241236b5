// quinn_b200: kernel 2 (log-posterior + gradient) and the HMC / MALA chain kernel on the tensor cores (tcgen05).
// Device code: qb_tcg.cuh.  Separate translation unit so that it compiles in parallel with qb_kernels.cu.
#include <cuda_runtime.h>
#include <string.h>
#include <algorithm>

#include "quinn_b200.h"
#include "qb_plan.h"
#include "qb_device.cuh"
#include "qb_chain.cuh"
#include "qb_tc.cuh"
#include "qb_tcg.cuh"
#include "qb_grad_tc.h"
#include "qb_launch.h"

bool qb_tcg_make_plan(const qb_net_t* net, int dtype, QbTcgPlan* tp) {
    memset(tp, 0, sizeof(*tp));
    if (dtype != QB_F32 || qb_env_int("QB_NO_TC", 0) || qb_env_int("QB_NO_TCG", 0)) return false;
    if (net->n_layers != 3 || net->in_dim > 7 || net->out_dim != 1 || net->final_exp) return false;
    const qb_layer_t& L0 = net->layers[0];
    const qb_layer_t& L1 = net->layers[1];
    const qb_layer_t& L2 = net->layers[2];
    if (L0.res_step != 0.0 || L1.res_step != 0.0 || L2.res_step != 0.0) return false;
    if (L0.n_terms > 1 || L1.n_terms > 1 || L2.n_terms > 1) return false;
    const int H = L0.n_out;
    if (L1.n_out != H || (H != 32 && H != 64)) return false;
    if (L0.act != L1.act || (L0.act != QB_ACT_TANH && L0.act != QB_ACT_RELU) || L2.act != QB_ACT_IDENTITY) return false;
    tp->in_dim = net->in_dim; tp->ni = net->in_dim <= 3 ? 4 : 8; tp->n_params = net->n_params;
    tp->h0 = H; tp->h1 = H; tp->act = L0.act;
    tp->G = H / 16; tp->nthreads = 128 * tp->G;
    tp->w0_off = L0.w_off; tp->b0_off = L0.b_off; tp->w1_off = L1.w_off; tp->b1_off = L1.b_off;
    tp->wl_off = L2.w_off; tp->bl_off = L2.b_off;
    int off = QB_TCG_HDR;
    tp->w1hi = off; off += H * H * 4;
    tp->w1lo = off; off += H * H * 4;
    tp->w1thi = off; off += H * H * 4;
    tp->w1tlo = off; off += H * H * 4;
    off = (off + 1023) / 1024 * 1024;
    const int atoms = (H + 31) / 32, sbo = 512 * atoms, pbytes = 32 * sbo;      // 128 points = 32 atoms of 4 points
    tp->a0_sbo = sbo; tp->z_sbo = sbo;
    tp->a0hi = off; off += pbytes;
    tp->a0lo = off; off += pbytes;
    tp->zhi = off; off += pbytes;
    tp->zlo = off; off += pbytes;
    off += 1024;            // M = 64 operands read (and ignore) one atom past the last row group
    tp->xt = off; off += 2 * QB_TCG_XT_TILE;
    tp->fl_base = off;
    int f = 0;
    tp->w0 = f; f += H * tp->ni;
    tp->b1 = f; f += H;
    tp->wl = f; f += H;
    tp->bl = f; f += 4;
    off += f * 4;
    off = (off + 15) / 16 * 16;
    tp->ybuf = off; off += tp->G * 128 * 4;
    tp->c_a0hi = 0; tp->c_a0lo = H; tp->c_zhi = 2 * H; tp->c_zlo = 3 * H; tp->c_d1 = 4 * H; tp->c_d0 = 5 * H;
    tp->c_dw1 = 6 * H; tp->c_db1 = 7 * H; tp->c_dw0 = 7 * H + 8;
    const int cols = 7 * H + 16;
    tp->tmem_cols = cols <= 256 ? 256 : 512;
    if (off > QB_SMEM_MAX) return false;
    tp->smem_bytes = (int)std::min<long long>(QB_SMEM_MAX, std::max<long long>(off, qb_tmem_smem_floor(tp->tmem_cols)));
    return true;
}

template <int H, int NI, int ACT>
__global__ void __launch_bounds__(H * 8, H == 32 ? 2 : 1) k_logpost_grad_tc(const __grid_constant__ QbTcgPlan tp, const EvalArgs<float> a) {
    extern __shared__ __align__(1024) unsigned char smem_g[];
    QbTcgCtx cx;
    qb_tcg_init(tp, smem_g, cx);
    const long long k = blockIdx.x, s = blockIdx.y;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    float* g = (a.S == 1) ? a.grad + k * tp.n_params : a.gpart + (k * a.S + s) * tp.n_params;
    qb_tcg_stage(tp, smem_g, a.theta + k * tp.n_params);
    const double ssq = qb_tcg_eval<H, NI, ACT>(tp, cx, smem_g, a.x + k * a.xs, a.y + k * a.ys, n0, n1, (float)a.lk.inv_sigma2, g);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

template <int H, int NI, int ACT> struct QbGradTc {
    const QbTcgPlan& tp; QbTcgCtx& cx; unsigned char* smem; const ChainArgs<float>& c; long long k;
    __device__ __forceinline__ double operator()(const float* th, float* g) const {
        const int P = tp.n_params;
        double* red = reinterpret_cast<double*>(smem);
        __syncthreads();
        qb_tcg_stage(tp, smem, th);
        const double ssq = qb_tcg_eval<H, NI, ACT>(tp, cx, smem, c.x, c.y, 0, c.N, (float)c.lk.inv_sigma2, g);
        double pss = 0.0;
        if (c.lk.has_prior) {
            pss = qb_prior_ss<float>(c.lk, th, k, P, red);
            qb_prior_grad_add<float>(c.lk, th, k, P, g);
        }
        __syncthreads();
        return qb_lp_from(c.lk, ssq, c.N, pss, P);
    }
};

template <int H, int NI, int ACT>
__global__ void __launch_bounds__(H * 8, H == 32 ? 2 : 1) k_hmc_tc(const __grid_constant__ QbTcgPlan tp, const __grid_constant__ ChainArgs<float> c,
                                                     const __grid_constant__ HmcArgs<float> h) {
    extern __shared__ __align__(1024) unsigned char smem_g[];
    QbTcgCtx cx;
    qb_tcg_init(tp, smem_g, cx);
    QbGradTc<H, NI, ACT> eval{tp, cx, smem_g, c, (long long)blockIdx.x};
    qb_hmc_body<float>(c, h, tp.n_params, reinterpret_cast<double*>(smem_g), eval);
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

template <int H, int NI, int ACT>
static cudaError_t launch_eval_t(const QbTcgPlan& tp, const EvalArgs<float>& a, dim3 grid, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_logpost_grad_tc<H, NI, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    k_logpost_grad_tc<H, NI, ACT><<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, a);
    return cudaGetLastError();
}
template <int H, int NI, int ACT>
static cudaError_t launch_hmc_t(const QbTcgPlan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_hmc_tc<H, NI, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    k_hmc_tc<H, NI, ACT><<<(unsigned)K, tp.nthreads, tp.smem_bytes, st>>>(tp, c, h);
    return cudaGetLastError();
}

#define QB_TCG_DISPATCH(FN, ...)                                                                          \
    do {                                                                                                  \
        const bool tanh_ = tp.act == QB_ACT_TANH;                                                         \
        if (tp.h0 == 64 && tp.ni == 4) return tanh_ ? FN<64, 4, QB_ACT_TANH>(__VA_ARGS__) : FN<64, 4, QB_ACT_RELU>(__VA_ARGS__); \
        if (tp.h0 == 64) return tanh_ ? FN<64, 8, QB_ACT_TANH>(__VA_ARGS__) : FN<64, 8, QB_ACT_RELU>(__VA_ARGS__);               \
        if (tp.ni == 4) return tanh_ ? FN<32, 4, QB_ACT_TANH>(__VA_ARGS__) : FN<32, 4, QB_ACT_RELU>(__VA_ARGS__);                \
        return tanh_ ? FN<32, 8, QB_ACT_TANH>(__VA_ARGS__) : FN<32, 8, QB_ACT_RELU>(__VA_ARGS__);                                \
    } while (0)

cudaError_t qb_tcg_launch_eval(const QbTcgPlan& tp, const EvalArgs<float>& a, dim3 grid, cudaStream_t st) {
    QB_TCG_DISPATCH(launch_eval_t, tp, a, grid, st);
}
cudaError_t qb_tcg_launch_hmc(const QbTcgPlan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st) {
    QB_TCG_DISPATCH(launch_hmc_t, tp, c, h, K, st);
}
