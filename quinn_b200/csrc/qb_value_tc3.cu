// quinn_b200: kernel 1 and the AMCMC chain kernel for the hot shape (in <= 7 -> 64 -> 64 -> 1, tanh, fp32) on the
// warp-specialised tensor-core value path (device code: qb_tc3.cuh).  Separate translation unit: it compiles in
// parallel with qb_kernels.cu and keeps the register allocation of the hot loops away from every other variant.
//
// The chain kernel keeps the chain's state IN SHARED MEMORY for the whole launch (current point, proposal, proposal
// scales: 3 P floats next to the staged operands) -- one chain-step is then
//   per-element phase (Haario moments streamed through global memory, proposal scale, Philox proposal: every thread
//   owns the same groups of 4 consecutive parameters in every phase, so no block barrier separates them)
//   -> staging of the proposal from shared memory -> 79 tiles on the tensor cores -> accept (shared-memory copy)
// and nothing on the step's critical path waits for a global-memory round trip.  The generic kernel (qb_kernels.cu,
// k_amcmc) moved every array through global memory between phases: ~27 us of a 183 us step at config 5.
// Semantics are those of qb_amcmc_pre / qb_amcmc_post / qb_mh_step (admcmc.py:52-70, mcmc.py:55-85), same arithmetic
// in the same order: replays and Philox runs give the decisions of the generic kernel.
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>

#include "quinn_b200.h"
#include "qb_plan.h"
#include "qb_device.cuh"
#include "qb_chain.cuh"
#include "qb_tc.cuh"
#include "qb_tc3.cuh"
#include "qb_value_tc3.h"

// x[N, in] -> operand tiles: tile u = points 128u .. 128u+127 as [hi 128 K0 floats | lo 128 K0 floats], element (m, k) at
// ((m/8)*(K0/4) + k/4)*32 + (m%8)*4 + k%4; k < in: x, k == in: 1 (the bias slot), else 0; rows past N: zeros (never used)
template <int K0>
__global__ void __launch_bounds__(128) k_tc3_xsplit(const float* __restrict__ x, long long N, int in_dim, float* __restrict__ out) {
    const long long u = blockIdx.x, p = u * 128 + threadIdx.x;
    const int m = threadIdx.x;
    float* hi = out + u * (2 * 128 * K0);
    float* lo = hi + 128 * K0;
#pragma unroll
    for (int k = 0; k < K0; ++k) {
        float w = 0.0f;
        if (k < in_dim && p < N) w = x[p * in_dim + k];
        if (k == in_dim) w = 1.0f;
        const float h = qb_tf32_hi(w);
        const int idx = ((m >> 3) * (K0 / 4) + (k >> 2)) * 32 + (m & 7) * 4 + (k & 3);
        hi[idx] = h; lo[idx] = w - h;
    }
}

// kernel-end drain of the issue warp: x tiles requested for a next evaluation that never came
__device__ __forceinline__ void qb_tc3_drain(const QbTcPlan& tp, const QbTcCtx& cx, unsigned char* smem, long long N, bool bulk) {
    if ((threadIdx.x >> 5) == 8 && cx.phase && bulk) {
        const int T = (int)((N + 127) / 128);
        for (int u = 0; u < 3 && u < T; ++u)
            qb_mbar_wait_timed(qb_smem_u32(smem) + (uint32_t)tp.v3_xbar + 8u * u, (cx.hphase >> u) & 1u);
    }
}

// the tile loop out of line: the chain kernel's own state stays out of the loop's register allocation
static __device__ __noinline__ double qb_tc3_eval_chain(const QbTcPlan& tp, QbTcCtx& cx, unsigned char* smem, const float* __restrict__ x,
                                                        const float* __restrict__ y, long long N, const float* __restrict__ xs) {
    QbTcCtx c2 = cx;
    const double r = qb_tc3_eval_any<64, true>(tp, c2, smem, x, y, 0, N, xs);
    cx.phase = c2.phase; cx.hphase = c2.hphase;
    return r;
}

template <int H>
__global__ void __launch_bounds__(Qb3Dim<H>::NCOMP + 32, H == 64 ? 2 : 1) k_logpost_tc3(const __grid_constant__ QbTcPlan tp, const EvalArgs<float> a) {
    extern __shared__ __align__(128) unsigned char smem_tc[];
    QbTcCtx cx;
    const long long k = blockIdx.x, s = blockIdx.y;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    qb_tc3_init<H>(tp, smem_tc, cx);
#ifdef QB3_TRACE
    if (threadIdx.x == 0 && blockIdx.x < QB3_TR_BLOCKS && blockIdx.y == 0) { unsigned int id; asm("mov.u32 %0, %%smid;" : "=r"(id)); qb3_trace_sm[blockIdx.x] = id; }
#endif
    qb_tc3_stage<H, Qb3K0<H>::value>(tp, smem_tc, a.theta + k * tp.n_params, -1.0f);
    const float* xs = a.xsplit ? a.xsplit + (n0 >> 7) * (2 * 128 * Qb3K0<H>::value) : nullptr;
    const double ssq = qb_tc3_eval_any<H, false>(tp, cx, smem_tc, a.x + k * a.xs, a.y + k * a.ys, n0, n1, xs);
    if (threadIdx.x == 0) a.part[k * a.S + s] = ssq;
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

__global__ void __launch_bounds__(288, 2)
k_amcmc_tc3(const __grid_constant__ QbTcPlan tp, const __grid_constant__ ChainArgs<float> c, const __grid_constant__ AmcmcArgs<float> a,
            const float* __restrict__ xs) {
    extern __shared__ __align__(128) unsigned char smem[];
    QbTcCtx cx;
    QB3_STAMP(80, 0);
    qb_tc3_init<64>(tp, smem, cx);
    QB3_STAMP(80, 1);
#ifdef QB3_TRACE
    if (threadIdx.x == 0 && blockIdx.x < QB3_TR_BLOCKS) { unsigned int id; asm("mov.u32 %0, %%smid;" : "=r"(id)); qb3_trace_sm[blockIdx.x] = id; }
#endif
    double* red = reinterpret_cast<double*>(smem);
    const long long k = blockIdx.x;
    const int P = tp.n_params, Pp = (P + 3) & ~3, tid = threadIdx.x, nt = blockDim.x;
    float* cur_s = reinterpret_cast<float*>(smem + tp.v3_state);
    float* prop_s = cur_s + Pp;
    float* ps_s = prop_s + Pp;
    float* curg = c.theta + k * P;
    float* mapth = c.map_theta + k * P;
    float* psg = a.pscale + k * P;
    float* xm = a.xm ? a.xm + k * P : nullptr;
    float* cov = a.cov ? a.cov + k * (long long)P : nullptr;           // diagonal: this kernel never sees track == 2
    const bool replay = c.rng_mode == QB_RNG_REPLAY;
    const long long chain = c.chain_offset + k;

    for (int i = tid; i < P; i += nt) { cur_s[i] = curg[i]; ps_s[i] = psg[i]; }
    double lp_cur = 0.0, map_lp = 0.0;
    long long na = 0;
    if (!c.init_lp) { lp_cur = c.lp[k]; map_lp = c.map_lp[k]; na = c.naccept[k]; }
    int kind = a.prop_kind[k];
    __syncthreads();
    QB3_STAMP(80, 2);

    for (long long s = c.init_lp ? -1 : 0; s < c.nsteps; ++s) {
        const float* evalp = cur_s;
        float wmax = -1.0f;                        // largest |W1| entry of the proposal seen by this thread (< 0: not computed)
        QB3_STAMP(81, 0);
        if (s >= 0) {
            // ---- running moments (admcmc.py:52-59), proposal scale (61-67), proposal (70): one pass, thread-owned elements
            const long long t = c.t_start + s;
            const bool first = t == 0;
            const bool adapt_now = !first && a.adapt != QB_ADAPT_NONE && t > a.t0 && (t % a.tadapt) == 0;
            if (first) kind = 0; else if (adapt_now) kind = 1;
            const bool track = a.track && xm;
            const double td = (double)t;
            const float rt = (float)((td - 1.0) / td), st = (float)((td + 1.0) / (td * td));
            const float tdf = (float)td, td1 = (float)(td + 1.0);
            const double fac = a.gamma * 2.4 * 2.4 / (double)P;
            float z0 = 0.0f;
            if (!replay && kind == 0) { float zz[4]; qb_normal4(qb_rand4(c.seed, chain, t, QB_STREAM_Z0, 0), zz); z0 = 0.1f * zz[0]; }
            const float* xi = replay ? c.incr + (s * c.K + k) * P : nullptr;
            // the thread's moments first: all global loads of the step are in flight together (one round trip, not one
            // per element; the stores below could alias them, so the compiler would not hoist them on its own)
            constexpr int JMAX = 5;                      // groups of 4 per thread: P <= 4 * 288 * 5
            float xmv[JMAX][4], cvv[JMAX][4];
            const bool ldm = track && !first, ldc = cov && (ldm || (!track && adapt_now));
#pragma unroll
            for (int j = 0; j < JMAX; ++j) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = (tid + j * nt) * 4 + q;
                    xmv[j][q] = (ldm && i < P) ? xm[i] : 0.0f;
                    cvv[j][q] = (ldc && i < P) ? cov[i] : 0.0f;
                }
            }
            const int w1lo = tp.L[1].w_off, w1hi = w1lo + 64 * 64;
            QB3_STAMP(81, 5);
#pragma unroll
            for (int j = 0; j < JMAX; ++j) {
                const int i4 = tid + j * nt;
                if (j == 1) QB3_STAMP(81, 6);
                if (j == 2) QB3_STAMP(81, 7);
                if (i4 * 4 < P) {
                    float z[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                    if (!replay) qb_normal4(qb_rand4(c.seed, chain, t, QB_STREAM_INCR, (uint32_t)i4), z);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < P) {
                            const float cu = cur_s[i];
                            float cv = cvv[j][q];
                            if (track) {
                                if (first) {
                                    xm[i] = cu;
                                    if (cov) cov[i] = 0.0f;
                                } else {
                                    const float m = qb_add<float>(qb_mul<float>(tdf, xmv[j][q]), cu) / td1;
                                    xm[i] = m;
                                    if (cov) {
                                        const float d = cu - m;
                                        cv = qb_add<float>(qb_mul<float>(rt, cv), qb_mul<float>(st, qb_mul<float>(d, d)));
                                        cov[i] = cv;
                                    }
                                }
                            }
                            float ps = ps_s[i];
                            if (first) { ps = (float)sqrt(0.09 * fabs((double)cu)); ps_s[i] = ps; }
                            else if (adapt_now) { ps = (float)sqrt(fac * ((double)cv + 1e-8)); ps_s[i] = ps; }
                            const float pr = replay ? qb_add<float>(cu, xi[i]) : cu + (z0 + ps * z[q]);
                            prop_s[i] = pr;
                            if (i >= w1lo && i < w1hi) wmax = fmaxf(wmax, fabsf(pr));
                        }
                    }
                }
            }
            wmax = fmaxf(wmax, 0.0f);             // every thread has looked at its share of W1
            evalp = prop_s;
        }
        // ---- evaluate
        QB3_STAMP(81, 1);
        __syncthreads();                           // the proposal is complete in shared memory
        qb_tc3_stage<64, 8>(tp, smem, evalp, wmax);
        QB3_STAMP(81, 2);
        const double ssq = qb_tc3_eval_chain(tp, cx, smem, c.x, c.y, c.N, xs);
        QB3_STAMP(81, 3);
        double pss = 0.0;
        if (c.lk.has_prior) pss = qb_prior_ss<float>(c.lk, evalp, k, P, red);
        const double lp_prop = qb_lp_from(c.lk, ssq, c.N, pss, P);
        // ---- accept / reject and bookkeeping (mcmc.py:55-61 for the initial state, 69-85 per step)
        if (s < 0) {
            lp_cur = lp_prop; map_lp = lp_prop; na = 0;
            if (tid == 0 && c.rec_lp0) c.rec_lp0[k] = lp_prop;
            for (int i = tid; i < P; i += nt) mapth[i] = cur_s[i];
        } else {
            const double mh = exp(lp_prop - lp_cur);                      // exp(cur_H - prop_H), unclipped; inf is normal
            double u;
            if (replay) u = c.unif[s * c.K + k];
            else u = qb_u01(qb_rand4(c.seed, chain, c.t_start + s, QB_STREAM_UNIF, 0).x);
            const bool acc = u < mh;                                      // strict <, NaN rejects
            if (acc) {
                lp_cur = lp_prop;
                na += 1;
                const bool newmap = lp_cur >= map_lp;
                if (newmap) map_lp = lp_cur;
                for (int i4 = tid; i4 * 4 < P; i4 += nt) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < P) { const float v = prop_s[i]; cur_s[i] = v; if (newmap) mapth[i] = v; }
                    }
                }
            }
            if (tid == 0) {
                if (c.rec_lp) c.rec_lp[k * c.rec_ld + s] = lp_cur;
                if (c.rec_alpha) c.rec_alpha[k * c.rec_ld + s] = mh;
                if (c.rec_acc) c.rec_acc[k * c.rec_ld + s] = acc ? 1 : 0;
            }
            if (c.samples && c.store_every > 0 && (s + 1) % c.store_every == 0) {
                const long long slot = (s + 1) / c.store_every - 1;
                if (slot < c.n_slots) {
                    __syncthreads();
                    float* dst = c.samples + (k * c.n_slots + slot) * P;
                    for (int i = tid; i < P; i += nt) dst[i] = cur_s[i];
                }
            }
        }
    }
    QB3_STAMP(81, 4);
    qb_tc3_drain(tp, cx, smem, c.N, xs != nullptr);
    __syncthreads();
    for (int i = tid; i < P; i += nt) { curg[i] = cur_s[i]; psg[i] = ps_s[i]; }
    if (tid == 0) { c.lp[k] = lp_cur; c.map_lp[k] = map_lp; c.naccept[k] = na; a.prop_kind[k] = kind; }
    QB3_STAMP(80, 3);
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

#ifdef QB3_TRACE
// development aid: copy the phase stamps of the last launches to the host
extern "C" int qb_tc3_trace_dump(unsigned int* buf, unsigned int* sm) {
    if (cudaMemcpyFromSymbol(buf, qb3_trace_buf, sizeof(unsigned int) * QB3_TR_BLOCKS * QB3_TR_WARPS * QB3_TR_TILES * QB3_TR_EV) != cudaSuccess) return -1;
    if (cudaMemcpyFromSymbol(sm, qb3_trace_sm, sizeof(unsigned int) * QB3_TR_BLOCKS) != cudaSuccess) return -1;
    return 0;
}
#endif

// kernel 4: network outputs of member blockIdx.x over its chunk of tiles -> out[m, p] (one output per point)
template <int H>
__global__ void __launch_bounds__(Qb3Dim<H>::NCOMP + 32, H == 64 ? 2 : 1)
k_predict_tc3(const __grid_constant__ QbTcPlan tp, const float* __restrict__ theta, const float* __restrict__ x, long long N,
              float* __restrict__ out, long long tiles_per_block) {
    extern __shared__ __align__(128) unsigned char smem_tc[];
    QbTcCtx cx;
    const long long m = blockIdx.x;
    const long long n0 = (long long)blockIdx.y * tiles_per_block * 128, n1 = min(N, n0 + tiles_per_block * 128);
    qb_tc3_init<H>(tp, smem_tc, cx);
#ifdef QB3_TRACE
    if (threadIdx.x == 0 && blockIdx.x < QB3_TR_BLOCKS && blockIdx.y == 0) { unsigned int id; asm("mov.u32 %0, %%smid;" : "=r"(id)); qb3_trace_sm[blockIdx.x] = id; }
#endif
    qb_tc3_stage<H, Qb3K0<H>::value>(tp, smem_tc, theta + m * tp.n_params, -1.0f);
    Qb3SinkStore sink;
    sink.out = out + m * N;
    qb_tc3_dispatch<H, false>(tp, cx, smem_tc, x, n0, n1, nullptr, sink);
    qb_tc_stop(cx.tmem, (uint32_t)tp.tmem_cols);
}

cudaError_t qb_tc3_launch_logpost(const QbTcPlan& tp, const EvalArgs<float>& a, dim3 grid, cudaStream_t st) {
    const unsigned nt = (unsigned)((a.N + 127) / 128);
    cudaError_t e;
    if (tp.v3 == 1) {
        e = cudaFuncSetAttribute(k_logpost_tc3<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
        if (e != cudaSuccess) return e;
        if (a.xsplit) k_tc3_xsplit<8><<<nt, 128, 0, st>>>(a.x, a.N, tp.in_dim, const_cast<float*>(a.xsplit));
        k_logpost_tc3<64><<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, a);
    } else {
        e = cudaFuncSetAttribute(k_logpost_tc3<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
        if (e != cudaSuccess) return e;
        if (a.xsplit) k_tc3_xsplit<16><<<nt, 128, 0, st>>>(a.x, a.N, tp.in_dim, const_cast<float*>(a.xsplit));
        k_logpost_tc3<128><<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, a);
    }
    return cudaGetLastError();
}

cudaError_t qb_tc3_launch_predict(const QbTcPlan& tp, const float* theta, const float* x, long long N, float* out,
                                  long long tiles_per_block, dim3 grid, cudaStream_t st) {
    cudaError_t e;
    if (tp.v3 == 1) {
        e = cudaFuncSetAttribute(k_predict_tc3<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
        if (e != cudaSuccess) return e;
        k_predict_tc3<64><<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, theta, x, N, out, tiles_per_block);
    } else {
        e = cudaFuncSetAttribute(k_predict_tc3<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
        if (e != cudaSuccess) return e;
        k_predict_tc3<128><<<grid, tp.nthreads, tp.smem_bytes, st>>>(tp, theta, x, N, out, tiles_per_block);
    }
    return cudaGetLastError();
}

cudaError_t qb_tc3_launch_amcmc(const QbTcPlan& tp, const ChainArgs<float>& c, const AmcmcArgs<float>& a, long long K, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(k_amcmc_tc3, cudaFuncAttributeMaxDynamicSharedMemorySize, tp.smem_bytes);
    if (e != cudaSuccess) return e;
    // the generic kernel's proposal scratch ([K,P] floats) is free here: it holds the x tiles when it is large enough
    float* xs = nullptr;
    if ((size_t)K * (size_t)tp.n_params * sizeof(float) >= qb_tc3_xsplit_bytes(c.N, 8)) {
        xs = a.prop;
        k_tc3_xsplit<8><<<(unsigned)((c.N + 127) / 128), 128, 0, st>>>(c.x, c.N, tp.in_dim, xs);
    }
    k_amcmc_tc3<<<(unsigned)K, tp.nthreads, tp.smem_bytes, st>>>(tp, c, a, xs);
    return cudaGetLastError();
}
