// Parallel tempering (replica exchange) for HMC / MALA: the tempered evaluation functor, the per-slot wrapper of
// qb_hmc_body the four k_pt_hmc* kernels share, and the deterministic even-odd swap round (Syed, Bouchard-Cote,
// Deligiannidis & Doucet, JRSSB 2022).
//
// K = T * G chains, slot-major: chain k = i * G + g is temperature slot i of group g and targets
// pi_i(theta) ~ exp(beta_i * lp(theta)), lp the log-posterior kernel 2 evaluates (likelihood and optional prior).
// Every lp, MAP value and gradient a chain keeps is its tempered one.
#pragma once
#include "qb_device.cuh"
#include "qb_chain.cuh"

enum { QB_STREAM_PT = 6 };

struct PtArgs {
    const double* beta;        // [T] device, beta[0] == 1, strictly decreasing, > 0 (validated by the caller)
    const double* eps;         // [T] device, the step size of each slot
    long long G;               // groups; slot of chain k is k / G
};

// beta * lp and beta * grad of an inner evaluation functor.  With beta == 1 every product is exact, so slot 0 computes
// bit for bit what the untempered chain computes.
template <typename T, typename Eval> struct QbTempered {
    Eval& inner; double beta; int P;
    __device__ __forceinline__ double operator()(const T* th, T* g) const {
        const double lp = inner(th, g);
        const T b = (T)beta;
        for (int i = threadIdx.x; i < P; i += blockDim.x) g[i] = qb_mul<T>(b, g[i]);
        __syncthreads();
        return beta * lp;
    }
};

// qb_hmc_body for chain blockIdx.x at its slot's beta and step size; draws are stored for the cold rows (k < G) only,
// into samples [G, n_slots, P].
template <typename T, typename Eval>
__device__ __forceinline__ void qb_pt_hmc_body(const ChainArgs<T>& c, const HmcArgs<T>& h, const PtArgs& a, int P, double* red,
                                               Eval& inner) {
    const long long k = blockIdx.x, slot = k / a.G;
    ChainArgs<T> cl = c;
    if (k >= a.G) cl.samples = nullptr;
    HmcArgs<T> hl = h;
    hl.eps = a.eps[slot];
    QbTempered<T, Eval> eval{inner, a.beta[slot], P};
    qb_hmc_body<T>(cl, hl, P, red, eval);
}

// One DEO swap round r of group blockIdx.x: the pairs (i, i+1) with i = r (mod 2).  Thread j decides pair j; then the
// block exchanges the theta and grad_cur rows of the accepted pairs.  With U = lp / beta (untempered), a pair is
// accepted when u < exp((beta_i - beta_{i+1}) (U_{i+1} - U_i)) (strict <, NaN rejects), u = word 0 of Philox
// (seed, chain_offset + k_i, r, QB_STREAM_PT, 0).  The lp and gradient that move from slot j to slot i are multiplied by
// beta_i / beta_j (in double, rounded once to T).  naccept and the MAP stay with their slot; replica [K] moves with the
// state, last_end [K] (by replica: +1 cold end, -1 hot end last visited) counts round trips hot -> cold.
struct PtSwapArgs {
    const double* beta; long long G; int T_;
    unsigned long long seed; long long chain_offset; long long r;
    double* lp; int* replica; signed char* last_end; long long* round_trips; long long* attempts; long long* accepts;
};

template <typename T>
__global__ void __launch_bounds__(256) k_pt_swap(const __grid_constant__ PtSwapArgs a, T* __restrict__ theta, T* __restrict__ gcur, int P) {
    extern __shared__ int acc_s[];
    const long long g = blockIdx.x, G = a.G;
    const int nt = a.T_, i0 = (int)(a.r & 1), npairs = (nt - i0) / 2;
    for (int j = threadIdx.x; j < npairs; j += blockDim.x) {
        const int i = i0 + 2 * j;
        const long long ka = i * G + g, kb = (i + 1) * G + g;
        const double ba = a.beta[i], bb = a.beta[i + 1];
        const double x = (ba - bb) * (a.lp[kb] / bb - a.lp[ka] / ba);
        const double u = qb_u01(qb_rand4(a.seed, a.chain_offset + ka, a.r, QB_STREAM_PT, 0).x);
        const bool acc = u < exp(x);
        acc_s[j] = acc ? 1 : 0;
        a.attempts[g * (nt - 1) + i] += 1;
        if (acc) {
            a.accepts[g * (nt - 1) + i] += 1;
            const double la = a.lp[ka], lb = a.lp[kb];
            a.lp[ka] = lb * (ba / bb);
            a.lp[kb] = la * (bb / ba);
            const int ra = a.replica[ka];
            a.replica[ka] = a.replica[kb];
            a.replica[kb] = ra;
        }
    }
    __syncthreads();
    for (int j = 0; j < npairs; ++j) {
        if (!acc_s[j]) continue;
        const int i = i0 + 2 * j;
        const long long ka = i * G + g, kb = (i + 1) * G + g;
        const double up = a.beta[i] / a.beta[i + 1], down = a.beta[i + 1] / a.beta[i];
        T* ta = theta + ka * P; T* tb = theta + kb * P;
        T* ga = gcur + ka * P; T* gb = gcur + kb * P;
        for (int e = threadIdx.x; e < P; e += blockDim.x) {
            const T t0 = ta[e]; ta[e] = tb[e]; tb[e] = t0;
            const T g0 = ga[e];
            ga[e] = (T)((double)gb[e] * up);
            gb[e] = (T)((double)g0 * down);
        }
    }
    if (threadIdx.x == 0 && nt > 1) {
        a.last_end[a.replica[(nt - 1) * G + g]] = -1;
        const int rc = a.replica[g];
        if (a.last_end[rc] == -1) { a.last_end[rc] = 1; a.round_trips[g] += 1; }
    }
}
