// No-U-Turn sampler (Hoffman & Gelman 2014), multinomial form (Betancourt 2017), with the iterative tree building of
// Phan, Pradhan & Jankowiak (2019) and per-chain dual-averaging step sizes (Hoffman & Gelman 2014 section 3.2, Stan's
// constants).  One thread block runs one chain for all its transitions; the identity metric is used.
//
// Transition t of chain k (global step t = t_start + s):
//   - momentum r0 ~ N(0, I) from QB_STREAM_INCR (as qb_hmc_body); H0 = -lp(z0) + |r0|^2 / 2; the tree is {z0}, weight 0.
//   - doubling j = 0, 1, ...: direction = bit 0 of word x of qb_rand4(seed, chain, t, QB_STREAM_NUTS, j) (1: forwards).
//     A subtree of 2^j leapfrog leaves grows from the tree's end in that direction.  Leaf n (counted over the whole
//     transition from 0) has weight w = H0 - H (H non-finite or lp non-finite: w = -inf) and joins the subtree's proposal
//     with probability exp(w - logaddexp(w_sub, w)) against word x of qb_rand4(..., QB_NUTS_LEAF0 + n) (uniform progressive
//     sampling; the subtree's first leaf is always taken).  The subtree stops early on a divergent leaf (H - H0 > 1000 or a
//     non-finite log-posterior) or on a U-turn of any of its power-of-two sub-subtrees ending at the new leaf, found
//     against the stored checkpoints (NumPyro's _iterative_build_subtree).  Then the subtree's proposal replaces the
//     tree's with probability min(1, exp(w_sub - w_tree)) against word y of the doubling's draw (biased progressive
//     sampling), 0 for a turning or divergent subtree.
//   - the tree stops on a divergence, a U-turn inside the new subtree or across the whole tree, or at max_depth doublings
//     (2^max_depth - 1 leapfrogs at most).
//   - U-turn of a trajectory with end momenta ra, rb and momentum sum rs: (rs - (ra + rb)/2) . ra <= 0 or ... . rb <= 0.
//   - acceptance statistic = mean over the new leaves of min(1, exp(H0 - H)); it drives the dual averaging while
//     t < n_adapt: m = t + 1, H_bar <- (1 - 1/(m+10)) H_bar + (target - stat)/(m+10), log eps = mu - sqrt(m) H_bar / 0.05,
//     log eps_bar <- m^-0.75 log eps + (1 - m^-0.75) log eps_bar, mu = log(10 eps0).  Transitions t < n_adapt use eps,
//     later ones eps_bar (n_adapt = 0: eps0 throughout).  init_lp resets log eps = log eps_bar = log eps0, H_bar = 0.
//
// Scratch per chain: (QB_NUTS_VECS + 2 max_depth) vectors of P elements, in this order: z, r, grad of the backward end;
// z, r, grad of the forward end; z and grad of the subtree's proposal; the running momentum sum of the tree and the
// growing subtree; max_depth checkpoint momenta; max_depth checkpoint running sums (a sub-subtree's momentum sum is the
// running sum at its last leaf minus the one at its first leaf plus that leaf's momentum).  The tree's proposal is kept in
// theta and grad_cur (the gradient at the current state, reused by the next transition).  Energies and dot products
// accumulate in double.
#pragma once
#include "qb_chain.cuh"

enum { QB_NUTS_MAX_DEPTH = 12, QB_NUTS_VECS = 9, QB_NUTS_LEAF0 = 16 };

template <typename T> struct NutsArgs {
    double eps0, target; int max_depth; long long n_adapt;
    double* log_eps; double* log_eps_bar; double* h_bar;    // [K] dual-averaging state
    T* gcur; T* scratch;
    int* rec_depth; int* rec_nleap; unsigned char* rec_div; double* rec_eps;    // [k * c.rec_ld + s], each optional
};

__device__ __forceinline__ double qb_logaddexp(double a, double b) {
    const double m = fmax(a, b);
    if (m == -INFINITY) return -INFINITY;
    return m + log1p(exp(-fabs(a - b)));
}

// U-turn test of the trajectory from checkpoint leaf (momentum rc, running momentum sum sc at that leaf) to the leaf with
// momentum r, where rs is the running momentum sum at r; rc == nullptr: the whole tree, ends ra / rb, sum rs.
template <typename T>
__device__ __forceinline__ bool qb_nuts_turning(const T* ra, const T* rb, const T* rs, const T* sc, int P, double* red) {
    double s1 = 0.0, s2 = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const double a = (double)ra[i], b = (double)rb[i];
        double sum = (double)rs[i];
        if (sc) sum = sum - (double)sc[i] + a;
        const double d = sum - (a + b) * 0.5;
        s1 += a * d;
        s2 += b * d;
    }
    s1 = qb_block_sum(s1, red);
    s2 = qb_block_sum(s2, red);
    return s1 <= 0.0 || s2 <= 0.0;
}

template <typename T>
__device__ __forceinline__ void qb_copy_vec(T* dst, const T* src, int P) {
    for (int i = threadIdx.x; i < P; i += blockDim.x) dst[i] = src[i];
}

// nsteps NUTS transitions of chain blockIdx.x.  `eval(theta, grad)` as in qb_hmc_body, called from ONE site: the loop
// below is a state machine whose every pass does one position update, one evaluation, then the momentum update and the
// tree bookkeeping (the pass with s == -1, only when init_lp, evaluates the incoming state instead).  Only the scalars
// of the transition in progress stay in registers across the evaluation; the chain's log-posterior, MAP and adaptation
// state are read and written in their [K] arrays (thread 0 writes, every thread reads after a barrier).
template <typename T, typename GradEval>
__device__ __forceinline__ void qb_nuts_body(const ChainArgs<T>& c, const NutsArgs<T>& a, int P, double* red, GradEval& eval) {
    const long long k = blockIdx.x, chain = c.chain_offset + k;
    const int tid = threadIdx.x, nt = blockDim.x, D = a.max_depth;
    T* cur = c.theta + k * P;
    T* gcur = a.gcur + k * P;
    T* w = a.scratch + k * (long long)(QB_NUTS_VECS + 2 * D) * P;     // zl rl gl | zr rr gr | zs gs | rsum | ck_r | ck_s
    T* rsum = w + 8 * P;
    T* ck_r = w + (long long)QB_NUTS_VECS * P;
    T* ck_s = ck_r + (long long)D * P;

    // the transition in progress (block-uniform: every thread holds the same values)
    double H0 = 0.0, w_tree = 0.0, w_sub = 0.0, lp_sub = 0.0, sum_acc = 0.0;
    int depth = 0, n_leap = 0, n_sub = 0;
    bool fwd = true, moved = false, begin = true;
    T e = T(0);

    for (long long s = c.init_lp ? -1 : 0; s < c.nsteps;) {
        const long long t = c.t_start + s;
        T* z = cur;
        T* r = w + P;
        T* g = gcur;
        if (s >= 0) {
            if (begin) {
                const double eps = (a.n_adapt > 0 && t >= a.n_adapt) ? exp(a.log_eps_bar[k]) : exp(a.log_eps[k]);
                e = (T)eps;
                double ksum = 0.0;
                for (int i4 = tid; i4 * 4 < P; i4 += nt) {
                    T zz[4];
                    qb_normal4(qb_rand4(c.seed, chain, t, QB_STREAM_INCR, (uint32_t)i4), zz);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < P) {
                            w[P + i] = zz[q]; w[4 * P + i] = zz[q]; rsum[i] = zz[q];
                            ksum += (double)zz[q] * (double)zz[q];
                        }
                    }
                }
                for (int i = tid; i < P; i += nt) { w[i] = cur[i]; w[3 * P + i] = cur[i]; w[2 * P + i] = gcur[i]; w[5 * P + i] = gcur[i]; }
                H0 = -c.lp[k] + qb_block_sum(ksum, red) / 2.0;      // the block sum's barriers also order the reads above
                if (tid == 0 && a.rec_eps) a.rec_eps[k * c.rec_ld + s] = eps;
                w_tree = 0.0; sum_acc = 0.0; n_leap = 0; depth = 0; n_sub = 0; moved = false;
                fwd = (qb_rand4(c.seed, chain, t, QB_STREAM_NUTS, 0).x & 1u) != 0;
                begin = false;
            }
            T* end = fwd ? w + 3 * P : w;
            z = end; r = end + P; g = end + 2 * P;
            const T es = fwd ? e : -e, eh = qb_mul<T>(es, T(0.5));
            for (int i = tid; i < P; i += nt) {
                const T ri = qb_add<T>(r[i], qb_mul<T>(eh, g[i]));
                r[i] = ri;
                z[i] = qb_add<T>(z[i], qb_mul<T>(es, ri));
            }
        }
        __syncthreads();
        const double lp = eval(z, g);
        if (s < 0) {
            if (tid == 0) {
                c.lp[k] = lp; c.map_lp[k] = lp; c.naccept[k] = 0;
                if (c.rec_lp0) c.rec_lp0[k] = lp;
                a.log_eps[k] = log(a.eps0); a.log_eps_bar[k] = log(a.eps0); a.h_bar[k] = 0.0;
            }
            qb_copy_vec<T>(c.map_theta + k * P, cur, P);
            __syncthreads();
            s = 0;
            continue;
        }
        const T eh = qb_mul<T>(fwd ? e : -e, T(0.5));
        double k2 = 0.0;
        for (int i = tid; i < P; i += nt) {
            const T ri = qb_add<T>(r[i], qb_mul<T>(eh, g[i]));
            r[i] = ri;
            rsum[i] = qb_add<T>(rsum[i], ri);
            k2 += (double)ri * (double)ri;
        }
        double dH = (-lp + qb_block_sum(k2, red) / 2.0) - H0;
        if (!isfinite(lp) || isnan(dH)) dH = INFINITY;
        const double wl = -dH;
        const bool div = dH > 1000.0;
        sum_acc += dH > 0.0 ? exp(-dH) : 1.0;
        ++n_leap;

        // uniform progressive sampling inside the subtree
        bool take = true;
        if (n_sub == 0) {
            w_sub = wl;
        } else {
            const double wn = qb_logaddexp(w_sub, wl);
            const double u = qb_u01(qb_rand4(c.seed, chain, t, QB_STREAM_NUTS, (uint32_t)(QB_NUTS_LEAF0 + n_leap - 1)).x);
            take = wl > -INFINITY && u < exp(wl - wn);
            w_sub = wn;
        }
        if (take) {
            qb_copy_vec<T>(w + 6 * P, z, P);
            qb_copy_vec<T>(w + 7 * P, g, P);
            lp_sub = lp;
        }

        // checkpoints and the U-turn checks of the sub-subtrees that end at this leaf
        const int leaf = n_sub++;
        const int idx_max = __popc(leaf >> 1), idx_min = idx_max - (__ffs(~leaf) - 1) + 1;
        if ((leaf & 1) == 0) {
            qb_copy_vec<T>(ck_r + (long long)idx_max * P, r, P);
            qb_copy_vec<T>(ck_s + (long long)idx_max * P, rsum, P);
        }
        bool turn = false;
        for (int ci = idx_max; ci >= idx_min && !turn && !div; --ci)
            turn = qb_nuts_turning<T>(ck_r + (long long)ci * P, r, rsum, ck_s + (long long)ci * P, P, red);

        if (div || turn || n_sub == (1 << depth)) {
            // the subtree joins the trajectory (biased progressive sampling)
            const double u = qb_u01(qb_rand4(c.seed, chain, t, QB_STREAM_NUTS, (uint32_t)depth).y);
            if (!div && !turn && u < fmin(1.0, exp(w_sub - w_tree))) {
                qb_copy_vec<T>(cur, w + 6 * P, P);
                qb_copy_vec<T>(gcur, w + 7 * P, P);
                if (tid == 0) c.lp[k] = lp_sub;
                moved = true;
            }
            w_tree = qb_logaddexp(w_tree, w_sub);
            ++depth;
            if (!div && !turn) turn = qb_nuts_turning<T>(w + P, w + 4 * P, rsum, (const T*)nullptr, P, red);
            if (div || turn || depth >= D) {
                const double stat = sum_acc / (double)n_leap;
                __syncthreads();
                const double lp_cur = c.lp[k];
                if (moved && lp_cur >= c.map_lp[k]) qb_copy_vec<T>(c.map_theta + k * P, cur, P);
                if (tid == 0) {
                    if (moved) {
                        c.naccept[k] += 1;
                        if (lp_cur >= c.map_lp[k]) c.map_lp[k] = lp_cur;
                    }
                    const long long ri = k * c.rec_ld + s;
                    if (c.rec_lp) c.rec_lp[ri] = lp_cur;
                    if (c.rec_alpha) c.rec_alpha[ri] = stat;
                    if (c.rec_acc) c.rec_acc[ri] = moved ? 1 : 0;
                    if (a.rec_depth) a.rec_depth[ri] = depth;
                    if (a.rec_nleap) a.rec_nleap[ri] = n_leap;
                    if (a.rec_div) a.rec_div[ri] = div ? 1 : 0;
                    if (t < a.n_adapt) {           // dual averaging (Stan: gamma 0.05, t0 10, kappa 0.75)
                        const double m = (double)(t + 1), eta = 1.0 / (m + 10.0);
                        const double hbar = (1.0 - eta) * a.h_bar[k] + eta * (a.target - stat);
                        const double log_eps = log(10.0 * a.eps0) - sqrt(m) / 0.05 * hbar;
                        const double xe = pow(m, -0.75);
                        a.h_bar[k] = hbar;
                        a.log_eps[k] = log_eps;
                        a.log_eps_bar[k] = xe * log_eps + (1.0 - xe) * a.log_eps_bar[k];
                    }
                }
                if (c.samples && c.store_every > 0 && (s + 1) % c.store_every == 0) {
                    const long long slot = (s + 1) / c.store_every - 1;
                    if (slot < c.n_slots) qb_copy_vec<T>(c.samples + (k * c.n_slots + slot) * P, cur, P);
                }
                ++s;
                begin = true;
            } else {
                fwd = (qb_rand4(c.seed, chain, t, QB_STREAM_NUTS, (uint32_t)depth).x & 1u) != 0;
                n_sub = 0;
            }
        }
        __syncthreads();
    }
}
