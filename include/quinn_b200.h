/*
 * quinn_b200.h -- C ABI of the B200-native QUiNN posterior-sampling hot path.
 *
 * The reference (sandialabs/quinn) has no FFI: its boundary for this path is Python
 * duck typing at two seams (SURVEY.md section 8b).  Every entry point below states the
 * reference interface it replaces (file:line under the reference tree).  A maintainer
 * binds these with ctypes (INTEGRATION.md shows the stub); quinn_b200/_lib.py is that
 * binding for this repository.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types cross the boundary.
 *   - every buffer is caller-owned DEVICE memory unless a comment says "host";
 *     the library never allocates persistent memory.
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*).
 *   - return value: 0 on success, negative on error; qb_last_error() gives the text.
 *     Nothing is thrown across the ABI.
 *   - dtype: QB_F32 or QB_F64 selects the arithmetic type of theta/x/y/grad/etc.
 *     Per-chain scalars (log-posteriors, alphas) are ALWAYS double.
 *   - flat parameter layout = quinn/nns/nnwrap.py:64-106: nnmodel.parameters() order, each
 *     tensor flattened C-order; a Linear weight is (n_out, n_in) row-major.
 */
#ifndef QUINN_B200_H
#define QUINN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QB_MAX_LAYERS 16
#define QB_MAX_TERMS 6

enum { QB_F32 = 0, QB_F64 = 1 };
enum { QB_ACT_IDENTITY = 0, QB_ACT_TANH = 1, QB_ACT_RELU = 2 };

/* One Linear(+activation) step.  res_step == 0: h <- act(W h + b)   (quinn/nns/mlp.py:59-86).
 * res_step != 0: h <- h + res_step * act(W h + b)                   (quinn/nns/rnet.py:150-158).
 * Several layers may name the same w_off/b_off (RNet with Poly(0), rnet.py:344-347). */
/* n_terms >= 2: weights that are a polynomial in the depth variable (RNet with Lin / Quad / Cubic / Poly(n),
 * quinn/nns/rnet.py:244-347):  W = sum_m coef[m] * theta[w_off + m*w_stride ...], b likewise with b_stride; coef[m] = t^m
 * of the residual step.  Gradients are scattered back to every term (chain rule).  n_terms 0 or 1: plain layer. */
typedef struct {
    int32_t n_in, n_out;
    int32_t w_off;          /* offset of W (n_out x n_in row-major) in the flat parameter vector */
    int32_t b_off;          /* offset of the bias, or -1 */
    int32_t act;            /* QB_ACT_* */
    int32_t n_terms;
    double  res_step;
    int32_t w_stride, b_stride;
    double  coef[QB_MAX_TERMS];
} qb_layer_t;

/* The network the kernels evaluate: MLP.forward (mlp.py:92-101) / RNet.forward (rnet.py:124-164). */
typedef struct {
    int32_t n_layers, in_dim, out_dim, n_params;
    int32_t final_exp;      /* 1: out <- exp(out)  (mlp.py:82-83 final_transform='exp') */
    int32_t reserved[3];
    qb_layer_t layers[QB_MAX_LAYERS];
} qb_net_t;

/* Gaussian likelihood + optional Gaussian prior: NegLogPost / NegLogPrior (quinn/nns/losses.py:186-256).
 *   -lp = 0.5*sum (y-M(x))^2/sigma^2 + N/2 log 2pi + N log sigma
 *         + prior_scale * [ sum (w-anchor)^2/(2 prior_sigma^2) + P/2 log(2 pi prior_sigma^2) ]
 * prior_scale is len(predictions)/fulldatasize (losses.py:204).  NN_MCMC uses no prior (nn_mcmc.py:64). */
typedef struct {
    double sigma;
    double prior_sigma;         /* <= 0: no prior */
    double prior_scale;
    const void* prior_anchor;   /* device, dtype elements: [P] or [K,P]; NULL = zeros */
    int32_t anchor_per_chain;   /* 1: anchor is [K,P] */
    int32_t reserved;
} qb_lik_t;

/* Training data, shared by all chains.  x: [N, in_dim], y: [N, out_dim], row-major, dtype elements. */
typedef struct {
    const void* x;
    const void* y;
    int64_t n;
} qb_data_t;

const char* qb_last_error(void);

/* ABI version: bumped with every change of a struct layout or a signature.  A binding must refuse a library whose
 * qb_version() differs from the QB_ABI_VERSION it was written against (quinn_b200/_lib.py does), and can check its
 * struct mirrors against qb_struct_sizes(): out[0..n) = sizeof of qb_layer_t, qb_net_t, qb_lik_t, qb_data_t, qb_chain_t,
 * qb_rng_t, qb_record_t, qb_amcmc_t, qb_hmc_t (declaration order); returns how many sizes exist. */
#define QB_ABI_VERSION 203
int qb_version(void);
int qb_struct_sizes(int64_t* out, int n);

/* Bytes of scratch the evaluation entry points need for (net, dtype, K chains, N points). */
size_t qb_eval_workspace_bytes(const qb_net_t* net, int dtype, int64_t K, int64_t N, int want_grad);

/* Kernel 1.  lp[k] = log p(theta_k | D) for K flat parameter vectors at once.
 * Replaces NN_MCMC.logpost (quinn/solvers/nn_mcmc.py:45-71) == -NNWrap.calc_loss(theta, NegLogPost, x, y)
 * (quinn/nns/nnwrap.py:109-126), called once per theta there.
 * theta: [K, P] dtype; lp: [K] double. */
int qb_logpost(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
               const qb_lik_t* lik, double* lp, void* workspace, size_t workspace_bytes, void* stream);

/* Kernel 2.  lp[k] and grad[k,:] = d lp / d theta_k (fused forward + reverse mode).
 * Replaces NN_MCMC.logpostgrad (nn_mcmc.py:73-98) == -NNWrap.calc_lossgrad (nnwrap.py:128-150).
 * grad: [K, P] dtype. */
int qb_logpost_grad(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
                    const qb_lik_t* lik, double* lp, void* grad, void* workspace, size_t workspace_bytes,
                    void* stream);

/* Kernel 5.  hv[k,:] = (d^2 lp / d theta^2) v_k at one theta[P] (lp exactly as qb_logpost_grad) for K directions.
 * v: [K,P] dtype, or NULL for the unit directions v_k = e_{col0+k} (rows col0 .. col0+K-1 of the Hessian).
 * Replaces NNWrap.calc_hess_full (quinn/nns/nnwrap.py:153-203).  lik->anchor_per_chain must be 0.  K == 0 does nothing.
 * A network whose weights, one direction and the smallest tile of activations and tangents (16 points in fp32, 8 in
 * fp64) exceed 227 KB of shared memory is refused; it is not streamed.  hv: [K,P] dtype.  Deterministic: fp64 results
 * are bit-identical run to run. */
size_t qb_hvp_workspace_bytes(const qb_net_t* net, int dtype, int64_t K, int64_t N);
int qb_logpost_hvp(const qb_net_t* net, int dtype, const void* theta, const void* v, int64_t col0, int64_t K,
                   const qb_data_t* data, const qb_lik_t* lik, void* hv, void* workspace, size_t workspace_bytes,
                   void* stream);
/* Launch plan of kernel 5 for K directions over N points: out[0..4] = {tile points TM, threads per block, dynamic smem
 * bytes, N-splits S, blocks}.  Returns -1 (with qb_last_error) for a network kernel 5 refuses. */
int qb_hvp_plan_info(const qb_net_t* net, int dtype, int64_t K, int64_t N, int64_t* out);

/* Kernel 6.  Kronecker factors of the per-point empirical Fisher of every layer at one theta[P], summed over the N points
 * (no 1/N, no prior).  For layer l with input activations a_i and pre-activation gradients delta_i = d log p_i / d z_l of
 * point i's data term -0.5 ||y_i - f(x_i)||^2 / sigma^2 (only lik->sigma is used):
 *     A_l = sum_i a_i a_i^T [n_in, n_in],  s_l = sum_i a_i [n_in] (layers with a bias only),  G_l = sum_i delta_i delta_i^T
 *     [n_out, n_out].
 * factors: device double, [A_0 | s_0 | G_0 | A_1 | s_1 | G_1 | ...], each matrix row-major, s_l absent without a bias.
 * Refused (error text says why): layers sharing weights (RNet Poly(0)), polynomial-in-depth weights (n_terms >= 2),
 * networks that kernel 2 evaluates on the layer-streamed path (plan code 5), lik->anchor_per_chain != 0.
 * N == 0 writes zero factors and launches no kernel.  Deterministic: fp64 results are bit-identical run to run. */
size_t qb_kfac_workspace_bytes(const qb_net_t* net, int dtype, int64_t N);
int qb_logpost_kfac(const qb_net_t* net, int dtype, const void* theta, const qb_data_t* data, const qb_lik_t* lik,
                    double* factors, void* workspace, size_t workspace_bytes, void* stream);
/* Launch plan of kernel 6 over N points: out[0..4] = {tile points TM, threads per block, dynamic smem bytes, N-splits S
 * (one block each), factor elements F}.  Returns -1 (with qb_last_error) for a network kernel 6 refuses. */
int qb_kfac_plan_info(const qb_net_t* net, int dtype, int64_t N, int64_t* out);

/* Kernel 7.  Network outputs and their per-point Jacobians with respect to theta[P] over x[N, in_dim] (dtype), as
 * per-layer pairs: for output j of point n, layer l's part of d f_j(x_n) / d [W_l | b_l] is outer(d_l[j, :, n],
 * [a_l[:, n]; 1]) with a_l the layer's input and d_l[j] = d f_j / d z_l its pre-activation gradient.  Polynomial terms
 * (each term gets coef_m times that part) and layers sharing weights (parts summed) are left to the caller.
 * out: [N, o] dtype, f(x_n) with final_exp applied.
 * fac: dtype, N * F elements with F = sum_l (n_in_l + o * n_out_l), unit-major; per layer, in order,
 *     a_l as [n_in_l, N], then d_l as [o, n_out_l, N].
 * Refused (error text says why): networks that kernel 2 evaluates on the layer-streamed path (plan code 5), NULL
 * arguments, N < 0.  N == 0 launches no kernel.  No reduction over the points: fp64 results are bit-identical run to
 * run.  Replaces nothing in the reference; it feeds NN_Laplace.predict_mom_glm (DESIGN.md section 4h). */
int qb_predict_jac(const qb_net_t* net, int dtype, const void* theta, const void* x, int64_t N, void* out, void* fac,
                   void* stream);
/* Launch plan of kernel 7 over N points: out[0..4] = {tile points TM, threads per block, dynamic smem bytes, blocks (runs
 * of whole tiles, 0 for N == 0), factor rows F}.  Returns -1 (with qb_last_error) for a network kernel 7 refuses. */
int qb_jac_plan_info(const qb_net_t* net, int dtype, int64_t N, int64_t* out);

/* ---- Batched ensemble training (SURVEY.md 8f rank 1) --------------------------------------------
 * NN_Ens.fit (quinn/solvers/nn_ens.py:51-69) trains nens members one after the other, each with
 * Learner.fit -> nnfit (quinn/ens/learner.py:59-73, quinn/nns/nnfit.py:125-166: minibatch loop, torch Adam, best
 * model by validation loss).  Here all members advance together: kernels 1 / 2 with per-member data, a flat Adam
 * update and a masked row copy for the best-model bookkeeping. */

/* Kernels 1 / 2 where member k sees x + k*x_stride and y + k*y_stride (strides in ELEMENTS, 0 = shared by all
 * members): every member has its own subset (dfrac) or minibatch of data->n points.  grad may be NULL (value only).
 * Workspace as qb_eval_workspace_bytes(net, dtype, K, data->n, grad != NULL). */
int qb_logpost_members(const qb_net_t* net, int dtype, const void* theta, int64_t K, const qb_data_t* data,
                       int64_t x_stride, int64_t y_stride, const qb_lik_t* lik, double* lp, void* grad,
                       void* workspace, size_t workspace_bytes, void* stream);

/* torch.optim.Adam step (nnfit.py:92-93 `optim.Adam(params, lr=lrate, weight_decay=wd)`) on flat arrays of n
 * elements: g = grad*grad_scale + wd*theta; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
 * theta -= lr/(1-b1^step) * m / (sqrt(v)/sqrt(1-b2^step) + eps).  step counts from 1. */
int qb_adam_step(int dtype, void* theta, const void* grad, void* m, void* v, int64_t n, double lr, double beta1,
                 double beta2, double eps, double wd, int64_t step, double grad_scale, void* stream);

/* dst[k,:] = src[k,:] for the rows with mask[k] != 0 (best-model tracking of nnfit.py:147-152, per member). */
int qb_copy_rows_where(int dtype, void* dst, const void* src, const unsigned char* mask, int64_t K, int64_t P,
                       void* stream);

/* ---- Kernel 3: fused chain steps (propose + evaluate + accept) ------------------------------
 * Replaces the loop body of MCMCBase.run (quinn/mcmc/mcmc.py:65-85) together with
 * AMCMC.sampler (admcmc.py:38-74), HMC.sampler (hmc.py:27-70), MALA.sampler (mala.py:24-53).
 * One thread block owns one chain for all `nsteps`; no host round trip per step. */

/* Per-chain state, [K,...] device arrays, updated in place. */
typedef struct {
    int64_t K;
    void*    theta;        /* [K,P] dtype: current state */
    double*  lp;           /* [K]: log-posterior of the current state */
    int64_t* naccept;      /* [K] */
    void*    map_theta;    /* [K,P] dtype: MAP state (updated on accept with >=, mcmc.py:79) */
    double*  map_lp;       /* [K] */
} qb_chain_t;

enum { QB_RNG_PHILOX = 0, QB_RNG_REPLAY = 1 };

/* Random draws.  PHILOX: counter-based, keyed by (seed, chain_offset + k) so results do not depend
 * on how chains are sharded over GPUs.  REPLAY: consume draws recorded from the reference:
 *   incr[s, k, :]  proposal increment (AMCMC, np.random.multivariate_normal of admcmc.py:70) or
 *                  momentum (HMC/MALA, np.random.randn of hmc.py:43 / mala.py:42), dtype [nsteps,K,P]
 *   unif[s, k]     np.random.random_sample() of mcmc.py:75, double [nsteps,K] */
typedef struct {
    int32_t mode;
    int32_t reserved;
    uint64_t seed;
    int64_t chain_offset;
    const void* incr;
    const double* unif;
} qb_rng_t;

/* Per-step records, each optional (NULL = do not record).  Index s is the step within this call.
 *   logpost[k*ld + s], alpha[k*ld + s] (double), accepted[k*ld + s] (uint8)      (mcmc.py:83-85)
 *   samples[(k*n_slots + slot)*P + :] dtype, slot = (s+1)/store_every - 1 when (s+1)%store_every==0 */
typedef struct {
    double*  logpost;
    double*  alpha;
    uint8_t* accepted;
    int64_t  ld;
    void*    samples;
    int64_t  store_every;
    int64_t  n_slots;
    double*  logpost0;     /* [K], optional: log-posterior of the incoming state, written when init_lp != 0 (mcmc.py:55-61) */
} qb_record_t;

enum { QB_ADAPT_NONE = 0, QB_ADAPT_DIAG = 1, QB_ADAPT_FULL = 2 };

/* AMCMC state (admcmc.py:34-36 `_Xm`, `_cov`, `_propcov`).
 *   adapt == NONE: proposal covariance stays the initial one for ever.
 *   adapt == FULL: the reference's recursion on a dense PxP covariance per chain + in-kernel Cholesky
 *                  at every adaptation step (only when K*P*P fits; small P).
 *   adapt == DIAG: the scalable deviation: only the diagonal of the recursion is kept.
 * The initial covariance is the reference's 0.01 + diag(0.09|theta0|) (admcmc.py:65: rank-1 + diagonal),
 * sampled in O(P) as 0.1*z0 + sqrt(0.09|theta0|)*z, unless chol_ini (lower Cholesky factor of a
 * user cov_ini, [P,P] dtype, shared by all chains) is given. */
typedef struct {
    double gamma;
    int64_t t0, tadapt;
    int32_t adapt;
    int32_t track_moments;   /* 0: off; 1: run the Xm recursion with the DIAGONAL of cov ([K,P]);
                                2: with the dense cov ([K,P,P]).  Forced to 1 / 2 by adapt DIAG / FULL. */
    void* xm;                /* [K,P] dtype */
    void* cov;               /* [K,P] or [K,P,P] (see track_moments); dtype */
    void* pscale;            /* [K,P] dtype: per-element proposal std (initial or adapted-diag) */
    void* chol;              /* FULL: [K,P,P] dtype lower factor of the adapted proposal covariance */
    const void* chol_ini;    /* optional [P,P] dtype */
    int32_t* prop_kind;      /* [K]: 0 = initial rank1+diag, 1 = adapted diag, 2 = adapted full, 3 = chol_ini */
} qb_amcmc_t;

/* nsteps AMCMC steps for K chains starting at absolute step t_start.  If init_lp != 0 the kernel first
 * evaluates lp of the incoming theta (mcmc.py:55-56) and initialises map_theta/map_lp/naccept.
 * scratch: [K,P] dtype (proposal). */
int qb_amcmc_run(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik,
                 qb_chain_t* chain, qb_amcmc_t* am, const qb_rng_t* rng, const qb_record_t* rec,
                 int64_t t_start, int64_t nsteps, int init_lp, void* scratch, void* stream);

/* HMC (method 0, hmc.py) / MALA (method 1, mala.py) state.  grad_cur caches the gradient at the current
 * state between steps (exactly what the reference recomputes at hmc.py:48 / mala.py:44). */
typedef struct {
    int32_t method;          /* 0 = HMC, 1 = MALA */
    int32_t L;               /* leapfrog steps (HMC) */
    double epsilon;
    void* grad_cur;          /* [K,P] dtype */
    void* mom;               /* [K,P] dtype scratch */
    void* prop;              /* [K,P] dtype scratch */
    void* grad_prop;         /* [K,P] dtype scratch */
} qb_hmc_t;

int qb_hmc_run(const qb_net_t* net, int dtype, const qb_data_t* data, const qb_lik_t* lik,
               qb_chain_t* chain, qb_hmc_t* hm, const qb_rng_t* rng, const qb_record_t* rec,
               int64_t t_start, int64_t nsteps, int init_lp, void* stream);

/* ---- Kernel 4: posterior predictive -----------------------------------------------------------
 * Replaces the M sequential forwards of nn_p (quinn/nns/nnwrap.py:330-347), NN_MCMC.predict_ens
 * (nn_mcmc.py:180-200), NN_Ens.predict_ens (nn_ens.py:85-110), QUiNNBase.predict_ens /
 * predict_mom_sample (solvers/quinn.py:51-104).
 * theta: [M,P]; x: [N,in_dim]; out (optional): [M,N,out_dim]; mean/var (optional): [N,out_dim],
 * var with ddof=1 (quinn.py:96).  All dtype elements. */
int qb_predict(const qb_net_t* net, int dtype, const void* theta, int64_t M, const void* x, int64_t N,
               void* out, void* mean, void* var, void* stream);

/* ---- Variational inference (Bayes by backprop) -------------------------------------------------
 * Replaces BNet.forward's sampling + log q + log prior (quinn/vi/bnet.py:142-166, rvar/rvs.py:96-127,
 * 159-173) for nsam weight samples at once.
 * w[s,:] = mu + exp(rho)*eps[s,:];  logq[s], logp[s] (double).
 * eps: [nsam,P] dtype; if rng_seed_or_0 != 0 eps is filled with Philox normals first. */
int qb_vi_sample(int dtype, const void* mu, const void* rho, void* eps, int64_t nsam, int64_t P,
                 double pi, double sigma1, double sigma2, uint64_t rng_seed_or_0, uint64_t rng_step,
                 void* w, double* logq, double* logp, void* stream);

/* Chain rule of BNet.sample_elbo / viloss (bnet.py:181-232) back to (mu, rho).  With
 * glp[s,:] = d lp_data(sigma=1)/d w_s from qb_logpost_grad (so d ssq_s/dw = -2 glp), for a scalar
 *   L = c_ssq * sum_s ssq_s + c_logp * sum_s logp_s + c_logq * sum_s logq_s
 * it returns gmu[p] = sum_s dL/dw_sp and grho[p] = sum_s (dL/dw_sp * exp(rho_p) eps_sp) - nsam*c_logq
 * (the total derivative of log q wrt mu is 0 and wrt rho is -1 per sample).
 * viloss uses c_ssq = 0.5*B/(nsam*B*o)/datanoise^2, c_logp = -1/(nsam*num_batches), c_logq = -c_logp. */
int qb_vi_backward(int dtype, const void* mu, const void* rho, const void* eps, const void* w,
                   const void* glp, int64_t nsam, int64_t P, double pi, double sigma1, double sigma2,
                   double c_ssq, double c_logp, double c_logq, void* gmu, void* grho, void* stream);

/* ---- measurement helper --------------------------------------------------------------------------
 * Dependent-chain FMA micro-benchmark used as the FP32 / FP64 CUDA-core roofline denominator
 * (MEASURED_PEAKS.json has no such entry).  Enqueues one launch doing `flops_out` floating point
 * operations (written to the host pointer); the caller times it with CUDA events. */
int qb_fma_peak(int dtype, int variant, int64_t iters, double* flops_out_host, void* sink, void* stream);

/* Launch-plan introspection for DESIGN.md / bench.py: fills out[0..7] =
 * {tile points TM, threads per block, dynamic smem bytes, N-splits S, blocks, inplace flag,
 *  tensor-core path (0: CUDA-core kernel, 1: tcgen05 3xTF32, 2: same, software-pipelined, 3: tcgen05 gradient kernel (3xTF32),
 *  4: tcgen05 gradient kernel with fp16-split operands, 5: CUDA cores, weights streamed through shared memory),
 *  tensor-memory columns}.
 * Code 5 serves networks whose weights do not fit in shared memory next to one tile of activations (in fp64 from about
 * 27 000 parameters): only activations stay resident and every layer's weights pass through a small shared-memory ring in
 * chunks of output rows, in every entry point (kernels 1-4).  It is chosen only when the resident plan does not fit;
 * a network whose activations of one tile (8 points in fp64, 16 in fp32) exceed 227 KB is refused.
 * The tensor-core VALUE path (qb_logpost, qb_amcmc_run, qb_predict) serves fp32 MLPs with <= 15 inputs, hidden widths
 * that are multiples of 16 (<= 128), <= 4 outputs and no residual layers; the tensor-core GRADIENT path
 * (qb_logpost_grad, qb_logpost_members, qb_hmc_run) serves fp32 MLPs in -> H -> H -> 1: tanh nets with H = 64 or 128 and
 * <= 15 inputs (code 4: 3xFP16; its operand scales come from max|x|, max|y| of the call, found by a small kernel ahead of
 * the evaluation in 256 bytes that qb_eval_workspace_bytes adds to the workspace), tanh / relu nets with H = 32 or 64 and
 * <= 7 inputs (code 3).  QB_NO_TC=1 disables both paths, QB_NO_TCG=1 only the gradient path, QB_NO_TG8=1 only code 4,
 * QB_TG8_64=0 keeps the 64-wide tanh nets on code 3. */
int qb_plan_info(const qb_net_t* net, int dtype, int64_t K, int64_t N, int want_grad, int64_t* out);

/* ---- device-side post-processing of chains / ensembles (SURVEY.md 8f rank 2) -------------------------------------
 * None of these has a counterpart kernel in the reference; they replace host numpy on arrays that should not leave
 * the device: the (M, N*, o) predictive array of QUiNNBase.predict_ens (quinn/solvers/quinn.py:51-70) and the per-step
 * records of MCMCBase.run (quinn/mcmc/mcmc.py:92-99). */

/* mean[k], var[k] (ddof = 1) of the rows of x[K, n] (doubles): per-chain moments of a monitored scalar, the inputs of the
 * Gelman-Rubin R-hat (quinn_b200/dist.py: rhat). */
int qb_row_moments(const double* x, int64_t K, int64_t n, double* mean, double* var, void* stream);

/* Effective sample size of every row of x[K, n]: n / tau with tau = -1 + 2 sum_m (rho_2m + rho_2m+1) over Geyer's initial
 * positive sequence (autocorrelations up to max_lag, <= 0: n - 1).  tau may be NULL. */
int qb_ess(const double* x, int64_t K, int64_t n, int64_t max_lag, double* ess, double* tau, void* stream);

/* out[p] = mean_k g[k,p]^2 (double).  With g = per-point loss gradients (qb_logpost_members, one point per member) this is
 * the diagonal Fisher of NNWrap.calc_hess_diag (quinn/nns/nnwrap.py:204-229). */
int qb_colsq_mean(int dtype, const void* g, int64_t K, int64_t P, double* out, void* stream);

/* out[iq, i] = quantile q[iq] of y[:, i] over the leading (member) axis of y[M, n], numpy's default linear interpolation:
 * the quantiles of get_stats (quinn/utils/stats.py:8-32: 0.25, 0.5, 0.75).  q: host array of nq <= 8 values in [0, 1]. */
int qb_quantiles(int dtype, const void* y, int64_t M, int64_t n, const double* q_host, int nq, void* out, void* stream);

/* Number of kernel launches this library has enqueued since load (bench.py's gpu_launches). */
int64_t qb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* QUINN_B200_H */
