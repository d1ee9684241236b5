// quinn_b200: kernels + C ABI (include/quinn_b200.h).  Build: see quinn_b200/build.py
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <atomic>

#include "quinn_b200.h"
#include "qb_plan.h"
#include "qb_device.cuh"
#include "qb_chain.cuh"
#include "qb_stream.cuh"
#include "qb_hvp.cuh"
#include "qb_kfac.cuh"
#include "qb_tc.cuh"
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
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int qb_fail(const char* fmt, const char* a = "", long long b = 0) {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return -1;
}
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

// =================================================================================================
// launch planning (host)
// =================================================================================================
static inline int rup(int v, int m) { return (v + m - 1) / m * m; }
static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }
static int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return (s && *s) ? atoi(s) : dflt;
}

static const int QB_SMEM_MAX = 227 * 1024;
static const int QB_SMEM_SM = 228 * 1024;    // shared memory per SM
// SM count of the current device (148 on B200), queried once per process
static int qb_num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) n = v;
        else n = 148;
    }
    return n;
}
#define QB_NUM_SMS (qb_num_sms())

static int validate_net(const qb_net_t* net) {
    if (!net) return qb_fail("net is NULL");
    if (net->n_layers < 1 || net->n_layers > QB_MAX_LAYERS) return qb_fail("n_layers out of range%s (%lld)", "", net->n_layers);
    int width = net->in_dim;
    for (int l = 0; l < net->n_layers; ++l) {
        const qb_layer_t& L = net->layers[l];
        if (L.n_in != width) return qb_fail("layer %s%lld: n_in does not match the previous width", "", l);
        if (L.n_in < 1 || L.n_out < 1) return qb_fail("layer %s%lld: empty layer", "", l);
        if (L.act < 0 || L.act > 2) return qb_fail("layer %s%lld: unknown activation", "", l);
        if (L.res_step != 0.0 && L.n_in != L.n_out) return qb_fail("layer %s%lld: residual layer must be square", "", l);
        if (L.w_off < 0 || L.w_off + L.n_in * L.n_out > net->n_params) return qb_fail("layer %s%lld: weight offset out of range", "", l);
        if (L.b_off >= 0 && L.b_off + L.n_out > net->n_params) return qb_fail("layer %s%lld: bias offset out of range", "", l);
        if (L.n_terms < 0 || L.n_terms > QB_MAX_TERMS) return qb_fail("layer %s%lld: n_terms out of range", "", l);
        if (L.n_terms > 1) {
            const long long lastw = (long long)L.w_off + (long long)(L.n_terms - 1) * L.w_stride;
            const long long lastb = (long long)L.b_off + (long long)(L.n_terms - 1) * L.b_stride;
            if (L.w_stride < 0 || lastw + (long long)L.n_in * L.n_out > net->n_params) return qb_fail("layer %s%lld: polynomial weight terms out of range", "", l);
            if (L.b_off >= 0 && (L.b_stride < 0 || lastb + L.n_out > net->n_params)) return qb_fail("layer %s%lld: polynomial bias terms out of range", "", l);
        }
        width = L.n_out;
    }
    if (width != net->out_dim) return qb_fail("out_dim does not match the last layer");
    return 0;
}

// Fill `P` for tile size TM; returns smem bytes (or -1 if a constraint fails).
static long long plan_for_tm(const qb_net_t* net, int dtype, bool want_grad, int TM, QbPlan* P, bool wr_global = false) {
    const int elem = dtype == QB_F64 ? 8 : 4;
    const int TU = dtype == QB_F64 ? 4 : 8, LDPAD = dtype == QB_F64 ? 2 : 4, PV = dtype == QB_F64 ? 2 : 4;
    // gradient kernel: TU x 4 thread tiles (twice the threads per tile) when some layer is >= 64 wide, else TU x 8
    int widest = 0;
    for (int l = 0; l < net->n_layers; ++l) widest = std::max(widest, net->layers[l].n_out);
    const int tpg = (dtype == QB_F64 || widest >= 64) ? 4 : 8;
    const int TP = want_grad ? env_int("QB_TPG", tpg) : TU;
    memset(P, 0, sizeof(*P));
    P->n_layers = net->n_layers; P->in_dim = net->in_dim; P->out_dim = net->out_dim;
    P->n_params = net->n_params; P->final_exp = net->final_exp;
    P->TM = TM; P->lda = TM + LDPAD; P->want_grad = want_grad ? 1 : 0; P->elem_size = elem;
    P->tpg = TP;
    const int PG = TM / TP;
    int max_items = 0, woff = 0;
    bool any_gemm = false;
    for (int l = 0; l < net->n_layers; ++l) {
        const qb_layer_t& S = net->layers[l];
        QbLayerPlan& L = P->L[l];
        L.n_in = S.n_in; L.n_out = S.n_out; L.n_in_pad = rup(S.n_in, TU); L.n_out_pad = rup(S.n_out, TU);
        L.w_off = S.w_off; L.b_off = S.b_off; L.act = S.act; L.res_step = S.res_step; L.has_res = S.res_step != 0.0;
        L.n_terms = S.n_terms > 1 ? S.n_terms : 0; L.w_stride = S.w_stride; L.b_stride = S.b_stride;
        for (int m = 0; m < QB_MAX_TERMS; ++m) L.coef[m] = S.coef[m];
        if (L.has_res) P->has_res = 1;
        const int UG = L.n_out_pad / TU;
        L.ug_shift = L.ugi_shift = L.ig_shift = -1;
        for (int sft = 0; sft < 16; ++sft) {
            if ((1 << sft) == UG) L.ug_shift = sft;
            if ((1 << sft) == L.n_in_pad / TU) L.ugi_shift = sft;
            if ((1 << sft) == (S.n_in + 3) / 4) L.ig_shift = sft;
        }
        L.nj = S.n_out == 1 ? 1 : (S.n_out == 2 ? 2 : 4);
        const long long cost_g = cdiv((long long)UG * PG, 256) * S.n_in * (TP * TU + 4);
        const long long cost_d = cdiv(TM, 256) * cdiv(S.n_out, L.nj) * S.n_in * (2 * L.nj + 1);
        L.mode = (cost_d < cost_g) ? QB_MODE_DOT : QB_MODE_GEMM;
        if (L.mode == QB_MODE_GEMM) { any_gemm = true; max_items = std::max(max_items, UG * PG); }
        if (want_grad && l > 0) max_items = std::max(max_items, (L.n_in_pad / TU) * PG), any_gemm = true;
        // shared weights: reuse an identical earlier staging
        int dup = -1;
        for (int m = 0; m < l; ++m) {
            const qb_layer_t& Sm = net->layers[m];
            bool same_terms = (Sm.n_terms > 1 ? Sm.n_terms : 0) == (S.n_terms > 1 ? S.n_terms : 0);
            if (same_terms && S.n_terms > 1)
                for (int q = 0; q < S.n_terms; ++q) same_terms = same_terms && Sm.coef[q] == S.coef[q];
            if (same_terms && Sm.w_off == S.w_off && Sm.b_off == S.b_off && Sm.n_in == S.n_in && Sm.n_out == S.n_out &&
                (Sm.act == QB_ACT_TANH) == (S.act == QB_ACT_TANH) &&      // fp32 tanh layers stage W * 2log2(e)
                P->L[m].mode == L.mode && (P->L[m].wr_off >= 0) == (want_grad && l > 0 && !wr_global)) { dup = m; break; }
        }
        if (dup >= 0) {
            L.wt_off = P->L[dup].wt_off; L.bias_off = P->L[dup].bias_off; L.wr_off = P->L[dup].wr_off;
        } else {
            L.wt_off = woff; woff += rup(L.n_in * L.n_out_pad, 4);
            L.bias_off = woff; woff += rup(L.n_out_pad, 4);
            L.wr_off = -1;
            if (want_grad && l > 0 && !wr_global) { L.wr_off = woff; woff += rup(L.n_out * L.n_in_pad, 4); }
        }
    }
    P->w_elems = woff;
    int nthreads = any_gemm ? max_items : TM;
    nthreads = std::min(want_grad ? 256 : 512, std::max(64, rup(nthreads, 32)));
    nthreads = env_int("QB_THREADS", nthreads);
    P->nthreads = nthreads;
    // value kernel: in place when every GEMM layer is a single pass and DOT layers are single-chunk
    int inplace = 1, buf_rows = rup(net->in_dim, TU);
    for (int l = 0; l < net->n_layers; ++l) {
        QbLayerPlan& L = P->L[l];
        buf_rows = std::max(buf_rows, std::max(L.n_in_pad, L.n_out_pad));
        if (L.mode == QB_MODE_GEMM && (L.n_out_pad / TU) * PG > nthreads) inplace = 0;
        if (L.mode == QB_MODE_DOT && L.n_out > L.nj) inplace = 0;
        // dW split-K chunks for narrow layers
        const int patches = ((L.n_out + 3) / 4) * ((L.n_in + 3) / 4);
        int C = 1;
        while (C < 32 && patches * C * 2 <= nthreads && TM / (C * 2) >= PV) C *= 2;
        L.dw_chunks = C;
        L.c_shift = 0;
        while ((1 << L.c_shift) < C) ++L.c_shift;
    }
    if (env_int("QB_NO_INPLACE", 0)) inplace = 0;
    // Warp-synchronous value kernel: when every GEMM layer's unit groups divide a warp, one warp can own WP
    // consecutive points for ALL layers (its lanes cover every unit of those points), so the tile loop needs
    // no block barrier and warps drift apart (MUFU / FMA / LDS phases of different warps overlap).
    P->ws = 0; P->WP = 0;
    if (!want_grad && any_gemm && !env_int("QB_NO_WS", 0)) {
        int ugmax = 0; bool ok = true;
        for (int l = 0; l < net->n_layers; ++l) {
            const QbLayerPlan& L = P->L[l];
            if (L.mode == QB_MODE_GEMM) {
                const int UG = L.n_out_pad / TU;
                if (UG > 32 || 32 % UG) ok = false;
                ugmax = std::max(ugmax, UG);
            } else if (L.n_out > L.nj) ok = false;
        }
        if (ok) {
            const int WP = (32 / ugmax) * TP;
            if (TM % WP == 0 && TM / WP >= 1 && TM / WP <= 16) {
                P->ws = 1; P->WP = WP; inplace = 1;
                nthreads = 32 * (TM / WP);
                P->nthreads = nthreads;
            }
        }
    }
    P->inplace = inplace; P->buf_rows = buf_rows;
    // fused tail: ... -> GEMM hidden layer -> narrow linear output layer (identity, no residual, n_out <= 4)
    P->fuse_tail = 0;
    // (off by default: the first implementation made ptxas keep the accumulators in local memory -- 8x slower,
    //  profiles/r1_notes.md; kept behind QB_TAIL=1 for the next round)
    if (P->ws && net->n_layers >= 2 && env_int("QB_TAIL", 0)) {
        const QbLayerPlan& Lh = P->L[net->n_layers - 2];
        const QbLayerPlan& Lo = P->L[net->n_layers - 1];
        if (Lh.mode == QB_MODE_GEMM && Lo.mode == QB_MODE_DOT && Lo.n_out <= 4 && Lo.act == QB_ACT_IDENTITY &&
            !Lo.has_res && Lh.ug_shift >= 0)
            P->fuse_tail = 1;
    }
    long long act_elems;
    if (!want_grad) {
        act_elems = (long long)(inplace ? 1 : 2) * buf_rows * P->lda;
        P->total_rows = buf_rows; P->d_row = -1;
    } else {
        int row = 0, dmax = 0;
        for (int l = 0; l < net->n_layers; ++l) {
            QbLayerPlan& L = P->L[l];
            L.row_in = row;
            row += (l == 0) ? rup(net->in_dim, TU) : P->L[l - 1].n_out_pad;
            if (L.has_res) dmax = std::max(dmax, L.n_out_pad);
        }
        for (int l = 0; l < net->n_layers; ++l) P->L[l].row_out = (l + 1 < net->n_layers) ? P->L[l + 1].row_in : row;
        row += P->L[net->n_layers - 1].n_out_pad;
        P->d_row = dmax ? row : -1;
        row += dmax;
        P->total_rows = row;
        act_elems = (long long)row * P->lda;
    }
    act_elems += P->lda;      // one pad row: the double-buffered hot loop prefetches one row past the end
    P->smem_bytes = 40 * 8 + (long long)woff * elem + act_elems * elem;
    return P->smem_bytes;
}

// Layer-streamed plan (qb_stream.cuh) for tile size TM: fills `P`, returns its shared-memory bytes, or -1 when the
// activations of one tile leave no room for a ring of chunks of TU rows per layer.
static long long stream_plan_for_tm(const qb_net_t* net, int dtype, bool want_grad, int TM, QbStreamPlan* P) {
    const int elem = dtype == QB_F64 ? 8 : 4;
    const int TU = dtype == QB_F64 ? 4 : 8, TP = 4, VW = dtype == QB_F64 ? 2 : 4, PV = dtype == QB_F64 ? 2 : 4;
    const int LDPAD = dtype == QB_F64 ? 2 : 4;
    const int NT = QS_THREADS, nl = net->n_layers;
    memset(P, 0, sizeof(*P));
    P->n_layers = nl; P->in_dim = net->in_dim; P->out_dim = net->out_dim; P->n_params = net->n_params;
    P->final_exp = net->final_exp; P->want_grad = want_grad ? 1 : 0;
    P->TM = TM; P->lda = TM + LDPAD;
    while ((TP << P->lg_pg) < TM) ++P->lg_pg;
    int widest = net->in_dim, row = 0;
    for (int l = 0; l < nl; ++l) {
        const qb_layer_t& S = net->layers[l];
        QbLayerPlan& L = P->L[l];
        L.n_in = S.n_in; L.n_out = S.n_out; L.n_in_pad = rup(S.n_in, TU); L.n_out_pad = rup(S.n_out, TU);
        L.w_off = S.w_off; L.b_off = S.b_off; L.act = S.act; L.res_step = S.res_step; L.has_res = S.res_step != 0.0;
        L.n_terms = S.n_terms > 1 ? S.n_terms : 0; L.w_stride = S.w_stride; L.b_stride = S.b_stride;
        for (int m = 0; m < QB_MAX_TERMS; ++m) L.coef[m] = S.coef[m];
        L.wt_off = L.wr_off = L.bias_off = -1;
        widest = std::max(widest, S.n_out);
        L.row_in = row; row += S.n_in; L.row_out = row;
        // weight-gradient split of qb_dw_accumulate (as in plan_for_tm)
        const int patches = ((S.n_out + 3) / 4) * ((S.n_in + 3) / 4);
        int C = 1;
        while (C < 32 && patches * C * 2 <= NT && TM / (C * 2) >= PV) C *= 2;
        L.dw_chunks = C; L.c_shift = 0;
        while ((1 << L.c_shift) < C) ++L.c_shift;
        L.ig_shift = -1;
        for (int sft = 0; sft < 16; ++sft) if ((1 << sft) == (S.n_in + 3) / 4) L.ig_shift = sft;
    }
    row += net->layers[nl - 1].n_out;
    P->buf_rows = widest; P->total_rows = row; P->da_rows = want_grad ? widest : 0;
    const long long act_elems = want_grad ? (long long)(row + widest) * P->lda : 2LL * widest * P->lda;
    const long long head = 384;          // 40 doubles of reduction scratch, then the ring's mbarriers
    const long long avail = QB_SMEM_MAX - head - act_elems * elem;
    if (avail <= 0) return -1;
    const long long slot_max = avail / (QS_STAGES * elem) / 4 * 4;
    long long slot = 0;
    int c = 0;
    for (int l = 0; l < nl; ++l) {
        const QbLayerPlan& L = P->L[l];
        QbStreamLayer& S = P->SL[l];
        const int nterm = L.n_terms > 1 ? L.n_terms : 1;
        S.ldw = rup(L.n_in, TU);
        const long long rmax = slot_max / ((long long)nterm * S.ldw) / TU * TU;
        if (rmax < TU) return -1;
        int R = (int)std::min<long long>(rmax, rup(L.n_out, TU));
        S.nch = (int)cdiv(L.n_out, R);
        R = rup((int)cdiv(L.n_out, S.nch), TU);
        S.R = R;
        slot = std::max<long long>(slot, rup(nterm * R * S.ldw, 4));
        const int nsub = (R / TU) * (TM / TP);
        while (S.lg_ks < 5 && qs_items(nsub, S.lg_ks + 1) <= NT && (L.n_in >> (S.lg_ks + 1)) >= 2 * VW) ++S.lg_ks;
        S.kl = rup((int)cdiv(L.n_in, 1 << S.lg_ks), VW);
        const int nsub_b = (int)cdiv(L.n_in, TU) * (TM / TP);
        while (S.lg_bks < 5 && qs_items(nsub_b, S.lg_bks + 1) <= NT && (R >> (S.lg_bks + 1)) >= 2) ++S.lg_bks;
        S.bkl = (int)cdiv(R, 1 << S.lg_bks);
        S.cp_dr = NT / L.n_in; S.cp_di = NT % L.n_in;
        S.fwd_c0 = c; c += S.nch;
        S.bwd_c0 = -1;
    }
    if (want_grad)
        for (int l = nl - 1; l >= 1; --l) { P->SL[l].bwd_c0 = c; c += P->SL[l].nch; }
    P->n_chunks = c;
    P->slot_elems = (int)slot;
    P->ring_off = (int)head;
    P->act_off = P->ring_off + QS_STAGES * (int)slot * elem;
    P->da_off = P->act_off + (want_grad ? row * P->lda * elem : 0);
    P->act_elems = (int)act_elems;
    P->smem_bytes = P->act_off + act_elems * elem;
    return P->smem_bytes;
}

struct QbLaunch { QbPlan plan; int S; long long pts_per_split; bool streamed; QbStreamPlan sp; };

// Networks whose weights do not fit next to one tile of activations: the layer-streamed kernels (qb_stream.cuh).
// The tile is chosen so that the rows of one chunk times its points fill the thread tiles of the block with as little
// split of the reduction as possible (larger tiles at equal fill: fewer passes of the weights through the ring).
static int make_stream_launch(const qb_net_t* net, int dtype, bool want_grad, long long K, long long N, bool force_single,
                              QbLaunch* out) {
    const int TU = dtype == QB_F64 ? 4 : 8, TP = 4;
    const int cands32[] = {128, 64, 32, 16}, cands64[] = {128, 64, 32, 16, 8};
    const int* cands = dtype == QB_F64 ? cands64 : cands32;
    const int nc = dtype == QB_F64 ? 5 : 4, mintm = cands[nc - 1];
    const int cap = std::max(mintm, rup((int)std::min<long long>(N, 256), mintm));
    QbStreamPlan tmp;
    int pick = -1;
    long long best = -1;
    for (int c = 0; c < nc; ++c) {
        const int TM = cands[c];
        if (TM > cap) continue;
        if (stream_plan_for_tm(net, dtype, want_grad, TM, &tmp) < 0) continue;
        long long fill = (long long)QS_THREADS * TU * TP;
        for (int l = 0; l < net->n_layers; ++l)
            if (net->layers[l].n_out > TU) fill = std::min<long long>(fill, (long long)tmp.SL[l].R * TM);
        if (fill > best) { best = fill; pick = TM; }
    }
    if (pick < 0)
        return qb_fail("network too large for the layer-streamed path: the activations of one %s%lld-point tile exceed 227 KB of shared memory",
                       "", mintm);
    stream_plan_for_tm(net, dtype, want_grad, pick, &out->sp);
    out->streamed = true;
    const int TM = pick;
    long long S = 1;
    if (!force_single) {
        // same rule as the resident kernels; with a gradient, the [K,S,P] partial rows stay under 256 MB
        const long long target = (long long)QB_NUM_SMS * 8;
        if (K < target) S = std::max<long long>(1, std::min(cdiv(N, 2LL * TM), cdiv(target, K)));
        if (want_grad) S = std::min<long long>(S, std::max<long long>(1, (256LL << 20) / (K * net->n_params * (dtype == QB_F64 ? 8 : 4))));
    }
    long long pps = rup((int)cdiv(N, S), TM);
    S = cdiv(N, pps);
    out->S = (int)S; out->pts_per_split = pps;
    return 0;
}

static int make_launch(const qb_net_t* net, int dtype, bool want_grad, long long K, long long N, bool force_single,
                       QbLaunch* out) {
    if (validate_net(net)) return -1;
    if (dtype != QB_F32 && dtype != QB_F64) return qb_fail("unknown dtype");
    if (K < 1 || N < 1) return qb_fail("K and N must be positive");
    const int cands32[] = {256, 128, 64, 32}, cands64[] = {128, 64, 32, 16};
    const int* cands = dtype == QB_F64 ? cands64 : cands32;
    const int mintm = cands[3];
    const int cap = std::max(mintm, rup((int)std::min<long long>(N, 256), mintm));
    int forced = env_int("QB_TM", 0);
    // Score every tile size by resident warps per SM (limited by shared memory, 128 registers/thread and 2048
    // threads); ties go to more, smaller blocks for the value kernel (their MUFU / FMA phases overlap better,
    // measured on config 5) and to larger tiles for the gradient kernel (fewer block barriers per point).
    // Gradient only: if nothing fits, drop the shared copy of W used by back-propagation (read from global).
    int pick = -1, best_score = -1;
    bool wr_global = false;
    QbPlan tmp;
    bool any_poly = false;
    for (int l = 0; l < net->n_layers; ++l) any_poly = any_poly || net->layers[l].n_terms > 1;
    for (int g = (want_grad && env_int("QB_WR_GLOBAL", 0)) ? 1 : 0; g < 2 && pick < 0; ++g) {
        if (g == 1 && (!want_grad || any_poly)) break;      // the global-W fallback reads theta directly: no polynomial terms
        for (int c = 0; c < 4; ++c) {
            int TM = cands[c];
            if (forced) TM = forced;
            else if (TM > cap) continue;
            const long long b = plan_for_tm(net, dtype, want_grad, TM, &tmp, g == 1);
            if (b <= QB_SMEM_MAX) {
                const int by_smem = (int)(QB_SMEM_SM / (b + 1024));
                const int by_regs = 512 / tmp.nthreads;
                const int blocks = std::max(1, std::min(std::min(by_smem, by_regs), 16));
                int score;
                if (want_grad) {
                    // gradient kernel (block barriers per layer): the largest tile that still leaves two blocks per SM,
                    // else the largest tile that fits at all
                    score = (blocks >= 2 ? 1000 : 0) + (3 - c);
                } else {
                    score = blocks * (tmp.nthreads / 32) * 16 + std::min(blocks, 8);
                }
                if (score > best_score) { best_score = score; pick = TM; wr_global = (g == 1); }
            }
            if (forced) break;
        }
    }
    out->streamed = false;
    if (pick < 0) {
        if (forced) return qb_fail("network too large for the fused shared-memory path (weights + one tile exceed 227 KB)");
        memset(&out->plan, 0, sizeof(out->plan));
        return make_stream_launch(net, dtype, want_grad, K, N, force_single, out);
    }
    plan_for_tm(net, dtype, want_grad, pick, &out->plan, wr_global);
    const int TM = out->plan.TM;
    long long S = 1;
    if (!force_single) {
        // few chains: split the data axis so that the grid is >= 8 waves of one block per SM (tail effect < 10 %),
        // keeping at least two tiles per block; partial sums / gradients are combined in fixed order by k_finalize
        const long long target = (long long)QB_NUM_SMS * 8;
        if (K < target) S = std::max<long long>(1, std::min(cdiv(N, 2LL * TM), cdiv(target, K)));
        S = env_int("QB_SPLIT", (int)S);
        if (S < 1) S = 1;
    }
    long long pps = rup((int)cdiv(N, S), TM);
    S = cdiv(N, pps);
    out->S = (int)S; out->pts_per_split = pps;
    return 0;
}


// Tensor-core (tcgen05 3xTF32) plan for the value path; returns false when the network is not eligible:
// fp32, >= 3 layers, no residual layers, n_in <= 15, hidden widths multiples of 16 (<= 128), <= 4 outputs.
// allow_v3: 1 = the caller can run the warp-specialised kernels (qb_value_tc3.cu); 2 = the chain kernel (hidden width 64
// only, with room for the chain state, 3 P floats, in shared memory); 3 = kernel 4
static bool make_tc_plan(const qb_net_t* net, int dtype, QbTcPlan* tp, int allow_v3 = 0) {
    memset(tp, 0, sizeof(*tp));
    if (dtype != QB_F32 || env_int("QB_NO_TC", 0)) return false;
    const int nl = net->n_layers;
    if (nl < 3 || net->in_dim > 15 || net->out_dim > 4) return false;
    int kmax = 0, nmax = 0;
    for (int l = 0; l < nl; ++l) {
        const qb_layer_t& S = net->layers[l];
        if (S.res_step != 0.0 || S.n_terms > 1) return false;
        if (l < nl - 1 && (S.n_out % 16 != 0 || S.n_out < 16 || S.n_out > 128)) return false;
        if (l >= 1 && l < nl - 1) { kmax = std::max(kmax, S.n_in); nmax = std::max(nmax, S.n_out); }
    }
    const bool pipe = nl == 3 && net->layers[0].act == net->layers[1].act &&
                      (net->layers[0].act == QB_ACT_TANH || net->layers[0].act == QB_ACT_RELU) && !env_int("QB_NO_PIPE", 0);
    const int grp = std::max(kmax, nmax) > 64 ? 4 : 2;       // column groups = warps per quarter of the tile
    const int cols = 2 * kmax + (pipe ? 2 : 1) * nmax;       // pipelined path: the accumulator is double-buffered
    if (cols > 512) return false;
    tp->n_layers = nl; tp->in_dim = net->in_dim; tp->out_dim = net->out_dim; tp->n_params = net->n_params;
    tp->ni = (net->in_dim < 4 && !(pipe && grp == 4)) ? 4 : 16;
    if (pipe && grp == 4 && net->in_dim <= 11 && net->layers[0].act == QB_ACT_TANH) tp->ni = 12;   // config 3: 10 inputs + bias
    tp->h0 = net->layers[0].n_out; tp->kl = net->layers[nl - 1].n_in;
    tp->act0 = net->layers[0].act; tp->act_last = net->layers[nl - 1].act; tp->final_exp = net->final_exp;
    tp->w0_off = net->layers[0].w_off; tp->b0_off = net->layers[0].b_off;
    tp->wl_off = net->layers[nl - 1].w_off; tp->bl_off = net->layers[nl - 1].b_off;
    tp->a_lo_col = kmax; tp->d_col = 2 * kmax;
    tp->pipe = pipe ? grp : 0;
    tp->tmem_cols = cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512;
    int off = QB_TC_HDR_BYTES;
    for (int l = 1; l < nl - 1; ++l) {
        const qb_layer_t& S = net->layers[l];
        QbTcLayer& L = tp->L[l];
        L.n_in = S.n_in; L.n_out = S.n_out; L.w_off = S.w_off; L.b_off = S.b_off; L.act = S.act;
        L.bhi = off; off += S.n_in * S.n_out * 4;
        L.blo = off; off += S.n_in * S.n_out * 4;
    }
    tp->fl_base = off;
    int f = 0;
    tp->w0 = f; f += tp->h0 * tp->ni;
    for (int l = 1; l < nl - 1; ++l) { tp->L[l].bias = f; f += rup(tp->L[l].n_out, 4); }
    tp->wl = f; f += rup(tp->out_dim * tp->kl, 4);
    tp->bl = f; f += 4;
    long long bytes = (long long)off + (long long)f * 4;
    bytes = (bytes + 15) / 16 * 16;
    tp->ybuf = (int)bytes; bytes += 2 * 3 * 4 * 128 * 4;
    tp->nthreads = tp->pipe ? 128 * tp->pipe : 128;
    if (bytes > QB_SMEM_MAX) return false;
    // tensor memory is 512 columns per SM: request enough shared memory that no more blocks than 512/tmem_cols
    // become resident (a further block would spin in tcgen05.alloc)
    const int max_blocks = 512 / tp->tmem_cols;
    const long long floor_bytes = QB_SMEM_SM / (max_blocks + 1) + 1;
    tp->smem_bytes = (int)std::min<long long>(QB_SMEM_MAX, std::max(bytes, floor_bytes));
    const int v3h = allow_v3 ? qb_tc_v3_shape(*tp) : 0;
    if (v3h && net->layers[1].act == QB_ACT_TANH && !env_int("QB_NO_V3", 0) && !(allow_v3 == 2 && v3h != 64)) {
        // warp-specialised path (qb_tc3.cuh): 4 H/32 compute warps + 1 issue warp, 4 H tensor-memory columns, own layout
        const int H = v3h, K0 = H == 64 ? 8 : 16, G = H / 32;
        tp->v3 = H == 64 ? 1 : 2; tp->nthreads = 128 * G + 32; tp->tmem_cols = 4 * H;
        int o = QB_TC_HDR_BYTES;
        tp->v3_w1 = o; o += 3 * H * H * 2;
        tp->v3_w0 = o; o += 2 * H * K0 * 4;
        tp->v3_x = o; o += 3 * 2 * 128 * K0 * 4;
        tp->fl_base = o;
        tp->L[1].bias = 0; tp->wl = H; tp->bl = 2 * H; tp->v3_c1 = 2 * H + 4;
        o += (2 * H + 8) * 4;
        tp->ybuf = o; o += 4 * (G - 1) * 128 * 4;
        tp->v3_xbar = o; o += 32;
        tp->v3_state = o;
        if (allow_v3 == 2) o += 3 * ((net->n_params + 3) / 4 * 4) * 4;
        const int max_blocks3 = 512 / tp->tmem_cols;
        tp->smem_bytes = (int)std::max<long long>(o, QB_SMEM_SM / (max_blocks3 + 1) + 1);
        if (tp->smem_bytes > (QB_SMEM_SM - 1024 * max_blocks3) / max_blocks3) return make_tc_plan(net, dtype, tp, 0);     // the blocks must fit
    }
    return true;
}

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
    qb_tc_fini(tp, cx);
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
    if (make_launch(net, dtype, want_grad, K, data->n, false, &L)) return -1;
    const size_t need = qb_eval_workspace_bytes(net, dtype, K, data->n, want_grad);
    if (ws_bytes < need || (need && !ws)) return qb_fail("workspace too small%s (need %lld bytes)", "", (long long)need);
    EvalArgs<T> a;
    a.theta = (const T*)theta; a.x = (const T*)data->x; a.y = (const T*)data->y;
    a.xs = x_stride; a.ys = y_stride;
    a.K = K; a.N = data->n; a.S = L.S; a.pps = L.pts_per_split;
    a.part = (double*)ws;
    a.grad = (T*)grad;
    const size_t part_bytes = ((size_t)K * L.S * sizeof(double) + 255) / 256 * 256;
    a.gpart = (L.S > 1 && want_grad) ? (T*)((char*)ws + part_bytes) : nullptr;
    a.lp = lp; a.lk = lik_dev(lik);
    a.xsplit = nullptr;
    dim3 grid((unsigned)K, (unsigned)L.S);
    if (L.streamed) {
        const dim3 sgrid((unsigned)(K * L.S));
        if (want_grad) {
            if (set_smem(k_logpost_stream<T, true>, L.sp.smem_bytes)) return -2;
            k_logpost_stream<T, true><<<sgrid, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, a);
        } else {
            if (set_smem(k_logpost_stream<T, false>, L.sp.smem_bytes)) return -2;
            k_logpost_stream<T, false><<<sgrid, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, a);
        }
    } else if (want_grad) {
        QbTcgPlan tg;
        QbTg8Plan t8;
        if (qb_tg8_make_plan(net, dtype, &t8)) {
            // tanh nets of width 64 / 128: fp16-split operands, scaled with max |x|, max |y| (8 bytes at the end of the workspace)
            if (launch_grad_tc128<T>(t8, a, (char*)ws + need - QB_TG8_SCRATCH_BYTES, grid, st)) return -2;
            g_launches += 1;
        } else if (qb_tcg_make_plan(net, dtype, &tg)) {
            if (launch_grad_tc<T>(tg, a, grid, st)) return -2;
        } else {
            if (set_smem(k_logpost_grad<T>, L.plan.smem_bytes)) return -2;
            k_logpost_grad<T><<<grid, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, a);
        }
    } else {
        QbTcPlan tp;
        if (make_tc_plan(net, dtype, &tp, 1)) {
            // hot shape with shared data: x goes to the kernel as ready-made operand tiles at the end of the workspace
            if (tp.v3 && x_stride == 0) a.xsplit = (const T*)((char*)ws + need - qb_tc3_xsplit_bytes(data->n, tp.v3 == 1 ? 8 : 16));
            if (launch_logpost_tc<T>(tp, a, grid, st)) return -2;
        } else {
            if (set_smem(k_logpost<T>, L.plan.smem_bytes)) return -2;
            k_logpost<T><<<grid, L.plan.nthreads, L.plan.smem_bytes, st>>>(L.plan, a);
        }
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

extern "C" size_t qb_eval_workspace_bytes(const qb_net_t* net, int dtype, int64_t K, int64_t N, int want_grad) {
    QbLaunch L;
    if (make_launch(net, dtype, want_grad != 0, K, N, false, &L)) return 0;
    size_t b = ((size_t)K * L.S * sizeof(double) + 255) / 256 * 256;
    if (want_grad && L.S > 1) b += (size_t)K * L.S * net->n_params * (dtype == QB_F64 ? 8 : 4);
    if (L.streamed) return b;
    QbTcPlan tp;
    if (!want_grad && make_tc_plan(net, dtype, &tp, 1) && tp.v3) b = (b + 255) / 256 * 256 + qb_tc3_xsplit_bytes(N, tp.v3 == 1 ? 8 : 16);
    QbTcgPlan tg;
    QbTg8Plan t8;
    (void)tg;
    if (want_grad && qb_tg8_make_plan(net, dtype, &t8)) b = (b + 255) / 256 * 256 + QB_TG8_SCRATCH_BYTES;
    return b;
}

extern "C" int qb_plan_info(const qb_net_t* net, int dtype, int64_t K, int64_t N, int want_grad, int64_t* out) {
    QbLaunch L;
    if (make_launch(net, dtype, want_grad != 0, K, N, false, &L)) return -1;
    out[0] = L.plan.TM; out[1] = L.plan.nthreads; out[2] = L.plan.smem_bytes; out[3] = L.S;
    out[4] = (int64_t)K * L.S; out[5] = L.plan.inplace; out[6] = 0; out[7] = 0;
    if (L.streamed) {
        // CUDA cores, weights streamed through shared memory (qb_stream.cuh): out[6] = 5
        out[0] = L.sp.TM; out[1] = QS_THREADS; out[2] = L.sp.smem_bytes; out[5] = 0; out[6] = 5;
        return 0;
    }
    QbTcgPlan tg;
    QbTg8Plan t8;
    if (want_grad && qb_tg8_make_plan(net, dtype, &t8)) {
        // gradient path on the tensor cores, fp16-split operands (qb_tg8.cuh: tanh nets of width 64 / 128): out[6] = 4
        out[0] = 128; out[1] = t8.nthreads; out[2] = t8.smem_bytes; out[5] = 0; out[6] = 4; out[7] = t8.tmem_cols;
    } else if (want_grad && qb_tcg_make_plan(net, dtype, &tg)) {
        // gradient path on the tensor cores, 3xTF32 (qb_tcg.cuh: widths 32 / 64, tanh / relu): out[6] = 3
        out[0] = 128; out[1] = tg.nthreads; out[2] = tg.smem_bytes; out[5] = 0; out[6] = 3; out[7] = tg.tmem_cols;
    }
    QbTcPlan tp;
    if (!want_grad && make_tc_plan(net, dtype, &tp, 1)) {
        // value path on the tensor cores: 128-point tiles, 128 or 256 threads, out[6] = 1 + pipelined flag,
        // out[7] = tensor-memory columns per block
        out[0] = 128; out[1] = tp.nthreads; out[2] = tp.smem_bytes; out[5] = 0; out[6] = tp.pipe ? 2 : 1; out[7] = tp.tmem_cols;
    }
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
// Plan for tile size TM: every layer in GEMM mode with TU x 4 thread tiles; returns the shared-memory bytes.
static long long hvp_plan_for_tm(const qb_net_t* net, int dtype, int TM, QbHvpPlan* H) {
    const int elem = dtype == QB_F64 ? 8 : 4;
    const int TU = dtype == QB_F64 ? 4 : 8, LDPAD = dtype == QB_F64 ? 2 : 4, PV = dtype == QB_F64 ? 2 : 4, TP = 4;
    const int nl = net->n_layers, PG = TM / TP;
    memset(H, 0, sizeof(*H));
    QbPlan* P = &H->P;
    P->n_layers = nl; P->in_dim = net->in_dim; P->out_dim = net->out_dim;
    P->n_params = net->n_params; P->final_exp = net->final_exp;
    P->TM = TM; P->lda = TM + LDPAD; P->want_grad = 1; P->elem_size = elem; P->tpg = TP;
    int woff = 0, max_items = 0, dmax = 0;
    for (int l = 0; l < nl; ++l) {
        const qb_layer_t& S = net->layers[l];
        QbLayerPlan& L = P->L[l];
        L.n_in = S.n_in; L.n_out = S.n_out; L.n_in_pad = rup(S.n_in, TU); L.n_out_pad = rup(S.n_out, TU);
        L.w_off = S.w_off; L.b_off = S.b_off; L.act = S.act; L.res_step = S.res_step; L.has_res = S.res_step != 0.0;
        L.n_terms = S.n_terms > 1 ? S.n_terms : 0; L.w_stride = S.w_stride; L.b_stride = S.b_stride;
        for (int m = 0; m < QB_MAX_TERMS; ++m) L.coef[m] = S.coef[m];
        L.mode = QB_MODE_GEMM; L.nj = 4;
        if (L.has_res) { P->has_res = 1; dmax = std::max(dmax, L.n_out_pad); }
        L.ug_shift = L.ugi_shift = L.ig_shift = -1;
        for (int sft = 0; sft < 16; ++sft) {
            if ((1 << sft) == L.n_out_pad / TU) L.ug_shift = sft;
            if ((1 << sft) == L.n_in_pad / TU) L.ugi_shift = sft;
            if ((1 << sft) == (S.n_in + 3) / 4) L.ig_shift = sft;
        }
        max_items = std::max(max_items, (L.n_out_pad / TU) * PG);
        if (l > 0) max_items = std::max(max_items, (L.n_in_pad / TU) * PG);
        // [W^T ; V^T], [b ; v_b], and for l > 0 [W ; V] (qb_hvp.cuh)
        L.wt_off = woff; woff += rup((L.n_in_pad + L.n_in) * L.n_out_pad, 4);
        L.bias_off = woff; woff += rup(2 * L.n_out_pad, 4);
        L.wr_off = -1;
        if (l > 0) { L.wr_off = woff; woff += rup((L.n_out_pad + L.n_out) * L.n_in_pad, 4); }
    }
    P->w_elems = woff;
    const int nthreads = std::min(256, std::max(64, rup(max_items, 32)));
    P->nthreads = nthreads;
    // activation rows: per layer boundary the tangent rows, then the activation rows
    int row = 0;
    for (int b = 0; b <= nl; ++b) {
        const int npad = b == 0 ? P->L[0].n_in_pad : P->L[b - 1].n_out_pad;
        row += npad;                                   // tangent rows
        if (b < nl) P->L[b].row_in = row;
        if (b > 0) P->L[b - 1].row_out = row;
        row += npad;
    }
    P->d_row = dmax ? row : -1; row += dmax;
    H->dd_row = dmax ? row : -1; row += dmax;
    P->total_rows = row;
    P->buf_rows = row;
    for (int l = 0; l < nl; ++l) {
        QbLayerPlan& L = P->L[l];
        const int patches = ((L.n_out + 3) / 4) * ((L.n_in + 3) / 4);
        int C = 1;
        while (C < 32 && patches * C * 2 <= nthreads && TM / (C * 2) >= PV) C *= 2;
        L.dw_chunks = C;
        L.c_shift = 0;
        while ((1 << L.c_shift) < C) ++L.c_shift;
        H->LA[l] = L; H->LA[l].row_out = L.row_out - L.n_out_pad;
        H->LB[l] = L; H->LB[l].row_in = L.row_in - L.n_in_pad; H->LB[l].b_off = -1;
    }
    // one pad row: the double-buffered hot loop prefetches one row past the end
    P->smem_bytes = (long long)woff * elem + (long long)(row + 1) * P->lda * elem;
    return P->smem_bytes;
}

struct QbHvpLaunch { QbHvpPlan H; int S; long long pps; };

static int make_hvp_launch(const qb_net_t* net, int dtype, long long K, long long N, QbHvpLaunch* out) {
    if (validate_net(net)) return -1;
    if (dtype != QB_F32 && dtype != QB_F64) return qb_fail("unknown dtype");
    if (K < 1 || N < 1) return qb_fail("K and N must be positive");
    const int cands32[] = {128, 64, 32, 16}, cands64[] = {64, 32, 16, 8};
    const int* cands = dtype == QB_F64 ? cands64 : cands32;
    const int mintm = cands[3];
    const int cap = std::max(mintm, rup((int)std::min<long long>(N, 256), mintm));
    // The largest tile that fits.  Measured on a B200 (DESIGN.md section 4f, profiles/r4_hessian_bench_*.json): more,
    // smaller blocks per SM lose, e.g. fp32 config 2 at TM 16 (six 64-thread blocks per SM) reaches 0.06 of the FMA peak
    // against 0.20 at TM 128, and fp32 config 5 at TM 16 0.07 against 0.30 at TM 128.
    int pick = -1;
    for (int c = 0; c < 4 && pick < 0; ++c) {
        const int TM = cands[c];
        if (TM <= cap && hvp_plan_for_tm(net, dtype, TM, &out->H) <= QB_SMEM_MAX) pick = TM;
    }
    if (pick < 0) {
        hvp_plan_for_tm(net, dtype, mintm, &out->H);
        return qb_fail("network too large for the Hessian-vector kernel: its weights, one direction and a %s%lld-point tile "
                       "exceed 227 KB of shared memory (use the diagonal curvature)", "", mintm);
    }
    hvp_plan_for_tm(net, dtype, pick, &out->H);
    // few directions: split the data axis as kernel 2 does; the [K,S,P] partial rows stay under 256 MB
    long long S = 1;
    const long long target = (long long)QB_NUM_SMS * 8;
    if (K < target) S = std::max<long long>(1, std::min(cdiv(N, 2LL * pick), cdiv(target, K)));
    S = std::min<long long>(S, std::max<long long>(1, (256LL << 20) / (K * net->n_params * (dtype == QB_F64 ? 8 : 4))));
    const long long pps = rup((int)cdiv(N, S), pick);
    out->S = (int)cdiv(N, pps); out->pps = pps;
    return 0;
}

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

extern "C" size_t qb_hvp_workspace_bytes(const qb_net_t* net, int dtype, int64_t K, int64_t N) {
    if (K == 0) return 0;
    QbHvpLaunch L;
    if (make_hvp_launch(net, dtype, K, N, &L)) return 0;
    return L.S > 1 ? (size_t)K * L.S * net->n_params * (dtype == QB_F64 ? 8 : 4) : 0;
}

extern "C" int qb_hvp_plan_info(const qb_net_t* net, int dtype, int64_t K, int64_t N, int64_t* out) {
    QbHvpLaunch L;
    if (make_hvp_launch(net, dtype, K, N, &L)) return -1;
    out[0] = L.H.P.TM; out[1] = L.H.P.nthreads; out[2] = L.H.P.smem_bytes; out[3] = L.S; out[4] = (int64_t)K * L.S;
    return 0;
}

template <typename T>
static int run_hvp(const qb_net_t* net, int dtype, const void* theta, const void* v, int64_t col0, int64_t K,
                   const qb_data_t* data, const qb_lik_t* lik, void* hv, void* ws, size_t ws_bytes, cudaStream_t st) {
    QbHvpLaunch L;
    if (make_hvp_launch(net, dtype, K, data->n, &L)) return -1;
    const size_t need = qb_hvp_workspace_bytes(net, dtype, K, data->n);
    if (ws_bytes < need || (need && !ws)) return qb_fail("workspace too small%s (need %lld bytes)", "", (long long)need);
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
// qb_dw_accumulate's split of one re-pointed factor pass (as in plan_for_tm, for the pass's own shape)
static void kfac_dw_split(QbLayerPlan& L, int nthreads, int TM, int PV) {
    const int patches = ((L.n_out + 3) / 4) * ((L.n_in + 3) / 4);
    int C = 1;
    while (C < 32 && patches * C * 2 <= nthreads && TM / (C * 2) >= PV) C *= 2;
    L.dw_chunks = C;
    L.c_shift = 0;
    while ((1 << L.c_shift) < C) ++L.c_shift;
    L.ig_shift = -1;
    for (int sft = 0; sft < 16; ++sft)
        if ((1 << sft) == (L.n_in + 3) / 4) L.ig_shift = sft;
}

struct QbKfacLaunch { QbKfacPlan K; int S; long long pps; };

// Kernel 2's resident CUDA-core plan for one theta, the factor passes of every layer, and the N-split: one block per
// split, the [S, F] partial rows (dtype) under 256 MB.
static int make_kfac_launch(const qb_net_t* net, int dtype, long long N, QbKfacLaunch* out) {
    if (validate_net(net)) return -1;
    if (dtype != QB_F32 && dtype != QB_F64) return qb_fail("unknown dtype");
    for (int l = 0; l < net->n_layers; ++l) {
        const qb_layer_t& S = net->layers[l];
        if (S.n_terms > 1)
            return qb_fail("Kronecker factors: layer %s%lld has polynomial-in-depth weights (n_terms >= 2); every layer "
                           "must own its weights", "", l);
        for (int m = 0; m < l; ++m)
            if (net->layers[m].w_off == S.w_off)
                return qb_fail("Kronecker factors: layer %s%lld shares its weights with an earlier layer; every layer must "
                               "own its weights", "", l);
    }
    QbLaunch L;
    if (make_launch(net, dtype, true, 1, N, true, &L)) return -1;
    if (L.streamed)
        return qb_fail("Kronecker factors: the network's weights do not fit in shared memory next to one tile of "
                       "activations, and the layer-streamed path (plan code 5) has no factor kernel");
    memset(&out->K, 0, sizeof(out->K));
    out->K.P = L.plan;
    const QbPlan& P = out->K.P;
    const int PV = dtype == QB_F64 ? 2 : 4;
    int off = 0;
    for (int l = 0; l < P.n_layers; ++l) {
        const QbLayerPlan& B = P.L[l];
        QbLayerPlan& A = out->K.LA[l];
        A = B;
        A.n_out = B.n_in; A.n_out_pad = B.n_in_pad; A.row_out = B.row_in;
        A.n_terms = 0;
        A.w_off = off; off += B.n_in * B.n_in;
        A.b_off = -1;
        if (B.b_off >= 0) { A.b_off = off; off += B.n_in; }
        kfac_dw_split(A, P.nthreads, P.TM, PV);
        QbLayerPlan& G = out->K.LG[l];
        G = B;
        G.n_in = B.n_out; G.n_in_pad = B.n_out_pad; G.row_in = B.row_out;
        G.n_terms = 0;
        G.w_off = off; off += B.n_out * B.n_out;
        G.b_off = -1;
        kfac_dw_split(G, P.nthreads, P.TM, PV);
    }
    out->K.n_factors = off;
    const int TM = P.TM;
    const long long row_bytes = (long long)off * (dtype == QB_F64 ? 8 : 4);
    long long S = std::max<long long>(1, std::min(cdiv(N, 2LL * TM), (long long)QB_NUM_SMS * 8));
    S = std::min<long long>(S, std::max<long long>(1, (256LL << 20) / row_bytes));
    const long long pps = rup((int)cdiv(N, S), TM);
    out->S = (int)cdiv(N, pps); out->pps = pps;
    return 0;
}

template <typename T> struct KfacArgs {
    const T* theta; const T* x; const T* y;
    long long N; int S; long long pps;
    T* part;            // [S, F]
    double* factors;    // [F]
    double inv_sigma2;
};

// fp32: one block per SM in the register budget (157 registers; at two, 128 registers spill the fp32 factor passes)
template <typename T>
__global__ void __launch_bounds__(256, sizeof(T) == 8 ? 2 : 1) k_logpost_kfac(const __grid_constant__ QbKfacPlan K, const KfacArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const QbSmem S = qb_carve<T>(K.P, smem_raw);
    const long long s = blockIdx.x;
    const long long n0 = s * a.pps, n1 = min(a.N, n0 + a.pps);
    qb_kfac_eval<T>(K, S, a.theta, a.x, a.y, n0, n1, a.inv_sigma2, a.part + s * K.n_factors);
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

extern "C" size_t qb_kfac_workspace_bytes(const qb_net_t* net, int dtype, int64_t N) {
    if (N <= 0) return 0;
    QbKfacLaunch L;
    if (make_kfac_launch(net, dtype, N, &L)) return 0;
    return (size_t)L.S * L.K.n_factors * (dtype == QB_F64 ? 8 : 4);
}

extern "C" int qb_kfac_plan_info(const qb_net_t* net, int dtype, int64_t N, int64_t* out) {
    QbKfacLaunch L;
    if (make_kfac_launch(net, dtype, std::max<int64_t>(N, 1), &L)) return -1;
    out[0] = L.K.P.TM; out[1] = L.K.P.nthreads; out[2] = L.K.P.smem_bytes; out[3] = L.S; out[4] = L.K.n_factors;
    return 0;
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
    const size_t need = (size_t)L.S * L.K.n_factors * sizeof(T);
    if (ws_bytes < need || !ws) return qb_fail("workspace too small%s (need %lld bytes)", "", (long long)need);
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
    if constexpr (TC) qb_tc_fini(tp, cx);
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
    if (make_launch(net, dtype, true, ch->K, data->n, true, &L)) return -1;
    if (!hm->grad_cur || !hm->mom || !hm->prop || !hm->grad_prop) return qb_fail("hmc state has NULL arrays");
    if (hm->method == 0 && hm->L < 1) return qb_fail("HMC needs L >= 1");
    ChainArgs<T> c; fill_chain_args<T>(c, data, lik, ch, rng, rec, t_start, nsteps, init_lp);
    HmcArgs<T> h;
    h.method = hm->method; h.L = hm->L; h.eps = hm->epsilon;
    h.gcur = (T*)hm->grad_cur; h.mom = (T*)hm->mom; h.prop = (T*)hm->prop; h.gprop = (T*)hm->grad_prop;
    QbTcgPlan tg;
    QbTg8Plan t8;
    if (L.streamed) {
        if (set_smem(k_hmc_stream<T>, L.sp.smem_bytes)) return -2;
        k_hmc_stream<T><<<(unsigned)ch->K, QS_THREADS, L.sp.smem_bytes, st>>>(L.sp, c, h);
    } else if (qb_tg8_make_plan(net, dtype, &t8)) {
        if (launch_hmc_tc128<T>(t8, c, h, ch->K, st)) return -2;
        g_launches += 1;
    } else if (qb_tcg_make_plan(net, dtype, &tg)) {
        if (launch_hmc_tc<T>(tg, c, h, ch->K, st)) return -2;
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
    qb_tc_fini(tp, cx);
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
        const long long tiles = cdiv(N, SP.TM);
        long long chunks = std::max<long long>(1, std::min<long long>(tiles, cdiv((long long)QB_NUM_SMS * 2, M)));
        a.tiles_per_block = cdiv(tiles, chunks);
        chunks = cdiv(tiles, a.tiles_per_block);
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
        const long long t128 = cdiv(N, 128);
        long long ch = std::max<long long>(1, std::min<long long>(t128, cdiv((long long)QB_NUM_SMS * 2 * 8, M)));
        a.tiles_per_block = cdiv(t128, ch);
        ch = cdiv(t128, a.tiles_per_block);
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
    if (!fused) {
        chunks = std::max<long long>(1, std::min<long long>(tiles, cdiv((long long)QB_NUM_SMS * 8, M)));
        a.tiles_per_block = cdiv(tiles, chunks);
        chunks = cdiv(tiles, a.tiles_per_block);
    }
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
    const int blocks = QB_NUM_SMS * 8, threads = 256;
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
