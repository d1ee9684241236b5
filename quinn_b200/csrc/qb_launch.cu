// quinn_b200: launch planning (host only, declarations in qb_launch.h): every planner and every C ABI function that only
// plans.  This unit defines no kernel.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>

#include "qb_launch.h"
#include "qb_value_tc3.h"
#include "qb_grad_tc.h"
#include "qb_grad_tc128.h"

extern thread_local char g_err[512];       // qb_kernels.cu

int qb_fail(const char* fmt, const char* a, long long b) {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return -1;
}

int qb_env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return (s && *s) ? atoi(s) : dflt;
}

static inline int rup(int v, int m) { return (v + m - 1) / m * m; }
static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

int qb_num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) n = v;
        else n = 148;
    }
    return n;
}

// per-dtype tiling constants: element bytes, units per thread tile, activation row padding, elements per 128-bit vector
struct QbDt { int elem, TU, LDPAD, PV; };
static QbDt dt_of(int dtype) { return dtype == QB_F64 ? QbDt{8, 4, 2, 2} : QbDt{4, 8, 4, 4}; }

// log2(v) if v is a power of two below 2^16, else -1
static int exact_log2(int v) {
    for (int sft = 0; sft < 16; ++sft)
        if ((1 << sft) == v) return sft;
    return -1;
}

// the layer descriptor part of a layer plan (units padded to TU)
static void copy_layer(const qb_layer_t& S, int TU, QbLayerPlan& L) {
    L.n_in = S.n_in; L.n_out = S.n_out; L.n_in_pad = rup(S.n_in, TU); L.n_out_pad = rup(S.n_out, TU);
    L.w_off = S.w_off; L.b_off = S.b_off; L.act = S.act; L.res_step = S.res_step; L.has_res = S.res_step != 0.0;
    L.n_terms = S.n_terms > 1 ? S.n_terms : 0; L.w_stride = S.w_stride; L.b_stride = S.b_stride;
    for (int m = 0; m < QB_MAX_TERMS; ++m) L.coef[m] = S.coef[m];
}

// split of qb_dw_accumulate for the layer's shape: split-K chunks of the points for narrow layers, while the patches
// times chunks fill the block and every chunk keeps a vector of points
static void dw_split(QbLayerPlan& L, int nthreads, int TM, int PV) {
    const int patches = ((L.n_out + 3) / 4) * ((L.n_in + 3) / 4);
    int C = 1;
    while (C < 32 && patches * C * 2 <= nthreads && TM / (C * 2) >= PV) C *= 2;
    L.dw_chunks = C;
    L.c_shift = exact_log2(C);
    L.ig_shift = exact_log2((L.n_in + 3) / 4);
}

// Wanted split count of the data axis: with few chains the grid gets >= 8 waves of one block per SM (tail effect
// < 10 %), keeping at least two tiles per split; row_bytes > 0: the [K, S] partial rows of row_bytes each stay under
// 256 MB.  The splits are combined in fixed order, so S fixes the summation order of a result.
static long long want_splits(long long N, int TM, long long K, long long row_bytes) {
    const long long target = (long long)qb_num_sms() * 8;
    long long S = 1;
    if (K < target) S = std::max<long long>(1, std::min(cdiv(N, 2LL * TM), cdiv(target, K)));
    if (row_bytes) S = std::min<long long>(S, std::max<long long>(1, (256LL << 20) / (K * row_bytes)));
    return S;
}

// S splits rounded to whole tiles: pps points per split, and the number of splits that then hold points
static void fit_splits(long long N, int TM, long long S, int* S_out, long long* pps) {
    *pps = rup((int)cdiv(N, S), TM);
    *S_out = (int)cdiv(N, *pps);
}

long long qb_tile_chunks(long long tiles, long long blocks_wanted, long long M, long long* tiles_per_block) {
    const long long ch = std::max<long long>(1, std::min<long long>(tiles, cdiv(blocks_wanted, M)));
    *tiles_per_block = cdiv(tiles, ch);
    return cdiv(tiles, *tiles_per_block);
}

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

// the network-wide fields of a CUDA-core plan (cleared first)
static void plan_head(const qb_net_t* net, const QbDt& D, int TM, bool want_grad, int TP, QbPlan* P) {
    memset(P, 0, sizeof(*P));
    P->n_layers = net->n_layers; P->in_dim = net->in_dim; P->out_dim = net->out_dim;
    P->n_params = net->n_params; P->final_exp = net->final_exp;
    P->TM = TM; P->lda = TM + D.LDPAD; P->want_grad = want_grad ? 1 : 0; P->elem_size = D.elem; P->tpg = TP;
}

// the arguments every planner takes: a valid network, a known dtype, K and N positive
static int check_args(const qb_net_t* net, int dtype, long long K, long long N) {
    if (validate_net(net)) return -1;
    if (dtype != QB_F32 && dtype != QB_F64) return qb_fail("unknown dtype");
    if (K < 1 || N < 1) return qb_fail("K and N must be positive");
    return 0;
}

// =================================================================================================
// kernels 1-4 on the CUDA cores
// =================================================================================================
// Fill `P` for tile size TM; returns smem bytes (or -1 if a constraint fails).
static long long plan_for_tm(const qb_net_t* net, int dtype, bool want_grad, int TM, QbPlan* P, bool wr_global = false) {
    const QbDt D = dt_of(dtype);
    const int TU = D.TU;
    // gradient kernel: TU x 4 thread tiles (twice the threads per tile) when some layer is >= 64 wide, else TU x 8
    int widest = 0;
    for (int l = 0; l < net->n_layers; ++l) widest = std::max(widest, net->layers[l].n_out);
    const int tpg = (dtype == QB_F64 || widest >= 64) ? 4 : 8;
    const int TP = want_grad ? qb_env_int("QB_TPG", tpg) : TU;
    plan_head(net, D, TM, want_grad, TP, P);
    const int PG = TM / TP;
    int max_items = 0, woff = 0;
    bool any_gemm = false;
    for (int l = 0; l < net->n_layers; ++l) {
        const qb_layer_t& S = net->layers[l];
        QbLayerPlan& L = P->L[l];
        copy_layer(S, TU, L);
        if (L.has_res) P->has_res = 1;
        const int UG = L.n_out_pad / TU;
        L.ug_shift = exact_log2(UG); L.ugi_shift = exact_log2(L.n_in_pad / TU);
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
    nthreads = qb_env_int("QB_THREADS", nthreads);
    P->nthreads = nthreads;
    // value kernel: in place when every GEMM layer is a single pass and DOT layers are single-chunk
    int inplace = 1, buf_rows = rup(net->in_dim, TU);
    for (int l = 0; l < net->n_layers; ++l) {
        QbLayerPlan& L = P->L[l];
        buf_rows = std::max(buf_rows, std::max(L.n_in_pad, L.n_out_pad));
        if (L.mode == QB_MODE_GEMM && (L.n_out_pad / TU) * PG > nthreads) inplace = 0;
        if (L.mode == QB_MODE_DOT && L.n_out > L.nj) inplace = 0;
        dw_split(L, nthreads, TM, D.PV);
    }
    if (qb_env_int("QB_NO_INPLACE", 0)) inplace = 0;
    // Warp-synchronous value kernel: when every GEMM layer's unit groups divide a warp, one warp can own WP
    // consecutive points for ALL layers (its lanes cover every unit of those points), so the tile loop needs
    // no block barrier and warps drift apart (MUFU / FMA / LDS phases of different warps overlap).
    P->ws = 0; P->WP = 0;
    if (!want_grad && any_gemm && !qb_env_int("QB_NO_WS", 0)) {
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
    if (P->ws && net->n_layers >= 2 && qb_env_int("QB_TAIL", 0)) {
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
    P->smem_bytes = 40 * 8 + (long long)woff * D.elem + act_elems * D.elem;
    return P->smem_bytes;
}

// Layer-streamed plan (qb_stream.cuh) for tile size TM: fills `P`, returns its shared-memory bytes, or -1 when the
// activations of one tile leave no room for a ring of chunks of TU rows per layer.
static long long stream_plan_for_tm(const qb_net_t* net, int dtype, bool want_grad, int TM, QbStreamPlan* P) {
    const QbDt D = dt_of(dtype);
    const int elem = D.elem, TU = D.TU, TP = 4, VW = D.PV;
    const int NT = QS_THREADS, nl = net->n_layers;
    memset(P, 0, sizeof(*P));
    P->n_layers = nl; P->in_dim = net->in_dim; P->out_dim = net->out_dim; P->n_params = net->n_params;
    P->final_exp = net->final_exp; P->want_grad = want_grad ? 1 : 0;
    P->TM = TM; P->lda = TM + D.LDPAD;
    while ((TP << P->lg_pg) < TM) ++P->lg_pg;
    int widest = net->in_dim, row = 0;
    for (int l = 0; l < nl; ++l) {
        const qb_layer_t& S = net->layers[l];
        QbLayerPlan& L = P->L[l];
        copy_layer(S, TU, L);
        L.wt_off = L.wr_off = L.bias_off = -1;
        widest = std::max(widest, S.n_out);
        L.row_in = row; row += S.n_in; L.row_out = row;
        dw_split(L, NT, TM, D.PV);
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

// Networks whose weights do not fit next to one tile of activations: the layer-streamed kernels (qb_stream.cuh).
// The tile is chosen so that the rows of one chunk times its points fill the thread tiles of the block with as little
// split of the reduction as possible (larger tiles at equal fill: fewer passes of the weights through the ring).
static int make_stream_launch(const qb_net_t* net, int dtype, bool want_grad, long long N, QbLaunch* out) {
    const int TU = dt_of(dtype).TU, TP = 4;
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
    return 0;
}

int make_launch(const qb_net_t* net, int dtype, bool want_grad, long long K, long long N, bool force_single, QbLaunch* out) {
    if (check_args(net, dtype, K, N)) return -1;
    const int cands32[] = {256, 128, 64, 32}, cands64[] = {128, 64, 32, 16};
    const int* cands = dtype == QB_F64 ? cands64 : cands32;
    const int mintm = cands[3];
    const int cap = std::max(mintm, rup((int)std::min<long long>(N, 256), mintm));
    int forced = qb_env_int("QB_TM", 0);
    // Score every tile size by resident warps per SM (limited by shared memory, 128 registers/thread and 2048
    // threads); ties go to more, smaller blocks for the value kernel (their MUFU / FMA phases overlap better,
    // measured on config 5) and to larger tiles for the gradient kernel (fewer block barriers per point).
    // Gradient only: if nothing fits, drop the shared copy of W used by back-propagation (read from global).
    int pick = -1, best_score = -1;
    bool wr_global = false;
    QbPlan tmp;
    bool any_poly = false;
    for (int l = 0; l < net->n_layers; ++l) any_poly = any_poly || net->layers[l].n_terms > 1;
    for (int g = (want_grad && qb_env_int("QB_WR_GLOBAL", 0)) ? 1 : 0; g < 2 && pick < 0; ++g) {
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
    out->streamed = pick < 0;
    long long S;
    if (out->streamed) {
        if (forced) return qb_fail("network too large for the fused shared-memory path (weights + one tile exceed 227 KB)");
        memset(&out->plan, 0, sizeof(out->plan));
        if (make_stream_launch(net, dtype, want_grad, N, out)) return -1;
        // with a gradient, the [K,S,P] partial rows stay under 256 MB
        S = want_splits(N, out->sp.TM, K, want_grad ? (long long)net->n_params * dt_of(dtype).elem : 0);
    } else {
        plan_for_tm(net, dtype, want_grad, pick, &out->plan, wr_global);
        S = std::max(1, qb_env_int("QB_SPLIT", (int)want_splits(N, pick, K, 0)));
    }
    fit_splits(N, out->streamed ? out->sp.TM : pick, force_single ? 1 : S, &out->S, &out->pts_per_split);
    return 0;
}

// =================================================================================================
// kernels 1 and 2: the kernel of a call and the workspace of qb_logpost*
// =================================================================================================
// Tensor-core (tcgen05 3xTF32) plan for the value path; returns false when the network is not eligible:
// fp32, >= 3 layers, no residual layers, n_in <= 15, hidden widths multiples of 16 (<= 128), <= 4 outputs.
// allow_v3: 1 = the caller can run the warp-specialised kernels (qb_value_tc3.cu); 2 = the chain kernel (hidden width 64
// only, with room for the chain state, 3 P floats, in shared memory); 3 = kernel 4
bool make_tc_plan(const qb_net_t* net, int dtype, QbTcPlan* tp, int allow_v3) {
    memset(tp, 0, sizeof(*tp));
    if (dtype != QB_F32 || qb_env_int("QB_NO_TC", 0)) return false;
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
                      (net->layers[0].act == QB_ACT_TANH || net->layers[0].act == QB_ACT_RELU) && !qb_env_int("QB_NO_PIPE", 0);
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
    tp->smem_bytes = (int)std::min<long long>(QB_SMEM_MAX, std::max(bytes, qb_tmem_smem_floor(tp->tmem_cols)));
    const int v3h = allow_v3 ? qb_tc_v3_shape(*tp) : 0;
    if (v3h && net->layers[1].act == QB_ACT_TANH && !qb_env_int("QB_NO_V3", 0) && !(allow_v3 == 2 && v3h != 64)) {
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
        tp->smem_bytes = (int)std::max<long long>(o, qb_tmem_smem_floor(tp->tmem_cols));
        if (tp->smem_bytes > (QB_SMEM_SM - 1024 * max_blocks3) / max_blocks3) return make_tc_plan(net, dtype, tp, 0);     // the blocks must fit
    }
    return true;
}

// The kernel of kernels 1 and 2: streamed when the weights do not fit next to a tile (tensor-core paths only for resident
// networks), then the fp16-split and 3xTF32 gradient kernels or the 3xTF32 value kernel, else the CUDA cores.  The
// N-split is the CUDA-core plan's in every case.
int plan_eval(const qb_net_t* net, int dtype, bool want_grad, long long K, long long N, bool force_single, QbLaunch* out) {
    if (make_launch(net, dtype, want_grad, K, N, force_single, out)) return -1;
    if (out->streamed) out->path = QB_PATH_STREAM;
    else if (want_grad && qb_tg8_make_plan(net, dtype, &out->t8)) out->path = QB_PATH_TG8;
    else if (want_grad && qb_tcg_make_plan(net, dtype, &out->tg)) out->path = QB_PATH_TCG;
    else if (!want_grad && make_tc_plan(net, dtype, &out->tp, 1)) out->path = out->tp.pipe ? QB_PATH_TC_PIPE : QB_PATH_TC;
    else out->path = QB_PATH_CUDA;
    size_t b = ((size_t)K * out->S * sizeof(double) + 255) / 256 * 256;
    out->gpart_off = b;
    if (want_grad && out->S > 1) b += (size_t)K * out->S * net->n_params * (dtype == QB_F64 ? 8 : 4);
    out->tail_off = (b + 255) / 256 * 256;
    if ((out->path == QB_PATH_TC || out->path == QB_PATH_TC_PIPE) && out->tp.v3)
        b = out->tail_off + qb_tc3_xsplit_bytes(N, out->tp.v3 == 1 ? 8 : 16);
    else if (out->path == QB_PATH_TG8)
        b = out->tail_off + QB_TG8_SCRATCH_BYTES;
    out->ws_bytes = b;
    return 0;
}

extern "C" size_t qb_eval_workspace_bytes(const qb_net_t* net, int dtype, int64_t K, int64_t N, int want_grad) {
    QbLaunch L;
    return plan_eval(net, dtype, want_grad != 0, K, N, false, &L) ? 0 : L.ws_bytes;
}

extern "C" int qb_plan_info(const qb_net_t* net, int dtype, int64_t K, int64_t N, int want_grad, int64_t* out) {
    QbLaunch L;
    if (plan_eval(net, dtype, want_grad != 0, K, N, false, &L)) return -1;
    out[0] = L.plan.TM; out[1] = L.plan.nthreads; out[2] = L.plan.smem_bytes; out[3] = L.S;
    out[4] = (int64_t)K * L.S; out[5] = L.plan.inplace; out[6] = L.path; out[7] = 0;
    if (L.path == QB_PATH_STREAM) { out[0] = L.sp.TM; out[1] = QS_THREADS; out[2] = L.sp.smem_bytes; out[5] = 0; }
    // tensor-core paths: 128-point tiles, out[7] = tensor-memory columns per block
    if (L.path == QB_PATH_TG8) { out[0] = 128; out[1] = L.t8.nthreads; out[2] = L.t8.smem_bytes; out[5] = 0; out[7] = L.t8.tmem_cols; }
    if (L.path == QB_PATH_TCG) { out[0] = 128; out[1] = L.tg.nthreads; out[2] = L.tg.smem_bytes; out[5] = 0; out[7] = L.tg.tmem_cols; }
    if (L.path == QB_PATH_TC || L.path == QB_PATH_TC_PIPE) {
        out[0] = 128; out[1] = L.tp.nthreads; out[2] = L.tp.smem_bytes; out[5] = 0; out[7] = L.tp.tmem_cols;
    }
    return 0;
}

// =================================================================================================
// kernel 5: Hessian-vector products (qb_hvp.cuh)
// =================================================================================================
// Plan for tile size TM: every layer in GEMM mode with TU x 4 thread tiles; returns the shared-memory bytes.
static long long hvp_plan_for_tm(const qb_net_t* net, int dtype, int TM, QbHvpPlan* H) {
    const QbDt D = dt_of(dtype);
    const int TU = D.TU, TP = 4;
    const int nl = net->n_layers, PG = TM / TP;
    memset(H, 0, sizeof(*H));
    QbPlan* P = &H->P;
    plan_head(net, D, TM, true, TP, P);
    int woff = 0, max_items = 0, dmax = 0;
    for (int l = 0; l < nl; ++l) {
        QbLayerPlan& L = P->L[l];
        copy_layer(net->layers[l], TU, L);
        L.mode = QB_MODE_GEMM; L.nj = 4;
        if (L.has_res) { P->has_res = 1; dmax = std::max(dmax, L.n_out_pad); }
        L.ug_shift = exact_log2(L.n_out_pad / TU); L.ugi_shift = exact_log2(L.n_in_pad / TU);
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
        dw_split(L, nthreads, TM, D.PV);
        H->LA[l] = L; H->LA[l].row_out = L.row_out - L.n_out_pad;
        H->LB[l] = L; H->LB[l].row_in = L.row_in - L.n_in_pad; H->LB[l].b_off = -1;
    }
    // one pad row: the double-buffered hot loop prefetches one row past the end
    P->smem_bytes = (long long)woff * D.elem + (long long)(row + 1) * P->lda * D.elem;
    return P->smem_bytes;
}

int make_hvp_launch(const qb_net_t* net, int dtype, long long K, long long N, QbHvpLaunch* out) {
    if (check_args(net, dtype, K, N)) return -1;
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
    const long long row_bytes = (long long)net->n_params * dt_of(dtype).elem;
    fit_splits(N, pick, want_splits(N, pick, K, row_bytes), &out->S, &out->pps);
    out->ws_bytes = out->S > 1 ? (size_t)K * out->S * row_bytes : 0;
    return 0;
}

extern "C" size_t qb_hvp_workspace_bytes(const qb_net_t* net, int dtype, int64_t K, int64_t N) {
    if (K == 0) return 0;
    QbHvpLaunch L;
    return make_hvp_launch(net, dtype, K, N, &L) ? 0 : L.ws_bytes;
}

extern "C" int qb_hvp_plan_info(const qb_net_t* net, int dtype, int64_t K, int64_t N, int64_t* out) {
    QbHvpLaunch L;
    if (make_hvp_launch(net, dtype, K, N, &L)) return -1;
    out[0] = L.H.P.TM; out[1] = L.H.P.nthreads; out[2] = L.H.P.smem_bytes; out[3] = L.S; out[4] = (int64_t)K * L.S;
    return 0;
}

// =================================================================================================
// kernel 6: Kronecker factors of the per-point empirical Fisher (qb_kfac.cuh)
// =================================================================================================
// Kernel 2's resident CUDA-core plan for one theta, the factor passes of every layer, and the N-split: one block per
// split, the [S, F] partial rows (dtype) under 256 MB.
int make_kfac_launch(const qb_net_t* net, int dtype, long long N, QbKfacLaunch* out) {
    if (check_args(net, dtype, 1, N)) return -1;
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
    const QbDt D = dt_of(dtype);
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
        dw_split(A, P.nthreads, P.TM, D.PV);
        QbLayerPlan& G = out->K.LG[l];
        G = B;
        G.n_in = B.n_out; G.n_in_pad = B.n_out_pad; G.row_in = B.row_out;
        G.n_terms = 0;
        G.w_off = off; off += B.n_out * B.n_out;
        G.b_off = -1;
        dw_split(G, P.nthreads, P.TM, D.PV);
    }
    out->K.n_factors = off;
    const long long row_bytes = (long long)off * D.elem;
    fit_splits(N, P.TM, want_splits(N, P.TM, 1, row_bytes), &out->S, &out->pps);
    out->ws_bytes = (size_t)out->S * row_bytes;
    return 0;
}

extern "C" size_t qb_kfac_workspace_bytes(const qb_net_t* net, int dtype, int64_t N) {
    if (N <= 0) return 0;
    QbKfacLaunch L;
    return make_kfac_launch(net, dtype, N, &L) ? 0 : L.ws_bytes;
}

extern "C" int qb_kfac_plan_info(const qb_net_t* net, int dtype, int64_t N, int64_t* out) {
    QbKfacLaunch L;
    if (make_kfac_launch(net, dtype, std::max<int64_t>(N, 1), &L)) return -1;
    out[0] = L.K.P.TM; out[1] = L.K.P.nthreads; out[2] = L.K.P.smem_bytes; out[3] = L.S; out[4] = L.K.n_factors;
    return 0;
}

// =================================================================================================
// kernel 7: per-point output Jacobians as per-layer pairs (qb_jac.cuh)
// =================================================================================================
// Kernel 2's resident CUDA-core plan for one theta, the factor rows of every layer, and the N-split: one block per run of
// whole tiles.  Nothing is reduced over the points, so there are no partial rows to cap.
int make_jac_launch(const qb_net_t* net, int dtype, long long N, QbJacLaunch* out) {
    if (check_args(net, dtype, 1, N)) return -1;
    QbLaunch L;
    if (make_launch(net, dtype, true, 1, N, true, &L)) return -1;
    if (L.streamed)
        return qb_fail("output Jacobians: the network's weights do not fit in shared memory next to one tile of "
                       "activations, and the layer-streamed path (plan code 5) has no Jacobian kernel");
    memset(&out->J, 0, sizeof(out->J));
    out->J.P = L.plan;
    const QbPlan& P = out->J.P;
    int row = 0;
    for (int l = 0; l < P.n_layers; ++l) {
        out->J.row0[l] = row;
        row += P.L[l].n_in + P.out_dim * P.L[l].n_out;
    }
    out->J.n_rows = row;
    fit_splits(N, P.TM, want_splits(N, P.TM, 1, 0), &out->S, &out->pps);
    return 0;
}

extern "C" int qb_jac_plan_info(const qb_net_t* net, int dtype, int64_t N, int64_t* out) {
    if (N < 0) return qb_fail("N must not be negative");
    QbJacLaunch L;
    if (make_jac_launch(net, dtype, std::max<int64_t>(N, 1), &L)) return -1;
    out[0] = L.J.P.TM; out[1] = L.J.P.nthreads; out[2] = L.J.P.smem_bytes; out[3] = N > 0 ? L.S : 0; out[4] = L.J.n_rows;
    return 0;
}
