// quinn_b200: launch planning of the library's kernels (host only, qb_launch.cu).  The plan structs live next to the
// device code that reads them.
#pragma once
#include "qb_plan.h"
#include "qb_stream.cuh"
#include "qb_hvp.cuh"
#include "qb_kfac.cuh"
#include "qb_jac.cuh"
#include "qb_tc.cuh"
#include "qb_tcg.cuh"
#include "qb_tg8_plan.h"

constexpr int QB_SMEM_MAX = 227 * 1024;    // shared memory of one block
constexpr int QB_SMEM_SM = 228 * 1024;     // shared memory per SM
// Tensor memory has 512 columns per SM, and a block whose tcgen05.alloc cannot be met spins until another block frees
// its columns.  A kernel that allocates tmem_cols columns asks for at least this much shared memory, so that no more
// than 512 / tmem_cols of its blocks become resident on one SM.
inline long long qb_tmem_smem_floor(int tmem_cols) { return QB_SMEM_SM / (512 / tmem_cols + 1) + 1; }

// sets the thread's error text (format: a string, then an integer) and returns -1
int qb_fail(const char* fmt, const char* a = "", long long b = 0);
// an environment variable as an integer, dflt when unset or empty (read on every call)
int qb_env_int(const char* name, int dflt);
// SM count of the current device, 148 when none is visible; queried once per process
int qb_num_sms();

// the kernel of kernels 1 and 2 for a call; the values are the qb_plan_info codes (out[6])
enum QbEvalPath { QB_PATH_CUDA = 0, QB_PATH_TC = 1, QB_PATH_TC_PIPE = 2, QB_PATH_TCG = 3, QB_PATH_TG8 = 4, QB_PATH_STREAM = 5 };

// make_launch: the resident (plan) or layer-streamed (sp) CUDA-core plan (the other is not cleared), S splits of
// pts_per_split points.  plan_eval adds the kernel and its tensor-core plan, and the workspace: [K, S] partial sums at 0,
// [K, S, P] gradient rows at gpart_off, tail scratch (x operand tiles or fp16-split scale words) at tail_off.
struct QbLaunch {
    QbPlan plan; int S; long long pts_per_split; bool streamed; QbStreamPlan sp;
    QbEvalPath path; QbTcPlan tp; QbTcgPlan tg; QbTg8Plan t8;
    size_t gpart_off, tail_off, ws_bytes;
};
struct QbHvpLaunch { QbHvpPlan H; int S; long long pps; size_t ws_bytes; };
struct QbKfacLaunch { QbKfacPlan K; int S; long long pps; size_t ws_bytes; };
struct QbJacLaunch { QbJacPlan J; int S; long long pps; };

// the planners return -1 with the error set when they refuse; force_single: one block per chain
int make_launch(const qb_net_t* net, int dtype, bool want_grad, long long K, long long N, bool force_single, QbLaunch* out);
int plan_eval(const qb_net_t* net, int dtype, bool want_grad, long long K, long long N, bool force_single, QbLaunch* out);
int make_hvp_launch(const qb_net_t* net, int dtype, long long K, long long N, QbHvpLaunch* out);
int make_kfac_launch(const qb_net_t* net, int dtype, long long N, QbKfacLaunch* out);
int make_jac_launch(const qb_net_t* net, int dtype, long long N, QbJacLaunch* out);
bool make_tc_plan(const qb_net_t* net, int dtype, QbTcPlan* tp, int allow_v3 = 0);
// kernel 4's member-parallel grid: chunks of tiles_per_block consecutive tiles, about blocks_wanted blocks over M members
long long qb_tile_chunks(long long tiles, long long blocks_wanted, long long M, long long* tiles_per_block);
