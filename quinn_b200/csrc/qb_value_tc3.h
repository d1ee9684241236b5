// Host interface of the warp-specialised hot-shape value path (qb_value_tc3.cu); called from qb_kernels.cu and qb_launch.cu.
#pragma once
#include <cuda_runtime.h>
#include "quinn_b200.h"
#include "qb_tc.cuh"

template <typename T> struct EvalArgs;
template <typename T> struct ChainArgs;
template <typename T> struct AmcmcArgs;

// tp.v3 != 0 (make_tc_plan); the chain kernel additionally needs the state area (tp.v3_state, plan mode 2), diagonal or
// no adaptation and no user-supplied Cholesky factor
// bytes of the operand-tile image of x[N, in] (tf32 hi | lo, canonical K-major [128 x K0] tiles: K0 KB per 128 points;
// K0 = 8 for the 64-wide shape, 16 for the 128-wide one)
static inline size_t qb_tc3_xsplit_bytes(long long N, int k0) { return (size_t)((N + 127) / 128) * 1024 * (size_t)k0; }
// a.xsplit (if not NULL) is filled from a.x by a small kernel launched ahead of the evaluation
cudaError_t qb_tc3_launch_logpost(const QbTcPlan& tp, const EvalArgs<float>& a, dim3 grid, cudaStream_t st);
// kernel 4 (one output per point): out[m, p], grid = (members, chunks of tiles_per_block tiles)
cudaError_t qb_tc3_launch_predict(const QbTcPlan& tp, const float* theta, const float* x, long long N, float* out,
                                  long long tiles_per_block, dim3 grid, cudaStream_t st);
// a.prop (the [K,P] scratch the generic kernel keeps proposals in) holds the x tiles here when it is large enough
cudaError_t qb_tc3_launch_amcmc(const QbTcPlan& tp, const ChainArgs<float>& c, const AmcmcArgs<float>& a, long long K, cudaStream_t st);
