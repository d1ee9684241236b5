// Host interface of the tensor-core gradient translation unit (qb_grad_tc.cu); called from qb_kernels.cu and qb_launch.cu.
#pragma once
#include <cuda_runtime.h>
#include "quinn_b200.h"
#include "qb_tcg.cuh"

template <typename T> struct EvalArgs;
template <typename T> struct ChainArgs;
template <typename T> struct HmcArgs;
template <typename T> struct NutsArgs;
struct PtArgs;

// eligibility + plan of the tcgen05 gradient path (fp32, in -> H -> H -> 1, H in {32, 64}, tanh / relu); false: not eligible
bool qb_tcg_make_plan(const qb_net_t* net, int dtype, QbTcgPlan* tp);
cudaError_t qb_tcg_launch_eval(const QbTcgPlan& tp, const EvalArgs<float>& a, dim3 grid, cudaStream_t st);
cudaError_t qb_tcg_launch_hmc(const QbTcgPlan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st);
cudaError_t qb_tcg_launch_nuts(const QbTcgPlan& tp, const ChainArgs<float>& c, const NutsArgs<float>& a, long long K, cudaStream_t st);
cudaError_t qb_tcg_launch_pt(const QbTcgPlan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, const PtArgs& a, long long K,
                             cudaStream_t st);
