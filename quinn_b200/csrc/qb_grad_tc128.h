// Host interface of the fp16-split tensor-core gradient translation unit (qb_grad_tc128.cu); called from qb_kernels.cu and qb_launch.cu.
#pragma once
#include <cuda_runtime.h>
#include "quinn_b200.h"
#include "qb_tg8_plan.h"

template <typename T> struct EvalArgs;
template <typename T> struct ChainArgs;
template <typename T> struct HmcArgs;

// eligibility + plan of the fp16-split tcgen05 gradient path (fp32, in <= 15 -> H -> H -> 1, H in {64, 128}, tanh); false: not eligible
bool qb_tg8_make_plan(const qb_net_t* net, int dtype, QbTg8Plan* tp);
// scratch: 8 bytes of device memory (max |x|, max |y| of the launch), written by a small kernel ahead of the evaluation
cudaError_t qb_tg8_launch_eval(const QbTg8Plan& tp, const EvalArgs<float>& a, void* scratch, dim3 grid, cudaStream_t st);
// HMC / MALA chains on the same evaluation (the scratch words live in a small per-(device, stream) buffer kept by the library)
cudaError_t qb_tg8_launch_hmc(const QbTg8Plan& tp, const ChainArgs<float>& c, const HmcArgs<float>& h, long long K, cudaStream_t st);
enum { QB_TG8_SCRATCH_BYTES = 256 };
