"""Throughput of kernel 5 (qb_logpost_hvp, quinn_b200/csrc/qb_hvp.cuh): K Hessian-vector products with random directions
and the full Hessian (P unit directions), on the config-2 (2-32-32-1) and config-5 (3-64-64-1) nets, fp64 and fp32,
N = 10^4, timed with CUDA events after a warm-up.  Kernel 2 (value + gradient) on the same net is timed alongside.

Algorithmic FLOPs per data point and direction, with S = sum of the layers' n_in*n_out and S0 = n_in*n_out of the first
layer (whose input tangent is zero):
    primal forward 2S, tangent forward 4S - 2 S0, W^T dz 2(S - S0), W^T dz_dot + V^T dz 4(S - S0),
    Hv_W = dz_dot a_in^T + dz a_dot_in^T 4S - 2 S0                       ->  F_hvp = 16 S - 10 S0
Kernel 2: F_vg = 6 S - 2 S0 (SURVEY.md section 8d); in fp32 it is timed as selected (tensor cores for these nets) and, with
QB_NO_TC=1, on the CUDA cores.  The fraction of peak uses the CUDA-core FMA rate measured in the same
process (qb_fma_peak: DFMA chains for fp64, FFMA2 chains for fp32).  Card name and power limit are printed with the numbers.

    python scripts/hessian_bench.py [--reps 5] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from oracle import quinn_oracle as qo            # noqa: E402
from golden_util import netdesc_from_layers      # noqa: E402
from quinn_b200 import ops                       # noqa: E402

N = 10000
NETS = [('config2_2-32-32-1', 2, (32, 32)), ('config5_3-64-64-1', 3, (64, 64))]
K_HVP = 64


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def timed(fn, reps):
    fn()
    fn()                                           # warm-up: module load, attributes, workspace
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'hessian_bench.py measures on the GPU'
    name, power = card()
    peak = {torch.float64: ops.fma_peak(torch.float64, 0), torch.float32: ops.fma_peak(torch.float32, 2)}
    res = dict(card=name, power_limit_and_max_sm_clock=power, N=N,
               fma_peak_tflops={'f64': peak[torch.float64] / 1e12, 'f32': peak[torch.float32] / 1e12}, legs=[])
    print(f'# {name}, power limit / max SM clock: {power}')
    print(f'# measured FMA peak: fp64 {peak[torch.float64] / 1e12:.1f} TFLOP/s, fp32 (FFMA2) {peak[torch.float32] / 1e12:.1f} TFLOP/s')
    rs = np.random.RandomState(0)
    for leg, indim, hls in NETS:
        layers, P = qo.mlp_layers(indim, 1, hls, True, 'tanh')
        desc = netdesc_from_layers(layers, P)
        S = sum(L['n_in'] * L['n_out'] for L in layers)
        S0 = layers[0]['n_in'] * layers[0]['n_out']
        x = rs.rand(N, indim) * 2 - 1
        y = np.sin(x.sum(1, keepdims=True))
        f_hvp, f_vg = (16.0 * S - 10.0 * S0) * N, (6.0 * S - 2.0 * S0) * N
        for dt in (torch.float64, torch.float32):
            prob = ops.Problem(desc, x, y, 0.1, dtype=dt, prior_sigma=1.0, prior_anchor=np.zeros(P), fulldatasize=N)
            theta = 0.2 * rs.randn(P)
            V = torch.as_tensor(rs.randn(K_HVP, P), dtype=dt, device='cuda')
            th = prob.theta(theta)
            thK = th.expand(K_HVP, P).contiguous()
            dts = str(dt).split('.')[-1]
            legs = [('hvp', f_hvp, K_HVP, lambda: ops.logpost_hvp(prob, th, V), ops.hvp_plan_info(prob, K_HVP)),
                    ('hessian', f_hvp, P, lambda: ops.logpost_hessian(prob, th), ops.hvp_plan_info(prob, P)),
                    ('kernel2_grad', f_vg, K_HVP, lambda: ops.logpost_grad(prob, thK), prob.plan_info(K_HVP, True))]
            if dt == torch.float32:
                # kernel 2 of fp32 tanh nets runs on the tensor cores; the CUDA-core leg is the like-for-like comparison
                legs.append(('kernel2_grad_cuda_cores', f_vg, K_HVP, lambda: ops.logpost_grad(prob, thK), None))
            for kind, flops, K, fn, info in legs:
                no_tc = info is None
                if no_tc:
                    os.environ['QB_NO_TC'] = '1'
                    info = prob.plan_info(K_HVP, True)
                t = timed(fn, args.reps)
                if no_tc:
                    del os.environ['QB_NO_TC']
                tf = K * flops / t
                row = dict(leg=leg, kind=kind, dtype=dts, P=P, K=K, plan=info, seconds_per_call=t, tflops=tf / 1e12,
                           fraction_of_fma_peak=tf / peak[dt])
                res['legs'].append(row)
                code = info.get('tensor_core', 0)
                print(f'{leg:18s} {dts:8s} {kind:24s} K={K:5d} TM={info["TM"]:3d} S={info["splits"]:3d} '
                      f'threads={info["threads"]:3d} smem={info["smem_bytes"]:6d} code={code}  {t * 1e3:9.3f} ms  '
                      f'{tf / 1e12:6.2f} TFLOP/s  {tf / peak[dt]:.3f} of peak')
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
