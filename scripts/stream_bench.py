"""Throughput of the layer-streamed kernels (quinn_b200/csrc/qb_stream.cuh) on networks whose weights do not fit in shared
memory: kernels 1 (value) and 2 (value + gradient) and one HMC(L=3) leg, timed with CUDA events after a warm-up.

Algorithmic FLOPs (SURVEY.md section 8d): F_v = 2*N*S, F_vg = 6*N*S - 2*N*n0*n1 per evaluation, S = sum of the layers'
n_in*n_out; an HMC(L) step costs L*F_vg.  The fraction of peak uses the CUDA-core FMA rate measured in the same process
(qb_fma_peak: DFMA chains for fp64, FFMA2 chains for fp32).  Card name and power limit are printed with the numbers.

    python scripts/stream_bench.py [--reps 10] [--out FILE.json]
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
LEGS = [  # name, hidden widths, dtype, K
    ('mlp_10_128x3_f64', (128, 128, 128), torch.float64, 256),
    ('mlp_10_256x3_f64', (256, 256, 256), torch.float64, 256),
    ('mlp_10_512x2_f32', (512, 512), torch.float32, 64),
]


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
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'stream_bench.py measures on the GPU'
    name, power = card()
    peak = {torch.float64: ops.fma_peak(torch.float64, 0), torch.float32: ops.fma_peak(torch.float32, 2)}
    res = dict(card=name, power_limit_and_max_sm_clock=power, N=N,
               fma_peak_tflops={'f64': peak[torch.float64] / 1e12, 'f32': peak[torch.float32] / 1e12}, legs=[])
    print(f'# {name}, power limit / max SM clock: {power}')
    print(f'# measured FMA peak: fp64 {peak[torch.float64] / 1e12:.1f} TFLOP/s, fp32 (FFMA2) {peak[torch.float32] / 1e12:.1f} TFLOP/s')
    rs = np.random.RandomState(0)
    for leg, hls, dt, K in LEGS:
        layers, P = qo.mlp_layers(10, 1, hls, True, 'tanh')
        desc = netdesc_from_layers(layers, P)
        S = sum(L['n_in'] * L['n_out'] for L in layers)
        n0n1 = layers[0]['n_in'] * layers[0]['n_out']
        x = rs.rand(N, 10) * 2 - 1
        y = np.sin(x.sum(1, keepdims=True))
        prob = ops.Problem(desc, x, y, 0.1, dtype=dt)
        th = (0.05 * torch.randn((K, P), dtype=torch.float64, device='cuda')).to(dt)
        lp = torch.empty(K, dtype=torch.float64, device='cuda')
        g = torch.empty_like(th)
        fv, fvg = 2.0 * N * S, 6.0 * N * S - 2.0 * N * n0n1
        for kind, flops, fn in (('value', fv, lambda: ops.logpost(prob, th, out=lp)),
                                ('value+grad', fvg, lambda: ops.logpost_grad(prob, th, lp=lp, grad=g))):
            info = prob.plan_info(K, kind != 'value')
            t = timed(fn, args.reps)
            tf = K * flops / t
            row = dict(leg=leg, kind=kind, P=P, K=K, dtype=str(dt).split('.')[-1], plan=info, seconds_per_call=t,
                       evals_per_s=K / t, tflops=tf / 1e12, fraction_of_fma_peak=tf / peak[dt])
            res['legs'].append(row)
            print(f'{leg:18s} {kind:10s} K={K:4d} TM={info["TM"]:3d} S={info["splits"]:3d} code={info["tensor_core"]}  '
                  f'{t * 1e3:9.3f} ms  {K / t:10.1f} evals/s  {tf / 1e12:6.2f} TFLOP/s  {tf / peak[dt]:.3f} of peak')
        if leg == 'mlp_10_128x3_f64':
            # HMC(L=3): one block per chain, L value+gradient evaluations per step
            nsteps, L = 4, 3
            st = ops.ChainState(prob, th.double().cpu().numpy())
            hm = ops.HmcState(st, epsilon=1e-4, L=L)
            ops.hmc_run(st, hm, 1, None, seed=1)           # initial gradient
            t = timed(lambda: ops.hmc_run(st, hm, nsteps, None, seed=2), max(2, args.reps // 5)) / nsteps
            tf = K * L * fvg / t
            res['legs'].append(dict(leg=leg, kind='hmc_L3_step', P=P, K=K, dtype='float64', seconds_per_step=t,
                                    chain_steps_per_s=K / t, tflops=tf / 1e12, fraction_of_fma_peak=tf / peak[dt]))
            print(f'{leg:18s} {"hmc L=3":10s} K={K:4d}  {t * 1e3:9.3f} ms/step  {K / t:10.1f} chain-steps/s  '
                  f'{tf / 1e12:6.2f} TFLOP/s  {tf / peak[dt]:.3f} of peak')
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
