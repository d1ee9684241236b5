"""Throughput of kernel 6 (qb_logpost_kfac, quinn_b200/csrc/qb_kfac.cuh): the Kronecker factors of every layer at one
theta, against kernel 2 (value + gradient, K = 1) on the CUDA cores over the same points, for the config-2 (2-32-32-1),
config-5 (3-64-64-1) and config-3/4 (10-128-128-1) nets, fp64 and fp32, N = 10^4 and 10^5; then NN_Laplace.la_calc with
la_type='kron' against 'diag' on the config-3/4 net at N = 10^5, fp64.  Timed with CUDA events after a warm-up.

Algorithmic FLOPs per data point, with S = sum of the layers' n_in*n_out and S0 = n_in*n_out of the first layer:
    forward 2S, back-propagation 2(S - S0), factors sum_l 2(n_in^2 + n_out^2)   (kernel 6)
    forward 2S, back-propagation 2(S - S0), dW 2S                                (kernel 2: 6S - 2S0)
Kernel 2 runs with QB_NO_TC=1 so that both kernels are on the CUDA cores.  The fraction of peak uses the CUDA-core FMA
rate measured in the same process (qb_fma_peak: DFMA chains for fp64, FFMA2 chains for fp32).  Card name and power limit
are recorded with the numbers.

    python scripts/kfac_bench.py [--reps 5] [--out profiles/r5_kfac_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from oracle import quinn_oracle as qo            # noqa: E402
from golden_util import netdesc_from_layers      # noqa: E402
from quinn_b200 import ops                       # noqa: E402

NETS = [('config2_2-32-32-1', 2, (32, 32)), ('config5_3-64-64-1', 3, (64, 64)), ('config34_10-128-128-1', 10, (128, 128))]


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


def la_calc_times(reps):
    """NN_Laplace.la_calc ('kron' vs 'diag') on the config-3/4 net at N = 10^5, fp64: host clock around a synchronise"""
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_Laplace
    rs = np.random.RandomState(1)
    N = 100000
    x = rs.rand(N, 10) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(N, 1)
    out = {}
    for la_type in ('kron', 'diag'):
        torch.manual_seed(0)
        uq = NN_Laplace(MLP(10, 1, (128, 128), activ='tanh').double(), la_type=la_type, datanoise=0.05)

        class _Learner:                            # la_calc reads learner.best_model only
            best_model = uq.nnmodel
        anchor = np.zeros(uq.nparams)
        ts = []
        for r in range(reps + 1):
            uq._factors = []
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            uq.la_calc(_Learner, x, y, anchor)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        out[la_type] = dict(seconds=min(ts[1:]), seconds_all=ts)
        print(f'la_calc {la_type:5s} config-3/4 N={N} fp64: {min(ts[1:]):8.3f} s  (first call {ts[0]:.3f} s)')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'kfac_bench.py measures on the GPU'
    name, power = card()
    peak = {torch.float64: ops.fma_peak(torch.float64, 0), torch.float32: ops.fma_peak(torch.float32, 2)}
    res = dict(card=name, power_limit_and_max_sm_clock=power,
               fma_peak_tflops={'f64': peak[torch.float64] / 1e12, 'f32': peak[torch.float32] / 1e12}, legs=[])
    print(f'# {name}, power limit / max SM clock: {power}')
    print(f'# measured FMA peak: fp64 {peak[torch.float64] / 1e12:.1f} TFLOP/s, fp32 (FFMA2) {peak[torch.float32] / 1e12:.1f} TFLOP/s')
    rs = np.random.RandomState(0)
    for leg, indim, hls in NETS:
        layers, P = qo.mlp_layers(indim, 1, hls, True, 'tanh')
        desc = netdesc_from_layers(layers, P)
        S = sum(L['n_in'] * L['n_out'] for L in layers)
        S0 = layers[0]['n_in'] * layers[0]['n_out']
        fac = sum(2 * (L['n_in'] ** 2 + L['n_out'] ** 2) for L in layers)
        f_kfac, f_vg = 2.0 * S + 2.0 * (S - S0) + fac, 6.0 * S - 2.0 * S0
        for N in (10 ** 4, 10 ** 5):
            x = rs.rand(N, indim) * 2 - 1
            y = np.sin(x.sum(1, keepdims=True))
            for dt in (torch.float64, torch.float32):
                prob = ops.Problem(desc, x, y, 0.1, dtype=dt)
                th = prob.theta(0.2 * rs.randn(P))
                dts = str(dt).split('.')[-1]
                for kind, flops, fn in (('kernel6_kfac', f_kfac, lambda: ops.logpost_kfac(prob, th)),
                                        ('kernel2_grad_cuda_cores', f_vg, lambda: ops.logpost_grad(prob, th))):
                    if kind.startswith('kernel2'):
                        os.environ['QB_NO_TC'] = '1'
                        info = prob.plan_info(1, True)
                    else:
                        info = ops.kfac_plan_info(prob)
                    t = timed(fn, args.reps)
                    os.environ.pop('QB_NO_TC', None)
                    tf = N * flops / t
                    res['legs'].append(dict(leg=leg, kind=kind, dtype=dts, N=N, P=P, flops_per_point=flops, plan=info,
                                            seconds_per_call=t, tflops=tf / 1e12, fraction_of_fma_peak=tf / peak[dt]))
                    print(f'{leg:22s} {dts:8s} N={N:6d} {kind:24s} TM={info["TM"]:3d} S={info["splits"]:4d} '
                          f'threads={info["threads"]:3d} smem={info["smem_bytes"]:6d}  {t * 1e3:9.3f} ms  '
                          f'{tf / 1e12:6.2f} TFLOP/s  {tf / peak[dt]:.3f} of peak')
    res['la_calc_config34_N1e5_f64'] = la_calc_times(max(1, args.reps // 2))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
