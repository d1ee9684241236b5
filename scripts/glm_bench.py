"""Throughput of kernel 7 (qb_predict_jac, quinn_b200/csrc/qb_jac.cuh): outputs and per-point Jacobian pairs at one theta
for the config-2 (2-32-32-1), config-5 (3-64-64-1) and config-3/4 (10-128-128-1) nets, fp64 and fp32, N = 10^4 and 10^5
(and 10^6 for config 3/4); then NN_Laplace.predict_mom_glm(msc=1) per la_type next to predict_mom_sample(msc=1,
nsam=1000) on the config-5 net at N = 10^5 test points, fp64.  Kernel 7 is timed with CUDA events after a warm-up, on
preallocated buffers; the predictive calls with a host clock around a synchronise.

Algorithmic FLOPs per point, with S = sum of the layers' n_in*n_out and S0 = n_in*n_out of the first layer:
    forward 2S, one back-propagation per output 2(S - S0):  2S + o*2(S - S0)
(the kernel runs the forward pass again for every output after the first; that work is not counted).  Store bytes per
point are F*elem, F = sum_l (n_in_l + o*n_out_l).  The fraction of peak uses the CUDA-core FMA rate measured in the same
process (qb_fma_peak: DFMA chains for fp64, FFMA2 chains for fp32).  Card name and power limit are recorded with the
numbers.

    python scripts/glm_bench.py [--reps 5] [--out profiles/r6_glm_bench.json]
"""
import argparse
import ctypes as C
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
from quinn_b200 import _lib, ops                 # noqa: E402

NETS = [('config2_2-32-32-1', 2, (32, 32), (10 ** 4, 10 ** 5)), ('config5_3-64-64-1', 3, (64, 64), (10 ** 4, 10 ** 5)),
        ('config34_10-128-128-1', 10, (128, 128), (10 ** 4, 10 ** 5, 10 ** 6))]
HBM_BYTES_PER_S = 7.7e12           # HGX B200 data sheet, one GPU


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
    fn()                                           # warm-up: module load, attributes
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def host_timed(fn, reps):
    ts = []
    for _ in range(reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return min(ts[1:]), ts


def predictive_times(reps):
    """predict_mom_glm(msc=1) per la_type and predict_mom_sample(msc=1, nsam=1000), config-5 net, 10^5 test points"""
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_Laplace
    rs = np.random.RandomState(1)
    x = rs.rand(10000, 3) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(10000, 1)
    xt = rs.rand(100000, 3) * 2 - 1
    out = {}
    for la_type in ('full', 'diag', 'kron'):
        np.random.seed(0)
        torch.manual_seed(0)
        uq = NN_Laplace(MLP(3, 1, (64, 64), activ='tanh').double(), la_type=la_type, datanoise=0.05)
        uq.fit(x, y, nepochs=20, lrate=0.01, batch_size=1000)
        t_glm, all_glm = host_timed(lambda: uq.predict_mom_glm(xt, msc=1), reps)
        np.random.seed(2)
        t_smp, all_smp = host_timed(lambda: uq.predict_mom_sample(xt, msc=1, nsam=1000), reps)
        out[la_type] = dict(glm_seconds=t_glm, glm_seconds_all=all_glm, sample_nsam1000_seconds=t_smp,
                            sample_seconds_all=all_smp, P=uq.nparams)
        print(f'config-5 N=1e5 fp64 {la_type:5s}: predict_mom_glm {t_glm:8.3f} s   predict_mom_sample(nsam=1000) '
              f'{t_smp:8.3f} s')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'glm_bench.py measures on the GPU'
    name, power = card()
    peak = {torch.float64: ops.fma_peak(torch.float64, 0), torch.float32: ops.fma_peak(torch.float32, 2)}
    res = dict(card=name, power_limit_and_max_sm_clock=power,
               fma_peak_tflops={'f64': peak[torch.float64] / 1e12, 'f32': peak[torch.float32] / 1e12}, legs=[])
    print(f'# {name}, power limit / max SM clock: {power}')
    print(f'# measured FMA peak: fp64 {peak[torch.float64] / 1e12:.1f} TFLOP/s, fp32 (FFMA2) {peak[torch.float32] / 1e12:.1f} TFLOP/s')
    lib = _lib.load()
    rs = np.random.RandomState(0)
    for leg, indim, hls, Ns in NETS:
        layers, P = qo.mlp_layers(indim, 1, hls, True, 'tanh')
        desc = netdesc_from_layers(layers, P)
        cnet = desc.to_c()
        o = 1
        S = sum(L['n_in'] * L['n_out'] for L in layers)
        S0 = layers[0]['n_in'] * layers[0]['n_out']
        flops = 2.0 * S + o * 2.0 * (S - S0)
        for N in Ns:
            x = rs.rand(N, indim) * 2 - 1
            for dt in (torch.float64, torch.float32):
                info = ops.jac_plan_info(desc, N, dt)
                elem = 8 if dt == torch.float64 else 4
                xs = ops.as_device(x, dt, 'cuda')
                th = ops.as_device(0.2 * rs.randn(P), dt, 'cuda')
                out = torch.empty((N, o), dtype=dt, device='cuda')
                fac = torch.empty(N * info['rows'], dtype=dt, device='cuda')

                def fn():
                    _lib.check(lib.qb_predict_jac(C.byref(cnet), ops.qb_dtype(dt), ops._ptr(th), ops._ptr(xs), N,
                                                  ops._ptr(out), ops._ptr(fac), ops._stream()), 'qb_predict_jac')
                t = timed(fn, args.reps)
                tf = N * flops / t
                store = N * (info['rows'] + o) * elem
                dts = str(dt).split('.')[-1]
                res['legs'].append(dict(leg=leg, dtype=dts, N=N, P=P, flops_per_point=flops,
                                        store_bytes_per_point=info['rows'] * elem, plan=info, seconds_per_call=t,
                                        tflops=tf / 1e12, fraction_of_fma_peak=tf / peak[dt],
                                        store_gbytes_per_s=store / t / 1e9,
                                        store_fraction_of_hbm_datasheet=store / t / HBM_BYTES_PER_S))
                print(f'{leg:22s} {dts:8s} N={N:7d} TM={info["TM"]:3d} blocks={info["blocks"]:5d} '
                      f'threads={info["threads"]:3d} smem={info["smem_bytes"]:6d}  {t * 1e3:9.3f} ms  '
                      f'{tf / 1e12:6.2f} TFLOP/s  {tf / peak[dt]:.3f} of peak  stores {store / t / 1e9:7.1f} GB/s')
                del fac, out
    res['predictive_config5_N1e5_f64'] = predictive_times(max(1, args.reps // 2))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
