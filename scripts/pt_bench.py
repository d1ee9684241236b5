"""Parallel tempering (qb_pt_run) against HMC(L=3) (qb_hmc_run) on the same net, dtype, K, N and kernel path:

1. throughput in chain-steps per second: PT-HMC with T = 8 temperatures and K / 8 groups, swap_every 1 and 10, against
   HMC at the same K.  Tempering adds one P-length pass per gradient evaluation, and a swap round a small kernel that
   moves two rows per accepted pair; the runs alternate HMC, PT(1), PT(10) twice, so the spread shows;
2. the share of device time in k_pt_swap, from a separate torch.profiler run of PT with swap_every = 1;
3. mixing on the two-mode net of tests/test_gpu_pt.py (MLP 1-1-1 tanh, prior sigma_p = 1: the posterior is symmetric
   under (w1, b1, w2) -> -(w1, b1, w2)): switches of the sign of w2 per 1000 cold steps and round trips per second;
4. the swap-acceptance profile along the ladder on config 2.

Shapes: config 2 (fp32, MLP 2-32-32-1, N = 10^3, K = 1024, fp16-split tensor-core path), the config-5 shape (fp32, MLP
3-64-64-1, N = 10^4, K = 1024) and an fp64 CUDA-core net (MLP 1-16-16-1, N = 10^3, K = 1024).  Every shape is warmed up
first.  Card name and power limit are read in the same run.

    python scripts/pt_bench.py [--out profiles/r9_pt_bench.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quinn_b200 import ops                      # noqa: E402
from quinn_b200.netdesc import NetDesc, Layer    # noqa: E402

T_PT = 8
SHAPES = [
    dict(name='c2', d=2, hls=(32, 32), N=1_000, K=1_024, sigma=0.02, dtype=torch.float32, eps=1e-4, path=4, nsteps=200),
    dict(name='c5_shape', d=3, hls=(64, 64), N=10_000, K=1_024, sigma=0.05, dtype=torch.float32, eps=2e-6, path=4,
         nsteps=100),
    dict(name='f64_cuda', d=1, hls=(16, 16), N=1_000, K=1_024, sigma=0.05, dtype=torch.float64, eps=1e-4, path=0,
         nsteps=200),
]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def mlp_desc(d, hls):
    widths = [d] + list(hls) + [1]
    layers, off = [], 0
    for l in range(len(widths) - 1):
        w = off
        off += widths[l] * widths[l + 1]
        layers.append(Layer(widths[l], widths[l + 1], w, off, 'tanh' if l < len(widths) - 2 else 'identity', 0.0))
        off += widths[l + 1]
    return NetDesc(d, 1, off, layers)


def data(s):
    """bench.py's data: Ackley for config 2, Sine otherwise"""
    rs = np.random.RandomState(0)
    if s['name'] == 'c2':
        x = rs.rand(s['N'], s['d']) * 3.0 - 1.5
        y = 0.02 * rs.randn(s['N'])
        for i in range(s['d'] - 1):
            y += np.exp(-0.2) * np.sqrt(x[:, i] ** 2 + x[:, i + 1] ** 2) + 3 * (np.cos(2 * x[:, i]) + np.sin(2 * x[:, i + 1]))
        return x, y.reshape(-1, 1)
    x = rs.rand(s['N'], s['d']) * 2 * math.pi - math.pi
    return x, s['sigma'] * rs.randn(s['N'], 1) + np.sin(x).sum(1, keepdims=True)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def pt_states(prob, th0, G, eps, swap_every):
    st = ops.ChainState(prob, np.tile(th0[:G], (T_PT, 1)))
    ps = ops.PtState(st, G, ops.pt_ladder(T_PT, 0.05), eps, 3, 'hmc', swap_every)
    return st, ps


def run_shape(s, seed=7):
    desc = mlp_desc(s['d'], s['hls'])
    x, y = data(s)
    prob = ops.Problem(desc, x, y, s['sigma'], dtype=s['dtype'], device='cuda')
    K, P, n = s['K'], desc.n_params, s['nsteps']
    G = K // T_PT
    path = prob.plan_info(K, True)['tensor_core']
    assert path == s['path'], (s['name'], path)
    th0 = 0.1 * np.random.RandomState(1234).randn(K, P)
    out = dict(net=f"MLP {s['d']}-{'-'.join(map(str, s['hls']))}-1 tanh", P=P, N=s['N'], K=K, T=T_PT, groups=G,
               dtype=str(s['dtype']), plan_code=path, steps_per_run=n, epsilon_cold=s['eps'], L=3)
    st_h = ops.ChainState(prob, th0)
    hm = ops.HmcState(st_h, epsilon=s['eps'], L=3, method='hmc')
    runs = {'hmc': lambda: ops.hmc_run(st_h, hm, n, None, seed=seed)}
    pts = {}
    for se in (1, 10):
        pts[se] = pt_states(prob, th0, G, s['eps'], se)
        runs[f'pt_swap{se}'] = (lambda se=se: ops.pt_run(pts[se][0], pts[se][1], n, None, seed=seed))
    for fn in runs.values():           # warm-up: module load, first launches, the PT step counters reach n
        fn()
    times = {k: [] for k in runs}
    for _ in range(2):
        for k, fn in runs.items():
            times[k].append(timed(fn))
    for k, ts in times.items():
        out[k] = dict(seconds=ts, chain_steps_per_s=[K * n / t for t in ts])
    best = {k: K * n / min(ts) for k, ts in times.items()}
    for se in (1, 10):
        out[f'pt_swap{se}_over_hmc_chain_steps_per_s'] = best[f'pt_swap{se}'] / best['hmc']
        st, ps = pts[se]
        out[f'pt_swap{se}']['swap_rate_by_pair'] = ps.swap_rate().mean(0).cpu().tolist()
        out[f'pt_swap{se}']['cold_accept_rate'] = (st.naccept[:G].double().mean() / st.t).item()
    out['hmc']['accept_rate'] = (st_h.naccept.double().mean() / st_h.t).item()
    # share of device time in the swap kernel, PT with swap_every = 1, in a profiler run of its own
    st, ps = pts[1]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ops.pt_run(st, ps, n, None, seed=seed)
        torch.cuda.synchronize()
    tot = swap = 0.0
    for ev in prof.key_averages():
        dt = getattr(ev, 'device_time_total', None)
        if dt is None:
            dt = ev.cuda_time_total
        if ev.key.startswith('k_') or ' k_' in ev.key:          # every kernel of the library is named k_*
            tot += dt
            if 'k_pt_swap' in ev.key:
                swap += dt
    out['swap_kernel_share_of_kernel_time_swap1'] = swap / tot if tot > 0 else float('nan')
    return out


def two_modes(seed=12):
    """tests/test_gpu_pt.py's two-mode net: mode switches of the cold chains and round trips per second"""
    from quinn_b200.nns import MLP
    from quinn_b200.netdesc import netdesc_from_module
    rs = np.random.RandomState(1)
    N = 20
    x = np.linspace(-1, 1, N)[:, None]
    y = np.tanh(2 * x) + 0.3 * rs.randn(N, 1)
    desc = netdesc_from_module(MLP(1, 1, (1,), activ='tanh').double())
    prob = ops.Problem(desc, x, y, 0.5, dtype=torch.float64, device='cuda', prior_sigma=1.0,
                       prior_anchor=np.zeros(desc.n_params), fulldatasize=N)
    G, burn, keep, iw = 64, 1000, 3000, desc.layers[-1].w_off
    th0 = np.zeros((G, desc.n_params))
    th0[:, desc.layers[0].w_off], th0[:, iw] = 2.0, 1.0
    betas = ops.pt_ladder(8, 0.02)
    st = ops.ChainState(prob, np.tile(th0, (len(betas), 1)))
    ps = ops.PtState(st, G, betas, 0.05, 3, 'hmc', 1)
    ops.pt_run(st, ps, burn, None, seed=seed)
    trips0 = ps.round_trips.sum().item()
    rec = ops.Recorder(st, keep, store_every=1, sample_rows=G)
    t = timed(lambda: ops.pt_run(st, ps, keep, rec, seed=seed))
    sign = (rec.samples[:, :, iw] < 0)
    switches = (sign[:, 1:] != sign[:, :-1]).sum().item()
    return dict(net='MLP 1-1-1 tanh, prior sigma_p 1, N 20, sigma 0.5', groups=G, T=len(betas), beta_min=0.02,
                epsilon_cold=0.05, steps=keep, burn_in=burn, cold_fraction_w2_negative=sign.double().mean().item(),
                mode_switches_per_1000_steps_per_group=switches / G / keep * 1000,
                round_trips=ps.round_trips.sum().item() - trips0, seconds=t,
                round_trips_per_s=(ps.round_trips.sum().item() - trips0) / t,
                swap_rate_by_pair=ps.swap_rate().mean(0).cpu().tolist())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r9_pt_bench.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('pt_bench.py measures on a GPU and found none')
    torch.cuda.set_device(0)
    name, power = card()
    print(f'# {name}, power limit / max SM clock: {power}')
    res = dict(card=name, power_limit_and_max_sm_clock=power, shapes={})
    for s in SHAPES:
        r = run_shape(s)
        res['shapes'][s['name']] = r
        print(json.dumps({s['name']: r}))
    res['two_modes'] = two_modes()
    print(json.dumps({'two_modes': res['two_modes']}))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
