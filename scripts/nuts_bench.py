"""NUTS (qb_nuts_run) against HMC(L=3) (qb_hmc_run) on the same net, dtype, K, N and kernel path:

1. gradient evaluations per second: HMC makes L = 3 per chain-step; NUTS makes one per leapfrog (the recorded n_leapfrog),
   so the ratio shows the per-leapfrog cost of the tree bookkeeping and of the launch tail (chains whose trees are deep
   keep their block while the others have finished);
2. mean tree depth after warm-up;
3. ESS of the log-posterior per second (quinn_b200.post.ess, summed over the chains) for NUTS with its adapted step sizes
   against HMC at bench.py's hand-picked epsilon (config 2: 1e-4; config-5 shape: 2e-6; the fp64 case has none in
   bench.py and uses 1e-4).

Both samplers first run their warm-up (NUTS: n_adapt transitions of step-size adaptation; HMC: as many steps) from the
same start, then the timed window, which ends in a device synchronise.  Shapes: config 2 (fp32, MLP 2-32-32-1, N = 10^3,
K = 1024; the fp16-split tensor-core path, plan code 4, which takes 32-wide tanh nets with zero-padded units), the config-5 shape (fp32, MLP 3-64-64-1, N = 10^4, TG8 path; fewer chains than bench.py's
10^5) and an fp64 CUDA-core case (MLP 1-16-16-1, N = 10^3).  Card name and power limit are read in the same run.

    python scripts/nuts_bench.py [--out profiles/r8_nuts_bench.json]
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

from quinn_b200 import ops, post                 # noqa: E402
from quinn_b200.netdesc import NetDesc, Layer    # noqa: E402

SHAPES = [
    dict(name='c2', d=2, hls=(32, 32), N=1_000, K=1_024, sigma=0.02, dtype=torch.float32, eps_hmc=1e-4, path=4,
         n_adapt=200, n_keep=200, max_depth=8),
    dict(name='c5_shape', d=3, hls=(64, 64), N=10_000, K=1_024, sigma=0.05, dtype=torch.float32, eps_hmc=2e-6, path=4,
         n_adapt=100, n_keep=100, max_depth=8),
    dict(name='f64_cuda', d=1, hls=(16, 16), N=1_000, K=512, sigma=0.05, dtype=torch.float64, eps_hmc=1e-4, path=0,
         n_adapt=200, n_keep=200, max_depth=8),
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


def run_shape(s, seed=7):
    desc = mlp_desc(s['d'], s['hls'])
    x, y = data(s)
    prob = ops.Problem(desc, x, y, s['sigma'], dtype=s['dtype'], device='cuda')
    K, P = s['K'], desc.n_params
    path = prob.plan_info(K, True)['tensor_core']
    assert path == s['path'], (s['name'], path)
    th0 = 0.1 * np.random.RandomState(1234).randn(K, P)
    out = dict(net=f"MLP {s['d']}-{'-'.join(map(str, s['hls']))}-1 tanh", P=P, N=s['N'], K=K, dtype=str(s['dtype']),
               plan_code=path, max_depth=s['max_depth'], n_adapt=s['n_adapt'], n_keep=s['n_keep'])

    # NUTS: warm-up with adaptation, then the timed window
    st = ops.ChainState(prob, th0)
    ns = ops.NutsState(st, epsilon=s['eps_hmc'] * 10, max_depth=s['max_depth'], n_adapt=s['n_adapt'], target_accept=0.8)
    wrec, wnrec = ops.Recorder(st, s['n_adapt'], store_every=0), ops.NutsRecords(st, s['n_adapt'])
    t_warm = timed(lambda: ops.nuts_run(st, ns, s['n_adapt'], wrec, wnrec, seed=seed))
    rec, nrec = ops.Recorder(st, s['n_keep'], store_every=0), ops.NutsRecords(st, s['n_keep'])
    t_nuts = timed(lambda: ops.nuts_run(st, ns, s['n_keep'], rec, nrec, seed=seed))
    nleap = int(nrec.n_leapfrog.sum().item())
    ess_nuts = post.ess(rec.logpost.contiguous())
    out['nuts'] = dict(
        warmup_s=t_warm, warmup_grad_evals=int(wnrec.n_leapfrog.sum().item()), timed_s=t_nuts, grad_evals=nleap,
        grad_evals_per_s=nleap / t_nuts, mean_tree_depth=nrec.tree_depth.double().mean().item(),
        max_tree_depth=int(nrec.tree_depth.max().item()), mean_n_leapfrog=nrec.n_leapfrog.double().mean().item(),
        divergences=int(nrec.diverging.sum().item()), mean_accept_stat=rec.alpha.mean().item(),
        moved_fraction=rec.accepted.double().mean().item(),
        step_size_median=float(nrec.step_size[:, -1].median().item()),
        step_size_range=[float(nrec.step_size[:, -1].min().item()), float(nrec.step_size[:, -1].max().item())],
        ess_logpost_sum=ess_nuts.sum().item(), ess_logpost_per_s=ess_nuts.sum().item() / t_nuts)

    # HMC(L=3) at the hand-picked epsilon, same start, same warm-up length
    st = ops.ChainState(prob, th0)
    hm = ops.HmcState(st, epsilon=s['eps_hmc'], L=3, method='hmc')
    t_hwarm = timed(lambda: ops.hmc_run(st, hm, s['n_adapt'], None, seed=seed))
    n_h = s['n_keep'] * 3
    hrec = ops.Recorder(st, n_h, store_every=0)
    t_hmc = timed(lambda: ops.hmc_run(st, hm, n_h, hrec, seed=seed))
    ess_hmc = post.ess(hrec.logpost.contiguous())
    out['hmc'] = dict(epsilon=s['eps_hmc'], L=3, warmup_s=t_hwarm, steps=n_h, timed_s=t_hmc, grad_evals=K * n_h * 3,
                      grad_evals_per_s=K * n_h * 3 / t_hmc, accept_rate=hrec.accepted.double().mean().item(),
                      ess_logpost_sum=ess_hmc.sum().item(), ess_logpost_per_s=ess_hmc.sum().item() / t_hmc)
    out['nuts_over_hmc_grad_evals_per_s'] = out['nuts']['grad_evals_per_s'] / out['hmc']['grad_evals_per_s']
    out['nuts_over_hmc_ess_per_s'] = out['nuts']['ess_logpost_per_s'] / max(out['hmc']['ess_logpost_per_s'], 1e-300)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r8_nuts_bench.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('nuts_bench.py measures on a GPU and found none')
    torch.cuda.set_device(0)
    name, power = card()
    print(f'# {name}, power limit / max SM clock: {power}')
    res = dict(card=name, power_limit_and_max_sm_clock=power, shapes={})
    for s in SHAPES:
        r = run_shape(s)
        res['shapes'][s['name']] = r
        print(json.dumps({s['name']: r}))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
