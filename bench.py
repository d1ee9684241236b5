#!/usr/bin/env python
"""Benchmark of the posterior-sampling hot path (contract: task statement "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c5|c5h|c2|c3|c4|c3fit] [--impl native|reference]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[4] / north_star target ("c5"): AMCMC, 10^5 chains TOTAL (sharded
over the N GPUs: strong scaling), MLP 3->64->64->1 (P=4481), N=10^4 synthetic points, fp32.  A "step" is one
AMCMC chain step of every chain (propose + log-posterior + accept, fused kernel 3).
metric = chain-steps/s, whole job.  Other workloads are selectable for the record:
  c5h HMC(L=3) on the config-5 shape (1e5 chains)                  (chain-steps/s)
  c2  HMC(L=3) 1,024 chains, MLP 2->32->32->1, N=1,000            (chain-steps/s)
  c3  256-member ensemble predictive mean/var over 10^6 points, MLP 10->128->128->1   (member-points/s)
  c4  VI ELBO value+grad, 128 MC samples, same net, N=10^5        (MC-sample evals/s)
One JSON line is printed by rank 0.  --dump-outputs DIR writes what the timed path computed in its last step to
DIR/<name>.npy; inputs and random streams are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

if 'reference' in sys.argv or any(a.startswith('--impl=ref') for a in sys.argv):
    # the reference arm uses every host thread; torchrun exports OMP_NUM_THREADS=1, which would also pin
    # numpy's LAPACK (the PxP SVD of admcmc.py:70) to one core -- undo that before numpy is imported
    for _v in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS', 'OPENBLAS_NUM_THREADS'):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


# ------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md section 8d)
# ------------------------------------------------------------------------------------------------
def scale01(xx, lo, hi):
    return xx * (hi - lo) + lo


def workload_spec(name):
    if name == 'c5':
        return dict(name='c5', d=3, hls=(64, 64), N=10_000, K=100_000, sigma=0.05, sampler='amcmc',
                    desc='AMCMC 1e5 chains (total), MLP 3-64-64-1 tanh, N=1e4 Sine data, gamma=0.01 t0=100 tadapt=1000')
    if name == 'c5h':
        return dict(name='c5', d=3, hls=(64, 64), N=10_000, K=100_000, sigma=0.05, sampler='hmc', L=3, eps=2e-6,
                    desc='HMC L=3 eps=2e-6, 1e5 chains (total), MLP 3-64-64-1 tanh, N=1e4 Sine data (north_star target shape)')
    if name == 'c2':
        return dict(name='c2', d=2, hls=(32, 32), N=1_000, K=1_024, sigma=0.02, sampler='hmc', L=3, eps=1e-4,
                    desc='HMC L=3 eps=1e-4, 1024 chains, MLP 2-32-32-1 tanh, N=1e3 Ackley data')
    if name == 'c3':
        return dict(name='c3', d=10, hls=(128, 128), N=1_000_000, K=256, sigma=0.05, sampler='predict',
                    desc='256-member ensemble predictive mean+var, MLP 10-128-128-1 tanh, 1e6 test points')
    if name == 'c4':
        return dict(name='c4', d=10, hls=(128, 128), N=100_000, K=128, sigma=0.05, sampler='vi',
                    desc='VI ELBO value+grad, 128 MC weight samples, MLP 10-128-128-1 tanh, N=1e5 Sine data')
    if name == 'c3fit':
        return dict(name='c3fit', d=10, hls=(128, 128), N=10_000, K=256, sigma=0.05, sampler='ensfit', dfrac=0.8,
                    desc='NN_Ens training (SURVEY 8f rank 1): 256 members trained together, MLP 10-128-128-1 tanh, N=1e4 Sine data, '
                         'dfrac=0.8, full-batch Adam epochs with best-model tracking')
    raise SystemExit(f'unknown workload {name}')


def make_data(spec):
    rs = np.random.RandomState(0)
    d, N = spec['d'], spec['N']
    if spec['name'] == 'c2':
        x = scale01(rs.rand(N, d), -1.5, 1.5)
        y = 0.02 * rs.randn(N)
        for i in range(d - 1):          # Ackley (func/funcs.py:90-109)
            y += np.exp(-0.2) * np.sqrt(x[:, i] ** 2 + x[:, i + 1] ** 2) + 3 * (np.cos(2 * x[:, i]) + np.sin(2 * x[:, i + 1]))
        return x, y.reshape(-1, 1)
    if spec['name'] == 'c5':
        x = scale01(rs.rand(N, d), -math.pi, math.pi)
    else:
        x = rs.rand(N, d)
    y = spec['sigma'] * rs.randn(N, 1) + np.sum(np.sin(x), axis=1).reshape(-1, 1)     # Sine (funcs.py:29-45)
    return x, y


def mlp_desc(d, hls, o=1):
    from quinn_b200.netdesc import NetDesc, Layer
    widths = [d] + list(hls) + [o]
    layers, off = [], 0
    for l in range(len(widths) - 1):
        w = off
        off += widths[l] * widths[l + 1]
        b = off
        off += widths[l + 1]
        layers.append(Layer(widths[l], widths[l + 1], w, b, 'tanh' if l < len(widths) - 2 else 'identity', 0.0))
    return NetDesc(d, o, off, layers)


def theta_init(spec, P, lo, hi):
    """theta0[k] for global chains lo..hi-1, a function of the GLOBAL chain index only (generated in blocks of 1024
    chains seeded by the block index), so the job is the same however it is sharded over GPUs.
    c5: rand(P) (nn_mcmc.py:124); c2: 0.1*randn(P); c3/c4: U(+-1/sqrt(fan_in))-like."""
    out = np.empty((hi - lo, P), dtype=np.float32)
    B = 1024
    for blk in range(lo // B, (hi + B - 1) // B):
        rs = np.random.RandomState(1234 + blk)
        if spec['name'] == 'c5':
            vals = rs.rand(B, P)
        elif spec['name'] == 'c2':
            vals = 0.1 * rs.randn(B, P)
        else:
            vals = (2 * rs.rand(B, P) - 1) / math.sqrt(spec['hls'][0])
        a, b = max(lo, blk * B), min(hi, (blk + 1) * B)
        out[a - lo:b - lo] = vals[a - blk * B:b - blk * B]
    return out


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md: the clocks line)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [c.strip() for c in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------
# the reference itself (pure Python): QUINN_REF -> baseline/_ref (pip --target install, travels to the GPU box) ->
# /root/reference (build container only); matplotlib is absent, so it is stubbed as SURVEY.md 8c describes
# ------------------------------------------------------------------------------------------------
def import_reference():
    from unittest.mock import MagicMock
    for n in ['matplotlib', 'matplotlib.pyplot', 'matplotlib.colors', 'matplotlib.lines', 'matplotlib.cm']:
        try:
            __import__(n)
        except Exception:
            sys.modules[n] = MagicMock()
    for cand in (os.environ.get('QUINN_REF'), os.path.join(ROOT, 'baseline', '_ref'), '/root/reference'):
        if cand and os.path.isdir(os.path.join(cand, 'quinn')):
            if cand not in sys.path:
                sys.path.insert(0, cand)
            try:
                import quinn.solvers.nn_mcmc      # noqa: F401
                return cand
            except Exception:
                sys.path.remove(cand)
    return None


def reference_baseline(spec, nsteps, nwarm):
    """The UNMODIFIED reference on the host cores, one chain / member (it has no batching; its rate per unit does not
    depend on how many units the job has).  Every reported step is actually executed."""
    import contextlib
    import io
    import torch
    where = import_reference()
    if where is None:
        return None
    torch.set_num_threads(os.cpu_count() or 1)
    from quinn.nns.mlp import MLP
    from quinn.solvers.nn_mcmc import NN_MCMC
    cores = torch.get_num_threads()
    x, y = make_data(spec)
    with contextlib.redirect_stdout(io.StringIO()):
        net = MLP(spec['d'], 1, spec['hls'], activ='tanh')
        uq = NN_MCMC(net, verbose=False)
    lpinfo = {'model': None, 'xd': x, 'yd': [yy for yy in y], 'ltype': 'classical', 'lparams': {'sigma': spec['sigma']}}
    rs = np.random.RandomState(7)
    th = rs.rand(uq.pdim)
    np.random.seed(7)

    def timed_run(sam, n):
        with contextlib.redirect_stdout(io.StringIO()):
            t0 = time.perf_counter()
            sam.run(n, th.copy())
            return time.perf_counter() - t0
    if spec['sampler'] == 'amcmc':
        from quinn.mcmc.admcmc import AMCMC
        sam = AMCMC(gamma=0.01, t0=100, tadapt=1000)
        sam.setLogPost(uq.logpost, None, lpinfo=lpinfo)
        if nwarm:
            timed_run(sam, nwarm)
        dt = timed_run(sam, nsteps)
        t0 = time.perf_counter()
        nlp = 0
        while time.perf_counter() - t0 < 3.0:
            uq.logpost(th, lpinfo)
            nlp += 1
        t_lp = (time.perf_counter() - t0) / nlp
        return dict(value=nsteps / dt, unit='chain-steps/s', cores=cores, kind='reference', where=where,
                    sample=f'reference AMCMC.run: {nsteps} steps of 1 chain of {spec["K"]} in {dt:.1f} s (every step: dense PxP '
                           f'np.random.multivariate_normal = SVD, admcmc.py:70, + NN_MCMC.logpost); chains are sequential in the '
                           f'reference, so the rate does not depend on the chain count; log-posterior alone: '
                           f'{1.0 / t_lp:.1f} evals/s ({t_lp * 1e3:.2f} ms)',
                    logpost_only_evals_per_s=1.0 / t_lp, step_s=dt / nsteps)
    if spec['sampler'] == 'hmc':
        from quinn.mcmc.hmc import HMC
        sam = HMC(epsilon=spec['eps'], L=spec['L'])
        sam.setLogPost(uq.logpost, uq.logpostgrad, lpinfo=lpinfo)
        if nwarm:
            timed_run(sam, nwarm)
        n = max(nsteps, 20)
        dt = timed_run(sam, n)
        return dict(value=n / dt, unit='chain-steps/s', cores=cores, kind='reference', where=where,
                    sample=f'reference HMC.run (L={spec["L"]}): {n} steps of 1 chain of {spec["K"]} in {dt:.2f} s '
                           f'({spec["L"] + 1} logpostgrad + 1 logpost per step, hmc.py:27-70)')
    if spec['sampler'] == 'predict':
        from quinn.ens.learner import Learner
        with contextlib.redirect_stdout(io.StringIO()):
            lrn = Learner(MLP(spec['d'], 1, spec['hls'], activ='tanh'))
        lrn.best_model, lrn.trained = lrn.nnmodel, True
        n = min(spec['N'], 200_000)
        lrn.predict(x[:1000])
        t0 = time.perf_counter()
        lrn.predict(x[:n])
        dt = time.perf_counter() - t0
        return dict(value=n / dt, unit='member-points/s', cores=cores, kind='reference', where=where,
                    sample=f'reference Learner.predict: 1 member x {n} points of {spec["N"]} (members are sequential, nn_ens.py:106-108)')
    return None


# ------------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference flow, timed on the host cores)
# ------------------------------------------------------------------------------------------------
def cpu_baseline(spec, budget_s=18.0):
    import torch
    from oracle.torch_port import RefPort, amcmc_proposal_draw
    torch.set_num_threads(os.cpu_count() or 1)
    x, y = make_data(spec)
    port = RefPort(spec['d'], 1, spec['hls'], 'tanh')
    ylist = [r for r in y]
    rs = np.random.RandomState(7)
    th = rs.rand(port.pdim)
    cores = torch.get_num_threads()
    if spec['sampler'] == 'predict':
        n = min(spec['N'], 200_000)
        t0 = time.perf_counter()
        port.forward(th, x[:n])
        dt = time.perf_counter() - t0
        return dict(value=n / dt, unit='member-points/s', cores=cores, kind='port',
                    sample=f'1 member x {n} points of {spec["N"]} (reference: Learner.predict per member, sequential)')

    def rate(fn, budget):
        for _ in range(2):
            fn()
        n, t0 = 0, time.perf_counter()
        while True:
            fn()
            n += 1
            dt = time.perf_counter() - t0
            if dt > budget or n >= 400:
                return dt / n
    if spec['sampler'] == 'amcmc':
        t_lp = rate(lambda: port.logpost(th, x, ylist, spec['sigma']), 5.0)
        t0 = time.perf_counter()
        amcmc_proposal_draw(th)                     # one dense-covariance draw (SVD of PxP), admcmc.py:70
        t_draw = time.perf_counter() - t0
        return dict(value=1.0 / (t_lp + t_draw), unit='chain-steps/s', cores=cores, kind='port',
                    sample=f'1 chain of {spec["K"]}: {t_lp * 1e3:.2f} ms/logpost (avg over ~5 s) + {t_draw:.2f} s/proposal draw '
                           f'(1 draw, PxP SVD); logpost-only rate {1.0 / t_lp:.1f} evals/s',
                    logpost_only_evals_per_s=1.0 / t_lp, proposal_draw_s=t_draw)
    if spec['sampler'] == 'hmc':
        t_g = rate(lambda: port.logpostgrad(th, x, ylist, spec['sigma']), 6.0)
        t_v = rate(lambda: port.logpost(th, x, ylist, spec['sigma']), 3.0)
        step = (spec['L'] + 1) * t_g + t_v          # hmc.py: L+1 gradients + 1 value per step
        return dict(value=1.0 / step, unit='chain-steps/s', cores=cores, kind='port',
                    sample=f'1 chain of {spec["K"]}: {(spec["L"] + 1)} grads ({t_g * 1e3:.2f} ms) + 1 value ({t_v * 1e3:.2f} ms) per step')
    if spec['sampler'] == 'ensfit':
        # the reference's procedure for ONE member (nnfit.py:125-166): torch Adam on the MSE, full batch, validation loss
        # on the member's own data before each update; members are trained one after the other (nn_ens.py:56-66)
        from quinn_b200.nns import MLP
        net = MLP(spec['d'], 1, spec['hls'], activ='tanh').double()
        nsub = int(spec['N'] * spec['dfrac'])
        xt, yt = torch.as_tensor(x[:nsub]), torch.as_tensor(y[:nsub])
        opt = torch.optim.Adam(net.parameters(), lr=0.01)
        mse = torch.nn.MSELoss(reduction='mean')

        def epoch():
            loss = mse(net(xt), yt)
            with torch.no_grad():
                mse(net(xt), yt).item()
            opt.zero_grad()
            loss.backward()
            opt.step()
        t_e = rate(epoch, 10.0)
        return dict(value=1.0 / t_e, unit='member-epochs/s', cores=cores, kind='port',
                    sample=f'1 member of {spec["K"]}: full-batch Adam epoch on {nsub} points ({t_e * 1e3:.2f} ms), members sequential')
    # vi: value+grad per MC sample
    t_g = rate(lambda: port.logpostgrad(th, x, ylist, spec['sigma']), 10.0)
    return dict(value=1.0 / t_g, unit='MC-sample evals/s', cores=cores, kind='port',
                sample='viloss fwd+bwd per MC weight sample, sequential over samples (bnet.py:202-205)')


def run_reference_arm(args, spec):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (rank 0 only): the installed
    reference (baseline/_ref) when it imports, else the oracle port.  Every step it reports is executed."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    t0 = time.perf_counter()
    base = None
    try:
        base = reference_baseline(spec, max(1, args.steps), max(0, args.warmup))
    except Exception as exc:        # pragma: no cover
        sys.stderr.write(f'reference import / run failed ({exc!r}); timing the oracle port instead\n')
    if base is None:
        base = cpu_baseline(spec, budget_s=10.0)
    v = float(base['value'])
    line = dict(impl='reference', metric=metric_name(spec), value=v, unit=base['unit'], n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 / v if v > 0 else None, higher_is_better=True, scaling='strong',
                vs_baseline=None, dtype='f64', data='synthetic', config=workload_config(spec),
                cpu_baseline=base, e2e=dict(value=v, unit=base['unit'], h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                note='a reference step is one chain-step of ONE chain (the reference has no batching: its chain-steps/s does not '
                     'depend on the number of chains); ms_per_step is that, so steps x ms_per_step is what this process ran',
                wall_s=time.perf_counter() - t0)
    print(json.dumps(line), flush=True)


def workload_config(spec):
    """The `config` object both arms print (same keys and values, so the driver's same_config check compares like with like)."""
    return dict(workload=spec['desc'], chains_or_units_total=spec['K'], N=spec['N'],
                l2='GPU arm: inputs larger than L2 (per-chain / per-member state is GBs and is streamed once per step)')


def metric_name(spec):
    return {'amcmc': 'MCMC chain-steps/sec', 'hmc': 'MCMC chain-steps/sec', 'predict': 'predictive member-points/sec',
            'vi': 'VI MC-sample evals/sec', 'ensfit': 'ensemble-training member-epochs/sec'}[spec['sampler']]


# ------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='c5')
    ap.add_argument('--impl', default='native')
    ap.add_argument('--chains', type=int, default=0, help='override the total chain count (development)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the c5h / c3 legs reported under "extra"')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the arrays the last timed step of the headline workload computed to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    spec = workload_spec(args.workload)
    if args.chains:
        spec['K'] = args.chains
    if args.impl == 'reference':
        run_reference_arm(args, spec)
        return

    import torch
    from quinn_b200 import dist, _lib
    rank, world, local = dist.init()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py (native arm) needs a CUDA device; there is no CPU fallback')
    torch.cuda.set_device(local)
    _lib.load()
    args.warmup = max(args.warmup, 3)
    line = run_native(spec, args, args.steps, args.warmup, rank, world, local, headline=True)
    # the other halves of BASELINE.json's metric ("log-post+grad evals/s", "predictive pts/s"), outside the headline timed
    # region: HMC at the north_star target shape (tensor-core gradient kernel), the config-3 predictive sweep, config 4 (VI ELBO
    # value + gradient) and the config-3 ensemble fit, each on its own tensor-core kernel
    if args.workload == 'c5' and not args.no_extra and not args.chains:
        extra = {}
        for name in ('c5h', 'c3', 'c4', 'c3fit', 'c2'):
            torch.cuda.empty_cache()
            sub = run_native(workload_spec(name), args, 3, 3, rank, world, local, headline=False)
            if rank == 0:
                extra[name] = {k: sub[k] for k in ('metric', 'value', 'unit', 'ms_per_step', 'steps', 'warmup', 'config', 'launch', 'roofline',
                                                   'gpu_launches', 'diagnostics') if k in sub}
        if rank == 0:
            line['extra'] = extra
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as td
        td.destroy_process_group()


def run_native(spec, args, steps, warmup, rank, world, local, headline):
    """Times `steps` steps of one workload (after `warmup`), device-timed with CUDA events between barriers, max over
    ranks; returns the JSON line as a dict (rank 0) -- the headline additionally carries e2e, cpu_baseline and clocks."""
    import torch
    from quinn_b200 import ops, dist, _lib
    lib = _lib.load()
    dev = torch.device('cuda', local)
    desc = mlp_desc(spec['d'], spec['hls'])
    P, S = desc.n_params, desc.macs_per_point()
    x, y = make_data(spec)
    lo, hi = dist.shard_range(spec['K'], rank, world)
    Kloc = hi - lo
    N = spec['N']
    dt = torch.float32
    F_v = 2.0 * N * S
    F_vg = 6.0 * N * S - 2.0 * N * desc.layers[0].n_in * desc.layers[0].n_out

    th0_host = torch.from_numpy(theta_init(spec, P, lo, hi)).pin_memory()
    st = None
    recs = {}        # per-step log-posteriors / MH ratios / accept flags of every chain are recorded, as in a real run
    if spec['sampler'] in ('amcmc', 'hmc'):
        prob = ops.Problem(desc, x, y, spec['sigma'], dtype=dt, device=dev)
        st = ops.ChainState(prob, th0_host)
        if spec['sampler'] == 'amcmc':
            samp = ops.AmcmcState(st, gamma=0.01, t0=100, tadapt=1000, adapt='diag')
            advance = lambda n: ops.amcmc_run(st, samp, n, recs[n], seed=2026, chain_offset=lo)      # noqa: E731
            flop_per_unit, kernel_name = F_v, 'k_amcmc<float>'
        else:
            samp = ops.HmcState(st, epsilon=spec['eps'], L=spec['L'], method='hmc')
            advance = lambda n: ops.hmc_run(st, samp, n, recs[n], seed=2026, chain_offset=lo)        # noqa: E731
            flop_per_unit, kernel_name = spec['L'] * F_vg, 'k_hmc<float>'
        for n in {warmup, steps}:           # record buffers are allocated outside the timed region
            recs[n] = ops.Recorder(st, n, store_every=0)
        units_per_step = spec['K']
        plan = prob.plan_info(Kloc, spec['sampler'] == 'hmc')
        # what MCMCBase.run returns for the last step (quinn_b200/mcmc/mcmc.py), per chain.  The recorded MH ratio is
        # unclipped and overflows to inf when a proposal is far more probable, so the acceptance probability
        # min(1, ratio) that decides the step is written instead
        outputs = lambda: (dict(theta=st.theta, mapparams=st.map_theta, maxpost=st.map_lp, naccept=st.naccept,   # noqa: E731
                                logpost=recs[steps].logpost[:, -1], accept_prob=recs[steps].alpha[:, -1].clamp(max=1.0),
                                accepted=recs[steps].accepted[:, -1]), {})
    elif spec['sampler'] == 'predict':
        # members stay whole on every rank; the 10^6 test points are sharded (no collective needed, SURVEY 8e)
        plo, phi = dist.shard_range(N, rank, world)
        xs = torch.as_tensor(x[plo:phi], dtype=dt, device=dev)
        th = torch.as_tensor(theta_init(spec, P, 0, spec['K']), device=dev)
        cnet = desc.to_c()
        last = {}

        def advance(n):
            for _ in range(n):
                last['moments'] = ops.predict(desc, th, xs, dtype=dt, device=dev, want_out=False, want_moments=True, cnet=cnet)[1:]
        # predictive mean and variance per test point (points are sharded over ranks)
        outputs = lambda: (dict(mean=last['moments'][0], var=last['moments'][1]), {})       # noqa: E731
        flop_per_unit, kernel_name = 2.0 * S, 'k_predict<float>'
        units_per_step = spec['K'] * N
        import ctypes as _C
        _pi = (_C.c_int64 * 8)()
        lib.qb_plan_info(_C.byref(cnet), _lib.QB_F32, spec['K'], xs.shape[0], 0, _pi)
        plan = dict(TM=_pi[0], threads=_pi[1], smem_bytes=_pi[2], tensor_core=int(_pi[6]), tmem_cols=int(_pi[7]))
    elif spec['sampler'] == 'ensfit':
        # members are sharded over ranks; every member has its own dfrac subset (nn_ens.py:62-63); one step = one
        # full-batch epoch of every member: kernel 2 with per-member data + best-model copy + Adam
        from quinn_b200.ens.batched import MemberTrainer
        nsub = int(N * spec['dfrac'])
        rs_s = np.random.RandomState(99)
        subsets = np.stack([rs_s.permutation(N)[:nsub] for _ in range(spec['K'])])[lo:hi]
        trainer = MemberTrainer(desc, theta_init(spec, P, lo, hi), x, y, subsets, val=None, lrate=0.01, dtype=dt, device=dev)
        epoch_no = [0]

        def advance(n):
            for _ in range(n):
                trainer.epoch(epoch_no[0])
                epoch_no[0] += 1
        # what fit_members returns (quinn_b200/ens/batched.py), per member
        outputs = lambda: (dict(theta=trainer.theta, best_theta=trainer.best_theta, best_loss=trainer.best_loss,     # noqa: E731
                                loss=trainer.last_crit), {})
        F_fit = 6.0 * nsub * S - 2.0 * nsub * desc.layers[0].n_in * desc.layers[0].n_out
        flop_per_unit, kernel_name = F_fit, 'k_logpost_grad<float>'
        units_per_step = spec['K']
        _pi = (__import__('ctypes').c_int64 * 8)()
        lib.qb_plan_info(__import__('ctypes').byref(desc.to_c()), _lib.QB_F32, Kloc, nsub, 1, _pi)
        plan = dict(TM=_pi[0], threads=_pi[1], smem_bytes=_pi[2], splits=_pi[3], blocks=_pi[4], tensor_core=int(_pi[6]))
    else:   # vi
        prob = ops.Problem(desc, x, y, 1.0, dtype=dt, device=dev)
        mu = torch.as_tensor(theta_init(spec, P, 0, 1)[0], device=dev)
        rho = torch.full((P,), -4.5, dtype=dt, device=dev)
        B = N
        c_ssq = 0.5 * B / (Kloc * world * B) / spec['sigma'] ** 2
        last = {}

        def advance(n):
            for i in range(n):
                w, eps, logq, logp = ops.vi_sample(mu, rho, Kloc, 0.5, 1.0, 1.0, seed=11 + rank, step=i + 1)
                lp, glp = ops.logpost_grad(prob, w)
                gmu, grho = ops.vi_backward(mu, rho, eps, w, glp, 0.5, 1.0, 1.0, c_ssq, -1.0 / spec['K'], 1.0 / spec['K'])
                if world > 1:          # the MC samples are sharded over ranks: sum their gradient contributions (2P floats)
                    dist._allreduce(gmu)
                    dist._allreduce(grho)
                last.update(logpost=lp, logq=logq, logprior=logp, grad_mu=gmu, grad_rho=grho)
        # the ELBO terms per MC sample and the ELBO gradient with respect to the variational parameters
        outputs = lambda: ({k: last[k] for k in ('logpost', 'logq', 'logprior')},                 # noqa: E731
                           {k: last[k] for k in ('grad_mu', 'grad_rho')})
        flop_per_unit, kernel_name = F_vg, 'k_logpost_grad<float>'
        units_per_step = spec['K']
        plan = prob.plan_info(Kloc, True)

    # ---- FP32 FMA peak, measured live (the roofline denominator of the CUDA-core kernels; MEASURED_PEAKS.json has none)
    fma_peak = ops.fma_peak(dt, 0, iters=20000, device=dev)

    # ---- warm-up, then the timed region (device-timed, barrier + sync on both sides, max over ranks)
    advance(warmup)
    torch.cuda.synchronize()
    dist.barrier()
    clocks = ClockSampler(local)
    if rank == 0 and headline:
        clocks.start()
    l0 = lib.qb_launch_count()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    advance(steps)
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms_local = e0.elapsed_time(e1)
    launches = lib.qb_launch_count() - l0
    ms = dist.max_over_ranks(ms_local)
    clk = clocks.stop() if (rank == 0 and headline) else None

    # cross-chain diagnostics reduced over NVLink: mean acceptance rate and the Gelman-Rubin R-hat of the log-posterior over
    # the timed steps (per-chain moments on each rank, small all-reduces, quinn_b200/dist.py)
    diag = None
    if spec['sampler'] in ('amcmc', 'hmc'):
        acc = st.naccept.double() / float(st.t)
        sacc = torch.stack([acc.sum(), (acc * acc).sum(), torch.tensor(float(Kloc), device=dev, dtype=torch.float64)])
        dist._allreduce(sacc)
        diag = dict(mean_accept_rate=(sacc[0] / sacc[2]).item())
        if steps >= 2:
            lph = recs[steps].logpost
            diag['rhat_logpost'] = dist.rhat(lph.mean(1), lph.var(1, unbiased=True), steps).item()

    if headline and args.dump_outputs:
        per_unit, whole = outputs()
        first, n_units = (plo, N) if spec['sampler'] == 'predict' else (lo, spec['K'])
        dump_outputs(args.dump_outputs, per_unit, whole, n_units, first, rank)

    value = units_per_step * steps / (ms * 1e-3)
    units_local = Kloc if spec['sampler'] != 'predict' else spec['K'] * xs.shape[0]
    achieved = units_local * steps * flop_per_unit / (ms_local * 1e-3)
    tc = int(plan.get('tensor_core', 0))
    # DRAM bytes of the dominant kernel per launch: dram__bytes_read.sum + dram__bytes_write.sum of ONE `ncu --set full`
    # capture of this build (profiles/r2_traffic.json, written from the committed capture by scripts/ncu_traffic.py),
    # scaled per chain-step / member-point to this launch; null when no capture of this kernel is committed
    traffic = measured_traffic(spec, tc, units_local * steps)
    roofline = dict(bound='fp32', kernel=kernel_name, achieved=achieved / 1e12, peak=fma_peak / 1e12, unit='TFLOP/s',
                    frac=achieved / fma_peak, traffic=traffic,
                    note='FP32 CUDA-core FMA bound (not hbm/tensor): peak = live FMA micro-benchmark qb_fma_peak; '
                         'achieved = algorithmic GEMM flops (2 flop/MAC, SURVEY 8d) / CUDA-event time of the timed launches')
    if tc:
        # The GEMMs run on the tensor cores (tcgen05 kind::tf32, operands split hi/lo = 3 MMA passes for fp32-level accuracy).
        # Denominator: the measured dense bf16 rate (sustained figure, the kernel is timed inside a long step); TF32 runs at
        # half of it and the 3 passes divide it by three again, so 1/6 of it is the ceiling of this algorithm on the tensor pipe.
        peak_bf16, src = measured_bf16_peak()
        sm_mhz = (clk or {}).get('sm_mhz') or 1965.0
        v3 = spec['sampler'] in ('amcmc', 'predict') and int(plan.get('threads', 0)) in (288, 544)      # warp-specialised kernels (qb_tc3.cuh)
        kname = {'amcmc': 'k_amcmc_tc3 (tcgen05.mma: layer 0 kind::tf32 x3 passes, hidden GEMM kind::f16 x3 passes with exact power-of-two '
                          'scaling, issued by a dedicated warp; sigmoid epilogues on MUFU; chain state in shared memory)' if v3 else
                          'k_amcmc<float,2> (tcgen05.mma kind::tf32 x3 passes + MUFU tanh epilogue)',
                 'predict': 'k_predict_tc3 (tcgen05.mma: layer 0 kind::tf32 x3 passes, hidden GEMM kind::f16 x3 passes, dedicated issue warp; '
                            'sigmoid epilogues on MUFU)' if v3 else 'k_predict_tc (tcgen05.mma kind::tf32 x3 passes + MUFU tanh epilogue)',
                 'hmc': 'k_hmc_tc (forward, back-propagation and weight-gradient GEMMs on tcgen05.mma kind::tf32 x3 passes)'
                 }.get(spec['sampler'], 'k_logpost_grad_tc (tcgen05.mma kind::tf32 x3 passes)')
        if tc == 4:            # fp16-split gradient kernels (qb_tg8.cuh)
            kname = ('k_hmc_tc128' if spec['sampler'] == 'hmc' else 'k_logpost_grad_tc128') + \
                    '<%d> (layer 0, forward, back-propagation and both weight-gradient GEMMs on tcgen05.mma kind::f16 x3 passes, fp16 hi/lo ' \
                    'operands with exact power-of-two scaling, one shared-memory image per matrix for its K-major and MN-major use, ' \
                    'dedicated issue warp%s)' % (max(64, int(spec['hls'][0])), '; the 32-wide net runs with zero-padded units' if int(spec['hls'][0]) == 32 else '')
        roofline = dict(bound='tensor', kernel=kname, achieved=achieved / 1e12, peak=peak_bf16, unit='TFLOP/s',
                        frac=achieved / 1e12 / peak_bf16, traffic=traffic, peak_source=src,
                        tf32_peak=peak_bf16 / 2.0, frac_of_tf32_peak=achieved / 1e12 / (peak_bf16 / 2.0),
                        tf32x3_peak=peak_bf16 / 6.0, frac_of_tf32x3_peak=achieved / 1e12 / (peak_bf16 / 6.0),
                        fp32_core_peak=fma_peak / 1e12, x_fp32_core_peak=achieved / fma_peak,
                        note='achieved = algorithmic fp32 GEMM flops (2 flop/MAC, SURVEY 8d) / CUDA-event time; peak = measured '
                             'dense bf16 TFLOP/s (%s); kind::tf32 runs at half of it (tf32_peak) and these kernels do 3 TF32 passes '
                             'per GEMM for fp32 accuracy (ceiling = peak/6, frac_of_tf32x3_peak); x_fp32_core_peak compares with the '
                             'live CUDA-core FMA peak that bounds the SIMT kernels' % src)
        if tc == 4:
            # every GEMM of the gradient kernel is 3 kind::f16 passes: ceiling of the algorithm on the tensor pipe = peak / 3
            roofline.update(f16x3_peak=peak_bf16 / 3.0, frac_of_f16x3_peak=achieved / 1e12 / (peak_bf16 / 3.0))
            roofline['note'] = ('achieved = algorithmic fp32 GEMM flops (2 flop/MAC, SURVEY 8d: value + gradient = 6 N S - 2 N n0 n1) / '
                                'CUDA-event time; peak = measured dense bf16 TFLOP/s (%s); this kernel does 3 kind::f16 passes per GEMM for '
                                'fp32-level accuracy (ceiling = peak/3, frac_of_f16x3_peak); its MMAs take both operands from shared memory '
                                'and are bound by that operand traffic (8 KB per 128x128x16 MMA = 64 cycles), see DESIGN.md 4d' % src)
        if v3:
            # tensor-pipe ceiling of THIS algorithm: per point 3 x (8 x 64) tf32 MAC slots (layer 0, K padded to 8; tf32 = half the
            # bf16 rate) + 3 x (64 x 64) f16 slots against S algorithmic MACs
            Hh = int(spec['hls'][0])
            K0 = 8 if Hh == 64 else 16
            slots = 2.0 * 3 * K0 * Hh + 3.0 * Hh * Hh
            roofline.update(algo_ceiling=peak_bf16 * S / slots, frac_of_algo_ceiling=achieved / 1e12 / (peak_bf16 * S / slots),
                            algo_ceiling_note='peak x S / (bf16-equivalent MMA slots per point): layer 0 3 tf32 passes over K=8 (16 for 128-wide nets), '
                                              'hidden layer 3 fp16 passes (hi*hi + lo*hi + hi*lo)')
        if spec['sampler'] in ('amcmc', 'predict'):
            # what bounds the value kernels is the sigmoid/tanh epilogue on the MUFU pipe (16 results/clk/SM): one ex2 per
            # activation + one reciprocal shared by 8 (hot-shape kernel: 1.125 MUFU per activation) or by 4 (1.25)
            n_tanh = N * sum(l.n_out for l in desc.layers[:-1])
            n_evals = Kloc if spec['sampler'] == 'amcmc' else spec['K'] * xs.shape[0] / N     # N-point sweeps per step
            mufu_ach = n_evals * steps * n_tanh * (1.125 if v3 else 1.25) / (ms_local * 1e-3)
            mufu_peak = 16.0 * 148 * sm_mhz * 1e6
            roofline['mufu'] = dict(achieved_gops=mufu_ach / 1e9, peak_gops=mufu_peak / 1e9, frac=mufu_ach / mufu_peak)

    if rank != 0 and not headline:
        return None
    line = dict(metric=metric_name(spec), value=value, unit=cpu_unit(spec), n_gpus=world, steps=steps,
                warmup=warmup, ms_per_step=ms / steps, higher_is_better=True, scaling='strong',
                vs_baseline=None, dtype='f32', data='synthetic', config=workload_config(spec),
                launch=dict(per_rank=Kloc, P=P, macs_per_point=S, plan=plan),
                gpu_launches=int(launches), roofline=roofline, diagnostics=diag)
    if headline:
        # ---- end to end through the public API with host buffers
        e2e = None
        if not args.no_e2e:
            del recs, advance
            if st is not None:
                del st, samp
            torch.cuda.empty_cache()
            e2e = run_e2e(spec, desc, x, y, th0_host, lo, args, dev, world)
        cb = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                cb = reference_baseline(spec, 2, 0)         # the real reference, 2 executed steps of one chain
            except Exception:       # pragma: no cover
                cb = None
            if cb is None:
                cb = cpu_baseline(spec)
        line.update(clocks=clk, e2e=e2e, cpu_baseline=cb)
    return line if rank == 0 else None


DUMP_BYTES = 60 * 10 ** 6          # array bytes of one dump; with the .npy headers the files stay under 64 MB


def dump_outputs(path, per_unit, whole, n_units, first, rank):
    """Write the outputs of the last timed step as path/<name>.npy, float64 where the device array is float64 or an
    integer count, float32 otherwise.  per_unit: arrays whose first dimension is this rank's units (chains, members,
    test points or MC samples), starting at global unit `first`; whole: arrays every rank holds in full.  When all units would
    take more than DUMP_BYTES, a fixed seeded sample of them is written (the same units for any number of GPUs), with
    its global indices as unit_index.npy."""
    import torch
    from quinn_b200 import dist
    conv = lambda t: t.detach().double() if t.dtype in (torch.float64, torch.int64) else t.detach().float()   # noqa: E731
    per_unit = {k: conv(t) for k, t in per_unit.items()}
    whole = {k: conv(t) for k, t in whole.items()}
    row_bytes = sum(math.prod(t.shape[1:]) * t.element_size() for t in per_unit.values())
    room = DUMP_BYTES - sum(t.numel() * t.element_size() for t in whole.values())
    keep = None
    if n_units * row_bytes > room:
        keep = np.sort(np.random.RandomState(0).choice(n_units, room // (row_bytes + 8), replace=False))
        n_local = next(iter(per_unit.values())).shape[0]
        rows = torch.as_tensor(keep[(keep >= first) & (keep < first + n_local)] - first)
        per_unit = {k: t[rows.to(t.device)] for k, t in per_unit.items()}
    per_unit = {k: dist.gather_to_rank0(t.contiguous()) for k, t in per_unit.items()}
    if rank != 0:
        return
    os.makedirs(path, exist_ok=True)
    for name, t in list(per_unit.items()) + list(whole.items()):
        np.save(os.path.join(path, name + '.npy'), t.cpu().numpy())
    if keep is not None:
        np.save(os.path.join(path, 'unit_index.npy'), keep.astype(np.float64))


def measured_traffic(spec, tc, units):
    """DRAM bytes (read + write) of the dominant kernel for `units` chain-steps / member-points, from the committed
    `ncu --set full` capture of this build (profiles/r2_traffic.json: bytes per unit per kernel), or None."""
    path = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    key = {'amcmc': 'k_amcmc_tc3' if tc else 'k_amcmc', 'hmc': ('k_hmc_tc128' if tc == 4 else 'k_hmc_tc') if tc else 'k_hmc',
           'predict': 'k_predict_tc' if tc else 'k_predict'}.get(spec['sampler'])
    if key == 'k_hmc_tc128' and int(spec['hls'][0]) != 64:
        return None                               # the committed capture is the 3-64-64-1 shape (config 5 / c5h)
    try:
        with open(path) as f:
            per_unit = json.load(f)[key]['dram_bytes_per_unit']
        return float(per_unit) * units
    except Exception:
        return None


def measured_bf16_peak():
    """Dense bf16 TFLOP/s of this pool's B200s as measured by the driver (sustained figure); fallback per
    B200_PROFILING.md when the file is absent."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            d = json.load(f)
        return float(d.get('bf16_tflops_sustained') or d['bf16_tflops']), 'of measured (MEASURED_PEAKS.json, sustained)'
    except Exception:
        return 1400.0, 'of fallback (1.4 PFLOP/s sustained)'


def cpu_unit(spec):
    return {'amcmc': 'chain-steps/s', 'hmc': 'chain-steps/s', 'predict': 'member-points/s', 'vi': 'MC-sample evals/s',
            'ensfit': 'member-epochs/s'}[spec['sampler']]


def run_e2e(spec, desc, x, y, th0_host, lo, args, dev, world):
    """Same metric through the public API (the reference-facing classes) with HOST inputs and outputs."""
    import torch
    from quinn_b200 import dist
    from quinn_b200.mcmc import AMCMC, HMC, DeviceLogPost
    from quinn_b200 import ops
    steps = args.steps
    P = desc.n_params
    if spec['sampler'] in ('amcmc', 'hmc'):
        # The call a user of the reference makes: NN_MCMC(net).fit(x, y, zflag=False, nmcmc, param_ini=host[K,P], sampler=...)
        # -> host result dict (nn_mcmc.py:100-139 with the many-chain extension).  Every call uploads the chain states
        # from pinned host memory and downloads final states, MAP states and the per-step log-posteriors / MH ratios /
        # accept flags of every chain.  Fixed per-call costs (GB-sized transfers) are amortised over e2e_steps >= 100 steps,
        # as in a real run (the reference's example runs 10,000).
        from quinn_b200.nns import MLP
        from quinn_b200.solvers import NN_MCMC
        e2e_steps = max(steps, 100 if spec['sampler'] == 'amcmc' else 30)
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            uq = NN_MCMC(MLP(spec['d'], 1, spec['hls'], activ='tanh'), verbose=False, dtype=torch.float32, device=dev)
        sp = dict(gamma=0.01, t0=100, tadapt=1000, adapt='diag') if spec['sampler'] == 'amcmc' else dict(epsilon=spec['eps'], L=spec['L'])

        def once(n):
            res = uq.fit(x, y, zflag=False, datanoise=spec['sigma'], nmcmc=n, param_ini=th0_host, sampler=spec['sampler'],
                         sampler_params=sp, seed=5, store_every=n, chain_offset=lo)
            torch.cuda.synchronize()
            return res['logpost'], res['accrate']
        once(2)                               # warm-up: library load, pinned buffers of the small shape
        once(e2e_steps)                       # warm-up at the timed shape (allocates its pinned result buffers once)
        dist.barrier()
        t0 = time.perf_counter()
        once(e2e_steps)
        dist.barrier()
        dtm = dist.max_over_ranks(time.perf_counter() - t0)
        Kl = th0_host.shape[0]
        h2d = (th0_host.numel() * 4 + x.size * 4 + y.size * 4) / e2e_steps
        d2h = (2 * Kl * P * 4 + Kl * P * 4 + Kl * (2 * (e2e_steps + 1) * 8 + e2e_steps + 16)) / e2e_steps     # chain[K,2,P], MAP, scalars
        return dict(value=spec['K'] * e2e_steps / dtm, unit='chain-steps/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                    steps=e2e_steps, wall_s=dtm,
                    api='NN_MCMC(net, dtype=float32).fit(x, y, zflag=False, nmcmc=steps, param_ini=pinned host [K,P], sampler=...) -> '
                        'host result dict (chain, mapparams, logpost, alphas, accrate); states above 256 MB go through 8 shards '
                        'pipelined on 2 streams')
    if spec['sampler'] == 'ensfit':
        from quinn_b200.nns import MLP
        from quinn_b200.solvers import NN_Ens
        Kl = th0_host.shape[0]
        net = MLP(spec['d'], 1, spec['hls'], activ='tanh')

        def once():
            np.random.seed(4)
            ens = NN_Ens(net, nens=Kl, dfrac=spec['dfrac'], dtype=torch.float32)
            ens.fit(x, y, nepochs=steps, lrate=0.01, freq_out=0)              # host data in, trained torch modules out
            torch.cuda.synchronize()
            return ens
        once()
        dist.barrier()
        t0 = time.perf_counter()
        once()
        dist.barrier()
        dtm = dist.max_over_ranks(time.perf_counter() - t0)
        return dict(value=spec['K'] * steps / dtm, unit='member-epochs/s', h2d_bytes_per_step=(x.size + y.size + Kl * P) * 4 / steps,
                    d2h_bytes_per_step=Kl * P * 4 / steps,
                    api='NN_Ens(net, nens, dfrac).fit(x, y, nepochs=steps) from host arrays -> trained member modules '
                        '(includes building the K learners and unflattening the best parameters)')
    if spec['sampler'] == 'predict':
        plo, phi = dist.shard_range(spec['N'], *dist.env_rank_world()[:2])
        xh = torch.from_numpy(np.ascontiguousarray(x[plo:phi], dtype=np.float32)).pin_memory()
        thh = torch.from_numpy(theta_init(spec, P, 0, spec['K'])).pin_memory()

        def once():
            _, m, v = ops.predict(desc, thh, xh, dtype=torch.float32, device=dev, want_out=False, want_moments=True)
            return m.cpu(), v.cpu()
        once()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            once()
        dist.barrier()
        dtm = dist.max_over_ranks(time.perf_counter() - t0)
        return dict(value=spec['K'] * spec['N'] * steps / dtm, unit='member-points/s', h2d_bytes_per_step=xh.numel() * 4 + thh.numel() * 4,
                    d2h_bytes_per_step=2 * xh.shape[0] * 4, api='ops.predict(host theta, host x) -> host mean, var')
    return None


if __name__ == '__main__':
    main()
