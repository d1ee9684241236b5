"""NN_MCMC with the reference's interface (quinn/solvers/nn_mcmc.py:15-200).

``logpost`` / ``logpostgrad`` evaluate in CUDA kernels 1 / 2; ``fit`` runs the fused chain-step kernel 3
for one chain (reference behaviour) or for K chains when ``param_ini`` is (K,P) / ``nchains`` is given;
the predictive calls run kernel 4."""
import copy

import numpy as np
import torch

from .. import ops
from ..mcmc.admcmc import AMCMC
from ..mcmc.hmc import HMC
from ..mcmc.mala import MALA
from ..mcmc.nuts import NUTS
from ..mcmc.pt import PT
from ..mcmc.mcmc import DeviceLogPost
from ..netdesc import netdesc_from_module
from ..nns.nnwrap import NNWrap, nn_p
from .quinn import QUiNNBase


class NN_MCMC(QUiNNBase):
    def __init__(self, nnmodel, verbose=True, dtype=torch.float64, device='cuda'):
        """``dtype`` (extension): arithmetic type of the kernels; float64 reproduces the reference
        (tchutils.py:9), float32 is the throughput mode."""
        super().__init__(nnmodel)
        self.verbose = verbose
        self.pdim = sum(p.numel() for p in self.nnmodel.parameters())
        print("Number of parameters:", self.pdim)
        if self.verbose:
            self.print_params(names_only=True)
        self.samples = None
        self.cmode = None
        self.lpinfo = {}
        self.dtype, self.device = dtype, device
        self.desc = netdesc_from_module(self.nnmodel)
        self._problems = {}

    # ---- device handle
    def device_logpost(self, lpinfo):
        """GPU-resident log-posterior for this lpinfo dict (built once, unlike nn_mcmc.py:55-66)."""
        if lpinfo['ltype'] != 'classical':
            raise ValueError('Likelihood type is not recognized.')
        # keyed by CONTENT (data bytes, shapes, sigma): mutating lpinfo in place, which is legal in the reference (it rebuilds
        # everything per call), gives a new key; calling fit() again with the same data reuses the resident copy
        import hashlib
        xd = np.ascontiguousarray(np.asarray(lpinfo['xd'], dtype=np.float64))
        yd = np.ascontiguousarray(np.asarray(lpinfo['yd'], dtype=np.float64))
        hsh = hashlib.blake2b(xd.tobytes(), digest_size=16)
        hsh.update(yd.tobytes())
        key = (xd.shape, yd.shape, float(lpinfo['lparams']['sigma']), str(self.dtype), str(self.device), hsh.hexdigest())
        h = self._problems.get(key)
        if h is None:
            prob = ops.Problem(self.desc, xd, yd, lpinfo['lparams']['sigma'], dtype=self.dtype, device=self.device)
            h = DeviceLogPost(prob)
            self._problems = {key: h}
        return h

    def logpost(self, modelpars, lpinfo):
        """log p(theta | D) as a float for theta (P,), or an array (K,) for theta (K,P) (nn_mcmc.py:45-71)."""
        modelpars = np.asarray(modelpars, dtype=np.float64)
        lp = ops.logpost(self.device_logpost(lpinfo).problem, modelpars)
        return float(lp[0].item()) if modelpars.ndim == 1 else lp.cpu().numpy()

    def logpostgrad(self, modelpars, lpinfo):
        """Gradient of the log-posterior, (P,) or (K,P) (nn_mcmc.py:73-98)."""
        modelpars = np.asarray(modelpars, dtype=np.float64)
        _, g = ops.logpost_grad(self.device_logpost(lpinfo).problem, modelpars)
        g = g.double().cpu().numpy()
        return g[0] if modelpars.ndim == 1 else g

    def fit(self, xtrn, ytrn, zflag=True, datanoise=0.05, nmcmc=6000, param_ini=None, sampler='amcmc',
            sampler_params=None, *, nchains=None, seed=None, store_every=1, replay=None, chain_offset=0,
            distributed=False, diag_every=None, gather=True, data_sharded=False, keep_on_device=False):
        """Sample the posterior of the flat parameters (nn_mcmc.py:100-139).

        ``sampler='nuts'`` runs the No-U-Turn sampler (quinn_b200.mcmc.NUTS, sampler_params: epsilon, max_depth, n_adapt,
        target_accept) in this process; its result dict adds ``tree_depth``, ``n_leapfrog``, ``diverging`` and
        ``step_size`` per transition.

        ``sampler='pt'`` runs parallel tempering on HMC or MALA (quinn_b200.mcmc.PT, sampler_params: base, epsilon, L,
        betas, n_temps, beta_min, swap_every) in this process.  ``nchains`` / the rows of ``param_ini`` count groups: each
        runs T tempered chains, and the result dict (and so predict_* and diagnose()) holds the cold ones; it adds
        ``betas``, ``step_sizes``, ``swap_rate`` and ``round_trips``.

        Extensions (keyword-only): ``nchains`` / a (K,P) ``param_ini`` run K chains at once (``samples``
        becomes (K, M+1, P)); ``seed``, ``store_every``, ``replay``, ``chain_offset`` are passed to the sampler.
        With ``zflag`` the start point is refined by BFGS on -logpost using the analytic gradient of kernel 2
        (the reference uses finite differences, nn_mcmc.py:126).

        Multi-GPU (one process per GPU under torchrun, ``quinn_b200.dist.init()`` or an initialised process group):
        ``distributed=True`` shards the K chains over the ranks (block partition, Philox keyed by the global chain index, so
        the chains are the ones a single process would run), reduces the R-hat of the log-posterior and the acceptance
        rate over all ranks every ``diag_every`` steps (default: the sampler's ``tadapt`` or nmcmc/10) on a side stream
        (``self.diagnostics``), and, with ``gather``, collects the result dict on rank 0 (other ranks keep their shard).
        ``keep_on_device=True`` leaves the result dict (and ``self.samples``) as CUDA tensors: predict_ens / predict_mom_sample
        / predict_stats then thin and evaluate the chain without a host round trip.
        ``data_sharded=True``: every rank passes ITS slice of the data and all chains; each step's log-posterior
        (and gradient) is the all-reduced sum of the per-rank partial sums (the N-sharded mode for data that exceed one
        GPU; propose / accept run redundantly and identically on every rank)."""
        assert xtrn.shape[0] == ytrn.shape[0]
        if sampler == 'pt' and (data_sharded or distributed or replay is not None):
            raise ValueError("sampler='pt' runs in a single process from Philox draws: distributed=True, "
                             "data_sharded=True and replay are not supported with it")
        if sampler == 'nuts' and (data_sharded or distributed):
            raise ValueError("sampler='nuts' runs in a single process: distributed=True and data_sharded=True are not "
                             "supported with it")
        if data_sharded:
            return self._fit_data_sharded(xtrn, ytrn, datanoise, nmcmc, param_ini, sampler, sampler_params, nchains, seed,
                                          store_every)
        if distributed:
            return self._fit_distributed(xtrn, ytrn, zflag, datanoise, nmcmc, param_ini, sampler, sampler_params, nchains,
                                         seed, store_every, chain_offset, diag_every, gather)
        self.lpinfo = {'model': nn_p, 'xd': xtrn, 'yd': [y for y in ytrn], 'ltype': 'classical',
                       'lparams': {'sigma': datanoise}}
        if param_ini is None:
            shape = (self.pdim,) if nchains is None else (nchains, self.pdim)
            param_ini = np.random.rand(*shape)
            if zflag:
                param_ini = self._map_start(param_ini)
        sampler_params = {} if sampler_params is None else sampler_params
        if sampler == 'amcmc':
            mymcmc = AMCMC(**sampler_params)
            mymcmc.setLogPost(self.logpost, None, lpinfo=self.lpinfo)
        elif sampler == 'hmc':
            mymcmc = HMC(**sampler_params)
            mymcmc.setLogPost(self.logpost, self.logpostgrad, lpinfo=self.lpinfo)
        elif sampler == 'mala':                     # promised by the docstring at nn_mcmc.py:110
            mymcmc = MALA(**sampler_params)
            mymcmc.setLogPost(self.logpost, self.logpostgrad, lpinfo=self.lpinfo)
        elif sampler == 'nuts':
            mymcmc = NUTS(**sampler_params)
            mymcmc.setLogPost(self.logpost, self.logpostgrad, lpinfo=self.lpinfo)
        elif sampler == 'pt':
            mymcmc = PT(**sampler_params)
            mymcmc.setLogPost(self.logpost, self.logpostgrad, lpinfo=self.lpinfo)
        else:
            raise ValueError(f"sampler {sampler!r} is not one of 'amcmc', 'hmc', 'mala', 'nuts', 'pt'")
        res = mymcmc.run(param_ini=param_ini, nmcmc=nmcmc, seed=seed, store_every=store_every, replay=replay,
                         chain_offset=chain_offset, verbose=self.verbose, keep_on_device=keep_on_device)
        self.sampler_obj, self.mcmc_results = mymcmc, res
        self.samples, self.cmode = res['chain'], res['mapparams']
        return res

    # ---- multi-GPU drivers ------------------------------------------------------------------------------------------
    def _make_sampler(self, sampler, sampler_params):
        sampler_params = {} if sampler_params is None else sampler_params
        if sampler == 'amcmc':
            m = AMCMC(**sampler_params)
            m.setLogPost(self.logpost, None, lpinfo=self.lpinfo)
        elif sampler == 'hmc':
            m = HMC(**sampler_params)
            m.setLogPost(self.logpost, self.logpostgrad, lpinfo=self.lpinfo)
        elif sampler == 'mala':
            m = MALA(**sampler_params)
            m.setLogPost(self.logpost, self.logpostgrad, lpinfo=self.lpinfo)
        else:
            raise ValueError(f"sampler {sampler!r} is not one of 'amcmc', 'hmc', 'mala'")
        return m

    def _fit_distributed(self, xtrn, ytrn, zflag, datanoise, nmcmc, param_ini, sampler, sampler_params, nchains, seed,
                         store_every, chain_offset, diag_every, gather):
        """Chains sharded over the ranks; diagnostics reduced on a side stream; results gathered on rank 0."""
        from .. import dist
        rank, world = dist.world()
        self.lpinfo = {'model': nn_p, 'xd': xtrn, 'yd': [y for y in ytrn], 'ltype': 'classical', 'lparams': {'sigma': datanoise}}
        dev = torch.device(self.device)
        # every rank must use the same start points and the same Philox seed: rank 0's are broadcast
        if param_ini is None:
            K = 1 if nchains is None else int(nchains)
            p0 = torch.as_tensor(np.random.rand(K, self.pdim), dtype=torch.float64)
        else:
            p0 = torch.as_tensor(np.atleast_2d(np.asarray(param_ini, dtype=np.float64)))
        sd = torch.tensor([int(seed) if seed is not None else int(np.random.randint(1, 2 ** 31 - 1))], dtype=torch.int64)
        if world > 1:
            on = dev if dev.type == 'cuda' else torch.device('cpu')
            p0 = dist.broadcast_from_rank0(p0.to(on)).cpu()
            sd = dist.broadcast_from_rank0(sd.to(on)).cpu()
        K = p0.shape[0]
        lo, hi = dist.shard_range(K, rank, world)
        mine = p0[lo:hi].numpy()
        if zflag:
            mine = np.atleast_2d(self._map_start(mine))
        mymcmc = self._make_sampler(sampler, sampler_params)
        every = int(diag_every or getattr(mymcmc, 'tadapt', 0) or max(1, nmcmc // 10))
        every = max(1, min(every, nmcmc))
        diag = dist.RunningDiagnostics(dev)
        res = mymcmc.run(param_ini=mine, nmcmc=nmcmc, seed=int(sd.item()), store_every=store_every,
                         chain_offset=chain_offset + lo, verbose=False, keep_on_device=True, segment_every=every, on_segment=diag)
        self.diagnostics = diag.finish()
        if self.verbose and rank == 0:
            for row in self.diagnostics:
                print('%d / %d completed, acceptance rate %lg, R-hat(logpost) %lg' % (row['step'], nmcmc, row['accept_rate'], row['rhat_logpost']))
        self.sampler_obj = mymcmc
        self.shard = (lo, hi)
        out = {}
        for k, v in res.items():
            if k == 'state':
                continue
            full = dist.gather_to_rank0(v.contiguous()) if (gather and world > 1) else v
            if full is None:            # not rank 0: keep the local shard
                full = v
            out[k] = full.cpu().numpy().astype(bool) if full.dtype in (torch.uint8, torch.bool) else full.cpu().numpy()
        self.mcmc_results = out
        self.samples, self.cmode = out['chain'], out['mapparams']
        return out

    def predict_moments_distributed(self, x, nens=10, nburn=1000):
        """Posterior-predictive mean / variance (ddof=1) over the thinned samples of ALL ranks' chains (quinn.py:85-99 with
        the thinning rule of nn_mcmc.py:194-196 applied to every chain): per-rank sums of y and y^2, one all-reduce each.
        Call after fit(distributed=True, gather=False); every rank returns the same arrays."""
        from .. import dist
        thetas = self._thinned(nens, nburn)
        dev = torch.device(self.device)
        out, _, _ = ops.predict(self.desc, thetas, np.asarray(x), dtype=self.dtype, device=dev)
        y = out.double()
        mean, var = dist.reduce_predictive_moments(y.sum(0), (y * y).sum(0), y.shape[0])
        return mean.cpu().numpy(), var.cpu().numpy()

    def _fit_data_sharded(self, xtrn, ytrn, datanoise, nmcmc, param_ini, sampler, sampler_params, nchains, seed, store_every):
        """N-sharded mode: this rank holds a slice of the data; log-posteriors / gradients are all-reduced partial sums."""
        from .. import dist
        from ..mcmc.mcmc import ShardedDataLogPost
        rank, world = dist.world()
        dev = torch.device(self.device)
        n_local = torch.tensor([float(xtrn.shape[0])], dtype=torch.float64, device=dev)
        n_total = int(dist.allreduce_sum_(n_local.clone()).item())
        prob = ops.Problem(self.desc, np.asarray(xtrn), np.asarray(ytrn), datanoise, dtype=self.dtype, device=dev)
        slp = ShardedDataLogPost(prob, n_total)
        if param_ini is None:
            K = 1 if nchains is None else int(nchains)
            param_ini = np.random.rand(K, self.pdim)
        p0 = torch.as_tensor(np.atleast_2d(np.asarray(param_ini, dtype=np.float64)), device=dev)
        sd = torch.tensor([int(seed) if seed is not None else int(np.random.randint(1, 2 ** 31 - 1))], dtype=torch.int64, device=dev)
        p0, sd = dist.broadcast_from_rank0(p0), dist.broadcast_from_rank0(sd)
        sampler_params = {} if sampler_params is None else sampler_params
        mymcmc = {'amcmc': AMCMC, 'hmc': HMC, 'mala': MALA}[sampler](**sampler_params)
        mymcmc.setLogPost(slp, slp.grad if sampler != 'amcmc' else None)
        res = mymcmc.run(param_ini=p0.cpu().numpy(), nmcmc=nmcmc, seed=int(sd.item()), store_every=store_every, verbose=False)
        self.sampler_obj, self.mcmc_results = mymcmc, res
        self.samples, self.cmode = res['chain'], res['mapparams']
        return res

    def _map_start(self, param_ini):
        from scipy.optimize import minimize

        def fg(th):
            lp, g = ops.logpost_grad(self.device_logpost(self.lpinfo).problem, th)
            return -float(lp[0].item()), -g[0].double().cpu().numpy()
        rows = np.atleast_2d(param_ini)
        if rows.shape[0] > self.map_batched_above:
            return self._map_start_batched(rows)
        out = np.array([minimize(fg, r, jac=True, method='BFGS', options={'gtol': 1e-13}).x for r in rows])
        return out[0] if np.ndim(param_ini) == 1 else out

    map_batched_above = 8          # more start points than this: one batched optimisation instead of K BFGS runs
    map_start_steps = 300          # Adam ascent steps of the batched MAP start

    def _map_start_batched(self, rows, nsteps=None, lrate=0.01):
        """MAP pre-conditioning of MANY chains at once (SURVEY 8f rank 3; the reference has one chain and BFGS with
        finite differences, nn_mcmc.py:125-127): Adam ascent on log p(theta|D) for all K starts together - kernel 2,
        qb_adam_step and qb_copy_rows_where, nothing leaves the device - returning the best state each chain visited."""
        import ctypes as C
        from .. import _lib
        from ..ops import _ptr, _stream, qb_dtype
        nsteps = self.map_start_steps if nsteps is None else nsteps
        prob = self.device_logpost(self.lpinfo).problem
        lib = _lib.load()
        theta = prob.theta(rows).clone()
        K, P = theta.shape
        m, v, best = torch.zeros_like(theta), torch.zeros_like(theta), theta.clone()
        best_lp = torch.full((K,), -float('inf'), dtype=torch.float64, device=theta.device)
        lp = torch.empty(K, dtype=torch.float64, device=theta.device)
        g = torch.empty_like(theta)
        qdt = qb_dtype(prob.dtype)
        for step in range(1, nsteps + 2):
            ops.logpost_grad(prob, theta, lp, g)
            better = lp > best_lp
            mask = better.to(torch.uint8)
            with torch.cuda.device(theta.device):
                _lib.check(lib.qb_copy_rows_where(qdt, _ptr(best), _ptr(theta), _ptr(mask), K, P, _stream()), 'qb_copy_rows_where')
            best_lp = torch.where(better, lp, best_lp)
            if step > nsteps:
                break
            with torch.cuda.device(theta.device):
                _lib.check(lib.qb_adam_step(qdt, _ptr(theta), _ptr(g), _ptr(m), _ptr(v), K * P, lrate, 0.9, 0.999, 1e-8, 0.0,
                                            step, -1.0, _stream()), 'qb_adam_step')
        self.map_start_logpost = best_lp.cpu().numpy()
        return best.double().cpu().numpy()

    # ---- predictive (nn_mcmc.py:142-200)
    def get_best_model(self, param):
        nnw = NNWrap(self.nnmodel)
        nnw.p_unflatten(param)
        return copy.deepcopy(nnw.nnmodel)

    def _forward(self, thetas, x):
        if not torch.is_tensor(thetas):                  # CUDA tensors (keep_on_device) are passed through untouched
            thetas = np.asarray(thetas, dtype=np.float64)
        out, _, _ = ops.predict(self.desc, thetas, np.asarray(x), dtype=self.dtype, device=self.device)
        return out.double().cpu().numpy()

    def predict_MAP(self, x):
        cm = self.cmode if torch.is_tensor(self.cmode) else np.asarray(self.cmode)
        return self._forward(cm, x)[0] if cm.ndim == 1 else self._forward(cm, x)

    def predict_sample(self, x, param):
        return self._forward(param, x)[0]

    def _thinned(self, nens, nburn):
        """Rows samples[nburn + j*nevery], nevery = int((M'-nburn)/nens) (nn_mcmc.py:194-196); for a
        multi-chain run the same rows of every chain, chain-major."""
        s = self.samples if torch.is_tensor(self.samples) else np.asarray(self.samples)      # device chains stay on the device
        nevery = int((s.shape[-2] - nburn) / nens)
        rows = [nburn + j * nevery for j in range(nens)]
        return s[..., rows, :].reshape(-1, s.shape[-1])

    def diagnose(self, max_lag=0):
        """Cross-chain diagnostics of the last fit computed on the device (qb_post.cu): R-hat of the log-posterior over the
        second half of the run and the effective sample size of the log-posterior per chain (extensions: the reference has
        neither)."""
        from .. import post
        lp = torch.as_tensor(self.mcmc_results['logpost'])
        lp = lp[None, :] if lp.dim() == 1 else lp
        half = lp[:, lp.shape[1] // 2:]
        r = post.rhat(half) if half.shape[0] > 1 else torch.full((1,), float('nan'))
        e = post.ess(half, max_lag)
        return dict(rhat_logpost=float(r.reshape(-1)[0].item()), ess_logpost=e.cpu().numpy(), nsteps=int(half.shape[1]))

    def predict_ens(self, x, nens=10, nburn=1000):
        return self._forward(self._thinned(nens, nburn), x)

    def _ens_thetas(self, nens):
        # predict_mom_sample -> base predict_ens(x, nens=nsam) in the reference calls the override with
        # nburn=1000 (quinn.py:84 -> nn_mcmc.py:180)
        return self.desc, self._thinned(nens, 1000), self.dtype
