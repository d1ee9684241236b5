"""No-U-Turn sampler (Hoffman & Gelman 2014) with per-chain dual-averaging step sizes; every transition of a chain runs
inside one fused kernel (qb_nuts_run, quinn_b200/csrc/qb_nuts.cuh)."""
import torch

from .. import ops
from .mcmc import MCMCBase


class NUTS(MCMCBase):
    """``epsilon``: initial step size (the dual averaging starts from it; with ``n_adapt=0`` it is kept).  ``max_depth``:
    at most 2^max_depth - 1 leapfrog steps per transition (1..12).  ``n_adapt``: transitions of step-size adaptation
    towards the acceptance statistic ``target_accept``; later transitions use each chain's averaged step size.

    NUTS needs a device log-posterior (``NN_MCMC.logpost`` with ``lpinfo=`` or a ``DeviceLogPost``).  Besides the usual
    keys, its result dict has ``tree_depth``, ``n_leapfrog``, ``diverging`` and ``step_size`` per transition; ``alphas``
    holds the acceptance statistic and ``accepted`` whether the chain moved."""

    def __init__(self, epsilon=0.05, max_depth=10, n_adapt=1000, target_accept=0.8):
        super().__init__()
        if not 1 <= int(max_depth) <= ops.NUTS_MAX_DEPTH:
            raise ValueError(f'max_depth must lie in [1, {ops.NUTS_MAX_DEPTH}]')
        if not 0.0 < float(target_accept) < 1.0:
            raise ValueError('target_accept must lie in (0, 1)')
        if not float(epsilon) > 0.0:
            raise ValueError('epsilon must be > 0')
        if int(n_adapt) < 0:
            raise ValueError('n_adapt must be >= 0')
        self.epsilon, self.max_depth = float(epsilon), int(max_depth)
        self.n_adapt, self.target_accept = int(n_adapt), float(target_accept)

    def run(self, nmcmc, param_ini, *, replay=None, **kw):
        if replay is not None:
            raise ValueError('NUTS has no replay mode: its draws come from Philox')
        if self.logPost is not None and self._device_lp is None:
            raise ValueError('NUTS needs a device log-posterior (NN_MCMC.logpost with lpinfo=, or a DeviceLogPost)')
        return super().run(nmcmc, param_ini, **kw)

    def _auto_shards(self, theta0, replay, keep_on_device):
        return 1            # the host-pipelined path has no buffers for the NUTS records

    def _run_fused(self, *args, **kw):
        self._nrecs = []
        res = super()._run_fused(*args, **kw)
        for key in ('tree_depth', 'n_leapfrog', 'diverging', 'step_size'):
            res[key] = torch.cat([getattr(r, key) for r in self._nrecs], dim=1)
        res['diverging'] = res['diverging'].bool()
        self._nrecs = []
        return res

    def _device_sampler_state(self, st):
        return ops.NutsState(st, epsilon=self.epsilon, max_depth=self.max_depth, n_adapt=self.n_adapt,
                             target_accept=self.target_accept)

    def _device_advance(self, st, samp, nsteps, rec, kw):
        nrec = ops.NutsRecords(st, nsteps)
        ops.nuts_run(st, samp, nsteps, rec, nrec, **kw)
        self._nrecs.append(nrec)

    def sampler(self, current, imcmc):
        raise ValueError('NUTS needs a device log-posterior (NN_MCMC.logpost with lpinfo=, or a DeviceLogPost)')
