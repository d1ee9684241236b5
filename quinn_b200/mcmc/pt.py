"""Parallel tempering (replica exchange) on HMC or MALA: T tempered copies of every chain run in the same kernel launch,
and a deterministic even-odd swap round between neighbouring temperatures follows every ``swap_every`` steps
(qb_pt_run, quinn_b200/csrc/qb_pt.cuh)."""
import torch

from .. import ops
from .mcmc import MCMCBase


class PT(MCMCBase):
    """``base``: 'hmc' or 'mala', run at every temperature with ``L`` leapfrog steps (HMC).  ``betas``: the inverse
    temperatures 1 = beta_0 > ... > beta_{T-1} > 0; without them a geometric ladder of ``n_temps`` values from 1 to
    ``beta_min``.  ``epsilon``: a scalar (slot i steps with epsilon * beta_i^-1/2) or one step size per temperature.
    Slot i targets exp(beta_i * lp), the whole log-posterior tempered.  Without a prior (NN_MCMC uses none) a hot target
    can be improper where the likelihood goes flat, e.g. along saturated tanh units; hot chains then drift there, which
    slows the swaps but does not bias the cold chain.

    Each row of ``param_ini`` is a group: all T slots of the group start there.  The result dict has the usual keys for
    the cold (beta = 1) chains, so ``logpost`` and ``maxpost`` are untempered, and adds ``betas`` [T], ``step_sizes``
    [T], ``swap_rate`` [G, T-1] (accepted / attempted swaps of each neighbouring pair) and ``round_trips`` [G] (replicas
    that went from the cold end to the hot end and back).  ``last_state`` keeps all K = T * G slots.  PT needs a device
    log-posterior and has no replay mode."""

    def __init__(self, base='hmc', epsilon=0.05, L=3, betas=None, n_temps=8, beta_min=0.05, swap_every=1):
        super().__init__()
        if base not in ('hmc', 'mala'):
            raise ValueError("base must be 'hmc' or 'mala'")
        if int(swap_every) < 1:
            raise ValueError('swap_every must be >= 1')
        if base == 'hmc' and int(L) < 1:
            raise ValueError('HMC needs L >= 1')
        ladder = ops.pt_ladder(n_temps, beta_min) if betas is None else betas
        self.betas, self.step_sizes = ops.pt_check_ladder(ladder, epsilon)
        self.base, self.epsilon, self.L, self.swap_every = base, epsilon, int(L), int(swap_every)

    def run(self, nmcmc, param_ini, *, replay=None, **kw):
        if replay is not None:
            raise ValueError("sampler='pt' has no replay mode: its draws come from Philox")
        if self.logPost is not None and self._device_lp is None:
            raise ValueError('PT needs a device log-posterior (NN_MCMC.logpost with lpinfo=, or a DeviceLogPost)')
        return super().run(nmcmc, param_ini, **kw)

    def _auto_shards(self, theta0, replay, keep_on_device):
        return 1            # the host-pipelined path has no buffers for the tempered slots

    def _run_fused(self, nmcmc, theta0, seed, store_every, replay, chain_offset, verbose, segment_every=None,
                   on_segment=None):
        prob = self._device_lp.problem
        th0 = prob.theta(theta0)
        G, T = th0.shape[0], self.betas.size
        st = ops.ChainState(prob, th0.repeat(T, 1))            # slot-major: row i * G + g is slot i of group g
        ps = ops.PtState(st, G, self.betas, self.step_sizes, self.L, self.base, self.swap_every)
        # segment ends fall on multiples of both swap_every and store_every
        unit = max(self.swap_every, store_every) if store_every > 0 else self.swap_every
        nseg = 10 if (verbose and nmcmc >= 10) else 1
        bounds = [int(round(i * nmcmc / nseg)) for i in range(nseg + 1)]
        if segment_every:
            bounds = list(range(0, nmcmc, int(segment_every))) + [nmcmc]
        bounds = sorted(set([0, nmcmc] + [b - b % unit for b in bounds[1:-1]]))
        recs = []
        for a, b in zip(bounds[:-1], bounds[1:]):
            if b <= a:
                continue
            rec = ops.Recorder(st, b - a, store_every=store_every, sample_rows=G)
            ops.pt_run(st, ps, b - a, rec, seed=seed, chain_offset=chain_offset)
            recs.append(rec)
            if on_segment is not None:
                on_segment(st, rec, b)
            if verbose:
                acc = st.naccept[:G].double().mean().item() / b
                print('%d / %d completed, cold-chain acceptance rate %lg' % (b, nmcmc, acc))
        dev = prob.device
        chain = torch.cat([th0[:, None, :]] + [r.samples for r in recs if r.samples is not None], dim=1)
        if not recs:
            lp0 = ops.logpost(prob, th0)
            recs_lp, recs_al, recs_acc = [], [], []
        else:
            lp0 = recs[0].logpost0[:G]
            recs_lp, recs_al, recs_acc = ([r.logpost[:G] for r in recs], [r.alpha[:G] for r in recs],
                                          [r.accepted[:G] for r in recs])
        logpost = torch.cat([lp0[:, None]] + recs_lp, dim=1)
        alphas = torch.cat([torch.zeros((G, 1), dtype=torch.float64, device=dev)] + recs_al, dim=1)
        accepted = torch.cat([torch.zeros((G, 0), dtype=torch.uint8, device=dev)] + recs_acc, dim=1)
        self._ladder = dict(betas=torch.as_tensor(self.betas), step_sizes=torch.as_tensor(self.step_sizes))
        self.pt_state = ps
        return dict(chain=chain, mapparams=st.map_theta[:G], maxpost=st.map_lp[:G],
                    accrate=st.naccept[:G].double() / max(nmcmc, 1), logpost=logpost, alphas=alphas, accepted=accepted,
                    swap_rate=ps.swap_rate(), round_trips=ps.round_trips.clone(), state=st)

    def _finish(self, res, single, keep_on_device):
        out = super()._finish(res, single, keep_on_device)
        for k, v in self._ladder.items():            # per temperature, not per group: no group axis to drop
            out[k] = v.to(self._device_lp.problem.device) if keep_on_device else v.numpy()
        if single and not keep_on_device:
            out['round_trips'] = int(out['round_trips'])
        return out

    def sampler(self, current, imcmc):
        raise ValueError('PT needs a device log-posterior (NN_MCMC.logpost with lpinfo=, or a DeviceLogPost)')
