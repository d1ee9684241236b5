"""TEST INFRASTRUCTURE (oracle): numpy restatement of parallel tempering as qb_pt_run runs it (quinn_b200/csrc/qb_pt.cuh)
-- the tempered HMC / MALA step on beta * lp and beta * grad with the momenta and uniforms of oracle/philox.hmc_draws,
the deterministic even-odd (DEO) swap round with its rescaling of lp and gradient, and the round-trip bookkeeping -- so
that a device run can be replayed step by step.  Each MH and swap decision also reports its margin: how far the log of
its uniform was from the log of its acceptance ratio, relative to the size of the quantities that ratio was formed from.
"""
import math

import numpy as np

from oracle import philox

STREAM_PT = 6              # QB_STREAM_PT of quinn_b200/csrc/qb_pt.cuh


def _margin(log_u, log_r, scale):
    if not np.isfinite(log_r):
        return math.inf if log_r == -math.inf or log_r == math.inf else 0.0
    return abs(log_u - log_r) / (scale + 1e-300)


def step(lpg, beta, eps, method, L, z, lp, g, seed, chain, t):
    """One tempered HMC (method 0) / MALA (method 1) step from (z, lp = beta * lp(z), g = beta * grad).  Returns
    (z, lp, g, accepted, mh, margin)."""
    P = z.size
    p = philox.normals(seed, chain, t, philox.STREAM_INCR, P)
    u = philox.uniform(seed, chain, t)

    def tl(th):
        v, gr = lpg(th)
        return beta * v, beta * gr
    K_cur = float(np.dot(p, p)) / 2.0
    if method == 0:
        mom = p + eps * g / 2
        prop = z.copy()
        for jj in range(L):
            prop = prop + eps * mom
            lpp, gp = tl(prop)
            mom = mom + (eps * gp if jj != L - 1 else eps * gp / 2)
    else:
        prop = z + (0.5 * eps * eps) * g + eps * p
        lpp, gp = tl(prop)
        mom = p + eps * (g + gp) / 2
    K_prop = float(np.dot(mom, mom)) / 2.0
    log_r = (-lp + K_cur) - (-lpp + K_prop)
    with np.errstate(over='ignore', invalid='ignore'):
        mh = math.exp(log_r) if log_r < 700 else math.inf
    acc = bool(u < mh)
    margin = _margin(math.log(u), log_r, abs(lp) + abs(lpp) + K_cur + K_prop)
    if acc:
        return prop, lpp, gp, True, mh, margin
    return z, lp, g, False, mh, margin


def swap_round(st, betas, G, seed, chain_offset, r):
    """DEO round r on st = dict(z [K,P], lp [K], g [K,P], replica [K], last_end [K], round_trips [G], attempts [G,T-1],
    accepts [G,T-1]) in place.  Returns the decision margins [(g, i, accepted, margin)]."""
    T = len(betas)
    out = []
    for grp in range(G):
        for i in range(r % 2, T - 1, 2):
            a, b = i * G + grp, (i + 1) * G + grp
            ba, bb = betas[i], betas[i + 1]
            Ua, Ub = st['lp'][a] / ba, st['lp'][b] / bb
            x = (ba - bb) * (Ub - Ua)
            u = float(philox.u01(philox.rand4(seed, chain_offset + a, r, STREAM_PT, np.zeros(1))[0])[0])
            with np.errstate(over='ignore'):
                acc = bool(u < math.exp(min(x, 700.0)))
            st['attempts'][grp, i] += 1
            out.append((grp, i, acc, _margin(math.log(u), x, (ba - bb) * (abs(Ua) + abs(Ub)))))
            if acc:
                st['accepts'][grp, i] += 1
                la, lb = st['lp'][a], st['lp'][b]
                st['lp'][a], st['lp'][b] = lb * (ba / bb), la * (bb / ba)
                ga, gb = st['g'][a].copy(), st['g'][b].copy()
                st['g'][a], st['g'][b] = gb * (ba / bb), ga * (bb / ba)
                st['z'][[a, b]] = st['z'][[b, a]]
                st['replica'][[a, b]] = st['replica'][[b, a]]
        if T > 1:
            round_trip_update(st, G, T, grp)
    return out


def round_trip_update(st, G, T, grp):
    """After a round: the replica in the hottest slot has last visited the hot end; the one in slot 0 completes a round
    trip if it last visited the hot end."""
    st['last_end'][st['replica'][(T - 1) * G + grp]] = -1
    rc = st['replica'][grp]
    if st['last_end'][rc] == -1:
        st['last_end'][rc] = 1
        st['round_trips'][grp] += 1


def init_state(lpg, theta0, betas):
    """K = T * G slot-major chains started at theta0 [G, P] (every slot of group g at theta0[g])."""
    theta0 = np.atleast_2d(np.asarray(theta0, dtype=np.float64))
    G, T = theta0.shape[0], len(betas)
    K = T * G
    z = np.tile(theta0, (T, 1))
    lp, g = np.zeros(K), np.zeros_like(z)
    for k in range(K):
        v, gr = lpg(z[k])
        lp[k], g[k] = betas[k // G] * v, betas[k // G] * gr
    last_end = np.zeros(K, dtype=np.int64)
    last_end[:G] = 1
    if T > 1:
        last_end[(T - 1) * G:] = -1
    return dict(z=z, lp=lp, g=g, map_lp=lp.copy(), map_z=z.copy(), naccept=np.zeros(K, dtype=np.int64),
                replica=np.arange(K), last_end=last_end, round_trips=np.zeros(G, dtype=np.int64),
                attempts=np.zeros((G, max(T - 1, 0)), dtype=np.int64), accepts=np.zeros((G, max(T - 1, 0)), dtype=np.int64))


def run(lpg, theta0, nsteps, betas, eps, method=0, L=3, swap_every=1, seed=0, chain_offset=0, t_start=0, st=None):
    """nsteps steps of qb_pt_run from absolute step t_start (st: a state from init_state / an earlier run, else a fresh
    one from theta0).  Returns (st, records) with records: lp [K, nsteps], acc [K, nsteps], mh_margin [K, nsteps],
    cold_z [nsteps, G, P] and swaps: one list of (g, i, accepted, margin) per round."""
    betas = np.asarray(betas, dtype=np.float64)
    eps = np.broadcast_to(np.asarray(eps, dtype=np.float64), betas.shape)
    st = init_state(lpg, theta0, betas) if st is None else st
    K = st['z'].shape[0]
    T = betas.size
    G = K // T
    rec = dict(lp=np.zeros((K, nsteps)), acc=np.zeros((K, nsteps), dtype=bool), mh_margin=np.zeros((K, nsteps)),
               cold_z=np.zeros((nsteps, G, st['z'].shape[1])), swaps=[])
    for s in range(nsteps):
        t = t_start + s
        for k in range(K):
            i = k // G
            z, lp, g, acc, _, m = step(lpg, betas[i], eps[i], method, L, st['z'][k], st['lp'][k], st['g'][k], seed,
                                       chain_offset + k, t)
            st['z'][k], st['lp'][k], st['g'][k] = z, lp, g
            if acc:
                st['naccept'][k] += 1
                if lp >= st['map_lp'][k]:
                    st['map_lp'][k], st['map_z'][k] = lp, z.copy()
            rec['lp'][k, s], rec['acc'][k, s], rec['mh_margin'][k, s] = lp, acc, m
        rec['cold_z'][s] = st['z'][:G]
        if (t + 1) % swap_every == 0:
            rec['swaps'].append(swap_round(st, betas, G, seed, chain_offset, (t + 1) // swap_every - 1))
    return st, rec
