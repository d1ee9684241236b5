"""TEST INFRASTRUCTURE (oracle): numpy restatement of the NUTS transition of quinn_b200/csrc/qb_nuts.cuh -- the
iterative multinomial tree with the generalised no-U-turn checks against stored checkpoints, and the dual averaging of
the step size -- on the Philox draws of oracle/philox.py, so that a device chain can be replayed transition by
transition.  Besides the states it reports each transition's smallest decision margin: how far each U-turn dot product and
each selection uniform was from flipping its decision, relative to the size of the compared quantities."""
import math

import numpy as np

from oracle import philox

STREAM_NUTS = 5            # QB_STREAM_NUTS of quinn_b200/csrc/qb_device.cuh
LEAF0 = 16                 # QB_NUTS_LEAF0: index of leapfrog n's selection uniform is 16 + n


def _logaddexp(a, b):
    m = max(a, b)
    if m == -math.inf:
        return -math.inf
    return m + math.log1p(math.exp(-abs(a - b)))


def _turning(ra, rb, rs, margin):
    d = rs - (ra + rb) * 0.5
    s1, s2 = float(np.dot(ra, d)), float(np.dot(rb, d))
    scale = float(np.dot(np.abs(ra) + np.abs(rb), np.abs(d))) + 1e-300
    margin[0] = min(margin[0], abs(s1) / scale, abs(s2) / scale)
    return s1 <= 0.0 or s2 <= 0.0


def _uniform_choice(u, p, margin):
    if p > 0.0:
        margin[0] = min(margin[0], abs(u - p) / p)
    return u < p


def transition(lpg, z0, lp0, g0, eps, max_depth, seed, chain, t):
    """One NUTS transition from (z0, lp0, g0) with step size eps.  lpg(theta) -> (lp, grad).
    Returns dict(z, lp, g, moved, stat, depth, n_leapfrog, diverging, margin)."""
    P = z0.size
    r0 = philox.normals(seed, chain, t, philox.STREAM_INCR, P)
    H0 = -lp0 + float(np.dot(r0, r0)) / 2.0
    ends = {False: [z0.copy(), r0.copy(), g0.copy()], True: [z0.copy(), r0.copy(), g0.copy()]}
    rsum = r0.copy()
    ck_r, ck_s = np.zeros((max_depth, P)), np.zeros((max_depth, P))
    z, lp, g = z0.copy(), lp0, g0.copy()
    w_tree, sum_acc, n_leap, depth, moved, div = 0.0, 0.0, 0, 0, False, False
    margin = [math.inf]
    while True:
        rd = philox.rand4(seed, chain, t, STREAM_NUTS, np.array([depth]))
        fwd, u_bias = (int(rd[0][0]) & 1) == 1, float(philox.u01(rd[1])[0])
        e = eps if fwd else -eps
        w_sub, zs, gs, lps, turn = 0.0, None, None, None, False
        for leaf in range(2 ** depth):
            ze, re, ge = ends[fwd]
            re = re + (e * 0.5) * ge
            ze = ze + e * re
            lpe, ge = lpg(ze)
            re = re + (e * 0.5) * ge
            ends[fwd] = [ze, re, ge]
            rsum = rsum + re
            dH = (-lpe + float(np.dot(re, re)) / 2.0) - H0
            if not np.isfinite(lpe) or np.isnan(dH):
                dH = math.inf
            wl = -dH
            div = dH > 1000.0
            sum_acc += math.exp(-dH) if dH > 0.0 else 1.0
            n_leap += 1
            take = True
            if leaf == 0:
                w_sub = wl
            else:
                wn = _logaddexp(w_sub, wl)
                u = float(philox.u01(philox.rand4(seed, chain, t, STREAM_NUTS, np.array([LEAF0 + n_leap - 1]))[0])[0])
                take = wl > -math.inf and _uniform_choice(u, math.exp(wl - wn), margin)
                w_sub = wn
            if take:
                zs, gs, lps = ze.copy(), ge.copy(), lpe
            idx_max = bin(leaf >> 1).count('1')
            trailing = 0
            while (leaf >> trailing) & 1:
                trailing += 1
            idx_min = idx_max - trailing + 1
            if leaf % 2 == 0:
                ck_r[idx_max], ck_s[idx_max] = re, rsum
            for ci in range(idx_max, idx_min - 1, -1):
                if div:
                    break
                if _turning(ck_r[ci], re, rsum - ck_s[ci] + ck_r[ci], margin):
                    turn = True
                    break
            if div or turn:
                break
        if not div and not turn:
            p = 1.0 if w_sub >= w_tree else math.exp(w_sub - w_tree)
            if _uniform_choice(u_bias, p, margin):
                z, g, lp, moved = zs, gs, lps, True
        w_tree = _logaddexp(w_tree, w_sub)
        depth += 1
        if not div and not turn:
            turn = _turning(ends[False][1], ends[True][1], rsum, margin)
        if div or turn or depth >= max_depth:
            break
    return dict(z=z, lp=lp, g=g, moved=moved, stat=sum_acc / n_leap, depth=depth, n_leapfrog=n_leap, diverging=div,
                margin=margin[0])


def dual_average(state, t, stat, eps0, target):
    """Stan's dual averaging after transition t (gamma 0.05, t0 10, kappa 0.75, mu = log(10 eps0)); state = dict(log_eps,
    log_eps_bar, h_bar), updated in place."""
    m = float(t + 1)
    eta = 1.0 / (m + 10.0)
    state['h_bar'] = (1.0 - eta) * state['h_bar'] + eta * (target - stat)
    log_eps = math.log(10.0 * eps0) - math.sqrt(m) / 0.05 * state['h_bar']
    xe = m ** -0.75
    state['log_eps'] = log_eps
    state['log_eps_bar'] = xe * log_eps + (1.0 - xe) * state['log_eps_bar']


def run_chain(lpg, theta0, nsteps, seed, chain, eps0=0.05, max_depth=10, n_adapt=1000, target_accept=0.8):
    """nsteps NUTS transitions of one chain, as qb_nuts_run with init_lp from step 0.  Returns the result dict of the
    device sampler for this chain (chain (nsteps+1, P), logpost (nsteps+1,), alphas, accepted, tree_depth, n_leapfrog,
    diverging, step_size, maxpost, mapparams) plus the per-transition decision margins."""
    z = np.array(theta0, dtype=np.float64)
    lp, g = lpg(z)
    da = dict(log_eps=math.log(eps0), log_eps_bar=math.log(eps0), h_bar=0.0)
    out = {k: [] for k in ('chain', 'logpost', 'alphas', 'accepted', 'tree_depth', 'n_leapfrog', 'diverging', 'step_size',
                           'margin')}
    out['chain'].append(z.copy())
    out['logpost'].append(lp)
    out['alphas'].append(0.0)
    map_lp, map_th = lp, z.copy()
    for t in range(nsteps):
        eps = math.exp(da['log_eps_bar'] if (n_adapt > 0 and t >= n_adapt) else da['log_eps'])
        tr = transition(lpg, z, lp, g, eps, max_depth, seed, chain, t)
        if tr['moved']:
            z, lp, g = tr['z'], tr['lp'], tr['g']
            if lp >= map_lp:
                map_lp, map_th = lp, z.copy()
        if t < n_adapt:
            dual_average(da, t, tr['stat'], eps0, target_accept)
        out['chain'].append(z.copy())
        out['logpost'].append(lp)
        out['alphas'].append(tr['stat'])
        out['accepted'].append(tr['moved'])
        out['tree_depth'].append(tr['depth'])
        out['n_leapfrog'].append(tr['n_leapfrog'])
        out['diverging'].append(tr['diverging'])
        out['step_size'].append(eps)
        out['margin'].append(tr['margin'])
    res = {k: np.array(v) for k, v in out.items()}
    res.update(maxpost=map_lp, mapparams=map_th, da=da)
    return res
