"""TEST INFRASTRUCTURE: the fp32 AMCMC chain arithmetic restated in numpy, and a per-step checker of device chains.

The fp32 chain kernels (k_amcmc_tc3 for the hot shape, k_amcmc<float, 2> and the CUDA-core k_amcmc<float>) draw their
proposals with the fp32 Box-Muller of qb_normal4(uint4, float (&)[4]) (quinn_b200/csrc/qb_device.cuh) on the special
function unit.  Its transcendental parts are approximations, so a draw is restated here as an interval: the 24-bit
uniforms and the angle exactly as the device forms them (np.float32), the logarithm, square root, sine and cosine in
float64, and an error bound from the documented accuracy of __logf, sqrt.approx.f32, __sinf and __cosf.  The Haario
moments and the proposal scales use correctly rounded fp32 operations and IEEE division on the device, so they are
emulated bit for bit.

check_amcmc_steps() then checks every step of a device chain given the device's OWN previous state, so a chain never
drifts away from its restatement and a decision tie at fp32 noise never ends a comparison.
"""
import math

import numpy as np

from oracle import philox

F32 = np.float32
_U24 = F32(5.9604644775390625e-8)                 # 2^-24
_ANG = F32(3.7450702829239286e-7)                 # 2 pi 2^-24
_PI = F32(3.14159265358979)
# documented accuracies (CUDA C Programming Guide, intrinsic functions; PTX ISA sqrt.approx.f32)
LOGF_ABS = 2.0 ** -21.41                          # __logf, x in [0.5, 2]: absolute error
LOGF_ULP = 3.0                                    # __logf elsewhere: ulp error
SQRT_REL = 2.0 ** -22                             # sqrt.approx.f32: relative error (documented ~2^-23, one bit of slack)
SINCOS_ABS = 2.0 ** -20.9                         # __sinf / __cosf on (-pi, pi): absolute error
EPS32 = 2.0 ** -24                                # unit round-off of an fp32 operation


def u24_f32(m):
    """u = ((float)m + 0.5f) * 2^-24 for the top 24 bits m of a Philox word, in fp32 as the device rounds it."""
    return (np.asarray(m, dtype=np.uint32).astype(F32) + F32(0.5)) * _U24


def _angle(m):
    """The angle (m + 0.5f) * 2 pi 2^-24 - pi: contracted into one FMA (one rounding) or computed with two roundings.
    Returns the FMA value and the largest distance to the two-rounding value."""
    s = np.asarray(m, dtype=np.uint32).astype(F32) + F32(0.5)
    a_fma = (s.astype(np.float64) * float(_ANG) - float(_PI)).astype(F32)     # exact in float64, then one rounding
    a_two = (s * _ANG) - _PI
    return a_fma.astype(np.float64), np.abs(a_fma.astype(np.float64) - a_two.astype(np.float64))


def _radius(m):
    """sqrt(-2 __logf(u)) as an interval: (mid, half-width)."""
    u = u24_f32(m).astype(np.float64)
    L = np.log(u)
    Lf = np.abs(L).astype(F32)
    eL = np.where((u >= 0.5) & (u <= 2.0), LOGF_ABS, LOGF_ULP * np.spacing(Lf).astype(np.float64))
    v = -2.0 * L
    mid = np.sqrt(v)
    lo = np.sqrt(np.maximum(v - 2.0 * eL, 0.0)) * (1.0 - SQRT_REL)
    hi = np.sqrt(v + 2.0 * eL) * (1.0 + SQRT_REL)
    return mid, np.maximum(hi - mid, mid - lo)


def normals_f32(seed, chain, step, stream, n, block_shift=0):
    """The first n fp32 normals of a stream as the device's qb_normal4(float) forms them: (z, err) in float64 with
    |z_device - z| <= err for any implementation within the documented accuracies.  Element i comes from Philox block
    i // 4 + block_shift, position i % 4 = (-r1 cos a1, -r1 sin a1, -r2 cos a2, -r2 sin a2).  block_shift != 0 only
    serves to model a wrong block index."""
    nb = (n + 3) // 4
    r = philox.rand4(seed, chain, step, stream, np.arange(nb) + block_shift)
    zs, es = [], []
    for wr, wa in ((r[0], r[1]), (r[2], r[3])):
        rad, erad = _radius(wr >> 8)
        a, da = _angle(wa >> 8)
        ec = SINCOS_ABS + da
        for f in (np.cos, np.sin):
            z = -rad * f(a)
            zs.append(z)
            es.append(erad * (1.0 + ec) + rad * ec + np.abs(z) * 2.0 * EPS32)
    z = np.stack([zs[0], zs[1], zs[2], zs[3]], axis=1).reshape(-1)[:n]
    e = np.stack([es[0], es[1], es[2], es[3]], axis=1).reshape(-1)[:n]
    return z, e


def amcmc_draws_f32(seed, chain, nsteps, P, t_start=0, step_shift=0, block_shift=0):
    """Draws an fp32 AMCMC chain consumes in Philox mode: z0[t] = 0.1f * (first normal of QB_STREAM_Z0), z[t, P] from
    QB_STREAM_INCR (with their error bounds) and the double uniform u[t].  step_shift / block_shift model a wrong step
    counter or block index."""
    z0, z0e, z, ze = [], [], [], []
    for t in range(t_start, t_start + nsteps):
        a, ea = normals_f32(seed, chain, t + step_shift, philox.STREAM_Z0, 1, block_shift)
        v = float(F32(0.1)) * a[0]
        z0.append(v)
        z0e.append(float(F32(0.1)) * ea[0] + abs(v) * EPS32)
        b, eb = normals_f32(seed, chain, t + step_shift, philox.STREAM_INCR, P, block_shift)
        z.append(b)
        ze.append(eb)
    u = np.array([philox.uniform(seed, chain, t) for t in range(t_start, t_start + nsteps)])
    return dict(z0=np.array(z0), z0_err=np.array(z0e), z=np.stack(z), z_err=np.stack(ze), u=u)


class AdaptF32:
    """Running moments and proposal scales of one fp32 chain (the per-element phase of k_amcmc_tc3 and qb_amcmc_pre):
    xm = (t * xm + cu) / (t + 1) and cov = rt * cov + st * d^2 with _rn products and sums and an IEEE quotient in fp32,
    rt and st formed in double and rounded, pscale = float(sqrt(0.09 |cu|)) at t = 0 and float(sqrt(fac (cov + eps)))
    at an adaptation step.  eps and adapt_shift exist to model faults."""

    def __init__(self, P, gamma, t0, tadapt, adapt, eps=1e-8, adapt_shift=0):
        self.P, self.t0, self.tadapt, self.adapt = P, t0, tadapt, adapt
        self.fac = gamma * 2.4 * 2.4 / P                     # same association as the kernel
        self.track = adapt == 'diag'
        self.eps, self.adapt_shift = eps, adapt_shift
        self.xm = self.cov = self.pscale = None
        self.kind = 0

    def load(self, xm, cov, pscale, kind):
        self.xm = None if xm is None else np.asarray(xm, F32).copy()
        self.cov = None if cov is None else np.asarray(cov, F32).copy()
        self.pscale, self.kind = np.asarray(pscale, F32).copy(), int(kind)

    def step(self, t, cu):
        """Advance to step t with current point cu (fp32); returns (kind, pscale) of the step's proposal."""
        cu = np.asarray(cu, F32)
        first = t == 0
        ta = t - self.adapt_shift
        adapt_now = not first and self.adapt != 'none' and t > self.t0 and ta % self.tadapt == 0
        if first:
            self.kind = 0
        elif adapt_now:
            self.kind = 1
        if self.track:
            if first:
                self.xm, self.cov = cu.copy(), np.zeros(self.P, F32)
            else:
                rt, st = F32((t - 1.0) / t), F32((t + 1.0) / (t * t))
                m = (F32(t) * self.xm + cu) / F32(t + 1.0)
                d = cu - m
                self.cov = rt * self.cov + st * (d * d)
                self.xm = m
        if first:
            self.pscale = np.sqrt(0.09 * np.abs(cu.astype(np.float64))).astype(F32)
        elif adapt_now:
            cv = self.cov.astype(np.float64) if self.cov is not None else np.zeros(self.P)
            self.pscale = np.sqrt(self.fac * (cv + self.eps)).astype(F32)
        return self.kind, self.pscale


def proposal(cu, kind, ps, draws, s):
    """Restated Philox proposal of step s: cu + (z0 + ps z) (kind 0) or cu + ps z (kind 1), as (mid, bound); the bound
    is the draws' error through ps plus two fp32 roundings."""
    cu = np.asarray(cu, np.float64)
    ps = np.asarray(ps, np.float64)
    z0, z0e = (draws['z0'][s], draws['z0_err'][s]) if kind == 0 else (0.0, 0.0)
    inner = z0 + ps * draws['z'][s]
    mid = cu + inner
    ulp = lambda v: np.spacing(np.abs(v).astype(F32)).astype(np.float64)          # noqa: E731
    return mid, ps * draws['z_err'][s] + z0e + ulp(inner) + ulp(mid)


def simulate_amcmc_f32(logpost_fn, theta0, draws, nsteps, gamma, t0, tadapt, adapt, fault=None, fault_step=None):
    """A numpy model of an fp32 chain kernel, for testing the checker: returns the records a device run with
    store_every=1 would give.  fault names a deliberate bug: 'flip' (one decision inverted), 'le' (u <= alpha),
    'no_eps' (scale without the 1e-8), 'adapt_shift' (adaptation one step late), 'map_gt' (MAP kept on > instead of >=).
    Faults in the draws (step or block index) are modelled by the draws passed in."""
    th = np.asarray(theta0, F32).copy()
    P = th.size
    ad = AdaptF32(P, gamma, t0, tadapt, adapt, eps=0.0 if fault == 'no_eps' else 1e-8,
                  adapt_shift=1 if fault == 'adapt_shift' else 0)
    lp = logpost_fn(th.astype(np.float64))
    out = dict(logpost0=lp, samples=[], logpost=[], alpha=[], accepted=[])
    map_lp, map_th, na = lp, th.copy(), 0
    for s in range(nsteps):
        kind, ps = ad.step(s, th)
        z0 = F32(draws['z0'][s]) if kind == 0 else F32(0.0)
        prop = th + (z0 + ps * draws['z'][s].astype(F32))
        lpp = logpost_fn(prop.astype(np.float64))
        with np.errstate(over='ignore', invalid='ignore'):
            mh = math.exp(lpp - lp) if np.isfinite(lpp - lp) else float('nan')
        u = draws['u'][s]
        acc = (u <= mh) if fault == 'le' else (u < mh)
        if fault == 'flip' and s == fault_step:
            acc = not acc
        if acc:
            th, lp, na = prop, lpp, na + 1
            if (lp > map_lp) if fault == 'map_gt' else (lp >= map_lp):
                map_lp, map_th = lp, th.copy()
        out['samples'].append(th.copy())
        out['logpost'].append(lp)
        out['alpha'].append(mh)
        out['accepted'].append(acc)
    out = {k: np.array(v) if isinstance(v, list) else v for k, v in out.items()}
    out.update(lp=lp, theta=th, map_lp=map_lp, map_theta=map_th, naccept=na, xm=ad.xm, cov=ad.cov, pscale=ad.pscale,
               prop_kind=ad.kind)
    return out


class CheckFailed(AssertionError):
    pass


def _need(cond, what, s):
    if not cond:
        raise CheckFailed(f'step {s}: {what}')


def check_amcmc_steps(rec, theta0, draws, logpost_grad, gamma, t0, tadapt, adapt, t_start=0, lp_rtol=1e-5,
                      start=None, lp_tol=None):
    """Check one chain's device records step by step against the restatement, each step given the device's own
    previous state.

    rec: numpy records of one chain run with store_every=1: samples[S, P], logpost[S], alpha[S], accepted[S],
      logpost0 (the log-posterior at theta0) and the final state: lp, theta, map_lp, map_theta, naccept, xm, cov,
      pscale, prop_kind (xm / cov None when not tracked).
    draws: amcmc_draws_f32(...) of the chain (Philox mode) or dict(xi=[S, P] fp32, u=[S]) (replay mode).
    logpost_grad: theta (float64) -> (lp, grad) of the fp64 oracle.
    lp_tol: theta -> absolute tolerance of a device log-posterior there; lp_rtol * |lp| by default.
    start: state in force before the first step when the run continues a chain: dict(map_lp, map_theta, naccept, xm,
      cov, pscale, prop_kind); None for a chain that starts at t_start = 0.
    Returns the number of steps checked and the largest deviation / tolerance of each tolerance-based check."""
    S, P = rec['samples'].shape
    replay = 'xi' in draws
    ad = AdaptF32(P, gamma, t0, tadapt, adapt)
    cur = np.asarray(theta0, F32)
    if lp_tol is None:
        lp_tol = lambda th: lp_rtol * max(abs(logpost_grad(th)[0]), 1.0)          # noqa: E731
    lp0_ref, _ = logpost_grad(cur.astype(np.float64))
    lp_cur = float(rec['logpost0'])
    margins = dict(lp=abs(lp_cur - lp0_ref) / lp_tol(cur.astype(np.float64)), proposal=0.0, log_alpha=0.0)
    _need(margins['lp'] <= 1.0, f'logpost0 {lp_cur} vs oracle {lp0_ref}', -1)
    if start is None:
        map_lp, map_th, na = lp_cur, cur.copy(), 0
    else:
        map_lp, map_th, na = start['map_lp'], np.asarray(start['map_theta'], F32), int(start['naccept'])
        ad.load(start['xm'], start['cov'], start['pscale'], start['prop_kind'])
    for s in range(S):
        t = t_start + s
        kind, ps = ad.step(t, cur)
        if replay:
            pmid = (cur + np.asarray(draws['xi'][s], F32)).astype(np.float64)     # qb_add: exact in fp32
            pbnd = np.zeros(P)
        else:
            pmid, pbnd = proposal(cur, kind, ps, draws, s)
        alpha, acc, u = float(rec['alpha'][s]), bool(rec['accepted'][s]), float(draws['u'][s])
        _need(acc == (u < alpha), f'decision {acc} but u = {u!r}, alpha = {alpha!r}', s)
        lpp, g = logpost_grad(pmid)
        if np.isfinite(lpp):
            _need(not math.isnan(alpha), f'alpha is NaN where the oracle gives lp = {lpp}', s)
        if acc:
            smp = rec['samples'][s].astype(np.float64)
            dev = np.abs(smp - pmid)
            _need(np.all(dev <= pbnd), f'proposal off by {dev.max()} (bound {pbnd[np.argmax(dev - pbnd)]}) at '
                                       f'parameter {int(np.argmax(dev - pbnd))}', s)
            if not replay:
                margins['proposal'] = max(margins['proposal'], float(np.max(dev / np.maximum(pbnd, 1e-300))))
            lp_ref, _ = logpost_grad(smp)
            dl = abs(rec['logpost'][s] - lp_ref) / lp_tol(smp)
            margins['lp'] = max(margins['lp'], dl)
            _need(dl <= 1.0, f'logpost {rec["logpost"][s]} vs oracle {lp_ref}', s)
            cur = rec['samples'][s].astype(F32)
            lp_cur_new = float(rec['logpost'][s])
            na += 1
            if lp_cur_new >= map_lp:
                map_lp, map_th = lp_cur_new, cur.copy()
        else:
            _need(np.array_equal(rec['samples'][s].view(np.uint32), cur.view(np.uint32)), 'rejected step moved', s)
            _need(rec['logpost'][s] == lp_cur, 'rejected step changed the log-posterior', s)
            lp_cur_new = lp_cur
        if np.isfinite(alpha) and alpha > 0.0 and np.isfinite(lpp):
            tol = lp_tol(pmid) + float(np.sum(np.abs(g) * pbnd))
            dla = abs(math.log(alpha) - (lpp - lp_cur))
            margins['log_alpha'] = max(margins['log_alpha'], dla / tol)
            _need(dla <= tol, f'log alpha {math.log(alpha)} vs oracle {lpp - lp_cur} (tol {tol})', s)
        lp_cur = lp_cur_new
    _need(rec['lp'] == lp_cur and np.array_equal(np.asarray(rec['theta'], F32), cur), 'final state', S)
    _need(rec['naccept'] == na, f'naccept {rec["naccept"]} vs {na}', S)
    _need(rec['map_lp'] == map_lp, f'map_lp {rec["map_lp"]} vs {map_lp}', S)
    _need(np.array_equal(np.asarray(rec['map_theta'], F32), map_th), 'map_theta', S)
    _need(int(rec['prop_kind']) == ad.kind, f'prop_kind {rec["prop_kind"]} vs {ad.kind}', S)
    _need(np.array_equal(np.asarray(rec['pscale'], F32), ad.pscale), 'pscale', S)
    if ad.track:
        _need(np.array_equal(np.asarray(rec['xm'], F32), ad.xm), 'xm', S)
        _need(np.array_equal(np.asarray(rec['cov'], F32), ad.cov), 'cov', S)
    return dict(steps=S, **margins)
