"""tests/chain_replay.py without a GPU: the fp32 draws against the fp64 Philox restatement, the fp32 uniforms at the
extreme words, the fp32 moment recursion against the oracle's, and the per-step checker against a numpy model of the
chain kernel, both as it is (the checker passes) and with each of a set of deliberate bugs (the checker fails).  The
second half is the evidence that the GPU replay tests (test_gpu_amcmc_tc3.py) would notice such a bug in a kernel."""
import numpy as np
import pytest

import chain_replay as cr
from oracle import philox
from oracle import quinn_oracle as qo
from test_gpu_tensorcore import make_net

F32 = np.float32


def test_normals_f32_track_the_fp64_stream():
    """Same Philox blocks, same layout and sign as the fp64 normals: they differ only by the 24- versus 32-bit
    quantisation of the uniforms and by the fp32 error bound."""
    n = 4 * 3000
    for seed, chain, step in [(2026, 0, 0), (7, 2 ** 33 + 5, 17), (2 ** 40 + 1, 3, 2 ** 32 + 9)]:
        z, e = cr.normals_f32(seed, chain, step, philox.STREAM_INCR, n)
        z64 = philox.normals(seed, chain, step, philox.STREAM_INCR, n)
        r = philox.rand4(seed, chain, step, philox.STREAM_INCR, np.arange(n // 4))
        rad24 = [cr._radius(w >> 8)[0] for w in (r[0], r[2])]
        rad32 = [np.sqrt(-2.0 * np.log(philox.u01(w))) for w in (r[0], r[2])]
        q = np.repeat(np.stack([np.abs(a - b) for a, b in zip(rad24, rad32)], 1), 2, axis=1).reshape(-1)
        q += np.repeat(np.stack(rad32, 1), 2, axis=1).reshape(-1) * 2 * np.pi * 2.0 ** -23
        assert np.all(np.abs(z - z64) <= e + q)
        assert np.all(e < 2e-5 * np.maximum(1.0, np.abs(z)) + 1e-3)     # the bound is tight except right at u -> 1
        assert abs(z.mean()) < 0.05 and abs(z.std() - 1.0) < 0.05


@pytest.mark.parametrize('m,u', [(0, 2.0 ** -25), (2 ** 23 - 1, 0.5 - 2.0 ** -25), (2 ** 23, 0.5),
                                 (2 ** 24 - 3, 1.0 - 2.0 ** -23), (2 ** 24 - 2, 1.0 - 2.0 ** -23), (2 ** 24 - 1, 1.0)])
def test_u1_emulation_at_extreme_words(m, u):
    """((float)m + 0.5f) * 2^-24 rounds to even: m = 2^23 loses its half, the top three words give 1 - 2^-23 or 1."""
    v = cr.u24_f32(np.array([m]))[0]
    assert v.dtype == F32 and float(v) == u
    mid, err = cr._radius(np.array([m]))
    if m >= 2 ** 24 - 3:
        assert mid[0] - err[0] <= 0.0                  # within __logf's error the radius may be 0: the interval says so
    else:
        assert err[0] < 1e-6 * max(1.0, mid[0])


def test_moment_recursion_matches_the_oracle():
    rs = np.random.RandomState(1)
    P, steps, gamma, t0, tadapt = 7, 60, 0.3, 5, 10
    chain = (rs.randn(steps, P) * 0.1 + 1.0).astype(F32)
    ad = cr.AdaptF32(P, gamma, t0, tadapt, 'diag')
    Xm = cov = None
    fac = gamma * 2.4 ** 2 / P
    for t in range(steps):
        kind, ps = ad.step(t, chain[t])
        Xm, cov = qo.amcmc_moments_update(Xm, cov, chain[t].astype(np.float64), t)
        np.testing.assert_allclose(ad.xm, Xm, rtol=1e-6)
        np.testing.assert_allclose(ad.cov, np.diag(cov), rtol=1e-4, atol=1e-9)
        if t == 0:
            np.testing.assert_allclose(ps, np.sqrt(0.09 * np.abs(chain[0])), rtol=1e-7)
        elif t > t0 and t % tadapt == 0:
            assert kind == 1
            np.testing.assert_allclose(ps, np.sqrt(fac * (np.diag(cov) + 1e-8)), rtol=1e-4)
        assert kind == (1 if t > t0 and t >= tadapt else 0)


# ---- the checker against a numpy model of the kernel ---------------------------------------------------------------
_LAYERS, _P = make_net([2, 4, 4, 1], ['tanh', 'tanh', 'identity'])
_RS = np.random.RandomState(5)
_X = _RS.rand(20, 2) * 2 - 1
_Y = np.sin(_X.sum(1, keepdims=True))
_TH0 = (0.2 * _RS.randn(_P)).astype(F32)
_STEPS, _GAMMA, _T0, _TADAPT = 40, 0.5, 5, 10
_SEED, _CHAIN = 2026, 11


def _lpg(th):
    return qo.logpost_grad(_LAYERS, th, _X, _Y, 0.5)


def _lp(th):
    return _lpg(th)[0]


def _flat(th):
    return -3.0, np.zeros_like(th)


def _run(fault=None, draws_fault=None, lpg=_lpg, tie=None):
    draws = cr.amcmc_draws_f32(_SEED, _CHAIN, _STEPS, _P)
    used = draws
    if draws_fault is not None:
        used = cr.amcmc_draws_f32(_SEED, _CHAIN, _STEPS, _P, **draws_fault)
    if tie is not None:
        # a uniform that equals the ratio of step `tie` exactly (found from a clean run of the same chain)
        clean = cr.simulate_amcmc_f32(lambda th: lpg(th)[0], _TH0, draws, _STEPS, _GAMMA, _T0, _TADAPT, 'diag')
        draws = dict(draws, u=draws['u'].copy())
        draws['u'][tie] = clean['alpha'][tie]
        used = draws
    rec = cr.simulate_amcmc_f32(lambda th: lpg(th)[0], _TH0, used, _STEPS, _GAMMA, _T0, _TADAPT, 'diag', fault=fault,
                                fault_step=17)
    return rec, draws


def _check(rec, draws, lpg=_lpg):
    return cr.check_amcmc_steps(rec, _TH0, draws, lpg, _GAMMA, _T0, _TADAPT, 'diag')


def test_checker_passes_the_model_chain():
    rec, draws = _run()
    acc = rec['accepted']
    for part in (acc[:_TADAPT], acc[_TADAPT:]):             # both proposal kinds are accepted and rejected
        assert part.any() and not part.all()
    m = _check(rec, draws)
    assert m['steps'] == _STEPS and m['proposal'] <= 1.0 and m['log_alpha'] <= 1.0 and m['lp'] <= 1.0


def test_checker_passes_a_tie_decided_by_strict_less_than():
    rec, draws = _run(tie=23)
    assert not rec['accepted'][23]
    _check(rec, draws)


FAULTS = {
    'one flipped decision': dict(fault='flip'),
    '<= in place of <': dict(fault='le', tie=23),
    "proposal from step t+1's draws": dict(draws_fault=dict(step_shift=1)),
    "proposal from step t-1's draws": dict(draws_fault=dict(step_shift=-1)),
    'block index off by one': dict(draws_fault=dict(block_shift=1)),
    'scale without the +1e-8': dict(fault='no_eps'),
    'scale from the wrong adaptation step': dict(fault='adapt_shift'),
}


@pytest.mark.parametrize('name', list(FAULTS))
def test_checker_fails_an_injected_fault(name):
    rec, draws = _run(**FAULTS[name])
    with pytest.raises(cr.CheckFailed):
        _check(rec, draws)


def test_checker_fails_a_map_update_on_strictly_greater():
    """On a flat target every accepted step ties the MAP: >= moves it to the newest state, > never moves it."""
    draws = cr.amcmc_draws_f32(_SEED, _CHAIN, _STEPS, _P)
    rec = cr.simulate_amcmc_f32(lambda th: -3.0, _TH0, draws, _STEPS, _GAMMA, _T0, _TADAPT, 'diag')
    assert rec['accepted'].all()
    _check(rec, draws, _flat)
    bad = cr.simulate_amcmc_f32(lambda th: -3.0, _TH0, draws, _STEPS, _GAMMA, _T0, _TADAPT, 'diag', fault='map_gt')
    with pytest.raises(cr.CheckFailed, match='map_theta'):
        _check(bad, draws, _flat)
