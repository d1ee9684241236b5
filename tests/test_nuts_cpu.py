"""CPU checks of the NUTS pieces: the numpy oracle (tests/nuts_oracle.py) samples a correlated 2-D Gaussian correctly and
respects the depth cap, the ABI symbol is declared and exported, and arguments that need no device are refused."""
import ctypes as C
import os

import numpy as np
import pytest

import nuts_oracle


def _gauss_2d():
    cov = np.array([[1.0, 0.8], [0.8, 1.0]])
    prec = np.linalg.inv(cov)
    return cov, lambda th: (-0.5 * float(th @ prec @ th), -(prec @ th))


def _batch_se(x, nb=20):
    """standard error of the mean of a correlated series by batch means"""
    b = x[:len(x) // nb * nb].reshape(nb, -1).mean(1)
    return b.std(ddof=1) / np.sqrt(nb)


def test_oracle_samples_a_correlated_gaussian():
    cov, lpg = _gauss_2d()
    draws = []
    for ch in range(4):
        res = nuts_oracle.run_chain(lpg, np.array([2.0, -1.0]), 900, seed=5, chain=ch, eps0=0.5, max_depth=6,
                                    n_adapt=150, target_accept=0.8)
        assert not res['diverging'][150:].any()
        draws.append(res['chain'][151:])
        assert abs(res['alphas'][151:].mean() - 0.8) < 0.15          # short warm-up: eps_bar sits below the target's eps
    x = np.concatenate(draws)
    for f, ref in ((x[:, 0], 0.0), (x[:, 1], 0.0), (x[:, 0] ** 2, cov[0, 0]), (x[:, 1] ** 2, cov[1, 1]),
                   (x[:, 0] * x[:, 1], cov[0, 1])):
        se = np.sqrt(np.mean([_batch_se(f.reshape(4, -1)[c]) ** 2 for c in range(4)]) / 4)
        assert abs(f.mean() - ref) <= 5 * se, (f.mean(), ref, se)


def test_oracle_depth_cap():
    """a tiny step size never turns within the cap: every transition runs the full 2^max_depth - 1 leapfrogs"""
    _, lpg = _gauss_2d()
    res = nuts_oracle.run_chain(lpg, np.array([0.3, 0.1]), 12, seed=1, chain=0, eps0=1e-3, max_depth=3, n_adapt=0)
    assert np.all(res['n_leapfrog'] <= 2 ** 3 - 1)
    assert np.all(res['tree_depth'] == 3) and np.all(res['n_leapfrog'] == 7)
    np.testing.assert_allclose(res['step_size'], 1e-3, rtol=1e-15)


def test_oracle_dual_averaging_moves_towards_the_target():
    """a step size far too large gives a low acceptance statistic, so the adaptation shrinks it"""
    _, lpg = _gauss_2d()
    res = nuts_oracle.run_chain(lpg, np.array([0.3, 0.1]), 60, seed=2, chain=0, eps0=5.0, max_depth=5, n_adapt=60)
    assert res['step_size'][-1] < 1.0 < res['step_size'][0]


def test_nuts_symbol_is_declared_and_exported():
    from quinn_b200 import _lib
    from golden_util import ROOT
    hdr = open(os.path.join(ROOT, 'include', 'quinn_b200.h')).read()
    lib = C.CDLL(_lib.lib_path()) if os.path.exists(_lib.lib_path()) else _lib.load()
    assert 'int qb_nuts_run(' in hdr and 'qb_nuts_run' in _lib.SYMBOLS and hasattr(lib, 'qb_nuts_run')
    from quinn_b200.mcmc import NUTS          # noqa: F401
    assert _lib.QB_ABI_VERSION == 204


def _call(mode=0, K=2, nsteps=3, eps=0.1, depth=5, target=0.8, null_state=False, with_rec=True, nrec=False):
    """qb_nuts_run with host dummies: every refusal below is decided before any device work"""
    from quinn_b200 import _lib
    lib = _lib.load()
    dummy = C.c_void_p(0x1000)
    net, data, lik = _lib.qb_net_t(), _lib.qb_data_t(), _lib.qb_lik_t()
    net.n_layers, net.in_dim, net.out_dim, net.n_params = 1, 1, 1, 2
    data.x = data.y = 0x1000
    data.n = 4
    ch = _lib.qb_chain_t(K, 0x1000, 0x1000, 0x1000, 0x1000, 0x1000)
    rng = _lib.qb_rng_t()
    rng.mode = mode
    rec = _lib.qb_record_t()
    arr = None if null_state else dummy
    rd = dummy if nrec else None
    rc = lib.qb_nuts_run(C.byref(net), _lib.QB_F64, C.byref(data), C.byref(lik), C.byref(ch), C.byref(rng),
                         C.byref(rec) if with_rec else None, 0, nsteps, 1, eps, depth, 10, target, arr, arr, arr, arr, arr,
                         rd, rd, rd, rd, None)
    return rc, lib.qb_last_error().decode()


@pytest.mark.parametrize('kw,match', [
    (dict(mode=1), 'replay'),
    (dict(null_state=True), 'NULL'),
    (dict(depth=0), 'max_depth'),
    (dict(depth=13), 'max_depth'),
    (dict(target=0.0), 'target_accept'),
    (dict(target=1.0), 'target_accept'),
    (dict(eps=0.0), 'epsilon'),
    (dict(eps=-0.1), 'epsilon'),
    (dict(eps=float('inf')), 'epsilon'),
    (dict(with_rec=False, nrec=True), 'records need rec'),
])
def test_nuts_run_refusals(kw, match):
    rc, msg = _call(**kw)
    assert rc != 0 and match in msg, msg


@pytest.mark.parametrize('kw', [dict(K=0), dict(nsteps=0)])
def test_nuts_run_empty_launches_nothing(kw):
    assert _call(**kw)[0] == 0


@pytest.mark.parametrize('kw', [dict(max_depth=0), dict(max_depth=13), dict(target_accept=1.0), dict(target_accept=0.0),
                                dict(epsilon=0.0), dict(n_adapt=-1)])
def test_sampler_constructor_refusals(kw):
    from quinn_b200.mcmc import NUTS
    with pytest.raises(ValueError):
        NUTS(**kw)


def test_sampler_refuses_generic_callables_and_replay():
    from quinn_b200.mcmc import NUTS
    m = NUTS()
    m.setLogPost(lambda th: -0.5 * float(np.sum(th ** 2)), lambda th: -th)
    with pytest.raises(ValueError, match='device log-posterior'):
        m.run(5, np.zeros(2), verbose=False)
    with pytest.raises(ValueError, match='replay'):
        m.run(5, np.zeros(2), replay=dict(incr=np.zeros((5, 2)), unif=np.zeros(5)), verbose=False)


@pytest.mark.parametrize('flag', ['distributed', 'data_sharded'])
def test_fit_refuses_multi_process_nuts(flag):
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_MCMC
    uq = NN_MCMC(MLP(1, 1, (3,), activ='tanh').double(), verbose=False)
    x = np.linspace(-1, 1, 8)[:, None]
    with pytest.raises(ValueError, match='nuts'):
        uq.fit(x, np.sin(x), sampler='nuts', nmcmc=4, **{flag: True})
