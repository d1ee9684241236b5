"""CPU checks of parallel tempering: the numpy oracle (tests/pt_oracle.py) samples each tempered target of a correlated
2-D Gaussian correctly, its DEO rounds alternate parity, round trips are counted on a hand-made index sequence, the
ladder is built and validated, the ABI symbol is declared and exported, and every argument refusal of PT, ops.PtState
and qb_pt_run is decided before any device work."""
import ctypes as C
import os

import numpy as np
import pytest

import pt_oracle


def _gauss_2d():
    mu = np.array([0.5, -0.3])
    cov = np.array([[1.0, 0.8], [0.8, 1.0]])
    prec = np.linalg.inv(cov)
    return mu, cov, lambda th: (-0.5 * float((th - mu) @ prec @ (th - mu)), -(prec @ (th - mu)))


def _batch_se(x, nb=20):
    b = x[:len(x) // nb * nb].reshape(nb, -1).mean(1)
    return b.std(ddof=1) / np.sqrt(nb)


@pytest.mark.parametrize('method', [0, 1])
def test_oracle_slots_sample_their_tempered_gaussians(method):
    """flat prior: slot i targets N(mu, cov / beta_i); every slot's draws match its moments within 5 standard errors"""
    mu, cov, lpg = _gauss_2d()
    betas = np.array([1.0, 0.5, 0.25])
    eps = (0.35 if method == 0 else 0.6) / np.sqrt(betas)
    G, n, burn = 2, 2500, 200
    T = betas.size
    st = pt_oracle.init_state(lpg, np.array([[2.0, -1.0], [-1.0, 1.0]]), betas)
    traces = np.zeros((n, T * G, 2))
    t = 0
    for s in range(n):
        st, _ = pt_oracle.run(lpg, None, 1, betas, eps, method=method, L=3, swap_every=1, seed=11, t_start=t, st=st)
        t += 1
        traces[s] = st['z']
    assert st['accepts'].sum() > 0.2 * st['attempts'].sum()
    for i, b in enumerate(betas):
        x = traces[burn:, i * G:(i + 1) * G, :]                       # [n, G, 2]
        c = cov / b
        for f, ref in ((x[..., 0], mu[0]), (x[..., 1], mu[1]), ((x[..., 0] - mu[0]) ** 2, c[0, 0]),
                       ((x[..., 1] - mu[1]) ** 2, c[1, 1]), ((x[..., 0] - mu[0]) * (x[..., 1] - mu[1]), c[0, 1])):
            se = np.sqrt(np.mean([_batch_se(f[:, g]) ** 2 for g in range(G)]) / G)
            assert abs(f.mean() - ref) <= 5 * se, (i, f.mean(), ref, se)


def test_deo_rounds_alternate_parity():
    _, _, lpg = _gauss_2d()
    betas = np.array([1.0, 0.6, 0.3, 0.1, 0.05])
    _, rec = pt_oracle.run(lpg, np.zeros((3, 2)), 12, betas, 0.2, swap_every=3, seed=2)
    assert len(rec['swaps']) == 4
    for r, dec in enumerate(rec['swaps']):
        pairs = sorted(set(i for _, i, _, _ in dec))
        assert pairs == ([0, 2] if r % 2 == 0 else [1, 3])
        assert len(dec) == 3 * len(pairs)


def test_swap_rescales_lp_and_gradient():
    betas = np.array([1.0, 0.5])
    st = dict(z=np.array([[1.0, 2.0], [3.0, 4.0]]), lp=np.array([-10.0, -1.0]), g=np.array([[1.0, 1.0], [2.0, 2.0]]),
              replica=np.arange(2), last_end=np.array([1, -1]), round_trips=np.zeros(1, dtype=np.int64),
              attempts=np.zeros((1, 1), dtype=np.int64), accepts=np.zeros((1, 1), dtype=np.int64))
    # U_0 = -10, U_1 = -2: x = 0.5 * 8 = 4 > log u for every u, so the swap is accepted
    dec = pt_oracle.swap_round(st, betas, 1, seed=0, chain_offset=0, r=0)
    assert dec[0][2]
    np.testing.assert_array_equal(st['z'], [[3.0, 4.0], [1.0, 2.0]])
    np.testing.assert_array_equal(st['lp'], [-2.0, -5.0])
    np.testing.assert_array_equal(st['g'], [[4.0, 4.0], [0.5, 0.5]])
    np.testing.assert_array_equal(st['replica'], [1, 0])
    assert st['round_trips'][0] == 1 and list(st['last_end']) == [-1, 1]


def test_round_trips_on_a_hand_made_index_sequence():
    """T = 3, one group: replica 0 goes cold -> hot -> cold (one trip), replica 2 starts hot and reaches cold (one trip)"""
    G, T = 1, 3
    st = dict(replica=np.arange(3), last_end=np.array([1, 0, -1]), round_trips=np.zeros(1, dtype=np.int64))
    seq = [[0, 1, 2], [1, 0, 2], [1, 2, 0], [2, 1, 0], [2, 0, 1], [0, 2, 1]]
    trips = []
    for order in seq:
        st['replica'] = np.array(order)
        pt_oracle.round_trip_update(st, G, T, 0)
        trips.append(int(st['round_trips'][0]))
    # replica 2 reaches slot 0 at [2, 1, 0] (it started at the hot end); replica 0 reaches slot 0 again at [0, 2, 1]
    assert trips == [0, 0, 0, 1, 1, 2]


def test_ladder_construction_and_validation():
    from quinn_b200 import ops
    b = ops.pt_ladder(5, 0.0625)
    np.testing.assert_allclose(b, [1.0, 0.5, 0.25, 0.125, 0.0625], rtol=1e-15)
    assert b[0] == 1.0 and ops.pt_ladder(1, 0.5).tolist() == [1.0]
    b, e = ops.pt_check_ladder([1.0, 0.25], 0.1)
    np.testing.assert_allclose(e, [0.1, 0.2], rtol=1e-15)
    b, e = ops.pt_check_ladder([1.0, 0.25], [0.1, 0.3])
    assert e.tolist() == [0.1, 0.3]
    for betas, eps in (([0.9, 0.5], 0.1), ([1.0, 1.0], 0.1), ([1.0, 0.5, 0.6], 0.1), ([1.0, 0.0], 0.1),
                       ([1.0, -0.5], 0.1), ([1.0, 0.5], 0.0), ([1.0, 0.5], float('nan')), ([1.0, 0.5], [0.1, 0.1, 0.1]),
                       ([1.0, 0.5], [0.1, -0.1]), ([1.0, 0.5], float('inf'))):
        with pytest.raises(ValueError):
            ops.pt_check_ladder(betas, eps)
    for kw in (dict(n_temps=0, beta_min=0.1), dict(n_temps=3, beta_min=1.0), dict(n_temps=3, beta_min=0.0)):
        with pytest.raises(ValueError):
            ops.pt_ladder(**kw)


@pytest.mark.parametrize('kw', [dict(base='nuts'), dict(swap_every=0), dict(L=0), dict(betas=[0.5, 0.2]),
                                dict(betas=[1.0, 0.5, 0.7]), dict(n_temps=0), dict(beta_min=1.5), dict(epsilon=0.0),
                                dict(epsilon=[0.1, 0.1], n_temps=3)])
def test_sampler_constructor_refusals(kw):
    from quinn_b200.mcmc import PT
    with pytest.raises(ValueError):
        PT(**kw)


def test_sampler_refuses_generic_callables_and_replay():
    from quinn_b200.mcmc import PT
    m = PT()
    m.setLogPost(lambda th: -0.5 * float(np.sum(th ** 2)), lambda th: -th)
    with pytest.raises(ValueError, match='device log-posterior'):
        m.run(5, np.zeros(2), verbose=False)
    with pytest.raises(ValueError, match='replay'):
        m.run(5, np.zeros(2), replay=dict(incr=np.zeros((5, 2)), unif=np.zeros(5)), verbose=False)


@pytest.mark.parametrize('flag', ['distributed', 'data_sharded', 'replay'])
def test_fit_refuses_multi_process_and_replayed_pt(flag):
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_MCMC
    uq = NN_MCMC(MLP(1, 1, (3,), activ='tanh').double(), verbose=False)
    x = np.linspace(-1, 1, 8)[:, None]
    val = dict(incr=np.zeros((4, uq.pdim)), unif=np.zeros(4)) if flag == 'replay' else True
    with pytest.raises(ValueError, match="'pt'"):
        uq.fit(x, np.sin(x), sampler='pt', nmcmc=4, **{flag: val})


class _HostState:
    """what ops.PtState reads of a ChainState, on the host"""
    def __init__(self, K, P=2):
        import torch

        class _Prob:
            device = torch.device('cpu')
        self.K, self.P, self.prob = K, P, _Prob()
        self.theta = torch.zeros((K, P), dtype=torch.float64)


@pytest.mark.parametrize('kw', [dict(n_groups=0), dict(n_groups=4), dict(method='nuts'), dict(swap_every=0),
                                dict(L=0), dict(betas=[0.9, 0.5, 0.2]), dict(betas=[1.0, 0.5, 0.5]), dict(epsilon=-1.0)])
def test_pt_state_refusals(kw):
    from quinn_b200 import ops
    args = dict(n_groups=2, betas=[1.0, 0.5, 0.25], epsilon=0.1, L=3, method='hmc', swap_every=1)
    args.update(kw)
    with pytest.raises(ValueError):
        ops.PtState(_HostState(6), **args)


def test_pt_symbol_is_declared_and_exported():
    from quinn_b200 import _lib
    from golden_util import ROOT
    hdr = open(os.path.join(ROOT, 'include', 'quinn_b200.h')).read()
    lib = C.CDLL(_lib.lib_path()) if os.path.exists(_lib.lib_path()) else _lib.load()
    assert 'int qb_pt_run(' in hdr and 'qb_pt_run' in _lib.SYMBOLS and hasattr(lib, 'qb_pt_run')
    from quinn_b200.build import HEADERS
    assert 'qb_pt.cuh' in HEADERS
    from quinn_b200.mcmc import PT          # noqa: F401
    assert _lib.QB_ABI_VERSION == 204


def _call(mode=0, K=6, G=2, nsteps=3, t_start=0, swap_every=1, store_every=1, null_state=False, with_samples=True):
    """qb_pt_run with host dummies: every refusal below is decided before any device work"""
    from quinn_b200 import _lib
    lib = _lib.load()
    dummy = C.c_void_p(0x1000)
    net, data, lik = _lib.qb_net_t(), _lib.qb_data_t(), _lib.qb_lik_t()
    net.n_layers, net.in_dim, net.out_dim, net.n_params = 1, 1, 1, 2
    data.x = data.y = 0x1000
    data.n = 4
    ch = _lib.qb_chain_t(K, 0x1000, 0x1000, 0x1000, 0x1000, 0x1000)
    hm = _lib.qb_hmc_t(0, 3, 0.1, 0x1000, 0x1000, 0x1000, 0x1000)
    rng = _lib.qb_rng_t()
    rng.mode = mode
    rec = _lib.qb_record_t()
    rec.store_every = store_every
    if with_samples:
        rec.samples = 0x1000
    arr = None if null_state else dummy
    rc = lib.qb_pt_run(C.byref(net), _lib.QB_F64, C.byref(data), C.byref(lik), C.byref(ch), C.byref(hm), C.byref(rng),
                       C.byref(rec), t_start, nsteps, 1, G, arr, arr, swap_every, arr, arr, arr, arr, arr, None)
    return rc, lib.qb_last_error().decode()


@pytest.mark.parametrize('kw,match', [
    (dict(mode=1), 'replay'),
    (dict(null_state=True), 'NULL'),
    (dict(G=0), 'n_groups'),
    (dict(G=4), 'multiple of n_groups'),
    (dict(swap_every=0), 'swap_every'),
    (dict(swap_every=3, t_start=4), 't_start'),
    (dict(swap_every=4, store_every=6), 'divide one another'),
    (dict(swap_every=6, store_every=4), 'divide one another'),
])
def test_pt_run_refusals(kw, match):
    rc, msg = _call(**kw)
    assert rc != 0 and match in msg, msg


@pytest.mark.parametrize('kw', [dict(K=0), dict(nsteps=0)])
def test_pt_run_empty_launches_nothing(kw):
    assert _call(**kw)[0] == 0
