"""NUTS on the device (qb_nuts_run, quinn_b200/csrc/qb_nuts.cuh) against the numpy oracle (tests/nuts_oracle.py) on every
gradient path, its determinism, an exactly Gaussian posterior, divergences, the solver and the refusals."""
import numpy as np
import pytest
import torch

import nuts_oracle
from golden_util import netdesc_from_layers
from oracle import quinn_oracle as qo

pytestmark = pytest.mark.gpu


def _problem(layers, P, N, dtype, seed, in_dim, sigma=0.1):
    from quinn_b200 import ops
    rs = np.random.RandomState(seed)
    x = rs.rand(N, in_dim) * 2 - 1
    y = np.sin(2 * x.sum(1, keepdims=True)) + 0.1 * rs.randn(N, 1)
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, sigma, dtype=dtype, device='cuda')
    return prob, x, y, rs


def _run(prob, th0, nsteps, seed, eps0, max_depth, n_adapt, target=0.8, splits=(None,)):
    """NUTS on the device over the segments `splits` (None: one launch); returns numpy records [K, nsteps(+1)]"""
    from quinn_b200 import ops
    st = ops.ChainState(prob, th0)
    ns = ops.NutsState(st, epsilon=eps0, max_depth=max_depth, n_adapt=n_adapt, target_accept=target)
    bounds = [0] + [b for b in splits if b is not None] + [nsteps]
    recs, nrecs = [], []
    for a, b in zip(bounds[:-1], bounds[1:]):
        rec, nrec = ops.Recorder(st, b - a, store_every=1), ops.NutsRecords(st, b - a)
        ops.nuts_run(st, ns, b - a, rec, nrec, seed=seed)
        recs.append(rec)
        nrecs.append(nrec)
    torch.cuda.synchronize()
    cat = lambda f: torch.cat([f(r) for r in recs], 1).cpu().numpy()          # noqa: E731
    ncat = lambda f: torch.cat([f(r) for r in nrecs], 1).cpu().numpy()        # noqa: E731
    chain = np.concatenate([st.prob.theta(th0).double().cpu().numpy()[:, None], cat(lambda r: r.samples.double())], 1)
    return dict(chain=chain, logpost=np.concatenate([recs[0].logpost0.cpu().numpy()[:, None], cat(lambda r: r.logpost)], 1),
                alphas=cat(lambda r: r.alpha), accepted=cat(lambda r: r.accepted).astype(bool),
                tree_depth=ncat(lambda r: r.tree_depth), n_leapfrog=ncat(lambda r: r.n_leapfrog),
                diverging=ncat(lambda r: r.diverging).astype(bool), step_size=ncat(lambda r: r.step_size),
                maxpost=st.map_lp.cpu().numpy(), mapparams=st.map_theta.double().cpu().numpy(),
                log_eps=ns.log_eps.cpu().numpy())


def _oracle(layers, x, y, sigma, th0, nsteps, seed, eps0, max_depth, n_adapt, target=0.8):
    lpg = lambda th: qo.logpost_grad(layers, th, x, y, sigma)           # noqa: E731
    return [nuts_oracle.run_chain(lpg, th0[k], nsteps, seed, k, eps0, max_depth, n_adapt, target) for k in range(len(th0))]


def _nets():
    yield 'mlp', qo.mlp_layers(1, 1, (5, 4), True, 'tanh'), 1
    yield 'rnet_c1', qo.rnet_layers(3, 3, 1, 1, biasorno=True, nonlin=True, mlp=False, shared=True), 1


@pytest.mark.parametrize('name', ['mlp', 'rnet_c1'])
def test_fp64_replays_the_oracle(name):
    (layers, P), in_dim = dict((n, (l, d)) for n, l, d in _nets())[name]
    prob, x, y, rs = _problem(layers, P, 40, torch.float64, 3, in_dim)
    assert prob.plan_info(8, True)['tensor_core'] == 0
    th0 = 0.5 * rs.randn(8, P)
    kw = dict(seed=17, eps0=0.05, max_depth=4, n_adapt=12)
    dev = _run(prob, th0, 30, **kw)
    # the device draws its normals with sincospi, the oracle with cos / sin of 2 pi u, and its sums run in another order;
    # trajectories amplify those 1e-16 differences (to ~1e-7 after 30 transitions of depth 7), so the trees are capped at
    # depth 4 here
    refs = _oracle(layers, x, y, 0.1, th0, 30, **kw)
    for k, ref in enumerate(refs):
        for key in ('tree_depth', 'n_leapfrog', 'diverging', 'accepted'):
            np.testing.assert_array_equal(dev[key][k], ref[key], err_msg=f'{key} chain {k}')
        for key in ('chain', 'logpost', 'step_size', 'alphas'):
            d, r = dev[key][k], ref[key][1:] if key == 'alphas' else ref[key]
            assert np.abs(d - r).max() <= 1e-9 * np.abs(r).max(), (key, k, np.abs(d - r).max(), np.abs(r).max())
        assert dev['maxpost'][k] == pytest.approx(ref['maxpost'], rel=1e-9)
    assert (dev['tree_depth'] > 1).mean() > 0.5               # the trees do grow and turn


def test_fp64_is_deterministic_and_segment_independent():
    layers, P = qo.mlp_layers(1, 1, (5, 4), True, 'tanh')
    prob, x, y, rs = _problem(layers, P, 40, torch.float64, 4, 1)
    th0 = 0.5 * rs.randn(8, P)
    kw = dict(seed=9, eps0=0.05, max_depth=7, n_adapt=10)
    a = _run(prob, th0, 30, **kw)
    b = _run(prob, th0, 30, **kw)
    c = _run(prob, th0, 30, splits=(15,), **kw)
    for key in a:
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
        np.testing.assert_array_equal(a[key], c[key], err_msg=key)


PATHS = [  # name, layers, in_dim, dtype, plan code, tolerance
    ('stream_f64', qo.mlp_layers(10, 1, (128, 128, 128), True, 'tanh'), 10, torch.float64, 5, 1e-9),
    ('tcg_h32', qo.mlp_layers(2, 1, (32, 32), True, 'relu'), 2, torch.float32, 3, 2e-3),      # tanh ones go to TG8
    ('tg8_h64', qo.mlp_layers(3, 1, (64, 64), True, 'tanh'), 3, torch.float32, 4, 2e-3),
    ('tg8_h128', qo.mlp_layers(10, 1, (128, 128), True, 'tanh'), 10, torch.float32, 4, 2e-3),
    ('cuda_f32', qo.mlp_layers(1, 1, (5, 4), True, 'tanh'), 1, torch.float32, 0, 2e-3),
]


@pytest.mark.parametrize('name', [p[0] for p in PATHS])
def test_every_path_agrees_with_the_oracle(name):
    _, (layers, P), in_dim, dtype, code, tol = [p for p in PATHS if p[0] == name][0]
    K, nsteps = 16, 3
    prob, x, y, rs = _problem(layers, P, 64, dtype, 5, in_dim)
    assert prob.plan_info(K, True)['tensor_core'] == code
    th0 = (0.3 * rs.randn(K, P)).astype(np.float32).astype(np.float64) if dtype == torch.float32 else 0.3 * rs.randn(K, P)
    # a step size that gives trees of a few doublings on these nets: the largest that the oracle accepts at ~0.8
    eps0 = 2e-3 if P > 1000 else 1e-2
    kw = dict(seed=31, eps0=eps0, max_depth=5, n_adapt=0)
    dev = _run(prob, th0, nsteps, **kw)
    refs = _oracle(layers, x, y, 0.1, th0, nsteps, **kw)
    compared = 0
    for k, ref in enumerate(refs):
        if ref['margin'].min() <= tol:
            continue
        compared += 1
        for key in ('tree_depth', 'n_leapfrog', 'diverging', 'accepted'):
            np.testing.assert_array_equal(dev[key][k], ref[key], err_msg=f'{key} chain {k}')
        scale = np.abs(ref['chain']).max()
        assert np.abs(dev['chain'][k] - ref['chain']).max() <= tol * scale, k
        np.testing.assert_allclose(dev['logpost'][k], ref['logpost'], rtol=tol, atol=tol)
    assert compared >= K // 2, compared


def test_exact_gaussian_posterior_of_a_linear_model():
    """Linear(d, 1): theta = [w, b] has posterior N(theta_hat, sigma^2 (X~^T X~)^-1) under the flat prior"""
    from quinn_b200 import ops, post
    from quinn_b200.netdesc import netdesc_from_module
    d, N, sigma, K = 4, 200, 0.3, 2048
    rs = np.random.RandomState(8)
    x = rs.randn(N, d)
    y = x @ rs.randn(d, 1) + 0.5 + sigma * rs.randn(N, 1)
    Xt = np.hstack([x, np.ones((N, 1))])
    cov = sigma ** 2 * np.linalg.inv(Xt.T @ Xt)
    mean = np.linalg.solve(Xt.T @ Xt, Xt.T @ y[:, 0])
    prob = ops.Problem(netdesc_from_module(torch.nn.Linear(d, 1)), x, y, sigma, dtype=torch.float64, device='cuda')
    n_adapt, n_keep = 1000, 400
    th0 = mean + 0.3 * rs.randn(K, d + 1)
    st = ops.ChainState(prob, th0)
    ns = ops.NutsState(st, epsilon=0.05, max_depth=8, n_adapt=n_adapt, target_accept=0.8)
    ops.nuts_run(st, ns, n_adapt, None, seed=4)
    rec, nrec = ops.Recorder(st, n_keep, store_every=1), ops.NutsRecords(st, n_keep)
    ops.nuts_run(st, ns, n_keep, rec, nrec, seed=4)
    draws = rec.samples                                               # [K, n_keep, P]
    assert not nrec.diverging.any().item()
    acc = rec.alpha.mean().item()
    assert abs(acc - 0.8) <= 0.05, acc
    for p in range(d + 1):
        for f, ref in ((draws[:, :, p], mean[p]), ((draws[:, :, p] - mean[p]) ** 2, cov[p, p])):
            ess = post.ess(f.contiguous()).sum().item()
            se = f.std().item() / np.sqrt(ess)
            assert abs(f.mean().item() - ref) <= 5 * se, (p, f.mean().item(), ref, se, ess)


def test_huge_step_size_diverges_and_keeps_the_state():
    layers, P = qo.mlp_layers(1, 1, (5, 4), True, 'tanh')
    prob, x, y, rs = _problem(layers, P, 40, torch.float64, 6, 1)
    dev = _run(prob, 0.5 * rs.randn(8, P), 10, seed=2, eps0=50.0, max_depth=6, n_adapt=0)
    assert dev['diverging'].mean() > 0.5
    assert np.isfinite(dev['chain']).all() and np.isfinite(dev['logpost']).all()
    stay = dev['diverging'] & ~dev['accepted']
    assert stay.any()
    for k, s in zip(*np.nonzero(stay)):
        np.testing.assert_array_equal(dev['chain'][k, s + 1], dev['chain'][k, s])


def _solver():
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_MCMC
    torch.manual_seed(3)
    rs = np.random.RandomState(3)
    x = rs.rand(50, 1) * 2 - 1
    return NN_MCMC(MLP(1, 1, (6,), activ='tanh').double(), verbose=False), x, np.sin(3 * x) + 0.1 * rs.randn(50, 1)


def test_solver_single_chain_and_many_chains():
    uq, x, y = _solver()
    P = uq.pdim
    sp = dict(epsilon=0.01, max_depth=6, n_adapt=10)
    res = uq.fit(x, y, datanoise=0.1, nmcmc=20, sampler='nuts', sampler_params=sp, seed=5)
    assert res['chain'].shape == (21, P) and res['logpost'].shape == (21,) and res['alphas'].shape == (21,)
    assert isinstance(res['maxpost'], float) and isinstance(res['accrate'], float)
    for key, dt in (('tree_depth', np.int32), ('n_leapfrog', np.int32), ('diverging', bool), ('step_size', np.float64)):
        assert res[key].shape == (20,) and res[key].dtype == dt, key
    assert np.all(res['n_leapfrog'] <= 2 ** 6 - 1) and np.all(res['n_leapfrog'] >= 1)
    assert res['accrate'] == pytest.approx(res['accepted'].mean())
    res = uq.fit(x, y, datanoise=0.1, nmcmc=20, sampler='nuts', sampler_params=sp, seed=5, nchains=4, zflag=False)
    assert res['chain'].shape == (4, 21, P) and res['tree_depth'].shape == (4, 20)
    assert res['step_size'].shape == (4, 20) and np.all(res['step_size'][:, 0] == pytest.approx(0.01))


def test_solver_refusals():
    from quinn_b200.mcmc import NUTS
    uq, x, y = _solver()
    with pytest.raises(ValueError, match='replay'):
        uq.fit(x, y, nmcmc=3, sampler='nuts', replay=dict(incr=np.zeros((3, uq.pdim)), unif=np.zeros(3)), zflag=False)
    for flag in ('distributed', 'data_sharded'):
        with pytest.raises(ValueError, match='nuts'):
            uq.fit(x, y, nmcmc=3, sampler='nuts', **{flag: True})
    m = NUTS()
    m.setLogPost(lambda th: -0.5 * float(np.sum(th ** 2)), None)
    with pytest.raises(ValueError, match='device log-posterior'):
        m.run(3, np.zeros(2), verbose=False)
