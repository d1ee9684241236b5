"""Kernel 6 (qb_logpost_kfac: Kronecker factors of the per-point empirical Fisher of every Linear layer) against the
numpy oracle (tests/kfac_oracle.py), and NN_Laplace(la_type='kron')."""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_util import netdesc_from_layers
from kfac_oracle import factors, kron_precision, layer_index, per_point
from oracle import quinn_oracle as qo
from test_hessian_cpu import case_data
from test_kfac_cpu import SUPPORTED

pytestmark = pytest.mark.gpu


def _np(t):
    return t.double().cpu().numpy()


def _check(got, ref, tol):
    """every factor within tol of its largest entry"""
    assert len(got) == len(ref)
    for g, r in zip(got, ref):
        for k in ('A', 's', 'G'):
            if r[k] is None:
                assert g[k] is None
                continue
            assert g[k].dtype == torch.float64 and g[k].is_cuda
            err = np.abs(_np(g[k]) - r[k]).max()
            assert err <= tol * max(np.abs(r[k]).max(), 1e-300), (k, err, np.abs(r[k]).max())


def _case_problem(name, dtype, N):
    from quinn_b200 import ops
    layers, P, final, x, y, theta, sigma, nfull, prior = case_data(name, N=N)
    if dtype == torch.float32:          # the oracle sees exactly the values the kernel sees
        x, y, theta = (a.astype(np.float32).astype(np.float64) for a in (x, y, theta))
    prob = ops.Problem(netdesc_from_layers(layers, P, final == 'exp'), x, y, sigma, dtype=dtype,
                       prior_sigma=prior['sigma'], prior_anchor=prior['anchor'], fulldatasize=nfull)
    return prob, layers, final, x, y, theta, sigma


@pytest.mark.parametrize('name', SUPPORTED)
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_kfac_matches_oracle(name, dtype):
    from quinn_b200 import ops
    prob, layers, final, x, y, theta, sigma = _case_problem(name, dtype, 300)
    got = ops.logpost_kfac(prob, theta)
    _check(got, factors(layers, theta, x, y, sigma, final), 1e-9 if dtype == torch.float64 else 1e-4)


def _config_net(name):
    hls, outdim, indim = {'mlp_c2': ((32, 32), 1, 2), 'mlp_c5': ((64, 64), 1, 3), 'mlp_c5_o4': ((64, 64), 4, 3),
                          'mlp_c34': ((128, 128), 1, 10)}[name]
    return qo.mlp_layers(indim, outdim, hls, True, 'tanh'), indim, outdim


def _config_problem(name, dtype, N, seed=5):
    from quinn_b200 import ops
    (layers, P), indim, outdim = _config_net(name)
    rs = np.random.RandomState(seed)
    x = rs.rand(N, indim) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True) * np.arange(1, outdim + 1)) + 0.05 * rs.randn(N, outdim)
    theta = 0.2 * rs.randn(P)
    if dtype == torch.float32:
        x, y, theta = (a.astype(np.float32).astype(np.float64) for a in (x, y, theta))
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, 0.05, dtype=dtype, prior_sigma=1.0,
                       prior_anchor=0.1 * rs.randn(P), fulldatasize=2 * N)
    return prob, layers, x, y, theta


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('name', ['mlp_c2', 'mlp_c5', 'mlp_c5_o4', 'mlp_c34'])
def test_kfac_config_nets(name, dtype):
    from quinn_b200 import ops
    prob, layers, x, y, theta = _config_problem(name, dtype, 2000)
    info = ops.kfac_plan_info(prob)
    got = ops.logpost_kfac(prob, theta)
    print(f'{name} {dtype}: plan {info}')
    _check(got, factors(layers, theta, x, y, 0.05), 1e-9 if dtype == torch.float64 else 1e-4)


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_kfac_point_counts(dtype):
    """N not a multiple of the tile, N below one tile, and N = 1 (Lambda without prior = the per-point g g^T)"""
    from quinn_b200 import ops
    TM = ops.kfac_plan_info(_config_problem('mlp_c5', dtype, 1000)[0])['TM']
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    for N in (3 * TM + 5, TM - 3, 1):
        prob, layers, x, y, theta = _config_problem('mlp_c5', dtype, N, seed=N)
        got = ops.logpost_kfac(prob, theta)
        _check(got, factors(layers, theta, x, y, 0.05), tol)
    for name in ('mlp_c5_o4', 'mlp_tanh', 'mlp_nobias', 'mlp_exp'):
        if name.startswith('mlp_c5'):
            prob, layers, x, y, theta = _config_problem(name, dtype, 1, seed=9)
            final, sigma = None, 0.05
        else:
            prob, layers, final, x, y, theta, sigma = _case_problem(name, dtype, 1)
        got = ops.logpost_kfac(prob, theta)
        for L, f, (at, d) in zip(layers, got, per_point(layers, theta, x, y, sigma, final)):
            A = _np(f['A'])
            if f['s'] is not None:
                s = _np(f['s'])
                A = np.block([[A, s[:, None]], [s[None, :], np.ones((1, 1))]])
            Lam = np.kron(_np(f['G']), A)
            g = np.outer(d[0], at[0]).ravel()
            ref = np.outer(g, g)
            assert np.abs(Lam - ref).max() <= tol * max(np.abs(ref).max(), 1e-300), name


def test_kfac_split_equals_unsplit_and_repeats_are_bit_identical():
    from quinn_b200 import ops
    N = 20000
    prob, layers, x, y, theta = _config_problem('mlp_c5', torch.float64, N, seed=6)
    info = ops.kfac_plan_info(prob)
    assert info['splits'] > 1
    a = ops.logpost_kfac(prob, theta)
    b = ops.logpost_kfac(prob, theta)
    for fa, fb in zip(a, b):
        for k in ('A', 's', 'G'):
            assert torch.equal(fa[k], fb[k])
    # unsplit launches: chunks of two tiles (one block each), summed here
    step = 2 * info['TM']
    acc = None
    for lo in range(0, N, step):
        sub = ops.Problem(prob.desc, x[lo:lo + step], y[lo:lo + step], 0.05, dtype=torch.float64)
        assert ops.kfac_plan_info(sub)['splits'] == 1
        part = ops.logpost_kfac(sub, theta)
        acc = [{k: _np(f[k]) for k in ('A', 's', 'G')} for f in part] if acc is None else \
            [{k: acc[i][k] + _np(f[k]) for k in ('A', 's', 'G')} for i, f in enumerate(part)]
    for fa, fr in zip(a, acc):
        for k in ('A', 's', 'G'):
            assert np.abs(_np(fa[k]) - fr[k]).max() <= 1e-12 * np.abs(fr[k]).max()


def test_kfac_errors_and_empty_data():
    from quinn_b200 import _lib, ops
    lib = _lib.load()
    rs = np.random.RandomState(8)
    for name, msg in (('rnet_poly0', 'shares its weights'), ('rnet_quad', 'polynomial')):
        prob, *_ , theta, _ = _case_problem(name, torch.float64, 20)
        with pytest.raises(RuntimeError, match=msg):
            ops.logpost_kfac(prob, theta)
    layers, P = qo.mlp_layers(10, 1, (256, 256), True, 'tanh')
    prob = ops.Problem(netdesc_from_layers(layers, P), rs.randn(50, 10), rs.randn(50, 1), 0.1, dtype=torch.float64)
    assert prob.plan_info(1, True)['tensor_core'] == 5
    with pytest.raises(RuntimeError, match='layer-streamed'):
        ops.logpost_kfac(prob, 0.1 * rs.randn(P))
    prob, layers, final, x, y, theta, sigma = _case_problem('mlp_tanh', torch.float64, 30)
    th = prob.theta(theta)
    F = ops.kfac_plan_info(prob)['factor_elems']
    fac = torch.full((F,), 7.0, dtype=torch.float64, device='cuda')
    ws = torch.empty(lib.qb_kfac_workspace_bytes(C.byref(prob.cnet), prob.qdt, prob.n), dtype=torch.uint8, device='cuda')
    lik = _lib.qb_lik_t(prob.clik.sigma, 1.0, 1.0, th.data_ptr(), 1, 0)          # anchor_per_chain = 1
    rc = lib.qb_logpost_kfac(C.byref(prob.cnet), prob.qdt, ops._ptr(th), C.byref(prob.cdata), C.byref(lik),
                             ops._ptr(fac), ops._ptr(ws), ws.numel(), ops._stream())
    assert rc != 0 and b'anchor_per_chain' in lib.qb_last_error()
    rc = lib.qb_logpost_kfac(C.byref(prob.cnet), prob.qdt, ops._ptr(th), C.byref(prob.cdata), C.byref(prob.clik),
                             ops._ptr(fac), None, 0, ops._stream())
    assert rc != 0 and b'workspace' in lib.qb_last_error()
    # N = 0: zero factors, no kernel launch
    empty = ops.Problem(prob.desc, np.zeros((0, 3)), np.zeros((0, 1)), sigma, dtype=torch.float64)
    assert lib.qb_kfac_workspace_bytes(C.byref(empty.cnet), empty.qdt, 0) == 0
    n0 = lib.qb_launch_count()
    rc = lib.qb_logpost_kfac(C.byref(empty.cnet), empty.qdt, ops._ptr(th), C.byref(empty.cdata), C.byref(empty.clik),
                             ops._ptr(fac), None, 0, ops._stream())
    assert rc == 0 and lib.qb_launch_count() == n0
    assert torch.count_nonzero(fac).item() == 0


# ---------------------------------------------------------------- NN_Laplace('kron')

def test_nn_laplace_kron():
    from test_gpu_hessian import _fit
    from quinn_b200.solvers import NN_Laplace, NN_RMS
    uq, x, y = _fit(NN_Laplace, 'mlp', 'kron', cov_scale=0.5)
    rms, _, _ = _fit(NN_RMS, 'mlp')
    assert uq.batched_fit
    np.testing.assert_array_equal(_np(uq.means), rms.member_thetas())
    layers = uq._desc().as_oracle_layers()
    ind = uq.subsets[0]
    mu = _np(uq.means[0])
    tau = (1.0 / len(ind)) / uq.priorsigma ** 2
    Lam = kron_precision(layers, mu, x[ind], y[ind], uq.datanoise, tau)
    cov_ref = np.linalg.inv(Lam)
    assert len(uq.cov_mats) == 1
    assert np.abs(uq.cov_mats[0] - cov_ref).max() <= 1e-8 * np.abs(cov_ref).max()
    # block-diagonal over the layers
    idx0 = layer_index(layers[0]).ravel()
    idx1 = layer_index(layers[1]).ravel()
    assert np.all(uq.cov_mats[0][np.ix_(idx0, idx1)] == 0)
    # 2e5 draws: mean and covariance within 5 Monte-Carlo standard errors of mu and cov_scale * Lambda^-1
    n = 200000
    np.random.seed(14)
    th = _np(uq._ens_thetas(n)[1])
    S = 0.5 * cov_ref
    d = np.sqrt(np.diag(S))
    assert np.all(np.abs(th.mean(0) - mu) <= 5 * d / np.sqrt(n))
    emp = np.cov(th, rowvar=False)
    se = np.sqrt((np.outer(d ** 2, d ** 2) + S ** 2) / n)
    assert np.all(np.abs(emp - S) <= 5 * se)
    # predictive moments through kernel 4 on the same draws
    xt = np.linspace(-1, 1, 7)[:, None]
    np.random.seed(15)
    th = _np(uq._ens_thetas(50)[1])
    np.random.seed(15)
    m, v, _ = uq.predict_mom_sample(xt, msc=1, nsam=50)
    ye = qo.predict_ens(layers, th, xt)
    np.testing.assert_allclose(m, ye.mean(0), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(v, ye.var(0, ddof=1), rtol=1e-8, atol=1e-14)
    assert uq.predict_sample(xt).shape == (7, 1)
    assert uq.predict_ens(xt, nens=3).shape == (3, 7, 1)


def test_nn_laplace_kron_errors_and_large_net():
    from test_gpu_hessian import _laplace_net
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_Laplace
    with pytest.raises(ValueError, match='shared'):
        NN_Laplace(_laplace_net('rnet_c1'), la_type='kron')
    with pytest.raises(ValueError):
        NN_Laplace(_laplace_net('mlp'), la_type='kfac')
    rs = np.random.RandomState(19)
    x = rs.rand(200, 10) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(200, 1)
    for la_type in ('full', 'kron'):
        np.random.seed(20)
        torch.manual_seed(20)
        uq = NN_Laplace(MLP(10, 1, (128, 128), activ='tanh').double(), la_type=la_type, datanoise=0.1, dfrac=1.0)
        if la_type == 'full':
            with pytest.raises(RuntimeError, match='227 KB'):
                uq.fit(x, y, nepochs=3, lrate=0.01)
            continue
        uq.fit(x, y, nepochs=3, lrate=0.01)
        assert uq.means.shape == (1, uq.nparams)
        np.random.seed(21)
        th = _np(uq._ens_thetas(64)[1])
        assert th.shape == (64, uq.nparams) and np.all(np.isfinite(th))
        assert np.abs(th - _np(uq.means[0])).max() > 0
        m, v, _ = uq.predict_mom_sample(x[:5], msc=1, nsam=16)
        assert m.shape == (5, 1) and np.all(np.isfinite(v))
