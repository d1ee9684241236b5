"""Kernel 5 (qb_logpost_hvp: exact Hessian-vector products of the log-posterior) against the numpy forward-over-reverse
oracle, the shipped gradient kernel and torch autograd; NNWrap.calc_hess_full and the NN_Laplace solver."""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_util import netdesc_from_layers
from hessian_oracle import logpost_hessian, logpost_hvp
from oracle import quinn_oracle as qo
from test_hessian_cpu import CASES, _torch_neg_log_post, case_data

pytestmark = pytest.mark.gpu


def _problem(name, dtype, N=13, with_prior=True):
    from quinn_b200 import ops
    layers, P, final, x, y, theta, sigma, nfull, prior = case_data(name, N=N)
    if dtype == torch.float32:          # the oracle sees exactly the values the kernel sees
        x, y, theta = (a.astype(np.float32).astype(np.float64) for a in (x, y, theta))
    desc = netdesc_from_layers(layers, P, final == 'exp')
    prob = ops.Problem(desc, x, y, sigma, dtype=dtype, prior_sigma=prior['sigma'] if with_prior else None,
                       prior_anchor=prior['anchor'] if with_prior else None, fulldatasize=nfull)
    return prob, layers, P, final, x, y, theta, sigma, nfull, (prior if with_prior else None)


def _np(t):
    return t.double().cpu().numpy()


@pytest.mark.parametrize('with_prior', [False, True])
@pytest.mark.parametrize('name', CASES)
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_hvp_matches_oracle(name, dtype, with_prior):
    from quinn_b200 import ops
    prob, layers, P, final, x, y, theta, sigma, nfull, prior = _problem(name, dtype, N=300, with_prior=with_prior)
    V = np.random.RandomState(3).randn(4, P)
    if dtype == torch.float32:
        V = V.astype(np.float32).astype(np.float64)
    hv = _np(ops.logpost_hvp(prob, theta, V))
    ref = logpost_hvp(layers, theta, x, y, sigma, nfull, prior, final, V)
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    assert np.abs(hv - ref).max() <= tol * np.abs(ref).max()
    H = _np(ops.logpost_hessian(prob, theta))                         # unit directions (v == NULL)
    Href = logpost_hessian(layers, theta, x, y, sigma, nfull, prior, final)
    assert np.abs(H - Href).max() <= tol * np.abs(Href).max()


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('name', ['mlp_c2', 'mlp_c5', 'mlp_c5_o4'])
def test_hvp_config_nets(name, dtype):
    """config-2 / config-5 nets (and a 4-output net of that size) at N = 2000: random directions and Hessian rows"""
    from quinn_b200 import ops
    hls, outdim, indim = {'mlp_c2': ((32, 32), 1, 2), 'mlp_c5': ((64, 64), 1, 3), 'mlp_c5_o4': ((64, 64), 4, 3)}[name]
    layers, P = qo.mlp_layers(indim, outdim, hls, True, 'tanh')
    rs = np.random.RandomState(5)
    x = rs.rand(2000, indim) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True) * np.arange(1, outdim + 1)) + 0.05 * rs.randn(2000, outdim)
    theta = 0.2 * rs.randn(P)
    anchor = 0.1 * rs.randn(P)
    if dtype == torch.float32:
        x, y, theta = (a.astype(np.float32).astype(np.float64) for a in (x, y, theta))
    prior = dict(sigma=1.0, anchor=anchor)
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, 0.05, dtype=dtype, prior_sigma=1.0, prior_anchor=anchor,
                       fulldatasize=4000)
    V = rs.randn(3, P)
    if dtype == torch.float32:
        V = V.astype(np.float32).astype(np.float64)
    hv = _np(ops.logpost_hvp(prob, theta, V))
    ref = logpost_hvp(layers, theta, x, y, 0.05, 4000, prior, None, V)
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    err = np.abs(hv - ref).max() / np.abs(ref).max()
    print(f'{name} {dtype}: max |hv - oracle| / max |oracle| = {err:.2e}')
    assert err <= tol
    H = ops.logpost_hessian(prob, theta, block=P // 3 + 1)
    rows = [0, P // 2, P - 1]
    Href = logpost_hvp(layers, theta, x, y, 0.05, 4000, prior, None, np.eye(P)[rows])
    assert np.abs(_np(H[rows]) - Href).max() <= tol * np.abs(Href).max()
    if dtype == torch.float64:
        Hn = _np(H)
        assert np.abs(Hn - Hn.T).max() <= 1e-10 * np.abs(Hn).max()


def test_unit_directions_equal_explicit_identity():
    from quinn_b200 import ops
    for name in ('mlp_tanh', 'rnet_quad', 'mlp_exp'):
        prob, layers, P, final, x, y, theta, *_ = _problem(name, torch.float64, N=50)
        H = _np(ops.logpost_hessian(prob, theta))
        Hv = _np(ops.logpost_hvp(prob, theta, np.eye(P)))
        np.testing.assert_array_equal(H, Hv)
        assert np.abs(H - H.T).max() <= 1e-10 * np.abs(H).max()
        H2 = _np(ops.logpost_hessian(prob, theta, block=5))            # column blocks, col0 > 0
        np.testing.assert_array_equal(H, H2)


def test_split_launch_equals_unsplit_and_repeats_are_bit_identical():
    from quinn_b200 import ops
    layers, P = qo.mlp_layers(3, 1, (64, 64), True, 'tanh')
    rs = np.random.RandomState(6)
    x = rs.rand(20000, 3) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(20000, 1)
    theta = 0.2 * rs.randn(P)
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, 0.05, dtype=torch.float64, prior_sigma=1.0,
                       prior_anchor=np.zeros(P), fulldatasize=20000)
    v = rs.randn(P)
    assert ops.hvp_plan_info(prob, 1)['splits'] > 1
    assert ops.hvp_plan_info(prob, 2048)['splits'] == 1
    a = _np(ops.logpost_hvp(prob, theta, v[None]))[0]
    b = _np(ops.logpost_hvp(prob, theta, v[None]))[0]
    np.testing.assert_array_equal(a, b)
    Vb = np.zeros((2048, P))
    Vb[7] = v
    c = _np(ops.logpost_hvp(prob, theta, Vb))[7]
    assert np.abs(a - c).max() <= 1e-12 * np.abs(c).max()
    np.testing.assert_array_equal(c, _np(ops.logpost_hvp(prob, theta, Vb))[7])


def test_hvp_is_the_derivative_of_the_gradient_kernel():
    """(g(theta + h v) - g(theta - h v)) / 2h from qb_logpost_grad against Hv, fp64, on the config-5 net and an RNet"""
    from quinn_b200 import ops
    for name in ('rnet_quad', 'mlp_c5'):
        if name == 'mlp_c5':
            layers, P = qo.mlp_layers(3, 1, (64, 64), True, 'tanh')
            rs = np.random.RandomState(7)
            x = rs.rand(3000, 3) * 2 - 1
            y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(3000, 1)
            theta = 0.2 * rs.randn(P)
            prob = ops.Problem(netdesc_from_layers(layers, P), x, y, 0.05, dtype=torch.float64, prior_sigma=1.0,
                               prior_anchor=0.1 * rs.randn(P), fulldatasize=6000)
        else:
            prob, layers, P, final, x, y, theta, *_ = _problem(name, torch.float64, N=500)
            rs = np.random.RandomState(7)
        v = rs.randn(P)
        h = 1e-5
        _, g = ops.logpost_grad(prob, np.stack([theta + h * v, theta - h * v]))
        fd = _np(g[0] - g[1]) / (2 * h)
        hv = _np(ops.logpost_hvp(prob, theta, v[None]))[0]
        assert np.abs(fd - hv).max() <= 1e-6 * np.abs(hv).max()


def test_errors_and_empty_call():
    from quinn_b200 import _lib, ops
    lib = _lib.load()
    layers, P = qo.mlp_layers(10, 1, (128, 128), True, 'tanh')           # config 3 / 4
    rs = np.random.RandomState(8)
    prob = ops.Problem(netdesc_from_layers(layers, P), rs.randn(50, 10), rs.randn(50, 1), 0.1, dtype=torch.float64)
    with pytest.raises(RuntimeError, match='227 KB'):
        ops.logpost_hvp(prob, rs.randn(P), rs.randn(2, P))
    prob, layers, P, *_ = _problem('mlp_tanh', torch.float64)
    theta = prob.theta(np.zeros(P))
    hv = torch.zeros((2, P), dtype=torch.float64, device='cuda')
    lik = _lib.qb_lik_t(prob.clik.sigma, 1.0, 1.0, theta.data_ptr(), 1, 0)         # anchor_per_chain = 1
    rc = lib.qb_logpost_hvp(C.byref(prob.cnet), prob.qdt, ops._ptr(theta), None, 0, 2, C.byref(prob.cdata), C.byref(lik),
                            ops._ptr(hv), None, 0, ops._stream())
    assert rc != 0 and b'anchor_per_chain' in lib.qb_last_error()
    rc = lib.qb_logpost_hvp(C.byref(prob.cnet), prob.qdt, ops._ptr(theta), None, P - 1, 2, C.byref(prob.cdata),
                            C.byref(prob.clik), ops._ptr(hv), None, 0, ops._stream())
    assert rc != 0                                                                    # unit rows beyond P
    rc = lib.qb_logpost_hvp(C.byref(prob.cnet), prob.qdt, ops._ptr(theta), None, 0, 0, C.byref(prob.cdata),
                            C.byref(prob.clik), None, None, 0, ops._stream())
    assert rc == 0                                                                    # K = 0: nothing to do
    n0 = lib.qb_launch_count()
    lib.qb_logpost_hvp(C.byref(prob.cnet), prob.qdt, ops._ptr(theta), None, 0, 0, C.byref(prob.cdata),
                       C.byref(prob.clik), None, None, 0, ops._stream())
    assert lib.qb_launch_count() == n0


def test_nnwrap_calc_hess_full_matches_autograd():
    from quinn_b200.netdesc import flatten_module
    from quinn_b200.nns import MLP
    from quinn_b200.nns.losses import NegLogPost
    from quinn_b200.nns.nnwrap import NNWrap
    torch.manual_seed(0)
    net = MLP(2, 2, (6, 5), activ='tanh').double()
    rs = np.random.RandomState(9)
    x, y = rs.rand(40, 2), rs.randn(40, 2)
    theta = flatten_module(net) + 0.3 * rs.randn(sum(p.numel() for p in net.parameters()))
    anchor = torch.as_tensor(0.2 * rs.randn(theta.size))
    wrap = NNWrap(net)
    for pp in (None, {'sigma': 0.8, 'anchor': anchor}):
        loss = NegLogPost(net, 100, 0.2, pp)
        H = wrap.calc_hess_full(theta, loss, x, y)
        layers = wrap.desc().as_oracle_layers()
        f = _torch_neg_log_post(layers, x, y, 0.2, 100, None if pp is None else dict(sigma=0.8, anchor=anchor.numpy()), None)
        ref = torch.autograd.functional.hessian(f, torch.as_tensor(theta)).numpy()
        assert H.shape == (theta.size, theta.size)
        assert np.abs(H - ref).max() <= 1e-9 * np.abs(ref).max()
    with pytest.raises(NotImplementedError):
        wrap.calc_hess_full(theta, torch.nn.MSELoss(), x, y)


# ---------------------------------------------------------------- NN_Laplace

def _laplace_net(kind):
    from quinn_b200.nns import MLP, Poly, RNet
    torch.manual_seed(11)
    if kind == 'rnet_c1':
        return RNet(3, 3, wp_function=Poly(0), indim=1, outdim=1, layer_pre=True, layer_post=True, biasorno=True,
                    nonlin=True, mlp=False, final_layer=None).double()
    return MLP(1, 1, (5,), activ='tanh').double()


def _laplace_data():
    rs = np.random.RandomState(12)
    x = rs.rand(60, 1) * 2 - 1
    return x, np.sin(3 * x) + 0.1 * rs.randn(60, 1)


def _fit(cls, kind, la_type=None, nens=1, **kw):
    x, y = _laplace_data()
    np.random.seed(13)
    torch.manual_seed(13)
    args = dict(nens=nens, datanoise=0.1, priorsigma=1.0, dfrac=0.8)
    if la_type is not None:
        args.update(la_type=la_type, **kw)
    uq = cls(_laplace_net(kind), **args)
    uq.fit(x, y, nepochs=1500, lrate=0.02, freq_out=1000)
    return uq, x, y


def _oracle_curvature(uq, k, x, y):
    """loss Hessian (full) or diagonal Fisher (diag) of member k at its MAP, from the numpy oracle"""
    layers = uq._desc().as_oracle_layers()
    ind = uq.subsets[k]
    mu = _np(uq.means[k])
    prior = dict(sigma=uq.priorsigma, anchor=uq.anchors[k])
    if uq.la_type == 'full':
        return -logpost_hessian(layers, mu, x[ind], y[ind], uq.datanoise, len(ind), prior)
    return qo.diag_fisher(layers, mu, x[ind], y[ind], uq.datanoise, len(ind), prior)


@pytest.mark.parametrize('la_type', ['full', 'diag'])
@pytest.mark.parametrize('kind', ['rnet_c1', 'mlp'])
def test_nn_laplace(kind, la_type):
    from quinn_b200.solvers import NN_Laplace, NN_RMS
    uq, x, y = _fit(NN_Laplace, kind, la_type, cov_scale=0.5)
    rms, _, _ = _fit(NN_RMS, kind)
    assert uq.batched_fit
    np.testing.assert_array_equal(_np(uq.means), rms.member_thetas())          # the MAP the batched trainer returns
    C0 = _oracle_curvature(uq, 0, x, y)
    if la_type == 'full':
        lam, U = np.linalg.eigh(C0)
        cov_ref = np.linalg.inv(C0)
        samp_cov = (U / np.abs(lam)) @ U.T
    else:
        cov_ref = samp_cov = np.diag(1.0 / C0)
    assert len(uq.cov_mats) == 1
    assert np.abs(uq.cov_mats[0] - cov_ref).max() <= 1e-8 * np.abs(cov_ref).max()
    # 2e5 draws: mean and covariance within 5 Monte-Carlo standard errors of mu and cov_scale * H^-1
    n = 200000
    np.random.seed(14)
    th = _np(uq._ens_thetas(n)[1])
    mu, S = _np(uq.means[0]), 0.5 * samp_cov
    d = np.sqrt(np.diag(S))
    assert np.all(np.abs(th.mean(0) - mu) <= 5 * d / np.sqrt(n))
    emp = np.cov(th, rowvar=False)
    se = np.sqrt((np.outer(d ** 2, d ** 2) + S ** 2) / n)
    assert np.all(np.abs(emp - S) <= 5 * se)
    # predictive moments through kernel 4 on the same draws
    xt = np.linspace(-1, 1, 7)[:, None]
    for msc in (0, 1, 2):
        m, v, c = uq.predict_mom_sample(xt, msc=msc, nsam=40)
        assert m.shape == (7, 1)
        assert (v is None) == (msc == 0) and (c is None) == (msc < 2)
        if msc == 2:
            assert v.shape == (7, 1) and c.shape == (7, 7, 1)
    np.random.seed(15)
    th = _np(uq._ens_thetas(50)[1])
    np.random.seed(15)
    m, v, _ = uq.predict_mom_sample(xt, msc=1, nsam=50)
    ye = qo.predict_ens(uq._desc().as_oracle_layers(), th, xt)
    np.testing.assert_allclose(m, ye.mean(0), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(v, ye.var(0, ddof=1), rtol=1e-8, atol=1e-14)
    assert uq.predict_sample(xt).shape == (7, 1)
    assert uq.predict_ens(xt, nens=3).shape == (3, 7, 1)


def test_nn_laplace_members_and_errors(monkeypatch):
    from quinn_b200.nns.nnwrap import NNWrap
    from quinn_b200.solvers import NN_Laplace
    with pytest.raises(ValueError):
        NN_Laplace(_laplace_net('mlp'), la_type='kfac')
    uq, x, y = _fit(NN_Laplace, 'mlp', 'diag', nens=3)
    assert uq.means.shape[0] == 3 and len(uq.cov_mats) == 3
    n = 30000
    np.random.seed(16)
    members = np.random.randint(0, 3, size=n)
    np.random.seed(16)
    th = _np(uq._ens_thetas(n)[1])
    assert set(members) == {0, 1, 2}
    for j in range(3):
        rows = th[members == j]
        sd = np.sqrt(np.diag(uq.cov_mats[j]))
        assert np.all(np.abs(rows.mean(0) - _np(uq.means[j])) <= 5 * sd / np.sqrt(len(rows)))
    # a zero diagonal entry is singular, as np.linalg.inv would find
    real = NNWrap.fisher_diag_device

    def with_zero(self, *a, **k):
        f = real(self, *a, **k)
        f[2] = 0.0
        return f
    monkeypatch.setattr(NNWrap, 'fisher_diag_device', with_zero)
    with pytest.raises(np.linalg.LinAlgError):
        uq.la_calc(uq.learners[0], x[uq.subsets[0]], y[uq.subsets[0]], uq.anchors[0])


def test_nn_laplace_indefinite_hessian_warns_and_samples_with_abs_eigenvalues():
    from quinn_b200.netdesc import unflatten_module
    from quinn_b200.solvers import NN_Laplace
    uq, x, y = _fit(NN_Laplace, 'mlp', 'full')
    learner = uq.learners[0]
    rs = np.random.RandomState(17)
    far = 2.0 * rs.randn(uq.nparams)                     # far from the MAP, weak prior: an indefinite Hessian
    unflatten_module(learner.best_model, far)
    uq.priorsigma = 30.0
    ind = uq.subsets[0]
    layers = uq._desc().as_oracle_layers()
    Hl = -logpost_hessian(layers, far, x[ind], y[ind], uq.datanoise, len(ind), dict(sigma=30.0, anchor=uq.anchors[0]))
    lam, U = np.linalg.eigh(Hl)
    assert lam.min() < 0 < lam.max()
    uq._factors = []
    with pytest.warns(RuntimeWarning, match='positive-semidefinite'):
        uq.la_calc(learner, x[ind], y[ind], uq.anchors[0])
    Uk, isq, _ = uq._factors[0]
    got = _np((Uk * isq ** 2) @ Uk.T)
    ref = (U / np.abs(lam)) @ U.T
    assert np.abs(got - ref).max() <= 1e-8 * np.abs(ref).max()


def test_nn_laplace_member_by_member_fit(monkeypatch):
    """options the batched trainer does not take keep NN_RMS's member-by-member fit; la_calc uses its subsets and anchors"""
    from quinn_b200.solvers import NN_Laplace
    monkeypatch.setenv('QB_ENS_SEQUENTIAL', '1')
    x, y = _laplace_data()
    np.random.seed(18)
    torch.manual_seed(18)
    uq = NN_Laplace(_laplace_net('mlp'), nens=2, la_type='full', datanoise=0.1, dfrac=0.8)
    uq.fit(x, y, nepochs=30, lrate=0.01)
    assert not uq.batched_fit and uq.subsets.shape == (2, 48) and uq.anchors.shape == (2, uq.nparams)
    for k in range(2):
        np.testing.assert_allclose(_np(uq.means[k]), uq.member_thetas()[k], rtol=0, atol=0)
        cov_ref = np.linalg.inv(_oracle_curvature(uq, k, x, y))
        assert np.abs(uq.cov_mats[k] - cov_ref).max() <= 1e-8 * np.abs(cov_ref).max()
