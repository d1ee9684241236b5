"""Kernel 7 (qb_predict_jac: network outputs and their per-point Jacobians as per-layer pairs) against the numpy oracle
(tests/glm_oracle.py), and NN_Laplace.predict_mom_glm (the linearised predictive)."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from glm_oracle import glm_moments, jacobian, pairs
from golden_util import netdesc_from_layers
from oracle import quinn_oracle as qo
from test_hessian_cpu import CASES, case_data

pytestmark = pytest.mark.gpu


def _np(t):
    return t.double().cpu().numpy()


def _check(desc, theta, x, dtype, layers, final):
    """f against the oracle and kernel 4, every a / d block within tol of its largest entry"""
    from quinn_b200 import ops
    f, prs = ops.predict_jac(desc, theta, x, dtype=dtype)
    fr, ref = pairs(layers, theta, x, final)
    tol = 1e-10 if dtype == torch.float64 else 1e-5
    assert f.dtype == dtype and f.shape == fr.shape
    assert np.abs(_np(f) - fr).max() <= tol * np.abs(fr).max()
    assert len(prs) == len(ref)
    for g, r in zip(prs, ref):
        for k in ('a', 'd'):
            assert g[k].dtype == dtype and tuple(g[k].shape) == r[k].shape
            err = np.abs(_np(g[k]) - r[k]).max()
            assert err <= tol * max(np.abs(r[k]).max(), 1e-300), (k, err, np.abs(r[k]).max())
    # f is kernel 4's prediction at the same theta
    k4, _, _ = ops.predict(desc, theta, x, dtype=dtype)
    k4 = _np(k4[0])
    rel = 1e-12 if dtype == torch.float64 else 1e-5
    assert np.abs(_np(f) - k4).max() <= rel * np.abs(k4).max()
    return f, prs


def _case(name, dtype, N):
    layers, P, final, x, y, theta, *_ = case_data(name, N=N)
    if dtype == torch.float32:          # the oracle sees exactly the values the kernel sees
        x, theta = (a.astype(np.float32).astype(np.float64) for a in (x, theta))
    return netdesc_from_layers(layers, P, final == 'exp'), layers, final, x, theta


@pytest.mark.parametrize('name', CASES)
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_jac_matches_oracle(name, dtype):
    desc, layers, final, x, theta = _case(name, dtype, 300)
    _check(desc, theta, x, dtype, layers, final)


def _config(name, dtype, N, seed=5):
    hls, outdim, indim = {'mlp_c2': ((32, 32), 1, 2), 'mlp_c5': ((64, 64), 1, 3), 'mlp_c5_o4': ((64, 64), 4, 3),
                          'mlp_c34': ((128, 128), 1, 10)}[name]
    layers, P = qo.mlp_layers(indim, outdim, hls, True, 'tanh')
    rs = np.random.RandomState(seed)
    x = rs.rand(N, indim) * 2 - 1
    theta = 0.2 * rs.randn(P)
    if dtype == torch.float32:
        x, theta = (a.astype(np.float32).astype(np.float64) for a in (x, theta))
    return netdesc_from_layers(layers, P), layers, x, theta


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('name', ['mlp_c2', 'mlp_c5', 'mlp_c5_o4', 'mlp_c34'])
def test_jac_config_nets(name, dtype):
    from quinn_b200 import ops
    desc, layers, x, theta = _config(name, dtype, 2000)
    print(f'{name} {dtype}: plan {ops.jac_plan_info(desc, 2000, dtype)}')
    _check(desc, theta, x, dtype, layers, None)


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_jac_point_counts(dtype):
    """N not a multiple of the tile, N below one tile, N = 1, and N = 0 (no launch)"""
    from quinn_b200 import _lib, ops
    TM = ops.jac_plan_info(_config('mlp_c5', dtype, 1)[0], 1000, dtype)['TM']
    for N in (3 * TM + 5, TM - 3, 1):
        for name in ('mlp_c5', 'mlp_c5_o4'):
            desc, layers, x, theta = _config(name, dtype, N, seed=N)
            _check(desc, theta, x, dtype, layers, None)
    desc, layers, x, theta = _config('mlp_c5', dtype, 0)
    lib = _lib.load()
    n0 = lib.qb_launch_count()
    f, prs = ops.predict_jac(desc, theta, x, dtype=dtype)
    assert lib.qb_launch_count() == n0
    assert f.shape == (0, 1) and prs[0]['a'].shape == (3, 0) and prs[-1]['d'].shape == (1, 1, 0)


def test_jac_repeats_are_bit_identical():
    from quinn_b200 import ops
    desc, layers, x, theta = _config('mlp_c5_o4', torch.float64, 20000, seed=6)
    assert ops.jac_plan_info(desc, 20000, torch.float64)['blocks'] > 1
    fa, pa = ops.predict_jac(desc, theta, x, dtype=torch.float64)
    fb, pb = ops.predict_jac(desc, theta, x, dtype=torch.float64)
    assert torch.equal(fa, fb)
    for a, b in zip(pa, pb):
        assert torch.equal(a['a'], b['a']) and torch.equal(a['d'], b['d'])


def test_jac_refusals():
    from quinn_b200 import _lib, ops
    rs = np.random.RandomState(8)
    layers, P = qo.mlp_layers(10, 1, (256, 256), True, 'tanh')
    desc = netdesc_from_layers(layers, P)
    for dtype in (torch.float64, torch.float32):
        with pytest.raises(RuntimeError, match='layer-streamed'):
            ops.predict_jac(desc, 0.1 * rs.randn(P), rs.randn(50, 10), dtype=dtype)
    lib = _lib.load()
    desc, layers, x, theta = _config('mlp_c5', torch.float64, 10)
    net = desc.to_c()
    th = torch.as_tensor(theta, device='cuda')
    xs = torch.as_tensor(x, device='cuda')
    out = torch.empty((10, 1), dtype=torch.float64, device='cuda')
    fac = torch.empty(10 * ops.jac_plan_info(desc, 10, torch.float64)['rows'], dtype=torch.float64, device='cuda')
    args = [ops._ptr(th), ops._ptr(xs), 10, ops._ptr(out), ops._ptr(fac)]
    for i in (0, 1, 3, 4):
        bad = list(args)
        bad[i] = None
        assert lib.qb_predict_jac(C.byref(net), _lib.QB_F64, *bad, ops._stream()) != 0
        assert b'NULL' in lib.qb_last_error()
    bad = list(args)
    bad[2] = -1
    assert lib.qb_predict_jac(C.byref(net), _lib.QB_F64, *bad, ops._stream()) != 0
    assert b'negative' in lib.qb_last_error()
    assert lib.qb_predict_jac(C.byref(net), _lib.QB_F64, *args, ops._stream()) == 0


# ---------------------------------------------------------------- NN_Laplace.predict_mom_glm

_FITS = {}


def _fitted(kind, la_type, nens):
    """one fit per (kind, la_type, nens), shared by the tests of this module"""
    from test_gpu_hessian import _fit
    from quinn_b200.solvers import NN_Laplace
    key = (kind, la_type, nens)
    if key not in _FITS:
        _FITS[key] = _fit(NN_Laplace, kind, la_type, nens=nens, cov_scale=0.5)
    return _FITS[key]


def _sampler_cov(uq, j):
    """the covariance _ens_thetas draws member j from (without cov_scale): for 'full' U |lambda|^-1 U^T, which differs
    from cov_mats where the Hessian has negative eigenvalues"""
    if uq.la_type == 'full':
        U, _, lam = uq._factors[j]
        return _np((U / lam.abs()) @ U.T)
    return uq.cov_mats[j]


def _oracle_members(uq, xt):
    layers = uq._desc().as_oracle_layers()
    final = 'exp' if uq._desc().final_exp else None
    return [(*jacobian(layers, _np(uq.means[j]), xt, final), _sampler_cov(uq, j)) for j in range(uq.nens)]


XT = np.linspace(-1, 1, 7)[:, None]
GLM_CASES = [('mlp', t, n) for t in ('full', 'diag', 'kron') for n in (1, 3)] + \
            [('rnet_c1', t, n) for t in ('full', 'diag') for n in (1, 3)]


@pytest.mark.parametrize('kind,la_type,nens', GLM_CASES)
def test_predict_mom_glm_matches_oracle(kind, la_type, nens):
    uq, x, y = _fitted(kind, la_type, nens)
    mean_r, var_r, cov_r = glm_moments(_oracle_members(uq, XT), uq.cov_scale)
    m0, v0, c0 = uq.predict_mom_glm(XT)
    assert v0 is None and c0 is None
    m1, v1, c1 = uq.predict_mom_glm(XT, msc=1)
    m2, v2, c2 = uq.predict_mom_glm(XT, msc=2)
    assert c1 is None and m1.shape == v1.shape == (7, 1) and c2.shape == (7, 7, 1)
    for m in (m0, m1, m2):
        assert np.abs(m - mean_r).max() <= 1e-8 * np.abs(mean_r).max()
    for v in (v1, v2):
        assert np.abs(v - var_r).max() <= 1e-8 * np.abs(var_r).max()
    assert np.abs(c2 - cov_r).max() <= 1e-8 * np.abs(cov_r).max()
    with pytest.raises(ValueError):
        uq.predict_mom_glm(XT, msc=3)


def test_predict_mom_glm_before_fit_raises():
    from test_gpu_hessian import _laplace_net
    from quinn_b200.solvers import NN_Laplace
    with pytest.raises(RuntimeError, match='fit'):
        NN_Laplace(_laplace_net('mlp')).predict_mom_glm(XT)


@pytest.mark.parametrize('la_type', ['full', 'diag', 'kron'])
def test_predict_mom_glm_multi_output(la_type):
    """two outputs: the diagonal of the msc=2 covariance is the msc=1 variance, both match the oracle"""
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_Laplace
    rs = np.random.RandomState(22)
    x = rs.rand(60, 1) * 2 - 1
    y = np.hstack([np.sin(3 * x), np.cos(2 * x)]) + 0.1 * rs.randn(60, 2)
    np.random.seed(23)
    torch.manual_seed(23)
    uq = NN_Laplace(MLP(1, 2, (5,), activ='tanh').double(), nens=2, la_type=la_type, cov_scale=0.5, datanoise=0.1,
                    dfrac=0.8)
    uq.fit(x, y, nepochs=500, lrate=0.02, freq_out=1000)
    m1, v1, _ = uq.predict_mom_glm(XT, msc=1)
    m2, v2, c2 = uq.predict_mom_glm(XT, msc=2)
    assert v1.shape == (7, 2) and c2.shape == (7, 7, 2)
    np.testing.assert_allclose(m1, m2, rtol=0, atol=1e-14)
    for j in range(2):
        np.testing.assert_allclose(np.diag(c2[:, :, j]), v1[:, j], rtol=1e-12, atol=1e-15)
    mean_r, var_r, cov_r = glm_moments(_oracle_members(uq, XT), uq.cov_scale)
    assert np.abs(v1 - var_r).max() <= 1e-8 * np.abs(var_r).max()
    assert np.abs(c2 - cov_r).max() <= 1e-8 * np.abs(cov_r).max()


@pytest.mark.parametrize('la_type', ['full', 'diag', 'kron'])
def test_predict_mom_glm_is_the_linearised_sampler(la_type):
    """the linearised model f(mu_m) + J_m (theta_s - mu_m) on 2e5 draws of _ens_thetas: its mean and variance are within
    5 Monte-Carlo standard errors of the GLM moments"""
    uq, x, y = _fitted('mlp', la_type, 3)
    n = 200000
    np.random.seed(31)
    members = np.random.randint(0, uq.nens, size=n)
    np.random.seed(31)
    th = _np(uq._ens_thetas(n)[1])
    lin = np.empty((n, XT.shape[0]))
    for j, (f, J, _) in enumerate(_oracle_members(uq, XT)):
        rows = members == j
        lin[rows] = f[:, 0] + (th[rows] - _np(uq.means[j])) @ J[:, 0].T
    m, v, _ = uq.predict_mom_glm(XT, msc=1)
    emp_m, emp_v = lin.mean(0), lin.var(0)
    m4 = ((lin - emp_m) ** 4).mean(0)
    assert np.all(np.abs(emp_m - m[:, 0]) <= 5 * np.sqrt(emp_v / n))
    assert np.all(np.abs(emp_v - v[:, 0]) <= 5 * np.sqrt((m4 - emp_v ** 2) / n))


def test_predict_mom_glm_small_cov_scale_matches_the_sampled_predictive():
    """at cov_scale = 1e-6 the net is linear over the posterior's spread: kernel 4's sampled variance agrees with the
    GLM variance within its Monte-Carlo error"""
    uq, x, y = _fitted('mlp', 'full', 1)
    uq = copy.copy(uq)
    uq.cov_scale = 1e-6
    nsam = 20000
    np.random.seed(32)
    m_s, v_s, _ = uq.predict_mom_sample(XT, msc=1, nsam=nsam)
    m, v, _ = uq.predict_mom_glm(XT, msc=1)
    assert np.all(np.abs(v_s - v) <= 5 * np.sqrt(2.0 / (nsam - 1)) * v)
    # the sampled mean also carries the second-order term cov_scale/2 tr(f'' Sigma), which the linearisation drops
    assert np.abs(m_s - m).max() <= 1e-4 * np.abs(m).max()


def test_predict_mom_glm_fp32_and_chunks(monkeypatch):
    """kernel 7 in fp32 at the same posterior agrees with fp64 to 1e-4; an fp32 fit runs; chunked and unchunked calls
    agree to 1e-12"""
    from quinn_b200.solvers import NN_Laplace, nn_laplace
    from test_gpu_hessian import _fit
    xt = np.linspace(-1, 1, 301)[:, None]
    for la_type in ('full', 'diag', 'kron'):
        uq, x, y = _fitted('mlp', la_type, 3)
        ref = uq.predict_mom_glm(xt, msc=1)
        u32 = copy.copy(uq)
        u32.dtype = torch.float32
        got = u32.predict_mom_glm(xt, msc=1)
        for g, r in zip(got[:2], ref[:2]):
            assert np.abs(g - r).max() <= 1e-4 * np.abs(r).max()
        with monkeypatch.context() as mp:
            mp.setattr(nn_laplace, '_GLM_CHUNK_BYTES', 8 * 16 * 37)         # chunks of 37 points (P = 16 > F)
            ch = uq.predict_mom_glm(xt, msc=1)
        for g, r in zip(ch[:2], ref[:2]):
            assert np.abs(g - r).max() <= 1e-12 * np.abs(r).max()
    uq, _, _ = _fit(NN_Laplace, 'mlp', 'full', cov_scale=0.5, dtype=torch.float32)
    m, v, _ = uq.predict_mom_glm(xt, msc=1)
    assert m.shape == v.shape == (301, 1) and np.all(np.isfinite(v)) and np.all(v > 0)
