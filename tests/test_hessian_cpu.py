"""CPU checks of the Hessian-vector path: the numpy forward-over-reverse oracle (tests/hessian_oracle.py) against torch
autograd of a float64 restatement of NegLogPost, and the launch plan of kernel 5 (qb_hvp_plan_info)."""
import ctypes

import numpy as np
import pytest
import torch

from golden_util import netdesc_from_layers
from hessian_oracle import logpost_hessian, logpost_hvp
from oracle import quinn_oracle as qo

F32, F64 = 0, 1
SMEM_MAX = 227 * 1024


def _torch_neg_log_post(layers, x, y, sigma, fulldatasize, prior, final):
    """NegLogPost.forward (losses.py:186-206) of the flat theta, in float64 torch."""
    x, y = torch.as_tensor(x), torch.as_tensor(y)

    def wb(L, th):
        nw = L['n_in'] * L['n_out']
        terms = L.get('terms', [(1.0, L['w_off'], L['b_off'])])
        W = sum(c * th[wo:wo + nw].reshape(L['n_out'], L['n_in']) for c, wo, _ in terms)
        b = sum(c * th[bo:bo + L['n_out']] for c, _, bo in terms) if L['b_off'] >= 0 else None
        return W, b

    def f(th):
        h = x
        for L in layers:
            W, b = wb(L, th)
            z = h @ W.T + (b if b is not None else 0.0)
            a = torch.tanh(z) if L['act'] == 'tanh' else (torch.relu(z) if L['act'] == 'relu' else z)
            h = h + L['res_step'] * a if L['res_step'] != 0.0 else a
        if final == 'exp':
            h = torch.exp(h)
        n = h.shape[0]
        val = 0.5 * torch.sum((y - h) ** 2) / sigma ** 2 + n / 2 * np.log(2 * np.pi) + n * np.log(sigma)
        if prior is not None:
            anchor = torch.as_tensor(prior['anchor'])
            val = val + n * (torch.sum((th - anchor) ** 2) / 2 / prior['sigma'] ** 2
                             + th.numel() / 2 * np.log(2 * np.pi * prior['sigma'] ** 2)) / fulldatasize
        return val
    return f


def _case(name):
    """(layers, P, final) of the networks the Hessian tests cover"""
    if name == 'mlp_tanh':
        layers, P = qo.mlp_layers(3, 1, (6, 5), True, 'tanh')
    elif name == 'mlp_relu':
        layers, P = qo.mlp_layers(2, 1, (7,), True, 'relu')
    elif name == 'mlp_identity':
        layers, P = qo.mlp_layers(3, 1, (4, 4), True, 'lin')
    elif name == 'mlp_nobias':
        layers, P = qo.mlp_layers(3, 1, (6,), False, 'tanh')
    elif name == 'mlp_o2':
        layers, P = qo.mlp_layers(3, 2, (5, 4), True, 'tanh')
    elif name == 'mlp_exp':
        layers, P = qo.mlp_layers(2, 1, (5,), True, 'tanh')
    elif name == 'rnet_poly0':
        layers, P = qo.rnet_layers(3, 3, 1, 1, shared=True)
    elif name == 'rnet_lin':
        layers, P = qo.rnet_layers(4, 2, 2, 1, poly_order=1)
    elif name == 'rnet_quad':
        layers, P = qo.rnet_layers(3, 3, 1, 2, poly_order=2)
    elif name == 'rnet_mlp':
        layers, P = qo.rnet_layers(4, 2, 2, 1, mlp=True, shared=False)
    else:
        raise KeyError(name)
    return layers, P, ('exp' if name == 'mlp_exp' else None)


CASES = ['mlp_tanh', 'mlp_relu', 'mlp_identity', 'mlp_nobias', 'mlp_o2', 'mlp_exp', 'rnet_poly0', 'rnet_lin',
         'rnet_quad', 'rnet_mlp']


def case_data(name, N=13, seed=0):
    """Inputs of a case: x, y, theta, sigma, fulldatasize and a prior (shared with tests/test_gpu_hessian.py)."""
    layers, P, final = _case(name)
    rs = np.random.RandomState(seed + sum(map(ord, name)))
    indim, outdim = layers[0]['n_in'], layers[-1]['n_out']
    x = rs.rand(N, indim) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True) * np.arange(1, outdim + 1)) + 0.1 * rs.randn(N, outdim)
    if final == 'exp':
        y = np.exp(y)
    theta = 0.6 * rs.randn(P)
    prior = dict(sigma=0.7, anchor=0.3 * rs.randn(P))
    return layers, P, final, x, y, theta, 0.3, 3 * N + 1, prior


def _relu_off_kinks(layers, theta, x):
    """min |z| over the relu pre-activations: the Hessian is only defined away from z = 0"""
    h, m = np.asarray(x), np.inf
    for L in layers:
        W, b = qo._layer_wb(L, theta)
        z = h @ W.T + (b if b is not None else 0.0)
        if L['act'] == 'relu':
            m = min(m, np.abs(z).min())
        a = qo._act(L['act'], z)
        h = h + L['res_step'] * a if L['res_step'] != 0.0 else a
    return m


@pytest.mark.parametrize('with_prior', [False, True])
@pytest.mark.parametrize('name', CASES)
def test_oracle_hvp_matches_torch_autograd(name, with_prior):
    layers, P, final, x, y, theta, sigma, nfull, prior = case_data(name)
    prior = prior if with_prior else None
    if name == 'mlp_relu':
        assert _relu_off_kinks(layers, theta, x) > 1e-3
    f = _torch_neg_log_post(layers, x, y, sigma, nfull, prior, final)
    H_loss = torch.autograd.functional.hessian(f, torch.as_tensor(theta)).numpy()
    rs = np.random.RandomState(1)
    V = rs.randn(3, P)
    hv = logpost_hvp(layers, theta, x, y, sigma, nfull, prior, final, V)
    ref = -(V @ H_loss.T)
    np.testing.assert_allclose(hv, ref, rtol=0, atol=1e-10 * np.abs(ref).max())
    H = logpost_hessian(layers, theta, x, y, sigma, nfull, prior, final)
    np.testing.assert_allclose(H, -H_loss, rtol=0, atol=1e-10 * np.abs(H_loss).max())


def test_oracle_hvp_is_the_derivative_of_the_oracle_gradient():
    layers, P, final, x, y, theta, sigma, nfull, prior = case_data('rnet_quad')
    v = np.random.RandomState(2).randn(P)
    h = 1e-5
    gp = qo.logpost_grad(layers, theta + h * v, x, y, sigma, nfull, prior, final)[1]
    gm = qo.logpost_grad(layers, theta - h * v, x, y, sigma, nfull, prior, final)[1]
    hv = logpost_hvp(layers, theta, x, y, sigma, nfull, prior, final, v)
    np.testing.assert_allclose((gp - gm) / (2 * h), hv, rtol=0, atol=1e-7 * np.abs(hv).max())


# ---- launch plan of kernel 5 (host code only: no device needed) ----------------------------------------------------

def _lib():
    from quinn_b200 import _lib as L
    return L.load()


def _plan(layers, P, dtype, K=64, N=10000, final_exp=False):
    desc = netdesc_from_layers(layers, P, final_exp)
    out = (ctypes.c_int64 * 8)()
    net = desc.to_c()
    rc = _lib().qb_hvp_plan_info(ctypes.byref(net), dtype, K, N, out)
    ws = _lib().qb_hvp_workspace_bytes(ctypes.byref(net), dtype, K, N)
    return rc, list(out[:5]), ws


REQUIRED = {
    'rnet_c1': lambda: qo.rnet_layers(3, 3, 1, 1, shared=True),
    'mlp_c2': lambda: qo.mlp_layers(2, 1, (32, 32), True, 'tanh'),
    'mlp_c5': lambda: qo.mlp_layers(3, 1, (64, 64), True, 'tanh'),
    'mlp_c5_o4_relu': lambda: qo.mlp_layers(3, 4, (64, 64), True, 'relu'),
}


@pytest.mark.parametrize('dtype', [F32, F64])
@pytest.mark.parametrize('name', sorted(REQUIRED))
def test_hvp_plan_fits_the_required_networks(name, dtype):
    layers, P = REQUIRED[name]()
    for K, N in ((1, 10000), (P, 10000), (P, 7), (3, 1)):
        rc, (TM, threads, smem, S, blocks), ws = _plan(layers, P, dtype, K, N)
        assert rc == 0, _lib().qb_last_error()
        assert 0 < smem <= SMEM_MAX
        assert threads % 32 == 0 and 64 <= threads <= 256
        assert TM % 4 == 0 and TM >= (16 if dtype == F32 else 8)
        assert blocks == K * S and S >= 1
        assert (S - 1) * TM < N or S == 1             # every split has points
        assert ws == (K * S * P * (8 if dtype == F64 else 4) if S > 1 else 0)
        assert ws <= 256 << 20


def test_hvp_split_workspace_is_capped():
    layers, P = REQUIRED['mlp_c5']()
    rc, (TM, threads, smem, S, blocks), ws = _plan(layers, P, F64, K=1, N=10 ** 7)
    assert rc == 0 and S > 1 and ws <= 256 << 20


@pytest.mark.parametrize('dtype', [F32, F64])
def test_hvp_refuses_a_network_beyond_shared_memory(dtype):
    layers, P = qo.mlp_layers(10, 1, (128, 128), True, 'tanh')        # config 3 / 4: fits in neither precision
    rc, _, ws = _plan(layers, P, dtype)
    assert rc != 0 and ws == 0
    assert b'227 KB' in _lib().qb_last_error()


def test_hvp_leaves_the_other_plans_alone():
    """qb_plan_info of kernels 1-4 (every field) equals what the library gave before kernel 5, for every golden net"""
    import json
    import os
    from golden_util import GOLDEN, NET_CASES, NET_CASES_R2, netdesc_from_spec
    ref = json.load(open(os.path.join(GOLDEN, 'plan_info_k1to4.json')))['plans']
    specs = {**NET_CASES, **NET_CASES_R2}
    assert len(ref) == 4 * len(specs)
    for key, want in ref.items():
        name, dtype, grad = key.split('/')
        net = netdesc_from_spec(specs[name]).to_c()
        out = (ctypes.c_int64 * 8)()
        assert _lib().qb_plan_info(ctypes.byref(net), int(dtype), 256, 10000, int(grad), out) == 0
        assert list(out) == want, key
