"""CPU checks of the Kronecker-factored curvature: the numpy oracle (tests/kfac_oracle.py) against torch autograd's
per-point gradients, and the launch plan of kernel 6 (qb_kfac_plan_info, qb_kfac_workspace_bytes)."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from golden_util import GOLDEN, netdesc_from_layers
from kfac_oracle import factors, layer_index, per_point
from oracle import quinn_oracle as qo
from test_hessian_cpu import CASES, _torch_neg_log_post, case_data

F32, F64 = 0, 1
SMEM_MAX = 227 * 1024
REFUSED = {'rnet_poly0': b'shares its weights', 'rnet_lin': b'polynomial', 'rnet_quad': b'polynomial'}
SUPPORTED = [c for c in CASES if c not in REFUSED]


@pytest.mark.parametrize('name', SUPPORTED)
def test_oracle_outer_products_are_the_per_point_gradients(name):
    """outer(delta_i, a~_i) = d log p_i / d [W | b] of every layer, for every point (torch autograd, float64)"""
    layers, P, final, x, y, theta, sigma, *_ = case_data(name)
    pp = per_point(layers, theta, x, y, sigma, final)
    for i in range(x.shape[0]):
        f = _torch_neg_log_post(layers, x[i:i + 1], y[i:i + 1], sigma, 1, None, final)
        th = torch.as_tensor(theta).requires_grad_(True)
        g = -torch.autograd.grad(f(th), th)[0].numpy()
        for L, (at, d) in zip(layers, pp):
            ref = g[layer_index(L)]
            got = np.outer(d[i], at[i])
            assert np.abs(got - ref).max() <= 1e-12 * max(np.abs(ref).max(), 1e-300), (name, i)
    fs = factors(layers, theta, x, y, sigma, final)
    for L, (at, d), f in zip(layers, pp, fs):
        a = at[:, :L['n_in']]
        np.testing.assert_allclose(f['A'], sum(np.outer(r, r) for r in a), rtol=1e-13, atol=1e-13)
        np.testing.assert_allclose(f['G'], sum(np.outer(r, r) for r in d), rtol=1e-13, atol=1e-13)


# ---- launch plan of kernel 6 (host code only: no device needed) ----------------------------------------------------

def _lib():
    from quinn_b200 import _lib as L
    return L.load()


def _plan(layers, P, dtype, N=10000, final_exp=False):
    desc = netdesc_from_layers(layers, P, final_exp)
    out = (ctypes.c_int64 * 8)()
    net = desc.to_c()
    rc = _lib().qb_kfac_plan_info(ctypes.byref(net), dtype, N, out)
    ws = _lib().qb_kfac_workspace_bytes(ctypes.byref(net), dtype, N)
    return rc, list(out[:5]), ws, desc


def _n_factors(layers):
    return sum(L['n_in'] ** 2 + (L['n_in'] if L['b_off'] >= 0 else 0) + L['n_out'] ** 2 for L in layers)


NETS = {
    'mlp_c2': lambda: qo.mlp_layers(2, 1, (32, 32), True, 'tanh'),
    'mlp_c5': lambda: qo.mlp_layers(3, 1, (64, 64), True, 'tanh'),
    'mlp_c5_o4_relu': lambda: qo.mlp_layers(3, 4, (64, 64), True, 'relu'),
    'mlp_c34': lambda: qo.mlp_layers(10, 1, (128, 128), True, 'tanh'),
    'mlp_nobias': lambda: qo.mlp_layers(3, 1, (6,), False, 'tanh'),
}


@pytest.mark.parametrize('dtype', [F32, F64])
@pytest.mark.parametrize('name', sorted(NETS))
def test_kfac_plan_and_factor_offsets(name, dtype):
    from quinn_b200 import ops
    layers, P = NETS[name]()
    elem = 8 if dtype == F64 else 4
    for N in (10000, 100000, 7, 1):
        rc, (TM, threads, smem, S, F), ws, desc = _plan(layers, P, dtype, N)
        assert rc == 0, _lib().qb_last_error()
        assert 0 < smem <= SMEM_MAX and threads % 32 == 0 and 64 <= threads <= 256
        assert F == _n_factors(layers)
        assert S >= 1 and ((S - 1) * TM < N or S == 1)
        assert ws == S * F * elem and ws <= 256 << 20
    # [A_l | s_l | G_l] layer by layer
    lay = ops.kfac_layout(desc)
    off = 0
    for L, (n_in, n_out, bias, a_off, s_off, g_off) in zip(layers, lay):
        assert (n_in, n_out, bias) == (L['n_in'], L['n_out'], L['b_off'] >= 0)
        assert a_off == off
        off += n_in * n_in
        assert s_off == (off if bias else -1)
        off += n_in if bias else 0
        assert g_off == off
        off += n_out * n_out
    assert off == F


@pytest.mark.parametrize('dtype', [F32, F64])
def test_kfac_split_rows_are_capped_at_256_mb(dtype):
    layers, P = NETS['mlp_c34']()
    elem = 8 if dtype == F64 else 4
    rc, (TM, threads, smem, S, F), ws, _ = _plan(layers, P, dtype, N=10 ** 7)
    assert rc == 0 and S > 1
    cap = (256 << 20) // (F * elem)
    assert cap // 2 < S <= cap and ws == S * F * elem <= 256 << 20


@pytest.mark.parametrize('name', sorted(REFUSED))
def test_kfac_refuses_shared_and_polynomial_weights(name):
    from test_hessian_cpu import _case
    layers, P, _ = _case(name)
    for dtype in (F32, F64):
        rc, _, ws, _ = _plan(layers, P, dtype)
        assert rc != 0 and ws == 0
        assert REFUSED[name] in _lib().qb_last_error()


def test_kfac_refuses_a_streamed_network():
    layers, P = qo.mlp_layers(10, 1, (256, 256), True, 'tanh')
    desc = netdesc_from_layers(layers, P)
    net = desc.to_c()
    out = (ctypes.c_int64 * 8)()
    assert _lib().qb_plan_info(ctypes.byref(net), F64, 1, 10000, 1, out) == 0 and out[6] == 5     # kernel 2: streamed
    rc, _, ws, _ = _plan(layers, P, F64)
    assert rc != 0 and ws == 0
    assert b'layer-streamed' in _lib().qb_last_error()


def test_kfac_leaves_the_kernel5_plans_alone():
    """qb_hvp_plan_info of the Hessian-vector kernel equals what the library gave before kernel 6 (kernels 1-4:
    test_hessian_cpu.test_hvp_leaves_the_other_plans_alone)"""
    from test_hessian_cpu import REQUIRED
    ref = json.load(open(os.path.join(GOLDEN, 'plan_info_k5.json')))['plans']
    assert len(ref) == 2 * 4 * len(REQUIRED)
    for key, want in ref.items():
        name, dtype, K, N = key.split('/')
        layers, P = REQUIRED[name]()
        net = netdesc_from_layers(layers, P).to_c()
        out = (ctypes.c_int64 * 8)()
        K = P if K == 'P' else int(K)
        assert _lib().qb_hvp_plan_info(ctypes.byref(net), int(dtype), K, int(N), out) == 0
        assert list(out[:5]) == want, key
