"""CPU checks of the linearised (GLM) predictive: the numpy Jacobian oracle (tests/glm_oracle.py) against torch autograd,
NN_Laplace's assembly of J from kernel 7's per-layer pairs, and the launch plan of kernel 7 (qb_jac_plan_info)."""
import ctypes

import numpy as np
import pytest
import torch

from glm_oracle import assemble, jacobian, pairs
from golden_util import netdesc_from_layers
from oracle import quinn_oracle as qo
from test_hessian_cpu import CASES, case_data

F32, F64 = 0, 1
SMEM_MAX = 227 * 1024


def _torch_forward(layers, x, final):
    """the network's outputs as a function of the flat theta, in float64 torch"""
    x = torch.as_tensor(x)

    def f(th):
        h = x
        for L in layers:
            nw = L['n_in'] * L['n_out']
            terms = L.get('terms', [(1.0, L['w_off'], L['b_off'])])
            W = sum(c * th[wo:wo + nw].reshape(L['n_out'], L['n_in']) for c, wo, _ in terms)
            z = h @ W.T
            if L['b_off'] >= 0:
                z = z + sum(c * th[bo:bo + L['n_out']] for c, _, bo in terms)
            a = torch.tanh(z) if L['act'] == 'tanh' else (torch.relu(z) if L['act'] == 'relu' else z)
            h = h + L['res_step'] * a if L['res_step'] != 0.0 else a
        return torch.exp(h) if final == 'exp' else h
    return f


@pytest.mark.parametrize('name', CASES)
def test_oracle_jacobian_matches_torch_autograd(name):
    layers, P, final, x, y, theta, *_ = case_data(name)
    f, J = jacobian(layers, theta, x, final)
    fn = _torch_forward(layers, x, final)
    th = torch.as_tensor(theta)
    ref = torch.autograd.functional.jacobian(fn, th).numpy()          # [N, o, P]
    np.testing.assert_allclose(f, fn(th).numpy(), rtol=0, atol=1e-14 * np.abs(f).max())
    assert J.shape == ref.shape == (x.shape[0], layers[-1]['n_out'], P)
    assert np.abs(J - ref).max() <= 1e-12 * np.abs(ref).max(), name


@pytest.mark.parametrize('name', CASES)
def test_solver_assembly_reproduces_the_oracle_jacobian(name):
    from quinn_b200.solvers.nn_laplace import assemble_jac
    layers, P, final, x, y, theta, *_ = case_data(name)
    f, prs = pairs(layers, theta, x, final)
    desc = netdesc_from_layers(layers, P, final == 'exp')
    got = assemble_jac(desc, [dict(a=torch.as_tensor(p['a']), d=torch.as_tensor(p['d'])) for p in prs])
    ref = assemble(layers, P, prs)
    assert got.dtype == torch.float64 and not got.is_cuda
    np.testing.assert_allclose(got.numpy(), ref, rtol=0, atol=1e-14 * np.abs(ref).max())
    np.testing.assert_allclose(ref, jacobian(layers, theta, x, final)[1], rtol=0, atol=0)


# ---- launch plan of kernel 7 (host code only: no device needed) ----------------------------------------------------

def _lib():
    from quinn_b200 import _lib as L
    return L.load()


def _plan(layers, P, dtype, N, final_exp=False):
    net = netdesc_from_layers(layers, P, final_exp).to_c()
    out = (ctypes.c_int64 * 8)()
    rc = _lib().qb_jac_plan_info(ctypes.byref(net), dtype, N, out)
    return rc, list(out[:5])


NETS = {
    'mlp_c2': lambda: qo.mlp_layers(2, 1, (32, 32), True, 'tanh'),
    'mlp_c5': lambda: qo.mlp_layers(3, 1, (64, 64), True, 'tanh'),
    'mlp_c5_o4_relu': lambda: qo.mlp_layers(3, 4, (64, 64), True, 'relu'),
    'mlp_c34': lambda: qo.mlp_layers(10, 1, (128, 128), True, 'tanh'),
    'rnet_poly0': lambda: qo.rnet_layers(3, 3, 1, 1, shared=True),
    'rnet_quad': lambda: qo.rnet_layers(3, 3, 1, 2, poly_order=2),
}


@pytest.mark.parametrize('dtype', [F32, F64])
@pytest.mark.parametrize('name', sorted(NETS))
def test_jac_plan_rows_and_blocks(name, dtype):
    layers, P = NETS[name]()
    o = layers[-1]['n_out']
    F = sum(L['n_in'] + o * L['n_out'] for L in layers)
    for N in (10 ** 6, 10 ** 5, 10000, 7, 1):
        rc, (TM, threads, smem, blocks, rows) = _plan(layers, P, dtype, N)
        assert rc == 0, _lib().qb_last_error()
        assert rows == F
        assert 0 < smem <= SMEM_MAX and threads % 32 == 0 and 64 <= threads <= 256
        tiles = -(-N // TM)
        # runs of whole tiles: about 8 blocks per SM (148 SMs when no device is visible), at least two tiles each
        want = max(1, min(-(-N // (2 * TM)), 148 * 8))
        per = -(-tiles // want)
        assert blocks == -(-tiles // per)
        assert (blocks - 1) * per * TM < N <= blocks * per * TM
    rc, (TM, threads, smem, blocks, rows) = _plan(layers, P, dtype, 0)
    assert rc == 0 and blocks == 0 and rows == F


def test_jac_plan_refusals():
    layers, P = qo.mlp_layers(10, 1, (256, 256), True, 'tanh')
    net = netdesc_from_layers(layers, P).to_c()
    out = (ctypes.c_int64 * 8)()
    assert _lib().qb_plan_info(ctypes.byref(net), F64, 1, 10000, 1, out) == 0 and out[6] == 5     # kernel 2: streamed
    for dtype in (F32, F64):
        rc, _ = _plan(layers, P, dtype, 10000)
        assert rc != 0 and b'layer-streamed' in _lib().qb_last_error()
    layers, P = NETS['mlp_c5']()
    rc, _ = _plan(layers, P, F64, -1)
    assert rc != 0 and b'negative' in _lib().qb_last_error()
    assert _lib().qb_jac_plan_info(None, F64, 10, out) != 0 and b'NULL' in _lib().qb_last_error()
