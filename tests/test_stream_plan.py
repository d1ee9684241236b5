"""CPU-only checks of the layer-streamed launch plan (quinn_b200/csrc/qb_stream.cuh): networks whose weights do not fit
in shared memory next to one tile of activations are planned on the streamed kernels (qb_plan_info code 5), everything
that fitted before keeps its kernel, and a network whose single smallest tile of activations does not fit is refused."""
import ctypes

import pytest

from golden_util import NET_CASES, NET_CASES_R2, netdesc_from_layers, netdesc_from_spec

F32, F64 = 0, 1
SMEM_MAX = 227 * 1024


def _lib():
    from quinn_b200 import _lib as L
    lib = L.load()
    lib.qb_last_error.restype = ctypes.c_char_p
    return lib


def _mlp(indim, outdim, hls, activ='tanh', final_exp=False):
    from oracle import quinn_oracle as qo
    layers, P = qo.mlp_layers(indim, outdim, hls, True, activ)
    return netdesc_from_layers(layers, P, final_exp)


def _rnet(rdim, nlayers, indim, outdim, poly):
    from oracle import quinn_oracle as qo
    layers, P = qo.rnet_layers(rdim, nlayers, indim, outdim, poly_order=poly)
    return netdesc_from_layers(layers, P)


def _info(desc, dtype, grad, K=256, N=10000):
    out = (ctypes.c_int64 * 8)()
    net = desc.to_c()
    rc = _lib().qb_plan_info(ctypes.byref(net), dtype, K, N, grad, out)
    return rc, list(out)


# the networks of the streamed path: (name, descriptor factory, P, dtypes that need streaming)
STREAMED = [
    ('mlp_160x2', lambda: _mlp(10, 1, (160, 160)), 27681, (F64,)),
    ('mlp_100x4', lambda: _mlp(10, 1, (100, 100, 100, 100)), 31501, (F64,)),
    ('mlp_128x3', lambda: _mlp(10, 1, (128, 128, 128)), 34561, (F64,)),
    ('rnet_128_poly1', lambda: _rnet(128, 3, 10, 1, 1), 34561, (F32, F64)),
    ('mlp_256x2', lambda: _mlp(10, 1, (256, 256)), 68865, (F32, F64)),
    ('mlp_512x2', lambda: _mlp(10, 1, (512, 512)), 268801, (F32, F64)),
    ('mlp_256x3_relu_o2', lambda: _mlp(5, 2, (256, 256, 256), 'relu'), None, (F32, F64)),
    ('mlp_512x2_exp', lambda: _mlp(3, 1, (512, 512), final_exp=True), None, (F32, F64)),
    ('rnet_256_poly0', lambda: _rnet(256, 2, 10, 1, None), None, (F32, F64)),
]

# qb_plan_info code (out[6]) of every golden network before the streamed path existed, per (dtype, want_grad):
# [f32 value, f32 grad, f64 value, f64 grad]
RESIDENT_CODES = {
    'mlp_tanh_o2': [0, 0, 0, 0], 'mlp_relu': [0, 0, 0, 0], 'mlp_lin_nob': [0, 0, 0, 0],
    'mlp_c2': [2, 4, 0, 0], 'mlp_c5': [2, 4, 0, 0], 'mlp_c3': [2, 4, 0, 0],
    'rnet_c1': [0, 0, 0, 0], 'rnet_nonpar': [0, 0, 0, 0], 'rnet_mlpmode': [0, 0, 0, 0],
    'rnet_lin': [0, 0, 0, 0], 'rnet_quad': [0, 0, 0, 0], 'rnet_cubic': [0, 0, 0, 0], 'rnet_poly4': [0, 0, 0, 0],
}


@pytest.mark.parametrize('name,make,P,streamed', STREAMED, ids=[s[0] for s in STREAMED])
def test_large_networks_plan_on_the_streamed_path(name, make, P, streamed):
    desc = make()
    if P is not None:
        assert desc.n_params == P
    for dtype in (F32, F64):
        for grad in (0, 1):
            for K, N in ((256, 10000), (2, 10000), (2048, 1000), (1, 5)):
                rc, out = _info(desc, dtype, grad, K, N)
                assert rc == 0, _lib().qb_last_error()
                if dtype in streamed:
                    assert out[6] == 5, (dtype, grad, out)
                    assert out[0] in (8, 16, 32, 64, 128) and out[1] == 256 and 0 < out[2] <= SMEM_MAX, out
                    assert out[3] >= 1 and out[4] == K * out[3]
                    if grad and out[3] > 1:                # partial gradient rows [K, S, P] stay bounded
                        assert K * out[3] * desc.n_params * (8 if dtype == F64 else 4) <= 256 << 20
                else:
                    assert out[6] != 5, (dtype, grad, out)


def test_config3_net_stays_resident():
    # MLP(10,1,(128,128)) (configs 3/4) fits in both dtypes: never streamed
    desc = _mlp(10, 1, (128, 128))
    assert desc.n_params == 18049
    for dtype in (F32, F64):
        for grad in (0, 1):
            rc, out = _info(desc, dtype, grad)
            assert rc == 0 and out[6] != 5


@pytest.mark.parametrize('name', list(RESIDENT_CODES))
def test_resident_networks_keep_their_kernel(name):
    spec = {**NET_CASES, **NET_CASES_R2}[name]
    desc = netdesc_from_spec(spec)
    for dtype in (F32, F64):
        for grad in (0, 1):
            for K, N in ((256, 10000), (2, 10000), (4096, 500)):
                rc, out = _info(desc, dtype, grad, K, N)
                assert rc == 0
                assert out[6] == RESIDENT_CODES[name][2 * dtype + grad], (dtype, grad, K, N, out)


def test_too_wide_for_one_tile_is_refused():
    desc = _mlp(10, 1, (8192, 8192))
    for dtype in (F32, F64):
        for grad in (0, 1):
            rc, _ = _info(desc, dtype, grad)
            assert rc != 0
            err = _lib().qb_last_error().decode()
            assert 'activations of one' in err and 'tile' in err and 'weights' not in err, err
    net = desc.to_c()
    assert _lib().qb_eval_workspace_bytes(ctypes.byref(net), F64, 4, 1000, 1) == 0


@pytest.mark.parametrize('name,make,P,streamed', STREAMED, ids=[s[0] for s in STREAMED])
def test_workspace_is_sized_for_the_streamed_path(name, make, P, streamed):
    lib = _lib()
    lib.qb_eval_workspace_bytes.restype = ctypes.c_size_t
    desc = make()
    net = desc.to_c()
    for dtype in streamed:
        elem = 8 if dtype == F64 else 4
        for grad in (0, 1):
            for K in (1, 4, 256, 2048):
                nb = lib.qb_eval_workspace_bytes(ctypes.byref(net), dtype, K, 10000, grad)
                _, out = _info(desc, dtype, grad, K, 10000)
                S = out[3]
                assert nb >= K * S * 8
                if grad and S > 1:
                    assert nb >= K * S * 8 + K * S * desc.n_params * elem
