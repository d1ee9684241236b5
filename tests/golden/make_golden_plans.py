#!/usr/bin/env python
"""Record the launch plans of kernels 1, 2, 5 and 6 (host code only, no device needed):

    python tests/golden/make_golden_plans.py

  plan_info_all.json   for every golden, streamed and config-3/4 network in fp32 and fp64: qb_plan_info and
                       qb_eval_workspace_bytes (value and gradient) over a grid of (K, N), qb_hvp_plan_info and
                       qb_hvp_workspace_bytes, qb_kfac_plan_info and qb_kfac_workspace_bytes; for a refused call the return
                       code and the error text; a few networks again under the kernel-selection and tiling overrides.

The values hold for a 148-SM device (B200), which is also what the planner assumes when no device is visible.
tests/test_launch_plan_cpu.py recomputes every entry with the current library and compares.
"""
import ctypes
import json
import os
import sys
from contextlib import contextmanager

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
for _p in (os.path.dirname(TESTS), TESTS):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from golden_util import NET_CASES, NET_CASES_R2, netdesc_from_spec     # noqa: E402
from test_stream_plan import STREAMED, _mlp                             # noqa: E402

OUT = os.path.join(HERE, 'plan_info_all.json')
F32, F64 = 0, 1
EVAL_KN = [(1, 1), (1, 7), (3, 10 ** 4), (256, 10 ** 4), (10 ** 5, 10 ** 4), (1, 10 ** 7)]
HVP_KN = [(1, 10 ** 4), ('P', 10 ** 4), (3, 1)]
KFAC_N = [0, 1, 10 ** 4, 10 ** 7]
SWITCHES = [('QB_NO_TC', '1'), ('QB_NO_TCG', '1'), ('QB_TG8_64', '0'), ('QB_SPLIT', '3'), ('QB_TM', '64')]
SWITCH_NETS = ['mlp_tanh_o2', 'mlp_c2', 'mlp_c5', 'mlp_c3', 'rnet_c1', 'mlp_256x2']
SWITCH_KN = [(3, 10 ** 4), (256, 10 ** 4)]


def nets():
    """name -> NetDesc: the golden nets (mlp_c3 is the config-3/4 net, 10-128-128-1 tanh), the streamed nets, and one
    net too wide for a single tile of activations"""
    d = {name: netdesc_from_spec(spec) for name, spec in {**NET_CASES, **NET_CASES_R2}.items()}
    d.update({name: make() for name, make, _, _ in STREAMED})
    d['mlp_8192x2'] = _mlp(10, 1, (8192, 8192))
    return d


def _lib():
    from quinn_b200 import _lib as L
    return L.load()


def _call(fn, ws_fn):
    """[rc, workspace bytes, out[0..8)] or [rc, workspace bytes, error text]"""
    out = (ctypes.c_int64 * 8)(*([-1] * 8))
    rc = fn(out)
    ws = ws_fn()
    return [rc, ws, list(out)] if rc == 0 else [rc, ws, _lib().qb_last_error().decode()]


@contextmanager
def env(name, value):
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        yield
    finally:
        if old is None:
            del os.environ[name]
        else:
            os.environ[name] = old


def _eval(lib, net, dtype, K, N, grad):
    return _call(lambda o: lib.qb_plan_info(ctypes.byref(net), dtype, K, N, grad, o),
                 lambda: lib.qb_eval_workspace_bytes(ctypes.byref(net), dtype, K, N, grad))


def _hvp(lib, net, dtype, K, N):
    return _call(lambda o: lib.qb_hvp_plan_info(ctypes.byref(net), dtype, K, N, o),
                 lambda: lib.qb_hvp_workspace_bytes(ctypes.byref(net), dtype, K, N))


def _kfac(lib, net, dtype, N):
    return _call(lambda o: lib.qb_kfac_plan_info(ctypes.byref(net), dtype, N, o),
                 lambda: lib.qb_kfac_workspace_bytes(ctypes.byref(net), dtype, N))


def record():
    """key -> entry; keys: eval/net/dtype/grad/K/N, hvp/net/dtype/K/N, kfac/net/dtype/N, args/..., env=value/..."""
    lib = _lib()
    all_nets = nets()
    cnets = {name: d.to_c() for name, d in all_nets.items()}
    r = {}
    for name, net in cnets.items():
        P = all_nets[name].n_params
        for dtype in (F32, F64):
            for grad in (0, 1):
                for K, N in EVAL_KN:
                    r[f'eval/{name}/{dtype}/{grad}/{K}/{N}'] = _eval(lib, net, dtype, K, N, grad)
            for K, N in HVP_KN:
                r[f'hvp/{name}/{dtype}/{K}/{N}'] = _hvp(lib, net, dtype, P if K == 'P' else K, N)
            for N in KFAC_N:
                r[f'kfac/{name}/{dtype}/{N}'] = _kfac(lib, net, dtype, N)
    net = cnets['mlp_c5']
    for dtype, K, N in ((2, 4, 100), (F32, 0, 100), (F32, 4, 0), (F64, -1, 100)):
        r[f'args/eval/{dtype}/{K}/{N}'] = _eval(lib, net, dtype, K, N, 1)
        r[f'args/hvp/{dtype}/{K}/{N}'] = _hvp(lib, net, dtype, K, N)
    r['args/kfac/2/100'] = _kfac(lib, net, 2, 100)
    for var, val in SWITCHES:
        with env(var, val):
            for name in SWITCH_NETS:
                net = cnets[name]
                for dtype in (F32, F64):
                    for grad in (0, 1):
                        for K, N in SWITCH_KN:
                            r[f'{var}={val}/eval/{name}/{dtype}/{grad}/{K}/{N}'] = _eval(lib, net, dtype, K, N, grad)
                    r[f'{var}={val}/hvp/{name}/{dtype}/1/10000'] = _hvp(lib, net, dtype, 1, 10 ** 4)
                    r[f'{var}={val}/kfac/{name}/{dtype}/10000'] = _kfac(lib, net, dtype, 10 ** 4)
    return r


if __name__ == '__main__':
    plans = record()
    with open(OUT, 'w') as f:
        f.write('{\n"about": "launch plans of kernels 1, 2, 5 and 6 on 148 SMs: key -> [return code, workspace bytes, '
                'out[0..8) of the *_plan_info call or its error text]; recorded before the planners moved to qb_launch.cu",\n'
                '"plans": {\n')
        f.write(',\n'.join(f'{json.dumps(k)}: {json.dumps(v)}' for k, v in plans.items()))
        f.write('\n}\n}\n')
    print(len(plans), 'plans ->', OUT)
