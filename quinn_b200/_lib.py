"""ctypes binding of include/quinn_b200.h -- the only way Python reaches the CUDA kernels.

There is no CPU fallback: if the shared library is missing it is built with nvcc; if that fails, or a
call returns an error, a RuntimeError is raised.
"""
import ctypes as C
import os

from . import build as _build

QB_MAX_LAYERS = 16
QB_F32, QB_F64 = 0, 1
QB_ACT_IDENTITY, QB_ACT_TANH, QB_ACT_RELU = 0, 1, 2
QB_RNG_PHILOX, QB_RNG_REPLAY = 0, 1
QB_ADAPT_NONE, QB_ADAPT_DIAG, QB_ADAPT_FULL = 0, 1, 2


QB_MAX_TERMS = 6


class qb_layer_t(C.Structure):
    _fields_ = [('n_in', C.c_int32), ('n_out', C.c_int32), ('w_off', C.c_int32), ('b_off', C.c_int32),
                ('act', C.c_int32), ('n_terms', C.c_int32), ('res_step', C.c_double),
                ('w_stride', C.c_int32), ('b_stride', C.c_int32), ('coef', C.c_double * QB_MAX_TERMS)]


class qb_net_t(C.Structure):
    _fields_ = [('n_layers', C.c_int32), ('in_dim', C.c_int32), ('out_dim', C.c_int32), ('n_params', C.c_int32),
                ('final_exp', C.c_int32), ('reserved', C.c_int32 * 3), ('layers', qb_layer_t * QB_MAX_LAYERS)]


class qb_lik_t(C.Structure):
    _fields_ = [('sigma', C.c_double), ('prior_sigma', C.c_double), ('prior_scale', C.c_double),
                ('prior_anchor', C.c_void_p), ('anchor_per_chain', C.c_int32), ('reserved', C.c_int32)]


class qb_data_t(C.Structure):
    _fields_ = [('x', C.c_void_p), ('y', C.c_void_p), ('n', C.c_int64)]


class qb_chain_t(C.Structure):
    _fields_ = [('K', C.c_int64), ('theta', C.c_void_p), ('lp', C.c_void_p), ('naccept', C.c_void_p),
                ('map_theta', C.c_void_p), ('map_lp', C.c_void_p)]


class qb_rng_t(C.Structure):
    _fields_ = [('mode', C.c_int32), ('reserved', C.c_int32), ('seed', C.c_uint64), ('chain_offset', C.c_int64),
                ('incr', C.c_void_p), ('unif', C.c_void_p)]


class qb_record_t(C.Structure):
    _fields_ = [('logpost', C.c_void_p), ('alpha', C.c_void_p), ('accepted', C.c_void_p), ('ld', C.c_int64),
                ('samples', C.c_void_p), ('store_every', C.c_int64), ('n_slots', C.c_int64), ('logpost0', C.c_void_p)]


class qb_amcmc_t(C.Structure):
    _fields_ = [('gamma', C.c_double), ('t0', C.c_int64), ('tadapt', C.c_int64), ('adapt', C.c_int32),
                ('track_moments', C.c_int32), ('xm', C.c_void_p), ('cov', C.c_void_p), ('pscale', C.c_void_p),
                ('chol', C.c_void_p), ('chol_ini', C.c_void_p), ('prop_kind', C.c_void_p)]


class qb_hmc_t(C.Structure):
    _fields_ = [('method', C.c_int32), ('L', C.c_int32), ('epsilon', C.c_double), ('grad_cur', C.c_void_p),
                ('mom', C.c_void_p), ('prop', C.c_void_p), ('grad_prop', C.c_void_p)]


QB_ABI_VERSION = 204          # include/quinn_b200.h
ABI_STRUCTS = (qb_layer_t, qb_net_t, qb_lik_t, qb_data_t, qb_chain_t, qb_rng_t, qb_record_t, qb_amcmc_t, qb_hmc_t)

# every symbol include/quinn_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    'qb_last_error': (C.c_char_p, []),
    'qb_version': (C.c_int, []),
    'qb_struct_sizes': (C.c_int, [C.POINTER(C.c_int64), C.c_int]),
    'qb_eval_workspace_bytes': (C.c_size_t, [C.POINTER(qb_net_t), C.c_int, C.c_int64, C.c_int64, C.c_int]),
    'qb_logpost': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, C.c_int64, C.POINTER(qb_data_t), C.POINTER(qb_lik_t),
                             _P, _P, C.c_size_t, _P]),
    'qb_logpost_grad': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, C.c_int64, C.POINTER(qb_data_t),
                                  C.POINTER(qb_lik_t), _P, _P, _P, C.c_size_t, _P]),
    'qb_logpost_members': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, C.c_int64, C.POINTER(qb_data_t), C.c_int64, C.c_int64,
                                     C.POINTER(qb_lik_t), _P, _P, _P, C.c_size_t, _P]),
    'qb_hvp_workspace_bytes': (C.c_size_t, [C.POINTER(qb_net_t), C.c_int, C.c_int64, C.c_int64]),
    'qb_logpost_hvp': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, _P, C.c_int64, C.c_int64, C.POINTER(qb_data_t),
                                 C.POINTER(qb_lik_t), _P, _P, C.c_size_t, _P]),
    'qb_hvp_plan_info': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.c_int64, C.c_int64, C.POINTER(C.c_int64)]),
    'qb_kfac_workspace_bytes': (C.c_size_t, [C.POINTER(qb_net_t), C.c_int, C.c_int64]),
    'qb_logpost_kfac': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, C.POINTER(qb_data_t), C.POINTER(qb_lik_t), _P, _P,
                                  C.c_size_t, _P]),
    'qb_kfac_plan_info': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.c_int64, C.POINTER(C.c_int64)]),
    'qb_predict_jac': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, _P, C.c_int64, _P, _P, _P]),
    'qb_jac_plan_info': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.c_int64, C.POINTER(C.c_int64)]),
    'qb_adam_step': (C.c_int, [C.c_int, _P, _P, _P, _P, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double,
                               C.c_double, C.c_int64, C.c_double, _P]),
    'qb_copy_rows_where': (C.c_int, [C.c_int, _P, _P, _P, C.c_int64, C.c_int64, _P]),
    'qb_amcmc_run': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.POINTER(qb_data_t), C.POINTER(qb_lik_t),
                               C.POINTER(qb_chain_t), C.POINTER(qb_amcmc_t), C.POINTER(qb_rng_t),
                               C.POINTER(qb_record_t), C.c_int64, C.c_int64, C.c_int, _P, _P]),
    'qb_hmc_run': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.POINTER(qb_data_t), C.POINTER(qb_lik_t),
                             C.POINTER(qb_chain_t), C.POINTER(qb_hmc_t), C.POINTER(qb_rng_t),
                             C.POINTER(qb_record_t), C.c_int64, C.c_int64, C.c_int, _P]),
    'qb_nuts_run': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.POINTER(qb_data_t), C.POINTER(qb_lik_t),
                              C.POINTER(qb_chain_t), C.POINTER(qb_rng_t), C.POINTER(qb_record_t), C.c_int64, C.c_int64,
                              C.c_int, C.c_double, C.c_int, C.c_int64, C.c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'qb_pt_run': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.POINTER(qb_data_t), C.POINTER(qb_lik_t), C.POINTER(qb_chain_t),
                            C.POINTER(qb_hmc_t), C.POINTER(qb_rng_t), C.POINTER(qb_record_t), C.c_int64, C.c_int64, C.c_int,
                            C.c_int64, _P, _P, C.c_int64, _P, _P, _P, _P, _P, _P]),
    'qb_predict': (C.c_int, [C.POINTER(qb_net_t), C.c_int, _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P]),
    'qb_vi_sample': (C.c_int, [C.c_int, _P, _P, _P, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_double,
                               C.c_uint64, C.c_uint64, _P, _P, _P, _P]),
    'qb_vi_backward': (C.c_int, [C.c_int, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_double, C.c_double,
                                 C.c_double, C.c_double, C.c_double, C.c_double, _P, _P, _P]),
    'qb_swag_step': (C.c_int, [C.c_int, _P, _P, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int64, _P, _P, _P,
                               C.c_int64, _P]),
    'qb_swag_sample': (C.c_int, [C.c_int, _P, _P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, _P, C.c_int64,
                                 C.c_uint64, C.c_int64, C.c_double, _P, _P]),
    'qb_fma_peak': (C.c_int, [C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_double), _P, _P]),
    'qb_plan_info': (C.c_int, [C.POINTER(qb_net_t), C.c_int, C.c_int64, C.c_int64, C.c_int, C.POINTER(C.c_int64)]),
    'qb_launch_count': (C.c_int64, []),
    'qb_row_moments': (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P, _P]),
    'qb_ess': (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P]),
    'qb_colsq_mean': (C.c_int, [C.c_int, _P, C.c_int64, C.c_int64, _P, _P]),
    'qb_quantiles': (C.c_int, [C.c_int, _P, C.c_int64, C.c_int64, C.POINTER(C.c_double), C.c_int, _P, _P]),
}

_lib = None


def lib_path():
    # QB_LIB: development aid for A/B timing of two builds in one GPU session
    return os.environ.get('QB_LIB') or _build.OUT


def load(build_if_missing=True):
    """Load (building first if needed) libquinn_b200.so and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    # build only when the library is absent: a stale-looking mtime must not trigger a multi-minute nvcc run inside
    # every rank of a job (rebuild explicitly with `python -m quinn_b200.build` / __graft_entry__.build())
    if build_if_missing and not os.environ.get('QB_LIB') and not os.path.exists(path):
        if os.path.exists('/usr/local/cuda/bin/nvcc') or os.environ.get('NVCC'):
            _build.build()
    if not os.path.exists(path):
        raise RuntimeError(f'quinn_b200: CUDA library {path} is missing and could not be built; '
                           'there is no CPU fallback (run `python -m quinn_b200.build`)')
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    # ABI guard: a stale library with other struct layouts would be called with mismatched structs and corrupt memory
    if lib.qb_version() != QB_ABI_VERSION:
        raise RuntimeError(f'quinn_b200: {path} has ABI version {lib.qb_version()}, this binding expects {QB_ABI_VERSION}; '
                           'rebuild with `python -m quinn_b200.build --force`')
    sizes = (C.c_int64 * len(ABI_STRUCTS))()
    n = lib.qb_struct_sizes(sizes, len(ABI_STRUCTS))
    mine = [C.sizeof(t) for t in ABI_STRUCTS]
    if n != len(ABI_STRUCTS) or list(sizes) != mine:
        raise RuntimeError(f'quinn_b200: struct sizes of {path} {list(sizes)} differ from the ctypes mirrors {mine}')
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().qb_last_error()
        raise RuntimeError(f'quinn_b200: {what} failed (rc={rc}): {msg.decode() if msg else ""}')
