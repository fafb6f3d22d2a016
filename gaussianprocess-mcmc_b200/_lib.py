"""ctypes binding of libgpmc.so (the C ABI declared in include/gpmc.h).

The library is built in-tree by ``build.py`` / ``__graft_entry__.build()``.  There is no CPU
fallback: if the shared object is missing, or a call is made without a CUDA device, this module
raises instead of computing anything on the host.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libgpmc.so')

KIND_SE_ISO, KIND_SE_ARD = 0, 1
KIND_MATERN1, KIND_MATERN3, KIND_MATERN5 = 2, 3, 4
ASM_ADD_S, ASM_LOWER_ONLY = 1, 2
JITTER_NONE, JITTER_PYGPS = 0, 1
INFO_NOT_PD = -1
OP_POTRF, OP_LOGLIK, OP_SDS, OP_LOGLIK_GRAD, OP_MARGINAL = 1, 2, 3, 4, 5
KC_NAMES = ('assemble', 'gemm_update', 'potf2', 'panel_trsm', 'solve_reduce', 'tri_inverse', 'syrk_R', 'vector_control',
            'band_clear', 'grad_contract')

_c_double_p = ctypes.c_void_p     # raw addresses (torch data_ptr() / numpy ctypes.data)
_vp = ctypes.c_void_p
_i = ctypes.c_int
_sz = ctypes.c_size_t

# name -> (restype, argtypes); every symbol include/gpmc.h declares
SIGNATURES = {
    'gpmc_version': (_i, []),
    'gpmc_panel_width': (_i, []),
    'gpmc_last_error': (ctypes.c_char_p, []),
    'gpmc_device_info': (_i, [ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_sz)]),
    'gpmc_workspace_bytes': (_sz, [_i, _i, _i, _i]),
    'gpmc_cov_assemble': (_i, [_vp, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    'gpmc_potrf_batched': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _sz, _vp]),
    'gpmc_loglik_batched': (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_loglik_grad_batched': (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_loglik_host': (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    'gpmc_sds_workspace_bytes': (_sz, [_i, _i, _i]),
    'gpmc_sds_sweep': (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i,
                            ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_ulonglong, ctypes.c_uint,
                            _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_sds_run': (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _i,
                          ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_ulonglong, ctypes.c_uint, _i, _i,
                          _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _sz, _vp]),
    'gpmc_marginal_run': (_i, [_vp, _i, _i, _vp, ctypes.c_double, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i,
                               ctypes.c_ulonglong, ctypes.c_uint, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_marginal_rounds': (_i, [_i, _vp, _vp]),
    'gpmc_aux_workspace_bytes': (_sz, [_i]),
    'gpmc_aux_var_model': (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_trsv_lower_batched': (_i, [_vp, _i, _i, ctypes.c_longlong, _vp, _i, _i, _vp, _vp, _vp]),
    'gpmc_cov_cross': (_i, [_vp, _i, _vp, _i, _i, _vp, _i, _i, _vp, _i, _vp]),
    'gpmc_tg2_loglik': (_i, [_vp, ctypes.c_double, _vp, _i, _i, _i, _vp, ctypes.c_double, ctypes.c_double, _vp, _vp]),
    'gpmc_predict_workspace_bytes': (_sz, [_i, _i, _i]),
    'gpmc_predict_batched': (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_ess_workspace_bytes': (_sz, [_i, _i]),
    'gpmc_ess_sweep': (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                            ctypes.c_ulonglong, ctypes.c_uint, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'gpmc_set_tuning': (_i, [_i, _i]),
    'gpmc_loglik_layout': (_i, [ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    'gpmc_bench_fp64_peak': (_i, [_i, _i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    'gpmc_bench_dmma_ilp': (_i, [_i, _i, _i, ctypes.POINTER(ctypes.c_double)]),
    'gpmc_sds_loop_stats': (_i, [ctypes.POINTER(ctypes.c_longlong)] * 3),
    'gpmc_profile_enable': (_i, [_i]),
    'gpmc_profile_read': (_i, [_i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)]),
    'gpmc_profile_reset': (_i, []),
    'gpmc_profile_timeline': (_i, [_i, _i, ctypes.POINTER(ctypes.c_double), ctypes.c_longlong, ctypes.POINTER(ctypes.c_longlong)]),
}

_lib = None


class GpmcError(RuntimeError):
    pass


def load():
    """dlopen libgpmc.so and attach the prototypes.  Raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise GpmcError('%s is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                        '(there is no CPU fallback for this path)' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().gpmc_last_error().decode('utf-8', 'replace')
        raise GpmcError('%s failed (rc=%d): %s' % (what, rc, msg))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise GpmcError('no CUDA device: the GP log-likelihood path has no CPU fallback')
    return torch
