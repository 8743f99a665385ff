"""
ctypes binding of libttm.so (C ABI declared in include/ttm.h).

The library is built in-tree by `__graft_entry__.build()`.  There is NO CPU fallback: if the shared
library is missing or no CUDA device is visible, constructing a map raises.
"""

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libttm.so')

c_void_p, c_int, c_int64, c_double = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
_dp = ctypes.POINTER(c_double)
_ip = ctypes.POINTER(ctypes.c_int32)

TTM_DTYPE_F64, TTM_DTYPE_F32 = 0, 1     # include/ttm.h: element type of the *_ld entry points

_lib = None


class TTMError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TTMError('libttm.so not found at %s: run `python __graft_entry__.py` (build()) first; '
                           'this package has no CPU fallback.' % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.ttm_last_error.restype = ctypes.c_char_p
        sig = {
            'ttm_device_sm_count': [c_int, ctypes.POINTER(c_int)],
            'ttm_host_is_pinned': [c_void_p, ctypes.POINTER(c_int)],
            'ttm_ctx_create': [c_int, ctypes.POINTER(c_void_p)],
            'ttm_ctx_destroy': [c_void_p],
            'ttm_ctx_set_quadrature': [c_void_p, _dp, _dp, c_int],
            'ttm_ctx_set_rectifier': [c_void_p, c_int, c_double],
            'ttm_ctx_set_blocks_per_sm': [c_void_p, c_int],
            'ttm_ctx_set_objgrad_kernel': [c_void_p, c_int],
            'ttm_plan_info': [c_void_p, ctypes.POINTER(c_int)],
            'ttm_plan_create': [c_void_p, _ip, c_int64, _dp, c_int64, ctypes.POINTER(c_void_p)],
            'ttm_plan_update_doubles': [c_void_p, _dp, c_int64],
            'ttm_plan_destroy': [c_void_p],
            'ttm_colstats': [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
            'ttm_standardize_transpose': [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                          c_void_p],
            'ttm_colstats_ld': [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                c_void_p],
            'ttm_standardize_transpose_ld': [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p, c_void_p,
                                             c_void_p, c_int64, c_void_p],
            'ttm_transpose_back': [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                   c_void_p],
            'ttm_basis_eval': [c_void_p, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p],
            'ttm_plan_set_gram_mode': [c_void_p, c_int],
            'ttm_plan_set_coeffs': [c_void_p, _dp, c_void_p],
            'ttm_objgrad_ir_launch': [c_void_p, c_void_p, c_int64, c_int64, c_void_p],
            'ttm_plan_get_out': [c_void_p, _dp, c_int, c_void_p],
            'ttm_objgrad_ir': [c_void_p, c_void_p, c_int64, c_int64, _dp, _dp, c_void_p],
            'ttm_eval_s_ir': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p],
            'ttm_sep_eval': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p],
            'ttm_map_fused': [c_void_p, ctypes.POINTER(c_void_p), c_int, _dp, c_void_p, c_int64, c_int, c_void_p, c_void_p,
                              c_void_p, c_int, c_void_p, c_void_p, c_void_p],
            'ttm_map_fused_ld': [c_void_p, ctypes.POINTER(c_void_p), c_int, _dp, c_void_p, c_int, c_int64, c_int64, c_int,
                                 c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
            'ttm_gram': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p],
            'ttm_gram_tail': [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p],
            'ttm_sep_objgrad': [c_void_p, c_void_p, c_int64, c_int64, _dp, _dp, c_void_p],
            'ttm_sep_objgrad_launch': [c_void_p, c_void_p, c_int64, c_int64, _dp, c_void_p],
            'ttm_sep_objgrad_wait': [c_void_p, _dp, c_void_p],
            'ttm_sep_reduced_batch': [c_int, ctypes.POINTER(c_void_p), c_void_p, c_int64, c_int64, ctypes.c_double,
                                      ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                      ctypes.POINTER(c_void_p), c_void_p],
            'ttm_mon_table': [c_void_p, c_int, c_void_p, c_void_p],
            'ttm_inverse_table': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p],
            'ttm_inverse_fused_apack_size': [c_int, c_int, c_int, ctypes.POINTER(c_int64)],
            'ttm_inverse_fused': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p,
                                  c_void_p, c_void_p, c_int, c_int, c_void_p],
            'ttm_inverse_rect_rpack_size': [c_int, c_int, c_int, ctypes.POINTER(c_int64)],
            'ttm_map_rect': [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                             c_int64, c_void_p],
            'ttm_sep_eval_base': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, ctypes.c_double, c_void_p, c_void_p],
            'ttm_inverse_fused_split': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int, c_int, c_int,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p],
            'ttm_inverse_bisect': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int, c_int,
                                   ctypes.POINTER(c_int), c_void_p],
            'ttm_density_accumulate': [c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_int, c_int64, c_void_p],
            'ttm_density_finish': [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p],
            'ttm_ir_logdet_accumulate': [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_double, c_int, c_void_p,
                                         c_void_p],
            'ttm_fp64_peak': [c_void_p, _dp],
        }
        for name, args in sig.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = c_int
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise TTMError('libttm error %d: %s' % (rc, lib().ttm_last_error().decode()))


def dptr(a):
    """numpy float64 array -> double* (the array must stay alive during the call)."""
    assert a.dtype == np.float64 and a.flags['C_CONTIGUOUS']
    return a.ctypes.data_as(_dp)


def iptr(a):
    assert a.dtype == np.int32 and a.flags['C_CONTIGUOUS']
    return a.ctypes.data_as(_ip)
