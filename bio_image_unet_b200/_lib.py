"""ctypes binding of the C-ABI library (include/biu_b200.h).

The product path has no CPU fallback: if ``libbiu_b200.so`` is missing or a call fails, an exception is raised.
"""
import ctypes
import os
from ctypes import (POINTER, c_char_p, c_double, c_float, c_int, c_longlong, c_uint, c_uint8, c_uint32, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libbiu_b200.so')

# every symbol include/biu_b200.h declares: name -> (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    'biu_last_error': (c_char_p, []),
    'biu_version': (c_int, []),
    'biu_net_create': (_P, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_char_p), c_int,
                            c_int, c_int]),
    'biu_net_set_param': (c_int, [_P, c_char_p, _P, c_int, POINTER(c_longlong)]),
    'biu_net_finalize': (c_int, [_P]),
    'biu_net_plan': (c_longlong, [_P, c_int, c_int, c_int, c_int]),
    'biu_net_forward': (c_int, [_P, _P, c_int, _P, _P, _P, _P, _P]),
    'biu_net_debug_copy': (c_int, [_P, c_char_p, _P, _P, c_longlong]),
    'biu_net_set_force_direct': (c_int, [_P, c_int]),
    'biu_net_set_fuse_pool': (c_int, [_P, c_int]),
    'biu_net_set_debug_stop': (c_int, [_P, c_int]),
    'biu_set_rows_kernel': (c_int, [c_int]),
    'biu_set_halo_cta2': (c_int, [c_int]),
    'biu_net_fallback_ops': (c_int, [_P]),
    'biu_net_set_siam_shared': (c_int, [_P, c_int]),
    'biu_net_destroy': (None, [_P]),
    'biu_histogram': (c_int, [_P, c_int, c_longlong, c_int, _P, _P]),
    'biu_hist_sum': (c_int, [_P, c_int, _P, _P]),
    'biu_norm_lut': (c_int, [_P, _P, c_longlong, c_longlong, c_int, c_double, c_double, c_int, _P, _P, _P]),
    'biu_apply_lut': (c_int, [_P, c_int, c_longlong, c_int, _P, c_longlong, _P, _P]),
    'biu_norm_lut_f32': (c_int, [_P, _P, c_longlong, c_longlong, c_int, c_double, c_double, c_int, _P, _P, _P]),
    'biu_apply_lut_f32': (c_int, [_P, c_int, c_longlong, c_int, _P, c_longlong, _P, _P]),
    'biu_gather_tiles_f32': (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                     c_int, _P, _P]),
    'biu_gather_tiles_lut': (c_int, [_P, c_int, _P, c_longlong, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int,
                                     c_int, c_int, c_int, c_int, _P, _P]),
    'biu_gather_tiles': (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                 c_int, _P, _P]),
    'biu_gather_tiles_tta': (c_int, [_P, c_int, _P, c_longlong, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int,
                                     c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    'biu_gather_tiles_f32_tta': (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                         c_int, c_int, c_int, _P, _P]),
    'biu_tta_accumulate': (c_int, [_P, c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    'biu_stitch_mean_u8': (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    'biu_stitch_mod3_u8': (c_int, [_P, c_int, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P,
                                   _P]),
    'biu_stitch_weighted_u8': (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, c_int,
                                       c_int, c_int, _P, _P, _P, _P, _P]),
    'biu_stitch_ramp_f32': (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, c_int,
                                    c_int, c_int, c_int, _P, _P]),
    'biu_normalize_f32_scratch_bytes': (ctypes.c_longlong, [ctypes.c_longlong, c_int]),
    'biu_normalize_f32': (c_int, [_P, ctypes.c_longlong, c_int, c_int, ctypes.c_double, ctypes.c_double, c_int, _P, _P, _P, _P, _P]),
    'biu_stitch_margin_f32': (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P,
                                      _P, _P]),
    'biu_conv_tc': (c_int, [c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int,
                            _P, _P, c_float, _P, c_int, c_int, _P]),
    'biu_up_tc': (c_int, [c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, _P, _P, c_int,
                          c_int, _P]),
    'biu_conv_direct': (c_int, [c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P,
                                c_int, _P, _P, c_float, _P, c_int, c_int, _P]),
    'biu_pool2': (c_int, [c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int,
                          _P]),
    'biu_device_fault': (c_int, [POINTER(c_uint)]),
    'biu_launch_count': (ctypes.c_ulonglong, []),
    'biu_net_set_profile': (c_int, [_P, c_int]),
    'biu_net_profile_read': (c_int, [_P, c_int, POINTER(c_int), POINTER(c_float), POINTER(c_int)]),
}

_lib = None


class BiuError(RuntimeError):
    pass


def load():
    """Load the shared library once and attach the prototypes. Raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BiuError(f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                       f'(there is no CPU fallback)')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        msg = load().biu_last_error().decode('utf-8', 'replace')
        raise BiuError(f'{what}: {msg}' if what else msg)


def last_error():
    return load().biu_last_error().decode('utf-8', 'replace')


def ptr(t):
    """Raw device/host pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
