"""ctypes binding of libv2ce_b200.so (declared in include/v2ce_b200.h).

The library is the product: if it is missing or a call fails we raise -- there is
no CPU or PyTorch fallback anywhere in this package.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t,
                    c_uint64, c_void_p)

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libv2ce_b200.so')


class V2ceError(RuntimeError):
    pass


class LdatiParams(Structure):
    _fields_ = [
        ('height', c_int32), ('width', c_int32), ('n_frames', c_int32), ('true_div', c_int32),
        ('frame_base', c_int64), ('seed', c_uint64),
        ('fps64', c_double), ('nbins64', c_double), ('r_fps64', c_double), ('r_nbins64', c_double),
        ('fps32', c_float), ('nbins32', c_float), ('r_fps32', c_float), ('r_nbins32', c_float),
        ('vs32', c_float), ('inv_vs32', c_float), ('vs2_32', c_float), ('r_vs2_32', c_float),
        ('six32', c_float), ('r6_32', c_float), ('eps6', c_float), ('eps8', c_float),
        ('binstart_t0_32', c_float * 16), ('bin_base_us', c_int64 * 16),
        ('key_span', c_int32), ('add_frame_offset', c_int32),
        ('multi_events', c_int32), ('bidirectional', c_int32),
        ('pooling', c_int32), ('pooling_kernel_size', c_int32),
    ]


class BaselineParams(Structure):
    """Mirror of v2ce_baseline_params (include/v2ce_b200.h)."""
    _fields_ = [
        ('height', c_int32), ('width', c_int32), ('n_frames', c_int32), ('mode', c_int32),
        ('frame_base', c_int64), ('seed', c_uint64),
        ('delta32', c_float), ('binstart_t0_32', c_float * 10),
        ('key_base_us', c_int64), ('key_span', c_int32), ('add_frame_offset', c_int32),
    ]


_SIGNATURES = {
    'v2ce_last_error': (c_char_p, []),
    'v2ce_version': (c_int, []),
    'v2ce_device_check': (c_int, [c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    'v2ce_ldati_params_size': (c_size_t, []),
    'v2ce_ldati_params_validate': (c_int, [POINTER(LdatiParams)]),
    'v2ce_ldati_count_workspace_bytes': (c_int, [POINTER(LdatiParams), POINTER(c_size_t)]),
    'v2ce_ldati_emit_workspace_bytes': (c_int, [POINTER(LdatiParams), c_int64, POINTER(c_size_t)]),
    'v2ce_ldati_count': (c_int, [c_void_p, POINTER(LdatiParams), c_void_p, c_size_t, c_void_p, c_void_p]),
    'v2ce_ldati_count_ef': (c_int, [c_void_p, POINTER(LdatiParams), c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    'v2ce_ldati_emit': (c_int, [c_void_p, POINTER(LdatiParams), c_void_p, c_void_p, c_size_t, c_void_p, c_int32,
                                c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    'v2ce_ldati_relocate': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    'v2ce_baseline_params_size': (c_size_t, []),
    'v2ce_baseline_count_workspace_bytes': (c_int, [POINTER(BaselineParams), POINTER(c_size_t)]),
    'v2ce_baseline_emit_workspace_bytes': (c_int, [POINTER(BaselineParams), c_int64, POINTER(c_size_t)]),
    'v2ce_baseline_count': (c_int, [c_void_p, POINTER(BaselineParams), c_void_p, c_size_t, c_void_p, c_void_p]),
    'v2ce_baseline_emit': (c_int, [c_void_p, POINTER(BaselineParams), c_void_p, c_void_p, c_size_t, c_void_p, c_int64,
                                   c_void_p, c_void_p, c_void_p]),
    'v2ce_ts_diff_workspace_bytes': (c_int, [c_int32, c_int32, c_int64, POINTER(c_size_t)]),
    'v2ce_ts_diff_metric': (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32, c_int32, c_double, c_void_p,
                                    c_size_t, c_void_p, c_void_p]),
    'v2ce_events_to_voxels': (c_int, [c_void_p, c_int64, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                      c_void_p]),
    'v2ce_peer_window_alloc': (c_int, [c_size_t, POINTER(c_void_p), c_void_p]),
    'v2ce_peer_window_free': (c_int, [c_void_p]),
    'v2ce_peer_window_open': (c_int, [c_void_p, POINTER(c_void_p)]),
    'v2ce_peer_window_close': (c_int, [c_void_p]),
    'v2ce_peer_copy_async': (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    'v2ce_ef_accumulate': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'v2ce_ef_select_workspace_bytes': (c_int, [POINTER(c_size_t)]),
    'v2ce_ef_select': (c_int, [c_void_p, c_int64, c_double, c_int32, c_void_p, c_size_t, c_void_p, c_void_p]),
    'v2ce_ef_normalize': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_double, c_void_p, c_void_p]),
    'v2ce_image_units': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'v2ce_assemble_windows': (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                      c_int32, c_void_p, c_void_p]),
    'v2ce_model_create': (c_int, [POINTER(c_void_p), c_int]),
    'v2ce_model_destroy': (c_int, [c_void_p]),
    'v2ce_model_set_tensor': (c_int, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int32]),
    'v2ce_model_finalize': (c_int, [c_void_p]),
    'v2ce_model_workspace_bytes': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, POINTER(c_size_t)]),
    'v2ce_model_workspace_layout': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, POINTER(c_int64), c_int32,
                                            POINTER(c_int32)]),
    'v2ce_model_forward': (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                   c_size_t, c_void_p]),
    'v2ce_model_forward_frames': (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                          c_size_t, c_void_p]),
    'v2ce_model_last_sigmas': (c_int, [c_void_p, POINTER(c_float)]),
    'v2ce_model_call_count': (c_int, [c_void_p, POINTER(c_int64)]),
    'v2ce_model_sn_advance': (c_int, [c_void_p, c_int32, c_void_p]),
    'v2ce_model_last_launches': (c_int, [c_void_p, POINTER(c_int32)]),
    'v2ce_conv3d_bf16_ex': (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32,
                                    c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                    c_int32, c_void_p, c_int32, c_void_p]),
    'v2ce_model_set_option': (c_int, [c_void_p, c_char_p, c_int64]),
    'v2ce_model_layer_times': (c_int, [c_void_p, c_int32, POINTER(c_float), c_char_p, POINTER(c_int32)]),
    'v2ce_debug_mma_rate': (c_int, [c_int32, c_int32, c_int32, c_int32, POINTER(c_double)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load the shared library (once).  Raises V2ceError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise V2ceError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                        '(nvcc, sm_100a).  There is no CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.v2ce_ldati_params_size() != ctypes.sizeof(LdatiParams):
        raise V2ceError(f'v2ce_ldati_params is {lib.v2ce_ldati_params_size()} bytes in {LIB_PATH} but the ctypes mirror has '
                        f'{ctypes.sizeof(LdatiParams)}: rebuild the library (python -c "import __graft_entry__ as g; g.build()")')
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load().v2ce_last_error()
        raise V2ceError(f'libv2ce_b200 error {code}: {msg.decode() if msg else "?"}')


def require_cuda(t, name='tensor'):
    import torch
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise V2ceError(f'{name} must be a CUDA tensor: the V2CE B200 path has no CPU fallback')
    return t


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)
