"""ctypes binding of the C ABI in include/stb.h.

The only library this module ever opens is the nvcc-built `libscannertools_b200.so` that sits
next to it.  There is no CPU fallback: if the library is missing, or no CUDA device is usable,
loading / the first compute call raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = 'libscannertools_b200.so'
LIB_PATH = os.path.join(_HERE, LIB_NAME)

_u8pp = C.POINTER(C.c_void_p)
_vp = C.c_void_p


class FarnebackParams(C.Structure):
    _fields_ = [('num_levels', C.c_int), ('pyr_scale', C.c_double), ('fast_pyramids', C.c_int),
                ('win_size', C.c_int), ('num_iters', C.c_int), ('poly_n', C.c_int),
                ('poly_sigma', C.c_double), ('flags', C.c_int)]


# name -> (restype, argtypes); this table is also what tests use to check that the shared
# library exports every symbol include/stb.h declares.
SIGNATURES = {
    'stb_version': (C.c_int, []),
    'stb_last_error': (C.c_char_p, []),
    'stb_device_count': (C.c_int, []),
    'stb_hist_rgb16': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'stb_hist_rgb16_strided': (C.c_int, [_vp, C.c_size_t, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'stb_shot_scores': (C.c_int, [_vp, C.c_int, _vp, _vp, _vp]),
    'stb_flow_hist': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'stb_flow_hist_strided': (C.c_int, [_vp, C.c_size_t, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'stb_frame_diff': (C.c_int, [_vp, _vp, _vp, C.c_size_t, _vp]),
    'stb_farneback_default_params': (None, [C.POINTER(FarnebackParams)]),
    'stb_farneback_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.POINTER(FarnebackParams)]),
    'stb_farneback_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(FarnebackParams), C.POINTER(_vp)]),
    'stb_farneback_destroy': (C.c_int, [_vp]),
    'stb_farneback_run': (C.c_int, [_vp, _u8pp, C.c_int, _u8pp, _vp]),
    'stb_farneback_run_gray': (C.c_int, [_vp, _u8pp, C.c_int, _u8pp, _vp]),
    'stb_farneback_run_hist': (C.c_int, [_vp, _u8pp, C.c_int, _u8pp, _vp, _vp]),
    'stb_farneback_levels': (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'stb_farneback_debug_set': (C.c_int, [_vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    'stb_resize_target': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'stb_resize_bilinear_u8': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, C.c_int, _u8pp, C.c_int, C.c_int, _vp]),
    'stb_resize_interp_code': (C.c_int, [C.c_char_p]),
    'stb_resize_u8': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, C.c_int, _u8pp, C.c_int, C.c_int, C.c_int, _vp]),
    'stb_resize_f32': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, C.c_int, _u8pp, C.c_int, C.c_int, C.c_int, _vp]),
    'stb_color_code': (C.c_int, [C.c_char_p]),
    'stb_color_in_channels': (C.c_int, [C.c_int]),
    'stb_color_out_channels': (C.c_int, [C.c_int]),
    'stb_convert_color_u8': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, C.c_int, _u8pp, _vp]),
    'stb_blur_u8': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8pp, _vp]),
    'stb_hist_hsv16': (C.c_int, [_u8pp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'stb_hist_hsv16_strided': (C.c_int, [_vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    'stb_launch_count': (C.c_longlong, []),
    'stb_farneback_profile': (C.c_int, [_vp, C.c_int]),
    'stb_farneback_profile_read': (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    'stb_pipe_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    'stb_pipe_destroy': (C.c_int, [_vp]),
    'stb_pipe_hist': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    'stb_pipe_flow': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    'stb_pipe_flow_async': (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.POINTER(C.c_int)]),
    'stb_pipe_wait': (C.c_int, [_vp, C.c_int]),
    'stb_host_alloc': (C.c_int, [C.c_size_t, C.c_int, C.POINTER(_vp)]),
    'stb_host_free': (C.c_int, [_vp]),
}


def bind(cdll, names=None):
    """Attach restype/argtypes for every declared entry point; raises AttributeError if the
    library lacks one."""
    for name, (res, args) in SIGNATURES.items():
        if names is not None and name not in names:
            continue
        fn = getattr(cdll, name)
        fn.restype = res
        fn.argtypes = args
    return cdll


class StbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('scannertools_b200: status %d: %s' % (code, msg))
        self.code = code


_lib = None


def load():
    """Open libscannertools_b200.so (built by `python __graft_entry__.py` / build.py)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError('%s not built: run `python -c "import __graft_entry__ as g; g.build()"` '
                              'at the repo root (needs nvcc); there is no CPU fallback' % LIB_PATH)
        _lib = bind(C.CDLL(LIB_PATH))
    return _lib


def check(code, lib=None):
    if code != 0:
        lib = lib or load()
        raise StbError(code, (lib.stb_last_error() or b'').decode('utf-8', 'replace'))


def ptr_table(ptrs):
    """HOST array of device pointers, as the `const T* const*` parameters expect."""
    arr = (C.c_void_p * len(ptrs))(*[int(p) for p in ptrs])
    return arr
