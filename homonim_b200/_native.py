"""
ctypes binding of ``libhomonim_b200.so`` (the sm_100a CUDA library behind ``include/homonim_b200.h``).

This is the binding a maintainer would drop into homonim itself (see INTEGRATION.md): plain pointers and sizes, no
torch types cross the boundary -- tensors only provide ``data_ptr()`` and the current CUDA stream handle.

There is NO CPU fallback: if the shared library is missing or cannot be loaded, :func:`lib` raises
:class:`~homonim_b200.errors.NativeLibraryError`; if a call fails, so does :func:`check`.
"""
import ctypes
import os
import pathlib
import threading
from ctypes import c_char_p, c_double, c_int, c_long, c_size_t, c_void_p

from homonim_b200.errors import NativeLibraryError

HB_U8, HB_U16, HB_F32, HB_I16 = 0, 1, 2, 3
HB_MODEL_GAIN, HB_MODEL_GAIN_BLK_OFFSET, HB_MODEL_GAIN_OFFSET = 0, 1, 2
HB_UP_CUBIC_SPLINE, HB_UP_NEAREST, HB_UP_BILINEAR, HB_UP_CUBIC, HB_UP_LANCZOS = 0, 1, 2, 3, 4
HB_STAT_MIN, HB_STAT_MAX, HB_STAT_MED, HB_STAT_Q1, HB_STAT_Q3, HB_STAT_MODE = 0, 1, 2, 3, 4, 5
ABI_VERSION = 11

_PKG_DIR = pathlib.Path(__file__).resolve().parent
LIB_PATH = _PKG_DIR / 'libhomonim_b200.so'

_lock = threading.Lock()
_lib = None

# name -> (restype, argtypes); must list every symbol declared in include/homonim_b200.h
SIGNATURES = {
    'hb_abi_version': (c_int, []),
    'hb_last_error': (c_char_p, []),
    'hb_device_count': (c_int, []),
    'hb_launch_count': (c_long, []),
    'hb_reset_launch_count': (None, []),
    'hb_downsample_average': (c_int, [c_void_p, c_int, c_long, c_long, c_int, c_double, c_void_p, c_long, c_long,
                                      c_double, c_double, c_double, c_double, c_void_p]),
    'hb_resample_stat': (c_int, [c_void_p, c_int, c_long, c_long, c_int, c_double, c_void_p, c_long, c_long, c_double,
                                 c_double, c_double, c_double, c_int, c_void_p]),
    'hb_block_norm_workspace_bytes': (c_size_t, [c_long]),
    'hb_block_norm': (c_int, [c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_void_p, c_void_p,
                              c_size_t, c_void_p]),
    'hb_block_norm_shard_workspace_bytes': (c_size_t, [c_long, c_long]),
    'hb_block_norm_message_bytes': (c_size_t, [c_long, c_long]),
    'hb_block_norm_partial': (c_int, [c_int, c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_long, c_long,
                                      c_void_p, c_size_t, c_void_p]),
    'hb_block_norm_merge': (c_int, [c_int, c_void_p, c_int, c_int, c_long, c_long, c_void_p, c_size_t, c_void_p,
                                    c_void_p]),
    'hb_fit_same_grid': (c_int, [c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_long, c_int, c_int,
                                 c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'hb_fit_apply_same_grid': (c_int, [c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_long, c_int,
                                       c_int, c_int, c_void_p, c_int, c_int, c_double, c_void_p, c_void_p]),
    'hb_fit_same_grid_rows': (c_int, [c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_long, c_long,
                                      c_long, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'hb_fit_apply_same_grid_rows': (c_int, [c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_long,
                                            c_long, c_long, c_int, c_int, c_int, c_void_p, c_int, c_int, c_double,
                                            c_void_p, c_void_p]),
    'hb_inpaint_workspace_bytes': (c_size_t, [c_long, c_long]),
    'hb_inpaint_refit': (c_int, [c_void_p, c_void_p, c_long, c_long, c_double, c_double, c_void_p, c_size_t,
                                 c_void_p]),
    'hb_apply_same_grid': (c_int, [c_void_p, c_int, c_int, c_double, c_int, c_void_p, c_long, c_long, c_int, c_int,
                                   c_double, c_void_p, c_void_p]),
    'hb_upsample_apply': (c_int, [c_void_p, c_int, c_long, c_long, c_int, c_double, c_void_p, c_long, c_long, c_double,
                                  c_double, c_double, c_double, c_void_p, c_int, c_int, c_double, c_void_p, c_int,
                                  c_void_p]),
    'hb_resample_up': (c_int, [c_void_p, c_long, c_long, c_long, c_int, c_double, c_void_p, c_long, c_long, c_double,
                               c_double, c_double, c_double, c_int, c_void_p]),
    'hb_full_coverage_mask': (c_int, [c_void_p, c_long, c_long, c_void_p, c_long, c_long, c_double, c_double, c_double,
                                      c_double, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'hb_convert_dtype': (c_int, [c_void_p, c_long, c_int, c_int, c_double, c_void_p, c_void_p]),
    'hb_valid_mask': (c_int, [c_void_p, c_int, c_long, c_int, c_double, c_void_p, c_void_p]),
    'hb_compare_sums_workspace_bytes': (c_size_t, []),
    'hb_compare_sums': (c_int, [c_void_p, c_int, c_double, c_void_p, c_int, c_double, c_long, c_void_p, c_void_p,
                                c_size_t, c_void_p]),
    'hb_fuse_refspace': (c_int, [c_void_p, c_int, c_long, c_long, c_int, c_double, c_void_p, c_long, c_long, c_int,
                                 c_double, c_double, c_double, c_double, c_double, c_int, c_int, c_int, c_int, c_int,
                                 c_double, c_int, c_int, c_double, c_void_p, c_void_p, c_void_p]),
    'hb_fuse_refspace_host': (c_int, [c_void_p, c_int, c_long, c_long, c_int, c_double, c_void_p, c_long, c_long,
                                      c_int, c_double, c_double, c_double, c_double, c_double, c_int, c_int, c_int,
                                      c_int, c_int, c_double, c_int, c_int, c_double, c_void_p, c_void_p, c_void_p]),
    'hb_build_overviews': (c_int, [c_void_p, c_int, c_long, c_long, c_long, c_int, c_double, c_int, c_void_p, c_void_p]),
}


def build_hint() -> str:
    return ("build it with `python -c 'import __graft_entry__ as g; g.build()'` or `make -C homonim_b200/csrc` "
            "(needs nvcc; targets sm_100a)")


def lib() -> ctypes.CDLL:
    """ Load (once) and return the native library.  Raises NativeLibraryError -- never falls back to the CPU. """
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                path = pathlib.Path(os.environ.get('HOMONIM_B200_LIB', LIB_PATH))
                if not path.exists():
                    raise NativeLibraryError(f'{path} not found: the CUDA library is required; {build_hint()}')
                try:
                    handle = ctypes.CDLL(str(path))
                except OSError as ex:
                    raise NativeLibraryError(f'could not load {path}: {ex}') from ex
                for name, (restype, argtypes) in SIGNATURES.items():
                    try:
                        fn = getattr(handle, name)
                    except AttributeError as ex:
                        raise NativeLibraryError(f'{path} does not export {name}: rebuild it; {build_hint()}') from ex
                    fn.restype = restype
                    fn.argtypes = argtypes
                if handle.hb_abi_version() != ABI_VERSION:
                    raise NativeLibraryError(f'{path} has ABI {handle.hb_abi_version()}, expected {ABI_VERSION}')
                _lib = handle
    return _lib


def check(rc: int, what: str = ''):
    """ Raise NativeLibraryError for a non-zero return code of a C-ABI call. """
    if rc != 0:
        msg = lib().hb_last_error()
        msg = msg.decode('utf-8', 'replace') if msg else 'unknown error'
        raise NativeLibraryError(f'{what or "native call"} failed (code {rc}): {msg}')


def require_device() -> int:
    """ Number of CUDA devices; raises when there is none (the product path has no CPU implementation). """
    n = lib().hb_device_count()
    if n <= 0:
        msg = lib().hb_last_error()
        raise NativeLibraryError(
            'no CUDA device is available: homonim_b200 has no CPU fallback'
            + (f' ({msg.decode("utf-8", "replace")})' if msg else '')
        )
    return n
