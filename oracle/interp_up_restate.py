"""
oracle/interp_up_restate.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes front-end for ``oracle/interp_up_restate.c``: the CPU restatement of ``rasterio.warp.reproject`` with
``resampling=bilinear | cubic | lanczos`` for up-sampling (see the C file's header: PARITY UNPINNED).

``reproject_array`` has the signature of ``oracle.gdal_restate.reproject_array`` and hands every other resampling to
it, so the oracle's kernel-model port (``oracle/kernel_model_np.py``, which resamples through
``gdal_restate.reproject_array``) covers the three methods once its ``reproject_array`` is replaced by this one
(``with_interp_up``).

Only ``tests/`` may import this module.
"""
import contextlib
import os
import pathlib
import subprocess
import tempfile
import ctypes

import numpy as np

from oracle import gdal_restate

_HERE = pathlib.Path(__file__).resolve().parent
_SRC = _HERE / 'interp_up_restate.c'
_SO = _HERE / '_build' / 'libinterp_up_restate.so'
_lib = None
_FUNCS = {'bilinear': 'gr_bilinear_up', 'cubic': 'gr_cubic_up', 'lanczos': 'gr_lanczos_up'}
METHODS = tuple(_FUNCS)


def build(force: bool = False) -> pathlib.Path:
    """ Compile the C restatement with gcc (OpenMP) into oracle/_build -- or, when the tree is read-only, into a new
    temporary directory.  Returns the library's path. """
    so = _SO
    if force or (not so.exists()) or so.stat().st_mtime < _SRC.stat().st_mtime:
        try:
            so.parent.mkdir(exist_ok=True)
        except OSError:
            pass
        if not os.access(so.parent, os.W_OK):
            so = pathlib.Path(tempfile.mkdtemp(prefix='interp_up_restate_')) / _SO.name
        subprocess.run(['gcc', '-O2', '-fopenmp', '-fno-fast-math', '-ffp-contract=off', '-shared', '-fPIC', '-o',
                        str(so), str(_SRC), '-lm'], check=True)
    return so


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(str(build()))
        c_long, c_int, c_dbl, c_vp = ctypes.c_long, ctypes.c_int, ctypes.c_double, ctypes.c_void_p
        for name in _FUNCS.values():
            getattr(lib, name).argtypes = [c_vp, c_long, c_long, c_long, c_int, c_dbl, c_vp, c_long, c_long, c_dbl,
                                           c_dbl, c_dbl, c_dbl]
            getattr(lib, name).restype = None
        _lib = lib
    return _lib


# the original, kept so that `with_interp_up` can delegate to it while it is replaced
_base_reproject_array = gdal_restate.reproject_array


def reproject_array(src, src_transform, src_nodata, dst_shape, dst_transform, dst_nodata, resampling,
                    out_dtype='float32'):
    """ ``gdal_restate.reproject_array`` extended with bilinear, cubic and lanczos up-sampling. """
    resampling = getattr(resampling, 'name', resampling)
    if resampling not in _FUNCS:
        return _base_reproject_array(src, src_transform, src_nodata, dst_shape, dst_transform, dst_nodata,
                                     resampling, out_dtype)
    lib = _load()
    src = np.asarray(src)
    squeeze = src.ndim == 2
    src3 = src[None] if squeeze else src
    nb, hs, ws = src3.shape
    hd, wd = int(dst_shape[0]), int(dst_shape[1])
    sx, ox, sy, oy = gdal_restate.grid_map(src_transform, dst_transform)
    if sx > 1.0 + 1e-12 or sy > 1.0 + 1e-12:
        raise NotImplementedError(f'{resampling} is only restated for up-sampling')
    has_nd, nd = (0, 0.0) if src_nodata is None else (1, float(src_nodata))
    dst = np.full((nb, hd, wd), 0.0 if dst_nodata is None else dst_nodata, dtype='float32')
    s64 = np.ascontiguousarray(src3, dtype='float64')
    getattr(lib, _FUNCS[resampling])(s64.ctypes.data, nb, hs, ws, has_nd, nd, dst.ctypes.data, hd, wd, sx, ox, sy, oy)
    dst = dst.astype(out_dtype, copy=False)
    return dst[0] if squeeze else dst


@contextlib.contextmanager
def with_interp_up():
    """ Within the block, ``gdal_restate.reproject_array`` -- and so every function of ``oracle.kernel_model_np`` --
    also restates bilinear, cubic and lanczos up-sampling. """
    gdal_restate.reproject_array = reproject_array
    try:
        yield
    finally:
        gdal_restate.reproject_array = _base_reproject_array
