"""
oracle/footprint_stats_restate.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes front-end for ``oracle/footprint_stats_restate.c``: the CPU restatement of ``rasterio.warp.reproject`` with
``resampling=min | max | med | q1 | q3 | mode`` on any geometry (see the C file's header: PARITY UNPINNED).

``reproject_array`` has the signature of ``oracle.gdal_restate.reproject_array`` and hands every other resampling to
``oracle.interp_up_restate.reproject_array`` (which hands what it does not restate to ``gdal_restate``), so the oracle's
kernel-model port (``oracle/kernel_model_np.py``) covers the six methods once ``gdal_restate.reproject_array`` is
replaced by this one (``with_footprint_stats``).

Only ``tests/`` may import this module.
"""
import contextlib
import ctypes
import os
import pathlib
import subprocess
import tempfile

import numpy as np

from oracle import gdal_restate, interp_up_restate

_HERE = pathlib.Path(__file__).resolve().parent
_SRC = _HERE / 'footprint_stats_restate.c'
_SO = _HERE / '_build' / 'libfootprint_stats_restate.so'
_lib = None
METHOD_CODES = {'min': 0, 'max': 1, 'med': 2, 'q1': 3, 'q3': 4, 'mode': 5}
METHODS = tuple(METHOD_CODES)


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
            so = pathlib.Path(tempfile.mkdtemp(prefix='footprint_stats_restate_')) / _SO.name
        subprocess.run(['gcc', '-O2', '-fopenmp', '-fno-fast-math', '-ffp-contract=off', '-shared', '-fPIC', '-o',
                        str(so), str(_SRC), '-lm'], check=True)
    return so


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(str(build()))
        c_long, c_int, c_dbl, c_vp = ctypes.c_long, ctypes.c_int, ctypes.c_double, ctypes.c_void_p
        lib.fs_resample_stat.argtypes = [c_vp, c_long, c_long, c_int, c_dbl, c_vp, c_long, c_long, c_dbl, c_dbl, c_dbl,
                                         c_dbl, c_int]
        lib.fs_resample_stat.restype = None
        _lib = lib
    return _lib


def reproject_array(src, src_transform, src_nodata, dst_shape, dst_transform, dst_nodata, resampling,
                    out_dtype='float32'):
    """ ``interp_up_restate.reproject_array`` extended with the min, max, med, q1, q3 and mode footprint statistics. """
    resampling = getattr(resampling, 'name', resampling)
    if resampling not in METHOD_CODES:
        return interp_up_restate.reproject_array(src, src_transform, src_nodata, dst_shape, dst_transform, dst_nodata,
                                                 resampling, out_dtype)
    lib = _load()
    src = np.asarray(src)
    squeeze = src.ndim == 2
    src3 = src[None] if squeeze else src
    nb, hs, ws = src3.shape
    hd, wd = int(dst_shape[0]), int(dst_shape[1])
    sx, ox, sy, oy = gdal_restate.grid_map(src_transform, dst_transform)
    has_nd, nd = (0, 0.0) if src_nodata is None else (1, float(src_nodata))
    dst = np.full((nb, hd, wd), 0.0 if dst_nodata is None else dst_nodata, dtype='float32')
    for b in range(nb):
        plane = np.ascontiguousarray(src3[b], dtype='float32')       # the reference's float32 read
        lib.fs_resample_stat(plane.ctypes.data, hs, ws, has_nd, nd, dst[b].ctypes.data, hd, wd, sx, ox, sy, oy,
                             METHOD_CODES[resampling])
    dst = dst.astype(out_dtype, copy=False)
    return dst[0] if squeeze else dst


@contextlib.contextmanager
def with_footprint_stats():
    """ Within the block, ``gdal_restate.reproject_array`` -- and so every function of ``oracle.kernel_model_np`` --
    also restates the six footprint statistics (and, through ``interp_up_restate``, bilinear, cubic and lanczos
    up-sampling). """
    base = gdal_restate.reproject_array
    gdal_restate.reproject_array = reproject_array
    try:
        yield
    finally:
        gdal_restate.reproject_array = base
