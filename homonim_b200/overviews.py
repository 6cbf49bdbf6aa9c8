"""
Internal overviews of the output GeoTIFFs (reference fuse.py:151-165, ``RasterFuse._build_overviews``): how many levels a
written image gets, and the 2x average pyramid of its device planes (``hb_build_overviews``, csrc/overviews.cu).  The
pyramid is built from the planes as written -- output dtype and nodata -- each level from the previous one as stored.
"""
import ctypes
from typing import List, Optional, Sequence

import numpy as np

from homonim_b200 import _native

try:
    import torch
except ImportError:  # pragma: no cover
    torch = None

_DTYPES = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'int16': _native.HB_I16, 'float32': _native.HB_F32}
OVERVIEW_DTYPES = tuple(_DTYPES)        # output dtypes whose files get overviews
MAX_LEVELS = 8


def overview_factors(shape: Sequence[int], max_num_levels: int = MAX_LEVELS, min_level_pixels: int = 256) -> List[int]:
    """ Decimation factors of the overviews the reference builds for an image of ``shape`` (..., height, width):
    ``[2, 4, ..., 2 ** n]`` with ``n = min(max_num_levels, int(log2(min(height, width) / min_level_pixels)))`` --
    none for a side under ``2 * min_level_pixels``. """
    height, width = shape[-2:]
    num_levels = min(max_num_levels, int(np.log2(min(height, width) / min_level_pixels)))
    return [2 ** m for m in range(1, num_levels + 1)]


def level_shape(shape: Sequence[int], factor: int):
    """ (..., ceil(height / factor), ceil(width / factor)): the shape of the overview of decimation ``factor``. """
    return tuple(shape[:-2]) + (-(-shape[-2] // factor), -(-shape[-1] // factor))


def build_overviews(plane, nodata: Optional[float], n_levels: int) -> list:
    """
    Levels ``1..n_levels`` (factors 2, 4, ..., ``2 ** n_levels``) of the average pyramid of ``plane``, a contiguous CUDA
    tensor ``[H, W]`` or ``[B, H, W]`` of uint8, uint16, int16 or float32 holding the values as written.  Pixel (i, j) of
    a level averages the valid pixels of the 2 x 2 window (i, j) of the level before it; ``nodata`` (None: none) and, in
    float32 planes, NaN mark invalid pixels, and a window without valid pixels is ``nodata`` (NaN for float32 without
    one).  Integer levels round half up; float32 levels sum in double.  Runs on the tensor's device and the current
    stream (two kernel launches at most); returns a list of CUDA tensors of the plane's dtype.
    """
    if torch is None or not isinstance(plane, torch.Tensor):
        raise TypeError('`plane` must be a CUDA tensor')
    if not plane.is_cuda:
        raise TypeError('`plane` must be a CUDA tensor (overviews are built on the GPU)')
    dtype = str(plane.dtype).replace('torch.', '')
    if dtype not in _DTYPES:
        raise ValueError(f'overviews are built for {", ".join(OVERVIEW_DTYPES)} planes, not {dtype}')
    if plane.ndim not in (2, 3) or plane.numel() == 0:
        raise ValueError('`plane` must be a non-empty [H, W] or [B, H, W] tensor')
    if not plane.is_contiguous():
        raise ValueError('`plane` must be contiguous')
    n_levels = int(n_levels)
    if not 0 <= n_levels <= MAX_LEVELS:
        raise ValueError(f'`n_levels` must be in [0, {MAX_LEVELS}]')
    if n_levels == 0:
        return []
    levels = [torch.empty(level_shape(plane.shape, 2 ** k), dtype=plane.dtype, device=plane.device)
              for k in range(1, n_levels + 1)]
    nb = plane.shape[0] if plane.ndim == 3 else 1
    has, nd = (0, 0.0) if nodata is None else (1, float(nodata))
    pointers = (ctypes.c_void_p * n_levels)(*[lv.data_ptr() for lv in levels])
    from homonim_b200 import kernel_model as km
    with torch.cuda.device(plane.device):
        km._call('hb_build_overviews', plane.data_ptr(), _DTYPES[dtype], nb, plane.shape[-2], plane.shape[-1], has, nd,
                 n_levels, pointers, km._stream())
    return levels
