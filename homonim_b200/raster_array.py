"""
Geo-referenced masked array container for the B200 kernel-model path.

Host-side mirror of the part of ``homonim.raster_array.RasterArray`` that the kernel-model path touches
(/root/reference/homonim/raster_array.py:43-127, 223-351, 389-391, 526-578; SURVEY.md 8(a) row a15): same
constructor, ``from_profile``, ``array`` / ``mask`` / ``nodata`` / ``profile`` / ``proj_profile`` / ``res`` /
``transform`` / ``shape`` / ``copy`` / ``mask_ra`` semantics and error behaviour.  Differences, all additive:

  * ``array`` may be a numpy array (host) OR a torch CUDA tensor (device-resident raster).  Results of
    ``KernelModel.fit/apply`` live where their inputs live.
  * integer rasters (uint8 / uint16 / int16) may be kept in their stored dtype: the CUDA kernels convert on load, which is
    what the reference's reader does on the host with ``out_dtype='float32'`` (raster_array.py:178-188).
  * no rasterio dependency: ``crs`` is an opaque comparable label, ``transform`` any 6-coefficient affine.
  * file I/O methods (``from_rio_dataset`` / ``to_rio_dataset`` / ``to_file``) are out of scope (SURVEY.md 8, 2).
"""
from typing import Dict, Optional, Tuple, Union

import numpy as np

from homonim_b200.errors import ImageProfileError
from homonim_b200.geometry import Affine, CRS, window_bounds

try:  # torch is plumbing for device memory; the container also works for pure-host use without it
    import torch
except ImportError:  # pragma: no cover
    torch = None

ArrayLike = Union[np.ndarray, 'torch.Tensor']


def is_tensor(a) -> bool:
    return torch is not None and isinstance(a, torch.Tensor)


def nan_equals(a, b):
    """ ``a == b`` treating nan as equal to nan (reference utils.py:54-56); works for numpy arrays and tensors. """
    if is_tensor(a):
        if isinstance(b, float) and np.isnan(b):
            return torch.isnan(a) if a.is_floating_point() else torch.zeros_like(a, dtype=torch.bool)
        return a == b
    with np.errstate(invalid='ignore'):
        return (a == b) | (np.isnan(a) & np.isnan(b))


def _dtype_name(a) -> str:
    return str(a.dtype).replace('torch.', '') if is_tensor(a) else a.dtype.name


class RasterArray:
    default_nodata = float('nan')   # reference raster_array.py:48
    default_dtype = 'float32'       # reference raster_array.py:49

    def __init__(self, array: ArrayLike, crs, transform, nodata: Optional[float] = default_nodata, window=None):
        if (array.ndim < 2) or (array.ndim > 3):
            raise ValueError('`array` must be have 2 or 3 dimensions with bands along the first dimension')
        self._array = array
        if crs is None:
            raise TypeError('`crs` must be provided')
        self._crs = crs
        try:
            self._transform = Affine.coerce(transform)
        except TypeError:
            raise TypeError('`transform` must be an affine transform with 6 coefficients')
        if window is not None:
            col_off, row_off, width, height = (getattr(window, k) for k in ('col_off', 'row_off', 'width', 'height'))
            if (height, width) != tuple(array.shape[-2:]):
                raise ValueError('`window` and `array` width and height must match')
            self._transform = self._transform * Affine.translation(col_off, row_off)
        self._nodata = nodata
        self._mask = None

    @classmethod
    def from_profile(cls, array: Optional[ArrayLike], profile: Dict, window=None) -> 'RasterArray':
        """ Reference raster_array.py:95-127. """
        if not {'crs', 'transform', 'nodata'} <= set(profile):
            raise ImageProfileError("'profile' should include 'crs', 'transform' and 'nodata' keys")
        if array is None:
            if not {'width', 'height', 'count', 'dtype'} <= set(profile):
                raise ImageProfileError("'profile' should include 'width', 'height', 'count' and 'dtype' keys")
            shape = (profile['count'], profile['height'], profile['width'])
            array = np.full(shape, fill_value=profile['nodata'], dtype=profile['dtype'])
        return cls(array, profile['crs'], profile['transform'], nodata=profile['nodata'], window=window)

    # ---- array / geometry properties ------------------------------------------------------------------------------
    @property
    def array(self) -> ArrayLike:
        return self._array

    @array.setter
    def array(self, value: ArrayLike):
        if tuple(value.shape[-2:]) == tuple(self._array.shape[-2:]):
            self._array = value
            self._mask = None
        else:
            raise ValueError("'value' and 'array' shapes must match")

    @property
    def is_device(self) -> bool:
        """ True when the raster lives in GPU memory (torch CUDA tensor). """
        return is_tensor(self._array) and self._array.is_cuda

    @property
    def crs(self):
        return self._crs

    @property
    def width(self) -> int:
        return self.shape[-1]

    @property
    def height(self) -> int:
        return self.shape[-2]

    @property
    def shape(self) -> Tuple[int, int]:
        return tuple(int(s) for s in self._array.shape[-2:])

    @property
    def count(self) -> int:
        return int(self._array.shape[0]) if self._array.ndim == 3 else 1

    @property
    def dtype(self) -> str:
        return _dtype_name(self._array)

    @property
    def transform(self) -> Affine:
        return self._transform

    @property
    def res(self) -> Tuple[float, float]:
        return self._transform.a, -self._transform.e

    @property
    def bounds(self) -> Tuple[float, float, float, float]:
        return window_bounds(self._transform, self.height, self.width)

    @property
    def profile(self) -> Dict:
        return dict(
            crs=self._crs, transform=self._transform, nodata=self._nodata, count=self.count, width=self.width,
            height=self.height, dtype=self.dtype
        )

    @property
    def proj_profile(self) -> Dict:
        return dict(crs=self._crs, transform=self._transform, shape=self.shape)

    # ---- mask / nodata (reference raster_array.py:298-351) --------------------------------------------------------
    @property
    def mask(self):
        """ 2D boolean mask of valid pixels (numpy bool array, or bool tensor for device rasters). """
        if self._mask is None:
            if self._nodata is None:
                if is_tensor(self._array):
                    self._mask = torch.ones(self.shape, dtype=torch.bool, device=self._array.device)
                else:
                    self._mask = np.full(self.shape, True)
            else:
                self._mask = ~nan_equals(self._array, self._nodata)
                if self._array.ndim > 2:
                    self._mask = self._mask.any(0) if is_tensor(self._array) else np.any(self._mask, axis=0)
        return self._mask

    @mask.setter
    def mask(self, value):
        if is_tensor(self._array) and not is_tensor(value):
            value = torch.as_tensor(np.asarray(value), device=self._array.device)
        if self._array.ndim == 2:
            self._array[~value] = self._nodata
        else:
            self._array[:, ~value] = self._nodata
        self._mask = None

    @property
    def mask_ra(self) -> 'RasterArray':
        mask = self.mask
        mask = mask.to(torch.uint8) if is_tensor(mask) else mask.astype('uint8', copy=False)
        return RasterArray(mask, crs=self._crs, transform=self._transform, nodata=None)

    @property
    def nodata(self) -> Optional[float]:
        return self._nodata

    @nodata.setter
    def nodata(self, value: Optional[float]):
        if value is None or self._nodata is None:
            self._nodata = value
            self._mask = None
        elif not bool(nan_equals(np.float64(value), np.float64(self._nodata))):
            nodata_mask = ~self.mask
            if self._array.ndim == 3:
                self._array[:, nodata_mask] = value
            else:
                self._array[nodata_mask] = value
            self._nodata = value
            self._mask = None

    # ---- copies / residency ---------------------------------------------------------------------------------------
    def copy(self) -> 'RasterArray':
        array = self._array.clone() if is_tensor(self._array) else self._array.copy()
        return RasterArray.from_profile(array, self.profile)

    def to_device(self, device='cuda') -> 'RasterArray':
        """ Copy of this raster whose array is a contiguous tensor on ``device`` (no dtype change). """
        if torch is None:
            raise RuntimeError('torch is required for device rasters')
        array = self._array if is_tensor(self._array) else torch.from_numpy(np.ascontiguousarray(self._array))
        return RasterArray(array.to(device, non_blocking=True).contiguous(), self._crs, self._transform,
                           nodata=self._nodata)

    def to_host(self) -> 'RasterArray':
        """ Copy of this raster whose array is a numpy array. """
        array = self._array.detach().cpu().numpy() if is_tensor(self._array) else self._array
        return RasterArray(array, self._crs, self._transform, nodata=self._nodata)

    def reproject(self, crs=None, transform=None, shape: Optional[Tuple[int, int]] = None,
                  nodata: float = default_nodata, dtype: str = default_dtype, resampling='average', **kwargs
                  ) -> 'RasterArray':
        """
        Resample onto another axis-aligned grid of the same CRS on the GPU (reference raster_array.py:526-578, which
        calls GDAL's warper).  Supported: ``average`` (down-sampling), ``cubic_spline`` and ``nearest`` (up-sampling).
        """
        from homonim_b200 import kernel_model   # deferred: avoids a cycle, and loading the native library eagerly
        return kernel_model.reproject_raster(self, crs=crs, transform=transform, shape=shape, nodata=nodata,
                                             dtype=dtype, resampling=resampling)
