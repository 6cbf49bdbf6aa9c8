"""
KernelModel / RefSpaceModel / SrcSpaceModel for B200: the host-side mirror of homonim's kernel-model API.

Same class names, constructor arguments, config keys, return layouts and exceptions as
/root/reference/homonim/kernel_model.py (KernelModel :35-463, RefSpaceModel :466-503, SrcSpaceModel :506-535), so that
``RasterFuse.process`` (fuse.py:376-377, 304-307) and the reference's tests can use these classes unchanged.  All
pixel arithmetic runs in the sm_100a CUDA library behind ``include/homonim_b200.h`` (``_native.py``); there is no
CPU implementation here and none is fallen back to.

Differences from the reference, all deliberate:
  * ``fit`` does not mutate its inputs (the reference zeroes invalid pixels in place, kernel_model.py:246-247).
  * rasters may be host numpy arrays (copied to the device and back) or torch CUDA tensors (stay on the device);
    uint8 / uint16 / int16 sources may be passed in their stored dtype.
  * ``RefSpaceModel.apply`` never materialises the up-sampled parameters: up-sampling and gain*src+offset are one
    kernel.
  * down-sampling is ``average``; up-sampling is ``cubic_spline`` (the default), ``bilinear``, ``cubic``,
    ``lanczos`` or ``nearest``, each as GDAL computes it when the destination is at least as fine as the source (spec:
    oracle/gdal_restate.c, oracle/interp_up_restate.c).  The footprint statistics ``min``, ``max``, ``med``, ``q1``,
    ``q3`` and ``mode`` take any geometry and serve either key (spec: oracle/footprint_stats_restate.c).  Other
    ``downsampling`` / ``upsampling`` choices, and the interpolating up-sampling methods on a down-sampling geometry,
    raise NotImplementedError rather than silently using something else.
  * ``RefSpaceModel.apply`` fuses up-sampling and apply for every up-sampling method but ``nearest``; the one-call
    ``RefSpaceModel.fuse`` (``can_fuse``) is the default resampling pair only.
"""
import functools
import warnings
from typing import Dict, Optional, Tuple

import numpy as np

from homonim_b200 import _native
from homonim_b200.enums import Model, Resampling
from homonim_b200.errors import ConfigWarning
from homonim_b200.geometry import grid_map
from homonim_b200.raster_array import RasterArray, is_tensor

try:
    import torch
except ImportError:  # pragma: no cover
    torch = None

NAN = float('nan')
_DTYPE_CODES = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'int16': _native.HB_I16, 'float32': _native.HB_F32}
_OUT_DTYPE_CODES = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'int16': _native.HB_I16, 'float32': _native.HB_F32}
_MODEL_CODES = {
    Model.gain: _native.HB_MODEL_GAIN,
    Model.gain_blk_offset: _native.HB_MODEL_GAIN_BLK_OFFSET,
    Model.gain_offset: _native.HB_MODEL_GAIN_OFFSET,
}
MAX_SEARCH_DISTANCE = 100.0   # rasterio.fill.fillnodata default used by the reference (kernel_model.py:366)


def validate_kernel_shape(kernel_shape: Tuple[int, int], model: Model = Model.gain_blk_offset) -> Tuple[int, int]:
    """ Reference utils.validate_kernel_shape (utils.py:104-133): same checks, messages and warning. """
    kernel_shape = np.array(kernel_shape).astype(int)
    if not np.all(np.mod(kernel_shape, 2) == 1):
        raise ValueError('`kernel_shape` must be odd in both dimensions.')
    if model == Model.gain_offset:
        if np.prod(kernel_shape) < 2:
            raise ValueError('`kernel_shape` area should contain at least 2 elements for the gain-offset model.')
        elif np.prod(kernel_shape) < 25:
            warnings.warn(
                'A `kernel_shape` of at least 25 elements is recommended for the gain-offset model.',
                category=ConfigWarning
            )
    if not np.all(kernel_shape >= 1):
        raise ValueError('`kernel_shape` must be a minimum of one in both dimensions.')
    return tuple(int(k) for k in kernel_shape)


def overlap_for_kernel(kernel_shape: Tuple[int, int]) -> Tuple[int, int]:
    """ Reference utils.overlap_for_kernel (utils.py:136-153): block overlap = ceil(kernel / 2). """
    kernel_shape = np.array(kernel_shape).astype(int)
    return tuple(int(v) for v in np.ceil(kernel_shape / 2).astype('int'))


# ---------------------------------------------------------------------------------------------------------------------
# device plumbing (torch owns device memory and streams; the kernels are ours)
# ---------------------------------------------------------------------------------------------------------------------
def _require_torch():
    if torch is None:
        raise _native.NativeLibraryError('torch is required for device memory management')
    _native.require_device()


def _stream() -> int:
    """ Raw cudaStream_t of torch's current stream on the current device.  (``torch.cuda.current_stream()`` without a
    device index walks through ``is_available()`` / NVML checks: ~14 us per call, which at 36 native calls per row-band
    step was a quarter of the host time of a step.) """
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def current_stream():
    """ torch's current stream on the current device, by explicit index (the cheap path of ``torch.cuda.current_stream``). """
    return torch.cuda.current_stream(torch._C._cuda_getDevice())


class on_stream:
    """ ``with on_stream(s):`` -- what ``torch.cuda.stream(s)`` does for a stream of the current device, without its
    per-entry device queries. """
    __slots__ = ('stream', 'prev')

    def __init__(self, stream):
        self.stream = stream

    def __enter__(self):
        self.prev = current_stream()
        torch.cuda.set_stream(self.stream)
        return self.stream

    def __exit__(self, *exc):
        torch.cuda.set_stream(self.prev)
        return False


def _on_raster_device(method):
    """ Run a public model method with the first device-resident raster's GPU as the current device: the native entry points
    launch on the current device's stream, and its per-device set-up (function attributes, scratch pool) is keyed by it. """
    @functools.wraps(method)
    def wrapper(self, *args, **kwargs):
        for a in args:
            arr = getattr(a, 'array', None)
            if is_tensor(arr) and arr.is_cuda:
                if arr.device.index != torch.cuda.current_device():
                    with torch.cuda.device(arr.device):
                        return method(self, *args, **kwargs)
                break
        return method(self, *args, **kwargs)
    return wrapper


class KernelTimer:
    """
    Optional per-launch device timing of the C-ABI calls (used by bench.py for the roofline numbers): while active,
    every native call is bracketed by CUDA events on the launching stream.  ``results()`` synchronises and returns
    {entry point: [milliseconds per call]}.
    """
    active: Optional['KernelTimer'] = None

    def __init__(self):
        self._events = []

    def __enter__(self):
        KernelTimer.active = self
        return self

    def __exit__(self, *exc):
        KernelTimer.active = None

    def record(self, name, fn, args):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        rc = fn(*args)
        end.record()
        self._events.append((name, start, end))
        return rc

    def results(self) -> Dict[str, list]:
        torch.cuda.synchronize()
        out: Dict[str, list] = {}
        for name, start, end in self._events:
            out.setdefault(name, []).append(start.elapsed_time(end))
        return out

    def timeline(self, origin) -> list:
        """ ``[(entry point, start ms, end ms)]`` relative to the CUDA event ``origin`` (recorded before the calls), in
        issue order -- where on the device's clock every native call of a multi-stream step ran. """
        torch.cuda.synchronize()
        return [(name, round(origin.elapsed_time(start), 3), round(origin.elapsed_time(end), 3))
                for name, start, end in self._events]


def _call(name: str, *args):
    """ Invoke C-ABI entry point ``name`` and raise on failure. """
    fn = getattr(_native.lib(), name)
    timer = KernelTimer.active
    rc = timer.record(name, fn, args) if timer is not None else fn(*args)
    _native.check(rc, name)


def _nodata_args(nodata) -> Tuple[int, float]:
    return (0, 0.0) if nodata is None else (1, float(nodata))


def _to_device(array, device=None):
    """ Contiguous CUDA tensor for a numpy array / tensor; float64 is narrowed to float32, other dtypes are kept. """
    if is_tensor(array):
        t = array if array.is_cuda else array.to(device or 'cuda', non_blocking=True)
    else:
        array = np.ascontiguousarray(array)
        if array.dtype == np.float64:
            array = array.astype('float32')
        elif array.dtype == np.bool_:
            array = array.astype('uint8')
        t = torch.from_numpy(array).to(device or 'cuda', non_blocking=True)
    if t.dtype == torch.float64:
        t = t.float()
    return t.contiguous()


def _plane_code(t) -> int:
    name = str(t.dtype).replace('torch.', '')
    if name not in _DTYPE_CODES:
        raise TypeError(f'unsupported raster dtype {name!r}: expected uint8, uint16, int16 or float32')
    return _DTYPE_CODES[name]


def _as_f32_plane(t, nodata):
    """ float32 view / copy of a plane for the same-grid kernels (integer planes are widened on the device). """
    if t.dtype == torch.float32:
        return t
    return t.to(torch.float32)


def _as_nan_nodata_f32(t, nodata):
    """ float32 plane whose nodata is NaN (input convention of the cubic-spline up-sampler). """
    f = t.to(torch.float32) if t.dtype != torch.float32 else t
    if nodata is None or (isinstance(nodata, float) and np.isnan(nodata)):
        return f
    return torch.where(f == float(nodata), torch.full_like(f, NAN), f)


def _out_args(out_t, out_nodata) -> Tuple[int, int, float]:
    """
    (out_dtype, out_has_nodata, out_nodata) of a corrected plane for the native apply calls: the tensor's dtype decides
    the stored type; the conversion of RasterArray._convert_array_dtype (raster_array.py:353-387: round half-to-even,
    clip, NaN -> nodata) happens inside the kernel's store.  float32 with NaN / no nodata = the values as they are.
    """
    name = str(out_t.dtype).replace('torch.', '')
    if name not in _OUT_DTYPE_CODES:
        raise TypeError(f'unsupported output dtype {name!r}: expected float32, uint8, uint16 or int16')
    if out_nodata is None or (isinstance(out_nodata, float) and np.isnan(out_nodata)):
        return _OUT_DTYPE_CODES[name], 0, 0.0
    return _OUT_DTYPE_CODES[name], 1, float(out_nodata)


def _result(array_dev, like_device: bool):
    """ Return results where the caller's rasters live. """
    if like_device:
        return array_dev
    return array_dev.cpu().numpy()


class KernelModel:
    default_kernel_shape = (5, 5)           # reference kernel_model.py:37
    default_model = Model.gain_blk_offset   # reference kernel_model.py:38

    def __init__(self, model: Model = default_model, kernel_shape: Tuple[int, int] = default_kernel_shape,
                 find_r2: bool = False, **kwargs):
        self._model = Model(model)
        self._kernel_shape = validate_kernel_shape(kernel_shape, model=model)
        self._find_r2 = find_r2
        config = self.create_config(**kwargs)     # unknown keys raise TypeError, as in the reference
        self._r2_inpaint_thresh: Optional[float] = config['r2_inpaint_thresh']
        self._mask_partial: bool = config['mask_partial']
        self._downsampling = config['downsampling']
        self._upsampling = config['upsampling']

    @property
    def model(self) -> Model:
        return self._model

    @property
    def kernel_shape(self) -> Tuple[int, int]:
        return tuple(self._kernel_shape)

    @property
    def find_r2(self) -> bool:
        return self._find_r2

    @staticmethod
    def create_config(r2_inpaint_thresh: float = 0.25, mask_partial: bool = False,
                      downsampling=Resampling.average, upsampling=Resampling.cubic_spline) -> Dict:
        """ Reference kernel_model.py:98-136: same keys and defaults. """
        return dict(r2_inpaint_thresh=r2_inpaint_thresh, mask_partial=mask_partial, downsampling=downsampling,
                    upsampling=upsampling)

    def _get_resampling(self, from_res, to_res) -> Resampling:
        """ Reference kernel_model.py:138-140. """
        choice = self._downsampling if np.prod(np.abs(from_res)) <= np.prod(np.abs(to_res)) else self._upsampling
        return Resampling.coerce(choice)

    # ---- native steps on device tensors ---------------------------------------------------------------------------
    def _wants_r2(self) -> bool:
        return bool(self._find_r2 or (self._model == Model.gain_offset and self._r2_inpaint_thresh is not None))

    @staticmethod
    def _block_norm(src_t, src_nodata, ref_t, ref_nodata):
        """ Block normalisation (reference kernel_model.py:216-229) of two float32 device planes -> 2 float64s on the
        device. """
        lib = _native.lib()
        src_t, ref_t = _as_f32_plane(src_t, src_nodata).contiguous(), _as_f32_plane(ref_t, ref_nodata).contiguous()
        n = int(src_t.numel())
        s_has, s_nd = _nodata_args(src_nodata)
        r_has, r_nd = _nodata_args(ref_nodata)
        norm = torch.empty(2, dtype=torch.float64, device=src_t.device)
        ws_bytes = lib.hb_block_norm_workspace_bytes(n)
        work = torch.empty(ws_bytes, dtype=torch.uint8, device=src_t.device)
        _call('hb_block_norm', src_t.data_ptr(), s_has, s_nd, ref_t.data_ptr(), r_has, r_nd, n, norm.data_ptr(),
              work.data_ptr(), ws_bytes, _stream())
        return norm

    def _fit_planes(self, src_t, src_nodata, ref_t, ref_nodata, norm=None, rows=None):
        """
        Same-grid fit of two float32 device planes -> float32 [2|3, H, W] parameter tensor.  ``norm``: block
        normalisation computed elsewhere (row-band sharding: the statistics of the WHOLE block, dist.py).  ``rows`` =
        ``(row0, nrows)``: fit only these rows of the planes (a row band inside its halo); the result then holds
        ``nrows`` rows.  With R2 in-painting the whole plane is fitted and in-painted (its search reaches 100 pixels)
        and the rows are cut out afterwards.
        """
        lib = _native.lib()
        h, w = int(src_t.shape[-2]), int(src_t.shape[-1])
        src_t, ref_t = _as_f32_plane(src_t, src_nodata).contiguous(), _as_f32_plane(ref_t, ref_nodata).contiguous()
        want_r2 = self._wants_r2()
        inpaint = self._model == Model.gain_offset and self._r2_inpaint_thresh is not None
        row0, nrows = (0, h) if (rows is None or inpaint) else (int(rows[0]), int(rows[1]))
        params = torch.empty((3 if want_r2 else 2, nrows, w), dtype=torch.float32, device=src_t.device)
        s_has, s_nd = _nodata_args(src_nodata)
        r_has, r_nd = _nodata_args(ref_nodata)
        stream = _stream()
        norm_ptr = None
        if self._model == Model.gain_blk_offset:
            if norm is None:
                norm = self._block_norm(src_t, src_nodata, ref_t, ref_nodata)
            norm_ptr = norm.data_ptr()
        sums = torch.empty((3, h, w), dtype=torch.float32, device=src_t.device) if inpaint else None
        kh, kw = self._kernel_shape
        _call('hb_fit_same_grid_rows', src_t.data_ptr(), s_has, s_nd, ref_t.data_ptr(), r_has, r_nd, h, w, row0, nrows,
              _MODEL_CODES[self._model], kh, kw, int(want_r2), norm_ptr, params.data_ptr(),
              sums.data_ptr() if inpaint else None, stream)
        if inpaint:
            ws_bytes = lib.hb_inpaint_workspace_bytes(h, w)
            work = torch.empty(ws_bytes, dtype=torch.uint8, device=src_t.device)
            _call('hb_inpaint_refit', params.data_ptr(), sums.data_ptr(), h, w,
                                               float(self._r2_inpaint_thresh), MAX_SEARCH_DISTANCE, work.data_ptr(),
                                               ws_bytes, stream)
            if rows is not None:
                params = params[:, int(rows[0]):int(rows[0]) + int(rows[1])].contiguous()
        return params

    def _fit_apply_rows(self, src_t, src_nodata, ref_t, ref_nodata, row0, nrows, norm=None, out=None, out_nodata=NAN):
        """
        Fit fused with apply (``hb_fit_apply_same_grid_rows``) for the rows ``[row0, row0 + nrows)`` of two float32 device
        planes on one grid -> corrected float32 ``[nrows, W]``.  The parameters are not materialised (models whose
        parameters are final after the fit: everything but gain-offset with R2 in-painting).
        """
        if self._model == Model.gain_offset and self._r2_inpaint_thresh is not None:
            raise ValueError('fit + apply in one kernel is not available with R2 in-painting')
        h, w = int(src_t.shape[-2]), int(src_t.shape[-1])
        if src_t.dtype != torch.float32 or ref_t.dtype != torch.float32 or not src_t.is_contiguous() \
                or not ref_t.is_contiguous():
            raise ValueError('fit + apply in one kernel needs contiguous float32 planes')
        corr = self._check_out(out, int(nrows), w, src_t.device)
        if self._model == Model.gain_blk_offset and norm is None:
            norm = self._block_norm(src_t, src_nodata, ref_t, ref_nodata)
        s_has, s_nd = _nodata_args(src_nodata)
        r_has, r_nd = _nodata_args(ref_nodata)
        kh, kw = self._kernel_shape
        _call('hb_fit_apply_same_grid_rows', src_t.data_ptr(), s_has, s_nd, ref_t.data_ptr(), r_has, r_nd, h, w,
              int(row0), int(nrows), _MODEL_CODES[self._model], kh, kw, norm.data_ptr() if norm is not None else None,
              *_out_args(corr, out_nodata), corr.data_ptr(), _stream())
        return corr

    def _full_coverage_mask(self, in_mask_t, in_transform, params_t, param_transform):
        """ Reference kernel_model.py:375-409 on device: uint8 [hp, wp] mask on the parameter grid. """
        lib = _native.lib()
        hp, wp = int(params_t.shape[-2]), int(params_t.shape[-1])
        hi, wi = int(in_mask_t.shape[-2]), int(in_mask_t.shape[-1])
        gm = grid_map(in_transform, param_transform)          # param grid -> in_mask grid
        out = torch.empty((hp, wp), dtype=torch.uint8, device=params_t.device)
        work = torch.empty((hp, wp), dtype=torch.uint8, device=params_t.device)
        kh, kw = self._kernel_shape
        _call('hb_full_coverage_mask', in_mask_t.data_ptr(), hi, wi, params_t.data_ptr(), hp, wp, gm.sx,
                                                gm.ox, gm.sy, gm.oy, kh, kw, out.data_ptr(), work.data_ptr(),
                                                _stream())
        return out

    @staticmethod
    def _valid_mask_u8(t, nodata):
        lib = _native.lib()
        has, nd = _nodata_args(nodata)
        mask = torch.empty(tuple(t.shape[-2:]), dtype=torch.uint8, device=t.device)
        _call('hb_valid_mask', t.data_ptr(), _plane_code(t), t.numel(), has, nd, mask.data_ptr(), _stream())
        return mask

    # ---- public API (reference kernel_model.py:411-463) -----------------------------------------------------------
    @_on_raster_device
    def fit(self, src_ra: RasterArray, ref_ra: RasterArray) -> RasterArray:
        if (ref_ra.transform != src_ra.transform) or (ref_ra.shape != src_ra.shape):
            raise ValueError("'ref_ra' and 'src_ra' must have the same CRS, transform and shape")
        _require_torch()
        on_device = src_ra.is_device and ref_ra.is_device
        src_t, ref_t = _to_device(src_ra.array), _to_device(ref_ra.array)
        params = self._fit_planes(src_t, src_ra.nodata, ref_t, ref_ra.nodata)
        return RasterArray(_result(params, on_device), src_ra.crs, src_ra.transform, nodata=NAN)

    @_on_raster_device
    def apply(self, src_ra: RasterArray, param_ra: RasterArray, out=None, out_nodata=NAN) -> RasterArray:
        """
        Reference kernel_model.py:442-463.  ``out`` (optional, additive): a CUDA tensor ``[H, W]`` to write the corrected
        band into (device-resident callers avoid a copy); the returned RasterArray then wraps it.  ``out`` may be
        float32 (the reference's result, nodata NaN) or uint8 / uint16 / int16 with ``out_nodata``: the output dtype
        conversion the reference performs when it writes the block (raster_array.py:353-387, 493-500) is then fused into
        the apply kernel.
        """
        if (param_ra.transform != src_ra.transform) or (param_ra.shape != src_ra.shape):
            raise ValueError("'param_ra' and 'src_ra' must have the same CRS, transform and shape")
        _require_torch()
        on_device = (src_ra.is_device and param_ra.is_device) or out is not None
        src_t, par_t = _to_device(src_ra.array), _to_device(param_ra.array)
        corr = self._apply_planes(src_t, src_ra.nodata, par_t, mask_src=False, out=out, out_nodata=out_nodata)
        return RasterArray(_result(corr, on_device), param_ra.crs, param_ra.transform,
                           nodata=param_ra.nodata if out is None else out_nodata)

    @staticmethod
    def _check_out(out, h, w, device):
        if out is None:
            return torch.empty((h, w), dtype=torch.float32, device=device)
        if (not is_tensor(out)) or (not out.is_cuda) or tuple(out.shape) != (h, w) or not out.is_contiguous() \
                or str(out.dtype).replace('torch.', '') not in _OUT_DTYPE_CODES:
            raise ValueError("'out' must be a contiguous float32 / uint8 / uint16 / int16 CUDA tensor with the shape of "
                             "'src_ra'")
        return out

    @staticmethod
    def _apply_planes(src_t, src_nodata, par_t, mask_src: bool, out=None, out_nodata=NAN):
        lib = _native.lib()
        if par_t.ndim != 3 or par_t.shape[0] < 2 or par_t.dtype != torch.float32:
            raise ValueError("'param_ra' must hold at least 2 float32 bands (gain, offset)")
        h, w = int(src_t.shape[-2]), int(src_t.shape[-1])
        corr = KernelModel._check_out(out, h, w, src_t.device)
        has, nd = _nodata_args(src_nodata)
        _call('hb_apply_same_grid', src_t.data_ptr(), _plane_code(src_t), has, nd, int(mask_src), par_t.data_ptr(), h, w,
              *_out_args(corr, out_nodata), corr.data_ptr(), _stream())
        return corr


# ---------------------------------------------------------------------------------------------------------------------
# resampling between grids (reference RasterArray.reproject, raster_array.py:526-578)
# ---------------------------------------------------------------------------------------------------------------------
def _downsample_average(src_t, src_transform, src_nodata, dst_shape, dst_transform):
    """ float32 [hd, wd] (NaN nodata) average of a uint8 / uint16 / int16 / float32 plane. """
    lib = _native.lib()
    gm = grid_map(src_transform, dst_transform)
    hs, ws = int(src_t.shape[-2]), int(src_t.shape[-1])
    hd, wd = int(dst_shape[0]), int(dst_shape[1])
    dst = torch.empty((hd, wd), dtype=torch.float32, device=src_t.device)
    has, nd = _nodata_args(src_nodata)
    _call('hb_downsample_average', src_t.data_ptr(), _plane_code(src_t), hs, ws, has, nd, dst.data_ptr(), hd,
                                            wd, gm.sx, gm.ox, gm.sy, gm.oy, _stream())
    return dst


# footprint statistics (any geometry) and their C-ABI codes
_STAT_METHODS = {
    Resampling.min: _native.HB_STAT_MIN,
    Resampling.max: _native.HB_STAT_MAX,
    Resampling.med: _native.HB_STAT_MED,
    Resampling.q1: _native.HB_STAT_Q1,
    Resampling.q3: _native.HB_STAT_Q3,
    Resampling.mode: _native.HB_STAT_MODE,
}


def _resample_stat(src_t, src_transform, src_nodata, dst_shape, dst_transform, method):
    """ float32 [hd, wd] (NaN nodata) footprint statistic ``method`` (an ``HB_STAT_*`` code) of a uint8 / uint16 /
    int16 / float32 plane. """
    gm = grid_map(src_transform, dst_transform)
    hs, ws = int(src_t.shape[-2]), int(src_t.shape[-1])
    hd, wd = int(dst_shape[0]), int(dst_shape[1])
    dst = torch.empty((hd, wd), dtype=torch.float32, device=src_t.device)
    has, nd = _nodata_args(src_nodata)
    _call('hb_resample_stat', src_t.data_ptr(), _plane_code(src_t), hs, ws, has, nd, dst.data_ptr(), hd, wd, gm.sx,
          gm.ox, gm.sy, gm.oy, method, _stream())
    return dst


# up-sampling methods with an sm_100a kernel, and their C-ABI codes
_UP_METHODS = {
    Resampling.cubic_spline: _native.HB_UP_CUBIC_SPLINE,
    Resampling.bilinear: _native.HB_UP_BILINEAR,
    Resampling.cubic: _native.HB_UP_CUBIC,
    Resampling.lanczos: _native.HB_UP_LANCZOS,
    Resampling.nearest: _native.HB_UP_NEAREST,
}
# the ones that up-sample with GDAL's tap rules (NaN nodata, 1 or 2 bands per native call) and have a fused apply
_UP_INTERP = (Resampling.cubic_spline, Resampling.bilinear, Resampling.cubic, Resampling.lanczos)


def _resample_up(src_t, src_transform, src_nodata, dst_shape, dst_transform, method=_native.HB_UP_CUBIC_SPLINE):
    """ float32 [nb, hd, wd] (NaN nodata) up-sampling of 1 or 2 float32 bands. """
    lib = _native.lib()
    gm = grid_map(src_transform, dst_transform)
    squeeze = src_t.ndim == 2
    src3 = src_t[None] if squeeze else src_t
    if method != _native.HB_UP_NEAREST:
        src3 = _as_nan_nodata_f32(src3, src_nodata).contiguous()
        has, nd = 1, NAN
    else:
        src3 = src3.to(torch.float32).contiguous()
        has, nd = _nodata_args(src_nodata)
    nb, hs, ws = (int(v) for v in src3.shape)
    hd, wd = int(dst_shape[0]), int(dst_shape[1])
    dst = torch.empty((nb, hd, wd), dtype=torch.float32, device=src_t.device)
    for b0 in range(0, nb, 2):     # the native up-sampler takes 1 or 2 bands per call
        nbc = min(2, nb - b0)
        _call('hb_resample_up', src3[b0:b0 + nbc].data_ptr(), nbc, hs, ws, has, nd, dst[b0:].data_ptr(), hd,
                                         wd, gm.sx, gm.ox, gm.sy, gm.oy, method, _stream())
    return dst[0] if squeeze else dst


def _resample_plane(t, transform, nodata, dst_shape, dst_transform, resampling: Resampling):
    """ Resample one plane to a float32, NaN-nodata plane on the destination grid. """
    if resampling == Resampling.average:
        return _downsample_average(t, transform, nodata, dst_shape, dst_transform)
    if resampling in _UP_METHODS:
        if resampling in (Resampling.bilinear, Resampling.cubic, Resampling.lanczos):
            gm = grid_map(transform, dst_transform)
            if gm.sx > 1.0 + 1e-9 or gm.sy > 1.0 + 1e-9:
                raise NotImplementedError(
                    f'resampling {resampling.value!r} is only implemented for up-sampling (a destination grid at least '
                    f'as fine as the source); down-sampling is implemented for average only'
                )
        return _resample_up(t, transform, nodata, dst_shape, dst_transform, _UP_METHODS[resampling])
    if resampling in _STAT_METHODS:
        return _resample_stat(t, transform, nodata, dst_shape, dst_transform, _STAT_METHODS[resampling])
    raise NotImplementedError(
        f'resampling {resampling.value!r} has no sm_100a kernel yet (available: average for down-sampling; '
        f'cubic_spline, bilinear, cubic, lanczos and nearest for up-sampling)'
    )


def reproject_raster(ra: RasterArray, crs=None, transform=None, shape=None, nodata=NAN, dtype='float32',
                     resampling='average') -> RasterArray:
    """ GPU stand-in for RasterArray.reproject on axis-aligned grids of one CRS (raster_array.py:526-578). """
    if transform is not None and shape is None:
        raise ValueError('If `transform` is specified, `shape` is required')
    if crs is not None and crs != ra.crs:
        raise NotImplementedError('re-projection between different CRSs is outside the B200 kernel-model path')
    _require_torch()
    transform = ra.transform if transform is None else transform
    shape = ra.shape if shape is None else shape
    resampling = Resampling.coerce(resampling)
    src_t = _to_device(ra.array)
    planes = [src_t] if src_t.ndim == 2 else list(src_t)
    out = torch.stack([_resample_plane(p.contiguous(), ra.transform, ra.nodata, shape, transform, resampling)
                       for p in planes])
    if nodata is not None and not np.isnan(nodata):
        out = torch.where(torch.isnan(out), torch.full_like(out, float(nodata)), out)
    elif nodata is None:
        out = torch.nan_to_num(out, nan=0.0)
    if dtype not in (None, 'float32'):
        out = out.to(getattr(torch, str(dtype)))
    out = out[0] if src_t.ndim == 2 else out
    return RasterArray(_result(out, ra.is_device), ra.crs, transform, nodata=nodata)


class RefSpaceModel(KernelModel):
    """ Fit on the reference grid, apply on the source grid (reference kernel_model.py:466-503). """

    @_on_raster_device
    def fit(self, src_ra: RasterArray, ref_ra: RasterArray) -> RasterArray:
        _require_torch()
        on_device = src_ra.is_device and ref_ra.is_device
        resampling = self._get_resampling(src_ra.res, ref_ra.res)                            # :478
        src_t, ref_t = _to_device(src_ra.array), _to_device(ref_ra.array)
        src_ds = _resample_plane(src_t, src_ra.transform, src_ra.nodata, ref_ra.shape, ref_ra.transform,
                                 resampling)                                                 # :480
        params = self._fit_planes(src_ds, NAN, ref_t, ref_ra.nodata)                         # :482
        return RasterArray(_result(params, on_device), ref_ra.crs, ref_ra.transform, nodata=NAN)

    def can_fuse(self, src_ra: RasterArray, ref_ra: RasterArray) -> bool:
        """ True when fit + apply of this pair can run as ONE native call (`fuse`): the default resampling pair, no
        partial-coverage masking, and no per-entry-point timer active. """
        if self._mask_partial or KernelTimer.active is not None:
            return False
        if self._get_resampling(src_ra.res, ref_ra.res) != Resampling.average:
            return False
        return self._get_resampling(ref_ra.res, src_ra.res) == Resampling.cubic_spline

    @_on_raster_device
    def fuse(self, src_ra: RasterArray, ref_ra: RasterArray, out=None, want_params: bool = False, out_nodata=NAN
             ) -> Tuple[RasterArray, Optional[RasterArray]]:
        """
        ``apply(src_ra, fit(src_ra, ref_ra))`` -- one (band, block) of ``RasterFuse._process_block`` (fuse.py:304-307)
        -- as a single native call (``hb_fuse_refspace``): the same kernels in the same order, without the host work
        between them.  Returns ``(corr_ra, param_ra or None)``.
        """
        _require_torch()
        on_device = (src_ra.is_device and ref_ra.is_device) or out is not None
        src_t, ref_t = _to_device(src_ra.array), _to_device(ref_ra.array)
        ref_t = _as_f32_plane(ref_t, ref_ra.nodata).contiguous()
        gm = grid_map(src_ra.transform, ref_ra.transform)         # reference grid -> source grid
        corr, params = self._fuse_planes(src_t, src_ra.nodata, ref_t, ref_ra.nodata, gm, out, want_params, out_nodata)
        corr_ra = RasterArray(_result(corr, on_device), src_ra.crs, src_ra.transform, nodata=out_nodata)
        param_ra = None
        if params is not None:
            param_ra = RasterArray(_result(params, on_device), ref_ra.crs, ref_ra.transform, nodata=NAN)
        return corr_ra, param_ra

    def _fuse_planes(self, src_t, src_nodata, ref_t, ref_nodata, gm, out=None, want_params: bool = False,
                     out_nodata=NAN):
        """ `fuse` on prepared device planes (``ref_t``: contiguous float32; ``gm``: reference grid -> source grid):
        returns ``(corr, params or None)`` device tensors.  The lean inner call of ``RasterFuse.process``. """
        hs, ws = int(src_t.shape[-2]), int(src_t.shape[-1])
        hr, wr = int(ref_t.shape[-2]), int(ref_t.shape[-1])
        corr = self._check_out(out, hs, ws, src_t.device)
        want_r2 = self._wants_r2()
        inpaint = self._model == Model.gain_offset and self._r2_inpaint_thresh is not None
        params = None
        if want_params:
            params = torch.empty((3 if want_r2 else 2, hr, wr), dtype=torch.float32, device=src_t.device)
        s_has, s_nd = _nodata_args(src_nodata)
        r_has, r_nd = _nodata_args(ref_nodata)
        kh, kw = self._kernel_shape
        _call('hb_fuse_refspace', src_t.data_ptr(), _plane_code(src_t), hs, ws, s_has, s_nd, ref_t.data_ptr(), hr, wr,
              r_has, r_nd, gm.sx, gm.ox, gm.sy, gm.oy, _MODEL_CODES[self._model], kh, kw, int(want_r2), int(inpaint),
              float(self._r2_inpaint_thresh) if inpaint else 0.0, *_out_args(corr, out_nodata), corr.data_ptr(),
              params.data_ptr() if params is not None else None, _stream())
        return corr, params

    @_on_raster_device
    def apply(self, src_ra: RasterArray, param_ra: RasterArray, out=None, out_nodata=NAN) -> RasterArray:
        _require_torch()
        lib = _native.lib()
        on_device = (src_ra.is_device and param_ra.is_device) or out is not None
        src_t, par_t = _to_device(src_ra.array), _to_device(param_ra.array)
        if par_t.ndim != 3 or par_t.shape[0] < 2 or par_t.dtype != torch.float32:
            raise ValueError("'param_ra' must hold at least 2 float32 bands (gain, offset)")
        par2 = par_t[:2].contiguous()                                                        # :487
        resampling = self._get_resampling(param_ra.res, src_ra.res)                          # :489
        hs, ws = src_ra.shape
        cover = None
        if self._mask_partial:
            src_mask = self._valid_mask_u8(src_t, src_ra.nodata)
            cover = self._full_coverage_mask(src_mask, src_ra.transform, par2, param_ra.transform)   # :495
        if resampling in _UP_INTERP:
            # fused up-sample + apply (:491, :497-503): the up-sampled parameters never reach memory
            gm = grid_map(param_ra.transform, src_ra.transform)       # source grid -> param grid
            hp, wp = int(par2.shape[-2]), int(par2.shape[-1])
            corr = self._check_out(out, hs, ws, src_t.device)
            has, nd = _nodata_args(src_ra.nodata)
            _call('hb_upsample_apply', src_t.data_ptr(), _plane_code(src_t), hs, ws, has, nd,
                                                par2.data_ptr(), hp, wp, gm.sx, gm.ox, gm.sy, gm.oy,
                                                cover.data_ptr() if cover is not None else None,
                                                *_out_args(corr, out_nodata), corr.data_ptr(),
                                                _UP_METHODS[resampling], _stream())
        else:
            # parameters finer than (or as fine as) the source: resample them, then the same-grid apply
            par_us = torch.stack([_resample_plane(par2[b], param_ra.transform, NAN, (hs, ws), src_ra.transform,
                                                  resampling) for b in range(2)])
            if cover is not None:
                cover_us = _resample_up(cover.to(torch.float32), param_ra.transform, None, (hs, ws),
                                        src_ra.transform, _native.HB_UP_NEAREST)
                par_us[:, ~(cover_us > 0)] = NAN                                             # :497-498
                corr = self._apply_planes(src_t, src_ra.nodata, par_us, mask_src=False, out=out, out_nodata=out_nodata)
            else:
                corr = self._apply_planes(src_t, src_ra.nodata, par_us, mask_src=True, out=out,
                                          out_nodata=out_nodata)                                      # :500
        return RasterArray(_result(corr, on_device), src_ra.crs, src_ra.transform,
                           nodata=NAN if out is None else out_nodata)


class SrcSpaceModel(KernelModel):
    """ Fit and apply on the source grid (reference kernel_model.py:506-535). """

    def can_fuse(self, src_ra: RasterArray, ref_ra: RasterArray) -> bool:
        """ True when apply(fit()) can run with the apply step fused into the fit kernel (`fuse`): the parameters are
        final after the fit (no R2 in-painting) and no partial-coverage masking.  (The fused form is still one C-ABI
        call per kernel, so a per-entry-point timer sees the same launches as an untimed call.) """
        if self._mask_partial:
            return False
        return not (self._model == Model.gain_offset and self._r2_inpaint_thresh is not None)

    @_on_raster_device
    def fuse(self, src_ra: RasterArray, ref_ra: RasterArray, out=None, out_nodata=NAN) -> RasterArray:
        """
        ``apply(src_ra, fit(src_ra, ref_ra))`` without materialising the parameters: the reference image is resampled to
        the source grid (kernel_model.py:518-520) and ``hb_fit_apply_same_grid`` writes the corrected pixels straight
        from the fit kernel's epilogue (8 bytes in + 4 out per pixel instead of 16 + 16).  Bit-identical to the two-step
        path.
        """
        _require_torch()
        on_device = (src_ra.is_device and ref_ra.is_device) or out is not None
        resampling = self._get_resampling(ref_ra.res, src_ra.res)
        src_t, ref_t = _to_device(src_ra.array), _to_device(ref_ra.array)
        ref_us = _resample_plane(ref_t, ref_ra.transform, ref_ra.nodata, src_ra.shape, src_ra.transform, resampling)
        src_f = _as_f32_plane(src_t, src_ra.nodata).contiguous()
        h, w = int(src_f.shape[-2]), int(src_f.shape[-1])
        corr = self._check_out(out, h, w, src_f.device)
        norm = None
        if self._model == Model.gain_blk_offset:
            norm = self._block_norm(src_f, src_ra.nodata, ref_us, NAN)
        s_has, s_nd = _nodata_args(src_ra.nodata)
        kh, kw = self._kernel_shape
        _call('hb_fit_apply_same_grid', src_f.data_ptr(), s_has, s_nd, ref_us.data_ptr(), 1, NAN, h, w,
              _MODEL_CODES[self._model], kh, kw, norm.data_ptr() if norm is not None else None,
              *_out_args(corr, out_nodata), corr.data_ptr(), _stream())
        return RasterArray(_result(corr, on_device), src_ra.crs, src_ra.transform, nodata=out_nodata)

    @_on_raster_device
    def fit(self, src_ra: RasterArray, ref_ra: RasterArray) -> RasterArray:
        _require_torch()
        on_device = src_ra.is_device and ref_ra.is_device
        resampling = self._get_resampling(ref_ra.res, src_ra.res)                            # :518
        src_t, ref_t = _to_device(src_ra.array), _to_device(ref_ra.array)
        ref_us = _resample_plane(ref_t, ref_ra.transform, ref_ra.nodata, src_ra.shape, src_ra.transform,
                                 resampling)                                                 # :520
        params = self._fit_planes(src_t, src_ra.nodata, ref_us, NAN)                         # :524
        if self._mask_partial:
            ref_mask = self._valid_mask_u8(ref_t, ref_ra.nodata)
            cover = self._full_coverage_mask(ref_mask, ref_ra.transform, params[:2].contiguous(),
                                             src_ra.transform)                               # :528-530
            params[:, cover == 0] = NAN                                                      # :531
        # (:533 -- re-masking with the source mask is a no-op: the fit already wrote NaN wherever src is invalid)
        return RasterArray(_result(params, on_device), src_ra.crs, src_ra.transform, nodata=NAN)
