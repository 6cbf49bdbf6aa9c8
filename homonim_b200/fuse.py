"""
RasterFuse for B200: the caller of the kernel-model path, for in-memory rasters and GeoTIFF files.

Mirrors the user-facing surface of ``homonim.RasterFuse`` that reaches the hot path
(/root/reference/homonim/fuse.py:44-149 config factories, :295-408 ``_process_block`` / ``process``;
raster_pair.py:194-225 ``proc_crs`` resolution, :280-296 processing windows): same constructor and ``process``
signatures, config dictionaries, model selection (``SrcSpaceModel if proc_crs == src else RefSpaceModel``,
fuse.py:376-377) and per-band fit -> apply flow (fuse.py:304-307).

Sources and references are :class:`~homonim_b200.raster_array.RasterArray` objects (host numpy or CUDA tensors), for
which ``process`` RETURNS the corrected (and optionally parameter) rasters, or GeoTIFF file names, for which it also
writes the corrected / parameter files as the reference does (band matching by wavelength, metadata, and -- with
``build_ovw=True``, the default -- internal average overviews built on the GPU from the planes as written; see
:mod:`homonim_b200.overviews`).  The reference's block grid exists to bound host memory (raster_pair.py:227-269); on a
180 GB B200 a whole band is one block, which is also the reference's own result for ``max_block_mem`` large enough
(SURVEY.md 7.4-5).
"""
import pathlib
import threading
import warnings
from multiprocessing import cpu_count
from typing import Dict, List, Optional, Tuple, Union

import numpy as np

from homonim_b200.enums import Model, ProcCrs
from homonim_b200.errors import ConfigWarning, ImageContentError, IoError
from homonim_b200.files import FilePair, is_path
from homonim_b200.geometry import Affine
from homonim_b200.kernel_model import (KernelModel, RefSpaceModel, SrcSpaceModel, current_stream, on_stream,
                                       overlap_for_kernel)
from homonim_b200.overviews import OVERVIEW_DTYPES, build_overviews, level_shape, overview_factors
from homonim_b200.raster_array import RasterArray, is_tensor

try:
    import torch
except ImportError:  # pragma: no cover
    torch = None


_STREAM_POOLS: Dict[int, list] = {}
_STREAM_POOLS_LOCK = threading.Lock()


def _band_streams(n: int) -> list:
    """
    Persistent per-device pool of CUDA streams for band-level concurrency.  Re-using the same streams lets torch's
    caching allocator re-use each stream's blocks from one ``process`` call to the next (fresh streams would mean
    fresh cudaMallocs for every band).
    """
    dev = torch.cuda.current_device()
    with _STREAM_POOLS_LOCK:
        pool = _STREAM_POOLS.setdefault(dev, [])
        while len(pool) < n:
            pool.append(torch.cuda.Stream(device=dev))
        return pool[:n]


def _validate_threads(threads: int) -> int:
    """ Reference utils.validate_threads (utils.py:156-164). """
    _cpu_count = cpu_count()
    threads = _cpu_count if threads == 0 else threads
    if threads > _cpu_count:
        raise ValueError(f"'threads' is limited to the number of processors ({_cpu_count})")
    return threads


def _band(ra: RasterArray, index: int) -> RasterArray:
    """ Single-band (2D) RasterArray view of 1-based band ``index`` (bands are read singly, raster_pair.py:333-339). """
    array = ra.array if ra.array.ndim == 2 else ra.array[index - 1]
    return RasterArray(array, ra.crs, ra.transform, nodata=ra.nodata)


def ref_window_for_src(src_ra: RasterArray, ref_ra: RasterArray) -> Tuple[int, int, int, int]:
    """
    (row_off, col_off, height, width) of the reference window covering the source extent, expanded to whole
    reference pixels (raster_pair.py:292-296, utils.expand_window_to_grid) and clipped to the reference raster.
    """
    left, bottom, right, top = src_ra.bounds
    inv = ~ref_ra.transform
    c0, r0 = inv * (left, top)
    c1, r1 = inv * (right, bottom)
    col0, col1 = int(np.floor(min(c0, c1))), int(np.ceil(max(c0, c1)))
    row0, row1 = int(np.floor(min(r0, r1))), int(np.ceil(max(r0, r1)))
    col0, row0 = max(col0, 0), max(row0, 0)
    col1, row1 = min(col1, ref_ra.width), min(row1, ref_ra.height)
    if col1 <= col0 or row1 <= row0:
        raise ImageContentError('The reference image does not overlap the source image.')
    return row0, col0, row1 - row0, col1 - col0


class RasterFuse:

    def __init__(self, src: RasterArray, ref: RasterArray, proc_crs: ProcCrs = ProcCrs.auto,
                 src_bands: Optional[List[int]] = None, ref_bands: Optional[List[int]] = None, force: bool = False):
        """
        Correct a source raster to surface reflectance by fusion with a reference (reference fuse.py:46-87,
        matched_pair.py:38-83).  ``src`` / ``ref`` are RasterArrays on north-up grids of the same CRS; ``src_bands`` /
        ``ref_bands`` are 1-based band indexes (default: all bands, matched in order).
        """
        self._files = None
        if is_path(src) and is_path(ref):
            # GeoTIFF file names, as the reference takes them: open, match the bands by wavelength (matched_pair.py),
            # and stage the matched bands (in matched order) for the GPU path
            self._files = FilePair(src, ref, src_bands=src_bands, ref_bands=ref_bands, force=force)
            src, ref, src_bands, ref_bands = self._files.src_ra, self._files.ref_ra, None, None
        if not isinstance(src, RasterArray) or not isinstance(ref, RasterArray):
            raise TypeError('`src` and `ref` must both be GeoTIFF file names, or both be RasterArray objects')
        if src.crs != ref.crs:
            raise NotImplementedError('source and reference must share a CRS (CRS re-projection is out of scope)')
        self._src, self._ref = src, ref
        self._src_bands = list(src_bands) if src_bands is not None else list(range(1, src.count + 1))
        self._ref_bands = list(ref_bands) if ref_bands is not None else list(range(1, ref.count + 1))
        if len(self._ref_bands) < len(self._src_bands):
            raise ImageContentError(
                f'The reference has fewer bands ({len(self._ref_bands)}) than the source ({len(self._src_bands)}).'
            )
        self._ref_bands = self._ref_bands[:len(self._src_bands)]
        self._proc_crs = self._resolve_proc_crs(src, ref, ProcCrs(proc_crs))
        self._closed = True
        # `process` keeps its working state in locals and may be called from several threads at once; the only state
        # they share is the per-band plan cache (the reference's write locks, fuse.py:92-93, guard its output FILES)
        self._plan_lock = threading.Lock()
        self._plans: Dict[int, tuple] = {}

    @staticmethod
    def _resolve_proc_crs(src: RasterArray, ref: RasterArray, proc_crs: ProcCrs = ProcCrs.auto) -> ProcCrs:
        """ Reference raster_pair.py:194-225. """
        src_pixel_smaller = np.prod(np.abs(src.res)) <= np.prod(np.abs(ref.res))
        if proc_crs == ProcCrs.auto:
            proc_crs = ProcCrs.ref if src_pixel_smaller else ProcCrs.src
        elif (proc_crs == ProcCrs.src and src_pixel_smaller) or (proc_crs == ProcCrs.ref and not src_pixel_smaller):
            rec = ProcCrs.ref if src_pixel_smaller else ProcCrs.src
            cmp_str = 'smaller' if src_pixel_smaller else 'larger'
            warnings.warn(
                f'proc_crs={rec} is recommended when the source pixel size is {cmp_str} than the reference.',
                category=ConfigWarning
            )
        return proc_crs

    # ---- context management (reference raster_pair.py:271-311) ----------------------------------------------------
    @property
    def proc_crs(self) -> ProcCrs:
        return self._proc_crs

    @property
    def src_bands(self) -> Tuple[int, ...]:
        """ 1-based source bands taking part (band numbers in the file, for a pair opened from files). """
        return tuple(self._files.src_bands) if self._files is not None else tuple(self._src_bands)

    @property
    def ref_bands(self) -> Tuple[int, ...]:
        """ The reference band matched to each source band. """
        return tuple(self._files.ref_bands) if self._files is not None else tuple(self._ref_bands)

    @property
    def closed(self) -> bool:
        return self._closed

    def open(self):
        self._closed = False

    def close(self):
        self._closed = True

    def __enter__(self):
        self.open()
        return self

    def __exit__(self, exc_type, exc_val, exc_tb):
        self.close()

    def _assert_open(self):
        if self.closed:
            raise IoError('The raster pair has not been opened: use `with RasterFuse(...) as fuse:` or `open()`')

    # ---- configuration factories (reference fuse.py:89-149) -------------------------------------------------------
    create_model_config = KernelModel.create_config

    @staticmethod
    def create_block_config(threads: int = 0, max_block_mem: float = 100) -> Dict:
        return dict(threads=_validate_threads(threads), max_block_mem=max_block_mem)

    @staticmethod
    def create_out_profile(driver: str = 'GTiff', dtype: str = RasterArray.default_dtype,
                           nodata: float = RasterArray.default_nodata, creation_options: Optional[Dict] = None) -> Dict:
        creation_options = creation_options or dict(
            tiled=True, blockxsize=512, blockysize=512, compress='deflate', interleave='band', photometric=None
        )
        return dict(driver=driver, dtype=dtype, nodata=nodata, **creation_options)

    # ---- the hot path ----------------------------------------------------------------------------------------------
    def _ref_block(self, band_i: int) -> RasterArray:
        """ Reference band cropped to the window covering the source (raster_pair.py:292-296). """
        ref_ra = _band(self._ref, self._ref_bands[band_i])
        row0, col0, height, width = ref_window_for_src(self._src, ref_ra)
        if (row0, col0, height, width) == (0, 0, ref_ra.height, ref_ra.width):
            return ref_ra
        array = ref_ra.array[row0:row0 + height, col0:col0 + width]
        transform = ref_ra.transform * Affine.translation(col0, row0)
        return RasterArray(array, ref_ra.crs, transform, nodata=ref_ra.nodata)

    def _band_plan(self, band_i: int):
        """
        Per-band inputs of the one-call path, prepared once and re-used by later ``process`` calls on unchanged rasters
        (the reference's reader likewise fixes its windows when the pair is opened, raster_pair.py:280-296): the source
        band view, the reference block as a contiguous float32 device plane, and the grid map between them.  The cache
        key holds the tensors' identities and version counters, so in-place edits of either raster invalidate it.
        """
        src_arr, ref_arr = self._src.array, self._ref.array
        key = (src_arr.data_ptr(), src_arr._version, tuple(src_arr.shape), ref_arr.data_ptr(), ref_arr._version,
               tuple(ref_arr.shape), self._src_bands[band_i], self._ref_bands[band_i])
        with self._plan_lock:
            plan = self._plans.get(band_i)
        if plan is not None and plan[0] == key:
            return plan[1:]
        from homonim_b200.geometry import grid_map
        src_ra = _band(self._src, self._src_bands[band_i])
        ref_ra = self._ref_block(band_i)
        ref_t = ref_ra.array
        if ref_t.dtype != torch.float32:
            ref_t = ref_t.to(torch.float32)
        ref_t = ref_t.contiguous()
        gm = grid_map(src_ra.transform, ref_ra.transform)         # reference grid -> source grid
        plan = (key, src_ra, ref_ra, ref_t, gm)
        with self._plan_lock:
            self._plans[band_i] = plan
        return plan[1:]

    def _process_band(self, band_i: int, model: KernelModel, out=None, stage: bool = False,
                      want_params: bool = True, out_nodata=float('nan')) -> Tuple[RasterArray, Optional[RasterArray]]:
        """
        One band of reference fuse.py:295-319 (``_process_block`` with a single block): read -> fit -> apply.
        ``stage``: copy a host band to the device once up front (fit and apply both read it) and leave the results
        on the device; otherwise results live where the inputs live.  ``out`` / ``out_nodata``: device plane of the
        OUTPUT dtype that the apply kernel writes directly (the reference converts when it writes the block,
        raster_array.py:493-500; here the conversion is part of the kernel's store).
        """
        if self._src.is_device and self._ref.is_device and isinstance(model, RefSpaceModel):
            # device-resident rasters, proc_crs = ref: one native call per band on cached, prepared planes
            src_ra, ref_ra, ref_t, gm = self._band_plan(band_i)
            if model.can_fuse(src_ra, ref_ra):
                corr, params = model._fuse_planes(src_ra.array, src_ra.nodata, ref_t, ref_ra.nodata, gm, out,
                                                  want_params, out_nodata)
                corr_ra = RasterArray(corr, src_ra.crs, src_ra.transform, nodata=out_nodata)
                param_ra = None
                if params is not None:
                    param_ra = RasterArray(params, ref_ra.crs, ref_ra.transform, nodata=float('nan'))
                return corr_ra, param_ra
        src_ra = _band(self._src, self._src_bands[band_i])
        ref_ra = self._ref_block(band_i)
        if stage and not src_ra.is_device:
            src_ra, ref_ra = src_ra.to_device(), ref_ra.to_device()
        if isinstance(model, SrcSpaceModel) and not want_params and model.can_fuse(src_ra, ref_ra):
            # fit + apply in one kernel: the parameters are not wanted, so they are never written
            return model.fuse(src_ra, ref_ra, out=out, out_nodata=out_nodata), None
        if isinstance(model, RefSpaceModel) and model.can_fuse(src_ra, ref_ra):
            # fit + apply as one native call (same kernels, same order; the parameters are only materialised for the
            # caller when a parameter raster was asked for)
            return model.fuse(src_ra, ref_ra, out=out, want_params=want_params, out_nodata=out_nodata)
        param_ra = model.fit(src_ra, ref_ra)          # fuse.py:306
        corr_ra = model.apply(src_ra, param_ra, out=out, out_nodata=out_nodata)       # fuse.py:307
        return corr_ra, param_ra

    def process(self, corr_filename=None, model: Model = KernelModel.default_model,
                kernel_shape: Tuple[int, int] = KernelModel.default_kernel_shape, param_filename=None,
                build_ovw: bool = True, overwrite: bool = False, model_config: Optional[Dict] = None,
                out_profile: Optional[Dict] = None, block_config: Optional[Dict] = None, corr_out=None
                ) -> Tuple[RasterArray, Optional[RasterArray]]:
        """
        Correct the source to surface reflectance (reference fuse.py:321-408).  Same arguments as the reference;
        ``corr_filename`` / ``param_filename`` only act as switches here (``param_filename is not None`` turns on the
        R2 band and returns the parameter raster, as ``find_r2=param_filename is not None`` does at fuse.py:377).

        ``corr_out`` (optional, additive): a pre-allocated ``[bands, H, W]`` tensor of the output dtype to receive the
        corrected image -- a CUDA tensor, or a (pinned) CPU tensor for host pipelines, where each band's device -> host
        copy then overlaps the other bands' work.

        Returns ``(corr_ra, param_ra or None)``: ``corr_ra`` has one band per source band on the source grid and lives
        where the source lives (CUDA tensor / numpy array) or in ``corr_out``; ``param_ra`` interleaves parameters
        band-major as the reference's parameter file does (index = param_i * n_bands + band_i, fuse.py:315).
        """
        self._assert_open()
        if self._files is not None and not overwrite:  # fuse.py:275-282: refuse before any work is done
            for name, what in ((corr_filename, 'Corrected'), (param_filename, 'Parameter')):
                if is_path(name) and pathlib.Path(name).exists():
                    raise FileExistsError(
                        f"{what} image file exists and won't be overwritten without the `overwrite` option: {name}")
        model_type = Model(model)
        _ = overlap_for_kernel(kernel_shape)           # fuse.py:371 (single block per band: no overlap is needed)
        if self._src.is_device and self._src.array.device.index != torch.cuda.current_device():
            with torch.cuda.device(self._src.array.device):        # the native calls launch on the current device
                return self.process(corr_filename, model, kernel_shape, param_filename, build_ovw, overwrite,
                                    model_config, out_profile, block_config, corr_out)
        model_config = RasterFuse.create_model_config(**(model_config or {}))
        block_config = RasterFuse.create_block_config(**(block_config or {}))
        out_profile = RasterFuse.create_out_profile(**(out_profile or {}))

        model_cls = SrcSpaceModel if self.proc_crs == ProcCrs.src else RefSpaceModel          # fuse.py:376
        kernel_model = model_cls(model_type, kernel_shape, find_r2=param_filename is not None, **model_config)

        if torch is None or not torch.cuda.is_available():
            from homonim_b200 import _native
            _native.require_device()                   # raises: there is no CPU implementation

        n_bands = len(self._src_bands)
        hs, ws = self._src.shape
        out_dtype = out_profile['dtype'] or 'float32'
        out_nodata = out_profile['nodata']
        plain_f32 = out_dtype == 'float32' and (out_nodata is None or (isinstance(out_nodata, float)
                                                                       and np.isnan(out_nodata)))
        src_on_device = self._src.is_device
        device = self._src.array.device if src_on_device else torch.device('cuda', torch.cuda.current_device())
        # where the corrected bands go: straight into a [bands, H, W] device tensor (no stacking copy), or band by
        # band to the host
        to_host = (corr_out is not None and not corr_out.is_cuda) or (corr_out is None and not src_on_device)
        if corr_out is not None:
            if tuple(corr_out.shape) != (n_bands, hs, ws) or str(corr_out.dtype).replace('torch.', '') != out_dtype:
                raise ValueError(f"'corr_out' must be a [{n_bands}, {hs}, {ws}] {out_dtype} tensor")
            corr_all = corr_out
        elif to_host:
            corr_all = torch.empty((n_bands, hs, ws), dtype=getattr(torch, out_dtype))
        else:
            corr_all = torch.empty((n_bands, hs, ws), dtype=getattr(torch, out_dtype), device=device)
        param_planes = [None] * n_bands

        # output dtypes the apply kernels store themselves (conversion fused into their epilogue); anything else goes through
        # a float32 plane and a separate conversion
        fused_out = out_dtype in ('float32', 'uint8', 'uint16', 'int16')

        # Internal overviews of the written files (reference fuse.py:151-165): every band's levels are built on the GPU from
        # its device plane as written (output dtype and nodata), on the band's stream, and copied to host buffers with the
        # band -- so that the writer encodes them band by band like the image's own tiles.
        write_files = self._files is not None and is_path(corr_filename)
        corr_levels = 0
        if write_files and build_ovw:
            if out_dtype in OVERVIEW_DTYPES:
                corr_levels = len(overview_factors((hs, ws)))
            else:
                warnings.warn(f'`build_ovw`: overviews are built for {", ".join(OVERVIEW_DTYPES)} outputs; the {out_dtype} '
                              f'output is written without them (use gdaladdo on it).', category=ConfigWarning)
        param_ovw = write_files and build_ovw and is_path(param_filename)
        corr_ovw = [torch.empty(level_shape((n_bands, hs, ws), 2 ** k), dtype=getattr(torch, out_dtype))
                    for k in range(1, corr_levels + 1)]
        param_ovw_planes = [None] * n_bands

        # File -> file (SURVEY.md 8f-4): the corrected image is encoded and written band by band WHILE the GPU works on the
        # later bands -- the writer waits on a band stream that a small completion thread feeds as every band's device ->
        # host copy lands.  (The reference's writer likewise runs inside its thread pool, fuse.py:254-293, 396-408.)
        meta = dict(model=model_type, kernel_shape=tuple(kernel_shape), **model_config,
                    **dict(block_config, max_block_mem='whole-band'))     # one block per band: recorded as applied
        streaming = self._files is not None and is_path(corr_filename) and to_host and corr_out is None
        band_stream = done_queue = writer = completer = None
        writer_error: list = []
        if streaming:
            import queue
            import types
            from homonim_b200.geotiff import BandStream
            band_stream = BandStream(corr_all.numpy(), overviews=[o.numpy() for o in corr_ovw])
            done_queue = queue.Queue()

            def _complete():
                while True:
                    item = done_queue.get()
                    if item is None:
                        return
                    band_i, event = item
                    try:
                        event.synchronize()
                        band_stream.set_ready(band_i)
                    except BaseException as ex:      # noqa
                        band_stream.fail(ex)
                        return

            def _write():
                try:
                    target = types.SimpleNamespace(array=band_stream, transform=self._src.transform, crs=self._src.crs)
                    self._files.write_corrected(target, corr_filename, self.proc_crs, out_profile, overwrite=overwrite,
                                                **meta)
                except BaseException as ex:          # noqa
                    writer_error.append(ex)
            completer = threading.Thread(target=_complete, daemon=True)
            writer = threading.Thread(target=_write, daemon=True)
            completer.start()
            writer.start()

        def run_band(band_i):
            want = param_filename is not None
            if fused_out:
                plane = corr_all[band_i] if not to_host else torch.empty((hs, ws), dtype=getattr(torch, out_dtype),
                                                                         device=device)
                corr_ra, param_ra = self._process_band(band_i, kernel_model, out=plane, stage=True, want_params=want,
                                                       out_nodata=out_nodata)
                if to_host:
                    corr_all[band_i].copy_(plane, non_blocking=True)
                if corr_levels:
                    for host, level in zip(corr_ovw, build_overviews(plane, out_nodata, corr_levels)):
                        host[band_i].copy_(level, non_blocking=True)
            else:
                corr_ra, param_ra = self._process_band(band_i, kernel_model, out=None, stage=True, want_params=want)
                plane = _convert_dtype(corr_ra, out_dtype, out_nodata)
                corr_all[band_i].copy_(plane, non_blocking=True)
            if param_ra is not None and param_ovw:
                levels = build_overviews(param_ra.array.contiguous(), float('nan'),
                                         len(overview_factors(param_ra.array.shape)))
                param_ovw_planes[band_i] = [torch.empty(lv.shape, dtype=lv.dtype).copy_(lv, non_blocking=True)
                                            for lv in levels]
            if param_ra is not None:
                param_planes[band_i] = param_ra if (src_on_device or param_filename is None) else param_ra.to_host()
            if streaming:
                landed = torch.cuda.Event()
                landed.record(current_stream())
                done_queue.put((band_i, landed))

        # Bands are independent (the reference runs (band, block) jobs on a thread pool, fuse.py:396-408).  On the
        # GPU each band is enqueued on its own CUDA stream, so that the small latency-bound kernels of one band (fit
        # on the proc grid, in-painting) overlap the bandwidth-bound resampling kernels of the others -- and, for host
        # rasters, one band's host <-> device copies overlap the other bands' kernels.
        n_streams = min(n_bands, max(1, int(block_config['threads'])), 4)
        try:
            self._run_bands(run_band, n_bands, n_streams, corr_all, param_planes)
        except BaseException as ex:
            if streaming:
                band_stream.fail(ex)
                done_queue.put(None)
                writer.join(timeout=60)
            raise
        if to_host or corr_ovw or param_ovw:
            current_stream().synchronize()  # the host copies have landed
        if streaming:
            done_queue.put(None)
            completer.join()
            writer.join()
            if writer_error:
                raise writer_error[0]

        corr_array = corr_all if (src_on_device or corr_out is not None or is_tensor(self._src.array)) \
            else corr_all.numpy()
        corr = RasterArray(corr_array, self._src.crs, self._src.transform, nodata=out_nodata)
        params = None
        if param_filename is not None:
            n_params = param_planes[0].count
            planes = [param_planes[b].array[p] for p in range(n_params) for b in range(n_bands)]
            stack = torch.stack if is_tensor(planes[0]) else np.stack
            params = RasterArray(stack(planes), param_planes[0].crs, param_planes[0].transform, nodata=float('nan'))
        param_levels = None
        if param_ovw and param_ovw_planes[0]:                 # (None without parameters, [] under 512 px)
            n_params = param_ovw_planes[0][0].shape[0]       # interleaved band-major, as the parameter image itself
            param_levels = [torch.stack([param_ovw_planes[b][k][p] for p in range(n_params) for b in range(n_bands)])
                            for k in range(len(param_ovw_planes[0]))]
        if self._files is not None and is_path(corr_filename):
            # a pair opened from files: write the outputs with the reference's metadata (fuse.py:264-293)
            if not streaming:
                self._files.write_corrected(corr.to_host(), corr_filename, self.proc_crs, out_profile,
                                            overwrite=overwrite, overviews=corr_ovw, **meta)
            if params is not None and is_path(param_filename):
                self._files.write_params(params.to_host(), param_filename, self.proc_crs, out_profile,
                                         overwrite=overwrite, overviews=param_levels, **meta)
        return corr, params

    @staticmethod
    def _run_bands(run_band, n_bands, n_streams, corr_all, param_planes):
        """ Enqueue every band, each on its own CUDA stream of the per-device pool (see `process`). """
        if n_streams > 1:
            main = current_stream()
            streams = _band_streams(n_streams)
            for st in streams:
                st.wait_stream(main)
            for band_i in range(n_bands):              # bands outermost, raster_pair.py:379-381
                with on_stream(streams[band_i % n_streams]):
                    run_band(band_i)
            for st in streams:
                main.wait_stream(st)
            for t in [corr_all] + [p.array for p in param_planes if p is not None]:
                if is_tensor(t) and t.is_cuda:
                    t.record_stream(main)
        else:
            for band_i in range(n_bands):
                run_band(band_i)


def _convert_dtype(ra: RasterArray, dtype: str, nodata):
    """
    Output dtype conversion of ``RasterArray._convert_array_dtype`` (raster_array.py:353-387): round half-to-even and
    clip when going to an integer type, then substitute the output nodata.  float32 / NaN output is a no-op.
    """
    array = ra.array
    is_nan_nd = nodata is not None and isinstance(nodata, float) and np.isnan(nodata)
    if dtype in ('float32', None) and (nodata is None or is_nan_nd):
        return array
    _OUT_CODES = {'uint8': 0, 'uint16': 1, 'float32': 2, 'int16': 3}
    if is_tensor(array) and array.is_cuda and array.dtype == torch.float32 and dtype in _OUT_CODES:
        # one native pass: round half-to-even, clip, cast, nodata substitution
        from homonim_b200 import kernel_model as km
        src = array.contiguous()
        out = torch.empty(src.shape, dtype=getattr(torch, dtype), device=src.device)
        has, nd = (0, 0.0) if nodata is None else (1, float(nodata))
        km._call('hb_convert_dtype', src.data_ptr(), src.numel(), _OUT_CODES[dtype], has, nd, out.data_ptr(),
                 km._stream())
        return out
    if is_tensor(array):
        mask = ~torch.isnan(array)
        out = array
        tdtype = getattr(torch, dtype)
        if not tdtype.is_floating_point:
            info = torch.iinfo(tdtype)
            out = torch.clamp(torch.round(out), info.min, info.max)
        out = torch.nan_to_num(out, nan=0.0).to(tdtype)
        if nodata is not None:
            out[~mask] = nodata
        return out
    mask = ~np.isnan(array)
    out = array
    if np.issubdtype(np.dtype(dtype), np.integer):
        info = np.iinfo(dtype)
        out = np.clip(np.round(out), info.min, info.max)
    with np.errstate(invalid='ignore'):
        out = np.nan_to_num(out, nan=0.0).astype(dtype)
    if nodata is not None:
        out[~mask] = nodata
    return out
