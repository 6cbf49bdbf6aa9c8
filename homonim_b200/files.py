"""
File front-end of ``RasterFuse`` / ``RasterCompare`` (SURVEY.md 8f-4): open a source / reference GeoTIFF pair, match
their bands, stage the matched bands as ``RasterArray`` objects for the GPU path, and write the corrected and
parameter images with the metadata the reference writes -- the parts of ``RasterPairReader`` / ``MatchedPairReader``
(raster_pair.py:104-311, matched_pair.py:38-94) and of ``RasterFuse``'s output handling (fuse.py:167-293) that sit on
either side of the kernel-model path.  Pixels go through :mod:`homonim_b200.geotiff`; nothing here computes on them.
"""
import logging
import pathlib
import warnings
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from homonim_b200.errors import ImageContentError
from homonim_b200.geometry import CRS
from homonim_b200.geotiff import GeoTiffReader, write_geotiff
from homonim_b200.matched_pair import match_bands
from homonim_b200.raster_array import RasterArray

try:
    import torch
except ImportError:  # pragma: no cover
    torch = None

logger = logging.getLogger(__name__)

_NATIVE_DTYPES = ('uint8', 'uint16', 'int16', 'float32')      # storage dtypes the kernels read directly


def is_path(obj) -> bool:
    return isinstance(obj, (str, pathlib.Path))


class FilePair:
    """
    A source / reference file pair opened for the kernel-model path.

    ``src_ra`` / ``ref_ra`` hold only the matched bands, in matched order (band ``i`` of one corrects / is corrected by
    band ``i`` of the other); ``src_bands`` / ``ref_bands`` are the 1-based band numbers they have in the files.
    """

    def __init__(self, src_filename, ref_filename, src_bands: Optional[Sequence[int]] = None,
                 ref_bands: Optional[Sequence[int]] = None, force: bool = False, pinned: bool = True):
        self.src_filename, self.ref_filename = pathlib.Path(src_filename), pathlib.Path(ref_filename)
        with GeoTiffReader(self.src_filename) as src_im, GeoTiffReader(self.ref_filename) as ref_im:
            for im in (src_im, ref_im):
                t = im.transform
                if not (t.a > 0 and t.e < 0 and t.b == 0 and t.d == 0):
                    raise NotImplementedError(f'{im.name}: only north-up rasters are supported (re-orientation needs '
                                              f'a warper, which is outside the B200 kernel-model path)')
            if src_im.crs != ref_im.crs:
                raise NotImplementedError(
                    f'{self.src_filename.name} and {self.ref_filename.name} are in different CRSs: re-projection '
                    f'between CRSs is outside the B200 kernel-model path (warp one of them first)')
            self.src_bands, self.ref_bands = match_bands(src_im, ref_im, src_bands, ref_bands, force)     # 1-based
            if not self.src_bands:
                raise ImageContentError('No source / reference bands could be matched.')
            for im in (src_im, ref_im):
                if im.nodata is None and 'alpha' in im.colorinterp:
                    # the reference masks with the alpha band then (dataset_mask, raster_array.py:170-197); reading the
                    # file as fully valid would let the masked pixels into the fit
                    raise NotImplementedError(f'{pathlib.Path(im.name).name}: alpha-band masks are not supported (give '
                                              f'the image a nodata value instead)')
            # the reference window that covers the source (whole reference pixels, 2 pixels to spare), clipped
            left, bottom, right, top = src_im.bounds
            rt = ref_im.transform
            c0 = int(np.floor((left - rt.c) / rt.a)) - 2
            c1 = int(np.ceil((right - rt.c) / rt.a)) + 2
            r0 = int(np.floor((top - rt.f) / rt.e)) - 2
            r1 = int(np.ceil((bottom - rt.f) / rt.e)) + 2
            c0, r0, c1, r1 = max(c0, 0), max(r0, 0), min(c1, ref_im.width), min(r1, ref_im.height)
            if c1 <= c0 or r1 <= r0:
                raise ImageContentError(f'{self.ref_filename.name} does not overlap {self.src_filename.name}.')
            self.src_ra = self._read(src_im, self.src_bands, None, pinned)
            self.ref_ra = self._read(ref_im, self.ref_bands, (c0, r0, c1 - c0, r1 - r0), pinned)
            self.src_profile, self.ref_profile = src_im.profile, ref_im.profile
            self.src_geokeys, self.ref_geokeys = src_im.geokeys, ref_im.geokeys
            self.src_descriptions = [src_im.descriptions[b - 1] for b in self.src_bands]
            self.ref_descriptions = [ref_im.descriptions[b - 1] for b in self.ref_bands]
            self.src_band_tags = [src_im.tags(b) for b in self.src_bands]
            self.ref_band_tags = [ref_im.tags(b) for b in self.ref_bands]

    @staticmethod
    def _read(im: GeoTiffReader, bands: Sequence[int], window, pinned: bool) -> RasterArray:
        """ The chosen bands as a [bands, H, W] RasterArray: uint8 / uint16 / int16 / float32 stay as stored (the kernels
        read them directly), other sample types are widened to float32 as the reference's reader does for every type
        (raster_array.py:178-188).  A file without a nodata value gets the default NaN nodata, as in the reference. """
        array = im.read(list(bands), window=window, pinned=pinned and im.dtype.name in _NATIVE_DTYPES)
        nodata = im.nodata
        if im.dtype.name not in _NATIVE_DTYPES:
            array = np.asarray(array).astype('float32')
            if torch is not None and pinned:
                array = torch.from_numpy(array)
                array = array.pin_memory() if torch.cuda.is_available() else array
        if nodata is None:
            nodata = RasterArray.default_nodata          # raster_array.py:166 (NaN: no integer pixel equals it)
        transform = im.transform
        if window is not None:
            from homonim_b200.geometry import Affine
            transform = transform * Affine.translation(window[0], window[1])
        return RasterArray(array, im.crs if im.crs is not None else CRS('unknown'), transform, nodata=nodata)

    # ---- outputs (reference fuse.py:167-293) ------------------------------------------------------------------------
    def _meta(self, proc_crs, **kwargs) -> Dict[str, str]:
        """ FUSE_* dataset metadata items (fuse.py:203-215). """
        meta = dict(FUSE_SRC_FILE=self.src_filename.name, FUSE_REF_FILE=self.ref_filename.name,
                    FUSE_PROC_CRS=getattr(proc_crs, 'name', str(proc_crs)))
        for key, value in kwargs.items():
            meta[f'FUSE_{key.upper()}'] = value.name if hasattr(value, 'name') else value
        return meta

    @staticmethod
    def _creation(out_profile: Dict) -> Dict:
        driver = out_profile.get('driver', 'GTiff')
        if driver != 'GTiff':
            raise NotImplementedError(f'output driver {driver!r} is not supported (GTiff is)')
        if not out_profile.get('tiled', True):
            logger.debug('untiled output was requested: a tiled GeoTIFF is written')
        compress = out_profile.get('compress', 'deflate')
        compress = None if compress in (None, 'none', 'NONE') else str(compress).lower()
        return dict(compress=compress, blocksize=int(out_profile.get('blockxsize', 512) or 512),
                    level=int(out_profile.get('zlevel', 6)),          # GDAL's ZLEVEL creation option (default 6)
                    interleave=str(out_profile.get('interleave', 'band')).lower(),
                    photometric=(str(out_profile['photometric']).lower() if out_profile.get('photometric') else
                                 'minisblack'))

    def write_corrected(self, corr_ra: RasterArray, corr_filename, proc_crs, out_profile: Dict, overwrite: bool = False,
                        overviews=None, **kwargs) -> pathlib.Path:
        """ The corrected image, in the source's grid and CRS, with the reference bands' wavelength metadata and
        descriptions copied to the bands they corrected (fuse.py:217-238), and its internal ``overviews`` (levels of
        factor 2, 4, ...; a band stream carries its own). """
        keep = ('center_wavelength', 'name', 'description', 'offset', 'scale')
        band_tags = [{k: v for k, v in tags.items() if k in keep} for tags in self.ref_band_tags]
        nodata = out_profile.get('nodata')
        if nodata is None:
            logger.debug('nodata=None: no internal mask is written; invalid pixels hold 0')
        return write_geotiff(corr_filename, corr_ra.array, corr_ra.transform, crs=corr_ra.crs, nodata=nodata,
                             descriptions=self.ref_descriptions, tags=self._meta(proc_crs, **kwargs),
                             band_tags=band_tags, geokeys=self.src_geokeys, overwrite=overwrite, overviews=overviews,
                             **self._creation(out_profile))

    def write_params(self, param_ra: RasterArray, param_filename, proc_crs, out_profile: Dict, overwrite: bool = False,
                     overviews=None, **kwargs) -> pathlib.Path:
        """ The parameter image (float32, NaN nodata; gains, then offsets, then R2, one of each per band,
        fuse.py:186-201, 240-262), with its internal ``overviews`` (interleaved as the image). """
        n_bands = len(self.src_bands)
        descriptions: List[Optional[str]] = [None] * param_ra.count
        band_tags: List[Dict] = [dict() for _ in range(param_ra.count)]
        for bi in range(n_bands):
            ref_descr = self.ref_descriptions[bi] or f'B{self.ref_bands[bi]}'
            for param_i, param_name in zip(range(bi, param_ra.count, n_bands), ('GAIN', 'OFFSET', 'R2')):
                descriptions[param_i] = f'{ref_descr}_{param_name}'
                band_tags[param_i] = {k: f'{v.upper()} {param_name}' for k, v in self.ref_band_tags[bi].items()
                                      if k in ('ABBREV', 'ID', 'NAME')}
        geokeys = self.ref_geokeys if getattr(proc_crs, 'name', str(proc_crs)) == 'ref' else self.src_geokeys
        creation = self._creation(out_profile)
        creation['photometric'] = 'minisblack'
        return write_geotiff(param_filename, param_ra.array, param_ra.transform, crs=param_ra.crs,
                             nodata=float('nan'), descriptions=descriptions, tags=self._meta(proc_crs, **kwargs),
                             band_tags=band_tags, geokeys=geokeys, overwrite=overwrite, overviews=overviews, **creation)


def create_out_postfix(proc_crs, model, kernel_shape: Tuple[int, int], driver: str = 'GTiff') -> str:
    """ File-name postfix of a corrected image, e.g. ``_FUSE_cREF_mGAIN-BLK-OFFSET_k5_5.tif`` (utils.py:167-173). """
    if driver != 'GTiff':
        raise NotImplementedError(f'output driver {driver!r} is not supported (GTiff is)')
    model_name = getattr(model, 'value', str(model))
    crs_name = getattr(proc_crs, 'name', str(proc_crs))
    return f'_FUSE_c{crs_name.upper()}_m{model_name.upper()}_k{kernel_shape[0]}_{kernel_shape[1]}.tif'


def create_param_filename(filename) -> pathlib.Path:
    """ ``<corrected stem>_PARAM<ext>`` next to the corrected image (utils.py:176-179). """
    filename = pathlib.Path(filename)
    return filename.parent.joinpath(f'{filename.stem}_PARAM{filename.suffix}')
