"""
GeoTIFF block reader / writer for the B200 kernel-model path (SURVEY.md 8f-4) -- the stand-in for the rasterio
dataset I/O the reference wraps in ``RasterArray.from_rio_dataset`` / ``to_rio_dataset`` (raster_array.py:129-199,
424-524) and ``RasterPairReader.read`` (raster_pair.py:313-340).  rasterio / GDAL are not available where this package
is built, so the container format is handled here directly: classic TIFF and BigTIFF; strips or tiles; chunky or
band-separate layout; uncompressed or deflate, horizontal predictor; 8 / 16 / 32-bit integer and 32 / 64-bit float
samples; north-up ModelPixelScale + ModelTiepoint (or ModelTransformation) geo-referencing; GDAL's nodata and metadata
tags.  Blocks are (de)compressed on a thread pool (zlib releases the GIL), and a read can land directly in pinned host
memory so that the host -> device copy of one band overlaps the decoding of the next.

What is NOT handled raises ``NotImplementedError`` instead of returning wrong pixels: LZW / JPEG / other codecs, the
floating-point predictor, internal mask IFDs, rotated geo-transforms.
"""
import concurrent.futures
import math
import os
import pathlib
import struct
import threading
import zlib
from typing import Dict, List, Optional, Sequence, Tuple
from xml.etree import ElementTree
from xml.sax.saxutils import escape, quoteattr

import numpy as np

from homonim_b200.geometry import Affine, CRS

try:
    import torch
except ImportError:  # pragma: no cover
    torch = None

# TIFF field types: code -> (struct char, size)
_FIELD = {1: ('B', 1), 2: ('c', 1), 3: ('H', 2), 4: ('I', 4), 5: ('II', 8), 6: ('b', 1), 7: ('B', 1), 8: ('h', 2),
          9: ('i', 4), 10: ('ii', 8), 11: ('f', 4), 12: ('d', 8), 16: ('Q', 8), 17: ('q', 8), 18: ('Q', 8)}
_SAMPLE_DTYPES = {(1, 8): 'u1', (1, 16): 'u2', (1, 32): 'u4', (2, 8): 'i1', (2, 16): 'i2', (2, 32): 'i4',
                  (3, 32): 'f4', (3, 64): 'f8'}
_DEFLATE = (8, 32946)
# GeoKeys that only carry citations / names: ignored when two CRSs are compared
_CITATION_KEYS = (1026, 2049, 3073)
_RASTER_TYPE_KEY = 1025          # GTRasterTypeGeoKey: 1 = RasterPixelIsArea, 2 = RasterPixelIsPoint (not part of the CRS)


def _raster_type(directory: Sequence[int]) -> int:
    """ GTRasterTypeGeoKey of a GeoKeyDirectory (1 = PixelIsArea when absent). """
    if directory and len(directory) >= 4:
        for i in range(directory[3]):
            key, loc, _, value = directory[4 + 4 * i:8 + 4 * i]
            if key == _RASTER_TYPE_KEY and loc == 0:
                return int(value)
    return 1


def _geokeys_pixel_is_area(geokeys):
    """ The GeoKeys with GTRasterTypeGeoKey rewritten to RasterPixelIsArea: `write_geotiff` always writes its tie point
    at the pixel CORNER, so keys passed through from a PixelIsPoint source must not keep saying "point". """
    directory = list(geokeys[0])
    if len(directory) >= 4:
        for i in range(directory[3]):
            if directory[4 + 4 * i] == _RASTER_TYPE_KEY and directory[5 + 4 * i] == 0:
                directory[7 + 4 * i] = 1
    return (tuple(directory),) + tuple(geokeys[1:])

_pool = None


def _codec_pool() -> concurrent.futures.ThreadPoolExecutor:
    global _pool
    if _pool is None:
        _pool = concurrent.futures.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 4),
                                                      thread_name_prefix='hb-tiff')
    return _pool


def _crs_from_geokeys(directory: Sequence[int], doubles: Sequence[float], ascii_params: str) -> Optional[CRS]:
    """ An opaque, comparable CRS label from the GeoKeyDirectory (citation keys left out of the comparison). """
    if not directory or len(directory) < 4:
        return None
    keys = []
    for i in range(directory[3]):
        key, loc, count, value = directory[4 + 4 * i:8 + 4 * i]
        if key in _CITATION_KEYS or key == _RASTER_TYPE_KEY:
            continue
        if loc == 0:
            keys.append((key, value))
        elif loc == 34736:
            keys.append((key, tuple(doubles[value:value + count])))
        elif loc == 34737:
            keys.append((key, ascii_params[value:value + count].rstrip('|')))
    return CRS(('geokeys', tuple(sorted(keys, key=lambda kv: kv[0]))))


class GeoTiffReader:
    """
    Read access to one GeoTIFF file.  Attribute names follow the rasterio dataset attributes the reference uses
    (``width``, ``height``, ``count``, ``dtypes``, ``nodata``, ``transform``, ``crs``, ``descriptions``, ``colorinterp``,
    ``tags()``, ``profile``), so that the pair / band-matching logic reads like the reference's.

    ``overview_level`` (rasterio's open option of that name): open internal overview ``overview_level`` instead of the
    full-resolution image, counted from 0 for the first (factor 2) overview.  Its pixels, size, blocks and transform are
    the overview's; CRS, nodata, metadata and descriptions are the image's.
    """

    def __init__(self, filename, overview_level: Optional[int] = None):
        self.name = str(filename)
        self._fh = open(filename, 'rb')
        self._closed = False
        try:
            self._parse_header(overview_level)
        except BaseException:
            self.close()
            raise

    # ---- header -----------------------------------------------------------------------------------------------------
    def _parse_header(self, overview_level: Optional[int] = None):
        fh = self._fh
        head = fh.read(16)
        if head[:2] not in (b'II', b'MM'):
            raise ValueError(f'{self.name}: not a TIFF file')
        bo = '<' if head[:2] == b'II' else '>'
        magic, = struct.unpack(bo + 'H', head[2:4])
        if magic == 42:
            self._big = False
            ifd_off, = struct.unpack(bo + 'I', head[4:8])
        elif magic == 43:
            self._big = True
            ifd_off, = struct.unpack(bo + 'Q', head[8:16])
        else:
            raise ValueError(f'{self.name}: not a TIFF file (magic {magic})')
        self._bo = bo
        tags = self._read_ifd(ifd_off)
        self._raw_tags = tags
        # GDAL per-dataset masks live in a LATER IFD (NewSubfileType bit 2) or in a `.msk` side-car; the reference honours
        # them through dataset_mask (raster_array.py:170-197).  They are not decoded here, and reading such a file as
        # "fully valid" would let invalid pixels into the fit, so refuse it.
        self.has_internal_mask = False
        self._overview_ifds: List[Dict[int, tuple]] = []          # reduced-resolution IFDs (NewSubfileType bit 0)
        next_off, seen = self._next_ifd, 0
        while next_off and seen < 64:
            sub = self._read_ifd(next_off)
            next_off, seen = self._next_ifd, seen + 1
            if 254 in sub and (int(sub[254][0]) & 4):
                self.has_internal_mask = True
            elif 254 in sub and (int(sub[254][0]) & 1):
                self._overview_ifds.append(sub)
        if os.path.exists(self.name + '.msk'):
            self.has_internal_mask = True
        if self.has_internal_mask:
            raise NotImplementedError(f'{self.name}: internal / side-car mask bands are not supported (give the image '
                                      f'a nodata value instead)')
        self._full_shape = (int(tags[257][0]), int(tags[256][0]))
        self.overview_level = overview_level
        if overview_level is not None:
            if not 0 <= int(overview_level) < len(self._overview_ifds):
                raise ValueError(f'{self.name}: overview level {overview_level} does not exist (the file has '
                                 f'{len(self._overview_ifds)})')
            tags = self._overview_ifds[int(overview_level)]     # the pixels' layout; the metadata stay IFD 0's
        self.width, self.height = int(tags[256][0]), int(tags[257][0])
        self.count = int(tags.get(277, (1,))[0])
        bits = tags.get(258, (1,))
        fmt = tags.get(339, (1,) * self.count)
        if len(set(bits)) != 1 or len(set(fmt)) != 1 or (fmt[0], bits[0]) not in _SAMPLE_DTYPES:
            raise NotImplementedError(f'{self.name}: unsupported sample layout (bits {bits}, format {fmt})')
        self.dtype = np.dtype(_SAMPLE_DTYPES[(fmt[0], bits[0])])
        self._file_dtype = self.dtype.newbyteorder(bo)
        self.compression = int(tags.get(259, (1,))[0])
        if self.compression != 1 and self.compression not in _DEFLATE:
            raise NotImplementedError(f'{self.name}: TIFF compression {self.compression} is not supported '
                                      f'(uncompressed and deflate are)')
        self.predictor = int(tags.get(317, (1,))[0])
        if self.predictor not in (1, 2) or (self.predictor == 2 and self.dtype.kind == 'f'):
            raise NotImplementedError(f'{self.name}: TIFF predictor {self.predictor} is not supported')
        self.planar = int(tags.get(284, (1,))[0])
        self.tiled = 322 in tags
        if self.tiled:
            self.block_shape = (int(tags[323][0]), int(tags[322][0]))                  # (rows, cols)
            self._offsets, self._counts = tags[324], tags[325]
        else:
            self.block_shape = (min(int(tags.get(278, (self.height,))[0]), self.height), self.width)
            self._offsets, self._counts = tags[273], tags[279]
        self._blocks_down = -(-self.height // self.block_shape[0])
        self._blocks_across = -(-self.width // self.block_shape[1])
        planes = self.count if self.planar == 2 else 1
        if len(self._offsets) != self._blocks_down * self._blocks_across * planes:
            raise ValueError(f'{self.name}: inconsistent block table')
        if 254 in tags and (tags[254][0] & 4):
            raise NotImplementedError(f'{self.name}: the first IFD is a mask')
        tags = self._raw_tags
        if overview_level is not None and int(tags.get(277, (1,))[0]) != self.count:
            raise ValueError(f'{self.name}: overview {overview_level} has a different band count')
        # geo-referencing
        if 33550 in tags and 33922 in tags:
            scale, tie = tags[33550], tags[33922]
            self.transform = Affine(float(scale[0]), 0.0, float(tie[3]) - float(tie[0]) * float(scale[0]), 0.0,
                                    -float(scale[1]), float(tie[4]) + float(tie[1]) * float(scale[1]))
        elif 34264 in tags:
            m = tags[34264]
            self.transform = Affine(float(m[0]), float(m[1]), float(m[3]), float(m[4]), float(m[5]), float(m[7]))
        else:
            self.transform = Affine.identity()
        self._geo = (tuple(tags.get(34735, ())), tuple(tags.get(34736, ())), tags.get(34737, ''))
        self.crs = _crs_from_geokeys(*self._geo)
        if self.crs is not None:
            self.crs.raw_geokeys = self._geo
            if _raster_type(self._geo[0]) == 2:                 # RasterPixelIsPoint: the tie point is a pixel centre
                self.transform = self.transform * Affine.translation(-0.5, -0.5)
        if overview_level is not None:                          # rasterio: the full transform scaled to the overview
            full_h, full_w = self._full_shape
            self.transform = self.transform * Affine.scale(full_w / self.width, full_h / self.height)
        nodata = tags.get(42113)
        self.nodata = None
        if nodata is not None:
            try:
                self.nodata = float(str(nodata).strip().strip('\x00'))
            except ValueError:
                self.nodata = None
        # GDAL metadata: dataset items, per-band items, band descriptions
        self._tags: Dict[str, str] = {}
        self._band_tags: List[Dict[str, str]] = [dict() for _ in range(self.count)]
        self.descriptions: List[Optional[str]] = [None] * self.count
        if 42112 in tags:
            try:
                root = ElementTree.fromstring(str(tags[42112]).strip('\x00').strip())
            except ElementTree.ParseError:
                root = None
            for item in (root.findall('Item') if root is not None else []):
                name, sample, role, text = item.get('name'), item.get('sample'), item.get('role'), item.text or ''
                if sample is None:
                    self._tags[name] = text
                elif 0 <= int(sample) < self.count:
                    if role == 'description':
                        self.descriptions[int(sample)] = text
                    elif role is None:
                        self._band_tags[int(sample)][name] = text
        # colour interpretation, as GDAL derives it from PhotometricInterpretation / ExtraSamples
        photometric = int(tags.get(262, (1,))[0])
        extra = tuple(tags.get(338, ()))
        base = self.count - len(extra)
        if photometric == 2 and base >= 3:
            interp = ['red', 'green', 'blue'] + ['undefined'] * (base - 3)
        else:
            interp = ['gray'] + ['undefined'] * max(base - 1, 0)
        interp += ['alpha' if e in (1, 2) else 'undefined' for e in extra]
        self.colorinterp = (interp + ['undefined'] * self.count)[:self.count]

    def _read_ifd(self, offset: int) -> Dict[int, tuple]:
        fh, bo = self._fh, self._bo
        fh.seek(offset)
        if self._big:
            n, = struct.unpack(bo + 'Q', fh.read(8))
            entries = fh.read(20 * n)
            esize, head_fmt, inline = 20, 'HHQ', 8
        else:
            n, = struct.unpack(bo + 'H', fh.read(2))
            entries = fh.read(12 * n)
            esize, head_fmt, inline = 12, 'HHI', 4
        hsize = struct.calcsize(bo + head_fmt)
        tags = {}
        for i in range(n):
            entry = entries[esize * i:esize * (i + 1)]
            tag, typ, cnt = struct.unpack(bo + head_fmt, entry[:hsize])
            if typ not in _FIELD:
                continue
            fmt, size = _FIELD[typ]
            total = size * cnt
            if total <= inline:
                data = entry[hsize:hsize + total]
            else:
                off, = struct.unpack(bo + ('Q' if self._big else 'I'), entry[hsize:hsize + inline])
                fh.seek(off)
                data = fh.read(total)
            if typ == 2:
                tags[tag] = data.decode('latin1').rstrip('\x00')
            elif typ in (5, 10):
                vals = struct.unpack(bo + fmt[0] * (2 * cnt), data)
                tags[tag] = tuple(vals[2 * k] / vals[2 * k + 1] if vals[2 * k + 1] else 0.0 for k in range(cnt))
            else:
                tags[tag] = struct.unpack(bo + fmt * cnt, data)
        fh.seek(offset + (8 if self._big else 2) + esize * n)
        nxt = fh.read(8 if self._big else 4)
        self._next_ifd = struct.unpack(bo + ('Q' if self._big else 'I'), nxt)[0] if len(nxt) in (4, 8) else 0
        return tags

    # ---- dataset-style attributes -------------------------------------------------------------------------------------
    @property
    def closed(self) -> bool:
        return self._closed

    def close(self):
        if not self._closed:
            self._fh.close()
            self._closed = True

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def shape(self) -> Tuple[int, int]:
        return self.height, self.width

    @property
    def dtypes(self) -> Tuple[str, ...]:
        return (self.dtype.name,) * self.count

    @property
    def res(self) -> Tuple[float, float]:
        return abs(self.transform.a), abs(self.transform.e)

    @property
    def bounds(self) -> Tuple[float, float, float, float]:
        t = self.transform
        xs, ys = (t.c, t.c + t.a * self.width), (t.f, t.f + t.e * self.height)
        return min(xs), min(ys), max(xs), max(ys)

    @property
    def profile(self) -> Dict:
        return dict(driver='GTiff', dtype=self.dtype.name, nodata=self.nodata, width=self.width, height=self.height,
                    count=self.count, crs=self.crs, transform=self.transform,
                    blockxsize=self.block_shape[1], blockysize=self.block_shape[0], tiled=self.tiled,
                    compress='deflate' if self.compression in _DEFLATE else None,
                    interleave='band' if self.planar == 2 else 'pixel')

    def overviews(self, bidx: int) -> List[int]:
        """ Decimation factors of the internal overviews of 1-based band ``bidx`` (rasterio ``DatasetReader.overviews``:
        ``round(width / overview width)``; every band has the same overviews here). """
        if not 1 <= bidx <= self.count:
            raise IndexError(f'{self.name}: band index out of range')
        return [int(round(self._full_shape[1] / int(sub[256][0]))) for sub in self._overview_ifds]

    def tags(self, bidx: Optional[int] = None) -> Dict[str, str]:
        """ Dataset metadata items, or those of 1-based band ``bidx`` (rasterio ``DatasetReader.tags``). """
        return dict(self._tags) if bidx is None else dict(self._band_tags[bidx - 1])

    @property
    def geokeys(self) -> Tuple[tuple, tuple, str]:
        """ The raw (GeoKeyDirectory, GeoDoubleParams, GeoAsciiParams) tags, to be written through unchanged. """
        return self._geo

    # ---- pixels -------------------------------------------------------------------------------------------------------
    def _decode_block(self, index: int, rows: int) -> np.ndarray:
        """ One strip / tile as an array [rows, block cols, samples per block pixel] in native byte order. """
        offset, nbytes = self._offsets[index], self._counts[index]
        raw = os.pread(self._fh.fileno(), nbytes, offset)
        if self.compression != 1:
            raw = zlib.decompress(raw)
        spp = self.count if self.planar == 1 else 1
        cols = self.block_shape[1]
        block = np.frombuffer(raw, dtype=self._file_dtype, count=rows * cols * spp).reshape(rows, cols, spp)
        if self.predictor == 2:
            block = np.cumsum(block, axis=1, dtype=self.dtype)
        return block.astype(self.dtype, copy=False)

    def read(self, indexes=None, window: Optional[Tuple[int, int, int, int]] = None, fill_value=None,
             out: Optional[np.ndarray] = None, pinned: bool = False):
        """
        Read bands ``indexes`` (1-based; an int gives a 2D array) over ``window`` = (col_off, row_off, width, height),
        which may reach beyond the raster ("boundless", raster_array.py:175-199): pixels outside are set to
        ``fill_value`` (default: the file's nodata, else 0).  ``pinned=True`` returns a torch tensor in pinned host
        memory (ready for an asynchronous host -> device copy) instead of a numpy array.
        """
        if self._closed:
            raise ValueError(f'{self.name}: the file is closed')
        squeeze = np.isscalar(indexes)
        bands = list(range(1, self.count + 1)) if indexes is None else ([int(indexes)] if squeeze else list(indexes))
        if any(b < 1 or b > self.count for b in bands):
            raise IndexError(f'{self.name}: band index out of range')
        col_off, row_off, width, height = (0, 0, self.width, self.height) if window is None else \
            tuple(int(v) for v in window)
        if fill_value is None:
            fill_value = self.nodata if self.nodata is not None else 0
        if self.dtype.kind != 'f' and isinstance(fill_value, float) and math.isnan(fill_value):
            fill_value = 0
        shape = (len(bands), height, width)
        if out is not None:
            array = out if out.ndim == 3 else out[None]
            if tuple(array.shape) != shape or array.dtype != self.dtype:
                raise ValueError('`out` does not match the window / bands / dtype')
            holder = None
        elif pinned and torch is not None:
            holder = torch.empty(shape, dtype=getattr(torch, self.dtype.name), pin_memory=torch.cuda.is_available())
            array = holder.numpy()
        else:
            holder = None
            array = np.empty(shape, dtype=self.dtype)
        # part of the window inside the raster
        r0, r1 = max(row_off, 0), min(row_off + height, self.height)
        c0, c1 = max(col_off, 0), min(col_off + width, self.width)
        if r0 > row_off or c0 > col_off or r1 < row_off + height or c1 < col_off + width or r1 <= r0 or c1 <= c0:
            array[...] = fill_value
        if r1 > r0 and c1 > c0:
            bh, bw = self.block_shape
            jobs = []
            for by in range(r0 // bh, (r1 - 1) // bh + 1):
                rows = bh if self.tiled else min(bh, self.height - by * bh)
                for bx in range(c0 // bw, (c1 - 1) // bw + 1):
                    if self.planar == 1:
                        jobs.append((by, bx, rows, None, (by * self._blocks_across) + bx))
                    else:
                        for k, b in enumerate(bands):
                            idx = ((b - 1) * self._blocks_down + by) * self._blocks_across + bx
                            jobs.append((by, bx, rows, k, idx))

            def run(job):
                by, bx, rows, k, idx = job
                block = self._decode_block(idx, rows)
                y0, x0 = by * bh, bx * bw
                ya, yb = max(y0, r0), min(y0 + rows, r1)
                xa, xb = max(x0, c0), min(x0 + bw, c1)
                part = block[ya - y0:yb - y0, xa - x0:xb - x0, :]
                dst = (slice(ya - row_off, yb - row_off), slice(xa - col_off, xb - col_off))
                if k is None:
                    for kk, b in enumerate(bands):
                        array[(kk,) + dst] = part[:, :, b - 1]
                else:
                    array[(k,) + dst] = part[:, :, 0]

            if len(jobs) > 1:
                list(_codec_pool().map(run, jobs))
            else:
                run(jobs[0])
        if out is not None:
            return out
        result = holder if holder is not None else array
        return result[0] if squeeze else result


# ---------------------------------------------------------------------------------------------------------------------
# writer
# ---------------------------------------------------------------------------------------------------------------------
def _gdal_metadata_xml(tags: Optional[Dict], band_tags: Optional[Sequence[Dict]],
                       descriptions: Optional[Sequence[Optional[str]]]) -> Optional[str]:
    items = []
    for key, value in (tags or {}).items():
        items.append(f'  <Item name={quoteattr(str(key))}>{escape(str(value))}</Item>')
    count = max(len(band_tags or ()), len(descriptions or ()))
    for b in range(count):
        if descriptions and b < len(descriptions) and descriptions[b]:
            items.append(f'  <Item name="DESCRIPTION" sample="{b}" role="description">'
                         f'{escape(str(descriptions[b]))}</Item>')
        if band_tags and b < len(band_tags):
            for key, value in (band_tags[b] or {}).items():
                items.append(f'  <Item name={quoteattr(str(key))} sample="{b}">{escape(str(value))}</Item>')
    if not items:
        return None
    return '<GDALMetadata>\n' + '\n'.join(items) + '\n</GDALMetadata>\n'


class BandStream:
    """
    A ``[bands, H, W]`` array whose bands become available one after the other -- what :func:`write_geotiff` takes to
    encode band ``b`` while the GPU is still producing band ``b + 1`` (SURVEY.md 8f-4).  ``array`` is the (host) buffer
    the producer fills; the producer calls ``set_ready(b)`` once band ``b`` is complete in it, or ``fail(exc)``.
    ``overviews``: optional ``[bands, h_k, w_k]`` host buffers of the image's overview levels (factors 2, 4, ...), whose
    band ``b`` the producer also fills before ``set_ready(b)``.
    """

    def __init__(self, array: np.ndarray, overviews: Optional[Sequence[np.ndarray]] = None):
        if array.ndim != 3:
            raise ValueError('BandStream needs a [bands, H, W] buffer')
        self.array = array
        self.overviews = list(overviews) if overviews else None
        self.shape, self.dtype, self.ndim = array.shape, array.dtype, 3
        self._ready = [threading.Event() for _ in range(array.shape[0])]
        self._error: Optional[BaseException] = None

    def set_ready(self, band: int) -> None:
        self._ready[band].set()

    def fail(self, exc: BaseException) -> None:
        self._error = exc
        for ev in self._ready:
            ev.set()

    def wait_band(self, band: int, timeout: float = 3600.0) -> np.ndarray:
        if not self._ready[band].wait(timeout):
            raise TimeoutError(f'band {band} was not produced within {timeout} s')
        if self._error is not None:
            raise RuntimeError('the producer of this band stream failed') from self._error
        return self.array[band]

    def wait_all(self) -> np.ndarray:
        for b in range(self.shape[0]):
            self.wait_band(b)
        return self.array


def _check_overviews(overviews, shape, dtype) -> list:
    """ The overview arrays as [bands, h_k, w_k] numpy arrays; level k (0-based) must have decimation factor 2^(k+1). """
    levels = []
    count, height, width = shape
    for k, level in enumerate(overviews or ()):
        if torch is not None and isinstance(level, torch.Tensor):
            level = level.detach().cpu().numpy()
        level = np.asarray(level)
        if level.ndim == 2:
            level = level[None]
        f = 2 ** (k + 1)
        expect = (count, -(-height // f), -(-width // f))
        if level.shape != expect:
            raise ValueError(f'overview {k} (factor {f}) must be {list(expect)}, not {list(level.shape)}')
        if np.dtype(level.dtype).newbyteorder('=') != dtype:
            raise ValueError(f'overview {k} has dtype {level.dtype}, the image {dtype}')
        levels.append(level)
    return levels


def write_geotiff(filename, array, transform, crs=None, nodata=None, descriptions=None, tags=None, band_tags=None,
                  geokeys=None, compress: Optional[str] = 'deflate', blocksize: int = 512, interleave: str = 'band',
                  photometric: Optional[str] = None, bigtiff: Optional[bool] = None, overwrite: bool = False,
                  level: int = 6, overviews: Optional[Sequence] = None):
    """
    Write ``array`` ([bands, H, W] or [H, W]; numpy or CPU torch tensor) as a tiled GeoTIFF -- what
    ``RasterArray.to_rio_dataset`` + the creation profile do in the reference (raster_array.py:424-524,
    fuse.py:167-215).  ``geokeys`` = (GeoKeyDirectory, GeoDoubleParams, GeoAsciiParams) as read by
    :class:`GeoTiffReader` is written through unchanged (the path never re-projects, so the output CRS is the source's).
    BigTIFF is chosen automatically when the pixels would not fit a classic TIFF.

    ``overviews``: internal overviews (what ``gdaladdo`` / the reference's ``_build_overviews`` add), a list of
    ``[bands, ceil(H / f), ceil(W / f)]`` arrays of the image's dtype for f = 2, 4, 8, ...  They are written as
    reduced-resolution IFDs (NewSubfileType = 1) chained after the image's, with its layout, compression and tile size.
    A :class:`BandStream` ``array`` carries its overviews itself.
    """
    path = pathlib.Path(filename)
    if path.exists() and not overwrite:
        raise FileExistsError(f"{path} exists and won't be overwritten without `overwrite`")
    stream = array if isinstance(array, BandStream) else None
    if stream is None:
        if torch is not None and isinstance(array, torch.Tensor):
            array = array.detach().cpu().numpy()
        array = np.asarray(array)
        if array.ndim == 2:
            array = array[None]
    elif overviews:
        raise ValueError('a BandStream carries its own overviews')
    else:
        overviews = stream.overviews
    if array.ndim != 3:
        raise ValueError('`array` must be [bands, H, W] or [H, W]')
    dtype = np.dtype(array.dtype).newbyteorder('=')
    sample = {v: k for k, v in _SAMPLE_DTYPES.items()}.get(dtype.str[1:])
    if sample is None:
        raise NotImplementedError(f'dtype {dtype} cannot be written')
    if compress not in (None, 'deflate', 'none'):
        raise NotImplementedError(f'compression {compress!r} is not supported (deflate or None)')
    deflate = compress == 'deflate'
    count, height, width = array.shape
    levels = _check_overviews(overviews, array.shape, dtype)
    blocksize = max(16, (int(blocksize) + 15) // 16 * 16)                 # TIFF: tile sides are multiples of 16
    th, tw = blocksize, blocksize
    # per IFD (the image, then each overview): (height, width, tiles down, tiles across)
    grids = [(h, w, -(-h // th), -(-w // tw)) for h, w in [(height, width)] + [lv.shape[1:] for lv in levels]]
    planar = 2 if (interleave == 'band' and count > 1) else 1
    raw_bytes = sum(count * h * w for h, w, _, _ in grids) * dtype.itemsize
    big = bool(bigtiff) if bigtiff is not None else raw_bytes > 3_900_000_000
    t = Affine.coerce(transform)
    if not t.is_rectilinear:
        raise NotImplementedError('rotated geo-transforms cannot be written')

    def source(ifd, plane):
        """ [bands or 1, h, w] pixels of IFD `ifd`: one band (planar 2) or all of them; a band stream blocks until the
        producer has finished them. """
        if stream is not None:
            stream.wait_band(plane) if planar == 2 else stream.wait_all()
        full = array if ifd == 0 else levels[ifd - 1]
        if stream is not None and ifd == 0:
            full = stream.array
        return full[plane:plane + 1] if planar == 2 else full

    def encode(job):
        ifd, plane, by, bx = job
        h, w = grids[ifd][:2]
        tile = np.zeros((th, tw, 1 if planar == 2 else count), dtype=dtype)
        ys, xs = slice(by * th, min((by + 1) * th, h)), slice(bx * tw, min((bx + 1) * tw, w))
        part = source(ifd, plane)[:, ys, xs]
        tile[:part.shape[1], :part.shape[2], :] = np.moveaxis(part, 0, 2)
        data = tile.tobytes()
        return zlib.compress(data, level) if deflate else data

    # file order: band by band (planar 2), each band's image tiles followed by its overview tiles -- so that a band
    # stream's overview tiles are encoded as soon as their band is ready
    jobs = [(i, p, by, bx) for p in range(count if planar == 2 else 1) for i, (_, _, down, across) in enumerate(grids)
            for by in range(down) for bx in range(across)]
    bo = '<'
    off_fmt, off_type = ('Q', 16) if big else ('I', 4)
    tmp = path.with_name(path.name + '.part')
    offsets = [[0] * (down * across * (count if planar == 2 else 1)) for _, _, down, across in grids]
    counts = [list(o) for o in offsets]
    try:
        with open(tmp, 'wb') as fh:
            fh.write(b'II' + (struct.pack('<HHHQ', 43, 8, 0, 0) if big else struct.pack('<HI', 42, 0)))
            # (a band stream gets its own workers: its jobs block while they wait for the producer, and must not starve the
            #  shared codec pool that readers decode on)
            own_pool = concurrent.futures.ThreadPoolExecutor(max_workers=max(2, os.cpu_count() or 2)) if stream is not None \
                else None
            try:
                for (ifd, plane, by, bx), data in zip(jobs, (own_pool if own_pool is not None else _codec_pool()).map(
                        encode, jobs)):
                    down, across = grids[ifd][2:]
                    index = (plane * down + by) * across + bx
                    offsets[ifd][index] = fh.tell()
                    counts[ifd][index] = len(data)
                    fh.write(data)
                    if fh.tell() % 2:
                        fh.write(b'\x00')
            finally:
                if own_pool is not None:
                    own_pool.shutdown(wait=True, cancel_futures=True)
            if photometric is None:
                photometric = 'rgb' if (count == 3 and dtype.kind == 'u' and dtype.itemsize == 1) else 'minisblack'
            base = 3 if photometric == 'rgb' else 1
            next_field = 8 if big else 4                            # where the first IFD's offset goes
            for ifd, (h, w, _, _) in enumerate(grids):
                # ---- IFD ----
                entries = []                                        # (tag, type, count, packed value bytes)

                def add(tag, typ, values):
                    if typ == 2:
                        data = str(values).encode('latin1', 'replace') + b'\x00'
                        entries.append((tag, 2, len(data), data))
                    else:
                        fmt = _FIELD[typ][0]
                        values = list(values)
                        entries.append((tag, typ, len(values), struct.pack(bo + fmt * len(values), *values)))

                if ifd > 0:
                    add(254, 4, [1])                                # NewSubfileType: reduced-resolution image
                add(256, 3 if w < 65536 else 4, [w])
                add(257, 3 if h < 65536 else 4, [h])
                add(258, 3, [sample[1]] * count)
                add(259, 3, [8 if deflate else 1])
                add(262, 3, [2 if photometric == 'rgb' else 1])
                add(277, 3, [count])
                add(284, 3, [planar])
                add(322, 3, [tw])
                add(323, 3, [th])
                add(324, off_type, offsets[ifd])
                add(325, off_type, counts[ifd])
                if count > base:
                    add(338, 3, [0] * (count - base))
                add(339, 3, [sample[0]] * count)
                if ifd == 0:
                    add(33550, 12, [abs(t.a), abs(t.e), 0.0])
                    add(33922, 12, [0.0, 0.0, 0.0, t.c, t.f, 0.0])
                    if geokeys is None:
                        geokeys = getattr(crs, 'raw_geokeys', None)  # a CRS read by GeoTiffReader carries its raw keys
                    if geokeys and geokeys[0]:
                        geokeys = _geokeys_pixel_is_area(geokeys)    # the tie point below is a pixel corner
                        add(34735, 3, geokeys[0])
                        if geokeys[1]:
                            add(34736, 12, geokeys[1])
                        if geokeys[2]:
                            add(34737, 2, geokeys[2])
                    xml = _gdal_metadata_xml(tags, band_tags, descriptions)
                    if xml:
                        add(42112, 2, xml)
                if nodata is not None:
                    add(42113, 2, 'nan' if (isinstance(nodata, float) and math.isnan(nodata)) else repr(
                        int(nodata) if float(nodata).is_integer() else float(nodata)))
                entries.sort(key=lambda e: e[0])
                if fh.tell() % 2:
                    fh.write(b'\x00')
                # out-of-line values first, then the directory
                inline = 8 if big else 4
                placed = []
                for tag, typ, cnt, data in entries:
                    if len(data) <= inline:
                        placed.append((tag, typ, cnt, data.ljust(inline, b'\x00')))
                    else:
                        pos = fh.tell()
                        fh.write(data)
                        if fh.tell() % 2:
                            fh.write(b'\x00')
                        placed.append((tag, typ, cnt, struct.pack(bo + off_fmt, pos)))
                ifd_pos = fh.tell()
                if big:
                    fh.write(struct.pack('<Q', len(placed)))
                    for tag, typ, cnt, value in placed:
                        fh.write(struct.pack('<HHQ', tag, typ, cnt) + value)
                    fh.write(struct.pack('<Q', 0))
                    end = fh.tell()
                    fh.seek(next_field)
                    fh.write(struct.pack('<Q', ifd_pos))
                    next_field = end - 8
                else:
                    if ifd_pos >= 2 ** 32:
                        raise ValueError('the image does not fit a classic TIFF: pass bigtiff=True')
                    fh.write(struct.pack('<H', len(placed)))
                    for tag, typ, cnt, value in placed:
                        fh.write(struct.pack('<HHI', tag, typ, cnt) + value)
                    fh.write(struct.pack('<I', 0))
                    end = fh.tell()
                    fh.seek(next_field)
                    fh.write(struct.pack('<I', ifd_pos))
                    next_field = end - 4
                fh.seek(end)
    except BaseException:
        # (a failed write -- e.g. a band stream whose producer failed -- leaves no partial file behind)
        try:
            os.unlink(tmp)
        except OSError:
            pass
        raise
    os.replace(tmp, path)
    return path
