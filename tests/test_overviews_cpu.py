"""
CPU tier, internal overviews of the output files (reference fuse.py:151-165): the number of levels, the pixel rule of the
numpy oracle on hand-worked windows, and the GeoTIFF writer / reader of reduced-resolution IFDs.  No GPU.
"""
import math
import pathlib
import threading
import time

import numpy as np
import pytest

from homonim_b200.geometry import Affine
from homonim_b200.geotiff import BandStream, GeoTiffReader, write_geotiff
from homonim_b200.overviews import level_shape, overview_factors
from oracle import overviews_np as ovnp

GEOKEYS = ((1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 3857), (), '')
TF = Affine(5.0, 0.0, -57129.5, 0.0, -5.0, -3723906.75)
NAN = float('nan')


@pytest.mark.parametrize('shape, factors', [
    ((805, 1421), [2]), ((5000, 5000), [2, 4, 8, 16]), ((511, 9000), []), ((100, 100), []), ((256, 256), []),
    ((512, 512), [2]), ((200000, 200000), [2, 4, 8, 16, 32, 64, 128, 256]), ((3, 1023, 2048), [2]),
])
def test_overview_factors_follow_the_reference_rule(shape, factors):
    assert overview_factors(shape) == factors
    assert ovnp.overview_factors(shape[-2:]) == factors
    assert overview_factors((5000, 5000), max_num_levels=2) == [2, 4]


def test_level_shape_rounds_up():
    assert level_shape((805, 1421), 2) == (403, 711)
    assert level_shape((4, 7, 1), 4) == (4, 2, 1)


def _one(values, dtype, nodata):
    """ Level 1 of a plane given as nested lists. """
    return ovnp.next_level(np.array(values, dtype=dtype), nodata)


def test_oracle_hand_worked_windows():
    # constant planes stay constant, at every level
    for dtype in ('uint8', 'uint16', 'int16', 'float32'):
        plane = np.full((13, 7), 9, dtype)
        for level in ovnp.build_overviews(plane, None, 3):
            assert level.dtype == plane.dtype and np.all(level == 9)
    # integer: round half up on the exact sum
    assert _one([[1, 1], [2, 2]], 'uint16', None)[0, 0] == 2                 # 6 / 4 = 1.5 -> 2
    assert _one([[1, 1], [2, 0]], 'uint16', 0)[0, 0] == 1                    # 4 / 3 = 1.33 -> 1
    assert _one([[1, 2], [2, 0]], 'uint16', 0)[0, 0] == 2                    # 5 / 3 = 1.67 -> 2
    assert _one([[255, 255], [255, 254]], 'uint8', None)[0, 0] == 255        # 254.75, no overflow
    assert _one([[-1, -2], [-2, -2]], 'int16', None)[0, 0] == -2             # -1.75 -> -2
    assert _one([[-1, -2], [-1, -2]], 'int16', None)[0, 0] == -1             # -1.5 -> -1 (half up)
    assert _one([[-3, -9999], [-4, -9999]], 'int16', -9999)[0, 0] == -3      # -3.5 -> -3
    # no valid pixel: nodata
    assert _one([[0, 0], [0, 0]], 'uint8', 0)[0, 0] == 0
    assert _one([[-9999, -9999], [-9999, -9999]], 'int16', -9999)[0, 0] == -9999
    assert np.isnan(_one([[NAN, NAN], [NAN, NAN]], 'float32', None)[0, 0])
    assert _one([[NAN, -9999], [NAN, -9999]], 'float32', -9999)[0, 0] == -9999
    # float: NaN is never valid; double sum, one rounding
    assert _one([[1, NAN], [2, NAN]], 'float32', None)[0, 0] == 1.5
    assert _one([[1, 2], [4, -9999]], 'float32', -9999)[0, 0] == np.float32(7 / 3)
    big = np.float32(3e38)
    assert _one([[big, big], [big, big]], 'float32', None)[0, 0] == big      # no float32 overflow in the sum
    # odd sizes: the edge windows hold 1 or 2 pixels; 1 x N planes
    level = _one([[1, 2, 3], [4, 5, 6], [7, 8, 9]], 'uint16', None)
    assert level.tolist() == [[3, 5], [8, 9]]                                 # (1+2+4+5)/4, (3+6)/2, (7+8)/2, 9
    assert _one([[1, 2, 3, 4, 5]], 'uint8', None).tolist() == [[2, 4, 5]]     # 1.5 -> 2, 3.5 -> 4, 5
    assert _one([[1], [2], [3]], 'float32', None).tolist() == [[1.5], [3.0]]
    assert ovnp.build_overviews(np.arange(5, dtype='uint8')[None], None, 4)[-1].shape == (1, 1)


def test_oracle_cascades_from_stored_values():
    """ Level 2 is computed from level 1 as stored (rounded), not from the base. """
    plane = np.array([[1, 2, 0, 0], [1, 2, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]], 'uint16')
    lv1, lv2 = ovnp.build_overviews(plane, None, 2)
    assert lv1.tolist() == [[2, 0], [0, 0]]                                   # 6 / 4 = 1.5 -> 2
    assert lv2[0, 0] == 1                                                     # (2 + 0 + 0 + 0) / 4 = 0.5 -> 1
    assert (2 * int(plane.sum()) + 16) // 32 == 0                             # the base average, 0.375, would give 0
    # a stored value equal to nodata is nodata at the next level
    plane = np.array([[-9998, -10000], [-9998, -10000]], 'int16')
    assert ovnp.build_overviews(plane, -9999, 1)[0][0, 0] == -9999


@pytest.mark.parametrize('dtype, nodata', [('uint8', 0), ('uint16', None), ('int16', -9999), ('float32', NAN),
                                           ('float32', -9999.0), ('float32', None)])
def test_oracle_vectorised_equals_per_window_loops(dtype, nodata):
    rng = np.random.default_rng(4)
    for shape in ((1, 9), (9, 1), (17, 23), (32, 31)):
        plane = rng.integers(-3 if dtype != 'uint8' and dtype != 'uint16' else 0, 6, shape).astype(dtype)
        if dtype == 'float32':
            plane = plane * np.float32(1.37)
            plane[rng.random(shape) < 0.2] = NAN
        if nodata is not None and not math.isnan(nodata):
            plane[rng.random(shape) < 0.3] = nodata
        fast = ovnp.build_overviews(plane, nodata, 4)
        slow = ovnp.build_overviews(plane, nodata, 4, reduce=ovnp.next_level_loops)
        for a, b in zip(fast, slow):
            assert a.dtype == b.dtype and np.array_equal(a, b, equal_nan=True)


def _pyramid(dtype, count, height, width, n, nodata, seed=3):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 200, (count, height, width)).astype(dtype)
    if nodata is not None and not math.isnan(nodata):
        base[:, :5, :7] = nodata
    elif dtype == 'float32':
        base[:, :5, :7] = NAN
    return base, ovnp.build_overviews(base, nodata, n)


@pytest.mark.parametrize('dtype, count, interleave, compress, bigtiff', [
    ('uint8', 3, 'band', 'deflate', None),
    ('uint16', 4, 'pixel', None, None),
    ('int16', 2, 'band', None, True),
    ('float32', 1, 'band', 'deflate', True),
    ('float32', 3, 'pixel', 'deflate', None),
    ('uint16', 2, 'band', 'deflate', True),
])
def test_geotiff_overviews_round_trip(tmp_path, dtype, count, interleave, compress, bigtiff):
    nodata = NAN if dtype == 'float32' else (-9999 if dtype == 'int16' else 0)
    height, width = 150, 97
    base, levels = _pyramid(dtype, count, height, width, 3, nodata)
    path = write_geotiff(tmp_path / 'o.tif', base, TF, nodata=nodata, geokeys=GEOKEYS, compress=compress, blocksize=32,
                         interleave=interleave, bigtiff=bigtiff, descriptions=[f'b{i}' for i in range(count)],
                         tags=dict(FUSE_MODEL='gain'), overviews=levels)
    with GeoTiffReader(path) as im:
        assert im._big == bool(bigtiff) and im.overview_level is None
        assert (im.height, im.width, im.count) == (height, width, count) and im.transform == TF
        assert np.array_equal(im.read(), base, equal_nan=True)
        # rasterio's factors, round(width / level width): 97 -> 49, 25, 13 gives 2, 4, 7
        assert [im.overviews(b) for b in range(1, count + 1)] == [[2, 4, 7]] * count
    for k, level in enumerate(levels):
        with GeoTiffReader(path, overview_level=k) as im:
            h, w = level.shape[1:]
            assert (im.height, im.width, im.count, im.dtype.name) == (h, w, count, dtype)
            assert im.block_shape == (32, 32) and im.planar == (2 if interleave == 'band' and count > 1 else 1)
            assert im.compression == (8 if compress else 1)
            assert np.array_equal(im.read(), level, equal_nan=True)
            assert im.transform == TF * Affine.scale(width / w, height / h)
            assert im.crs is not None and im.descriptions == [f'b{i}' for i in range(count)]
            assert im.tags() == dict(FUSE_MODEL='gain')
            assert (math.isnan(im.nodata) if dtype == 'float32' else im.nodata == nodata)
            assert im.overviews(1) == [2, 4, 7]
    with pytest.raises(ValueError, match='overview level'):
        GeoTiffReader(path, overview_level=3)


def test_geotiff_without_overviews_is_unchanged(tmp_path):
    """ overviews=None and overviews=[] write the same bytes; a file without overviews reports none. """
    base = np.arange(3 * 40 * 50, dtype='uint16').reshape(3, 40, 50)
    a = write_geotiff(tmp_path / 'a.tif', base, TF, nodata=0, blocksize=16)
    b = write_geotiff(tmp_path / 'b.tif', base, TF, nodata=0, blocksize=16, overviews=[])
    assert pathlib.Path(a).read_bytes() == pathlib.Path(b).read_bytes()
    with GeoTiffReader(a) as im:
        assert im.overviews(1) == []
        with pytest.raises(IndexError):
            im.overviews(4)
    with pytest.raises(ValueError):
        GeoTiffReader(a, overview_level=0)


def test_geotiff_rejects_wrong_overviews(tmp_path):
    base = np.zeros((2, 41, 30), 'uint16')
    good = [np.zeros((2, 21, 15), 'uint16'), np.zeros((2, 11, 8), 'uint16')]
    write_geotiff(tmp_path / 'ok.tif', base, TF, overviews=good)
    for bad in ([np.zeros((2, 20, 15), 'uint16')],                      # floor instead of ceil
                [good[1]],                                              # factor 4 given as the first level
                [np.zeros((1, 21, 15), 'uint16')],                      # band count
                [good[0].astype('float32')],                            # dtype
                [good[0], good[0]]):                                    # a repeated level
        with pytest.raises(ValueError, match='overview'):
            write_geotiff(tmp_path / 'bad.tif', base, TF, overviews=bad)
        assert not (tmp_path / 'bad.tif').exists()
    stream = BandStream(base.copy(), overviews=good)
    with pytest.raises(ValueError, match='BandStream'):
        write_geotiff(tmp_path / 'bad.tif', stream, TF, overviews=good)


def test_band_stream_writer_with_overviews_equals_eager_writer(tmp_path):
    """ Overview tiles fed band by band through the band stream give the same bytes as the eager call. """
    base, levels = _pyramid('uint16', 3, 300, 420, 2, 0, seed=8)
    tf = Affine(2.0, 0, 100.0, 0, -2.0, 900.0)
    for compress, interleave in (('deflate', 'band'), (None, 'band'), ('deflate', 'pixel')):
        eager = write_geotiff(tmp_path / f'eager_{compress}_{interleave}.tif', base, tf, nodata=0, compress=compress,
                              blocksize=64, interleave=interleave, overviews=levels)
        buf = np.zeros_like(base)
        lv_bufs = [np.zeros_like(lv) for lv in levels]
        stream = BandStream(buf, overviews=lv_bufs)

        def produce():
            for b in range(3):
                time.sleep(0.05)
                buf[b] = base[b]
                for dst, src in zip(lv_bufs, levels):
                    dst[b] = src[b]
                stream.set_ready(b)
        t = threading.Thread(target=produce)
        t.start()
        lazy = write_geotiff(tmp_path / f'lazy_{compress}_{interleave}.tif', stream, tf, nodata=0, compress=compress,
                             blocksize=64, interleave=interleave)
        t.join()
        assert pathlib.Path(eager).read_bytes() == pathlib.Path(lazy).read_bytes()
        with GeoTiffReader(lazy, overview_level=1) as im:
            assert np.array_equal(im.read(), levels[1])


def test_mask_check_ignores_overview_ifds(tmp_path):
    """ Reduced-resolution IFDs (NewSubfileType = 1) are not masks: the file opens. """
    base, levels = _pyramid('uint8', 1, 64, 64, 2, 0)
    path = write_geotiff(tmp_path / 'o.tif', base, TF, nodata=0, overviews=levels, compress=None)
    with GeoTiffReader(path) as im:
        assert not im.has_internal_mask and im.overviews(1) == [2, 4]
