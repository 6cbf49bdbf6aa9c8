"""
CPU tier: the footprint-statistics restatement (oracle/footprint_stats_restate.c: min, max, med, q1, q3, mode) against
the independent numpy restatement (oracle/footprint_stats_alt.py), bit for bit, and the properties the rules promise.
"""
import math

import numpy as np
import pytest

from oracle import footprint_stats_restate as fsr
from oracle.footprint_stats_alt import footprint_stats_alt

METHODS = fsr.METHODS
NAN = float('nan')


def _c(src, nodata, dst_shape, sx, ox, sy, oy, method):
    """ the C restatement through reproject_array, on transforms that give exactly (sx, ox, sy, oy) """
    return fsr.reproject_array(src, (1.0, 0.0, 0.0, 0.0, -1.0, 0.0), nodata, dst_shape, (sx, 0.0, ox, 0.0, -sy, -oy),
                               NAN, method)


def _bits_equal(a, b):
    return np.array_equal(np.asarray(a, 'float32').view('uint32'), np.asarray(b, 'float32').view('uint32'))


def _raster(rng, h, w, dtype, nodata, nan_holes=False, patch=(4, 9)):
    """ few distinct values (so mode has ties and quantiles have repeats), nodata holes, an all-nodata top-left
    ``patch`` (rows, columns), optional NaN pixels """
    if dtype == 'float32':
        src = rng.choice(np.array([-3.5, -0.0, 0.0, 1.25, 2.0, 7.0, 1e6], 'float32'), (h, w))
        noisy = rng.random((h, w)) < 0.3
        src[noisy] = rng.normal(0, 10, int(noisy.sum())).astype('float32')
    else:
        src = rng.integers(0, 6 if dtype == 'uint8' else 9, (h, w)).astype(dtype)
        src[rng.random((h, w)) < 0.2] = 200 if dtype == 'uint8' else 40000
    if nodata is not None:
        src[rng.random((h, w)) < 0.1] = nodata
        src[:patch[0], :patch[1]] = nodata
    if nan_holes:
        src[rng.random((h, w)) < 0.1] = np.nan
    return src


GEOMS = [
    # (hs, ws, hd, wd, sx, ox, sy, oy)
    (40, 42, 20, 21, 2.0, 0.0, 2.0, 0.0),                       # ratio 2
    (39, 40, 14, 14, 3.0, -1.0, 3.0, 1.0),                      # ratio 3, windows partly outside the raster
    (100, 90, 6, 5, 20.0, 0.0, 20.0, -5.0),                     # ratio 20, the first row of windows partly outside
    (43, 41, 17, 16, 2.7, 0.35, 2.7, -0.45),                    # ratio 2.7, sub-pixel offsets
    (70, 66, 12, 11, 6.4, 0.2, 6.4, 0.7),                       # ratio 6.4
    (12, 13, 31, 34, 0.4, 0.15, 0.4, -0.3),                     # up-sampling at 0.4
    (30, 60, 40, 18, 3.3, 0.1, 0.75, 0.2),                      # mixed axes: x down, y up
]
CASES = [('uint8', None, False), ('uint8', 0, False), ('uint16', 40000, False), ('uint16', None, False),
         ('float32', None, False), ('float32', NAN, False), ('float32', 2.0, True), ('float32', None, True)]


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('case', range(len(CASES)))
@pytest.mark.parametrize('geom', range(len(GEOMS)))
def test_c_vs_numpy_restatement(method, case, geom):
    hs, ws, hd, wd, sx, ox, sy, oy = GEOMS[geom]
    dtype, nodata, nan_holes = CASES[case]
    rng = np.random.default_rng(1000 * geom + 10 * case + METHODS.index(method))
    # (the patch covers the whole window of destination pixel (0, 0): an all-invalid window)
    patch = (math.ceil(sy + abs(oy)) + 1, math.ceil(sx + abs(ox)) + 1)
    src = _raster(rng, hs, ws, dtype, nodata, nan_holes, patch)
    got = _c(src, nodata, (hd, wd), sx, ox, sy, oy, method)
    exp = footprint_stats_alt(src, nodata, (hd, wd), sx, ox, sy, oy, method)
    assert _bits_equal(got, exp)
    assert (~np.isnan(got)).any()
    if nodata is not None:
        assert np.isnan(got[0, 0])


@pytest.mark.parametrize('geom', range(len(GEOMS)))
def test_order_and_membership(geom):
    """ min <= q1 <= med <= q3 <= max where valid, and every output is a valid value of its own window """
    from oracle.footprint_stats_alt import window
    hs, ws, hd, wd, sx, ox, sy, oy = GEOMS[geom]
    rng = np.random.default_rng(7 + geom)
    src = rng.normal(0, 50, (hs, ws)).astype('float32').round()
    src[rng.random((hs, ws)) < 0.15] = -9999
    src[rng.random((hs, ws)) < 0.05] = np.nan
    out = {m: _c(src, -9999, (hd, wd), sx, ox, sy, oy, m) for m in METHODS}
    valid = ~np.isnan(out['min'])
    for m in METHODS:
        assert np.array_equal(np.isnan(out[m]), ~valid), m
    chain = [out[m][valid] for m in ('min', 'q1', 'med', 'q3', 'max')]
    for lo, hi in zip(chain, chain[1:]):
        assert np.all(lo <= hi)
    for i in range(hd):
        y0, y1 = window(sy, oy, i, hs)
        for j in range(wd):
            x0, x1 = window(sx, ox, j, ws)
            win = src[y0:y1, x0:x1].ravel()
            win = win[~np.isnan(win) & (win != -9999)]
            for m in METHODS:
                assert (win.size == 0) == np.isnan(out[m][i, j])
                if win.size:
                    assert out[m][i, j] in win, (m, i, j)
    assert np.all(out['mode'][valid] >= out['min'][valid]) and np.all(out['mode'][valid] <= out['max'][valid])


def _one_window(values, method, nodata=None):
    """ the statistic of one destination pixel whose footprint is the 1 x n row ``values`` """
    src = np.asarray(values, dtype='float32')[None, :]
    return _c(src, nodata, (1, 1), float(src.shape[1]), 0.0, 1.0, 0.0, method)[0, 0]


@pytest.mark.parametrize('n', range(1, 9))
def test_quantile_indices(n):
    """ v[ceil(q n - 1)], checked by hand: for even n the median is the lower one """
    expected_index = {
        'med': [0, 0, 1, 1, 2, 2, 3, 3],
        'q1': [0, 0, 0, 0, 1, 1, 1, 1],
        'q3': [0, 1, 2, 2, 3, 4, 5, 5],
    }
    values = np.arange(10.0, 10.0 + n)[::-1]                   # descending, so sorting matters
    sorted_v = np.sort(values)
    for method, idx in expected_index.items():
        assert idx[n - 1] == math.ceil({'med': 0.5, 'q1': 0.25, 'q3': 0.75}[method] * n - 1)
        assert _one_window(values, method) == sorted_v[idx[n - 1]], (method, n)
    assert _one_window(values, 'min') == sorted_v[0]
    assert _one_window(values, 'max') == sorted_v[-1]


def test_mode_tie_rules():
    # all distinct: the first valid pixel in scan order
    assert _one_window([5.0, 3.0, 9.0, 1.0], 'mode') == 5.0
    assert _one_window([-1.0, 5.0, 3.0, 9.0], 'mode', nodata=-1.0) == 5.0
    # the highest count wins regardless of position
    assert _one_window([1.0, 2.0, 3.0, 3.0], 'mode') == 3.0
    # ties: the value whose LAST occurrence comes first (4 reaches 2 at position 2, 7 only at position 3)
    assert _one_window([7.0, 4.0, 4.0, 7.0], 'mode') == 4.0
    assert _one_window([4.0, 7.0, 7.0, 4.0], 'mode') == 7.0
    # (not the first occurrence: 7 occurs first, but 4 completes its count first)
    assert _one_window([7.0, 4.0, 4.0, 7.0, 1.0], 'mode') == 4.0
    # -0.0 and +0.0 are one value, stored as +0.0
    got = _one_window([-0.0, 2.0, 0.0, 2.0, -0.0], 'mode')
    assert got == 0.0 and not np.signbit(got)
    assert not np.signbit(_one_window([-0.0, -0.0, 1.0], 'min'))
    # NaN is never counted, not even under a numeric nodata
    assert _one_window([np.nan, np.nan, np.nan, 3.0], 'mode') == 3.0
    assert _one_window([np.nan, np.nan, 8.0, 3.0], 'mode', nodata=3.0) == 8.0
    assert np.isnan(_one_window([np.nan, 3.0], 'mode', nodata=3.0))


def test_two_dimensional_scan_order():
    """ scan order is row-major over the clipped window """
    src = np.array([[6.0, 2.0],
                    [2.0, 6.0]], dtype='float32')          # 2 completes at index 2, 6 at index 3
    assert _c(src, None, (1, 1), 2.0, 0.0, 2.0, 0.0, 'mode')[0, 0] == 2.0
    assert _c(src.T.copy()[:, ::-1].copy(), None, (1, 1), 2.0, 0.0, 2.0, 0.0, 'mode')[0, 0] == 6.0


def test_enum_names():
    from homonim_b200.enums import Resampling

    class RasterioLike:
        def __init__(self, name):
            self.name = name

    for name in ('min', 'max', 'med', 'q1', 'q3', 'mode'):
        assert Resampling.coerce(name) == Resampling(name) == name
        assert Resampling.coerce(RasterioLike(name)) is Resampling(name)
    from homonim_b200 import RefSpaceModel
    RefSpaceModel(downsampling='med', upsampling='mode')
