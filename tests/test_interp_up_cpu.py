"""
CPU tier: the bilinear, cubic and lanczos up-sampling restatement (oracle/interp_up_restate.c) against the independent
numpy restatement (oracle/interp_up_alt.py), and properties each method must have.
"""
import math

import numpy as np
import pytest

from oracle import interp_up_restate
from oracle.interp_up_alt import interp_up_alt

METHODS = ('bilinear', 'cubic', 'lanczos')


def _c(src, nodata, dst_shape, sx, ox, sy, oy, method):
    """ the C restatement through reproject_array, on transforms that give exactly (sx, ox, sy, oy) """
    src_tf = (1.0, 0.0, 0.0, 0.0, -1.0, 0.0)
    dst_tf = (sx, 0.0, ox, 0.0, -sy, -oy)
    return interp_up_restate.reproject_array(src, src_tf, nodata, dst_shape, dst_tf, float('nan'), method)


def _raster(rng, nb, h, w, holes=0.1, band_holes=0.05):
    src = rng.uniform(-5.0, 50.0, (nb, h, w))
    src[:, rng.random((h, w)) < holes] = np.nan
    if nb > 1:
        src[1, rng.random((h, w)) < band_holes] = np.nan                   # single-band holes
    return src


def _rel_err(a, b):
    m = ~np.isnan(b)
    return float(np.max(np.abs(a[m].astype('float64') - b[m]) / np.maximum(np.abs(b[m]), 1.0))) if m.any() else 0.0


GEOMS = [
    # (hs, ws, hd, wd, sx, ox, sy, oy)
    (9, 11, 36, 44, 0.25, 0.0, 0.25, 0.0),                      # integer ratio, aligned
    (7, 8, 21, 24, 1 / 3, 0.1, 1 / 3, -0.2),                    # integer ratio, sub-pixel shift
    (10, 9, 16, 14, 0.625, 0.0, 0.625, 0.0),                    # ratio 1.6
    (12, 13, 13, 14, 0.91, -0.3, 0.91, 0.4),                    # ratio 1.1, shifted past the edges
    (6, 7, 6, 7, 1.0, 0.0, 1.0, 0.0),                           # same grid
    (5, 6, 23, 29, 0.2, -0.7, 0.2, 0.3),                        # ratio 5, destination overhanging the source
]


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('nb', [1, 2])
@pytest.mark.parametrize('geom', range(len(GEOMS)))
def test_c_vs_numpy_restatement(method, nb, geom):
    hs, ws, hd, wd, sx, ox, sy, oy = GEOMS[geom]
    rng = np.random.default_rng(100 * geom + 10 * nb + METHODS.index(method))
    src = _raster(rng, nb, hs, ws)
    got = _c(src, float('nan'), (hd, wd), sx, ox, sy, oy, method)
    exp = interp_up_alt(src, float('nan'), (hd, wd), sx, ox, sy, oy, method)
    assert np.array_equal(np.isnan(got), np.isnan(exp))
    assert _rel_err(got, exp) <= 1e-12
    assert (~np.isnan(got)).any()


@pytest.mark.parametrize('method', METHODS)
def test_integer_nodata_and_no_nodata(method):
    rng = np.random.default_rng(3)
    src = rng.integers(0, 4, (2, 8, 9)).astype('float64')
    for nodata in (0.0, None):
        got = _c(src, nodata, (20, 22), 0.4, 0.05, 0.4, 0.0, method)
        exp = interp_up_alt(src, nodata, (20, 22), 0.4, 0.05, 0.4, 0.0, method)
        assert np.array_equal(np.isnan(got), np.isnan(exp))
        assert _rel_err(got, exp) <= 1e-12


@pytest.mark.parametrize('method', METHODS)
def test_constant_field_stays_constant(method):
    src = np.full((10, 12), 7.25)
    src[4, 5] = np.nan
    got = _c(src, float('nan'), (33, 40), 0.3, 0.1, 0.3, -0.05, method)
    m = ~np.isnan(got)
    assert m.sum() > 0.9 * got.size
    if method == 'lanczos':
        # lanczos weights do not sum to 1 and GDAL leaves a sum within 1e-5 of 1 undivided: kept to 1e-5 only
        assert np.max(np.abs(got[m] - 7.25)) <= 7.25 * 1e-5
    else:
        # weights summing to 1 (or divided by their sum): an error below 1e-12 rounds to the float32 value itself
        assert np.all(got[m] == np.float32(7.25))
    alt = interp_up_alt(src, float('nan'), (33, 40), 0.3, 0.1, 0.3, -0.05, method)
    assert np.array_equal(np.isnan(alt), ~m)


def test_bilinear_reproduces_linear_ramp():
    y, x = np.mgrid[0:12, 0:14].astype('float64')
    src = 3.0 + 0.5 * x - 1.25 * y
    hd, wd, s = 48, 56, 0.25
    got = _c(src, None, (hd, wd), s, 0.0, s, 0.0, 'bilinear').astype('float64')
    cx = s * (np.arange(wd) + 0.5) - 0.5                        # source pixel-centre coordinates of the centres
    cy = s * (np.arange(hd) + 0.5) - 0.5
    exp = 3.0 + 0.5 * cx[None, :] - 1.25 * cy[:, None]
    inner = (slice(4, -4), slice(4, -4))
    assert np.max(np.abs(got[inner] - exp[inner])) <= 1e-5


def test_cubic_reproduces_quadratic():
    y, x = np.mgrid[0:12, 0:14].astype('float64')
    src = 1.0 + 0.1 * x * x - 0.05 * y * y + 0.02 * x * y
    hd, wd, s = 36, 42, 1 / 3
    got = _c(src, None, (hd, wd), s, 0.0, s, 0.0, 'cubic').astype('float64')
    cx = s * (np.arange(wd) + 0.5) - 0.5
    cy = s * (np.arange(hd) + 0.5) - 0.5
    exp = 1.0 + 0.1 * cx[None, :] ** 2 - 0.05 * cy[:, None] ** 2 + 0.02 * cx[None, :] * cy[:, None]
    inner = (slice(6, -6), slice(6, -6))
    assert np.max(np.abs(got[inner] - exp[inner]) / np.abs(exp[inner])) <= 1e-6


def test_cubic_falls_back_to_bilinear_bit_for_bit():
    rng = np.random.default_rng(5)
    src = _raster(rng, 1, 10, 11, holes=0.08, band_holes=0.0)[0]
    args = ((31, 35), 0.31, 0.02, 0.31, -0.1)
    cub = _c(src, float('nan'), *args, 'cubic')
    bil = _c(src, float('nan'), *args, 'bilinear')
    hd, wd = args[0]
    _, ky, _ = (None,) + tuple(_kd(hd, 0.31, -0.1))
    _, kx, _ = (None,) + tuple(_kd(wd, 0.31, 0.02))
    h, w = src.shape
    n_fallback = 0
    for i in range(hd):
        for j in range(wd):
            ys = np.arange(ky[i] - 1, ky[i] + 3)
            xs = np.arange(kx[j] - 1, kx[j] + 3)
            leaves = ys.min() < 0 or ys.max() >= h or xs.min() < 0 or xs.max() >= w
            if leaves or np.isnan(src[np.ix_(ys, xs)]).any():
                n_fallback += 1
                assert np.array_equal(cub[i, j], bil[i, j], equal_nan=True)
    assert n_fallback > 50


def _kd(n, s, o):
    src = s * (np.arange(n) + 0.5) + o
    k = np.floor(src - 0.5)
    return k.astype('int64'), src - 0.5 - k


def test_lanczos_reach_is_three_taps():
    # a destination pixel whose cell is (k, k+1) reads taps k-2 .. k+3: a hole at k+3 changes it, one at k+4 does not
    src = np.arange(1.0, 1.0 + 14 * 14).reshape(14, 14) % 7 + 1.0
    hd = wd = 14 * 4
    base = _c(src, float('nan'), (hd, wd), 0.25, 0.0, 0.25, 0.0, 'lanczos')
    i = j = 4 * 5 + 3                                          # src_y = src_x = 5.875: k = 5, d = 0.375
    for dk, changes in ((3, True), (4, False), (-2, True), (-3, False)):
        holed = src.copy()
        holed[5 + dk, 5] = np.nan
        got = _c(holed, float('nan'), (hd, wd), 0.25, 0.0, 0.25, 0.0, 'lanczos')
        assert (got[i, j] != base[i, j]) == changes, dk


@pytest.mark.parametrize('method', METHODS)
def test_centre_rule(method):
    src = np.full((8, 8), 3.0)
    src[3, 4] = np.nan
    got = _c(src, float('nan'), (32, 32), 0.25, 0.0, 0.25, 0.0, method)
    assert np.isnan(got[12:16, 16:20]).all()                   # centres inside the hole
    assert not np.isnan(got[11, 16]) and not np.isnan(got[16, 16])
    # 2 bands: the centre rule is unified (any band valid); each band's own taps decide its value
    two = np.stack([src, np.full((8, 8), 2.0)])
    got2 = _c(two, float('nan'), (32, 32), 0.25, 0.0, 0.25, 0.0, method)
    assert not np.isnan(got2[:, 12:16, 16:20]).any()
    assert not np.isnan(got2[1, 12:16, 16:20]).any()


@pytest.mark.parametrize('method', METHODS)
def test_downsampling_not_restated(method):
    with pytest.raises(NotImplementedError):
        _c(np.ones((8, 8)), None, (4, 4), 2.0, 0.0, 2.0, 0.0, method)
