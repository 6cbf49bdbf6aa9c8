"""
GPU tier: each C-ABI entry point of include/homonim_b200.h against the matching oracle function, plus
size-independent properties at BASELINE.json's full raster sizes (where the oracle would take too long).
"""
import ctypes

import numpy as np
import pytest

from conftest import RTOL, assert_same_mask, check_corr, rel_err

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from homonim_b200 import Affine, _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402

NAN = float('nan')
TF_LO = Affine(10, 0, 2000, 0, -10, 9000)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _oracle():
    from oracle import gdal_restate, kernel_model_np
    return gdal_restate, kernel_model_np


def _rand_src(rng, h, w, dtype, nodata, holes=True):
    if dtype == 'float32':
        a = rng.normal(0.3, 0.1, (h, w)).astype('float32')
    else:
        a = rng.integers(1, np.iinfo(dtype).max, (h, w)).astype(dtype)
    if holes:
        a[rng.integers(0, h, 50), rng.integers(0, w, 50)] = nodata
        a[h // 3:h // 3 + 7, w // 4:w // 4 + 9] = nodata
    return a


@pytest.mark.parametrize('dtype, nodata, ratio, shift, hw', [
    ('uint16', 0, 20, (0, 0), (30, 37)),          # C2 geometry: aligned, exact integer sums -> bit-exact
    ('uint8', 0, 4, (0, 0), (50, 64)),
    ('float32', NAN, 20, (0, 0), (30, 37)),
    ('float32', NAN, 2, (0, 0), (100, 91)),
    ('uint16', 0, 5, (1.3, 2.6), (40, 33)),       # mis-aligned: fractional edge weights
    ('float32', NAN, 3, (0.5, 0.25), (41, 50)),
    ('float32', -9999.0, 2.5, (0.2, 0.7), (40, 44)),   # non-integer ratio, value nodata
    ('uint16', 0, 100, (0, 0), (9, 11)),          # few destination pixels per warp strip
    ('uint8', 0, 300, (7.0, 3.0), (12, 13)),      # very large ratio (0.1 m drone imagery vs 30 m Landsat)
])
def test_downsample_average(dtype, nodata, ratio, shift, hw):
    gr, _ = _oracle()
    rng = np.random.default_rng(1)
    hd, wd = hw
    hs, ws = int(hd * ratio) - 3, int(wd * ratio) - 5          # source does not quite cover the last cells
    src = _rand_src(rng, hs, ws, dtype, nodata)
    src_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
    expected = gr.reproject_array(src, tuple(src_tf), nodata, (hd, wd), tuple(TF_LO), NAN, 'average')
    got = hkm._downsample_average(torch.from_numpy(src).cuda(), src_tf, nodata, (hd, wd), TF_LO).cpu().numpy()
    inside = np.ones((hd, wd), bool)      # cells whose footprint leaves the raster follow the padded-source convention
    gm = hkm.grid_map(src_tf, TF_LO)
    jj, ii = np.meshgrid(np.arange(wd), np.arange(hd))
    inside &= (gm.sx * jj + gm.ox >= 0) & (gm.sx * (jj + 1) + gm.ox <= ws)
    inside &= (gm.sy * ii + gm.oy >= 0) & (gm.sy * (ii + 1) + gm.oy <= hs)
    assert inside.mean() > 0.8
    assert_same_mask(got[inside], expected[inside], 'average')
    if dtype != 'float32' and shift == (0, 0):
        assert np.array_equal(got[inside], expected[inside], equal_nan=True)       # bit-exact
    else:
        assert rel_err(got[inside], expected[inside], 1e-3 * np.nanmean(np.abs(expected))) <= 1e-6


@pytest.mark.parametrize('nb', [1, 2])
@pytest.mark.parametrize('ratio, shift', [(20, (0, 0)), (2, (0, 0)), (4, (1.3, 2.6)), (3, (0.5, 0.25)), (1.6, (0, 0))])
def test_resample_up_cubic_spline(nb, ratio, shift):
    gr, _ = _oracle()
    rng = np.random.default_rng(2)
    hp, wp = 40, 33
    coarse = rng.normal(1.0, 0.2, (nb, hp, wp)).astype('float32')
    coarse[:, 10:13, 5:9] = NAN
    coarse[0, 30, 20] = NAN                                    # invalid in one band only
    coarse[:, :, -1] = NAN
    hd, wd = int(hp * ratio) + 3, int(wp * ratio) + 2          # destination slightly larger than the coarse raster
    dst_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
    arr = coarse if nb == 2 else coarse[0]
    expected = gr.reproject_array(arr, tuple(TF_LO), NAN, (hd, wd), tuple(dst_tf), NAN, 'cubic_spline')
    got = hkm._resample_up(torch.from_numpy(arr).cuda(), TF_LO, NAN, (hd, wd), dst_tf).cpu().numpy()
    assert_same_mask(got, expected, 'cubic_spline')
    assert rel_err(got, expected, 1e-3) <= 1e-6


def test_resample_up_nearest():
    gr, _ = _oracle()
    rng = np.random.default_rng(3)
    coarse = rng.normal(1.0, 0.2, (25, 31)).astype('float32')
    coarse[3:6, 4:8] = NAN
    dst_tf = TF_LO * Affine.scale(1.0 / 3) * Affine.translation(0.5, 0.25)
    expected = gr.reproject_array(coarse, tuple(TF_LO), NAN, (80, 95), tuple(dst_tf), NAN, 'nearest')
    got = hkm._resample_up(torch.from_numpy(coarse).cuda(), TF_LO, NAN, (80, 95), dst_tf,
                           _native.HB_UP_NEAREST).cpu().numpy()
    assert np.array_equal(got, expected, equal_nan=True)


@pytest.mark.parametrize('dtype, nodata, ratio, shift, partial', [
    ('uint16', 0, 20, (0, 0), False), ('uint8', 0, 4, (0, 0), True), ('float32', NAN, 5, (1.3, 2.6), False),
    ('float32', NAN, 2, (0, 0), True), ('uint16', 0, 3, (0.5, 0.25), True),
])
def test_upsample_apply(dtype, nodata, ratio, shift, partial):
    """ hb_upsample_apply (+ hb_valid_mask + hb_full_coverage_mask) against RefSpaceModel.apply of the oracle. """
    _, kmnp = _oracle()
    rng = np.random.default_rng(4)
    hp, wp = 36, 30
    hs, ws = hp * ratio - 2, wp * ratio - 3
    src = _rand_src(rng, hs, ws, dtype, nodata)
    params = np.stack([rng.normal(0.7, 0.1, (hp, wp)), rng.normal(20.0, 50.0, (hp, wp))]).astype('float32')
    params[:, 8:12, 10:15] = NAN
    params[:, :2, :] = NAN
    src_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
    # the reference reads its source block boundlessly (nodata beyond the raster, raster_array.py:175-199): give the
    # oracle the padded block, and compare on the un-padded extent
    pad = 2 * ratio
    src_pad = np.full((hs + 2 * pad, ws + 2 * pad), nodata, dtype=src.dtype)
    src_pad[pad:pad + hs, pad:pad + ws] = src
    pad_tf = src_tf * Affine.translation(-pad, -pad)
    expected = kmnp.refspace_apply(src_pad, tuple(pad_tf), nodata, params, tuple(TF_LO), (3, 5),
                                   mask_partial=partial)[pad:pad + hs, pad:pad + ws]
    from homonim_b200 import CRS, Model, RasterArray, RefSpaceModel
    crs = CRS.from_epsg(3857)
    km = RefSpaceModel(Model.gain_blk_offset, (3, 5), mask_partial=partial)
    got = km.apply(RasterArray(src, crs, src_tf, nodata=nodata), RasterArray(params, crs, TF_LO, nodata=NAN)).array
    check_corr(got, expected.astype('float32'), 'upsample_apply')


def test_block_norm():
    _, kmnp = _oracle()
    lib = _native.lib()
    rng = np.random.default_rng(5)
    # 2**22: the largest block of the single cooperative launch; 2**22 + 1: the smallest of the multi-kernel path
    for n, nodata in ((1, NAN), (7, NAN), (9, NAN), (129, NAN), (1000, NAN), (4097, 0.0), (250_000, 0.0), (1_000_003, NAN),
                      (2**22, NAN), (2**22 + 1, 0.0), (9_000_000, NAN)):
        src = rng.normal(3000, 900, n).astype('float32')
        ref = (0.7 * src + 100 + rng.normal(0, 30, n)).astype('float32')
        bad = rng.random(n) < 0.05
        src[bad & (np.arange(n) % 2 == 0)] = nodata
        ref[bad & (np.arange(n) % 2 == 1)] = NAN
        if n < 10:
            src[:] = np.abs(src) + 1
            ref[:] = np.abs(ref) + 1
        mask = ~kmnp.nan_equals(src, nodata) & ~np.isnan(ref)
        with np.errstate(all='ignore'):
            expected = kmnp.block_norm(src, ref, mask)
        s, r = torch.from_numpy(src).cuda(), torch.from_numpy(ref).cuda()
        norm = torch.zeros(2, dtype=torch.float64, device='cuda')
        nbytes = lib.hb_block_norm_workspace_bytes(n)
        work = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
        _native.check(lib.hb_block_norm(s.data_ptr(), 1, nodata, r.data_ptr(), 1, NAN, n, norm.data_ptr(),
                                        work.data_ptr(), nbytes, _stream()))
        got = norm.cpu().numpy()
        if n == 1:
            assert np.isnan(got[0]) == np.isnan(expected[0])      # std == 0 -> 0/0
            continue
        # bit for bit: the float32 standard deviations replay numpy's pairwise summation (np.std of `array[mask]`), the
        # order statistics are exact and the interpolation follows numpy's float32 arithmetic
        assert got[0] == expected[0], (n, got, expected)
        assert got[1] == expected[1], (n, got, expected)


def test_block_norm_empty_mask():
    lib = _native.lib()
    s = torch.full((100,), NAN, device='cuda')
    norm = torch.ones(2, dtype=torch.float64, device='cuda')
    nbytes = lib.hb_block_norm_workspace_bytes(100)
    work = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    _native.check(lib.hb_block_norm(s.data_ptr(), 1, NAN, s.data_ptr(), 1, NAN, 100, norm.data_ptr(), work.data_ptr(),
                                    nbytes, _stream()))
    assert norm.cpu().tolist() == [0.0, 0.0]                       # kernel_model.py:223-226


def test_fuse_refspace_host_entry_point():
    """ hb_fuse_refspace_host with HOST buffers equals the device-pointer pipeline and the oracle. """
    _, kmnp = _oracle()
    lib = _native.lib()
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(60, 52, 10, bands=1, dtype='uint16', seed=9, device='cpu', src_nodata=0, ref_pad=0)
    src = np.ascontiguousarray(src_ra.array[0].numpy())
    ref = np.ascontiguousarray(ref_ra.array[0].numpy())
    gm = hkm.grid_map(src_ra.transform, ref_ra.transform)
    corr = np.empty(src.shape, 'float32')
    params = np.empty((3,) + ref.shape, 'float32')
    _native.check(lib.hb_fuse_refspace_host(
        src.ctypes.data, _native.HB_U16, src.shape[0], src.shape[1], 1, 0.0, ref.ctypes.data, ref.shape[0],
        ref.shape[1], 1, NAN, gm.sx, gm.ox, gm.sy, gm.oy, _native.HB_MODEL_GAIN_OFFSET, 15, 15, 1, 1, 0.25,
        _native.HB_F32, 0, 0.0, corr.ctypes.data, params.ctypes.data, _stream()))
    # the same call with the output dtype conversion fused in: uint16, nodata 0 (raster_array.py:353-387)
    corr16 = np.empty(src.shape, 'uint16')
    _native.check(lib.hb_fuse_refspace_host(
        src.ctypes.data, _native.HB_U16, src.shape[0], src.shape[1], 1, 0.0, ref.ctypes.data, ref.shape[0],
        ref.shape[1], 1, NAN, gm.sx, gm.ox, gm.sy, gm.oy, _native.HB_MODEL_GAIN_OFFSET, 15, 15, 1, 1, 0.25,
        _native.HB_U16, 1, 0.0, corr16.ctypes.data, None, _stream()))
    exp16 = np.where(np.isnan(corr), 0, np.clip(np.round(np.nan_to_num(corr)), 0, 65535)).astype('uint16')
    assert np.array_equal(corr16, exp16)
    exp_params, _, exp_corr = kmnp.fuse_band_blocks(src, tuple(src_ra.transform), 0, ref, tuple(ref_ra.transform), NAN,
                                                    'gain-offset', (15, 15), 'ref', True, 0.25)
    from conftest import check_params
    check_params(params, exp_params, float(src[src != 0].mean()), 'host entry params')
    check_corr(corr, exp_corr.astype('float32'), 'host entry corr')


def test_error_reporting():
    lib = _native.lib()
    a = torch.zeros((8, 8), device='cuda')
    rc = lib.hb_fit_same_grid(a.data_ptr(), 0, 0.0, a.data_ptr(), 0, 0.0, 8, 8, 0, 4, 4, 0, None, a.data_ptr(), None,
                              _stream())
    assert rc != 0 and b'odd' in lib.hb_last_error()
    with pytest.raises(_native.NativeLibraryError):
        _native.check(rc, 'hb_fit_same_grid')
    before = lib.hb_launch_count()
    m = torch.empty(64, dtype=torch.uint8, device='cuda')
    _native.check(lib.hb_valid_mask(a.data_ptr(), _native.HB_F32, 64, 1, 0.0, m.data_ptr(), _stream()))
    assert lib.hb_launch_count() == before + 1 and int(m.sum()) == 0


# ---- size-independent properties at the full sizes of BASELINE.json ----------------------------------------------------
def test_full_size_refspace_properties():
    """
    10 000 x 10 000 uint16 band against a 10 m reference (BASELINE.json configs[1]): with ref = 2 * avg(src) the
    gain model must return gain == 2 exactly on every valid proc pixel, the corrected band 2 * src where the spline
    sees constant parameters, and NaN exactly on the source nodata.
    """
    from homonim_b200 import CRS, Model, RasterArray, RefSpaceModel
    hp = wp = 500
    ratio = 20
    g = torch.Generator(device='cuda').manual_seed(1)
    src = torch.randint(1, 5000, (hp * ratio, wp * ratio), generator=g, device='cuda', dtype=torch.int32)
    src[:777, :1234] = 0
    src = src.to(torch.uint16)
    crs = CRS.from_epsg(32735)
    src_tf = Affine(0.5, 0, 0, 0, -0.5, 0)
    ref_tf = Affine(10, 0, 0, 0, -10, 0)
    src_ra = RasterArray(src, crs, src_tf, nodata=0)
    avg = hkm._downsample_average(src, src_tf, 0, (hp, wp), ref_tf)
    blocks = src.view(hp, ratio, wp, ratio).to(torch.float64)
    cnt = (blocks != 0).sum(dim=(1, 3))
    mean = blocks.sum(dim=(1, 3)) / cnt
    assert torch.equal(torch.isnan(avg), cnt == 0)
    assert torch.equal(avg[cnt > 0], mean[cnt > 0].to(torch.float32))            # exact integer sums
    ref_ra = RasterArray((2 * avg).nan_to_num(1.0), crs, ref_tf, nodata=NAN)
    km = RefSpaceModel(Model.gain, (1, 1))
    param_ra = km.fit(src_ra, ref_ra)
    gain = param_ra.array[0]
    assert torch.equal(torch.isnan(gain), cnt == 0)
    assert bool((gain[cnt > 0] == 2).all()) and bool((param_ra.array[1][cnt > 0] == 0).all())
    corr = km.apply(src_ra, param_ra).array
    assert torch.equal(torch.isnan(corr), src == 0)
    # away from the nodata block and from the raster edge every spline tap is present and equal: 2 * src up to the
    # float32 rounding of the spline weights (their sum is 1 to a few 1e-7; GDAL's double sum is then rounded to
    # float32 as well) -- two orders of magnitude inside the 1e-4 contract.  (Within 2 coarse pixels of an edge GDAL
    # drops the out-of-range taps and, when their weight is < 1e-5, does not renormalise: 2 * src * (1 - O(1e-6)).)
    interior = torch.zeros_like(src, dtype=torch.bool)
    interior[900:-60, 1400:-60] = src[900:-60, 1400:-60] != 0
    expect = 2 * src.to(torch.int32)[interior].to(torch.float32)
    assert float(((corr[interior] - expect).abs() / expect).max()) <= 1e-6


def test_full_size_same_grid_properties():
    """
    8 192 x 8 192 float32 planes on one grid (the C3 / C5b regime): with ref = 0.5 * src + 0.125 (exact in float32) the
    gain-offset fit is exact up to float32 cancellation, R2 ~ 1, and a shifted band decomposition gives the same
    parameters (row-band / column-strip independence of the kernel).
    """
    from homonim_b200 import CRS, KernelModel, Model, RasterArray
    n = 8192
    g = torch.Generator(device='cuda').manual_seed(2)
    src = (torch.rand((n, n), generator=g, device='cuda') * 0.5 + 0.25)
    src = (src * 1024).round() / 1024
    ref = 0.5 * src + 0.125
    src[4000:4100, 100:300] = NAN
    crs, tf = CRS.from_epsg(32735), Affine(1, 0, 0, 0, -1, 0)
    km = KernelModel(Model.gain_offset, (15, 15), find_r2=True, r2_inpaint_thresh=None)
    p = km.fit(RasterArray(src, crs, tf), RasterArray(ref, crs, tf)).array
    valid = ~torch.isnan(src)
    assert torch.equal(torch.isnan(p[0]), ~valid)
    assert float((p[0][valid] - 0.5).abs().max()) < 2e-3
    assert float((p[2][valid] - 1).abs().max()) < 1e-2
    # a crop with its own tiling must reproduce the full-raster parameters away from the crop border
    y0, x0, m = 3000, 2001, 2048
    pc = km.fit(RasterArray(src[y0:y0 + m, x0:x0 + m].contiguous(), crs, tf),
                RasterArray(ref[y0:y0 + m, x0:x0 + m].contiguous(), crs, tf)).array
    a, b = p[:, y0 + 8:y0 + m - 8, x0 + 8:x0 + m - 8], pc[:, 8:-8, 8:-8]
    same = (a == b) | (torch.isnan(a) & torch.isnan(b))
    assert float(same.float().mean()) > 0.999
    fin = torch.isfinite(a) & torch.isfinite(b)
    assert float(((a - b).abs()[fin] / a.abs()[fin].clamp_min(1e-3)).max()) <= RTOL


# ---- the polynomial fast path of the up-sampler (csrc/upsample.cu): destination >= ~3.4x finer, width % 4 == 0 ---------
_POLY_CASES = [
    # dtype, nodata, ratio, shift (source-grid pixels), extra destination pixels beyond the coarse raster, pattern
    ('uint16', 0, 20, (0, 0), 0, 'holes'),
    ('uint16', 0, 4, (0, 0), 0, 'holes'),
    ('uint8', 0, 7, (2.0, 3.0), 0, 'holes'),
    ('float32', NAN, 5, (1.3, 2.6), 0, 'holes'),           # mis-aligned grids
    ('float32', NAN, 3.5, (0.4, 0.9), 0, 'holes'),         # non-integer ratio, near the eligibility limit
    ('float32', -9999.0, 6.4, (0.0, 0.0), 0, 'band'),      # value nodata; one band invalid where the other is not
    ('uint16', 0, 8, (-12.0, -20.0), 24, 'holes'),         # destination larger than the coarse raster on every side
    ('uint16', 65535, 10, (0, 0), 0, 'single'),            # isolated invalid coarse pixels
    ('float32', NAN, 12, (0, 0), 0, 'spikes'),             # parameter spikes / infinities next to normal values
    ('uint8', None, 16, (0, 0), 0, 'none'),                # no nodata at all
    ('float32', NAN, 33, (5.0, 1.0), 0, 'checker'),        # every cell dirty
    # small ratios: the "y first" kernel (a lane spans up to 3 coarse cells)
    ('uint16', 0, 2, (0, 0), 0, 'holes'),
    ('float32', NAN, 2, (0.5, 0.5), 0, 'single'),
    ('uint8', 0, 3, (0, 0), 0, 'holes'),                   # Landsat 30 m vs Sentinel-2 10 m
    ('float32', NAN, 2.5, (0.3, 0.7), 4, 'band'),
    ('uint16', 0, 1.7, (0, 0), 0, 'holes'),
    ('float32', NAN, 8, (3.0, 2.0), 0, 'spikes'),
    ('uint16', 0, 5, (0, 0), 0, 'checker'),
]


@pytest.mark.parametrize('dtype, nodata, ratio, shift, extra, pattern', _POLY_CASES)
def test_upsample_apply_fast_path(dtype, nodata, ratio, shift, extra, pattern):
    """ hb_upsample_apply on geometries that take the packed-float32 polynomial kernel + classification pre-pass +
    double-precision fix-up, against RefSpaceModel.apply of the oracle: masks exact, values within 1e-4. """
    _, kmnp = _oracle()
    rng = np.random.default_rng(11)
    hp, wp = 31, 27
    hs = int(hp * ratio) + 2 * extra
    ws = (int(wp * ratio) + 2 * extra) // 4 * 4               # the fast path needs a width that is a multiple of 4
    src = _rand_src(rng, hs, ws, dtype, nodata if nodata is not None else 0, holes=nodata is not None)
    yy, xx = np.mgrid[0:hp, 0:wp]
    params = np.stack([0.7 + 0.1 * np.sin(xx / 5.0) + 0.05 * rng.normal(size=(hp, wp)),
                       20.0 + 30.0 * np.cos(yy / 7.0) + 5.0 * rng.normal(size=(hp, wp))]).astype('float32')
    if pattern == 'holes':
        params[:, 8:12, 10:15] = NAN
        params[:, :2, :] = NAN
        params[:, 20, 3] = NAN
    elif pattern == 'band':
        params[0, 5:9, 5:9] = NAN
        params[1, 7:12, 8:13] = NAN
    elif pattern == 'single':
        params[:, rng.integers(0, hp, 12), rng.integers(0, wp, 12)] = NAN
    elif pattern == 'spikes':
        params[0, 10, 10] = 4000.0
        params[0, 15, 4] = -3.0
        params[0, 22, 20] = np.inf
        params[1, 22, 20] = -np.inf
        params[0, 3, 18] = 0.0
    elif pattern == 'checker':
        params[:, (yy + xx) % 3 == 0] = NAN
    src_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(shift[0] - extra, shift[1] - extra)
    pad = int(2 * ratio) + 4
    fill = nodata if nodata is not None else 0
    src_pad = np.full((hs + 2 * pad, ws + 2 * pad), fill, dtype=src.dtype)
    src_pad[pad:pad + hs, pad:pad + ws] = src
    pad_tf = src_tf * Affine.translation(-pad, -pad)
    with np.errstate(all='ignore'):
        expected = kmnp.refspace_apply(src_pad, tuple(pad_tf), nodata, params, tuple(TF_LO), (3, 5))[pad:pad + hs,
                                                                                                       pad:pad + ws]
    from homonim_b200 import CRS, Model, RasterArray, RefSpaceModel
    crs = CRS.from_epsg(3857)
    km = RefSpaceModel(Model.gain_blk_offset, (3, 5))
    lib = _native.lib()
    lib.hb_reset_launch_count()
    got = km.apply(RasterArray(torch.from_numpy(src).cuda(), crs, src_tf, nodata=nodata),
                   RasterArray(torch.from_numpy(params).cuda(), crs, TF_LO, nodata=NAN)).array.cpu().numpy()
    assert lib.hb_launch_count() == 3, 'expected the pre-pass + polynomial + fix-up kernels'
    expected = expected.astype('float32')
    assert_same_mask(got, expected, 'fast up-sample + apply')
    # infinities must agree exactly; finite values within the 1e-4 contract relative to the magnitude of the terms of
    # gain*src + offset (next to a spike the sum cancels: a purely relative test on the result is ill-posed)
    inf = np.isinf(expected)
    assert np.array_equal(got[inf], expected[inf])
    fin = np.isfinite(expected)
    scale = np.maximum(np.abs(expected[fin]), 1e-3 * np.mean(np.abs(expected[fin])))
    assert np.max(np.abs(got[fin].astype('float64') - expected[fin]) / scale) <= RTOL


@pytest.mark.parametrize('nb', [1, 2])
@pytest.mark.parametrize('ratio, shift', [(2, (0, 0)), (3, (0.5, 0.25)), (2.5, (1.0, 0.0)), (6, (0, 0)), (24, (2.0, 5.0))])
def test_resample_up_fast_paths(nb, ratio, shift):
    """ Plain cubic-spline up-sampling (SrcSpaceModel's reference up-sampling) on widths that take the fast kernel: it
    feeds a fit whose float32 arithmetic amplifies last-bit differences, so it has to round like GDAL (double). """
    gr, _ = _oracle()
    rng = np.random.default_rng(5)
    hp, wp = 38, 36
    coarse = rng.normal(1.0, 0.2, (nb, hp, wp)).astype('float32')
    coarse[:, 10:13, 5:9] = NAN
    coarse[0, 30, 20] = NAN
    coarse[:, :, -1] = NAN
    hd, wd = int(hp * ratio) + 3, (int(wp * ratio) + 2) // 4 * 4
    dst_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
    arr = coarse if nb == 2 else coarse[0]
    expected = gr.reproject_array(arr, tuple(TF_LO), NAN, (hd, wd), tuple(dst_tf), NAN, 'cubic_spline')
    lib = _native.lib()
    lib.hb_reset_launch_count()
    got = hkm._resample_up(torch.from_numpy(arr).cuda(), TF_LO, NAN, (hd, wd), dst_tf).cpu().numpy()
    # one band: ONE double-precision "y first" kernel (invalid taps handled inline); two bands: the general kernel
    assert lib.hb_launch_count() == 1
    assert_same_mask(got, expected, 'cubic_spline')
    assert rel_err(got, expected, 1e-3) <= 1e-6


@pytest.mark.parametrize('dtype, nodata', [('uint8', 0), ('uint16', 0), ('uint16', 65535), ('int16', -32768),
                                           ('uint16', None), ('float32', -9999.0)])
def test_convert_dtype(dtype, nodata):
    """ hb_convert_dtype against RasterArray._convert_array_dtype (raster_array.py:353-387) restated with numpy: round
    half to even in float32, clip to the integer range, cast, nodata where the corrected pixel is NaN. """
    rng = np.random.default_rng(8)
    n = 100003
    corr = (rng.normal(300.0, 400.0, n)).astype('float32')
    corr[::7] = np.round(corr[::7]) + 0.5                           # exact ties
    corr[5:50] = [-1e9, 1e9, 65535.4, 65535.5, 65536.0, -0.5, 0.5, 1.5, 2.5, 254.5, 255.5, 32767.5, -32768.5] + [0.0] * 32
    corr[rng.integers(0, n, 5000)] = NAN
    mask = ~np.isnan(corr)
    exp = corr.copy()
    if dtype != 'float32':
        info = np.iinfo(dtype)
        with np.errstate(invalid='ignore'):
            exp = np.clip(np.round(exp), info.min, info.max)
            exp = np.where(mask, exp, 0).astype(dtype)
    if nodata is not None:
        exp[~mask] = nodata
    lib = _native.lib()
    src = torch.from_numpy(corr).cuda()
    out = torch.empty(n, dtype=getattr(torch, dtype), device='cuda')
    code = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'int16': _native.HB_I16, 'float32': _native.HB_F32}[dtype]
    _native.check(lib.hb_convert_dtype(src.data_ptr(), n, code, int(nodata is not None),
                                       float(nodata) if nodata is not None else 0.0, out.data_ptr(), _stream()))
    got = out.cpu().numpy()
    if dtype == 'float32':
        assert np.array_equal(got, exp)
    else:
        assert np.array_equal(got.astype('int64'), exp.astype('int64'))


def test_process_out_profile_dtype():
    """ RasterFuse.process(out_profile=dict(dtype='uint16', nodata=0)): the corrected image converted on the device. """
    from homonim_b200 import Model, RasterFuse
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(40, 36, 8, bands=2, dtype='uint16', mu=3000.0, seed=3, device='cuda', src_nodata=0)
    with RasterFuse(src_ra, ref_ra) as fuse:
        f32, _ = fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5))
        u16, _ = fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5), out_profile=dict(dtype='uint16', nodata=0))
    assert u16.array.dtype == torch.uint16 and u16.nodata == 0
    a = f32.array.cpu().numpy()
    exp = np.where(np.isnan(a), 0, np.clip(np.round(np.nan_to_num(a)), 0, 65535)).astype('uint16')
    assert np.array_equal(u16.array.cpu().numpy().view('uint16'), exp)


@pytest.mark.parametrize('dtype, nodata', [('uint8', 0), ('uint16', 0), ('uint16', 65535), ('int16', -32768),
                                           ('float32', -9999.0)])
@pytest.mark.parametrize('proc_crs, ratio, shape', [('ref', 20, (37, 41)), ('ref', 2, (150, 130)), ('ref', 7, (64, 53)),
                                                    ('src', 2, (150, 130))])
def test_fused_output_dtype_equals_reference_conversion(dtype, nodata, proc_crs, ratio, shape):
    """ The output dtype conversion fused into the apply kernels' stores (every up-sampling kernel variant: polynomial,
    'y first', fix-up, general; the same-grid fit + apply kernel) equals the reference's own `_convert_array_dtype`
    (raster_array.py:353-387; oracle restatement pinned to tests/golden/convert_dtype.npz) of the float32 result, and the
    host-staged path (device -> host copy of the narrow plane) gives the same. """
    from homonim_b200 import Model, ProcCrs, RasterFuse
    from homonim_b200.synthetic import make_pair
    _, kmnp = _oracle()
    mu = 120.0 if dtype == 'uint8' else 3000.0
    src_ra, ref_ra = make_pair(shape[0], shape[1], ratio, bands=2, dtype='float32' if proc_crs == 'src' else 'uint16',
                               mu=mu, seed=5, device='cuda', src_nodata=NAN if proc_crs == 'src' else 0)
    kw = dict(model=Model.gain_blk_offset, kernel_shape=(5, 5))
    with RasterFuse(src_ra, ref_ra, proc_crs=ProcCrs(proc_crs)) as fuse:
        f32, _ = fuse.process(**kw)
        out, _ = fuse.process(out_profile=dict(dtype=dtype, nodata=nodata), **kw)
    assert str(out.array.dtype).replace('torch.', '') == dtype
    a = f32.array.cpu().numpy()
    exp = kmnp.convert_dtype(a, dtype, nodata)
    got = out.array.cpu().numpy()
    if dtype == 'uint16':
        got = got.view('uint16')
    assert np.array_equal(got, exp, equal_nan=True), f'{int((got != exp).sum())} pixels differ'
    # host rasters: the narrow plane is what crosses PCIe
    with RasterFuse(src_ra.to_host(), ref_ra.to_host(), proc_crs=ProcCrs(proc_crs)) as fuse:
        out_h, _ = fuse.process(out_profile=dict(dtype=dtype, nodata=nodata), **kw)
    got_h = np.asarray(out_h.array)
    assert np.array_equal(got_h.view(exp.dtype) if got_h.dtype != exp.dtype else got_h, exp, equal_nan=True)


def test_bench_contract_on_gpu(tmp_path):
    """ `python bench.py` prints ONE JSON line with the driver's contract (value, e2e, roofline, cpu_baseline, clocks,
    gpu_launches ...); run on the tiny workload.  `--dump-outputs` writes the corrected image of the last timed step. """
    import json
    import pathlib
    import subprocess
    import sys
    repo = pathlib.Path(__file__).resolve().parent.parent
    out = subprocess.run([sys.executable, str(repo / 'bench.py'), '--workload', 'tiny', '--steps', '3', '--warmup', '3',
                          '--dump-outputs', str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=str(repo))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline',
                'parity', 'row_band'):
        assert key in line, key
    assert line['value'] > 0 and line['gpu_launches'] > 0 and line['n_gpus'] == 1 and line['steps'] == 3
    assert line['e2e']['value'] > 0 and line['e2e']['h2d_bytes_per_step'] > 0 and line['e2e']['d2h_bytes_per_step'] > 0
    roof = line['roofline']
    for key in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert key in roof, key
    assert roof['bound'] == 'hbm' and roof['achieved'] > 0
    assert line['cpu_baseline']['kind'] in ('reference', 'port') and line['cpu_baseline']['value'] > 0
    # the GPU result of the sampled band against the reference's own result on the same inputs
    par = line['parity']
    assert par['masks_identical'] and par['within_tolerance'], par
    assert par['max_rel_err_corr'] <= 1e-4 and par['max_rel_err_gain'] <= 1e-4 and par['max_rel_err_offset'] <= 1e-4
    # the one-raster (row band) regime measured in the same invocation
    rb = line['row_band']
    assert rb['value'] > 0 and rb['scaling'] == 'strong' and rb['gpu_launches'] > 0
    assert 'workload' in line['config'] and 'model' not in line['config']
    # tiny: 2 bands of 320 x 288 source pixels, small enough to be written whole; nodata as 0 plus a validity mask
    corr, valid = np.load(tmp_path / 'corr.npy'), np.load(tmp_path / 'corr_valid.npy')
    assert corr.dtype == valid.dtype == np.float32 and corr.shape == valid.shape == (2, 320, 288)
    assert np.isfinite(corr).all() and set(np.unique(valid)) <= {0.0, 1.0} and valid.mean() > 0.5
    assert np.all(corr[valid == 0] == 0)


def test_convert_dtype_vs_reference_golden():
    """ hb_convert_dtype against RasterArray._convert_array_dtype of the unmodified reference
    (tests/golden/convert_dtype.npz). """
    import pathlib
    lib = _native.lib()
    codes = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'int16': _native.HB_I16, 'float32': _native.HB_F32}
    with np.load(pathlib.Path(__file__).resolve().parent / 'golden' / 'convert_dtype.npz') as data:
        corr = torch.from_numpy(data['corr']).cuda().contiguous()
        for key in data.files:
            if key == 'corr':
                continue
            dtype, nodata = key.rsplit('_', 1)
            out = torch.empty(corr.shape, dtype=getattr(torch, dtype), device='cuda')
            _native.check(lib.hb_convert_dtype(corr.data_ptr(), corr.numel(), codes[dtype], 1, float(nodata),
                                               out.data_ptr(), _stream()))
            got = out.cpu().numpy()
            exp = data[key]
            if dtype == 'float32':
                assert np.array_equal(got, exp), key
            else:
                assert np.array_equal(got.astype('int64'), exp.astype('int64')), key


@pytest.mark.parametrize('n, offset, src_nodata, ref_nodata', [
    (1, 0, NAN, NAN),
    (1000003, 0, NAN, NAN),                 # vector path with a scalar tail
    (262144, 1, NAN, -9999.0),              # planes not 16-byte aligned -> scalar path; a value nodata
    (5000000, 0, None, NAN),                # every source pixel valid; more pixels than one trip of the grid
    (4097, 0, NAN, NAN),
])
def test_compare_sums(n, offset, src_nodata, ref_nodata):
    """ hb_compare_sums against get_block_sums (compare.py:243-253) restated with numpy: the same float32 terms summed
    in double (tolerance 1e-12: the two double summation orders); deterministic from call to call. """
    _, knp = _oracle()
    from homonim_b200.compare import SUM_KEYS, compare_sums_device
    rng = np.random.default_rng(n)
    ref = rng.normal(900.0, 300.0, n + offset).astype('float32')
    src = (0.7 * ref + 40 + rng.normal(0.0, 50.0, n + offset)).astype('float32')
    if src_nodata is not None:
        src[rng.integers(0, n + offset, n // 10)] = src_nodata
    ref[rng.integers(0, n + offset, n // 17)] = ref_nodata
    if n == 1:
        src[:], ref[:] = 3.0, 5.0
    exp = knp.compare_sums(src[offset:], src_nodata, ref[offset:], ref_nodata, dtype='float64')
    src_t, ref_t = torch.from_numpy(src).cuda()[offset:], torch.from_numpy(ref).cuda()[offset:]
    got = compare_sums_device(src_t, src_nodata, ref_t, ref_nodata).cpu().numpy()
    again = compare_sums_device(src_t, src_nodata, ref_t, ref_nodata).cpu().numpy()
    assert np.array_equal(got, again)
    for key, value in zip(SUM_KEYS, got):
        assert abs(value - float(exp[key])) <= 1e-12 * max(abs(float(exp[key])), 1.0), key
    assert got[-1] == int(exp['mask_sum'])


def test_compare_sums_all_invalid():
    """ An empty mask gives seven zeros (the statistics are then NaN, as in the reference). """
    from homonim_b200.compare import RasterCompare, compare_sums_device
    src = torch.full((37, 41), NAN, device='cuda')
    ref = torch.ones((37, 41), device='cuda')
    got = compare_sums_device(src, NAN, ref, NAN).cpu().numpy()
    assert np.array_equal(got, np.zeros(7))
    stats = RasterCompare._band_stats(*got)
    assert stats['n'] == 0 and np.isnan(stats['r2']) and np.isnan(stats['rmse'])


def test_concurrent_process_and_fit_from_host_threads():
    """ The reference runs its (band, block) jobs on a thread pool (fuse.py:396-408); here the equivalent is several
    host threads driving one RasterFuse / one model object at once.  Every thread must get exactly the result a single
    thread gets (shared state: the band-plan cache, the stream pool, the native side streams and one-time set-up). """
    import threading
    from homonim_b200 import Model, ProcCrs, RasterArray, RasterFuse, RefSpaceModel, SrcSpaceModel
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(128, 96, 12, bands=4, dtype='uint16', seed=5, device='cuda')
    jobs = [(Model.gain_blk_offset, (5, 5), None), (Model.gain_offset, (5, 5), 0.25), (Model.gain, (1, 1), None),
            (Model.gain_offset, (7, 5), None)]
    with RasterFuse(src_ra, ref_ra, proc_crs=ProcCrs.ref) as fuse:
        def run(job):
            model, kshape, thresh = job
            corr, params = fuse.process(model=model, kernel_shape=kshape, param_filename='p',
                                        model_config=dict(r2_inpaint_thresh=thresh))
            return corr.array.clone(), params.array.clone()
        expected = [run(job) for job in jobs]
        torch.cuda.synchronize()
        results, errors = {}, []

        def worker(i):
            try:
                for rep in range(3):
                    results[(i, rep)] = run(jobs[i % len(jobs)])
                torch.cuda.current_stream().synchronize()
            except Exception as ex:     # noqa
                errors.append(repr(ex))
        threads = [threading.Thread(target=worker, args=(i,)) for i in range(8)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        torch.cuda.synchronize()
        assert not errors, errors
        for (i, rep), (corr, params) in results.items():
            exp_c, exp_p = expected[i % len(jobs)]
            assert torch.equal(corr.view(torch.int32), exp_c.view(torch.int32)), (i, rep)
            assert torch.equal(params.view(torch.int32), exp_p.view(torch.int32)), (i, rep)
    # one model object, fit() + apply() from 8 threads, both processing spaces
    s1 = RasterArray(src_ra.array[0].float().contiguous(), src_ra.crs, src_ra.transform, nodata=0.0)
    r1 = RasterArray(ref_ra.array[0].float().contiguous(), ref_ra.crs, ref_ra.transform, nodata=ref_ra.nodata)
    for model in (RefSpaceModel(Model.gain_offset, (5, 5), find_r2=True),
                  SrcSpaceModel(Model.gain_blk_offset, (9, 9), find_r2=True)):
        exp_p = model.fit(s1, r1)
        exp_c = model.apply(s1, exp_p).array.clone()
        out, errors = {}, []

        def fit_worker(i):
            try:
                p_ra = model.fit(s1, r1)
                out[i] = (p_ra.array.clone(), model.apply(s1, p_ra).array.clone())
            except Exception as ex:     # noqa
                errors.append(repr(ex))
        threads = [threading.Thread(target=fit_worker, args=(i,)) for i in range(8)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        torch.cuda.synchronize()
        assert not errors, errors
        for i, (p_t, c_t) in out.items():
            assert torch.equal(p_t.view(torch.int32), exp_p.array.view(torch.int32)), (type(model).__name__, i)
            assert torch.equal(c_t.view(torch.int32), exp_c.view(torch.int32)), (type(model).__name__, i)
