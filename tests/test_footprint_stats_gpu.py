"""
GPU tier: the footprint-statistics kernels (csrc/footprint_stats.cu: min, max, med, q1, q3, mode) against the C
restatement (oracle/footprint_stats_restate.c) bit for bit, and the public paths that reach them -- RefSpaceModel.fit,
RasterFuse, RasterCompare, SrcSpaceModel, reproject_raster and row bands -- against the oracle's kernel-model port.
"""
import os
import socket

import numpy as np
import pytest

from conftest import check_corr, check_params
from test_footprint_stats_cpu import CASES, GEOMS, _raster

torch = pytest.importorskip('torch')
import torch.distributed as dist   # noqa: E402
import torch.multiprocessing as mp   # noqa: E402

from homonim_b200 import Affine, CRS, Model, RasterArray, RefSpaceModel, SrcSpaceModel, _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402

pytestmark = pytest.mark.gpu

NAN = float('nan')
CRS_ = CRS.from_epsg(3857)
METHODS = ('min', 'max', 'med', 'q1', 'q3', 'mode')
CODES = {'min': _native.HB_STAT_MIN, 'max': _native.HB_STAT_MAX, 'med': _native.HB_STAT_MED, 'q1': _native.HB_STAT_Q1,
         'q3': _native.HB_STAT_Q3, 'mode': _native.HB_STAT_MODE}
DTYPE_CODES = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'float32': _native.HB_F32}


@pytest.fixture(autouse=True)
def _oracle_with_footprint_stats():
    """ the oracle's kernel-model port, with its re-projection extended to the footprint statistics """
    from oracle.footprint_stats_restate import with_footprint_stats
    with with_footprint_stats():
        yield


def _restated(src, nodata, dst_shape, sx, ox, sy, oy, method):
    from oracle import footprint_stats_restate as fsr
    return fsr.reproject_array(src, (1.0, 0.0, 0.0, 0.0, -1.0, 0.0), nodata, dst_shape, (sx, 0.0, ox, 0.0, -sy, -oy),
                               NAN, method)


def _kernel(src_t, nodata, dst_shape, sx, ox, sy, oy, method, dtype=None):
    """ hb_resample_stat on a device plane (``src_t`` may be a view with any element offset) """
    hs, ws = int(src_t.shape[0]), int(src_t.shape[1])
    dst = torch.empty(dst_shape, dtype=torch.float32, device='cuda')
    has, nd = (0, 0.0) if nodata is None else (1, float(nodata))
    code = DTYPE_CODES[dtype or str(src_t.dtype).replace('torch.', '')]
    hkm._call('hb_resample_stat', src_t.data_ptr(), code, hs, ws, has, nd, dst.data_ptr(), dst_shape[0], dst_shape[1],
              sx, ox, sy, oy, CODES[method], hkm._stream())
    return dst.cpu().numpy()


def _assert_bits(got, exp, what):
    assert got.shape == exp.shape, what
    same = got.view('uint32') == exp.view('uint32')
    assert same.all(), f'{what}: {int((~same).sum())} pixels differ, e.g. at {np.argwhere(~same)[:3].tolist()}'


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('case', range(len(CASES)))
@pytest.mark.parametrize('geom', range(len(GEOMS)))
def test_kernel_vs_restatement(method, case, geom):
    import math
    hs, ws, hd, wd, sx, ox, sy, oy = GEOMS[geom]
    dtype, nodata, nan_holes = CASES[case]
    rng = np.random.default_rng(1000 * geom + 10 * case + METHODS.index(method))
    patch = (math.ceil(sy + abs(oy)) + 1, math.ceil(sx + abs(ox)) + 1)
    src = _raster(rng, hs, ws, dtype, nodata, nan_holes, patch)
    exp = _restated(src, nodata, (hd, wd), sx, ox, sy, oy, method)
    got = _kernel(torch.from_numpy(src).cuda(), nodata, (hd, wd), sx, ox, sy, oy, method)
    _assert_bits(got, exp, f'{method} {dtype} geom {geom}')


def _big(rng, h, w, dtype, nodata):
    if dtype == 'float32':
        src = rng.normal(300.0, 80.0, (h, w)).astype('float32').round(1)       # (repeats, for mode)
    else:
        src = rng.integers(1, 255 if dtype == 'uint8' else 4000, (h, w)).astype(dtype)
    src[rng.random((h, w)) < 0.02] = nodata
    src[:50, :70] = nodata
    return src


@pytest.mark.parametrize('shape, dtype, nodata, ratio', [
    ((10000, 10000), 'uint16', 0, 20.0),          # the C2 band
    ((1800, 1920), 'uint16', 0, 60.0),
    ((1800, 1920), 'float32', NAN, 60.0),
    ((1425, 807), 'uint8', 0, 2.0),               # C1-sized
    ((400, 1001), 'uint16', 0, 7.3),              # a width that is not a multiple of the 16-byte load vector
    ((2100, 2000), 'float32', NAN, 19.6),
])
def test_large_shapes(shape, dtype, nodata, ratio):
    rng = np.random.default_rng(int(ratio * 10))
    src = _big(rng, *shape, dtype, nodata)
    src_t = torch.from_numpy(src).cuda()
    dst_shape = (int(shape[0] / ratio), int(shape[1] / ratio))
    for method in METHODS:
        exp = _restated(src, nodata, dst_shape, ratio, 0.0, ratio, 0.0, method)
        got = _kernel(src_t, nodata, dst_shape, ratio, 0.0, ratio, 0.0, method)
        _assert_bits(got, exp, f'{method} {shape} {dtype} ratio {ratio}')


@pytest.mark.parametrize('dtype', ['uint8', 'uint16', 'float32'])
@pytest.mark.parametrize('ratio, offset', [(128.0, 0.0), (127.3, 0.6)])
def test_largest_ratio(dtype, ratio, offset):
    """ 128 source pixels per destination pixel on each axis (non-integer: windows of up to 129 x 129) """
    rng = np.random.default_rng(3)
    src = _big(rng, 400, 530, dtype, 0 if dtype != 'float32' else NAN)
    nodata = 0 if dtype != 'float32' else NAN
    src_t = torch.from_numpy(src).cuda()
    for method in METHODS:
        exp = _restated(src, nodata, (3, 4), ratio, offset, ratio, offset, method)
        got = _kernel(src_t, nodata, (3, 4), ratio, offset, ratio, offset, method)
        _assert_bits(got, exp, f'{method} {dtype} ratio {ratio}')


@pytest.mark.parametrize('dtype', ['uint8', 'uint16', 'float32'])
@pytest.mark.parametrize('ratio', [2.0, 20.0])
def test_unaligned_source_pointer(dtype, ratio):
    """ a source plane that starts one element past a 16-byte boundary, with an odd width """
    rng = np.random.default_rng(5)
    hs, ws = 201, 163
    src = _big(rng, hs, ws, dtype, 0 if dtype != 'float32' else NAN)
    nodata = 0 if dtype != 'float32' else NAN
    flat = torch.zeros(hs * ws + 1, dtype=getattr(torch, dtype), device='cuda')
    flat[1:] = torch.from_numpy(src.ravel()).cuda()
    view = flat[1:].view(hs, ws)
    assert view.data_ptr() % 16 != 0
    dst_shape = (int(hs / ratio), int(ws / ratio))
    for method in METHODS:
        exp = _restated(src, nodata, dst_shape, ratio, 0.0, ratio, 0.0, method)
        got = _kernel(view, nodata, dst_shape, ratio, 0.0, ratio, 0.0, method)
        _assert_bits(got, exp, f'{method} {dtype}')


@pytest.mark.parametrize('sx, sy', [(129.0, 2.0), (2.0, 128.5)])
def test_ratio_over_limit_is_an_error(sx, sy):
    src_t = torch.ones((300, 300), dtype=torch.uint16, device='cuda')
    with pytest.raises(_native.NativeLibraryError, match='maximum of 128'):
        _kernel(src_t, None, (2, 2), sx, 0.0, sy, 0.0, 'med')


# ---- public paths against the oracle's kernel-model port ---------------------------------------------------------------
@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('dtype, nodata', [('uint16', 0), ('float32', NAN)])
def test_refspace_fit_vs_oracle(method, dtype, nodata):
    from oracle import kernel_model_np as kmnp
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(40, 36, 5, bands=1, dtype=dtype, mu=3000.0 if dtype == 'uint16' else 0.3, seed=6,
                               src_nodata=nodata)
    src, ref = src_ra.array[0], ref_ra.array[0]
    km = RefSpaceModel(Model.gain_offset, (5, 5), r2_inpaint_thresh=None, downsampling=method)
    got = km.fit(RasterArray(src, CRS_, src_ra.transform, nodata=nodata),
                 RasterArray(ref, CRS_, ref_ra.transform, nodata=ref_ra.nodata)).array
    exp = kmnp.refspace_fit(src, tuple(src_ra.transform), nodata, ref, tuple(ref_ra.transform), ref_ra.nodata,
                            'gain-offset', (5, 5), r2_inpaint_thresh=None, downsampling=method)
    check_params(got, exp, float(np.nanmean(src)), f'refspace fit {method}')


def _fuse_band_oracle(kmnp, src, src_tf, src_nd, ref, ref_tf, ref_nd, kshape, proc_crs, **resampling):
    """ kernel_model_np.fuse_band_blocks with the `downsampling` / `upsampling` choices passed through """
    src_blk, src_blk_tf, ref_blk, ref_blk_tf, (r0, c0) = kmnp.block_windows(src, src_tf, src_nd, ref, ref_tf)
    hs, ws = np.shape(src)
    model = 'gain-blk-offset'
    if proc_crs == 'src':
        params = kmnp.srcspace_fit(src_blk, src_blk_tf, src_nd, ref_blk, ref_blk_tf, ref_nd, model, kshape, False, None,
                                   False, **resampling)
        corr = kmnp.srcspace_apply(src_blk, params)
    else:
        params = kmnp.refspace_fit(src_blk, src_blk_tf, src_nd, ref_blk, ref_blk_tf, ref_nd, model, kshape, False, None,
                                   **resampling)
        corr = kmnp.refspace_apply(src_blk, src_blk_tf, src_nd, params, ref_blk_tf, kshape, False, **resampling)
    return np.ascontiguousarray(corr[r0:r0 + hs, c0:c0 + ws])


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('proc_crs', ['ref', 'src'])
def test_raster_fuse_vs_oracle(method, proc_crs):
    """ proc_crs=ref down-samples the source with `method`; proc_crs=src up-samples the reference with it.  (No
    `bad_blobs`: inside them the source does not follow the reference, the fitted offsets cancel gain * src, and corrected
    values near zero are differences of terms ~1e3 times larger, where the fused apply's single rounding, DESIGN §4.5,
    exceeds the relative tolerance whatever the down-sampling.) """
    from oracle import kernel_model_np as kmnp
    from homonim_b200 import ProcCrs, RasterFuse
    from homonim_b200.synthetic import make_pair
    key = 'downsampling' if proc_crs == 'ref' else 'upsampling'
    src_ra, ref_ra = make_pair(48, 40, 6, bands=1, dtype='uint16', seed=17, device='cuda:0', src_nodata=0, bad_blobs=0)
    with RasterFuse(src_ra, ref_ra, proc_crs=ProcCrs(proc_crs)) as fuse:
        corr_ra, _ = fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5),
                                  model_config={key: method, 'r2_inpaint_thresh': None})
    src, ref = src_ra.to_host(), ref_ra.to_host()
    exp = _fuse_band_oracle(kmnp, src.array[0], tuple(src.transform), src.nodata, ref.array[0], tuple(ref.transform),
                            ref.nodata, (5, 5), proc_crs, **{key: method})
    check_corr(corr_ra.to_host().array[0], exp.astype('float32'), f'fuse {method} {proc_crs}')


@pytest.mark.parametrize('method', METHODS)
def test_compare_vs_oracle(method):
    from oracle import kernel_model_np as kmnp
    from homonim_b200 import ProcCrs, RasterCompare
    from homonim_b200.compare import SUM_KEYS
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(48, 40, 5, bands=1, dtype='uint16', seed=8, src_nodata=0)
    with RasterCompare(src_ra, ref_ra, proc_crs=ProcCrs.ref) as cmp:
        got = cmp._band_sums_device(0, downsampling=method).cpu().numpy()
        stats = cmp.process(downsampling=method)
    exp = kmnp.compare_band(src_ra.array[0], tuple(src_ra.transform), src_ra.nodata, ref_ra.array[0],
                            tuple(ref_ra.transform), ref_ra.nodata, proc_crs='ref', downsampling=method)
    for key, value in zip(SUM_KEYS, got):
        assert abs(value - float(exp[key])) <= 1e-6 * max(abs(float(exp[key])), 1.0), key
    assert len(stats) >= 1


@pytest.mark.parametrize('method', METHODS)
def test_srcspace_fit_finer_reference_vs_oracle(method):
    """ SrcSpaceModel with a reference finer than the source: the reference is down-sampled with `method` """
    from oracle import kernel_model_np as kmnp
    from homonim_b200.synthetic import make_pair
    hi_ra, lo_ra = make_pair(40, 36, 4, bands=1, dtype='float32', mu=0.3, seed=5, src_nodata=NAN)
    src, src_tf = lo_ra.array[0], lo_ra.transform                   # the coarse image is the source here
    ref, ref_tf = hi_ra.array[0], hi_ra.transform
    km = SrcSpaceModel(Model.gain_offset, (5, 5), r2_inpaint_thresh=None, downsampling=method)
    got = km.fit(RasterArray(src, CRS_, src_tf, nodata=NAN), RasterArray(ref, CRS_, ref_tf, nodata=NAN)).array
    exp = kmnp.srcspace_fit(src, tuple(src_tf), NAN, ref, tuple(ref_tf), NAN, 'gain-offset', (5, 5),
                            r2_inpaint_thresh=None, downsampling=method)
    check_params(got, exp, float(np.nanmean(src)), f'srcspace {method}')


@pytest.mark.parametrize('dtype', ['uint16', 'float32'])
def test_reproject_raster_mode_upsampling(dtype):
    from oracle import gdal_restate
    from homonim_b200.kernel_model import reproject_raster
    rng = np.random.default_rng(12)
    src = rng.integers(1, 6, (30, 41)).astype(dtype)
    src[rng.random(src.shape) < 0.1] = 0
    src_tf = Affine(10, 0, 2000, 0, -10, 9000)
    dst_tf = src_tf * Affine.scale(0.4) * Affine.translation(0.3, -0.2)
    got = reproject_raster(RasterArray(src, CRS_, src_tf, nodata=0), transform=dst_tf, shape=(70, 100),
                           resampling='mode').array
    exp = gdal_restate.reproject_array(src, tuple(src_tf), 0, (70, 100), tuple(dst_tf), NAN, 'mode')
    _assert_bits(np.asarray(got, dtype='float32'), exp, f'reproject_raster mode {dtype}')


# ---- row bands ----------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _rowband_worker(rank, world, port, result_dir, method):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from homonim_b200.dist import (RowBands, fuse_refspace_sharded_begin, fuse_refspace_sharded_end,
                                       source_band_for_proc_rows)
        from homonim_b200.synthetic import make_pair
        src_ra, ref_ra = make_pair(90, 64, 20, bands=1, dtype='uint16', seed=21, device='cuda:0', src_nodata=0,
                                   ref_pad=0)
        src = RasterArray(src_ra.array[0].contiguous(), src_ra.crs, src_ra.transform, nodata=0)
        ref = RasterArray(ref_ra.array[0].contiguous(), ref_ra.crs, ref_ra.transform, nodata=NAN)
        model = RefSpaceModel(Model.gain_blk_offset, (15, 15), find_r2=True, downsampling=method)
        full_ds = hkm._resample_plane(src.array, src.transform, 0, ref.shape, ref.transform,
                                      hkm.Resampling.coerce(method))
        full_corr = model.apply(src, model.fit(src, ref)).array
        bands = RowBands.split(ref.height, world)
        a, b = bands.band(rank)
        r0, r1 = source_band_for_proc_rows(src.shape, src.transform, ref.transform, bands.band(rank))
        src_local = RasterArray(src.array[r0:r1].contiguous(), src.crs, src.transform * Affine.translation(0, r0),
                                nodata=0)
        shard = fuse_refspace_sharded_begin(model, src_local, ref, bands)
        ds_same = torch.equal(shard.src_ds_local.view(torch.int32), full_ds[a:b].contiguous().view(torch.int32))
        corr_local, _ = fuse_refspace_sharded_end(shard)
        exp_c, got_c = full_corr[r0:r1], corr_local.array
        ok = torch.equal(torch.isnan(got_c), torch.isnan(exp_c))
        fin = torch.isfinite(exp_c)
        rel = ((got_c - exp_c).abs()[fin] / exp_c.abs()[fin].clamp_min(1e-3 * exp_c[fin].abs().mean())).max().item()
        open(os.path.join(result_dir, f'r{rank}'), 'w').write(f'{int(ds_same)} {int(ok)} {rel}')
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('method', ['med', 'mode'])
def test_row_bands_equal_unsharded(tmp_path, method):
    mp.spawn(_rowband_worker, args=(2, _free_port(), str(tmp_path), method), nprocs=2, join=True)
    res = [open(tmp_path / f'r{r}').read().split() for r in range(2)]
    assert all(int(d) for d, _, _ in res), 'rank-local down-sampled rows differ from the unsharded plane'
    assert all(int(m) for _, m, _ in res), 'masks differ'
    assert max(float(e) for _, _, e in res) <= 1e-4
