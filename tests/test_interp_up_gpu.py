"""
GPU tier: the bilinear, cubic and lanczos up-sampling methods of the general up-sampling kernel (csrc/upsample.cu)
against the oracle's restatement (oracle/interp_up_restate.c): plain up-sampling, the fused up-sample + apply of
RefSpaceModel.apply, SrcSpaceModel, RasterFuse, RasterCompare and lanczos row bands.
"""
import os
import socket

import numpy as np
import pytest

from conftest import RTOL, assert_same_mask, check_corr, rel_err

torch = pytest.importorskip('torch')
import torch.distributed as dist   # noqa: E402
import torch.multiprocessing as mp   # noqa: E402

from homonim_b200 import Affine, CRS, Model, RasterArray, RefSpaceModel, SrcSpaceModel, _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402

pytestmark = pytest.mark.gpu

NAN = float('nan')
TF_LO = Affine(10, 0, 2000, 0, -10, 9000)
CRS_ = CRS.from_epsg(3857)
METHODS = ('bilinear', 'cubic', 'lanczos')
CODES = {'bilinear': _native.HB_UP_BILINEAR, 'cubic': _native.HB_UP_CUBIC, 'lanczos': _native.HB_UP_LANCZOS}


def _oracle():
    from oracle import interp_up_restate, kernel_model_np
    return interp_up_restate, kernel_model_np


@pytest.fixture(autouse=True)
def _oracle_with_interp_up():
    """ the oracle's kernel-model port, with its re-projection extended to bilinear / cubic / lanczos up-sampling """
    from oracle.interp_up_restate import with_interp_up
    with with_interp_up():
        yield


def _params(rng, hp, wp):
    p = np.stack([rng.normal(0.7, 0.1, (hp, wp)), rng.normal(20.0, 50.0, (hp, wp))]).astype('float32')
    p[:, 8:11, 10:14] = NAN                          # holes in both bands
    p[1, 3, 4:7] = NAN                               # offset-only holes
    p[0, 15, 20] = NAN                               # gain-only hole
    p[:, :2, :] = NAN
    return p


def _rand_src(rng, h, w, dtype, nodata):
    if dtype == 'float32':
        s = rng.normal(300.0, 80.0, (h, w)).astype('float32')
    else:
        hi = 255 if dtype == 'uint8' else 4000
        s = rng.integers(1, hi, (h, w)).astype(dtype)
    holes = rng.random((h, w)) < 0.02
    s[holes] = nodata
    return s


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('nb', [1, 2])
@pytest.mark.parametrize('ratio, shift', [(20, (0, 0)), (4, (0, 0)), (3, (0.4, -0.3)), (1.6, (0, 0)), (1.1, (0.2, 0.1))])
def test_resample_up_vs_oracle(method, nb, ratio, shift):
    gr, _ = _oracle()
    rng = np.random.default_rng(11)
    hp, wp = 30, 41
    par = _params(rng, hp, wp)[:nb]
    hd, wd = int(hp * ratio) - 1, int(wp * ratio) - 2
    dst_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
    expected = gr.reproject_array(par, tuple(TF_LO), NAN, (hd, wd), tuple(dst_tf), NAN, method)
    got = hkm._resample_up(torch.from_numpy(par).cuda(), TF_LO, NAN, (hd, wd), dst_tf, CODES[method]).cpu().numpy()
    for b in range(nb):
        assert_same_mask(got[b], expected[b], f'{method} band {b}')
        assert rel_err(got[b], expected[b], 1e-3) <= 1e-6


def _apply_case(method, dtype, nodata, ratio, shift, partial, hp=36, wp=30, seed=4):
    _, kmnp = _oracle()
    rng = np.random.default_rng(seed)
    hs, ws = int(hp * ratio) - 2, int(wp * ratio) - 3
    src = _rand_src(rng, hs, ws, dtype, nodata)
    params = _params(rng, hp, wp)
    src_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
    pad = int(np.ceil(3 * ratio))
    src_pad = np.full((hs + 2 * pad, ws + 2 * pad), nodata, dtype=src.dtype)
    src_pad[pad:pad + hs, pad:pad + ws] = src
    pad_tf = src_tf * Affine.translation(-pad, -pad)
    expected = kmnp.refspace_apply(src_pad, tuple(pad_tf), nodata, params, tuple(TF_LO), (3, 5), mask_partial=partial,
                                   upsampling=method)[pad:pad + hs, pad:pad + ws]
    return src, src_tf, params, expected.astype('float32')


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('dtype, nodata, ratio, shift, partial', [
    ('uint16', 0, 20, (0, 0), False), ('uint8', 0, 4, (0, 0), True), ('float32', NAN, 5, (1.3, 2.6), False),
    ('float32', NAN, 2, (0, 0), True), ('uint16', 0, 3, (0.5, 0.25), True), ('uint16', 0, 1.25, (0.3, 0), False),
])
def test_upsample_apply_vs_oracle_and_two_step(method, dtype, nodata, ratio, shift, partial):
    src, src_tf, params, expected = _apply_case(method, dtype, nodata, ratio, shift, partial)
    km = RefSpaceModel(Model.gain_blk_offset, (3, 5), mask_partial=partial, upsampling=method)
    src_ra, par_ra = RasterArray(src, CRS_, src_tf, nodata=nodata), RasterArray(params, CRS_, TF_LO, nodata=NAN)
    got = km.apply(src_ra, par_ra).array
    check_corr(got, expected, f'upsample_apply {method}')
    assert_same_mask(got, expected, method)
    # the fused kernel == the two-step composition: up-sample both bands, then the same-grid apply
    if not partial:
        src_t = torch.from_numpy(src).cuda()
        par_us = hkm._resample_up(torch.from_numpy(params).cuda(), TF_LO, NAN, src.shape, src_tf, CODES[method])
        two = hkm.KernelModel._apply_planes(src_t, nodata, par_us, mask_src=True).cpu().numpy()
        assert np.array_equal(got.view('uint32'), two.view('uint32')) or np.array_equal(got, two, equal_nan=True)
    # uint16 output with a nodata value
    out = torch.empty(src.shape, dtype=torch.uint16, device='cuda')
    got16 = km.apply(RasterArray(torch.from_numpy(src).cuda(), CRS_, src_tf, nodata=nodata),
                     RasterArray(torch.from_numpy(params).cuda(), CRS_, TF_LO, nodata=NAN), out=out,
                     out_nodata=0).array.cpu().numpy()
    _, kmnp = _oracle()
    exp16 = kmnp.convert_dtype(expected, 'uint16', 0)
    close = np.abs(got16.astype('int64') - exp16.astype('int64')) <= 1
    assert close.all() and (got16 == exp16).mean() > 0.999


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('ratio', [10.0, 1.07])
def test_upsample_apply_large(method, ratio):
    """ >= 4000^2 at ratio 10, and ratio ~1 more than two CTAs wide (the widest-ncols instantiation) """
    hp, wp = (400, 410) if ratio > 2 else (300, 2200)
    src, src_tf, params, expected = _apply_case(method, 'uint16', 0, ratio, (0, 0), False, hp=hp, wp=wp, seed=9)
    km = RefSpaceModel(Model.gain_blk_offset, (3, 5), upsampling=method)
    got = km.apply(RasterArray(src, CRS_, src_tf, nodata=0), RasterArray(params, CRS_, TF_LO, nodata=NAN)).array
    check_corr(got, expected, f'large {method} {ratio}')


def _fuse_band_oracle(kmnp, src, src_tf, src_nd, ref, ref_tf, ref_nd, model, kshape, proc_crs, method):
    """ kernel_model_np.fuse_band_blocks with the `upsampling` choice passed through """
    src_blk, src_blk_tf, ref_blk, ref_blk_tf, (r0, c0) = kmnp.block_windows(src, src_tf, src_nd, ref, ref_tf)
    hs, ws = np.shape(src)
    if proc_crs == 'src':
        params = kmnp.srcspace_fit(src_blk, src_blk_tf, src_nd, ref_blk, ref_blk_tf, ref_nd, model, kshape, False, None,
                                   False, upsampling=method)
        corr = kmnp.srcspace_apply(src_blk, params)
    else:
        params = kmnp.refspace_fit(src_blk, src_blk_tf, src_nd, ref_blk, ref_blk_tf, ref_nd, model, kshape, False, None,
                                   upsampling=method)
        corr = kmnp.refspace_apply(src_blk, src_blk_tf, src_nd, params, ref_blk_tf, kshape, False, upsampling=method)
    return np.ascontiguousarray(corr[r0:r0 + hs, c0:c0 + ws])


@pytest.mark.parametrize('method', METHODS)
@pytest.mark.parametrize('proc_crs', ['ref', 'src'])
def test_raster_fuse_vs_oracle(method, proc_crs):
    _, kmnp = _oracle()
    from homonim_b200 import ProcCrs, RasterFuse
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(48, 40, 6, bands=1, dtype='uint16', seed=17, device='cuda:0', src_nodata=0)
    with RasterFuse(src_ra, ref_ra, proc_crs=ProcCrs(proc_crs)) as fuse:
        corr_ra, _ = fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5),
                                  model_config=dict(upsampling=method, r2_inpaint_thresh=None))
    src, ref = src_ra.to_host(), ref_ra.to_host()
    exp = _fuse_band_oracle(kmnp, src.array[0], tuple(src.transform), src.nodata, ref.array[0], tuple(ref.transform),
                            ref.nodata, 'gain-blk-offset', (5, 5), proc_crs, method)
    check_corr(corr_ra.to_host().array[0], exp.astype('float32'), f'fuse {method} {proc_crs}')


@pytest.mark.parametrize('method', METHODS)
def test_srcspace_fit_vs_oracle(method):
    _, kmnp = _oracle()
    from homonim_b200.synthetic import make_pair
    from conftest import check_params
    src_ra, ref_ra = make_pair(40, 36, 4, bands=1, dtype='float32', mu=0.3, seed=5, src_nodata=NAN)
    src, ref = src_ra.array[0], ref_ra.array[0]
    km = SrcSpaceModel(Model.gain_offset, (5, 5), r2_inpaint_thresh=None, upsampling=method)
    got = km.fit(RasterArray(src, CRS_, src_ra.transform, nodata=src_ra.nodata),
                 RasterArray(ref, CRS_, ref_ra.transform, nodata=ref_ra.nodata)).array
    exp = kmnp.srcspace_fit(src, tuple(src_ra.transform), src_ra.nodata, ref, tuple(ref_ra.transform), ref_ra.nodata,
                            'gain-offset', (5, 5), r2_inpaint_thresh=None, upsampling=method)
    check_params(got, exp, float(np.nanmean(src)), f'srcspace {method}')


def test_compare_lanczos_vs_oracle():
    _, kmnp = _oracle()
    from homonim_b200 import ProcCrs, RasterCompare
    from homonim_b200.compare import SUM_KEYS
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(48, 40, 5, bands=1, dtype='uint16', seed=8, src_nodata=0)
    with RasterCompare(src_ra, ref_ra, proc_crs=ProcCrs.src) as cmp:
        got = cmp._band_sums_device(0, upsampling='lanczos').cpu().numpy()
        stats = cmp.process(upsampling='lanczos')
    exp = kmnp.compare_band(src_ra.array[0], tuple(src_ra.transform), src_ra.nodata, ref_ra.array[0],
                            tuple(ref_ra.transform), ref_ra.nodata, proc_crs='src', upsampling='lanczos')
    for key, value in zip(SUM_KEYS, got):
        assert abs(value - float(exp[key])) <= 1e-6 * max(abs(float(exp[key])), 1.0), key
    assert len(stats) >= 1


def test_fused_apply_rejects_nearest():
    src = torch.ones((8, 8), dtype=torch.float32, device='cuda')
    par = torch.ones((2, 2, 2), dtype=torch.float32, device='cuda')
    out = torch.empty_like(src)
    with pytest.raises(Exception, match='nearest'):
        hkm._call('hb_upsample_apply', src.data_ptr(), _native.HB_F32, 8, 8, 0, 0.0, par.data_ptr(), 2, 2, 0.25, 0.0,
                  0.25, 0.0, None, _native.HB_F32, 0, 0.0, out.data_ptr(), _native.HB_UP_NEAREST, hkm._stream())


@pytest.mark.parametrize('method', METHODS)
def test_downsampling_geometry_not_implemented(method):
    from homonim_b200.enums import Resampling
    t = torch.ones((16, 16), dtype=torch.float32, device='cuda')
    with pytest.raises(NotImplementedError, match='up-sampling'):
        hkm._resample_plane(t, TF_LO, NAN, (8, 8), TF_LO * Affine.scale(2.0), Resampling(method))


# ---- lanczos row bands ------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _rowband_worker(rank, world, port, result_dir, reach):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from homonim_b200 import dist as hdist
        from homonim_b200.dist import RowBands, fuse_refspace_sharded, source_band_for_proc_rows
        from homonim_b200.synthetic import make_pair
        if reach is not None:                             # (the row window of the 4-tap methods, for the control run)
            hdist.up_reach = lambda upsampling: reach
        src_ra, ref_ra = make_pair(90, 64, 20, bands=1, dtype='float32', mu=0.3, seed=21, device='cuda:0',
                                   src_nodata=NAN, ref_pad=0)
        src = RasterArray(src_ra.array[0].contiguous(), src_ra.crs, src_ra.transform, nodata=NAN)
        ref = RasterArray(ref_ra.array[0].contiguous(), ref_ra.crs, ref_ra.transform, nodata=NAN)
        model = RefSpaceModel(Model.gain_blk_offset, (15, 15), find_r2=True, upsampling='lanczos')
        full_corr = model.apply(src, model.fit(src, ref)).array
        bands = RowBands.split(ref.height, world)
        r0, r1 = source_band_for_proc_rows(src.shape, src.transform, ref.transform, bands.band(rank))
        src_local = RasterArray(src.array[r0:r1].contiguous(), src.crs, src.transform * Affine.translation(0, r0),
                                nodata=NAN)
        corr_local, _ = fuse_refspace_sharded(model, src_local, ref, bands)
        exp_c, got_c = full_corr[r0:r1], corr_local.array
        ok = torch.equal(torch.isnan(got_c), torch.isnan(exp_c))
        fin = torch.isfinite(exp_c)
        rel = ((got_c - exp_c).abs()[fin] / exp_c.abs()[fin].clamp_min(1e-3 * exp_c[fin].abs().mean())).max().item()
        open(os.path.join(result_dir, f'r{rank}'), 'w').write(f'{int(ok)} {rel}')
    finally:
        dist.destroy_process_group()


def _rowbands(tmp_path, reach):
    mp.spawn(_rowband_worker, args=(2, _free_port(), str(tmp_path), reach), nprocs=2, join=True)
    res = [open(tmp_path / f'r{r}').read().split() for r in range(2)]
    return all(int(m) for m, _ in res), max(float(e) for _, e in res)


def test_lanczos_row_bands_equal_unsharded(tmp_path):
    same_mask, rel = _rowbands(tmp_path, None)
    assert same_mask and rel <= 1e-4, rel


def test_lanczos_row_bands_need_three_rows(tmp_path):
    """ control: with the 4-tap methods' reach of 2 rows, the pixels next to the band seam differ """
    same_mask, rel = _rowbands(tmp_path, 2)
    assert not (same_mask and rel <= 1e-4), rel
