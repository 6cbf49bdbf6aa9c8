"""
GPU tier: int16 source and reference planes, read in their stored dtype by every kernel that reads a stored plane.

1. Same as float32: each entry point gives the same bits for an int16 plane as for the same plane widened to float32
   (with the nodata value as a float).  Each case's geometry sends both dtypes to the same kernel by the launch rules
   of launch_downsample / launch_upsample (element sizes 2 and 4: alignment is judged per element), and the kernel is
   named in the case id.  The one exception is the exact-box down-sampler, which only integer planes have: there the
   float32 twin takes the general down-sampler, and both give the same bits because both divide the same exact
   integer sum by the same count in double.
2. Same as uint16: non-negative int16 data gives the bits of the same values stored as uint16 (same element size, so
   the same kernel).
3. The public paths against the oracle's kernel-model port, which gets the plane widened to float32 -- what the
   reference's reader hands its kernels.
4. Production size, GeoTIFF files and row bands.
"""
import os
import socket

import numpy as np
import pytest

from conftest import check_corr, check_params

torch = pytest.importorskip('torch')
import torch.distributed as dist   # noqa: E402
import torch.multiprocessing as mp   # noqa: E402

from homonim_b200 import Affine, CRS, KernelModel, Model, ProcCrs, RasterArray, RasterFuse, RefSpaceModel  # noqa: E402
from homonim_b200 import SrcSpaceModel, _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402

pytestmark = pytest.mark.gpu

NAN = float('nan')
CRS_ = CRS.from_epsg(3857)
DEV = 'cuda:0'
# -1 was the "no integer nodata" sentinel of the integer kernels; 40000 and NaN match no int16 pixel
NODATAS = [-9999, -32768, 32767, -1, 0, None, 40000, NAN]
STATS = {'min': _native.HB_STAT_MIN, 'max': _native.HB_STAT_MAX, 'med': _native.HB_STAT_MED, 'q1': _native.HB_STAT_Q1,
         'q3': _native.HB_STAT_Q3, 'mode': _native.HB_STAT_MODE}
UP = {'cubic_spline': _native.HB_UP_CUBIC_SPLINE, 'bilinear': _native.HB_UP_BILINEAR, 'cubic': _native.HB_UP_CUBIC,
      'lanczos': _native.HB_UP_LANCZOS}
OUT_NODATA = {torch.float32: NAN, torch.uint8: 0, torch.uint16: 0, torch.int16: -32768}


def _nd_id(nd):
    return 'none' if nd is None else ('nan' if nd != nd else str(nd))


def _int16_plane(rng, h, w, nodata, nonneg=False):
    """ values across [-32768, 32767] (or [0, 32767]), with runs of -1, the extremes, and nodata pixels when the nodata
    value is an int16 """
    lo = 0 if nonneg else -32768
    a = rng.integers(lo // 8, 32767 // 8, (h, w)).astype('int16')
    for v, frac in ((-1, 0.01), (-32768, 0.005), (32767, 0.005), (0, 0.01)):
        if v >= lo:
            a[rng.random((h, w)) < frac] = v
    if _in_int16(nodata) and nodata >= lo:
        a[rng.random((h, w)) < 0.04] = nodata
        a[5:9, 3:40] = nodata                                      # whole footprints of nodata
    return a


def _twin(a, nodata, twin):
    """ the same plane as float32 (nodata as a float) or uint16 """
    if twin == 'float32':
        return a.astype('float32'), (None if nodata is None else float(nodata))
    return a.astype('uint16'), nodata


def _dev(a, misalign=False):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if not misalign:
        return t.to(DEV)
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=DEV)   # base pointer one element past an allocation
    view = flat[1:].view(t.shape)
    view.copy_(t.to(DEV))
    return view


def _same_bits(got, exp, what):
    got, exp = got.detach().cpu().contiguous().numpy(), exp.detach().cpu().contiguous().numpy()
    assert got.dtype == exp.dtype and got.shape == exp.shape, what
    assert np.array_equal(got.view(f'u{got.itemsize}'), exp.view(f'u{exp.itemsize}')), \
        f'{what}: {int((got.view(f"u{got.itemsize}") != exp.view(f"u{exp.itemsize}")).sum())} pixels differ'


# ---- down-sampling: hb_downsample_average, hb_resample_stat ----------------------------------------------------------
# (id, source shape, source -> destination scale and offset, misaligned base pointer)
DS_GEOMS = [
    ('int_aligned-vs-average_r20', (400, 480), 20.0, 0.0, False),      # exact box (int16) / general (float32)
    ('average_aligned_r5_shift', (203, 400), 5.0, 0.37, False),        # ws % 8 == 0: vector loads for both dtypes
    ('average_scalar_r5_w397', (203, 397), 5.0, 0.37, False),          # ws % 4 != 0: scalar loads for both
    ('average_scalar_r5_misaligned', (203, 400), 5.0, 0.37, True),     # base pointer 2 / 4 bytes off: scalar loads
]


def _ds_dst(shape, s, o):
    hs, ws = shape
    return (int(np.floor((hs - o) / s)), int(np.floor((ws - o) / s)))


def _downsample(t, nodata, s, o, dst_shape):
    tf = Affine(1, 0, 0, 0, -1, 0)
    return hkm._downsample_average(t, tf, nodata, dst_shape, Affine(s, 0, o, 0, -s, -o))


def _stat(t, nodata, s, o, dst_shape, code):
    tf = Affine(1, 0, 0, 0, -1, 0)
    return hkm._resample_stat(t, tf, nodata, dst_shape, Affine(s, 0, o, 0, -s, -o), code)


@pytest.mark.parametrize('nodata', NODATAS, ids=_nd_id)
@pytest.mark.parametrize('gid, shape, s, o, misalign', DS_GEOMS, ids=[g[0] for g in DS_GEOMS])
def test_downsample_average_same_as_float32(gid, shape, s, o, misalign, nodata):
    rng = np.random.default_rng(1)
    a = _int16_plane(rng, *shape, nodata)
    f, fnd = _twin(a, nodata, 'float32')
    dst = _ds_dst(shape, s, o)
    got = _downsample(_dev(a, misalign), nodata, s, o, dst)
    exp = _downsample(_dev(f, misalign), fnd, s, o, dst)
    _same_bits(got, exp, gid)
    assert torch.isfinite(got).any()


@pytest.mark.parametrize('method', list(STATS))
@pytest.mark.parametrize('nodata', [-9999, -1, 40000, None], ids=_nd_id)
@pytest.mark.parametrize('gid, s, o', [('stat_thread_r5', 5.0, 0.37), ('stat_warp_r20', 20.0, 0.0)])
def test_resample_stat_same_as_float32(gid, s, o, nodata, method):
    rng = np.random.default_rng(2)
    a = _int16_plane(rng, 200, 240, nodata)
    a[20:60, 20:60] = rng.integers(-3, 3, (40, 40))                # many ties: the mode's tie-break
    f, fnd = _twin(a, nodata, 'float32')
    dst = _ds_dst(a.shape, s, o)
    _same_bits(_stat(_dev(a), nodata, s, o, dst, STATS[method]), _stat(_dev(f), fnd, s, o, dst, STATS[method]),
               f'{gid} {method}')


# ---- up-sampling + apply: hb_upsample_apply --------------------------------------------------------------------------
# (id, coarse grid, destination grid, destination -> coarse scale and offset); ws % 4 == 0 and 256-byte aligned
# allocations: every case is "aligned" for both element sizes, so the method and the ratio alone pick the kernel
UP_GEOMS = [
    ('poly_r20', (14, 16), (280, 320), 1 / 20, 0.0),
    ('yfirst_r2', (60, 70), (120, 140), 0.5, 0.0),
    ('general_r1.25_shift', (90, 100), (104, 120), 0.8, 0.13),
]


def _params(rng, hp, wp):
    p = np.stack([rng.normal(1.0, 0.1, (hp, wp)), rng.normal(0.0, 200.0, (hp, wp))]).astype('float32')
    p[:, 3:5, 4:7] = NAN
    p[1, 8, 2:4] = NAN
    return torch.from_numpy(p).to(DEV)


def _upsample_apply(t, nodata, par, s, o, method, out_dtype):
    hs, ws = int(t.shape[0]), int(t.shape[1])
    out = torch.empty((hs, ws), dtype=out_dtype, device=DEV)
    has, nd = hkm._nodata_args(nodata)
    hkm._call('hb_upsample_apply', t.data_ptr(), hkm._plane_code(t), hs, ws, has, nd, par.data_ptr(),
              int(par.shape[1]), int(par.shape[2]), s, o, s, o, None,
              *hkm._out_args(out, OUT_NODATA[out_dtype]), out.data_ptr(), UP[method], hkm._stream())
    return out


def _kernel_id(gid, method):
    """ the kernel launch_upsample picks: the fast paths are cubic spline only """
    return gid if method == 'cubic_spline' else f'general_{gid}'


UP_CASES = [(g, m) for g in UP_GEOMS for m in UP]


@pytest.mark.parametrize('nodata', NODATAS, ids=_nd_id)
@pytest.mark.parametrize('geom, method', UP_CASES, ids=[_kernel_id(g[0], m) + f'_{m}' for g, m in UP_CASES])
def test_upsample_apply_same_as_float32(geom, method, nodata):
    gid, (hp, wp), (hs, ws), s, o = geom
    rng = np.random.default_rng(3)
    a = _int16_plane(rng, hs, ws, nodata)
    f, fnd = _twin(a, nodata, 'float32')
    par = _params(rng, hp, wp)
    got = _upsample_apply(_dev(a), nodata, par, s, o, method, torch.float32)
    exp = _upsample_apply(_dev(f), fnd, par, s, o, method, torch.float32)
    _same_bits(got, exp, f'{gid} {method}')


@pytest.mark.parametrize('out_dtype', [torch.uint8, torch.uint16, torch.int16, torch.float32], ids=str)
@pytest.mark.parametrize('geom', UP_GEOMS, ids=[g[0] for g in UP_GEOMS])
def test_upsample_apply_output_dtypes_same_as_float32(geom, out_dtype):
    gid, (hp, wp), (hs, ws), s, o = geom
    rng = np.random.default_rng(4)
    a = (_int16_plane(rng, hs, ws, -9999) // 64).astype('int16')   # corrected values inside the uint8 range too
    f, fnd = _twin(a, -9999, 'float32')
    par = _params(rng, hp, wp)
    _same_bits(_upsample_apply(_dev(a), -9999, par, s, o, 'cubic_spline', out_dtype),
               _upsample_apply(_dev(f), fnd, par, s, o, 'cubic_spline', out_dtype), f'{gid} {out_dtype}')


@pytest.mark.parametrize('nodata', [-9999, -1, None], ids=_nd_id)
def test_mask_partial_general_kernel_same_as_float32(nodata):
    """ RefSpaceModel fit + apply with mask_partial: hb_valid_mask, the coverage mask and the general up-sampling kernel
    (ratio 1.25 with a shift) """
    rng = np.random.default_rng(5)
    a = _int16_plane(rng, 104, 120, nodata)
    f, fnd = _twin(a, nodata, 'float32')
    ref = torch.from_numpy(rng.normal(500.0, 100.0, (84, 98)).astype('float32')).to(DEV)
    src_tf, ref_tf = Affine(1, 0, 0, 0, -1, 0), Affine(1.25, 0, -0.4, 0, -1.25, 0.4)
    ref_ra = RasterArray(ref, CRS_, ref_tf, nodata=NAN)
    km = RefSpaceModel(Model.gain_blk_offset, (3, 3), mask_partial=True)
    outs = []
    for plane, nd in ((a, nodata), (f, fnd)):
        src_ra = RasterArray(_dev(plane), CRS_, src_tf, nodata=nd)
        outs.append(km.apply(src_ra, km.fit(src_ra, ref_ra)).array)
    _same_bits(outs[0], outs[1], 'mask_partial')
    mask = KernelModel._valid_mask_u8(_dev(a), nodata)
    _same_bits(mask, KernelModel._valid_mask_u8(_dev(f), fnd), 'hb_valid_mask')


# ---- same-grid apply, the one-call fuse and its host form -------------------------------------------------------------
@pytest.mark.parametrize('out_dtype', [torch.float32, torch.int16, torch.uint16], ids=str)
@pytest.mark.parametrize('nodata', NODATAS, ids=_nd_id)
def test_apply_same_grid_same_as_float32(nodata, out_dtype):
    rng = np.random.default_rng(6)
    a = _int16_plane(rng, 60, 77, nodata)
    f, fnd = _twin(a, nodata, 'float32')
    par = torch.from_numpy(np.stack([rng.normal(1.0, 0.1, a.shape), rng.normal(0.0, 9.0, a.shape)]).astype('float32'))
    par = par.to(DEV)
    outs = [KernelModel._apply_planes(_dev(p), nd, par, True, torch.empty(a.shape, dtype=out_dtype, device=DEV),
                                      OUT_NODATA[out_dtype]) for p, nd in ((a, nodata), (f, fnd))]
    _same_bits(outs[0], outs[1], 'apply_same_grid')


def _in_int16(nodata):
    return nodata is not None and nodata == nodata and -32768 <= nodata <= 32767 and nodata == int(nodata)


def _fuse_pair(nodata, seed=9):
    """ a make_pair int16 source (nodata pixels = `nodata` where an int16 can hold it, else -9999) and its reference """
    from homonim_b200.synthetic import make_pair
    src_ra, ref_ra = make_pair(30, 26, 8, bands=1, dtype='int16', seed=seed,
                               src_nodata=nodata if _in_int16(nodata) else -9999)
    return src_ra.array[0].numpy(), ref_ra.array[0].contiguous(), src_ra.transform, ref_ra.transform


@pytest.mark.parametrize('nodata', [-9999, -1, 0, None, 40000], ids=_nd_id)
@pytest.mark.parametrize('model', [Model.gain_blk_offset, Model.gain_offset], ids=lambda m: m.value)
def test_fuse_refspace_same_as_float32(model, nodata):
    a, ref, src_tf, ref_tf = _fuse_pair(nodata)
    f, fnd = _twin(a, nodata, 'float32')
    km = RefSpaceModel(model, (5, 5), r2_inpaint_thresh=None)
    ref_ra = RasterArray(ref.to(DEV), CRS_, ref_tf, nodata=NAN)
    outs = []
    for plane, nd in ((a, nodata), (f, fnd)):
        corr, params = km.fuse(RasterArray(_dev(plane), CRS_, src_tf, nodata=nd), ref_ra, want_params=True)
        outs.append((corr.array, params.array))
    _same_bits(outs[0][0], outs[1][0], 'hb_fuse_refspace corr')
    _same_bits(outs[0][1], outs[1][1], 'hb_fuse_refspace params')
    # hb_fuse_refspace_host: host buffers in and out (its copy is sized by the source's element size)
    lib = _native.lib()
    hosts = []
    for plane, nd in ((a, nodata), (f, fnd)):
        plane = np.ascontiguousarray(plane)
        refh = np.ascontiguousarray(ref.numpy())
        corr = np.empty(plane.shape, 'float32')
        params = np.empty((2,) + refh.shape, 'float32')
        gm = hkm.grid_map(src_tf, ref_tf)
        has, ndv = hkm._nodata_args(nd)
        _native.check(lib.hb_fuse_refspace_host(
            plane.ctypes.data, hkm._plane_code(torch.from_numpy(plane)), plane.shape[0], plane.shape[1], has, ndv,
            refh.ctypes.data, refh.shape[0], refh.shape[1], 1, NAN, gm.sx, gm.ox, gm.sy, gm.oy,
            hkm._MODEL_CODES[model], 5, 5, 0, 0, 0.0, _native.HB_F32, 0, 0.0, corr.ctypes.data, params.ctypes.data,
            None), 'hb_fuse_refspace_host')
        hosts.append(corr)
    _same_bits(torch.from_numpy(hosts[0]), torch.from_numpy(hosts[1]), 'hb_fuse_refspace_host')
    _same_bits(torch.from_numpy(hosts[0]), outs[0][0], 'host vs device')


# ---- 2. same as uint16 ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nodata', [0, 32767, 1234, None, 40000], ids=_nd_id)
def test_nonnegative_int16_same_as_uint16(nodata):
    rng = np.random.default_rng(10)
    for gid, shape, s, o, misalign in DS_GEOMS:
        a = _int16_plane(rng, *shape, nodata, nonneg=True)
        u, und = _twin(a, nodata, 'uint16')
        dst = _ds_dst(shape, s, o)
        _same_bits(_downsample(_dev(a, misalign), nodata, s, o, dst), _downsample(_dev(u, misalign), und, s, o, dst),
                   f'{gid} vs uint16')
        for method, code in STATS.items():
            _same_bits(_stat(_dev(a), nodata, s, o, dst, code), _stat(_dev(u), und, s, o, dst, code),
                       f'{gid} {method} vs uint16')
    for (gid, (hp, wp), (hs, ws), s, o), method in UP_CASES:
        a = _int16_plane(rng, hs, ws, nodata, nonneg=True)
        u, und = _twin(a, nodata, 'uint16')
        par = _params(rng, hp, wp)
        for out_dtype in (torch.float32, torch.int16):
            _same_bits(_upsample_apply(_dev(a), nodata, par, s, o, method, out_dtype),
                       _upsample_apply(_dev(u), und, par, s, o, method, out_dtype), f'{gid} {method} vs uint16')
    a = _int16_plane(rng, 60, 77, nodata, nonneg=True)
    u, und = _twin(a, nodata, 'uint16')
    _same_bits(KernelModel._valid_mask_u8(_dev(a), nodata), KernelModel._valid_mask_u8(_dev(u), und), 'valid mask')
    par = torch.from_numpy(np.stack([rng.normal(1.0, 0.1, a.shape), rng.normal(0.0, 9.0, a.shape)]).astype('float32'))
    _same_bits(KernelModel._apply_planes(_dev(a), nodata, par.to(DEV), True),
               KernelModel._apply_planes(_dev(u), und, par.to(DEV), True), 'apply_same_grid vs uint16')
    a, ref, src_tf, ref_tf = _fuse_pair(0, seed=11)
    holes = a == 0
    a = np.clip(a, 1, None).astype('int16')
    if _in_int16(nodata):
        a[holes] = nodata
    u, und = _twin(a, nodata, 'uint16')
    ref_ra = RasterArray(ref.to(DEV), CRS_, ref_tf, nodata=NAN)
    km = RefSpaceModel(Model.gain_blk_offset, (5, 5))
    outs = [km.fuse(RasterArray(_dev(p), CRS_, src_tf, nodata=nd), ref_ra)[0].array
            for p, nd in ((a, nodata), (u, und))]
    _same_bits(outs[0], outs[1], 'hb_fuse_refspace vs uint16')


# ---- 3. the public paths against the oracle ------------------------------------------------------------------------------
def _pair(seed=12, nodata=-9999, hp=40, wp=36, ratio=5, **kw):
    from homonim_b200.synthetic import make_pair
    return make_pair(hp, wp, ratio, bands=1, dtype='int16', seed=seed, src_nodata=nodata, **kw)


def test_refspace_fit_apply_int16_source_vs_oracle():
    from oracle import kernel_model_np as kmnp
    src_ra, ref_ra = _pair()
    src, ref = src_ra.array[0].numpy(), ref_ra.array[0].numpy()
    assert (src[src != -9999] < 0).any()
    km = RefSpaceModel(Model.gain_offset, (5, 5), r2_inpaint_thresh=None)
    s_ra = RasterArray(src, CRS_, src_ra.transform, nodata=-9999)
    param_ra = km.fit(s_ra, RasterArray(ref, CRS_, ref_ra.transform, nodata=NAN))
    corr = km.apply(s_ra, param_ra).array
    srcf = src.astype('float32')
    exp = kmnp.refspace_fit(srcf, tuple(src_ra.transform), -9999.0, ref, tuple(ref_ra.transform), NAN, 'gain-offset',
                            (5, 5), r2_inpaint_thresh=None)
    bad = check_params(param_ra.array, exp, float(np.mean(srcf[src != -9999])), 'refspace fit int16')
    exp_corr = kmnp.refspace_apply(srcf, tuple(src_ra.transform), -9999.0, exp, tuple(ref_ra.transform), (5, 5))
    check_corr(corr, exp_corr.astype('float32'), 'refspace apply int16')


@pytest.mark.parametrize('method', ['average', 'med'])
def test_srcspace_int16_reference_vs_oracle(method):
    """ SrcSpaceModel with a reference finer than the source: the int16 reference is down-sampled with `method` """
    from oracle import kernel_model_np as kmnp
    from oracle.footprint_stats_restate import with_footprint_stats
    hi_ra, lo_ra = _pair(seed=13, nodata=-9999, ratio=4)
    src, src_tf = lo_ra.array[0].numpy(), lo_ra.transform                  # the coarse image is the source here
    ref, ref_tf = hi_ra.array[0].numpy(), hi_ra.transform
    km = SrcSpaceModel(Model.gain_offset, (5, 5), r2_inpaint_thresh=None, downsampling=method)
    got = km.fit(RasterArray(src, CRS_, src_tf, nodata=NAN), RasterArray(ref, CRS_, ref_tf, nodata=-9999)).array
    with with_footprint_stats():
        exp = kmnp.srcspace_fit(src, tuple(src_tf), NAN, ref.astype('float32'), tuple(ref_tf), -9999.0, 'gain-offset',
                                (5, 5), r2_inpaint_thresh=None, downsampling=method)
    check_params(got, exp, float(np.nanmean(src)), f'srcspace int16 reference {method}')


@pytest.mark.parametrize('proc_crs', ['ref', 'src'])
def test_raster_fuse_int16_vs_oracle(proc_crs):
    from oracle import kernel_model_np as kmnp
    src_ra, ref_ra = _pair(seed=14, nodata=-9999, hp=48, wp=40, ratio=6, bad_blobs=0)
    with RasterFuse(src_ra, ref_ra, proc_crs=ProcCrs(proc_crs)) as fuse:
        corr_ra, _ = fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5),
                                  model_config={'r2_inpaint_thresh': None})
    src, ref = src_ra.to_host(), ref_ra.to_host()
    exp = kmnp.fuse_band_blocks(src.array[0].astype('float32'), tuple(src.transform), -9999.0, ref.array[0],
                                tuple(ref.transform), NAN, 'gain-blk-offset', (5, 5), proc_crs, False, None)[2]
    check_corr(corr_ra.to_host().array[0], np.asarray(exp, 'float32'), f'fuse int16 {proc_crs}')


def test_compare_int16_reference_vs_oracle():
    from oracle import kernel_model_np as kmnp
    from homonim_b200 import RasterCompare
    from homonim_b200.compare import SUM_KEYS
    hi_ra, lo_ra = _pair(seed=15, nodata=-9999, ratio=4)
    src_ra = RasterArray(lo_ra.array[0].numpy(), CRS_, lo_ra.transform, nodata=NAN)
    ref_ra = RasterArray(hi_ra.array[0].numpy(), CRS_, hi_ra.transform, nodata=-9999)
    with RasterCompare(src_ra, ref_ra, proc_crs=ProcCrs.src) as cmp:
        got = cmp._band_sums_device(0).cpu().numpy()
    exp = kmnp.compare_band(src_ra.array, tuple(src_ra.transform), NAN, ref_ra.array.astype('float32'),
                            tuple(ref_ra.transform), -9999.0, proc_crs='src')
    for key, value in zip(SUM_KEYS, got):
        assert abs(value - float(exp[key])) <= 1e-6 * max(abs(float(exp[key])), 1.0), key


# ---- 4. production size, files, row bands -------------------------------------------------------------------------------
def test_production_size_fuse_same_as_float32():
    """ one 10 000 x 10 000 int16 band at ratio 20 through RasterFuse (the one-call hb_fuse_refspace path) """
    src_ra, ref_ra = _pair(seed=16, nodata=-9999, hp=500, wp=500, ratio=20, device=DEV)
    src_f = RasterArray(src_ra.array.to(torch.float32), src_ra.crs, src_ra.transform, nodata=-9999.0)
    outs = []
    for s in (src_ra, src_f):
        with RasterFuse(s, ref_ra) as fuse:
            outs.append(fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5))[0].array)
    _same_bits(outs[0], outs[1], '10000^2 int16 vs float32')
    del outs


@pytest.mark.parametrize('out_dtype', ['float32', 'int16'])
def test_int16_files_through_raster_fuse(tmp_path, out_dtype):
    from homonim_b200.geotiff import GeoTiffReader, write_geotiff
    src_ra, ref_ra = _pair(seed=17, nodata=-9999, hp=48, wp=40, ratio=6)
    src = src_ra.array.numpy()
    geokeys = ((1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 32735), (), '')
    src_path = write_geotiff(tmp_path / 'src.tif', src, src_ra.transform, nodata=-9999, geokeys=geokeys,
                             compress='deflate', blocksize=64)
    ref_path = write_geotiff(tmp_path / 'ref.tif', ref_ra.array.numpy(), ref_ra.transform, nodata=NAN,
                             geokeys=geokeys, compress='deflate', blocksize=64)
    with GeoTiffReader(src_path) as im:
        assert im.dtype.name == 'int16' and np.array_equal(im.read(), src)
    out_nodata = NAN if out_dtype == 'float32' else -32768
    profile = dict(dtype=out_dtype, nodata=out_nodata)
    corr_path = tmp_path / 'corr.tif'
    with RasterFuse(src_path, ref_path) as fuse:
        fuse.process(corr_path, Model.gain_blk_offset, (5, 5), out_profile=profile, build_ovw=False)
    with RasterFuse(src_ra, RasterArray(ref_ra.array, ref_ra.crs, ref_ra.transform, nodata=NAN)) as fuse:
        exp = fuse.process(model=Model.gain_blk_offset, kernel_shape=(5, 5), out_profile=profile)[0].array
    exp = exp.cpu().numpy() if hasattr(exp, 'cpu') else np.asarray(exp)
    with GeoTiffReader(corr_path) as im:
        got = im.read()
    assert got.dtype == exp.dtype
    assert np.array_equal(got, exp, equal_nan=True)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _rowband_worker(rank, world, port, result_dir):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from homonim_b200.dist import RowBands, fuse_refspace_sharded, source_band_for_proc_rows
        src_ra, ref_ra = _pair(seed=18, nodata=-9999, hp=90, wp=64, ratio=20, ref_pad=0, device=DEV)
        src = RasterArray(src_ra.array[0].contiguous(), src_ra.crs, src_ra.transform, nodata=-9999)
        ref = RasterArray(ref_ra.array[0].contiguous(), ref_ra.crs, ref_ra.transform, nodata=NAN)
        model = RefSpaceModel(Model.gain_blk_offset, (15, 15), find_r2=True)
        full_corr = model.apply(src, model.fit(src, ref)).array
        bands = RowBands.split(ref.height, world)
        r0, r1 = source_band_for_proc_rows(src.shape, src.transform, ref.transform, bands.band(rank))
        src_local = RasterArray(src.array[r0:r1].contiguous(), src.crs, src.transform * Affine.translation(0, r0),
                                nodata=-9999)
        corr_local, _ = fuse_refspace_sharded(model, src_local, ref, bands)
        exp_c, got_c = full_corr[r0:r1], corr_local.array
        ok = torch.equal(torch.isnan(got_c), torch.isnan(exp_c))
        fin = torch.isfinite(exp_c)
        rel = ((got_c - exp_c).abs()[fin] / exp_c.abs()[fin].clamp_min(1e-3 * exp_c[fin].abs().mean())).max().item()
        open(os.path.join(result_dir, f'r{rank}'), 'w').write(f'{int(ok)} {rel}')
    finally:
        dist.destroy_process_group()


def test_int16_row_bands_equal_unsharded(tmp_path):
    mp.spawn(_rowband_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    res = [open(tmp_path / f'r{r}').read().split() for r in range(2)]
    assert all(int(m) for m, _ in res)
    assert max(float(e) for _, e in res) <= 1e-5
