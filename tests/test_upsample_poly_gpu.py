"""
GPU tier: upsample_poly_kernel (csrc/upsample.cu) on the geometries its row loop distinguishes -- rasters several
CTAs wide with a partial last CTA, widths that are not a multiple of 8, CTAs whose row count is not a multiple of the
rows handled per loop iteration, cell rows that start in the middle of an iteration, and the output conversion to
uint8 / uint16 -- against RefSpaceModel.apply of the oracle.
"""
import numpy as np
import pytest

from conftest import RTOL, assert_same_mask

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from homonim_b200 import CRS, Affine, Model, RasterArray, RefSpaceModel, _native   # noqa: E402

NAN = float('nan')
TF_LO = Affine(10, 0, 2000, 0, -10, 9000)


def _case(dtype, nodata, ratio, hs, ws, seed):
    rng = np.random.default_rng(seed)
    hp, wp = int(np.ceil(hs / ratio)) + 1, int(np.ceil(ws / ratio)) + 1
    if dtype == 'float32':
        src = rng.normal(0.3, 0.1, (hs, ws)).astype('float32')
    else:
        src = rng.integers(1, np.iinfo(dtype).max, (hs, ws)).astype(dtype)
    src[rng.integers(0, hs, 200), rng.integers(0, ws, 200)] = nodata
    src[hs // 3:hs // 3 + 7, ws // 4:ws // 4 + 9] = nodata
    yy, xx = np.mgrid[0:hp, 0:wp]
    params = np.stack([0.7 + 0.1 * np.sin(xx / 5.0) + 0.05 * rng.normal(size=(hp, wp)),
                       20.0 + 30.0 * np.cos(yy / 7.0) + 5.0 * rng.normal(size=(hp, wp))]).astype('float32')
    params[:, 8:11, 10:14] = NAN                              # DIRTY and DEAD cells in the middle of the raster
    params[:, rng.integers(0, hp, 6), rng.integers(0, wp, 6)] = NAN
    src_tf = TF_LO * Affine.scale(1.0 / ratio) * Affine.translation(0.25, 0.5)
    return src, src_tf, params


def _oracle(src, src_tf, nodata, params):
    from oracle import kernel_model_np as kmnp
    hs, ws = src.shape
    pad = 64
    src_pad = np.full((hs + 2 * pad, ws + 2 * pad), nodata, dtype=src.dtype)
    src_pad[pad:pad + hs, pad:pad + ws] = src
    pad_tf = src_tf * Affine.translation(-pad, -pad)
    with np.errstate(all='ignore'):
        exp = kmnp.refspace_apply(src_pad, tuple(pad_tf), nodata, params, tuple(TF_LO), (3, 5))
    return exp[pad:pad + hs, pad:pad + ws].astype('float32')


def _apply(src, src_tf, nodata, params, out=None, out_nodata=NAN):
    crs = CRS.from_epsg(3857)
    km = RefSpaceModel(Model.gain_blk_offset, (3, 5))
    lib = _native.lib()
    lib.hb_reset_launch_count()
    res = km.apply(RasterArray(torch.from_numpy(src).cuda(), crs, src_tf, nodata=nodata),
                   RasterArray(torch.from_numpy(params).cuda(), crs, TF_LO, nodata=NAN), out=out, out_nodata=out_nodata)
    torch.cuda.synchronize()
    assert lib.hb_launch_count() == 3, 'expected the pre-pass + polynomial + fix-up kernels'
    return res.array.cpu().numpy()


@pytest.mark.parametrize('dtype, nodata, ratio, hs, ws', [
    ('uint16', 0, 20, 203, 2600),         # 3 CTAs across, the last one partial; 203 rows: a partial last stage
    ('uint16', 0, 20, 130, 2604),         # width % 8 == 4
    ('uint16', 0, 7, 389, 1100),          # cell rows start at every position inside a 4-row stage
    ('uint8', 0, 5, 257, 2052),           # 257 rows: one row in the last CTA's last stage
    ('uint8', 0, 6.4, 301, 1284),         # non-integer ratio
    ('float32', NAN, 9, 262, 1540),       # float32 source (the row-band instantiation)
    ('float32', -9999.0, 13, 515, 3076),
])
def test_poly_row_loop_vs_oracle(dtype, nodata, ratio, hs, ws):
    src, src_tf, params = _case(dtype, nodata, ratio, hs, ws, seed=hs + ws)
    got = _apply(src, src_tf, nodata, params)
    exp = _oracle(src, src_tf, nodata, params)
    assert_same_mask(got, exp, 'poly up-sample + apply')
    fin = np.isfinite(exp)
    scale = np.maximum(np.abs(exp[fin]), 1e-3 * np.mean(np.abs(exp[fin])))
    assert np.max(np.abs(got[fin].astype('float64') - exp[fin]) / scale) <= RTOL


@pytest.mark.parametrize('out_dtype', ['uint8', 'uint16'])
@pytest.mark.parametrize('dtype, nodata, ratio, hs, ws', [
    ('uint16', 0, 20, 203, 2600),
    ('uint8', 0, 7, 131, 1028),
    ('float32', NAN, 11, 150, 1544),
])
def test_poly_convert_store(dtype, nodata, ratio, hs, ws, out_dtype):
    """ The output conversion fused into the store: the float32 result of the same call, rounded half to even, clipped,
    nodata -> the output nodata value -- and that float32 result against the oracle. """
    src, src_tf, params = _case(dtype, nodata, ratio, hs, ws, seed=7 * hs + ws)
    if dtype == 'float32':
        src = (src * 200.0).astype('float32')                  # values in the integer output's range (NaN stays NaN)
    f32 = _apply(src, src_tf, nodata, params)
    exp = _oracle(src, src_tf, nodata, params)
    assert_same_mask(f32, exp, 'poly up-sample + apply (float32)')
    out_nd = 255 if out_dtype == 'uint8' else 65535
    out = torch.empty((hs, ws), dtype=getattr(torch, out_dtype), device='cuda')
    got = _apply(src, src_tf, nodata, params, out=out, out_nodata=out_nd)
    info = np.iinfo(out_dtype)
    want = np.where(np.isnan(f32), out_nd, np.clip(np.round(f32), info.min, info.max)).astype(out_dtype)
    assert np.array_equal(got, want)
