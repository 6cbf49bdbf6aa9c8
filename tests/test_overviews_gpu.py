"""
GPU tier, internal overviews (reference fuse.py:151-165): ``hb_build_overviews`` bit for bit against the numpy oracle
(oracle/overviews_np.py) for every dtype x nodata, odd / prime / 1 x N shapes and 1-8 levels, and the file -> file flow
of ``RasterFuse.process(..., build_ovw=True)``.
"""
import math
import warnings

import numpy as np
import pytest

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from homonim_b200 import Model, RasterFuse, _native   # noqa: E402
from homonim_b200.errors import ConfigWarning   # noqa: E402
from homonim_b200.geotiff import GeoTiffReader, write_geotiff   # noqa: E402
from homonim_b200.overviews import build_overviews, overview_factors   # noqa: E402
from homonim_b200.synthetic import make_pair   # noqa: E402
from oracle import overviews_np as ovnp   # noqa: E402

NAN = float('nan')
GEOKEYS = ((1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 32735), (), '')


def _plane(dtype, shape, nodata, seed):
    """ Random pixels over the dtype's range, with scattered and blocked nodata (and NaN in float planes). """
    rng = np.random.default_rng(seed)
    if dtype == 'float32':
        plane = (rng.normal(0, 1000, shape) * rng.choice([1e-3, 1, 1e3], shape)).astype('float32')
        plane[rng.random(shape) < 0.1] = NAN
    else:
        info = np.iinfo(dtype)
        plane = rng.integers(info.min, int(info.max) + 1, shape).astype(dtype)
    if nodata is not None and not math.isnan(nodata):
        plane[rng.random(shape) < 0.25] = nodata
        plane[..., :9, :13] = nodata                      # whole windows without a valid pixel
    return plane


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape
    return np.array_equal(a.view(f'u{a.dtype.itemsize}'), b.view(f'u{b.dtype.itemsize}'))


DTYPE_NODATA = [('uint8', None), ('uint8', 0), ('uint16', None), ('uint16', 0), ('int16', None), ('int16', -9999),
                ('float32', None), ('float32', NAN), ('float32', -9999.0)]
SHAPES_LEVELS = [((1, 64, 64), 6), ((1, 67, 45), 3), ((4, 131, 257), 8), ((1, 1, 97), 7), ((1, 97, 1), 2),
                 ((4, 1031, 515), 8), ((1, 509, 1021), 1), ((1, 1, 1), 4)]


@pytest.mark.parametrize('dtype, nodata', DTYPE_NODATA)
@pytest.mark.parametrize('shape, n_levels', SHAPES_LEVELS)
def test_build_overviews_bit_identical_to_oracle(dtype, nodata, shape, n_levels):
    plane = _plane(dtype, shape, nodata, seed=sum(shape) + len(dtype) + n_levels)
    dev = torch.from_numpy(plane).cuda()
    lib = _native.lib()
    lib.hb_reset_launch_count()
    got = build_overviews(dev if shape[0] > 1 else dev[0], nodata, n_levels)
    torch.cuda.synchronize()
    assert lib.hb_launch_count() <= 2
    expect = ovnp.build_overviews(plane if shape[0] > 1 else plane[0], nodata, n_levels)
    assert len(got) == n_levels
    for k, (g, e) in enumerate(zip(got, expect)):
        assert str(g.dtype) == f'torch.{dtype}'
        assert _same_bits(g.cpu().numpy(), e), f'level {k + 1} differs at {int((g.cpu().numpy() != e).sum())} pixels'


def test_build_overviews_full_size_plane():
    """ A 20000 x 20000 float32 plane (larger than L2), 6 levels, bit for bit. """
    gen = torch.Generator(device='cuda').manual_seed(5)
    dev = torch.randn((20000, 20000), generator=gen, device='cuda') * 500
    dev[torch.rand((20000, 20000), generator=gen, device='cuda') < 0.05] = -9999.0
    got = build_overviews(dev, -9999.0, 6)
    expect = ovnp.build_overviews(dev.cpu().numpy(), -9999.0, 6)
    for g, e in zip(got, expect):
        assert _same_bits(g.cpu().numpy(), e)


def test_build_overviews_rejects_bad_input():
    with pytest.raises(TypeError):
        build_overviews(torch.zeros((8, 8), dtype=torch.uint16), None, 1)           # host tensor
    with pytest.raises(TypeError):
        build_overviews(np.zeros((8, 8), 'uint16'), None, 1)
    with pytest.raises(ValueError):
        build_overviews(torch.zeros((8, 8), dtype=torch.float64, device='cuda'), None, 1)
    with pytest.raises(ValueError):
        build_overviews(torch.zeros((8, 16), dtype=torch.float32, device='cuda')[:, ::2], None, 1)
    with pytest.raises(ValueError):
        build_overviews(torch.zeros((8, 8), dtype=torch.float32, device='cuda'), None, 9)
    assert build_overviews(torch.zeros((8, 8), dtype=torch.float32, device='cuda'), None, 0) == []


def test_build_overviews_runs_on_the_current_stream():
    plane = torch.from_numpy(_plane('uint16', (2, 300, 200), 0, 1)).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = build_overviews(plane, 0, 3)
    side.synchronize()
    for g, e in zip(got, ovnp.build_overviews(plane.cpu().numpy(), 0, 3)):
        assert _same_bits(g.cpu().numpy(), e)


# ---- file -> file ------------------------------------------------------------------------------------------------------
def _files(tmp_path, src_ra, ref_ra):
    wl = [dict(center_wavelength=w) for w in (0.48, 0.56, 0.66, 0.83)[:src_ra.count]]
    src = write_geotiff(tmp_path / 'src.tif', src_ra.to_host().array, src_ra.transform, nodata=0, geokeys=GEOKEYS,
                        band_tags=wl)
    ref = write_geotiff(tmp_path / 'ref.tif', ref_ra.to_host().array, ref_ra.transform, geokeys=GEOKEYS, band_tags=wl)
    return src, ref


def _run(src, ref, out, proc_crs, out_dtype, nodata, build_ovw, param=None):
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter('always')
        with RasterFuse(src, ref, proc_crs=proc_crs) as fuse:
            fuse.process(out, Model.gain_offset, (5, 5), param_filename=param, build_ovw=build_ovw,
                         out_profile=dict(dtype=out_dtype, nodata=nodata))
    return [w for w in caught if issubclass(w.category, ConfigWarning)]


def _check_levels(path, nodata):
    """ The file's overviews are the oracle's pyramid of its base as read back; returns the factors. """
    with GeoTiffReader(path) as im:
        base, factors = im.read(), im.overviews(1)
        assert factors == overview_factors(base.shape)
    expect = ovnp.build_overviews(base, nodata, len(factors))
    for k, e in enumerate(expect):
        with GeoTiffReader(path, overview_level=k) as im:
            assert _same_bits(im.read(), e), f'{path}: overview {k} differs'
    return factors, base


@pytest.mark.parametrize('out_dtype, nodata', [('uint16', 0), ('float32', NAN)])
def test_file_flow_writes_overviews_proc_crs_ref(tmp_path, out_dtype, nodata):
    src_ra, ref_ra = make_pair(110, 104, 20, bands=2, dtype='uint16', seed=11, device='cuda', src_nodata=0.0)
    src, ref = _files(tmp_path, src_ra, ref_ra)
    corr, param = tmp_path / 'corr.tif', tmp_path / 'corr_PARAM.tif'
    assert _run(src, ref, corr, 'ref', out_dtype, nodata, True, param=param) == []
    factors, base = _check_levels(corr, nodata)
    assert factors == [2, 4, 8]                                    # 2080 x 2200
    with GeoTiffReader(param) as im:
        assert im.overviews(1) == []                               # the reference grid: under 512 px
    assert _run(src, ref, tmp_path / 'plain.tif', 'ref', out_dtype, nodata, False) == []
    with GeoTiffReader(tmp_path / 'plain.tif') as im:
        assert im.overviews(1) == [] and _same_bits(im.read(), base)


def test_file_flow_writes_overviews_proc_crs_src(tmp_path):
    src_ra, ref_ra = make_pair(2048, 2100, 1, bands=2, dtype='uint16', seed=12, device='cuda', src_nodata=0.0)
    src, ref = _files(tmp_path, src_ra, ref_ra)
    corr, param = tmp_path / 'corr.tif', tmp_path / 'corr_PARAM.tif'
    caught = _run(src, ref, corr, 'src', 'float32', NAN, True, param=param)
    # (the only warning: proc_crs=src on grids of equal resolution is not the recommended choice)
    assert all('proc_crs' in str(w.message) for w in caught) and len(caught) <= 1
    assert _check_levels(corr, NAN)[0] == [2, 4, 8]
    assert _check_levels(param, NAN)[0] == [2, 4, 8]
    with GeoTiffReader(param) as im:
        assert im.count == 6 and im.descriptions[0] == 'B1_GAIN'


def test_file_flow_other_dtypes_warn_without_overviews(tmp_path):
    src_ra, ref_ra = make_pair(110, 104, 20, bands=1, dtype='uint16', seed=13, device='cuda', src_nodata=0.0)
    src, ref = _files(tmp_path, src_ra, ref_ra)
    caught = _run(src, ref, tmp_path / 'f64.tif', 'ref', 'float64', NAN, True)
    assert len(caught) == 1 and 'overviews' in str(caught[0].message)
    with GeoTiffReader(tmp_path / 'f64.tif') as im:
        assert im.dtype.name == 'float64' and im.overviews(1) == []
