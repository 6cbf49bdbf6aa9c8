"""
CPU tier: int16 source and reference planes -- the dtype code the kernels receive, the dtypes that stay rejected, and
the int16 form of the synthetic pair generator (whose other dtypes must not change: the benchmark uses them).
"""
import pathlib

import numpy as np
import pytest

torch = pytest.importorskip('torch')

from homonim_b200 import _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402
from homonim_b200.synthetic import make_pair   # noqa: E402

GOLDEN = pathlib.Path(__file__).resolve().parent / 'golden'


def test_int16_plane_code():
    assert hkm._plane_code(torch.zeros((2, 2), dtype=torch.int16)) == _native.HB_I16


@pytest.mark.parametrize('dtype', [torch.int32, torch.int8, torch.uint32])
def test_other_integer_dtypes_stay_rejected(dtype):
    with pytest.raises(TypeError, match='uint8, uint16, int16 or float32'):
        hkm._plane_code(torch.zeros((2, 2), dtype=dtype))


@pytest.mark.parametrize('nodata', [-9999, -32768, 32767])
def test_make_pair_int16(nodata):
    src_ra, ref_ra = make_pair(24, 20, 4, bands=2, dtype='int16', seed=3, src_nodata=nodata)
    a = src_ra.array.numpy()
    assert a.dtype == np.int16 and src_ra.nodata == nodata and ref_ra.array.dtype == torch.float32
    valid = a != nodata
    assert (a[valid] < 0).any() and (a[valid] > 0).any()          # values on both sides of zero
    assert (~valid).mean() > 0.02                                  # the nodata wedge and holes


def test_make_pair_existing_dtypes_unchanged():
    """ make_pair(12, 10, 4, bands=2, seed=3) as the generator produced it before int16 existed (arrays stored from
    that version).  torch's CPU kernels may round differently on another CPU, so integers may differ by one where a
    value sat on a rounding boundary and floats by a few ulps; any change to the generator itself moves everything. """
    with np.load(GOLDEN / 'make_pair_seed3.npz') as data:
        golden = {k: data[k] for k in data.files}
    for dtype, nodata in (('uint8', 0.0), ('uint16', 0.0), ('float32', float('nan'))):
        src_ra, ref_ra = make_pair(12, 10, 4, bands=2, dtype=dtype, seed=3, src_nodata=nodata)
        src, ref = src_ra.array.numpy(), ref_ra.array.numpy()
        exp_src, exp_ref = golden[f'{dtype}_src'], golden[f'{dtype}_ref']
        assert src.dtype == exp_src.dtype and src.shape == exp_src.shape
        if dtype == 'float32':
            np.testing.assert_allclose(src, exp_src, rtol=1e-5, equal_nan=True)
        else:
            diff = np.abs(src.astype('int64') - exp_src.astype('int64'))
            assert diff.max() <= 1 and (diff > 0).mean() <= 0.005, dtype
        np.testing.assert_allclose(ref, exp_ref, rtol=1e-4, atol=1e-2)
