"""
GPU tier: the launch-time variants of the in-painting, down-sampling and fit kernels that the rest of the suite does not
reach, each against an independent answer.  Every case also checks, with torch.profiler, that the variant it exists for
is the kernel that ran, so that a change to the dispatch cannot quietly move a case onto another variant.

  A. ``inpaint_scan_kernel`` (planes taller than 8192 rows) and ``inpaint_scan_small_kernel`` through
     ``hb_inpaint_refit``, bit for bit against numpy + the GDALFillNodata restatement;
  B. the same in-painting end to end on tall planes (same-grid at C = 1 and C = 4, RefSpace fuse);
  C. ``downsample_int_aligned_kernel`` (the exact-box down-sampler), bit for bit against GRA_Average, with a twin per
     case that breaks one of its eligibility conditions and so runs ``downsample_average_kernel``;
  D. ``fit_same_grid_kernel`` at C = 4 in its general form (value nodata, kh = 1 / kw = 1), with scalar loads
     (w % 4 != 0, misaligned base pointer), fused into a uint16 store, and on both sides of the C = 1 / C = 4 switch.

Tall, narrow planes keep the oracle (cv2 box filters, OpenMP fill) at a few million pixels.
"""
import re
import warnings

import numpy as np
import pytest

from conftest import check_corr, check_params

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

from homonim_b200 import CRS, Affine, KernelModel, Model, RasterArray, RasterFuse, _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402
from homonim_b200.synthetic import make_pair   # noqa: E402

NAN = float('nan')
F32 = np.float32
CRS0 = CRS.from_epsg(3857)
TF1 = Affine(1.0, 0.0, 0.0, 0.0, -1.0, 0.0)


def _oracle():
    from oracle import gdal_restate, kernel_model_np
    return gdal_restate, kernel_model_np


def _stream():
    return torch.cuda.current_stream().cuda_stream


def launched_kernels(fn):
    """ Run ``fn`` under torch.profiler; returns (fn's result, names of the CUDA kernels it launched). """
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [ev.name for ev in prof.events() if ev.device_type.name == 'CUDA']


def kernel_launches(names, kernel):
    """ Template arguments of every launch of ``kernel`` in ``names`` (a list per launch, casts such as ``(bool)`` and
    ``true`` / ``false`` normalised to ``1`` / ``0``; ``[]`` for a non-template kernel). """
    out = []
    for name in names:
        m = re.search(r'\b' + kernel + r'\b(<([^>]*)>)?', name)
        if m is None:
            continue
        args = [] if m.group(2) is None else [re.sub(r'^\([\w ]+\)', '', a.strip()) for a in m.group(2).split(',')]
        out.append([{'true': '1', 'false': '0'}.get(a, a) for a in args])
    return out


def assert_ran(names, kernel, args=None, absent=()):
    """ ``kernel`` was launched (with template arguments ``args``, given as strings, where not None) and none of
    ``absent`` was. """
    launches = kernel_launches(names, kernel)
    assert launches, f'{kernel} did not run; launched: {names}'
    if args is not None:
        assert all(a == list(args) for a in launches), f'{kernel}: expected <{", ".join(args)}>, launched {launches}'
    for other in absent:
        assert not kernel_launches(names, other), f'{other} ran; launched: {names}'


def assert_bits_equal(got, exp, what):
    """ Same NaN pattern and the same bits everywhere else. """
    got, exp = np.asarray(got, F32), np.asarray(exp, F32)
    assert got.shape == exp.shape, what
    gn, en = np.isnan(got), np.isnan(exp)
    assert np.array_equal(gn, en), f'{what}: NaN patterns differ at {int((gn != en).sum())} pixels'
    diff = got[~gn].view(np.uint32) != exp[~en].view(np.uint32)
    assert not diff.any(), f'{what}: {int(diff.sum())} pixels differ, e.g. got {got[~gn][diff][:5]} ' \
                           f'expected {exp[~en][diff][:5]}'


# =====================================================================================================================
# A. in-painting tables, kernel level
# =====================================================================================================================
INPAINT_THRESH = 0.3
INPAINT_SHAPES = [(8192, 37), (8193, 37), (8193, 1), (9000, 33), (20000, 64), (12000, 70)]
INPAINT_PATTERNS = ['random_low_r2', 'column_without_source', 'sources_in_first_chunk_only', 'reach_100_101',
                    'runs_across_chunk_boundaries', 'rows_outside_mask', 'nonpositive_gain_nan_r2',
                    'r2_at_threshold']


def inpaint_planes(h, w, pattern, seed):
    """ params [3, h, w] (gain, offset, R2: NaN outside the mask, as the fit leaves them) and sums [3, h, w]
    (ref_sum, src_sum, valid count; the count is -1 outside the mask), host float32. """
    rng = np.random.default_rng(seed)
    rc = -(-h // 32)                                                 # rows per chunk of inpaint_scan_kernel
    gain = rng.uniform(0.5, 1.5, (h, w)).astype(F32)
    off = rng.normal(0.0, 50.0, (h, w)).astype(F32)
    r2 = rng.uniform(0.5, 1.0, (h, w)).astype(F32)
    cnt = rng.integers(1, 26, (h, w)).astype(F32)
    ref_sum = (cnt * rng.uniform(100.0, 4000.0, (h, w))).astype(F32)
    src_sum = (cnt * rng.uniform(100.0, 4000.0, (h, w))).astype(F32)
    mask = np.ones((h, w), bool)
    low = np.zeros((h, w), bool)                                     # pixels that fail the R2 test
    xc = w // 2
    if pattern == 'random_low_r2':
        while low.mean() < 0.3:
            y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
            low[y:y + int(rng.integers(1, 200)), x:x + int(rng.integers(1, w + 1))] = True
    elif pattern == 'column_without_source':
        low[:, xc] = True
    elif pattern == 'sources_in_first_chunk_only':
        # column xc has sources only in rows < rc - 20; its neighbours within 30 columns have none in the 150 rows
        # below, so the targets of chunk 1 within reach take their top source from chunk 0 through the carry
        low[rc - 20:, xc] = True
        low[rc - 20:rc + 130, max(xc - 30, 0):xc + 31] = True
    elif pattern == 'reach_100_101':
        # one source at (a, xc) in a block of targets: (a + 100, xc) is within reach of it alone, (a + 101, xc) of
        # nothing (the next sources are more than 100 pixels away in every quadrant)
        a = h // 2
        low[a - 150:a + 202, :] = True
        low[a, xc] = False
    elif pattern == 'runs_across_chunk_boundaries':
        for k in range(1, 32):
            b = k * rc
            low[max(b - 2, 0):min(b + 3, h), :] = True
    elif pattern == 'rows_outside_mask':
        rows = np.concatenate([rng.integers(0, h, 30), [0, h - 1, rc - 1, rc, 5 * rc + 1]])
        mask[rows, :] = False
        low |= rng.random((h, w)) < 0.15
    elif pattern == 'nonpositive_gain_nan_r2':
        pick = rng.random((h, w))
        gain[pick < 0.04] = -1.0
        gain[(pick >= 0.04) & (pick < 0.06)] = 0.0
        gain[(pick >= 0.06) & (pick < 0.07)] = -0.0
        r2[(pick >= 0.07) & (pick < 0.12)] = NAN
    elif pattern == 'r2_at_threshold':
        t = F32(INPAINT_THRESH)
        pick = rng.random((h, w))
        r2[pick < 0.1] = t
        r2[(pick >= 0.1) & (pick < 0.15)] = np.nextafter(t, F32(1))
        r2[(pick >= 0.15) & (pick < 0.2)] = np.nextafter(t, F32(0))
    else:
        raise ValueError(pattern)
    r2[low] = rng.uniform(0.0, 0.25, int(low.sum())).astype(F32)
    gain[~mask] = off[~mask] = r2[~mask] = NAN
    cnt[~mask] = -1.0
    return np.stack([gain, off, r2]), np.stack([ref_sum, src_sum, cnt])


def inpaint_expected(params, sums, thresh):
    """ kernel_model.py:363-371 in numpy with the GDALFillNodata restatement (oracle.fit_gain_offset :192-199). """
    gr, _ = _oracle()
    gain, off, r2 = (p.copy() for p in params)
    ref_sum, src_sum, cnt = sums
    mask = cnt >= 0
    with np.errstate(invalid='ignore'):
        r2_mask = (r2 > F32(thresh)) & (gain > 0) & mask
    off = gr.fillnodata(off, r2_mask)
    off[~mask] = NAN
    refit = ~r2_mask & mask
    gain[refit] = (ref_sum[refit] - cnt[refit] * off[refit]) / src_sum[refit]
    return np.stack([gain, off, r2])


@pytest.mark.parametrize('pattern', INPAINT_PATTERNS)
@pytest.mark.parametrize('shape', INPAINT_SHAPES)
def test_inpaint_tables_vs_numpy(shape, pattern):
    """ hb_inpaint_refit on host-built planes: gain, offset and R2 bit-identical to the numpy statement. """
    h, w = shape
    params, sums = inpaint_planes(h, w, pattern, seed=h + w)
    expected = inpaint_expected(params, sums, INPAINT_THRESH)
    lib = _native.lib()
    p, s = torch.from_numpy(params).cuda(), torch.from_numpy(sums).cuda()
    nbytes = lib.hb_inpaint_workspace_bytes(h, w)
    work = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    _, names = launched_kernels(lambda: _native.check(lib.hb_inpaint_refit(
        p.data_ptr(), s.data_ptr(), h, w, INPAINT_THRESH, hkm.MAX_SEARCH_DISTANCE, work.data_ptr(), nbytes,
        _stream()), 'hb_inpaint_refit'))
    if h <= 8192:
        assert_ran(names, 'inpaint_scan_small_kernel', absent=['inpaint_scan_kernel'])
    else:
        assert_ran(names, 'inpaint_scan_kernel', absent=['inpaint_scan_small_kernel'])
    assert_ran(names, 'inpaint_fill_kernel')
    got = p.cpu().numpy()
    # the planes give the fill work to do (a single column without a source pixel has none)
    filled = np.isfinite(params[1]) & (got[1] != params[1])
    assert filled.any() or (pattern == 'column_without_source' and w == 1)
    for b, what in enumerate(('gain', 'offset', 'R2')):
        assert_bits_equal(got[b], expected[b], f'{shape} {pattern}: {what}')


# =====================================================================================================================
# B. in-painting end to end on tall planes
# =====================================================================================================================
def _assert_r2_clear_of(r2, thresh, what):
    """ No expected R2 lies within rounding of the threshold (such a pixel may flip legitimately and move nearby
    offsets). """
    fin = r2[np.isfinite(r2)].astype('float64')
    gap = float(np.min(np.abs(fin - float(F32(thresh)))))
    assert gap > 1e-5, f'{what}: an expected R2 lies {gap:.2g} from the threshold; choose another seed'


@pytest.mark.parametrize('shape, seed, c', [((8704, 96), 2, 1), ((9000, 480), 2, 4)])
def test_same_grid_inpaint_tall_vs_oracle(shape, seed, c):
    """ KernelModel gain-offset 5 x 5, r2_inpaint_thresh = 0.25, on same-grid float32 planes taller than 8192 rows: the
    fit at C = 1 (< 4 M pixels) or C = 4 (lean form) followed by the large-raster in-painting tables. """
    _, kmnp = _oracle()
    h, w = shape
    src_ra, ref_ra = make_pair(h, w, 1, bands=1, dtype='float32', mu=0.3, seed=seed, src_nodata=NAN, ref_pad=0,
                               bad_blobs=40)
    src, ref = src_ra.array[0].numpy(), ref_ra.array[0].numpy()
    exp_params = kmnp.fit_same_grid(src, NAN, ref, NAN, Model.gain_offset, (5, 5), False, 0.25)
    _assert_r2_clear_of(exp_params[2], 0.25, f'{shape}')
    km = KernelModel(Model.gain_offset, (5, 5), r2_inpaint_thresh=0.25)
    s_ra = RasterArray(torch.from_numpy(src).cuda(), CRS0, src_ra.transform, nodata=NAN)
    r_ra = RasterArray(torch.from_numpy(ref).cuda(), CRS0, src_ra.transform, nodata=NAN)
    param_ra, names = launched_kernels(lambda: km.fit(s_ra, r_ra))
    assert_ran(names, 'fit_same_grid_kernel', args=fit_variant(Model.gain_offset, True, c=c, lean=c == 4))
    assert_ran(names, 'inpaint_scan_kernel', absent=['inpaint_scan_small_kernel'])
    corr_ra = km.apply(s_ra, param_ra)
    got = param_ra.to_host().array
    bad = check_params(got, exp_params, float(np.nanmean(src)), 'params')
    check_corr(corr_ra.to_host().array, kmnp.apply_same_grid(src, exp_params), 'corr', bad=bad)
    same = (got[0] == exp_params[0]) | (np.isnan(got[0]) & np.isnan(exp_params[0]))
    assert same.mean() > 0.99


def test_refspace_inpaint_tall_reference_vs_oracle():
    """ RasterFuse proc_crs = ref whose reference grid is taller than 8192 rows: the fused RefSpace call in-paints with
    the large-raster tables. """
    _, kmnp = _oracle()
    src_ra, ref_ra = make_pair(8300, 40, 2, bands=1, dtype='uint16', mu=3000.0, seed=1, src_nodata=0, bad_blobs=40)
    src, ref = src_ra.array[0].numpy(), ref_ra.array[0].numpy()
    exp_params, _, exp_corr = kmnp.fuse_band_blocks(src, tuple(src_ra.transform), 0, ref, tuple(ref_ra.transform), NAN,
                                                    Model.gain_offset, (5, 5), 'ref', True, 0.25)
    assert exp_params.shape[1] > 8192
    _assert_r2_clear_of(exp_params[2], 0.25, 'refspace')
    s_ra, r_ra = src_ra.to_device(), ref_ra.to_device()

    def run():
        with RasterFuse(s_ra, r_ra) as fuse:
            return fuse.process(model=Model.gain_offset, kernel_shape=(5, 5), param_filename='params',
                                model_config=dict(r2_inpaint_thresh=0.25))
    (corr_ra, param_ra), names = launched_kernels(run)
    assert_ran(names, 'inpaint_scan_kernel', absent=['inpaint_scan_small_kernel'])
    got = param_ra.to_host().array
    valid = src[src != 0].astype('float64')
    check_params(got, exp_params, float(np.mean(valid)), 'params')
    check_corr(corr_ra.to_host().array[0], exp_corr.astype('float32'), 'corr')


# =====================================================================================================================
# C. the exact-box down-sampler
# =====================================================================================================================
def _borrow_values(dtype, nodata):
    """ Values whose XOR with the nodata pattern borrows in the packed has-zero test. """
    raw = (1, 0x0100, 0x8000, 0x7FFF) if dtype == 'uint16' else (1, 0x80)
    nd = 0 if nodata is None else int(nodata)
    return [v ^ nd for v in raw]


def downsample_source(dtype, nodata, rx, ry, ox, oy, hd, wd, extra_cols, extra_rows, seed, fill=None):
    """ Source covering a (hd, wd) destination of (ry, rx) boxes from source offset (oy, ox), plus ``extra_rows`` /
    ``extra_cols`` (may be negative), with all-nodata footprints and nodata at every position of a 32-bit word next to
    borrowing values. """
    rng = np.random.default_rng(seed)
    hs, ws = oy + hd * ry + extra_rows, ox + wd * rx + extra_cols
    top = np.iinfo(dtype).max
    if fill is not None:
        return np.full((hs, ws), fill, dtype=dtype)
    src = rng.integers(0, top + 1, (hs, ws)).astype(dtype)
    if nodata is not None:
        # all-nodata footprints: destination (0, 0), (hd - 1, wd - 1) and one in the middle
        for (i, j) in ((0, 0), (hd - 1, wd - 1), (hd // 2, wd // 2)):
            src[oy + i * ry:oy + (i + 1) * ry, ox + j * rx:ox + (j + 1) * rx] = nodata
        # nodata at each position of a word, the other fields borrowing values, across a band of rows
        g = 4 // np.dtype(dtype).itemsize
        vals = _borrow_values(dtype, nodata)
        y0 = oy + (hd // 3) * ry
        for r in range(min(ry * 2, hs - y0)):
            for c in range(ox, min(ws, ox + 16 * g * 8), g):
                pos = (c // g + r) % (g + 1)             # (one word in g + 1 has no nodata field)
                for f in range(g):
                    src[y0 + r, c + f] = nodata if f == pos else vals[(r + c + f) % len(vals)]
        src[rng.random((hs, ws)) < 0.01] = nodata
    return src


# name: dtype, nodata, (rx, ry), (ox, oy), (hd, wd), extra (cols, rows), fill value
DS_CASES = {
    'u16_8x8_nd-none_ends-on-last-pixel': ('uint16', None, (8, 8), (0, 0), (40, 300), (0, 0), None),
    'u16_20x20_nd0_offset': ('uint16', 0, (20, 20), (4, 7), (30, 120), (4, 3), None),
    'u16_24x1_nd65535': ('uint16', 65535, (24, 1), (2, 1), (200, 100), (6, 0), None),
    'u16_16x40_nd0_ends-on-last-pixel': ('uint16', 0, (16, 40), (8, 40), (12, 150), (0, 0), None),
    'u16_254x255_all-65535_nd-none': ('uint16', None, (254, 255), (0, 0), (2, 9), (2, 0), 65535),
    'u16_254x255_all-65535_nd0': ('uint16', 0, (254, 255), (2, 1), (2, 9), (0, 0), 65535),
    'u16_8x255_nd0': ('uint16', 0, (8, 255), (6, 0), (3, 260), (2, 0), None),
    'u8_8x8_nd-none': ('uint8', None, (8, 8), (0, 0), (40, 300), (0, 0), None),
    'u8_20x20_nd0_offset': ('uint8', 0, (20, 20), (4, 5), (30, 120), (12, 0), None),
    'u8_24x1_nd255': ('uint8', 255, (24, 1), (8, 3), (200, 100), (8, 0), None),
    'u8_16x40_nd255_ends-on-last-pixel': ('uint8', 255, (16, 40), (0, 0), (12, 150), (0, 0), None),
    'u8_252x255_all-255_nd0': ('uint8', 0, (252, 255), (0, 0), (2, 9), (4, 0), 255),
}
# per eligible case, the twin that breaks one condition of the exact-box kernel
DS_TWINS = {
    'u16_8x8_nd-none_ends-on-last-pixel': 'rx_256',
    'u16_20x20_nd0_offset': 'pitch_not_16_bytes',
    'u16_24x1_nd65535': 'offset_1',
    'u16_16x40_nd0_ends-on-last-pixel': 'one_row_short',
    'u16_254x255_all-65535_nd-none': 'rx_odd',
    'u16_254x255_all-65535_nd0': 'base_pointer_plus_1',
    'u16_8x255_nd0': 'rx_odd',
    'u8_8x8_nd-none': 'base_pointer_plus_1',
    'u8_20x20_nd0_offset': 'pitch_not_16_bytes',
    'u8_24x1_nd255': 'one_row_short',
    'u8_16x40_nd255_ends-on-last-pixel': 'rx_256',
    'u8_252x255_all-255_nd0': 'offset_1',
}


def _twin_geometry(kind, dtype, rxy, oxy, hdw, extra):
    (rx, ry), (ox, oy), (hd, wd), (ec, er) = rxy, oxy, hdw, extra
    g = 4 // np.dtype(dtype).itemsize
    if kind == 'rx_256':
        rx, wd = 256, 7
        ec = (-(ox + wd * rx)) % 16
    elif kind == 'rx_odd':
        rx = rx + 1 if rx % 2 == 0 else rx
        rx = 255 if rx > 255 else rx
        ec = (-(ox + wd * rx)) % 16
    elif kind == 'offset_1':
        ox = 1
        ec = (-(ox + wd * rx)) % 16 + (16 if g == 4 else 0)
    elif kind == 'pitch_not_16_bytes':
        ec = ec + 16 // np.dtype(dtype).itemsize // 2
    elif kind == 'one_row_short':
        er = -1
    return (rx, ry), (ox, oy), (hd, wd), (ec, er)


def _downsample(src_t, rxy, oxy, hdw, nodata):
    (rx, ry), (ox, oy), (hd, wd) = rxy, oxy, hdw
    dst_tf = Affine(float(rx), 0.0, float(ox), 0.0, -float(ry), -float(oy))
    return launched_kernels(lambda: hkm._downsample_average(src_t, TF1, nodata, (hd, wd), dst_tf))


def _downsample_expected(src, rxy, oxy, hdw, nodata):
    gr, _ = _oracle()
    (rx, ry), (ox, oy), (hd, wd) = rxy, oxy, hdw
    dst_tf = Affine(float(rx), 0.0, float(ox), 0.0, -float(ry), -float(oy))
    return gr.reproject_array(src, tuple(TF1), nodata, (hd, wd), tuple(dst_tf), NAN, 'average')


@pytest.mark.parametrize('case', sorted(DS_CASES))
def test_downsample_exact_box_vs_oracle(case):
    """ Integer ratio, G-aligned integer offset, destination inside the source, 16-byte pitch and base: the exact-box
    kernel, bit-identical to GRA_Average.  Its twin breaks one of those conditions, runs the general kernel, and is
    bit-identical to GRA_Average on every cell whose footprint lies inside the source. """
    dtype, nodata, rxy, oxy, hdw, extra, fill = DS_CASES[case]
    itemsize = np.dtype(dtype).itemsize
    src = downsample_source(dtype, nodata, *rxy, *oxy, *hdw, *extra, seed=len(case), fill=fill)
    assert (src.shape[1] * itemsize) % 16 == 0 and oxy[0] % (4 // itemsize) == 0
    assert oxy[1] + hdw[0] * rxy[1] <= src.shape[0] and oxy[0] + hdw[1] * rxy[0] <= src.shape[1]
    expected = _downsample_expected(src, rxy, oxy, hdw, nodata)
    got, names = _downsample(torch.from_numpy(src).cuda(), rxy, oxy, hdw, nodata)
    ctype = 'unsigned short' if dtype == 'uint16' else 'unsigned char'
    assert_ran(names, 'downsample_int_aligned_kernel', args=[ctype, '1' if nodata is not None else '0'],
               absent=['downsample_average_kernel'])
    got = got.cpu().numpy()
    assert np.array_equal(got, expected, equal_nan=True), \
        f'{case}: {int((got != expected).sum())} cells differ; max |d| {np.nanmax(np.abs(got - expected))}'
    if fill is not None:
        assert np.all(got == float(fill))                             # the largest sums: exact, no wrap-around
    if nodata is not None and fill is None:
        assert np.isnan(got[0, 0]) and np.isnan(got[-1, -1])          # all-nodata footprints
        assert np.isfinite(got).mean() > 0.9
    # the twin
    kind = DS_TWINS[case]
    trxy, toxy, thdw, textra = _twin_geometry(kind, dtype, rxy, oxy, hdw, extra)
    tsrc = downsample_source(dtype, nodata, *trxy, *toxy, *thdw, *textra, seed=len(case) + 1, fill=fill)
    texp = _downsample_expected(tsrc, trxy, toxy, thdw, nodata)
    if kind == 'base_pointer_plus_1':
        buf = torch.empty(tsrc.size + 1, dtype=getattr(torch, dtype), device='cuda')
        tsrc_t = buf[1:].view(tsrc.shape)
        tsrc_t.copy_(torch.from_numpy(tsrc))
        assert tsrc_t.data_ptr() % 16 != 0
    else:
        tsrc_t = torch.from_numpy(tsrc).cuda()
    tgot, tnames = _downsample(tsrc_t, trxy, toxy, thdw, nodata)
    assert_ran(tnames, 'downsample_average_kernel', absent=['downsample_int_aligned_kernel'])
    tgot = tgot.cpu().numpy()
    inside = np.ones(thdw, bool)
    if kind == 'one_row_short':
        inside[-1, :] = False
    assert inside.mean() > 0.5
    assert np.array_equal(tgot[inside], texp[inside], equal_nan=True), \
        f'{case} twin {kind}: {int((tgot[inside] != texp[inside]).sum())} cells differ'


# =====================================================================================================================
# D. the fit at C = 4: general form, scalar loads, fused store, the C = 1 / C = 4 switch
# =====================================================================================================================
FIT_H, FIT_W = 2100, 2050                                            # 4.3 M pixels (C = 4), w % 4 == 2


def fit_pair(h, w, seed, src_dtype='float32', src_nodata=NAN, ref_nodata=NAN):
    """ Seeded same-grid source / reference planes (host numpy) with nodata holes on both and decorrelated blobs. """
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype('float64')
    # (the pixel-scale term gives every window a variance well above the rounding of the reference's float32 R2
    #  recipe, whose terms cancel: on smooth texture its own R2 is off by up to 1e-3 in small windows)
    tex = (np.sin(xx / 23.0) * np.cos(yy / 31.0) + 0.5 * np.sin((xx + 2 * yy) / 13.0)
           + 0.6 * (np.sin(xx / 1.3) + np.sin(yy / 1.7)))
    mu = 3000.0 if src_dtype == 'uint16' else 0.3
    src = mu * (1.0 + 0.3 * tex) + 0.03 * mu * rng.standard_normal((h, w))
    gain = 0.7 + 0.1 * np.sin(xx / 150.0 + yy / 230.0)
    ref = gain * src + 0.05 * mu * np.cos(yy / 170.0) + 0.01 * mu * rng.standard_normal((h, w))
    for _ in range(12):
        y, x = int(rng.integers(0, h - 40)), int(rng.integers(0, w - 40))
        ref[y:y + 40, x:x + 40] = mu * (0.7 + 0.2 * rng.standard_normal((40, 40)))
    if src_dtype == 'uint16':
        src = np.clip(np.round(src), 1, 65535)
    src, ref = src.astype(src_dtype), ref.astype('float32')
    for (r0, r1, c0, c1) in ((0, 30, 0, 200), (h - 9, h, 500, 900), (700, 760, w - 33, w), (1000, 1200, 1000, 1003),
                             (300, 301, 0, w)):
        src[r0:r1, c0:c1] = src_nodata
    src[rng.random((h, w)) < 0.002] = src_nodata
    ref[40:80, 1200:1300] = ref_nodata
    ref[rng.random((h, w)) < 0.002] = ref_nodata
    return src, ref


def fit_variant(model, want_r2, c, fused=False, lean=False):
    """ Template arguments <MODEL, WANT_R2, NQ, C, FUSED, LEAN> of the fit_same_grid_kernel a case must launch. """
    nq = 5 if want_r2 else (4 if model == Model.gain_offset else 2)
    return [str(v) for v in (hkm._MODEL_CODES[model], int(want_r2), nq, c, int(fused), int(lean))]


def _fit_vs_oracle(params_t, src, src_nodata, ref, ref_nodata, model, kshape, find_r2, thresh, what):
    _, kmnp = _oracle()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        exp = kmnp.fit_same_grid(src, src_nodata, ref, ref_nodata, model, kshape, find_r2, thresh)
    if thresh is not None:
        _assert_r2_clear_of(exp[2], thresh, what)
    got = params_t.cpu().numpy() if torch.is_tensor(params_t) else params_t
    valid = src[kmnp.valid_mask(src, src_nodata)].astype('float64')
    bad = check_params(got, exp, float(valid.mean()), what)
    same = (got[0] == exp[0]) | (np.isnan(got[0]) & np.isnan(exp[0]))
    assert same.mean() > 0.99, f'{what}: only {same.mean():.4f} of the gains are bit-identical'
    return exp, bad


@pytest.mark.parametrize('model, kshape, find_r2, thresh', [
    (Model.gain, (5, 5), False, None),
    (Model.gain_blk_offset, (5, 5), True, None),
    (Model.gain_offset, (15, 15), False, 0.25),
])
def test_fit_c4_value_nodata_vs_oracle(model, kshape, find_r2, thresh):
    """ KernelModel.fit of a uint16 source with nodata 0 (widened to float32, nodata kept) and a float32 reference with
    nodata -9999: the general form at C = 4 with scalar loads (w % 4 == 2), then apply, against the oracle. """
    _, kmnp = _oracle()
    src, ref = fit_pair(FIT_H, FIT_W, seed=9, src_dtype='uint16', src_nodata=0, ref_nodata=-9999.0)
    km = KernelModel(model, kshape, find_r2=find_r2, r2_inpaint_thresh=thresh)
    s_ra = RasterArray(torch.from_numpy(src).cuda(), CRS0, TF1, nodata=0)
    r_ra = RasterArray(torch.from_numpy(ref).cuda(), CRS0, TF1, nodata=-9999.0)
    param_ra, names = launched_kernels(lambda: km.fit(s_ra, r_ra))
    assert_ran(names, 'fit_same_grid_kernel', args=fit_variant(model, find_r2 or thresh is not None, c=4))
    exp, bad = _fit_vs_oracle(param_ra.array, src, 0, ref, -9999.0, model, kshape, find_r2, thresh, f'{model} {kshape}')
    corr = km.apply(s_ra, param_ra).array.cpu().numpy()
    check_corr(corr, kmnp.apply_same_grid(src, exp), 'corr', bad=bad)


@pytest.mark.parametrize('variant', ['nan_nodata_w_mod_4', 'misaligned_base_pointer'])
def test_fit_c4_lean_scalar_loads_vs_oracle(variant):
    """ The lean form (NaN nodata) at C = 4 without 16-byte loads: across a whole raster whose width is not a multiple
    of 4, and on a plane whose base pointer is one float past a 16-byte boundary (a view at storage offset 1). """
    w = FIT_W if variant == 'nan_nodata_w_mod_4' else 2052
    src, ref = fit_pair(FIT_H, w, seed=4)
    src_t = torch.from_numpy(src).cuda()
    if variant == 'misaligned_base_pointer':
        buf = torch.empty(src.size + 1, dtype=torch.float32, device='cuda')
        src_t = buf[1:].view(src.shape)
        src_t.copy_(torch.from_numpy(src))
        assert src_t.is_contiguous() and src_t.data_ptr() % 16 == 4
        assert hkm._as_f32_plane(src_t, NAN).data_ptr() == src_t.data_ptr()
    ref_t = torch.from_numpy(ref).cuda()
    km = KernelModel(Model.gain_offset, (15, 15), find_r2=True, r2_inpaint_thresh=None)
    params, names = launched_kernels(lambda: km._fit_planes(src_t, NAN, ref_t, NAN))
    assert_ran(names, 'fit_same_grid_kernel', args=fit_variant(Model.gain_offset, True, c=4, lean=True))
    _fit_vs_oracle(params, src, NAN, ref, NAN, Model.gain_offset, (15, 15), True, None, variant)


@pytest.mark.parametrize('model, kshape, find_r2', [
    (Model.gain_offset, (1, 15), True),
    (Model.gain_blk_offset, (15, 1), True),
    (Model.gain, (1, 1), False),
])
def test_fit_c4_single_row_or_column_kernel_vs_oracle(model, kshape, find_r2):
    """ kh = 1 or kw = 1 at C = 4: general form only (the lean form needs a kernel of at least 3 x 3), NaN nodata. """
    src, ref = fit_pair(FIT_H, FIT_W, seed=5)
    km = KernelModel(model, kshape, find_r2=find_r2, r2_inpaint_thresh=None)
    src_t, ref_t = torch.from_numpy(src).cuda(), torch.from_numpy(ref).cuda()
    params, names = launched_kernels(lambda: km._fit_planes(src_t, NAN, ref_t, NAN))
    assert_ran(names, 'fit_same_grid_kernel', args=fit_variant(model, find_r2, c=4))
    _fit_vs_oracle(params, src, NAN, ref, NAN, model, kshape, find_r2, None, f'{kshape}')


def test_fit_apply_c4_uint16_output_vs_oracle():
    """ The fit fused with apply (_fit_apply_rows), general form at C = 4 (value nodata on both planes), storing a uint16
    plane with nodata 0, against the oracle's apply followed by the reference's dtype conversion. """
    _, kmnp = _oracle()
    src, ref = fit_pair(FIT_H, FIT_W, seed=6, src_dtype='uint16', src_nodata=0, ref_nodata=-9999.0)
    src_f = src.astype('float32')
    km = KernelModel(Model.gain_offset, (15, 15), r2_inpaint_thresh=None)
    s_t, r_t = torch.from_numpy(src_f).cuda(), torch.from_numpy(ref).cuda()
    out = torch.empty((FIT_H, FIT_W), dtype=torch.uint16, device='cuda')
    _, names = launched_kernels(lambda: km._fit_apply_rows(s_t, 0, r_t, -9999.0, 0, FIT_H, out=out, out_nodata=0))
    assert_ran(names, 'fit_same_grid_kernel', args=fit_variant(Model.gain_offset, False, c=4, fused=True))
    exp_params = kmnp.fit_same_grid(src_f, 0, ref, -9999.0, Model.gain_offset, (15, 15), False, None)
    expected = kmnp.convert_dtype(kmnp.apply_same_grid(src_f, exp_params), 'uint16', 0).astype('int64')
    got = out.cpu().numpy().astype('int64')
    assert np.array_equal(got == 0, expected == 0), 'nodata masks differ'
    assert np.abs(got - expected).max() <= 1
    assert (got == expected).mean() >= 0.999


@pytest.mark.parametrize('shape, c', [((2048, 2047), 1), ((2048, 2048), 4)])
def test_fit_c1_c4_switch_vs_oracle(shape, c):
    """ One plane just below the 4 M-pixel switch from one column per thread (C = 1) to four (C = 4), one at it. """
    h, w = shape
    src, ref = fit_pair(h, w, seed=7)
    km = KernelModel(Model.gain_offset, (5, 5), find_r2=True, r2_inpaint_thresh=None)
    src_t, ref_t = torch.from_numpy(src).cuda(), torch.from_numpy(ref).cuda()
    params, names = launched_kernels(lambda: km._fit_planes(src_t, NAN, ref_t, NAN))
    assert_ran(names, 'fit_same_grid_kernel', args=fit_variant(Model.gain_offset, True, c=c, lean=c == 4))
    _fit_vs_oracle(params, src, NAN, ref, NAN, Model.gain_offset, (5, 5), True, None, f'{shape}')
