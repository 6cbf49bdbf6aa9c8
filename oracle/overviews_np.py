"""
Numpy restatement of the overview pyramid (reference fuse.py:151-165: RasterFuse._build_overviews, average resampling,
factors 2, 4, ..., 2^L) under the pixel rule of DESIGN.md section 7, written window by window from the rule itself and
independent of the product's code: the checker of ``hb_build_overviews`` and of the overviews in written files.

Level k is computed from level k - 1 as stored (level 0 = the written plane).  Pixel (i, j) of level k averages the valid
pixels among rows 2i, 2i+1 and columns 2j, 2j+1 of level k - 1; rows / columns past an odd edge are absent.  Valid = not
nodata (when there is one) and, in float planes, not NaN.  No valid pixel -> nodata (NaN for float without one).
Integer planes: floor((2s + n) / 2n) of the exact sum s of the n valid pixels.  float32: the valid values summed in
float64 in the order top-left, top-right, bottom-left, bottom-right, divided by n in float64, rounded once to float32.
"""
import math

import numpy as np


def overview_factors(shape, max_num_levels=8, min_level_pixels=256):
    """ Reference fuse.py:155-158. """
    num_levels = min(max_num_levels, int(np.log2(min(shape) / min_level_pixels)))
    return [2 ** m for m in range(1, num_levels + 1)]


def _valid(values, nodata):
    values = np.asarray(values)
    valid = np.ones(values.shape, bool)
    if values.dtype.kind == 'f':
        valid &= ~np.isnan(values)
        if nodata is not None and not math.isnan(nodata):
            valid &= values != np.float32(nodata)
    elif nodata is not None and not math.isnan(nodata) and float(nodata).is_integer():
        info = np.iinfo(values.dtype)
        if info.min <= nodata <= info.max:
            valid &= values.astype('int64') != int(nodata)
    return valid


def _fill(dtype, nodata):
    if np.dtype(dtype).kind == 'f':
        return np.float32('nan') if nodata is None else np.float32(nodata)
    return 0 if nodata is None or math.isnan(nodata) else int(nodata)


def next_level(plane, nodata):
    """ One 2x reduction of a 2D plane under the rule above (vectorised over the four window positions). """
    plane = np.asarray(plane)
    h, w = plane.shape
    ho, wo = -(-h // 2), -(-w // 2)
    # the four window positions, padded with "absent" past the edges
    vals = np.zeros((4, ho, wo), dtype=plane.dtype)
    ok = np.zeros((4, ho, wo), dtype=bool)
    for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):       # TL, TR, BL, BR
        part = plane[dy::2, dx::2]
        vals[k, :part.shape[0], :part.shape[1]] = part
        ok[k, :part.shape[0], :part.shape[1]] = _valid(part, nodata)
    n = ok.sum(axis=0)
    fill = _fill(plane.dtype, nodata)
    if plane.dtype.kind == 'f':
        s = np.zeros((ho, wo), dtype='float64')
        for k in range(4):                                  # row-major order, one float64 add per valid pixel
            s = np.where(ok[k], s + vals[k].astype('float64'), s)
        with np.errstate(invalid='ignore', divide='ignore'):
            out = (s / np.maximum(n, 1)).astype('float32')
        return np.where(n > 0, out, np.float32(fill)).astype(plane.dtype)
    s = np.where(ok, vals.astype('int64'), 0).sum(axis=0)
    out = np.floor_divide(2 * s + n, 2 * np.maximum(n, 1))
    return np.where(n > 0, out, fill).astype(plane.dtype)


def next_level_loops(plane, nodata):
    """ The same reduction written as explicit per-window loops (slow: small planes only). """
    plane = np.asarray(plane)
    h, w = plane.shape
    out = np.empty((-(-h // 2), -(-w // 2)), dtype=plane.dtype)
    valid = _valid(plane, nodata)
    for i in range(out.shape[0]):
        for j in range(out.shape[1]):
            window = [(y, x) for y in (2 * i, 2 * i + 1) for x in (2 * j, 2 * j + 1) if y < h and x < w and valid[y, x]]
            if not window:
                out[i, j] = _fill(plane.dtype, nodata)
            elif plane.dtype.kind == 'f':
                s = 0.0
                for y, x in window:
                    s += float(plane[y, x])
                out[i, j] = np.float32(s / len(window))
            else:
                s, n = sum(int(plane[y, x]) for y, x in window), len(window)
                out[i, j] = (2 * s + n) // (2 * n)
    return out


def build_overviews(plane, nodata, n_levels, reduce=next_level):
    """ Levels 1..n_levels of a [H, W] or [B, H, W] plane, each computed from the previous one as stored. """
    plane = np.asarray(plane)
    if plane.ndim == 3:
        per_band = [build_overviews(b, nodata, n_levels, reduce) for b in plane]
        return [np.stack([lv[k] for lv in per_band]) for k in range(n_levels)]
    levels, cur = [], plane
    for _ in range(n_levels):
        cur = reduce(cur, nodata)
        levels.append(cur)
    return levels
