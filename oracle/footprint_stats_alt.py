"""
oracle/footprint_stats_alt.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A second, independent restatement of the footprint statistics (min, max, med, q1, q3, mode) specified in the header
of ``oracle/footprint_stats_restate.c``, in plain numpy: a brute-force gather of each destination pixel's window and
``np.sort`` / ``np.unique``.  It shares no code with the C file; tests compare the two bit for bit.
"""
import math

import numpy as np

METHODS = ('min', 'max', 'med', 'q1', 'q3', 'mode')
_Q = {'med': 0.5, 'q1': 0.25, 'q3': 0.75}


def window(s, o, i, n):
    """ Footprint of destination index ``i`` on one axis: ``[a, b)`` clipped to ``[0, n)`` (may be empty). """
    lo, hi = s * float(i) + o, s * float(i + 1) + o
    a, b = math.floor(lo + 1e-10), math.ceil(hi - 1e-10)
    if a == b:
        b += 1
    return max(a, 0), min(b, n)


def pick(values, method):
    """ The statistic of the valid float32 ``values`` (1-D, in scan order, NaN and nodata already removed, n >= 1). """
    n = values.size
    if method == 'mode':
        uniq, inverse, counts = np.unique(values, return_inverse=True, return_counts=True)
        last = np.full(uniq.size, -1)
        last[inverse] = np.arange(n)                  # (later positions overwrite earlier ones: the last occurrence)
        top = counts == counts.max()
        return uniq[top][np.argmin(last[top])]
    v = np.sort(values)
    if method == 'min':
        return v[0]
    if method == 'max':
        return v[-1]
    return v[int(math.ceil(_Q[method] * n - 1.0))]


def footprint_stats_alt(src, nodata, dst_shape, sx, ox, sy, oy, method):
    """ float32 [hd, wd] statistic of a 2-D ``src`` (any dtype: read as float32); NaN where no value is valid. """
    src = np.asarray(src).astype('float32')
    hs, ws = src.shape
    hd, wd = dst_shape
    valid = ~np.isnan(src)
    if nodata is not None and not np.isnan(nodata):
        valid &= src != np.float32(nodata)
    out = np.full((hd, wd), np.nan, dtype='float32')
    for i in range(hd):
        y0, y1 = window(sy, oy, i, hs)
        for j in range(wd):
            x0, x1 = window(sx, ox, j, ws)
            if y1 <= y0 or x1 <= x0:
                continue
            vals = src[y0:y1, x0:x1][valid[y0:y1, x0:x1]] + np.float32(0.0)     # (-0.0 + 0.0 = +0.0)
            if vals.size:
                out[i, j] = pick(vals, method)
    return out
