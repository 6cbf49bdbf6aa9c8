"""
oracle/interp_up_alt.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A second, independent restatement of GDAL's bilinear, cubic and lanczos UP-sampling (``rasterio.warp.reproject`` with a
destination at least as fine as the source), written from the rules below rather than from
oracle/interp_up_restate.c, to catch transcription errors in the latter (GDAL itself cannot be installed in this
image: parity with GDAL is UNPINNED for these methods).  Vectorised over destination pixels, one tap at a time; numpy only, for small rasters.

The rules (notation of oracle/interp_up_restate.c: src_x = sx (j + 0.5) + ox, k = floor(src_x - 0.5),
d = src_x - 0.5 - k, the same in y; nb bands share a "unified" validity = valid in any band):
  * centre rule: the source pixel containing the destination centre (floor(src + 1e-10), the last pixel when it falls
    exactly on the far edge) must be in range and valid in at least one band, else the pixel is nodata;
  * a tap counts only when it is in range and valid in its own band; every decision is taken per band;
  * bilinear: taps k, k+1 per axis, weights (1 - d, d); valid taps summed UL, UR, LR, LL; nodata if the weight sum is
    < 1e-5, unchanged if it is exactly 1.0, else divided by it;
  * cubic: taps k-1 .. k+2, Keys (a = -0.5) weights, each row convolved in x then the rows in y, no normalisation;
    when the 4 x 4 footprint leaves the raster or has an invalid tap in the band: exactly the bilinear result;
  * lanczos: taps k-2 .. k+3, weights L(i - d), L(0) = 1, L(t) = sin(pi t) sin(pi t / 3) / (pi^2 t^2 / 3) for
    0 < |t| < 3, else 0; valid taps of each row summed in x (values and weights), then the rows in y; nodata if the
    weight sum is < 1e-6, divided by it when outside [0.99999, 1.00001].
Accumulation in double, result stored as float32; nodata pixels hold ``dst_nodata``.
"""
import math

import numpy as np


def _axis(n_dst, scale, off):
    src = scale * (np.arange(n_dst, dtype='float64') + 0.5) + off
    k = np.floor(src - 0.5)
    return src, k.astype('int64'), src - 0.5 - k


def _centre(src, n):
    c = np.floor(src + 1e-10).astype('int64')
    c = np.where(c == n, c - 1, c)
    return c, (src >= 0.0) & (c >= 0) & (c < n)


def _keys(d):
    return [0.5 * d * (-1.0 + d * (2.0 - d)), 1.0 + 0.5 * d * d * (-5.0 + 3.0 * d), 0.5 * d * (1.0 + d * (4.0 - 3.0 * d)),
            0.5 * d * d * (-1.0 + d)]


def _lanczos(t):
    t = np.asarray(t, dtype='float64')
    out = np.zeros_like(t)
    inner = (t != 0.0) & (np.abs(t) < 3.0)
    pt = math.pi * t[inner]
    out[inner] = np.sin(pt) * np.sin(pt / 3.0) / (pt * pt / 3.0)
    out[t == 0.0] = 1.0
    return out


def interp_up_alt(src, nodata, dst_shape, sx, ox, sy, oy, method, dst_nodata=np.nan):
    """ ``src``: [nb, hs, ws] (or 2D); (sx, ox, sy, oy) maps destination to source pixel-edge coordinates. """
    src = np.asarray(src, dtype='float64')
    squeeze = src.ndim == 2
    src = src[None] if squeeze else src
    nb, hs, ws = src.shape
    hd, wd = dst_shape
    if sx > 1.0 + 1e-12 or sy > 1.0 + 1e-12:
        raise NotImplementedError('up-sampling only')
    valid = np.ones(src.shape, bool) if nodata is None else (
        ~np.isnan(src) if np.isnan(nodata) else src != nodata)
    src_y, ky, dy = _axis(hd, sy, oy)
    src_x, kx, dx = _axis(wd, sx, ox)
    Y, X = np.meshgrid(np.arange(hd), np.arange(wd), indexing='ij')
    KY, KX, DY, DX = ky[Y], kx[X], dy[Y], dx[X]
    cy, oky = _centre(src_y, hs)
    cx, okx = _centre(src_x, ws)
    CY, CX = np.clip(cy[Y], 0, hs - 1), np.clip(cx[X], 0, ws - 1)
    centre_ok = oky[Y] & okx[X] & valid.any(axis=0)[CY, CX]

    def tap(b, ty, tx):
        """ value (0 where not counted) and whether the tap counts """
        inr = (ty >= 0) & (ty < hs) & (tx >= 0) & (tx < ws)
        yy, xx = np.clip(ty, 0, hs - 1), np.clip(tx, 0, ws - 1)
        ok = inr & valid[b][yy, xx]
        return np.where(ok, src[b][yy, xx], 0.0), ok

    def bilinear(b):
        acc = np.zeros((hd, wd))
        acc_w = np.zeros((hd, wd))
        for oy_, ox_, wy, wx in ((0, 0, 1 - DY, 1 - DX), (0, 1, 1 - DY, DX), (1, 1, DY, DX), (1, 0, DY, 1 - DX)):
            v, ok = tap(b, KY + oy_, KX + ox_)
            w = wx * wy
            acc_w = np.where(ok, acc_w + w, acc_w)
            acc = np.where(ok, acc + v * w, acc)
        good = acc_w >= 0.00001
        res = np.where(acc_w == 1.0, acc, acc / np.where(good, acc_w, 1.0))
        return res, good

    out = np.full((nb, hd, wd), dst_nodata, dtype='float32')
    for b in range(nb):
        if method == 'bilinear':
            res, good = bilinear(b)
        elif method == 'cubic':
            bil, bil_good = bilinear(b)
            cwx, cwy = _keys(DX), _keys(DY)
            full = np.ones((hd, wd), bool)
            rows = []
            for tj in range(4):
                r = np.zeros((hd, wd))
                terms = []
                for ti in range(4):
                    v, ok = tap(b, KY - 1 + tj, KX - 1 + ti)
                    full &= ok
                    terms.append(cwx[ti] * v)
                r = ((terms[0] + terms[1]) + terms[2]) + terms[3]
                rows.append(r)
            cub = ((cwy[0] * rows[0] + cwy[1] * rows[1]) + cwy[2] * rows[2]) + cwy[3] * rows[3]
            res = np.where(full, cub, bil)
            good = full | bil_good
        elif method == 'lanczos':
            lwx = [_lanczos(i - DX) for i in range(-2, 4)]
            lwy = [_lanczos(i - DY) for i in range(-2, 4)]
            acc = np.zeros((hd, wd))
            acc_w = np.zeros((hd, wd))
            for tj in range(6):
                r = np.zeros((hd, wd))
                r_w = np.zeros((hd, wd))
                for ti in range(6):
                    v, ok = tap(b, KY - 2 + tj, KX - 2 + ti)
                    r = np.where(ok, r + v * lwx[ti], r)
                    r_w = np.where(ok, r_w + lwx[ti], r_w)
                acc = acc + r * lwy[tj]
                acc_w = acc_w + r_w * lwy[tj]
            good = acc_w >= 0.000001
            norm = (acc_w < 0.99999) | (acc_w > 1.00001)
            res = np.where(norm, acc / np.where(good, acc_w, 1.0), acc)
        else:
            raise NotImplementedError(method)
        keep = centre_ok & good
        out[b][keep] = res[keep].astype('float32')
    return out[0] if squeeze else out
