"""
Deterministic synthetic source / reference raster pairs for parity tests and benchmarks (SURVEY.md section 8d).

There is no network for real imagery, so the named configurations are instantiated from a band-limited random
texture: white noise smoothed with a Gaussian (sigma = 3 proc-grid pixels) guarantees local variance inside every
kernel window, which keeps the reference's float32 least-squares solves well-conditioned (SURVEY.md 7.4-1).

    src  = clip(mu + 0.3 * mu * T_hi, lo, hi)                 T_hi = bilinear up-sample of T (+ 2 % hi-res noise)
    ref  = G * avg_down(src) + O + N(0, 0.01 * mu)            G = 0.6 + 0.2 sin(.), O = 0.05 mu cos(.)  (period ~200 px)

Source nodata: a wedge in one corner (~3 % of the area) and a few rectangular holes.  The reference is fully valid,
aligned with the source (integer ratio) and padded by one reference pixel on every side so that it encompasses the
source.  A few reference blobs are replaced by noise so that the gain-offset R2 in-painting has work to do.

Generation uses torch on ``device`` (CPU here, CUDA on the GPU box); parity tests always hand the SAME tensors to the
oracle and to the CUDA path, so cross-device RNG differences never matter.
"""
import math
from typing import Tuple

import numpy as np
import torch
import torch.nn.functional as F

from homonim_b200.geometry import Affine, CRS
from homonim_b200.raster_array import RasterArray

_DTYPES = {'uint8': (torch.uint8, 1.0, 255.0), 'uint16': (torch.uint16, 1.0, 65535.0),
           'int16': (torch.int16, -32768.0, 32767.0), 'float32': (torch.float32, -3.0e38, 3.0e38)}


def _gauss_kernel(sigma: float, device) -> torch.Tensor:
    radius = int(math.ceil(3 * sigma))
    x = torch.arange(-radius, radius + 1, dtype=torch.float32, device=device)
    k = torch.exp(-0.5 * (x / sigma) ** 2)
    return k / k.sum()


def _smooth(x: torch.Tensor, sigma: float) -> torch.Tensor:
    k = _gauss_kernel(sigma, x.device)
    r = k.numel() // 2
    x = F.pad(x[None, None], (r, r, r, r), mode='reflect')
    x = F.conv2d(x, k.view(1, 1, 1, -1))
    x = F.conv2d(x, k.view(1, 1, -1, 1))
    return x[0, 0]


def make_pair(hp: int, wp: int, ratio: int, bands: int = 1, dtype: str = 'uint16', mu: float = 3000.0, seed: int = 0,
              device='cpu', src_nodata=0.0, holes: int = 6, bad_blobs: int = 3, ref_pad: int = 1,
              src_res: float = 0.5) -> Tuple[RasterArray, RasterArray]:
    """
    Source raster of ``hp*ratio x wp*ratio`` pixels per band and its coarser reference.

    hp, wp:      proc (reference) grid size covered by the source.
    ratio:       integer source pixels per reference pixel (aligned grids).
    dtype:       source storage dtype: 'uint8', 'uint16', 'int16' or 'float32'.  int16 sources are shifted down by
                 mu / 2 per band (before the reference is derived), so that a few percent of their values are negative,
                 as in surface-reflectance products stored as int16.
    src_nodata:  source nodata value (use float('nan') for float32 sources).
    Returns (src_ra [bands, hs, ws], ref_ra [bands, hp + 2*ref_pad, wp + 2*ref_pad] float32, fully valid, nodata nan).
    """
    tdtype, lo, hi = _DTYPES[dtype]
    gen = torch.Generator(device=device)
    hs, ws = hp * ratio, wp * ratio
    yy = torch.arange(hp, dtype=torch.float32, device=device)[:, None]
    xx = torch.arange(wp, dtype=torch.float32, device=device)[None, :]
    period = 200.0
    src_planes, ref_planes = [], []
    for b in range(bands):
        gen.manual_seed(1000003 * seed + 7919 * b + 17)
        t = _smooth(torch.randn((hp, wp), generator=gen, device=device), 3.0)
        t = t / t.std()
        mu_b = mu * (1.0 + 0.15 * b)
        lo_res = mu_b + 0.3 * mu_b * t
        if ratio > 1:
            hi_res = F.interpolate(lo_res[None, None], size=(hs, ws), mode='bilinear', align_corners=False)[0, 0]
            hi_res = hi_res + 0.02 * mu_b * torch.randn((hs, ws), generator=gen, device=device)
        else:
            hi_res = lo_res + 0.02 * mu_b * torch.randn((hs, ws), generator=gen, device=device)
        if dtype == 'int16':
            hi_res = hi_res - 0.5 * mu_b
        hi_res = hi_res.clamp(lo, hi)
        if dtype != 'float32':
            hi_res = hi_res.round()
        # reference from the (valid everywhere) source surface
        avg = F.avg_pool2d(hi_res[None, None], ratio)[0, 0] if ratio > 1 else hi_res.clone()
        gain = 0.6 + 0.2 * torch.sin(2 * math.pi * (xx / period + 0.3 * yy / period) + b)
        off = 0.05 * mu_b * torch.cos(2 * math.pi * (yy / period - 0.2 * xx / period) + 0.5 * b)
        ref = gain * avg + off + 0.01 * mu_b * torch.randn((hp, wp), generator=gen, device=device)
        # decorrelated blobs: low R2 there
        for k in range(bad_blobs):
            by = int(torch.randint(0, max(hp - 12, 1), (1,), generator=gen, device=device))
            bx = int(torch.randint(0, max(wp - 12, 1), (1,), generator=gen, device=device))
            bh, bw = min(12, hp - by), min(12, wp - bx)
            ref[by:by + bh, bx:bx + bw] = mu_b * (0.5 + 0.3 * torch.randn((bh, bw), generator=gen, device=device))
        # source nodata: corner wedge + rectangular holes (at least 3 x 3 proc pixels)
        nd_mask = ((yy / hp + xx / wp) < 0.245).expand(hp, wp).clone()
        for k in range(holes):
            hy = int(torch.randint(0, max(hp - 8, 1), (1,), generator=gen, device=device))
            hx = int(torch.randint(0, max(wp - 8, 1), (1,), generator=gen, device=device))
            hh = 3 + int(torch.randint(0, 5, (1,), generator=gen, device=device))
            hw = 3 + int(torch.randint(0, 5, (1,), generator=gen, device=device))
            nd_mask[hy:hy + hh, hx:hx + hw] = True
        if ratio > 1:
            nd_hi = nd_mask.repeat_interleave(ratio, 0).repeat_interleave(ratio, 1)
        else:
            nd_hi = nd_mask
        if src_nodata is not None:
            hi_res = torch.where(nd_hi, torch.full_like(hi_res, float(src_nodata)), hi_res)
        src_planes.append(hi_res.to(tdtype))
        if ref_pad:
            ref = F.pad(ref[None, None], (ref_pad,) * 4, mode='replicate')[0, 0]
        ref_planes.append(ref.contiguous())
        del hi_res, avg, t, lo_res
    crs = CRS.from_epsg(32735)
    # north-up grids, same origin for the source and the (unpadded) proc grid
    x0, y0 = 500000.0, 6200000.0
    ref_res = src_res * ratio
    src_tf = Affine(src_res, 0.0, x0, 0.0, -src_res, y0)
    ref_tf = Affine(ref_res, 0.0, x0 - ref_pad * ref_res, 0.0, -ref_res, y0 + ref_pad * ref_res)
    src_ra = RasterArray(torch.stack(src_planes), crs, src_tf, nodata=src_nodata)
    ref_ra = RasterArray(torch.stack(ref_planes), crs, ref_tf, nodata=float('nan'))
    return src_ra, ref_ra


def to_numpy_pair(src_ra: RasterArray, ref_ra: RasterArray) -> Tuple[RasterArray, RasterArray]:
    """ Host (numpy) copies of a pair, for the oracle. """
    return src_ra.to_host(), ref_ra.to_host()
