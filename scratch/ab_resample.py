"""Compare two builds of the library bit for bit on the resampling entry points.

    python scratch/ab_resample.py --out DIR --ab OLD.so NEW.so

Each build runs in its own process (HOMONIM_B200_LIB selects the library) on the same seeded inputs (numpy, generated
on the host) and saves every output; the parent then compares the outputs byte for byte.  Cases:
  * hb_upsample_apply: cubic spline, bilinear, cubic, lanczos x uint8 / uint16 / float32 sources x a width that is a
    multiple of 4 and one that is not x ratios 1.25, 2, 20 x without / with a coverage mask.  Cubic spline at ratios 2
    and 20 on the aligned width without a mask takes the fast paths (pre-pass, poly / y-first kernels, DIRTY-cell
    fix-up); everything else takes the general kernel;
  * hb_resample_up: 1 and 2 bands, every method including nearest, the same ratios and widths (one band of cubic
    spline on the aligned width at ratios 2 and 20 takes the double-precision y-first kernel);
  * hb_downsample_average: integer ratios on aligned grids (the integer-aligned kernel for uint8 / uint16) and a
    fractional, shifted ratio (the general kernel), every source dtype;
  * hb_resample_stat: min, max, med, q1, q3, mode at ratio 2.5 (one thread per pixel) and 12 (one warp per pixel);
  * hb_full_coverage_mask: an integer and a fractional, shifted ratio, two kernel shapes.
The coarse parameter planes carry NaN holes (DIRTY and DEAD cells) and a patch of -0.0 (signed zeros must survive).
Writes DIR/ab_resample.json: per case the SHA-256 of both builds' output and the number of differing bytes.
"""
import argparse
import hashlib
import json
import os
import pathlib
import subprocess
import sys
import tempfile

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
U8, U16, F32 = 0, 1, 2
UP = {'cubic_spline': 0, 'nearest': 1, 'bilinear': 2, 'cubic': 3, 'lanczos': 4}
STAT = {'min': 0, 'max': 1, 'med': 2, 'q1': 3, 'q3': 4, 'mode': 5}
NP = {U8: np.uint8, U16: np.uint16, F32: np.float32}


def source(rng, dtype, h, w):
    """ a source plane with a nodata patch and scattered nodata pixels; returns (array, nodata) """
    if dtype == F32:
        a = (rng.random((h, w), dtype=np.float32) * 0.5 + 0.05).astype(np.float32)
        nd = float('nan')
    else:
        a = rng.integers(1, 255 if dtype == U8 else 20000, (h, w)).astype(NP[dtype])
        nd = 0
    a[h // 3:h // 3 + 7, w // 4:w // 4 + 9] = nd
    a.reshape(-1)[rng.integers(0, h * w, h * w // 200)] = nd
    return a, nd


def params(rng, nb, hp, wp):
    """ smooth coarse bands with NaN holes and a -0.0 patch """
    yy, xx = np.mgrid[0:hp, 0:wp].astype(np.float32)
    g = 0.9 + 0.1 * np.sin(xx / 7.0) * np.cos(yy / 5.0) + 0.01 * rng.random((hp, wp), dtype=np.float32)
    o = 3.0 * np.cos(xx / 5.0 + yy / 9.0)
    p = np.stack([g, o])[:nb].astype(np.float32)
    p[:, hp // 2:hp // 2 + 2, wp // 2:wp // 2 + 3] = np.nan
    p[0, 1, 2] = np.nan
    if nb > 1:
        p[1, hp - 2, 1] = np.nan
    p[:, 0:2, wp - 3:wp - 1] = -0.0
    return np.ascontiguousarray(p)


def run_cases(out_path):
    import torch
    sys.path.insert(0, str(ROOT))
    from homonim_b200 import _native
    lib = _native.lib()
    dev = torch.device('cuda:0')

    def dev_t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    def call(name, *args):
        _native.check(getattr(lib, name)(*args), name)

    outs = {}
    rng = np.random.default_rng(20261022)
    hs = 240
    for ws in (1200, 1203):
        for ratio in (1.25, 2.0, 20.0):
            hp, wp = int(np.ceil(hs / ratio)), int(np.ceil(ws / ratio))
            sx = sy = 1.0 / ratio
            p2 = dev_t(params(rng, 2, hp, wp))
            cover = dev_t((rng.random((hp, wp)) < 0.9).astype(np.uint8))
            for dtype in (U8, U16, F32):
                src, nd = source(rng, dtype, hs, ws)
                src_t = dev_t(src)
                for method in ('cubic_spline', 'bilinear', 'cubic', 'lanczos'):
                    for cov in (False, True):
                        out = torch.empty((hs, ws), dtype=torch.float32, device=dev)
                        call('hb_upsample_apply', src_t.data_ptr(), dtype, hs, ws, 1, float(nd), p2.data_ptr(), hp, wp,
                             sx, 0.0, sy, 0.0, cover.data_ptr() if cov else None, F32, 0, 0.0, out.data_ptr(),
                             UP[method], None)
                        outs[f'apply/{method}/{NP[dtype].__name__}/w{ws}/r{ratio}/cover{int(cov)}'] = out
            for nb in (1, 2):
                p = dev_t(params(rng, nb, hp, wp))
                for method in UP:
                    out = torch.empty((nb, hs, ws), dtype=torch.float32, device=dev)
                    call('hb_resample_up', p.data_ptr(), nb, hp, wp, 1, float('nan'), out.data_ptr(), hs, ws, sx, 0.0,
                         sy, 0.0, UP[method], None)
                    outs[f'resample_up/{method}/nb{nb}/w{ws}/r{ratio}'] = out
    # down-sampling: (ratio, offset) -- integer ratios on aligned grids, a fractional ratio with a shift
    hs, ws = 960, 1280
    for ratio, off in ((8.0, 0.0), (16.0, 0.0), (3.7, 0.3)):
        hd, wd = int((hs - off) // ratio), int((ws - off) // ratio)
        for dtype in (U8, U16, F32):
            src, nd = source(rng, dtype, hs, ws)
            src_t = dev_t(src)
            out = torch.empty((hd, wd), dtype=torch.float32, device=dev)
            call('hb_downsample_average', src_t.data_ptr(), dtype, hs, ws, 1, float(nd), out.data_ptr(), hd, wd, ratio,
                 off, ratio, off, None)
            outs[f'downsample_average/{NP[dtype].__name__}/r{ratio}'] = out
    for ratio, off in ((2.5, 0.25), (12.0, 0.0)):
        hd, wd = int((hs - off) // ratio), int((ws - off) // ratio)
        for dtype in (U8, U16, F32):
            src, nd = source(rng, dtype, hs, ws)
            src_t = dev_t(src)
            for method in STAT:
                out = torch.empty((hd, wd), dtype=torch.float32, device=dev)
                call('hb_resample_stat', src_t.data_ptr(), dtype, hs, ws, 1, float(nd), out.data_ptr(), hd, wd, ratio,
                     off, ratio, off, STAT[method], None)
                outs[f'resample_stat/{method}/{NP[dtype].__name__}/r{ratio}'] = out
    for ratio, off in ((20.0, 0.0), (7.3, -0.4)):
        hp, wp = int(np.ceil(hs / ratio)), int(np.ceil(ws / ratio))
        mask = dev_t((rng.random((hs, ws)) < 0.999).astype(np.uint8))
        p = dev_t(params(rng, 2, hp, wp))
        for kh, kw in ((1, 1), (3, 5)):
            out = torch.empty((hp, wp), dtype=torch.uint8, device=dev)
            work = torch.empty((hp, wp), dtype=torch.uint8, device=dev)
            call('hb_full_coverage_mask', mask.data_ptr(), hs, ws, p.data_ptr(), hp, wp, ratio, off, ratio, off, kh, kw,
                 out.data_ptr(), work.data_ptr(), None)
            outs[f'full_coverage_mask/r{ratio}/k{kh}x{kw}'] = out
    torch.cuda.synchronize()
    np.savez(out_path, **{k.replace('/', '|'): v.cpu().numpy() for k, v in outs.items()})
    print(f'{len(outs)} outputs -> {out_path}', flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, metavar='DIR', help='directory the JSON result is written to')
    ap.add_argument('--ab', nargs=2, metavar=('OLD', 'NEW'))
    ap.add_argument('--save', help=argparse.SUPPRESS)   # (child: where to save this build's outputs)
    a = ap.parse_args()
    if a.save:
        run_cases(a.save)
        return
    if not a.ab:
        raise SystemExit('--ab OLD.so NEW.so is required')
    out_dir = pathlib.Path(a.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        for tag, lib in zip(('old', 'new'), a.ab):
            subprocess.run([sys.executable, __file__, '--out', str(out_dir), '--save', f'{tmp}/{tag}.npz'], check=True,
                           env=dict(os.environ, HOMONIM_B200_LIB=str(pathlib.Path(lib).resolve())))
        old, new = np.load(f'{tmp}/old.npz'), np.load(f'{tmp}/new.npz')
        assert sorted(old.files) == sorted(new.files)
        for k in old.files:
            bo, bn = old[k].tobytes(), new[k].tobytes()
            diff = int(np.count_nonzero(np.frombuffer(bo, np.uint8) != np.frombuffer(bn, np.uint8)))
            res[k.replace('|', '/')] = {'sha256_old': hashlib.sha256(bo).hexdigest(),
                                        'sha256_new': hashlib.sha256(bn).hexdigest(), 'bytes_differing': diff,
                                        'nan_share': float(np.mean(np.isnan(new[k]))) if new[k].dtype == np.float32
                                        else None}
    n_diff = sum(1 for r in res.values() if r['bytes_differing'])
    summary = {'cases': len(res), 'cases_differing': n_diff, 'results': res}
    (out_dir / 'ab_resample.json').write_text(json.dumps(summary, indent=1))
    print(f'{len(res)} cases, {n_diff} differing')
    for k, r in res.items():
        if r['bytes_differing']:
            print('  DIFFERS', k, r['bytes_differing'])
    if n_diff:
        raise SystemExit(1)


if __name__ == '__main__':
    main()
