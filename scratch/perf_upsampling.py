"""Time the up-sampling methods: the fused up-sample + apply and plain up-sampling, per method.

    python scratch/perf_upsampling.py --out DIR [--n 25]

Per method (cubic_spline, bilinear, cubic, lanczos), with CUDA events (median of --n calls after a warm-up; the
256 MB L2 flush buffer is overwritten before each call, so every input is read from HBM):
  * RefSpaceModel.apply (hb_upsample_apply) on a 10 000^2 uint16 band at ratio 20, float32 and uint16 output;
  * the same at ratio 1.25 with a sub-pixel shift (unaligned with the coarse grid);
  * the unfused composition it replaces: _resample_plane of gain and offset to the source grid + the same-grid apply;
  * _resample_up of one 1 000^2 band to 20 000^2.
Bytes are the algorithmic ones (source pixel in + output pixel out; float32 out for plain up-sampling).  Writes
DIR/perf_upsampling.json with the card's name and power limit.
"""
import argparse
import json
import pathlib
import statistics
import subprocess
import sys

METHODS = ('cubic_spline', 'bilinear', 'cubic', 'lanczos')


def timed(fn, n, flush):
    import torch
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(n):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) * 1e3)
    return statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--n', type=int, default=25)
    args = ap.parse_args()
    import torch
    sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
    from homonim_b200 import CRS, Affine, Model, RasterArray, RefSpaceModel
    from homonim_b200 import kernel_model as hkm
    from homonim_b200.enums import Resampling
    if not torch.cuda.is_available():
        raise SystemExit('needs a GPU')
    dev = torch.device('cuda:0')
    smi = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                          '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    crs = CRS.from_epsg(3857)
    tf_lo = Affine(200, 0, 2000, 0, -200, 9_000_000)
    flush = torch.empty(256 * 2**20, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(5)
    res = {'device': torch.cuda.get_device_properties(dev).name, 'nvidia_smi': smi, 'n': args.n, 'cases': []}

    def params(hp, wp):
        yy = torch.arange(hp, device=dev, dtype=torch.float32)[:, None]
        xx = torch.arange(wp, device=dev, dtype=torch.float32)[None, :]
        gain = 0.9 + 0.1 * torch.sin(xx / 17.0) * torch.cos(yy / 13.0)
        off = 30.0 * torch.cos(xx / 11.0) + 5.0 * torch.sin(yy / 7.0)
        p = torch.stack([gain, off]).contiguous()
        p[:, hp // 2:hp // 2 + 3, wp // 3:wp // 3 + 4] = float('nan')
        return p

    for shape, (hs, ws, ratio, shift) in {'r20': (10000, 10000, 20, (0.0, 0.0)),
                                          'r1.25_shift': (10000, 10000, 1.25, (0.3, 0.2))}.items():
        src = torch.randint(1, 20000, (hs, ws), generator=g, device=dev, dtype=torch.int32).to(torch.uint16)
        hp, wp = int(-(-hs // ratio)) + 1, int(-(-ws // ratio)) + 1
        par = params(hp, wp)
        src_tf = tf_lo * Affine.scale(1.0 / ratio) * Affine.translation(*shift)
        src_ra, par_ra = RasterArray(src, crs, src_tf, nodata=0), RasterArray(par, crs, tf_lo, nodata=float('nan'))
        for method in METHODS:
            km = RefSpaceModel(Model.gain_offset, (15, 15), upsampling=method)
            for odt, ob in (('float32', 4), ('uint16', 2)):
                out = torch.empty((hs, ws), dtype=getattr(torch, odt), device=dev)
                us = timed(lambda: km.apply(src_ra, par_ra, out=out, out_nodata=0), args.n, flush)
                res['cases'].append({'case': f'apply_{shape}_{odt}', 'method': method, 'us': us,
                                     'GBps': hs * ws * (2 + ob) / us / 1e3})
            # the unfused composition: up-sampled parameters in memory, then the same-grid apply
            out = torch.empty((hs, ws), dtype=torch.float32, device=dev)

            def unfused():
                par_us = torch.stack([hkm._resample_plane(par[b], tf_lo, float('nan'), (hs, ws), src_tf,
                                                          Resampling(method)) for b in range(2)])
                hkm.KernelModel._apply_planes(src, 0, par_us, mask_src=True, out=out)
            us = timed(unfused, args.n, flush)
            res['cases'].append({'case': f'unfused_{shape}_float32', 'method': method, 'us': us,
                                 'GBps': hs * ws * (2 + 4) / us / 1e3})
            print(json.dumps(res['cases'][-3:]), flush=True)
        del src, par
    coarse = params(1000, 1000)[:1].contiguous()
    dst_tf = tf_lo * Affine.scale(1.0 / 20)
    for method in METHODS:
        code = hkm._UP_METHODS[Resampling(method)]
        us = timed(lambda: hkm._resample_up(coarse, tf_lo, float('nan'), (20000, 20000), dst_tf, code), args.n, flush)
        res['cases'].append({'case': 'resample_up_1000_to_20000', 'method': method, 'us': us,
                             'GBps': 20000 * 20000 * 4 / us / 1e3})
        print(json.dumps(res['cases'][-1]), flush=True)
    out_dir = pathlib.Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    (out_dir / 'perf_upsampling.json').write_text(json.dumps(res, indent=1))
    print(smi)


if __name__ == '__main__':
    main()
