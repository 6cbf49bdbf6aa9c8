"""Time the footprint statistics (hb_resample_stat) beside the average down-sampler on the same inputs.

    python scratch/perf_footprint_stats.py --out DIR [--n 25]

Shapes: 10 000^2 uint16 at ratio 20 (the C2 band), 10 000^2 float32 at ratio 20, 1 425 x 807 uint8 at ratio 2
(C1-sized) and 12 000^2 uint16 at ratio 60.  Per shape, hb_downsample_average and hb_resample_stat for min, max, med,
q1, q3 and mode, with CUDA events: the median of --n launches after a warm-up, a 256 MB buffer overwritten before
every launch so that each input is read from HBM, not L2.  Bytes are the algorithmic ones: the source dtype's size per
source pixel plus 4 B per destination pixel.  Writes DIR/perf_footprint_stats.json with the card's name and power limit.
"""
import argparse
import json
import pathlib
import statistics
import subprocess
import sys

METHODS = ('min', 'max', 'med', 'q1', 'q3', 'mode')


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
    from homonim_b200 import _native
    from homonim_b200 import kernel_model as hkm
    if not torch.cuda.is_available():
        raise SystemExit('needs a GPU')
    dev = torch.device('cuda:0')
    smi = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                          '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 * 2**20, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(7)
    res = {'device': torch.cuda.get_device_properties(dev).name, 'nvidia_smi': smi, 'n': args.n, 'cases': []}
    codes = {'uint8': _native.HB_U8, 'uint16': _native.HB_U16, 'float32': _native.HB_F32}
    sizes = {'uint8': 1, 'uint16': 2, 'float32': 4}
    shapes = [('C2_uint16_r20', 10000, 10000, 'uint16', 20), ('float32_r20', 10000, 10000, 'float32', 20),
              ('C1_uint8_r2', 1425, 807, 'uint8', 2), ('uint16_r60', 12000, 12000, 'uint16', 60)]
    for name, hs, ws, dtype, ratio in shapes:
        if dtype == 'float32':
            src = (300.0 + 80.0 * torch.randn((hs, ws), generator=g, device=dev)).contiguous()
        else:
            hi = 255 if dtype == 'uint8' else 4000
            src = torch.randint(1, hi, (hs, ws), generator=g, device=dev, dtype=torch.int32).to(getattr(torch, dtype))
        hd, wd = hs // ratio, ws // ratio
        dst = torch.empty((hd, wd), dtype=torch.float32, device=dev)
        nbytes = hs * ws * sizes[dtype] + hd * wd * 4
        st = hkm._stream()

        def average():
            hkm._call('hb_downsample_average', src.data_ptr(), codes[dtype], hs, ws, 1, 0.0, dst.data_ptr(), hd, wd,
                      float(ratio), 0.0, float(ratio), 0.0, st)

        def stat(code):
            return lambda: hkm._call('hb_resample_stat', src.data_ptr(), codes[dtype], hs, ws, 1, 0.0, dst.data_ptr(),
                                     hd, wd, float(ratio), 0.0, float(ratio), 0.0, code, st)

        for method, fn in [('average', average)] + [(m, stat(hkm._STAT_METHODS[hkm.Resampling(m)])) for m in METHODS]:
            us = timed(fn, args.n, flush)
            res['cases'].append({'shape': name, 'method': method, 'us': round(us, 2),
                                 'GBps': round(nbytes / us / 1e3, 1)})
            print(json.dumps(res['cases'][-1]), flush=True)
        del src, dst
    out_dir = pathlib.Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    (out_dir / 'perf_footprint_stats.json').write_text(json.dumps(res, indent=1))
    print(smi)


if __name__ == '__main__':
    main()
