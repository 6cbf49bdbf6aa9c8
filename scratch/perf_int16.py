"""int16 sources read natively against the same values stored as uint16, and against widening to float32 first.

    PYTHONPATH=. python scratch/perf_int16.py [--out DIR] [--reps 30]

One 10 000 x 10 000 band at ratio 20 (the C2 geometry: 500 x 500 reference pixels), values in [0, 32767] so that int16
and uint16 hold the same numbers, nodata 0 in the wedge and holes of synthetic.make_pair.  Timed, alternating the
dtypes launch by launch:
  * hb_downsample_average (the exact-box down-sampler for both integer dtypes);
  * hb_upsample_apply, cubic spline, float32 and int16 output (the poly fast path);
  * the whole hb_fuse_refspace call (gain-blk-offset 5 x 5);
and each of them as the composition a caller without int16 kernels would run: widen the source to float32 with torch,
then the float32 call.  CUDA events around each call, median of --reps launches, a 256 MB buffer overwritten between
launches so that no input is served from L2.  Prints the card name and power limit of the same run and one JSON line;
writes it to DIR/perf_int16.json when --out is given.  Bytes per pixel are the compulsory traffic of each call.
"""
import argparse
import json
import pathlib
import subprocess
import sys

import torch

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))

from homonim_b200 import Model, RasterArray, RefSpaceModel, _native   # noqa: E402
from homonim_b200 import kernel_model as hkm   # noqa: E402
from homonim_b200.geometry import grid_map   # noqa: E402
from homonim_b200.synthetic import make_pair   # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out')
    ap.add_argument('--reps', type=int, default=30)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    src_ra, ref_ra = make_pair(500, 500, 20, bands=1, dtype='uint16', mu=12000.0, seed=4, device=dev, src_nodata=0)
    u16 = src_ra.array[0].to(torch.int32).clamp(max=32767).to(torch.uint16).contiguous()
    i16 = u16.to(torch.int16)
    assert torch.equal(i16.to(torch.int32), u16.to(torch.int32))
    ref = ref_ra.array[0].contiguous()
    hs, ws = u16.shape
    hr, wr = ref.shape
    gm = grid_map(src_ra.transform, ref_ra.transform)
    lib = _native.lib()
    stream = torch.cuda.current_stream().cuda_stream
    km = RefSpaceModel(Model.gain_blk_offset, (5, 5))
    params = km.fit(RasterArray(u16, src_ra.crs, src_ra.transform, nodata=0),
                    RasterArray(ref, ref_ra.crs, ref_ra.transform, nodata=float('nan'))).array[:2].contiguous()
    ds = torch.empty((hr, wr), dtype=torch.float32, device=dev)
    outs = {torch.float32: torch.empty((hs, ws), dtype=torch.float32, device=dev),
            torch.int16: torch.empty((hs, ws), dtype=torch.int16, device=dev)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def downsample(t):
        _native.check(lib.hb_downsample_average(t.data_ptr(), hkm._plane_code(t), hs, ws, 1, 0.0, ds.data_ptr(), hr, wr,
                                                gm.sx, gm.ox, gm.sy, gm.oy, stream))

    def up(t, out):
        _native.check(lib.hb_upsample_apply(t.data_ptr(), hkm._plane_code(t), hs, ws, 1, 0.0, params.data_ptr(), hr, wr,
                                            1.0 / gm.sx, -gm.ox / gm.sx, 1.0 / gm.sy, -gm.oy / gm.sy, None,
                                            *hkm._out_args(out, -32768 if out.dtype == torch.int16 else float('nan')),
                                            out.data_ptr(), _native.HB_UP_CUBIC_SPLINE, stream))

    def fuse(t):
        _native.check(lib.hb_fuse_refspace(t.data_ptr(), hkm._plane_code(t), hs, ws, 1, 0.0, ref.data_ptr(), hr, wr, 1,
                                           float('nan'), gm.sx, gm.ox, gm.sy, gm.oy, _native.HB_MODEL_GAIN_BLK_OFFSET,
                                           5, 5, 0, 0, 0.0, _native.HB_F32, 0, 0.0, outs[torch.float32].data_ptr(), None,
                                           stream))

    def widened(fn):
        return lambda t, *a: fn(t.to(torch.float32), *a)

    steps = {
        'downsample_average': (downsample, ()),
        'upsample_apply_f32_out': (up, (outs[torch.float32],)),
        'upsample_apply_i16_out': (up, (outs[torch.int16],)),
        'fuse_refspace': (fuse, ()),
    }
    out_bytes = {'downsample_average': 0, 'upsample_apply_f32_out': 4, 'upsample_apply_i16_out': 2, 'fuse_refspace': 4}
    arms = {'int16': (i16, False), 'uint16': (u16, False), 'widen_f32': (i16, True)}
    result = dict(card=card(), shape=[hs, ws], ratio=20, reps=args.reps, steps={})
    for name, (fn, extra) in steps.items():
        # the fuse call reads the source twice (down-sampling, then up-sampling + apply); every other call once
        reads = 2 if name == 'fuse_refspace' else 1
        times = {arm: [] for arm in arms}
        for arm, (t, widen) in arms.items():                    # warm-up of every shape
            (widened(fn) if widen else fn)(t, *extra)
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for arm, (t, widen) in arms.items():                # alternate the arms launch by launch
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                (widened(fn) if widen else fn)(t, *extra)
                e1.record()
                e1.synchronize()
                times[arm].append(e0.elapsed_time(e1) * 1e3)
        row = {}
        for arm, ts in times.items():
            med = sorted(ts)[len(ts) // 2]
            # widening reads 2 B and writes 4 B per pixel, then the float32 call reads 4 B per pass over the source
            per_px = (2 + 4 + 4 * reads) if arm == 'widen_f32' else 2 * reads
            b = hs * ws * (per_px + out_bytes[name])
            row[arm] = dict(median_us=round(med, 1), min_us=round(min(ts), 1), max_us=round(max(ts), 1),
                            bytes_per_px=round(b / (hs * ws), 1), gbps=round(b / med / 1e3, 1))
        row['int16_vs_uint16'] = round(row['int16']['median_us'] / row['uint16']['median_us'], 4)
        row['widen_vs_int16'] = round(row['widen_f32']['median_us'] / row['int16']['median_us'], 3)
        result['steps'][name] = row
        print(name, json.dumps(row), flush=True)
    print(f'card: {result["card"]}')
    print(json.dumps(result))
    if args.out:
        pathlib.Path(args.out).mkdir(parents=True, exist_ok=True)
        (pathlib.Path(args.out) / 'perf_int16.json').write_text(json.dumps(result, indent=1))


if __name__ == '__main__':
    main()
