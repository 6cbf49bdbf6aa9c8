"""Time hb_upsample_apply and upsample_poly_kernel alone on the shapes the fused up-sample + apply runs at.

    python scratch/perf_poly.py --out DIR [--n 25]                    # the library the package loads
    python scratch/perf_poly.py --out DIR --ab OLD.so NEW.so [--rounds 3]   # two builds alternating, bits compared

One measurement per process (HOMONIM_B200_LIB selects the library).  Per shape: hb_upsample_apply timed with CUDA events
(median of --n launches after a warm-up; every input is larger than L2 or L2 is overwritten before each launch), and the
poly kernel's own duration from torch.profiler (median over the same number of launches, a separate pass).  Bytes are
the algorithmic ones: source pixels read once, output pixels written once.  The output's SHA-256 lets --ab check that
two builds compute the same bits.  Results go to DIR/perf_poly_<tag>.json; --ab also writes DIR/perf_poly_ab.json.
"""
import argparse
import hashlib
import json
import os
import pathlib
import re
import statistics
import subprocess
import sys

HBM_TBS = 7.7          # B200 data sheet, one GPU
# name: (dtype, rows, cols, ratio, output dtype)
SHAPES = {
    'c2_u16_f32': ('uint16', 10000, 10000, 20, 'float32'),    # bench.py c2 band
    'c2_u16_u16': ('uint16', 10000, 10000, 20, 'uint16'),     # same band, uint16 output (conversion fused in the store)
    'c4_u16_f32': ('uint16', 8000, 8000, 20, 'float32'),      # bench.py c4 band
    'c5a_f32_f32': ('float32', 1024, 60000, 20, 'float32'),   # one row band of a 60 000-wide float32 raster (c5a)
    'u8_u8': ('uint8', 10000, 10000, 20, 'uint8'),            # uint8 source -> uint8 output
}


def measure(out_dir, tag, n):
    import torch
    sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
    from homonim_b200 import CRS, Affine, Model, RasterArray, RefSpaceModel
    dev = torch.device('cuda:0')
    props = torch.cuda.get_device_properties(dev)
    smi = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                          '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    crs = CRS.from_epsg(3857)
    tf_lo = Affine(200, 0, 2000, 0, -200, 9_000_000)
    km = RefSpaceModel(Model.gain_offset, (15, 15))
    l2_flush = torch.empty(256 * 2**20, dtype=torch.uint8, device=dev)
    res = {'tag': tag, 'lib': os.environ.get('HOMONIM_B200_LIB', 'default'), 'device': props.name, 'nvidia_smi': smi,
           'shapes': {}}
    for name, (dtype, hs, ws, ratio, odt) in SHAPES.items():
        g = torch.Generator(device=dev).manual_seed(5)
        hp, wp = -(-hs // ratio), -(-ws // ratio)
        if dtype == 'float32':
            src = torch.rand((hs, ws), generator=g, device=dev) * 0.5 + 0.05
            nodata = float('nan')
        else:
            hi = 255 if dtype == 'uint8' else 20000
            src = torch.randint(1, hi, (hs, ws), generator=g, device=dev, dtype=torch.int32).to(getattr(torch, dtype))
            nodata = 0
        src[hs // 3:hs // 3 + 40, ws // 4:ws // 4 + 90] = nodata
        yy = torch.arange(hp, device=dev, dtype=torch.float32)[:, None]
        xx = torch.arange(wp, device=dev, dtype=torch.float32)[None, :]
        gain = (0.9 + 0.1 * torch.sin(xx / 17.0) * torch.cos(yy / 13.0)
                + 0.01 * torch.rand((hp, wp), generator=g, device=dev))
        off = (5.0 if dtype != 'float32' else 0.01) * torch.cos(xx / 11.0 + yy / 23.0)
        params = torch.stack([gain, off.expand(hp, wp)]).contiguous()
        params[:, hp // 2:hp // 2 + 3, wp // 2:wp // 2 + 4] = float('nan')          # a few DIRTY / DEAD cells
        src_tf = tf_lo * Affine.scale(1.0 / ratio)
        sra = RasterArray(src, crs, src_tf, nodata=nodata)
        pra = RasterArray(params, crs, tf_lo, nodata=float('nan'))
        out = torch.empty((hs, ws), dtype=getattr(torch, odt), device=dev)
        out_nd = float('nan') if odt == 'float32' else 0

        def run():
            km.apply(sra, pra, out=out, out_nodata=out_nd)
        small = hs * ws * (src.element_size() + out.element_size()) < 2 * 126e6
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        ts = []
        for _ in range(n):
            if small:
                l2_flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                if small:
                    l2_flush.zero_()
                run()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.events():
            m = re.search(r'(upsample_\w+)', ev.name)
            if ev.device_type.name == 'CUDA' and m:
                key = m.group(1)
                kern.setdefault(key, []).append(ev.device_time if hasattr(ev, 'device_time') else ev.cuda_time)
        nbytes = hs * ws * (src.element_size() + out.element_size())
        poly = statistics.median(kern.get('upsample_poly_kernel', [float('nan')]))
        apply_us = statistics.median(ts)
        digest = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()
        res['shapes'][name] = {
            'src': dtype, 'out': odt, 'shape': [hs, ws], 'ratio': ratio, 'bytes': nbytes,
            'apply_us': round(apply_us, 2), 'apply_gbs': round(nbytes / apply_us / 1e3, 1),
            'poly_us': round(poly, 2), 'poly_gbs': round(nbytes / poly / 1e3, 1),
            'poly_share_of_hbm': round(nbytes / poly / 1e6 / HBM_TBS, 3),
            'kernels_us': {k: round(statistics.median(v), 2) for k, v in kern.items()},
            'sha256': digest}
        print(name, json.dumps(res['shapes'][name]), flush=True)
    out_dir.mkdir(parents=True, exist_ok=True)
    (out_dir / f'perf_poly_{tag}.json').write_text(json.dumps(res, indent=1))
    print(res['device'], '|', smi)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, metavar='DIR', help='directory the JSON results are written to')
    ap.add_argument('--n', type=int, default=25)
    ap.add_argument('--tag', default='run')
    ap.add_argument('--ab', nargs=2, metavar=('OLD', 'NEW'))
    ap.add_argument('--rounds', type=int, default=3)
    a = ap.parse_args()
    out_dir = pathlib.Path(a.out)
    if not a.ab:
        measure(out_dir, a.tag, a.n)
        return
    runs = {'old': [], 'new': []}
    for i in range(a.rounds):
        for tag, lib in (('old', a.ab[0]), ('new', a.ab[1])):
            t = f'{tag}{i}'
            subprocess.run([sys.executable, __file__, '--out', str(out_dir), '--n', str(a.n), '--tag', t], check=True,
                           env=dict(os.environ, HOMONIM_B200_LIB=str(pathlib.Path(lib).resolve())))
            runs[tag].append(json.loads((out_dir / f'perf_poly_{t}.json').read_text()))
    summary = {'device': runs['new'][0]['device'], 'nvidia_smi': runs['new'][0]['nvidia_smi'], 'shapes': {}}
    for name in SHAPES:
        row = {}
        for tag in ('old', 'new'):
            for k in ('apply_us', 'poly_us'):
                row[f'{k}_{tag}'] = statistics.median(r['shapes'][name][k] for r in runs[tag])
        nbytes = runs['new'][0]['shapes'][name]['bytes']
        row['poly_gbs_new'] = round(nbytes / row['poly_us_new'] / 1e3, 1)
        row['poly_share_of_hbm_new'] = round(nbytes / row['poly_us_new'] / 1e6 / HBM_TBS, 3)
        digests = {r['shapes'][name]['sha256'] for tag in runs for r in runs[tag]}
        row['identical_outputs'] = len(digests) == 1
        summary['shapes'][name] = row
        print(name, json.dumps(row))
    (out_dir / 'perf_poly_ab.json').write_text(json.dumps(summary, indent=1))
    if not all(r['identical_outputs'] for r in summary['shapes'].values()):
        raise SystemExit('outputs differ between the builds')


if __name__ == '__main__':
    main()
