"""
Cost of the output overviews (RasterFuse.process(..., build_ovw=True)).
usage: python scratch/perf_overviews.py [repeats=3]

1. The pyramid kernel alone (hb_build_overviews, CUDA events around each launch, median of 20): a 5000^2 uint16 band with
   4 levels (the plane fits the 126 MB L2, so a 512 MB buffer is overwritten before every timed launch), and 20000^2
   uint16 / float32 planes with 6 levels (larger than L2, no flush).  Bytes = one read of the plane + the levels written.
2. File -> file on the perf_files.py workload (4-band uint16 5000^2 source, gain-offset 15 x 15): deflate float32 output
   and uncompressed uint16 output, build_ovw=False / True alternating in one run, median wall time of `repeats` each.
"""
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, '.')
from homonim_b200 import Model, RasterFuse   # noqa: E402
from homonim_b200.geotiff import GeoTiffReader, write_geotiff   # noqa: E402
from homonim_b200.overviews import build_overviews, level_shape   # noqa: E402
from homonim_b200.synthetic import make_pair   # noqa: E402

repeats = int(sys.argv[1]) if len(sys.argv) > 1 else 3
assert torch.cuda.is_available(), 'needs a CUDA device'
smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                     capture_output=True, text=True).stdout.strip()
print(f'device: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi}')

# ---- 1. kernel ------------------------------------------------------------------------------------------------------
flush = torch.empty(512 << 20, dtype=torch.uint8, device='cuda')


def time_kernel(plane, nodata, levels, flush_l2, n=20):
    for _ in range(3):
        build_overviews(plane, nodata, levels)
    times = []
    for _ in range(n):
        if flush_l2:
            flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        build_overviews(plane, nodata, levels)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e3)
    out_bytes = sum(torch.Size(level_shape(plane.shape, 2 ** k)).numel() for k in range(1, levels + 1))
    nbytes = (plane.numel() + out_bytes) * plane.element_size()
    us = statistics.median(times)
    return us, nbytes, nbytes / us / 1e3


gen = torch.Generator(device='cuda').manual_seed(1)
for shape, dtype, levels, flush_l2 in (((5000, 5000), torch.uint16, 4, True), ((20000, 20000), torch.uint16, 6, False),
                                       ((20000, 20000), torch.float32, 6, False)):
    plane = (torch.rand(shape, generator=gen, device='cuda') * 4000).to(dtype)
    us, nbytes, gbs = time_kernel(plane, 0, levels, flush_l2)
    print(f'kernel {shape[0]}^2 {str(dtype)[6:]} {levels} levels ({"L2 flushed" if flush_l2 else "no flush"}): '
          f'{us:.1f} us, {nbytes / 1e6:.1f} MB moved, {gbs:.0f} GB/s')
    del plane
del flush
torch.cuda.empty_cache()

# ---- 2. file -> file ------------------------------------------------------------------------------------------------
src_ra, ref_ra = make_pair(250, 250, 20, bands=4, dtype='uint16', mu=3000.0, seed=2, device='cuda', src_nodata=0.0)
tmp = tempfile.mkdtemp(prefix='hb_ovw_')
geokeys = ((1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 32735), (), '')
wl = [dict(center_wavelength=w) for w in (0.48, 0.56, 0.66, 0.83)]
src_path = write_geotiff(os.path.join(tmp, 'src.tif'), src_ra.to_host().array, src_ra.transform, nodata=0,
                         geokeys=geokeys, band_tags=wl)
ref_path = write_geotiff(os.path.join(tmp, 'ref.tif'), ref_ra.to_host().array, ref_ra.transform, geokeys=geokeys,
                         band_tags=wl)
del src_ra, ref_ra
torch.cuda.empty_cache()
print(f'file -> file: 4-band uint16 5000^2 source, gain-offset 15 x 15, cores {os.cpu_count()}')
for compress, out_dtype, nodata in (('deflate', 'float32', float('nan')), (None, 'uint16', 0)):
    profile = dict(dtype=out_dtype, nodata=nodata, creation_options=dict(tiled=True, blockxsize=512, blockysize=512,
                                                                          compress=compress, interleave='band',
                                                                          photometric=None))
    times = {False: [], True: []}
    sizes = {}
    for rep in range(repeats + 1):                       # the first pair is a warm-up
        for ovw in (False, True):
            out = os.path.join(tmp, f'corr_{ovw}.tif')
            t0 = time.perf_counter()
            with RasterFuse(src_path, ref_path) as fuse:
                fuse.process(out, Model.gain_offset, (15, 15), build_ovw=ovw, overwrite=True, out_profile=profile)
            if rep:
                times[ovw].append(time.perf_counter() - t0)
            sizes[ovw] = os.path.getsize(out)
    with GeoTiffReader(os.path.join(tmp, 'corr_True.tif')) as im:
        factors = im.overviews(1)
    off, on = statistics.median(times[False]), statistics.median(times[True])
    print(f'  {out_dtype} {compress or "uncompressed"}: build_ovw=False {off:.3f} s ({sizes[False] / 1e6:.0f} MB) | '
          f'build_ovw=True {on:.3f} s ({sizes[True] / 1e6:.0f} MB, factors {factors}) | +{on - off:.3f} s '
          f'(runs: {[round(t, 3) for t in times[False]]} / {[round(t, 3) for t in times[True]]})')
