/*
 * oracle/footprint_stats_restate.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C, OpenMP over destination rows) of rasterio.warp.reproject(..., resampling=min | max | med |
 * q1 | q3 | mode): GDAL's footprint statistics, computed in the same routine as GRA_Average (GWKAverageOrModeThread)
 * over the same source window per destination pixel.  A companion of oracle/gdal_restate.c, with the same grid
 * convention (destination pixel-edge coordinate u maps to source coordinate sx*u + ox, rows sy*v + oy).
 *
 * GDAL is not installed in this image, no published known answer exists for these methods, and GDAL's handling of
 * them has changed between releases: PARITY UNPINNED.  The rules below are this project's specification;
 * oracle/footprint_stats_alt.py restates them independently in numpy.
 *
 *   1. Footprint window (that of the average down-sampler, csrc/resample.cu): with y_min = sy i + oy and
 *      y_max = sy (i + 1) + oy, rows run from floor(y_min + 1e-10) to ceil(y_max - 1e-10), end exclusive; a footprint
 *      inside one source row takes that row; the window is then clipped to the raster.  Columns likewise.  The methods
 *      are UNWEIGHTED: a partly covered edge pixel counts as one value like any other.
 *   2. Valid values: a pixel counts when it is not the nodata value (compared as float32) and is not NaN -- NaN never
 *      counts, even under a numeric nodata.  Values are compared as float32 (the reference's float32 read; exact for
 *      uint8 and uint16).  -0.0 and +0.0 are one value, and a zero result is +0.0.  A window without a valid pixel is
 *      not written (the caller pre-fills the destination with its nodata, NaN on the processing grid).
 *   3. min, max, med, q1, q3: with v[0..n) the valid values sorted ascending, min = v[0], max = v[n - 1], and
 *      med / q1 / q3 = v[ceil(q n - 1)] with q = 0.5 / 0.25 / 0.75 computed in double (GDAL's quantile index as read
 *      here; for even n, the lower median).
 *   4. mode: the most frequent value; among values tied for the highest count, the one whose LAST occurrence comes
 *      first in row-major scan order of the clipped window -- the value that first reaches the winning count in a
 *      scan, which is what GDAL's float mode scan intends.  So with all values distinct, the first valid pixel.  This
 *      float rule applies to every source dtype (the reference hands GDAL float32 arrays); GDAL's integer histogram
 *      rule (ties to the smallest value) does not apply.
 *   5. Geometry: any -- down-sampling, up-sampling (footprints of 1-2 pixels per axis) and mixed axes.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

enum { FS_MIN = 0, FS_MAX = 1, FS_MED = 2, FS_Q1 = 3, FS_Q3 = 4, FS_MODE = 5 };

typedef struct {
    float v;
    long pos;
} fs_item;

static int fs_cmp_value(const void *a, const void *b)
{
    const float x = *(const float *)a, y = *(const float *)b;
    return (x < y) ? -1 : (x > y ? 1 : 0);
}

/* by value, then by scan position */
static int fs_cmp_item(const void *a, const void *b)
{
    const fs_item *x = (const fs_item *)a, *y = (const fs_item *)b;
    if (x->v < y->v) return -1;
    if (x->v > y->v) return 1;
    return (x->pos < y->pos) ? -1 : (x->pos > y->pos ? 1 : 0);
}

/* rule 1 on one axis */
static void fs_axis(double s, double o, long i, long n, long *a, long *b)
{
    const double lo = s * (double)i + o, hi = s * (double)(i + 1) + o;
    const long a0 = (long)floor(lo + 1e-10);
    long b0 = (long)ceil(hi - 1e-10);
    if (a0 == b0) b0++;
    *a = a0 < 0 ? 0 : a0;
    *b = b0 > n ? n : b0;
}

/* src: float32 [hs][ws]; dst: float32 [hd][wd], pre-filled with the destination nodata */
void fs_resample_stat(const float *src, long hs, long ws, int has_nd, double nd, float *dst, long hd, long wd,
                      double sx, double ox, double sy, double oy, int method)
{
    const float ndf = (float)nd;
    const int nd_nan = isnan(nd);
    _Pragma("omp parallel")
    {
        fs_item *items = NULL;
        float *vals = NULL;
        long cap = 0;
        _Pragma("omp for schedule(static)")
        for (long i = 0; i < hd; i++) {
            long y0, y1;
            fs_axis(sy, oy, i, hs, &y0, &y1);
            for (long j = 0; j < wd; j++) {
                long x0, x1;
                fs_axis(sx, ox, j, ws, &x0, &x1);
                const long need = (y1 > y0 && x1 > x0) ? (y1 - y0) * (x1 - x0) : 0;
                if (need > cap) {
                    cap = need;
                    items = (fs_item *)realloc(items, (size_t)cap * sizeof(fs_item));
                    vals = (float *)realloc(vals, (size_t)cap * sizeof(float));
                }
                long n = 0;
                for (long y = y0; y < y1; y++)
                    for (long x = x0; x < x1; x++) {
                        float v = src[y * ws + x];
                        if (isnan(v)) continue;
                        if (has_nd && !nd_nan && v == ndf) continue;
                        if (v == 0.0f) v = 0.0f;                    /* -0.0 -> +0.0 */
                        vals[n] = v;
                        items[n].v = v;
                        items[n].pos = n;
                        n++;
                    }
                if (n == 0) continue;
                float out;
                if (method == FS_MODE) {
                    qsort(items, (size_t)n, sizeof(fs_item), fs_cmp_item);
                    long best_cnt = 0, best_last = 0;
                    out = items[0].v;
                    for (long a = 0; a < n;) {
                        long b = a;
                        while (b + 1 < n && items[b + 1].v == items[a].v) b++;
                        const long cnt = b - a + 1, last = items[b].pos;
                        if (cnt > best_cnt || (cnt == best_cnt && last < best_last)) {
                            best_cnt = cnt;
                            best_last = last;
                            out = items[a].v;
                        }
                        a = b + 1;
                    }
                } else {
                    qsort(vals, (size_t)n, sizeof(float), fs_cmp_value);
                    long k;
                    if (method == FS_MIN) k = 0;
                    else if (method == FS_MAX) k = n - 1;
                    else {
                        const double q = (method == FS_MED) ? 0.5 : (method == FS_Q1 ? 0.25 : 0.75);
                        k = (long)ceil(q * (double)n - 1.0);
                    }
                    out = vals[k];
                }
                dst[i * wd + j] = out;
            }
        }
        free(items);
        free(vals);
    }
}
