/*
 * oracle/interp_up_restate.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C, OpenMP over destination rows) of rasterio.warp.reproject(..., resampling=bilinear |
 * cubic | lanczos) for UP-sampling -- the `upsampling` config choices other than the default cubic_spline -- as GDAL
 * computes them (alg/gdalwarpkernel.cpp: GWKBilinearResample4Sample, GWKCubicResample4Sample, GWKResample /
 * GWKResampleOptimizedLanczos; no kernel scaling at a scale >= 0.95).  A companion of oracle/gdal_restate.c, with the
 * same grid convention (destination pixel-edge coordinate u maps to source coordinate sx*u + ox, rows sy*v + oy) and
 * the same nb-band "unified" validity as its gr_cubic_spline_up.
 *
 * GDAL is not installed in this image and no published known answer exists for these methods: PARITY UNPINNED.  The
 * rules below are their specification; oracle/interp_up_alt.py restates them independently in numpy.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

static inline int gr_invalid(double v, int has_nd, double nd)
{
    if (!has_nd) return 0;
    if (isnan(nd)) return isnan(v);
    return v == nd;
}

/* ------------------------------------------------------------------------------------------------------------------
 * GRA_Bilinear, GRA_Cubic and GRA_Lanczos for UP-sampling (scale >= 0.95 in GDAL: no kernel scaling), with the nb-band
 * unified validity of gr_cubic_spline_up.  Shared rules, per destination pixel:
 *   - centre rule: the source pixel containing the destination centre must be in range and unified-valid, else skip;
 *   - a tap counts only when it is in range and valid in its own band (band-valid implies unified-valid);
 *   - every decision is taken per band; accumulation in double, stored as float.
 * With src_x = sx (j + 0.5) + ox, k = floor(src_x - 0.5), d = src_x - 0.5 - k (the same in y):
 *   bilinear  (GWKBilinearResample4Sample)  taps k, k+1, weights (1-d, d); valid taps summed in the order UL, UR, LR,
 *             LL; skip if sum(w) < 1e-5, keep if sum(w) == 1.0 exactly, else divide by sum(w).
 *   cubic     (GWKCubicResample4Sample)  taps k-1 .. k+2, Keys a = -0.5; each row convolved in x, then the four rows
 *             in y, no normalisation.  If the 4x4 footprint leaves the raster or any of its taps is invalid for the
 *             band, the result is exactly the bilinear one.
 *   lanczos   (GWKResample)  taps k-2 .. k+3, weights L(i - d), i = -2 .. 3, L(0) = 1,
 *             L(t) = sin(pi t) sin(pi t / 3) / (pi^2 t^2 / 3) for 0 < |t| < 3, 0 otherwise; the valid taps of each row
 *             summed in x (values and weights), the rows then in y; skip if sum(w) < 1e-6, divide by sum(w) if it is
 *             outside [0.99999, 1.00001].
 * src is [nb, hs, ws] double; dst is [nb, hd, wd] float pre-filled with the destination nodata.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct {
    const double *src;
    long nb, hs, ws;
    int has_nd;
    double nd;
} gr_raster;

/* tap (y, x) of band b: 1 and its value when in range and valid in band b (band-valid implies unified-valid) */
static inline int gr_tap(const gr_raster *r, long b, long y, long x, double *v)
{
    if (y < 0 || y >= r->hs || x < 0 || x >= r->ws) return 0;
    *v = r->src[b * r->hs * r->ws + y * r->ws + x];
    return !gr_invalid(*v, r->has_nd, r->nd);
}

/* centre rule: the source pixel containing the destination centre is in range and valid in some band */
static inline int gr_centre_ok(const gr_raster *r, double src_y, double src_x)
{
    if (src_y < 0.0 || src_x < 0.0) return 0;
    long cy = (long)floor(src_y + 1e-10), cx = (long)floor(src_x + 1e-10);
    if (cy == r->hs) cy--;
    if (cx == r->ws) cx--;
    if (cy < 0 || cy >= r->hs || cx < 0 || cx >= r->ws) return 0;
    int any_valid = 0;
    for (long b = 0; b < r->nb; b++)
        any_valid |= !gr_invalid(r->src[b * r->hs * r->ws + cy * r->ws + cx], r->has_nd, r->nd);
    return any_valid;
}

static int gr_bilinear_px(const gr_raster *r, long b, long ky, double dy, long kx, double dx, double *out)
{
    const long ty[4] = {ky, ky, ky + 1, ky + 1}, tx[4] = {kx, kx + 1, kx + 1, kx};      /* UL, UR, LR, LL */
    const double wy[4] = {1.0 - dy, 1.0 - dy, dy, dy}, wx[4] = {1.0 - dx, dx, dx, 1.0 - dx};
    double acc = 0.0, acc_w = 0.0, v;
    for (int t = 0; t < 4; t++) {
        if (!gr_tap(r, b, ty[t], tx[t], &v)) continue;
        const double w = wx[t] * wy[t];
        acc_w += w;
        acc += v * w;
    }
    if (acc_w < 0.00001) return 0;
    *out = (acc_w == 1.0) ? acc : acc / acc_w;
    return 1;
}

static inline void gr_keys(double d, double *c)
{
    c[0] = 0.5 * d * (-1.0 + d * (2.0 - d));
    c[1] = 1.0 + 0.5 * d * d * (-5.0 + 3.0 * d);
    c[2] = 0.5 * d * (1.0 + d * (4.0 - 3.0 * d));
    c[3] = 0.5 * d * d * (-1.0 + d);
}

static int gr_cubic_px(const gr_raster *r, long b, long ky, double dy, long kx, double dx, double *out)
{
    double cx[4], cy[4], row[4];
    gr_keys(dx, cx);
    gr_keys(dy, cy);
    for (int tj = 0; tj < 4; tj++) {
        double v[4];
        for (int ti = 0; ti < 4; ti++)
            if (!gr_tap(r, b, ky - 1 + tj, kx - 1 + ti, &v[ti])) return gr_bilinear_px(r, b, ky, dy, kx, dx, out);
        row[tj] = cx[0] * v[0] + cx[1] * v[1] + cx[2] * v[2] + cx[3] * v[3];
    }
    *out = cy[0] * row[0] + cy[1] * row[1] + cy[2] * row[2] + cy[3] * row[3];
    return 1;
}

static inline double gr_lanczos3(double t)
{
    if (t == 0.0) return 1.0;
    if (fabs(t) >= 3.0) return 0.0;
    const double pt = M_PI * t;
    return sin(pt) * sin(pt / 3.0) / (pt * pt / 3.0);
}

static int gr_lanczos_px(const gr_raster *r, long b, long ky, double dy, long kx, double dx, double *out)
{
    double wx[6], wy[6], acc = 0.0, acc_w = 0.0, v;
    for (int i = 0; i < 6; i++) {
        wx[i] = gr_lanczos3((double)(i - 2) - dx);
        wy[i] = gr_lanczos3((double)(i - 2) - dy);
    }
    for (int tj = 0; tj < 6; tj++) {
        double row = 0.0, row_w = 0.0;
        for (int ti = 0; ti < 6; ti++) {
            if (!gr_tap(r, b, ky - 2 + tj, kx - 2 + ti, &v)) continue;
            row += v * wx[ti];
            row_w += wx[ti];
        }
        acc += row * wy[tj];
        acc_w += row_w * wy[tj];
    }
    if (acc_w < 0.000001) return 0;
    if (acc_w < 0.99999 || acc_w > 1.00001) acc /= acc_w;
    *out = acc;
    return 1;
}

typedef int (*gr_px_fn)(const gr_raster *, long, long, double, long, double, double *);

static void gr_interp_up(gr_px_fn px, const double *src, long nb, long hs, long ws, int has_nd, double nd, float *dst,
                         long hd, long wd, double sx, double ox, double sy, double oy)
{
    const gr_raster r = {src, nb, hs, ws, has_nd, nd};
    const long dplane = hd * wd;
    #pragma omp parallel for schedule(static)
    for (long i = 0; i < hd; i++) {
        const double src_y = sy * ((double)i + 0.5) + oy;
        const long ky = (long)floor(src_y - 0.5);
        const double dy = src_y - 0.5 - (double)ky;
        for (long j = 0; j < wd; j++) {
            const double src_x = sx * ((double)j + 0.5) + ox;
            if (!gr_centre_ok(&r, src_y, src_x)) continue;
            const long kx = (long)floor(src_x - 0.5);
            const double dx = src_x - 0.5 - (double)kx;
            for (long b = 0; b < nb; b++) {
                double v;
                if (px(&r, b, ky, dy, kx, dx, &v)) dst[b * dplane + i * wd + j] = (float)v;
            }
        }
    }
}

void gr_bilinear_up(const double *src, long nb, long hs, long ws, int has_nd, double nd, float *dst, long hd, long wd,
                    double sx, double ox, double sy, double oy)
{
    gr_interp_up(gr_bilinear_px, src, nb, hs, ws, has_nd, nd, dst, hd, wd, sx, ox, sy, oy);
}

void gr_cubic_up(const double *src, long nb, long hs, long ws, int has_nd, double nd, float *dst, long hd, long wd,
                 double sx, double ox, double sy, double oy)
{
    gr_interp_up(gr_cubic_px, src, nb, hs, ws, has_nd, nd, dst, hd, wd, sx, ox, sy, oy);
}

void gr_lanczos_up(const double *src, long nb, long hs, long ws, int has_nd, double nd, float *dst, long hd, long wd,
                   double sx, double ox, double sy, double oy)
{
    gr_interp_up(gr_lanczos_px, src, nb, hs, ws, has_nd, nd, dst, hd, wd, sx, ox, sy, oy);
}
