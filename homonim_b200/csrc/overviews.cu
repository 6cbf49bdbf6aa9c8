// overviews.cu -- 2x average overview pyramid of a written plane (RasterFuse._build_overviews, homonim/fuse.py:151-165:
// internal overviews with Resampling.average, levels 2, 4, 8, ...).
//
// Pixel rule (level 0 = the plane as written, level k computed from level k-1 as STORED in the output dtype): pixel
// (i, j) of level k averages the valid pixels among rows 2i, 2i+1 and columns 2j, 2j+1 of level k-1; rows / columns past
// the edge of an odd-sized level are absent.  Valid = not equal to the nodata value (when there is one) and, in float
// planes, not NaN.  No valid pixel -> nodata (NaN for float32 without one).  Integer types: exact sum s of the n valid
// pixels, floor((2s + n) / 2n) (round half up).  float32: sum in double in the order TL, TR, BL, BR, divided by n in
// double, rounded once to float.  Level k has ceil(H / 2^k) x ceil(W / 2^k) pixels.
//
// With this rule an aligned 64 x 64 tile of level 0 maps to aligned 32 x 32, 16 x 16, ..., 1 x 1 tiles of levels 1..6,
// so one CTA reads its base tile once (8 pixels per thread and row, 16-byte loads where the rows allow) and builds every
// level of that tile in shared memory.  Levels 7 and 8 are a second launch of the same kernel on level 6.
#include "hb_common.cuh"

namespace {

constexpr int OV_TILE = 64;            // base tile side
constexpr int OV_PASS_LEVELS = 6;      // levels built from one tile: 64 -> 32 -> ... -> 1
constexpr int OV_THREADS = 256;        // 32 level-1 rows x 8 threads, 4 level-1 pixels each

struct OvLevels {
    void *dst[OV_PASS_LEVELS];         // level k of this pass -> dst[k - 1], [nb][h[k]][w[k]]
    long h[OV_PASS_LEVELS + 1], w[OV_PASS_LEVELS + 1];     // [0]: the input plane
    int n;                             // levels of this pass (1..6)
};

template <typename T> struct OvNoData {
    int has;     // a stored pixel can equal the nodata value
    T value;     // nodata as stored; also what a window without valid pixels gets
};

template <typename T> __device__ __forceinline__ bool ov_valid(T v, const OvNoData<T> &nd)
{
    return !(nd.has && v == nd.value);
}
template <> __device__ __forceinline__ bool ov_valid<float>(float v, const OvNoData<float> &nd)
{
    return !(v != v) && !(nd.has && v == nd.value);
}

// average of the present + valid pixels of one window (a, b: top row; c, d: bottom row)
template <typename T>
__device__ __forceinline__ T ov_average(T a, T b, T c, T d, bool pb, bool pc, bool pd, const OvNoData<T> &nd)
{
    const bool va = ov_valid(a, nd), vb = pb && ov_valid(b, nd), vc = pc && ov_valid(c, nd), vd = pd && ov_valid(d, nd);
    const int n = (int)va + (int)vb + (int)vc + (int)vd;
    if (n == 0) return nd.value;
    const int s = (va ? (int)a : 0) + (vb ? (int)b : 0) + (vc ? (int)c : 0) + (vd ? (int)d : 0);
    const int num = 2 * s + n, den = 2 * n;
    int q = num / den;                           // C division truncates: make it a floor for negative sums
    if (num % den != 0 && num < 0) q -= 1;
    return (T)q;
}
template <>
__device__ __forceinline__ float ov_average<float>(float a, float b, float c, float d, bool pb, bool pc, bool pd,
                                                   const OvNoData<float> &nd)
{
    double s = 0.0;
    int n = 0;
    if (ov_valid(a, nd)) { s += (double)a; ++n; }
    if (pb && ov_valid(b, nd)) { s += (double)b; ++n; }
    if (pc && ov_valid(c, nd)) { s += (double)c; ++n; }
    if (pd && ov_valid(d, nd)) { s += (double)d; ++n; }
    return n ? (float)(s / (double)n) : nd.value;
}

// 8 consecutive pixels of one row (16-byte aligned when `vec`), or the present ones of them
template <typename T> __device__ __forceinline__ void ov_load8(const T *p, bool vec, long avail, T (&v)[8])
{
    if (vec && avail >= 8) {
        if (sizeof(T) == 1) {
            const uint2 r = hb_ldg_stream8(p);
            memcpy(v, &r, 8);
        } else if (sizeof(T) == 2) {
            const uint4 r = hb_ldg_stream16(p);
            memcpy(v, &r, 16);
        } else {
            const uint4 r0 = hb_ldg_stream16(p), r1 = hb_ldg_stream16(p + 4);
            memcpy(v, &r0, 16);
            memcpy(v + 4, &r1, 16);
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = (k < avail) ? p[k] : T(0);
}

template <typename T>
__global__ void __launch_bounds__(OV_THREADS) overview_pyramid_kernel(const T *__restrict__ src, OvNoData<T> nd,
                                                                      OvLevels lv, int vec)
{
    __shared__ T buf[2][(OV_TILE / 2) * (OV_TILE / 2)];
    const long band = blockIdx.z;
    const long ty0 = (long)blockIdx.y * OV_TILE, tx0 = (long)blockIdx.x * OV_TILE;
    const long h0 = lv.h[0], w0 = lv.w[0];

    // ---- level 1 from the input tile: thread -> level-1 row r, columns cq .. cq + 3 of the tile ----
    const int r = threadIdx.x >> 3, cq = (threadIdx.x & 7) * 4;
    const long gy = ty0 + 2 * r, gx = tx0 + 2 * cq;
    T top[8], bot[8];
    const long avail = w0 - gx;
    const bool has_top = gy < h0 && avail > 0, has_bot = gy + 1 < h0 && avail > 0;
    const T *row = src + (band * h0 + gy) * w0 + gx;
    if (has_top) ov_load8(row, vec, avail, top);
    if (has_bot) ov_load8(row + w0, vec, avail, bot);
    {
        const long h1 = lv.h[1], w1 = lv.w[1];
        const long oy = (ty0 >> 1) + r, ox = (tx0 >> 1) + cq;
        T *dst = reinterpret_cast<T *>(lv.dst[0]) + band * h1 * w1 + oy * w1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (has_top && 2 * j < avail) {
                const T v = ov_average(top[2 * j], top[2 * j + 1], bot[2 * j], bot[2 * j + 1], 2 * j + 1 < avail, has_bot,
                                       has_bot && 2 * j + 1 < avail, nd);
                dst[ox + j] = v;
                buf[0][r * (OV_TILE / 2) + cq + j] = v;
            }
        }
    }

    // ---- levels 2 .. n from the previous level's tile in shared memory ----
    for (int k = 2; k <= lv.n; ++k) {
        __syncthreads();
        const int side = OV_TILE >> k, pside = 2 * side;
        const T *prev = buf[k & 1];
        T *cur = buf[(k + 1) & 1];
        const long ph = lv.h[k - 1], pw = lv.w[k - 1], hk = lv.h[k], wk = lv.w[k];
        const long py0 = ty0 >> (k - 1), px0 = tx0 >> (k - 1);     // the previous level's tile origin
        T *dst = reinterpret_cast<T *>(lv.dst[k - 1]) + band * hk * wk;
        for (int idx = threadIdx.x; idx < side * side; idx += OV_THREADS) {
            const int i = idx / side, j = idx - i * side;
            const long y = py0 + 2 * i, x = px0 + 2 * j;
            if (y >= ph || x >= pw) continue;
            const bool pr = x + 1 < pw, pd = y + 1 < ph;
            const T *p = prev + (2 * i) * pside + 2 * j;
            const T v = ov_average(p[0], pr ? p[1] : p[0], pd ? p[pside] : p[0], (pr && pd) ? p[pside + 1] : p[0], pr, pd,
                                   pr && pd, nd);
            dst[(y >> 1) * wk + (x >> 1)] = v;
            cur[i * side + j] = v;
        }
    }
}

template <typename T> OvNoData<T> ov_make_nodata(int has_nodata, double nodata)
{
    OvNoData<T> nd;
    const double lo = (T)(-1) < (T)0 ? -32768.0 : 0.0, hi = sizeof(T) == 1 ? 255.0 : (lo < 0 ? 32767.0 : 65535.0);
    nd.has = has_nodata && nodata >= lo && nodata <= hi && nodata == floor(nodata);
    nd.value = nd.has ? (T)nodata : (T)0;   // (an unrepresentable nodata matches no pixel: every window has one)
    return nd;
}
template <> OvNoData<float> ov_make_nodata<float>(int has_nodata, double nodata)
{
    OvNoData<float> nd;
    nd.has = has_nodata && !isnan(nodata);
    nd.value = has_nodata ? (float)nodata : __builtin_nanf("");
    return nd;
}

template <typename T>
int launch_pyramid(const void *src_dev, long nb, long h, long w, int has_nodata, double nodata, int n_levels,
                   void *const *levels_dev, cudaStream_t st)
{
    const OvNoData<T> nd = ov_make_nodata<T>(has_nodata, nodata);
    const void *in = src_dev;
    long ih = h, iw = w;
    for (int first = 1; first <= n_levels; first += OV_PASS_LEVELS) {
        OvLevels lv;
        lv.n = n_levels - first + 1 < OV_PASS_LEVELS ? n_levels - first + 1 : OV_PASS_LEVELS;
        lv.h[0] = ih;
        lv.w[0] = iw;
        for (int k = 1; k <= OV_PASS_LEVELS; ++k) {
            lv.h[k] = (lv.h[k - 1] + 1) / 2;
            lv.w[k] = (lv.w[k - 1] + 1) / 2;
            lv.dst[k - 1] = k <= lv.n ? levels_dev[first + k - 2] : nullptr;
        }
        const int vec = (iw % 8 == 0) && ((uintptr_t)in % 16 == 0);
        const dim3 grid((unsigned)((iw + OV_TILE - 1) / OV_TILE), (unsigned)((ih + OV_TILE - 1) / OV_TILE), (unsigned)nb);
        overview_pyramid_kernel<T><<<grid, OV_THREADS, 0, st>>>((const T *)in, nd, lv, vec);
        HB_LAUNCH_OK("overview_pyramid_kernel");
        in = lv.dst[lv.n - 1];
        ih = lv.h[lv.n];
        iw = lv.w[lv.n];
    }
    return 0;
}

}  // namespace

extern "C" int hb_build_overviews(const void *src_dev, int dtype, long nb, long h, long w, int has_nodata, double nodata,
                                  int n_levels, void *const *levels_dev, void *stream)
{
    HB_REQUIRE(src_dev && levels_dev && nb >= 1 && nb <= 65535 && h > 0 && w > 0 && n_levels >= 1 && n_levels <= 8,
               "hb_build_overviews: bad arguments");
    HB_REQUIRE((h + OV_TILE - 1) / OV_TILE <= 65535, "hb_build_overviews: the plane has too many rows (%ld)", h);
    for (int k = 0; k < n_levels; ++k) HB_REQUIRE(levels_dev[k], "hb_build_overviews: level %d has no buffer", k + 1);
    cudaStream_t st = (cudaStream_t)stream;
    switch (dtype) {
        case HB_U8: return launch_pyramid<uint8_t>(src_dev, nb, h, w, has_nodata, nodata, n_levels, levels_dev, st);
        case HB_U16: return launch_pyramid<uint16_t>(src_dev, nb, h, w, has_nodata, nodata, n_levels, levels_dev, st);
        case HB_I16: return launch_pyramid<int16_t>(src_dev, nb, h, w, has_nodata, nodata, n_levels, levels_dev, st);
        case HB_F32: return launch_pyramid<float>(src_dev, nb, h, w, has_nodata, nodata, n_levels, levels_dev, st);
    }
    HB_REQUIRE(false, "hb_build_overviews: unsupported dtype %d", dtype);
}
