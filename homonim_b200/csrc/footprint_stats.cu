// footprint_stats.cu -- footprint statistics of the kernel-model path (sm_100a):
//   * hb_resample_stat : RasterArray.reproject(resampling=min | max | med | q1 | q3 | mode)   (reference
//                        raster_array.py:526-578, GDAL GWKAverageOrModeThread)
// Each destination pixel takes one of the valid source values under its footprint: no arithmetic on the values, so the
// result is exact and does not depend on launch or scheduling order.  The rules (footprint window, validity, quantile
// index, mode tie-break) are specified in oracle/footprint_stats_restate.c.
//
// Values are compared through order-preserving 32-bit keys: the value itself for uint8 / uint16, v + 32768 for int16,
// the float_key map of block_norm.cu for float32 (after -0.0 -> +0.0).  Two paths, chosen at launch from the largest
// footprint the geometry allows:
//   * stat_thread_kernel  (<= kStatSmallMax pixels: up-sampling and ratios up to ~5)  one thread per destination pixel;
//     the thread's valid keys sit in a shared-memory column and a rank / count double loop over them selects the value.
//   * stat_warp_kernel    (larger footprints)  one warp per destination pixel; the warp stages the footprint's valid keys
//     in scan order into its shared-memory slice, then: min / max by a warp reduction; med / q1 / q3 by radix select
//     (8-bit digits, one level for uint8, two for uint16 / int16, four for float32, shared-memory histograms); mode by a
//     bitonic sort of (key, scan index) pairs, whose runs give each value's count and last occurrence.
#include "hb_common.cuh"

namespace {

constexpr int kStatMaxRatio = 128;           // source pixels per destination pixel, each axis
constexpr int kStatSmallMax = 49;            // largest footprint of the thread-per-pixel path
constexpr int kStatThreads = 128;            // threads per CTA of the thread-per-pixel path
constexpr int kStatWarpsMax = 8;
constexpr int kStatSmemMax = 227 * 1024;     // sm_100 opt-in shared memory per CTA
constexpr int kStatHistBytes = 256 * 4;      // per warp: radix-select digit histogram
constexpr unsigned kFull = 0xffffffffu;

template <typename T> struct StatKey;
template <> struct StatKey<uint8_t> {
    static constexpr int kTopShift = 0;       // keys < 2^8: one 8-bit digit
    static __device__ __forceinline__ bool load(const uint8_t *p, const NoData &nd, uint32_t &k)
    {
        k = __ldg(p);
        return hb_valid_int(k, nd);
    }
    static __device__ __forceinline__ float value(uint32_t k) { return (float)k; }
};
template <> struct StatKey<uint16_t> {
    static constexpr int kTopShift = 8;       // keys < 2^16: two digits
    static __device__ __forceinline__ bool load(const uint16_t *p, const NoData &nd, uint32_t &k)
    {
        k = __ldg(p);
        return hb_valid_int(k, nd);
    }
    static __device__ __forceinline__ float value(uint32_t k) { return (float)k; }
};
template <> struct StatKey<int16_t> {
    static constexpr int kTopShift = 8;       // keys < 2^16: two digits
    // v ^ 0x8000 on the 16-bit pattern is v + 32768: order-preserving
    static __device__ __forceinline__ bool load(const int16_t *p, const NoData &nd, uint32_t &k)
    {
        const int16_t v = __ldg(p);
        k = (uint32_t)(uint16_t)v ^ 0x8000u;
        return hb_valid_int((uint32_t)(int)v, nd);
    }
    static __device__ __forceinline__ float value(uint32_t k) { return __uint_as_float(0x4B000000u | k) - 8421376.0f; }
};
template <> struct StatKey<float> {
    static constexpr int kTopShift = 24;      // four digits
    // NaN never counts, even under a numeric nodata; -0.0 and +0.0 share the key of +0.0
    static __device__ __forceinline__ bool load(const float *p, const NoData &nd, uint32_t &k)
    {
        const float v = __ldg(p);
        uint32_t b = __float_as_uint(v);
        if ((b << 1) == 0u) b = 0u;
        k = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
        return hb_valid(v, nd) && !isnan(v);
    }
    static __device__ __forceinline__ float value(uint32_t k)
    {
        return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
    }
};

// Footprint of destination index i on one axis: GDAL's window (hb_footprint) clipped to [0, n), capped at wmax pixels --
// the most the geometry allows, so the cap never binds; it only bounds the shared-memory writes.
__device__ __forceinline__ void stat_axis(double s, double o, long i, long n, long wmax, long &a, long &b)
{
    const HbFootprint f = hb_footprint(s, o, i);
    a = max(f.a0, 0L);
    b = min(min(f.b0, n), a + wmax);
}

// 0-based rank of min / max / med / q1 / q3 among n >= 1 sorted values: v[ceil(q n - 1)], in double
__device__ __forceinline__ int stat_rank(int method, int n)
{
    if (method == HB_STAT_MIN) return 0;
    if (method == HB_STAT_MAX) return n - 1;
    const double q = (method == HB_STAT_MED) ? 0.5 : (method == HB_STAT_Q1 ? 0.25 : 0.75);
    return (int)ceil(q * (double)n - 1.0);
}

// ---- small footprints: one thread per destination pixel --------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kStatThreads)
stat_thread_kernel(const T *__restrict__ src, long hs, long ws, NoData nd, float *__restrict__ dst, long hd, long wd,
                   double sx, double ox, double sy, double oy, int method, int wxmax, int wymax)
{
    extern __shared__ uint32_t s_keys[];                       // [wxmax * wymax][kStatThreads]: one column per thread
    const long p = (long)blockIdx.x * kStatThreads + threadIdx.x;
    if (p >= hd * wd) return;
    const long i = p / wd, j = p - i * wd;
    long y0, y1, x0, x1;
    stat_axis(sy, oy, i, hs, wymax, y0, y1);
    stat_axis(sx, ox, j, ws, wxmax, x0, x1);
    uint32_t *keys = s_keys + threadIdx.x;
    int n = 0;
    for (long y = y0; y < y1; y++)
        for (long x = x0; x < x1; x++) {
            uint32_t k;
            if (StatKey<T>::load(src + y * ws + x, nd, k)) keys[(n++) * kStatThreads] = k;
        }
    float out = __int_as_float(0x7fc00000);
    if (n > 0) {
        uint32_t sel = 0u;
        if (method == HB_STAT_MODE) {
            // highest count wins; among equal counts, the value whose last occurrence comes first
            int best_cnt = 0, best_last = 0;
            for (int a = 0; a < n; a++) {
                const uint32_t ka = keys[a * kStatThreads];
                int cnt = 0, last = 0;
                for (int b = 0; b < n; b++)
                    if (keys[b * kStatThreads] == ka) { cnt++; last = b; }
                if (cnt > best_cnt || (cnt == best_cnt && last < best_last)) { best_cnt = cnt; best_last = last; sel = ka; }
            }
        } else {
            // the value whose run of equal values in sorted order covers rank r
            const int r = stat_rank(method, n);
            for (int a = 0; a < n; a++) {
                const uint32_t ka = keys[a * kStatThreads];
                int less = 0, eq = 0;
                for (int b = 0; b < n; b++) {
                    const uint32_t kb = keys[b * kStatThreads];
                    less += (kb < ka) ? 1 : 0;
                    eq += (kb == ka) ? 1 : 0;
                }
                if (less <= r && r < less + eq) { sel = ka; break; }
            }
        }
        out = StatKey<T>::value(sel);
    }
    dst[p] = out;
}

// ---- large footprints: one warp per destination pixel ---------------------------------------------------------------
// key of rank r among the n keys by radix select: per 8-bit digit from the top, histogram the keys that match the digits
// chosen so far and descend into the bucket that holds rank r
__device__ uint32_t warp_radix_select(const uint32_t *keys, int n, int r, uint32_t *hist, int lane, int top_shift)
{
    uint32_t prefix = 0u, pmask = 0u;
    for (int shift = top_shift; shift >= 0; shift -= 8) {
        for (int b = lane; b < 256; b += 32) hist[b] = 0u;
        __syncwarp();
        for (int e = lane; e < n; e += 32) {
            const uint32_t k = keys[e];
            if ((k & pmask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
        }
        __syncwarp();
        uint32_t c[8], s = 0u;                                  // lane owns buckets [8 lane, 8 lane + 8)
#pragma unroll
        for (int q = 0; q < 8; q++) { c[q] = hist[8 * lane + q]; s += c[q]; }
        uint32_t incl = s;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(kFull, incl, off);
            if (lane >= off) incl += t;
        }
        const uint32_t excl = incl - s;
        const bool mine = excl <= (uint32_t)r && (uint32_t)r < incl;
        const int owner = __ffs(__ballot_sync(kFull, mine)) - 1;
        uint32_t bucket = 0u, below = excl;
        if (mine) {
            bool found = false;
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (!found && (uint32_t)r < below + c[q]) { bucket = 8u * lane + q; found = true; }
                else if (!found) below += c[q];
            }
        }
        bucket = __shfl_sync(kFull, bucket, owner);
        below = __shfl_sync(kFull, below, owner);
        r -= (int)below;
        prefix |= bucket << shift;
        pmask |= 255u << shift;
        __syncwarp();
    }
    return prefix;
}

// mode of the n (key << 32 | scan index) entries: bitonic sort (every comparator ascending, so the entries past n act as
// +infinity without being stored), then each run of one key ends at its last occurrence; its start is found by binary
// search.  The winner maximises (count, -last occurrence).
__device__ uint32_t warp_mode(unsigned long long *v, int n, int lane)
{
    int npow = 1;
    while (npow < n) npow <<= 1;
    for (int k = 2; k <= npow; k <<= 1) {
        for (int j = k >> 1; j >= 1; j >>= 1) {
            for (int t = lane; t < (npow >> 1); t += 32) {
                int lo, hi;
                if (j == (k >> 1)) {                            // first step of a merge: mirrored partner
                    const int blk = t / j, o = t - blk * j;
                    lo = blk * k + o;
                    hi = blk * k + k - 1 - o;
                } else {
                    const int blk = t / j, o = t - blk * j;
                    lo = blk * 2 * j + o;
                    hi = lo + j;
                }
                if (hi < n) {
                    const unsigned long long a = v[lo], b = v[hi];
                    if (a > b) { v[lo] = b; v[hi] = a; }
                }
            }
            __syncwarp();
        }
    }
    unsigned long long best = 0ull;
    uint32_t best_key = 0u;
    for (int e = lane; e < n; e += 32) {
        const uint32_t key = (uint32_t)(v[e] >> 32);
        if (e + 1 < n && (uint32_t)(v[e + 1] >> 32) == key) continue;
        int lo = 0, hi = e;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((uint32_t)(v[mid] >> 32) < key) lo = mid + 1; else hi = mid;
        }
        const unsigned long long cand = ((unsigned long long)(e - lo + 1) << 32) | (0xffffffffu - (uint32_t)v[e]);
        if (cand > best) { best = cand; best_key = key; }
    }
    unsigned long long all = best;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const unsigned long long o = __shfl_xor_sync(kFull, all, off);
        all = o > all ? o : all;
    }
    const int owner = __ffs(__ballot_sync(kFull, best == all)) - 1;
    return __shfl_sync(kFull, best_key, owner);
}

template <typename T>
__global__ void __launch_bounds__(32 * kStatWarpsMax)
stat_warp_kernel(const T *__restrict__ src, long hs, long ws, NoData nd, float *__restrict__ dst, long hd, long wd,
                 double sx, double ox, double sy, double oy, int method, int wxmax, int wymax, int buf_bytes)
{
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const long p = (long)blockIdx.x * warps + w;
    if (p >= hd * wd) return;                                   // (whole warps: no CTA-wide barrier below)
    uint32_t *hist = reinterpret_cast<uint32_t *>(s_raw) + 256 * w;
    unsigned char *buf = s_raw + (size_t)kStatHistBytes * warps + (size_t)buf_bytes * w;
    uint32_t *keys = reinterpret_cast<uint32_t *>(buf);
    unsigned long long *pairs = reinterpret_cast<unsigned long long *>(buf);
    const bool mode = method == HB_STAT_MODE;

    const long i = p / wd, j = p - i * wd;
    long y0, y1, x0, x1;
    stat_axis(sy, oy, i, hs, wymax, y0, y1);
    stat_axis(sx, ox, j, ws, wxmax, x0, x1);
    const int nc = (int)max(x1 - x0, 0L), ne = (int)max(y1 - y0, 0L) * nc;

    // stage the valid keys in row-major scan order (lane e of a step reads window element e0 + e); the loads of
    // kStageBatch steps are issued before the first is used, so that a warp has that many in flight, not one
    constexpr int kStageBatch = 8;
    int n = 0;
    if (ne > 0) {
        const int dr = 32 / nc, dc = 32 - dr * nc;
        int r = lane / nc, c = lane - (lane / nc) * nc;
        const unsigned lt = (1u << lane) - 1u;
        for (int e0 = 0; e0 < ne; e0 += 32 * kStageBatch) {
            uint32_t kb[kStageBatch];
            bool okb[kStageBatch];
#pragma unroll
            for (int u = 0; u < kStageBatch; u++) {
                kb[u] = 0u;
                okb[u] = (e0 + 32 * u + lane < ne) && StatKey<T>::load(src + (y0 + r) * ws + x0 + c, nd, kb[u]);
                r += dr;
                c += dc;
                if (c >= nc) { c -= nc; r++; }
            }
#pragma unroll
            for (int u = 0; u < kStageBatch; u++) {
                const unsigned bal = __ballot_sync(kFull, okb[u]);
                if (okb[u]) {
                    const int at = n + __popc(bal & lt);
                    if (mode) pairs[at] = ((unsigned long long)kb[u] << 32) | (unsigned)at;
                    else keys[at] = kb[u];
                }
                n += __popc(bal);
            }
        }
    }
    __syncwarp();

    float out = __int_as_float(0x7fc00000);
    if (n > 0) {
        uint32_t sel;
        if (method == HB_STAT_MIN || method == HB_STAT_MAX) {
            uint32_t m = (method == HB_STAT_MIN) ? 0xffffffffu : 0u;
            for (int e = lane; e < n; e += 32) m = (method == HB_STAT_MIN) ? min(m, keys[e]) : max(m, keys[e]);
            sel = (method == HB_STAT_MIN) ? __reduce_min_sync(kFull, m) : __reduce_max_sync(kFull, m);
        } else if (mode) {
            sel = warp_mode(pairs, n, lane);
        } else {
            sel = warp_radix_select(keys, n, stat_rank(method, n), hist, lane, StatKey<T>::kTopShift);
        }
        out = StatKey<T>::value(sel);
    }
    if (lane == 0) dst[p] = out;
}

template <typename T>
int launch_stat(const void *src, long hs, long ws, NoData nd, float *dst, long hd, long wd, double sx, double ox,
                double sy, double oy, int method, cudaStream_t stream)
{
    // most pixels a footprint can span on each axis: floor(ratio) + 2 (a fractional start and end)
    const int wxmax = (int)floor(sx) + 2, wymax = (int)floor(sy) + 2;
    const long nmax = (long)wxmax * wymax;
    const long npix = hd * wd;
    if (nmax <= kStatSmallMax) {
        const long blocks = (npix + kStatThreads - 1) / kStatThreads;
        HB_REQUIRE(blocks < 2147483647L, "hb_resample_stat: grid too large");
        const size_t smem = (size_t)nmax * kStatThreads * sizeof(uint32_t);
        stat_thread_kernel<T><<<(unsigned)blocks, kStatThreads, smem, stream>>>(
            (const T *)src, hs, ws, nd, dst, hd, wd, sx, ox, sy, oy, method, wxmax, wymax);
        HB_LAUNCH_OK("stat_thread_kernel");
        return 0;
    }
    static HbOncePerDevice once;
    const int rc = hb_once_per_device(once, [] {
        HB_CUDA_OK(cudaFuncSetAttribute(stat_warp_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, kStatSmemMax));
        return 0;
    });
    if (rc) return rc;
    const int buf_bytes = (int)(((method == HB_STAT_MODE ? 8 : 4) * nmax + 15) / 16 * 16);
    const int per_warp = kStatHistBytes + buf_bytes;
    // warps per CTA: 4 when many fit (several CTAs then share an SM), otherwise as many as the shared memory holds
    const int fit = kStatSmemMax / per_warp;
    const int warps = fit >= 2 * 4 ? 4 : min(fit, kStatWarpsMax);
    const long blocks = (npix + warps - 1) / warps;
    HB_REQUIRE(blocks < 2147483647L, "hb_resample_stat: grid too large");
    stat_warp_kernel<T><<<(unsigned)blocks, 32 * warps, (size_t)per_warp * warps, stream>>>(
        (const T *)src, hs, ws, nd, dst, hd, wd, sx, ox, sy, oy, method, wxmax, wymax, buf_bytes);
    HB_LAUNCH_OK("stat_warp_kernel");
    return 0;
}

}  // namespace

// =====================================================================================================================
// C-ABI
// =====================================================================================================================
extern "C" int hb_resample_stat(const void *src_dev, int src_dtype, long hs, long ws, int has_nodata, double nodata,
                                float *dst_dev, long hd, long wd, double sx, double ox, double sy, double oy, int method,
                                void *stream)
{
    HB_REQUIRE(src_dev && dst_dev && hs > 0 && ws > 0 && hd > 0 && wd > 0, "hb_resample_stat: bad arguments");
    HB_REQUIRE(sx > 0 && sy > 0, "hb_resample_stat: grids must have the same orientation");
    HB_REQUIRE(sx <= kStatMaxRatio && sy <= kStatMaxRatio,
               "hb_resample_stat: %.4g x %.4g source pixels per destination pixel exceed the maximum of %d on each axis",
               sx, sy, kStatMaxRatio);
    HB_REQUIRE(method >= HB_STAT_MIN && method <= HB_STAT_MODE, "hb_resample_stat: unknown method %d", method);
    const NoData nd = hb_make_nodata(has_nodata, nodata, src_dtype);
    cudaStream_t st = (cudaStream_t)stream;
    switch (src_dtype) {
        case HB_U8: return launch_stat<uint8_t>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, method, st);
        case HB_U16: return launch_stat<uint16_t>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, method, st);
        case HB_I16: return launch_stat<int16_t>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, method, st);
        case HB_F32: return launch_stat<float>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, method, st);
    }
    HB_REQUIRE(false, "hb_resample_stat: unknown dtype %d", src_dtype);
}
