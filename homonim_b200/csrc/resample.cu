// resample.cu -- down-sampling and element-wise kernels of the kernel-model path (sm_100a):
//   * hb_downsample_average : RasterArray.reproject(resampling=average)     (reference raster_array.py:526-578,
//                             kernel_model.py:480)                            [HBM-bound: reads every hi-res pixel]
//   * hb_apply_same_grid, hb_valid_mask, hb_full_coverage_mask                (kernel_model.py:375-409, 442-463)
//   * hb_convert_dtype      : output dtype conversion                         (raster_array.py:353-387)
// Up-sampling (hb_upsample_apply, hb_resample_up) lives in upsample.cu.
//
// The GDAL algorithms restated here are specified in oracle/gdal_restate.c (GDAL itself is not in this image).
#include <type_traits>

#include "hb_common.cuh"

namespace {

// =====================================================================================================================
// 1. average down-sampling
// =====================================================================================================================
constexpr int kDsVec = 8;                        // source pixels per thread per row
#ifndef HB_DS_THREADS
#define HB_DS_THREADS 256
#endif
#ifndef HB_DS_MIN_CTAS
#define HB_DS_MIN_CTAS 3
#endif
constexpr int kDsThreads = HB_DS_THREADS;
constexpr int kDsSpan = kDsThreads * kDsVec;     // source columns staged per CTA

template <typename T> struct Raw8;               // 8 consecutive source pixels, vector-loaded
template <> struct Raw8<uint16_t> {
    static __device__ __forceinline__ void load(const uint16_t *p, uint16_t (&v)[8])
    {
        const uint4 w = hb_ldg_stream16(p);
        v[0] = (uint16_t)(w.x & 0xFFFFu); v[1] = (uint16_t)(w.x >> 16);
        v[2] = (uint16_t)(w.y & 0xFFFFu); v[3] = (uint16_t)(w.y >> 16);
        v[4] = (uint16_t)(w.z & 0xFFFFu); v[5] = (uint16_t)(w.z >> 16);
        v[6] = (uint16_t)(w.w & 0xFFFFu); v[7] = (uint16_t)(w.w >> 16);
    }
};
template <> struct Raw8<int16_t> {
    static __device__ __forceinline__ void load(const int16_t *p, int16_t (&v)[8])
    {
        const uint4 w = hb_ldg_stream16(p);
        v[0] = (int16_t)(w.x & 0xFFFFu); v[1] = (int16_t)(w.x >> 16);
        v[2] = (int16_t)(w.y & 0xFFFFu); v[3] = (int16_t)(w.y >> 16);
        v[4] = (int16_t)(w.z & 0xFFFFu); v[5] = (int16_t)(w.z >> 16);
        v[6] = (int16_t)(w.w & 0xFFFFu); v[7] = (int16_t)(w.w >> 16);
    }
};
template <> struct Raw8<uint8_t> {
    static __device__ __forceinline__ void load(const uint8_t *p, uint8_t (&v)[8])
    {
        const uint2 w = hb_ldg_stream8(p);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            v[k] = (uint8_t)((w.x >> (8 * k)) & 0xFFu);
            v[4 + k] = (uint8_t)((w.y >> (8 * k)) & 0xFFu);
        }
    }
};
template <> struct Raw8<float> {
    static __device__ __forceinline__ void load(const float *p, float (&v)[8])
    {
        const uint4 a = hb_ldg_stream16(p), b = hb_ldg_stream16(p + 4);
        v[0] = __uint_as_float(a.x); v[1] = __uint_as_float(a.y); v[2] = __uint_as_float(a.z);
        v[3] = __uint_as_float(a.w); v[4] = __uint_as_float(b.x); v[5] = __uint_as_float(b.y);
        v[6] = __uint_as_float(b.z); v[7] = __uint_as_float(b.w);
    }
};

template <typename T> struct IsInt { static constexpr bool value = true; };
template <> struct IsInt<float> { static constexpr bool value = false; };

template <typename T> __device__ __forceinline__ bool ds_valid(T v, const NoData &nd)
{
    if (IsInt<T>::value) return hb_valid_int((uint32_t)v, nd);         // (int16: sign-extended)
    return hb_valid((float)v, nd);
}

// The integer paths sum raw 32-bit words of packed pixels.  int16 words hold two's-complement fields: they are summed by
// the signed form of dp2a, their nodata pattern is the value's 16-bit two's complement, and the 32-bit sums (exact: at
// most 65025 * 32768 < 2^31 in magnitude) are read back as signed.
template <typename T> __device__ __forceinline__ uint32_t ds_nd_field(const NoData &nd)
{
    return std::is_same<T, int16_t>::value ? hb_nd_bits16(nd) : (uint32_t)nd.ivalue;
}
template <typename T> __device__ __forceinline__ uint32_t ds_dp2a_lo(uint32_t w, uint32_t b, uint32_t acc)
{
    if constexpr (std::is_same<T, int16_t>::value) return (uint32_t)__dp2a_lo((int)w, (int)b, (int)acc);
    else return __dp2a_lo(w, b, acc);
}
template <typename T> __device__ __forceinline__ double ds_sum(uint32_t s)
{
    return std::is_same<T, int16_t>::value ? (double)(int)s : (double)s;
}

// fetch 8 pixels of row `row` starting at column c (may be partially / wholly outside [0, ws))
template <typename T, bool ALIGNED>
__device__ __forceinline__ void ds_fetch(const T *row, long c, long ws, T (&v)[8], uint32_t &inb)
{
    if (ALIGNED && c >= 0 && c + 8 <= ws) {
        Raw8<T>::load(row + c, v);
        inb = 0xFFu;
    } else {
        inb = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const long x = c + k;
            if (x >= 0 && x < ws) { v[k] = row[x]; inb |= (1u << k); } else v[k] = (T)0;
        }
    }
}

// One CTA: one destination row, `ndc` destination columns.  Phase 1: every thread owns 8 source columns and sums them
// down the footprint rows (interior rows have weight 1: exact integer sums for uint8/uint16/int16, double for float32;
// the <= 2 fractionally covered rows are added in double).  Phase 2: one thread per destination pixel combines its
// footprint columns from shared memory with the fractional edge weights.
template <typename T, bool ALIGNED>
__global__ void __launch_bounds__(kDsThreads, (sizeof(T) == 4) ? HB_DS_MIN_CTAS - 1 : HB_DS_MIN_CTAS)
downsample_average_kernel(const T *__restrict__ src, long hs, long ws, NoData nd, float *__restrict__ dst, long hd,
                          long wd, double sx, double ox, double sy, double oy, int ndc, int chunks)
{
    __shared__ double s_sum[kDsSpan];
    __shared__ double s_w[kDsSpan];

    const long i = blockIdx.x / chunks;
    const int chunk = (int)(blockIdx.x % chunks);
    const long j0 = (long)chunk * ndc;
    const long j1 = min(j0 + (long)ndc, wd);
    const int t = threadIdx.x;
    const float qnan = __int_as_float(0x7fc00000);

    // Footprint rows.  Weights follow GDAL's COMPUTE_WEIGHT_Y on the UNCLAMPED footprint and rows outside the raster
    // are skipped -- i.e. the result equals GDAL's on a source padded with nodata, which is how the reference reads
    // its source blocks (boundless windows, raster_array.py:175-199).
    const HbFootprint fy = hb_footprint(sy, oy, i);
    const long iy0u = fy.a0, iy1u = fy.b0;
    const long iy0 = max(iy0u, 0L), iy1 = min(iy1u, hs);
    if (iy0 >= iy1) {
        for (long j = j0 + t; j < j1; j += kDsThreads) dst[i * wd + j] = qnan;
        return;
    }
    const double wy_first = (iy0u + 1 == iy1u) ? 1.0 : 1.0 - (fy.lo - (double)iy0u);
    const double wy_last = 1.0 - ((double)iy1u - fy.hi);
    const bool first_frac = (iy0u >= 0) && (wy_first != 1.0);
    const bool last_frac = (iy1u <= hs) && (iy0u + 1 < iy1u) && (wy_last != 1.0);
    const long ya = iy0 + (first_frac ? 1 : 0), yb = iy1 - (last_frac ? 1 : 0);   // interior rows [ya, yb)

    const long c_lo = max(hb_footprint(sx, ox, j0).a0, 0L);
    const long c_base = (c_lo / kDsVec) * kDsVec;
    const long c = c_base + (long)t * kDsVec;

    const NoData ndk = nd;

    // ---- phase 1: column sums over interior rows ------------------------------------------------------------------
    double colsum[8], colw[8];
    if (IsInt<T>::value) {
        uint32_t isum[8], icnt[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { isum[k] = 0; icnt[k] = 0; }
        if (ALIGNED && c >= 0 && c + 8 <= ws) {
            // Fast path (every vector of this thread lies inside the raster).  Sum ALL pixels with one integer
            // dot-product instruction per pixel (IDP: dp2a / dp4a against a one-hot byte vector -- no unpacking), and
            // only look for nodata with a packed "has a zero field" test on (word ^ nodata pattern); the exact
            // per-pixel count of nodata pixels runs only for words that may contain one.  Afterwards
            //     sum(valid) = sum(all) - nodata * count(nodata),  count(valid) = rows - count(nodata)   (exact).
            constexpr int NW = (sizeof(T) == 2) ? 4 : 2;                   // 32-bit words per 8 pixels
            constexpr uint32_t kOnes = (sizeof(T) == 2) ? 0x00010001u : 0x01010101u;
            constexpr uint32_t kHigh = (sizeof(T) == 2) ? 0x80008000u : 0x80808080u;
            const bool scan_nd = ndk.int_ok && (sizeof(T) == 2 || ndk.ivalue <= 255);
            const uint32_t ndpat = scan_nd ? ds_nd_field<T>(ndk) * kOnes : 0u;
            uint32_t ndc[8];
#pragma unroll
            for (int k = 0; k < 8; k++) ndc[k] = 0;
            const T *p = src + ya * ws + c;
            // rows are fetched kDsBatch at a time, ALL loads of a batch issued before the first is used (the rare
            // nodata branch below would otherwise keep the compiler from hoisting loads: 1-3 in flight per thread)
#ifndef HB_DS_BATCH
#define HB_DS_BATCH 10
#endif
            constexpr int kDsBatch = HB_DS_BATCH;
            for (long yb0 = ya; yb0 < yb; yb0 += kDsBatch) {
            uint32_t wb[kDsBatch][NW];
#pragma unroll
            for (int u = 0; u < kDsBatch; u++) {
                const T *pu = p + (yb0 + u < yb ? (long)u : yb - 1 - yb0) * ws;      // (clamped: re-reads the last row)
                if (sizeof(T) == 2) {
                    const uint4 v = hb_ldg_stream16(pu);
                    wb[u][0] = v.x; wb[u][1] = v.y; wb[u][NW > 2 ? 2 : 0] = v.z; wb[u][NW > 3 ? 3 : 0] = v.w;
                } else {
                    const uint2 v = hb_ldg_stream8(pu);
                    wb[u][0] = v.x; wb[u][1] = v.y;
                }
            }
            p += (long)kDsBatch * ws;
#pragma unroll
            for (int u = 0; u < kDsBatch; u++) {
                if (yb0 + u >= yb) break;
                uint32_t w[4];
#pragma unroll
                for (int i = 0; i < 4; i++) w[i] = (i < NW) ? wb[u][i] : 0u;
                uint32_t anyz = 0;
#pragma unroll
                for (int i = 0; i < NW; i++) {
                    if (sizeof(T) == 2) {
                        isum[2 * i] = ds_dp2a_lo<T>(w[i], 0x0001u, isum[2 * i]);
                        isum[2 * i + 1] = ds_dp2a_lo<T>(w[i], 0x0100u, isum[2 * i + 1]);
                    } else {
                        isum[4 * i] = __dp4a(w[i], 0x00000001u, isum[4 * i]);
                        isum[4 * i + 1] = __dp4a(w[i], 0x00000100u, isum[4 * i + 1]);
                        isum[4 * i + 2] = __dp4a(w[i], 0x00010000u, isum[4 * i + 2]);
                        isum[4 * i + 3] = __dp4a(w[i], 0x01000000u, isum[4 * i + 3]);
                    }
                    const uint32_t x = w[i] ^ ndpat;
                    anyz |= (x - kOnes) & ~x;
                }
                if (scan_nd && (anyz & kHigh)) {                            // rare: some pixel may be nodata
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        const uint32_t word = (sizeof(T) == 2) ? w[k >> 1] : w[k >> 2];
                        const uint32_t v = (sizeof(T) == 2) ? ((word >> (16 * (k & 1))) & 0xFFFFu)
                                                            : ((word >> (8 * (k & 3))) & 0xFFu);
                        ndc[k] += (v == ds_nd_field<T>(ndk)) ? 1u : 0u;
                    }
                }
            }
            }
            const uint32_t nrows = (uint32_t)(yb > ya ? yb - ya : 0);
#pragma unroll
            for (int k = 0; k < 8; k++) {
                colsum[k] = ds_sum<T>(isum[k] - (scan_nd ? (uint32_t)ndk.ivalue * ndc[k] : 0u));
                colw[k] = (double)(nrows - ndc[k]);
            }
        } else {
#pragma unroll 4
            for (long y = ya; y < yb; y++) {
                T v[8]; uint32_t inb;
                ds_fetch<T, ALIGNED>(src + y * ws, c, ws, v, inb);
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const bool ok = ((inb >> k) & 1u) && ds_valid<T>(v[k], ndk);
                    isum[k] += ok ? (uint32_t)v[k] : 0u;
                    icnt[k] += ok ? 1u : 0u;
                }
            }
#pragma unroll
            for (int k = 0; k < 8; k++) { colsum[k] = ds_sum<T>(isum[k]); colw[k] = (double)icnt[k]; }
        }
    } else {
        uint32_t icnt[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { colsum[k] = 0.0; icnt[k] = 0; }
        if (ALIGNED && c >= 0 && c + 8 <= ws) {
            // fast path (every vector of this thread inside the raster): 5 rows = ten 16-byte loads issued together
            constexpr int kFb = 5;
            const T *p = src + ya * ws + c;
            for (long yb0 = ya; yb0 < yb; yb0 += kFb) {
                uint4 raw[kFb][2];
#pragma unroll
                for (int u = 0; u < kFb; u++) {
                    const T *pu = p + (yb0 + u < yb ? (long)u : yb - 1 - yb0) * ws;   // (clamped: re-reads the last row)
                    raw[u][0] = hb_ldg_stream16(pu);
                    raw[u][1] = hb_ldg_stream16(pu + 4);
                }
                p += (long)kFb * ws;
#pragma unroll
                for (int u = 0; u < kFb; u++) {
                    if (yb0 + u >= yb) break;
                    const float v[8] = {__uint_as_float(raw[u][0].x), __uint_as_float(raw[u][0].y),
                                        __uint_as_float(raw[u][0].z), __uint_as_float(raw[u][0].w),
                                        __uint_as_float(raw[u][1].x), __uint_as_float(raw[u][1].y),
                                        __uint_as_float(raw[u][1].z), __uint_as_float(raw[u][1].w)};
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        const bool ok = hb_valid(v[k], ndk);
                        colsum[k] += ok ? (double)v[k] : 0.0;
                        icnt[k] += ok ? 1u : 0u;
                    }
                }
            }
        } else {
#pragma unroll 4
            for (long y = ya; y < yb; y++) {
                T v[8]; uint32_t inb;
                ds_fetch<T, ALIGNED>(src + y * ws, c, ws, v, inb);
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const bool ok = ((inb >> k) & 1u) && ds_valid<T>(v[k], ndk);
                    colsum[k] += ok ? (double)v[k] : 0.0;
                    icnt[k] += ok ? 1u : 0u;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) colw[k] = (double)icnt[k];
    }
    // fractionally covered first / last rows
    if (first_frac || last_frac) {
#pragma unroll 1
        for (int e = 0; e < 2; e++) {
            if ((e == 0 && !first_frac) || (e == 1 && !last_frac)) continue;
            const long y = (e == 0) ? iy0u : iy1u - 1;
            const double wy = (e == 0) ? wy_first : wy_last;
            T v[8]; uint32_t inb;
            ds_fetch<T, ALIGNED>(src + y * ws, c, ws, v, inb);
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const bool ok = ((inb >> k) & 1u) && ds_valid<T>(v[k], ndk);
                if (ok) { colsum[k] += wy * (double)v[k]; colw[k] += wy; }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; k++) { s_sum[t * kDsVec + k] = colsum[k]; s_w[t * kDsVec + k] = colw[k]; }
    __syncthreads();

    // ---- phase 2: one thread per destination pixel ----------------------------------------------------------------
    for (long j = j0 + t; j < j1; j += kDsThreads) {
        const HbFootprint fx = hb_footprint(sx, ox, j);
        const long ix0u = fx.a0, ix1u = fx.b0;
        const long ix0 = max(ix0u, 0L), ix1 = min(ix1u, ws);
        float out = qnan;
        double total = 0.0, total_w = 0.0;
        // neighbouring threads start `ratio` columns apart: rotate each thread's starting column so that the 64-bit
        // shared-memory reads of a warp spread over the banks (the sum is over the same terms, in a fixed order)
        const long ncol = ix1 - ix0;
        long x = ix0 + ((ncol > 0) ? (long)(t % (int)ncol) : 0);
        for (long it = 0; it < ncol; it++) {
            double wx = 1.0;
            if (x == ix0u) wx = (ix0u + 1 == ix1u) ? 1.0 : 1.0 - (fx.lo - (double)ix0u);
            else if (x + 1 == ix1u) wx = 1.0 - ((double)ix1u - fx.hi);
            const int s = (int)(x - c_base);
            total += wx * s_sum[s];
            total_w += wx * s_w[s];
            if (++x == ix1) x = ix0;
        }
        if (total_w > 0.0) out = (float)(total / total_w);
        dst[i * wd + j] = out;
    }
}

// ---- integer sources on aligned grids with an integer ratio (the benchmark configurations; any "aerial image against a
//      coarser, snapped reference" case) ------------------------------------------------------------------------------------
// Every destination pixel is then the exact box of ry x rx source pixels (all GDAL weights are 1), and with rx a multiple
// of the G = 2 (uint16 / int16) / 4 (uint8) pixels of a 32-bit word no word straddles two destination pixels.  The kernel
// is instruction-issue bound, not DRAM bound, in its general form (ncu: 9.6 lane-instructions per pixel, issue-active ~45 %),
// so this variant spends as few instructions per WORD as it can:
//   * one integer dot-product per word sums its G pixels at once (dp2a / dp4a against all-ones);
//   * nodata is not counted per pixel: a packed running minimum of (word ^ nodata pattern) -- one min.u16x2 per word --
//     tells after the loop whether ANY field of the thread's columns was nodata; only then are the rows re-read (L2
//     hits) and counted exactly.  sum(valid) = sum(all) - nodata * count(nodata), count(valid) = all - count(nodata);
//   * whole batches of rows are loaded without per-row clamps; the footprint rows are exactly ry;
//   * the per-destination-pixel combination is a shared-memory integer atomic per thread and destination pixel (at most
//     two per thread) instead of a serial loop over the footprint columns.
// Sums are exact integers, so the result is bit-identical to the general kernel's (and to GDAL's double accumulation).
template <typename T, bool NDSCAN>
__global__ void __launch_bounds__(kDsThreads, 4)
downsample_int_aligned_kernel(const T *__restrict__ src, long ws, NoData nd, float *__restrict__ dst, long wd, int rx,
                              int ry, long cx0, long cy0, int ndc, int chunks)
{
    constexpr int NW = (sizeof(T) == 2) ? 4 : 2;                           // 32-bit words per thread and row (8 pixels)
    constexpr int G = 4 / (int)sizeof(T);                                  // pixels per word
    constexpr uint32_t kOnes = (sizeof(T) == 2) ? 0x00010001u : 0x01010101u;
    constexpr uint32_t kHigh = (sizeof(T) == 2) ? 0x80008000u : 0x80808080u;
    __shared__ unsigned int s_sum[kDsSpan / 8 + 8], s_cnt[kDsSpan / 8 + 8];   // per destination pixel of this CTA (rx >= 8)

    const long i = blockIdx.x / chunks;
    const int chunk = (int)(blockIdx.x % chunks);
    const long j0 = (long)chunk * ndc;
    const int nj = (int)min((long)ndc, wd - j0);
    const int t = threadIdx.x;
    for (int k = t; k < nj; k += kDsThreads) { s_sum[k] = 0u; s_cnt[k] = 0u; }
    __syncthreads();

    const long c_first = cx0 + j0 * rx;                                    // first source column of this CTA's footprint
    const long c_base = (c_first / kDsVec) * kDsVec;                       // 16-byte aligned start of the staged span
    const long c = c_base + (long)t * kDsVec;                              // this thread's 8 columns
    const long c_end = c_first + (long)nj * rx;                            // one past the footprint's last column
    const uint32_t ndpat = NDSCAN ? ds_nd_field<T>(nd) * kOnes : 0u;
    if (c + kDsVec > c_first && c < c_end) {                               // (threads wholly outside the footprint idle)
        uint32_t acc[NW], mn[NW];
#pragma unroll
        for (int w = 0; w < NW; w++) { acc[w] = 0u; mn[w] = 0xFFFFFFFFu; }
        const T *p = src + (cy0 + i * ry) * ws + c;
        auto add_row = [&](const uint32_t (&w)[NW]) {
#pragma unroll
            for (int k = 0; k < NW; k++) {
                // (dp2a.lo multiplies the two 16-bit halves of the word by the two LOW BYTES of its second operand)
                if (sizeof(T) == 2) acc[k] = ds_dp2a_lo<T>(w[k], 0x0101u, acc[k]);
                else acc[k] = __dp4a(w[k], 0x01010101u, acc[k]);
                if (NDSCAN) {
                    const uint32_t x = w[k] ^ ndpat;
                    if (sizeof(T) == 2) asm("min.u16x2 %0, %0, %1;" : "+r"(mn[k]) : "r"(x));
                    else mn[k] &= ~((x - kOnes) & ~x);                   // (a cleared high bit marks "some byte was zero")
                }
            }
        };
        auto load_row = [&](const T *q, uint32_t (&w)[NW]) {
            if (sizeof(T) == 2) { const uint4 v = hb_ldg_stream16(q); w[0] = v.x; w[1] = v.y; w[NW > 2 ? 2 : 0] = v.z; w[NW > 3 ? 3 : 0] = v.w; }
            else { const uint2 v = hb_ldg_stream8(q); w[0] = v.x; w[1] = v.y; }
        };
        constexpr int B = 10;
        int r = 0;
        for (; r + B <= ry; r += B) {                                      // whole batches: all loads issued before the first use
            uint32_t wb[B][NW];
#pragma unroll
            for (int u = 0; u < B; u++) load_row(p + (long)(r + u) * ws, wb[u]);
#pragma unroll
            for (int u = 0; u < B; u++) add_row(wb[u]);
        }
        for (; r < ry; r++) { uint32_t w1[NW]; load_row(p + (long)r * ws, w1); add_row(w1); }
        // nodata fields seen?  (uint16: a zero half-word in the running minimum; uint8: a cleared marker bit)
        uint32_t ndcnt[NW];
#pragma unroll
        for (int k = 0; k < NW; k++) ndcnt[k] = 0u;
        if (NDSCAN) {
            bool any = false;
#pragma unroll
            for (int k = 0; k < NW; k++) {
                if (sizeof(T) == 2) any = any || (((mn[k] - kOnes) & ~mn[k] & kHigh) != 0u);
                else any = any || ((mn[k] & kHigh) != kHigh);
            }
            if (any) {                                                     // rare: count the nodata pixels exactly (rows are L2 hits)
                for (int rr = 0; rr < ry; rr++) {
                    uint32_t w1[NW];
                    load_row(p + (long)rr * ws, w1);
#pragma unroll
                    for (int k = 0; k < NW; k++) {
#pragma unroll
                        for (int f = 0; f < G; f++) {
                            const uint32_t v = (w1[k] >> (f * 8 * (int)sizeof(T))) & ((sizeof(T) == 2) ? 0xFFFFu : 0xFFu);
                            ndcnt[k] += (v == ds_nd_field<T>(nd)) ? 1u : 0u;
                        }
                    }
                }
            }
        }
        // every word lies inside ONE destination pixel (rx % G == 0, cx0 % G == 0): merge this thread's words per
        // destination pixel and add them with one shared-memory atomic each
        int jprev = -1;
        uint32_t psum = 0u, pcnt = 0u;
#pragma unroll
        for (int k = 0; k < NW; k++) {
            const long col = c + (long)k * G;
            const bool inside = (col >= c_first) && (col < c_end);
            const int jd = inside ? (int)((col - c_first) / rx) : -1;
            const uint32_t vs = acc[k] - (NDSCAN ? (uint32_t)nd.ivalue * ndcnt[k] : 0u);
            const uint32_t vc = (uint32_t)(G * ry) - ndcnt[k];
            if (jd != jprev) {
                if (jprev >= 0) { atomicAdd(&s_sum[jprev], psum); atomicAdd(&s_cnt[jprev], pcnt); }
                jprev = jd; psum = 0u; pcnt = 0u;
            }
            if (inside) { psum += vs; pcnt += vc; }
        }
        if (jprev >= 0) { atomicAdd(&s_sum[jprev], psum); atomicAdd(&s_cnt[jprev], pcnt); }
    }
    __syncthreads();
    const float qnan = __int_as_float(0x7fc00000);
    for (int k = t; k < nj; k += kDsThreads) {
        const uint32_t n = s_cnt[k];
        dst[i * wd + j0 + k] = n ? (float)(ds_sum<T>(s_sum[k]) / (double)n) : qnan;
    }
}

template <typename T>
int launch_downsample(const void *src, long hs, long ws, NoData nd, float *dst, long hd, long wd, double sx, double ox,
                      double sy, double oy, cudaStream_t stream)
{
    // destination columns per CTA so that their footprint (plus alignment slack) fits the staged span
    long ndc = (long)floor(((double)kDsSpan - kDsVec - 2.0) / sx);
    HB_REQUIRE(ndc >= 1, "hb_downsample_average: down-sampling ratio %.1f is too large (max %d)", sx, kDsSpan - 10);
    if (ndc > wd) ndc = wd;
    const long chunks = (wd + ndc - 1) / ndc;
    const long blocks = hd * chunks;
    HB_REQUIRE(blocks > 0 && blocks < 2147483647L, "hb_downsample_average: grid too large");
    const bool aligned = ((ws * (long)sizeof(T)) % 16 == 0) && (((uintptr_t)src) % 16 == 0);
    if constexpr (IsInt<T>::value) {
        // integer ratio, integer offset, destination wholly inside the source, words never straddling destination pixels:
        // the exact-box kernel (see downsample_int_aligned_kernel)
        constexpr int G = 4 / (int)sizeof(T);
        const double rxd = floor(sx + 0.5), ryd = floor(sy + 0.5), oxd = floor(ox + 0.5), oyd = floor(oy + 0.5);
        const bool integral = fabs(sx - rxd) < 1e-12 && fabs(sy - ryd) < 1e-12 && fabs(ox - oxd) < 1e-9 && fabs(oy - oyd) < 1e-9;
        if (aligned && integral && rxd >= 8 && rxd <= 255 && ryd >= 1 && ryd <= 255 && ((long)rxd % G) == 0 &&
            oxd >= 0 && oyd >= 0 && ((long)oxd % G) == 0 && (long)oxd + wd * (long)rxd <= ws &&
            (long)oyd + hd * (long)ryd <= hs) {
            const bool ndscan = nd.has && nd.int_ok && (sizeof(T) == 2 || nd.ivalue <= 255);
            if (ndscan)
                downsample_int_aligned_kernel<T, true><<<(unsigned)blocks, kDsThreads, 0, stream>>>(
                    (const T *)src, ws, nd, dst, wd, (int)rxd, (int)ryd, (long)oxd, (long)oyd, (int)ndc, (int)chunks);
            else
                downsample_int_aligned_kernel<T, false><<<(unsigned)blocks, kDsThreads, 0, stream>>>(
                    (const T *)src, ws, nd, dst, wd, (int)rxd, (int)ryd, (long)oxd, (long)oyd, (int)ndc, (int)chunks);
            HB_LAUNCH_OK("downsample_int_aligned_kernel");
            return 0;
        }
    }
    if (aligned)
        downsample_average_kernel<T, true><<<(unsigned)blocks, kDsThreads, 0, stream>>>(
            (const T *)src, hs, ws, nd, dst, hd, wd, sx, ox, sy, oy, (int)ndc, (int)chunks);
    else
        downsample_average_kernel<T, false><<<(unsigned)blocks, kDsThreads, 0, stream>>>(
            (const T *)src, hs, ws, nd, dst, hd, wd, sx, ox, sy, oy, (int)ndc, (int)chunks);
    HB_LAUNCH_OK("downsample_average_kernel");
    return 0;
}

// =====================================================================================================================
// 2. element-wise kernels
// =====================================================================================================================
template <typename T>
__global__ void apply_same_grid_kernel(const T *__restrict__ src, NoData nd, int mask_src,
                                       const float *__restrict__ params, long n, void *__restrict__ corr, OutSpec os)
{
    const float qnan = __int_as_float(0x7fc00000);
    const long stride = (long)gridDim.x * blockDim.x;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float s = hb_to_f32<T>(src[i]);
        float r = __fadd_rn(__fmul_rn(__ldg(params + i), s), __ldg(params + n + i));   // kernel_model.py:461
        if (mask_src && !hb_valid(s, nd)) r = qnan;
        hb_store1_out(corr, i, r, os);                       // (output dtype conversion fused into the store)
    }
}

template <typename T>
__global__ void valid_mask_kernel(const T *__restrict__ src, long n, NoData nd, uint8_t *__restrict__ mask)
{
    const long stride = (long)gridDim.x * blockDim.x;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        mask[i] = hb_valid(hb_to_f32<T>(src[i]), nd) ? 1 : 0;
}

// ---- output dtype conversion (raster_array.py:353-387) ------------------------------------------------------------------
template <typename O> struct OutCvt;
template <> struct OutCvt<float> {
    static __device__ __forceinline__ float cvt(float v, float nd) { return isnan(v) ? nd : v; }
};
template <typename O> struct OutCvt {
    // np.round (half to even) in float32, clip to the integer range, cast; NaN -> nodata
    static __device__ __forceinline__ O cvt(float v, float nd)
    {
        constexpr float lo = std::is_signed<O>::value ? -32768.f : 0.f;
        constexpr float hi = sizeof(O) == 1 ? 255.f : (std::is_signed<O>::value ? 32767.f : 65535.f);
        const float r = fminf(fmaxf(rintf(v), lo), hi);
        return isnan(v) ? (O)nd : (O)(int)r;
    }
};

template <typename O>
__global__ void convert_dtype_kernel(const float *__restrict__ src, long n, float nd, O *__restrict__ dst)
{
    const long stride = (long)gridDim.x * blockDim.x;
    const long n4 = n / 4;
    const bool vec = (((uintptr_t)src) % 16 == 0) && (((uintptr_t)dst) % (4 * sizeof(O)) == 0);
    long done = 0;
    if (vec) {
        for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < n4; g += stride) {
            const uint4 raw = hb_ldg_stream16(src + 4 * g);
            const float v[4] = {__uint_as_float(raw.x), __uint_as_float(raw.y), __uint_as_float(raw.z),
                                __uint_as_float(raw.w)};
            struct __align__(4 * sizeof(O)) Pack { O o[4]; } pk;
#pragma unroll
            for (int k = 0; k < 4; k++) pk.o[k] = OutCvt<O>::cvt(v[k], nd);
            reinterpret_cast<Pack *>(dst)[g] = pk;
        }
        done = n4 * 4;
    }
    for (long i = done + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = OutCvt<O>::cvt(src[i], nd);
}

// ---- full-coverage mask (kernel_model.py:375-409) -------------------------------------------------------------------
// step 1: param pixel is "covered" iff it is valid and every in-range pixel of the other image's mask under its
//         footprint is valid (== GDAL average of the 0/1 mask is exactly 1) and the footprint is not empty.
__global__ void coverage_kernel(const uint8_t *__restrict__ in_mask, long hi, long wi, const float *__restrict__ params,
                                long hp, long wp, double sx, double ox, double sy, double oy,
                                uint8_t *__restrict__ covered)
{
    const long n = hp * wp;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long)gridDim.x * blockDim.x) {
        const long i = idx / wp, j = idx - i * wp;
        bool ok = !(isnan(params[idx]) && isnan(params[n + idx]));
        if (ok) {
            const HbFootprint fy = hb_footprint(sy, oy, i), fx = hb_footprint(sx, ox, j);
            const long iy0 = fy.a0, iy1 = fy.b0, ix0 = fx.a0, ix1 = fx.b0;
            // a footprint that leaves the other image's raster is covered by nodata there (boundless read)
            if (iy0 < 0 || ix0 < 0 || iy1 > hi || ix1 > wi) ok = false;
            for (long y = iy0; ok && y < iy1; y++)
                for (long x = ix0; x < ix1; x++)
                    if (!in_mask[y * wi + x]) { ok = false; break; }
        }
        covered[idx] = ok ? 1 : 0;
    }
}

// step 2: erosion with a (kh+2) x (kw+2) rectangle, zero border (cv.erode BORDER_CONSTANT 0, kernel_model.py:407-408)
__global__ void erode_kernel(const uint8_t *__restrict__ in, long h, long w, int eh, int ew, uint8_t *__restrict__ out)
{
    const long n = h * w;
    const int ry = eh / 2, rx = ew / 2;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long)gridDim.x * blockDim.x) {
        const long i = idx / w, j = idx - i * w;
        bool ok = (i - ry >= 0) && (i + ry < h) && (j - rx >= 0) && (j + rx < w);
        for (long y = i - ry; ok && y <= i + ry; y++)
            for (long x = j - rx; x <= j + rx; x++)
                if (!in[y * w + x]) { ok = false; break; }
        out[idx] = ok ? 1 : 0;
    }
}

}  // namespace

// =====================================================================================================================
// C-ABI
// =====================================================================================================================
extern "C" int hb_downsample_average(const void *src_dev, int src_dtype, long hs, long ws, int has_nodata,
                                     double nodata, float *dst_dev, long hd, long wd, double sx, double ox, double sy,
                                     double oy, void *stream)
{
    HB_REQUIRE(src_dev && dst_dev && hs > 0 && ws > 0 && hd > 0 && wd > 0, "hb_downsample_average: bad arguments");
    HB_REQUIRE(sx > 0 && sy > 0, "hb_downsample_average: grids must have the same orientation");
    const NoData nd = hb_make_nodata(has_nodata, nodata, src_dtype);
    cudaStream_t st = (cudaStream_t)stream;
    switch (src_dtype) {
        case HB_U8: return launch_downsample<uint8_t>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, st);
        case HB_U16: return launch_downsample<uint16_t>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, st);
        case HB_I16: return launch_downsample<int16_t>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, st);
        case HB_F32: return launch_downsample<float>(src_dev, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy, oy, st);
    }
    HB_REQUIRE(false, "hb_downsample_average: unknown dtype %d", src_dtype);
}

extern "C" int hb_apply_same_grid(const void *src_dev, int src_dtype, int has_nodata, double nodata, int mask_src,
                                  const float *params_dev, long h, long w, int out_dtype, int out_has_nodata,
                                  double out_nodata, void *corr_dev, void *stream)
{
    HB_REQUIRE(src_dev && params_dev && corr_dev && h > 0 && w > 0, "hb_apply_same_grid: bad arguments");
    HB_REQUIRE(hb_outspec_error(out_dtype, out_has_nodata, out_nodata) == nullptr, "hb_apply_same_grid: %s",
               hb_outspec_error(out_dtype, out_has_nodata, out_nodata));
    const NoData nd = hb_make_nodata(has_nodata, nodata, src_dtype);
    const OutSpec os = hb_make_outspec(out_dtype, out_has_nodata, out_nodata);
    cudaStream_t st = (cudaStream_t)stream;
    const long n = h * w;
    const unsigned grid = hb_grid_for(n, 256, 16);
    switch (src_dtype) {
        case HB_U8:
            apply_same_grid_kernel<uint8_t><<<grid, 256, 0, st>>>((const uint8_t *)src_dev, nd, mask_src, params_dev, n,
                                                                  corr_dev, os);
            break;
        case HB_U16:
            apply_same_grid_kernel<uint16_t><<<grid, 256, 0, st>>>((const uint16_t *)src_dev, nd, mask_src, params_dev,
                                                                   n, corr_dev, os);
            break;
        case HB_I16:
            apply_same_grid_kernel<int16_t><<<grid, 256, 0, st>>>((const int16_t *)src_dev, nd, mask_src, params_dev,
                                                                  n, corr_dev, os);
            break;
        case HB_F32:
            apply_same_grid_kernel<float><<<grid, 256, 0, st>>>((const float *)src_dev, nd, mask_src, params_dev, n,
                                                                corr_dev, os);
            break;
        default: HB_REQUIRE(false, "hb_apply_same_grid: unknown dtype %d", src_dtype);
    }
    HB_LAUNCH_OK("apply_same_grid_kernel");
    return 0;
}

extern "C" int hb_convert_dtype(const float *src_dev, long n, int out_dtype, int has_nodata, double nodata, void *dst_dev,
                                void *stream)
{
    HB_REQUIRE(src_dev && dst_dev && n > 0, "hb_convert_dtype: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const float nd = has_nodata ? (float)nodata : 0.f;
    const unsigned grid = hb_grid_for((n + 3) / 4, 256, 16);
    switch (out_dtype) {
        case HB_U8:
            HB_REQUIRE(!has_nodata || (nodata >= 0 && nodata <= 255 && nodata == floor(nodata)),
                       "hb_convert_dtype: nodata %g cannot be safely cast to uint8", nodata);
            convert_dtype_kernel<uint8_t><<<grid, 256, 0, st>>>(src_dev, n, nd, (uint8_t *)dst_dev);
            break;
        case HB_U16:
            HB_REQUIRE(!has_nodata || (nodata >= 0 && nodata <= 65535 && nodata == floor(nodata)),
                       "hb_convert_dtype: nodata %g cannot be safely cast to uint16", nodata);
            convert_dtype_kernel<uint16_t><<<grid, 256, 0, st>>>(src_dev, n, nd, (uint16_t *)dst_dev);
            break;
        case HB_I16:
            HB_REQUIRE(!has_nodata || (nodata >= -32768 && nodata <= 32767 && nodata == floor(nodata)),
                       "hb_convert_dtype: nodata %g cannot be safely cast to int16", nodata);
            convert_dtype_kernel<int16_t><<<grid, 256, 0, st>>>(src_dev, n, nd, (int16_t *)dst_dev);
            break;
        case HB_F32:
            convert_dtype_kernel<float><<<grid, 256, 0, st>>>(src_dev, n, has_nodata ? (float)nodata : __builtin_nanf(""),
                                                             (float *)dst_dev);
            break;
        default: HB_REQUIRE(false, "hb_convert_dtype: unsupported output dtype %d", out_dtype);
    }
    HB_LAUNCH_OK("convert_dtype_kernel");
    return 0;
}

extern "C" int hb_valid_mask(const void *src_dev, int src_dtype, long n, int has_nodata, double nodata,
                             uint8_t *mask_dev, void *stream)
{
    HB_REQUIRE(src_dev && mask_dev && n > 0, "hb_valid_mask: bad arguments");
    const NoData nd = hb_make_nodata(has_nodata, nodata, src_dtype);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = hb_grid_for(n, 256, 16);
    switch (src_dtype) {
        case HB_U8: valid_mask_kernel<uint8_t><<<grid, 256, 0, st>>>((const uint8_t *)src_dev, n, nd, mask_dev); break;
        case HB_U16:
            valid_mask_kernel<uint16_t><<<grid, 256, 0, st>>>((const uint16_t *)src_dev, n, nd, mask_dev);
            break;
        case HB_I16:
            valid_mask_kernel<int16_t><<<grid, 256, 0, st>>>((const int16_t *)src_dev, n, nd, mask_dev);
            break;
        case HB_F32: valid_mask_kernel<float><<<grid, 256, 0, st>>>((const float *)src_dev, n, nd, mask_dev); break;
        default: HB_REQUIRE(false, "hb_valid_mask: unknown dtype %d", src_dtype);
    }
    HB_LAUNCH_OK("valid_mask_kernel");
    return 0;
}

extern "C" int hb_full_coverage_mask(const uint8_t *in_mask_dev, long hi, long wi, const float *params_dev, long hp,
                                     long wp, double sx, double ox, double sy, double oy, int kh, int kw,
                                     uint8_t *out_dev, void *workspace_dev, void *stream)
{
    HB_REQUIRE(in_mask_dev && params_dev && out_dev && workspace_dev && hi > 0 && wi > 0 && hp > 0 && wp > 0,
               "hb_full_coverage_mask: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *covered = (uint8_t *)workspace_dev;
    coverage_kernel<<<hb_grid_for(hp * wp, 256), 256, 0, st>>>(in_mask_dev, hi, wi, params_dev, hp, wp, sx, ox, sy, oy,
                                                               covered);
    HB_LAUNCH_OK("coverage_kernel");
    erode_kernel<<<hb_grid_for(hp * wp, 256), 256, 0, st>>>(covered, hp, wp, kh + 2, kw + 2, out_dev);
    HB_LAUNCH_OK("erode_kernel");
    return 0;
}
