// upsample.cu -- GDAL GRA_CubicSpline up-sampling of parameter planes (sm_100a), behind two entry points:
//   * hb_upsample_apply : RefSpaceModel.apply = cubic-spline up-sampling of (gain, offset) fused with
//                         corr = gain*src + offset                        (kernel_model.py:484-503, 442-463)
//   * hb_resample_up    : plain cubic-spline / nearest up-sampling        (kernel_model.py:491, 497, 520)
//
// launch_upsample picks the kernel.  Aligned rasters >= ~1.6x finer than the coarse grid, with no coverage mask, take a
// fast path:
//   upsample_poly_kernel        fused up-sample + apply, >= ~3.4 destination pixels per coarse pixel (packed float32)
//   upsample_yfirst_kernel      fused up-sample + apply at smaller ratios (packed float32)
//   upsample_yfirst_f64_kernel  plain one-band up-sampling in double (SrcSpaceModel's reference up-sampling)
// Everything else -- small ratios, unaligned rasters, the coverage mask, plain two-band up-sampling, and the bilinear,
// cubic and lanczos methods -- runs on the general upsample_kernel.
//
// GDAL's rules are each written once and every kernel takes them from there: up_tap (a destination index's taps,
// fractional position and centre pixel), up_weights<METHOD> (the taps' weights) and gwk_normalise (GWKResample's
// weight-sum rule; up_normalise<METHOD> picks each method's rule).
//
// Replaces, for RefSpaceModel.apply (reference kernel_model.py:484-503): the GDAL GRA_CubicSpline warp of the gain and
// offset planes onto the source grid, the two float32 planes it writes, and numpy's gain*src + offset pass (:461).
// GDAL's algorithm is restated in oracle/gdal_restate.c (gr_cubic_spline_up); the fused fast paths evaluate the same
// interpolant with a different arithmetic organisation:
//
//   * Inside one coarse cell the interpolated surface is a bicubic polynomial.  A lane owns 4 adjacent destination
//     columns; whenever the tap rows change (once per `ratio` destination rows) it interpolates its 4 pixel COLUMNS
//     through the 4 tap rows with the columns' x-weights and keeps the 4 results per pixel column and band in
//     registers.  A destination row then costs 4 multiply-adds per pixel and band with the row's 4 y-weights (which
//     are per-row scalars from a small per-CTA table).  This is GDAL's sum of 16 weighted taps, re-associated; all
//     weights are positive, so there is no cancellation (a monomial-basis cubic in dy would save one operation but
//     cancels catastrophically next to parameter spikes).
//   * All of that is float32 arithmetic on PACKED pairs (FFMA2 / FADD2 / FMUL2: two adjacent pixels per
//     instruction), because the kernel is instruction-issue bound, not memory bound, when evaluated in double
//     (profiles/README.md, round 1).  B-spline weights are a convex combination, so float32 evaluation stays within a
//     few 1e-7 relative of GDAL's double accumulation -- inside the 1e-4 contract of BASELINE.json (tests:
//     test_upsample_apply, test_refspace_fuse_vs_oracle).  The geometry (tap indices, fractional offsets, weights)
//     is computed in double.
//   * A tiny pre-pass on the coarse grid classifies every cell: CLEAN (all 4x4 taps in range and valid in every
//     band: the polynomial form is exact, GDAL does not renormalise), DEAD (no destination pixel of the cell can
//     have a valid centre pixel: output is nodata) or DIRTY (anything else: taps dropped, weights renormalised).
//     Lanes touching a DIRTY cell store nothing; the DIRTY cells are appended to a list and a small fix-up kernel
//     re-does their destination pixels with GDAL's general rules in double, tap by tap.
//   * Source pixels arrive through a per-warp cp.async ring (each lane copies, and later reads, only its own bytes:
//     no barriers); one CTA barrier in total.
#include <limits.h>

#include <mutex>

#include "hb_common.cuh"

namespace {

// A small per-device pool of HIGH-PRIORITY side streams with a fork / join event pair each; nullptr when none could be
// made.  Pending kernels of equal priority are dispatched in launch order, so a small kernel launched behind a streaming
// kernel of another band only runs once that kernel has handed out all its CTAs; on a high-priority stream it slips in
// between.  The caller holds `mu` from the fork record to the join wait (a few host-side enqueues): the events of a slot
// are re-recorded by every user, so two host threads must not interleave on one slot.
struct SideStream { cudaStream_t s; cudaEvent_t fork, join; bool ok; std::mutex mu; };

SideStream *side_stream()
{
    constexpr int kPool = 8, kMaxDev = 64;
    static SideStream pool[kMaxDev][kPool];
    static bool made[kMaxDev] = {false};
    static unsigned next[kMaxDev] = {0};
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDev) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!made[dev]) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);             // (hi is the numerically smallest = highest priority)
        for (int i = 0; i < kPool; i++) {
            SideStream &ss = pool[dev][i];
            ss.ok = cudaStreamCreateWithPriority(&ss.s, cudaStreamNonBlocking, hi) == cudaSuccess &&
                    cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming) == cudaSuccess &&
                    cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming) == cudaSuccess;
        }
        cudaGetLastError();
        made[dev] = true;
    }
    SideStream *ss = &pool[dev][next[dev]++ % kPool];
    return ss->ok ? ss : nullptr;
}

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMinCtas = 2;                // resident CTAs per SM the streaming kernels are compiled for
constexpr int kPpt = 4;                    // destination pixels per lane
constexpr int kWarpW = 32 * kPpt;          // destination columns per warp
constexpr int kRb = 4;                     // rows per cp.async stage
constexpr int kStages = 4;                 // stages in flight per warp (kStages * kRb: a power of two)
constexpr int kMaxRows = 128;              // destination rows per CTA of the fast paths (upper bound)
constexpr int kRowTableBytes = kMaxRows * (16 + 4 + 4);   // per-CTA row table: 4 float y-weights + tap row + weight sum per row

// kernel parameters of the fast paths (the general kernel's are UpGeom)
struct UpPolyGeom {
    long hs, ws;              // destination (fine) grid
    long hp, wp;              // coarse grid
    double sx, ox, sy, oy;    // destination pixel index -> coarse pixel coordinate: c = s * (i + 0.5) + o
    OutSpec ospec;            // output dtype / nodata of the corrected plane (apply mode); plain float32 otherwise
};

// ---- packed float32 pairs -------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c)
{
    unsigned long long ua = *reinterpret_cast<unsigned long long *>(&a), ub = *reinterpret_cast<unsigned long long *>(&b),
                       uc = *reinterpret_cast<unsigned long long *>(&c), ud;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(ud) : "l"(ua), "l"(ub), "l"(uc));
    return *reinterpret_cast<float2 *>(&ud);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b)
{
    unsigned long long ua = *reinterpret_cast<unsigned long long *>(&a), ub = *reinterpret_cast<unsigned long long *>(&b), ud;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(ud) : "l"(ua), "l"(ub));
    return *reinterpret_cast<float2 *>(&ud);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b)
{
    unsigned long long ua = *reinterpret_cast<unsigned long long *>(&a), ub = *reinterpret_cast<unsigned long long *>(&b), ud;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(ud) : "l"(ua), "l"(ub));
    return *reinterpret_cast<float2 *>(&ud);
}
__device__ __forceinline__ float2 splat(float v) { return make_float2(v, v); }

// the same on values that LIVE in 64-bit registers (long-lived packed state: keeps the register allocator from
// scattering the halves of a pair, which costs two moves per use)
typedef unsigned long long pk2;
__device__ __forceinline__ pk2 pk(float lo, float hi)
{
    pk2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float pk_lo(pk2 v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); (void)hi; return lo; }
__device__ __forceinline__ float pk_hi(pk2 v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); (void)lo; return hi; }
__device__ __forceinline__ pk2 pk_fma(pk2 a, pk2 b, pk2 c) { pk2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ pk2 pk_mul(pk2 a, pk2 b) { pk2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// ---- geometry shared by the fast kernel and the fix-up kernel (identical expressions => identical cell indices) -----
__device__ __forceinline__ double up_src_coord(double scale, double off, long i) { return scale * ((double)i + 0.5) + off; }
__device__ __forceinline__ long up_cell(double scale, double off, long i)
{
    return (long)floor(up_src_coord(scale, off, i) - 0.5);
}

// first destination index i in [0, n] with up_cell(i) >= k (up_cell is monotone in i)
__device__ __forceinline__ long up_first_index(double scale, double off, long k, long n)
{
    long i = (long)floor(((double)k + 0.5 - off) / scale - 0.5) - 1;
    i = min(max(i, 0L), n);
    while (i < n && up_cell(scale, off, i) < k) i++;
    return i;
}

// GDAL's tap / centre geometry of destination index i along one axis of a coarse grid of n pixels: source coordinate
// c = s (i + 0.5) + o, first tap k - 1 with k = floor(c - 0.5), fractional position d = c - 0.5 - k in [0, 1); the
// centre pixel is floor(c + 1e-10), moved back to n - 1 when it is n, and `ok` says it exists (c >= 0, centre in
// [0, n)).  Every kernel takes its tap and centre indices from here, so that all of them agree on every pixel.
struct UpTap { double c, d; long k, centre; bool ok; };
__device__ __forceinline__ UpTap up_tap(double scale, double off, long i, long n)
{
    UpTap t;
    t.c = up_src_coord(scale, off, i);
    const double kd = floor(t.c - 0.5);
    t.k = (long)kd;
    t.d = t.c - 0.5 - kd;
    t.centre = (long)floor(t.c + 1e-10);
    if (t.centre == n) t.centre--;
    t.ok = (t.c >= 0.0) && t.centre >= 0 && t.centre < n;
    return t;
}

// ---- the up-sampling methods (spec: oracle/gdal_restate.c, oracle/interp_up_restate.c) ----------------------------
// Taps per axis: 6 for lanczos (k-2 .. k+3), 4 otherwise (k-1 .. k+2; bilinear uses the inner two).
__host__ __device__ constexpr int up_taps(int method) { return method == HB_UP_LANCZOS ? 6 : 4; }

// Weights of the up_taps(METHOD) taps at fractional position d in [0, 1): cubic spline: B(tap - d), the cubic B-spline;
// bilinear (0, 1-d, d, 0); cubic: Keys, a = -0.5; lanczos: L(i - d), i = -2 .. 3,
// L(t) = sin(pi t) sin(pi t / 3) / (pi^2 t^2 / 3), L(0) = 1.
template <int METHOD> __device__ __forceinline__ void up_weights(double d, double (&w)[up_taps(METHOD)])
{
    if constexpr (METHOD == HB_UP_CUBIC_SPLINE) {
        const double u = 1.0 - d, d2 = d * d, u2 = u * u;
        w[0] = u2 * u * (1.0 / 6.0);
        w[1] = (4.0 + d2 * (3.0 * d - 6.0)) * (1.0 / 6.0);
        w[2] = (4.0 + u2 * (3.0 * u - 6.0)) * (1.0 / 6.0);
        w[3] = d2 * d * (1.0 / 6.0);
    } else if constexpr (METHOD == HB_UP_BILINEAR) {
        w[0] = 0.0; w[1] = 1.0 - d; w[2] = d; w[3] = 0.0;
    } else if constexpr (METHOD == HB_UP_CUBIC) {
        w[0] = 0.5 * d * (-1.0 + d * (2.0 - d));
        w[1] = 1.0 + 0.5 * d * d * (-5.0 + 3.0 * d);
        w[2] = 0.5 * d * (1.0 + d * (4.0 - 3.0 * d));
        w[3] = 0.5 * d * d * (-1.0 + d);
    } else {
        // (sinpi: |t| < 4 needs no general argument reduction, and sin(pi t) of the six taps is +-sin(pi d))
        const double pi = 3.14159265358979323846;
        const double s = sinpi(d);
#pragma unroll
        for (int i = 0; i < 6; i++) {
            const double t = (double)(i - 2) - d;
            double l = 0.0;
            if (t == 0.0) l = 1.0;
            else if (fabs(t) < 3.0) l = ((i & 1) ? s : -s) * sinpi(t / 3.0) / (pi * pi * t * t / 3.0);
            w[i] = l;
        }
    }
}

// GWKResample's normalisation of a weighted sum `v` by its weight sum `w` (cubic spline, lanczos): false, the pixel is
// nodata, below 1e-6; divide unless within 1e-5 of 1.
__device__ __forceinline__ bool gwk_normalise(double &v, double w)
{
    if (w < 0.000001) return false;
    if (w < 0.99999 || w > 1.00001) v /= w;
    return true;
}

// GDAL's normalisation of a weighted sum `v` by its weight sum `w`; false: the pixel is nodata.  Bilinear / cubic's
// bilinear fallback (GWKBilinearResample4Sample): nodata below 1e-5, divide unless exactly 1.  Cubic spline and
// lanczos: GWKResample's rule.
template <int METHOD> __device__ __forceinline__ bool up_normalise(double &v, double w)
{
    if constexpr (METHOD == HB_UP_CUBIC_SPLINE || METHOD == HB_UP_LANCZOS) {
        return gwk_normalise(v, w);
    } else {
        if (w < 0.00001) return false;
        if (w != 1.0) v /= w;
        return true;
    }
}

// B-spline weights of one destination index along one axis with out-of-range taps zeroed, their sum, and whether no
// tap was dropped (for GDAL's exact rule on the PRODUCT of the two axis sums).  Returns the tap / centre geometry.
__device__ __forceinline__ UpTap up_axis_weights_raw(double scale, double off, long i, long n, double (&w)[4], double &sum,
                                                     bool &all_in)
{
    const UpTap tp = up_tap(scale, off, i, n);
    up_weights<HB_UP_CUBIC_SPLINE>(tp.d, w);
    sum = 0.0;
    all_in = true;
#pragma unroll
    for (int t = 0; t < 4; t++) {
        const long tap = tp.k - 1 + t;
        if (tap < 0 || tap >= n) { w[t] = 0.0; all_in = false; }
        sum += w[t];
    }
    return tp;
}

// The same with GDAL's edge rules folded in: the remaining weights are divided by their sum unless it is within 1e-5 of
// 1 (GWKResample's rule, applied per axis -- GDAL applies it to the product of the two axis sums; the two differ by
// <= 2e-5 relative, and only where taps are dropped on both axes); all weights are NaN when the pixel's centre coarse
// pixel is out of range (GDAL skips such pixels).  `k` returns the first tap index + 1.
__device__ __forceinline__ void up_axis_weights(double scale, double off, long i, long n, double (&w)[4], long &k)
{
    double sum;
    bool all_in;
    const UpTap tp = up_axis_weights_raw(scale, off, i, n, w, sum, all_in);
    k = tp.k;
    if (!tp.ok || sum < 0.99999 || sum > 1.00001) {         // (rare: only next to the raster's edges)
        const double norm = tp.ok ? 1.0 / sum : __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
        for (int t = 0; t < 4; t++) w[t] *= norm;
    }
}

// ---- cp.async (LDGSTS) ---------------------------------------------------------------------------------------------
template <int BYTES> __device__ __forceinline__ void cp_async_lane(uint32_t smem_dst, const void *gmem_src)
{
    if (BYTES == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_dst), "l"(gmem_src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- 4 source pixels of storage type T -> two float32 pairs + validity ---------------------------------------------
// Key: the nodata test, prepared once per thread (integer storage: the bit pattern of 2^23 + nodata, or a pattern no
// pixel can produce when the nodata value is not representable in the storage type).
template <typename T> struct SrcQuad;
template <> struct SrcQuad<uint16_t> {
    static constexpr int kBytes = 8;
    typedef uint32_t Key;
    static __device__ __forceinline__ Key key(const NoData &nd)
    {
        return (nd.ivalue >= 0 && nd.ivalue <= 65535) ? (0x4B000000u | (uint32_t)nd.ivalue) : 0xFFFFFFFFu;
    }
    static __device__ __forceinline__ void get_shared(uint32_t sa, const Key magic, float2 (&s)[2], bool (&ok)[4])
    {
        uint2 w;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(w.x), "=r"(w.y) : "r"(sa));
        // 2^23 + v has v in its mantissa: one byte-permute per pixel and one packed subtract per pair (exact)
        const float2 m0 = make_float2(__uint_as_float(__byte_perm(w.x, 0x4B000000u, 0x7410)),
                                      __uint_as_float(__byte_perm(w.x, 0x4B000000u, 0x7432)));
        const float2 m1 = make_float2(__uint_as_float(__byte_perm(w.y, 0x4B000000u, 0x7410)),
                                      __uint_as_float(__byte_perm(w.y, 0x4B000000u, 0x7432)));
        s[0] = fadd2(m0, splat(-8388608.0f));
        s[1] = fadd2(m1, splat(-8388608.0f));
        ok[0] = __float_as_uint(m0.x) != magic;
        ok[1] = __float_as_uint(m0.y) != magic;
        ok[2] = __float_as_uint(m1.x) != magic;
        ok[3] = __float_as_uint(m1.y) != magic;
    }
};
template <> struct SrcQuad<int16_t> {
    static constexpr int kBytes = 8;
    typedef uint32_t Key;
    static __device__ __forceinline__ Key key(const NoData &nd)
    {
        return nd.int_ok ? (0x4B000000u | (hb_nd_bits16(nd) ^ 0x8000u)) : 0xFFFFFFFFu;
    }
    static __device__ __forceinline__ void get_shared(uint32_t sa, const Key magic, float2 (&s)[2], bool (&ok)[4])
    {
        uint2 w;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(w.x), "=r"(w.y) : "r"(sa));
        // flipping the sign bits turns each field into v + 32768 (one LOP per two pixels); then as uint16, with
        // 2^23 + 32768 subtracted (exact)
        w.x ^= 0x80008000u;
        w.y ^= 0x80008000u;
        const float2 m0 = make_float2(__uint_as_float(__byte_perm(w.x, 0x4B000000u, 0x7410)),
                                      __uint_as_float(__byte_perm(w.x, 0x4B000000u, 0x7432)));
        const float2 m1 = make_float2(__uint_as_float(__byte_perm(w.y, 0x4B000000u, 0x7410)),
                                      __uint_as_float(__byte_perm(w.y, 0x4B000000u, 0x7432)));
        s[0] = fadd2(m0, splat(-8421376.0f));
        s[1] = fadd2(m1, splat(-8421376.0f));
        ok[0] = __float_as_uint(m0.x) != magic;
        ok[1] = __float_as_uint(m0.y) != magic;
        ok[2] = __float_as_uint(m1.x) != magic;
        ok[3] = __float_as_uint(m1.y) != magic;
    }
};
template <> struct SrcQuad<uint8_t> {
    static constexpr int kBytes = 4;
    typedef uint32_t Key;
    static __device__ __forceinline__ Key key(const NoData &nd)
    {
        return (nd.ivalue >= 0 && nd.ivalue <= 255) ? (0x4B000000u | (uint32_t)nd.ivalue) : 0xFFFFFFFFu;
    }
    static __device__ __forceinline__ void get_shared(uint32_t sa, const Key magic, float2 (&s)[2], bool (&ok)[4])
    {
        uint32_t w;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(sa));
        const float2 m0 = make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7440)),
                                      __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7441)));
        const float2 m1 = make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7442)),
                                      __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7443)));
        s[0] = fadd2(m0, splat(-8388608.0f));
        s[1] = fadd2(m1, splat(-8388608.0f));
        ok[0] = __float_as_uint(m0.x) != magic;
        ok[1] = __float_as_uint(m0.y) != magic;
        ok[2] = __float_as_uint(m1.x) != magic;
        ok[3] = __float_as_uint(m1.y) != magic;
    }
};
template <> struct SrcQuad<float> {
    static constexpr int kBytes = 16;
    typedef NoData Key;
    static __device__ __forceinline__ Key key(const NoData &nd) { return nd; }
    static __device__ __forceinline__ void get_shared(uint32_t sa, const Key &nd, float2 (&s)[2], bool (&ok)[4])
    {
        float4 w;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w.x), "=f"(w.y), "=f"(w.z), "=f"(w.w) : "r"(sa));
        s[0] = make_float2(w.x, w.y);
        s[1] = make_float2(w.z, w.w);
        ok[0] = hb_valid(w.x, nd); ok[1] = hb_valid(w.y, nd); ok[2] = hb_valid(w.z, nd); ok[3] = hb_valid(w.w, nd);
    }
};

// =====================================================================================================================
// pre-pass: classify the coarse cells, interleave the two bands, list the DIRTY cells
// =====================================================================================================================
// Cell (ky, kx), ky in [-1, hp], kx in [-1, wp]: the destination pixels whose first tap is (ky - 1, kx - 1).
// flags[(ky + 1) * (wp + 2) + (kx + 1)]: bit0 CLEAN, bit1 DEAD, bit2 OUT (DEAD because the centre pixels are out of range).
// A cell is only CLEAN if the gain band's taps are within a factor ~16 of each other.  Next to a parameter spike (an
// ill-conditioned solve of the reference, SURVEY.md 7.4-1) corr = gain*src + offset cancels heavily and float32
// interpolation errors would be amplified past 1e-4; such cells take the double-precision fix-up instead.
// One CTA = 32 x 8 cells.  The per-pixel facts (in range, usable in every band, valid in some band, binary exponent of
// |gain|) of the 35 x 11 coarse pixels under the tile's tap windows are packed into 16-bit words in shared memory once;
// every cell then combines its 4 x 4 window from there.
constexpr int kPrepW = 32, kPrepH = 8;

__global__ void __launch_bounds__(kPrepW * kPrepH)
upsample_prep_kernel(const float *__restrict__ coarse, long hp, long wp, float2 *__restrict__ coarse2,
                     uint8_t *__restrict__ flags, int *__restrict__ list, int *__restrict__ count)
{
    constexpr int TW = kPrepW + 3, TH = kPrepH + 3;
    __shared__ unsigned short s_px[TH][TW + 1];
    const long fw = wp + 2, plane = hp * wp;
    const long ky0 = (long)blockIdx.y * kPrepH - 1, kx0 = (long)blockIdx.x * kPrepW - 1;   // first cell of the tile
    // pixel tile: rows ky0 - 1 .. ky0 + kPrepH + 1, columns kx0 - 1 .. kx0 + kPrepW + 1
    for (int i = threadIdx.x; i < TW * TH; i += kPrepW * kPrepH) {
        const int ty = i / TW, tx = i % TW;
        const long y = ky0 - 1 + ty, x = kx0 - 1 + tx;
        unsigned v = 0;
        if (y >= 0 && y < hp && x >= 0 && x < wp) {
            const float g0 = __ldg(coarse + y * wp + x);
            const float g1 = __ldg(coarse + plane + y * wp + x);
            // (an infinite tap is data for GDAL; the fast path cannot multiply it by a zero weight: not usable)
            v = 4u | ((isfinite(g0) && isfinite(g1)) ? 1u : 0u) | ((!isnan(g0) || !isnan(g1)) ? 2u : 0u);
            if (!isnan(g0)) v |= 8u | (((__float_as_uint(g0) >> 23) & 0xFFu) << 8);
            // the interleaved copy is written by the tile that owns the pixel as a cell
            if (ty >= 1 && ty <= kPrepH && tx >= 1 && tx <= kPrepW) coarse2[y * wp + x] = make_float2(g0, g1);
        }
        s_px[ty][tx] = (unsigned short)v;
    }
    __syncthreads();
    const int cx = threadIdx.x % kPrepW, cy = threadIdx.x / kPrepW;
    const long ky = ky0 + cy, kx = kx0 + cx;
    const bool live = (ky <= hp) && (kx <= wp);
    // bit (j*4+i) of `all` = usable in every band, of `any` = valid in some band, of `inr` = inside the raster
    unsigned all = 0, any = 0, inr = 0;
    int emin = 255, emax = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const unsigned v = s_px[cy + j][cx + i];
            const unsigned bit = 1u << (j * 4 + i);
            if (v & 1u) all |= bit;
            if (v & 2u) any |= bit;
            if (v & 4u) inr |= bit;
            if (v & 8u) { emin = min(emin, (int)(v >> 8)); emax = max(emax, (int)(v >> 8)); }
        }
    }
    // centre-pixel candidates of the cell's destination pixels: rows {ky, ky+1} (+ ky-1 when ky == hp, GDAL's
    // "cy == hs -> cy--" rule), same for the columns; window bit (j, i) is row ky-1+j, column kx-1+i
    unsigned rows_m = 0x6u, cols_m = 0x6u;                      // j (i) in {1, 2}
    if (ky == hp) rows_m |= 0x1u;
    if (kx == wp) cols_m |= 0x1u;
    unsigned cand = 0;
#pragma unroll
    for (int j = 0; j < 4; j++)
        if ((rows_m >> j) & 1u) cand |= (cols_m & 0xFu) << (j * 4);
    const bool dead = (any & cand) == 0;                      // no destination pixel of the cell has a valid centre
    const bool outr = (inr & cand) == 0;                      // ... because no centre candidate is inside the raster
    // CLEAN: every tap inside the raster is usable in every band (taps outside it are handled by the edge weights);
    // and the gains' binary exponents differ by <= 3, i.e. their magnitudes by less than a factor 16
    const bool clean = !dead && (all == inr) && emax - emin <= 3;
    const long idx = (ky + 1) * fw + (kx + 1);
    if (live) flags[idx] = (uint8_t)((clean ? 1 : 0) | (dead ? 2 : 0) | (outr ? 4 : 0));
    // append the DIRTY cells: one atomic per warp
    const bool dirty = live && !clean && !dead;
    const unsigned vote = __ballot_sync(0xffffffffu, dirty);
    if (vote) {
        const int lane = threadIdx.x & 31, leader = __ffs(vote) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(count, __popc(vote));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (dirty) list[base + __popc(vote & ((1u << lane) - 1u))] = (int)idx;
    }
}

// =====================================================================================================================
// fast kernel
// =====================================================================================================================
struct __align__(16) RowEntry { float wy[4]; };            // the row's B-spline y-weights (taps ky-1 .. ky+2)

// upsample_poly_kernel's row table: everything a destination row needs in one 32-byte entry (one LDS.128 + one LDS.64)
struct __align__(32) PolyRow {
    float wy[4];    // the row's B-spline y-weights (taps ky-1 .. ky+2)
    int ky;         // first tap row + 1, clamped to [-4, hp + 4] (non-decreasing: sy > 0); INT_MAX past the CTA's rows
    float sy;       // sum of the y-weights: exactly 1.0f unless taps were dropped
    int pad[2];
};
constexpr int kPolyRowTableBytes = (kMaxRows + kRb - 1) * (int)sizeof(PolyRow);   // (+ pad entries of a partial stage)

// corr = up(gain) * src + up(offset).  T: storage type of the source plane; coarse2: interleaved (gain, offset) [hp][wp];
// CONVERT: an output dtype / nodata other than plain float32 (g.ospec).
// rows_per_cta (<= kMaxRows) is chosen by the host so that the grid fills whole waves.
template <typename T, bool CONVERT>
__global__ void __launch_bounds__(kThreads, kMinCtas)
upsample_poly_kernel(const T *__restrict__ src, NoData nd, const float2 *__restrict__ coarse2,
                     const uint8_t *__restrict__ flags, UpPolyGeom g, int rows_per_cta, float *__restrict__ out)
{
    constexpr int kLaneBytes = SrcQuad<T>::kBytes;
    constexpr int kRowBytes = 32 * kLaneBytes;
    constexpr int kStageBytes = kRb * kRowBytes;
    constexpr int kRingBytes = kStages * kStageBytes;
    constexpr int kWBytes = 6 * 32 * (int)sizeof(float4);                  // x-weights (+ their sums) of one warp
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long Y0 = (long)blockIdx.y * rows_per_cta;
    const int nrows = (int)min((long)rows_per_cta, g.hs - Y0);
    const float qnan = __int_as_float(0x7fc00000);

    // per-CTA row table of the CTA's destination rows, padded to whole stages (rows are processed a stage at a time)
    PolyRow *s_rows = reinterpret_cast<PolyRow *>(smem_raw);
    if ((int)threadIdx.x < nrows + kRb - 1) {
        PolyRow e = {{0.f, 0.f, 0.f, 0.f}, INT_MAX, 0.f, {0, 0}};
        if ((int)threadIdx.x < nrows) {
            double wy[4];
            long ky;
            up_axis_weights(g.sy, g.oy, Y0 + threadIdx.x, g.hp, wy, ky);
#pragma unroll
            for (int j = 0; j < 4; j++) e.wy[j] = (float)wy[j];
            e.ky = (int)min(max(ky, -4L), g.hp + 4);
            e.sy = (float)(((wy[0] + wy[1]) + wy[2]) + wy[3]);
        }
        s_rows[threadIdx.x] = e;
    }
    __syncthreads();                                        // the only CTA barrier

    const long X0 = ((long)blockIdx.x * kWarps + warp) * kWarpW + (long)lane * kPpt;
    if (X0 - lane * kPpt >= g.ws) return;                   // the whole warp is beyond the raster
    int lane_in_i = X0 < g.ws;                              // (ws % 4 == 0: a lane is wholly inside or outside)
    asm("" : "+r"(lane_in_i));                              // (kept in a register, not re-derived at every stage)
    const bool lane_in = lane_in_i != 0;
    unsigned char *warp_base = smem_raw + kPolyRowTableBytes + warp * (kWBytes + kRingBytes);
    float4 *s_w = reinterpret_cast<float4 *>(warp_base) + lane;            // s_w[i * 32]: tap i of the lane's 4 pixels
    const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(warp_base + kWBytes + lane * kLaneBytes);

    // ---- cp.async ring of source rows: every lane copies, and later reads, only its own 4 pixels ----------------------
    const long pitch_b = g.ws * (long)sizeof(T);
    const char *pf = reinterpret_cast<const char *>(src + Y0 * g.ws + X0);   // next row to prefetch
    int pf_left = nrows;
    uint32_t pf_dst = ring_sa;
    auto prefetch = [&]() {
        if (lane_in) {
            if (pf_left >= kRb) {
#pragma unroll
                for (int rr = 0; rr < kRb; rr++) {
                    cp_async_lane<kLaneBytes>(pf_dst + rr * kRowBytes, pf);
                    pf += pitch_b;
                }
            } else {                                        // (the CTA's last, partial stage)
#pragma unroll 1
                for (int rr = 0; rr < pf_left; rr++) {
                    cp_async_lane<kLaneBytes>(pf_dst + rr * kRowBytes, pf);
                    pf += pitch_b;
                }
            }
        }
        pf_left -= kRb;
        pf_dst = (pf_dst + kStageBytes == ring_sa + kRingBytes) ? ring_sa : pf_dst + kStageBytes;
        cp_async_commit();
    };
#pragma unroll
    for (int st = 0; st < kStages - 1; st++) prefetch();

    // ---- row-invariant lane geometry (double): edge-aware x-weights over the lane's 5-column tap window -> shared ------
    int col0 = 0;                                           // first tap column of the lane's window
    int cellA = 0, cellB = 0;                               // flag columns (kx + 1) of the lane's first / last pixel
    {
        float w5[kPpt][5], sx[kPpt];
        long kx0 = 0;
#pragma unroll
        for (int k = 0; k < kPpt; k++) {
            double wx[4];
            long kx;
            up_axis_weights(g.sx, g.ox, X0 + k, g.wp, wx, kx);
            sx[k] = (float)(((wx[0] + wx[1]) + wx[2]) + wx[3]);
            if (k == 0) kx0 = kx;
            const bool sh = (kx != kx0);                    // the pixel's window starts 0 or 1 column into the lane's
            if (k == kPpt - 1) cellB = (int)min(max(kx + 1, -1L), g.wp + 2);
            w5[k][0] = sh ? 0.f : (float)wx[0];
            w5[k][1] = (float)(sh ? wx[0] : wx[1]);
            w5[k][2] = (float)(sh ? wx[1] : wx[2]);
            w5[k][3] = (float)(sh ? wx[2] : wx[3]);
            w5[k][4] = sh ? (float)wx[3] : 0.f;
        }
        col0 = (int)min(max(kx0 - 1, -8L), g.wp + 8);
        cellA = (int)min(max(kx0 + 1, -1L), g.wp + 2);
#pragma unroll
        for (int i = 0; i < 5; i++) s_w[i * 32] = make_float4(w5[0][i], w5[1][i], w5[2][i], w5[3][i]);
        s_w[5 * 32] = make_float4(sx[0], sx[1], sx[2], sx[3]);
    }
    const int fw = (int)g.wp + 2, hp = (int)g.hp, wp = (int)g.wp;
    // cells outside the flag table hold no pixel with an in-range centre: DEAD
    auto cell_flags = [&](int ky, int cell) -> unsigned {
        if (ky < -1 || ky > hp || cell < 0 || cell >= fw) return 6u;
        return flags[(ky + 1) * fw + cell];
    };
    // the lane's tap columns; taps outside the raster have weight 0 (x-weights / row table): read the clamped position
    int coff[5];
#pragma unroll
    for (int i = 0; i < 5; i++) coff[i] = min(max(col0 + i, 0), wp - 1);
    const bool five = (cellB != cellA);                     // some pixel's window starts one column in: 5th column is used

    typename SrcQuad<T>::Key nd_key = SrcQuad<T>::key(nd);
    if constexpr (sizeof(nd_key) == 4) asm("" : "+r"(nd_key));   // (kept in a register, not re-derived at every row)
    // x-interpolated tap rows per pixel PAIR and band.  CLEAN lanes: the interpolated values; DEAD lanes: NaN (so that
    // the row arithmetic produces nodata by itself); DIRTY lanes / lanes beyond the raster: stale, never stored.
    //
    // The taps are interpolated RELATIVE TO A BASE VALUE `base` (the coarse pixel at the centre of the lane's window):
    //     sum_i w_i t_i  =  base * sum_i w_i  +  sum_i w_i (t_i - base)
    // The parameter planes are smooth, so the second term is small and its float32 rounding errors vanish against the
    // result, while the first is exact (sum_i w_i == 1.0f wherever no tap was dropped) -- the float32 parameter the
    // reference gets from GDAL's double-precision accumulation comes out correctly rounded in all but near-tie cases.
    float2 q[2][2][4];                                      // [pixel pair][band: gain, offset][tap row]
    float base[2];
    float2 base2[2];                                        // (base, base): an operand of every row's packed FMA
#pragma unroll
    for (int b = 0; b < 2; b++) base[b] = 0.f, base2[b] = splat(0.f);
    const float4 sx4 = s_w[5 * 32];
    int q_ky = INT_MIN;
    bool do_store = false;

    // ---- new tap rows `ky` (once per cell row): re-classify the lane, re-interpolate its pixel columns -----------------
    auto reinterpolate = [&](int ky) {
        q_ky = ky;
        const unsigned fa = cell_flags(ky, cellA), fb = cell_flags(ky, cellB);
        if (lane_in) {
            // next cell row's flags -> L1 (the flag load heads the dependency chain of every re-interpolation)
            const int nf = min(max(ky + 2, 0), hp + 1) * fw;
            asm volatile("prefetch.global.L1 [%0];" ::"l"(flags + nf + min(max(cellA, 0), fw - 1)));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(flags + nf + min(max(cellB, 0), fw - 1)));
        }
        // 0: CLEAN, 1: SKIP (DIRTY: left to the fix-up kernel; or a lane beyond the raster), 2: DEAD.
        // A CLEAN cell next to an OUT cell: the OUT cell's pixel columns carry NaN x-weights.
        const bool clean2 = ((fa | fb) & 1u) && (fa & 5u) && (fb & 5u);
        const int state = !lane_in ? 1 : (clean2 ? 0 : ((fa & fb & 2u) ? 2 : 1));
        do_store = (state != 1);
        if (state == 2) {
#pragma unroll
            for (int p = 0; p < 2; p++)
#pragma unroll
                for (int b = 0; b < 2; b++)
#pragma unroll
                    for (int j = 0; j < 4; j++) q[p][b][j] = splat(qnan);
        }
        if (lane_in) {
            // the NEXT cell row re-uses 3 of these tap rows (L1 hits by then); pull its one new row into L1 now, so
            // that the whole CTA does not stall on L2 at its next (simultaneous) re-interpolation
            const int nrow = min(max(ky + 3, 0), hp - 1) * wp + coff[0];
            const float2 *np = coarse2 + nrow;
            asm volatile("prefetch.global.L1 [%0];" ::"l"(np));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(np + 4));
        }
        if (state == 0) {
            float2 wp01[5], wp23[5];
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const float4 w = s_w[i * 32];
                wp01[i] = make_float2(w.x, w.y);
                wp23[i] = make_float2(w.z, w.w);
            }
            {
                // base: the coarse pixel at tap row 1, tap column 1 of the lane's window (inside the raster, hence
                // usable in a CLEAN cell)
                const int boff = min(max(ky, 0), hp - 1) * wp + coff[1];
                const float2 v = __ldg(coarse2 + boff);
                base[0] = v.x;
                base[1] = v.y;
#pragma unroll
                for (int b = 0; b < 2; b++) base2[b] = splat(base[b]);
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int row_off = min(max(ky - 1 + j, 0), hp - 1) * wp;     // (hp * wp < 2^31: launch_poly)
                float t[2][5];
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    // (the 5th column has weight 0 when unused, but may be NaN: skip it)
                    const float2 v = (i < 4 || five) ? __ldg(coarse2 + (row_off + coff[i])) : make_float2(base[0], base[1]);
                    t[0][i] = __fsub_rn(v.x, base[0]);
                    t[1][i] = __fsub_rn(v.y, base[1]);
                }
#pragma unroll
                for (int b = 0; b < 2; b++) {              // x-interpolation of tap row j at the lane's 4 pixel columns
                    float2 r0 = fmul2(wp01[0], splat(t[b][0])), r1 = fmul2(wp23[0], splat(t[b][0]));
#pragma unroll
                    for (int i = 1; i < 5; i++) {
                        r0 = ffma2(wp01[i], splat(t[b][i]), r0);
                        r1 = ffma2(wp23[i], splat(t[b][i]), r1);
                    }
                    q[0][b][j] = r0;
                    q[1][b][j] = r1;
                }
            }
        }
    };

    // ---- one destination row: 4 multiply-adds per pixel pair and band with the row's y-weights, fused apply ------------
    // `rd`: the lane's source pixels of the row in the ring; `pix`: pixel index of the lane's 4 pixels in the output plane
    auto dest_row = [&](const PolyRow &e, uint32_t rd, long pix) {
        const float2 w0 = splat(e.wy[0]), w1 = splat(e.wy[1]), w2 = splat(e.wy[2]), w3 = splat(e.wy[3]);
        float2 gv[2], ov[2];
#pragma unroll
        for (int p = 0; p < 2; p++) {
            // weight sum of the pixel = (sum of its x-weights) * (sum of the row's y-weights): 1.0f away from the edges
            const float2 wsum = fmul2(p == 0 ? make_float2(sx4.x, sx4.y) : make_float2(sx4.z, sx4.w), splat(e.sy));
            const float2 dg = ffma2(q[p][0][3], w3, ffma2(q[p][0][2], w2, ffma2(q[p][0][1], w1, fmul2(q[p][0][0], w0))));
            gv[p] = ffma2(base2[0], wsum, dg);
            const float2 dof = ffma2(q[p][1][3], w3, ffma2(q[p][1][2], w2, ffma2(q[p][1][1], w1, fmul2(q[p][1][0], w0))));
            ov[p] = ffma2(base2[1], wsum, dof);
        }
        float2 s[2];
        bool ok[4];
        SrcQuad<T>::get_shared(rd, nd_key, s, ok);
        // corr = gain * src + offset as ONE fused multiply-add, rounded once (DESIGN.md 4.5)
        const float2 c0 = ffma2(gv[0], s[0], ov[0]), c1 = ffma2(gv[1], s[1], ov[1]);
        const float4 res = make_float4(ok[0] ? c0.x : qnan, ok[1] ? c0.y : qnan, ok[2] ? c1.x : qnan, ok[3] ? c1.y : qnan);
        if (do_store) {                                     // (DIRTY lanes are written by the fix-up kernel)
            if constexpr (CONVERT) hb_store4_out(out, pix, res, g.ospec);   // output dtype conversion in the store
            else hb_stg_stream16(out + pix, res);
        }
    };

    // ---- the rows, one ring stage (kRb rows) per iteration ----------------------------------------------------------------
    long opix = Y0 * g.ws + X0;
    const long out_pitch = g.ws;
#pragma unroll 1
    for (int r = 0; r < nrows; r += kRb, opix += kRb * out_pitch) {
        prefetch();                                         // keep the ring full, wait for this stage
        cp_async_wait<kStages - 1>();
        const uint32_t rd = ring_sa + (uint32_t)(r & (kStages * kRb - 1)) * kRowBytes;
        // (warp-uniform) the tap rows are non-decreasing in the row and q_ky is the previous row's: if the stage's last
        // row still has them, so does every row of the stage
        if (s_rows[r + kRb - 1].ky == q_ky) {
#pragma unroll
            for (int h = 0; h < kRb; h++) dest_row(s_rows[r + h], rd + h * kRowBytes, opix + h * out_pitch);
        } else {                                            // new tap rows in this stage, or the CTA's partial last stage
            const int n = min(kRb, nrows - r);
#pragma unroll 1
            for (int h = 0; h < n; h++) {
                const PolyRow e = s_rows[r + h];
                if (e.ky != q_ky) reinterpolate(e.ky);
                dest_row(e, rd + h * kRowBytes, opix + h * out_pitch);
            }
        }
    }
}

// =====================================================================================================================
// fast kernel for small ratios (about 1.6 .. 9 destination pixels per coarse pixel): "y first"
// =====================================================================================================================
// At small ratios the tap rows change every few destination rows and re-interpolating 4 pixel columns through them
// (upsample_poly_kernel) would dominate.  Here a lane keeps the 4 tap rows x 6 window columns of its 4 pixels in
// registers (shifted / reloaded when the tap rows change) and every destination row (1) combines the 4 tap rows with
// the row's y-weights per window column (packed over column pairs) and (2) combines the 6 columns with each pixel's
// x-weights (packed over pixel pairs; a pixel's 4 weights sit at its window offset 0..2 inside the 6-column window,
// zeros elsewhere).  Same classification / fix-up / edge rules / cp.async ring as upsample_poly_kernel.
constexpr int kYfCols = 6;

template <typename T, bool CONVERT>
__global__ void __launch_bounds__(kThreads, kMinCtas)
upsample_yfirst_kernel(const T *__restrict__ src, NoData nd, const float2 *__restrict__ coarse2,
                       const uint8_t *__restrict__ flags, UpPolyGeom g, int rows_per_cta, float *__restrict__ out)
{
    constexpr int kLaneBytes = SrcQuad<T>::kBytes;
    constexpr int kRowBytes = 32 * kLaneBytes;
    constexpr int kStageBytes = kRb * kRowBytes;
    constexpr int kRingBytes = kStages * kStageBytes;
    constexpr int kWBytes = kYfCols * 32 * (int)sizeof(float4);            // x-weights of one warp
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long Y0 = (long)blockIdx.y * rows_per_cta;
    const int nrows = (int)min((long)rows_per_cta, g.hs - Y0);
    const float qnan = __int_as_float(0x7fc00000);

    RowEntry *s_rows = reinterpret_cast<RowEntry *>(smem_raw);
    int *s_ky = reinterpret_cast<int *>(smem_raw + kMaxRows * sizeof(RowEntry));
    if ((int)threadIdx.x < nrows) {
        double wy[4];
        long ky;
        up_axis_weights(g.sy, g.oy, Y0 + threadIdx.x, g.hp, wy, ky);
        RowEntry e;
#pragma unroll
        for (int j = 0; j < 4; j++) e.wy[j] = (float)wy[j];
        s_rows[threadIdx.x] = e;
        s_ky[threadIdx.x] = (int)min(max(ky, -4L), g.hp + 4);
    }
    __syncthreads();                                        // the only CTA barrier

    const long X0 = ((long)blockIdx.x * kWarps + warp) * kWarpW + (long)lane * kPpt;
    if (X0 - lane * kPpt >= g.ws) return;
    const bool lane_in = X0 < g.ws;
    unsigned char *warp_base = smem_raw + kRowTableBytes + warp * (kWBytes + kRingBytes);
    float4 *s_w = reinterpret_cast<float4 *>(warp_base) + lane;            // s_w[c * 32]: window column c, 4 pixels
    const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(warp_base + kWBytes + lane * kLaneBytes);

    const long pitch_b = g.ws * (long)sizeof(T);
    const char *pf = reinterpret_cast<const char *>(src + Y0 * g.ws + X0);
    int pf_left = nrows;
    uint32_t pf_dst = ring_sa;
    auto prefetch = [&]() {
        if (lane_in) {
            for (int rr = 0; rr < kRb; rr++) {
                if (rr < pf_left) cp_async_lane<kLaneBytes>(pf_dst + rr * kRowBytes, pf);
                pf += pitch_b;
            }
        }
        pf_left -= kRb;
        pf_dst = (pf_dst + kStageBytes == ring_sa + kRingBytes) ? ring_sa : pf_dst + kStageBytes;
        cp_async_commit();
    };
#pragma unroll
    for (int st = 0; st < kStages - 1; st++) prefetch();

    // ---- row-invariant lane geometry: edge-aware x-weights placed in the lane's 6-column window -> shared memory -------
    int col0 = 0, cellA = 0, ncell = 1;                     // first window column; first flag column; cells spanned
    bool geom_ok = lane_in;
    {
        float w6[kPpt][kYfCols];
        long kx0 = 0, kx3 = 0;
#pragma unroll
        for (int k = 0; k < kPpt; k++) {
            double wx[4];
            long kx;
            up_axis_weights(g.sx, g.ox, X0 + k, g.wp, wx, kx);
            if (k == 0) kx0 = kx;
            kx3 = kx;
            const long sh = kx - kx0;                       // 0 .. 2
            geom_ok = geom_ok && sh >= 0 && sh <= 2;
#pragma unroll
            for (int c = 0; c < kYfCols; c++) {
                const long i = c - sh;
                w6[k][c] = (i >= 0 && i < 4) ? (float)wx[i < 0 ? 0 : (i > 3 ? 3 : i)] : 0.f;
            }
        }
        col0 = (int)min(max(kx0 - 1, -8L), g.wp + 8);
        cellA = (int)min(max(kx0 + 1, -1L), g.wp + 2);
        ncell = (int)min(max(kx3 - kx0, 0L), 2L) + 1;
#pragma unroll
        for (int c = 0; c < kYfCols; c++) s_w[c * 32] = make_float4(w6[0][c], w6[1][c], w6[2][c], w6[3][c]);
    }
    const int fw = (int)g.wp + 2, hp = (int)g.hp, wp = (int)g.wp;
    auto cell_flags = [&](int ky, int cell) -> unsigned {
        if (ky < -1 || ky > hp || cell < 0 || cell >= fw) return 6u;
        return flags[(long)(ky + 1) * fw + cell];
    };
    int coff[kYfCols];                                      // clamped window columns (taps outside have weight 0)
#pragma unroll
    for (int c = 0; c < kYfCols; c++) coff[c] = min(max(col0 + c, 0), wp - 1);
    const int ncols_used = 3 + ncell;                       // columns beyond are never weighted: not read (may be NaN)

    const typename SrcQuad<T>::Key nd_key = SrcQuad<T>::key(nd);
    pk2 t[2][4][kYfCols / 2];                               // bands x tap rows x window column pairs (packed float32 pairs)
    int q_ky = INT_MIN;
    bool do_store = false;
    long opix = Y0 * g.ws + X0;                             // pixel index of the lane's 4 pixels in the output plane
    const long out_pitch = g.ws;
    uint32_t ring_rd = ring_sa;
    auto load_tap_row = [&](int ky, int j) {
        const long row_off = (long)min(max(ky - 1 + j, 0), hp - 1) * wp;
        float v[2][kYfCols];
#pragma unroll
        for (int c = 0; c < kYfCols; c++) {
            const float2 x = (c < ncols_used) ? __ldg(coarse2 + row_off + coff[c]) : make_float2(0.f, 0.f);
            v[0][c] = x.x; v[1][c] = x.y;
        }
#pragma unroll
        for (int b = 0; b < 2; b++)
#pragma unroll
            for (int p = 0; p < kYfCols / 2; p++) t[b][j][p] = pk(v[b][2 * p], v[b][2 * p + 1]);
    };
#pragma unroll 1
    for (int r = 0; r < nrows; r++, opix += out_pitch) {
        if ((r & (kRb - 1)) == 0) {
            prefetch();
            cp_async_wait<kStages - 1>();
        }
        const int ky = s_ky[r];
        if (ky != q_ky) {                                   // (warp-uniform) new tap rows
            // 0: CLEAN, 1: SKIP (DIRTY -> fix-up kernel, or beyond the raster), 2: DEAD; the lane spans ncell cells
            unsigned f_or = 0, f_and = 7u;
            bool each_ok = true;                            // every cell CLEAN or OUT
            for (int c = 0; c < ncell; c++) {
                const unsigned f = cell_flags(ky, cellA + c);
                f_or |= f; f_and &= f;
                each_ok = each_ok && (f & 5u);
            }
            const int state = (!lane_in || !geom_ok) ? 1 : ((each_ok && (f_or & 1u)) ? 0 : ((f_and & 2u) ? 2 : 1));
            do_store = (state != 1);
            if (state == 2) {
#pragma unroll
                for (int b = 0; b < 2; b++)
#pragma unroll
                    for (int j = 0; j < 4; j++)
#pragma unroll
                        for (int p = 0; p < kYfCols / 2; p++) t[b][j][p] = pk(qnan, qnan);
            } else if (state == 0) {
                // (always reload all four rows: the lane may have been DEAD / DIRTY for the previous tap rows)
#pragma unroll
                for (int j = 0; j < 4; j++) load_tap_row(ky, j);
            }
            q_ky = ky;
        }
        // ---- one destination row ---------------------------------------------------------------------------------------
        const RowEntry ri = s_rows[r];
        pk2 A[2][kYfCols / 2];                              // y-combination per band and window column pair
        {
            const pk2 y0 = pk(ri.wy[0], ri.wy[0]), y1 = pk(ri.wy[1], ri.wy[1]), y2 = pk(ri.wy[2], ri.wy[2]),
                      y3 = pk(ri.wy[3], ri.wy[3]);
#pragma unroll
            for (int b = 0; b < 2; b++)
#pragma unroll
                for (int p = 0; p < kYfCols / 2; p++)
                    A[b][p] = pk_fma(t[b][3][p], y3, pk_fma(t[b][2][p], y2, pk_fma(t[b][1][p], y1, pk_mul(t[b][0][p], y0))));
        }
        pk2 o[2][2];                                        // per band, pixel pairs (0,1) and (2,3)
#pragma unroll
        for (int c = 0; c < kYfCols; c++) {
            const float4 w = s_w[c * 32];
            const pk2 w01 = pk(w.x, w.y), w23 = pk(w.z, w.w);
#pragma unroll
            for (int b = 0; b < 2; b++) {
                const float a = (c & 1) ? pk_hi(A[b][c / 2]) : pk_lo(A[b][c / 2]);
                const pk2 aa = pk(a, a);
                o[b][0] = (c == 0) ? pk_mul(w01, aa) : pk_fma(w01, aa, o[b][0]);
                o[b][1] = (c == 0) ? pk_mul(w23, aa) : pk_fma(w23, aa, o[b][1]);
            }
        }
        float2 s[2];
        bool ok[4];
        SrcQuad<T>::get_shared(ring_rd, nd_key, s, ok);
        ring_rd = (ring_rd + kRowBytes == ring_sa + kRingBytes) ? ring_sa : ring_rd + kRowBytes;
        // corr = gain * src + offset as ONE fused multiply-add, rounded once (DESIGN.md 4.5)
        const pk2 c0 = pk_fma(o[0][0], pk(s[0].x, s[0].y), o[1][0]);
        const pk2 c1 = pk_fma(o[0][1], pk(s[1].x, s[1].y), o[1][1]);
        const float4 res = make_float4(ok[0] ? pk_lo(c0) : qnan, ok[1] ? pk_hi(c0) : qnan, ok[2] ? pk_lo(c1) : qnan,
                                       ok[3] ? pk_hi(c1) : qnan);
        if (do_store) {
            if constexpr (CONVERT) hb_store4_out(out, opix, res, g.ospec);   // output dtype conversion in the store
            else hb_stg_stream16(out + opix, res);
        }
    }
}

// =====================================================================================================================
// plain up-sampling of ONE band in double precision ("y first" organisation)
// =====================================================================================================================
// SrcSpaceModel up-samples the reference image onto the source grid and FITS on the result (kernel_model.py:518-524).
// The reference's float32 numerator N*sum(sr) - sum(s)*sum(r) cancels catastrophically, so last-bit differences of the
// up-sampled pixels are amplified past 1e-4 in the parameters: this path must round like GDAL does -- double
// accumulation, one rounding to float32 -- and cannot use the packed-float32 kernels above.
struct __align__(16) RowEntryD { double wy[4]; double sum; double jc; };   // sum: NaN when the row's centre is out of range;
                                                                            // jc: tap row (0..3) of the centre coarse row, -1: none
// Self-contained (no classification pre-pass, no fix-up kernel): a lane keeps the 4 tap rows x 6 window columns of its 4
// pixels in registers -- when the tap rows advance by one coarse row (every `ratio` destination rows) the window is
// SHIFTED and only the new row is loaded -- and evaluates every destination row with the fast separable formula (all
// taps valid).  A NaN result means some tap was invalid (or the pixel has no valid centre): those pixels, and only
// those, are re-evaluated from the same registers with GDAL's general rule (invalid / out-of-range taps dropped,
// renormalised unless the remaining weights sum to 1 within 1e-5, nodata when the centre coarse pixel is invalid or the
// weights sum to < 1e-6), in the accumulation order of the fix-up kernel of the two-band path.
__global__ void __launch_bounds__(kThreads, kMinCtas)
upsample_yfirst_f64_kernel(const float *__restrict__ coarse, UpPolyGeom g, int rows_per_cta, float *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long Y0 = (long)blockIdx.y * rows_per_cta;
    const int nrows = (int)min((long)rows_per_cta, g.hs - Y0);
    const double dnan = __longlong_as_double(0x7ff8000000000000LL);

    RowEntryD *s_rows = reinterpret_cast<RowEntryD *>(smem_raw);
    int *s_ky = reinterpret_cast<int *>(smem_raw + kMaxRows * sizeof(RowEntryD));
    if ((int)threadIdx.x < nrows) {
        RowEntryD e;
        bool all_in;
        const UpTap ty = up_axis_weights_raw(g.sy, g.oy, Y0 + threadIdx.x, g.hp, e.wy, e.sum, all_in);
        if (all_in) e.sum = 1.0;                            // (the four weights sum to 1 up to rounding)
        if (!ty.ok) e.sum = dnan;
        const long jc = ty.centre - (ty.k - 1);
        e.jc = (ty.ok && jc >= 0 && jc <= 3) ? (double)jc : -1.0;
        s_rows[threadIdx.x] = e;
        s_ky[threadIdx.x] = (int)min(max(ty.k, -4L), g.hp + 4);
    }
    __syncthreads();

    const long X0 = ((long)blockIdx.x * kWarps + warp) * kWarpW + (long)lane * kPpt;
    if (X0 >= g.ws) return;                                 // (ws % 4 == 0: a lane is wholly inside or outside)
    // x-weights of the warp: s_w[(c * 2 + h) * 32 + lane] = window column c, pixels (2h, 2h + 1), as double2
    double2 *s_w = reinterpret_cast<double2 *>(smem_raw + kMaxRows * (sizeof(RowEntryD) + sizeof(int)) +
                                               warp * (kYfCols * 2 * 32 * sizeof(double2))) + lane;
    int col0 = 0, ncell = 1;
    int cc[kPpt];                                           // window column of every pixel's centre coarse pixel (-1: none)
    double xsum[kPpt];                                      // sum of the in-range x-weights per pixel (NaN: centre out of range)
    {
        double w6[kPpt][kYfCols];
        long kx0 = 0, kx3 = 0;
#pragma unroll
        for (int k = 0; k < kPpt; k++) {
            double wx[4];
            bool all_in;
            const UpTap tx = up_axis_weights_raw(g.sx, g.ox, X0 + k, g.wp, wx, xsum[k], all_in);
            if (all_in) xsum[k] = 1.0;
            if (!tx.ok) xsum[k] = dnan;
            const long kx = tx.k;
            if (k == 0) kx0 = kx;
            kx3 = kx;
            const long sh = kx - kx0;                       // 0 .. 2 (>= 1.6 destination pixels per coarse pixel)
#pragma unroll
            for (int c = 0; c < kYfCols; c++) {
                const long i = c - sh;
                w6[k][c] = (i >= 0 && i < 4) ? wx[i < 0 ? 0 : (i > 3 ? 3 : i)] : 0.0;
            }
            const long ci = tx.centre - (kx0 - 1);
            cc[k] = (tx.ok && ci >= 0 && ci < kYfCols) ? (int)ci : -1;
        }
        col0 = (int)min(max(kx0 - 1, -8L), g.wp + 8);
        ncell = (int)min(max(kx3 - kx0, 0L), 2L) + 1;
#pragma unroll
        for (int c = 0; c < kYfCols; c++) {
            s_w[(c * 2 + 0) * 32] = make_double2(w6[0][c], w6[1][c]);
            s_w[(c * 2 + 1) * 32] = make_double2(w6[2][c], w6[3][c]);
        }
    }
    const int hp = (int)g.hp, wp = (int)g.wp;
    int coff[kYfCols];
#pragma unroll
    for (int c = 0; c < kYfCols; c++) coff[c] = min(max(col0 + c, 0), wp - 1);
    const int ncols_used = 3 + ncell;
    auto load_tap_row = [&](int row, double (&dst)[kYfCols]) {
        // (rows / columns outside the raster carry weight 0: read the clamped position)
        const float *p = coarse + (long)min(max(row, 0), hp - 1) * wp;
#pragma unroll
        for (int c = 0; c < kYfCols; c++) dst[c] = (c < ncols_used) ? (double)__ldg(p + coff[c]) : 0.0;
    };

    const bool x_plain = (xsum[0] == 1.0) && (xsum[1] == 1.0) && (xsum[2] == 1.0) && (xsum[3] == 1.0);
    double t[4][kYfCols];
    int q_ky = INT_MIN;
    float *orow = out + Y0 * g.ws + X0;
#pragma unroll 1
    for (int r = 0; r < nrows; r++, orow += g.ws) {
        const int ky = s_ky[r];
        if (ky != q_ky) {                                   // (warp-uniform)
            if (ky == q_ky + 1) {                           // one coarse row further: shift the window, load the new row
#pragma unroll
                for (int j = 0; j < 3; j++)
#pragma unroll
                    for (int c = 0; c < kYfCols; c++) t[j][c] = t[j + 1][c];
                load_tap_row(ky + 2, t[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) load_tap_row(ky - 1 + j, t[j]);
            }
            q_ky = ky;
        }
        const RowEntryD ri = s_rows[r];
        double A[kYfCols];
#pragma unroll
        for (int c = 0; c < kYfCols; c++)
            A[c] = fma(t[3][c], ri.wy[3], fma(t[2][c], ri.wy[2], fma(t[1][c], ri.wy[1], t[0][c] * ri.wy[0])));
        double o[kPpt];
#pragma unroll
        for (int c = 0; c < kYfCols; c++) {
            const double2 w01 = s_w[(c * 2 + 0) * 32], w23 = s_w[(c * 2 + 1) * 32];
            if (c == 0) { o[0] = w01.x * A[0]; o[1] = w01.y * A[0]; o[2] = w23.x * A[0]; o[3] = w23.y * A[0]; }
            else {
                o[0] = fma(w01.x, A[c], o[0]); o[1] = fma(w01.y, A[c], o[1]);
                o[2] = fma(w23.x, A[c], o[2]); o[3] = fma(w23.y, A[c], o[3]);
            }
        }
        // GDAL's rule on the sum of the usable weights = (x sum) * (y sum): divide unless within 1e-5 of 1; a NaN sum
        // marks a pixel whose centre coarse pixel is out of range
        if (!(ri.sum == 1.0 && x_plain)) {
#pragma unroll
            for (int k = 0; k < kPpt; k++) {
                const double wsum = xsum[k] * ri.sum;
                if (wsum != wsum) o[k] = dnan;
                else if (wsum < 0.99999 || wsum > 1.00001) o[k] /= wsum;
            }
        }
        // pixels with an invalid tap (NaN result): GDAL's general rule from the same registers
        if ((o[0] != o[0]) || (o[1] != o[1]) || (o[2] != o[2]) || (o[3] != o[3])) {
            const int jc = (int)ri.jc;
#pragma unroll
            for (int k = 0; k < kPpt; k++) {
                if (o[k] == o[k]) continue;
                double acc = 0.0, acc_w = 0.0, centre = dnan;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    double a = 0.0, m = 0.0;
#pragma unroll
                    for (int c = 0; c < kYfCols; c++) {
                        const double2 wp2 = s_w[(c * 2 + (k >> 1)) * 32];
                        const double wx = (k & 1) ? wp2.y : wp2.x;
                        const double v = t[j][c];
                        const bool ok = (wx != 0.0) && (v == v);
                        a = fma(ok ? v : 0.0, ok ? wx : 0.0, a);     // dropped taps add exact zeros
                        m += ok ? wx : 0.0;
                        if (j == jc && c == cc[k]) centre = v;
                    }
                    acc = fma(ri.wy[j], a, acc);
                    acc_w = fma(ri.wy[j], m, acc_w);
                }
                o[k] = (jc >= 0 && cc[k] >= 0 && centre == centre && gwk_normalise(acc, acc_w)) ? acc : dnan;
            }
        }
        hb_stg_stream16(orow, make_float4((float)o[0], (float)o[1], (float)o[2], (float)o[3]));
    }
}

// =====================================================================================================================
// fix-up kernel: the destination pixels of the DIRTY cells, GDAL's general rules, double arithmetic, tap by tap
// =====================================================================================================================
// (gr_cubic_spline_up in oracle/gdal_restate.c: centre pixel in range and valid in some band; out-of-range / invalid
// taps dropped; pixel dropped if sum(w) < 1e-6; renormalised unless sum(w) is within 1e-5 of 1.)
constexpr int kFixThreads = 128;
constexpr int kFixSplit = 1;

// One warp per DIRTY cell (grid-stride over the list), one lane per destination pixel COLUMN of the 4-pixel groups that
// touch the cell.  A lane first combines its column's 4x4 taps along x -- values A[j] = sum_i wx[i] v[j][i] over the
// usable taps, and their weights M[j] = sum_i wx[i] -- and then walks down the cell's rows: acc = sum_j wy[j] A[j],
// acc_w = sum_j wy[j] M[j], which is GDAL's double sum over the usable taps, re-associated.
template <typename T>
__global__ void __launch_bounds__(kFixThreads, 4)
upsample_fixup_kernel(const T *__restrict__ src, NoData nd, const float *__restrict__ coarse, UpPolyGeom g,
                      float *__restrict__ out, const int *__restrict__ list, const int *__restrict__ count)
{
    constexpr int kFixWarps = kFixThreads / 32;
    __shared__ double s_wy[kFixWarps][32][4];
    __shared__ int s_jc[kFixWarps][32];
    const int lane = threadIdx.x & 31;
    const long warp_id = (long)blockIdx.x * kFixWarps + (threadIdx.x >> 5);
    const long n_warps = (long)gridDim.x * kFixWarps;
    const long fw = g.wp + 2, plane = g.hp * g.wp;
    const float qnan = __int_as_float(0x7fc00000);
    // every cell is split into kFixSplit row chunks (one warp each): short dependent chains, more warps in flight
    const long n = (long)*count * kFixSplit;
    for (long e = warp_id; e < n; e += n_warps) {
        const long idx = list[e / kFixSplit];
        const int part = (int)(e % kFixSplit);
        const long ky = idx / fw - 1, kx = idx % fw - 1;
        // destination rows / columns of the cell: the i with up_cell(i) == k (monotone in i); the four bounds are
        // independent chains of double-precision operations: one lane each
        long ya, yb, xa, xb;
        {
            long mine = 0;
            if (lane == 0) mine = up_first_index(g.sy, g.oy, ky, g.hs);
            else if (lane == 1) mine = up_first_index(g.sy, g.oy, ky + 1, g.hs);
            else if (lane == 2) mine = up_first_index(g.sx, g.ox, kx, g.ws);
            else if (lane == 3) mine = up_first_index(g.sx, g.ox, kx + 1, g.ws);
            ya = __shfl_sync(0xffffffffu, mine, 0); yb = __shfl_sync(0xffffffffu, mine, 1);
            xa = __shfl_sync(0xffffffffu, mine, 2); xb = __shfl_sync(0xffffffffu, mine, 3);
        }
        if (yb <= ya || xb <= xa) continue;
        {
            const long chunk = (yb - ya + kFixSplit - 1) / kFixSplit;
            ya += part * chunk;
            yb = min(yb, ya + chunk);
            if (yb <= ya) continue;
        }
        // the rows' y-weights and centre rows are the same for every column: lane r prepares row ya + r once
        const bool cached = (yb - ya) <= 32;
        __syncwarp();
        // (every row of the cell has k == ky: its d and centre row are relative to the cell's tap rows)
        if (cached && ya + lane < yb) {
            const UpTap ty = up_tap(g.sy, g.oy, ya + lane, g.hp);
            const long jc = ty.centre - (ky - 1);
            double wy[4];
            up_weights<HB_UP_CUBIC_SPLINE>(ty.d, wy);
#pragma unroll
            for (int j = 0; j < 4; j++) s_wy[threadIdx.x >> 5][lane][j] = wy[j];
            s_jc[threadIdx.x >> 5][lane] = (ty.ok && jc >= 0 && jc <= 2) ? (int)jc : -1;
        }
        __syncwarp();
        // every 4-pixel group (= lane of the fast kernel) that touches the cell was skipped there: do whole groups
        const long ga = (xa / kPpt) * kPpt, gb = min(((xb - 1) / kPpt + 1) * kPpt, g.ws);
        for (long X = ga + lane; X < gb; X += 32) {
            const UpTap tx = up_tap(g.sx, g.ox, X, g.wp);
            const long cx = tx.centre, kxx = tx.k;
            const bool cx_ok = tx.ok;
            double wx[4];
            up_weights<HB_UP_CUBIC_SPLINE>(tx.d, wx);
            // x-combination of the 4 tap rows ky-1 .. ky+2 (every row of the cell has the same tap rows)
            double A[2][4], M[2][4];                       // [band: gain, offset][tap row]
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const long y = ky - 1 + j;
                float v[2][4];
                bool in[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const long x = kxx - 1 + i;
                    in[i] = y >= 0 && y < g.hp && x >= 0 && x < g.wp;
                    const long a = min(max(y, 0L), g.hp - 1) * g.wp + min(max(x, 0L), g.wp - 1);
#pragma unroll
                    for (int b = 0; b < 2; b++) v[b][i] = __ldg(coarse + b * plane + a);
                }
#pragma unroll
                for (int b = 0; b < 2; b++) {
                    double a = 0.0, m = 0.0;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const bool ok = in[i] && !isnan(v[b][i]);
                        a = fma(ok ? (double)v[b][i] : 0.0, ok ? wx[i] : 0.0, a);   // dropped taps add exact zeros
                        m += ok ? wx[i] : 0.0;
                    }
                    A[b][j] = a;
                    M[b][j] = m;
                }
            }
            // validity (in some band) of the centre-pixel candidates: coarse rows ky-1, ky, ky+1 at column cx
            bool cen[3];
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const long y = ky - 1 + j;
                bool any = false;
                if (cx_ok && y >= 0 && y < g.hp) {
                    any = !isnan(__ldg(coarse + y * g.wp + cx)) || !isnan(__ldg(coarse + plane + y * g.wp + cx));
                }
                cen[j] = any;
            }
            constexpr int kBatch = 8;                        // source pixels of 8 rows in flight per lane
            for (long Yc = ya; Yc < yb; Yc += kBatch) {
                float sv[kBatch];
#pragma unroll
                for (int u = 0; u < kBatch; u++)
                    sv[u] = (Yc + u < yb) ? hb_to_f32<T>(src[(Yc + u) * g.ws + X]) : 0.f;
#pragma unroll
                for (int u = 0; u < kBatch; u++) {
                    const long Y = Yc + u;
                    if (Y >= yb) break;
                    int jc;                                  // tap row of the centre pixel (0 .. 2), -1: out of range
                    double wy[4];
                    if (cached) {
                        const int ri = (int)(Y - ya);
                        jc = s_jc[threadIdx.x >> 5][ri];
#pragma unroll
                        for (int j = 0; j < 4; j++) wy[j] = s_wy[threadIdx.x >> 5][ri][j];
                    } else {
                        const UpTap ty = up_tap(g.sy, g.oy, Y, g.hp);
                        const long j0 = ty.centre - (ky - 1);
                        jc = (ty.ok && j0 >= 0 && j0 <= 2) ? (int)j0 : -1;
                        up_weights<HB_UP_CUBIC_SPLINE>(ty.d, wy);
                    }
                    bool c_ok = (jc == 0 ? cen[0] : (jc == 1 ? cen[1] : (jc == 2 ? cen[2] : false)));
                    const float s = sv[u];
                    c_ok = c_ok && hb_valid(s, nd);
                    float r[2] = {qnan, qnan};
                    if (c_ok) {
#pragma unroll
                        for (int b = 0; b < 2; b++) {
                            double acc = 0.0, acc_w = 0.0;
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                acc = fma(wy[j], A[b][j], acc);
                                acc_w = fma(wy[j], M[b][j], acc_w);
                            }
                            if (gwk_normalise(acc, acc_w)) r[b] = (float)acc;
                        }
                    }
                    hb_store1_out(out, Y * g.ws + X, __fadd_rn(__fmul_rn(r[0], s), r[1]), g.ospec);   // two roundings, as numpy
                }
            }
        }
    }
}

// =====================================================================================================================
// general kernel: every up-sampling ratio, any alignment, the coverage mask
// =====================================================================================================================
// GDAL GRA_CubicSpline (4x4 cubic B-spline taps, invalid / out-of-range taps dropped and the rest renormalised; spec in
// oracle/gdal_restate.c).  After a one-off per-CTA table of the rows' y-geometry, every WARP is autonomous (no further
// CTA barrier): it owns a 128-pixel-wide column strip (4 pixels per lane, vector stores) and walks down it row by row.
// Source pixels arrive through a 4-deep cp.async ring (each lane copies, and later reads, only its own bytes).
//
//   (Aligned destinations >= ~1.6x finer than the coarse grid take the fast paths above instead; this kernel handles
//   smaller ratios, unaligned rasters, the coverage mask of mask_partial and plain two-band up-sampling.)
//   Per destination row:
//     A. lane <-> coarse column: combine the column's 4 tap rows (register cache, invalid taps zeroed + validity mask)
//        with the row's y-weights into warp-private shared memory (values, weight sums, flags);
//     C. lane <-> 4 pixels: sum the 4 column combinations with the pixel's x-weights, apply GDAL's centre-pixel and
//        renormalisation rules.
// In APPLY mode the up-sampled parameters never exist in memory.
struct __align__(16) Pair { double g, o; };          // band 0 (gain) and band 1 (offset)
struct __align__(16) RowInfo {
    double dy;        // fractional row position inside the cell row
    int ky;           // first tap row + 1
    int jc;           // tap row hosting the centre pixel (1 or 2; 0 when clamped), -1: centre row out of range
    int cy;           // coarse row of the centre pixel
    int pad;
};

constexpr int kUpMaxRows = 64;                        // destination rows per CTA (upper bound)

// 4 source pixels of storage type T -> float32, plus their validity against the nodata value
template <typename T> struct Src4;
template <> struct Src4<uint16_t> {
    static constexpr int kBytes = 8;
    static __device__ __forceinline__ void get(const void *p, const NoData &nd, float (&v)[4], bool (&ok)[4])
    {
        const uint2 w = *reinterpret_cast<const uint2 *>(p);
        const uint32_t r[4] = {w.x & 0xFFFFu, w.x >> 16, w.y & 0xFFFFu, w.y >> 16};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            v[k] = __uint_as_float(0x4B000000u | r[k]) - 8388608.0f;      // exact, no I2F
            ok[k] = (int)r[k] != nd.ivalue;                                // (kHbNoIntNodata when no integer nodata)
        }
    }
};
template <> struct Src4<int16_t> {
    static constexpr int kBytes = 8;
    static __device__ __forceinline__ void get(const void *p, const NoData &nd, float (&v)[4], bool (&ok)[4])
    {
        uint2 w = *reinterpret_cast<const uint2 *>(p);
        w.x ^= 0x80008000u;                                                 // fields: v + 32768
        w.y ^= 0x80008000u;
        const uint32_t r[4] = {w.x & 0xFFFFu, w.x >> 16, w.y & 0xFFFFu, w.y >> 16};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            v[k] = __uint_as_float(0x4B000000u | r[k]) - 8421376.0f;      // exact, no I2F
            ok[k] = (int)r[k] - 32768 != nd.ivalue;
        }
    }
};
template <> struct Src4<uint8_t> {
    static constexpr int kBytes = 4;
    static __device__ __forceinline__ void get(const void *p, const NoData &nd, float (&v)[4], bool (&ok)[4])
    {
        const uint32_t w = *reinterpret_cast<const uint32_t *>(p);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t r = (w >> (8 * k)) & 0xFFu;
            v[k] = __uint_as_float(0x4B000000u | r) - 8388608.0f;
            ok[k] = (int)r != nd.ivalue;
        }
    }
};
template <> struct Src4<float> {
    static constexpr int kBytes = 16;
    static __device__ __forceinline__ void get(const void *p, const NoData &nd, float (&v)[4], bool (&ok)[4])
    {
        const float4 w = *reinterpret_cast<const float4 *>(p);
        v[0] = w.x; v[1] = w.y; v[2] = w.z; v[3] = w.w;
#pragma unroll
        for (int k = 0; k < 4; k++) ok[k] = hb_valid(v[k], nd);
    }
};

struct UpGeom {
    long hs, ws;          // destination (fine) grid
    long hp, wp;          // coarse grid
    double sx, ox, sy, oy;
    int ncols;            // coarse columns staged per warp (cells + 3)
    int rows_per_cta;
    OutSpec ospec;        // output dtype / nodata of the corrected plane (APPLY); plain float32 otherwise
};

// T: storage type of the source plane (APPLY); NB: coarse bands (1 or 2); APPLY: fuse gain*src+offset;
// MC: coarse columns per lane (ncols <= 32 * MC); METHOD: HB_UP_CUBIC_SPLINE, HB_UP_BILINEAR, HB_UP_CUBIC or
// HB_UP_LANCZOS.
//   All methods share the geometry, the centre / cover rules, phase C and the stores; every column stores per-band
//   "tap missing" flags (bit0 gain, bit2 offset) and "centre usable" (bit1).  Phase A has two forms: cubic spline keeps
//   its tap rows in a register cache (MC = 1 / 3 / 5); the other methods re-read the taps through L1 every row (nothing
//   persists across rows, so even MC = 5 stays clear of spills with 6 taps), and cubic stores a second column
//   combination of the two inner taps with its own weight sum (its bilinear fallback, s_val2 / s_wgt).
template <typename T, int NB, bool APPLY, bool ALIGNED, int MC, int METHOD>
__global__ void __launch_bounds__(kThreads, kMinCtas)
upsample_kernel(const T *__restrict__ src, NoData nd, const float *__restrict__ coarse, UpGeom g,
                const uint8_t *__restrict__ cover, float *__restrict__ out)
{
    constexpr bool kSpline = (METHOD == HB_UP_CUBIC_SPLINE);
    constexpr int NT = up_taps(METHOD);                                   // taps per axis
    constexpr int kLo = NT / 2 - 1;                                       // taps before the cell's first row / column
    constexpr int kPairs = (METHOD == HB_UP_CUBIC) ? 3 : 2;               // Pairs per staged column
    constexpr int NOUT = (NB == 2 && !APPLY) ? 2 : 1;
    constexpr int kLaneBytes = APPLY ? Src4<T>::kBytes : 0;
    constexpr int kRowBytes = 32 * kLaneBytes;                            // one staged source row of the warp
    constexpr int kRingBytes = kStages * kRb * kRowBytes;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int ncols = g.ncols;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float qnan = __int_as_float(0x7fc00000);

    auto row_info = [&](long Y) {
        const UpTap ty = up_tap(g.sy, g.oy, Y, g.hp);
        RowInfo ri;
        ri.dy = ty.d;
        ri.ky = (int)ty.k;
        ri.jc = ty.ok ? (int)(ty.centre - (ty.k - kLo)) : -1;   // kLo or kLo + 1 (kLo - 1 when clamped at the bottom edge)
        ri.cy = (int)ty.centre;
        ri.pad = 0;
        return ri;
    };

    // ---- per-CTA row table: y-geometry of the CTA's destination rows ---------------------------------------------------
    RowInfo *s_rows = reinterpret_cast<RowInfo *>(smem_raw);
    const long Y0 = (long)blockIdx.y * g.rows_per_cta;
    const long Y1 = min(Y0 + (long)g.rows_per_cta, g.hs);
    const long strip = (long)blockIdx.x * kWarps + warp;
    if ((long)threadIdx.x < Y1 - Y0) s_rows[threadIdx.x] = row_info(Y0 + threadIdx.x);
    __syncthreads();                                        // the only CTA barrier

    // warp-private shared memory: values [ncols], weights [ncols], column flags [ncols] of ONE row, source ring
    const int comb_bytes = ((ncols * (kPairs * (int)sizeof(Pair) + 1)) + 15) / 16 * 16;
    unsigned char *base = smem_raw + kUpMaxRows * sizeof(RowInfo) + warp * (comb_bytes + kRingBytes);
    Pair *s_val = reinterpret_cast<Pair *>(base);
    Pair *s_wgt = s_val + ncols;
    Pair *s_val2 = s_wgt + ncols;                                          // (cubic only)
    uint8_t *s_colf = reinterpret_cast<uint8_t *>(s_wgt + (kPairs - 1) * ncols);   // bit0: a tap missing, bit1: centre usable
    const unsigned char *s_ring = base + comb_bytes + lane * kLaneBytes;   // this lane's slot in a staged row
    const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(s_ring);

    const long Xw0 = strip * kWarpW;                      // first destination column of the warp
    if (Xw0 >= g.ws) return;
    const long X0 = Xw0 + (long)lane * kPpt;
    const long plane = g.hp * g.wp;

    // coarse column window of the warp: the taps of its first pixel start at column kx - 1
    const long col_base = up_tap(g.sx, g.ox, Xw0, g.wp).k - kLo;

    // ---- per-pixel, row-invariant geometry (recomputed on demand: keeps it out of the hot loop's registers) ------------
    auto px_geom = [&](int k, double &dxk, int &clk, int &ctk) {
        const UpTap tx = up_tap(g.sx, g.ox, X0 + k, g.wp);
        dxk = tx.d;                                         // fractional column position inside the cell
        long c = tx.k - kLo - col_base;                     // first tap column, relative to col_base
        int ct = -1;                                        // tap column hosting the centre (0..NT-1), -1: none usable
        if (c < 0 || c + (NT - 1) >= ncols) c = 0;          // only for X >= ws (never stored)
        else if (tx.ok) ct = (int)(tx.centre - (tx.k - kLo));   // kLo or kLo + 1 (kLo - 1 when clamped at the right edge)
        clk = (int)c;
        ctk = (ct >= 0 && ct < NT) ? ct : -1;
    };
    const bool full_vec = (X0 + kPpt <= g.ws);
    const bool use_async = APPLY && ALIGNED && full_vec;   // pixels come through the cp.async ring
    double wxr[kPpt][NT];                                   // x-weights, first tap column, centre tap column per pixel
    double dxr[kPpt];                                       // (cubic: the bilinear fallback's fractional column)
    int clr[kPpt], ctr[kPpt];
#pragma unroll
    for (int k = 0; k < kPpt; k++) {
        px_geom(k, dxr[k], clr[k], ctr[k]);
        up_weights<METHOD>(dxr[k], wxr[k]);
    }

    // ---- tap rows cached per lane column ---------------------------------------------------------------------------
    float tv[MC][NB][4];
    unsigned tmask[MC];
#pragma unroll
    for (int m = 0; m < MC; m++) tmask[m] = 0;
    int a_ky = INT_MIN;

    auto prefetch = [&](long Yp, int stage) {
        if (use_async) {
#pragma unroll
            for (int rr = 0; rr < kRb; rr++)
                if (Yp + rr < Y1)
                    cp_async_lane<kLaneBytes>(ring_sa + (stage * kRb + rr) * kRowBytes, src + (Yp + rr) * g.ws + X0);
        }
        cp_async_commit();
    };
    if (APPLY) {
#pragma unroll
        for (int st = 0; st < kStages - 1; st++) prefetch(Y0 + (long)st * kRb, st);
    }

    // (APPLY: the corrected plane's output dtype conversion is fused into the store; `opix` = pixel index of the lane's
    //  first pixel in the output plane)
    auto store_row = [&](long opix, const float (&res)[NOUT][kPpt]) {
        if (ALIGNED && full_vec) {
            if constexpr (APPLY) hb_store4_out(out, opix, make_float4(res[0][0], res[0][1], res[0][2], res[0][3]), g.ospec);
            else hb_stg_stream16(out + opix, make_float4(res[0][0], res[0][1], res[0][2], res[0][3]));
            if constexpr (NOUT == 2)
                hb_stg_stream16(out + g.hs * g.ws + opix, make_float4(res[1][0], res[1][1], res[1][2], res[1][3]));
        } else {
#pragma unroll
            for (int k = 0; k < kPpt; k++) {
                if ((X0 + k) < g.ws) {
                    if constexpr (APPLY) hb_store1_out(out, opix + k, res[0][k], g.ospec);
                    else out[opix + k] = res[0][k];
                    if constexpr (NOUT == 2) out[g.hs * g.ws + opix + k] = res[1][k];
                }
            }
        }
    };
    auto load_src = [&](long Y, const unsigned char *ring_row, float (&s)[kPpt], bool (&ok)[kPpt]) {
        if constexpr (APPLY) {
            if (use_async) {
                Src4<T>::get(ring_row, nd, s, ok);
            } else {
                const T *row = src + Y * g.ws;
#pragma unroll
                for (int k = 0; k < kPpt; k++) {
                    const bool in_row = (X0 + k) < g.ws;
                    s[k] = in_row ? hb_to_f32<T>(row[X0 + k]) : 0.f;
                    ok[k] = in_row && hb_valid(s[k], nd);
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < kPpt; k++) { s[k] = 0.f; ok[k] = (X0 + k) < g.ws; }
        }
    };

    int batch = 0;
    for (long Yb = Y0; Yb < Y1; Yb += kRb, batch++) {
        const int nrows = (int)min((long)kRb, Y1 - Yb);
        if (APPLY) {
            prefetch(Yb + (long)(kStages - 1) * kRb, (batch + kStages - 1) % kStages);
            cp_async_wait<kStages - 1>();                 // this stage's source rows have landed
        }
        const unsigned char *ring_b = s_ring + ((batch % kStages) * kRb) * kRowBytes;

        for (int rr = 0; rr < nrows; rr++) {
            const long orow = (Yb + rr) * g.ws + X0;
            const long Y = Yb + rr;
            const RowInfo ri = s_rows[Y - Y0];

            float s[kPpt];
            bool ok[kPpt];
            float res[NOUT][kPpt];

            // ---- GENERAL row, phase A: column combinations ------------------------------------------------------------
            double wy[NT];
            up_weights<METHOD>(ri.dy, wy);
            if constexpr (kSpline) {
                if (ri.ky != a_ky) {                            // (warp-uniform) fetch / shift the tap rows
                    const bool shift1 = (ri.ky - a_ky) == 1;
#pragma unroll
                    for (int m = 0; m < MC; m++) {
                        const long col = col_base + lane + 32 * m;
                        const bool col_in = (lane + 32 * m < ncols) && col >= 0 && col < g.wp;
                        unsigned mask = shift1 ? ((tmask[m] >> 1) & 0x77u) : 0u;
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const long row = (long)ri.ky - 1 + j;
                            const bool inside = col_in && row >= 0 && row < g.hp;
#pragma unroll
                            for (int b = 0; b < NB; b++) {
                                if (shift1 && j < 3) {
                                    tv[m][b][j] = tv[m][b][j + 1];
                                } else {
                                    const float v = inside ? __ldg(coarse + b * plane + row * g.wp + col) : qnan;
                                    const bool okv = !isnan(v);
                                    tv[m][b][j] = okv ? v : 0.f;
                                    if (okv) mask |= 1u << (b * 4 + j);
                                }
                            }
                        }
                        tmask[m] = mask;
                    }
                    a_ky = ri.ky;
                }
#pragma unroll
                for (int m = 0; m < MC; m++) {
                    const int c = lane + 32 * m;
                    if (c < ncols) {
                        Pair val;                               // invalid taps are stored as 0: no predication needed
                        val.g = fma(wy[3], (double)tv[m][0][3], fma(wy[2], (double)tv[m][0][2],
                                fma(wy[1], (double)tv[m][0][1], wy[0] * (double)tv[m][0][0])));
                        val.o = 0.0;
                        if (NB > 1)
                            val.o = fma(wy[3], (double)tv[m][1][3], fma(wy[2], (double)tv[m][1][2],
                                    fma(wy[1], (double)tv[m][1][1], wy[0] * (double)tv[m][1][0])));
                        s_val[c] = val;
                        const unsigned mask = tmask[m];
                        const unsigned miss = ((mask & 0xFu) != 0xFu ? 1u : 0u) | ((NB > 1 && (mask >> 4) != 0xFu) ? 4u : 0u);
                        // centre pixel: its coarse pixel must be in range and valid in any band (+ the coverage mask)
                        bool c_ok = (ri.jc >= 0) && (((mask | (mask >> 4)) >> ri.jc) & 1u);
                        if (c_ok && cover != nullptr) c_ok = cover[(long)ri.cy * g.wp + col_base + c] != 0;
                        // a band's tap counts iff that band is valid there (band-valid implies "any band" validity)
                        Pair wgt = {0.0, 0.0};
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            if ((mask >> j) & 1u) wgt.g += wy[j];
                            if (NB > 1 && ((mask >> (4 + j)) & 1u)) wgt.o += wy[j];
                        }
                        s_wgt[c] = wgt;
                        s_colf[c] = (uint8_t)(miss | (c_ok ? 2u : 0u));
                    }
                }
            } else {
                const double by[2] = {1.0 - ri.dy, ri.dy};      // (cubic: the bilinear fallback's y-weights)
#pragma unroll 1
                for (int m = 0; m < MC; m++) {
                    const int c = lane + 32 * m;
                    if (c < ncols) {
                        const long col = col_base + c;
                        const bool col_in = col >= 0 && col < g.wp;
                        double acc[NB], wsum[NB], acc2[NB], wsum2[NB];
#pragma unroll
                        for (int b = 0; b < NB; b++) acc[b] = wsum[b] = acc2[b] = wsum2[b] = 0.0;
                        unsigned miss = 0;
                        bool c_any = false;
#pragma unroll
                        for (int j = 0; j < NT; j++) {
                            // bilinear weighs only the inner two rows; an outer row is read only when it hosts the centre
                            const bool weighed = METHOD != HB_UP_BILINEAR || (j == 1 || j == 2);
                            const long row = (long)ri.ky - kLo + j;
                            const bool inside = (weighed || j == ri.jc) && col_in && row >= 0 && row < g.hp;
                            bool any = false;
#pragma unroll
                            for (int b = 0; b < NB; b++) {
                                const float v = inside ? __ldg(coarse + b * plane + row * g.wp + col) : qnan;
                                const bool okv = !isnan(v);
                                any |= okv;
                                if (!weighed) continue;
                                if (okv) {
                                    acc[b] = fma(wy[j], (double)v, acc[b]);
                                    wsum[b] += wy[j];
                                    if (METHOD == HB_UP_CUBIC && (j == 1 || j == 2)) {
                                        acc2[b] = fma(by[j - 1], (double)v, acc2[b]);
                                        wsum2[b] += by[j - 1];
                                    }
                                } else {
                                    miss |= 1u << (2 * b);
                                }
                            }
                            if (j == ri.jc) c_any = any;
                        }
                        // centre pixel: its coarse pixel must be in range and valid in any band (+ the coverage mask)
                        bool c_ok = (ri.jc >= 0) && c_any;
                        if (c_ok && cover != nullptr) c_ok = cover[(long)ri.cy * g.wp + col] != 0;
                        s_val[c] = Pair{acc[0], NB > 1 ? acc[NB - 1] : 0.0};
                        if constexpr (METHOD == HB_UP_CUBIC) {
                            s_val2[c] = Pair{acc2[0], NB > 1 ? acc2[NB - 1] : 0.0};
                            s_wgt[c] = Pair{wsum2[0], NB > 1 ? wsum2[NB - 1] : 0.0};
                        } else {
                            s_wgt[c] = Pair{wsum[0], NB > 1 ? wsum[NB - 1] : 0.0};
                        }
                        s_colf[c] = (uint8_t)(miss | (c_ok ? 2u : 0u));
                    }
                }
            }
            __syncwarp();

            // ---- GENERAL row, phase C: destination pixels -------------------------------------------------------------
            if (X0 < g.ws) {
                load_src(Y, ring_b + rr * kRowBytes, s, ok);
#pragma unroll
                for (int k = 0; k < kPpt; k++) {
                    const double (&wx)[NT] = wxr[k];
                    const int clk = clr[k], ctk = ctr[k];
                    const Pair *v = s_val + clk;
                    // (cubic spline starts from -0.0, and fma(w, a, -0.0) == w * a: its sum starts with a product, as
                    //  in its phase A and its fast paths, so that a sum of negative zeros stays -0.0 on every path)
                    double gv = kSpline ? -0.0 : 0.0, ov = gv;
                    unsigned fm = 0;                        // per-band "tap missing" over the footprint's columns
#pragma unroll
                    for (int i = 0; i < NT; i++) {
                        if (METHOD == HB_UP_BILINEAR && (i == 0 || i == 3)) continue;
                        const Pair a = v[i];
                        gv = fma(wx[i], a.g, gv);
                        if (NB > 1) ov = fma(wx[i], a.o, ov);
                        fm |= s_colf[clk + i];
                    }
                    const unsigned fc = (ctk >= 0) ? s_colf[clk + ctk] : 0u;
                    bool g_ok = ok[k] && (fc & 2u), o_ok = g_ok;
                    const Pair *w = s_wgt + clk;
                    if constexpr (METHOD == HB_UP_CUBIC) {
                        // the 4x4 Keys sum where every tap of the band is valid and in range, else the bilinear result
                        const double bx0 = 1.0 - dxr[k], bx1 = dxr[k];
                        const Pair *v2 = s_val2 + clk;
                        if (fm & 1u) {
                            gv = fma(bx1, v2[2].g, bx0 * v2[1].g);
                            g_ok = g_ok && up_normalise<METHOD>(gv, fma(bx1, w[2].g, bx0 * w[1].g));
                        }
                        if (NB > 1 && (fm & 4u)) {
                            ov = fma(bx1, v2[2].o, bx0 * v2[1].o);
                            o_ok = o_ok && up_normalise<METHOD>(ov, fma(bx1, w[2].o, bx0 * w[1].o));
                        }
                    } else if (METHOD == HB_UP_LANCZOS || (fm & 5u)) {
                        // lanczos: its weights do not sum to 1, so every pixel is normalised
                        double wg = 0.0, wo = 0.0;
#pragma unroll
                        for (int i = 0; i < NT; i++) {
                            if (METHOD == HB_UP_BILINEAR && (i == 0 || i == 3)) continue;
                            wg = fma(wx[i], w[i].g, wg);
                            if (NB > 1) wo = fma(wx[i], w[i].o, wo);
                        }
                        g_ok = g_ok && up_normalise<METHOD>(gv, wg);
                        if (NB > 1) o_ok = o_ok && up_normalise<METHOD>(ov, wo);
                    }
                    const float gf = g_ok ? (float)gv : qnan;
                    const float of = o_ok ? (float)ov : qnan;
                    if (APPLY) {
                        res[0][k] = __fadd_rn(__fmul_rn(gf, s[k]), of);
                    } else {
                        res[0][k] = gf;
                        if constexpr (NOUT == 2) res[1][k] = of;
                    }
                }
                store_row(orow, res);
            }
            __syncwarp();
        }
    }
}

// nearest-neighbour up-sampling of float planes (kernel_model.py:497 semantics for float data)
__global__ void nearest_kernel(const float *__restrict__ src, long nb, long hs, long ws, NoData nd,
                               float *__restrict__ dst, long hd, long wd, double sx, double ox, double sy, double oy)
{
    const long n = hd * wd;
    const float qnan = __int_as_float(0x7fc00000);
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long)gridDim.x * blockDim.x) {
        const long i = idx / wd, j = idx - i * wd;
        const UpTap ty = up_tap(sy, oy, i, hs), tx = up_tap(sx, ox, j, ws);
        for (long b = 0; b < nb; b++) {
            float v = qnan;
            if (ty.ok && tx.ok) {
                const float s = src[b * hs * ws + ty.centre * ws + tx.centre];
                if (hb_valid(s, nd)) v = s;
            }
            dst[b * n + idx] = v;
        }
    }
}

// Rows per CTA of the fast paths: as many as possible (fewer row tables / weight set-ups per pixel) such that the grid of
// gx CTA columns is just under a whole number of waves of `slots` resident CTAs (every warp streams the same amount: no
// ragged tail).
long wave_rows_per_cta(long gx, long hs, long slots)
{
    long rpc = kMaxRows;
    double best = -1.0;
    for (long cand = kMaxRows; cand >= 32; cand -= kRb) {
        const long ctas = gx * ((hs + cand - 1) / cand);
        const long waves = (ctas + slots - 1) / slots;
        const double eff = (double)ctas / (double)(waves * slots) * (cand >= 64 ? 1.0 : 0.97);
        if (eff > best + 0.02) { best = eff; rpc = cand; }
    }
    return rpc;
}

// The fix-up kernel only depends on the pre-pass and writes pixels the streaming kernel skips: it runs on a side stream
// forked after the pre-pass (a few latency-bound warps that would otherwise add ~15-20 us in front of / behind the
// streaming kernel), joined before the scratch is released.  A small per-device pool of high-priority side streams.
template <typename T>
int launch_poly(const T *src, NoData nd, const float *coarse, const UpPolyGeom &g, float *out, cudaStream_t stream)
{
    const long fw = g.wp + 2, ncell = (g.hp + 2) * fw;
    HB_REQUIRE(ncell < 2147483000L, "up-sampling: coarse raster too large");
    // workspace: [count (16 B)] [list: ncell ints] [flags: ncell bytes] [interleaved bands: hp*wp float2]
    const size_t off_list = 16, off_flags = off_list + (((size_t)ncell * 4 + 15) / 16) * 16;
    const size_t off_c2 = off_flags + (((size_t)ncell + 15) / 16) * 16;
    const size_t total = off_c2 + (size_t)g.hp * g.wp * sizeof(float2);
    char *wsb = nullptr;
    HB_CUDA_OK(hb_pool_keep_memory());
    HB_CUDA_OK(cudaMallocAsync((void **)&wsb, total, stream));
    int *count = (int *)wsb, *list = (int *)(wsb + off_list);
    uint8_t *flags = (uint8_t *)(wsb + off_flags);
    float2 *coarse2 = (float2 *)(wsb + off_c2);
    HB_CUDA_OK(cudaMemsetAsync(count, 0, 16, stream));
    {
        dim3 pgrid((unsigned)((fw + kPrepW - 1) / kPrepW), (unsigned)((g.hp + 2 + kPrepH - 1) / kPrepH));
        HB_REQUIRE(pgrid.y <= 65535u, "up-sampling: coarse raster has too many rows (%ld)", g.hp);
        upsample_prep_kernel<<<pgrid, kPrepW * kPrepH, 0, stream>>>(coarse, g.hp, g.wp, coarse2, flags, list, count);
        HB_LAUNCH_OK("upsample_prep_kernel");
    }
    // fork: the fix-up kernel on a side stream, concurrently with the streaming kernel below
    SideStream *side = side_stream();
    std::unique_lock<std::mutex> side_lock;
    if (side != nullptr) {
        side_lock = std::unique_lock<std::mutex>(side->mu);
        if (cudaEventRecord(side->fork, stream) != cudaSuccess || cudaStreamWaitEvent(side->s, side->fork, 0) != cudaSuccess) {
            cudaGetLastError();
            side = nullptr;
        }
    }
    if (side != nullptr) {
        const unsigned blocks = (unsigned)hb_sm_count() * 16;
        upsample_fixup_kernel<T><<<blocks, kFixThreads, 0, side->s>>>(src, nd, coarse, g, out, list, count);
        HB_LAUNCH_OK("upsample_fixup_kernel");
        HB_CUDA_OK(cudaEventRecord(side->join, side->s));
    }
    {
        // a lane spanning 3 coarse cells (fewer than ~3.4 destination pixels per coarse pixel): the "y first" kernel
        const bool yfirst = (g.sx > 0.3);
        const size_t ring = (size_t)kStages * kRb * 32 * kPpt * sizeof(T);
        const size_t smem = (yfirst ? kRowTableBytes : kPolyRowTableBytes) +
                            ((yfirst ? kYfCols : 6) * 32 * sizeof(float4) + ring) * kWarps;
        const long cta_w = (long)kWarpW * kWarps;
        const long gx = (g.ws + cta_w - 1) / cta_w;
        // (CONVERT: an output dtype / nodata other than plain float32 -- its own instantiation, so that the float32 path's
        //  store stays a single 16-byte instruction)
        const bool convert = !g.ospec.plain;
        auto kern = yfirst ? (convert ? upsample_yfirst_kernel<T, true> : upsample_yfirst_kernel<T, false>)
                           : (convert ? upsample_poly_kernel<T, true> : upsample_poly_kernel<T, false>);
        if (smem > 48 * 1024)
            HB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        static int ctas_cache[4] = {0, 0, 0, 0};
        int &ctas_per_sm = ctas_cache[(yfirst ? 1 : 0) + (convert ? 2 : 0)];
        if (ctas_per_sm == 0) {
            int n = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, kThreads, smem) != cudaSuccess || n < 1) n = 1;
            ctas_per_sm = n;
        }
        const long rpc = wave_rows_per_cta(gx, g.hs, (long)hb_sm_count() * ctas_per_sm);
        dim3 grid((unsigned)gx, (unsigned)((g.hs + rpc - 1) / rpc));
        HB_REQUIRE(grid.y <= 65535u, "up-sampling destination has too many rows (%ld)", g.hs);
        kern<<<grid, kThreads, smem, stream>>>(src, nd, coarse2, flags, g, (int)rpc, out);
        HB_LAUNCH_OK("upsample_poly_kernel");
    }
    if (side != nullptr) {
        HB_CUDA_OK(cudaStreamWaitEvent(stream, side->join, 0));            // join before the scratch is released
    } else {
        const unsigned blocks = (unsigned)hb_sm_count() * 16;
        upsample_fixup_kernel<T><<<blocks, kFixThreads, 0, stream>>>(src, nd, coarse, g, out, list, count);
        HB_LAUNCH_OK("upsample_fixup_kernel");
    }
    HB_CUDA_OK(cudaFreeAsync(wsb, stream));
    return 0;
}

// plain up-sampling of ONE band in double precision: one kernel (see upsample_yfirst_f64_kernel)
int launch_yfirst_f64(const float *coarse, const UpPolyGeom &g, float *out, cudaStream_t stream)
{
    const size_t smem = kMaxRows * (sizeof(RowEntryD) + sizeof(int)) + (size_t)kWarps * kYfCols * 2 * 32 * sizeof(double2);
    static HbOncePerDevice attr_once;
    const int arc = hb_once_per_device(attr_once, [&]() -> int {
        HB_CUDA_OK(cudaFuncSetAttribute(upsample_yfirst_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        return 0;
    });
    if (arc) return arc;
    const long cta_w = (long)kWarpW * kWarps;
    const long gx = (g.ws + cta_w - 1) / cta_w;
    const long rpc = wave_rows_per_cta(gx, g.hs, (long)hb_sm_count() * kMinCtas);
    dim3 grid((unsigned)gx, (unsigned)((g.hs + rpc - 1) / rpc));
    HB_REQUIRE(grid.y <= 65535u, "up-sampling destination has too many rows (%ld)", g.hs);
    upsample_yfirst_f64_kernel<<<grid, kThreads, smem, stream>>>(coarse, g, (int)rpc, out);
    HB_LAUNCH_OK("upsample_yfirst_f64_kernel");
    return 0;
}

// the general kernel for one method: coarse columns per lane (MC) and alignment picked from the geometry
template <typename T, int NB, bool APPLY, int METHOD>
int launch_general(const void *src, NoData ndk, const float *coarse, const UpGeom &g, bool aligned, dim3 grid,
                   size_t smem, const uint8_t *cover, float *out, cudaStream_t stream)
{
#define HB_UP_LAUNCH(AL_, MC_)                                                                                        \
    do {                                                                                                              \
        auto kern = upsample_kernel<T, NB, APPLY, AL_, MC_, METHOD>;                                                  \
        if (smem > 48 * 1024)                                                                                         \
            HB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));          \
        kern<<<grid, kThreads, smem, stream>>>((const T *)src, ndk, coarse, g, cover, out);                          \
    } while (0)
    if constexpr (METHOD == HB_UP_CUBIC_SPLINE) {
        if (g.ncols <= 32) { if (aligned) HB_UP_LAUNCH(true, 1); else HB_UP_LAUNCH(false, 1); }
        else if (g.ncols <= 96) { if (aligned) HB_UP_LAUNCH(true, 3); else HB_UP_LAUNCH(false, 3); }
        else { if (aligned) HB_UP_LAUNCH(true, 5); else HB_UP_LAUNCH(false, 5); }
    } else {
        // (the other methods walk their staged columns in a loop that is not unrolled: MC only bounds it)
        if (aligned) HB_UP_LAUNCH(true, 5); else HB_UP_LAUNCH(false, 5);
    }
#undef HB_UP_LAUNCH
    HB_LAUNCH_OK("upsample_kernel");
    return 0;
}

template <typename T, int NB, bool APPLY>
int launch_upsample(const void *src, NoData nd, const float *coarse, long hs, long ws, long hp, long wp, double sx,
                    double ox, double sy, double oy, const uint8_t *cover, float *out, cudaStream_t stream,
                    OutSpec ospec, int method)
{
    HB_REQUIRE(sx > 0 && sy > 0 && sx <= 1.0 + 1e-9 && sy <= 1.0 + 1e-9,
               "up-sampling needs a destination grid at least as fine as the source (scale %.4f, %.4f)", sx, sy);
    HB_REQUIRE(hp < 2147483000L && wp < 2147483000L, "coarse raster too large");
    UpGeom g;
    g.hs = hs; g.ws = ws; g.hp = hp; g.wp = wp; g.sx = sx; g.ox = ox; g.sy = sy; g.oy = oy;
    g.ospec = ospec;
    // coarse columns under a warp's 128 destination columns: the cells they span + the taps' reach on either side
    g.ncols = (int)ceil((double)kWarpW * sx) + up_taps(method) + 1;
    // rows per CTA: a couple of coarse rows' worth, so that the per-cell-row work is amortised
    long rpc = (long)ceil(2.0 / sy);
    rpc = ((rpc + kRb - 1) / kRb) * kRb;
    if (rpc < 16) rpc = 16;
    if (rpc > kUpMaxRows) rpc = kUpMaxRows;
    g.rows_per_cta = (int)rpc;
    const size_t ring = APPLY ? (size_t)kStages * kRb * 32 * kPpt * sizeof(T) : 0;
    const size_t pairs = (method == HB_UP_CUBIC) ? 3 : 2;    // (must match the kernel's kPairs)
    const size_t per_warp = ((size_t)g.ncols * (pairs * sizeof(Pair) + 1) + 15) / 16 * 16 + ring;
    const size_t smem = kUpMaxRows * sizeof(RowInfo) + per_warp * kWarps;
    const long cta_w = (long)kWarpW * kWarps;
    dim3 grid((unsigned)((ws + cta_w - 1) / cta_w), (unsigned)((hs + rpc - 1) / rpc));
    HB_REQUIRE(grid.y <= 65535u, "up-sampling destination has too many rows (%ld)", hs);
    const size_t align = APPLY ? sizeof(T) * kPpt : 16;
    const bool aligned = (!APPLY || (((ws * (long)sizeof(T)) % (long)align == 0) && (((uintptr_t)src) % align == 0))) &&
                         (ws % 4 == 0) && (((uintptr_t)out) % (4 * hb_out_size(ospec.dtype)) == 0);
    // ---- cubic-spline fast paths: aligned rasters, no coverage mask, >= ~1.6 destination pixels per coarse pixel (a
    //      lane's 4 pixels must span at most 3 coarse cells: 3 * sx < 2, with margin; the row direction only needs
    //      sy <= 1).  The other methods always take the general kernel.
    if (method == HB_UP_CUBIC_SPLINE && aligned && cover == nullptr && sx <= 0.62 && sy <= 1.0 + 1e-9 &&
        ws % kPpt == 0) {
        const UpPolyGeom pg = {hs, ws, hp, wp, sx, ox, sy, oy, ospec};
        if constexpr (APPLY) return launch_poly<T>((const T *)src, nd, coarse, pg, out, stream);
        // plain up-sampling: one band in double precision (it feeds a fit); two bands stay on the general kernel
        if constexpr (NB == 1) return launch_yfirst_f64(coarse, pg, out, stream);
    }
    switch (method) {
        case HB_UP_CUBIC_SPLINE:
            return launch_general<T, NB, APPLY, HB_UP_CUBIC_SPLINE>(src, nd, coarse, g, aligned, grid, smem, cover, out,
                                                                    stream);
        case HB_UP_BILINEAR:
            return launch_general<T, NB, APPLY, HB_UP_BILINEAR>(src, nd, coarse, g, aligned, grid, smem, cover, out,
                                                                stream);
        case HB_UP_CUBIC:
            return launch_general<T, NB, APPLY, HB_UP_CUBIC>(src, nd, coarse, g, aligned, grid, smem, cover, out,
                                                             stream);
        case HB_UP_LANCZOS:
            return launch_general<T, NB, APPLY, HB_UP_LANCZOS>(src, nd, coarse, g, aligned, grid, smem, cover, out,
                                                               stream);
    }
    HB_REQUIRE(false, "up-sampling: unknown method %d", method);
}

}  // namespace

// =====================================================================================================================
// C-ABI
// =====================================================================================================================
extern "C" int hb_upsample_apply(const void *src_dev, int src_dtype, long hs, long ws, int has_nodata, double nodata,
                                 const float *params_dev, long hp, long wp, double sx, double ox, double sy, double oy,
                                 const uint8_t *cover_dev, int out_dtype, int out_has_nodata, double out_nodata,
                                 void *corr_dev, int method, void *stream)
{
    HB_REQUIRE(src_dev && params_dev && corr_dev && hs > 0 && ws > 0 && hp > 0 && wp > 0,
               "hb_upsample_apply: bad arguments");
    HB_REQUIRE(method != HB_UP_NEAREST,
               "hb_upsample_apply: nearest has no fused form (up-sample with hb_resample_up, then hb_apply_same_grid)");
    HB_REQUIRE(method == HB_UP_CUBIC_SPLINE || method == HB_UP_BILINEAR || method == HB_UP_CUBIC ||
               method == HB_UP_LANCZOS, "hb_upsample_apply: unknown method %d", method);
    HB_REQUIRE(hb_outspec_error(out_dtype, out_has_nodata, out_nodata) == nullptr, "hb_upsample_apply: %s",
               hb_outspec_error(out_dtype, out_has_nodata, out_nodata));
    const NoData nd = hb_make_nodata(has_nodata, nodata, src_dtype);
    const OutSpec os = hb_make_outspec(out_dtype, out_has_nodata, out_nodata);
    cudaStream_t st = (cudaStream_t)stream;
    float *out = (float *)corr_dev;                          // (typed by `os`; the kernels index it in pixels)
    switch (src_dtype) {
        case HB_U8:
            return launch_upsample<uint8_t, 2, true>(src_dev, nd, params_dev, hs, ws, hp, wp, sx, ox, sy, oy, cover_dev,
                                                     out, st, os, method);
        case HB_U16:
            return launch_upsample<uint16_t, 2, true>(src_dev, nd, params_dev, hs, ws, hp, wp, sx, ox, sy, oy,
                                                      cover_dev, out, st, os, method);
        case HB_I16:
            return launch_upsample<int16_t, 2, true>(src_dev, nd, params_dev, hs, ws, hp, wp, sx, ox, sy, oy,
                                                     cover_dev, out, st, os, method);
        case HB_F32:
            return launch_upsample<float, 2, true>(src_dev, nd, params_dev, hs, ws, hp, wp, sx, ox, sy, oy, cover_dev,
                                                   out, st, os, method);
    }
    HB_REQUIRE(false, "hb_upsample_apply: unknown dtype %d", src_dtype);
}

extern "C" int hb_resample_up(const float *src_dev, long nb, long hs, long ws, int has_nodata, double nodata,
                              float *dst_dev, long hd, long wd, double sx, double ox, double sy, double oy, int method,
                              void *stream)
{
    HB_REQUIRE(src_dev && dst_dev && nb >= 1 && hs > 0 && ws > 0 && hd > 0 && wd > 0, "hb_resample_up: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const NoData nd = hb_make_nodata(has_nodata, nodata);
    if (method == HB_UP_NEAREST) {
        nearest_kernel<<<hb_grid_for(hd * wd, 256), 256, 0, st>>>(src_dev, nb, hs, ws, nd, dst_dev, hd, wd, sx, ox, sy,
                                                                  oy);
        HB_LAUNCH_OK("nearest_kernel");
        return 0;
    }
    HB_REQUIRE(method == HB_UP_CUBIC_SPLINE || method == HB_UP_BILINEAR || method == HB_UP_CUBIC ||
               method == HB_UP_LANCZOS, "hb_resample_up: unknown method %d", method);
    HB_REQUIRE(has_nodata && isnan(nodata), "hb_resample_up: cubic-spline, bilinear, cubic and lanczos input must use "
               "NaN as nodata");
    HB_REQUIRE(nb <= 2, "hb_resample_up: cubic-spline, bilinear, cubic and lanczos support 1 or 2 bands per call "
               "(got %ld)", nb);
    const NoData none = hb_make_nodata(0, 0.0);
    const OutSpec f32 = hb_make_outspec(HB_F32, 0, 0.0);
    if (nb == 1)
        return launch_upsample<float, 1, false>(nullptr, none, src_dev, hd, wd, hs, ws, sx, ox, sy, oy, nullptr,
                                                dst_dev, st, f32, method);
    return launch_upsample<float, 2, false>(nullptr, none, src_dev, hd, wd, hs, ws, sx, ox, sy, oy, nullptr, dst_dev,
                                            st, f32, method);
}
