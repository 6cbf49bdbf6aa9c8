// hb_common.cuh -- shared device / host helpers for the sm_100a kernel-model kernels.
#pragma once

#include <cuda_runtime.h>
#include <limits.h>
#include <math.h>
#include <mutex>
#include <stdint.h>
#include <stdio.h>

#include "../../include/homonim_b200.h"

// ---- error plumbing (thread-local message, C-ABI returns non-zero) -------------------------------------------------
void hb_set_error(const char *fmt, ...);
void hb_count_launch(int n = 1);

#define HB_CUDA_OK(call)                                                                                     \
    do {                                                                                                     \
        cudaError_t err__ = (call);                                                                          \
        if (err__ != cudaSuccess) {                                                                          \
            hb_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(err__));    \
            return 1;                                                                                        \
        }                                                                                                    \
    } while (0)

#define HB_LAUNCH_OK(name)                                                                                   \
    do {                                                                                                     \
        cudaError_t err__ = cudaGetLastError();                                                              \
        if (err__ != cudaSuccess) {                                                                          \
            hb_set_error("launch of %s failed at %s:%d: %s", name, __FILE__, __LINE__,                       \
                         cudaGetErrorString(err__));                                                         \
            return 1;                                                                                        \
        }                                                                                                    \
        hb_count_launch();                                                                                   \
    } while (0)

#define HB_REQUIRE(cond, ...)                                                                                \
    do {                                                                                                     \
        if (!(cond)) {                                                                                       \
            hb_set_error(__VA_ARGS__);                                                                       \
            return 2;                                                                                        \
        }                                                                                                    \
    } while (0)

static inline size_t hb_dtype_size(int dtype) { return dtype == HB_U8 ? 1 : ((dtype == HB_U16 || dtype == HB_I16) ? 2 : 4); }

// ---- nodata ---------------------------------------------------------------------------------------------------------
// A pixel is invalid iff it equals the nodata value, or both are NaN (homonim/utils.py:54-56).  The comparison is
// done in float32, as numpy does for a float32 array against a Python float (NEP 50 weak scalar).
struct NoData {
    int has;       // 0: every pixel valid
    int is_nan;    // nodata is NaN
    float value;   // nodata as float32
    int int_ok;    // nodata is an integer in the range of the plane's storage type: only then can an integer pixel equal
                   // it ([0, 65535] for uint8 / uint16 -- the uint8 kernels also check <= 255 -- [-32768, 32767] for int16)
    int ivalue;    // nodata as integer when int_ok, otherwise kHbNoIntNodata
};
// ivalue when there is no integer nodata: no uint8, uint16 or int16 pixel, zero- or sign-extended, can equal it
constexpr int kHbNoIntNodata = INT_MIN;

// `dtype`: storage type of the plane the nodata value belongs to (HB_U8 / HB_U16 / HB_I16 / HB_F32)
static inline NoData hb_make_nodata(int has, double nodata, int dtype = HB_F32)
{
    const double lo = (dtype == HB_I16) ? -32768.0 : 0.0, hi = (dtype == HB_I16) ? 32767.0 : 65535.0;
    NoData nd;
    nd.has = has ? 1 : 0;
    nd.is_nan = (has && isnan(nodata)) ? 1 : 0;
    nd.value = (float)nodata;
    nd.int_ok = (has && !nd.is_nan && nodata >= lo && nodata <= hi && nodata == floor(nodata)) ? 1 : 0;
    nd.ivalue = nd.int_ok ? (int)nodata : kHbNoIntNodata;
    return nd;
}

__device__ __forceinline__ bool hb_valid(float v, const NoData &nd)
{
    if (!nd.has) return true;
    return nd.is_nan ? !isnan(v) : (v != nd.value);
}
// integer storage: compare as integers (exact; `v` is the pixel zero-extended -- uint8 / uint16 -- or sign-extended --
// int16 -- so a pixel can only equal an in-range integer nodata)
__device__ __forceinline__ bool hb_valid_int(uint32_t v, const NoData &nd) { return !(nd.int_ok && (int)v == nd.ivalue); }
// the stored 16-bit pattern of an int16 nodata value (two's complement), for packed comparisons with raw words
__device__ __forceinline__ uint32_t hb_nd_bits16(const NoData &nd) { return (uint32_t)nd.ivalue & 0xFFFFu; }

// ---- GDAL's down-sampling footprint (GWKAverageOrModeThread) ------------------------------------------------------
// Destination index i on one axis covers source coordinates [lo, hi) = [s i + o, s (i + 1) + o); its source window is
// [a0, b0) = [floor(lo + 1e-10), ceil(hi - 1e-10)), and a footprint inside one source pixel takes that pixel.  The window
// is NOT clamped to the raster: clamping, edge weights and what a window leaving the raster means are the caller's.
struct HbFootprint { double lo, hi; long a0, b0; };
__device__ __forceinline__ HbFootprint hb_footprint(double s, double o, long i)
{
    HbFootprint f;
    f.lo = s * (double)i + o;
    f.hi = s * (double)(i + 1) + o;
    f.a0 = (long)floor(f.lo + 1e-10);
    f.b0 = (long)ceil(f.hi - 1e-10);
    if (f.a0 == f.b0) f.b0++;
    return f;
}

// ---- storage dtype -> float32 (what the reference's reader does with out_dtype='float32') -------------------------
template <typename T> __device__ __forceinline__ float hb_to_f32(T v) { return (float)v; }
// exact small-integer -> float without the (slow) I2F pipe: 2^23 + v has v in its mantissa
template <> __device__ __forceinline__ float hb_to_f32<uint8_t>(uint8_t v)
{
    return __uint_as_float(0x4B000000u | (uint32_t)v) - 8388608.0f;
}
template <> __device__ __forceinline__ float hb_to_f32<uint16_t>(uint16_t v)
{
    return __uint_as_float(0x4B000000u | (uint32_t)v) - 8388608.0f;
}
// int16: v ^ 0x8000 is the 16-bit pattern of v + 32768, so the float is 2^23 + 32768 + v
template <> __device__ __forceinline__ float hb_to_f32<int16_t>(int16_t v)
{
    return __uint_as_float(0x4B000000u | ((uint32_t)(uint16_t)v ^ 0x8000u)) - 8421376.0f;
}

// ---- streaming loads / stores (read-once data: keep it out of L1) -------------------------------------------------
__device__ __forceinline__ uint4 hb_ldg_stream16(const void *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 hb_ldg_stream8(const void *p)
{
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t hb_ldg_stream4(const void *p)
{
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void hb_stg_stream16(void *p, float4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// ---- output dtype of a corrected plane, fused into the apply kernels' stores ---------------------------------------------
// RasterArray._convert_array_dtype (raster_array.py:353-387) as used by to_rio_dataset (:493-500): integer outputs are
// rounded half-to-even (np.round) and clipped to the type's range, NaN (the corrected image's nodata) becomes the output
// nodata value (0 when there is none); float32 output only substitutes the nodata value.
struct OutSpec {
    int dtype;      // HB_U8 / HB_U16 / HB_I16 / HB_F32
    int plain;      // float32 with NaN nodata: store the values as they are
    float nd;       // output nodata as float (integer types: cast on store)
    float lo, hi;   // clip range of the integer types
};

static inline OutSpec hb_make_outspec(int out_dtype, int has_nodata, double nodata)
{
    OutSpec o;
    o.dtype = out_dtype;
    o.nd = has_nodata ? (float)nodata : (out_dtype == HB_F32 ? __builtin_nanf("") : 0.f);
    o.plain = (out_dtype == HB_F32 && o.nd != o.nd) ? 1 : 0;
    o.lo = (out_dtype == HB_I16) ? -32768.f : 0.f;
    o.hi = (out_dtype == HB_U8) ? 255.f : (out_dtype == HB_I16 ? 32767.f : 65535.f);
    return o;
}
static inline const char *hb_outspec_error(int out_dtype, int has_nodata, double nodata)
{
    if (out_dtype != HB_U8 && out_dtype != HB_U16 && out_dtype != HB_I16 && out_dtype != HB_F32) return "unsupported output dtype";
    if (out_dtype != HB_F32 && has_nodata) {
        const double lo = (out_dtype == HB_I16) ? -32768.0 : 0.0, hi = (out_dtype == HB_U8) ? 255.0 : (out_dtype == HB_I16 ? 32767.0 : 65535.0);
        if (!(nodata >= lo && nodata <= hi && nodata == floor(nodata))) return "output nodata cannot be safely cast to the output dtype";
    }
    return nullptr;
}
static inline size_t hb_out_size(int out_dtype) { return out_dtype == HB_U8 ? 1 : (out_dtype == HB_F32 ? 4 : 2); }

__device__ __forceinline__ int hb_out_int(float v, const OutSpec &o)
{
    const float r = fminf(fmaxf(rintf(v), o.lo), o.hi);
    return (v != v) ? (int)o.nd : (int)r;
}
// 4 adjacent pixels starting at pixel index `pix` (a multiple of 4; the plane is 16 / 8 / 4-byte aligned accordingly)
__device__ __forceinline__ void hb_store4_out(void *base, long pix, float4 v, const OutSpec &o)
{
    if (o.plain) {
        hb_stg_stream16(reinterpret_cast<float *>(base) + pix, v);
    } else if (o.dtype == HB_F32) {
        hb_stg_stream16(reinterpret_cast<float *>(base) + pix,
                        make_float4(v.x != v.x ? o.nd : v.x, v.y != v.y ? o.nd : v.y, v.z != v.z ? o.nd : v.z,
                                    v.w != v.w ? o.nd : v.w));
    } else {
        const unsigned a = (unsigned)hb_out_int(v.x, o), b = (unsigned)hb_out_int(v.y, o), c = (unsigned)hb_out_int(v.z, o),
                       d = (unsigned)hb_out_int(v.w, o);
        if (o.dtype == HB_U8) {
            const unsigned w = (a & 0xffu) | ((b & 0xffu) << 8) | ((c & 0xffu) << 16) | (d << 24);
            asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(reinterpret_cast<unsigned char *>(base) + pix), "r"(w) : "memory");
        } else {
            const unsigned w0 = (a & 0xffffu) | (b << 16), w1 = (c & 0xffffu) | (d << 16);
            asm volatile("st.global.cs.v2.u32 [%0], {%1,%2};" ::"l"(reinterpret_cast<unsigned short *>(base) + pix), "r"(w0), "r"(w1)
                         : "memory");
        }
    }
}
__device__ __forceinline__ void hb_store1_out(void *base, long pix, float v, const OutSpec &o)
{
    if (o.dtype == HB_F32) reinterpret_cast<float *>(base)[pix] = (!o.plain && v != v) ? o.nd : v;
    else if (o.dtype == HB_U8) reinterpret_cast<unsigned char *>(base)[pix] = (unsigned char)hb_out_int(v, o);
    else reinterpret_cast<unsigned short *>(base)[pix] = (unsigned short)hb_out_int(v, o);
}

// Stream-ordered scratch (cudaMallocAsync) comes from the device's default memory pool.  By default the pool hands
// freed memory back to the OS at every synchronisation, so that each call would pay for a fresh allocation.  Keep a
// BOUNDED amount cached (the pool is shared with the host application: an existing higher threshold is left alone, and
// nothing is pinned for ever): 4 GiB (2 % of a B200's HBM) covers the scratch of four concurrent bands at BASELINE.json's
// largest configuration (~0.25 GB of parameter-grid planes and work lists per band of the 60k x 60k raster; full-resolution
// planes are the caller's).
static inline cudaError_t hb_pool_keep_memory()
{
    static thread_local int done_for = -1;
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess || dev == done_for) return err;
    cudaMemPool_t pool;
    err = cudaDeviceGetDefaultMemPool(&pool, dev);
    if (err != cudaSuccess) return err;
    unsigned long long keep = 4ull << 30, have = 0ull;
    err = cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &have);
    if (err == cudaSuccess && have < keep) err = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    if (err == cudaSuccess) done_for = dev;
    return err;
}
// Per-device one-time set-up such as cudaFuncSetAttribute (function attributes belong to the device that is current
// when they are set).  `once` is a call-site static; the set-up runs under its mutex and the device's bit is only set
// AFTER it succeeded, so a second thread can never launch before the attribute is in place.
struct HbOncePerDevice {
    std::mutex mu;
    unsigned long long done = 0ull;
};
template <class F> static inline int hb_once_per_device(HbOncePerDevice &once, F &&setup)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return setup();
    const unsigned long long bit = 1ull << dev;
    std::lock_guard<std::mutex> lock(once.mu);
    if (once.done & bit) return 0;
    const int rc = setup();
    if (rc == 0) once.done |= bit;
    return rc;
}

static inline int hb_sm_count()
{
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
            sms = 148;
    }
    return sms;
}

// blocks of a grid-stride launch over n items: one item per thread, at most `per_sm` blocks per SM
static inline unsigned hb_grid_for(long n, int threads, int per_sm = 8)
{
    long blocks = (n + threads - 1) / threads;
    const long cap = (long)hb_sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}
