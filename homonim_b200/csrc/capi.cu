// capi.cu -- C-ABI plumbing: error reporting, launch accounting, and the host-buffer convenience entry point.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>


#include "hb_common.cuh"

static thread_local char g_error[512] = "";
static thread_local long g_launches = 0;

void hb_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

void hb_count_launch(int n) { g_launches += n; }

extern "C" int hb_abi_version(void) { return HB_ABI_VERSION; }
extern "C" const char *hb_last_error(void) { return g_error; }
extern "C" long hb_launch_count(void) { return g_launches; }
extern "C" void hb_reset_launch_count(void) { g_launches = 0; }

extern "C" int hb_device_count(void)
{
    int n = 0;
    const cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess) {
        hb_set_error("cudaGetDeviceCount failed: %s", cudaGetErrorString(err));
        return -1;
    }
    return n;
}

namespace {
struct DevBuf {
    void *p = nullptr;
    cudaStream_t st;
    explicit DevBuf(cudaStream_t s) : st(s) {}
    cudaError_t alloc(size_t bytes)
    {
        const cudaError_t err = hb_pool_keep_memory();
        return err != cudaSuccess ? err : cudaMallocAsync(&p, bytes ? bytes : 16, st);
    }
    ~DevBuf() { if (p) cudaFreeAsync(p, st); }
};
}  // namespace

// One (band, block) of RasterFuse._process_block (homonim/fuse.py:304-307) for proc_crs = ref on DEVICE buffers:
// down-sample -> [block normalisation] -> fit -> [in-paint + refit] -> up-sample + apply, all enqueued on `stream`.
static int fuse_refspace_direct(const void *src_dev, int src_dtype, long hs, long ws, int src_has_nodata,
                                double src_nodata, const float *ref_dev, long hr, long wr, int ref_has_nodata,
                                double ref_nodata, double sx, double ox, double sy, double oy, int model, int kh, int kw,
                                int want_r2, int do_inpaint, double r2_thresh, int out_dtype, int out_has_nodata,
                                double out_nodata, void *corr_dev, float *params_dev, void *stream)
{
    HB_REQUIRE(src_dev && ref_dev && corr_dev && hs > 0 && ws > 0 && hr > 0 && wr > 0, "hb_fuse_refspace: bad arguments");
    HB_REQUIRE(src_dtype == HB_U8 || src_dtype == HB_U16 || src_dtype == HB_I16 || src_dtype == HB_F32,
               "hb_fuse_refspace: bad dtype");
    cudaStream_t st = (cudaStream_t)stream;
    const bool inpaint = (model == HB_MODEL_GAIN_OFFSET) && do_inpaint;
    const int r2 = (want_r2 || inpaint) ? 1 : 0;
    const size_t nr = (size_t)hr * wr;
    const double nan = __builtin_nan("");

    // one stream-ordered allocation for all the proc-grid scratch of this call
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    const bool blk = (model == HB_MODEL_GAIN_BLK_OFFSET);
    const size_t b_ds = al(nr * sizeof(float)), b_params = params_dev ? 0 : al(nr * sizeof(float) * 3),
                 b_sums = inpaint ? al(nr * sizeof(float) * 3) : 0, b_norm = blk ? al(2 * sizeof(double)) : 0,
                 b_work = blk ? al(hb_block_norm_workspace_bytes((long)nr)) : 0,
                 b_work2 = inpaint ? al(hb_inpaint_workspace_bytes(hr, wr)) : 0;
    DevBuf scratch(st);
    HB_CUDA_OK(scratch.alloc(b_ds + b_params + b_sums + b_norm + b_work + b_work2));
    char *base = (char *)scratch.p;
    float *d_ds = (float *)base;
    float *params = params_dev ? params_dev : (float *)(base + b_ds);
    float *d_sums = (float *)(base + b_ds + b_params);
    double *d_norm = (double *)(base + b_ds + b_params + b_sums);
    void *d_work = base + b_ds + b_params + b_sums + b_norm;
    void *d_work2 = base + b_ds + b_params + b_sums + b_norm + b_work;

    int rc = hb_downsample_average(src_dev, src_dtype, hs, ws, src_has_nodata, src_nodata, d_ds, hr, wr, sx, ox, sy, oy,
                                   stream);
    if (rc) return rc;
    const double *norm = nullptr;
    if (blk) {
        rc = hb_block_norm(d_ds, 1, nan, ref_dev, ref_has_nodata, ref_nodata, (long)nr, d_norm, d_work, b_work, stream);
        if (rc) return rc;
        norm = d_norm;
    }
    rc = hb_fit_same_grid(d_ds, 1, nan, ref_dev, ref_has_nodata, ref_nodata, hr, wr, model, kh, kw, r2, norm, params,
                          inpaint ? d_sums : nullptr, stream);
    if (rc) return rc;
    if (inpaint) {
        rc = hb_inpaint_refit(params, d_sums, hr, wr, r2_thresh, 100.0, d_work2, b_work2, stream);
        if (rc) return rc;
    }
    // source grid -> reference (param) grid is the inverse of the reference -> source map
    return hb_upsample_apply(src_dev, src_dtype, hs, ws, src_has_nodata, src_nodata, params, hr, wr, 1.0 / sx, -ox / sx,
                             1.0 / sy, -oy / sy, nullptr, out_dtype, out_has_nodata, out_nodata, corr_dev,
                             HB_UP_CUBIC_SPLINE, stream);
}

// No CUDA-graph cache here: replaying a captured band step (8 kernels + stream-ordered allocations) saved 0.18 ms of host
// time per call on one idle GPU but was 2x slower with 8 processes driving 8 GPUs of one box (graph launches with memory
// allocation nodes), and the direct path is not host-bound in either case -- measured in round 1, removed in round 2.
extern "C" int hb_fuse_refspace(const void *src_dev, int src_dtype, long hs, long ws, int src_has_nodata,
                                double src_nodata, const float *ref_dev, long hr, long wr, int ref_has_nodata,
                                double ref_nodata, double sx, double ox, double sy, double oy, int model, int kh, int kw,
                                int want_r2, int do_inpaint, double r2_thresh, int out_dtype, int out_has_nodata,
                                double out_nodata, void *corr_dev, float *params_dev, void *stream)
{
    return fuse_refspace_direct(src_dev, src_dtype, hs, ws, src_has_nodata, src_nodata, ref_dev, hr, wr, ref_has_nodata,
                                ref_nodata, sx, ox, sy, oy, model, kh, kw, want_r2, do_inpaint, r2_thresh, out_dtype,
                                out_has_nodata, out_nodata, corr_dev, params_dev, stream);
}

// One (band, block) of RasterFuse._process_block (homonim/fuse.py:304-307) for proc_crs = ref, host buffers in/out.
extern "C" int hb_fuse_refspace_host(const void *src_host, int src_dtype, long hs, long ws, int src_has_nodata,
                                     double src_nodata, const float *ref_host, long hr, long wr, int ref_has_nodata,
                                     double ref_nodata, double sx, double ox, double sy, double oy, int model, int kh,
                                     int kw, int want_r2, int do_inpaint, double r2_thresh, int out_dtype,
                                     int out_has_nodata, double out_nodata, void *corr_host, float *params_host,
                                     void *stream)
{
    HB_REQUIRE(src_host && ref_host && corr_host && hs > 0 && ws > 0 && hr > 0 && wr > 0,
               "hb_fuse_refspace_host: bad arguments");
    HB_REQUIRE(src_dtype == HB_U8 || src_dtype == HB_U16 || src_dtype == HB_I16 || src_dtype == HB_F32,
               "hb_fuse_refspace_host: bad dtype");
    cudaStream_t st = (cudaStream_t)stream;
    const bool inpaint = (model == HB_MODEL_GAIN_OFFSET) && do_inpaint;
    const int r2 = (want_r2 || inpaint) ? 1 : 0;
    const size_t ns = (size_t)hs * ws, nr = (size_t)hr * wr;
    const size_t src_bytes = ns * hb_dtype_size(src_dtype);

    DevBuf d_src(st), d_ref(st), d_params(st), d_corr(st);
    HB_CUDA_OK(d_src.alloc(src_bytes));
    HB_CUDA_OK(d_ref.alloc(nr * sizeof(float)));
    HB_CUDA_OK(d_params.alloc(nr * sizeof(float) * 3));
    HB_REQUIRE(hb_outspec_error(out_dtype, out_has_nodata, out_nodata) == nullptr, "hb_fuse_refspace_host: %s",
               hb_outspec_error(out_dtype, out_has_nodata, out_nodata));
    const size_t corr_bytes = ns * hb_out_size(out_dtype);
    HB_CUDA_OK(d_corr.alloc(corr_bytes));
    HB_CUDA_OK(cudaMemcpyAsync(d_src.p, src_host, src_bytes, cudaMemcpyHostToDevice, st));
    HB_CUDA_OK(cudaMemcpyAsync(d_ref.p, ref_host, nr * sizeof(float), cudaMemcpyHostToDevice, st));
    const int rc = hb_fuse_refspace(d_src.p, src_dtype, hs, ws, src_has_nodata, src_nodata, (const float *)d_ref.p, hr, wr,
                                    ref_has_nodata, ref_nodata, sx, ox, sy, oy, model, kh, kw, want_r2, do_inpaint,
                                    r2_thresh, out_dtype, out_has_nodata, out_nodata, d_corr.p, (float *)d_params.p,
                                    stream);
    if (rc) return rc;
    HB_CUDA_OK(cudaMemcpyAsync(corr_host, d_corr.p, corr_bytes, cudaMemcpyDeviceToHost, st));
    if (params_host)
        HB_CUDA_OK(cudaMemcpyAsync(params_host, d_params.p, nr * sizeof(float) * (r2 ? 3 : 2), cudaMemcpyDeviceToHost,
                                   st));
    HB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}
