/*
 * homonim_b200.h -- C-ABI of the B200-native (sm_100a) kernel-model fit / apply path.
 *
 * This is the drop-in boundary for the hot path of leftfield-geospatial/homonim: the work done by
 * homonim/kernel_model.py (KernelModel / RefSpaceModel / SrcSpaceModel .fit() / .apply()) and by the
 * RasterArray.reproject() / rasterio.fill.fillnodata() calls it makes.  The reference has no FFI of its own (it is
 * pure Python over cv2 / GDAL / numpy); the entry points below are what a ctypes binding inside
 * homonim/kernel_model.py would call (see INTEGRATION.md).  homonim_b200/_native.py is exactly such a binding.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - every raster plane is dense row-major [rows][cols]; multi-band arrays are band-major [bands][rows][cols].
 *   - pointers named *_dev are DEVICE pointers (cudaMalloc / torch CUDA storage); `stream` is a cudaStream_t passed
 *     as void*.  All device entry points are asynchronous on `stream` and never synchronise.
 *   - nodata: `has_nodata` = 0 means "no nodata value" (every pixel valid).  `nodata` may be NaN.  A pixel is invalid
 *     iff value == (T)nodata, or both are NaN  (homonim/utils.py:54-56, raster_array.py:298-308).
 *   - grid maps: destination pixel-EDGE coordinates (col u, row v) map to source pixel-edge coordinates
 *         src_col = sx * u + ox,   src_row = sy * v + oy          (sx, sy > 0; north-up grids of one CRS)
 *     so destination pixel j covers [j, j+1) and its centre is j + 0.5.
 *   - corrected planes (`corr_dev`) are written in the OUTPUT dtype the caller asks for: `out_dtype` (HB_F32, HB_U8, HB_U16,
 *     HB_I16) with `out_has_nodata` / `out_nodata`.  The conversion of RasterArray._convert_array_dtype
 *     (homonim/raster_array.py:353-387, used by to_rio_dataset :493-500) -- round half-to-even, clip to the type's range,
 *     NaN -> nodata (0 when there is none) -- is fused into the apply kernels' stores.  HB_F32 with no nodata (or NaN)
 *     writes the float32 values as they are (nodata = NaN), which is the reference's default output profile.
 *   - return value: 0 on success, non-zero on failure; hb_last_error() then returns a message (thread-local).
 *     There is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef HOMONIM_B200_H
#define HOMONIM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_ABI_VERSION 11

/* storage dtype of a raster plane.  Every dtype is a source dtype of the entry points that read a stored source plane
 * (hb_downsample_average, hb_resample_stat, hb_apply_same_grid, hb_upsample_apply, hb_valid_mask, hb_fuse_refspace,
 * hb_fuse_refspace_host) and an output dtype.  A stored pixel v reads as the float32 value (float)v; an integer pixel
 * equals the nodata value only when that is an integer in the dtype's range. */
enum { HB_U8 = 0, HB_U16 = 1, HB_F32 = 2, HB_I16 = 3 };
/* homonim.enums.Model (homonim/enums.py:22-42) */
enum { HB_MODEL_GAIN = 0, HB_MODEL_GAIN_BLK_OFFSET = 1, HB_MODEL_GAIN_OFFSET = 2 };
/* up-sampling methods of hb_resample_up and hb_upsample_apply (GDAL GRA_CubicSpline, GRA_NearestNeighbour,
 * GRA_Bilinear, GRA_Cubic, GRA_Lanczos; spec: oracle/gdal_restate.c, oracle/interp_up_restate.c) */
enum { HB_UP_CUBIC_SPLINE = 0, HB_UP_NEAREST = 1, HB_UP_BILINEAR = 2, HB_UP_CUBIC = 3, HB_UP_LANCZOS = 4 };
/* footprint statistics of hb_resample_stat (rasterio Resampling min, max, med, q1, q3, mode; spec:
 * oracle/footprint_stats_restate.c) */
enum { HB_STAT_MIN = 0, HB_STAT_MAX = 1, HB_STAT_MED = 2, HB_STAT_Q1 = 3, HB_STAT_Q3 = 4, HB_STAT_MODE = 5 };

int hb_abi_version(void);
const char *hb_last_error(void);
/* number of visible CUDA devices, or -1 (with hb_last_error set) when the CUDA runtime cannot initialise */
int hb_device_count(void);
/* kernels launched by this library on the calling thread since the last reset (for bench.py's gpu_launches) */
long hb_launch_count(void);
void hb_reset_launch_count(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Down-sampling: RasterArray.reproject(..., resampling=average)  (homonim/raster_array.py:526-578, called from
 * RefSpaceModel.fit kernel_model.py:480).  dst[hd][wd] float32, nodata = NaN: weighted mean of the valid source
 * pixels under each destination pixel's footprint (GDAL GRA_Average); NaN where no valid source pixel contributes.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_downsample_average(const void *src_dev, int src_dtype, long hs, long ws, int has_nodata, double nodata,
                          float *dst_dev, long hd, long wd, double sx, double ox, double sy, double oy,
                          void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Footprint statistics: RasterArray.reproject(..., resampling=min | max | med | q1 | q3 | mode) on any geometry
 * (down-sampling, up-sampling or mixed axes).  dst[hd][wd] float32, nodata = NaN.  Each destination pixel takes one of
 * the valid source values under its footprint -- the window of hb_downsample_average, unweighted: a partly covered
 * pixel counts as one value.  Valid = passes the nodata test and is not NaN; values compare as float32, -0.0 == +0.0,
 * a zero result is +0.0.  With v[0..n) the n valid values sorted ascending: HB_STAT_MIN v[0], HB_STAT_MAX v[n-1],
 * HB_STAT_MED / Q1 / Q3 v[ceil(q n - 1)] with q = 0.5 / 0.25 / 0.75 in double; HB_STAT_MODE the most frequent value,
 * ties going to the value whose last occurrence comes first in row-major scan order.  NaN where no value is valid.
 * Exact and deterministic.  At most 128 source pixels per destination pixel on each axis (sx, sy <= 128); beyond that
 * the call fails.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_resample_stat(const void *src_dev, int src_dtype, long hs, long ws, int has_nodata, double nodata,
                     float *dst_dev, long hd, long wd, double sx, double ox, double sy, double oy, int method,
                     void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Block normalisation statistics: KernelModel._fit_block_norm (kernel_model.py:216-229).
 *   norm[0] = std(ref[mask]) / std(src[mask]);  norm[1] = P1(ref[mask]) - P1(src[mask]) * norm[0]
 * over mask = valid(src) & valid(ref), numpy-linear 1st percentile; {0, 0} for an empty mask.
 * norm_dev: 2 doubles on the device.  workspace_dev: hb_block_norm_workspace_bytes(n) bytes of device scratch,
 * 256-byte aligned.  Up to 2^28 pixels the float32 standard deviations replay numpy's pairwise float32 np.std to the bit
 * (compaction of the valid pixels in C order + numpy's summation tree); larger blocks use double accumulation.
 * --------------------------------------------------------------------------------------------------------------- */
size_t hb_block_norm_workspace_bytes(long n);
int hb_block_norm(const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                  int ref_has_nodata, double ref_nodata, long n, double *norm_dev, void *workspace_dev,
                  size_t workspace_bytes, void *stream);

/* Row-band shards (one raster split by rows over several GPUs, SURVEY.md 8e): _fit_block_norm is a statistic of the
 * WHOLE block (kernel_model.py:216-229), so the three streaming passes of hb_block_norm are run per shard and resolved
 * after an exchange.  Per level (0, 1, 2, in this order), every rank calls
 *     hb_block_norm_partial(level, its rows of both planes, n_local, ...)             -- accumulate only
 * all-gathers the first hb_block_norm_message_bytes(n_local_max, n_total) bytes of its workspace (the level's counts,
 * sums, histograms, the shard's first / last valid pixels and its pairwise-leaf sums) into `gathered_dev` = world x
 * message_bytes, in rank order, and calls
 *     hb_block_norm_merge(level, gathered_dev, world, rank, ...)                      -- sum over ranks + resolve
 * n_local_max = pixels of the largest shard, n_total = pixels of the whole block (both the same on every rank); the
 * workspace holds hb_block_norm_shard_workspace_bytes(n_local_max, n_total) bytes, 256-byte aligned.  The merge adds the
 * shards' accumulators in rank order, so every rank derives bit-identical statistics, and up to 2^28 pixels per block
 * the float32 standard deviations replay numpy's pairwise np.std over the concatenation of the shards' valid pixels:
 * after level 2 norm_dev holds exactly the two doubles hb_block_norm gives for the unsharded planes.  n_local may be 0;
 * at most 64 shards. */
size_t hb_block_norm_shard_workspace_bytes(long n_local_max, long n_total);
size_t hb_block_norm_message_bytes(long n_local_max, long n_total);
int hb_block_norm_partial(int level, const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                          int ref_has_nodata, double ref_nodata, long n_local, long n_local_max, long n_total,
                          void *workspace_dev, size_t workspace_bytes, void *stream);
int hb_block_norm_merge(int level, const void *gathered_dev, int world, int rank, long n_local_max, long n_total,
                        void *workspace_dev, size_t workspace_bytes, double *norm_dev, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Same-grid fit: KernelModel.fit -> _fit_gain / _fit_gain_blk_offset / _fit_gain_offset + _r2_array
 * (kernel_model.py:142-373, 411-440), without the in-painting step.
 *   src, ref   float32 [h][w] on the same grid; they are NOT modified.
 *   params     float32 [2 or 3][h][w]: gain, offset, (R2 when want_r2); NaN outside mask = valid(src)&valid(ref).
 *   norm_dev   device pointer to the 2 doubles of hb_block_norm (HB_MODEL_GAIN_BLK_OFFSET only, else NULL).
 *   sums_dev   optional float32 [3][h][w] receiving the window sums (sum ref, sum src, count) that
 *              hb_inpaint_refit needs; NULL to skip.
 * Window sums are centred kh x kw box sums with zero padding (cv.boxFilter BORDER_CONSTANT), accumulated in
 * double and rounded exactly where OpenCV / numpy round them (SURVEY.md 8a numerics note).  kh, kw odd, <= 127.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_fit_same_grid(const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                     int ref_has_nodata, double ref_nodata, long h, long w, int model, int kh, int kw, int want_r2,
                     const double *norm_dev, float *params_dev, float *sums_dev, void *stream);

/* hb_fit_same_grid for the output rows [row0, row0 + nrows) only: the planes still hold h rows (the windows of the
 * first / last output rows reach into the rows around them), params_dev / sums_dev hold nrows rows per plane.  What a
 * row band of a sharded raster calls on its rows + halo (SURVEY.md 8e; the reference's block overlap, utils.py:136-153):
 * rows outside [0, h) are the reference's zero padding, rows inside are real neighbours. */
int hb_fit_same_grid_rows(const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                          int ref_has_nodata, double ref_nodata, long h, long w, long row0, long nrows, int model, int kh,
                          int kw, int want_r2, const double *norm_dev, float *params_dev, float *sums_dev, void *stream);

/* Same-grid fit fused with the apply step: corr = gain * src + offset (KernelModel.apply, kernel_model.py:442-463) of the
 * parameters hb_fit_same_grid would produce, written straight from the fit kernel's epilogue -- the parameters never
 * reach memory (8 bytes in + 4 out per pixel instead of 16 + 16 for fit then apply).  For the models / options whose
 * parameters are final after the fit: gain, gain-blk-offset (norm_dev as for hb_fit_same_grid), and gain-offset without
 * R2 in-painting.  corr_dev: float32 [h][w]; NaN where either input is invalid. */
int hb_fit_apply_same_grid(const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                           int ref_has_nodata, double ref_nodata, long h, long w, int model, int kh, int kw,
                           const double *norm_dev, int out_dtype, int out_has_nodata, double out_nodata, void *corr_dev,
                           void *stream);

/* hb_fit_apply_same_grid for the output rows [row0, row0 + nrows) only (see hb_fit_same_grid_rows); corr_dev holds
 * nrows rows. */
int hb_fit_apply_same_grid_rows(const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                                int ref_has_nodata, double ref_nodata, long h, long w, long row0, long nrows, int model,
                                int kh, int kw, const double *norm_dev, int out_dtype, int out_has_nodata,
                                double out_nodata, void *corr_dev, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Low-R2 in-painting and gain refit: kernel_model.py:361-371 (rasterio.fill.fillnodata == GDALFillNodata with
 * max_search_distance = 100, no smoothing).  params float32 [3][h][w] from hb_fit_same_grid(want_r2 = 1), sums from
 * the same call.  Offsets of pixels failing (R2 > thresh) & (gain > 0) & mask are inverse-distance filled from the
 * pixels passing it; their gains are re-estimated as (sum ref - N * offset) / sum src.
 * --------------------------------------------------------------------------------------------------------------- */
size_t hb_inpaint_workspace_bytes(long h, long w);
int hb_inpaint_refit(float *params_dev, const float *sums_dev, long h, long w, double r2_thresh,
                     double max_search_dist, void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Same-grid apply: KernelModel.apply (kernel_model.py:442-463): corr = params[0] * src + params[1] in float32 (two
 * roundings).  `mask_src` != 0 additionally writes NaN where src is nodata (the SrcSpaceModel.fit re-mask,
 * kernel_model.py:533, folded in for callers that did not materialise it).
 * --------------------------------------------------------------------------------------------------------------- */
int hb_apply_same_grid(const void *src_dev, int src_dtype, int has_nodata, double nodata, int mask_src,
                       const float *params_dev, long h, long w, int out_dtype, int out_has_nodata, double out_nodata,
                       void *corr_dev, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Fused parameter up-sampling + apply: RefSpaceModel.apply (kernel_model.py:484-503).
 *   params     float32 [2][hp][wp] (gain, offset; NaN = nodata) on the coarse grid.
 *   (sx, ox, sy, oy) maps SOURCE-grid pixel-edge coordinates to PARAM-grid pixel-edge coordinates.
 *   cover_dev  optional uint8 [hp][wp] full-coverage mask (mask_partial=True, kernel_model.py:493-498), looked up
 *              with nearest resampling; NULL = mask with the source nodata mask (kernel_model.py:500).
 *   corr       [hs][ws] of the output dtype = up(gain) * src + up(offset) (two float32 roundings, as numpy), nodata where
 *              masked.  The up-sampled parameters are never written to memory.
 *   method     HB_UP_CUBIC_SPLINE (GDAL GRA_CubicSpline: 4x4 cubic B-spline taps, invalid taps skipped and the rest
 *              renormalised), HB_UP_BILINEAR, HB_UP_CUBIC or HB_UP_LANCZOS.  HB_UP_NEAREST is rejected: nearest
 *              parameters are up-sampled with hb_resample_up and applied with hb_apply_same_grid.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_upsample_apply(const void *src_dev, int src_dtype, long hs, long ws, int has_nodata, double nodata,
                      const float *params_dev, long hp, long wp, double sx, double ox, double sy, double oy,
                      const uint8_t *cover_dev, int out_dtype, int out_has_nodata, double out_nodata, void *corr_dev,
                      int method, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Plain up-sampling of nb float32 bands (NaN nodata in, NaN nodata out): RasterArray.reproject(...,
 * resampling=cubic_spline | nearest | bilinear | cubic | lanczos), used by SrcSpaceModel.fit (kernel_model.py:520)
 * and RefSpaceModel.apply when the up-sampled parameters themselves are wanted.  (sx, ox, sy, oy) maps destination to
 * source coordinates; the destination must be at least as fine as the source.  Every method but nearest needs NaN
 * nodata and 1 or 2 bands per call (2 bands: a tap counts where its own band is valid, the centre pixel where any
 * band is).
 * --------------------------------------------------------------------------------------------------------------- */
int hb_resample_up(const float *src_dev, long nb, long hs, long ws, int has_nodata, double nodata, float *dst_dev,
                   long hd, long wd, double sx, double ox, double sy, double oy, int method, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Full-coverage mask: KernelModel._full_coverage_mask (kernel_model.py:375-409).
 *   in_mask    uint8 [hi][wi] validity mask of the OTHER image (source mask for RefSpace, reference mask for
 *              SrcSpace); (sx, ox, sy, oy) maps param-grid coordinates to in_mask-grid coordinates.
 *   params     float32 [2][hp][wp]; a param pixel is valid if either band is not NaN.
 *   out        uint8 [hp][wp] = erode( (average(in_mask) >= 1) & valid(params), ones(kh + 2, kw + 2) ), border 0.
 *   workspace  hp * wp bytes of device scratch.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_full_coverage_mask(const uint8_t *in_mask_dev, long hi, long wi, const float *params_dev, long hp, long wp,
                          double sx, double ox, double sy, double oy, int kh, int kw, uint8_t *out_dev,
                          void *workspace_dev, void *stream);

/* Stand-alone output dtype conversion of a float32 plane (nodata = NaN) -- for callers that already hold a float32
 * corrected plane; the apply entry points above fuse the same conversion into their stores.  RasterArray._convert_array_dtype
 * (raster_array.py:353-387) as used by to_rio_dataset (:493-500): integer outputs are rounded half-to-even and clipped
 * to the type's range; NaN pixels become `nodata` (0 when has_nodata == 0).  out_dtype: HB_U8, HB_U16, HB_I16 or HB_F32
 * (nodata substitution only).  One pass: 4 bytes read + sizeof(out) written per pixel. */
int hb_convert_dtype(const float *src_dev, long n, int out_dtype, int has_nodata, double nodata, void *dst_dev,
                     void *stream);

/* validity mask of a raster plane as uint8 (RasterArray.mask / mask_ra, raster_array.py:298-327) */
int hb_valid_mask(const void *src_dev, int src_dtype, long n, int has_nodata, double nodata, uint8_t *mask_dev,
                  void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Accuracy sums of RasterCompare: `get_block_sums` of RasterCompare.process (homonim/compare.py:232-256) for two
 * float32 planes of n pixels on one grid (the source and the reference after one of them was re-projected onto the
 * other's grid).  mask = valid(src) & valid(ref); pixels outside it count as zero in both planes.
 *   sums_dev   7 doubles on the device, in the reference's order:
 *              sum(src), sum(ref), sum(src^2), sum(ref^2), sum(src*ref), sum((ref-src)^2), sum(mask)
 * The per-pixel terms are rounded to float32 as numpy rounds them and accumulated in double in a fixed order.
 * workspace_dev: hb_compare_sums_workspace_bytes() bytes of 16-byte aligned device scratch.  8 bytes read per pixel.
 * --------------------------------------------------------------------------------------------------------------- */
size_t hb_compare_sums_workspace_bytes(void);
int hb_compare_sums(const float *src_dev, int src_has_nodata, double src_nodata, const float *ref_dev,
                    int ref_has_nodata, double ref_nodata, long n, double *sums_dev, void *workspace_dev,
                    size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * One (band, block) of RasterFuse._process_block (homonim/fuse.py:304-307: model.fit + model.apply) for proc_crs = ref
 * with DEVICE pointers, in one call: hb_downsample_average -> [hb_block_norm] -> hb_fit_same_grid ->
 * [hb_inpaint_refit] -> hb_upsample_apply, all enqueued on `stream` (asynchronous).  Device scratch is allocated with
 * cudaMallocAsync on `stream`.  params_dev: optional [2|3][hr][wr] float32 output of the fitted parameters (3 planes
 * when want_r2 != 0 or in-painting is on); may be NULL.  (sx, ox, sy, oy) maps REFERENCE-grid coordinates to
 * SOURCE-grid coordinates.  r2_thresh is ignored unless model == HB_MODEL_GAIN_OFFSET and do_inpaint != 0.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_fuse_refspace(const void *src_dev, int src_dtype, long hs, long ws, int src_has_nodata, double src_nodata,
                     const float *ref_dev, long hr, long wr, int ref_has_nodata, double ref_nodata, double sx, double ox,
                     double sy, double oy, int model, int kh, int kw, int want_r2, int do_inpaint, double r2_thresh,
                     int out_dtype, int out_has_nodata, double out_nodata, void *corr_dev, float *params_dev,
                     void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Host-buffer convenience entry point: one (band, block) of RasterFuse._process_block (homonim/fuse.py:304-307)
 * for proc_crs = ref, with HOST pointers.  Copies the source / reference planes to the device, runs
 * hb_downsample_average -> [hb_block_norm] -> hb_fit_same_grid -> [hb_inpaint_refit] -> hb_upsample_apply, and copies
 * the corrected plane (and, when params_host != NULL, the [2|3][hr][wr] parameters) back; synchronises `stream`
 * before returning.  Device scratch is allocated with cudaMallocAsync on `stream`.
 * (sx, ox, sy, oy) maps REFERENCE-grid coordinates to SOURCE-grid coordinates.
 * r2_thresh is ignored unless model == HB_MODEL_GAIN_OFFSET and do_inpaint != 0.
 * --------------------------------------------------------------------------------------------------------------- */
int hb_fuse_refspace_host(const void *src_host, int src_dtype, long hs, long ws, int src_has_nodata,
                          double src_nodata, const float *ref_host, long hr, long wr, int ref_has_nodata,
                          double ref_nodata, double sx, double ox, double sy, double oy, int model, int kh, int kw,
                          int want_r2, int do_inpaint, double r2_thresh, int out_dtype, int out_has_nodata,
                          double out_nodata, void *corr_host, float *params_host, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Overview pyramid of written planes: RasterFuse._build_overviews (homonim/fuse.py:151-165, Resampling.average) on the
 * corrected / parameter planes as they are stored in the output file.
 *   src        [nb][h][w] of `dtype` (HB_U8, HB_U16, HB_I16 or HB_F32), the written values (output dtype and nodata).
 *   levels_dev HOST array of n_levels (1..8) DEVICE pointers; level k (1-based) is [nb][ceil(h / 2^k)][ceil(w / 2^k)] of
 *              the same dtype.
 * Level k is computed from level k - 1 as stored (level 0 = src): pixel (i, j) averages the valid pixels among rows 2i,
 * 2i+1 and columns 2j, 2j+1 of level k - 1 (rows / columns past an odd edge are absent).  Valid = not equal to nodata
 * (when has_nodata) and, for HB_F32, not NaN; a window without valid pixels gets nodata (NaN for HB_F32 without one).
 * Integer types: floor((2s + n) / 2n) of the exact sum s of the n valid pixels (round half up).  HB_F32: the valid
 * values summed in double in the order top-left, top-right, bottom-left, bottom-right, divided by n in double, rounded
 * once to float.  Two kernel launches at most (levels 1-6 from one read of the plane, then levels 7-8).
 * --------------------------------------------------------------------------------------------------------------- */
int hb_build_overviews(const void *src_dev, int dtype, long nb, long h, long w, int has_nodata, double nodata,
                       int n_levels, void *const *levels_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HOMONIM_B200_H */
