/*
 * hipr_b200.h -- C ABI of libhipr_b200.so, the B200 (sm_100a) implementation of the HiPR-FISH
 * spectral-segmentation front end.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch/numpy types.  Every entry
 * point names the reference code it replaces (paths relative to the reference repository;
 * eco/ = hiprfish-image-analysis-ecoli, bio/ = hiprfish-image-analysis-biofilm,
 * syn/ = hiprfish-image-analysis-synthetic-community).  INTEGRATION.md shows the ctypes
 * binding a reference maintainer adds.
 *
 * Conventions
 *  - All arrays are C-contiguous, channel (or line sample) fastest, exactly as the reference's
 *    numpy arrays are.  "dev" pointers are device pointers, "host" pointers host memory.
 *  - dtype codes: HIPR_F32 = 0 (float), HIPR_F64 = 1 (double); the label entry points and
 *    hipr_paint_labels also take HIPR_I32 = 2, HIPR_I64 = 3 and HIPR_U8 = 4 (uint8 / bool).
 *  - Every function returns 0 on success, a negative HIPR_E* code for a rejected argument, or
 *    a positive cudaError_t value.  hipr_error_string() describes either.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device entry
 *    points only enqueue work; they never synchronise.
 *  - Line tables are passed as HOST int32 arrays in patch coordinates (0 .. patch_size-1),
 *    shape (n_dirs, patch_size, ndim), as built by eco/neighbor2d.pyx:32-55 or
 *    bio/neighbor.pyx:141-170; the library never recomputes them (they depend on libm
 *    rounding, SURVEY.md section 4).
 */
#ifndef HIPR_B200_H
#define HIPR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HIPR_ABI_VERSION 1

#define HIPR_F32 0
#define HIPR_F64 1
#define HIPR_I32 2
#define HIPR_I64 3
#define HIPR_U8  4

/* epilogue flavours (SURVEY.md section 8a) */
#define HIPR_FLAVOUR_F1  1  /* syn/..._measurement.py:111-124 */
#define HIPR_FLAVOUR_F2  2  /* bio/..._analysis.py:905-917 */
#define HIPR_FLAVOUR_F3  3  /* bio/..._analysis.py:1114-1125 */
#define HIPR_FLAVOUR_ME2 4  /* bio/neighbor.pyx:256-262 + bio/..._analysis.py:812-817 */
#define HIPR_FLAVOUR_V3  5  /* bio/neighbor.pyx:335-348 */

#define HIPR_OK            0
#define HIPR_E_ARG        -1  /* null pointer / non-positive size */
#define HIPR_E_DTYPE      -2
#define HIPR_E_PATCH      -3  /* patch_size even, < 3 or too large; image smaller than patch */
#define HIPR_E_TABLE      -4  /* table entry outside the patch / table too large */
#define HIPR_E_FLAVOUR    -5
#define HIPR_E_ALIGN      -6
#define HIPR_E_RANGE      -7  /* size overflows the kernel's index type */
#define HIPR_E_NODEVICE   -8
#define HIPR_E_UNSUPPORTED -9 /* valid request outside this entry point's fast path; use the general one */

#define HIPR_MAX_PATCH     31
#define HIPR_MAX_TABLE     960   /* n_dirs * patch_size, fits the kernel parameter bank */
#define HIPR_MAX_DIRS      128

int         hipr_abi_version(void);
const char *hipr_error_string(int code);
/* number of kernels this library has launched in the calling process (for bench.py) */
int64_t     hipr_launch_count(void);
/* multiprocessor count of the current device, or a negative error */
int         hipr_sm_count(void);

/* ---- prologue: channel sum (+ global max) -------------------------------------------------
 * Replaces `np.sum(image_channel, axis=2)` and the np.max that follows it,
 * syn/..._measurement.py:105-106 (bio/..._analysis.py:347-348, 451-452, 808-809).
 *   cube_dev   (npix, C) float32
 *   calib_dev  NULL, or (npix, C) float32 flat-field divisor (syn/..._measurement.py:104)
 *   sum_dev    (npix) of sum_dtype; channel sums are accumulated in float64 either way
 *   maxkey_dev NULL, or TWO uint64: [0] receives an order-preserving key of max(sum), [1] of
 *              min(sum) (decode with hipr_maxkey_decode; consumed by hipr_normalize,
 *              hipr_lne2d, hipr_lne2d_q); both are reset by this call
 */
int hipr_chansum(const float *cube_dev, const float *calib_dev, int64_t npix, int C,
                 void *sum_dev, int sum_dtype, uint64_t *maxkey_dev, void *stream);

/* Channel sum of RAW detector counts: cube_dev (npix, C) of uint16 (sample_bytes 2) or uint8 (1).  Each sample
 * becomes the float32 value python-bioformats' load_image(rescale=True) hands the scripts at
 * syn/..._measurement.py:81, image.astype(np.float32) / float(scale), one correctly rounded float32 divide,
 * before the float64 channel sum: the same sums as hipr_chansum on the rescaled float32 cube, from half (a
 * quarter) of the bytes.  sum_dev (npix) float64; maxkey_dev as hipr_chansum. */
int hipr_chansum_raw(const void *cube_dev, int sample_bytes, double scale, int64_t npix, int C,
                     double *sum_dev, uint64_t *maxkey_dev, void *stream);

/* ---- registration paste + channel stack + flat field + channel sum, one pass --------------------
 * Replaces syn/..._measurement.py:86-105 (bio/..._analysis.py:330-348; eco/..._measurement.py:147-148
 * with zero shifts): the per-excitation images are pasted at their integer registration shifts
 *   registered_e[r, c, :] = stack_e[r - shift_row[e], c - shift_col[e], :]      (0 where that falls outside)
 * stacked along the channel axis (np.dstack), divided by the flat field, and channel-summed.
 *   stacks_dev  HOST array of n_stacks device pointers, stack e is (H, W, chans[e]) float32
 *   chans, shift_row, shift_col   HOST int32 arrays of length n_stacks (<= 8; sum of chans <= 192)
 *   calib_dev   NULL, or (H, W, C) float32 divisor, C = sum(chans)
 *   cube_dev    NULL, or (H, W, C) float32: receives the registered (and flat-fielded) cube, the
 *               `image_registered` the scripts save and run the per-cell reduction on
 *   sum_dev     (H, W) float64 channel sums of the registered, flat-fielded cube
 *   maxkey_dev  NULL or two keys (max, min of the sums), as hipr_chansum
 * The shifts can be estimated on the device from the same stacks with hipr_excitation_shifts (below).
 */
int hipr_register_stacks(const float *const *stacks_dev, const int32_t *chans, const int32_t *shift_row,
                         const int32_t *shift_col, int n_stacks, int H, int W, const float *calib_dev,
                         float *cube_dev, double *sum_dev, uint64_t *maxkey_dev, void *stream);

/* ---- registration shifts: float64 FFT cross-correlation (csrc/xcorr2d.cu) ---------------------------------------
 * Replaces skimage.feature.register_translation(src, target)[0] with its defaults (upsample_factor 1, space "real"),
 * syn/..._measurement.py:83-85: cc = ifftn(fftn(src) * conj(fftn(target))), the peak of |cc| by numpy's argmax
 * (a NaN wins over any number, ties go to the lowest flat index), and an index i > n // 2 wrapped to i - n.
 * Parity unpinned: scikit-image is not pinned by the reference (tests/shift_oracle.py::register_translation).
 * H and W are each a power of two in [2, 8192] (HIPR_E_UNSUPPORTED otherwise).  All arithmetic is float64.
 * hipr_xcorr2d_workspace_bytes: device scratch for n_images (2 for hipr_register_translation_2d, n_stacks for
 *   hipr_excitation_shifts; at most 8); negative for an unsupported size.  A smaller workspace is HIPR_E_RANGE.
 * hipr_register_translation_2d: src_dev, target_dev (H, W) of dtype; shift_dev receives (row, col) float64 with
 *   integer values; corr_dev NULL or (H, W) float64 receives |cc|.
 * hipr_excitation_shifts: the scripts' shifts for the excitation stacks of hipr_register_stacks (same stacks_dev,
 *   chans): per stack the float64 channel sum (hipr_chansum), transformed (transform 0: none; 1: log(sum + eps)),
 *   then register_translation(T(sum_0), T(sum_e)) for e >= 1; shifts_dev (n_stacks, 2) float64, row 0 = (0, 0).
 * Both only enqueue work on `stream`. */
int64_t hipr_xcorr2d_workspace_bytes(int H, int W, int n_images);
int hipr_register_translation_2d(const void *src_dev, const void *target_dev, int dtype, int H, int W,
                                 void *work_dev, int64_t work_bytes, double *shift_dev, double *corr_dev,
                                 void *stream);
int hipr_excitation_shifts(const float *const *stacks_dev, const int32_t *chans, int n_stacks, int H, int W,
                           int transform, double eps, void *work_dev, int64_t work_bytes, double *shifts_dev,
                           void *stream);

/* global min / max of any image as keys: range_dev[0] = max key, range_dev[1] = min key */
int hipr_image_range(const void *image_dev, int dtype, int64_t n, uint64_t *range_dev, void *stream);
/* out_dev[i] = (float)(sum_dev[i] / max), out of place from a float64 sum image
 * (maxkey_dev NULL: plain float64 -> float32 cast) */
int hipr_normalize_cast(const double *sum_dev, int64_t npix, const uint64_t *maxkey_dev, float *out_dev,
                        void *stream);

/* sum_dev[i] /= max   (syn/..._measurement.py:106).  maxkey_dev from hipr_chansum. */
int hipr_normalize(void *sum_dev, int sum_dtype, int64_t npix, const uint64_t *maxkey_dev,
                   void *stream);
/* decode the key into a double on the device (for callers that want the scalar) */
int hipr_maxkey_decode(const uint64_t *maxkey_dev, double *max_dev, void *stream);

/* range keys <-> doubles on the device: maxmin_dev[0] = max, [1] = min (used around the
 * cross-GPU all-reduce of a split mosaic's range) */
int hipr_range_decode(const uint64_t *range_dev, double *maxmin_dev, void *stream);
int hipr_range_encode(const double *maxmin_dev, uint64_t *range_dev, void *stream);

/* ---- non-local-means denoise of the sum image --------------------------------------------------
 * Replaces skimage.restoration.denoise_nl_means(image, h = h) as the 2-D callers use it (fast mode,
 * patch_size 7, patch_distance 11, sigma 0): syn/..._measurement.py:108, bio/..._analysis.py:350, 592, 668,
 * 725, 989.  image_dev, out_dev (H, W) of dtype; H, W > offset + patch_distance + 1 (a single reflection of
 * the border, as np.pad(mode='reflect') on such images).  patch_size 7 (or 6, which skimage makes 7) only,
 * patch_distance <= 15 (HIPR_E_UNSUPPORTED otherwise).  scikit-image is not pinned by the reference and is
 * not available to the oracle: parity is against the restated algorithm (oracle/hipr_oracle.py).
 */
int hipr_denoise_nl_means_2d(const void *image_dev, int H, int W, int dtype, int patch_size,
                             int patch_distance, double h, void *out_dev, void *stream);

/* The same for a z-stack: skimage.restoration.denoise_nl_means(volume, h = 0.03) on the (X, Y, Z) normalised sum
 * volume, bio/..._analysis.py:454 (fast mode, patch_size 7, patch_distance 11, sigma 0; a 3-D array read as a
 * volume, scikit-image >= 0.15 -- parity unpinned like the 2-D form).  volume_dev, out_dev (X, Y, Z) of dtype;
 * X, Y, Z > offset + patch_distance + 1.  workspace_dev: hipr_denoise_nl_means_3d_workspace(X, Y, Z,
 * patch_distance) bytes of device memory (the reflect-padded float64 copy); HIPR_E_RANGE if smaller. */
int hipr_denoise_nl_means_3d(const void *volume_dev, int X, int Y, int Z, int dtype, int patch_size,
                             int patch_distance, double h, void *out_dev, void *workspace_dev,
                             int64_t workspace_bytes, void *stream);
int64_t hipr_denoise_nl_means_3d_workspace(int X, int Y, int Z, int patch_distance);

/* ---- 2-D literal stencil ------------------------------------------------------------------
 * Replaces line_profile_2d_v2(image_padded, patch_size, phi_range), eco/neighbor2d.pyx:8-64:
 *   out[i, j, t, li] = image_padded[i + table[t, li, 0], j + table[t, li, 1]]
 *   image_padded_dev (Hp, Wp) of dtype;  out_dev (Hp-P+1, Wp-P+1, n_dirs, P) of dtype
 */
int hipr_line_profile_2d(const void *image_padded_dev, int Hp, int Wp, int dtype,
                         int patch_size, int n_dirs, const int32_t *table_host,
                         void *out_dev, void *stream);

/* The same gather from and to HOST arrays: what `from neighbor2d import line_profile_2d_v2`
 * (syn/..._measurement.py:30, :110) binds when the caller holds numpy arrays.
 *   image_padded_host (Hp, Wp) float64, C order
 *   out_host          (Hp-P+1, Wp-P+1, n_dirs, P) float64 -- 792 B per pixel at (11, 9)
 * The image is uploaded once; the gather runs in row bands on the device while the previous
 * bands cross PCIe (straight into out_host when it is page-locked, through the library's
 * page-locked staging ring and host threads when it is ordinary pageable memory).  Blocking;
 * hipr_host_last_elapsed_ms() gives the device-side time. */
int hipr_line_profile_2d_host(const double *image_padded_host, int Hp, int Wp, int patch_size,
                              int n_dirs, const int32_t *table_host, double *out_host);

/* ---- 2-D fused stencil + epilogue ("local neighbourhood enhancement") ---------------------
 * Replaces line_profile_2d_v2 (eco/neighbor2d.pyx:56-63) + the numpy epilogue of `flavour`
 * (F1 syn/..._measurement.py:111-124, F2 bio/..._analysis.py:671-683, F3 :1114-1125) and,
 * when padded == 0, the edge pad before it (syn/..._measurement.py:109).
 *   image_dev  (Hs, Ws) of dtype, row pitch `ld` elements.  padded != 0: it is the padded
 *              image and the output is (Hs-P+1, Ws-P+1); padded == 0: it is the unpadded
 *              image, border samples clamp to the edge, output is (Hs, Ws)
 *   maxkey_dev NULL, or the key from hipr_chansum: samples are divided by the max on load
 *   out_dev    (H, W) of dtype
 */
int hipr_lne2d(const void *image_dev, int Hs, int Ws, int64_t ld, int padded, int dtype,
               int patch_size, int n_dirs, const int32_t *table_host, int flavour,
               const uint64_t *maxkey_dev, void *out_dev, void *stream);

/* Same operation on a 31-bit fixed-point copy of the image (exact min / max / differences; see
 * csrc/lne2d_q.cu).  This is what the cube -> score pipeline uses: image_dev is the float64 (or
 * float32) channel-sum image, range_dev the two keys from hipr_chansum / hipr_image_range; the
 * division by max is implied (the score is invariant to it; F3's epsilon is rescaled).
 * range_dev NULL (F1 / F2 only): every 32x32 tile is quantised with its own min / max.
 * patch_size must be 11 and n_dirs 9 (HIPR_E_TABLE otherwise: use hipr_lne2d).  out is float32.
 */
int hipr_lne2d_q(const void *image_dev, int Hs, int Ws, int64_t ld, int padded, int dtype,
                 int patch_size, int n_dirs, const int32_t *table_host, int flavour,
                 const uint64_t *range_dev, float *out_dev, void *stream);

/* ---- the whole 2-D front end in one call, kernels overlapped --------------------------------
 * cube_dev (H, W, C) float32 -> score_dev (H, W) float32 (same semantics as
 * hipr_neighbor2d_fused), as row bands: the channel sum of band b+1 (HBM-bound) runs on `stream`
 * while the fixed-point stencil of band b (SM-bound, tile-local quantisation) runs on an internal
 * side stream; `stream` is joined before returning control (csrc/pipeline2d.cu).
 *   sum_dev   (H, W) float64, receives the channel sums (required: it is the intermediate)
 *   range_dev 2 keys, receive max / min of the sums (reset by this call)
 *   bands     number of row bands (<= 0: default 1 = the two kernels back to back; banding
 *             measured slower on B200, see DESIGN.md); F3 always runs unbanded (global epsilon)
 * patch_size 11 / n_dirs 9 only (HIPR_E_UNSUPPORTED otherwise).
 */
int hipr_neighbor2d(const float *cube_dev, int H, int W, int C, int patch_size, int n_dirs,
                    const int32_t *table_host, int flavour, float *score_dev, double *sum_dev,
                    uint64_t *range_dev, int bands, void *stream);

/* ---- the whole 2-D front end in one launch -------------------------------------------------
 * cube_dev (H, W, C) float32 -> score_dev (H, W) float32: channel sum -> [/max] -> edge pad ->
 * line profiles -> epilogue, i.e. syn/..._measurement.py:105-124 without the skimage denoise
 * (flavour F1) or the F2 variant (bio/..._analysis.py:665-683).  The sum image stays on chip
 * (csrc/fused2d.cu).  sum_dev: NULL, or (H, W) float64 that receives the (unnormalised) channel
 * sums, with range_dev (2 keys, may be NULL) their max / min.
 * Handles patch_size 11 / 9 directions with the reference's table, flavours F1 and F2, W % 4 == 0,
 * a 16-byte aligned cube and C up to ~130; anything else returns HIPR_E_UNSUPPORTED and the
 * caller runs hipr_chansum + hipr_lne2d_q (same arithmetic, two launches).
 */
int hipr_neighbor2d_fused(const float *cube_dev, int H, int W, int C, int patch_size, int n_dirs,
                          const int32_t *table_host, int flavour, float *score_dev,
                          double *sum_dev, uint64_t *range_dev, void *stream);

/* ---- 3-D stencils -------------------------------------------------------------------------
 * hipr_line_profile_3d replaces line_profile_v2, bio/neighbor.pyx:115-181
 *   out (X, Y, Z, n_dirs, P).
 * hipr_lne3d_dirs replaces line_profile_memory_efficient_v2, bio/neighbor.pyx:186-263
 *   out (X, Y, Z, n_dirs): (centre - min) / max(max - min, 1e-8) per direction.
 * hipr_lne3d replaces the stencil + epilogue: F2 (bio/..._analysis.py:904-917), F3
 *   (:1112-1125), ME2 (:811-817), V3 = line_profile_memory_efficient_v3
 *   (bio/neighbor.pyx:268-349; pass the v3 table, reads use flat addressing, see DESIGN.md).
 * volume_dev is the PADDED volume (Xp, Yp, Zp) unless padded == 0 (edge clamp, as 2-D).
 */
int hipr_line_profile_3d(const void *volume_padded_dev, int Xp, int Yp, int Zp, int dtype,
                         int patch_size, int n_dirs, const int32_t *table_host,
                         void *out_dev, void *stream);
int hipr_lne3d_dirs(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype,
                    int patch_size, int n_dirs, const int32_t *table_host,
                    const uint64_t *maxkey_dev, void *out_dev, void *stream);
/* line_profile_memory_efficient_v2 from and to HOST arrays (what `from neighbor import
 * line_profile_memory_efficient_v2`, bio/..._analysis.py:39, :456, :812, binds for numpy callers):
 * padded float64 volume (Xp, Yp, Zp) in, (X, Y, Z, n_dirs) float64 out (576 B per voxel at 72
 * directions), computed in bands of x-planes under the device -> host copy of the previous bands
 * (page-locked out_host directly, pageable through the staging ring).  Blocking. */
int hipr_lne3d_dirs_host(const double *volume_padded_host, int Xp, int Yp, int Zp, int patch_size,
                         int n_dirs, const int32_t *table_host, double *out_host);
/* line_profile_v2 (bio/neighbor.pyx:115-181) from and to host arrays, same banding:
 * out_host (X, Y, Z, n_dirs, P) float64, 6,336 B per voxel at (11, 9, 9). */
int hipr_line_profile_3d_host(const double *volume_padded_host, int Xp, int Yp, int Zp, int patch_size,
                              int n_dirs, const int32_t *table_host, double *out_host);
int hipr_lne3d(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype,
               int patch_size, int n_dirs, const int32_t *table_host, int flavour,
               const uint64_t *maxkey_dev, void *out_dev, void *stream);

/* Fixed-point 3-D stencil (csrc/lne3d.cu, lne3d_q_kernel): the float64 (or float32) sum volume is
 * quantised brick by brick onto 31-bit integers, min / max / differences along the lines are
 * exact; float32 out.  dirs_only != 0: the (X, Y, Z, 72) output of
 * line_profile_memory_efficient_v2; else the fused score of `flavour` (F2 / F3 / ME2).
 * maxkey_dev: key of the global max (hipr_chansum) used to scale the 1e-8 epsilons of F3 / ME2;
 * NULL = the volume is already normalised.  The reference's (11, 9, 9) table only
 * (HIPR_E_UNSUPPORTED otherwise: use hipr_lne3d).
 */
int hipr_lne3d_q(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype,
                 int patch_size, int n_dirs, const int32_t *table_host, int flavour, int dirs_only,
                 const uint64_t *maxkey_dev, float *out_dev, void *stream);

/* ---- per-cell mean spectra ----------------------------------------------------------------
 * Replaces the regionprops loop, syn/..._measurement.py:167-172 (eco/...:151-157,
 * ref/...:177-183, bio/..._analysis.py:1214-1220, 1364-1369).
 * hipr_label_max:   max label (int64, >= 0) of a label image; label_bytes is 4 or 8.
 * hipr_cell_spectra_accumulate:
 *   cube_dev (npix, C) float32; labels_dev (npix) int32/int64, <= 0 = background;
 *   row_len = length of the label image's fastest axis (W, or Z for volumes), so that the
 *   kernel can walk 32 x 32 tiles; 0 (or a value that does not divide npix) = flat array;
 *   sums_dev (max_label+1, C) float64 and counts_dev (max_label+1) int32 are ADDED to (zero
 *   them first, or keep accumulating slabs / all-reduce them across ranks); labels above
 *   max_label are counted in *overflow_dev (int32, may be NULL).
 * hipr_cell_spectra_finalize:
 *   compacts to the labels present, ascending (regionprops order):
 *   n_cells_dev (1) int32; labels_out (max_label) int64; area_out (max_label) int64;
 *   avgint_out, avgint_norm_out (max_label, C) float64 -- the first n_cells rows are valid;
 *   avgint_norm = avgint / max(avgint, axis=1) (syn/..._measurement.py:172).
 */
int hipr_label_max(const void *labels_dev, int label_bytes, int64_t npix, int64_t *max_dev,
                   void *stream);
int hipr_cell_spectra_accumulate(const float *cube_dev, const void *labels_dev,
                                 int label_bytes, int64_t npix, int64_t row_len, int C,
                                 int64_t max_label,
                                 double *sums_dev, int32_t *counts_dev, int32_t *overflow_dev,
                                 void *stream);
/* zero the accumulators (cudaMemsetAsync on `stream`) */
int hipr_cell_spectra_reset(double *sums_dev, int32_t *counts_dev, int64_t max_label, int C,
                            void *stream);
int hipr_cell_spectra_finalize(const double *sums_dev, const int32_t *counts_dev,
                               int64_t max_label, int C, int32_t *n_cells_dev,
                               int64_t *labels_out, int64_t *area_out, double *avgint_out,
                               double *avgint_norm_out, void *stream);

/* ---- per-cell geometry and paint-by-label ---------------------------------------------------
 * hipr_cell_moments + hipr_cell_geometry_finalize replace skimage.measure.regionprops(segmentation) as
 * syn/hiprfish_imaging_classify_spectra.py:38-46 and bio/..._analysis.py:1232-1240 read it: label, centroid,
 * major_axis_length, minor_axis_length, eccentricity, orientation, area.
 *   labels_dev   (H, W) int32 / int64, <= 0 background;
 *   moments_dev  (max_label + 1, 6) uint64, zeroed by the call: count, sum r, sum c, sum r^2, sum c^2, sum r c
 *                (integer atomics: exact and order independent; slabs of a split mosaic can be all-reduced
 *                after offsetting rows on the host side);
 *   finalize: counts_scratch_dev (max_label + 1) int32 scratch; n_cells_dev (1) int32; labels_out, area_out
 *   (max_label) int64; geometry_out (max_label, 9) float64, the first n_cells rows valid, ascending label:
 *   [centroid_row, centroid_col, major_axis_length, minor_axis_length, eccentricity, orientation,
 *    mu20, mu02, mu11] (central moments of (row, col)).  Axis lengths and eccentricity are the eigenvalues of
 *   the coordinate covariance (4 sqrt(l)), the same in every scikit-image version; orientation follows the
 *   'rc' convention of scikit-image >= 0.16 (the reference does not pin its version).
 * hipr_paint_labels replaces the `image[segmentation == label] = value` loops,
 *   eco/hiprfish_imaging_image_classification.py:64-70, bio/..._analysis.py:1247-1257:
 *   out_dev[p, :] = values_dev[labels_dev[p], :], values_dev (max_label + 1, K) of dtype (row 0 = background);
 *   labels outside [0, max_label] take row 0.  dtype HIPR_F32 / HIPR_F64, or HIPR_I32 / HIPR_I64 / HIPR_U8 for the
 *   per-label lookup tables of the connected-component operators below.
 */
int hipr_cell_moments(const void *labels_dev, int label_bytes, int H, int W, int64_t max_label,
                      uint64_t *moments_dev, void *stream);
int hipr_cell_geometry_finalize(const uint64_t *moments_dev, int64_t max_label, int32_t *counts_scratch_dev,
                                int32_t *n_cells_dev, int64_t *labels_out, int64_t *area_out,
                                double *geometry_out, void *stream);
int hipr_paint_labels(const void *labels_dev, int label_bytes, int64_t npix, const void *values_dev, int K,
                      int64_t max_label, int dtype, void *out_dev, void *stream);

/* ---- connected components (csrc/label.cu) ----------------------------------------------------------------------
 * The segmentation back end between the k-means mask and the label image: syn/..._measurement.py:125-158,
 * eco/..._measurement.py:73-127, bio/..._analysis.py:367-419, 463-501.
 * hipr_label: scipy.ndimage.label(mask, generate_binary_structure(ndim, connectivity)) for a mask, and
 *   skimage.measure.label(image, background=0, connectivity=connectivity) for a label image (neighbours connect
 *   when their values are equal and non-zero; negative values are ordinary values).
 *   image_dev   C-order (d0, d1) (ndim 2) or (d0, d1, d2) (ndim 3); dtype HIPR_U8: a mask, non-zero is foreground
 *               (invert != 0: zero is foreground); HIPR_I32 / HIPR_I64: a label image
 *   connectivity 1 .. ndim (4 / 8 neighbours in 2-D, 6 / 18 / 26 in 3-D)
 *   labels_out  label_bytes 4 (int32) or 8 (int64): components numbered 1 .. n in raster order of their first
 *               pixel (scipy's and scikit-image's numbering), 0 for the background
 *   n_dev       one int64: n
 *   workspace   hipr_label_workspace_bytes(ndim, d0, d1, d2) bytes (negative: HIPR_E_RANGE when the image has
 *               2^31 pixels or more); what it holds before the call does not matter
 *   Five launches whatever the image holds; no host synchronisation.
 * hipr_label_counts: np.bincount of a label image into counts_dev (max_label + 1) int32, zeroed by the call.
 *   border >= 0: only pixels within `border` of an edge count (skimage clear_border's band of buffer_size + 1
 *   pixels); border < 0: all pixels.  Labels below 0 or above max_label are counted in *overflow_dev (may be NULL).
 * hipr_label_clear: clear_border's write, out[p] = flagged_dev[labels_dev[p]] != 0 ? fill : image[p];
 *   image_dev and out_dev (npix) of dtype HIPR_U8 / HIPR_I32 / HIPR_I64, labels_dev (npix) int32 in [0, n],
 *   flagged_dev (n + 1) int32 (the border counts of hipr_label_counts).
 * The per-label tables between these calls go through hipr_paint_labels (integer and uint8 values) and
 * hipr_label_max.
 */
int64_t hipr_label_workspace_bytes(int ndim, int d0, int d1, int d2);
int hipr_label(const void *image_dev, int dtype, int invert, int ndim, int d0, int d1, int d2, int connectivity,
               void *workspace_dev, int64_t workspace_bytes, void *labels_out, int label_bytes, int64_t *n_dev,
               void *stream);
int hipr_label_counts(const void *labels_dev, int label_bytes, int ndim, int d0, int d1, int d2, int border,
                      int64_t max_label, int32_t *counts_dev, int32_t *overflow_dev, void *stream);
int hipr_label_clear(const void *image_dev, int dtype, const int32_t *labels_dev, int64_t npix,
                     const int32_t *flagged_dev, int64_t fill, void *out_dev, void *stream);

/* ---- binary morphology (csrc/morphology.cu) ---------------------------------------------------------------------
 * The opening of the k-means mask before remove_small_objects / binary_fill_holes (syn/..._measurement.py:125-158,
 * bio/..._analysis.py:367-419, 463-501) and the erosion that makes the watershed seeds (eco/..._measurement.py:44-127).
 * hipr_binary_morphology: scipy.ndimage.binary_erosion(mask, structure, iterations, border_value=border_value)
 *   (dilate == 0) or scipy.ndimage.binary_dilation(...) (dilate != 0), origin 0, bit for bit.  Erosion:
 *   out[p] = AND over members o of in[p + o]; dilation: out[p] = OR over members o of in[p - o]; every pixel outside
 *   the image is border_value (non-zero = 1) in every pass.  An empty structure erodes to all 1 and dilates to all 0.
 *   mask_dev       C-order (d0, d1) (ndim 2) or (d0, d1, d2) (ndim 3) uint8, non-zero = 1
 *   structure_host C-order (s0, s1) (ndim 2) or (s0, s1, s2) (ndim 3) uint8 in HOST memory, non-zero = member; every
 *                  extent odd and <= HIPR_MORPH_MAX_EXTENT, at most HIPR_MORPH_MAX_RUNS runs (hipr_morphology_runs);
 *                  read during the call and passed to the kernel by value
 *   iterations     >= 1 passes, each a launch; the passes alternate between out_dev and the workspace, the last
 *                  writes out_dev
 *   out_dev        same shape, uint8 0 / 1; must not overlap mask_dev
 *   workspace      hipr_morphology_workspace_bytes(ndim, d0, d1, d2, iterations) bytes (0 for one pass; negative:
 *                  HIPR_E_RANGE when the image has 2^31 pixels or more); what it holds before the call does not matter
 *   No host synchronisation, no copy.  binary_opening is erosion then dilation, binary_closing dilation then erosion,
 *   each with the same iterations and border_value: two calls.
 * hipr_morphology_runs: the run table behind the kernel, host only.  Writes up to `capacity` runs of a (s0, s1, s2)
 *   structure (pass s0 = 1 for a 2-D one) into runs_out (capacity, 4) int32: (d0, d1, first d2, last d2), offsets from
 *   the centre, one per maximal run of members along the last axis, in C order; returns the number of runs (which may
 *   exceed capacity), HIPR_E_ARG for an even or non-positive extent, HIPR_E_RANGE for an extent above the limit.
 */
#define HIPR_MORPH_MAX_EXTENT 31
#define HIPR_MORPH_MAX_RUNS   1000  /* the run table travels in the 4 KB kernel parameter space; a full 31^3 cube has 961 */
int64_t hipr_morphology_workspace_bytes(int ndim, int d0, int d1, int d2, int iterations);
int hipr_binary_morphology(const uint8_t *mask_dev, int ndim, int d0, int d1, int d2, const uint8_t *structure_host,
                           int s0, int s1, int s2, int dilate, int border_value, int iterations, void *workspace_dev,
                           int64_t workspace_bytes, uint8_t *out_dev, void *stream);
int hipr_morphology_runs(const uint8_t *structure_host, int s0, int s1, int s2, int32_t *runs_out, int capacity);

/* ---- marker watershed (csrc/watershed.cu) -----------------------------------------------------------------------
 * skimage.segmentation.watershed(image, markers, connectivity=connectivity, mask=mask) (no compactness, no watershed
 * line), the last step of the segmentation back end: syn/..._measurement.py:125-158, eco/..._measurement.py:44-127,
 * bio/..._analysis.py:367-419, 463-501.  scikit-image floods from a heap keyed by (value, age); where two neighbours of
 * a pixel tie for the lowest level with different labels ("tie-decided" pixels: plateaus, quantised data, markers of
 * equal value) its answer depends on the age order.  This entry point computes a fully specified rule instead, which
 * equals the heap wherever no pixel is tie-decided (DESIGN.md K11): every flooded pixel gets the key (L, d, l) --
 * level (minimax path value from the markers, -0.0 equal to +0.0), hop count within the level group, label (signed)
 * -- a marker (v, 0, its label), any other in-mask pixel f(min over its in-mask neighbours of their keys), with
 * f((L, d, l), p) = (L, d + 1, l) if v(p) <= L, else (v(p), 1, l); its label is l.  At ties it prefers markers, then
 * fewer hops, then the smaller label.  Parity unpinned (scikit-image is not pinned by the reference).
 *   image_dev    C-order (d0, d1) (ndim 2) or (d0, d1, d2) (ndim 3) of image_dtype HIPR_F32 / HIPR_F64; no NaN inside
 *                the mask (the result is unspecified there)
 *   markers_dev  same shape, int32 (label_bytes 4) or int64 (8): any non-zero value is a marker; markers outside the
 *                mask are dropped (scikit-image's markers * mask)
 *   mask_dev     NULL (every pixel) or uint8, non-zero = inside
 *   connectivity 1 .. ndim, the offsets of hipr_label
 *   labels_out   same shape and dtype as the markers: the label of every flooded pixel; 0 outside the mask and
 *                where no marker reaches
 *   status_dev   8 int64, written by the call: [0] status (0 ok; k = 1, 2, 3: phase k still changed after its cap of
 *                npix + 1 rounds, which the algorithm never reaches -- treat as an internal error), [1..3] rounds of
 *                the three phases, [4..6] tile visits of the three phases, [7] CTAs of the launch
 *   workspace    hipr_watershed_workspace_bytes(...) bytes (negative: HIPR_E_RANGE when the image has 2^31 pixels or
 *                more); what it holds before the call does not matter
 * One memset and one cooperative launch whatever the image holds (HIPR_E_UNSUPPORTED without cooperative launch);
 * no host synchronisation.
 */
int64_t hipr_watershed_workspace_bytes(int ndim, int d0, int d1, int d2, int image_dtype, int label_bytes);
int hipr_watershed(const void *image_dev, int image_dtype, const void *markers_dev, int label_bytes,
                   const uint8_t *mask_dev, int ndim, int d0, int d1, int d2, int connectivity, void *workspace_dev,
                   int64_t workspace_bytes, void *labels_out, int64_t *status_dev, void *stream);

/* ---- 1-D k-means thresholding ---------------------------------------------------------------------------
 * Replaces KMeans(n_clusters = k, random_state = seed).fit_predict(image.reshape(-1, 1)) on the score map, the
 * denoised sum image or their logarithms, and the mask orientation that follows it:
 *   syn/..._measurement.py:125-149; bio/..._analysis.py:367-392, 463-486, 819-846, 1128-1156;
 *   eco/..._measurement.py:73-85 (log(sum + 1e-2)); ref/..._measurement.py:112-124.
 * Oracle: scikit-learn 1.9.0 (k-means++ seeding, Lloyd, tol = 1e-4 * var, labels from the final centres, best of
 * n_init by inertia).  scikit-learn's random draws are data independent in number, so the CALLER draws them:
 *   uniforms_host = numpy.random.RandomState(seed).random_sample(hipr_kmeans1d_uniforms(k, n_init))
 * (per initialisation: 1 for the first seed, then 2 + int(log(k)) per further seed).
 *   image_dev     (n) of dtype; sample value = image (transform 0), log10(image + eps) (1) or ln(image + eps) (2),
 *                 computed in float64; positive_only != 0: only samples with image > 0 take part (the
 *                 `image_final[image_final > 0]` call sites), in raster order
 *   workspace_dev hipr_kmeans1d_workspace_bytes() bytes of device scratch
 *   labels_out_dev NULL or (n) int32: scikit-learn's label of every sample; fill_label where positive_only excludes it
 *   mask_out_dev  NULL or (n) uint8: 1 where the sample belongs to the cluster with the largest mean of its positive
 *                 image values (the scripts' `i0 < i1` / np.argmax([i0, i1, i2]) orientation), else 0
 *   result_dev    32 doubles: [0] status (0 ok; 2 non-finite sample; 3 a cluster ran empty; 4 fewer samples than k),
 *                 [1] samples used, [2] their mean, [3] absolute tolerance, [4] Lloyd iterations, [5] inertia,
 *                 [6] index of the winning initialisation, [7] label of the brightest cluster,
 *                 [8..8+k) cluster_centers_, [16..16+k) cluster sizes, [24..24+k) mean of the positive image values
 * One cooperative launch (csrc/kmeans1d.cu); k <= 8; k * n_init bounded by hipr_kmeans1d_uniforms (HIPR_E_RANGE).
 */
int64_t hipr_kmeans1d_workspace_bytes(void);
int hipr_kmeans1d_uniforms(int k, int n_init);
int hipr_kmeans1d(const void *image_dev, int dtype, int64_t n, int transform, double eps, int positive_only, int k,
                  int n_init, const double *uniforms_host, int max_iter, double tol, void *workspace_dev,
                  int32_t *labels_out_dev, int fill_label, uint8_t *mask_out_dev, double *result_dev, void *stream);

/* ---- split mosaic over NVLink peer memory (BASELINE config 5) -------------------------------------------
 * The reference has no multi-GPU path; this is the exchange step of a stitched mosaic cut into row slabs, done by
 * this library's kernels through peer-mapped memory instead of a collective library (csrc/mosaic_p2p.cu).
 * Each rank allocates one buffer (hipr_p2p_alloc, hipr_mosaic_p2p_bytes), publishes its 64-byte IPC handle
 * (hipr_p2p_get_handle) and opens every other rank's (hipr_p2p_open_handle).  Per exchange (same `epoch` = 1, 2, ...
 * and parity = epoch & 1 on every rank): the caller's channel-sum kernel writes the slab's sums to
 * hipr_mosaic_p2p_rows_ptr(..., with_top_halo = 0); hipr_mosaic_p2p_exchange pushes the 5 edge rows into the
 * neighbours' halo rows and keys_local_dev (2 keys from hipr_chansum) into every rank's table, releases a flag,
 * then waits (bounded; *error_dev = 1 on timeout) for every rank's flag and writes the global max / min keys to
 * range_out_dev.  The extended image for hipr_lne2d_q starts at hipr_mosaic_p2p_rows_ptr(..., with_top_halo = rank > 0).
 *   bases_host  HOST array of `world` device pointers: entry r = rank r's buffer as mapped in this process
 *   rows, rows_up  height of this rank's slab and of the slab above (ignored for rank 0); rows_max = max over ranks
 */
int64_t hipr_mosaic_p2p_bytes(int rows_max, int W, int world);
int hipr_p2p_alloc(void **ptr, int64_t bytes);
int hipr_p2p_free(void *ptr);
int hipr_p2p_get_handle(void *ptr, void *handle64);
int hipr_p2p_open_handle(const void *handle64, void **peer_ptr);
int hipr_p2p_close_handle(void *peer_ptr);
int hipr_mosaic_p2p_rows_ptr(void *base, int rows_max, int W, int world, int parity, int with_top_halo,
                             double **rows_ptr);
int hipr_mosaic_p2p_exchange(void *const *bases_host, int rank, int world, int rows, int rows_up, int rows_max,
                             int W, int parity, const uint64_t *keys_local_dev, uint64_t epoch,
                             uint64_t *range_out_dev, int32_t *error_dev, void *stream);

/* Failure handling.  A wait kernel that does not see every peer's flag within the timeout (default ~10 s of SM
 * clocks; hipr_mosaic_p2p_set_timeout_ms changes it process-wide) sets *error_dev = 1 instead of hanging the GPU.
 * hipr_mosaic_p2p_guard, enqueued after the stencil, then overwrites that call's score with NaN, so a stale halo can
 * never pass as a result even if the caller does not poll error_dev (hipr_mosaic_p2p_score calls it itself). */
int hipr_mosaic_p2p_set_timeout_ms(double ms);
int hipr_mosaic_p2p_guard(const int32_t *error_dev, float *score_dev, int64_t n, void *stream);

/* The whole slab in one call, cube_slab_dev (rows, W, C) float32 -> score_dev (rows, W) float32, with the exchange
 * and the stencil hidden under the channel sum: row bands, first and last band summed first and their edge rows
 * pushed, then the channel sum of band b + 1 on `stream` while the stencil of band b runs on an internal side
 * stream (tile-local quantisation, flavours F1 / F2); F3, or bands < 3, runs sum -> exchange -> stencil in order.
 * keys_local_dev / range_dev: 2 uint64 of scratch each. */
int hipr_mosaic_p2p_score(const float *cube_slab_dev, int C, void *const *bases_host, int rank, int world, int rows,
                          int rows_up, int rows_max, int W, int parity, uint64_t epoch, const int32_t *table_host,
                          int flavour, int bands, uint64_t *keys_local_dev, uint64_t *range_dev, int32_t *error_dev,
                          float *score_dev, void *stream);

/* ---- host-buffer entry points (what a numpy caller binds; copies are inside) --------------
 * hipr_neighbor2d_host: cube_host (H, W, C) float32 -> score_host (H, W) float32:
 *   channel sum -> /max -> edge pad -> line profiles -> epilogue `flavour`, i.e.
 *   syn/..._measurement.py:105-124 without the skimage denoise (as bio/...:807-817 does).
 *   sum_host may be NULL or receives the (H, W) float32 normalised sum image.
 *   The cube is streamed to the device in row bands overlapped with the channel sum.
 *   Pinned host memory (hipr_host_alloc) gives full PCIe rate; pageable memory works.
 * hipr_cell_spectra_host: cube_host (npix, C) float32, labels_host (npix) int32/int64 ->
 *   *n_cells, labels_out/area_out (capacity) int64, avgint/avgint_norm (capacity, C) float64;
 *   returns HIPR_E_RANGE if capacity < number of cells.
 */
int hipr_neighbor2d_host(const float *cube_host, int H, int W, int C, int patch_size,
                         int n_dirs, const int32_t *table_host, int flavour,
                         float *score_host, float *sum_host);
/* hipr_neighbor3d_host: cube_host (X, Y, Z, C) float32 -> score_host (X, Y, Z) float32: channel sum -> /max -> edge
 * pad -> 3-D line profiles -> epilogue `flavour` (ME2: bio/..._analysis.py:807-817; F2: :900-917; F3: :1102-1125),
 * the cube streamed to the device in bands of x-planes under the channel sum. */
int hipr_neighbor3d_host(const float *cube_host, int X, int Y, int Z, int C, int patch_size, int n_dirs,
                         const int32_t *table_host, int flavour, float *score_host);
/* hipr_neighbor3d_host with the denoise of bio/..._analysis.py:454 between the normalisation and the stencil
 * (hipr_denoise_nl_means_3d, patch 7, distance denoise_distance (11 in the reference), h = denoise_h; the float64
 * stencil follows): lines 452-462 in full from a host cube. */
int hipr_neighbor3d_host_denoise(const float *cube_host, int X, int Y, int Z, int C, int patch_size, int n_dirs,
                                 const int32_t *table_host, int flavour, double denoise_h, int denoise_distance,
                                 float *score_host);
/* hipr_neighbor2d_host with the denoise of syn/..._measurement.py:108 between the normalisation and the stencil
 * (hipr_denoise_nl_means_2d, patch 7, distance 11, h = denoise_h; the float64 stencil follows): lines 105-124 in
 * full.  sum_host (may be NULL) receives the DENOISED normalised sum image (the scripts' image_registered_sum_nl). */
int hipr_neighbor2d_host_denoise(const float *cube_host, int H, int W, int C, int patch_size, int n_dirs,
                                 const int32_t *table_host, int flavour, double denoise_h, float *score_host,
                                 float *sum_host);
/* hipr_neighbor2d_host_batch: n_fov cubes (H, W, C) float32 -> n_fov score maps (H, W) float32, one FOV after
 * another as the scripts process a sample's fields of view (syn/..._measurement.py:161-173 under the Snakefile's
 * loop), pipelined across FOVs: FOV i + 1 is uploaded and summed while FOV i's normalisation, NL-means denoise
 * (denoise_h > 0: syn/..._measurement.py:106-124 in full; 0: without it, as hipr_neighbor2d_host), stencil and score
 * read-back run on a third stream.  Results are bit-identical to the single-FOV entry points. */
int hipr_neighbor2d_host_batch(const float *const *cubes_host, int n_fov, int H, int W, int C, int patch_size,
                               int n_dirs, const int32_t *table_host, int flavour, double denoise_h,
                               float *const *scores_host);
/* hipr_neighbor2d_host on raw uint16 / uint8 counts (see hipr_chansum_raw): half / a quarter of the PCIe
 * traffic of the float32 cube, same score. */
int hipr_neighbor2d_host_raw(const void *cube_host, int sample_bytes, double scale, int H, int W, int C,
                             int patch_size, int n_dirs, const int32_t *table_host, int flavour,
                             float *score_host, float *sum_host);
int hipr_cell_spectra_host(const float *cube_host, const void *labels_host, int label_bytes,
                           int64_t npix, int64_t row_len, int C, int64_t capacity,
                           int64_t *n_cells,
                           int64_t *labels_out, int64_t *area_out, double *avgint_out,
                           double *avgint_norm_out);
/* After hipr_cell_spectra_host returned HIPR_E_RANGE (*n_cells > capacity): copies that call's table, still on the
 * device, into arrays of sufficient capacity without recomputing it. */
int hipr_cell_spectra_host_fetch(int64_t capacity, int64_t *labels_out, int64_t *area_out, double *avgint_out,
                                 double *avgint_norm_out);
/* ---- field-of-view handle: one upload for the score map AND the per-cell spectra ------------------------------
 * The scripts hold `image_registered` across both steps (syn/..._measurement.py:161-173: generate_2d_segmentation
 * returns it, the regionprops loop at :167-172 reads it again after the watershed).  hipr_fov_upload streams the
 * (H, W, C) float32 cube to the CURRENT device once (row bands under the channel sum; page-locked memory from
 * hipr_host_alloc goes at the PCIe rate) and keeps cube, float64 channel sums and their range resident:
 *   hipr_fov_score         = hipr_neighbor2d_host without the upload (score_host / sum_host as there)
 *   hipr_fov_cell_spectra  = hipr_cell_spectra_host without the upload (HIPR_E_RANGE with *n_cells set when
 *                            capacity is too small: call again, the cube is still resident)
 *   hipr_fov_device_arrays   device pointers of the resident cube / sums / range keys (any may be NULL)
 *   hipr_fov_release         frees everything
 * A handle belongs to the device it was created on; calls switch to that device and restore the caller's.  Calls on
 * one handle are serialised; different handles are independent (own streams). */
int hipr_fov_upload(const float *cube_host, int H, int W, int C, void **handle_out);
int hipr_fov_score(void *handle, int patch_size, int n_dirs, const int32_t *table_host, int flavour,
                   float *score_host, float *sum_host);
int hipr_fov_cell_spectra(void *handle, const void *labels_host, int label_bytes, int64_t capacity, int64_t *n_cells,
                          int64_t *labels_out, int64_t *area_out, double *avgint_out, double *avgint_norm_out);
int hipr_fov_device_arrays(void *handle, const float **cube_dev, const double **sum_dev, const uint64_t **range_dev);
int hipr_fov_release(void *handle);

/* device-clock duration (CUDA events: before the first H2D .. after the last D2H) of the calling thread's most
 * recent host-buffer or handle call, in ms; negative if none yet */
double hipr_host_last_elapsed_ms(void);
int hipr_host_alloc(void **ptr, int64_t bytes);   /* page-locked host memory */
int hipr_host_free(void *ptr);
int hipr_host_release_workspace(void);            /* frees cached device buffers/streams */

#ifdef __cplusplus
}
#endif
#endif /* HIPR_B200_H */
