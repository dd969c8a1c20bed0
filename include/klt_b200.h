/*
 * klt_b200.h -- C ABI of libkltb200.so: the B200 (sm_100a) implementation of PyFeatureTrack's KLT hot path.
 *
 * This is the drop-in boundary.  The reference's "plugin" layer for this path is its two Cython
 * extension modules plus the SciPy call in convolve.py; each entry point below names the reference
 * interface it replaces (file:line into TimSC/PyFeatureTrack).  The Python modules in
 * pyfeaturetrack_b200/ (klt, convolve, pyramid, selectGoodFeatures, trackFeatures, goodFeaturesUtils,
 * trackFeaturesUtils) are thin ctypes shims over these functions; INTEGRATION.md shows the binding a
 * reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative klt_status;
 *     klt_last_error(ctx) returns a human-readable message for the last failure on that context.
 *   - no exceptions or exit() cross the ABI; the caller owns every host buffer; the library owns device
 *     memory behind opaque handles.
 *   - one klt_ctx per (GPU, stream).  A context is not thread-safe; distinct contexts may run concurrently.
 *   - pointer arguments documented "host or device" are classified with cudaPointerGetAttributes; host
 *     buffers are copied with cudaMemcpyAsync on the context's stream (pinned memory from
 *     klt_host_alloc makes those copies truly asynchronous).
 *   - there is NO CPU fallback: without a CUDA device klt_ctx_create fails with KLT_ERR_CUDA.
 *   - images are row-major; `pitch` arguments are in ELEMENTS, not bytes.
 */
#ifndef KLT_B200_H
#define KLT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLT_B200_ABI_VERSION 4
#define KLT_MAX_TAPS 71   /* convolve.py:28 maxKernelWidth */
#define KLT_MAX_LEVELS 8

/* error codes (return values) */
typedef enum klt_status {
    KLT_OK = 0,
    KLT_ERR_INVALID = -1,     /* bad argument */
    KLT_ERR_CUDA = -2,        /* CUDA runtime error (message has the cudaError string) */
    KLT_ERR_NOMEM = -3,
    KLT_ERR_UNSUPPORTED = -4, /* e.g. even-length kernel, border smaller than window half-size + 1 */
    KLT_ERR_ASSERT = -5       /* the reference would raise AssertionError (trackFeaturesUtils.pyx:35) */
} klt_status;

/* feature status codes == kltState (klt.py:23-29) */
#define KLT_TRACKED 0
#define KLT_NOT_FOUND (-1)
#define KLT_SMALL_DET (-2)
#define KLT_MAX_ITERATIONS (-3)
#define KLT_OOB (-4)
#define KLT_LARGE_RESIDUE (-5)
/* beyond the reference: the forward-backward check rejected the feature (klt_track_features_fb) */
#define KLT_FB_ERROR (-6)

/* arithmetic mode of the convolution / pyramid kernels */
#define KLT_PRECISION_FAST 0   /* fp32 FMA accumulation (<= 1e-6 relative-to-max of the reference images) */
#define KLT_PRECISION_STRICT 1 /* fp64 accumulation in SciPy's exact operation order: bit-identical images */
/* FAST arithmetic, pyramid builds only: write the intensity planes and skip the gradient planes.  klt_track_features
 * then evaluates the gradient pair (convolve.py:245-246) inside the windows the features visit, in shared memory;
 * anything that asks for a gradient plane (klt_pyr_download, klt_pyr_ensure_gradients, the affine tracker, window sizes
 * or gradient kernels the windowed tracker does not cover) builds the planes on demand, so results never depend on it. */
#define KLT_PRECISION_FAST_WINDOWED 2

typedef struct klt_ctx klt_ctx; /* one per (device, stream) */
typedef struct klt_pyr klt_pyr; /* a batch of image pyramids: intensity, gradx, grady for every level */
typedef struct klt_affine klt_affine; /* per-feature affine-consistency state (templates, template centre, 2x2 map) */
typedef struct klt_sequence klt_sequence; /* B lock-stepped sequences: rotating pyramid batches, device-resident feature lists */

/* how the minimum-eigenvalue map of a selection is computed */
#define KLT_SELECT_STRICT 0 /* float32 summed-area tables built by the reference's sequential chains (goodFeaturesUtils.pyx:49-51):
                             * on STRICT gradients the selection is bit-identical to the reference's */
#define KLT_SELECT_FAST 1   /* gradients + direct window sums + eigenvalue fused in one pass over the level-0 image; same
                             * feature SET as the reference for ~99.8 % of the features, not the same slots (SURVEY 7.3) */

/* One 1-D kernel, as produced by _computeKernels (convolve.py:27-93).  Computed on the host. */
typedef struct klt_kernel1d {
    int32_t n;                 /* odd, <= KLT_MAX_TAPS */
    int32_t reserved;
    double taps[KLT_MAX_TAPS]; /* convolution taps, index 0 = leftmost */
} klt_kernel1d;

/* The kernels one pyramid build uses (the reference's kernel cache can hand a stale kernel to any of
 * these roles, convolve.py:236,258 -- so they are per call, not per context). */
typedef struct klt_taps {
    klt_kernel1d smooth;     /* gauss(sigma = smooth_sigma_fact * max(window))      trackFeatures.py:166 */
    klt_kernel1d pyramid;    /* gauss(sigma = subsampling * pyramid_sigma_fact)     pyramid.py:42,60     */
    klt_kernel1d grad_gauss; /* gauss(grad_sigma)                                   convolve.py:245-246  */
    klt_kernel1d grad_deriv; /* gaussderiv(grad_sigma)                                                   */
} klt_taps;

/* The fields of KLT_TrackingContext (klt.py:44-73) read by selection and tracking. */
typedef struct klt_params {
    int32_t window_width, window_height;
    int32_t n_levels, subsampling;
    double borderx, bordery;      /* Python floats in the reference (quirk Q1: true division) */
    int32_t mindist, min_eigenvalue;
    int32_t n_skipped_pixels;
    int32_t max_iterations;
    float min_determinant, min_displacement, step_factor;
    int32_t has_max_residue;      /* 0 == tc.max_residue is None (klt.py:57) */
    float max_residue;
    int32_t retain_trackers;
    int32_t lighting_insensitive; /* gain/bias-normalised windows as in the C the reference carries as comments
                                   * (trackFeaturesUtils.pyx:152-239; the reference itself raises, :434-437): honoured by
                                   * klt_track_features (exact-order kernel), refused by klt_track_iterate and together
                                   * with the affine check.  Parity: against the oracle's restatement only. */
    /* affine consistency check (klt.py:67-73); only read by klt_track_features_affine */
    int32_t affine_consistency_check;        /* -1 off, 0 translation, 1 similarity, 2 affine */
    int32_t affine_window_width, affine_window_height;
    int32_t affine_max_iterations;
    float affine_max_residue, affine_min_displacement, affine_max_displacement_differ;
    float min_eigenvalue_f;       /* tc.min_eigenvalue when it is not an integer (the reference compares val >= min_eigenvalue in
                                   * floating point, selectGoodFeatures.py:116): if > 0 it replaces min_eigenvalue; pass the smallest
                                   * float32 >= the Python value */
} klt_params;

/* ---- library / context ------------------------------------------------------------------------- */
int klt_abi_version(void);
/* stream: a cudaStream_t to launch on (e.g. torch.cuda.current_stream().cuda_stream) or NULL to let
 * the context create its own non-blocking stream. */
int klt_ctx_create(int device, void *stream, klt_ctx **out);
int klt_ctx_destroy(klt_ctx *ctx);
const char *klt_last_error(const klt_ctx *ctx); /* ctx may be NULL: message of the last failed klt_ctx_create */
/* cudaStreamSynchronize on the context's stream.  Returns KLT_ERR_ASSERT (once) if a call that returned without waiting --
 * klt_track_features* on DEVICE arrays without n_iterations, klt_track_pairs_u8_async -- hit the reference's AssertionError
 * case since the last klt_sync / klt_async_result. */
int klt_sync(klt_ctx *ctx);
void *klt_ctx_stream(klt_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t klt_launch_count(const klt_ctx *ctx);
/* pinned host memory for asynchronous copies */
int klt_host_alloc(size_t bytes, void **out);
int klt_host_free(void *p);
/* device memory helpers for callers that want device-resident inputs without torch */
int klt_device_alloc(klt_ctx *ctx, size_t bytes, void **out);
int klt_device_free(klt_ctx *ctx, void *p);
int klt_memcpy(klt_ctx *ctx, void *dst, const void *src, size_t bytes); /* async on the ctx stream, any direction */
/* device timing on the context's stream: start/stop record CUDA events, elapsed synchronises */
int klt_timer_start(klt_ctx *ctx);
int klt_timer_stop(klt_ctx *ctx);
int klt_timer_elapsed_ms(klt_ctx *ctx, float *ms);

/* per-kernel device timing: while enabled, every kernel launch is bracketed by CUDA events on the context's stream.
 * klt_profile_get returns, per kernel name, the summed duration, launch count and summed ALGORITHMIC bytes
 * (each launch's compulsory traffic: inputs read once + outputs written once).  Used by bench.py's roofline. */
int klt_profile_enable(klt_ctx *ctx, int on);
int klt_profile_reset(klt_ctx *ctx);
int klt_profile_count(klt_ctx *ctx);
int klt_profile_get(klt_ctx *ctx, int index, const char **name, double *total_ms, int64_t *launches, double *bytes);

/* diagnostics: what this GPU sustains for the read/write MIX and launch size of one of the pyramid kernels, moved by a trivial
 * linear kernel that computes nothing (bench.py states each HBM-bound kernel against the ceiling of its own mix; no counterpart
 * in the reference).  total_bytes = bytes one launch moves; runs `reps` launches between two events on the context's stream. */
#define KLT_MIX_COPY 0     /* 16 B read : 16 B written */
#define KLT_MIX_SMOOTH0 1  /* 1 B read : 4 B written per pixel   (stream_smooth0) */
#define KLT_MIX_DOWN2 2    /* 16 B read : 4 B written per output pixel   (stream_down2) */
#define KLT_MIX_LEVEL01 3  /* 1 B read : 4 B + 1 B written per pixel, two output planes   (stream_level01) */
int klt_probe_traffic_mix(klt_ctx *ctx, int kind, double total_bytes, int reps, double *ms_per_rep, double *bytes_moved);

/* ---- operator level: replaces scipy.ndimage.convolve1d pairs behind convolve.py -------------------
 * klt_convolve_separable_f32  == _convolveSeparate(img, hk, vk)         convolve.py:208-214
 * klt_smooth_f32              == KLTComputeSmoothedImage's convolution  convolve.py:254-264
 * klt_gradients_f32           == KLTComputeGradients                    convolve.py:226-248
 * in/out: float32 [h][w] contiguous, host or device.  Reflect ('half-sample symmetric') borders. */
int klt_convolve_separable_f32(klt_ctx *ctx, const float *in, int w, int h, const klt_kernel1d *hk,
                               const klt_kernel1d *vk, int precision, float *out);
int klt_smooth_f32(klt_ctx *ctx, const float *in, int w, int h, const klt_kernel1d *gauss, int precision, float *out);
int klt_gradients_f32(klt_ctx *ctx, const float *in, int w, int h, const klt_kernel1d *gauss,
                      const klt_kernel1d *deriv, int precision, float *gradx, float *grady);

/* ---- pyramids: replaces ComputeImagePyramids (trackFeatures.py:146-196) and KLTPyramid (pyramid.py:14-77)
 * A klt_pyr holds `batch` independent images' three pyramids in one device allocation.
 * level dims follow pyramid.py:60-64: w_i = int(w_{i-1}/ss).                                           */
int klt_pyr_create(klt_ctx *ctx, int w, int h, int n_levels, int subsampling, int batch, klt_pyr **out);
int klt_pyr_destroy(klt_ctx *ctx, klt_pyr *pyr);
int klt_pyr_dims(const klt_pyr *pyr, int level, int *w, int *h, int *pitch);
size_t klt_pyr_bytes(const klt_pyr *pyr);
/* frames: uint8 [batch][h][pitch] (host or device), frame_stride in elements between images.
 * = img.convert("F") -> smooth -> KLTPyramid.Compute -> KLTComputeGradients per level, for every image.
 * precision KLT_PRECISION_FAST_WINDOWED defers the last step (see above); klt_select_good_features on such a pyramid
 * builds level 0's gradient planes first, klt_track_features_affine all of them. */
int klt_pyr_build_u8(klt_ctx *ctx, klt_pyr *pyr, const uint8_t *frames, size_t pitch, size_t frame_stride,
                     const klt_taps *taps, int precision);
/* same from float32 images (host or device).  already_smoothed != 0: the images ARE level 0 (pyramid.py:56 takes
 * the smoothed image as level 0 by reference); == 0: they are first smoothed with taps->smooth like the u8 path. */
int klt_pyr_build_f32(klt_ctx *ctx, klt_pyr *pyr, const float *images, size_t pitch, size_t frame_stride,
                      const klt_taps *taps, int precision, int already_smoothed);
/* which: 0 = intensity, 1 = gradx, 2 = grady.  out: float32 [h_level][w_level] contiguous, host or device. */
int klt_pyr_download(klt_ctx *ctx, const klt_pyr *pyr, int image, int which, int level, float *out);
/* device pointer of a level (for callers that keep working on the device).  A gradient plane of an image-only
 * (KLT_PRECISION_FAST_WINDOWED) pyramid does not exist until klt_pyr_ensure_gradients or klt_pyr_download has built
 * it: KLT_ERR_UNSUPPORTED until then. */
int klt_pyr_level_ptr(const klt_pyr *pyr, int image, int which, int level, const float **ptr);
/* Build the gradient planes of an image-only pyramid with the kernels of its last build (_KLTComputeGradients per
 * level, trackFeatures.py:171-176); no-op when they are valid. */
int klt_pyr_ensure_gradients(klt_ctx *ctx, klt_pyr *pyr);

/* ---- selection: replaces goodFeaturesUtils.ScanImageForGoodFeatures (goodFeaturesUtils.pyx:35-73),
 * the sort (selectGoodFeatures.py:234-236) and _enforceMinimumDistance (selectGoodFeatures.py:45-135).
 * klt_scan_good_features: gradx/grady float32 [h][w] (host or device) -> val float32 [ny][nx]
 *   (row-major over y in [by, h-by) step s, x in [bx, w-bx) step s), exactly the reference's pointlistval order. */
int klt_scan_good_features(klt_ctx *ctx, const float *gradx, const float *grady, int w, int h, int borderx,
                           int bordery, int window_hw, int window_hh, int n_skipped_pixels, float *val);
/* klt_select_good_features: full selection on level-0 gradients of image `image` of a pyramid batch
 * (pass pyr) or on explicit gradient images (pyr == NULL).  x, y, val: n_features host arrays.
 * replace == 0: SELECTING_ALL (all slots overwritten; unfilled slots get x=y=-1, val=KLT_NOT_FOUND);
 * replace == 1: REPLACING_SOME (slots with val >= 0 are kept and pre-marked, only val < 0 slots are filled).
 * n_consumed (optional): how many sorted candidates the greedy walk looked at. */
int klt_select_good_features(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr, int image,
                             const float *gradx, const float *grady, int w, int h, int n_features, int replace,
                             double *x, double *y, int32_t *val, int64_t *n_consumed);

/* The same for EVERY image of a pyramid batch in one chain of launches without host synchronisation (the candidate count,
 * the sort and the greedy walk are sized and driven on the device): KLTSelectGoodFeatures (replace == 0) or
 * KLTReplaceLostFeatures (replace == 1) for pyr->batch images.  x, y, val: [batch][n_features], host or device (device
 * arrays are updated in place and the call returns without waiting).  select_mode: KLT_SELECT_STRICT / KLT_SELECT_FAST. */
int klt_select_good_features_batch(klt_ctx *ctx, const klt_params *params, klt_pyr *pyr, int n_features, int replace,
                                   int select_mode, double *x, double *y, int32_t *val);

/* The minimum-eigenvalue maps alone, for every image of a pyramid batch, by either method: what ScanImageForGoodFeatures
 * returns as pointlistval (goodFeaturesUtils.pyx:53-71), val [batch][ny][nx] (host or device; NULL: only report nx, ny). */
int klt_eigen_map_batch(klt_ctx *ctx, const klt_params *params, klt_pyr *pyr, int select_mode, float *val, int *nx, int *ny);

/* ---- tracking: replaces KLTTrackFeatures' per-feature loop (trackFeatures.py:250-346), _trackFeature
 * (:67-136) and trackFeaturesUtils.trackFeatureIterateCKLT / extractImagePatch* / _compute* / _solveEquation
 * (trackFeaturesUtils.pyx:14-51,61-128,246-340,393-459).
 * pyr1/pyr2: pyramids of the first/second images (same geometry and batch).  x, y, val: [batch][n_per_image]
 * host or device arrays, updated in place exactly like the reference mutates the feature list
 * (lost features: x=y=-1, val=status; tracked: val=0).  Features with val < 0 are skipped.
 * n_iterations (optional, host): total Newton iterations executed.
 * Host arrays (or n_iterations != NULL): the call waits and returns KLT_ERR_ASSERT where the reference raises AssertionError
 * (a window leaves the image at some level, trackFeaturesUtils.pyx:35).  Device arrays with n_iterations == NULL: the call only
 * enqueues; that condition is then reported by the next klt_sync / klt_async_result on the context. */
int klt_track_features(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2,
                       int n_per_image, double *x, double *y, int32_t *val, int64_t *n_iterations);
/* ---- forward-backward check (Kalal, Mikolajczyk, Matas, ICPR 2010; beyond the reference and C-KLT).
 * klt_track_features, then every feature it reports KLT_TRACKED at (xf, yf) is tracked back from pyr2 to pyr1 with the same
 * params and kernels.  With e = sqrt(dx*dx + dy*dy) in double (dx = xb - x0, dy = yb - y0, (x0, y0) its position on entry),
 * the feature becomes x = y = -1, val = KLT_FB_ERROR when the backward track is lost or !(e <= max_fb_error); otherwise it keeps
 * the forward result.  A backward template that leaves the image rejects the feature and raises no KLT_ERR_ASSERT.
 * max_fb_error: level-0 pixels, finite and > 0.  fb_error (optional, [batch][n_per_image]): (float)e where the backward track
 * completed, -1 elsewhere.  x, y, val, fb_error host or device, same waiting / deferred-assert rules as klt_track_features;
 * n_iterations counts both passes. */
int klt_track_features_fb(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2,
                          int n_per_image, float max_fb_error, double *x, double *y, int32_t *val, float *fb_error,
                          int64_t *n_iterations);
/* ---- affine consistency check: the block at trackFeatures.py:347-399.  The reference's callees there
 * (_KLTCreateFloatImage, _am_getSubFloatImage, _am_trackFeatureAffine) are undefined (NameError); these entry points
 * implement the C-KLT 1.3.4 routines of those names (parity against oracle/klt_oracle.c, unpinned by the reference).
 * A klt_affine holds, for n_features_total feature slots, what the reference keeps on each KLT_Feature:
 * aff_img / aff_img_gradx / aff_img_grady ((aw+2) x (ah+2) templates), aff_x, aff_y, aff_Axx, aff_Ayx, aff_Axy, aff_Ayy. */
int klt_affine_create(klt_ctx *ctx, int n_features_total, int affine_window_width, int affine_window_height, klt_affine **out);
int klt_affine_destroy(klt_ctx *ctx, klt_affine *a);
/* mask (host, n_features_total ints, or NULL = all): slots to reset to "no template, aff_x = aff_y = -1, A = identity"
 * (what selectGoodFeatures.py:120-128 does to a (re)selected feature) */
int klt_affine_reset(klt_ctx *ctx, klt_affine *a, const int32_t *mask);
/* host copies of the state: has_template[n], aff_x[n], aff_y[n], A[n][4] = (Axx, Ayx, Axy, Ayy); any pointer may be NULL */
int klt_affine_download(klt_ctx *ctx, const klt_affine *a, int32_t *has_template, float *aff_x, float *aff_y, float *A);
/* template of one slot: float32 [3][(ah+2)][(aw+2)] (img, gradx, grady), host */
int klt_affine_download_template(klt_ctx *ctx, const klt_affine *a, int slot, float *out);
/* klt_track_features followed by the affine block for every feature the translational tracker reports KLT_TRACKED:
 * first successful track stores the template from pyr1 level 0; later tracks run the affine tracker against pyr2
 * level 0 and turn the feature's val into its status (x = y = -1 when lost).  x, y, val: host or device. */
int klt_track_features_affine(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2,
                              int n_per_image, double *x, double *y, int32_t *val, klt_affine *a, int64_t *n_iterations);

/* trackFeaturesUtils.extractImagePatchSlow(img, x, y, height, width) (trackFeaturesUtils.pyx:14-18):
 * img float32 [h][w] host or device, out float32 [height][width] host. */
int klt_extract_patch(klt_ctx *ctx, const float *img, int w, int h, float x, float y, int height, int width,
                      float *out);

/* trackFeaturesUtils.trackFeatureIterateCKLT(x2, y2, gxPatch, gyPatch, imgPatch, img2, gradx2, grady2, tc)
 * (trackFeaturesUtils.pyx:393-459): the Newton loop for ONE feature on caller-provided template patches.
 * patches: float32 [window_height][window_width] host; img2/gradx2/grady2: float32 [h][w] host or device. */
int klt_track_iterate(klt_ctx *ctx, const klt_params *params, float x2, float y2, const float *gx_patch,
                      const float *gy_patch, const float *img_patch, const float *img2, const float *gradx2,
                      const float *grady2, int w, int h, float *x2_out, float *y2_out, int32_t *status,
                      int32_t *iterations);
/* computeIntensityDifference (mode 0: out = patch1 - patch(img2 at x2,y2), pyx:61-97) and computeGradientSum
 * (mode 1: out = -patch1 - patch(img2 at x2,y2), pyx:107-142); out: float32 [height][width] host */
int klt_patch_combine(klt_ctx *ctx, const float *patch1, const float *img2, int w, int h, float x2, float y2, int height,
                      int width, int mode, float *out);
/* _enforceMinimumDistance(pointlist, featurelist, ncols, nrows, mindist, min_eigenvalue, overwriteAllFeatures)
 * (selectGoodFeatures.py:45-135) on a caller-ordered candidate list (host arrays, walked front to back) */
int klt_enforce_min_distance(klt_ctx *ctx, int n_points, const float *pval, const int32_t *px, const int32_t *py,
                             int ncols, int nrows, int mindist, double min_eigenvalue, int overwrite_all, int n_features,
                             double *x, double *y, int32_t *val);

/* ---- whole-call convenience: KLTTrackFeatures(tc, img1, img2, fl) for `batch` independent frame pairs with
 * HOST (ideally pinned) or device uint8 frames: upload, two pyramid builds, tracking, download.
 * pyr1/pyr2 are caller-provided scratch pyramids of matching geometry (reused across calls). */
int klt_track_pairs_u8(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int precision, klt_pyr *pyr1,
                       klt_pyr *pyr2, const uint8_t *frames1, const uint8_t *frames2, size_t pitch,
                       size_t frame_stride, int n_per_image, double *x, double *y, int32_t *val);
/* The same without waiting: everything, including the download of x / y / val, is only enqueued (pass pinned host
 * memory from klt_host_alloc, or device pointers; the frames must stay untouched until the stream has consumed them).
 * Two staging halves alternate between calls, so the upload of call k+1 overlaps the kernels of call k on ONE context
 * and one host thread -- SURVEY 8(f) rank 2.  klt_async_result waits for the stream and reports whether any of the calls
 * since the last klt_async_result hit the reference's AssertionError case (KLT_ERR_ASSERT), else KLT_OK. */
int klt_track_pairs_u8_async(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int precision,
                             klt_pyr *pyr1, klt_pyr *pyr2, const uint8_t *frames1, const uint8_t *frames2,
                             size_t pitch, size_t frame_stride, int n_per_image, double *x, double *y, int32_t *val);
int klt_async_result(klt_ctx *ctx);
/* Host-side completion marks for pipelining asynchronous calls: klt_async_mark(slot) records "everything enqueued so far"
 * (slot 0..15), klt_async_wait(slot) blocks the host until that point has been reached -- e.g. before reusing the pinned
 * buffers of the call before last. */
int klt_async_mark(klt_ctx *ctx, int slot);
int klt_async_wait(klt_ctx *ctx, int slot);

/* ---- sequences: KLTTrackFeatures in tc.sequentialMode (pyramid reuse, trackFeatures.py:152-161,401-404) followed by
 * KLTReplaceLostFeatures (_KLTSelectGoodFeatures(REPLACING_SOME) on tc.pyramid_last's gradients,
 * selectGoodFeatures.py:176-179,45-135) for n_sequences independent, lock-stepped sequences -- BASELINE config D.
 * A klt_sequence owns three pyramid batches and eigenvalue maps in rotation (previous / current frame / the frame whose
 * build is already running), the device-resident feature lists [n_sequences][n_features] and the selection workspace.
 * One step = one pyramid build + one tracking launch + one selection chain for all sequences, enqueued without any host
 * synchronisation; the frame-only half of a step (build, eigenvalue maps) runs on the sequence's own stream and overlaps the
 * list-dependent half of the previous step when the caller does not wait in between; after a warm-up both halves are
 * replayed from CUDA graphs.  precision: KLT_PRECISION_* of the pyramid builds (and with it the tracker's arithmetic); select_mode:
 * KLT_SELECT_*.  With KLT_PRECISION_STRICT + KLT_SELECT_STRICT every list equals the reference's bit for bit. */
int klt_sequence_create(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int w, int h, int n_sequences,
                        int n_features, int precision, int select_mode, klt_sequence **out);
int klt_sequence_destroy(klt_ctx *ctx, klt_sequence *seq);
/* first frames: uint8 [n_sequences][h][pitch], host (ideally pinned) or device.  Builds the pyramids; select != 0 also
 * runs KLTSelectGoodFeatures(tc, frame, n_features) for every sequence (else call klt_sequence_set_features). */
int klt_sequence_start_u8(klt_ctx *ctx, klt_sequence *seq, const uint8_t *frames, size_t pitch, size_t frame_stride,
                          int select);
/* x, y, val: [n_sequences][n_features], host or device */
int klt_sequence_set_features(klt_ctx *ctx, klt_sequence *seq, const double *x, const double *y, const int32_t *val);
/* next frames: KLTTrackFeatures(prev, cur) and, if replace != 0, KLTReplaceLostFeatures(cur) for every sequence.
 * Everything is only enqueued.  Optional outputs ([n_sequences][n_features]; pinned host memory or device; they are
 * written when the stream gets there -- klt_sequence_sync / klt_sync / klt_async_wait): x, y, val = the lists after the
 * step (tracked features val 0, new features val > 0, lost and not replaced val < 0); val_tracked = val after tracking,
 * before replacement (the kltState codes).  The frames must stay untouched until the stream has consumed them. */
int klt_sequence_step_u8(klt_ctx *ctx, klt_sequence *seq, const uint8_t *frames, size_t pitch, size_t frame_stride,
                         int replace, double *x, double *y, int32_t *val, int32_t *val_tracked);
/* synchronous download of the current lists (any pointer may be NULL) */
int klt_sequence_get_features(klt_ctx *ctx, klt_sequence *seq, double *x, double *y, int32_t *val, int32_t *val_tracked);
/* waits for the stream; KLT_ERR_ASSERT if a window left the image in one of the steps since the last call (the
 * reference's AssertionError, trackFeaturesUtils.pyx:35); n_iterations (optional): Newton iterations since then */
int klt_sequence_sync(klt_ctx *ctx, klt_sequence *seq, int64_t *n_iterations);
/* diagnostics of the last selection of every sequence: out [n_sequences][4] = candidates the greedy walk consumed, 1 if
 * the candidates ran out before every slot was filled, slots filled, number of times the walk had to widen its range */
int klt_sequence_select_stats(klt_ctx *ctx, klt_sequence *seq, int64_t *out);
/* the pyramid batch of the latest frame (owned by the sequence; valid until the next step) */
int klt_sequence_pyramid(klt_sequence *seq, klt_pyr **out);
/* 1 once steps are replayed from CUDA graphs (0: plain launches, e.g. while profiling or with $KLT_B200_NO_GRAPH) */
int klt_sequence_uses_graph(const klt_sequence *seq);
/* from the next step on: max_fb_error > 0 runs the forward-backward check of klt_track_features_fb inside the step's tracking
 * (before val_tracked is taken and before replacement, so rejected slots are refilled in the same step); 0 turns it off.
 * Drops the captured graphs. */
int klt_sequence_set_fb_check(klt_ctx *ctx, klt_sequence *seq, float max_fb_error);
/* synchronous download of the last step's fb_error [n_sequences][n_features] (host or device; -1 where no backward track
 * completed, everywhere when that step ran without the check) */
int klt_sequence_get_fb_error(klt_ctx *ctx, klt_sequence *seq, float *out);

#ifdef __cplusplus
}
#endif
#endif /* KLT_B200_H */
