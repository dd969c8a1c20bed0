// Internal declarations shared by the translation units of libkltb200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/klt_b200.h"

// Kernel taps passed BY VALUE as a kernel parameter (constant bank): no global state, no symbol copies.
// c[j] is the tap that multiplies in[x + j - r]  (convolution: c[j] = taps[n-1-j]).
struct TapsF {
    int n, r, sym;   // sym: +1 symmetric, -1 antisymmetric, 0 general (SciPy's DBL_EPSILON test)
    float c[KLT_MAX_TAPS];
};
struct TapsD {
    int n, r, sym;
    int pad;
    double c[KLT_MAX_TAPS];
};

struct LevelDesc {
    int w, h, pitch;          // pitch in floats (multiple of 4)
    size_t off;               // offset in floats of image 0 inside the component plane
};

// host-only part of a pyramid (kept behind a pointer so that klt_pyr stays a small by-value kernel argument)
struct KltPyrHost {
    klt_taps taps;            // kernels of the last build (its level loops, lazy gradient builds and the windowed tracker read them)
    bool taps_valid;
    bool grad_valid;          // gradient planes of ALL levels hold the gradients of the current images
    bool grad0_valid;         // at least level 0 does (selection on a tracking pyramid needs only that one)
};

struct klt_pyr {
    KltPyrHost *hx;
    int w, h, n_levels, ss, batch;
    int precision;            // KLT_PRECISION_* of the last build (selects the tracking kernel's arithmetic)
    LevelDesc lv[KLT_MAX_LEVELS];
    size_t plane_floats;      // floats of ONE image's ONE component over all levels
    float *base;              // [which(3)][image(batch)][plane_floats]
    __host__ __device__ inline float *level(int which, int image, int l) const {
        return base + ((size_t)which * batch + image) * plane_floats + lv[l].off;
    }
};

struct klt_affine {
    int n, aw, ah;
    int *has;                 // [n] template present
    float *aff_x, *aff_y;     // [n] template centre
    float *A;                 // [n][4] Axx, Ayx, Axy, Ayy
    float *tmpl;              // [n][3][(ah+2)*(aw+2)]
    void *block;              // the single allocation behind the arrays above
};

// Per-kernel device timing (klt_profile_* in klt_b200.h): CUDA events recorded on the context's stream around
// every launch while profiling is enabled; resolved lazily.
struct KltProfRec {
    std::string name;
    double bytes;       // algorithmic bytes of all launches (compulsory reads + writes of that kernel)
    double ms;
    long count;
};
struct KltProfPending { int rec; cudaEvent_t e0, e1; };

struct klt_ctx {
    bool profiling;
    std::vector<KltProfRec> prof;
    std::vector<KltProfPending> prof_pending;
    std::vector<cudaEvent_t> prof_pool;
    int device;
    cudaStream_t stream;
    bool own_stream;
    std::string err;
    int64_t launches;
    cudaEvent_t ev0, ev1;
    // upload pipeline of klt_track_pairs_u8: copy stream, per-chunk events, device staging for the frames
    cudaStream_t copy_stream;
    cudaStream_t aux_stream;    // second compute stream: the second pyramid build of a device-resident klt_track_pairs_u8
    cudaEvent_t ov_ev[2];       // [0] entry, [1] "second pyramid built"
    cudaEvent_t chunk_ev[16];
    cudaEvent_t half_free[2];   // recorded on the compute stream once the builds have consumed that staging half
    int half_next;
    void *frames_dev;           // two staging halves, so that the upload of call k+1 overlaps the kernels of call k
    size_t frames_bytes;        // bytes of ONE half
    cudaEvent_t marks[16];      // klt_async_mark / klt_async_wait
    int *async_flag_dev;        // sticky "a window left the image" flag of the asynchronous calls (klt_async_result)
    // grow-only device workspace
    void *ws;
    size_t ws_bytes;
    int num_sms;
    int select_chunk;           // chunk capacity of select_walk_kernel (4096; $KLT_B200_SELECT_CHUNK shrinks it for tests)
};

int klt_fail(klt_ctx *ctx, int code, const char *fmt, ...);
#define KLT_CUDA(ctx, call)                                                                           \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return klt_fail(ctx, KLT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                            __FILE__, __LINE__);                                                      \
    } while (0)
#define KLT_CHECK_LAUNCH(ctx)                   \
    do {                                        \
        (ctx)->launches++;                      \
        KLT_CUDA(ctx, cudaGetLastError());      \
    } while (0)
// bracket a kernel launch: `bytes` = that launch's algorithmic bytes (inputs read once + outputs written once)
int klt_prof_begin(klt_ctx *ctx, const char *name, double bytes);
void klt_prof_end(klt_ctx *ctx, int token);
#define KLT_LAUNCH(ctx, name, bytes, ...)                       \
    do {                                                        \
        const int tok__ = klt_prof_begin(ctx, name, bytes);     \
        __VA_ARGS__;                                            \
        klt_prof_end(ctx, tok__);                               \
        KLT_CHECK_LAUNCH(ctx);                                  \
    } while (0)

// Grow-only workspace.  Every extern "C" entry point that uses ctx->ws reserves it once, for its whole layout (klt_ws_layout),
// before it enqueues anything into it, and nothing it calls reserves again: a reserve that grows frees the old block, and
// with it whatever the caller has already staged there.
int klt_ws_reserve(klt_ctx *ctx, size_t bytes);
bool klt_is_device_ptr(const void *p);

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Bump carver of one device block into 256-byte aligned buffers.  A layout is written once, as code that takes its buffers
// from a carver: run on a null base it only counts the bytes (off), run on the block it hands out the pointers.
struct KltCarver {
    char *base;
    size_t off;
    template <class T> T *take(size_t count) {
        T *p = base ? (T *)(base + off) : nullptr;
        off += align_up(count * sizeof(T), 256);
        return p;
    }
};

// layout(KltCarver &) sizes the workspace, which is reserved, then carves ctx->ws
template <class F> int klt_ws_layout(klt_ctx *ctx, F &&layout) {
    KltCarver c{nullptr, 0};
    layout(c);
    int rc = klt_ws_reserve(ctx, c.off);
    if (rc) return rc;
    c = KltCarver{(char *)ctx->ws, 0};
    layout(c);
    return KLT_OK;
}

// layout(KltCarver &) sizes one new allocation *block (what: the error message's name for it), then carves it
template <class F> int klt_alloc_layout(klt_ctx *ctx, void **block, const char *what, F &&layout) {
    KltCarver c{nullptr, 0};
    layout(c);
    cudaError_t e = cudaMalloc(block, c.off);
    if (e != cudaSuccess) {
        *block = nullptr;
        return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for %s failed: %s", c.off, what, cudaGetErrorString(e));
    }
    c = KltCarver{(char *)*block, 0};
    layout(c);
    return KLT_OK;
}

// A "host or device" array of a call.  klt_arg classifies the pointer once: a device array is used in place (dev == user), a
// host array gets a slot in the call's layout (place).  klt_arg_staged always goes through a slot.  klt_stage_in fills the
// slot from the caller's array, klt_stage_out copies it back, both on ctx->stream; without a slot they do nothing.
template <class T> struct KltArg {
    T *user;
    size_t n;
    bool host;
    T *dev;
    void place(KltCarver &c) { if (host) dev = c.take<T>(n); }
};
template <class T> KltArg<T> klt_arg(T *p, size_t n) { return {p, n, p && !klt_is_device_ptr(p), p}; }
template <class T> KltArg<T> klt_arg_staged(T *p, size_t n) { return {p, n, true, p}; }
template <class T> int klt_stage_in(klt_ctx *ctx, const KltArg<T> &a) {
    if (a.host) KLT_CUDA(ctx, cudaMemcpyAsync((void *)a.dev, a.user, a.n * sizeof(T), cudaMemcpyDefault, ctx->stream));
    return KLT_OK;
}
template <class T> int klt_stage_out(klt_ctx *ctx, const KltArg<T> &a) {
    if (a.host) KLT_CUDA(ctx, cudaMemcpyAsync(a.user, a.dev, a.n * sizeof(T), cudaMemcpyDefault, ctx->stream));
    return KLT_OK;
}

// the x, y, val arrays of a feature call
struct KltFeatures {
    KltArg<double> x, y;
    KltArg<int32_t> val;
    void place(KltCarver &c) { x.place(c); y.place(c); val.place(c); }
};
// classifies x, y and val, which must all be host or all be device
static inline int klt_features(klt_ctx *ctx, double *x, double *y, int32_t *val, size_t n, KltFeatures *f) {
    *f = KltFeatures{klt_arg(x, n), klt_arg(y, n), klt_arg(val, n)};
    if (f->y.host != f->x.host || f->val.host != f->x.host)
        return klt_fail(ctx, KLT_ERR_INVALID, "x, y, val must all be host or all be device");
    return KLT_OK;
}
static inline int klt_stage_in(klt_ctx *ctx, const KltFeatures &f) {
    int rc;
    if ((rc = klt_stage_in(ctx, f.x)) || (rc = klt_stage_in(ctx, f.y)) || (rc = klt_stage_in(ctx, f.val))) return rc;
    return KLT_OK;
}
static inline int klt_stage_out(klt_ctx *ctx, const KltFeatures &f) {
    int rc;
    if ((rc = klt_stage_out(ctx, f.x)) || (rc = klt_stage_out(ctx, f.y)) || (rc = klt_stage_out(ctx, f.val))) return rc;
    return KLT_OK;
}

// Status words of tracking: one call's (track_impl) or a sequence's since its last klt_sequence_sync.  Cleared by one memset
// and read back by one copy; the kernels get plain pointers to the fields.
struct KltTrackStatus {
    unsigned long long iters;     // Newton iterations
    int asserted;                 // a feature window left the image (the reference raises AssertionError)
    int scratch_assert;           // the backward pass's assert word under the forward-backward check (marks features only)
};

static inline bool klt_pyr_has_gradients(const klt_pyr *p) { return !p->hx || p->hx->grad_valid; }

int klt_make_taps(klt_ctx *ctx, const klt_kernel1d *k, TapsF *f, TapsD *d);

// ---- klt_api.cu: the pyramid build, shared with klt_select.cu and klt_sequence.cu ------------------------
extern "C" {   // (defined inside klt_api.cu's extern "C" block; not part of the public ABI)
// host state of a build with the caller's KLT_PRECISION_* (arithmetic, kernels, which gradient planes exist); enqueues
// nothing, so a graph replay of a build calls it in place of the captured klt_build_u8_device
void klt_pyr_note_build(klt_pyr *p, const klt_taps *taps, int precision);
// device frames -> pyramids for images [first, first+count) with the caller's KLT_PRECISION_*; dframes points at image
// `first`.  Records level0_done (may be null) right after the kernel that writes level 0.
int klt_build_u8_device(klt_ctx *ctx, klt_pyr *p, const uint8_t *dframes, size_t pitch, size_t frame_stride,
                        const klt_taps *taps, int precision, int first, int count, cudaEvent_t level0_done);
// gradient planes of levels [0, levels) of a built pyramid, built now where the last build left them out
int klt_ensure_gradients(klt_ctx *ctx, klt_pyr *p, int levels);
}

// ---- launchers (klt_conv.cu) -- all pointers are DEVICE pointers, pitches in elements ----------------
// separable convolution out = vk_v( hk_h(in) ), batched over `batch` images
int klt_launch_conv_sep_f32(klt_ctx *ctx, const float *in, size_t in_pitch, size_t in_stride, float *out,
                            size_t out_pitch, size_t out_stride, int w, int h, int batch, const klt_kernel1d *hk,
                            const klt_kernel1d *vk, int precision);
int klt_launch_conv_sep_u8(klt_ctx *ctx, const uint8_t *in, size_t in_pitch, size_t in_stride, float *out,
                           size_t out_pitch, size_t out_stride, int w, int h, int batch, const klt_kernel1d *hk,
                           const klt_kernel1d *vk, int precision);
// gradient pair: gx = g_v(d_h(in)), gy = d_v(g_h(in))
int klt_launch_grad_pair(klt_ctx *ctx, const float *in, size_t in_pitch, size_t in_stride, float *gx, float *gy,
                         size_t out_pitch, size_t out_stride, int w, int h, int batch, const klt_kernel1d *g,
                         const klt_kernel1d *d, int precision);
// pyramid step: out[y][x] = smooth(in)[ss*y+ss/2][ss*x+ss/2], only sampled outputs are evaluated
int klt_launch_pyr_down(klt_ctx *ctx, const float *in, size_t in_pitch, size_t in_stride, int w, int h, float *out,
                        size_t out_pitch, size_t out_stride, int ow, int oh, int ss, int batch,
                        const klt_kernel1d *g, int precision);

// ---- klt_stream.cu: warp-streaming FAST-path kernels; return 1 = launched, 0 = configuration not covered ----
// (first, count): the sub-range of the pyramid batch to build; `frames` points at image `first`
int klt_stream_level0(klt_ctx *ctx, const uint8_t *frames, size_t pitch, size_t frame_stride, klt_pyr *p, const klt_taps *taps,
                      int first, int count);
// u8 frame -> smoothed level-0 image only (image-only pyramids)
int klt_stream_smooth0(klt_ctx *ctx, const uint8_t *frames, size_t pitch, size_t frame_stride, klt_pyr *p, const klt_taps *taps,
                       int first, int count);
int klt_stream_level01(klt_ctx *ctx, const uint8_t *frames, size_t pitch, size_t frame_stride, klt_pyr *p, const klt_taps *taps,
                       int first, int count);
int klt_stream_grad(klt_ctx *ctx, klt_pyr *p, int level, const klt_taps *taps, int first, int count);
int klt_stream_down2(klt_ctx *ctx, klt_pyr *p, int level, const klt_taps *taps, int first, int count);

// ---- klt_select.cu -----------------------------------------------------------------------------------
// sat_dev: the summed-area tables, [3][w * h]
int klt_launch_scan(klt_ctx *ctx, const float *gx, const float *gy, size_t pitch, int w, int h, int bx, int by,
                    int hw, int hh, int skip, float *sat_dev, float *val_dev /* [ny][nx] */, int nx, int ny);
// full selection for every image of `pyr` (or, pyr == NULL, for B explicit device gradient images img_stride apart);
// x, y, val: [B][n_features] host or device; mask (optional, host or device): uint8 [B][h][mask_pitch], mask_stride apart
// (0: one mask for all images), nonzero = candidates allowed there
int klt_select_batch(klt_ctx *ctx, const klt_params *p, int select_mode, klt_pyr *pyr, const float *gx0, const float *gy0,
                     size_t img_stride, size_t pitch, int w, int h, int B, int n_features, int replace, double *x, double *y,
                     int32_t *val, int64_t *n_consumed, const uint8_t *mask = nullptr, size_t mask_pitch = 0,
                     size_t mask_stride = 0);

int klt_eigen_maps(klt_ctx *ctx, const klt_params *p, int select_mode, klt_pyr *pyr, float *val, int *nx_out, int *ny_out);

// ---- klt_track.cu ------------------------------------------------------------------------------------
// features of the images [first_image, first_image + n_images) of the batch (n_images < 0: all from first_image on);
// assert_marks_feature: see TrackArgs
int klt_launch_track(klt_ctx *ctx, const klt_params *p, const klt_pyr *p1, const klt_pyr *p2, int n_per_image,
                     double *x_dev, double *y_dev, int32_t *val_dev, unsigned long long *iters_dev, int *assert_dev,
                     int first_image = 0, int n_images = -1, int assert_marks_feature = 0);
// device scratch of the forward-backward check, [batch][n_per_image] each; scratch_assert: the backward pass's assert word
struct FbArrays { double *x0, *y0, *xb, *yb; int32_t *vb; int *scratch_assert; };
// klt_launch_track p1 -> p2 with the forward-backward check: (x0, y0) saved, forward track, fb_prepare, the backward track
// p2 -> p1 on (xb, yb, vb) (its template assertions mark the feature and raise only *scratch_assert), fb_check.  fb_error may
// be null.  All pointers are device pointers; graph-capturable.
int klt_launch_track_fb(klt_ctx *ctx, const klt_params *p, const klt_pyr *p1, const klt_pyr *p2, int n_per_image,
                        float max_fb_error, double *x, double *y, int32_t *val, const FbArrays &fa, float *fb_error,
                        unsigned long long *iters_dev, int *assert_dev);
int klt_launch_extract_patch(klt_ctx *ctx, const float *img, size_t pitch, int w, int h, float x, float y,
                             int height, int width, float *out_dev, int *ok_dev);
int klt_launch_iterate(klt_ctx *ctx, const klt_params *p, const float *tpatch_dev, const float *img2, const float *gx2,
                       const float *gy2, int w_img, int h_img, float x2, float y2, float *out_dev);
int klt_launch_patch_combine(klt_ctx *ctx, const float *p1_dev, const float *img, int w, int h, float x, float y, int height,
                             int width, int mode, float *out_dev, int *ok_dev);
int klt_greedy_presorted(klt_ctx *ctx, const unsigned long long *keys_host, unsigned int nkeys, int w, int h, int mindist,
                         int n_features, int overwrite, double *x, double *y, int32_t *val);

// ---- klt_affine.cu -----------------------------------------------------------------------------------
int klt_launch_affine(klt_ctx *ctx, const klt_params *p, const klt_pyr *p1, const klt_pyr *p2, int n_per_image,
                      const double *x_in, const double *y_in, const int32_t *val_in, double *x, double *y, int32_t *val,
                      klt_affine *st, int *assert_dev);
int klt_launch_affine_reset(klt_ctx *ctx, klt_affine *st, const int *mask_dev);

__host__ __device__ static inline int klt_reflect(int i, int n) {
    // scipy 'reflect' (half-sample symmetric); loop handles kernels wider than the image
    if (n == 1) return 0;
    while (i < 0 || i >= n) {
        if (i < 0) i = -i - 1;
        if (i >= n) i = 2 * n - i - 1;
    }
    return i;
}
