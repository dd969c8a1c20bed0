// C ABI of libkltb200.so (see include/klt_b200.h): contexts, pyramids and the entry points that the Python
// shims in pyfeaturetrack_b200/ bind with ctypes.  Host-side orchestration only; kernels live in
// klt_conv.cu, klt_select.cu and klt_track.cu.
#include <cfloat>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "klt_common.cuh"
#include "klt_track_args.cuh"

static thread_local std::string g_create_error;

int klt_fail(klt_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return code;
}

bool klt_is_device_ptr(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

int klt_ws_reserve(klt_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->ws_bytes) return KLT_OK;
    if (ctx->ws) { KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); KLT_CUDA(ctx, cudaFree(ctx->ws)); ctx->ws = nullptr; ctx->ws_bytes = 0; }
    const size_t want = bytes + bytes / 4;
    cudaError_t e = cudaMalloc(&ctx->ws, want);
    if (e != cudaSuccess) return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for workspace failed: %s", want, cudaGetErrorString(e));
    ctx->ws_bytes = want;
    return KLT_OK;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int klt_prof_begin(klt_ctx *ctx, const char *name, double bytes) {
    if (!ctx->profiling) return -1;
    int rec = -1;
    for (size_t i = 0; i < ctx->prof.size(); i++)
        if (ctx->prof[i].name == name) { rec = (int)i; break; }
    if (rec < 0) { ctx->prof.push_back(KltProfRec{name, 0.0, 0.0, 0}); rec = (int)ctx->prof.size() - 1; }
    ctx->prof[rec].bytes += bytes;
    ctx->prof[rec].count += 1;
    KltProfPending pd;
    pd.rec = rec;
    for (cudaEvent_t *e : {&pd.e0, &pd.e1}) {
        if (!ctx->prof_pool.empty()) { *e = ctx->prof_pool.back(); ctx->prof_pool.pop_back(); }
        else cudaEventCreate(e);
    }
    cudaEventRecord(pd.e0, ctx->stream);
    ctx->prof_pending.push_back(pd);
    return (int)ctx->prof_pending.size() - 1;
}
void klt_prof_end(klt_ctx *ctx, int token) {
    if (token < 0) return;
    cudaEventRecord(ctx->prof_pending[token].e1, ctx->stream);
}
static void prof_resolve(klt_ctx *ctx) {
    cudaStreamSynchronize(ctx->stream);
    for (auto &pd : ctx->prof_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, pd.e0, pd.e1) == cudaSuccess) ctx->prof[pd.rec].ms += ms;
        ctx->prof_pool.push_back(pd.e0);
        ctx->prof_pool.push_back(pd.e1);
    }
    ctx->prof_pending.clear();
}

extern "C" {

int klt_profile_enable(klt_ctx *ctx, int on) {
    if (!ctx) return KLT_ERR_INVALID;
    prof_resolve(ctx);
    ctx->profiling = on != 0;
    return KLT_OK;
}
int klt_profile_reset(klt_ctx *ctx) {
    if (!ctx) return KLT_ERR_INVALID;
    prof_resolve(ctx);
    ctx->prof.clear();
    return KLT_OK;
}
int klt_profile_count(klt_ctx *ctx) {
    if (!ctx) return KLT_ERR_INVALID;
    prof_resolve(ctx);
    return (int)ctx->prof.size();
}
int klt_profile_get(klt_ctx *ctx, int index, const char **name, double *total_ms, int64_t *launches, double *bytes) {
    if (!ctx || index < 0 || index >= (int)ctx->prof.size()) return KLT_ERR_INVALID;
    const KltProfRec &r = ctx->prof[index];
    if (name) *name = r.name.c_str();
    if (total_ms) *total_ms = r.ms;
    if (launches) *launches = r.count;
    if (bytes) *bytes = r.bytes;
    return KLT_OK;
}


int klt_abi_version(void) { return KLT_B200_ABI_VERSION; }

int klt_ctx_create(int device, void *stream, klt_ctx **out) {
    if (!out) return klt_fail(nullptr, KLT_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return klt_fail(nullptr, KLT_ERR_CUDA, "no CUDA device available (%s); libkltb200 has no CPU fallback",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= count) return klt_fail(nullptr, KLT_ERR_INVALID, "device %d out of range (%d devices)", device, count);
    if ((e = cudaSetDevice(device)) != cudaSuccess) return klt_fail(nullptr, KLT_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return klt_fail(nullptr, KLT_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major < 10)       // the library carries sm_100a code only; fail loudly here instead of at the first launch
        return klt_fail(nullptr, KLT_ERR_UNSUPPORTED, "device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU", device, prop.name, prop.major, prop.minor);
    klt_ctx *ctx = new klt_ctx();
    ctx->device = device;
    ctx->profiling = false;
    ctx->launches = 0;
    ctx->ws = nullptr; ctx->ws_bytes = 0;
    ctx->own_stream = stream == nullptr;
    if (stream) ctx->stream = (cudaStream_t)stream;
    else if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        delete ctx;
        return klt_fail(nullptr, KLT_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    cudaEventCreate(&ctx->ev0);
    cudaEventCreate(&ctx->ev1);
    cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2; i++) cudaEventCreateWithFlags(&ctx->ov_ev[i], cudaEventDisableTiming);
    for (int i = 0; i < 16; i++) cudaEventCreateWithFlags(&ctx->chunk_ev[i], cudaEventDisableTiming);
    for (int i = 0; i < 2; i++) cudaEventCreateWithFlags(&ctx->half_free[i], cudaEventDisableTiming);
    ctx->half_next = 0;
    ctx->frames_dev = nullptr; ctx->frames_bytes = 0;
    ctx->async_flag_dev = nullptr;
    for (int i = 0; i < 16; i++) cudaEventCreateWithFlags(&ctx->marks[i], cudaEventDisableTiming);
    if (cudaMalloc(&ctx->async_flag_dev, 256) == cudaSuccess) cudaMemset(ctx->async_flag_dev, 0, 256);
    ctx->num_sms = prop.multiProcessorCount;
    ctx->select_chunk = 4096;
    if (const char *e2 = getenv("KLT_B200_SELECT_CHUNK")) {
        const int v = atoi(e2);
        if (v >= 32 && v <= 4096 && (v & (v - 1)) == 0) ctx->select_chunk = v;
    }
    *out = ctx;
    return KLT_OK;
}

int klt_ctx_destroy(klt_ctx *ctx) {
    if (!ctx) return KLT_OK;
    cudaSetDevice(ctx->device);
    prof_resolve(ctx);
    for (cudaEvent_t e : ctx->prof_pool) cudaEventDestroy(e);
    if (ctx->ws) cudaFree(ctx->ws);
    if (ctx->frames_dev) cudaFree(ctx->frames_dev);
    cudaStreamDestroy(ctx->copy_stream);
    cudaStreamDestroy(ctx->aux_stream);
    for (int i = 0; i < 2; i++) cudaEventDestroy(ctx->ov_ev[i]);
    for (int i = 0; i < 16; i++) cudaEventDestroy(ctx->chunk_ev[i]);
    for (int i = 0; i < 2; i++) cudaEventDestroy(ctx->half_free[i]);
    if (ctx->async_flag_dev) cudaFree(ctx->async_flag_dev);
    for (int i = 0; i < 16; i++) cudaEventDestroy(ctx->marks[i]);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return KLT_OK;
}

const char *klt_last_error(const klt_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int klt_sync(klt_ctx *ctx) {
    if (!ctx) return KLT_ERR_INVALID;
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->async_flag_dev) {      // the sticky flag of calls that returned without waiting (see klt_track_features)
        int flag = 0;
        KLT_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->async_flag_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (flag) {
            KLT_CUDA(ctx, cudaMemsetAsync(ctx->async_flag_dev, 0, sizeof(int), ctx->stream));
            return klt_fail(ctx, KLT_ERR_ASSERT, "a feature window left the image at a pyramid level in a call that did not wait for its result: the reference raises AssertionError (trackFeaturesUtils.pyx:35)");
        }
    }
    return KLT_OK;
}
void *klt_ctx_stream(klt_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
int64_t klt_launch_count(const klt_ctx *ctx) { return ctx ? ctx->launches : 0; }

int klt_host_alloc(size_t bytes, void **out) {
    if (!out) return KLT_ERR_INVALID;
    return cudaMallocHost(out, bytes) == cudaSuccess ? KLT_OK : KLT_ERR_NOMEM;
}
int klt_host_free(void *p) { return cudaFreeHost(p) == cudaSuccess ? KLT_OK : KLT_ERR_CUDA; }
int klt_device_alloc(klt_ctx *ctx, size_t bytes, void **out) {
    if (!ctx || !out) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return KLT_OK;
}
int klt_device_free(klt_ctx *ctx, void *p) {
    if (!ctx) return KLT_ERR_INVALID;
    KLT_CUDA(ctx, cudaFree(p));
    return KLT_OK;
}
int klt_memcpy(klt_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx || (bytes && (!dst || !src))) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->stream));
    return KLT_OK;
}
int klt_timer_start(klt_ctx *ctx) { if (!ctx) return KLT_ERR_INVALID; KLT_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream)); return KLT_OK; }
int klt_timer_stop(klt_ctx *ctx) { if (!ctx) return KLT_ERR_INVALID; KLT_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream)); return KLT_OK; }
int klt_timer_elapsed_ms(klt_ctx *ctx, float *ms) {
    if (!ctx || !ms) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
    KLT_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return KLT_OK;
}

// ---- operator level ---------------------------------------------------------------------------------------
// Stages host images in the workspace when needed.  Layout: [in][out0][out1].
static int stage_in(klt_ctx *ctx, const float *in, size_t n, size_t slot, size_t nslots, const float **dev) {
    const size_t plane = align_up(n * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, nslots * plane);
    if (rc) return rc;
    float *d = (float *)((char *)ctx->ws + slot * plane);
    KLT_CUDA(ctx, cudaMemcpyAsync(d, in, n * sizeof(float), cudaMemcpyDefault, ctx->stream));
    *dev = d;
    return KLT_OK;
}

int klt_convolve_separable_f32(klt_ctx *ctx, const float *in, int w, int h, const klt_kernel1d *hk,
                               const klt_kernel1d *vk, int precision, float *out) {
    if (!ctx || !in || !out || w <= 0 || h <= 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)w * h, plane = align_up(n * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, 2 * plane);
    if (rc) return rc;
    const float *din = in;
    float *dout = out;
    const bool in_host = !klt_is_device_ptr(in), out_host = !klt_is_device_ptr(out);
    if (in_host && (rc = stage_in(ctx, in, n, 0, 2, &din))) return rc;
    if (out_host) dout = (float *)((char *)ctx->ws + plane);
    if ((rc = klt_launch_conv_sep_f32(ctx, din, w, 0, dout, w, 0, w, h, 1, hk, vk, precision))) return rc;
    if (out_host) {
        KLT_CUDA(ctx, cudaMemcpyAsync(out, dout, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KLT_OK;
}

int klt_smooth_f32(klt_ctx *ctx, const float *in, int w, int h, const klt_kernel1d *gauss, int precision, float *out) {
    return klt_convolve_separable_f32(ctx, in, w, h, gauss, gauss, precision, out);
}

int klt_gradients_f32(klt_ctx *ctx, const float *in, int w, int h, const klt_kernel1d *gauss, const klt_kernel1d *deriv,
                      int precision, float *gradx, float *grady) {
    if (!ctx || !in || !gradx || !grady || w <= 0 || h <= 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)w * h, plane = align_up(n * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, 3 * plane);
    if (rc) return rc;
    const float *din = in;
    const bool in_host = !klt_is_device_ptr(in), out_host = !klt_is_device_ptr(gradx);
    if (out_host != !klt_is_device_ptr(grady)) return klt_fail(ctx, KLT_ERR_INVALID, "gradx and grady must both be host or both be device");
    if (in_host && (rc = stage_in(ctx, in, n, 0, 3, &din))) return rc;
    float *dgx = out_host ? (float *)((char *)ctx->ws + plane) : gradx;
    float *dgy = out_host ? (float *)((char *)ctx->ws + 2 * plane) : grady;
    if ((rc = klt_launch_grad_pair(ctx, din, w, 0, dgx, dgy, w, 0, w, h, 1, gauss, deriv, precision))) return rc;
    if (out_host) {
        KLT_CUDA(ctx, cudaMemcpyAsync(gradx, dgx, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(grady, dgy, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return KLT_OK;
}

// ---- pyramids -----------------------------------------------------------------------------------------------
int klt_pyr_create(klt_ctx *ctx, int w, int h, int n_levels, int subsampling, int batch, klt_pyr **out) {
    if (!ctx || !out || w <= 0 || h <= 0 || batch <= 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (n_levels < 1 || n_levels > KLT_MAX_LEVELS) return klt_fail(ctx, KLT_ERR_INVALID, "n_levels %d out of range 1..%d", n_levels, KLT_MAX_LEVELS);
    if (subsampling != 2 && subsampling != 4 && subsampling != 8 && subsampling != 16 && subsampling != 32)
        return klt_fail(ctx, KLT_ERR_INVALID, "Pyramid's subsampling must be either 2, 4, 8, 16, or 32");   // pyramid.py:17-20
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    klt_pyr *p = new klt_pyr();
    p->hx = new KltPyrHost();
    p->hx->taps_valid = false; p->hx->grad_valid = false; p->hx->grad0_valid = false;
    p->w = w; p->h = h; p->n_levels = n_levels; p->ss = subsampling; p->batch = batch;
    p->precision = KLT_PRECISION_STRICT;
    size_t off = 0;
    int lw = w, lh = h;
    for (int l = 0; l < n_levels; l++) {
        if (lw < 1 || lh < 1) { delete p->hx; delete p; return klt_fail(ctx, KLT_ERR_INVALID, "pyramid level %d is empty", l); }
        p->lv[l].w = lw; p->lv[l].h = lh; p->lv[l].pitch = (lw + 3) & ~3; p->lv[l].off = off;
        off += align_up((size_t)p->lv[l].pitch * lh, 64);    // 256-byte aligned levels
        lw /= subsampling; lh /= subsampling;               // int(n / ss), pyramid.py:63-64
    }
    p->plane_floats = off;
    const size_t bytes = 3 * (size_t)batch * off * sizeof(float);
    cudaError_t e = cudaMalloc(&p->base, bytes);
    if (e != cudaSuccess) { delete p->hx; delete p; return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for pyramid failed: %s", bytes, cudaGetErrorString(e)); }
    *out = p;
    return KLT_OK;
}

int klt_pyr_destroy(klt_ctx *ctx, klt_pyr *pyr) {
    if (!pyr) return KLT_OK;
    if (ctx) cudaStreamSynchronize(ctx->stream);
    cudaFree(pyr->base);
    delete pyr->hx;
    delete pyr;
    return KLT_OK;
}

int klt_pyr_dims(const klt_pyr *pyr, int level, int *w, int *h, int *pitch) {
    if (!pyr || level < 0 || level >= pyr->n_levels) return KLT_ERR_INVALID;
    if (w) *w = pyr->lv[level].w;
    if (h) *h = pyr->lv[level].h;
    if (pitch) *pitch = pyr->lv[level].pitch;
    return KLT_OK;
}
size_t klt_pyr_bytes(const klt_pyr *pyr) { return pyr ? 3 * (size_t)pyr->batch * pyr->plane_floats * sizeof(float) : 0; }

static int check_taps(klt_ctx *ctx, const klt_taps *t) {
    if (!t) return klt_fail(ctx, KLT_ERR_INVALID, "taps is NULL");
    return KLT_OK;
}

// Host state of a build with the caller's KLT_PRECISION_*: the arithmetic (FAST_WINDOWED computes in FAST), the kernels,
// and which gradient planes exist (none in an image-only FAST_WINDOWED build).  Builds, their lazy gradient passes and
// graph replays of a build all keep it through this one function; it enqueues nothing.
void klt_pyr_note_build(klt_pyr *p, const klt_taps *taps, int precision) {
    const bool windowed = precision == KLT_PRECISION_FAST_WINDOWED;
    p->precision = windowed ? KLT_PRECISION_FAST : precision;
    p->hx->taps = *taps; p->hx->taps_valid = true;
    p->hx->grad_valid = p->hx->grad0_valid = !windowed;
}

// build_levels: levels [from, n_levels) of images [first, first + count), each decimated from the level below;
// build_grads: the gradient pairs of levels [from, to).  Both run with the arithmetic and kernels of the last build: FAST
// arithmetic takes the warp-streaming kernel where it covers the level, everything else the generic tiled kernel.
static int build_levels(klt_ctx *ctx, klt_pyr *p, int from, int first, int count) {
    const klt_taps *taps = &p->hx->taps;
    const size_t stride = p->plane_floats;
    for (int l = from; l < p->n_levels; l++) {
        const LevelDesc &a = p->lv[l - 1], &b = p->lv[l];
        int rc = p->precision == KLT_PRECISION_FAST ? klt_stream_down2(ctx, p, l, taps, first, count) : 0;
        if (rc < 0) return rc;
        if (rc == 0 && (rc = klt_launch_pyr_down(ctx, p->level(0, first, l - 1), a.pitch, stride, a.w, a.h, p->level(0, first, l),
                                                 b.pitch, stride, b.w, b.h, p->ss, count, &taps->pyramid, p->precision))) return rc;
    }
    return KLT_OK;
}

static int build_grads(klt_ctx *ctx, klt_pyr *p, int from, int to, int first, int count) {
    const klt_taps *taps = &p->hx->taps;
    const size_t stride = p->plane_floats;
    for (int l = from; l < to; l++) {
        const LevelDesc &a = p->lv[l];
        int rc = p->precision == KLT_PRECISION_FAST ? klt_stream_grad(ctx, p, l, taps, first, count) : 0;
        if (rc < 0) return rc;
        if (rc == 0 && (rc = klt_launch_grad_pair(ctx, p->level(0, first, l), a.pitch, stride, p->level(1, first, l),
                                                  p->level(2, first, l), a.pitch, stride, a.w, a.h, count, &taps->grad_gauss,
                                                  &taps->grad_deriv, p->precision))) return rc;
    }
    return KLT_OK;
}

// gradient planes of levels [0, levels) of a built pyramid (an image-only build leaves them to its first reader; selection
// on a tracking pyramid, KLTReplaceLostFeatures in sequentialMode, reads level 0 only).  Only klt_pyr_ensure_gradients
// sets grad_valid: it sends tracking to the plane-based kernels, so a selection must leave an image-only pyramid on the
// windowed tracker even when level 0 is its only level.
int klt_ensure_gradients(klt_ctx *ctx, klt_pyr *p, int levels) {
    if (!p->hx || p->hx->grad_valid) return KLT_OK;
    if (!p->hx->taps_valid) return klt_fail(ctx, KLT_ERR_INVALID, "pyramid has not been built");
    int rc = build_grads(ctx, p, p->hx->grad0_valid ? 1 : 0, levels, 0, p->batch);
    if (rc) return rc;
    p->hx->grad0_valid = true;
    return KLT_OK;
}

int klt_pyr_ensure_gradients(klt_ctx *ctx, klt_pyr *p) {
    if (!ctx || !p) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = klt_ensure_gradients(ctx, p, p->n_levels);
    if (rc == KLT_OK && p->hx) p->hx->grad_valid = true;
    return rc;
}

// device frames -> pyramids for images [first, first+count); dframes points at image `first`.  level0_done (may be null) is
// recorded right after the kernel that writes level 0, for a caller that forks work reading only that level.
int klt_build_u8_device(klt_ctx *ctx, klt_pyr *p, const uint8_t *dframes, size_t pitch, size_t frame_stride,
                        const klt_taps *taps, int precision, int first, int count, cudaEvent_t level0_done) {
    klt_pyr_note_build(p, taps, precision);
    const bool windowed = precision == KLT_PRECISION_FAST_WINDOWED;
    int rc = 0, levels_done = 1;       // levels the level-0 step writes
    bool grad0_done = false;           // ... and whether it also writes level 0's gradient pair
    if (windowed) {
        // u8 -> smoothed image + level 1 in one pass, else u8 -> smoothed image only
        // a caller that forks after level 0 (klt_sequence's eigenvalue pass) forks after the fused kernel instead: measured
        // 0.273 against 0.276 ms per step of 8 sequences with the two-kernel build, one launch fewer
        if ((rc = klt_stream_level01(ctx, dframes, pitch, frame_stride, p, taps, first, count)) == 1) levels_done = 2;
        else if (rc == 0) rc = klt_stream_smooth0(ctx, dframes, pitch, frame_stride, p, taps, first, count);
    } else if (precision == KLT_PRECISION_FAST) {
        // fused u8 -> smoothed image + gradient pair of level 0 (one read of the frame, three writes)
        grad0_done = (rc = klt_stream_level0(ctx, dframes, pitch, frame_stride, p, taps, first, count)) == 1;
    }
    if (rc < 0) return rc;
    // img.convert("F") + KLTComputeSmoothedImage (trackFeatures.py:165-166): one kernel, u8 in, f32 out
    if (rc == 0 && (rc = klt_launch_conv_sep_u8(ctx, dframes, pitch, frame_stride, p->level(0, first, 0), p->lv[0].pitch,
                                                p->plane_floats, p->w, p->h, count, &taps->smooth, &taps->smooth, p->precision))) return rc;
    if (level0_done) KLT_CUDA(ctx, cudaEventRecord(level0_done, ctx->stream));
    if ((rc = build_levels(ctx, p, levels_done, first, count))) return rc;
    return windowed ? KLT_OK : build_grads(ctx, p, grad0_done ? 1 : 0, p->n_levels, first, count);
}

int klt_pyr_build_u8(klt_ctx *ctx, klt_pyr *p, const uint8_t *frames, size_t pitch, size_t frame_stride,
                     const klt_taps *taps, int precision) {
    if (!ctx || !p || !frames) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    int rc;
    if ((rc = check_taps(ctx, taps))) return rc;
    if (pitch < (size_t)p->w) return klt_fail(ctx, KLT_ERR_INVALID, "pitch %zu smaller than width %d", pitch, p->w);
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint8_t *dframes = frames;
    if (!klt_is_device_ptr(frames)) {
        const size_t bytes = (size_t)(p->batch - 1) * frame_stride + (size_t)(p->h - 1) * pitch + p->w;
        if ((rc = klt_ws_reserve(ctx, bytes))) return rc;
        KLT_CUDA(ctx, cudaMemcpyAsync(ctx->ws, frames, bytes, cudaMemcpyHostToDevice, ctx->stream));
        dframes = (const uint8_t *)ctx->ws;
    }
    return klt_build_u8_device(ctx, p, dframes, pitch, frame_stride, taps, precision, 0, p->batch, nullptr);
}

int klt_pyr_build_f32(klt_ctx *ctx, klt_pyr *p, const float *images, size_t pitch, size_t frame_stride,
                      const klt_taps *taps, int precision, int already_smoothed) {
    if (!ctx || !p || !images) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    int rc;
    if ((rc = check_taps(ctx, taps))) return rc;
    if (pitch < (size_t)p->w) return klt_fail(ctx, KLT_ERR_INVALID, "pitch %zu smaller than width %d", pitch, p->w);
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    klt_pyr_note_build(p, taps, precision);
    if (already_smoothed) {
        for (int b = 0; b < p->batch; b++)
            KLT_CUDA(ctx, cudaMemcpy2DAsync(p->level(0, b, 0), p->lv[0].pitch * sizeof(float), images + (size_t)b * frame_stride,
                                            pitch * sizeof(float), p->w * sizeof(float), p->h, cudaMemcpyDefault, ctx->stream));
    } else {
        const float *dimg = images;
        if (!klt_is_device_ptr(images)) {
            const size_t elems = (size_t)(p->batch - 1) * frame_stride + (size_t)(p->h - 1) * pitch + p->w;
            if ((rc = klt_ws_reserve(ctx, elems * sizeof(float)))) return rc;
            KLT_CUDA(ctx, cudaMemcpyAsync(ctx->ws, images, elems * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
            dimg = (const float *)ctx->ws;
        }
        if ((rc = klt_launch_conv_sep_f32(ctx, dimg, pitch, frame_stride, p->level(0, 0, 0), p->lv[0].pitch, p->plane_floats, p->w,
                                          p->h, p->batch, &taps->smooth, &taps->smooth, p->precision))) return rc;
    }
    if ((rc = build_levels(ctx, p, 1, 0, p->batch))) return rc;
    return precision == KLT_PRECISION_FAST_WINDOWED ? KLT_OK : build_grads(ctx, p, 0, p->n_levels, 0, p->batch);
}

int klt_pyr_download(klt_ctx *ctx, const klt_pyr *p, int image, int which, int level, float *out) {
    if (!ctx || !p || !out || image < 0 || image >= p->batch || which < 0 || which > 2 || level < 0 || level >= p->n_levels)
        return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (which > 0) {
        int rc = klt_pyr_ensure_gradients(ctx, const_cast<klt_pyr *>(p));
        if (rc) return rc;
    }
    const LevelDesc &a = p->lv[level];
    KLT_CUDA(ctx, cudaMemcpy2DAsync(out, a.w * sizeof(float), p->level(which, image, level), a.pitch * sizeof(float),
                                    a.w * sizeof(float), a.h, cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_pyr_level_ptr(const klt_pyr *p, int image, int which, int level, const float **ptr) {
    if (!p || !ptr || image < 0 || image >= p->batch || which < 0 || which > 2 || level < 0 || level >= p->n_levels) return KLT_ERR_INVALID;
    if (which > 0 && !klt_pyr_has_gradients(p)) return KLT_ERR_UNSUPPORTED;   // image-only pyramid: download builds them
    *ptr = p->level(which, image, level);
    return KLT_OK;
}

// ---- selection ----------------------------------------------------------------------------------------------
int klt_scan_good_features(klt_ctx *ctx, const float *gradx, const float *grady, int w, int h, int borderx, int bordery,
                           int window_hw, int window_hh, int n_skipped_pixels, float *val) {
    if (!ctx || !gradx || !grady || !val || w <= 0 || h <= 0 || n_skipped_pixels < 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (borderx < window_hw + 1 || bordery < window_hh + 1)
        return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "border (%d,%d) smaller than window half-size + 1: the reference reads out of bounds here", borderx, bordery);
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const int step = n_skipped_pixels + 1;
    int nx = 0, ny = 0;
    if (w - borderx > borderx) nx = (w - 2 * borderx + step - 1) / step;
    if (h - bordery > bordery) ny = (h - 2 * bordery + step - 1) / step;
    const size_t n = (size_t)w * h, plane = align_up(n * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, 6 * plane);
    if (rc) return rc;
    char *wsp = (char *)ctx->ws;
    float *dval = (float *)(wsp + 3 * plane);
    const float *dgx = gradx, *dgy = grady;
    if (!klt_is_device_ptr(gradx)) {
        float *d = (float *)(wsp + 4 * plane);
        KLT_CUDA(ctx, cudaMemcpyAsync(d, gradx, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        dgx = d;
    }
    if (!klt_is_device_ptr(grady)) {
        float *d = (float *)(wsp + 5 * plane);
        KLT_CUDA(ctx, cudaMemcpyAsync(d, grady, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        dgy = d;
    }
    if ((rc = klt_launch_scan(ctx, dgx, dgy, w, w, h, borderx, bordery, window_hw, window_hh, n_skipped_pixels, dval, nx, ny))) return rc;
    if (nx > 0 && ny > 0)
        KLT_CUDA(ctx, cudaMemcpyAsync(val, dval, (size_t)nx * ny * sizeof(float), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_select_good_features(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr, int image, const float *gradx,
                             const float *grady, int w, int h, int n_features, int replace, double *x, double *y,
                             int32_t *val, int64_t *n_consumed) {
    if (!ctx || !params || !x || !y || !val || n_features < 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    if (pyr) {
        if (image < 0 || image >= pyr->batch) return klt_fail(ctx, KLT_ERR_INVALID, "image index out of range");
        if (pyr->batch == 1) return klt_select_batch(ctx, params, KLT_SELECT_STRICT, const_cast<klt_pyr *>(pyr), nullptr, nullptr, 0, 0, pyr->w, pyr->h, 1, n_features, replace, x, y, val, n_consumed);
        int rc = klt_ensure_gradients(ctx, const_cast<klt_pyr *>(pyr), 1);      // image-only pyramids: build level 0's planes now
        if (rc) return rc;
        return klt_select_batch(ctx, params, KLT_SELECT_STRICT, nullptr, pyr->level(1, image, 0), pyr->level(2, image, 0), 0, pyr->lv[0].pitch, pyr->w, pyr->h,
                                1, n_features, replace, x, y, val, n_consumed);
    }
    if (!gradx || !grady || w <= 0 || h <= 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (!klt_is_device_ptr(gradx) || !klt_is_device_ptr(grady))
        return klt_fail(ctx, KLT_ERR_INVALID, "explicit gradient images must be device pointers (use a pyramid or klt_device_alloc)");
    return klt_select_batch(ctx, params, KLT_SELECT_STRICT, nullptr, gradx, grady, 0, w, w, h, 1, n_features, replace, x, y, val, n_consumed);
}

int klt_select_good_features_batch(klt_ctx *ctx, const klt_params *params, klt_pyr *pyr, int n_features, int replace,
                                   int select_mode, double *x, double *y, int32_t *val) {
    if (!ctx || !params || !pyr || !x || !y || !val || n_features < 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (select_mode != KLT_SELECT_STRICT && select_mode != KLT_SELECT_FAST) return klt_fail(ctx, KLT_ERR_INVALID, "select_mode must be KLT_SELECT_STRICT or KLT_SELECT_FAST");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    return klt_select_batch(ctx, params, select_mode, pyr, nullptr, nullptr, 0, 0, pyr->w, pyr->h, pyr->batch, n_features, replace, x, y, val, nullptr);
}

int klt_eigen_map_batch(klt_ctx *ctx, const klt_params *params, klt_pyr *pyr, int select_mode, float *val, int *nx, int *ny) {
    if (!ctx || !params || !pyr) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    return klt_eigen_maps(ctx, params, select_mode, pyr, val, nx, ny);
}

// ---- tracking -----------------------------------------------------------------------------------------------
static int check_track_args(klt_ctx *ctx, const klt_params *p, const klt_pyr *p1, const klt_pyr *p2) {
    if (p1->w != p2->w || p1->h != p2->h || p1->n_levels != p2->n_levels || p1->ss != p2->ss || p1->batch != p2->batch)
        return klt_fail(ctx, KLT_ERR_INVALID, "pyramids differ in geometry");
    if (p->n_levels != p1->n_levels || p->subsampling != p1->ss)
        return klt_fail(ctx, KLT_ERR_INVALID, "params (levels %d, subsampling %d) do not match the pyramids (%d, %d)", p->n_levels, p->subsampling, p1->n_levels, p1->ss);
    if (p->window_width < 3 || p->window_height < 3 || !(p->window_width & 1) || !(p->window_height & 1))
        return klt_fail(ctx, KLT_ERR_INVALID, "window must be odd and >= 3");
    if (p->window_width != p->window_height)
        return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "non-square tracking windows corrupt memory in the reference (quirk Q10); refused");
    return KLT_OK;
}

// max_fb_error > 0: the forward-backward check after the forward track (fb_error may then be null, host or device)
static int track_impl(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2, int n_per_image,
                      double *x, double *y, int32_t *val, klt_affine *aff, int64_t *n_iterations, bool async = false,
                      float max_fb_error = 0.f, float *fb_error = nullptr) {
    if (!ctx || !params || !pyr1 || !pyr2 || !x || !y || !val || n_per_image < 0) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    const bool fb = max_fb_error > 0.f;
    int rc;
    if ((rc = check_track_args(ctx, params, pyr1, pyr2))) return rc;
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    if (aff && params->lighting_insensitive)
        return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "lighting_insensitive together with the affine consistency check is not supported");
    if (aff || params->lighting_insensitive || !klt_windowed_supported(params, pyr1, pyr2)) {
        // the affine tracker and the configurations the windowed tracker does not cover read gradient planes
        if ((rc = klt_pyr_ensure_gradients(ctx, const_cast<klt_pyr *>(pyr1)))) return rc;
        if ((rc = klt_pyr_ensure_gradients(ctx, const_cast<klt_pyr *>(pyr2)))) return rc;
    }
    const size_t total = (size_t)n_per_image * pyr1->batch;
    if (aff) {
        if ((size_t)aff->n != total) return klt_fail(ctx, KLT_ERR_INVALID, "affine state has %d slots, %zu features given", aff->n, total);
        if (params->affine_consistency_check < 0 || params->affine_consistency_check > 2) return klt_fail(ctx, KLT_ERR_INVALID, "affine_consistency_check must be 0, 1 or 2");
        if (params->affine_window_width != aff->aw || params->affine_window_height != aff->ah) return klt_fail(ctx, KLT_ERR_INVALID, "affine window differs from the affine state's");
    }
    const bool host = !klt_is_device_ptr(x);
    if (host != !klt_is_device_ptr(y) || host != !klt_is_device_ptr(val)) return klt_fail(ctx, KLT_ERR_INVALID, "x, y, val must all be host or all be device");
    const size_t fbytes = align_up(total * sizeof(double), 256);
    // [iterations, assert word, backward assert word][x, y, val staging][affine: x_in, y_in, val_in | fb: x0, y0, vb, xb, yb, fb_error staging]
    if ((rc = klt_ws_reserve(ctx, (fb ? 9 : 6) * fbytes + 256))) return rc;
    char *wsp = (char *)ctx->ws;
    unsigned long long *iters = (unsigned long long *)wsp;
    // calls that return without reading the flag back (asynchronous, or device arrays without n_iterations) raise the context's
    // sticky flag instead: klt_sync / klt_async_result report it
    const bool deferred = async || (!host && !n_iterations);
    if (deferred && !ctx->async_flag_dev) return klt_fail(ctx, KLT_ERR_NOMEM, "the context has no status word");
    int *aflag = deferred ? ctx->async_flag_dev : (int *)(wsp + 8);
    double *dx = x, *dy = y;
    int32_t *dval = val;
    KLT_CUDA(ctx, cudaMemsetAsync(wsp, 0, 16, ctx->stream));
    if (host) {
        dx = (double *)(wsp + 256); dy = (double *)(wsp + 256 + fbytes); dval = (int32_t *)(wsp + 256 + 2 * fbytes);
        KLT_CUDA(ctx, cudaMemcpyAsync(dx, x, total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(dy, y, total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(dval, val, total * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    double *x_in = nullptr, *y_in = nullptr;
    int32_t *val_in = nullptr;
    if (aff) {   // the affine block needs the pre-track positions (xloc, yloc) and which features were live
        x_in = (double *)(wsp + 256 + 3 * fbytes); y_in = (double *)(wsp + 256 + 4 * fbytes); val_in = (int32_t *)(wsp + 256 + 5 * fbytes);
        KLT_CUDA(ctx, cudaMemcpyAsync(x_in, dx, total * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(y_in, dy, total * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(val_in, dval, total * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    const bool fb_host = fb && fb_error && !klt_is_device_ptr(fb_error);
    float *dfb = fb_host ? (float *)(wsp + 256 + 8 * fbytes) : fb_error;
    if (fb) {
        const FbArrays fa{(double *)(wsp + 256 + 3 * fbytes), (double *)(wsp + 256 + 4 * fbytes), (double *)(wsp + 256 + 6 * fbytes),
                          (double *)(wsp + 256 + 7 * fbytes), (int32_t *)(wsp + 256 + 5 * fbytes), (int *)(wsp + 12)};
        if ((rc = klt_launch_track_fb(ctx, params, pyr1, pyr2, n_per_image, max_fb_error, dx, dy, dval, fa, dfb, iters, aflag))) return rc;
    } else if ((rc = klt_launch_track(ctx, params, pyr1, pyr2, n_per_image, dx, dy, dval, iters, aflag))) return rc;
    if (aff && (rc = klt_launch_affine(ctx, params, pyr1, pyr2, n_per_image, x_in, y_in, val_in, dx, dy, dval, aff, aflag))) return rc;
    if (host) {
        KLT_CUDA(ctx, cudaMemcpyAsync(x, dx, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(y, dy, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(val, dval, total * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (fb_host) KLT_CUDA(ctx, cudaMemcpyAsync(fb_error, dfb, total * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (async) return KLT_OK;                    // results land when the stream gets there: klt_sync / klt_async_result
    if (host || n_iterations) {
        unsigned long long res[2] = {0, 0};
        KLT_CUDA(ctx, cudaMemcpyAsync(res, wsp, 16, cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (n_iterations) *n_iterations = (int64_t)res[0];
        if ((int)(res[1] & 0xffffffffull))
            return klt_fail(ctx, KLT_ERR_ASSERT, "a feature window leaves the image at a pyramid level: the reference raises AssertionError (trackFeaturesUtils.pyx:35)");
    }
    return KLT_OK;
}

int klt_track_features(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2, int n_per_image,
                       double *x, double *y, int32_t *val, int64_t *n_iterations) {
    return track_impl(ctx, params, pyr1, pyr2, n_per_image, x, y, val, nullptr, n_iterations);
}

int klt_track_features_fb(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2, int n_per_image,
                          float max_fb_error, double *x, double *y, int32_t *val, float *fb_error, int64_t *n_iterations) {
    if (!(max_fb_error > 0.f && max_fb_error <= FLT_MAX))
        return klt_fail(ctx, KLT_ERR_INVALID, "max_fb_error must be finite and > 0 (got %g)", (double)max_fb_error);
    return track_impl(ctx, params, pyr1, pyr2, n_per_image, x, y, val, nullptr, n_iterations, false, max_fb_error, fb_error);
}

int klt_track_features_affine(klt_ctx *ctx, const klt_params *params, const klt_pyr *pyr1, const klt_pyr *pyr2, int n_per_image,
                              double *x, double *y, int32_t *val, klt_affine *a, int64_t *n_iterations) {
    if (!a) return klt_fail(ctx, KLT_ERR_INVALID, "affine state is NULL");
    return track_impl(ctx, params, pyr1, pyr2, n_per_image, x, y, val, a, n_iterations);
}

int klt_affine_create(klt_ctx *ctx, int n, int aw, int ah, klt_affine **out) {
    if (!ctx || !out || n < 0 || aw < 3 || ah < 3 || !(aw & 1) || !(ah & 1)) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    klt_affine *a = new klt_affine();
    a->n = n; a->aw = aw; a->ah = ah;
    const size_t tn = (size_t)(aw + 2) * (ah + 2);
    const size_t b_has = align_up((size_t)n * 4 + 4, 256), b_f = align_up((size_t)n * 4 + 4, 256), b_A = align_up((size_t)n * 16 + 16, 256);
    const size_t bytes = b_has + 2 * b_f + b_A + (size_t)n * 3 * tn * 4 + 256;
    cudaError_t e = cudaMalloc(&a->block, bytes);
    if (e != cudaSuccess) { delete a; return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for affine state failed: %s", bytes, cudaGetErrorString(e)); }
    char *b = (char *)a->block;
    a->has = (int *)b; b += b_has;
    a->aff_x = (float *)b; b += b_f;
    a->aff_y = (float *)b; b += b_f;
    a->A = (float *)b; b += b_A;
    a->tmpl = (float *)b;
    int rc = klt_launch_affine_reset(ctx, a, nullptr);
    if (rc) { cudaFree(a->block); delete a; return rc; }
    *out = a;
    return KLT_OK;
}

int klt_affine_destroy(klt_ctx *ctx, klt_affine *a) {
    if (!a) return KLT_OK;
    if (ctx) cudaStreamSynchronize(ctx->stream);
    cudaFree(a->block);
    delete a;
    return KLT_OK;
}

int klt_affine_reset(klt_ctx *ctx, klt_affine *a, const int32_t *mask) {
    if (!ctx || !a) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!mask) return klt_launch_affine_reset(ctx, a, nullptr);
    int rc = klt_ws_reserve(ctx, (size_t)a->n * 4 + 256);
    if (rc) return rc;
    KLT_CUDA(ctx, cudaMemcpyAsync(ctx->ws, mask, (size_t)a->n * 4, cudaMemcpyDefault, ctx->stream));
    return klt_launch_affine_reset(ctx, a, (const int *)ctx->ws);
}

int klt_affine_download(klt_ctx *ctx, const klt_affine *a, int32_t *has_template, float *aff_x, float *aff_y, float *A) {
    if (!ctx || !a) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    const size_t n = (size_t)a->n;
    if (has_template) KLT_CUDA(ctx, cudaMemcpyAsync(has_template, a->has, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (aff_x) KLT_CUDA(ctx, cudaMemcpyAsync(aff_x, a->aff_x, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (aff_y) KLT_CUDA(ctx, cudaMemcpyAsync(aff_y, a->aff_y, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (A) KLT_CUDA(ctx, cudaMemcpyAsync(A, a->A, n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_affine_download_template(klt_ctx *ctx, const klt_affine *a, int slot, float *out) {
    if (!ctx || !a || !out || slot < 0 || slot >= a->n) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    const size_t tn = (size_t)(a->aw + 2) * (a->ah + 2);
    KLT_CUDA(ctx, cudaMemcpyAsync(out, a->tmpl + (size_t)slot * 3 * tn, 3 * tn * 4, cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_extract_patch(klt_ctx *ctx, const float *img, int w, int h, float x, float y, int height, int width, float *out) {
    if (!ctx || !img || !out || w <= 0 || h <= 0 || width < 1 || height < 1) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)w * h, plane = align_up(n * sizeof(float), 256), pbytes = align_up((size_t)width * height * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, plane + pbytes + 256);
    if (rc) return rc;
    char *wsp = (char *)ctx->ws;
    const float *dimg = img;
    if (!klt_is_device_ptr(img)) {
        KLT_CUDA(ctx, cudaMemcpyAsync(wsp, img, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        dimg = (const float *)wsp;
    }
    float *dout = (float *)(wsp + plane);
    int *dok = (int *)(wsp + plane + pbytes);
    if ((rc = klt_launch_extract_patch(ctx, dimg, w, w, h, x, y, height, width, dout, dok))) return rc;
    int ok = 0;
    KLT_CUDA(ctx, cudaMemcpyAsync(out, dout, (size_t)width * height * sizeof(float), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(&ok, dok, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!ok) return klt_fail(ctx, KLT_ERR_ASSERT, "patch out of bounds (trackFeaturesUtils.pyx:35)");
    return KLT_OK;
}

// ---- operator-level entry points of the reference's Cython modules --------------------------------------------------
static int stage_image(klt_ctx *ctx, const float *img, size_t n, char *slot, const float **dev) {
    *dev = img;
    if (!klt_is_device_ptr(img)) {
        KLT_CUDA(ctx, cudaMemcpyAsync(slot, img, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        *dev = (const float *)slot;
    }
    return KLT_OK;
}

int klt_track_iterate(klt_ctx *ctx, const klt_params *params, float x2, float y2, const float *gx_patch, const float *gy_patch,
                      const float *img_patch, const float *img2, const float *gradx2, const float *grady2, int w, int h,
                      float *x2_out, float *y2_out, int32_t *status, int32_t *iterations) {
    if (!ctx || !params || !gx_patch || !gy_patch || !img_patch || !img2 || !gradx2 || !grady2 || w <= 0 || h <= 0)
        return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (params->lighting_insensitive) return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "lighting_insensitive: Not implemented (trackFeaturesUtils.pyx:435)");
    if (params->window_width != params->window_height) return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "non-square windows are refused (quirk Q10)");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)w * h, plane = align_up(n * sizeof(float), 256);
    const size_t pn = (size_t)params->window_width * params->window_height, pbytes = align_up(3 * pn * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, 3 * plane + pbytes + 256);
    if (rc) return rc;
    char *wsp = (char *)ctx->ws;
    const float *d2, *dgx, *dgy;
    if ((rc = stage_image(ctx, img2, n, wsp, &d2))) return rc;
    if ((rc = stage_image(ctx, gradx2, n, wsp + plane, &dgx))) return rc;
    if ((rc = stage_image(ctx, grady2, n, wsp + 2 * plane, &dgy))) return rc;
    float *tp = (float *)(wsp + 3 * plane), *dout = (float *)(wsp + 3 * plane + pbytes);
    KLT_CUDA(ctx, cudaMemcpyAsync(tp, img_patch, pn * sizeof(float), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(tp + pn, gx_patch, pn * sizeof(float), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(tp + 2 * pn, gy_patch, pn * sizeof(float), cudaMemcpyDefault, ctx->stream));
    if ((rc = klt_launch_iterate(ctx, params, tp, d2, dgx, dgy, w, h, x2, y2, dout))) return rc;
    float res[4];
    KLT_CUDA(ctx, cudaMemcpyAsync(res, dout, sizeof(res), cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (x2_out) *x2_out = res[0];
    if (y2_out) *y2_out = res[1];
    if (status) *status = (int32_t)res[2];
    if (iterations) *iterations = (int32_t)res[3];
    return KLT_OK;
}

int klt_patch_combine(klt_ctx *ctx, const float *patch1, const float *img2, int w, int h, float x2, float y2, int height,
                      int width, int mode, float *out) {
    if (!ctx || !patch1 || !img2 || !out || w <= 0 || h <= 0 || width < 1 || height < 1 || mode < 0 || mode > 1)
        return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)w * h, plane = align_up(n * sizeof(float), 256), pn = (size_t)width * height, pbytes = align_up(pn * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, plane + 2 * pbytes + 256);
    if (rc) return rc;
    char *wsp = (char *)ctx->ws;
    const float *dimg;
    if ((rc = stage_image(ctx, img2, n, wsp, &dimg))) return rc;
    float *dp1 = (float *)(wsp + plane), *dout = (float *)(wsp + plane + pbytes);
    int *dok = (int *)(wsp + plane + 2 * pbytes);
    KLT_CUDA(ctx, cudaMemcpyAsync(dp1, patch1, pn * sizeof(float), cudaMemcpyDefault, ctx->stream));
    if ((rc = klt_launch_patch_combine(ctx, dp1, dimg, w, h, x2, y2, height, width, mode, dout, dok))) return rc;
    int ok = 0;
    KLT_CUDA(ctx, cudaMemcpyAsync(out, dout, pn * sizeof(float), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(&ok, dok, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!ok) return klt_fail(ctx, KLT_ERR_ASSERT, "patch out of bounds (trackFeaturesUtils.pyx:35)");
    return KLT_OK;
}

int klt_enforce_min_distance(klt_ctx *ctx, int n_points, const float *pval, const int32_t *px, const int32_t *py, int ncols,
                             int nrows, int mindist, double min_eigenvalue, int overwrite_all, int n_features, double *x,
                             double *y, int32_t *val) {
    if (!ctx || n_points < 0 || (n_points && (!pval || !px || !py)) || !x || !y || !val || n_features < 0)
        return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!(min_eigenvalue >= 1.0)) min_eigenvalue = 1.0;               // selectGoodFeatures.py:53
    std::vector<unsigned long long> keys;
    keys.reserve((size_t)n_points);
    for (int i = 0; i < n_points; i++) {
        if (px[i] < 0 || px[i] >= ncols || py[i] < 0 || py[i] >= nrows)
            return klt_fail(ctx, KLT_ERR_ASSERT, "candidate %d out of bounds (selectGoodFeatures.py:104-107)", i);
        if (!((double)pval[i] >= min_eigenvalue)) continue;          // can never be accepted (:116, compared as numbers); skipping keeps the walk order
        unsigned int bits;
        memcpy(&bits, &pval[i], 4);
        keys.push_back(~(((unsigned long long)bits << 26) | ((unsigned long long)px[i] << 13) | (unsigned long long)py[i]));
    }
    return klt_greedy_presorted(ctx, keys.data(), (unsigned int)keys.size(), ncols, nrows, mindist, n_features, overwrite_all ? 1 : 0,
                                x, y, val);
}

static int track_pairs_impl(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int precision, klt_pyr *pyr1,
                            klt_pyr *pyr2, const uint8_t *frames1, const uint8_t *frames2, size_t pitch, size_t frame_stride,
                            int n_per_image, double *x, double *y, int32_t *val, bool async) {
    if (!ctx || !params || !taps || !pyr1 || !pyr2 || !frames1 || !frames2) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    int rc;
    const bool host1 = !klt_is_device_ptr(frames1), host2 = !klt_is_device_ptr(frames2);
    if (!host1 && !host2) {
        if (!ctx->profiling && pyr1 != pyr2) {
            // the two (independent) pyramid builds on two streams: the CTAs of one fill the SM slots the other's last wave
            // leaves idle (0.774 -> 0.733 ms per 64 pairs at 1080p).  Profiling brackets every launch with events on the
            // context's stream, and one pyramid cannot be built twice at once, so those two cases build serially below.
            cudaStream_t main = ctx->stream;
            KLT_CUDA(ctx, cudaEventRecord(ctx->ov_ev[0], main));
            KLT_CUDA(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ov_ev[0], 0));
            if ((rc = klt_pyr_build_u8(ctx, pyr1, frames1, pitch, frame_stride, taps, precision))) return rc;
            ctx->stream = ctx->aux_stream;
            rc = klt_pyr_build_u8(ctx, pyr2, frames2, pitch, frame_stride, taps, precision);
            ctx->stream = main;
            if (rc) return rc;
            KLT_CUDA(ctx, cudaEventRecord(ctx->ov_ev[1], ctx->aux_stream));
            KLT_CUDA(ctx, cudaStreamWaitEvent(main, ctx->ov_ev[1], 0));
            return track_impl(ctx, params, pyr1, pyr2, n_per_image, x, y, val, nullptr, nullptr, async);
        }
        if ((rc = klt_pyr_build_u8(ctx, pyr1, frames1, pitch, frame_stride, taps, precision))) return rc;
        if ((rc = klt_pyr_build_u8(ctx, pyr2, frames2, pitch, frame_stride, taps, precision))) return rc;
        return track_impl(ctx, params, pyr1, pyr2, n_per_image, x, y, val, nullptr, nullptr, async);
    }
    if (host1 != host2) return klt_fail(ctx, KLT_ERR_INVALID, "frames1 and frames2 must both be host or both be device");
    if (pyr1->batch != pyr2->batch || pyr1->w != pyr2->w || pyr1->h != pyr2->h) return klt_fail(ctx, KLT_ERR_INVALID, "pyramids differ in geometry");
    if (pitch < (size_t)pyr1->w) return klt_fail(ctx, KLT_ERR_INVALID, "pitch smaller than width");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    // Host frames: the batch is cut into chunks; the H2D copy of chunk k+1 (copy stream) overlaps the pyramid builds of
    // chunk k (compute stream), and the two staging halves alternate between calls, so the upload of the NEXT call overlaps
    // the tracking kernels of this one when the caller does not wait in between (klt_track_pairs_u8_async, or a second
    // context on another thread).  PCIe, not the kernels, bounds this path.
    const int B = pyr1->batch;
    const size_t one = (size_t)(pyr1->h - 1) * pitch + pyr1->w;                 // bytes actually read of one frame
    const size_t per_set = (size_t)(B - 1) * frame_stride + one;
    const size_t set_stride = (per_set + 255) / 256 * 256;
    if (2 * set_stride > ctx->frames_bytes) {
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
        if (ctx->frames_dev) { KLT_CUDA(ctx, cudaFree(ctx->frames_dev)); ctx->frames_dev = nullptr; ctx->frames_bytes = 0; }
        cudaError_t e = cudaMalloc(&ctx->frames_dev, 4 * set_stride);
        if (e != cudaSuccess) return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for frame staging failed: %s", 4 * set_stride, cudaGetErrorString(e));
        ctx->frames_bytes = 2 * set_stride;
    }
    const int half = ctx->half_next;
    ctx->half_next ^= 1;
    uint8_t *d1 = (uint8_t *)ctx->frames_dev + (size_t)half * ctx->frames_bytes, *d2 = d1 + set_stride;
    const int nchunks = B < 4 ? 1 : (B < 16 ? 2 : 4);
    const int per_chunk = (B + nchunks - 1) / nchunks;
    // this half may still be read by the builds of the call before last
    KLT_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->half_free[half], 0));
    int k = 0;
    for (int first = 0; first < B; first += per_chunk, k++) {
        const int count = first + per_chunk <= B ? per_chunk : B - first;
        const size_t off = (size_t)first * frame_stride, bytes = (size_t)(count - 1) * frame_stride + one;
        KLT_CUDA(ctx, cudaMemcpyAsync(d1 + off, frames1 + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(d2 + off, frames2 + off, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        KLT_CUDA(ctx, cudaEventRecord(ctx->chunk_ev[k], ctx->copy_stream));
    }
    k = 0;
    for (int first = 0; first < B; first += per_chunk, k++) {
        const int count = first + per_chunk <= B ? per_chunk : B - first;
        const size_t off = (size_t)first * frame_stride;
        KLT_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->chunk_ev[k], 0));
        if ((rc = klt_build_u8_device(ctx, pyr1, d1 + off, pitch, frame_stride, taps, precision, first, count, nullptr))) return rc;
        if ((rc = klt_build_u8_device(ctx, pyr2, d2 + off, pitch, frame_stride, taps, precision, first, count, nullptr))) return rc;
    }
    KLT_CUDA(ctx, cudaEventRecord(ctx->half_free[half], ctx->stream));
    return track_impl(ctx, params, pyr1, pyr2, n_per_image, x, y, val, nullptr, nullptr, async);
}

int klt_track_pairs_u8(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int precision, klt_pyr *pyr1,
                       klt_pyr *pyr2, const uint8_t *frames1, const uint8_t *frames2, size_t pitch, size_t frame_stride,
                       int n_per_image, double *x, double *y, int32_t *val) {
    return track_pairs_impl(ctx, params, taps, precision, pyr1, pyr2, frames1, frames2, pitch, frame_stride, n_per_image, x, y, val, false);
}

int klt_track_pairs_u8_async(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int precision, klt_pyr *pyr1,
                             klt_pyr *pyr2, const uint8_t *frames1, const uint8_t *frames2, size_t pitch,
                             size_t frame_stride, int n_per_image, double *x, double *y, int32_t *val) {
    if (!ctx || !ctx->async_flag_dev) return klt_fail(ctx, KLT_ERR_NOMEM, "asynchronous calls need the context's status word");
    return track_pairs_impl(ctx, params, taps, precision, pyr1, pyr2, frames1, frames2, pitch, frame_stride, n_per_image, x, y, val, true);
}

int klt_async_mark(klt_ctx *ctx, int slot) {
    if (!ctx || slot < 0 || slot >= 16) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaEventRecord(ctx->marks[slot], ctx->stream));
    return KLT_OK;
}

int klt_async_wait(klt_ctx *ctx, int slot) {
    if (!ctx || slot < 0 || slot >= 16) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaEventSynchronize(ctx->marks[slot]));
    return KLT_OK;
}

int klt_async_result(klt_ctx *ctx) {
    if (!ctx || !ctx->async_flag_dev) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    int flag = 0;
    KLT_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->async_flag_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaMemsetAsync(ctx->async_flag_dev, 0, sizeof(int), ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (flag)
        return klt_fail(ctx, KLT_ERR_ASSERT, "a feature window left the image at a pyramid level in one of the asynchronous calls: the reference raises AssertionError (trackFeaturesUtils.pyx:35)");
    return KLT_OK;
}

}  // extern "C"
