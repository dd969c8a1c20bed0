// klt_sequence: B lock-stepped frame sequences in sequentialMode with per-frame feature replacement -- BASELINE config D.
//
// Reference flow per frame (one sequence): KLTTrackFeatures(tc, prev, cur, fl) with tc.sequentialMode (pyramid reuse,
// trackFeatures.py:152-161,401-404), then KLTReplaceLostFeatures(tc, cur, fl) = _KLTSelectGoodFeatures(REPLACING_SOME) on the
// gradients of tc.pyramid_last (selectGoodFeatures.py:176-179, 45-135).  Here one step does that for B independent sequences at
// once: ONE pyramid build (the new frames), ONE tracking launch, ONE selection chain, all on device-resident feature lists,
// with no host synchronisation anywhere.
//
// A step has two halves with different inputs:
//   FRONT  (needs only the new frames)     pyramid build + eigenvalue maps of the new frames (the latter on a third stream
//                                          beside the decimations, forked right after the level-0 kernel)
//   BACK   (needs FRONT + the lists of     tracking prev -> cur (with the forward-backward check: then back cur -> prev),
//           the previous step)             status copy, pre-marking of the survivors, histogram, plan, scatter, greedy walk
// FRONT runs on the sequence's own stream, BACK on the context's: when the caller does not wait between steps, FRONT of frame
// k + 1 overlaps BACK of frame k (the walk and the plan are one CTA per sequence; the eigenvalue pass fills the other SMs).
// That needs three pyramid batches and three eigenvalue maps in rotation (BACK(k) still tracks out of the pyramid FRONT(k + 2)
// will overwrite, hence FRONT(k) waits for BACK(k - 2)).  Each half is captured into a CUDA graph per rotation slot once it has
// run as plain launches; from then on a step is two graph launches and four event operations.  Host frames are uploaded on
// the copy stream into the staging buffer of the step's rotation slot.  $KLT_B200_SEQ_OVERLAP=0 (and profiling) puts everything on one stream.
#include <cfloat>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "klt_common.cuh"
#include "klt_select.cuh"

#define SEQ_ROT 3                    // rotation depth of the pyramid batches and eigenvalue maps

struct klt_sequence {
    klt_params params;
    klt_taps taps;
    int w, h, B, n, precision, select_mode;
    klt_pyr *pyr[SEQ_ROT];
    float *vmap[SEQ_ROT];            // eigenvalue maps, one per rotation slot ([0] is the one carved out of `block`)
    int cur;                         // rotation slot that holds the latest frame
    int started;
    long steps;
    SelDev S_all, S_rep;
    float *sat;
    bool fast_select_ok;
    char *block;                     // selection workspace + feature lists + counters (one allocation)
    double *fx, *fy;
    int *fval, *fval_tracked;
    unsigned long long *iters;       // [0] Newton iterations since the last klt_sequence_sync
    int *aflag;                      // sticky "a window left the image" flag (the reference's AssertionError case)
    uint8_t *stage[SEQ_ROT];         // device staging of the frames, one per rotation slot (the captured graphs carry the pointer)
    size_t stage_bytes, cap_pitch, cap_stride;
    cudaEvent_t stage_free[SEQ_ROT], stage_ready[SEQ_ROT];
    cudaStream_t front_stream;       // FRONT halves (own stream unless overlap is off)
    cudaStream_t eigen_stream;       // the eigenvalue pass inside FRONT, beside the decimations
    cudaEvent_t fork_ev, join_ev;    // eigenvalue pass beside the decimations (inside FRONT)
    cudaEvent_t front_done[SEQ_ROT], back_done[SEQ_ROT];
    bool back_recorded[SEQ_ROT];
    int overlap;
    int use_graph;
    cudaGraphExec_t graph[2][SEQ_ROT][2];     // [half: 0 front, 1 back][rotation slot][replace]
    bool graph_ok[2][SEQ_ROT][2];
    int warm[2][SEQ_ROT][2];
    int64_t graph_launches[2][SEQ_ROT][2];
    // forward-backward check (klt_sequence_set_fb_check): threshold (0 = off) and its arrays, allocated on first use
    float fb_max;
    bool fb_ran;                     // the last step ran the check (fb_err is current)
    char *fb_block;
    FbArrays fb;
    float *fb_err;
};

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// selection on the level-0 planes of `p` (all images) into the sequence's feature lists, one stream
static int select_on(klt_ctx *ctx, klt_sequence *q, klt_pyr *p, const SelDev *S) {
    int rc;
    if ((rc = klt_sel_launch_begin(ctx, S, q->B))) return rc;
    if ((rc = klt_sel_launch_eigen(ctx, S, q->B, p, q->select_mode, q->sat))) return rc;
    return klt_sel_launch_pick(ctx, S, q->B);
}

static SelDev sel_for_slot(const klt_sequence *q, int slot) {
    SelDev S = q->S_rep;
    S.vmap = q->vmap[slot];
    return S;
}

// FRONT of a step on ctx->stream (the caller points it at the stream it wants): frames in stage[par] -> pyramid `slot`,
// and (replacement steps) its eigenvalue maps
static int enqueue_front(klt_ctx *ctx, klt_sequence *q, int par, int slot, int replace) {
    const SelDev S = sel_for_slot(q, slot);
    int rc;
    // the fused fast eigenvalue pass reads the level-0 image only: it forks right after the level-0 kernel and runs beside the
    // decimations; the table-based pass needs the gradient planes, i.e. the whole build
    const bool fork = replace && q->overlap && !ctx->profiling && q->eigen_stream && q->fast_select_ok;
    if ((rc = klt_build_u8_device(ctx, q->pyr[slot], q->stage[par], q->cap_pitch, q->cap_stride, &q->taps, q->precision, 0, q->B,
                                  fork ? q->fork_ev : nullptr))) return rc;
    if (!replace) return KLT_OK;
    if (fork) {
        cudaStream_t mine = ctx->stream;
        KLT_CUDA(ctx, cudaStreamWaitEvent(q->eigen_stream, q->fork_ev, 0));
        ctx->stream = q->eigen_stream;
        rc = klt_sel_launch_eigen(ctx, &S, q->B, q->pyr[slot], q->select_mode, q->sat);
        ctx->stream = mine;
        if (rc) return rc;
        KLT_CUDA(ctx, cudaEventRecord(q->join_ev, q->eigen_stream));
        KLT_CUDA(ctx, cudaStreamWaitEvent(mine, q->join_ev, 0));
        return KLT_OK;
    }
    return klt_sel_launch_eigen(ctx, &S, q->B, q->pyr[slot], q->select_mode, q->sat);
}

// BACK of a step on ctx->stream: tracking prev -> slot and the list-dependent part of the replacement
static int enqueue_back(klt_ctx *ctx, klt_sequence *q, int prev, int slot, int replace) {
    int rc;
    // both pyramids stay alive until BACK ends (rotation of three), so the backward pass needs no further synchronisation
    if (q->fb_max > 0.f) {
        if ((rc = klt_launch_track_fb(ctx, &q->params, q->pyr[prev], q->pyr[slot], q->n, q->fb_max, q->fx, q->fy, q->fval, q->fb,
                                      q->fb_err, q->iters, q->aflag))) return rc;
    } else if ((rc = klt_launch_track(ctx, &q->params, q->pyr[prev], q->pyr[slot], q->n, q->fx, q->fy, q->fval, q->iters, q->aflag))) return rc;
    KLT_CUDA(ctx, cudaMemcpyAsync(q->fval_tracked, q->fval, (size_t)q->B * q->n * sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
    if (!replace) return KLT_OK;
    const SelDev S = sel_for_slot(q, slot);
    if ((rc = klt_sel_launch_begin(ctx, &S, q->B))) return rc;
    return klt_sel_launch_pick(ctx, &S, q->B);
}

static void drop_graphs(klt_sequence *q) {
    for (int hf = 0; hf < 2; hf++)
        for (int a = 0; a < SEQ_ROT; a++)
            for (int r = 0; r < 2; r++) {
                if (q->graph_ok[hf][a][r]) { cudaGraphExecDestroy(q->graph[hf][a][r]); q->graph_ok[hf][a][r] = false; }
                q->warm[hf][a][r] = 0;
            }
}

// frames -> stage[par]; the stream `consumer` (the one FRONT runs on) waits for them
static int stage_frames(klt_ctx *ctx, klt_sequence *q, int par, const uint8_t *frames, size_t pitch, size_t frame_stride,
                        cudaStream_t consumer) {
    if (pitch < (size_t)q->w) return klt_fail(ctx, KLT_ERR_INVALID, "pitch %zu smaller than width %d", pitch, q->w);
    const size_t bytes = (size_t)(q->B - 1) * frame_stride + (size_t)(q->h - 1) * pitch + q->w;
    if (bytes > q->stage_bytes) {
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(q->front_stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
        for (int i = 0; i < SEQ_ROT; i++) {
            if (q->stage[i]) KLT_CUDA(ctx, cudaFree(q->stage[i]));
            q->stage[i] = nullptr;
            KLT_CUDA(ctx, cudaMalloc(&q->stage[i], bytes + 256));
        }
        drop_graphs(q);
        q->stage_bytes = bytes;
    }
    if (pitch != q->cap_pitch || frame_stride != q->cap_stride) {      // captured graphs carry the frame layout
        drop_graphs(q);
        q->cap_pitch = pitch; q->cap_stride = frame_stride;
    }
    if (klt_is_device_ptr(frames)) {
        // (the consumer stream itself orders this copy behind the build that last read the buffer)
        KLT_CUDA(ctx, cudaMemcpyAsync(q->stage[par], frames, bytes, cudaMemcpyDeviceToDevice, consumer));
    } else {
        KLT_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, q->stage_free[par], 0));     // the build of three steps ago has read it
        KLT_CUDA(ctx, cudaMemcpyAsync(q->stage[par], frames, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        KLT_CUDA(ctx, cudaEventRecord(q->stage_ready[par], ctx->copy_stream));
        KLT_CUDA(ctx, cudaStreamWaitEvent(consumer, q->stage_ready[par], 0));
    }
    return KLT_OK;
}

// One half of a step on `stream`: plain launches the first time a (slot, replace) combination comes up, captured into a graph
// the second time, replayed afterwards.  half 0 = FRONT, 1 = BACK.
static int run_half(klt_ctx *ctx, klt_sequence *q, int half, cudaStream_t stream, int par, int prev, int slot, int rep) {
    int rc = KLT_OK;
    cudaStream_t saved = ctx->stream;
    auto enqueue = [&]() { return half == 0 ? enqueue_front(ctx, q, par, slot, rep) : enqueue_back(ctx, q, prev, slot, rep); };
    bool launched = false;
    ctx->stream = stream;
    if (q->use_graph && !ctx->profiling) {
        if (!q->graph_ok[half][slot][rep] && q->warm[half][slot][rep]) {
            const int64_t l0 = ctx->launches;
            cudaGraph_t g = nullptr;
            if (cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                rc = enqueue();
                const cudaError_t ee = cudaStreamEndCapture(stream, &g);
                if (rc == KLT_OK && ee == cudaSuccess && g && cudaGraphInstantiate(&q->graph[half][slot][rep], g, 0) == cudaSuccess) {
                    q->graph_ok[half][slot][rep] = true;
                    q->graph_launches[half][slot][rep] = ctx->launches - l0;
                } else {
                    cudaGetLastError();
                    q->use_graph = 0;                      // this configuration cannot be captured: plain launches from now on
                }
                if (g) cudaGraphDestroy(g);
                ctx->launches = l0;
                rc = KLT_OK;
            } else {
                cudaGetLastError();
                q->use_graph = 0;
            }
        }
        if (q->graph_ok[half][slot][rep]) {
            if (half == 0) {                               // host-side bookkeeping the captured calls would have done
                klt_pyr_note_build(q->pyr[slot], &q->taps, q->precision);
                if (rep && !q->fast_select_ok) q->pyr[slot]->hx->grad0_valid = true;
            }
            const cudaError_t e = cudaGraphLaunch(q->graph[half][slot][rep], stream);
            if (e != cudaSuccess) { ctx->stream = saved; return klt_fail(ctx, KLT_ERR_CUDA, "cudaGraphLaunch failed: %s", cudaGetErrorString(e)); }
            ctx->launches += q->graph_launches[half][slot][rep];
            launched = true;
        }
    }
    if (!launched) {
        rc = enqueue();
        q->warm[half][slot][rep] = 1;
    }
    ctx->stream = saved;
    return rc;
}

extern "C" {

int klt_sequence_create(klt_ctx *ctx, const klt_params *params, const klt_taps *taps, int w, int h, int n_sequences,
                        int n_features, int precision, int select_mode, klt_sequence **out) {
    if (!ctx || !params || !taps || !out || w <= 0 || h <= 0 || n_sequences <= 0 || n_features <= 0)
        return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (select_mode != KLT_SELECT_STRICT && select_mode != KLT_SELECT_FAST) return klt_fail(ctx, KLT_ERR_INVALID, "select_mode must be KLT_SELECT_STRICT or KLT_SELECT_FAST");
    if (precision < 0 || precision > 2) return klt_fail(ctx, KLT_ERR_INVALID, "bad precision");
    if (params->affine_consistency_check >= 0 || params->lighting_insensitive)
        return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "klt_sequence covers translational tracking; use klt_track_features_affine per frame for the affine check");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    *out = nullptr;
    klt_sequence *q = new klt_sequence();
    memset(q, 0, sizeof *q);
    q->params = *params; q->taps = *taps;
    q->w = w; q->h = h; q->B = n_sequences; q->n = n_features; q->precision = precision; q->select_mode = select_mode;
    q->use_graph = getenv("KLT_B200_NO_GRAPH") ? 0 : 1;
    q->overlap = (getenv("KLT_B200_SEQ_OVERLAP") && atoi(getenv("KLT_B200_SEQ_OVERLAP")) == 0) ? 0 : 1;
    int rc;
    for (int i = 0; i < SEQ_ROT; i++)
        if ((rc = klt_pyr_create(ctx, w, h, params->n_levels, params->subsampling, n_sequences, &q->pyr[i]))) { klt_sequence_destroy(ctx, q); return rc; }
    if ((rc = klt_sel_geometry(ctx, params, w, h, n_features, 1, &q->S_rep))) { klt_sequence_destroy(ctx, q); return rc; }
    q->fast_select_ok = select_mode == KLT_SELECT_FAST && klt_sel_fast_covers(&q->S_rep, &taps->grad_gauss, &taps->grad_deriv);
    const bool need_sat = !q->fast_select_ok;
    const size_t total = (size_t)q->B * q->n;
    const size_t sel_b = klt_sel_workspace_bytes(&q->S_rep, q->B, need_sat, true);
    const size_t extra = align_up(total * sizeof(int), 256) + 512;
    cudaError_t e = cudaMalloc(&q->block, sel_b + extra);
    if (e != cudaSuccess) { klt_sequence_destroy(ctx, q); return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for the sequence workspace failed: %s", sel_b + extra, cudaGetErrorString(e)); }
    klt_sel_carve(&q->S_rep, q->B, need_sat, true, q->block, &q->sat);
    q->vmap[0] = q->S_rep.vmap;
    for (int i = 1; i < SEQ_ROT; i++) {
        e = cudaMalloc(&q->vmap[i], (size_t)q->B * (q->S_rep.ncand + 1) * sizeof(float));
        if (e != cudaSuccess) { klt_sequence_destroy(ctx, q); return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc for an eigenvalue map failed: %s", cudaGetErrorString(e)); }
    }
    q->fx = q->S_rep.fx; q->fy = q->S_rep.fy; q->fval = q->S_rep.fval;
    q->fval_tracked = (int *)(q->block + sel_b);
    q->iters = (unsigned long long *)(q->block + sel_b + align_up(total * sizeof(int), 256));
    q->aflag = (int *)(q->iters + 4);
    cudaMemsetAsync(q->block + sel_b, 0, extra, ctx->stream);
    q->S_all = q->S_rep;                    // same buffers, SELECTING_ALL semantics
    q->S_all.replace = 0; q->S_all.premap = nullptr; q->S_all.target_mul = 32u; q->S_all.target_add = 8192u;
    if ((rc = klt_sel_prepare_kernels(ctx, &q->S_rep))) { klt_sequence_destroy(ctx, q); return rc; }
    for (int i = 0; i < SEQ_ROT; i++) {
        cudaEventCreateWithFlags(&q->stage_free[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&q->stage_ready[i], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&q->fork_ev, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&q->join_ev, cudaEventDisableTiming);
    for (int i = 0; i < SEQ_ROT; i++) {
        cudaEventCreateWithFlags(&q->front_done[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&q->back_done[i], cudaEventDisableTiming);
    }
    if (q->overlap) {
        // (lowest-priority streams for FRONT -- BACK is the critical path -- measured no better, with outliers: default priority)
        if (cudaStreamCreateWithFlags(&q->front_stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); q->front_stream = nullptr; }
        if (cudaStreamCreateWithFlags(&q->eigen_stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); q->eigen_stream = nullptr; }
    }
    *out = q;
    return KLT_OK;
}

int klt_sequence_destroy(klt_ctx *ctx, klt_sequence *q) {
    if (!q) return KLT_OK;
    if (ctx) { cudaStreamSynchronize(ctx->stream); cudaStreamSynchronize(ctx->copy_stream); if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream); }
    if (q->front_stream) cudaStreamSynchronize(q->front_stream);
    if (q->eigen_stream) cudaStreamSynchronize(q->eigen_stream);
    drop_graphs(q);
    for (int i = 0; i < SEQ_ROT; i++) {
        if (q->pyr[i]) klt_pyr_destroy(ctx, q->pyr[i]);
        if (i > 0 && q->vmap[i]) cudaFree(q->vmap[i]);
        if (q->front_done[i]) cudaEventDestroy(q->front_done[i]);
        if (q->back_done[i]) cudaEventDestroy(q->back_done[i]);
    }
    for (int i = 0; i < SEQ_ROT; i++) {
        if (q->stage[i]) cudaFree(q->stage[i]);
        if (q->stage_free[i]) cudaEventDestroy(q->stage_free[i]);
        if (q->stage_ready[i]) cudaEventDestroy(q->stage_ready[i]);
    }
    if (q->fork_ev) cudaEventDestroy(q->fork_ev);
    if (q->join_ev) cudaEventDestroy(q->join_ev);
    if (q->front_stream) cudaStreamDestroy(q->front_stream);
    if (q->eigen_stream) cudaStreamDestroy(q->eigen_stream);
    if (q->block) cudaFree(q->block);
    if (q->fb_block) cudaFree(q->fb_block);
    delete q;
    return KLT_OK;
}

int klt_sequence_start_u8(klt_ctx *ctx, klt_sequence *q, const uint8_t *frames, size_t pitch, size_t frame_stride, int select) {
    if (!ctx || !q || !frames) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    const int par = 0, slot = 0;
    // a restart must not overtake FRONT halves still in flight
    if (q->front_stream) KLT_CUDA(ctx, cudaStreamSynchronize(q->front_stream));
    for (int i = 0; i < SEQ_ROT; i++) q->back_recorded[i] = false;
    if ((rc = stage_frames(ctx, q, par, frames, pitch, frame_stride, ctx->stream))) return rc;
    if ((rc = klt_build_u8_device(ctx, q->pyr[slot], q->stage[par], pitch, frame_stride, &q->taps, q->precision, 0, q->B, nullptr))) return rc;
    KLT_CUDA(ctx, cudaEventRecord(q->stage_free[par], ctx->stream));
    if (select) {
        SelDev S = q->S_all;
        S.vmap = q->vmap[slot];
        if ((rc = select_on(ctx, q, q->pyr[slot], &S))) return rc;
    }
    KLT_CUDA(ctx, cudaEventRecord(q->back_done[slot], ctx->stream));
    q->back_recorded[slot] = true;
    q->cur = slot; q->started = 1; q->steps = 0;
    q->fb_ran = false;
    return KLT_OK;
}

int klt_sequence_set_features(klt_ctx *ctx, klt_sequence *q, const double *x, const double *y, const int32_t *val) {
    if (!ctx || !q || !x || !y || !val) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    const size_t total = (size_t)q->B * q->n;
    KLT_CUDA(ctx, cudaMemcpyAsync(q->fx, x, total * sizeof(double), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(q->fy, y, total * sizeof(double), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(q->fval, val, total * sizeof(int32_t), cudaMemcpyDefault, ctx->stream));
    return KLT_OK;
}

static int copy_out(klt_ctx *ctx, klt_sequence *q, double *x, double *y, int32_t *val, int32_t *val_tracked) {
    const size_t total = (size_t)q->B * q->n;
    if (x) KLT_CUDA(ctx, cudaMemcpyAsync(x, q->fx, total * sizeof(double), cudaMemcpyDefault, ctx->stream));
    if (y) KLT_CUDA(ctx, cudaMemcpyAsync(y, q->fy, total * sizeof(double), cudaMemcpyDefault, ctx->stream));
    if (val) KLT_CUDA(ctx, cudaMemcpyAsync(val, q->fval, total * sizeof(int32_t), cudaMemcpyDefault, ctx->stream));
    if (val_tracked) KLT_CUDA(ctx, cudaMemcpyAsync(val_tracked, q->fval_tracked, total * sizeof(int32_t), cudaMemcpyDefault, ctx->stream));
    return KLT_OK;
}

int klt_sequence_step_u8(klt_ctx *ctx, klt_sequence *q, const uint8_t *frames, size_t pitch, size_t frame_stride, int replace,
                         double *x, double *y, int32_t *val, int32_t *val_tracked) {
    if (!ctx || !q || !frames) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (!q->started) return klt_fail(ctx, KLT_ERR_INVALID, "klt_sequence_start_u8 has not been called");
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    const int rep = replace ? 1 : 0;
    const int prev = q->cur, slot = (q->cur + 1) % SEQ_ROT, par = slot;      // frames of slot s are staged in stage[s]
    const bool split = q->overlap && q->front_stream && !ctx->profiling;
    cudaStream_t fs = split ? q->front_stream : ctx->stream;
    // FRONT(k) overwrites the pyramid and the eigenvalue map of slot k mod 3, which BACK(k - 2) (tracking out of that pyramid)
    // and BACK(k - 3) were the last to read: wait for BACK(k - 2), recorded under slot (k - 2) mod 3 = (slot + 1) mod 3
    if (split && q->back_recorded[(slot + 1) % SEQ_ROT]) KLT_CUDA(ctx, cudaStreamWaitEvent(fs, q->back_done[(slot + 1) % SEQ_ROT], 0));
    // the first FRONT also waits for klt_sequence_start_u8, whose selection runs on the context's stream and shares the
    // summed-area-table workspace with the FRONT halves
    if (split && q->steps == 0 && q->back_recorded[q->cur]) KLT_CUDA(ctx, cudaStreamWaitEvent(fs, q->back_done[q->cur], 0));
    if ((rc = stage_frames(ctx, q, par, frames, pitch, frame_stride, fs))) return rc;
    if ((rc = run_half(ctx, q, 0, fs, par, prev, slot, rep))) return rc;
    KLT_CUDA(ctx, cudaEventRecord(q->stage_free[par], fs));
    if (split) {
        KLT_CUDA(ctx, cudaEventRecord(q->front_done[slot], fs));
        KLT_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, q->front_done[slot], 0));
    }
    if ((rc = run_half(ctx, q, 1, ctx->stream, par, prev, slot, rep))) return rc;
    KLT_CUDA(ctx, cudaEventRecord(q->back_done[slot], ctx->stream));
    q->back_recorded[slot] = true;
    q->cur = slot;
    q->steps++;
    q->fb_ran = q->fb_max > 0.f;
    return copy_out(ctx, q, x, y, val, val_tracked);
}

int klt_sequence_get_features(klt_ctx *ctx, klt_sequence *q, double *x, double *y, int32_t *val, int32_t *val_tracked) {
    if (!ctx || !q) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    int rc = copy_out(ctx, q, x, y, val, val_tracked);
    if (rc) return rc;
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_sequence_sync(klt_ctx *ctx, klt_sequence *q, int64_t *n_iterations) {
    if (!ctx || !q) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    unsigned long long res[5] = {0, 0, 0, 0, 0};
    KLT_CUDA(ctx, cudaMemcpyAsync(res, q->iters, sizeof res, cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaMemsetAsync(q->iters, 0, sizeof res, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (n_iterations) *n_iterations = (int64_t)res[0];
    if ((int)(res[4] & 0xffffffffull))
        return klt_fail(ctx, KLT_ERR_ASSERT, "a feature window left the image at a pyramid level: the reference raises AssertionError (trackFeaturesUtils.pyx:35)");
    return KLT_OK;
}

int klt_sequence_select_stats(klt_ctx *ctx, klt_sequence *q, int64_t *out) {
    if (!ctx || !q || !out) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    KLT_CUDA(ctx, cudaMemcpyAsync(out, q->S_rep.status, (size_t)q->B * SEL_STATUS_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_sequence_pyramid(klt_sequence *q, klt_pyr **out) {
    if (!q || !out) return KLT_ERR_INVALID;
    *out = q->pyr[q->cur];
    return KLT_OK;
}

int klt_sequence_set_fb_check(klt_ctx *ctx, klt_sequence *q, float max_fb_error) {
    if (!ctx || !q) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    if (!(max_fb_error == 0.f || (max_fb_error > 0.f && max_fb_error <= FLT_MAX)))
        return klt_fail(ctx, KLT_ERR_INVALID, "max_fb_error must be 0 (off) or finite and > 0 (got %g)", (double)max_fb_error);
    KLT_CUDA(ctx, cudaSetDevice(ctx->device));
    if (max_fb_error > 0.f && !q->fb_block) {
        const size_t total = (size_t)q->B * q->n, db = align_up(total * sizeof(double), 256), ib = align_up(total * sizeof(int), 256);
        const size_t bytes = 4 * db + 2 * ib + 256;
        cudaError_t e = cudaMalloc(&q->fb_block, bytes);
        if (e != cudaSuccess) { q->fb_block = nullptr; return klt_fail(ctx, KLT_ERR_NOMEM, "cudaMalloc(%zu) for the forward-backward arrays failed: %s", bytes, cudaGetErrorString(e)); }
        char *b = q->fb_block;
        q->fb.x0 = (double *)b; b += db;
        q->fb.y0 = (double *)b; b += db;
        q->fb.xb = (double *)b; b += db;
        q->fb.yb = (double *)b; b += db;
        q->fb.vb = (int32_t *)b; b += ib;
        q->fb_err = (float *)b; b += ib;
        q->fb.scratch_assert = (int *)b;
    }
    if (max_fb_error != q->fb_max) drop_graphs(q);      // the captured BACK halves carry the check and its threshold
    q->fb_max = max_fb_error;
    return KLT_OK;
}

int klt_sequence_get_fb_error(klt_ctx *ctx, klt_sequence *q, float *out) {
    if (!ctx || !q || !out) return klt_fail(ctx, KLT_ERR_INVALID, "bad argument");
    const size_t total = (size_t)q->B * q->n;
    if (q->fb_ran) {
        KLT_CUDA(ctx, cudaMemcpyAsync(out, q->fb_err, total * sizeof(float), cudaMemcpyDefault, ctx->stream));
    } else {
        std::vector<float> none(total, -1.f);
        KLT_CUDA(ctx, cudaMemcpyAsync(out, none.data(), total * sizeof(float), cudaMemcpyDefault, ctx->stream));
    }
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

int klt_sequence_uses_graph(const klt_sequence *q) {
    if (!q) return 0;
    for (int hf = 0; hf < 2; hf++)
        for (int a = 0; a < SEQ_ROT; a++)
            for (int r = 0; r < 2; r++)
                if (q->graph_ok[hf][a][r]) return 1;
    return 0;
}

}  // extern "C"
