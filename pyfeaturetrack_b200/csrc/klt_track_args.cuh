// Kernel-argument structs and per-feature decisions shared by the tracking translation units (klt_track.cu,
// klt_track_windowed.cu).
#pragma once
#include "klt_common.cuh"

#define KLT_INTERNAL_ASSERT (-100)

struct TrackArgs {
    klt_pyr p1, p2;
    int w, h;               // window
    int n_levels, ss;
    int max_iterations;
    float small_det, th, step_factor;
    int has_max_residue;
    float max_residue;
    int retain;
    double borderx, bordery;
    int n_per_image, total;     // features per image; END of the feature range of this launch
    int f_begin;                // first feature of this launch (a sub-range of the batch: [f_begin, total))
    int lighting_insensitive;   // gain / bias normalisation of trackFeaturesUtils.pyx:152-239 (exact-order kernel only)
    int assert_marks_feature;   // 1: a feature whose template leaves the image is written (-1, -1, KLT_OOB) instead of being
                                // left untouched (the backward pass of the forward-backward check; the flag is still raised)
};

// ---- the reference's per-feature policy (trackFeatures.py / trackFeaturesUtils.pyx), shared by the three trackers ----

// start position on the top level (trackFeatures.py:260-262); ss is a power of two, so x * (1/ss) == x / ss bit for bit
__device__ __forceinline__ void lk_top_level(double &x, double &y, int n_levels, double ss) {
    const double inv_ss = 1.0 / ss;
    for (int r = n_levels - 1; r >= 0; r--) { x = __dmul_rn(x, inv_ss); y = __dmul_rn(y, inv_ss); }
}

// the template's bilinear footprint lies inside the level (extractImagePatchOptimised's assertion, pyx:35)
__device__ __forceinline__ bool lk_template_inside(int ix, int iy, int hw, int hh, int nc, int nr) {
    return ix - hw >= 0 && iy - hh >= 0 && ix + hw + 2 <= nc && iy + hh + 2 <= nr;
}

// window check at the top of every Newton step, float32 with integer half-widths (trackFeatureIterateCKLT, pyx:393-459)
__device__ __forceinline__ bool lk_window_inside_f(float x, float y, float fhw, float fhh, float fnc, float fnr) {
    return !(__fsub_rn(x, fhw) < 0.f || __fsub_rn(fnc, __fadd_rn(x, fhw)) < 1.001f ||
             __fsub_rn(y, fhh) < 0.f || __fsub_rn(fnr, __fadd_rn(y, fhh)) < 1.001f);
}

// _trackFeature's re-check of the result (trackFeatures.py:108-136): doubles, and hw = width / 2.0 by true division
__device__ __forceinline__ bool lk_window_inside_d(float x, float y, int w, int h, int nc, int nr) {
    const double xd = (double)x, yd = (double)y, hw = w / 2.0, hh = h / 2.0;
    return !(__dsub_rn(xd, hw) < 0.0 || __dsub_rn((double)nc, __dadd_rn(xd, hw)) < 1.001 ||
             __dsub_rn(yd, hh) < 0.0 || __dsub_rn((double)nr, __dadd_rn(yd, hh)) < 1.001);
}

// a level's status as KLTTrackFeatures records it (trackFeatures.py:276-283)
__device__ __forceinline__ int lk_level_verdict(const TrackArgs &A, int status, int iteration) {
    if (A.retain) return KLT_TRACKED;
    if (status == KLT_SMALL_DET || status == KLT_OOB || status == KLT_LARGE_RESIDUE) return status;
    if (iteration >= A.max_iterations) return KLT_MAX_ITERATIONS;
    return KLT_TRACKED;
}

// the verdicts that end tracking before level 0 (trackFeatures.py:284-285)
__device__ __forceinline__ bool lk_level_lost(int st) { return st == KLT_SMALL_DET || st == KLT_OOB; }

// the feature's record after the last level, written by the one lane that owns it.  A template that left the image
// (KLT_INTERNAL_ASSERT) makes the host raise and leaves the feature untouched, unless the launch marks it lost.
__device__ __forceinline__ void lk_write_feature(const TrackArgs &A, int f, int st, double xout, double yout,
                                                 unsigned int my_iters, double *xs, double *ys, int *vals,
                                                 unsigned long long *iters_total) {
    if (my_iters) atomicAdd(iters_total, (unsigned long long)my_iters);
    if (st == KLT_INTERNAL_ASSERT) {
        if (A.assert_marks_feature) { xs[f] = -1.0; ys[f] = -1.0; vals[f] = KLT_OOB; }
        return;
    }
    const int W0 = A.p1.lv[0].w, H0 = A.p1.lv[0].h;
    const bool oob = xout < A.borderx || xout > __dsub_rn((double)(W0 - 1), A.borderx) || yout < A.bordery ||
                     yout > __dsub_rn((double)(H0 - 1), A.bordery);                         // _outOfBounds :140-141
    if (st == KLT_OOB || oob) { xs[f] = -1.0; ys[f] = -1.0; vals[f] = KLT_OOB; }
    else if (st == KLT_SMALL_DET || st == KLT_LARGE_RESIDUE || st == KLT_MAX_ITERATIONS) { xs[f] = -1.0; ys[f] = -1.0; vals[f] = st; }
    else { xs[f] = xout; ys[f] = yout; vals[f] = KLT_TRACKED; }
}

// float32 bilinear weights of the FAST trackers, and a sample of the four taps (i00 top left, i01 its right neighbour)
struct Bilinear {
    float w00, w01, w10, w11;
    __device__ __forceinline__ Bilinear(float ax, float ay) {
        w11 = ax * ay; w01 = ax - w11; w10 = ay - w11; w00 = 1.f - ax - ay + w11;
    }
    __device__ __forceinline__ float operator()(float i00, float i01, float i10, float i11) const {
        return fmaf(w11, i11, fmaf(w10, i10, fmaf(w01, i01, w00 * i00)));
    }
};

// gradient kernels of the two pyramids (the reference's kernel cache can hand different ones to the two images,
// convolve.py:236,258); c[j] multiplies in[x + j - 3]
struct WindowedTaps { float g1[7], d1[7], g2[7], d2[7]; int same; /* both images share their kernels (the normal case) */ };

bool klt_windowed_supported(const klt_params *p, const klt_pyr *p1, const klt_pyr *p2);
int klt_launch_track_windowed(klt_ctx *ctx, const TrackArgs &A, const klt_pyr *p1, const klt_pyr *p2, double *x_dev,
                              double *y_dev, int32_t *val_dev, unsigned long long *iters_dev, int *assert_dev);
