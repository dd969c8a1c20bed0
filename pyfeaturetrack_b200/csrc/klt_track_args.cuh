// Kernel-argument structs shared by the tracking translation units (klt_track.cu, klt_track_windowed.cu).
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

// gradient kernels of the two pyramids (the reference's kernel cache can hand different ones to the two images,
// convolve.py:236,258); c[j] multiplies in[x + j - 3]
struct WindowedTaps { float g1[7], d1[7], g2[7], d2[7]; int same; /* both images share their kernels (the normal case) */ };

bool klt_windowed_supported(const klt_params *p, const klt_pyr *p1, const klt_pyr *p2);
int klt_launch_track_windowed(klt_ctx *ctx, const TrackArgs &A, const klt_pyr *p1, const klt_pyr *p2, double *x_dev,
                              double *y_dev, int32_t *val_dev, unsigned long long *iters_dev, int *assert_dev);
