// Pyramidal Lucas-Kanade tracking: one warp per feature, all pyramid levels in one launch (sm_100a).
//
// Replaces the per-feature loop of KLTTrackFeatures (trackFeatures.py:250-346), _trackFeature (:67-136)
// and the Cython inner loops trackFeatureIterateCKLT / extractImagePatchOptimised /
// _computeIntensityDifference / _computeGradientSum / _compute2by2GradientMatrix / _compute2by1ErrorVector /
// _solveEquation (trackFeaturesUtils.pyx:20-51,61-128,246-340,393-459).
//
// Arithmetic follows the reference's operand types EXACTLY (taken from the Cython-generated C):
//   * bilinear sample: three products in double, the (ax*ay)*I11 product in float, summed left to right in
//     double, rounded to float once;
//   * gradient sums, products and the five window sums in float32 without FMA contraction; the window
//     sums run SEQUENTIALLY in row-major order (one lane per sum), because float addition order is part
//     of the reference's result;
//   * 2x2 solve in float32 with separately rounded products;
//   * the Python-level re-check uses doubles and hw = width/2 = 3.5 (true division, quirk Q2);
//   * the residue uses NumPy's float32 pairwise summation order.
// Given bit-identical pyramids (STRICT mode) the positions and status codes are bit-identical to the
// reference's; with FAST pyramids they agree to ~1e-4 px.
#include "klt_common.cuh"
#include "klt_track_args.cuh"

// bilinear sample with the reference's mixed precision (trackFeaturesUtils.pyx:44-47)
__device__ __forceinline__ float bilerp_ref(const float *__restrict__ p, int pitch, float ax, float ay) {
    const double dax = (double)ax, day = (double)ay;
    const double omx = __dsub_rn(1.0, dax), omy = __dsub_rn(1.0, day);
    const float i00 = p[0], i01 = p[1], i10 = p[pitch], i11 = p[pitch + 1];
    double v = __dmul_rn(__dmul_rn(omx, omy), (double)i00);
    v = __dadd_rn(v, __dmul_rn(__dmul_rn(dax, omy), (double)i01));
    v = __dadd_rn(v, __dmul_rn(__dmul_rn(omx, day), (double)i10));
    v = __dadd_rn(v, (double)__fmul_rn(__fmul_rn(ax, ay), i11));
    return __double2float_rn(v);
}

// NumPy FLOAT_pairwise_sum (numpy/_core/src/umath/loops_utils.h.src), executed by one lane.
__device__ float np_pairwise_sum(const float *a, int n) {
    if (n < 8) {
        float res = 0.f;
        for (int i = 0; i < n; i++) res = __fadd_rn(res, a[i]);
        return res;
    } else if (n <= 128) {
        float r[8];
        int i;
#pragma unroll
        for (i = 0; i < 8; i++) r[i] = a[i];
        for (i = 8; i < n - (n % 8); i += 8) {
#pragma unroll
            for (int j = 0; j < 8; j++) r[j] = __fadd_rn(r[j], a[i + j]);
        }
        float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                              __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
        for (; i < n; i++) res = __fadd_rn(res, a[i]);
        return res;
    } else {
        int n2 = n / 2;
        n2 -= n2 % 8;
        return __fadd_rn(np_pairwise_sum(a, n2), np_pairwise_sum(a + n2, n - n2));
    }
}

// Gain / bias normalisation of the lighting-insensitive mode (the C carried as comments in trackFeaturesUtils.pyx:152-239;
// the reference itself raises "Not implemented", so parity is against the oracle's restatement only).  T, P: the two
// windows in shared memory.  Lanes 0..3 run one sequential float32 sum each, in the C's row-major order:
//   alpha = sqrt((sum T^2/n)/(sum P^2/n)), belta = sum T/n - alpha * sum P/n; alphag = sqrt((sum T/n)/(sum P/n)) is what
//   the gradient routine computes (it accumulates the plain values into its sum*_squared variables, pyx:222-224).
struct LiCoeffs { float alpha, belta, alphag; };
__device__ __forceinline__ LiCoeffs li_coefficients(const float *T, const float *P, int n, int lane) {
    float acc = 0.f;
    if (lane < 4) {
        const float *s = (lane & 1) ? P : T;
        if (lane < 2) for (int k = 0; k < n; k++) acc = __fadd_rn(acc, s[k]);
        else for (int k = 0; k < n; k++) acc = __fadd_rn(acc, __fmul_rn(s[k], s[k]));
    }
    const float sum1 = __shfl_sync(0xffffffffu, acc, 0), sum2 = __shfl_sync(0xffffffffu, acc, 1);
    const float sq1 = __shfl_sync(0xffffffffu, acc, 2), sq2 = __shfl_sync(0xffffffffu, acc, 3);
    const float fn = (float)n;
    LiCoeffs c;
    c.alpha = __double2float_rn(__dsqrt_rn((double)__fdiv_rn(__fdiv_rn(sq1, fn), __fdiv_rn(sq2, fn))));
    const float m1 = __fdiv_rn(sum1, fn), m2 = __fdiv_rn(sum2, fn);
    c.belta = __fsub_rn(m1, __fmul_rn(c.alpha, m2));
    c.alphag = __double2float_rn(__dsqrt_rn((double)__fdiv_rn(m1, m2)));
    return c;
}

// trackFeatureIterateCKLT (trackFeaturesUtils.pyx:393-459) for one feature, executed by one warp with the reference's
// exact float32 operation order.  T/Tgx/Tgy: the w*h template patches (shared memory), S: 5*w*h floats of scratch.
__device__ __forceinline__ int iterate_exact(const float *T, const float *Tgx, const float *Tgy, float *S,
                                             const float *__restrict__ I2, const float *__restrict__ GX2,
                                             const float *__restrict__ GY2, int pitch, int nc, int nr, int w, int h,
                                             float step_factor, float small_det, float th, int max_iterations, int lane,
                                             float &x2, float &y2, int &iteration, bool lighting_insensitive = false) {
    const int n = w * h, hw = w / 2, hh = h / 2;
    const float fhw = (float)hw, fhh = (float)hh, fnc = (float)nc, fnr = (float)nr;
    int status = KLT_TRACKED;
    while (true) {
        if (!lk_window_inside_f(x2, y2, fhw, fhh, fnc, fnr)) { status = KLT_OOB; break; }
        const int ix = (int)x2, iy = (int)y2;
        const float ax = __double2float_rn(__dsub_rn((double)x2, (double)ix));
        const float ay = __double2float_rn(__dsub_rn((double)y2, (double)iy));
        if (lighting_insensitive) {
            // second image's patches first (the normalisation needs whole-window sums), then the products in place:
            // element k is read and overwritten by the same lane
            for (int k = lane; k < n; k += 32) {
                const int j = k / w, i = k - j * w;
                const size_t o = (size_t)(iy + j - hh) * pitch + (ix + i - hw);
                S[k] = bilerp_ref(I2 + o, pitch, ax, ay);
                S[n + k] = bilerp_ref(GX2 + o, pitch, ax, ay);
                S[2 * n + k] = bilerp_ref(GY2 + o, pitch, ax, ay);
            }
            __syncwarp();
            const LiCoeffs c = li_coefficients(T, S, n, lane);
            for (int k = lane; k < n; k += 32) {
                const float diff = __fsub_rn(__fsub_rn(T[k], __fmul_rn(S[k], c.alpha)), c.belta);
                const float gx = __fadd_rn(Tgx[k], __fmul_rn(S[n + k], c.alphag));
                const float gy = __fadd_rn(Tgy[k], __fmul_rn(S[2 * n + k], c.alphag));
                S[k] = __fmul_rn(gx, gx);
                S[n + k] = __fmul_rn(gx, gy);
                S[2 * n + k] = __fmul_rn(gy, gy);
                S[3 * n + k] = __fmul_rn(diff, gx);
                S[4 * n + k] = __fmul_rn(diff, gy);
            }
        } else {
            for (int k = lane; k < n; k += 32) {
                const int j = k / w, i = k - j * w;
                const size_t o = (size_t)(iy + j - hh) * pitch + (ix + i - hw);
                const float diff = __fsub_rn(T[k], bilerp_ref(I2 + o, pitch, ax, ay));       // pyx:61-88
                const float gx = __fadd_rn(Tgx[k], bilerp_ref(GX2 + o, pitch, ax, ay));      // -jacobian[:,0], pyx:107-128
                const float gy = __fadd_rn(Tgy[k], bilerp_ref(GY2 + o, pitch, ax, ay));
                S[k] = __fmul_rn(gx, gx);
                S[n + k] = __fmul_rn(gx, gy);
                S[2 * n + k] = __fmul_rn(gy, gy);
                S[3 * n + k] = __fmul_rn(diff, gx);
                S[4 * n + k] = __fmul_rn(diff, gy);
            }
        }
        __syncwarp();
        float acc = 0.f;                      // lanes 0..4: one sequential float32 sum each (pyx:246-305)
        if (lane < 5) {
            const float *s = S + lane * n;
#pragma unroll 7
            for (int k = 0; k < n; k++) acc = __fadd_rn(acc, s[k]);
        }
        __syncwarp();
        const float gxx = __shfl_sync(0xffffffffu, acc, 0), gxy = __shfl_sync(0xffffffffu, acc, 1),
                    gyy = __shfl_sync(0xffffffffu, acc, 2);
        const float ex = __fmul_rn(__shfl_sync(0xffffffffu, acc, 3), step_factor),
                    ey = __fmul_rn(__shfl_sync(0xffffffffu, acc, 4), step_factor);
        const float det = __fsub_rn(__fmul_rn(gxx, gyy), __fmul_rn(gxy, gxy));            // pyx:318-340
        if (det < small_det) { status = KLT_SMALL_DET; break; }
        const float dx = __fdiv_rn(__fsub_rn(__fmul_rn(gyy, ex), __fmul_rn(gxy, ey)), det);
        const float dy = __fdiv_rn(__fsub_rn(__fmul_rn(gxx, ey), __fmul_rn(gxy, ex)), det);
        x2 = __fadd_rn(x2, dx); y2 = __fadd_rn(y2, dy);
        iteration++;
        if (!((fabsf(dx) >= th || fabsf(dy) >= th) && iteration < max_iterations)) break;
    }
    return status;
}

// Shared memory per warp: T, Tgx, Tgy (templates) + 5 product arrays, each n = w*h floats.
__global__ void __launch_bounds__(128)
lk_track_kernel(const __grid_constant__ TrackArgs A, double *__restrict__ xs, double *__restrict__ ys,
                int *__restrict__ vals, unsigned long long *__restrict__ iters_total, int *__restrict__ assert_flag) {
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = A.f_begin + blockIdx.x * (blockDim.x >> 5) + warp;
    if (f >= A.total) return;
    if (vals[f] < 0) return;                                  // trackFeatures.py:253
    const int n = A.w * A.h;
    float *T = smem + (size_t)warp * 8 * n;
    float *Tgx = T + n, *Tgy = T + 2 * n, *S = T + 3 * n;     // S: 5 arrays of products / |diff|
    const int image = f / A.n_per_image;
    const int hw = A.w / 2, hh = A.h / 2;
    const double ss = (double)A.ss;

    double xloc = xs[f], yloc = ys[f];
    lk_top_level(xloc, yloc, A.n_levels, ss);
    double xout = xloc, yout = yloc;
    int st = KLT_TRACKED;
    unsigned int my_iters = 0;

    for (int r = A.n_levels - 1; r >= 0; r--) {
        xloc = __dmul_rn(xloc, ss); yloc = __dmul_rn(yloc, ss);
        xout = __dmul_rn(xout, ss); yout = __dmul_rn(yout, ss);
        const int nc = A.p1.lv[r].w, nr = A.p1.lv[r].h, pitch = A.p1.lv[r].pitch;
        const float *I1 = A.p1.level(0, image, r), *GX1 = A.p1.level(1, image, r), *GY1 = A.p1.level(2, image, r);
        const float *I2 = A.p2.level(0, image, r), *GX2 = A.p2.level(1, image, r), *GY2 = A.p2.level(2, image, r);

        // ---- _trackFeature: templates at (x1,y1) (trackFeatures.py:102-104) ----
        const float x1 = __double2float_rn(xloc), y1 = __double2float_rn(yloc);
        {
            const int ix = (int)x1, iy = (int)y1;
            if (!lk_template_inside(ix, iy, hw, hh, nc, nr)) {
                if (lane == 0) { atomicExch(assert_flag, 1); }
                st = KLT_INTERNAL_ASSERT;
                break;
            }
            const float ax = __double2float_rn(__dsub_rn((double)x1, (double)ix));
            const float ay = __double2float_rn(__dsub_rn((double)y1, (double)iy));
            for (int k = lane; k < n; k += 32) {
                const int j = k / A.w, i = k - j * A.w;
                const size_t o = (size_t)(iy + j - hh) * pitch + (ix + i - hw);
                T[k] = bilerp_ref(I1 + o, pitch, ax, ay);
                Tgx[k] = bilerp_ref(GX1 + o, pitch, ax, ay);
                Tgy[k] = bilerp_ref(GY1 + o, pitch, ax, ay);
            }
        }
        __syncwarp();

        // ---- trackFeatureIterateCKLT (pyx:393-459), float32 state ----
        float x2 = __double2float_rn(xout), y2 = __double2float_rn(yout);
        int iteration = 0;
        const int status0 = iterate_exact(T, Tgx, Tgy, S, I2, GX2, GY2, pitch, nc, nr, A.w, A.h, A.step_factor, A.small_det, A.th,
                                          A.max_iterations, lane, x2, y2, iteration, A.lighting_insensitive != 0);
        int status = status0;
        my_iters += iteration;

        // ---- back in _trackFeature (trackFeatures.py:108-136) ----
        if (!lk_window_inside_d(x2, y2, A.w, A.h, nc, nr)) status = KLT_OOB;
        if (status == KLT_TRACKED && A.has_max_residue) {
            const int ix = (int)x2, iy = (int)y2;
            const float ax = __double2float_rn(__dsub_rn((double)x2, (double)ix));
            const float ay = __double2float_rn(__dsub_rn((double)y2, (double)iy));
            if (A.lighting_insensitive) {         // trackFeatures.py:120-121 (the callee is undefined in the reference)
                for (int k = lane; k < n; k += 32) {
                    const int j = k / A.w, i = k - j * A.w;
                    S[k] = bilerp_ref(I2 + (size_t)(iy + j - hh) * pitch + (ix + i - hw), pitch, ax, ay);
                }
                __syncwarp();
                const LiCoeffs c = li_coefficients(T, S, n, lane);
                for (int k = lane; k < n; k += 32) S[k] = fabsf(__fsub_rn(__fsub_rn(T[k], __fmul_rn(S[k], c.alpha)), c.belta));
            } else {
                for (int k = lane; k < n; k += 32) {
                    const int j = k / A.w, i = k - j * A.w;
                    const size_t o = (size_t)(iy + j - hh) * pitch + (ix + i - hw);
                    S[k] = fabsf(__fsub_rn(T[k], bilerp_ref(I2 + o, pitch, ax, ay)));
                }
            }
            __syncwarp();
            float res = 0.f;
            if (lane == 0) res = __fdiv_rn(np_pairwise_sum(S, n), (float)n);
            res = __shfl_sync(0xffffffffu, res, 0);
            if (res > A.max_residue) status = KLT_LARGE_RESIDUE;
            __syncwarp();
        }
        xout = (double)x2; yout = (double)y2;
        st = lk_level_verdict(A, status, iteration);
        if (lk_level_lost(st)) break;
    }
    if (lane == 0) lk_write_feature(A, f, st, xout, yout, my_iters, xs, ys, vals, iters_total);
}


// ---------------------------------------------------------------------------------------------------------------------
// FAST tracking kernel (used when the pyramids were built in KLT_PRECISION_FAST): same algorithm and status logic,
// float32 bilinear weights and shuffle reductions instead of the reference's exact operation order.
// Mapping: one LANE per window COLUMN, G = 8 (W <= 7) or 16 (W <= 15) lanes per feature, 32/G features per warp.
// A lane loads the W+1 source pixels of its column and of the column to its right once per patch (vertically adjacent
// samples share corners: 2.3 loads per sample instead of 4; the lanes of a feature touch one or two 32-byte sectors
// per source row), keeps its column of the three templates in registers, accumulates the five window sums over its
// column with FMAs, and the G lanes of a feature combine them with log2(G) shuffle steps.
// ---------------------------------------------------------------------------------------------------------------------
// Lane i of a feature's lane group owns window COLUMN i and lane W the extra right-hand column: each lane loads ONE value
// per source row (the group reads W+1 consecutive addresses: coalesced) and takes the right-hand neighbour of the
// bilinear footprint from the next lane by shuffle, which halves the L1 wavefronts of the naive 4-tap gather.  Every
// lane of the warp must call these (the shuffles are warp-wide); `ld` says whether this lane really loads.
template <int W>
__device__ __forceinline__ void patch_col(const float *__restrict__ img, int pitch, int ix, int iy, int i, bool ld,
                                          const Bilinear &w, float (&out)[W]) {
    const float *p = img + (ld ? (size_t)(iy - W / 2) * pitch + (ix - W / 2 + i) : 0);
    float a[W + 1], b[W + 1];
#pragma unroll
    for (int j = 0; j < W + 1; j++) a[j] = ld ? __ldg(p + (size_t)j * pitch) : 0.f;
#pragma unroll
    for (int j = 0; j < W + 1; j++) b[j] = __shfl_down_sync(0xffffffffu, a[j], 1);
#pragma unroll
    for (int j = 0; j < W; j++) out[j] = w(a[j], b[j], a[j + 1], b[j + 1]);
}

// the three patches (image, gradx, grady) of one position: all 3*(W+1) loads are issued before the first use, so one
// memory round trip covers the whole phase
template <int W>
__device__ __forceinline__ void patch_col3(const float *__restrict__ i0, const float *__restrict__ i1,
                                           const float *__restrict__ i2, int pitch, int ix, int iy, int i, bool ld,
                                           const Bilinear &w, float (&o0)[W], float (&o1)[W], float (&o2)[W]) {
    const size_t off = ld ? (size_t)(iy - W / 2) * pitch + (ix - W / 2 + i) : 0;
    const float *p0 = i0 + off, *p1 = i1 + off, *p2 = i2 + off;
    float a0[W + 1], b0[W + 1], a1[W + 1], b1[W + 1], a2[W + 1], b2[W + 1];
#pragma unroll
    for (int j = 0; j < W + 1; j++) {
        const size_t r = (size_t)j * pitch;
        a0[j] = ld ? __ldg(p0 + r) : 0.f;
        a1[j] = ld ? __ldg(p1 + r) : 0.f;
        a2[j] = ld ? __ldg(p2 + r) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < W + 1; j++) {
        b0[j] = __shfl_down_sync(0xffffffffu, a0[j], 1);
        b1[j] = __shfl_down_sync(0xffffffffu, a1[j], 1);
        b2[j] = __shfl_down_sync(0xffffffffu, a2[j], 1);
    }
#pragma unroll
    for (int j = 0; j < W; j++) {
        o0[j] = w(a0[j], b0[j], a0[j + 1], b0[j + 1]);
        o1[j] = w(a1[j], b1[j], a1[j + 1], b1[j + 1]);
        o2[j] = w(a2[j], b2[j], a2[j + 1], b2[j + 1]);
    }
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = 1; o < G; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int W>
__global__ void __launch_bounds__(128)
lk_track_rows_kernel(const __grid_constant__ TrackArgs A, double *__restrict__ xs, double *__restrict__ ys,
                     int *__restrict__ vals, unsigned long long *__restrict__ iters_total, int *__restrict__ assert_flag) {
    constexpr int G = W <= 7 ? 8 : 16;
    constexpr int FPW = 32 / G;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = A.f_begin + (blockIdx.x * (blockDim.x >> 5) + warp) * FPW + lane / G;
    const int j = lane % G;                       // window column handled by this lane
    const bool row_ok = j < W;                    // lane owns a window column
    const bool col_ld = j <= W;                   // lane loads a source column (lane W: the right-hand extra one)
    bool alive = f < A.total;
    if (alive) alive = vals[f] >= 0;              // trackFeatures.py:253
    if (!__any_sync(0xffffffffu, alive)) return;
    const int image = alive ? f / A.n_per_image : 0;
    constexpr int hw = W / 2;
    const double ss = (double)A.ss;
    double xloc = alive ? xs[f] : 0.0, yloc = alive ? ys[f] : 0.0;
    lk_top_level(xloc, yloc, A.n_levels, ss);
    double xout = xloc, yout = yloc;
    int st = KLT_TRACKED;
    unsigned int my_iters = 0;
    const bool was_alive = alive;

    for (int r = A.n_levels - 1; r >= 0; r--) {
        xloc *= ss; yloc *= ss; xout *= ss; yout *= ss;
        const int nc = A.p1.lv[r].w, nr = A.p1.lv[r].h, pitch = A.p1.lv[r].pitch;
        const float *I1 = A.p1.level(0, image, r), *GX1 = A.p1.level(1, image, r), *GY1 = A.p1.level(2, image, r);
        const float *I2 = A.p2.level(0, image, r), *GX2 = A.p2.level(1, image, r), *GY2 = A.p2.level(2, image, r);
        float T[W], Tgx[W], Tgy[W];
        {
            const float x1 = (float)xloc, y1 = (float)yloc;
            const int ix = (int)x1, iy = (int)y1;
            if (alive && !lk_template_inside(ix, iy, hw, hw, nc, nr)) {
                if (j == 0) atomicExch(assert_flag, 1);
                st = KLT_INTERNAL_ASSERT;
                alive = false;
            }
            patch_col3<W>(I1, GX1, GY1, pitch, ix, iy, j, alive && col_ld, Bilinear(x1 - (float)ix, y1 - (float)iy), T, Tgx,
                          Tgy);
            if (!(alive && row_ok)) {
#pragma unroll
                for (int i = 0; i < W; i++) { T[i] = 0.f; Tgx[i] = 0.f; Tgy[i] = 0.f; }
            }
        }
        float x2 = (float)xout, y2 = (float)yout;
        int status = KLT_TRACKED, iteration = 0;
        const float fnc = (float)nc, fnr = (float)nr, fhw = (float)hw;
        bool iterating = alive;
        while (__any_sync(0xffffffffu, iterating)) {
            if (iterating && !lk_window_inside_f(x2, y2, fhw, fhw, fnc, fnr)) {
                status = KLT_OOB;
                iterating = false;
            }
            float gxx = 0.f, gxy = 0.f, gyy = 0.f, ex = 0.f, ey = 0.f;
            {
                const int ix = (int)x2, iy = (int)y2;
                float P[W], Px[W], Py[W];
                patch_col3<W>(I2, GX2, GY2, pitch, ix, iy, j, iterating && col_ld, Bilinear(x2 - (float)ix, y2 - (float)iy), P,
                              Px, Py);
                if (iterating && row_ok) {
#pragma unroll
                    for (int i = 0; i < W; i++) {
                        const float diff = T[i] - P[i], gx = Tgx[i] + Px[i], gy = Tgy[i] + Py[i];
                        gxx = fmaf(gx, gx, gxx); gxy = fmaf(gx, gy, gxy); gyy = fmaf(gy, gy, gyy);
                        ex = fmaf(diff, gx, ex); ey = fmaf(diff, gy, ey);
                    }
                }
            }
            gxx = group_sum<G>(gxx); gxy = group_sum<G>(gxy); gyy = group_sum<G>(gyy);
            ex = group_sum<G>(ex) * A.step_factor; ey = group_sum<G>(ey) * A.step_factor;
            if (iterating) {
                const float det = __fsub_rn(__fmul_rn(gxx, gyy), __fmul_rn(gxy, gxy));
                if (det < A.small_det) {
                    status = KLT_SMALL_DET;
                    iterating = false;
                } else {
                    const float dx = __fdiv_rn(__fsub_rn(__fmul_rn(gyy, ex), __fmul_rn(gxy, ey)), det);
                    const float dy = __fdiv_rn(__fsub_rn(__fmul_rn(gxx, ey), __fmul_rn(gxy, ex)), det);
                    x2 += dx; y2 += dy;
                    iteration++;
                    if (!((fabsf(dx) >= A.th || fabsf(dy) >= A.th) && iteration < A.max_iterations)) iterating = false;
                }
            }
        }
        my_iters += iteration;
        if (alive && !lk_window_inside_d(x2, y2, W, W, nc, nr)) status = KLT_OOB;
        const bool need_res = alive && status == KLT_TRACKED && A.has_max_residue;
        if (__any_sync(0xffffffffu, need_res)) {
            float res = 0.f;
            {
                const int ix = (int)x2, iy = (int)y2;
                float P[W];
                patch_col<W>(I2, pitch, ix, iy, j, need_res && col_ld, Bilinear(x2 - (float)ix, y2 - (float)iy), P);
                if (need_res && row_ok) {
#pragma unroll
                    for (int i = 0; i < W; i++) res += fabsf(T[i] - P[i]);
                }
            }
            res = group_sum<G>(res) / (float)(W * W);
            if (need_res && res > A.max_residue) status = KLT_LARGE_RESIDUE;
        }
        if (alive) {
            xout = (double)x2; yout = (double)y2;
            st = lk_level_verdict(A, status, iteration);
            if (lk_level_lost(st)) alive = false;
        }
    }
    if (was_alive && j == 0) lk_write_feature(A, f, st, xout, yout, my_iters, xs, ys, vals, iters_total);
}

template <int W>
static int launch_rows(klt_ctx *ctx, const TrackArgs &A, double *x, double *y, int32_t *v, unsigned long long *it, int *af) {
    constexpr int FPW = 32 / (W <= 7 ? 8 : 16);
    const int per_block = 4 * FPW;
    const int blocks = (A.total - A.f_begin + per_block - 1) / per_block;
    KLT_LAUNCH(ctx, "lk_track_rows", 0.0, (lk_track_rows_kernel<W><<<blocks, 128, 0, ctx->stream>>>(A, x, y, v, it, af)));
    return KLT_OK;
}

int klt_launch_track(klt_ctx *ctx, const klt_params *p, const klt_pyr *p1, const klt_pyr *p2, int n_per_image,
                     double *x_dev, double *y_dev, int32_t *val_dev, unsigned long long *iters_dev, int *assert_dev,
                     int first_image, int n_images, int assert_marks_feature) {
    // bit-exact arithmetic only pays off on bit-exact (STRICT) pyramids
    const bool exact = p1->precision == KLT_PRECISION_STRICT && p2->precision == KLT_PRECISION_STRICT;
    TrackArgs A;
    A.assert_marks_feature = assert_marks_feature;
    A.p1 = *p1; A.p2 = *p2;
    A.w = p->window_width; A.h = p->window_height;
    A.n_levels = p->n_levels; A.ss = p->subsampling;
    A.max_iterations = p->max_iterations;
    A.small_det = p->min_determinant; A.th = p->min_displacement; A.step_factor = p->step_factor;
    A.has_max_residue = p->has_max_residue; A.max_residue = p->max_residue;
    A.retain = p->retain_trackers;
    A.borderx = p->borderx; A.bordery = p->bordery;
    if (n_images < 0) n_images = p1->batch - first_image;
    A.n_per_image = n_per_image; A.f_begin = n_per_image * first_image; A.total = n_per_image * (first_image + n_images);
    A.lighting_insensitive = p->lighting_insensitive ? 1 : 0;
    if (A.total <= A.f_begin) return KLT_OK;
    // image-only pyramids (FAST_WINDOWED builds): gradients are evaluated inside the tracking windows
    if (!A.lighting_insensitive && (!klt_pyr_has_gradients(p1) || !klt_pyr_has_gradients(p2))) {
        if (!klt_windowed_supported(p, p1, p2))
            return klt_fail(ctx, KLT_ERR_INVALID, "image-only pyramid reached the plane-based tracker (internal error)");
        return klt_launch_track_windowed(ctx, A, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
    }
    if (!exact && A.w == A.h && !A.lighting_insensitive) {   // FAST pyramids: float32 row-per-lane kernel for the common window sizes
        switch (A.w) {
            case 3: return launch_rows<3>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            case 5: return launch_rows<5>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            case 7: return launch_rows<7>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            case 9: return launch_rows<9>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            case 11: return launch_rows<11>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            case 13: return launch_rows<13>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            case 15: return launch_rows<15>(ctx, A, x_dev, y_dev, val_dev, iters_dev, assert_dev);
            default: break;               // larger windows: the generic (exact-order) kernel below
        }
    }
    const int n = A.w * A.h;
    int warps = 4;
    size_t smem = (size_t)warps * 8 * n * sizeof(float);
    while (smem > 200 * 1024 && warps > 1) { warps /= 2; smem = (size_t)warps * 8 * n * sizeof(float); }
    if (smem > 200 * 1024) return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "tracking window %dx%d too large", A.w, A.h);
    KLT_CUDA(ctx, cudaFuncSetAttribute(lk_track_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    const int blocks = (A.total - A.f_begin + warps - 1) / warps;
    KLT_LAUNCH(ctx, "lk_track", 0.0, (lk_track_kernel<<<blocks, warps * 32, smem, ctx->stream>>>(A, x_dev, y_dev, val_dev, iters_dev, assert_dev)));
    return KLT_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Forward-backward check (Kalal, Mikolajczyk, Matas, ICPR 2010; no counterpart in the reference or in C-KLT).  The backward
// pass is an ordinary klt_launch_track with the two pyramids swapped; these two element-wise kernels surround it.
// ---------------------------------------------------------------------------------------------------------------------
// the forward result becomes the backward pass's input (features the forward pass lost keep val < 0: the tracker skips them)
__global__ void fb_prepare_kernel(int total, const double *__restrict__ x, const double *__restrict__ y,
                                  const int32_t *__restrict__ val, double *__restrict__ xb, double *__restrict__ yb,
                                  int32_t *__restrict__ vb) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total) return;
    xb[f] = x[f]; yb[f] = y[f]; vb[f] = val[f];
}

// decision: a forward-tracked feature whose backward track was lost, or came back farther than max_fb_error from where it
// started, becomes (-1, -1, KLT_FB_ERROR).  e = sqrt(dx*dx + dy*dy) in double without FMA (NumPy's result bit for bit).
__global__ void fb_check_kernel(int total, float max_fb_error, const double *__restrict__ x0, const double *__restrict__ y0,
                                const double *__restrict__ xb, const double *__restrict__ yb, const int32_t *__restrict__ vb,
                                double *__restrict__ x, double *__restrict__ y, int32_t *__restrict__ val,
                                float *__restrict__ fb_error) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total) return;
    float fe = -1.f;
    if (val[f] == KLT_TRACKED) {
        bool reject = true;
        if (vb[f] == KLT_TRACKED) {
            const double dx = __dsub_rn(xb[f], x0[f]), dy = __dsub_rn(yb[f], y0[f]);
            const double e = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
            fe = (float)e;
            reject = !(e <= (double)max_fb_error);
        }
        if (reject) { x[f] = -1.0; y[f] = -1.0; val[f] = KLT_FB_ERROR; }
    }
    if (fb_error) fb_error[f] = fe;
}

int klt_launch_track_fb(klt_ctx *ctx, const klt_params *p, const klt_pyr *p1, const klt_pyr *p2, int n_per_image,
                        float max_fb_error, double *x, double *y, int32_t *val, const FbArrays &fa, float *fb_error,
                        unsigned long long *iters_dev, int *assert_dev) {
    const int total = n_per_image * p1->batch;
    if (total <= 0) return KLT_OK;
    const int blocks = (total + 255) / 256;
    int rc;
    // (x0, y0): the start positions, which the forward track overwrites
    KLT_CUDA(ctx, cudaMemcpyAsync(fa.x0, x, total * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(fa.y0, y, total * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    if ((rc = klt_launch_track(ctx, p, p1, p2, n_per_image, x, y, val, iters_dev, assert_dev))) return rc;
    KLT_LAUNCH(ctx, "fb_prepare", 36.0 * total,
               (fb_prepare_kernel<<<blocks, 256, 0, ctx->stream>>>(total, x, y, val, fa.xb, fa.yb, fa.vb)));
    if ((rc = klt_launch_track(ctx, p, p2, p1, n_per_image, fa.xb, fa.yb, fa.vb, iters_dev, fa.scratch_assert, 0, -1, 1))) return rc;
    KLT_LAUNCH(ctx, "fb_check", 76.0 * total,
               (fb_check_kernel<<<blocks, 256, 0, ctx->stream>>>(total, max_fb_error, fa.x0, fa.y0, fa.xb, fa.yb, fa.vb, x, y, val,
                                                                 fb_error)));
    return KLT_OK;
}

// trackFeaturesUtils.extractImagePatchSlow (pyx:14-18) for operator-level parity tests.
__global__ void extract_patch_kernel(const float *__restrict__ img, int pitch, int nc, int nr, float x, float y,
                                     int height, int width, float *__restrict__ out, int *__restrict__ ok) {
    const int ix = (int)x, iy = (int)y, hw = width / 2, hh = height / 2;
    if (!lk_template_inside(ix, iy, hw, hh, nc, nr)) {
        if (threadIdx.x == 0) *ok = 0;
        return;
    }
    if (threadIdx.x == 0) *ok = 1;
    const float ax = __double2float_rn(__dsub_rn((double)x, (double)ix));
    const float ay = __double2float_rn(__dsub_rn((double)y, (double)iy));
    for (int k = threadIdx.x; k < width * height; k += blockDim.x) {
        const int j = k / width, i = k - j * width;
        out[k] = bilerp_ref(img + (size_t)(iy + j - hh) * pitch + (ix + i - hw), pitch, ax, ay);
    }
}

// Operator-level entry: trackFeaturesUtils.trackFeatureIterateCKLT on caller-provided template patches (one warp).
__global__ void __launch_bounds__(32)
lk_iterate_kernel(const float *__restrict__ tpatch /* [3][h*w]: img, gx, gy */, const float *__restrict__ img2,
                  const float *__restrict__ gx2, const float *__restrict__ gy2, int pitch, int nc, int nr, int w, int h,
                  float step_factor, float small_det, float th, int max_iterations, float x2, float y2, float *out /* x2,y2,status,iteration */) {
    extern __shared__ float smem[];
    const int lane = threadIdx.x, n = w * h;
    float *T = smem, *Tgx = T + n, *Tgy = T + 2 * n, *S = T + 3 * n;
    for (int k = lane; k < 3 * n; k += 32) T[k] = tpatch[k];
    __syncwarp();
    int iteration = 0;
    const int status = iterate_exact(T, Tgx, Tgy, S, img2, gx2, gy2, pitch, nc, nr, w, h, step_factor, small_det, th,
                                     max_iterations, lane, x2, y2, iteration);
    if (lane == 0) { out[0] = x2; out[1] = y2; out[2] = (float)status; out[3] = (float)iteration; }
}

int klt_launch_iterate(klt_ctx *ctx, const klt_params *p, const float *tpatch_dev, const float *img2, const float *gx2,
                       const float *gy2, int w_img, int h_img, float x2, float y2, float *out_dev) {
    const int n = p->window_width * p->window_height;
    const size_t smem = (size_t)8 * n * sizeof(float);
    if (smem > 200 * 1024) return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "window too large");
    KLT_CUDA(ctx, cudaFuncSetAttribute(lk_iterate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    KLT_LAUNCH(ctx, "lk_iterate", 0.0, (lk_iterate_kernel<<<1, 32, smem, ctx->stream>>>(tpatch_dev, img2, gx2, gy2, w_img, w_img, h_img,
                                                                                      p->window_width, p->window_height, p->step_factor,
                                                                                      p->min_determinant, p->min_displacement,
                                                                                      p->max_iterations, x2, y2, out_dev)));
    return KLT_OK;
}

// computeIntensityDifference (mode 0: p1 - patch(img2)) / computeGradientSum (mode 1: -p1 - patch(img2)), pyx:61-142
__global__ void patch_combine_kernel(const float *__restrict__ p1, const float *__restrict__ img, int pitch, int nc, int nr,
                                     float x, float y, int height, int width, int mode, float *__restrict__ out, int *__restrict__ ok) {
    const int ix = (int)x, iy = (int)y, hw = width / 2, hh = height / 2;
    if (!lk_template_inside(ix, iy, hw, hh, nc, nr)) {
        if (threadIdx.x == 0) *ok = 0;
        return;
    }
    if (threadIdx.x == 0) *ok = 1;
    const float ax = __double2float_rn(__dsub_rn((double)x, (double)ix));
    const float ay = __double2float_rn(__dsub_rn((double)y, (double)iy));
    for (int k = threadIdx.x; k < width * height; k += blockDim.x) {
        const int j = k / width, i = k - j * width;
        const float g2 = bilerp_ref(img + (size_t)(iy + j - hh) * pitch + (ix + i - hw), pitch, ax, ay);
        out[k] = mode == 0 ? __fsub_rn(p1[k], g2) : __fsub_rn(-p1[k], g2);
    }
}

int klt_launch_patch_combine(klt_ctx *ctx, const float *p1_dev, const float *img, int w, int h, float x, float y, int height,
                             int width, int mode, float *out_dev, int *ok_dev) {
    KLT_LAUNCH(ctx, "patch_combine", 0.0, (patch_combine_kernel<<<1, 128, 0, ctx->stream>>>(p1_dev, img, w, w, h, x, y, height, width, mode, out_dev, ok_dev)));
    return KLT_OK;
}

int klt_launch_extract_patch(klt_ctx *ctx, const float *img, size_t pitch, int w, int h, float x, float y, int height,
                             int width, float *out_dev, int *ok_dev) {
    extract_patch_kernel<<<1, 128, 0, ctx->stream>>>(img, (int)pitch, w, h, x, y, height, width, out_dev, ok_dev);
    KLT_CHECK_LAUNCH(ctx);
    return KLT_OK;
}
