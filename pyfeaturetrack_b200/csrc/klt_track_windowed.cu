// Pyramidal Lucas-Kanade on IMAGE-ONLY pyramids (KLT_PRECISION_FAST_WINDOWED, the default tracker).
// Replaces the `KLTTrackFeatures` loop (trackFeatures.py:205-409: `_trackFeature` :56-149, `trackFeatureIterateCKLT`
// trackFeaturesUtils.pyx:393-459) together with `_KLTComputeGradients` (trackFeatures.py:171-176, convolve.py:245-246):
// the gradient planes of the reference are never written to HBM.  A tracked feature only ever reads gradients inside its
// (W+1)^2 window -- ~3 % of a 1080p frame for 1000 features -- so the 7-tap separable gradient pair is evaluated just for
// the pixels a feature's window visits, from regions of the smoothed images staged in shared memory; every bilinear sample
// of the Newton loop reads shared memory (one global round trip per level instead of one per Newton step); when the window
// moves to another integer position the second image's gradients are re-evaluated there (0.2 times per level on the
// benchmark), and when it walks out of the staged region that is re-staged around the current position.
// Arithmetic: float32 FMA, tolerances of KLT_PRECISION_FAST (positions agree with the dense FAST path to ~1e-5 px); STRICT
// pyramids never come here.  Mapping onto the machine (second generation; the first -- one feature per warp, `cp.async`
// element staging, 1 330 warp instructions per feature and level against 850 here -- is in the history):
//
//   * TWO features per warp for windows up to 7x7 (one half-warp each; one per warp for larger windows): the per-level
//     scalar work (coordinates, bounds, staging decisions, the 2x2 solve) is issued once for both, which is where the
//     first generation spent 40 % of its issue slots;
//   * staging by TMA: an elected lane of each feature issues ONE `cp.async.bulk.tensor.3d` box per image and level
//     (tensor maps over [image][row][column] of every pyramid level, 16-byte aligned start column, completion on a
//     per-feature mbarrier) and one
//     `cp.async.bulk.prefetch.tensor` per image for the next level's regions.  Regions that cross the image border need
//     SciPy's 'reflect' indices (TMA can only zero-fill) and take a `cp.async` element path into the same layout;
//   * a TMA box lands densely (pitch = box width), so the separable gradient pair runs VERTICAL pass first with one region
//     COLUMN per lane (consecutive lanes, consecutive banks, any pitch), then the horizontal pass with one (plane, row)
//     per lane on an odd-pitch intermediate: no bank conflicts in either pass;
//   * window pixels map to lanes by rows (LPR lanes per window row), so every shared-memory offset of the Newton loop is
//     an immediate.
//
// gx = deriv_h(gauss_v(img)), gy = gauss_h(deriv_v(img)): the same separable products as convolve.py:245-246 with the
// two 1-D passes in the other order (they commute; float32 rounding differs in the last bit).
#include <cuda.h>

#include "klt_common.cuh"
#include "klt_track_args.cuh"

namespace {

constexpr int RG = 3;      // gradient kernel radius served here (grad_sigma = 1.0: 7 taps)
constexpr int MARGIN = 2;  // pixels of slack around the start window of the second image
constexpr unsigned FULL = 0xffffffffu;

struct alignas(64) WindowedMaps {
    CUtensorMap m1[KLT_MAX_LEVELS], m2[KLT_MAX_LEVELS];   // first / second pyramid, one map per level
};

template <int W>
struct Cfg2 {
    static constexpr int FPW = W <= 7 ? 2 : 1;              // features per warp
    static constexpr int LPF = 32 / FPW;                    // lanes per feature
    static constexpr int S = W + 1;                         // gradient footprint of a window (bilinear taps)
    static constexpr int NG = S + 2 * RG;                   // smoothed-image rows / columns that footprint needs
    static constexpr int N1 = NG, N2 = NG + 2 * MARGIN;     // staged regions (rows = columns) of image 1 / image 2
    // TMA boxes: the inner extent is a multiple of 16 bytes AND the start column must be 16-byte aligned (an unaligned start
    // coordinate is an illegal instruction: tools/tma_probe2.cu), so a box starts at the region's column rounded down to a
    // multiple of 4 and is 3 columns wider; the region then sits at column offset (start & 3) of the staged rows
    static constexpr int P1 = (N1 + 3 + 3) & ~3, P2 = (N2 + 3 + 3) & ~3;   // box widths = shared-memory pitches
    static constexpr int LPR = W <= 4 ? 4 : (W <= 8 ? 8 : 16);      // lanes per window row
    static constexpr int RPR = LPF / LPR;                   // window rows per round
    static constexpr int PX = (W + RPR - 1) / RPR;          // rounds = window pixels per lane
    static constexpr int TP = NG | 1;                       // intermediate planes [feature][gauss_v, deriv_v][S rows], odd pitch:
                                                            // row-per-lane walks of up to 32 rows hit 32 different banks
    static constexpr int GP = S | 1;                        // gradient planes: (gx, gy) PAIRS per row, odd
    static constexpr int r32(int n) { return (n + 31) & ~31; }
    static constexpr int IN1SZ = r32(N1 * P1), IN2SZ = r32(N2 * P2);     // TMA destinations: 128-byte aligned
    static constexpr int GSZ0 = 2 * S * GP;
    static constexpr int GSZ = FPW == 2 ? GSZ0 + ((16 - GSZ0 % 32) + 32) % 32 : r32(GSZ0);   // two features: 16 banks apart
    static constexpr int IN1 = 0, IN2 = IN1 + FPW * IN1SZ;
    static constexpr int T = IN2 + FPW * IN2SZ, TSZ = FPW * 2 * S * TP;
    static constexpr int G2 = r32(T + TSZ), G1 = G2 + FPW * GSZ;
    static constexpr int MB = r32(G1 + FPW * GSZ);          // one mbarrier (8 bytes) per feature
    static constexpr int FLOATS = MB + 32;
    static constexpr unsigned BYTES1 = (unsigned)(N1 * P1 * 4), BYTES2 = (unsigned)(N2 * P2 * 4);
    static_assert(NG <= LPF && 2 * S <= LPF, "a region column / a (plane, row) task per lane");
    static_assert(GSZ % 2 == 0 && G2 % 2 == 0, "64-bit gradient taps");
};

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async4(float *smem_dst, const float *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void mbar_init(unsigned mb, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mb), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned mb, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mb, unsigned parity) {
    unsigned ok = 0;
    for (int spin = 0; !ok; spin++) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(mb), "r"(parity) : "memory");
        if (spin > (1 << 22)) __trap();          // a lost TMA completion becomes a CUDA error, not a hang
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap *map, int x, int y, int z, unsigned mb) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(dst), "l"(reinterpret_cast<unsigned long long>(map)), "r"(x), "r"(y), "r"(z), "r"(mb) : "memory");
}
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap *map, int x, int y, int z) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];"
                 ::"l"(reinterpret_cast<unsigned long long>(map)), "r"(x), "r"(y), "r"(z) : "memory");
}

// element path for a region that crosses the image border (SciPy 'reflect'); LPF lanes of one feature
template <int N, int P, int LPF>
__device__ __forceinline__ void stage_reflect(float *__restrict__ dst, const float *__restrict__ img, int pitch, int nc, int nr,
                                              int sx0, int sy0, int q) {
#pragma unroll 1
    for (int idx = q; idx < N * N; idx += LPF) {
        const int ry = idx / N, rx = idx - ry * N;
        cp_async4(dst + ry * P + rx, img + (size_t)klt_reflect(sy0 + ry, nr) * pitch + klt_reflect(sx0 + rx, nc));
    }
}

__device__ __forceinline__ float bil(const float *p, int P, const Bilinear &w) { return w(p[0], p[1], p[P], p[P + 1]); }
// bilinear sample of an interleaved (gx, gy) plane: four 64-bit loads for both gradients; P = pitch in pairs
__device__ __forceinline__ float2 bil2(const float *p, int P, const Bilinear &w) {
    const float2 a = *reinterpret_cast<const float2 *>(p), b = *reinterpret_cast<const float2 *>(p + 2);
    const float2 c = *reinterpret_cast<const float2 *>(p + 2 * P), d = *reinterpret_cast<const float2 *>(p + 2 * P + 2);
    return make_float2(w(a.x, b.x, c.x, d.x), w(a.y, b.y, c.y, d.y));
}

// sum over the LPF lanes of a feature, result in every lane of the group.  Not lk_track_rows' group_sum: that one
// pairs the lanes in the opposite order, and the order is part of the rounded result.
template <int LPF>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = LPF / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
// Five group-wide sums at once: after the first exchange the lower half of the group owns a, b, c and the upper one d, e;
// after the second each quarter owns one of a, b, d, e (c rides along on the lower half); plain butterfly rounds finish
// them and five broadcasts hand the totals to every lane (16 shuffles for 32 lanes instead of 25, 14 instead of 20 for 16).
template <int LPF>
__device__ __forceinline__ void group_sum5(float &a, float &b, float &c, float &d, float &e, int q) {
    constexpr int H1 = LPF / 2, H2 = LPF / 4;
    const bool up1 = (q & H1) != 0, up2 = (q & H2) != 0;
    const float t0 = __shfl_xor_sync(FULL, up1 ? a : d, H1);
    const float t1 = __shfl_xor_sync(FULL, up1 ? b : e, H1);
    const float t2 = __shfl_xor_sync(FULL, up1 ? c : 0.f, H1);
    const float A = (up1 ? d : a) + t0, B = (up1 ? e : b) + t1;
    float Cc = up1 ? 0.f : c + t2;
    float X = (up2 ? B : A) + __shfl_xor_sync(FULL, up2 ? A : B, H2);
    Cc += __shfl_xor_sync(FULL, Cc, H2);
#pragma unroll
    for (int o = H2 / 2; o > 0; o >>= 1) { X += __shfl_xor_sync(FULL, X, o); Cc += __shfl_xor_sync(FULL, Cc, o); }
    a = __shfl_sync(FULL, X, 0, LPF); b = __shfl_sync(FULL, X, H2, LPF); d = __shfl_sync(FULL, X, H1, LPF);
    e = __shfl_sync(FULL, X, H1 + H2, LPF);
    c = __shfl_sync(FULL, Cc, 0, LPF);
}

// Gradient pair of ONE image for the features of this warp whose `on` is set (warp-uniform call, `on` uniform per feature).
//   in:   top-left input pixel of the NG x NG neighbourhood of the footprint, pitch P
//   tpl:  this feature's intermediate planes [2][S][TP];  gdst: this feature's (gx, gy) plane, GP pairs per row
//   g, d: gauss / derivative taps (constant bank);  th: this lane's horizontal taps (plane 0 = gx: d, plane 1 = gy: g)
template <int W, int P>
__device__ __forceinline__ void gradient_pair(const float *__restrict__ in, float *__restrict__ tpl, float *__restrict__ gdst,
                                              bool on, const float (&g)[7], const float (&d)[7], const float (&th)[7], int q) {
    using C = Cfg2<W>;
    if (on && q < C::NG) {                          // vertical pass: one region column per lane, both kernels
        float v[C::NG];
#pragma unroll
        for (int i = 0; i < C::NG; i++) v[i] = in[i * P + q];
#pragma unroll
        for (int j = 0; j < C::S; j++) {
            float tg = g[0] * v[j], td = d[0] * v[j];
#pragma unroll
            for (int k = 1; k < 7; k++) { tg = fmaf(g[k], v[j + k], tg); td = fmaf(d[k], v[j + k], td); }
            tpl[j * C::TP + q] = tg;
            tpl[(C::S + j) * C::TP + q] = td;
        }
    }
    __syncwarp();
    if (on && q < 2 * C::S) {                       // horizontal pass: lane q = (plane, row) = row q of the [2 S][TP] planes
        const int p = q / C::S, j = q - p * C::S;
        const float *row = tpl + q * C::TP;
        float v[C::NG];
#pragma unroll
        for (int i = 0; i < C::NG; i++) v[i] = row[i];
        float *o = gdst + 2 * j * C::GP + p;
#pragma unroll
        for (int c = 0; c < C::S; c++) {
            float acc = th[0] * v[c];
#pragma unroll
            for (int k = 1; k < 7; k++) acc = fmaf(th[k], v[c + k], acc);
            o[2 * c] = acc;
        }
    }
    __syncwarp();
}

// NW warps per CTA (2: see launch_windowed)
template <int W, int MINB, int NW>
__global__ void __launch_bounds__(NW * 32, MINB)
lk_windowed_kernel(const __grid_constant__ TrackArgs A, const __grid_constant__ WindowedTaps K,
                    const __grid_constant__ WindowedMaps M, double *__restrict__ xs, double *__restrict__ ys,
                    int *__restrict__ vals, unsigned long long *__restrict__ iters_total, int *__restrict__ assert_flag) {
    using C = Cfg2<W>;
    extern __shared__ __align__(128) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int h = lane / C::LPF, q = lane % C::LPF;            // feature slot of the warp, lane inside the feature
    const int f = A.f_begin + (blockIdx.x * NW + warp) * C::FPW + h;
    bool alive = f < A.total;
    if (alive) alive = vals[f] >= 0;                           // trackFeatures.py:253
    if (!__any_sync(FULL, alive)) return;
    const bool was_alive = alive;
    float *const s = smem + warp * C::FLOATS;
    float *const in1 = s + C::IN1 + h * C::IN1SZ, *const in2 = s + C::IN2 + h * C::IN2SZ;
    float *const tpl = s + C::T + h * (2 * C::S * C::TP);
    float *const g2 = s + C::G2 + h * C::GSZ, *const g1 = s + C::G1 + h * C::GSZ;
    const unsigned mb = smem_u32(s + C::MB + 2 * h);
    unsigned phase = 0;
    if (q == 0) mbar_init(mb, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fence_proxy_async();
    __syncwarp();

    const int image = alive ? f / A.n_per_image : 0;
    const float *const plane1 = A.p1.base + (size_t)image * A.p1.plane_floats;      // intensity planes of this feature's pair
    const float *const plane2 = A.p2.base + (size_t)image * A.p2.plane_floats;
    constexpr int hw = W / 2;
    const double ss = (double)A.ss;
    double xloc = alive ? xs[f] : 0.0, yloc = alive ? ys[f] : 0.0;
    lk_top_level(xloc, yloc, A.n_levels, ss);
    double xout = xloc, yout = yloc;
    int st = KLT_TRACKED;
    unsigned int my_iters = 0;
    // this lane's taps of the horizontal pass: plane 0 (gx) takes the derivative kernel, plane 1 (gy) the Gaussian
    const bool same_taps = K.same != 0;
    const bool hp = (q / C::S) != 0;
    float th2[7];
#pragma unroll
    for (int k = 0; k < 7; k++) th2[k] = hp ? K.g2[k] : K.d2[k];
    // this lane's window pixels: rows RPR * i + rr, column pc
    const int rr = q / C::LPR, pc = q % C::LPR;
    const bool col_on = pc < W;
    const int po = 2 * (rr * C::GP + pc);                      // offset in a gradient plane (floats)

    for (int r = A.n_levels - 1; r >= 0; r--) {
        xloc *= ss; yloc *= ss; xout *= ss; yout *= ss;
        if (!__any_sync(FULL, alive)) continue;
        const int nc = A.p1.lv[r].w, nr = A.p1.lv[r].h, pitch = A.p1.lv[r].pitch;
        const float x1 = (float)xloc, y1 = (float)yloc;
        const int ix1 = (int)x1, iy1 = (int)y1;
        if (alive && !lk_template_inside(ix1, iy1, hw, hw, nc, nr)) {
            if (q == 0) atomicExch(assert_flag, 1);
            st = KLT_INTERNAL_ASSERT;
            alive = false;
        }
        float x2 = (float)xout, y2 = (float)yout;
        int status = KLT_TRACKED, iteration = 0;
        const float fnc = (float)nc, fnr = (float)nr, fhw = (float)hw;
        // (rx0, ry0): window position at offset (0, 0) of the staged region of the second image; the start window sits
        // MARGIN pixels inside.  (gix, giy): window position the gradients in shared memory belong to.
        int rx0 = (int)x2 - hw - MARGIN, ry0 = (int)y2 - hw - MARGIN;
        int gix = -0x40000000, giy = -0x40000000;
        const bool start_inside = alive && lk_window_inside_f(x2, y2, fhw, fhw, fnc, fnr);

        // ---- one memory round trip: both regions of this level (TMA boxes; 'reflect' regions by element) ----
        // issue(do1, do2): group-uniform flags; returns whether the group has to wait on its mbarrier
        const float *i1 = in1, *i2 = in2;          // staged regions: buffer + column offset of the aligned box
        auto issue = [&](bool do1, bool do2) -> bool {
            const int sx1 = ix1 - hw - RG, sy1 = iy1 - hw - RG, sx2 = rx0 - RG, sy2 = ry0 - RG;
            const bool t1 = do1 && sx1 >= 0 && sy1 >= 0 && sx1 + C::N1 <= nc && sy1 + C::N1 <= nr;
            const bool t2 = do2 && sx2 >= 0 && sy2 >= 0 && sx2 + C::N2 <= nc && sy2 + C::N2 <= nr;
            if (do1) i1 = in1 + (t1 ? (sx1 & 3) : 0);
            if (do2) i2 = in2 + (t2 ? (sx2 & 3) : 0);
            if (q == 0 && (t1 || t2)) {
                fence_proxy_async();                   // earlier generic-proxy reads of these buffers are ordered before the TMA writes
                mbar_expect_tx(mb, (t1 ? C::BYTES1 : 0u) + (t2 ? C::BYTES2 : 0u));
                if (t1) tma_load_3d(smem_u32(in1), &M.m1[r], sx1 & ~3, sy1, image, mb);
                if (t2) tma_load_3d(smem_u32(in2), &M.m2[r], sx2 & ~3, sy2, image, mb);
            }
            if (do1 && !t1) stage_reflect<C::N1, C::P1, C::LPF>(in1, plane1 + A.p1.lv[r].off, pitch, nc, nr, sx1, sy1, q);
            if (do2 && !t2) stage_reflect<C::N2, C::P2, C::LPF>(in2, plane2 + A.p2.lv[r].off, pitch, nc, nr, sx2, sy2, q);
            return t1 || t2;
        };
        auto arrive = [&](bool tma) {
            cp_async_wait_all();
            if (tma) { mbar_wait(mb, phase); phase ^= 1u; }
            __syncwarp();
        };
        const bool tma0 = issue(alive, start_inside);
        if (r > 0 && alive && q == 0) {
            // pull the next (finer) level's regions towards L2 while this level computes
            const float xn1 = (float)(xloc * ss), yn1 = (float)(yloc * ss);
            const float xn2 = (float)((double)x2 * ss), yn2 = (float)((double)y2 * ss);
            tma_prefetch_3d(&M.m2[r - 1], ((int)xn2 - hw - MARGIN - RG) & ~3, (int)yn2 - hw - MARGIN - RG, image);
            tma_prefetch_3d(&M.m1[r - 1], ((int)xn1 - hw - RG) & ~3, (int)yn1 - hw - RG, image);
        }
        arrive(tma0);

        // ---- gradients of both windows ----
        gradient_pair<W, C::P2>(i2 + MARGIN * C::P2 + MARGIN, tpl, g2, start_inside, K.g2, K.d2, th2, q);
        if (start_inside) { gix = (int)x2; giy = (int)y2; }
        if (same_taps) {
            gradient_pair<W, C::P1>(i1, tpl, g1, alive, K.g2, K.d2, th2, q);
        } else {
            float th1[7];
#pragma unroll
            for (int k = 0; k < 7; k++) th1[k] = hp ? K.g1[k] : K.d1[k];
            gradient_pair<W, C::P1>(i1, tpl, g1, alive, K.g1, K.d1, th1, q);
        }

        // ---- template: the first image's window, gradients interpolated like the image (trackFeatures.py:87-92) ----
        float T[C::PX], Tgx[C::PX], Tgy[C::PX];
        {
            const Bilinear w(x1 - (float)ix1, y1 - (float)iy1);
#pragma unroll
            for (int i = 0; i < C::PX; i++) {
                const bool on = alive && col_on && (C::RPR * i + rr < W);
                T[i] = 0.f; Tgx[i] = 0.f; Tgy[i] = 0.f;
                if (on) {
                    T[i] = bil(i1 + (C::RPR * i + rr + RG) * C::P1 + pc + RG, C::P1, w);
                    const float2 tg = bil2(g1 + po + 2 * C::RPR * i * C::GP, C::GP, w);
                    Tgx[i] = tg.x; Tgy[i] = tg.y;
                }
            }
        }

        // ---- Newton iterations (trackFeaturesUtils.pyx:393-459) ----
        int ox = MARGIN, oy = MARGIN;
        bool iterating = alive;
        for (;;) {
            if (iterating && !lk_window_inside_f(x2, y2, fhw, fhw, fnc, fnr)) {
                status = KLT_OOB;
                iterating = false;
            }
            if (!__any_sync(FULL, iterating)) break;
            const int ix = (int)x2, iy = (int)y2;
            const bool moved = iterating && (ix != gix || iy != giy);      // the window sits on another pixel: new gradients
            if (__any_sync(FULL, moved)) {
                if (moved) { ox = ix - hw - rx0; oy = iy - hw - ry0; }
                const bool left = moved && (ox < 0 || oy < 0 || ox > 2 * MARGIN || oy > 2 * MARGIN);   // it even left the staged region
                __syncwarp();
                if (__any_sync(FULL, left)) {
                    if (left) { rx0 = ix - hw - MARGIN; ry0 = iy - hw - MARGIN; ox = MARGIN; oy = MARGIN; }
                    arrive(issue(false, left));
                }
                gradient_pair<W, C::P2>(i2 + oy * C::P2 + ox, tpl, g2, moved, K.g2, K.d2, th2, q);
                if (moved) { gix = ix; giy = iy; }
            }
            const Bilinear w(x2 - (float)ix, y2 - (float)iy);
            const float *bi = i2 + (oy + rr + RG) * C::P2 + ox + pc + RG;
            float gxx = 0.f, gxy = 0.f, gyy = 0.f, ex = 0.f, ey = 0.f;
            if (iterating && col_on) {
#pragma unroll
                for (int i = 0; i < C::PX; i++) {
                    if (C::RPR * (i + 1) <= W || C::RPR * i + rr < W) {      // (compile-time true except in the last round)
                        const float Pv = bil(bi + C::RPR * i * C::P2, C::P2, w);
                        const float2 Pg = bil2(g2 + po + 2 * C::RPR * i * C::GP, C::GP, w);
                        const float diff = T[i] - Pv, gx = Tgx[i] + Pg.x, gy = Tgy[i] + Pg.y;
                        gxx = fmaf(gx, gx, gxx); gxy = fmaf(gx, gy, gxy); gyy = fmaf(gy, gy, gyy);
                        ex = fmaf(diff, gx, ex); ey = fmaf(diff, gy, ey);
                    }
                }
            }
            group_sum5<C::LPF>(gxx, gxy, gyy, ex, ey, q);
            if (iterating) {
                ex *= A.step_factor; ey *= A.step_factor;
                const float det = __fsub_rn(__fmul_rn(gxx, gyy), __fmul_rn(gxy, gxy));
                if (det < A.small_det) {
                    status = KLT_SMALL_DET;
                    iterating = false;
                } else {
                    const float inv = __frcp_rn(det);             // one reciprocal instead of two divisions (within 1 ulp of them)
                    const float dx = __fsub_rn(__fmul_rn(gyy, ex), __fmul_rn(gxy, ey)) * inv;
                    const float dy = __fsub_rn(__fmul_rn(gxx, ey), __fmul_rn(gxy, ex)) * inv;
                    x2 += dx; y2 += dy;
                    iteration++;
                    if (!((fabsf(dx) >= A.th || fabsf(dy) >= A.th) && iteration < A.max_iterations)) iterating = false;
                }
            }
        }
        my_iters += iteration;
        if (alive && !lk_window_inside_d(x2, y2, W, W, nc, nr)) status = KLT_OOB;
        const bool need_res = alive && status == KLT_TRACKED && A.has_max_residue;
        if (__any_sync(FULL, need_res)) {
            const int ix = (int)x2, iy = (int)y2;
            if (need_res) { ox = ix - hw - rx0; oy = iy - hw - ry0; }
            const bool left = need_res && (ox < 0 || oy < 0 || ox > 2 * MARGIN || oy > 2 * MARGIN);
            if (__any_sync(FULL, left)) {
                __syncwarp();
                if (left) { rx0 = ix - hw - MARGIN; ry0 = iy - hw - MARGIN; ox = MARGIN; oy = MARGIN; }
                arrive(issue(false, left));
            }
            const Bilinear w(x2 - (float)ix, y2 - (float)iy);
            const float *bi = i2 + (oy + rr + RG) * C::P2 + ox + pc + RG;
            float res = 0.f;
            if (need_res && col_on) {
#pragma unroll
                for (int i = 0; i < C::PX; i++)
                    if (C::RPR * (i + 1) <= W || C::RPR * i + rr < W)
                        res += fabsf(T[i] - bil(bi + C::RPR * i * C::P2, C::P2, w));
            }
            res = group_sum<C::LPF>(res) / (float)(W * W);
            if (need_res && res > A.max_residue) status = KLT_LARGE_RESIDUE;
        }
        __syncwarp();                              // all lanes are done with the regions before the next level overwrites them
        if (alive) {
            xout = (double)x2; yout = (double)y2;
            st = lk_level_verdict(A, status, iteration);
            if (lk_level_lost(st)) alive = false;
        }
    }
    if (was_alive && q == 0) lk_write_feature(A, f, st, xout, yout, my_iters, xs, ys, vals, iters_total);
}

// ---- host side: tensor maps ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// map over the intensity component of level l: dims (column, row, image), box (bw, bh, 1), zero fill outside
bool make_map(CUtensorMap *m, const klt_pyr *p, int l, int bw, int bh) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)p->lv[l].w, (cuuint64_t)p->lv[l].h, (cuuint64_t)p->batch};
    const cuuint64_t strides[2] = {(cuuint64_t)p->lv[l].pitch * 4, (cuuint64_t)p->plane_floats * 4};
    const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, 1};
    const cuuint32_t es[3] = {1, 1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)(p->base + p->lv[l].off), dims, strides, box, es,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int W>
int launch_windowed(klt_ctx *ctx, const TrackArgs &A, const WindowedTaps &K, const klt_pyr *p1, const klt_pyr *p2, double *x,
                    double *y, int32_t *v, unsigned long long *it, int *af) {
    using C = Cfg2<W>;
    WindowedMaps M;
    for (int l = 0; l < A.n_levels; l++)
        if (!make_map(&M.m1[l], p1, l, C::P1, C::N1) || !make_map(&M.m2[l], p2, l, C::P2, C::N2))
            return klt_fail(ctx, KLT_ERR_CUDA, "cuTensorMapEncodeTiled failed for pyramid level %d (driver without TMA support?)", l);
    const int nfeat = A.total - A.f_begin;
    // algorithmic bytes: the staged regions of both images on every level (restaging not counted) + the feature records
    const double bytes = (double)nfeat * (A.n_levels * 4.0 * (C::N1 * C::N1 + C::N2 * C::N2) + 40.0);
    constexpr int MINB = W <= 7 ? 5 : 3;
    // 2-warp CTAs at twice the CTAs per SM: the same resident warps, and finer CTAs shorten the tail of the grid.  4-warp CTAs
    // for large grids measured 220 against 216-217 us per 64 000 features on a B200 at 1000 W.
    const int blocks = (nfeat + 2 * C::FPW - 1) / (2 * C::FPW);
    const size_t smem = (size_t)2 * C::FLOATS * sizeof(float);
    KLT_LAUNCH(ctx, "lk_windowed", bytes, (lk_windowed_kernel<W, 2 * MINB, 2><<<blocks, 64, smem, ctx->stream>>>(A, K, M, x, y, v, it, af)));
    return KLT_OK;
}

bool radius3(const klt_kernel1d &k) { return k.n == 2 * RG + 1; }
void flip7(const klt_kernel1d &k, float *dst) { for (int j = 0; j < 7; j++) dst[j] = (float)k.taps[6 - j]; }

}  // namespace

bool klt_windowed_supported(const klt_params *p, const klt_pyr *p1, const klt_pyr *p2) {
    if (p1->precision == KLT_PRECISION_STRICT || p2->precision == KLT_PRECISION_STRICT) return false;
    if (p->window_width != p->window_height || (p->window_width & 1) == 0 || p->window_width < 3 || p->window_width > 15) return false;
    if (!p1->hx || !p2->hx || !p1->hx->taps_valid || !p2->hx->taps_valid) return false;
    return radius3(p1->hx->taps.grad_gauss) && radius3(p1->hx->taps.grad_deriv) && radius3(p2->hx->taps.grad_gauss) &&
           radius3(p2->hx->taps.grad_deriv);
}

int klt_launch_track_windowed(klt_ctx *ctx, const TrackArgs &A, const klt_pyr *p1, const klt_pyr *p2, double *x_dev,
                              double *y_dev, int32_t *val_dev, unsigned long long *iters_dev, int *assert_dev) {
    WindowedTaps K;
    flip7(p1->hx->taps.grad_gauss, K.g1); flip7(p1->hx->taps.grad_deriv, K.d1);
    flip7(p2->hx->taps.grad_gauss, K.g2); flip7(p2->hx->taps.grad_deriv, K.d2);
    K.same = 1;
    for (int j = 0; j < 7; j++) K.same = K.same && K.g1[j] == K.g2[j] && K.d1[j] == K.d2[j];
    switch (A.w) {
        case 3: return launch_windowed<3>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
        case 5: return launch_windowed<5>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
        case 7: return launch_windowed<7>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
        case 9: return launch_windowed<9>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
        case 11: return launch_windowed<11>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
        case 13: return launch_windowed<13>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
        case 15: return launch_windowed<15>(ctx, A, K, p1, p2, x_dev, y_dev, val_dev, iters_dev, assert_dev);
    }
    return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "windowed tracking: window %d not covered", A.w);
}
