// FAST eigenvalue map: gradients, window sums and the minimum eigenvalue from ONE pass over the level-0 image
// (north_star (2): "the per-pixel 2x2 gradient-matrix minimum-eigenvalue scan fused with the gradient pass").
//
// Replaces, for select="fast", KLTComputeGradients (convolve.py:226-248) + ScanImageForGoodFeatures
// (goodFeaturesUtils.pyx:35-73): the gradient planes and the three summed-area tables never exist.  Arithmetic is plain
// fp32 with direct window sums, so the values differ from the reference's SAT-rounded ones by the SAT's own rounding error
// (SURVEY 7.3: same feature SET for ~99.8 %, not the same slots) -- the mode is judged by set overlap and labelled as such.
//
// Shape: a block of 128 threads owns a strip of 128 columns of one image and marches down a row segment; a thread owns one
// column.  Per input row: (1) the row goes through a shared-memory line, every thread forms d_h(I) and g_h(I) from its 7
// neighbours; (2) the vertical 7-tap filters run as accumulate-and-shift FMAs in registers (no memory), yielding one row of
// gx, gy; (3) gx^2, gx*gy, gy^2 enter the vertical window sums, again accumulate-and-shift in registers; (4) the completed row
// of column sums goes through shared memory once for the horizontal window sum; (5) eigenvalue, map store, histogram.
// Compulsory traffic: 4 B/px read + 4 B/candidate written (the strict path moves 52 B/px).
#include "klt_common.cuh"
#include "klt_select.cuh"

#define FS_THREADS 128
#define FS_R 3                  // gradient kernel radius (grad_sigma = 1.0 -> 7 taps)
#define FS_PF 4                 // rows loaded ahead

struct FastTaps { float g[7], d[7]; };   // c[j] multiplies in[x + j - 3]

template <int HH>
__global__ void __launch_bounds__(FS_THREADS)
eigen_fast_kernel(const float *__restrict__ img0, size_t img_stride, size_t pitch, const __grid_constant__ SelDev S,
                  const __grid_constant__ FastTaps T, int rows_per_seg) {
    __shared__ float rowI[2][FS_THREADS];
    __shared__ float rowV[2][3][FS_THREADS];
    const int t = threadIdx.x, b = blockIdx.z;
    const int W = S.W, H = S.H, hw = S.hw;
    const int halo = FS_R + hw, span = FS_THREADS - 2 * halo;
    const int x = S.bx - halo + (int)blockIdx.x * span + t;            // this thread's column
    const int xr = klt_reflect(x, W);
    const float *img = img0 + (size_t)b * img_stride + xr;
    // candidate rows of this segment
    const int ys = S.by + (int)blockIdx.y * rows_per_seg, ye = min(ys + rows_per_seg, H - S.by);
    if (ys >= ye) return;
    const int ci = x - S.bx;
    const bool cand_col = t >= halo && t < FS_THREADS - halo && x < W - S.bx && (ci % S.step) == 0;
    const int i_c = ci / S.step;
    float *vmap = S.vmap + (size_t)b * S.ncand;
    float Px[6], Py[6];                   // pending gx / gy rows (vertical 7-tap filters)
    float Qxx[2 * HH], Qxy[2 * HH], Qyy[2 * HH];   // pending vertical window sums
#pragma unroll
    for (int m = 0; m < 6; m++) { Px[m] = 0.f; Py[m] = 0.f; }
#pragma unroll
    for (int m = 0; m < 2 * HH; m++) { Qxx[m] = 0.f; Qxy[m] = 0.f; Qyy[m] = 0.f; }
    const int y0 = ys - HH - FS_R;        // first input row; input row y completes gradient row y-3 and window row y-3-HH
    float q[FS_PF];
#pragma unroll
    for (int i = 0; i < FS_PF; i++) q[i] = img[(size_t)klt_reflect(y0 + i, H) * pitch];
    __syncthreads();
    const int y_end = ye - 1 + HH + FS_R;  // last input row (inclusive)
    for (int y = y0; y <= y_end; y++) {
        const int par = (y - y0) & 1;
        const float cur = q[0];
#pragma unroll
        for (int i = 0; i < FS_PF - 1; i++) q[i] = q[i + 1];
        q[FS_PF - 1] = img[(size_t)klt_reflect(min(y + FS_PF, y_end), H) * pitch];
        rowI[par][t] = cur;
        __syncthreads();
        float dh = 0.f, gh = 0.f;
        if (t >= FS_R && t < FS_THREADS - FS_R) {
            const float *r = &rowI[par][t];
            const float a1 = r[1] + r[-1], a2 = r[2] + r[-2], a3 = r[3] + r[-3];
            const float b1 = r[1] - r[-1], b2 = r[2] - r[-2], b3 = r[3] - r[-3];
            // the reference's kernels are symmetric (gauss) / antisymmetric (derivative): c[3+k] = +-c[3-k]
            gh = fmaf(T.g[6], a3, fmaf(T.g[5], a2, fmaf(T.g[4], a1, T.g[3] * r[0])));
            dh = fmaf(T.d[6], b3, fmaf(T.d[5], b2, T.d[4] * b1));
        }
        // vertical filters: gx = g_v(d_h), gy = d_v(g_h); row y completes output row y - 3
        const float gx = fmaf(T.g[6], dh, Px[0]), gy = fmaf(T.d[6], gh, Py[0]);
#pragma unroll
        for (int m = 0; m < 5; m++) { Px[m] = fmaf(T.g[5 - m], dh, Px[m + 1]); Py[m] = fmaf(T.d[5 - m], gh, Py[m + 1]); }
        Px[5] = T.g[0] * dh; Py[5] = T.d[0] * gh;
        // vertical window sums: gradient row y-3 completes window row y - 3 - HH
        const float pxx = gx * gx, pxy = gx * gy, pyy = gy * gy;
        const float vxx = Qxx[0] + pxx, vxy = Qxy[0] + pxy, vyy = Qyy[0] + pyy;
#pragma unroll
        for (int m = 0; m < 2 * HH - 1; m++) { Qxx[m] = Qxx[m + 1] + pxx; Qxy[m] = Qxy[m + 1] + pxy; Qyy[m] = Qyy[m + 1] + pyy; }
        Qxx[2 * HH - 1] = pxx; Qxy[2 * HH - 1] = pxy; Qyy[2 * HH - 1] = pyy;
        const int yc = y - FS_R - HH;
        if (yc >= ys) {                                   // block-uniform
            rowV[par][0][t] = vxx; rowV[par][1][t] = vxy; rowV[par][2][t] = vyy;
            __syncthreads();
            const int cj = yc - S.by;
            if (cand_col && (cj % S.step) == 0) {
                float gxx = 0.f, gxy = 0.f, gyy = 0.f;
                for (int k = -hw; k <= hw; k++) { gxx += rowV[par][0][t + k]; gxy += rowV[par][1][t + k]; gyy += rowV[par][2][t + k]; }
                const float dd = gxx - gyy;
                vmap[(size_t)(cj / S.step) * S.nx + i_c] = 0.5f * ((gxx + gyy) - sqrtf(fmaf(dd, dd, 4.f * gxy * gxy)));
            }
        }
    }
}

// ---- windows up to 7x7: the same pass with no shared memory and no barriers -------------------------------------------
// A WARP owns 32 * NC adjacent columns and marches down its row segment; a lane owns NC = 4 adjacent columns (one 128-bit load
// per row).  Horizontal neighbours -- three image columns for the 7-tap gradient filters, HH columns of window sums -- come
// from the adjacent lanes by shuffle; the outermost HL = ceil(6 / NC) lanes on either side are halo lanes.  Everything else is
// arithmetic on NC independent columns; the vertical window sums run as add-new / subtract-old on a warp-private ring.
#define FQ_L2PF 16           // rows ahead of the L2 prefetch (the register queue covers an L2 hit, this covers DRAM)
#define FQ_NC 4              // columns per lane
// MUFU.SQRT: within 1 ulp of sqrtf without its Newton step and special-case branch (this mode is judged by set overlap)
__device__ __forceinline__ float sqrt_approx(float x) { float r; asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

template <int HH, bool STEP1>
__global__ void __launch_bounds__(FS_THREADS)
eigen_fast_quad_kernel(const float *__restrict__ img0, size_t img_stride, size_t pitch, const __grid_constant__ SelDev S,
                       const __grid_constant__ FastTaps T, int rows_per_seg, int n_strips, int vec_ok) {
    constexpr int NC = FQ_NC;
    constexpr int HL = (FS_R + HH + NC - 1) / NC;                   // halo lanes per side
    constexpr int USE = (32 - 2 * HL) * NC;                         // output columns per warp
    constexpr int NB = (FS_R + NC - 1) / NC, NBH = (HH + NC - 1) / NC;   // neighbour lanes that hold the 3 / HH adjacent columns
    typedef float4 vec_t;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, b = blockIdx.z;
    const int W = S.W, H = S.H;
    const int strip = blockIdx.x * (FS_THREADS / 32) + warp;
    const int ys = S.by + (int)blockIdx.y * rows_per_seg, ye = min(ys + rows_per_seg, H - S.by);
    if (strip >= n_strips || ys >= ye) return;
    const int xa = S.bx & ~(NC - 1);
    const int xl = xa - HL * NC + strip * USE + NC * lane;          // first of this lane's NC columns (multiple of NC)
    const bool vec = xl >= 0 && xl + NC - 1 < W && vec_ok;
    int cr[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) cr[c] = klt_reflect(xl + c, W);
    const float *img = img0 + (size_t)b * img_stride;
    float cur[NC], nxt[NC];
    // rows of a segment reach at most HH + 3 <= 6 rows beyond the image: one bounce of SciPy's 'reflect' covers them when the
    // image is taller than that (the launcher sends smaller images to the generic kernel)
    auto refl = [&](int y) { return y < 0 ? -y - 1 : (y >= H ? 2 * H - y - 1 : y); };
    auto load_row = [&](int y, float (&o)[NC]) {
        const float *r = img + (size_t)refl(y) * pitch;
        if (vec) {
            const vec_t v = *reinterpret_cast<const vec_t *>(r + xl);
            const float *pv = reinterpret_cast<const float *>(&v);
#pragma unroll
            for (int c = 0; c < NC; c++) o[c] = pv[c];
        } else {
#pragma unroll
            for (int c = 0; c < NC; c++) o[c] = r[cr[c]];
        }
    };
    const bool out_lane = lane >= HL && lane < 32 - HL;
    float *vmap = S.vmap + (size_t)b * S.ncand;
    // vertical window sums: running sums in registers, the last 2 HH + 1 rows of products in a warp-private shared-memory ring
    // (each lane only ever touches its own NC columns of it: no barrier).  The sums restart with every row segment, so the
    // rounding drift of add-new / subtract-old stays ~1e-6 relative.
    constexpr int KR = 2 * HH + 1;
    extern __shared__ __align__(16) float fq_ring[];                 // [warp][KR][3][32 lanes][NC]
    vec_t *ring = reinterpret_cast<vec_t *>(fq_ring) + (size_t)warp * KR * 3 * 32 + lane;
    float Px[NC][6], Py[NC][6], Sxx[NC], Sxy[NC], Syy[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) {
#pragma unroll
        for (int m = 0; m < 6; m++) { Px[c][m] = 0.f; Py[c][m] = 0.f; }
        Sxx[c] = 0.f; Sxy[c] = 0.f; Syy[c] = 0.f;
    }
    {
        vec_t z;
        float *pz = reinterpret_cast<float *>(&z);
#pragma unroll
        for (int c = 0; c < NC; c++) pz[c] = 0.f;
        for (int k = 0; k < KR * 3; k++) ring[k * 32] = z;
    }
    int slot = 0;
    // V[k] = value of column xl - R + k gathered from this lane (cols R .. R+NC-1) and its neighbours
    auto gather = [&](const float (&v)[NC], float *V, int R, int nb) {
#pragma unroll
        for (int k = 0; k < R; k++) {
            // column xl - R + k lives in lane - ceil((R-k)/NC), element NC*that - (R-k)
            const int d = (R - k + NC - 1) / NC, e = d * NC - (R - k);
            V[k] = __shfl_up_sync(0xffffffffu, v[e], d);
            const int kk = R + NC + k;                                // column xl + NC + k lives in lane + 1 + k/NC, element k % NC
            V[kk] = __shfl_down_sync(0xffffffffu, v[k % NC], 1 + k / NC);
        }
#pragma unroll
        for (int c = 0; c < NC; c++) V[R + c] = v[c];
        (void)nb;
    };
    const int y0 = ys - HH - FS_R, y_end = ye - 1 + HH + FS_R;
    // one row of both gradients for this lane's NC columns: horizontal 7-tap pair from the neighbours' columns, vertical pair
    // as accumulate-and-shift FMAs (input row y completes gradient row y - 3)
    auto gradients = [&](const float (&row)[NC], float (&gx)[NC], float (&gy)[NC]) {
        float I[NC + 2 * FS_R];                                       // columns xl-3 .. xl+NC+2
        gather(row, I, FS_R, NB);
#pragma unroll
        for (int c = 0; c < NC; c++) {
            const float *r = &I[FS_R + c];
            const float a1 = r[1] + r[-1], a2 = r[2] + r[-2], a3 = r[3] + r[-3];
            const float b1 = r[1] - r[-1], b2 = r[2] - r[-2], b3 = r[3] - r[-3];
            const float gh = fmaf(T.g[6], a3, fmaf(T.g[5], a2, fmaf(T.g[4], a1, T.g[3] * r[0])));
            const float dh = fmaf(T.d[6], b3, fmaf(T.d[5], b2, T.d[4] * b1));
            gx[c] = fmaf(T.g[6], dh, Px[c][0]); gy[c] = fmaf(T.d[6], gh, Py[c][0]);
#pragma unroll
            for (int m = 0; m < 5; m++) { Px[c][m] = fmaf(T.g[5 - m], dh, Px[c][m + 1]); Py[c][m] = fmaf(T.d[5 - m], gh, Py[c][m + 1]); }
            Px[c][5] = T.g[0] * dh; Py[c][5] = T.d[0] * gh;
        }
    };
    load_row(y0, nxt);
    // the first 6 rows of a segment only warm the vertical filters up: their "gradients" never enter the window sums
#pragma unroll 1
    for (int y = y0; y < y0 + 2 * FS_R; y++) {
#pragma unroll
        for (int c = 0; c < NC; c++) cur[c] = nxt[c];
        load_row(min(y + 1, y_end), nxt);
        float gx[NC], gy[NC];
        gradients(cur, gx, gy);
    }
#pragma unroll 1
    for (int y = y0 + 2 * FS_R; y <= y_end; y++) {
#pragma unroll
        for (int c = 0; c < NC; c++) cur[c] = nxt[c];
        load_row(min(y + 1, y_end), nxt);
        if (y + FQ_L2PF <= y_end && (lane & 7) == 0)       // one touch per 128-byte line
            asm volatile("prefetch.global.L2 [%0];" ::"l"(img + (size_t)refl(y + FQ_L2PF) * pitch + cr[0]));
        float vxx[NC], vxy[NC], vyy[NC];
        __align__(16) float nxx[NC], nxy[NC], nyy[NC];
        {
            float gx[NC], gy[NC];
            gradients(cur, gx, gy);
#pragma unroll
            for (int c = 0; c < NC; c++) { nxx[c] = gx[c] * gx[c]; nxy[c] = gx[c] * gy[c]; nyy[c] = gy[c] * gy[c]; }
        }
        {
            vec_t *rs = ring + (size_t)slot * 3 * 32;
            const vec_t oxx = rs[0], oxy = rs[32], oyy = rs[64];
            const float *po0 = reinterpret_cast<const float *>(&oxx), *po1 = reinterpret_cast<const float *>(&oxy), *po2 = reinterpret_cast<const float *>(&oyy);
#pragma unroll
            for (int c = 0; c < NC; c++) {
                Sxx[c] += nxx[c] - po0[c]; Sxy[c] += nxy[c] - po1[c]; Syy[c] += nyy[c] - po2[c];
                vxx[c] = Sxx[c]; vxy[c] = Sxy[c]; vyy[c] = Syy[c];
            }
            rs[0] = *reinterpret_cast<const vec_t *>(nxx); rs[32] = *reinterpret_cast<const vec_t *>(nxy); rs[64] = *reinterpret_cast<const vec_t *>(nyy);
            slot = slot + 1 == KR ? 0 : slot + 1;
        }
        const int yc = y - FS_R - HH;
        if (yc >= ys) {                                          // warp-uniform
            // horizontal window sums over columns xl-HH .. xl+NC-1+HH of the three planes
            float sx[NC], sxy_[NC], sy[NC];
            auto hbox = [&](const float (&v)[NC], float (&o)[NC]) {
                float V[NC + 2 * HH];
                gather(v, V, HH, NBH);
                float s0 = V[0];
#pragma unroll
                for (int k = 1; k <= 2 * HH; k++) s0 += V[k];
                o[0] = s0;
#pragma unroll
                for (int c = 1; c < NC; c++) o[c] = o[c - 1] + V[c + 2 * HH] - V[c - 1];
            };
            hbox(vxx, sx); hbox(vxy, sxy_); hbox(vyy, sy);
            const int cj = yc - S.by;
            if (out_lane && (STEP1 || (cj % S.step) == 0)) {
                float *vrow = vmap + (size_t)(STEP1 ? cj : cj / S.step) * S.nx;
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    const int x = xl + c, ci = x - S.bx;
                    if (ci >= 0 && x < W - S.bx && (STEP1 || (ci % S.step) == 0)) {
                        const float dd = sx[c] - sy[c];
                        vrow[STEP1 ? ci : ci / S.step] = 0.5f * ((sx[c] + sy[c]) - sqrt_approx(fmaf(dd, dd, 4.f * sxy_[c] * sxy_[c])));
                    }
                }
            }
        }
    }
}

template <int HH>
static int launch_fast_quad(klt_ctx *ctx, const SelDev *S, int B, const float *img0, size_t img_stride, size_t pitch, const FastTaps &T) {
    constexpr int NC = FQ_NC;
    constexpr int HL = (FS_R + HH + NC - 1) / NC, USE = (32 - 2 * HL) * NC;
    const int ncols = S->W - S->bx - (S->bx & ~(NC - 1)), nrows = S->H - 2 * S->by;
    if (S->W - 2 * S->bx <= 0 || nrows <= 0) return 1;
    const int n_strips = (ncols + USE - 1) / USE;
    const int strip_blocks = (n_strips + FS_THREADS / 32 - 1) / (FS_THREADS / 32);
    // about one wave of resident blocks; a segment re-reads 2*(HH+3) warm-up rows: keep it >= 64 rows
    long nseg = ((long)ctx->num_sms * 4) / ((long)strip_blocks * B);
    if (nseg < 1) nseg = 1;
    int rows = (int)((nrows + nseg - 1) / nseg);
    if (rows < 64) rows = 64;
    if (rows > nrows) rows = nrows;
    const dim3 grid(strip_blocks, (nrows + rows - 1) / rows, B);
    const double bytes = (4.0 * S->W * S->H + 4.0 * S->ncand) * B;
    const int vec_ok = (pitch % 4) == 0 && (img_stride % 4) == 0 && (reinterpret_cast<uintptr_t>(img0) & 15) == 0;
    const size_t smem = (size_t)(FS_THREADS / 32) * (2 * HH + 1) * 3 * 32 * NC * sizeof(float);      // <= 43 KB
    if (S->step == 1)
        KLT_LAUNCH(ctx, "eigen_fast", bytes, (eigen_fast_quad_kernel<HH, true><<<grid, FS_THREADS, smem, ctx->stream>>>(img0, img_stride, pitch, *S, T, rows, n_strips, vec_ok)));
    else
        KLT_LAUNCH(ctx, "eigen_fast", bytes, (eigen_fast_quad_kernel<HH, false><<<grid, FS_THREADS, smem, ctx->stream>>>(img0, img_stride, pitch, *S, T, rows, n_strips, vec_ok)));
    return 1;
}

template <int HH>
static int launch_fast(klt_ctx *ctx, const SelDev *S, int B, const float *img0, size_t img_stride, size_t pitch, const FastTaps &T) {
    const int span = FS_THREADS - 2 * (FS_R + S->hw);
    const int ncols = S->W - 2 * S->bx, nrows = S->H - 2 * S->by;
    if (ncols <= 0 || nrows <= 0) return 1;
    const int strips = (ncols + span - 1) / span;
    // about two waves of 8 resident blocks per SM; a segment re-reads 2*(HH+3) warm-up rows, so keep segments >= 64 rows
    long nseg = ((long)ctx->num_sms * 16) / ((long)strips * B);
    if (nseg < 1) nseg = 1;
    int rows = (int)((nrows + nseg - 1) / nseg);
    if (rows < 64) rows = 64;
    if (rows > nrows) rows = nrows;
    const dim3 grid(strips, (nrows + rows - 1) / rows, B);
    const double bytes = (4.0 * S->W * S->H + 4.0 * S->ncand) * B;
    KLT_LAUNCH(ctx, "eigen_fast_rows", bytes, (eigen_fast_kernel<HH><<<grid, FS_THREADS, 0, ctx->stream>>>(img0, img_stride, pitch, *S, T, rows)));
    return 1;
}

// the fused pass covers 7-tap gradient kernels and square windows of half-size 1..7
bool klt_sel_fast_covers(const SelDev *S, const klt_kernel1d *gauss, const klt_kernel1d *deriv) {
    if (gauss->n != 2 * FS_R + 1 || deriv->n != 2 * FS_R + 1) return false;
    if (S->hw != S->hh || S->hw < 1 || S->hw > 7) return false;
    for (int k = 1; k <= 3; k++)            // the folded form needs the symmetry the reference's kernels have
        if (fabs(gauss->taps[3 + k] - gauss->taps[3 - k]) > 1e-12 || fabs(deriv->taps[3 + k] + deriv->taps[3 - k]) > 1e-12) return false;
    return fabs(deriv->taps[3]) <= 1e-12;
}

// 1 = launched, 0 = configuration not covered (caller builds gradient planes and takes the table-based pass), < 0 error
int klt_sel_launch_eigen_fast(klt_ctx *ctx, const SelDev *S, int B, const float *img0, size_t img_stride, size_t pitch,
                              const klt_kernel1d *gauss, const klt_kernel1d *deriv) {
    if (!klt_sel_fast_covers(S, gauss, deriv)) return 0;
    FastTaps T;
    for (int j = 0; j < 7; j++) { T.g[j] = (float)gauss->taps[6 - j]; T.d[j] = (float)deriv->taps[6 - j]; }
    if (S->H < 16 && S->hh <= 3) {          // the quad kernel's one-bounce row reflection needs an image taller than its halo
        switch (S->hh) {
            case 1: return launch_fast<1>(ctx, S, B, img0, img_stride, pitch, T);
            case 2: return launch_fast<2>(ctx, S, B, img0, img_stride, pitch, T);
            case 3: return launch_fast<3>(ctx, S, B, img0, img_stride, pitch, T);
        }
    }
    switch (S->hh) {
        case 1: return launch_fast_quad<1>(ctx, S, B, img0, img_stride, pitch, T);
        case 2: return launch_fast_quad<2>(ctx, S, B, img0, img_stride, pitch, T);
        case 3: return launch_fast_quad<3>(ctx, S, B, img0, img_stride, pitch, T);
        case 4: return launch_fast<4>(ctx, S, B, img0, img_stride, pitch, T);
        case 5: return launch_fast<5>(ctx, S, B, img0, img_stride, pitch, T);
        case 6: return launch_fast<6>(ctx, S, B, img0, img_stride, pitch, T);
        case 7: return launch_fast<7>(ctx, S, B, img0, img_stride, pitch, T);
    }
    return 0;
}
