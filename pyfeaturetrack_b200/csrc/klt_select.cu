// Good-feature selection on the GPU (sm_100a), batched over the images of a pyramid batch and free of host
// synchronisation: every decision (how many candidates to sort, when to stop, when to widen the candidate set) is taken
// on the device, so a whole selection -- or a whole sequence step (klt_sequence.cu) -- is one chain of launches that can
// be captured in a CUDA graph.
//
// Replaces goodFeaturesUtils.ScanImageForGoodFeatures (goodFeaturesUtils.pyx:35-73), the candidate sort
// (selectGoodFeatures.py:234-236) and _enforceMinimumDistance (selectGoodFeatures.py:45-135).
//
// STRICT eigenvalues: the reference's values carry the rounding of three float32 summed-area tables built by strictly
// sequential additions (np.cumsum along rows, then along columns); selection ORDER depends on that rounding (SURVEY 7.3),
// so the tables are rebuilt with the same chains: one lane per row (tiles transposed through shared memory so that
// global traffic stays coalesced), then one thread per column, then the four-corner combine.  A parallel prefix scan would
// be faster per element but produces different float32 sums.
// FAST eigenvalues (klt_select_fast.cu): gradients, window sums and the eigenvalue from one shared-memory tile.
//
// Sort + greedy: the reference sorts every candidate (1.87 M at 1080p) although the greedy walk consumes only the best
// ~8.5 N.  Here the eigen kernels also build a 4096-bin histogram of the values (exponent + 7 mantissa bits, 0.8 %
// resolution); select_plan_kernel picks the bin range that holds about 32 N + 8192 candidates; select_scatter_kernel
// writes those candidates grouped by bin (descending) -- a one-pass MSD radix step; select_walk_kernel (one CTA per
// image) then takes bin groups of up to 4096 candidates at a time: drops the ones a feature accepted earlier already
// suppresses, sorts the rest in shared memory (bitonic) and runs the exact sequential greedy recurrence on them.  If the
// range runs out before every slot is filled the CTA widens it by itself (gathers the next bins from the eigenvalue map)
// until the map is exhausted, so the result is always the exact greedy result.  Replacement mode (KLTReplaceLostFeatures)
// leaves the candidates that surviving features suppress out of the histogram and the keys.
#include <cuda_pipeline.h>

#include "klt_common.cuh"
#include "klt_select.cuh"

// ---- summed-area tables: row pass -----------------------------------------------------------------------
// rows: s[y][x] = s[y][x-1] + p[y][x], p = exact fp32 product (np.power(g,2.) / g*g, pyx:49-51).
// One warp owns 32 rows of one image.  32x32 tiles of gx, gy are brought in with cp.async (ring of 4, coalesced), each
// lane then walks ITS row of the tile sequentially (the float32 chain of np.cumsum), and the three result tiles go back
// transposed so that the stores are coalesced too.
#define SAT_T 32
#define SAT_NBUF 4                      // cp.async ring: tiles are requested 3 chunks ahead of their use
struct SatSmem {
    float in[SAT_NBUF][2][SAT_T][SAT_T + 1];   // [buffer][gx|gy][row][col]
    float out[3][SAT_T][SAT_T + 1];
};

__global__ void __launch_bounds__(32)
sat_rows_kernel(const float *__restrict__ gx0, const float *__restrict__ gy0, size_t img_stride, size_t pitch, int W, int H,
                float *__restrict__ sat, size_t plane) {
    __shared__ SatSmem sm;
    const int lane = threadIdx.x;
    const int y0 = blockIdx.x * SAT_T;
    const float *gx = gx0 + (size_t)blockIdx.y * img_stride, *gy = gy0 + (size_t)blockIdx.y * img_stride;
    float *sxx = sat + (size_t)blockIdx.y * 3 * plane, *sxy = sxx + plane, *syy = sxy + plane;
    const int nchunks = (W + SAT_T - 1) / SAT_T;
    auto issue = [&](int chunk, int buf) {
        const int x = chunk * SAT_T + lane;
        if (x < W) {
#pragma unroll 8
            for (int i = 0; i < SAT_T; i++) {
                const int y = min(y0 + i, H - 1);
                __pipeline_memcpy_async(&sm.in[buf][0][i][lane], gx + (size_t)y * pitch + x, 4);
                __pipeline_memcpy_async(&sm.in[buf][1][i][lane], gy + (size_t)y * pitch + x, 4);
            }
        }
        __pipeline_commit();
    };
    float axx = 0.f, axy = 0.f, ayy = 0.f;     // 0 + p == p exactly, so starting from 0 equals cumsum's first copy
    for (int c = 0; c < SAT_NBUF - 1; c++) {
        if (c < nchunks) issue(c, c); else __pipeline_commit();
    }
    for (int c = 0; c < nchunks; c++) {
        const int buf = c % SAT_NBUF;
        if (c + SAT_NBUF - 1 < nchunks) issue(c + SAT_NBUF - 1, (c + SAT_NBUF - 1) % SAT_NBUF); else __pipeline_commit();
        __pipeline_wait_prior(SAT_NBUF - 1);
        __syncwarp();
        const int ncol = min(SAT_T, W - c * SAT_T);
        for (int k = 0; k < ncol; k++) {       // lane = row: sequential chain along x
            const float a = sm.in[buf][0][lane][k], b = sm.in[buf][1][lane][k];
            axx = __fadd_rn(axx, __fmul_rn(a, a));
            axy = __fadd_rn(axy, __fmul_rn(a, b));
            ayy = __fadd_rn(ayy, __fmul_rn(b, b));
            sm.out[0][lane][k] = axx; sm.out[1][lane][k] = axy; sm.out[2][lane][k] = ayy;
        }
        __syncwarp();
        const int x = c * SAT_T + lane;
        if (x < W) {
#pragma unroll 8
            for (int i = 0; i < SAT_T; i++) {
                const int y = y0 + i;
                if (y < H) {
                    const size_t o = (size_t)y * W + x;
                    sxx[o] = sm.out[0][i][lane]; sxy[o] = sm.out[1][i][lane]; syy[o] = sm.out[2][i][lane];
                }
            }
        }
        __syncwarp();
    }
}

// Same algorithm for W % 32 == 0 and 16-byte aligned rows: 128-bit cp.async, 128-bit shared loads/stores (row stride 36
// floats keeps every quarter-warp on distinct banks), fully unrolled so that only the 32-step float32 add chains are serial.
#define SAT_S 36
struct SatSmemV {
    float in[SAT_NBUF][2][SAT_T][SAT_S];
    float out[3][SAT_T][SAT_S];
};
__global__ void __launch_bounds__(32)
sat_rows_vec_kernel(const float *__restrict__ gx0, const float *__restrict__ gy0, size_t img_stride, size_t pitch, int W, int H,
                    float *__restrict__ sat, size_t plane) {
    extern __shared__ __align__(16) unsigned char sat_raw[];
    SatSmemV &sm = *reinterpret_cast<SatSmemV *>(sat_raw);
    const int lane = threadIdx.x;
    const int y0 = blockIdx.x * SAT_T;
    const float *gx = gx0 + (size_t)blockIdx.y * img_stride, *gy = gy0 + (size_t)blockIdx.y * img_stride;
    float *sxx = sat + (size_t)blockIdx.y * 3 * plane, *sxy = sxx + plane, *syy = sxy + plane;
    const int nchunks = W / SAT_T;
    const int q = lane & 7, r8 = lane >> 3;            // 16-byte chunk within a tile row, row within a group of 4
    auto issue = [&](int chunk, int buf) {
        const int x = chunk * SAT_T + 4 * q;
#pragma unroll
        for (int g = 0; g < SAT_T / 4; g++) {
            const int i = 4 * g + r8;
            const int y = min(y0 + i, H - 1);
            __pipeline_memcpy_async(&sm.in[buf][0][i][4 * q], gx + (size_t)y * pitch + x, 16);
            __pipeline_memcpy_async(&sm.in[buf][1][i][4 * q], gy + (size_t)y * pitch + x, 16);
        }
        __pipeline_commit();
    };
    float axx = 0.f, axy = 0.f, ayy = 0.f;
    for (int c = 0; c < SAT_NBUF - 1; c++) {
        if (c < nchunks) issue(c, c); else __pipeline_commit();
    }
    for (int c = 0; c < nchunks; c++) {
        const int buf = c % SAT_NBUF;
        if (c + SAT_NBUF - 1 < nchunks) issue(c + SAT_NBUF - 1, (c + SAT_NBUF - 1) % SAT_NBUF); else __pipeline_commit();
        __pipeline_wait_prior(SAT_NBUF - 1);
        __syncwarp();
        float4 va[8], vb[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            va[k] = *reinterpret_cast<const float4 *>(&sm.in[buf][0][lane][4 * k]);
            vb[k] = *reinterpret_cast<const float4 *>(&sm.in[buf][1][lane][4 * k]);
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {          // lane = row: the sequential float32 chain of np.cumsum along x
            float4 oxx, oxy, oyy;
            axx = __fadd_rn(axx, __fmul_rn(va[k].x, va[k].x)); axy = __fadd_rn(axy, __fmul_rn(va[k].x, vb[k].x)); ayy = __fadd_rn(ayy, __fmul_rn(vb[k].x, vb[k].x));
            oxx.x = axx; oxy.x = axy; oyy.x = ayy;
            axx = __fadd_rn(axx, __fmul_rn(va[k].y, va[k].y)); axy = __fadd_rn(axy, __fmul_rn(va[k].y, vb[k].y)); ayy = __fadd_rn(ayy, __fmul_rn(vb[k].y, vb[k].y));
            oxx.y = axx; oxy.y = axy; oyy.y = ayy;
            axx = __fadd_rn(axx, __fmul_rn(va[k].z, va[k].z)); axy = __fadd_rn(axy, __fmul_rn(va[k].z, vb[k].z)); ayy = __fadd_rn(ayy, __fmul_rn(vb[k].z, vb[k].z));
            oxx.z = axx; oxy.z = axy; oyy.z = ayy;
            axx = __fadd_rn(axx, __fmul_rn(va[k].w, va[k].w)); axy = __fadd_rn(axy, __fmul_rn(va[k].w, vb[k].w)); ayy = __fadd_rn(ayy, __fmul_rn(vb[k].w, vb[k].w));
            oxx.w = axx; oxy.w = axy; oyy.w = ayy;
            *reinterpret_cast<float4 *>(&sm.out[0][lane][4 * k]) = oxx;
            *reinterpret_cast<float4 *>(&sm.out[1][lane][4 * k]) = oxy;
            *reinterpret_cast<float4 *>(&sm.out[2][lane][4 * k]) = oyy;
        }
        __syncwarp();
        const int x = c * SAT_T + 4 * q;
#pragma unroll
        for (int g = 0; g < SAT_T / 4; g++) {
            const int i = 4 * g + r8, y = y0 + i;
            if (y < H) {
                const size_t o = (size_t)y * W + x;
                *reinterpret_cast<float4 *>(sxx + o) = *reinterpret_cast<const float4 *>(&sm.out[0][i][4 * q]);
                *reinterpret_cast<float4 *>(sxy + o) = *reinterpret_cast<const float4 *>(&sm.out[1][i][4 * q]);
                *reinterpret_cast<float4 *>(syy + o) = *reinterpret_cast<const float4 *>(&sm.out[2][i][4 * q]);
            }
        }
        __syncwarp();
    }
}

// min eigenvalue (pyx:17-19), operand types as in the Cython-generated C
__device__ __forceinline__ float min_eigenvalue(float gxx, float gxy, float gyy) {
    const float d = __fsub_rn(gxx, gyy);
    const float dd = __fmul_rn(d, d);
    const double t = __dadd_rn((double)dd, __dmul_rn(__dmul_rn(4.0, (double)gxy), (double)gxy));
    const float sqrtTerm = __double2float_rn(sqrt(t));   // reference: pow(t, 0.5); IEEE sqrt is the correctly rounded value
    const float s = __fsub_rn(__fadd_rn(gxx, gyy), sqrtTerm);
    return __double2float_rn(__dmul_rn((double)s, 0.5));   // s / 2. exactly (a power of two)
}

// ---- column pass -----------------------------------------------------------------------------------------------------
// columns: s[y][x] = s[y-1][x] + s[y][x] (np.cumsum(axis 0), sequential), in place.  One thread owns one column of one
// table of one image; 16 independent loads are in flight per thread while the add chain runs.  (A variant that kept the
// running sums in a shared-memory ring and evaluated the eigenvalues from it -- no write-back of the tables -- was
// measured at 914 us per 8 images against 130 + 40 us for this pass plus the eigen kernel: with one chain per thread the
// fused kernel cannot hide the latency of the eigenvalue's float64 sqrt behind anything.)
__global__ void __launch_bounds__(64)
sat_cols_kernel(float *__restrict__ sat, size_t plane, int W, int H) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= W) return;
    float *s = sat + ((size_t)blockIdx.z * 3 + blockIdx.y) * plane + x;
    float acc = s[0];
    int y = 1;
    for (; y + 16 <= H; y += 16) {
        float v[16];
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = s[(size_t)(y + i) * W];
#pragma unroll
        for (int i = 0; i < 16; i++) { acc = __fadd_rn(acc, v[i]); s[(size_t)(y + i) * W] = acc; }
    }
    for (; y < H; y++) { acc = __fadd_rn(acc, s[(size_t)y * W]); s[(size_t)y * W] = acc; }
}

// four-corner combine (pyx:23-31): (c + a - b - d) in float32, in that order
__device__ __forceinline__ float window_sum(const float *__restrict__ s, int W, int x, int y, int hw, int hh) {
    const float a = s[(size_t)(y - hh - 1) * W + (x - hw - 1)], b = s[(size_t)(y - hh - 1) * W + (x + hw)];
    const float c = s[(size_t)(y + hh) * W + (x + hw)], d = s[(size_t)(y + hh) * W + (x - hw - 1)];
    return __fsub_rn(__fsub_rn(__fadd_rn(c, a), b), d);
}

// eigenvalue map.  One block = 256 candidate columns x EIG_ROWS candidate rows of one image.
#define EIG_ROWS 8
__global__ void __launch_bounds__(256)
eigen_kernel(const float *__restrict__ sat, size_t plane, const __grid_constant__ SelDev S) {
    const int b = blockIdx.z;
    const float *sxx = sat + (size_t)b * 3 * plane, *sxy = sxx + plane, *syy = sxy + plane;
    float *vmap = S.vmap + (size_t)b * S.ncand;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= S.nx) return;
    for (int jj = 0; jj < EIG_ROWS; jj++) {
        const int j = blockIdx.y * EIG_ROWS + jj;
        if (j < S.ny) {
            const int x = S.bx + i * S.step, y = S.by + j * S.step;
            vmap[(size_t)j * S.nx + i] = min_eigenvalue(window_sum(sxx, S.W, x, y, S.hw, S.hh), window_sum(sxy, S.W, x, y, S.hw, S.hh),
                                                        window_sum(syy, S.W, x, y, S.hw, S.hh));
        }
    }
}

// ---- histogram of the eigenvalue map (candidates >= min_val that no surviving feature suppresses) -----------------------
// Separate from the eigen kernels on purpose: those are register- and latency-critical; this pass re-reads 4 B per candidate
// at full occupancy (~2 us per 1080p image).
#define HIST_ROWS 8
#define HIST_COPIES 1          // same-address shared-memory atomics serialise and neighbouring candidates share bins; per 8 x 1080p:
                               // 1 copy, one atomic per candidate 66-73 us; four copies selected by lane 162 us; __match_any_sync
                               // aggregation 146 us; run-length aggregation by shuffle + ballot (below): see profiles/
__global__ void __launch_bounds__(256)
select_hist_kernel(const __grid_constant__ SelDev S) {
    extern __shared__ unsigned int hsm[];                // [HIST_COPIES][SEL_BINS]
    const int b = blockIdx.y;
    for (int k = threadIdx.x; k < HIST_COPIES * SEL_BINS; k += 256) hsm[k] = 0;
    __syncthreads();
    unsigned int *h = hsm + (threadIdx.x & (HIST_COPIES - 1)) * SEL_BINS;
    const float *vmap = S.vmap + (size_t)b * S.ncand;
    const unsigned char *pm = S.premap ? S.premap + (size_t)b * S.map_stride : nullptr;
    // few, long-lived blocks: the flush below costs up to SEL_BINS global atomics per block
    const int tiles_x = (S.nx + 255) / 256, tiles = tiles_x * ((S.ny + HIST_ROWS - 1) / HIST_ROWS);
    // All loads of a tile are issued together (eigenvalues AND pre-mark bytes, 16 independent requests per thread) and one
    // tile AHEAD of the counting: with the byte load behind the `v >= min_val` test the kernel exposed one memory latency per
    // row (79 us per 8 x 1080p at 16 % issue), without the look-ahead one per tile (58 us).
    float v[HIST_ROWS], vn[HIST_ROWS];
    unsigned char m[HIST_ROWS], mn[HIST_ROWS];
    // (32-bit element offsets -- one image's map and frame are far below 2^31 elements -- and the range test once per tile:
    // with 64-bit index chains per load the kernel was instruction-bound at 54 instructions per warp-row)
    auto load_tile = [&](int tile, float (&vv)[HIST_ROWS], unsigned char (&mm)[HIST_ROWS]) {
        const int i = (tile % tiles_x) * 256 + threadIdx.x, j0 = (tile / tiles_x) * HIST_ROWS;
        const int nrows = (tile < tiles && i < S.nx) ? S.ny - j0 : 0;               // rows [0, nrows) of the tile exist
        const int voff = j0 * S.nx + i, moff = (S.by + j0 * S.step) * S.W + S.bx + i * S.step, mrow = S.step * S.W;
#pragma unroll
        for (int jj = 0; jj < HIST_ROWS; jj++) {
            const bool in = jj < nrows;
            vv[jj] = in ? vmap[voff + jj * S.nx] : 0.f;
            mm[jj] = in ? (pm ? pm[moff + jj * mrow] : (unsigned char)0) : (unsigned char)1;
        }
    };
    const int lane = threadIdx.x & 31;
    load_tile(blockIdx.x, v, m);
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        load_tile(tile + gridDim.x, vn, mn);
        // Neighbouring candidates often share a bin and same-address shared-memory atomics serialise, so a warp counts RUNS:
        // a lane whose bin differs from its left neighbour's adds the length of the run it starts.
#pragma unroll
        for (int jj = 0; jj < HIST_ROWS; jj++) {
            const bool ok = !m[jj] && v[jj] >= S.min_val;
            const int bin = ok ? eig_rbin(v[jj]) : -1;
            const int left = __shfl_up_sync(0xffffffffu, bin, 1);
            const bool head = lane == 0 || bin != left;
            const unsigned int heads = __ballot_sync(0xffffffffu, head);
            if (head && bin >= 0) {
                const unsigned int above = lane == 31 ? 0u : heads & (0xfffffffeu << lane);
                const int next = above ? __ffs(above) - 1 : 32;
                atomicAdd(&h[bin], (unsigned int)(next - lane));
            }
        }
#pragma unroll
        for (int jj = 0; jj < HIST_ROWS; jj++) { v[jj] = vn[jj]; m[jj] = mn[jj]; }
    }
    __syncthreads();
    unsigned int *hist = S.hist + (size_t)b * SEL_BINS;
    for (int k = threadIdx.x; k < SEL_BINS; k += 256) {
        unsigned int c = 0;
#pragma unroll
        for (int q = 0; q < HIST_COPIES; q++) c += hsm[q * SEL_BINS + k];
        if (c) atomicAdd(&hist[k], c);
    }
}

// ---- plan: which bins to sort first ---------------------------------------------------------------------------------
// block-wide inclusive scan of one value per thread (WALK_THREADS threads)
__device__ __forceinline__ unsigned int block_scan_incl(unsigned int v, unsigned int *warp_tot /* [32] shared */, unsigned int *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
    __syncthreads();                                    // warp_tot may still be read by a previous call
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    unsigned int base = 0, tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { const unsigned int c = warp_tot[w]; if (w < warp) base += c; tot += c; }
    if (total) *total = tot;
    return incl + base;
}

// Range of reversed bins [rb_lo, rb_hi] holding at least `target` candidates (or everything that is left).  Fills
// pre[rb] = candidates in bins [rb_lo, rb) for every rb (pre[SEL_BINS] = all of them; bins below rb_lo count as empty) and,
// if given, cur[rb] = the same (the gather's append cursors).  WALK_THREADS threads, 4 bins each; results through shared scalars.
__device__ void plan_range(const unsigned int *__restrict__ hist, unsigned int rb_lo, unsigned int target, unsigned int *pre,
                           unsigned int *cur, unsigned int *warp_tot, unsigned int *s_rb_hi, unsigned int *s_nkeys) {
    const int t = threadIdx.x;
    unsigned int c[4], sum = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const unsigned int rb = 4 * t + j;
        c[j] = rb >= rb_lo ? hist[rb] : 0u;
        sum += c[j];
    }
    if (t == 0) *s_rb_hi = SEL_BINS - 1;
    const unsigned int incl = block_scan_incl(sum, warp_tot, nullptr);     // contains two __syncthreads
    unsigned int run = incl - sum;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const unsigned int rb = 4 * t + j;
        pre[rb] = run;
        if (cur) cur[rb] = run;
        if (run < target && run + c[j] >= target) atomicMin(s_rb_hi, rb);  // the bin in which the running count reaches the target
        run += c[j];
    }
    if (t == WALK_THREADS - 1) pre[SEL_BINS] = run;
    __syncthreads();
    if (t == 0) *s_nkeys = pre[*s_rb_hi + 1];
    __syncthreads();
}

__device__ __forceinline__ unsigned int count_lost(const int *__restrict__ fval, int n, unsigned int *warp_tot) {
    unsigned int mine = 0;
    for (int f = threadIdx.x; f < n; f += blockDim.x) mine += fval[f] < 0 ? 1u : 0u;
    unsigned int tot;
    block_scan_incl(mine, warp_tot, &tot);
    return tot;
}

__global__ void __launch_bounds__(WALK_THREADS)
select_plan_kernel(const __grid_constant__ SelDev S) {
    __shared__ unsigned int pre[SEL_BINS + 1];
    __shared__ unsigned int warp_tot[32];
    __shared__ unsigned int s_rb_hi, s_nkeys;
    const int b = blockIdx.x, t = threadIdx.x;
    const unsigned int slots = S.replace ? count_lost(S.fval + (size_t)b * S.n_features, S.n_features, warp_tot) : (unsigned int)S.n_features;
    const unsigned int target = slots ? S.target_mul * slots + S.target_add : 0u;
    unsigned int *plan = S.plan + (size_t)b * SEL_PLAN_WORDS;
    unsigned int *offs = S.offs + (size_t)b * (SEL_BINS + 1), *cursor = S.cursor + (size_t)b * SEL_BINS;
    if (target == 0) {          // nothing to fill: no keys at all
        if (t == 0) { plan[SEL_PLAN_RB_HI] = 0xFFFFFFFFu; plan[SEL_PLAN_NKEYS] = 0; plan[SEL_PLAN_SLOTS] = 0; }
        return;
    }
    plan_range(S.hist + (size_t)b * SEL_BINS, 0u, target, pre, nullptr, warp_tot, &s_rb_hi, &s_nkeys);
    for (int k = t; k < SEL_BINS; k += WALK_THREADS) { offs[k] = pre[k]; cursor[k] = 0; }
    if (t == 0) { offs[SEL_BINS] = pre[SEL_BINS]; plan[SEL_PLAN_RB_HI] = s_rb_hi; plan[SEL_PLAN_NKEYS] = s_nkeys; plan[SEL_PLAN_SLOTS] = slots; }
}

// ---- scatter: candidates of the planned bin range -> keys grouped by bin (descending value) -----------------------------
// key layout (ascending sort of ~key == descending (val, x, y)): [val bits 32][x 13][y 13]
__device__ __forceinline__ unsigned long long make_key(float val, int x, int y) {
    const unsigned long long k = ((unsigned long long)__float_as_uint(val) << 26) | ((unsigned long long)x << 13) |
                                 (unsigned long long)y;
    return ~k;
}

#define SCAT_ROWS 16
__global__ void __launch_bounds__(256)
select_scatter_kernel(const __grid_constant__ SelDev S) {
    const int b = blockIdx.z;
    const unsigned int rb_hi = S.plan[(size_t)b * SEL_PLAN_WORDS + SEL_PLAN_RB_HI];
    if (rb_hi == 0xFFFFFFFFu) return;
    const int i = blockIdx.x * 256 + threadIdx.x;
    const float *vmap = S.vmap + (size_t)b * S.ncand;
    const unsigned char *pm = S.premap ? S.premap + (size_t)b * S.map_stride : nullptr;
    const unsigned int *offs = S.offs + (size_t)b * (SEL_BINS + 1);
    unsigned int *cursor = S.cursor + (size_t)b * SEL_BINS;
    unsigned long long *keys = S.keys + (size_t)b * S.key_stride;
    const int lane = threadIdx.x & 31;
    // the planned range holds ~0.1-2 % of the candidates: the smallest value that can be in it, as a float threshold
    // (reversed bin <= rb_hi  <=>  (bits >> 16) >= 0x4F7F - rb_hi); values above the histogram's top land in bin 0
    const float vmin = fmaxf(S.min_val, __uint_as_float((0x4F7Fu - min(rb_hi, (unsigned int)(SEL_BINS - 1))) << 16));
    float v[SCAT_ROWS];
    {
        const int j0 = blockIdx.y * SCAT_ROWS;
        const int nrows = i < S.nx ? min(SCAT_ROWS, S.ny - j0) : 0;
        const float *vp = vmap + (size_t)j0 * S.nx + i;
#pragma unroll
        for (int jj = 0; jj < SCAT_ROWS; jj++) {
            v[jj] = jj < nrows ? *vp : 0.f;
            vp += S.nx;
        }
    }
#pragma unroll
    for (int jj = 0; jj < SCAT_ROWS; jj++) {
        const int j = blockIdx.y * SCAT_ROWS + jj;
        bool keep = v[jj] >= vmin;                    // candidates below min_eigenvalue can never be accepted (:116)
        if (!__any_sync(0xffffffffu, keep)) continue;
        const int x = S.bx + i * S.step, y = S.by + j * S.step;
        const int rb = eig_rbin(v[jj]);
        keep = keep && (unsigned int)rb <= rb_hi && !(pm && pm[(size_t)y * S.W + x]);
        // warp-aggregated append: one atomic per distinct bin in the warp
        const unsigned int peers = __match_any_sync(0xffffffffu, keep ? rb : SEL_BINS + lane);
        if (keep) {
            const int leader = __ffs(peers) - 1;
            unsigned int base = 0;
            if (lane == leader) base = atomicAdd(&cursor[rb], (unsigned int)__popc(peers));
            base = __shfl_sync(peers, base, leader);
            keys[offs[rb] + base + __popc(peers & ((1u << lane) - 1u))] = make_key(v[jj], x, y);
        }
    }
}

// ---- pre-marking of the surviving features (replacement mode, selectGoodFeatures.py:64-69) ---------------------------
__global__ void __launch_bounds__(128)
premark_kernel(const __grid_constant__ SelDev S) {
    const int f = blockIdx.x, b = blockIdx.y;
    const size_t fo = (size_t)b * S.n_features + f;
    if (S.fval[fo] < 0) return;
    unsigned char *map = S.premap + (size_t)b * S.map_stride;
    const int x = (int)S.fx[fo], y = (int)S.fy[fo], r = S.r, side = 2 * r + 1;
    for (int idx = threadIdx.x; idx < side * side; idx += blockDim.x) {
        const int iy = y - r + idx / side, ix = x - r + idx % side;
        if (ix >= 0 && ix < S.W && iy >= 0 && iy < S.H) map[(size_t)iy * S.W + ix] = 1;
    }
}

// ---- the walk: sort + greedy minimum-distance suppression (_enforceMinimumDistance) -----------------------------------
// Accepted features are remembered in a grid of cells of side cs = r + 1 (r = mindist - 1): two features in one cell would
// be closer than mindist, so a cell holds at most one and a candidate only has to look at its 3x3 cell neighbourhood
// (shared memory, or global memory for very large images).  Features that survive from a previous frame (replacement
// mode) are not in the grid -- they may be closer to each other than mindist -- the candidates they suppress never become
// keys.
__device__ __forceinline__ bool grid_conflict(const unsigned short *grid, int gw, int gh, int cs, int r, int x, int y) {
    const int cx = x / cs, cy = y / cs;
    bool hit = false;
#pragma unroll
    for (int dy = -1; dy <= 1; dy++)
#pragma unroll
        for (int dx = -1; dx <= 1; dx++) {
            const int ncx = cx + dx, ncy = cy + dy;
            if (ncx >= 0 && ncx < gw && ncy >= 0 && ncy < gh) {
                const unsigned int g = grid[ncy * gw + ncx];
                if (g != 0xFFFFu) {
                    const int fx = ncx * cs + (int)(g >> 8), fy = ncy * cs + (int)(g & 255u);
                    hit |= abs(fx - x) <= r && abs(fy - y) <= r;
                }
            }
        }
    return hit;
}

// in-place ascending bitonic sort of s[0..P), P a power of two, whole block
__device__ void bitonic_sort(unsigned long long *s, int P) {
    for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < P; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = s[i], b = s[ixj];
                    if ((a > b) == ((i & k) == 0)) { s[i] = b; s[ixj] = a; }
                }
            }
            __syncthreads();
        }
}

// Slow path for a bin that holds more keys than a chunk (massive ties, e.g. periodic patterns): stable LSD radix sort of
// keys[0..m) in global memory by ONE CTA, 4-bit digits, ping-pong with tmp; the sorted keys end in `keys`.
__device__ void block_radix_sort(unsigned long long *keys, unsigned long long *tmp, unsigned int m, unsigned int *warp_tot) {
    __shared__ unsigned int dh[16], dbase[16];
    __shared__ unsigned int wh[WALK_THREADS / 32][16];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    unsigned long long *src = keys, *dst = tmp;
    for (int shift = 0; shift < 60; shift += 4) {
        if (t < 16) dh[t] = 0;
        __syncthreads();
        for (unsigned int i = t; i < m; i += WALK_THREADS) atomicAdd(&dh[(unsigned int)(src[i] >> shift) & 15u], 1u);
        __syncthreads();
        bool skip = false;
        if (t < 16) {
            unsigned int base = 0;
            for (int d = 0; d < t; d++) base += dh[d];
            dbase[t] = base;
        }
        for (int d = 0; d < 16; d++) skip |= dh[d] == m;              // every key has the same digit: nothing moves
        __syncthreads();
        if (skip) continue;
        for (unsigned int tile = 0; tile < m; tile += WALK_THREADS) {
            const unsigned int i = tile + t;
            const bool valid = i < m;
            const unsigned long long key = valid ? src[i] : 0ull;
            const unsigned int d = valid ? ((unsigned int)(key >> shift) & 15u) : (16u + lane);
            const unsigned int peers = __match_any_sync(0xffffffffu, d);
            const unsigned int rank = __popc(peers & ((1u << lane) - 1u));
            if (lane < 16) wh[warp][lane] = 0;
            __syncwarp();
            if (valid && rank == 0) wh[warp][d] = __popc(peers);
            __syncthreads();
            if (valid) {
                unsigned int o = dbase[d] + rank;
                for (int w = 0; w < warp; w++) o += wh[w][d];
                dst[o] = key;
            }
            __syncthreads();
            if (t < 16) {
                unsigned int tot = 0;
                for (int w = 0; w < WALK_THREADS / 32; w++) tot += wh[w][t];
                dbase[t] += tot;
            }
            __syncthreads();
        }
        unsigned long long *x = src; src = dst; dst = x;
        __threadfence_block();
    }
    if (src != keys) {
        for (unsigned int i = t; i < m; i += WALK_THREADS) keys[i] = src[i];
    }
    __syncthreads();
    (void)warp_tot;
}

__global__ void __launch_bounds__(WALK_THREADS, 1)
select_walk_kernel(const __grid_constant__ SelDev S, int presorted) {
    extern __shared__ __align__(16) unsigned char wsm[];
    unsigned long long *sk = reinterpret_cast<unsigned long long *>(wsm);      // survivors of phase 1 of the current chunk, sorted
    unsigned int *pre = reinterpret_cast<unsigned int *>(sk + S.ch);            // [SEL_BINS + 1] keys of the current range above each reversed bin
    unsigned int *off = pre + SEL_BINS + 4;                                     // [SEL_BINS] append cursors of the fallback gather
    __shared__ unsigned int warp_cnt[32];
    __shared__ int s_filled, s_slots, s_full, s_ns;
    __shared__ unsigned int s_m, s_e, s_big, s_rb_hi, s_nkeys;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_features = S.n_features;
    double *fx = S.fx + (size_t)b * n_features, *fy = S.fy + (size_t)b * n_features;
    int *fval = S.fval + (size_t)b * n_features;
    int *free_slots = S.free_slots + (size_t)b * n_features;
    unsigned long long *keys = S.keys + (size_t)b * S.key_stride, *keys2 = S.keys2 + (size_t)b * S.key_stride;
    const unsigned int *hist = S.hist + (size_t)b * SEL_BINS;
    const unsigned int *offs_planned = S.offs + (size_t)b * (SEL_BINS + 1);
    unsigned long long *status = S.status + (size_t)b * SEL_STATUS_WORDS;
    // accepted features (one per cell at most) and, during a round of phase 2, the smallest live rank per cell
    unsigned int *cellmin = S.grid_in_smem ? off + SEL_BINS : S.cellmin_global + (size_t)b * S.grid_stride;
    unsigned short *grid = S.grid_in_smem ? reinterpret_cast<unsigned short *>(cellmin + S.gw * S.gh) : S.grid_global + (size_t)b * S.grid_stride;
    const int overwrite = S.replace ? 0 : 1;
    const unsigned char *pm_walk = (presorted && S.premap) ? S.premap + (size_t)b * S.map_stride : nullptr;
    if (S.r >= 0)
        for (int c = tid; c < S.gw * S.gh; c += WALK_THREADS) { grid[c] = 0xFFFFu; cellmin[c] = 0xFFFFFFFFu; }
    // fillable slots: every slot (SELECTING_ALL) or, in list order, the slots of lost features (:64-69, :110-112)
    if (tid == 0) { s_slots = overwrite ? n_features : 0; s_filled = 0; }
    __syncthreads();
    if (!overwrite) {
        for (int f0 = 0; f0 < n_features; f0 += WALK_THREADS) {
            const int f = f0 + tid;
            const bool lost = f < n_features && fval[f] < 0;
            const unsigned int m = __ballot_sync(0xffffffffu, lost);
            if (lane == 0) warp_cnt[warp] = __popc(m);
            __syncthreads();
            if (warp == 0) {
                unsigned int c = warp_cnt[lane], incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
                warp_cnt[lane] = incl - c;
                if (lane == 31) s_ns = (int)incl;
            }
            __syncthreads();
            if (lost) free_slots[s_slots + warp_cnt[warp] + __popc(m & ((1u << lane) - 1u))] = f;
            __syncthreads();
            if (tid == 0) s_slots += s_ns;
            __syncthreads();
        }
    }
    if (tid == 0) s_full = s_slots == 0;
    __syncthreads();
    const int slots = s_slots;
    const unsigned int target = slots ? S.target_mul * (unsigned int)slots + S.target_add : 0u;
    unsigned long long consumed = 0ull;
    unsigned int fallbacks = 0;
    unsigned int rb_lo = 0, rb_hi, nkeys;
    if (presorted) { rb_hi = 0; nkeys = S.plan[(size_t)b * SEL_PLAN_WORDS + SEL_PLAN_NKEYS]; }
    else { rb_hi = S.plan[(size_t)b * SEL_PLAN_WORDS + SEL_PLAN_RB_HI]; nkeys = S.plan[(size_t)b * SEL_PLAN_WORDS + SEL_PLAN_NKEYS]; }
    if (!s_full && rb_hi != 0xFFFFFFFFu) {
        if (!presorted)
            for (int k = tid; k <= SEL_BINS; k += WALK_THREADS) pre[k] = offs_planned[k];
        for (;;) {                                       // candidate ranges: the planned one, then fallbacks
            __syncthreads();
            unsigned int rb = rb_lo;
            while (rb <= rb_hi && !s_full) {
                if (tid == 0) {
                    unsigned int m, e, big = 0;
                    if (presorted) { m = nkeys; e = rb_hi + 1; big = 1; }
                    else {
                        // the longest run of bins [rb, e) that fits a chunk: binary search in the prefix counts
                        const unsigned int p0 = pre[rb];
                        unsigned int lo = rb, hi = rb_hi + 1;             // pre[lo] - p0 <= ch always holds
                        while (lo < hi) {
                            const unsigned int mid = (lo + hi + 1) >> 1;
                            if (pre[mid] - p0 <= (unsigned int)S.ch) lo = mid; else hi = mid - 1;
                        }
                        e = lo; m = pre[e] - p0;
                        if (e == rb) { e = rb + 1; m = pre[e] - p0; big = 1; }      // one bin larger than a chunk
                    }
                    s_m = m; s_e = e; s_big = big;
                }
                __syncthreads();
                const unsigned int pos = presorted ? 0u : pre[rb];
                const unsigned int m = s_m, e = s_e, big = s_big;
                if (big && !presorted && m > 1) block_radix_sort(keys + pos, keys2 + pos, m, warp_cnt);
                for (unsigned int piece = 0; piece < m && !s_full; piece += S.ch) {
                    const int mm = (int)min((unsigned int)S.ch, m - piece);
                    // ---- phase 1: drop what the features accepted so far suppress; ordered compaction of the rest ----
                    if (tid == 0) s_ns = 0;
                    __syncthreads();
                    for (int i0 = 0; i0 < mm; i0 += WALK_THREADS) {
                        const int i = i0 + tid;
                        bool live = i < mm;
                        unsigned long long kk = 0ull;
                        if (live) {
                            kk = keys[pos + piece + i];
                            const unsigned long long k = ~kk;
                            const int x = (int)((k >> 13) & 8191ull), y = (int)(k & 8191ull);
                            if (pm_walk && pm_walk[(size_t)y * S.W + x]) live = false;      // only a caller-ordered list can still hold these (:109-116)
                            if (live && S.r >= 0 && grid_conflict(grid, S.gw, S.gh, S.cs, S.r, x, y)) live = false;
                        }
                        const unsigned int bm = __ballot_sync(0xffffffffu, live);
                        if (lane == 0) warp_cnt[warp] = __popc(bm);
                        __syncthreads();
                        const int base = s_ns;
                        unsigned int before = 0, tot = 0;
                        for (int w = 0; w < WALK_THREADS / 32; w++) { const unsigned int c = warp_cnt[w]; if (w < warp) before += c; tot += c; }
                        if (live) sk[base + before + __popc(bm & ((1u << lane) - 1u))] = kk;
                        __syncthreads();
                        if (tid == 0) s_ns = base + (int)tot;
                        __syncthreads();
                    }
                    const int ns = s_ns;
                    if (!big && ns > 1) {
                        int P = 2;
                        while (P < ns) P <<= 1;
                        for (int i = ns + tid; i < P; i += WALK_THREADS) sk[i] = ~0ull;
                        __syncthreads();
                        bitonic_sort(sk, P);
                    }
                    // ---- phase 2: the exact greedy result by parallel rounds.  Greedy over a sorted list = the lexicographically first
                    // maximal independent set (SURVEY 7.3): a live candidate with no live candidate of smaller rank within distance r
                    // is accepted; what the accepted ones suppress dies; repeat.  "No smaller rank within r" is tested conservatively
                    // on cells: every live candidate publishes its rank with atomicMin in its cell (side r + 1), and a candidate is
                    // accepted when no cell of its 3x3 neighbourhood holds a smaller rank.  That can only delay an acceptance to a
                    // later round, never change it; the smallest live rank is always accepted, so the rounds terminate.
                    // The sorted survivors are taken in rank windows (256, 768, then 1024 at a time), one candidate per thread: a
                    // window first drops what the earlier windows' features suppress, and the walk stops with the window that
                    // fills the last slot -- replacement (a handful of slots) usually ends inside the first one.  Within a window
                    // the k-th accepted candidate in rank order takes the k-th fillable slot.
                    for (int w0 = 0; w0 < ns && !s_full; ) {
                        const int wlen = w0 == 0 ? 256 : (w0 == 256 ? 768 : WALK_THREADS);
                        const int i = w0 + tid;
                        const bool valid = tid < wlen && i < ns;
                        const unsigned long long k = valid ? ~sk[i] : 0ull;
                        const int px = (int)((k >> 13) & 8191ull), py = (int)(k & 8191ull);
                        const int ccx = px / S.cs, ccy = py / S.cs, pcell = ccy * S.gw + ccx;
                        int pst = valid ? (S.r >= 0 ? 0 : 1) : 2;                     // 0 live, 1 accepted, 2 dead / none
                        if (S.r >= 0) {
                            if (pst == 0 && w0 > 0 && grid_conflict(grid, S.gw, S.gh, S.cs, S.r, px, py)) pst = 2;
                            while (__syncthreads_count(pst == 0) != 0) {
                                if (pst == 0) atomicMin(&cellmin[pcell], (unsigned int)tid);
                                __syncthreads();
                                bool acc_now = false;
                                if (pst == 0) {
                                    unsigned int m = 0xFFFFFFFFu;
#pragma unroll
                                    for (int dy = -1; dy <= 1; dy++)
#pragma unroll
                                        for (int dx = -1; dx <= 1; dx++) {
                                            const int ncx = ccx + dx, ncy = ccy + dy;
                                            if (ncx >= 0 && ncx < S.gw && ncy >= 0 && ncy < S.gh) m = min(m, cellmin[ncy * S.gw + ncx]);
                                        }
                                    acc_now = m == (unsigned int)tid;
                                }
                                __syncthreads();                      // every read of cellmin is done
                                if (pst == 0) {
                                    cellmin[pcell] = 0xFFFFFFFFu;     // leave the array clean for the next round / window
                                    if (acc_now) {
                                        pst = 1;
                                        grid[pcell] = (unsigned short)(((px - ccx * S.cs) << 8) | (py - ccy * S.cs));
                                    }
                                }
                                __syncthreads();
                                if (pst == 0 && grid_conflict(grid, S.gw, S.gh, S.cs, S.r, px, py)) pst = 2;
                            }
                        }
                        unsigned int tot;
                        const unsigned int incl = block_scan_incl(pst == 1 ? 1u : 0u, warp_cnt, &tot);
                        const int filled = s_filled, room = slots - filled;
                        if (pst == 1 && (int)incl - 1 < room) {
                            const int slot = overwrite ? filled + (int)incl - 1 : free_slots[filled + (int)incl - 1];
                            fx[slot] = (double)px; fy[slot] = (double)py; fval[slot] = (int)__uint_as_float((unsigned int)(k >> 26));
                        }
                        __syncthreads();                              // s_filled has been read by everyone
                        if (tid == 0) {
                            s_filled = filled + ((int)tot < room ? (int)tot : room);
                            if ((int)tot >= room) s_full = 1;
                        }
                        __syncthreads();
                        w0 += wlen;
                    }
                    __syncthreads();
                    consumed += (unsigned long long)mm;
                }
                rb = e;
                __syncthreads();                          // pre[] / s_m are read above; thread 0 rewrites s_m next
            }
            if (s_full || presorted || rb_hi >= SEL_BINS - 1) break;
            // ---- fallback: the range ran out before every slot was filled: gather the next bins from the eigenvalue map ----
            fallbacks++;
            rb_lo = rb_hi + 1;
            plan_range(hist, rb_lo, target, pre, off, warp_cnt, &s_rb_hi, &s_nkeys);
            rb_hi = s_rb_hi; nkeys = s_nkeys;
            if (nkeys == 0) break;                       // nothing left above min_eigenvalue
            const float *vmap = S.vmap + (size_t)b * S.ncand;
            const unsigned char *pm = S.premap ? S.premap + (size_t)b * S.map_stride : nullptr;
            for (size_t c = tid; c < S.ncand; c += WALK_THREADS) {
                const float v = vmap[c];
                if (v >= S.min_val) {
                    const unsigned int rbk = (unsigned int)eig_rbin(v);
                    if (rbk >= rb_lo && rbk <= rb_hi) {
                        const int j = (int)(c / S.nx), i = (int)(c - (size_t)j * S.nx);
                        const int x = S.bx + i * S.step, y = S.by + j * S.step;
                        if (!(pm && pm[(size_t)y * S.W + x])) keys[atomicAdd(&off[rbk], 1u)] = make_key(v, x, y);
                    }
                }
            }
            __syncthreads();
        }
    }
    __syncthreads();
    // SELECTING_ALL: slots the walk could not fill get x = y = -1, val = KLT_NOT_FOUND (C-KLT behaviour, quirk Q6)
    if (overwrite)
        for (int f = s_filled + tid; f < n_features; f += WALK_THREADS) { fx[f] = -1.0; fy[f] = -1.0; fval[f] = KLT_NOT_FOUND; }
    if (tid == 0) {
        status[0] = consumed;
        status[1] = s_full ? 0ull : 1ull;
        status[2] = (unsigned long long)s_filled;
        status[3] = (unsigned long long)fallbacks;
    }
}

// ---------------------------------------------------------------------------------------------------------
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int klt_sel_geometry(klt_ctx *ctx, const klt_params *p, int w, int h, int n_features, int replace, SelDev *S) {
    if (w > 8191 || h > 8191) return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "image larger than 8191 pixels per side");
    // border and window exactly as selectGoodFeatures.py:168-169,215-221,230 (true division, then int truncation)
    double window_hw = p->window_width / 2.0, window_hh = p->window_height / 2.0;
    double bxd = p->borderx, byd = p->bordery;
    if (bxd < window_hw) bxd = window_hw;
    if (byd < window_hh) byd = window_hh;
    const int bx = (int)bxd, by = (int)byd, hw = (int)window_hw, hh = (int)window_hh;
    if (bx < hw + 1 || by < hh + 1)
        return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "border (%d,%d) smaller than window half-size + 1: the reference reads out of bounds here", bx, by);
    const int step = p->n_skipped_pixels + 1;
    int nx = 0, ny = 0;
    if (w - bx > bx) nx = (w - 2 * bx + step - 1) / step;
    if (h - by > by) ny = (h - 2 * by + step - 1) / step;
    const int mindist = p->mindist < 0 ? 0 : p->mindist;                 // :241-243
    const int r = mindist - 1;                                           // :61
    if (r > 254) return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "mindist larger than 255");
    memset(S, 0, sizeof *S);
    S->W = w; S->H = h; S->bx = bx; S->by = by; S->hw = hw; S->hh = hh; S->step = step; S->nx = nx; S->ny = ny;
    S->r = r; S->cs = r >= 0 ? r + 1 : 1; S->gw = (w + S->cs - 1) / S->cs; S->gh = (h + S->cs - 1) / S->cs;
    S->n_features = n_features; S->replace = replace ? 1 : 0;
    // :53 (min_eigenvalue < 1 -> 1) and :116 (val >= min_eigenvalue, a float/int comparison in the reference)
    S->min_val = p->min_eigenvalue_f > 0.f ? p->min_eigenvalue_f : (float)p->min_eigenvalue;
    if (!(S->min_val >= 1.0f)) S->min_val = 1.0f;
    S->ncand = (size_t)nx * ny;
    S->key_stride = align_up(S->ncand + 1, 32);
    S->map_stride = align_up((size_t)w * h, 256);
    S->grid_stride = align_up((size_t)S->gw * S->gh, 128);
    S->ch = ctx->select_chunk;
    // replacement mode only sees the candidates no surviving feature suppresses: a smaller first range suffices
    S->target_mul = replace ? 128u : 32u;
    S->target_add = replace ? 1024u : 8192u;
    const size_t grid_b = (size_t)S->gw * S->gh * (sizeof(unsigned short) + sizeof(unsigned int));     // cell grid + per-cell minimum rank
    const size_t fixed = (size_t)S->ch * sizeof(unsigned long long) + (2 * SEL_BINS + 4) * sizeof(unsigned int);
    S->grid_in_smem = fixed + grid_b + 2048 <= 220 * 1024 ? 1 : 0;
    return KLT_OK;
}

size_t klt_sel_workspace_bytes(const SelDev *S, int B, bool strict_sat, bool own_features) {
    size_t t = 0;
    if (strict_sat) t += align_up((size_t)B * 3 * S->W * S->H * sizeof(float), 256);
    t += align_up((size_t)B * (S->ncand + 1) * sizeof(float), 256);              // vmap
    t += align_up((size_t)B * (SEL_BINS * 3 + 1) * sizeof(unsigned int), 256);   // hist, cursor, offs
    t += align_up((size_t)B * (SEL_PLAN_WORDS * sizeof(unsigned int) + SEL_STATUS_WORDS * sizeof(unsigned long long)), 256);
    t += 2 * align_up((size_t)B * S->key_stride * sizeof(unsigned long long), 256);
    if (S->replace) t += align_up((size_t)B * S->map_stride, 256);
    if (!S->grid_in_smem) t += align_up((size_t)B * S->grid_stride * sizeof(unsigned short), 256) + align_up((size_t)B * S->grid_stride * sizeof(unsigned int), 256);
    t += align_up((size_t)B * S->n_features * sizeof(int) + 64, 256);            // free slots
    if (own_features) t += align_up((size_t)B * S->n_features * (2 * sizeof(double) + sizeof(int)) + 64, 256);
    return t + 1024;
}

void klt_sel_carve(SelDev *S, int B, bool strict_sat, bool own_features, char *base, float **sat) {
    char *p = base;
    auto take = [&](size_t bytes) { char *q = p; p += align_up(bytes, 256); return q; };
    if (sat) *sat = nullptr;
    if (strict_sat) { float *s = (float *)take((size_t)B * 3 * S->W * S->H * sizeof(float)); if (sat) *sat = s; }
    S->vmap = (float *)take((size_t)B * (S->ncand + 1) * sizeof(float));
    unsigned int *h3 = (unsigned int *)take((size_t)B * (SEL_BINS * 3 + 1) * sizeof(unsigned int));
    S->hist = h3; S->cursor = h3 + (size_t)B * SEL_BINS; S->offs = h3 + (size_t)2 * B * SEL_BINS;      // offs: [B][SEL_BINS + 1]
    char *ps = take((size_t)B * (SEL_PLAN_WORDS * sizeof(unsigned int) + SEL_STATUS_WORDS * sizeof(unsigned long long)));
    S->status = (unsigned long long *)ps; S->plan = (unsigned int *)(ps + (size_t)B * SEL_STATUS_WORDS * sizeof(unsigned long long));
    S->keys = (unsigned long long *)take((size_t)B * S->key_stride * sizeof(unsigned long long));
    S->keys2 = (unsigned long long *)take((size_t)B * S->key_stride * sizeof(unsigned long long));
    S->premap = S->replace ? (unsigned char *)take((size_t)B * S->map_stride) : nullptr;
    S->grid_global = S->grid_in_smem ? nullptr : (unsigned short *)take((size_t)B * S->grid_stride * sizeof(unsigned short));
    S->cellmin_global = S->grid_in_smem ? nullptr : (unsigned int *)take((size_t)B * S->grid_stride * sizeof(unsigned int));
    S->free_slots = (int *)take((size_t)B * S->n_features * sizeof(int) + 64);
    if (own_features) {
        char *f = take((size_t)B * S->n_features * (2 * sizeof(double) + sizeof(int)) + 64);
        S->fx = (double *)f; S->fy = S->fx + (size_t)B * S->n_features; S->fval = (int *)(S->fy + (size_t)B * S->n_features);
    }
}

static size_t walk_smem(const SelDev *S) {
    size_t s = (size_t)S->ch * sizeof(unsigned long long) + (2 * SEL_BINS + 4) * sizeof(unsigned int);
    if (S->grid_in_smem) s += (size_t)S->gw * S->gh * (sizeof(unsigned short) + sizeof(unsigned int));
    return s;
}

int klt_sel_prepare_kernels(klt_ctx *ctx, const SelDev *S) {
    // function attributes are set outside any stream capture
    KLT_CUDA(ctx, cudaFuncSetAttribute(sat_rows_vec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SatSmemV)));
    KLT_CUDA(ctx, cudaFuncSetAttribute(select_walk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)walk_smem(S)));
    KLT_CUDA(ctx, cudaFuncSetAttribute(select_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(HIST_COPIES * SEL_BINS * sizeof(unsigned int))));
    return KLT_OK;
}

// histogram reset + (replacement mode) pre-marking of the surviving features; must precede the eigen pass
int klt_sel_launch_begin(klt_ctx *ctx, const SelDev *S, int B) {
    KLT_CUDA(ctx, cudaMemsetAsync(S->hist, 0, (size_t)B * SEL_BINS * sizeof(unsigned int), ctx->stream));
    if (S->replace) {
        KLT_CUDA(ctx, cudaMemsetAsync(S->premap, 0, (size_t)B * S->map_stride, ctx->stream));
        if (S->r >= 0 && S->n_features > 0)
            KLT_LAUNCH(ctx, "premark", (double)B * S->map_stride, (premark_kernel<<<dim3(S->n_features, B), 128, 0, ctx->stream>>>(*S)));
    }
    return KLT_OK;
}

// STRICT eigenvalue map (+ histogram) of B images from their level-0 gradient planes
int klt_sel_launch_eigen_strict(klt_ctx *ctx, const SelDev *S, int B, const float *gx0, const float *gy0, size_t img_stride,
                                size_t pitch, float *sat) {
    const int w = S->W, h = S->H;
    const size_t plane = (size_t)w * h;
    const bool vec = (w % SAT_T) == 0 && (pitch % 4) == 0 && (img_stride % 4) == 0 &&
                     ((reinterpret_cast<uintptr_t>(gx0) | reinterpret_cast<uintptr_t>(gy0)) & 15) == 0;
    const dim3 grid((h + SAT_T - 1) / SAT_T, B);
    if (vec)
        KLT_LAUNCH(ctx, "sat_rows", 20.0 * plane * B, (sat_rows_vec_kernel<<<grid, 32, sizeof(SatSmemV), ctx->stream>>>(gx0, gy0, img_stride, pitch, w, h, sat, plane)));
    else
        KLT_LAUNCH(ctx, "sat_rows", 20.0 * plane * B, (sat_rows_kernel<<<grid, 32, 0, ctx->stream>>>(gx0, gy0, img_stride, pitch, w, h, sat, plane)));
    KLT_LAUNCH(ctx, "sat_cols", 24.0 * plane * B, (sat_cols_kernel<<<dim3((w + 63) / 64, 3, B), 64, 0, ctx->stream>>>(sat, plane, w, h)));
    if (S->ncand) {
        const dim3 g2((S->nx + 255) / 256, (S->ny + EIG_ROWS - 1) / EIG_ROWS, B);
        const double bytes = (12.0 * plane + 4.0 * S->ncand) * B;
        KLT_LAUNCH(ctx, "eigen", bytes, (eigen_kernel<<<g2, 256, 0, ctx->stream>>>(sat, plane, *S)));
    }
    return KLT_OK;
}

int klt_sel_launch_eigen(klt_ctx *ctx, const SelDev *S, int B, klt_pyr *pyr, int select_mode, float *sat) {
    int rc;
    if (select_mode == KLT_SELECT_FAST && pyr->hx->taps_valid) {
        rc = klt_sel_launch_eigen_fast(ctx, S, B, pyr->level(0, 0, 0), pyr->plane_floats, pyr->lv[0].pitch, &pyr->hx->taps.grad_gauss,
                                       &pyr->hx->taps.grad_deriv);
        if (rc) return rc < 0 ? rc : KLT_OK;
    }
    if ((rc = klt_ensure_gradients(ctx, pyr, 1))) return rc;
    return klt_sel_launch_eigen_strict(ctx, S, B, pyr->level(1, 0, 0), pyr->level(2, 0, 0), pyr->plane_floats, pyr->lv[0].pitch, sat);
}

// plan + scatter + walk on the eigenvalue maps and histograms of B images
int klt_sel_launch_pick(klt_ctx *ctx, const SelDev *S, int B) {
    if (S->ncand) {
        const int tiles = ((S->nx + 255) / 256) * ((S->ny + HIST_ROWS - 1) / HIST_ROWS);
        int nblk = (ctx->num_sms * 4 + B - 1) / B;           // about four blocks per SM over all images
        if (nblk > tiles) nblk = tiles;
        if (nblk < 1) nblk = 1;
        KLT_LAUNCH(ctx, "select_hist", 4.0 * S->ncand * B, (select_hist_kernel<<<dim3(nblk, B), 256, HIST_COPIES * SEL_BINS * sizeof(unsigned int), ctx->stream>>>(*S)));
    }
    KLT_LAUNCH(ctx, "select_plan", 0.0, (select_plan_kernel<<<B, WALK_THREADS, 0, ctx->stream>>>(*S)));
    if (S->ncand)
        KLT_LAUNCH(ctx, "select_scatter", 4.0 * S->ncand * B, (select_scatter_kernel<<<dim3((S->nx + 255) / 256, (S->ny + SCAT_ROWS - 1) / SCAT_ROWS, B), 256, 0, ctx->stream>>>(*S)));
    KLT_LAUNCH(ctx, "select_walk", 0.0, (select_walk_kernel<<<B, WALK_THREADS, walk_smem(S), ctx->stream>>>(*S, 0)));
    return KLT_OK;
}

int klt_launch_scan(klt_ctx *ctx, const float *gx, const float *gy, size_t pitch, int w, int h, int bx, int by, int hw,
                    int hh, int skip, float *val_dev, int nx, int ny) {
    SelDev S;
    memset(&S, 0, sizeof S);
    S.W = w; S.H = h; S.bx = bx; S.by = by; S.hw = hw; S.hh = hh; S.step = skip + 1; S.nx = nx; S.ny = ny;
    S.ncand = (size_t)nx * ny; S.vmap = val_dev; S.min_val = 1.f;
    const size_t plane = align_up((size_t)w * h * sizeof(float), 256);
    int rc = klt_ws_reserve(ctx, 3 * plane);
    if (rc) return rc;
    if ((rc = klt_sel_prepare_kernels_scan(ctx, &S))) return rc;
    return klt_sel_launch_eigen_strict(ctx, &S, 1, gx, gy, 0, pitch, (float *)ctx->ws);
}

int klt_sel_prepare_kernels_scan(klt_ctx *ctx, const SelDev *S) {
    (void)S;
    KLT_CUDA(ctx, cudaFuncSetAttribute(sat_rows_vec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SatSmemV)));
    return KLT_OK;
}

// Full selection for B images with host or device feature arrays [B][n_features]; synchronises only to hand host arrays back.
// Source: the level-0 planes of `pyr` (all its images), or explicit device gradient images (pyr == NULL, B images img_stride apart).
int klt_select_batch(klt_ctx *ctx, const klt_params *p, int select_mode, klt_pyr *pyr, const float *gx0, const float *gy0,
                     size_t img_stride, size_t pitch, int w, int h, int B, int n_features, int replace, double *x, double *y,
                     int32_t *val, int64_t *n_consumed) {
    SelDev S;
    int rc = klt_sel_geometry(ctx, p, w, h, n_features, replace, &S);
    if (rc) return rc;
    const bool host = !klt_is_device_ptr(x);
    if (host != !klt_is_device_ptr(y) || host != !klt_is_device_ptr(val)) return klt_fail(ctx, KLT_ERR_INVALID, "x, y, val must all be host or all be device");
    if ((rc = klt_ws_reserve(ctx, klt_sel_workspace_bytes(&S, B, true, host)))) return rc;
    float *sat;
    klt_sel_carve(&S, B, true, host, (char *)ctx->ws, &sat);
    const size_t total = (size_t)B * n_features;
    if (host) {
        if (replace) {
            KLT_CUDA(ctx, cudaMemcpyAsync(S.fx, x, total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            KLT_CUDA(ctx, cudaMemcpyAsync(S.fy, y, total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            KLT_CUDA(ctx, cudaMemcpyAsync(S.fval, val, total * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        }
    } else { S.fx = x; S.fy = y; S.fval = val; }
    if ((rc = klt_sel_prepare_kernels(ctx, &S))) return rc;
    if ((rc = klt_sel_launch_begin(ctx, &S, B))) return rc;
    rc = pyr ? klt_sel_launch_eigen(ctx, &S, B, pyr, select_mode, sat) : klt_sel_launch_eigen_strict(ctx, &S, B, gx0, gy0, img_stride, pitch, sat);
    if (rc) return rc;
    if ((rc = klt_sel_launch_pick(ctx, &S, B))) return rc;
    if (host) {
        KLT_CUDA(ctx, cudaMemcpyAsync(x, S.fx, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(y, S.fy, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(val, S.fval, total * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (host || n_consumed) {
        unsigned long long st[SEL_STATUS_WORDS] = {0, 0, 0, 0};
        KLT_CUDA(ctx, cudaMemcpyAsync(st, S.status, sizeof st, cudaMemcpyDeviceToHost, ctx->stream));
        KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (n_consumed) *n_consumed = (int64_t)st[0];
    }
    return KLT_OK;
}

// eigenvalue maps of every image of a pyramid batch by either method (diagnostics and tests): val [B][ny][nx], host or device
int klt_eigen_maps(klt_ctx *ctx, const klt_params *p, int select_mode, klt_pyr *pyr, float *val, int *nx_out, int *ny_out) {
    SelDev S;
    int rc = klt_sel_geometry(ctx, p, pyr->w, pyr->h, 1, 0, &S);
    if (rc) return rc;
    const int B = pyr->batch;
    if (nx_out) *nx_out = S.nx;
    if (ny_out) *ny_out = S.ny;
    if (!val || !S.ncand) return KLT_OK;
    if (select_mode == KLT_SELECT_FAST && pyr->hx->taps_valid && !klt_sel_fast_covers(&S, &pyr->hx->taps.grad_gauss, &pyr->hx->taps.grad_deriv))
        return klt_fail(ctx, KLT_ERR_UNSUPPORTED, "the fused eigenvalue pass does not cover this window / gradient kernel");
    if ((rc = klt_ws_reserve(ctx, klt_sel_workspace_bytes(&S, B, true, false)))) return rc;
    float *sat;
    klt_sel_carve(&S, B, true, false, (char *)ctx->ws, &sat);
    if ((rc = klt_sel_prepare_kernels(ctx, &S))) return rc;
    if ((rc = klt_sel_launch_begin(ctx, &S, B))) return rc;
    if ((rc = klt_sel_launch_eigen(ctx, &S, B, pyr, select_mode, sat))) return rc;
    KLT_CUDA(ctx, cudaMemcpyAsync(val, S.vmap, (size_t)B * S.ncand * sizeof(float), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}

// _enforceMinimumDistance on a caller-provided, already ordered candidate list (selectGoodFeatures.py:45-135):
// keys_host[i] = ~((val_bits << 26) | (x << 13) | y) in walk order.
int klt_greedy_presorted(klt_ctx *ctx, const unsigned long long *keys_host, unsigned int nk, int w, int h, int mindist,
                         int n_features, int overwrite, double *x, double *y, int32_t *val) {
    klt_params p;
    memset(&p, 0, sizeof p);
    p.window_width = p.window_height = 3; p.borderx = p.bordery = 2; p.mindist = mindist; p.min_eigenvalue = 1;
    SelDev S;
    int rc = klt_sel_geometry(ctx, &p, w, h, n_features, overwrite ? 0 : 1, &S);
    if (rc) return rc;
    S.ncand = nk; S.key_stride = align_up((size_t)nk + 1, 32);        // the key buffer holds the caller's list
    if ((rc = klt_ws_reserve(ctx, klt_sel_workspace_bytes(&S, 1, false, true)))) return rc;
    klt_sel_carve(&S, 1, false, true, (char *)ctx->ws, nullptr);
    unsigned int plan[SEL_PLAN_WORDS] = {0};
    plan[SEL_PLAN_RB_HI] = 0; plan[SEL_PLAN_NKEYS] = nk;
    KLT_CUDA(ctx, cudaMemcpyAsync(S.plan, plan, sizeof plan, cudaMemcpyHostToDevice, ctx->stream));
    if (nk) KLT_CUDA(ctx, cudaMemcpyAsync(S.keys, keys_host, (size_t)nk * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
    if (!overwrite) {
        KLT_CUDA(ctx, cudaMemcpyAsync(S.fx, x, n_features * sizeof(double), cudaMemcpyDefault, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(S.fy, y, n_features * sizeof(double), cudaMemcpyDefault, ctx->stream));
        KLT_CUDA(ctx, cudaMemcpyAsync(S.fval, val, n_features * sizeof(int), cudaMemcpyDefault, ctx->stream));
    }
    if ((rc = klt_sel_prepare_kernels(ctx, &S))) return rc;
    if ((rc = klt_sel_launch_begin(ctx, &S, 1))) return rc;
    KLT_LAUNCH(ctx, "select_walk", 0.0, (select_walk_kernel<<<1, WALK_THREADS, walk_smem(&S), ctx->stream>>>(S, 1)));
    KLT_CUDA(ctx, cudaMemcpyAsync(x, S.fx, n_features * sizeof(double), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(y, S.fy, n_features * sizeof(double), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaMemcpyAsync(val, S.fval, n_features * sizeof(int), cudaMemcpyDefault, ctx->stream));
    KLT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KLT_OK;
}
