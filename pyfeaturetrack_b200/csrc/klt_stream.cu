// Warp-streaming pyramid kernels for the FAST (fp32) path (sm_100a).
//
// Why this shape: at level 0 the pipeline is u8 -> 5-tap smooth (h, v) -> 7-tap gradient pair (h, v for gx and gy):
// 38 FMAs per pixel for 13 bytes of compulsory traffic.  At 6.5 TB/s each SM must retire ~1.8 pixels per clock, i.e.
// ~70 FMA/clk of its 128 -- the kernel is as much issue-bound as HBM-bound, so the design goal is to spend issue slots
// on FMAs only:
//   * one WARP owns a strip of columns and marches down the rows of its segment; every lane owns 4 adjacent columns;
//   * vertical filters never touch memory: each lane keeps the 2r partially accumulated output rows of its 4 columns
//     in registers; a new input row updates them with one FMA each, and the FMA's destination register performs the
//     shift (acc[m] = fma(c, v, acc[m+1])), so there are no moves and no unrolling by the kernel length;
//   * horizontal filters get the neighbour columns from the adjacent lanes with warp shuffles (float rows) or from the
//     neighbour quads through L1 (u8 rows); no shared memory, no block barriers; lanes 0 and 31 are halo lanes whose own
//     outputs are discarded (30/32 = 94 % efficiency);
//   * no vertical halo recomputation inside a segment (a 2-D tile design recomputes ~30 %); segments overlap by the
//     filter radii only (warm-up rows);
//   * loads and stores are 128-bit (32-bit for the u8 frame: 4 pixels), coalesced along the warp's strip; the next
//     row is loaded one iteration ahead and an L2 prefetch runs a few rows further ahead.
//
// Borders: the reference filters with SciPy's mode='reflect' (half-sample symmetric).  A SYMMETRIC filter commutes with
// that extension, so the fused level-0 kernel simply reads the u8 frame through reflected row/column indices and treats
// the smoothed image on the extended domain as the reflect-extension of the smoothed image (exact in real arithmetic,
// ~1e-7 relative in fp32).  Decimation does not commute with it, so levels >= 1 run as two streaming kernels (decimate,
// then gradients) and the gradient kernel reflects its input indices directly.
// Widths are required to be multiples of 4: then every aligned quad of columns is either fully inside the image or
// fully outside, and an outside quad is the element-reversed quad at the mirrored position -- all loads stay
// branch-free 32/128-bit loads.
//
// These kernels serve KLT_PRECISION_FAST only.  STRICT (bit-exact) mode and configurations not covered here
// (other radii, widths not divisible by 4, subsampling 4/8) use the generic tiled kernels of klt_conv.cu.
#include "klt_common.cuh"

#define WARPS_PER_CTA 4
#define FULLMASK 0xffffffffu
#define PREFETCH_ROWS 6

struct StreamTaps {
    // c[j] multiplies in[x + j - r] (convolution order), zero padded and centred in a fixed-radius slot
    float p[12];     // pyramid gauss (radius 5) + one zero; first, so that the pairs (p[2m], p[2m+1]) are 8-byte aligned in the
                     // parameter bank and the packed kernels can read them as uniform register pairs
    float s[9];      // level-0 smoothing gauss (radius <= 4)
    float g[7];      // gradient gauss / deriv (radius 3)
    float d[7];
};

// single reflection (|overshoot| < n is guaranteed by the launchers)
__device__ __forceinline__ int reflect1(int i, int n) { return i < 0 ? -i - 1 : (i >= n ? 2 * n - i - 1 : i); }
// quad starting at column c (multiple of 4), W % 4 == 0: position of the quad to load and whether to reverse it
// (quads further than one quad beyond the image only feed discarded outputs; their address is clamped into the image)
__device__ __forceinline__ int mirror_quad(int c, int W, bool &rev) {
    rev = c < 0 || c >= W;
    const int m = c < 0 ? -c - 4 : (c >= W ? 2 * W - c - 4 : c);
    return min(max(m, 0), W - 4);
}
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// one I2F.U8 with a byte selector (conversion pipe, a quarter of the FMA rate -- plenty for 4..8 pixels per lane-row)
__device__ __forceinline__ float u8_byte_to_f32(unsigned int word, int byte) { return (float)((word >> (8 * byte)) & 0xffu); }

// vertical accumulate-and-shift: returns the completed output row value; acc[m] <- acc[m+1] + c[2R-1-m]*v
template <int R>
__device__ __forceinline__ float vacc(float (&acc)[2 * R], const float *c, float v) {
    const float out = fmaf(c[2 * R], v, acc[0]);
#pragma unroll
    for (int m = 0; m < 2 * R - 1; m++) acc[m] = fmaf(c[2 * R - 1 - m], v, acc[m + 1]);
    acc[2 * R - 1] = c[0] * v;
    return out;
}

// ---- gradient stage shared by the level-0 kernel and the gradient-only kernel -----------------------------------
struct GradState {
    float ax[4][6], ay[4][6];   // pending gx / gy rows (radius 3)
};
__device__ __forceinline__ void grad_init(GradState &st) {
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int m = 0; m < 6; m++) { st.ax[i][m] = 0.f; st.ay[i][m] = 0.f; }
}
// s[0..3] = this lane's 4 columns of the (smoothed) image row; neighbours come from lanes +-1.
__device__ __forceinline__ void grad_row(GradState &st, const StreamTaps &T, const float (&s)[4], float4 &gx, float4 &gy) {
    float e[10];                 // columns c-3 .. c+6
    e[0] = __shfl_up_sync(FULLMASK, s[1], 1);
    e[1] = __shfl_up_sync(FULLMASK, s[2], 1);
    e[2] = __shfl_up_sync(FULLMASK, s[3], 1);
    e[3] = s[0]; e[4] = s[1]; e[5] = s[2]; e[6] = s[3];
    e[7] = __shfl_down_sync(FULLMASK, s[0], 1);
    e[8] = __shfl_down_sync(FULLMASK, s[1], 1);
    e[9] = __shfl_down_sync(FULLMASK, s[2], 1);
    float ox[4], oy[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float hd = T.d[0] * e[i], hg = T.g[0] * e[i];
#pragma unroll
        for (int j = 1; j < 7; j++) { hd = fmaf(T.d[j], e[i + j], hd); hg = fmaf(T.g[j], e[i + j], hg); }
        ox[i] = vacc<3>(st.ax[i], T.g, hd);      // gx = gauss_v( deriv_h )
        oy[i] = vacc<3>(st.ay[i], T.d, hg);      // gy = deriv_v( gauss_h )
    }
    gx = make_float4(ox[0], ox[1], ox[2], ox[3]);
    gy = make_float4(oy[0], oy[1], oy[2], oy[3]);
}

// ---- level 0: u8 frame -> smoothed image, gradx, grady -----------------------------------------------------------
// Lane l of a warp owns columns c = 120*strip + 4*(l-1) .. c+3; lanes 1..30 store outputs.
template <int RS>
struct L0State {
    const unsigned char *b0, *bl, *br;     // frame base + (mirrored) column of the own / left / right quad
    unsigned int sel0, sell, selr;          // byte-reversal selectors for mirrored quads
    unsigned int w0, wl, wr;                // quads of the row loaded one iteration ahead
    float sa[4][2 * RS];                    // pending smoothed rows
    GradState gs;
    float *p_img, *p_gx, *p_gy;             // next output rows
    size_t opitch;                          // output pitch in floats
    unsigned int pitch;
    int H, ys, ye, t1, writer;
};

// One input row t: finish smoothed row r = t - RS, feed it to the gradient stage (finishing gradient row r - 3).
// LEAN = steady state of a segment: every store happens, no warm-up tests.
template <int RS, bool LEAN>
__device__ __forceinline__ void l0_row(L0State<RS> &S, const StreamTaps &T, int t) {
    // ---- consume the row loaded one iteration ago, then immediately issue the next row's loads ----
    // (the halo lanes 0 and 31 need their OUTER neighbour columns too -- their smoothed values feed the gradient stage of
    // lanes 1 and 30 -- so every lane reads its neighbour quads through L1 instead of shuffling them)
    const unsigned int q0 = __byte_perm(S.w0, 0u, S.sel0), ql = __byte_perm(S.wl, 0u, S.sell), qr = __byte_perm(S.wr, 0u, S.selr);
    float u[4 + 2 * RS];                             // columns c-RS .. c+3+RS
#pragma unroll
    for (int i = 0; i < 4; i++) u[RS + i] = u8_byte_to_f32(q0, i);
#pragma unroll
    for (int k = 0; k < RS; k++) {
        u[k] = u8_byte_to_f32(ql, 4 - RS + k);
        u[RS + 4 + k] = u8_byte_to_f32(qr, k);
    }
    {
        const unsigned int ro = (unsigned int)reflect1(min(t + 1, S.t1 - 1), S.H) * S.pitch;
        S.w0 = __ldg(reinterpret_cast<const unsigned int *>(S.b0 + ro));
        S.wl = __ldg(reinterpret_cast<const unsigned int *>(S.bl + ro));
        S.wr = __ldg(reinterpret_cast<const unsigned int *>(S.br + ro));
        const int tp = t + PREFETCH_ROWS;
        if (tp < S.t1) prefetch_l2(S.b0 + (unsigned int)reflect1(tp, S.H) * S.pitch);
    }
    // ---- horizontal + vertical smooth ----
    float s[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float h = T.s[0] * u[i];
#pragma unroll
        for (int j = 1; j < 2 * RS + 1; j++) h = fmaf(T.s[j], u[i + j], h);
        s[i] = vacc<RS>(S.sa[i], T.s, h);
    }
    const int r = t - RS;
    if (!LEAN && r < S.ys - 3) return;                   // vertical smooth still warming up (warp-uniform)
    if (LEAN || (r >= S.ys && r < S.ye)) {
        if (S.writer) *reinterpret_cast<float4 *>(S.p_img) = make_float4(s[0], s[1], s[2], s[3]);
        S.p_img += S.opitch;
    }
    float4 gx, gy;
    grad_row(S.gs, T, s, gx, gy);                        // completes gradient row q = r - 3
    if (LEAN || r - 3 >= S.ys) {                         // q < ye by construction
        if (S.writer) {
            __stcs(reinterpret_cast<float4 *>(S.p_gx), gx);      // gradients are not re-read by the build: stream them
            __stcs(reinterpret_cast<float4 *>(S.p_gy), gy);      // past L2 so that the smoothed image stays resident
        }
        S.p_gx += S.opitch;
        S.p_gy += S.opitch;
    }
}

template <int RS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
stream_level0_kernel(const unsigned char *__restrict__ frames, size_t pitch, size_t frame_stride, float *__restrict__ img,
                     float *__restrict__ gxo, float *__restrict__ gyo, int out_pitch, size_t out_stride, int W, int H,
                     int rows_per_seg, int n_strips, const __grid_constant__ StreamTaps T) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x * WARPS_PER_CTA + warp;
    if (strip >= n_strips) return;
    const int ys = blockIdx.y * rows_per_seg, ye = min(H, ys + rows_per_seg);
    const int c = strip * 120 + 4 * (lane - 1);
    const unsigned char *src = frames + (size_t)blockIdx.z * frame_stride;
    L0State<RS> S;
    // own quad and the two neighbour quads (through L1: the neighbour lanes load them as their own)
    bool rv0, rvl, rvr;
    const int m0 = mirror_quad(c, W, rv0), ml = mirror_quad(c - 4, W, rvl), mr = mirror_quad(c + 4, W, rvr);
    S.b0 = src + m0; S.bl = src + ml; S.br = src + mr;
    S.sel0 = rv0 ? 0x0123u : 0x3210u; S.sell = rvl ? 0x0123u : 0x3210u; S.selr = rvr ? 0x0123u : 0x3210u;
    S.writer = (lane >= 1 && lane <= 30 && c < W) ? 1 : 0;
    const size_t ooff = (size_t)blockIdx.z * out_stride + (size_t)c + (size_t)ys * out_pitch;
    S.p_img = img + ooff; S.p_gx = gxo + ooff; S.p_gy = gyo + ooff;
    S.opitch = (size_t)out_pitch; S.pitch = (unsigned int)pitch;
    S.H = H; S.ys = ys; S.ye = ye;
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int m = 0; m < 2 * RS; m++) S.sa[i][m] = 0.f;
    grad_init(S.gs);

    const int t0 = ys - 3 - RS, t1 = ye + 3 + RS;       // input rows [t0, t1) of the reflect-extended frame
    S.t1 = t1;
    {
        const unsigned int ro = (unsigned int)reflect1(t0, H) * S.pitch;
        S.w0 = __ldg(reinterpret_cast<const unsigned int *>(S.b0 + ro));
        S.wl = __ldg(reinterpret_cast<const unsigned int *>(S.bl + ro));
        S.wr = __ldg(reinterpret_cast<const unsigned int *>(S.br + ro));
    }
    // warm-up rows and the first three stored rows (tests inside), the steady state (no tests), the last three rows
    int t = t0;
    const int lean0 = min(ys + 3 + RS, t1), lean1 = max(lean0, ye + RS);
    for (; t < lean0; t++) l0_row<RS, false>(S, T, t);
    for (; t < lean1; t++) l0_row<RS, true>(S, T, t);
    for (; t < t1; t++) l0_row<RS, false>(S, T, t);
}

// ---- level 0 of an image-only pyramid: u8 frame -> smoothed image (KLT_PRECISION_FAST_WINDOWED) -----------------------
// The strip/lane geometry of stream_level0_kernel without the gradient stage: 1 B read + 4 B written per pixel,
// 2*(2*RS+1) FMAs.  With so little arithmetic per byte the row loop is kept minimal: each lane loads and converts only its own
// quad (the RS neighbour columns come from the adjacent lanes by shuffle), and segments that do not touch the top/bottom
// border walk a running row offset (no reflection arithmetic).
// sm_100 has packed fp32 arithmetic (PTX fma.rn.f32x2, SASS
// FFMA2: two FMAs per issue slot, a scalar multiplier may come from the uniform register file), so here one warp marches
// down TWO adjacent strips A and B = A + 120 columns and every filter value lives in a 64-bit register pair (A, B):
// the horizontal taps and the pending vertical sums are FFMA2s on such pairs, the conversions and shuffles write the two
// halves of a pair directly (no packing moves), and the LAST vertical FMA of a row runs as two scalar FFMAs whose
// destinations are the four consecutive registers each 128-bit store needs (no unpacking moves either): 44 floating
// point instructions per 8 pixels instead of 80, 46 instead of 65 instructions per 4 pixels overall.  An image of one strip
// (W <= 120) leaves strip B wholly outside: its loads are clamped into the image and its stores are off.
// The instruction count is not what bounds this kernel: a scalar one-strip-per-warp version (30 % more instructions) and a
// version with whole-row CTAs that stored through bulk copies took the same 123-124 us per 64 x 1080p on a B200, because a
// trivial kernel with the same 1 : 4 read/write mix and size stops at 119 us (tools/mix_probe.cu, DESIGN "How close are the
// streaming kernels ...").  This one stays for its fewer instructions (less power), and it is the first user of the packed
// idiom the fused kernel below depends on.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) { f32x2 d; asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(a), "f"(b)); return d; }
__device__ __forceinline__ float lo2(f32x2 v) { [[maybe_unused]] float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return a; }
__device__ __forceinline__ float hi2(f32x2 v) { [[maybe_unused]] float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return b; }
__device__ __forceinline__ f32x2 fma2(float c, f32x2 v, f32x2 acc) {
    f32x2 d; const f32x2 cc = pack2(c, c);
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(cc), "l"(v), "l"(acc));
    return d;
}
__device__ __forceinline__ f32x2 mul2(float c, f32x2 v) {
    f32x2 d; const f32x2 cc = pack2(c, c);
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(cc), "l"(v));
    return d;
}

template <int RS, bool INTERIOR, bool STORE>
__device__ __forceinline__ void smooth0x2_row(const unsigned char *__restrict__ bA, const unsigned char *__restrict__ bB,
                                              unsigned int &offs, unsigned int &wA, unsigned int &wB, unsigned int selA,
                                              unsigned int selB, unsigned int upitch, unsigned int pf_delta, int H, int t, int t1,
                                              bool writerA, bool writerB, float *&pA, float *&pB, int out_pitch,
                                              f32x2 (&sa)[4][2 * RS], const StreamTaps &T) {
    const unsigned int qA = __byte_perm(wA, 0u, selA), qB = __byte_perm(wB, 0u, selB);
    float uA[4], uB[4];
#pragma unroll
    for (int i = 0; i < 4; i++) { uA[i] = u8_byte_to_f32(qA, i); uB[i] = u8_byte_to_f32(qB, i); }
    if (INTERIOR) {
        offs += upitch;                                            // one row past the segment is still inside the image
        wA = __ldg(reinterpret_cast<const unsigned int *>(bA + offs));
        wB = __ldg(reinterpret_cast<const unsigned int *>(bB + offs));
        prefetch_l2(bA + offs + pf_delta);                         // lanes 0..15 pull strip A's line, 16..31 strip B's
    } else {
        const unsigned int ro = (unsigned int)reflect1(min(t + 1, t1 - 1), H) * upitch;
        wA = __ldg(reinterpret_cast<const unsigned int *>(bA + ro));
        wB = __ldg(reinterpret_cast<const unsigned int *>(bB + ro));
        const int tp = t + PREFETCH_ROWS;
        if (tp < t1) {
            const unsigned int rp = (unsigned int)reflect1(tp, H) * upitch;
            prefetch_l2(bA + rp);
            prefetch_l2(bB + rp);
        }
    }
    f32x2 U[4 + 2 * RS];
#pragma unroll
    for (int i = 0; i < 4; i++) U[RS + i] = pack2(uA[i], uB[i]);
#pragma unroll
    for (int k = 0; k < RS; k++) {
        U[k] = pack2(__shfl_up_sync(FULLMASK, uA[4 - RS + k], 1), __shfl_up_sync(FULLMASK, uB[4 - RS + k], 1));
        U[RS + 4 + k] = pack2(__shfl_down_sync(FULLMASK, uA[k], 1), __shfl_down_sync(FULLMASK, uB[k], 1));
    }
    float oA[4], oB[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        f32x2 h = mul2(T.s[0], U[i]);
#pragma unroll
        for (int j = 1; j < 2 * RS + 1; j++) h = fma2(T.s[j], U[i + j], h);
        // vertical accumulate-and-shift on the pair; the completed row leaves through two scalar FMAs
        if (STORE) {
            oA[i] = fmaf(T.s[2 * RS], lo2(h), lo2(sa[i][0]));
            oB[i] = fmaf(T.s[2 * RS], hi2(h), hi2(sa[i][0]));
        }
#pragma unroll
        for (int m = 0; m < 2 * RS - 1; m++) sa[i][m] = fma2(T.s[2 * RS - 1 - m], h, sa[i][m + 1]);
        sa[i][2 * RS - 1] = mul2(T.s[0], h);
    }
    if (STORE) {
        if (writerA) *reinterpret_cast<float4 *>(pA) = make_float4(oA[0], oA[1], oA[2], oA[3]);
        if (writerB) *reinterpret_cast<float4 *>(pB) = make_float4(oB[0], oB[1], oB[2], oB[3]);
        pA += out_pitch;
        pB += out_pitch;
    }
}

template <int RS, bool INTERIOR>
__device__ __forceinline__ void smooth0x2_rows(const unsigned char *__restrict__ bA, const unsigned char *__restrict__ bB,
                                               unsigned int selA, unsigned int selB, unsigned int upitch, unsigned int pf_delta,
                                               int H, int t0, int t1, bool writerA, bool writerB, float *pA, float *pB,
                                               int out_pitch, const StreamTaps &T) {
    f32x2 sa[4][2 * RS];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int m = 0; m < 2 * RS; m++) sa[i][m] = 0ull;
    unsigned int offs = (unsigned int)(INTERIOR ? t0 : reflect1(t0, H)) * upitch;
    unsigned int wA = __ldg(reinterpret_cast<const unsigned int *>(bA + offs));
    unsigned int wB = __ldg(reinterpret_cast<const unsigned int *>(bB + offs));
    int t = t0;
    for (; t < t0 + 2 * RS; t++)                       // warm-up rows: nothing to store yet (t - RS < ys)
        smooth0x2_row<RS, INTERIOR, false>(bA, bB, offs, wA, wB, selA, selB, upitch, pf_delta, H, t, t1, writerA, writerB, pA, pB,
                                           out_pitch, sa, T);
#pragma unroll 2
    for (; t < t1; t++)
        smooth0x2_row<RS, INTERIOR, true>(bA, bB, offs, wA, wB, selA, selB, upitch, pf_delta, H, t, t1, writerA, writerB, pA, pB,
                                          out_pitch, sa, T);
}

template <int RS>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
stream_smooth0x2_kernel(const unsigned char *__restrict__ frames, size_t pitch, size_t frame_stride, float *__restrict__ img,
                        int out_pitch, size_t out_stride, int W, int H, int rows_per_seg, int n_pairs,
                        const __grid_constant__ StreamTaps T) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int pair = blockIdx.x * WARPS_PER_CTA + warp;           // strips 2 * pair (A) and 2 * pair + 1 (B)
    if (pair >= n_pairs) return;
    const int ys = blockIdx.y * rows_per_seg, ye = min(H, ys + rows_per_seg);
    const int cA = pair * 240 + 4 * (lane - 1), cB = cA + 120;
    const unsigned char *src = frames + (size_t)blockIdx.z * frame_stride;
    bool rvA, rvB;
    const int mA = mirror_quad(cA, W, rvA), mB = mirror_quad(cB, W, rvB);
    const unsigned char *bA = src + mA, *bB = src + mB;
    const unsigned int selA = rvA ? 0x0123u : 0x3210u, selB = rvB ? 0x0123u : 0x3210u;
    const bool inner = lane >= 1 && lane <= 30;
    const bool writerA = inner && cA < W, writerB = inner && cB < W;
    float *pA = img + (size_t)blockIdx.z * out_stride + (size_t)ys * out_pitch + cA, *pB = pA + 120;
    const int t0 = ys - RS, t1 = ye + RS;
    const unsigned int upitch = (unsigned int)pitch;
    // L2 prefetch PREFETCH_ROWS - 1 rows below the row being loaded: the 32 lanes spread over the 248 bytes of the two
    // strips (8 bytes apart), so that every 128-byte line of the row segment is touched by one instruction
    const int pc = min(max(pair * 240 - 4 + 8 * lane, 0), W - 4);
    const unsigned int pf_delta = (PREFETCH_ROWS - 1) * upitch + (unsigned int)(pc - mA);
    if (t0 >= 0 && t1 + PREFETCH_ROWS <= H)
        smooth0x2_rows<RS, true>(bA, bB, selA, selB, upitch, pf_delta, H, t0, t1, writerA, writerB, pA, pB, out_pitch, T);
    else
        smooth0x2_rows<RS, false>(bA, bB, selA, selB, upitch, pf_delta, H, t0, t1, writerA, writerB, pA, pB, out_pitch, T);
}

// ---- gradients only: float image -> gradx, grady (levels >= 1) ---------------------------------------------------
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
stream_grad_kernel(const float *__restrict__ in, int in_pitch, size_t in_stride, float *__restrict__ gxo,
                   float *__restrict__ gyo, int out_pitch, size_t out_stride, int W, int H, int rows_per_seg,
                   int n_strips, const __grid_constant__ StreamTaps T) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x * WARPS_PER_CTA + warp;
    if (strip >= n_strips) return;
    const int ys = blockIdx.y * rows_per_seg, ye = min(H, ys + rows_per_seg);
    const int c = strip * 120 + 4 * (lane - 1);
    const float *src = in + (size_t)blockIdx.z * in_stride;
    bool rev;
    const int m0 = mirror_quad(c, W, rev);
    const bool warp_rev = __any_sync(FULLMASK, rev);      // interior warps skip the reversal code entirely
    const bool writer = lane >= 1 && lane <= 30 && c < W;
    const size_t ooff = (size_t)blockIdx.z * out_stride + (size_t)c + (size_t)ys * out_pitch;
    float *p_gx = gxo + ooff, *p_gy = gyo + ooff;
    GradState gs;
    grad_init(gs);
    const int t0 = ys - 3, t1 = ye + 3;
    float4 nxt = __ldg(reinterpret_cast<const float4 *>(src + (size_t)reflect1(t0, H) * in_pitch + m0));
    for (int t = t0; t < t1; t++) {
        float s[4] = {nxt.x, nxt.y, nxt.z, nxt.w};
        if (warp_rev && rev) { s[0] = nxt.w; s[1] = nxt.z; s[2] = nxt.y; s[3] = nxt.x; }
        {
            const int tn = min(t + 1, t1 - 1);
            nxt = __ldg(reinterpret_cast<const float4 *>(src + (size_t)reflect1(tn, H) * in_pitch + m0));
            const int tp = t + PREFETCH_ROWS;
            if (tp < t1) prefetch_l2(src + (size_t)reflect1(tp, H) * in_pitch + m0);
        }
        float4 gx, gy;
        grad_row(gs, T, s, gx, gy);
        if (t - 3 >= ys) {
            if (writer) {
                __stcs(reinterpret_cast<float4 *>(p_gx), gx);
                __stcs(reinterpret_cast<float4 *>(p_gy), gy);
            }
            p_gx += out_pitch;
            p_gy += out_pitch;
        }
    }
}

// ---- pyramid step for subsampling 2: out[Y][X] = smooth11(in)[2Y+1][2X+1] -----------------------------------------
// Lane l owns output columns X..X+3, X = 120*strip + 4*(l-1), i.e. input columns ci = 2X .. ci+7; it needs ci-4 .. ci+12.
// Lanes 0 and 31 only feed their neighbours.  Vertical: input rows arrive in (even, odd) pairs; output Y completes with
// even row 2Y+6; five partial outputs are pending per column.  A scalar form of this step issues ~225 instructions per lane
// and row pair (4 output pixels), 132 of them FFMA/FMUL, and measured co-limited by issue (60-65 % of the slots) and DRAM
// (63-72 %), so the arithmetic is packed:
//   * horizontal: the 128-bit loads deliver even-aligned column pairs (e[2k], e[2k+1]) in adjacent registers, so taps
//     (p[2m], p[2m+1]) are applied to such pairs with one FFMA2 (per-half multipliers), the two halves are added at the end
//     and the eleventh tap is a scalar FMA: 7 instead of 11 instructions per output and input row;
//   * vertical: the pending sums of output columns (0, 1) and (2, 3) are pairs, updated by FFMA2 with a uniform tap
//     (11 instead of 22 per row pair and column pair); the completed pairs are the four consecutive registers of the store;
//   * segments whose rows (including the look-ahead loads and prefetches) lie inside the image walk running pointers
//     instead of reflecting and multiplying row indices.
// 78 floating-point instructions per row pair instead of 132.  The sums are associated differently from a plain 11-tap sum
// (even and odd taps separately), so the two agree to rounding (~1e-7 relative), not bit for bit.
struct RowPair { float4 ea, eb, oa, ob; };   // even row: quads at ci, ci+4; odd row: the same

__device__ __forceinline__ f32x2 fma2v(f32x2 c, f32x2 v, f32x2 acc) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(c), "l"(v), "l"(acc));
    return d;
}
__device__ __forceinline__ f32x2 mul2v(f32x2 c, f32x2 v) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(c), "l"(v));
    return d;
}

__device__ __forceinline__ void down2p_hrow(const f32x2 (&pk)[5], float p10, float4 a, float4 b, bool warp_rev, bool rva,
                                            bool rvb, f32x2 (&h2)[2]) {
    if (warp_rev) {                                  // warp-uniform: only warps touching an image edge reverse quads
        if (rva) a = make_float4(a.w, a.z, a.y, a.x);
        if (rvb) b = make_float4(b.w, b.z, b.y, b.x);
    }
    f32x2 E[8];                                      // E[k] = input columns (ci - 4 + 2k, ci - 3 + 2k)
    E[2] = pack2(a.x, a.y); E[3] = pack2(a.z, a.w); E[4] = pack2(b.x, b.y); E[5] = pack2(b.z, b.w);
    E[0] = pack2(__shfl_up_sync(FULLMASK, b.x, 1), __shfl_up_sync(FULLMASK, b.y, 1));
    E[1] = pack2(__shfl_up_sync(FULLMASK, b.z, 1), __shfl_up_sync(FULLMASK, b.w, 1));
    const float r0 = __shfl_down_sync(FULLMASK, a.x, 1), r1 = __shfl_down_sync(FULLMASK, a.y, 1);
    const float r2 = __shfl_down_sync(FULLMASK, a.z, 1), r3 = __shfl_down_sync(FULLMASK, a.w, 1);
    const float r4 = __shfl_down_sync(FULLMASK, b.x, 1);
    E[6] = pack2(r0, r1); E[7] = pack2(r2, r3);
    const float last[4] = {b.z, r0, r2, r4};        // input column ci + 2i + 6: the eleventh tap of output X + i
    float h[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {                    // output column X+i is centred on input column ci + 2i + 1
        f32x2 acc = mul2v(pk[0], E[i]);
#pragma unroll
        for (int m = 1; m < 5; m++) acc = fma2v(pk[m], E[i + m], acc);
        h[i] = fmaf(p10, last[i], lo2(acc) + hi2(acc));
    }
    h2[0] = pack2(h[0], h[1]);
    h2[1] = pack2(h[2], h[3]);
}

template <bool INTERIOR>
__device__ __forceinline__ void down2p_rows(const float *__restrict__ src, int in_pitch, int H, int ma, int mb, bool rva, bool rvb,
                                            bool writer, float *p_out, int out_pitch, int ys, int ye, const StreamTaps &T) {
    f32x2 pk[5];
#pragma unroll
    for (int m = 0; m < 5; m++) pk[m] = pack2(T.p[2 * m], T.p[2 * m + 1]);
    f32x2 P[2][5];
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int m = 0; m < 5; m++) P[i][m] = 0ull;
    // c[j] multiplies in[2Y+1 + j - 5]; input row r contributes to output Y with j = r - 2Y + 4
    // pair j: rows 2j, 2j+1; even row 2j completes output Y = j - 3.  The loop takes two pairs per trip, so an odd number of
    // pairs starts one pair early (that pair only feeds outputs above the segment).
    const int j1 = ye + 3, j0 = ys - 2 - ((ye - ys + 5) & 1);
    const bool warp_rev = __any_sync(FULLMASK, rva || rvb);
    const size_t pitch2 = 2 * (size_t)in_pitch;
    const float *pn = src + (size_t)(INTERIOR ? 2 * j0 : 0) * in_pitch;     // INTERIOR: even row of the next pair to load
    int jn = j0;                                                            // otherwise: its index
    auto load_pair = [&](RowPair &rp) {
        const float *re, *ro;
        if (INTERIOR) { re = pn; ro = pn + in_pitch; pn += pitch2; }
        else {
            const int j = min(jn, j1 - 1);
            jn++;
            re = src + (size_t)reflect1(2 * j, H) * in_pitch; ro = src + (size_t)reflect1(2 * j + 1, H) * in_pitch;
        }
        rp.ea = __ldg(reinterpret_cast<const float4 *>(re + ma)); rp.eb = __ldg(reinterpret_cast<const float4 *>(re + mb));
        rp.oa = __ldg(reinterpret_cast<const float4 *>(ro + ma)); rp.ob = __ldg(reinterpret_cast<const float4 *>(ro + mb));
    };
    auto step = [&](const RowPair &cur, int j) {
        // L2 prefetch of pair j + 3 (INTERIOR: the load pointer stands at pair j + 2)
        if (INTERIOR) {
            prefetch_l2(pn + pitch2 + ma);
            prefetch_l2(pn + pitch2 + in_pitch + ma);
        } else if (j + 3 < j1) {
            prefetch_l2(src + (size_t)reflect1(2 * j + 6, H) * in_pitch + ma);
            prefetch_l2(src + (size_t)reflect1(2 * j + 7, H) * in_pitch + ma);
        }
        f32x2 he[2], ho[2];
        down2p_hrow(pk, T.p[10], cur.ea, cur.eb, warp_rev, rva, rvb, he);
        down2p_hrow(pk, T.p[10], cur.oa, cur.ob, warp_rev, rva, rvb, ho);
        f32x2 o[2];
#pragma unroll
        for (int i = 0; i < 2; i++) {
            // even row 2j: outputs Y=j-3..j+2 take taps 10, 8, 6, 4, 2, 0; odd row 2j+1: Y=j-2..j+2 take 9, 7, 5, 3, 1
            o[i] = fma2(T.p[10], he[i], P[i][0]);
            const f32x2 a0 = fma2(T.p[8], he[i], P[i][1]);
            const f32x2 a1 = fma2(T.p[6], he[i], P[i][2]);
            const f32x2 a2 = fma2(T.p[4], he[i], P[i][3]);
            const f32x2 a3 = fma2(T.p[2], he[i], P[i][4]);
            const f32x2 a4 = mul2(T.p[0], he[i]);
            P[i][0] = fma2(T.p[9], ho[i], a0);
            P[i][1] = fma2(T.p[7], ho[i], a1);
            P[i][2] = fma2(T.p[5], ho[i], a2);
            P[i][3] = fma2(T.p[3], ho[i], a3);
            P[i][4] = fma2(T.p[1], ho[i], a4);
        }
        if (j - 3 >= ys) {                               // Y = j - 3 < ye by construction
            if (writer) *reinterpret_cast<float4 *>(p_out) = make_float4(lo2(o[0]), hi2(o[0]), lo2(o[1]), hi2(o[1]));
            p_out += out_pitch;
        }
    };
    // two row-pair buffers, loop unrolled by two: each buffer is reloaded right after it has been consumed, one full
    // step before its next use, without register-to-register copies
    RowPair A, B;
    load_pair(A);
    load_pair(B);
    for (int j = j0; j < j1; j += 2) {
        step(A, j);
        load_pair(A);
        step(B, j + 1);
        load_pair(B);
    }
}

__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
stream_down2p_kernel(const float *__restrict__ in, int in_pitch, size_t in_stride, int W, int H, float *__restrict__ out,
                     int out_pitch, size_t out_stride, int OW, int OH, int rows_per_seg, int n_strips,
                     const __grid_constant__ StreamTaps T) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x * WARPS_PER_CTA + warp;
    if (strip >= n_strips) return;
    const int ys = blockIdx.y * rows_per_seg, ye = min(OH, ys + rows_per_seg);
    const int X = strip * 120 + 4 * (lane - 1);
    const int ci = 2 * X;
    const float *src = in + (size_t)blockIdx.z * in_stride;
    bool rva, rvb;
    const int ma = mirror_quad(ci, W, rva), mb = mirror_quad(ci + 4, W, rvb);
    const bool writer = lane >= 1 && lane <= 30 && X < OW;
    float *p_out = out + (size_t)blockIdx.z * out_stride + (size_t)ys * out_pitch + X;
    // interior: every row the loop loads (two pairs of look-ahead past the last one it needs) or prefetches (one more) is
    // inside the image: rows 2 (ys - 3) .. 2 (ye + 5) + 1
    if (ys >= 3 && 2 * (ye + 5) + 1 < H) down2p_rows<true>(src, in_pitch, H, ma, mb, rva, rvb, writer, p_out, out_pitch, ys, ye, T);
    else down2p_rows<false>(src, in_pitch, H, ma, mb, rva, rvb, writer, p_out, out_pitch, ys, ye, T);
}

// ---- levels 0 and 1 of an image-only pyramid in ONE pass --------------------------------------------------------------
// stream_smooth0 + the first stream_down2 move 5 + 5 bytes per level-0 pixel, 4 of them the re-read of the level-0 image
// that the decimation needs (64 frames no longer fit L2).  Both kernels sit at 95-97 % of what a trivial linear kernel
// reaches with their read/write mix (tools/mix_probe.cu), so the only way left to go faster is to move fewer bytes.  Round 1
// tried this fusion with scalar arithmetic and found it bound by instruction issue (0.143 ms against 0.140 ms for the two
// kernels); with packed arithmetic it fits.  A lane owns 8 level-0 columns (one 64-bit load of the frame, one 256-bit store
// of the smoothed row) = 4 level-1 columns; the smoothing runs on pairs (column i, column i + 4), its completed row leaves
// through scalar FMAs into the eight consecutive registers that are both the store's operand and the (a, b) quads the
// decimation's horizontal pass wants; even and odd smoothed rows feed the packed vertical accumulators of the decimation
// exactly as in stream_down2p_kernel.  Beyond the image the smoothed values are those of the reflect-extended frame, which
// is the reflect-extension of the smoothed image (symmetric filter; see the header comment) -- what the decimation reads
// there in the two-kernel version.  6 bytes per level-0 pixel instead of 10.
__device__ __forceinline__ int mirror_oct(int c, int W, bool &rev) {     // aligned block of 8 columns, W % 8 == 0
    rev = c < 0 || c >= W;
    const int m = c < 0 ? -c - 8 : (c >= W ? 2 * W - c - 8 : c);
    return min(max(m, 0), W - 8);
}

#define L01_WARPS 2            // warps per CTA: 8 CTAs of 2 warps per SM at 128 registers

struct L01State {
    f32x2 sa[4][4];            // pending smoothed rows: pairs (column i, column i + 4), radius 2
    f32x2 P[2][5];             // pending level-1 rows: pairs of output columns (0, 1), (2, 3)
};

// one frame row (8 bytes of the lane, already mirrored): completes smoothed row t - 2 of the lane's 8 columns (s[0..7]);
// OUT = the vertical filter is warm
template <bool OUT>
__device__ __forceinline__ void l01_smooth_row(L01State &S, uint2 w, unsigned int selx, unsigned int sely, const StreamTaps &T,
                                               float (&s)[8]) {
    const unsigned int q0 = __byte_perm(w.x, w.y, selx), q1 = __byte_perm(w.x, w.y, sely);
    float x[8];
#pragma unroll
    for (int i = 0; i < 4; i++) { x[i] = u8_byte_to_f32(q0, i); x[4 + i] = u8_byte_to_f32(q1, i); }
    const float xl0 = __shfl_up_sync(FULLMASK, x[6], 1), xl1 = __shfl_up_sync(FULLMASK, x[7], 1);
    const float xr0 = __shfl_down_sync(FULLMASK, x[0], 1), xr1 = __shfl_down_sync(FULLMASK, x[1], 1);
    // U[k] = (column k - 2, column k + 2): the windows of the first and of the second quad, side by side
    f32x2 U[8];
    U[0] = pack2(xl0, x[2]); U[1] = pack2(xl1, x[3]); U[2] = pack2(x[0], x[4]); U[3] = pack2(x[1], x[5]);
    U[4] = pack2(x[2], x[6]); U[5] = pack2(x[3], x[7]); U[6] = pack2(x[4], xr0); U[7] = pack2(x[5], xr1);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        f32x2 h = mul2(T.s[0], U[i]);
#pragma unroll
        for (int j = 1; j < 5; j++) h = fma2(T.s[j], U[i + j], h);
        if (OUT) {
            s[i] = fmaf(T.s[4], lo2(h), lo2(S.sa[i][0]));
            s[4 + i] = fmaf(T.s[4], hi2(h), hi2(S.sa[i][0]));
        }
#pragma unroll
        for (int m = 0; m < 3; m++) S.sa[i][m] = fma2(T.s[3 - m], h, S.sa[i][m + 1]);
        S.sa[i][3] = mul2(T.s[0], h);
    }
}

__device__ __forceinline__ void st256(float *p, const float (&s)[8]) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(s[0]), "f"(s[1]), "f"(s[2]), "f"(s[3]),
                 "f"(s[4]), "f"(s[5]), "f"(s[6]), "f"(s[7])
                 : "memory");
}

template <bool INTERIOR>
__device__ __forceinline__ void l01_rows(const unsigned char *__restrict__ b0, unsigned int selx, unsigned int sely,
                                         unsigned int upitch, int H, int ys, int ye, int r_end, bool writer0, bool writer1,
                                         float *p0, int pitch0, float *p1, int pitch1, int pf_rows, const StreamTaps &T) {
    L01State S;
    const unsigned int pf_bytes = (unsigned int)pf_rows * upitch;       // L2 prefetch distance below the row being loaded
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int m = 0; m < 4; m++) S.sa[i][m] = 0ull;
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int m = 0; m < 5; m++) S.P[i][m] = 0ull;
    f32x2 pk[5];
#pragma unroll
    for (int m = 0; m < 5; m++) pk[m] = pack2(T.p[2 * m], T.p[2 * m + 1]);
    // level-1 row Y needs smoothed rows 2Y - 4 .. 2Y + 6: pairs j = ys - 2 .. ye + 2 of smoothed rows (2j, 2j + 1), i.e.
    // frame rows 2 (ys - 2) - 2 .. 2 (ye + 2) + 3.  The frame rows of a pair are loaded one whole pair ahead.
    const int j0 = ys - 2, j1 = ye + 3;
    const int t0 = 2 * j0 - 2, t_last = 2 * (j1 - 1) + 3;
    unsigned int offs = (unsigned int)(INTERIOR ? t0 : 0) * upitch;       // INTERIOR: byte offset of the next row to load
    int tn = t0;                                                           // otherwise: its index
    auto load_row = [&]() -> uint2 {
        uint2 w;
        if (INTERIOR) {
            w = __ldg(reinterpret_cast<const uint2 *>(b0 + offs));
            offs += upitch;
        } else {
            w = __ldg(reinterpret_cast<const uint2 *>(b0 + (unsigned int)reflect1(min(tn, t_last), H) * upitch));
            tn++;
        }
        return w;
    };
    float s[8];
    uint2 wa = load_row(), wb = load_row();
#pragma unroll 1
    for (int k = 0; k < 2; k++) {                      // four frame rows: the smoothing filter warms up
        l01_smooth_row<false>(S, wa, selx, sely, T, s);
        wa = load_row();
        l01_smooth_row<false>(S, wb, selx, sely, T, s);
        wb = load_row();
    }
#pragma unroll 2
    for (int j = j0; j < j1; j++) {
        f32x2 he[2], ho[2];
        const int r = 2 * j;
        if (INTERIOR) prefetch_l2(b0 + offs + pf_bytes);
        else if (tn + pf_rows <= t_last) prefetch_l2(b0 + (unsigned int)reflect1(tn + pf_rows, H) * upitch);
        l01_smooth_row<true>(S, wa, selx, sely, T, s);
        wa = load_row();
        if (writer0 && r >= 2 * ys && r < r_end) st256(p0, s);
        down2p_hrow(pk, T.p[10], make_float4(s[0], s[1], s[2], s[3]), make_float4(s[4], s[5], s[6], s[7]), false, false, false, he);
        if (INTERIOR) prefetch_l2(b0 + offs + pf_bytes);
        else if (tn + pf_rows <= t_last) prefetch_l2(b0 + (unsigned int)reflect1(tn + pf_rows, H) * upitch);
        l01_smooth_row<true>(S, wb, selx, sely, T, s);
        wb = load_row();
        if (writer0 && r + 1 >= 2 * ys && r + 1 < r_end) st256(p0 + pitch0, s);
        p0 += 2 * (size_t)pitch0;
        down2p_hrow(pk, T.p[10], make_float4(s[0], s[1], s[2], s[3]), make_float4(s[4], s[5], s[6], s[7]), false, false, false, ho);
        f32x2 o[2];
#pragma unroll
        for (int i = 0; i < 2; i++) {
            o[i] = fma2(T.p[10], he[i], S.P[i][0]);
            const f32x2 a0 = fma2(T.p[8], he[i], S.P[i][1]);
            const f32x2 a1 = fma2(T.p[6], he[i], S.P[i][2]);
            const f32x2 a2 = fma2(T.p[4], he[i], S.P[i][3]);
            const f32x2 a3 = fma2(T.p[2], he[i], S.P[i][4]);
            const f32x2 a4 = mul2(T.p[0], he[i]);
            S.P[i][0] = fma2(T.p[9], ho[i], a0);
            S.P[i][1] = fma2(T.p[7], ho[i], a1);
            S.P[i][2] = fma2(T.p[5], ho[i], a2);
            S.P[i][3] = fma2(T.p[3], ho[i], a3);
            S.P[i][4] = fma2(T.p[1], ho[i], a4);
        }
        if (j - 3 >= ys) {                               // Y = j - 3 < ye by construction
            if (writer1) *reinterpret_cast<float4 *>(p1) = make_float4(lo2(o[0]), hi2(o[0]), lo2(o[1]), hi2(o[1]));
            p1 += pitch1;
        }
    }
}

// 128 registers = 8 CTAs of 2 warps per SM: 166 us per 64 x 1080p on a B200.  A 112-register budget (9 CTAs, a few spills)
// measured 170 us: more warps do not help, the kernel is near its traffic mix's ceiling.
__global__ void __maxnreg__(128)
stream_level01_kernel(const unsigned char *__restrict__ frames, size_t pitch, size_t frame_stride, float *__restrict__ img0,
                      int pitch0, float *__restrict__ img1, int pitch1, size_t out_stride, int W, int H, int OW, int OH,
                      int rows_per_seg, int n_strips, int pf_rows, const __grid_constant__ StreamTaps T) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x * L01_WARPS + warp;
    if (strip >= n_strips) return;
    const int ys = blockIdx.y * rows_per_seg, ye = min(OH, ys + rows_per_seg);
    const int c0 = strip * 240 + 8 * (lane - 1), X = strip * 120 + 4 * (lane - 1);
    bool rev;
    const int m0 = mirror_oct(c0, W, rev);
    const unsigned char *b0 = frames + (size_t)blockIdx.z * frame_stride + m0;
    const unsigned int selx = rev ? 0x4567u : 0x3210u, sely = rev ? 0x0123u : 0x7654u;
    const bool inner = lane >= 1 && lane <= 30;
    const bool writer0 = inner && c0 < W, writer1 = inner && X < OW;
    const int r_end = ye == OH ? H : 2 * ye;
    float *p0 = img0 + (size_t)blockIdx.z * out_stride + c0 + ((ptrdiff_t)2 * (ys - 2)) * pitch0;
    float *p1 = img1 + (size_t)blockIdx.z * out_stride + (size_t)ys * pitch1 + X;
    const int t0 = 2 * (ys - 2) - 2, t_end = 2 * (ye + 2) + 3 + 2 + 2 + pf_rows;
    if (t0 >= 0 && t_end < H) l01_rows<true>(b0, selx, sely, (unsigned int)pitch, H, ys, ye, r_end, writer0, writer1, p0, pitch0, p1, pitch1, pf_rows, T);
    else l01_rows<false>(b0, selx, sely, (unsigned int)pitch, H, ys, ye, r_end, writer0, writer1, p0, pitch0, p1, pitch1, pf_rows, T);
}

// ---- pyramid step for subsampling SS with a (2R+1)-tap gauss, generic form of the kernel above ------------------------
// (used for SS = 4, R = 10: the reference's DEFAULT pyramid, sigma = 0.9 * 4 -> 21 taps).
// Lane owns 4 output columns = 4*SS input columns [ci, ci + 4*SS); it needs NL = R - SS/2 more on the left and
// NR = NL + 1 on the right, all of which the adjacent lanes own.  Input rows r = SS*j + ph update the pending outputs
// Y = j + m with tap index ph - SS*m - SS/2 + R; output Y = j + m_min completes at phase 0 of period j.
template <int R> struct DownTaps { float c[2 * R + 1]; };

template <int SS, int R>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
stream_down_kernel(const float *__restrict__ in, int in_pitch, size_t in_stride, int W, int H, float *__restrict__ out,
                   int out_pitch, size_t out_stride, int OW, int OH, int rows_per_seg, int n_strips,
                   const __grid_constant__ DownTaps<R> T) {
    static_assert(SS % 2 == 0 && (R + SS / 2) % SS == 0, "the completing tap must fall on phase 0");
    constexpr int NQ = SS;                       // own quads per input row
    constexpr int NL = R - SS / 2, NR = NL + 1;
    static_assert(NL >= 0 && NR <= 4 * SS, "neighbour columns must come from the adjacent lanes");
    constexpr int M_MAX = (R - SS / 2) / SS, M_MIN = -((R + SS / 2) / SS);
    constexpr int NP = M_MAX - M_MIN;            // outputs pending between periods
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x * WARPS_PER_CTA + warp;
    if (strip >= n_strips) return;
    const int ys = blockIdx.y * rows_per_seg, ye = min(OH, ys + rows_per_seg);
    const int X = strip * 120 + 4 * (lane - 1);
    const int ci = SS * X;
    const float *src = in + (size_t)blockIdx.z * in_stride;
    int mq[NQ];
    bool rvq[NQ], any_rev = false;
#pragma unroll
    for (int q = 0; q < NQ; q++) { mq[q] = mirror_quad(ci + 4 * q, W, rvq[q]); any_rev |= rvq[q]; }
    const bool warp_rev = __any_sync(FULLMASK, any_rev);
    const bool writer = lane >= 1 && lane <= 30 && X < OW;
    float *p_out = out + (size_t)blockIdx.z * out_stride + (size_t)ys * out_pitch + X;
    float Q[4][NP];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int m = 0; m < NP; m++) Q[i][m] = 0.f;

    const int j0 = ys - M_MAX, j1 = ye - M_MIN;          // periods; period j completes output Y = j + M_MIN
    const int r_last = SS * j1 - 1;
    float4 bufA[NQ], bufB[NQ];
    auto load_row = [&](int r, float4 (&b)[NQ]) {
        const float *row = src + (size_t)reflect1(min(r, r_last), H) * in_pitch;
#pragma unroll
        for (int q = 0; q < NQ; q++) b[q] = __ldg(reinterpret_cast<const float4 *>(row + mq[q]));
    };
    // horizontal (2R+1)-tap filter at the 4 sampled columns of one buffered row
    auto hrow = [&](const float4 (&b)[NQ], float (&h)[4]) {
        float e[NL + 4 * SS + NR];
#pragma unroll
        for (int q = 0; q < NQ; q++) {
            float4 v = b[q];
            if (warp_rev && rvq[q]) v = make_float4(v.w, v.z, v.y, v.x);
            e[NL + 4 * q] = v.x; e[NL + 4 * q + 1] = v.y; e[NL + 4 * q + 2] = v.z; e[NL + 4 * q + 3] = v.w;
        }
#pragma unroll
        for (int k = 0; k < NL; k++) e[k] = __shfl_up_sync(FULLMASK, e[NL + 4 * SS - NL + k], 1);
#pragma unroll
        for (int k = 0; k < NR; k++) e[NL + 4 * SS + k] = __shfl_down_sync(FULLMASK, e[NL + k], 1);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            float acc = T.c[0] * e[SS * i];
#pragma unroll
            for (int t = 1; t < 2 * R + 1; t++) acc = fmaf(T.c[t], e[SS * i + t], acc);
            h[i] = acc;
        }
    };
    load_row(SS * j0, bufA);
    load_row(SS * j0 + 1, bufB);
    for (int j = j0; j < j1; j++) {
#pragma unroll
        for (int ph = 0; ph < SS; ph++) {
            const int r = SS * j + ph;
            float h[4];
            if (ph & 1) { hrow(bufB, h); load_row(r + 2, bufB); }
            else { hrow(bufA, h); load_row(r + 2, bufA); }
            if (ph == 0) {
                if (j + 2 < j1) prefetch_l2(src + (size_t)reflect1(min(r + 2 * SS, r_last), H) * in_pitch + mq[0]);
                float o[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    o[i] = fmaf(T.c[-SS * M_MIN - SS / 2 + R], h[i], Q[i][0]);
#pragma unroll
                    for (int k = 0; k < NP - 1; k++) Q[i][k] = fmaf(T.c[-SS * (M_MIN + 1 + k) - SS / 2 + R], h[i], Q[i][k + 1]);
                    Q[i][NP - 1] = T.c[-SS * M_MAX - SS / 2 + R] * h[i];
                }
                const int Y = j + M_MIN;
                if (Y >= ys) {                           // Y < ye by construction
                    if (writer) *reinterpret_cast<float4 *>(p_out) = make_float4(o[0], o[1], o[2], o[3]);
                    p_out += out_pitch;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int k = 0; k < NP; k++) Q[i][k] = fmaf(T.c[ph - SS * (M_MIN + 1 + k) - SS / 2 + R], h[i], Q[i][k]);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Segment height: fill the GPU with (at most) ONE wave of resident CTAs, so that equal-sized segments finish together
// and the warm-up rows (2*(radius) per segment) stay a small fraction of the work.
template <typename K>
static int pick_rows_per_seg(klt_ctx *ctx, K kernel, int H, int strip_ctas, int batch, int min_rows) {
    int per_sm = 4;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, WARPS_PER_CTA * 32, 0) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 4;
    }
    const long capacity = (long)ctx->num_sms * per_sm;
    const long columns = (long)strip_ctas * batch;
    long nseg = capacity / columns;
    if (nseg < 1) nseg = 1;
    long rows = (H + nseg - 1) / nseg;
    if (rows < min_rows) rows = min_rows;
    if (rows > H) rows = H;
    return (int)rows;
}

static bool fill_taps(const klt_kernel1d *k, float *dst, int cap) {
    if (!k || k->n > cap || !(k->n & 1)) return false;
    const int pad = (cap - k->n) / 2;                   // centre shorter kernels inside the fixed-radius slot
    for (int j = 0; j < cap; j++) dst[j] = 0.f;
    for (int j = 0; j < k->n; j++) dst[pad + j] = (float)k->taps[k->n - 1 - j];
    return true;
}
static bool is_symmetric(const klt_kernel1d *k) {
    for (int i = 0; i < k->n / 2; i++)
        if (fabs(k->taps[i] - k->taps[k->n - 1 - i]) > 2.220446049250313e-16) return false;
    return true;
}
static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Returns 1 if the streaming kernel was launched, 0 if the configuration is not covered (caller falls back), <0 on error.
int klt_stream_level0(klt_ctx *ctx, const uint8_t *frames, size_t pitch, size_t frame_stride, klt_pyr *p,
                      const klt_taps *taps, int first, int count) {
    StreamTaps T;
    const int ns = taps->smooth.n;
    if (ns != 3 && ns != 5 && ns != 7 && ns != 9) return 0;
    if (!is_symmetric(&taps->smooth)) return 0;          // the reflect-extension argument needs a symmetric smoother
    const int RS = ns / 2;
    if (!fill_taps(&taps->smooth, T.s, ns)) return 0;
    if (!fill_taps(&taps->grad_gauss, T.g, 7) || !fill_taps(&taps->grad_deriv, T.d, 7)) return 0;
    for (int j = 0; j < 12; j++) T.p[j] = 0.f;
    const int W = p->w, H = p->h;
    if (W < 16 || H < 16 || (W & 3)) return 0;
    if ((reinterpret_cast<uintptr_t>(frames) & 3) || (pitch & 3) || (frame_stride & 3)) return 0;
    const int n_strips = (W + 119) / 120;
    const int strip_ctas = (n_strips + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    int rows = 0;
    switch (RS) {
        case 1: rows = pick_rows_per_seg(ctx, stream_level0_kernel<1>, H, strip_ctas, count, 32); break;
        case 2: rows = pick_rows_per_seg(ctx, stream_level0_kernel<2>, H, strip_ctas, count, 32); break;
        case 3: rows = pick_rows_per_seg(ctx, stream_level0_kernel<3>, H, strip_ctas, count, 32); break;
        default: rows = pick_rows_per_seg(ctx, stream_level0_kernel<4>, H, strip_ctas, count, 32); break;
    }
    dim3 grid(strip_ctas, (H + rows - 1) / rows, count), block(WARPS_PER_CTA * 32);
    const double bytes = 13.0 * W * H * count;        // 1 B read + 3 x 4 B written per pixel
    float *img = p->level(0, first, 0), *gx = p->level(1, first, 0), *gy = p->level(2, first, 0);
#define LAUNCH_L0(R)                                                                                                   \
    KLT_LAUNCH(ctx, "stream_level0", bytes,                                                                            \
               (stream_level0_kernel<R><<<grid, block, 0, ctx->stream>>>(frames, pitch, frame_stride, img, gx, gy,      \
                                                                         p->lv[0].pitch, p->plane_floats, W, H, rows,  \
                                                                         n_strips, T)))
    switch (RS) {
        case 1: LAUNCH_L0(1); break;
        case 2: LAUNCH_L0(2); break;
        case 3: LAUNCH_L0(3); break;
        case 4: LAUNCH_L0(4); break;
        default: return 0;
    }
#undef LAUNCH_L0
    return 1;
}

int klt_stream_smooth0(klt_ctx *ctx, const uint8_t *frames, size_t pitch, size_t frame_stride, klt_pyr *p,
                       const klt_taps *taps, int first, int count) {
    StreamTaps T;
    const int ns = taps->smooth.n;
    if (ns != 3 && ns != 5 && ns != 7 && ns != 9) return 0;
    if (!is_symmetric(&taps->smooth)) return 0;
    const int RS = ns / 2;
    if (!fill_taps(&taps->smooth, T.s, ns)) return 0;
    for (int j = 0; j < 12; j++) T.p[j] = 0.f;
    for (int j = 0; j < 7; j++) T.g[j] = T.d[j] = 0.f;
    const int W = p->w, H = p->h;
    if (W < 16 || H < 16 || (W & 3)) return 0;
    if ((reinterpret_cast<uintptr_t>(frames) & 3) || (pitch & 3) || (frame_stride & 3)) return 0;
    const int n_strips = (W + 119) / 120;
    const double bytes = 5.0 * W * H * count;         // 1 B read + 4 B written per pixel
    float *img = p->level(0, first, 0);
    const int n_pairs = (n_strips + 1) / 2;
    const int pair_ctas = (n_pairs + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    int rows = 0;
    switch (RS) {
        case 1: rows = pick_rows_per_seg(ctx, stream_smooth0x2_kernel<1>, H, pair_ctas, count, 32); break;
        case 2: rows = pick_rows_per_seg(ctx, stream_smooth0x2_kernel<2>, H, pair_ctas, count, 32); break;
        case 3: rows = pick_rows_per_seg(ctx, stream_smooth0x2_kernel<3>, H, pair_ctas, count, 32); break;
        default: rows = pick_rows_per_seg(ctx, stream_smooth0x2_kernel<4>, H, pair_ctas, count, 32); break;
    }
    dim3 grid(pair_ctas, (H + rows - 1) / rows, count), block(WARPS_PER_CTA * 32);
#define LAUNCH_S0X2(R)                                                                                                 \
    KLT_LAUNCH(ctx, "stream_smooth0", bytes,                                                                           \
               (stream_smooth0x2_kernel<R><<<grid, block, 0, ctx->stream>>>(frames, pitch, frame_stride, img,           \
                                                                            p->lv[0].pitch, p->plane_floats, W, H,     \
                                                                            rows, n_pairs, T)))
    switch (RS) {
        case 1: LAUNCH_S0X2(1); break;
        case 2: LAUNCH_S0X2(2); break;
        case 3: LAUNCH_S0X2(3); break;
        default: LAUNCH_S0X2(4); break;
    }
#undef LAUNCH_S0X2
    return 1;
}

// levels 0 and 1 of an image-only pyramid in one launch; returns 0 when the configuration is not covered
int klt_stream_level01(klt_ctx *ctx, const uint8_t *frames, size_t pitch, size_t frame_stride, klt_pyr *p,
                       const klt_taps *taps, int first, int count) {
    if (p->n_levels < 2 || p->ss != 2) return 0;
    StreamTaps T;
    if (taps->smooth.n != 5 || !is_symmetric(&taps->smooth) || !fill_taps(&taps->smooth, T.s, 5)) return 0;
    if (taps->pyramid.n > 11 || !fill_taps(&taps->pyramid, T.p, 11)) return 0;
    T.p[11] = 0.f;
    for (int j = 5; j < 9; j++) T.s[j] = 0.f;
    for (int j = 0; j < 7; j++) { T.g[j] = 0.f; T.d[j] = 0.f; }
    const LevelDesc &a = p->lv[0], &b = p->lv[1];
    const int W = p->w, H = p->h;
    if (W < 64 || H < 32 || (W & 7) || (b.w & 3) || b.w < 8 || b.h < 8) return 0;
    if ((reinterpret_cast<uintptr_t>(frames) & 7) || (pitch & 7) || (frame_stride & 7)) return 0;
    float *img0 = p->level(0, first, 0), *img1 = p->level(0, first, 1);
    if ((reinterpret_cast<uintptr_t>(img0) & 31) || (a.pitch & 7) || (p->plane_floats & 7) || !aligned16(img1)) return 0;
    const int n_strips = (W + 239) / 240;
    const int strip_ctas = (n_strips + L01_WARPS - 1) / L01_WARPS;
    const int pf_rows = 4;                             // L2 prefetch distance in frame rows
    int per_sm = 8;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stream_level01_kernel, L01_WARPS * 32, 0) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 8;
    }
    long nseg = (long)ctx->num_sms * per_sm / ((long)strip_ctas * count);
    if (nseg < 1) nseg = 1;
    int rows = (int)((b.h + nseg - 1) / nseg);
    if (rows < 16) rows = 16;
    if (rows > b.h) rows = b.h;
    dim3 grid(strip_ctas, (b.h + rows - 1) / rows, count), block(L01_WARPS * 32);
    const double bytes = (5.0 * W * H + 4.0 * b.w * b.h) * count;     // 1 B read, 4 B + 1 B (a quarter of 4 B) written per pixel
    KLT_LAUNCH(ctx, "stream_level01", bytes,
               (stream_level01_kernel<<<grid, block, 0, ctx->stream>>>(frames, pitch, frame_stride, img0, a.pitch, img1, b.pitch,
                                                                       p->plane_floats, W, H, b.w, b.h, rows, n_strips, pf_rows, T)));
    return 1;
}

int klt_stream_grad(klt_ctx *ctx, klt_pyr *p, int level, const klt_taps *taps, int first, int count) {
    StreamTaps T;
    if (!fill_taps(&taps->grad_gauss, T.g, 7) || !fill_taps(&taps->grad_deriv, T.d, 7)) return 0;
    for (int j = 0; j < 9; j++) T.s[j] = 0.f;
    for (int j = 0; j < 12; j++) T.p[j] = 0.f;
    const LevelDesc &a = p->lv[level];
    if (a.w < 16 || a.h < 8 || (a.w & 3) || !aligned16(p->level(0, first, level)) || (p->plane_floats & 3)) return 0;
    const int n_strips = (a.w + 119) / 120;
    const int strip_ctas = (n_strips + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    const int rows = pick_rows_per_seg(ctx, stream_grad_kernel, a.h, strip_ctas, count, 8);
    dim3 grid(strip_ctas, (a.h + rows - 1) / rows, count), block(WARPS_PER_CTA * 32);
    const double bytes = 12.0 * a.w * a.h * count;
    KLT_LAUNCH(ctx, "stream_grad", bytes,
               (stream_grad_kernel<<<grid, block, 0, ctx->stream>>>(p->level(0, first, level), a.pitch, p->plane_floats,
                                                                    p->level(1, first, level), p->level(2, first, level), a.pitch,
                                                                    p->plane_floats, a.w, a.h, rows, n_strips, T)));
    return 1;
}

static int stream_down4(klt_ctx *ctx, klt_pyr *p, int level, const klt_taps *taps, int first, int count) {
    constexpr int R = 10;
    DownTaps<R> T;
    const klt_kernel1d *k = &taps->pyramid;
    if (k->n > 2 * R + 1 || !(k->n & 1)) return 0;
    const int pad = (2 * R + 1 - k->n) / 2;
    for (int j = 0; j < 2 * R + 1; j++) T.c[j] = 0.f;
    for (int j = 0; j < k->n; j++) T.c[pad + j] = (float)k->taps[k->n - 1 - j];
    const LevelDesc &a = p->lv[level - 1], &b = p->lv[level];
    if (b.w < 8 || b.h < 8 || a.w < 64 || a.h < 32 || (a.w & 3) || (b.w & 3)) return 0;
    if (!aligned16(p->level(0, first, level - 1)) || !aligned16(p->level(0, first, level)) || (p->plane_floats & 3)) return 0;
    const int n_strips = (b.w + 119) / 120;
    const int strip_ctas = (n_strips + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    const int rows = pick_rows_per_seg(ctx, stream_down_kernel<4, R>, b.h, strip_ctas, count, 8);
    dim3 grid(strip_ctas, (b.h + rows - 1) / rows, count), block(WARPS_PER_CTA * 32);
    const double bytes = 4.0 * ((double)a.w * a.h + (double)b.w * b.h) * count;
    KLT_LAUNCH(ctx, "stream_down4", bytes,
               (stream_down_kernel<4, R><<<grid, block, 0, ctx->stream>>>(p->level(0, first, level - 1), a.pitch, p->plane_floats,
                                                                          a.w, a.h, p->level(0, first, level), b.pitch,
                                                                          p->plane_floats, b.w, b.h, rows, n_strips, T)));
    return 1;
}

int klt_stream_down2(klt_ctx *ctx, klt_pyr *p, int level, const klt_taps *taps, int first, int count) {
    if (level < 1) return 0;
    if (p->ss == 4) return stream_down4(ctx, p, level, taps, first, count);
    if (p->ss != 2) return 0;
    StreamTaps T;
    if (taps->pyramid.n > 11 || !fill_taps(&taps->pyramid, T.p, 11)) return 0;
    T.p[11] = 0.f;
    for (int j = 0; j < 9; j++) T.s[j] = 0.f;
    for (int j = 0; j < 7; j++) { T.g[j] = 0.f; T.d[j] = 0.f; }
    const LevelDesc &a = p->lv[level - 1], &b = p->lv[level];
    if (b.w < 8 || b.h < 8 || a.w < 32 || a.h < 16 || (a.w & 3) || (b.w & 3)) return 0;
    if (!aligned16(p->level(0, first, level - 1)) || !aligned16(p->level(0, first, level)) || (p->plane_floats & 3)) return 0;
    const int n_strips = (b.w + 119) / 120;
    const int strip_ctas = (n_strips + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    const double bytes = 4.0 * ((double)a.w * a.h + (double)b.w * b.h) * count;
    int rows = pick_rows_per_seg(ctx, stream_down2p_kernel, b.h, strip_ctas, count, 8);
    if (!(rows & 1) && rows < b.h) rows++;           // rows + 5 row pairs per segment: even, so no extra leading pair
    dim3 grid(strip_ctas, (b.h + rows - 1) / rows, count), block(WARPS_PER_CTA * 32);
    KLT_LAUNCH(ctx, "stream_down2", bytes,
               (stream_down2p_kernel<<<grid, block, 0, ctx->stream>>>(p->level(0, first, level - 1), a.pitch, p->plane_floats,
                                                                      a.w, a.h, p->level(0, first, level), b.pitch,
                                                                      p->plane_floats, b.w, b.h, rows, n_strips, T)));
    return 1;
}
