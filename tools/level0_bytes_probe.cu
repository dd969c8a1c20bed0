// Would a byte level 0 make the image-only pair build pay?  Times the library's stream_level01 (float level 0 and float
// level 1 out) against a copy of it that stores the 8 frame bytes a lane already holds into a byte plane instead of its
// 256-bit float store of level 0 (3 instead of 6 B per level-0 pixel), alternating, with CUDA events, on 64 x 1080p.
// Then checks that the byte plane equals the frames and that level 1 is bit-identical.  DESIGN section 8 has the result.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o tools/level0_bytes_probe tools/level0_bytes_probe.cu
#include "../pyfeaturetrack_b200/csrc/klt_stream.cu"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

int klt_fail(klt_ctx *, int code, const char *, ...) { return -code; }
int klt_prof_begin(klt_ctx *, const char *, double) { return 0; }
void klt_prof_end(klt_ctx *, int) {}

// l01_rows with the level-0 store replaced: frame row t = r + 2, the row that completes smoothed row r, goes to p8
template <bool INTERIOR>
__device__ __forceinline__ void l01_rows_bytes(const unsigned char *__restrict__ b0, unsigned int selx, unsigned int sely,
                                               unsigned int upitch, int H, int ys, int ye, int r_end, bool writer0, bool writer1,
                                               unsigned char *p8, int pitch8, float *p1, int pitch1, int pf_rows, const StreamTaps &T) {
    L01State S;
    const unsigned int pf_bytes = (unsigned int)pf_rows * upitch;
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
    const int j0 = ys - 2, j1 = ye + 3;
    const int t0 = 2 * j0 - 2, t_last = 2 * (j1 - 1) + 3;
    unsigned int offs = (unsigned int)(INTERIOR ? t0 : 0) * upitch;
    int tn = t0;
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
    for (int k = 0; k < 2; k++) {
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
        if (writer0 && r + 2 >= 2 * ys && r + 2 < r_end) *reinterpret_cast<uint2 *>(p8) = wa;
        l01_smooth_row<true>(S, wa, selx, sely, T, s);
        wa = load_row();
        down2p_hrow(pk, T.p[10], make_float4(s[0], s[1], s[2], s[3]), make_float4(s[4], s[5], s[6], s[7]), false, false, false, he);
        if (INTERIOR) prefetch_l2(b0 + offs + pf_bytes);
        else if (tn + pf_rows <= t_last) prefetch_l2(b0 + (unsigned int)reflect1(tn + pf_rows, H) * upitch);
        if (writer0 && r + 3 >= 2 * ys && r + 3 < r_end) *reinterpret_cast<uint2 *>(p8 + pitch8) = wb;
        l01_smooth_row<true>(S, wb, selx, sely, T, s);
        wb = load_row();
        p8 += 2 * (size_t)pitch8;
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
        if (j - 3 >= ys) {
            if (writer1) *reinterpret_cast<float4 *>(p1) = make_float4(lo2(o[0]), hi2(o[0]), lo2(o[1]), hi2(o[1]));
            p1 += pitch1;
        }
    }
}

__global__ void __maxnreg__(128)
stream_level01_bytes_kernel(const unsigned char *__restrict__ frames, size_t pitch, size_t frame_stride, unsigned char *__restrict__ u8,
                            int pitch8, size_t stride8, float *__restrict__ img1, int pitch1, size_t out_stride, int W, int H, int OW,
                            int OH, int rows_per_seg, int n_strips, int pf_rows, const __grid_constant__ StreamTaps T) {
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
    unsigned char *p8 = u8 + (size_t)blockIdx.z * stride8 + c0 + ((ptrdiff_t)2 * (ys - 2) + 2) * pitch8;
    float *p1 = img1 + (size_t)blockIdx.z * out_stride + (size_t)ys * pitch1 + X;
    const int t0 = 2 * (ys - 2) - 2, t_end = 2 * (ye + 2) + 3 + 2 + 2 + pf_rows;
    if (t0 >= 0 && t_end < H)
        l01_rows_bytes<true>(b0, selx, sely, (unsigned int)pitch, H, ys, ye, r_end, writer0, writer1, p8, pitch8, p1, pitch1, pf_rows, T);
    else
        l01_rows_bytes<false>(b0, selx, sely, (unsigned int)pitch, H, ys, ye, r_end, writer0, writer1, p8, pitch8, p1, pitch1, pf_rows, T);
}

int main() {
    const int W = 1920, H = 1080, B = 64, OW = 960, OH = 540;
    const int pitch0 = 1920, pitch1 = 960, pitch8 = 1920;
    const size_t plane = (size_t)pitch0 * H + (size_t)pitch1 * OH + 4096;        // floats per image: level 0, level 1
    const size_t fbytes = (size_t)W * H * B;
    unsigned char *fr, *u8;
    float *img;
    if (cudaMalloc(&fr, fbytes) || cudaMalloc(&u8, (size_t)pitch8 * H * B) || cudaMalloc(&img, plane * B * 4)) {
        printf("cudaMalloc failed\n");
        return 1;
    }
    std::vector<unsigned char> h(fbytes);
    unsigned s = 12345;
    for (size_t i = 0; i < fbytes; i++) { s = s * 1664525u + 1013904223u; h[i] = s >> 24; }
    cudaMemcpy(fr, h.data(), fbytes, cudaMemcpyHostToDevice);
    StreamTaps T;
    memset(&T, 0, sizeof T);
    const float sm[5] = {0.054f, 0.244f, 0.403f, 0.244f, 0.054f};
    for (int j = 0; j < 5; j++) T.s[j] = sm[j];
    for (int j = 0; j < 11; j++) T.p[j] = 1.f / 11;
    int dev, nsm;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const int n_strips = (W + 239) / 240, strip_ctas = (n_strips + L01_WARPS - 1) / L01_WARPS, pf_rows = 4;
    int per_sm[2];
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], stream_level01_kernel, L01_WARPS * 32, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], stream_level01_bytes_kernel, L01_WARPS * 32, 0);
    printf("occupancy: float %d, byte %d CTAs per SM, %d SMs\n", per_sm[0], per_sm[1], nsm);
    float *img1 = img + (size_t)pitch0 * H;
    auto launch = [&](int bytes) {                     // segment heights as klt_stream_level01 picks them
        long nseg = (long)nsm * per_sm[bytes] / ((long)strip_ctas * B);
        if (nseg < 1) nseg = 1;
        int rows = (int)((OH + nseg - 1) / nseg);
        rows = rows < 16 ? 16 : (rows > OH ? OH : rows);
        dim3 grid(strip_ctas, (OH + rows - 1) / rows, B), block(L01_WARPS * 32);
        if (bytes)
            stream_level01_bytes_kernel<<<grid, block>>>(fr, W, (size_t)W * H, u8, pitch8, (size_t)pitch8 * H, img1, pitch1, plane, W, H,
                                                         OW, OH, rows, n_strips, pf_rows, T);
        else
            stream_level01_kernel<<<grid, block>>>(fr, W, (size_t)W * H, img, pitch0, img1, pitch1, plane, W, H, OW, OH, rows, n_strips,
                                                   pf_rows, T);
    };
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    for (int i = 0; i < 5; i++) { launch(0); launch(1); }
    cudaDeviceSynchronize();
    const int reps = 50;
    for (int round = 0; round < 4; round++)
        for (int v = 0; v < 2; v++) {
            cudaEventRecord(e0);
            for (int i = 0; i < reps; i++) launch(v);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            float ms;
            cudaEventElapsedTime(&ms, e0, e1);
            printf("round %d %s: %.2f us per launch\n", round, v ? "byte level 0 " : "float level 0", ms * 1e3f / reps);
        }
    const size_t n1 = (size_t)pitch1 * OH;
    std::vector<float> l1a(n1), l1b(n1);
    launch(0);
    cudaMemcpy(l1a.data(), img1 + plane * (B - 1), n1 * 4, cudaMemcpyDeviceToHost);
    cudaMemset(u8, 0, (size_t)pitch8 * H * B);
    cudaMemset(img1 + plane * (B - 1), 0, n1 * 4);
    launch(1);
    cudaMemcpy(l1b.data(), img1 + plane * (B - 1), n1 * 4, cudaMemcpyDeviceToHost);
    std::vector<unsigned char> hb(fbytes);
    cudaMemcpy(hb.data(), u8, fbytes, cudaMemcpyDeviceToHost);
    const cudaError_t e = cudaDeviceSynchronize();
    const bool same8 = memcmp(hb.data(), h.data(), fbytes) == 0, same1 = memcmp(l1a.data(), l1b.data(), n1 * 4) == 0;
    printf("byte plane == frames: %d, level 1 identical: %d, CUDA: %s\n", same8, same1, cudaGetErrorString(e));
    return same8 && same1 && e == cudaSuccess ? 0 : 1;
}
