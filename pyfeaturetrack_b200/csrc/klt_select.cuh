// Shared by the selection translation units (klt_select.cu, klt_select_fast.cu) and their callers (klt_api.cu,
// klt_sequence.cu): the by-value kernel argument that describes a batch of selections and the launch helpers.
#pragma once
#include "klt_common.cuh"

#define SEL_BINS 4096            // histogram of the eigenvalues: exponent + 7 mantissa bits, reversed (bin 0 = largest values)
#define WALK_THREADS 1024
#define SEL_PLAN_WORDS 4         // per image: [0] last reversed bin of the planned range (0xFFFFFFFF: nothing to do), [1] keys, [2] slots
#define SEL_PLAN_RB_HI 0
#define SEL_PLAN_NKEYS 1
#define SEL_PLAN_SLOTS 2
#define SEL_STATUS_WORDS 4       // per image: [0] candidates consumed, [1] 1 if they ran out, [2] slots filled, [3] fallback ranges used

struct SelDev {
    // geometry (selectGoodFeatures.py:168-169,215-230) and suppression grid
    int W, H, bx, by, hw, hh, step, nx, ny;
    int r, cs, gw, gh, grid_in_smem;
    int n_features, replace;
    float min_val;
    int ch;                           // chunk capacity of the walk (power of two)
    unsigned int target_mul, target_add;
    size_t ncand, key_stride, map_stride, grid_stride;
    // per-image buffers, image b at index b * stride
    float *vmap;                      // [B][ncand] eigenvalue map, row-major over (y, x) candidates
    unsigned int *hist, *offs, *cursor;   // [B][SEL_BINS]
    unsigned int *plan;               // [B][SEL_PLAN_WORDS]
    unsigned long long *status;       // [B][SEL_STATUS_WORDS]
    unsigned long long *keys, *keys2; // [B][key_stride]
    unsigned char *premap;            // [B][map_stride], replacement mode only
    unsigned short *grid_global;      // [B][grid_stride] when the cell grid does not fit in shared memory
    unsigned int *cellmin_global;     // [B][grid_stride] ditto, the per-cell minimum live rank of the walk's rounds
    int *free_slots;                  // [B][n_features]
    double *fx, *fy;                  // [B][n_features] feature lists, updated in place
    int *fval;
};

// reversed histogram bin of an eigenvalue >= 1: ascending bin = descending value
__device__ __forceinline__ int eig_rbin(float v) {
    const int rb = 0x4F7F - (int)(__float_as_uint(v) >> 16);
    return min(max(rb, 0), SEL_BINS - 1);
}

int klt_sel_geometry(klt_ctx *ctx, const klt_params *p, int w, int h, int n_features, int replace, SelDev *S);
size_t klt_sel_workspace_bytes(const SelDev *S, int B, bool strict_sat, bool own_features);
void klt_sel_carve(SelDev *S, int B, bool strict_sat, bool own_features, char *base, float **sat);
int klt_sel_prepare_kernels(klt_ctx *ctx, const SelDev *S);          // cudaFuncSetAttribute calls: outside stream capture
int klt_sel_prepare_kernels_scan(klt_ctx *ctx, const SelDev *S);
int klt_sel_launch_begin(klt_ctx *ctx, const SelDev *S, int B);
int klt_sel_launch_eigen_strict(klt_ctx *ctx, const SelDev *S, int B, const float *gx0, const float *gy0, size_t img_stride,
                                size_t pitch, float *sat);
// FAST eigenvalue map straight from the level-0 intensity planes (klt_select_fast.cu), where klt_sel_fast_covers says so
bool klt_sel_fast_covers(const SelDev *S, const klt_kernel1d *gauss, const klt_kernel1d *deriv);
int klt_sel_launch_eigen_fast(klt_ctx *ctx, const SelDev *S, int B, const float *img0, size_t img_stride, size_t pitch,
                              const klt_kernel1d *gauss, const klt_kernel1d *deriv);
// eigenvalue maps of the level-0 planes of every image of a built pyramid: the fused pass if select_mode is KLT_SELECT_FAST
// and it covers the configuration, else level 0's gradient planes (built now if the build left them out) and the table pass
int klt_sel_launch_eigen(klt_ctx *ctx, const SelDev *S, int B, klt_pyr *pyr, int select_mode, float *sat);
int klt_sel_launch_pick(klt_ctx *ctx, const SelDev *S, int B);
