// Shared definitions of the surfel rasteriser kernels (sm_100a).
// Algorithm: github.com/hbb1/diff-surfel-rasterization as called by
// /root/reference/nsr/gs_surfel.py:85-114; constants per SURVEY.md App. A.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define GA_BLOCK_X 16
#define GA_BLOCK_Y 16
#define GA_NEAR_N 0.2f
#define GA_FAR_N 100.0f
#define GA_FILTER_SIZE 0.707106f
#define GA_FILTER_INV_SQUARE 2.0f
#define GA_CUTOFF 3.0f
#define GA_REC_F 24
#define GA_GRAD_F 18

// record float offsets (6 x float4):
//  q0 = Tu.x Tu.y Tu.z Tv.x | q1 = Tv.y Tv.z Tw.x Tw.y | q2 = Tw.z xy.x xy.y opacity
//  q3 = n.x n.y n.z r        | q4 = bbox x0 x1 y0 y1    | q5 = g b - -
// gradient accumulator float offsets:
//  0-8 dL/dT (Tu,Tv,Tw) | 9-10 dL/dmean2D | 11-13 dL/dnormal | 14 dL/dopacity | 15-17 dL/drgb

struct RasterDims {
    int batch, P, views, NV;   // NV = batch*views images
    int H, W, gx, gy, T;       // T = gx*gy tiles per image
    float scale_modifier;
    int64_t max_instances;
    // the two unpinned judgement calls of the restatement (DESIGN.md 1), switchable so that pinning against
    // upstream is a flip of the defaults below; ga_raster_set_variant() overrides them at run time (tests)
    int list_k;                // > 0: the forward records every pixel's contributions (<= list_k per pixel), see RasterWs.lists
    int radius_formula;        // 0: ceil(max(ex, ey, 3*FilterSize))   1: ceil(3*max(ex, ey, FilterSize))
    int quat_norm_grad;        // 0: quaternion vjp not chained through q/|q| (upstream)   1: chained
};
#ifndef GA_RADIUS_FORMULA
#define GA_RADIUS_FORMULA 0
#endif
#ifndef GA_QUAT_NORM_GRAD
#define GA_QUAT_NORM_GRAD 0
#endif

struct RasterWs {
    int32_t *status;
    float *rec;
    float *depth;
    uint32_t *rect;
    uint32_t *tile_count;
    uint32_t *tile_start;
    unsigned long long *keys;
    uint32_t *ids;
    float *final_T;
    int32_t *n_contrib;
    // per-pixel contribution lists written by the forward when list_k > 0 (the backward then neither culls nor
    // re-evaluates pairs): entry k of pixel p of tile t at lists[(t * list_k + k) * 256 + p] = {list position, alpha
    // bits, depth bits, 0}; n_list[pixel] = contributions of the pixel; tile_flag[t] = 1 when a pixel of the tile had
    // more than list_k (that tile's backward recomputes instead)
    uint4 *lists;
    int32_t *n_list;
    uint32_t *tile_flag;
    uint32_t *tile_rec_start;  // (list_k > 0) [NV*T + 1] slice layout of the backward's record buffer, computed by the forward
    uint32_t *inst_off;        // backward (split path): start of every instance's record slice
    uint32_t *inst_cnt;        // ... and the number of records in it
};

// global-memory record lists of the split backward (carved from the backward scratch buffer)
struct BwdLists {
    uint32_t *tile_rec_start;  // [NV*T + 1] exclusive scan of the per-tile slice totals; [NV*T] = records needed
                               // (> capacity: the split kernels exit and the fused kernel runs)
    uint4 *records;
    uint32_t capacity;         // records the buffer holds
    uint32_t *inst_off, *inst_cnt;
};

// a side stream + fork/join events per device for kernels that are independent of the main stream's next kernel
// (few long CTAs that would otherwise serialise behind / in front of a grid-filling kernel); defined in raster_api.cu
struct GaSide { cudaStream_t st = nullptr; cudaEvent_t fork = nullptr, join = nullptr; };
GaSide *ga_side();

// kernel launchers (defined in the .cu files, called from raster_api.cu)
cudaError_t ga_launch_preprocess(const RasterDims &d, const RasterWs &w, const float *gauss13,
                                 const float *viewmats, const float *projmats,
                                 int32_t *out_radii, cudaStream_t s);
// status_host / status_event (both optional): after the tile scan -- the first point where the instance count and
// the overflow flag are known -- status[0..3] is copied to pinned host memory and the event recorded, so the host
// can look at them while the scatter / sort / composite kernels are still running.
// Tile counters / scatter cursors are kept in GA_TILE_REPLICAS copies per tile (replica = warp index mod R): the
// 1.05M atomics of the C2 scene otherwise queue up on 6144 addresses, ~170 deep, and L2 serialises same-address
// atomics (scatter: 48 us for 1M atomics).  The scan sums the replicas of a tile and hands every replica its own
// sub-range of the tile's slots; the order inside a tile is fixed afterwards by the sort, so results do not change.
#ifndef GA_TILE_REPLICAS
#define GA_TILE_REPLICAS 8
#endif

cudaError_t ga_launch_binning(const RasterDims &d, const RasterWs &w, cudaStream_t s, int32_t *status_host = nullptr,
                              cudaEvent_t status_event = nullptr);
cudaError_t ga_launch_render_fwd(const RasterDims &d, const RasterWs &w, const float *bg,
                                 float *out_color, float *out_allmap, cudaStream_t s);
cudaError_t ga_launch_render_fwd_with_slices(const RasterDims &d, const RasterWs &w, const float *bg, float *out_color,
                                             float *out_allmap, cudaStream_t s);
#ifndef GA_LIST_K
#define GA_LIST_K 32               /* default per-pixel list capacity callers pass as list_k */
#endif
cudaError_t ga_launch_render_bwd(const RasterDims &d, const RasterWs &w, const float *bg,
                                 const float *dL_dcolor, const float *dL_dallmap,
                                 float *grad_acc, const BwdLists &lists, cudaStream_t s);
// per-tile record totals of the split backward and their scan into tile_rec_start[NV*T + 1] ([NV*T] = total)
cudaError_t ga_launch_bwd_slices(const RasterDims &d, const RasterWs &w, uint32_t *tile_rec_start, cudaStream_t s);
cudaError_t ga_launch_preprocess_bwd(const RasterDims &d, const RasterWs &w, const float *gauss13,
                                     const float *viewmats, const float *projmats,
                                     const int32_t *radii, const float *grad_acc,
                                     float *grad_gauss13, cudaStream_t s);
