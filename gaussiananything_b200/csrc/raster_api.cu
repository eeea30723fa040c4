// C-ABI entry points of the surfel rasteriser (see include/ga_b200.h).
#include "../../include/ga_b200.h"
#include "raster_common.cuh"

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- optional per-stage timing (bench.py's roofline leg) -------------------
static int g_profile = 0;
static cudaEvent_t g_ev[7];
static bool g_ev_init = false;
static inline void prof(int i, cudaStream_t s) { if (g_profile) cudaEventRecord(g_ev[i], s); }

extern "C" int ga_profile_enable(int on)
{
    if (on && !g_ev_init) {
        for (int i = 0; i < 7; i++)
            if (cudaEventCreate(&g_ev[i]) != cudaSuccess) return GA_ERR_BADARG;
        g_ev_init = true;
    }
    g_profile = on ? 1 : 0;
    return 0;
}

extern "C" int ga_profile_read(float *ms, int n)
{
    if (!g_ev_init || !ms || n < 5) return 0;
    if (cudaEventSynchronize(g_ev[6]) != cudaSuccess) return 0;
    const int a[5] = {0, 1, 2, 4, 5}, b[5] = {1, 2, 3, 5, 6};
    for (int i = 0; i < 5; i++)
        if (cudaEventElapsedTime(&ms[i], g_ev[a[i]], g_ev[b[i]]) != cudaSuccess) return 0;
    return 5;
}

// side stream + events for work that is independent of the main stream's next kernel (one set per device)
GaSide *ga_side()
{
    static GaSide sides[64];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return nullptr;
    GaSide &g = sides[dev];
    if (!g.st) {
        if (cudaStreamCreateWithFlags(&g.st, cudaStreamNonBlocking) != cudaSuccess) { g.st = nullptr; return nullptr; }
        cudaEventCreateWithFlags(&g.fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g.join, cudaEventDisableTiming);
    }
    return &g;
}


static int g_radius_formula = GA_RADIUS_FORMULA, g_quat_norm_grad = GA_QUAT_NORM_GRAD;

extern "C" int ga_raster_set_variant(int radius_formula, int quat_norm_grad)
{
    g_radius_formula = radius_formula ? 1 : 0;
    g_quat_norm_grad = quat_norm_grad ? 1 : 0;
    return 0;
}

extern "C" int ga_raster_get_variant(int *radius_formula, int *quat_norm_grad)
{
    if (!radius_formula || !quat_norm_grad) return GA_ERR_BADARG;
    *radius_formula = g_radius_formula; *quat_norm_grad = g_quat_norm_grad;
    return 0;
}

static int make_dims(int batch, int P, int views, int H, int W, float scale_modifier,
                     int64_t max_instances, RasterDims *d, int list_k = 0)
{
    if (list_k < 0 || list_k > 1024) return GA_ERR_BADARG;
    d->list_k = list_k;
    if (batch <= 0 || P <= 0 || views <= 0 || H <= 0 || W <= 0 || max_instances < 0) return GA_ERR_BADARG;
    d->batch = batch; d->P = P; d->views = views; d->NV = batch * views;
    d->H = H; d->W = W;
    d->gx = (W + GA_BLOCK_X - 1) / GA_BLOCK_X;
    d->gy = (H + GA_BLOCK_Y - 1) / GA_BLOCK_Y;
    d->T = d->gx * d->gy;
    d->scale_modifier = scale_modifier;
    d->max_instances = max_instances;
    d->radius_formula = g_radius_formula; d->quat_norm_grad = g_quat_norm_grad;
    if (d->gx > 255 || d->gy > 255) return GA_ERR_SIZE;
    if ((int64_t)d->NV * P > 0x7fffffffLL || max_instances > 0xfffffff0LL) return GA_ERR_SIZE;
    if (d->NV > 65535) return GA_ERR_SIZE;
    return 0;
}

extern "C" int ga_raster_layout(int batch, int P, int views, int H, int W,
                                int64_t max_instances, GaRasterLayout *L)
{
    return ga_raster_layout_ex(batch, P, views, H, W, max_instances, 0, L);
}

extern "C" int ga_raster_layout_ex(int batch, int P, int views, int H, int W,
                                   int64_t max_instances, int list_k, GaRasterLayout *L)
{
    RasterDims d;
    int rc = make_dims(batch, P, views, H, W, 1.0f, max_instances, &d, list_k);
    if (rc) return rc;
    if (!L) return GA_ERR_BADARG;
    const size_t NVP = (size_t)d.NV * P, NVT = (size_t)d.NV * d.T, HW = (size_t)H * W;
    const size_t mi = (size_t)(max_instances > 0 ? max_instances : 1);
    size_t off = 0;
    L->status = off;     off = align_up(off + 16 * sizeof(int32_t), 256);
    L->rec = off;        off = align_up(off + NVP * GA_REC_F * sizeof(float), 256);
    L->depth = off;      off = align_up(off + NVP * sizeof(float), 256);
    L->rect = off;       off = align_up(off + NVP * sizeof(uint32_t), 256);
    L->tile_count = off; off = align_up(off + NVT * GA_TILE_REPLICAS * sizeof(uint32_t), 256);
    L->tile_start = off; off = align_up(off + (NVT + 1) * sizeof(uint32_t), 256);
    L->keys = off;       off = align_up(off + mi * sizeof(uint64_t), 256);
    L->ids = off;        off = align_up(off + mi * sizeof(uint32_t), 256);
    L->final_T = off;    off = align_up(off + (size_t)d.NV * 3 * HW * sizeof(float), 256);
    L->n_contrib = off;  off = align_up(off + (size_t)d.NV * 2 * HW * sizeof(int32_t), 256);
    L->inst_off = off;   off = align_up(off + mi * sizeof(uint32_t), 256);
    L->inst_cnt = off;   off = align_up(off + mi * sizeof(uint32_t), 256);
    L->n_list = off;     off = align_up(off + (list_k ? (size_t)d.NV * HW * sizeof(int32_t) : 0), 256);
    L->tile_flag = off;  off = align_up(off + (list_k ? NVT * sizeof(uint32_t) : 0), 256);
    L->tile_rec_start = off; off = align_up(off + (list_k ? (NVT + 1) * sizeof(uint32_t) : 0), 256);
    L->lists = off;      off = align_up(off + (size_t)list_k * NVT * 256 * 16, 256);
    L->total_bytes = off;
    return 0;
}

static void carve(const GaRasterLayout &L, void *base, RasterWs *w)
{
    char *p = (char *)base;
    w->status = (int32_t *)(p + L.status);
    w->rec = (float *)(p + L.rec);
    w->depth = (float *)(p + L.depth);
    w->rect = (uint32_t *)(p + L.rect);
    w->tile_count = (uint32_t *)(p + L.tile_count);
    w->tile_start = (uint32_t *)(p + L.tile_start);
    w->keys = (unsigned long long *)(p + L.keys);
    w->ids = (uint32_t *)(p + L.ids);
    w->final_T = (float *)(p + L.final_T);
    w->n_contrib = (int32_t *)(p + L.n_contrib);
    w->inst_off = (uint32_t *)(p + L.inst_off);
    w->inst_cnt = (uint32_t *)(p + L.inst_cnt);
    w->n_list = (int32_t *)(p + L.n_list);
    w->tile_flag = (uint32_t *)(p + L.tile_flag);
    w->tile_rec_start = (uint32_t *)(p + L.tile_rec_start);
    w->lists = (uint4 *)(p + L.lists);
}

static int raster_forward_impl(int stage, const float *gauss13, int batch, int P, int views,
                               const float *viewmats, const float *projmats, const float *bg,
                               int H, int W, float scale_modifier,
                               float *out_color, float *out_allmap, int32_t *out_radii,
                               void *workspace, size_t workspace_bytes, int64_t max_instances,
                               void *stream, int32_t *status_host = nullptr, void *status_event = nullptr, int list_k = 0)
{
    RasterDims d;
    int rc = make_dims(batch, P, views, H, W, scale_modifier, max_instances, &d, list_k);
    if (rc) return rc;
    if (!gauss13 || !viewmats || !projmats || !bg || !out_color || !out_allmap || !out_radii || !workspace)
        return GA_ERR_BADARG;
    GaRasterLayout L;
    ga_raster_layout_ex(batch, P, views, H, W, max_instances, list_k, &L);
    if (workspace_bytes < L.total_bytes) return GA_ERR_WORKSPACE;
    RasterWs w;
    carve(L, workspace, &w);
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    if (stage == 0 || stage == 1) {
        if ((e = cudaMemsetAsync(w.status, 0, 16 * sizeof(int32_t), s)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(w.tile_count, 0, (size_t)d.NV * d.T * GA_TILE_REPLICAS * sizeof(uint32_t), s)) != cudaSuccess) return (int)e;
        prof(0, s);
        if ((e = ga_launch_preprocess(d, w, gauss13, viewmats, projmats, out_radii, s)) != cudaSuccess) return (int)e;
        prof(1, s);
        if ((e = ga_launch_binning(d, w, s, status_host, (cudaEvent_t)status_event)) != cudaSuccess) return (int)e;
        prof(2, s);
    }
    if (stage == 0 || stage == 2) {
        if (list_k && (e = cudaMemsetAsync(w.tile_flag, 0, (size_t)d.NV * d.T * sizeof(uint32_t), s)) != cudaSuccess) return (int)e;
        if (list_k) e = ga_launch_render_fwd_with_slices(d, w, bg, out_color, out_allmap, s);
        else e = ga_launch_render_fwd(d, w, bg, out_color, out_allmap, s);
        if (e != cudaSuccess) return (int)e;
        prof(3, s);
    }
    return 0;
}

extern "C" int ga_raster_forward(const float *gauss13, int batch, int P, int views,
                                 const float *viewmats, const float *projmats, const float *bg,
                                 int H, int W, float scale_modifier,
                                 float *out_color, float *out_allmap, int32_t *out_radii,
                                 void *workspace, size_t workspace_bytes, int64_t max_instances,
                                 void *stream)
{
    return raster_forward_impl(0, gauss13, batch, P, views, viewmats, projmats, bg, H, W, scale_modifier, out_color,
                               out_allmap, out_radii, workspace, workspace_bytes, max_instances, stream);
}

extern "C" int ga_raster_forward_async(const float *gauss13, int batch, int P, int views,
                                       const float *viewmats, const float *projmats, const float *bg,
                                       int H, int W, float scale_modifier,
                                       float *out_color, float *out_allmap, int32_t *out_radii,
                                       void *workspace, size_t workspace_bytes, int64_t max_instances,
                                       int32_t *status_host, void *status_event, void *stream)
{
    if (!status_host || !status_event) return GA_ERR_BADARG;
    return raster_forward_impl(0, gauss13, batch, P, views, viewmats, projmats, bg, H, W, scale_modifier, out_color,
                               out_allmap, out_radii, workspace, workspace_bytes, max_instances, stream, status_host,
                               status_event);
}

extern "C" int ga_raster_forward_ex(const float *gauss13, int batch, int P, int views,
                                    const float *viewmats, const float *projmats, const float *bg,
                                    int H, int W, float scale_modifier,
                                    float *out_color, float *out_allmap, int32_t *out_radii,
                                    void *workspace, size_t workspace_bytes, int64_t max_instances, int list_k,
                                    int32_t *status_host, void *status_event, void *stream)
{
    if ((status_host == nullptr) != (status_event == nullptr)) return GA_ERR_BADARG;
    return raster_forward_impl(0, gauss13, batch, P, views, viewmats, projmats, bg, H, W, scale_modifier, out_color,
                               out_allmap, out_radii, workspace, workspace_bytes, max_instances, stream, status_host,
                               status_event, list_k);
}

extern "C" int ga_raster_forward_bin(const float *gauss13, int batch, int P, int views,
                                     const float *viewmats, const float *projmats, const float *bg,
                                     int H, int W, float scale_modifier,
                                     float *out_color, float *out_allmap, int32_t *out_radii,
                                     void *workspace, size_t workspace_bytes, int64_t max_instances,
                                     void *stream)
{
    return raster_forward_impl(1, gauss13, batch, P, views, viewmats, projmats, bg, H, W, scale_modifier, out_color,
                               out_allmap, out_radii, workspace, workspace_bytes, max_instances, stream);
}

extern "C" int ga_raster_forward_render(const float *gauss13, int batch, int P, int views,
                                        const float *viewmats, const float *projmats, const float *bg,
                                        int H, int W, float scale_modifier,
                                        float *out_color, float *out_allmap, int32_t *out_radii,
                                        void *workspace, size_t workspace_bytes, int64_t max_instances,
                                        void *stream)
{
    return raster_forward_impl(2, gauss13, batch, P, views, viewmats, projmats, bg, H, W, scale_modifier, out_color,
                               out_allmap, out_radii, workspace, workspace_bytes, max_instances, stream);
}

// Backward scratch = gradient accumulators [NV*P][18] | tile slice starts (room for the largest tile grid, 255 x 255
// per image) | flag | record lists of the split backward: GA_BWD_RECORDS_PER_SURFEL 16-byte records per (surfel,
// view).  The lists need sum over instances of the cull-box area inside the tile (~26 per instance on C2, i.e. ~45 per
// surfel-view); scenes that need more fall back to the fused kernel on the device (no error, no host sync).
#ifndef GA_BWD_RECORDS_PER_SURFEL
#define GA_BWD_RECORDS_PER_SURFEL 64
#endif
static size_t bwd_acc_bytes(int batch, int P, int views) { return align_up((size_t)batch * views * P * GA_GRAD_F * sizeof(float), 256); }
static size_t bwd_tiles_bytes(int batch, int views) { return align_up(((size_t)batch * views * 255 * 255 + 1) * sizeof(uint32_t), 256); }
// scratch bytes in front of the record lists: accumulators | tile slice starts | flag
static size_t bwd_fixed_bytes(int batch, int P, int views) { return bwd_acc_bytes(batch, P, views) + bwd_tiles_bytes(batch, views) + 256; }
// records the split backward's lists hold in `scratch_bytes`; 0: the buffer holds (little more than) the accumulators and
// the fused kernel is chosen on the host
static uint32_t bwd_list_capacity(int batch, int P, int views, size_t scratch_bytes)
{
    const size_t fixed = bwd_fixed_bytes(batch, P, views);
    if (scratch_bytes <= fixed + 4096) return 0;
    const size_t cap = (scratch_bytes - fixed) / 16;
    return (uint32_t)(cap > 0xfffffff0ull ? 0xfffffff0ull : cap);
}

extern "C" size_t ga_raster_backward_scratch_bytes(int batch, int P, int views)
{
    if (batch <= 0 || P <= 0 || views <= 0) return 0;
    return bwd_acc_bytes(batch, P, views) + bwd_tiles_bytes(batch, views) + 256 +
           align_up((size_t)batch * views * P * GA_BWD_RECORDS_PER_SURFEL * 16, 256);
}

extern "C" int ga_raster_backward(const float *gauss13, int batch, int P, int views,
                                  const float *viewmats, const float *projmats, const float *bg,
                                  int H, int W, float scale_modifier,
                                  const int32_t *radii,
                                  const float *dL_dcolor, const float *dL_dallmap,
                                  const void *workspace, size_t workspace_bytes, int64_t max_instances,
                                  void *scratch, size_t scratch_bytes,
                                  float *grad_gauss13, void *stream)
{
    return ga_raster_backward_ex(gauss13, batch, P, views, viewmats, projmats, bg, H, W, scale_modifier, radii, dL_dcolor,
                                 dL_dallmap, workspace, workspace_bytes, max_instances, 0, scratch, scratch_bytes,
                                 grad_gauss13, stream);
}

extern "C" int ga_raster_backward_ex(const float *gauss13, int batch, int P, int views,
                                     const float *viewmats, const float *projmats, const float *bg,
                                     int H, int W, float scale_modifier,
                                     const int32_t *radii,
                                     const float *dL_dcolor, const float *dL_dallmap,
                                     const void *workspace, size_t workspace_bytes, int64_t max_instances, int list_k,
                                     void *scratch, size_t scratch_bytes,
                                     float *grad_gauss13, void *stream)
{
    RasterDims d;
    int rc = make_dims(batch, P, views, H, W, scale_modifier, max_instances, &d, list_k);
    if (rc) return rc;
    if (!gauss13 || !viewmats || !projmats || !bg || !radii || !dL_dcolor || !dL_dallmap ||
        !workspace || !scratch || !grad_gauss13)
        return GA_ERR_BADARG;
    GaRasterLayout L;
    ga_raster_layout_ex(batch, P, views, H, W, max_instances, list_k, &L);
    if (workspace_bytes < L.total_bytes) return GA_ERR_WORKSPACE;
    const size_t need = bwd_acc_bytes(batch, P, views);                 // the accumulators are mandatory, the lists optional
    if (scratch_bytes < need) return GA_ERR_WORKSPACE;
    RasterWs w;
    carve(L, const_cast<void *>(workspace), &w);
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    float *grad_acc = (float *)scratch;
    prof(4, s);
    if ((e = cudaMemsetAsync(grad_acc, 0, need, s)) != cudaSuccess) return (int)e;
    BwdLists lists = {};
    {
        // a caller that passes only the accumulators (the round-1 scratch size) gets the fused kernel
        const uint32_t cap = bwd_list_capacity(batch, P, views, scratch_bytes);
        if (cap > 0) {
            char *p = (char *)scratch + need;
            lists.tile_rec_start = (uint32_t *)p;
            lists.records = (uint4 *)(p + bwd_tiles_bytes(batch, views) + 256);
            lists.capacity = cap;
            lists.inst_off = w.inst_off;
            lists.inst_cnt = w.inst_cnt;
            const size_t mi = (size_t)(max_instances > 0 ? max_instances : 1);
            if ((e = cudaMemsetAsync(w.inst_cnt, 0, mi * sizeof(uint32_t), s)) != cudaSuccess) return (int)e;
        }
    }
    if ((e = ga_launch_render_bwd(d, w, bg, dL_dcolor, dL_dallmap, grad_acc, lists, s)) != cudaSuccess) return (int)e;
    prof(5, s);
    if ((e = ga_launch_preprocess_bwd(d, w, gauss13, viewmats, projmats, radii, grad_acc, grad_gauss13, s)) != cudaSuccess)
        return (int)e;
    prof(6, s);
    return 0;
}

extern "C" int ga_raster_backward_records(int batch, int P, int views, int H, int W,
                                          const void *workspace, size_t workspace_bytes, int64_t max_instances,
                                          int list_k, void *scratch, size_t scratch_bytes,
                                          uint64_t *total, uint64_t *capacity, void *stream)
{
    RasterDims d;
    int rc = make_dims(batch, P, views, H, W, 1.0f, max_instances, &d, list_k);
    if (rc) return rc;
    if (!workspace || !total || !capacity) return GA_ERR_BADARG;
    GaRasterLayout L;
    ga_raster_layout_ex(batch, P, views, H, W, max_instances, list_k, &L);
    if (workspace_bytes < L.total_bytes) return GA_ERR_WORKSPACE;
    RasterWs w;
    carve(L, const_cast<void *>(workspace), &w);
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    const uint32_t *dev_total;
    if (list_k > 0) {
        dev_total = w.tile_rec_start + (size_t)d.NV * d.T;                  // laid out by the forward
    } else {
        // the slice layout the backward would compute, in the same place of the scratch
        if (!scratch || scratch_bytes < bwd_fixed_bytes(batch, P, views)) return GA_ERR_WORKSPACE;
        uint32_t *trs = (uint32_t *)((char *)scratch + bwd_acc_bytes(batch, P, views));
        if ((e = ga_launch_bwd_slices(d, w, trs, s)) != cudaSuccess) return (int)e;
        dev_total = trs + (size_t)d.NV * d.T;
    }
    int32_t overflow = 0;
    uint32_t t32 = 0;
    if ((e = cudaMemcpyAsync(&overflow, w.status + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpyAsync(&t32, dev_total, sizeof(uint32_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return (int)e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return (int)e;
    if (overflow) return GA_ERR_WORKSPACE;                                    // the forward binned nothing
    *total = t32;
    *capacity = bwd_list_capacity(batch, P, views, scratch_bytes);
    return 0;
}

extern "C" const char *ga_b200_version(void) { return "ga_b200 0.1 (sm_100a)"; }
