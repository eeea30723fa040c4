// K3 / K4: forward and backward alpha compositing of surfels, one CTA per
// 16x16 tile of one image, all images of the batch in one launch.
//
// Restates upstream forward.cu / backward.cu renderCUDA
// (github.com/hbb1/diff-surfel-rasterization; called from
// /root/reference/nsr/gs_surfel.py:100-114).  Differences in HOW, not WHAT:
//  * each warp owns an 8x4 pixel block; for every group of 32 staged surfels
//    the lanes test the surfels' conservative cull boxes (computed in K1)
//    against the warp's block and the warp only evaluates the hits.  The cull
//    box contains every pixel that can reach alpha >= 1/255, so results are
//    identical to evaluating every (pixel, surfel) pair.
//  * the backward recomputes the forward per tile, reduces each surfel's
//    gradient over the warp with shuffles, over the CTA in shared memory, and
//    issues one global atomic per (tile, surfel, component).
#include "raster_common.cuh"
#include "sm100_ptx.cuh"
#include "device_once.cuh"
#include <cstdlib>

#define CHUNK 256
#ifndef GA_LIST_STCS
#define GA_LIST_STCS 0
#endif
#ifndef GA_FWD_GROUP_DEFAULT
#define GA_FWD_GROUP_DEFAULT 8
#endif

// single-instruction approximations (MUFU.RCP / MUFU.EX2, <= 2 ulp): the IEEE division and the range-checked
// __expf cost ~10 instructions each in the inner loop; parity with the oracle stays ~1e-6 relative.
__device__ __forceinline__ float fast_rcp(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float fast_ex2(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
#define GA_M_C0 (GA_FAR_N / (GA_FAR_N - GA_NEAR_N))              /* m = C0 - C1 / depth */
#define GA_M_C1 (GA_FAR_N * GA_NEAR_N / (GA_FAR_N - GA_NEAR_N))
#define GA_NEG_HALF_LOG2E (-0.72134752044448170368f)              /* exp(-0.5 rho) = 2^(rho * this) */

struct PixelGeom {
    float s0, s1, p2, rho3d, rho2d, dx, dy, depth, G, alpha;
    bool use3d;
};

// Evaluates one (pixel, surfel) pair up to alpha; returns false when the pair
// is skipped (upstream's `continue` conditions).
__device__ __forceinline__ bool eval_pair(const float4 a, const float4 b, const float4 c,
                                          float pfx, float pfy, PixelGeom &o,
                                          float &k0, float &k1, float &k2,
                                          float &l0, float &l1, float &l2)
{
    // Tu = a.xyz, Tv = (a.w, b.x, b.y), Tw = (b.z, b.w, c.x), xy = (c.y, c.z), opacity = c.w
    k0 = pfx * b.z - a.x; k1 = pfx * b.w - a.y; k2 = pfx * c.x - a.z;
    l0 = pfy * b.z - a.w; l1 = pfy * b.w - b.x; l2 = pfy * c.x - b.y;
    const float p0 = k1 * l2 - k2 * l1, p1 = k2 * l0 - k0 * l2, p2 = k0 * l1 - k1 * l0;
    if (p2 == 0.0f) return false;
    const float ip = fast_rcp(p2);
    o.p2 = p2;
    o.s0 = p0 * ip; o.s1 = p1 * ip;
    o.rho3d = o.s0 * o.s0 + o.s1 * o.s1;
    o.dx = c.y - pfx; o.dy = c.z - pfy;
    o.rho2d = GA_FILTER_INV_SQUARE * (o.dx * o.dx + o.dy * o.dy);
    o.use3d = o.rho3d <= o.rho2d;
    const float rho = fminf(o.rho3d, o.rho2d);
    o.depth = o.use3d ? (o.s0 * b.z + o.s1 * b.w) + c.x : c.x;
    if (o.depth < GA_NEAR_N) return false;
    o.G = fast_ex2(rho * GA_NEG_HALF_LOG2E);         // rho >= 0, so upstream's `power > 0` never fires
    o.alpha = fminf(0.99f, c.w * o.G);
    return o.alpha >= 1.0f / 255.0f;
}

// pixels of the tile with origin (ox, oy) inside the cull box bb = (x0, x1, y0, y1): the record-slice length of an
// instance in the split backward, and an upper bound of its list length in the fused one.  An empty box (a surfel
// too transparent to reach alpha 1/255 anywhere: +-1e30 bounds) has no pixel.  The bounds are clamped to one pixel
// beyond the tile, which changes no count: unclamped, +-1e30 saturates the float -> int conversions and the wrapped
// difference counts 2 x 2 pixels.
__device__ __forceinline__ int clipped_box_area(const float4 bb, int ox, int oy)
{
    const float x0 = fminf(fmaxf(bb.x, (float)ox), (float)(ox + 16)), x1 = fmaxf(fminf(bb.y, (float)(ox + 15)), (float)(ox - 1));
    const float y0 = fminf(fmaxf(bb.z, (float)oy), (float)(oy + 16)), y1 = fmaxf(fminf(bb.w, (float)(oy + 15)), (float)(oy - 1));
    const int wx = max(0, (int)floorf(x1) - (int)ceilf(x0) + 1), wy = max(0, (int)floorf(y1) - (int)ceilf(y0) + 1);
    return wx * wy;
}

// Forward staging record (tile-local, computed once per (tile, surfel) by the
// staging thread): with o = tile origin, k_o = o.x*Tw - Tu, l_o = o.y*Tw - Tv,
//   p(dx,dy) = (k_o + dx*Tw) x (l_o + dy*Tw) = C + dx*A + dy*B,
//   C = k_o x l_o, A = Tw x l_o, B = k_o x Tw            (Tw x Tw = 0)
// which is upstream's cross(k, l) re-associated around the tile origin (all
// terms stay O(tile size), so no precision is lost) and costs 6 FMAs per pixel.
//  f0 = C.x C.y C.z A.x | f1 = A.y A.z B.x B.y | f2 = B.z Tw.x Tw.y Tw.z
//  f3 = xy.x-o.x xy.y-o.y opacity - | f4 = cull box (tile-local x0 x1 y0 y1)
//  f5 = n.x n.y n.z r | f6 = g b - -
// Lane groups.  A warp owns an 8x4 pixel block; GS = 32 evaluates one surfel per round for the whole block
// (warp-uniform shared-memory reads).  With the C2 scene a surfel's cull box covers ~25 pixels, so only ~9 of the 32
// lanes of a hit carry a contributing pixel.  GS = 16 splits the warp into two 4x4 blocks, GS = 8 into four 4x2
// blocks; every group walks ITS OWN list of hits, so a round evaluates up to 32 / GS different surfels (2 or 4
// distinct shared-memory addresses per load instead of one).  C2 scene (tools/raster_rounds.py): 44 rounds per warp
// and chunk with GS = 32, 32 with GS = 16, 26 with GS = 8 (17.5 with one list per lane, but per-lane lists make every
// load a 32-address gather: 0.208 vs 0.199 ms in round 1).  Measured: 209 / 181 / 176 us per 6-view launch.  Results do not depend on GS:
// the per-pixel sequence of contributing surfels is the same.
//
// LISTS: the kernel also records, per pixel, every surfel that contributed -- {position in the tile list, alpha,
// depth} -- into a tile-major array (entry k of the tile's 256 pixels is one contiguous 4 KB row, so a warp's store is
// four full 128-byte lines).  The backward then walks exactly these entries: no cull tests, no pair re-evaluation for
// pairs that do not contribute, and the contribution decisions are the forward's own bits.
template <int GS, bool LISTS>
__global__ void __launch_bounds__(256, 4)
render_fwd_kernel(RasterDims d, RasterWs ws, const float *__restrict__ bg,
                  float *__restrict__ out_color, float *__restrict__ out_allmap)
{
    constexpr int NG = 32 / GS;                                  // groups per warp
    constexpr int GW = GS == 32 ? 8 : 4;                         // group block width / height in pixels
    constexpr int GH = GS == 8 ? 2 : 4;
    __shared__ float4 s_rec[7][CHUNK];
    __shared__ uint32_t s_area;                                  // LISTS: sum of the clipped cull-box areas of this chunk
    __shared__ unsigned long long s_area_sum;                    // ... and of all chunks staged so far (thread 0)
    if (ws.status[1]) return;
    const int view = blockIdx.z;
    const int tile = blockIdx.y * d.gx + blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane / GS, gl = lane % GS;
    if (LISTS && threadIdx.x == 0) { s_area = 0; s_area_sum = 0; }
    const int ox = blockIdx.x * GA_BLOCK_X, oy = blockIdx.y * GA_BLOCK_Y;
    const int wx0 = (warp & 1) * 8, wy0 = (warp >> 1) * 4;       // warp's 8x4 block, tile-local
    // group blocks tile the warp block: GS=16 -> 2 side by side (4x4); GS=8 -> 2x2 arrangement of 4x2 blocks
    const int lx0 = wx0 + (GS == 32 ? 0 : (grp & 1) * 4), ly0 = wy0 + (GS == 8 ? (grp >> 1) * 2 : 0);
    const int lxi = lx0 + (gl % GW), lyi = ly0 + (gl / GW);
    const int pxi = ox + lxi, pyi = oy + lyi;
    const bool inside = pxi < d.W && pyi < d.H;
    const float dxf = (float)lxi, dyf = (float)lyi;
    const float oxf = (float)ox, oyf = (float)oy;

    const uint32_t start = ws.tile_start[(size_t)view * d.T + tile];
    const uint32_t end = ws.tile_start[(size_t)view * d.T + tile + 1];
    const int total = (int)(end - start);
    const float *rec_base = ws.rec + (size_t)view * d.P * GA_REC_F;

    bool done = !inside;
    float T = 1.0f, C0 = 0, C1 = 0, C2 = 0, N0 = 0, N1 = 0, N2 = 0;
    float Dacc = 0, M1 = 0, M2 = 0, dist = 0, median_depth = 0;
    int last_contributor = 0, median_contributor = -1;
    int nl = 0;                                                    // LISTS: contributions of this pixel so far
    uint4 *my_list = nullptr;
    if (LISTS) my_list = ws.lists + ((size_t)view * d.T + tile) * (size_t)d.list_k * 256 + (lyi * 16 + lxi);

    for (int c0 = 0; c0 < total; c0 += CHUNK) {
        if (__syncthreads_count(done) == 256) break;
        const int cnt = min(CHUNK, total - c0);
        uint32_t area = 0;
        if ((int)threadIdx.x < cnt) {
            const uint32_t id = ws.ids[start + c0 + threadIdx.x];
            const float4 *src = reinterpret_cast<const float4 *>(rec_base + (size_t)id * GA_REC_F);
            const float4 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
            const float4 nr = __ldg(src + 3), bb = __ldg(src + 4), gb = __ldg(src + 5);
            // Tu = a.xyz, Tv = (a.w,b.x,b.y), Tw = (b.z,b.w,c.x), xy = (c.y,c.z), opacity = c.w
            const float k0 = oxf * b.z - a.x, k1 = oxf * b.w - a.y, k2 = oxf * c.x - a.z;
            const float l0 = oyf * b.z - a.w, l1 = oyf * b.w - b.x, l2 = oyf * c.x - b.y;
            const float Cx = k1 * l2 - k2 * l1, Cy = k2 * l0 - k0 * l2, Cz = k0 * l1 - k1 * l0;
            const float Ax = b.w * l2 - c.x * l1, Ay = c.x * l0 - b.z * l2, Az = b.z * l1 - b.w * l0;
            const float Bx = k1 * c.x - k2 * b.w, By = k2 * b.z - k0 * c.x, Bz = k0 * b.w - k1 * b.z;
            s_rec[0][threadIdx.x] = make_float4(Cx, Cy, Cz, Ax);
            s_rec[1][threadIdx.x] = make_float4(Ay, Az, Bx, By);
            s_rec[2][threadIdx.x] = make_float4(Bz, b.z, b.w, c.x);
            s_rec[3][threadIdx.x] = make_float4(c.y - oxf, c.z - oyf, c.w, 0.f);
            s_rec[4][threadIdx.x] = make_float4(bb.x - oxf, bb.y - oxf, bb.z - oyf, bb.w - oyf);
            s_rec[5][threadIdx.x] = nr;
            s_rec[6][threadIdx.x] = gb;
            if (LISTS) area = (uint32_t)clipped_box_area(bb, ox, oy);    // slice length in the backward's record buffer
        }
        if (LISTS) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) area += __shfl_xor_sync(0xffffffffu, area, o);
            if (lane == 0 && area) atomicAdd(&s_area, area);
        }
        __syncthreads();
        // 64-bit running sum (a tile of 2^24 full-tile instances reaches 2^32); s_area is next written after the
        // barrier at the top of the loop
        if (LISTS && threadIdx.x == 0) { s_area_sum += s_area; s_area = 0; }
        for (int g0 = 0; g0 < cnt; g0 += 32) {
            if (__all_sync(0xffffffffu, done)) break;
            const int j = g0 + lane;
            // lane tests surfel j against the block of every group of the warp; each lane keeps its group's ballot
            unsigned mask = 0;
            {
                float4 bb = make_float4(1e30f, -1e30f, 1e30f, -1e30f);
                if (j < cnt) bb = s_rec[4][j];
#pragma unroll
                for (int q = 0; q < NG; q++) {
                    const float qx0 = (float)(wx0 + (GS == 32 ? 0 : (q & 1) * 4)), qy0 = (float)(wy0 + (GS == 8 ? (q >> 1) * 2 : 0));
                    const bool hit = !(bb.y < qx0 || bb.x > qx0 + (float)(GW - 1) || bb.w < qy0 || bb.z > qy0 + (float)(GH - 1));
                    const unsigned m = __ballot_sync(0xffffffffu, hit);
                    if (q == grp) mask = m;
                }
            }
            while (__any_sync(0xffffffffu, mask != 0)) {
                const bool active = mask != 0;
                const int jj = g0 + (active ? __ffs(mask) - 1 : 0);
                mask &= mask - 1;
                const float4 f0 = s_rec[0][jj], f1 = s_rec[1][jj], f2 = s_rec[2][jj], f3 = s_rec[3][jj];
                const float p0 = f0.x + dxf * f0.w + dyf * f1.z;
                const float p1 = f0.y + dxf * f1.x + dyf * f1.w;
                const float p2 = f0.z + dxf * f1.y + dyf * f2.x;
                const float ip = fast_rcp(p2);
                const float s0 = p0 * ip, s1 = p1 * ip;
                const float rho3d = s0 * s0 + s1 * s1;
                const float ddx = f3.x - dxf, ddy = f3.y - dyf;
                const float rho2d = GA_FILTER_INV_SQUARE * (ddx * ddx + ddy * ddy);
                const float rho = fminf(rho3d, rho2d);
                const float depth = (rho3d <= rho2d) ? (s0 * f2.y + s1 * f2.z) + f2.w : f2.w;
                // power = -0.5*rho > 0 never happens for rho >= 0; NaN rho (p2 == 0) fails the alpha test
                const float alpha = fminf(0.99f, f3.z * fast_ex2(rho * GA_NEG_HALF_LOG2E));
                bool ok = active && !done && p2 != 0.0f && depth >= GA_NEAR_N && alpha >= 1.0f / 255.0f;
                float test_T = 0.f;
                if (ok) {
                    test_T = T * (1 - alpha);
                    if (test_T < 0.0001f) { done = true; ok = false; }
                }
                if (__any_sync(0xffffffffu, ok)) {
                    const float4 nr = s_rec[5][jj], gb = s_rec[6][jj];
                    if (ok) {
                        const int contributor = c0 + jj + 1;
                        const float w = alpha * T;
                        const float A = 1 - T;
                        const float m = GA_M_C0 - GA_M_C1 * fast_rcp(depth);
                        dist += (m * m * A + M2 - 2 * m * M1) * w;
                        Dacc += depth * w;
                        M1 += m * w;
                        M2 += m * m * w;
                        if (T > 0.5f) { median_depth = depth; median_contributor = contributor; }
                        N0 += nr.x * w; N1 += nr.y * w; N2 += nr.z * w;
                        C0 += nr.w * w; C1 += gb.x * w; C2 += gb.y * w;
                        T = test_T;
                        last_contributor = contributor;
                        if (LISTS) {
                            if (nl < d.list_k) {
                                const uint4 ent = make_uint4((uint32_t)(contributor - 1), __float_as_uint(alpha),
                                                             __float_as_uint(depth), 0u);
#if GA_LIST_STCS
                                __stcs(my_list + (size_t)nl * 256, ent);       // written once, read once by the backward
#else
                                my_list[(size_t)nl * 256] = ent;
#endif
                            }
                            nl++;
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    if (LISTS) {
        if (inside) ws.n_list[(size_t)view * d.H * d.W + (size_t)pyi * d.W + pxi] = nl;
        if (nl > d.list_k) ws.tile_flag[(size_t)view * d.T + tile] = 1u;      // this tile's backward recomputes
        // every chunk the backward can reach (positions below the last contributor) has been staged here, so the sum
        // covers its slices; bwd_scan_area_kernel turns the per-tile sums into offsets
        if (threadIdx.x == 0) ws.tile_rec_start[(size_t)view * d.T + tile] = (uint32_t)min(s_area_sum, 0xffffffffull);
    }
    if (inside) {
        const size_t HW = (size_t)d.H * d.W;
        const size_t pix = (size_t)pyi * d.W + pxi;
        float *fT = ws.final_T + (size_t)view * 3 * HW;
        int32_t *nc = ws.n_contrib + (size_t)view * 2 * HW;
        fT[pix] = T; fT[pix + HW] = M1; fT[pix + 2 * HW] = M2;
        nc[pix] = last_contributor; nc[pix + HW] = median_contributor;
        float *oc = out_color + (size_t)view * 3 * HW;
        oc[pix] = C0 + T * bg[0]; oc[pix + HW] = C1 + T * bg[1]; oc[pix + 2 * HW] = C2 + T * bg[2];
        float *oa = out_allmap + (size_t)view * 7 * HW;
        oa[pix] = Dacc;
        oa[pix + HW] = 1 - T;
        oa[pix + 2 * HW] = N0; oa[pix + 3 * HW] = N1; oa[pix + 4 * HW] = N2;
        oa[pix + 5 * HW] = median_depth;
        oa[pix + 6 * HW] = dist;
    }
}

// GA_B200_FWD_GROUP=32|16|8 (or ga_raster_set_tuning) selects the lane-group size; see the kernel comment
static int g_fwd_group = -1;
extern "C" int ga_raster_set_tuning(int fwd_group)
{
    if (fwd_group != 32 && fwd_group != 16 && fwd_group != 8) return -1;
    g_fwd_group = fwd_group;
    return 0;
}

cudaError_t ga_launch_render_fwd(const RasterDims &d, const RasterWs &w, const float *bg,
                                 float *out_color, float *out_allmap, cudaStream_t s)
{
    if (g_fwd_group < 0) {
        const char *e = getenv("GA_B200_FWD_GROUP");
        const int v = e ? atoi(e) : GA_FWD_GROUP_DEFAULT;
        g_fwd_group = (v == 32 || v == 16 || v == 8) ? v : GA_FWD_GROUP_DEFAULT;
    }
    dim3 grid(d.gx, d.gy, d.NV);
    if (d.list_k > 0) {
        if (g_fwd_group == 32) render_fwd_kernel<32, true><<<grid, 256, 0, s>>>(d, w, bg, out_color, out_allmap);
        else if (g_fwd_group == 16) render_fwd_kernel<16, true><<<grid, 256, 0, s>>>(d, w, bg, out_color, out_allmap);
        else render_fwd_kernel<8, true><<<grid, 256, 0, s>>>(d, w, bg, out_color, out_allmap);
    } else {
        if (g_fwd_group == 32) render_fwd_kernel<32, false><<<grid, 256, 0, s>>>(d, w, bg, out_color, out_allmap);
        else if (g_fwd_group == 16) render_fwd_kernel<16, false><<<grid, 256, 0, s>>>(d, w, bg, out_color, out_allmap);
        else render_fwd_kernel<8, false><<<grid, 256, 0, s>>>(d, w, bg, out_color, out_allmap);
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K4 backward
//
// Two phases per group of G staged surfels (G = 128, 64, 32 or 16, picked per chunk so that a surfel's cull box
// clipped to the tile never holds more pixels than its list capacity BWD_LIST_RECORDS/G):
//   phase A (pixel-parallel, back to front): every lane walks its own stream of surfels whose cull box
//     contains its pixel, recomputes alpha, runs the compositing recurrences and appends a 16-byte record
//     (pixel, dL/dalpha, dL/dz, w) to the surfel's list in shared memory;
//   phase B (surfel-parallel): 256/G threads share a surfel, re-derive the ray-splat geometry of each
//     recorded pixel, accumulate the 18 gradient components in registers and reduce-scatter them over the
//     256/G lanes; one global atomic per (tile, surfel, component).
// This replaces a 32-lane reduction per (warp, surfel) hit -- where typically 8 of 32 lanes carried data --
// by register accumulation over the pixels a surfel actually touches.
// ---------------------------------------------------------------------------
#ifndef BWD_CTAS
#define BWD_CTAS 2                  /* CTAs per SM the backward is sized for (registers and shared memory) */
#endif
#if BWD_CTAS >= 3
#define BWD_LIST_RECORDS 2560
#else
#define BWD_LIST_RECORDS 4096
#endif
#define BWD_MAXG 128
#ifndef BWD_A_CTAS
#define BWD_A_CTAS 4                /* resident CTAs per SM kernel A is compiled for (64 registers, no spills) */
#endif
#ifndef BWD_B_UNROLL
#define BWD_B_UNROLL 2              /* records per loop iteration and lane in kernel B */
#endif
#ifndef BWD_B_THREADS
#define BWD_B_THREADS 128           /* threads per CTA (= per tile) in kernel B: 128 -> 6 CTAs per SM; 256: +22 us, 64: +56 us on C2 */
#endif
#ifndef BWD_B_CTAS
#define BWD_B_CTAS (768 / BWD_B_THREADS)
#endif
#ifndef BWD_B_TPI
#define BWD_B_TPI 2                 /* lanes per instance in kernel B (2: 364 us, 4: 375 us, 8: 400+ us on C2) */
#endif

struct BwdSmem {
    float4 rec[6][CHUNK];
    uint4 list[BWD_LIST_RECORDS];
    float4 up[2][256];              // per pixel: {dL/dcolor (3), dL/dnormal.x}, {dL/dnormal.yz, -, -}: two conflict-light LDS.128
    uint32_t id[CHUNK];
    int cnt[2][BWD_MAXG];
    int maxc;
};

// reduce-scatter of 18 components over TPI (2/4/8/16) consecutive lanes by recursive halving: after level l a lane
// is responsible for half of the components it held before; the fully reduced leftovers are added to dst.
template <int TPI>
__device__ __forceinline__ void reduce_scatter18(const float (&g)[GA_GRAD_F], int lane, float *__restrict__ dst)
{
    int off = 0, size = 9;
    float a9[10];
    {
        const bool u = lane & (TPI >> 1);
#pragma unroll
        for (int i = 0; i < 9; i++) {
            const float keep = u ? g[9 + i] : g[i], send = u ? g[i] : g[9 + i];
            a9[i] = keep + __shfl_xor_sync(0xffffffffu, send, TPI >> 1);
        }
        a9[9] = 0.f;
        off += u ? 9 : 0;
    }
    if constexpr (TPI == 2) {
#pragma unroll
        for (int i = 0; i < 9; i++)
            if (a9[i] != 0.f) atomicAdd(dst + off + i, a9[i]);
        return;
    } else {
        float b5[6];
        {
            const bool u = lane & (TPI >> 2);
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const float keep = u ? a9[5 + i] : a9[i], send = u ? a9[i] : a9[5 + i];
                b5[i] = keep + __shfl_xor_sync(0xffffffffu, send, TPI >> 2);
            }
            b5[5] = 0.f;
            off += u ? 5 : 0; size = u ? 4 : 5;
        }
        if constexpr (TPI == 4) {
#pragma unroll
            for (int i = 0; i < 5; i++)
                if (i < size && b5[i] != 0.f) atomicAdd(dst + off + i, b5[i]);
            return;
        } else {
            float c3[4];
            {
                const bool u = lane & (TPI >> 3);
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    const float keep = u ? b5[3 + i] : b5[i], send = u ? b5[i] : b5[3 + i];
                    c3[i] = keep + __shfl_xor_sync(0xffffffffu, send, TPI >> 3);
                }
                c3[3] = 0.f;
                off += u ? 3 : 0; size = u ? size - 3 : 3;
            }
            if constexpr (TPI == 8) {
#pragma unroll
                for (int i = 0; i < 3; i++)
                    if (i < size && c3[i] != 0.f) atomicAdd(dst + off + i, c3[i]);
                return;
            } else {
                const bool u = lane & (TPI >> 4);
                float d2[2];
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const float keep = u ? c3[2 + i] : c3[i], send = u ? c3[i] : c3[2 + i];
                    d2[i] = keep + __shfl_xor_sync(0xffffffffu, send, TPI >> 4);
                }
                off += u ? 2 : 0; size = u ? max(size - 2, 0) : min(size, 2);
#pragma unroll
                for (int i = 0; i < 2; i++)
                    if (i < size && d2[i] != 0.f) atomicAdd(dst + off + i, d2[i]);
            }
        }
    }
}

template <int TPI>
__device__ __forceinline__ void bwd_phase_b(BwdSmem &sm, const int *cnt, int g0, int gcnt, int cap, int ox, int oy,
                                            float *__restrict__ acc_base)
{
    const int tid = threadIdx.x, lane = tid & 31;
    const int inst = tid / TPI, sub = tid % TPI;
    const bool valid = inst < gcnt;
    const int n = valid ? min(cnt[inst], cap) : 0;
    float g[GA_GRAD_F];
#pragma unroll
    for (int f = 0; f < GA_GRAD_F; f++) g[f] = 0.f;
    if (n > 0) {
        const int jj = g0 + inst;
        const float4 a = sm.rec[0][jj], b = sm.rec[1][jj], c = sm.rec[2][jj];
        const float opa = c.w;
        for (int r = sub; r < n; r += TPI) {
            const uint4 rc = sm.list[inst * cap + r];
            const int pix = (int)rc.x;
            const float dL_dalpha = __uint_as_float(rc.y), dL_dz = __uint_as_float(rc.z), w = __uint_as_float(rc.w);
            const float pfx = (float)(ox + (pix & 15)), pfy = (float)(oy + (pix >> 4));
            PixelGeom pg;
            float k0, k1, k2, l0, l1, l2;
            eval_pair(a, b, c, pfx, pfy, pg, k0, k1, k2, l0, l1, l2);      // same code path as phase A: same bits
            const float G = pg.G;
            const float dL_dG = opa * dL_dalpha;                           // 0.99 clamp passed through (upstream)
            if (pg.use3d) {
                const float dL_ds0 = dL_dG * -G * pg.s0 + dL_dz * b.z;
                const float dL_ds1 = dL_dG * -G * pg.s1 + dL_dz * b.w;
                const float ip = fast_rcp(pg.p2);
                const float q0 = dL_ds0 * ip, q1 = dL_ds1 * ip;
                const float q2 = -(q0 * pg.s0 + q1 * pg.s1);
                const float dk0 = l1 * q2 - l2 * q1, dk1 = l2 * q0 - l0 * q2, dk2 = l0 * q1 - l1 * q0;
                const float dl0 = q1 * k2 - q2 * k1, dl1 = q2 * k0 - q0 * k2, dl2 = q0 * k1 - q1 * k0;
                g[0] -= dk0; g[1] -= dk1; g[2] -= dk2;
                g[3] -= dl0; g[4] -= dl1; g[5] -= dl2;
                g[6] += pfx * dk0 + pfy * dl0 + dL_dz * pg.s0;
                g[7] += pfx * dk1 + pfy * dl1 + dL_dz * pg.s1;
                g[8] += pfx * dk2 + pfy * dl2 + dL_dz;
            } else {
                g[9] += dL_dG * (-G * GA_FILTER_INV_SQUARE * pg.dx);
                g[10] += dL_dG * (-G * GA_FILTER_INV_SQUARE * pg.dy);
                g[8] += dL_dz;
            }
            g[14] += G * dL_dalpha;
            const float4 ua = sm.up[0][pix], ub = sm.up[1][pix];
            g[15] += w * ua.x; g[16] += w * ua.y; g[17] += w * ua.z;
            g[11] += w * ua.w; g[12] += w * ub.x; g[13] += w * ub.y;
        }
    }
    // all lanes of the warp take part in the shuffles; groups whose surfel recorded nothing carry zeros
    const int any = __any_sync(0xffffffffu, n > 0);
    if (any) {
        float *dst = acc_base + (size_t)(valid ? sm.id[g0 + inst] : 0) * GA_GRAD_F;
        reduce_scatter18<TPI>(g, lane, dst);
    }
}

// Two CTAs per SM (96 KB of shared memory, 128 registers).  Three per SM (2560-record lists, 80 registers) were
// measured at 0.85 ms against 0.55 ms: the phase-A recurrences do not fit 80 registers (192 B of spills).
__global__ void __launch_bounds__(256, BWD_CTAS)
render_bwd_kernel(RasterDims d, RasterWs ws, const float *__restrict__ bg,
                  const float *__restrict__ dL_dcolor, const float *__restrict__ dL_dallmap,
                  float *__restrict__ grad_acc, const uint32_t *__restrict__ split_total, uint32_t split_capacity)
{
    extern __shared__ __align__(16) uint8_t bwd_smem_raw[];
    BwdSmem &sm = *reinterpret_cast<BwdSmem *>(bwd_smem_raw);
    if (ws.status[1]) return;
    if (split_total && split_total[0] <= split_capacity) return;      // the split kernels (below) did the work
    const int view = blockIdx.z;
    const int tile = blockIdx.y * d.gx + blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ox = blockIdx.x * GA_BLOCK_X, oy = blockIdx.y * GA_BLOCK_Y;
    const int lx0 = (warp & 1) * 8, ly0 = (warp >> 1) * 4;
    const int lxi = lx0 + (lane & 7), lyi = ly0 + (lane >> 3);
    const int pxi = ox + lxi, pyi = oy + lyi;
    const int pix_local = lyi * 16 + lxi;
    const bool inside = pxi < d.W && pyi < d.H;
    const float pfx = (float)pxi, pfy = (float)pyi;
    const float bx_lo = (float)(ox + lx0), bx_hi = (float)(ox + lx0 + 7);
    const float by_lo = (float)(oy + ly0), by_hi = (float)(oy + ly0 + 3);

    const uint32_t start = ws.tile_start[(size_t)view * d.T + tile];
    const size_t HW = (size_t)d.H * d.W;
    const size_t pix = inside ? (size_t)pyi * d.W + pxi : 0;
    const float *fT = ws.final_T + (size_t)view * 3 * HW;
    const int32_t *nc = ws.n_contrib + (size_t)view * 2 * HW;
    const float *rec_base = ws.rec + (size_t)view * d.P * GA_REC_F;
    float *acc_base = grad_acc + (size_t)view * d.P * GA_GRAD_F;

    const float T_final = inside ? fT[pix] : 0.f;
    float T = T_final;
    const int last_contributor = inside ? nc[pix] : 0;
    const int median_contributor = inside ? nc[pix + HW] : 0;
    float dpx0 = 0, dpx1 = 0, dpx2 = 0, dL_ddepth = 0, dL_daccum = 0, dL_dreg = 0;
    float dn0 = 0, dn1 = 0, dn2 = 0, dL_dmedian = 0;
    if (inside) {
        const float *gc = dL_dcolor + (size_t)view * 3 * HW;
        const float *ga = dL_dallmap + (size_t)view * 7 * HW;
        dpx0 = gc[pix]; dpx1 = gc[pix + HW]; dpx2 = gc[pix + 2 * HW];
        dL_ddepth = ga[pix]; dL_daccum = ga[pix + HW];
        dn0 = ga[pix + 2 * HW]; dn1 = ga[pix + 3 * HW]; dn2 = ga[pix + 4 * HW];
        dL_dmedian = ga[pix + 5 * HW]; dL_dreg = ga[pix + 6 * HW];
    }
    sm.up[0][pix_local] = make_float4(dpx0, dpx1, dpx2, dn0);
    sm.up[1][pix_local] = make_float4(dn1, dn2, 0.f, 0.f);
    const float final_D = inside ? fT[pix + HW] : 0.f, final_D2 = inside ? fT[pix + 2 * HW] : 0.f;
    const float final_A = 1 - T_final;
    const float bg_dot_dpixel = bg[0] * dpx0 + bg[1] * dpx1 + bg[2] * dpx2;
    // Upstream keeps one suffix accumulator per output channel (colour 3, depth, alpha, normal 3), all with the same
    // recurrence acc = last_alpha * last_value + (1 - last_alpha) * acc, and adds (value - acc) * dL/dchannel to
    // dL/dalpha.  The sum over channels is linear, so ONE scalar recurrence on v = sum_ch value_ch * dL/dchannel does
    // the same work (8 recurrences and ~20 registers less per pair).
    float last_alpha = 0, v_last = 0, v_acc = 0, last_dL_dT = 0;

    // nothing behind the deepest contributor of the tile can receive gradient
    if (threadIdx.x == 0) sm.maxc = 0;
    sm.cnt[threadIdx.x >> 7][threadIdx.x & 127] = 0;
    __syncthreads();
    {
        int m = last_contributor;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) atomicMax(&sm.maxc, m);
    }
    __syncthreads();
    const int total = sm.maxc;          // list positions [0,total) matter
    int parity = 0;

    for (int hi = total; hi > 0; hi -= CHUNK) {
        const int lo = max(0, hi - CHUNK);
        const int cnt = hi - lo;
        // stage positions lo..hi-1; slot t holds position hi-1-t (back to front)
        int big0 = 0, big1 = 0, big2 = 0, big3 = 0;
        if ((int)threadIdx.x < cnt) {
            const uint32_t id = ws.ids[start + (hi - 1 - threadIdx.x)];
            sm.id[threadIdx.x] = id;
            const float4 *src = reinterpret_cast<const float4 *>(rec_base + (size_t)id * GA_REC_F);
            float4 q[6];
#pragma unroll
            for (int k = 0; k < 6; k++) { q[k] = __ldg(src + k); sm.rec[k][threadIdx.x] = q[k]; }
            // pixels of this tile inside the cull box (upper bound of the surfel's list length)
            const int area = clipped_box_area(q[4], ox, oy);
            big0 = area > BWD_LIST_RECORDS / 128; big1 = area > BWD_LIST_RECORDS / 64;
            big2 = area > BWD_LIST_RECORDS / 32; big3 = area > BWD_LIST_RECORDS / 16;
        }
        const int any0 = __syncthreads_or(big0);
        const int any1 = __syncthreads_or(big1);
        const int any2 = __syncthreads_or(big2);
        const int any3 = __syncthreads_or(big3);
        // list capacity per surfel = BWD_LIST_RECORDS / G must cover the pixels of its cull box inside the tile
        // (G = 8: capacity >= 256 = the whole tile)
        const int G = any3 ? 8 : (any2 ? 16 : (any1 ? 32 : (any0 ? 64 : 128)));
        const int cap = BWD_LIST_RECORDS / G;

        for (int g0 = 0; g0 < cnt; g0 += G, parity ^= 1) {
            const int gcnt = min(G, cnt - g0);
            int *cntp = sm.cnt[parity];
            // ---------------- phase A: sub-blocks of 32 surfels, no block barrier in between.  (Walking one per-lane
            // list over the whole group of 128 instead needs 22 % fewer rounds, tools/raster_rounds.py, but was measured
            // slower: 573 vs 537 us -- the list bookkeeping costs more than the rounds it saves.)
            for (int sb = 0; sb < gcnt; sb += 32) {
                const int base = g0 + sb;
                bool hit = false;
                if (sb + lane < gcnt) {
                    const float4 bb = sm.rec[4][base + lane];
                    hit = !(bb.y < bx_lo || bb.x > bx_hi || bb.w < by_lo || bb.z > by_hi);
                }
                unsigned mask = __ballot_sync(0xffffffffu, hit);
                unsigned mine = 0;
                while (mask) {
                    const int b = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const float4 bb = sm.rec[4][base + b];
                    if (pfx >= bb.x && pfx <= bb.y && pfy >= bb.z && pfy <= bb.w && (hi - 1 - (base + b)) < last_contributor)
                        mine |= 1u << b;
                }
                if (!inside) mine = 0;
                while (__any_sync(0xffffffffu, mine != 0)) {
                    const bool active = mine != 0;
                    const int bsel = active ? __ffs(mine) - 1 : 0;
                    mine &= mine - 1;
                    const int jj = base + bsel;
                    const int contributor = hi - 1 - jj;       // 0-based list position
                    const float4 a = sm.rec[0][jj], b = sm.rec[1][jj], c = sm.rec[2][jj];
                    PixelGeom pg;
                    float k0, k1, k2, l0, l1, l2;
                    const bool ok = active && eval_pair(a, b, c, pfx, pfy, pg, k0, k1, k2, l0, l1, l2);
                    if (ok) {
                        const float4 nr = sm.rec[3][jj], gb = sm.rec[5][jj];
                        const float alpha = pg.alpha, c_d = pg.depth;
                        const float inv1ma = fast_rcp(1.f - alpha);
                        T = T * inv1ma;
                        const float w = alpha * T;
                        float dL_dz = 0.0f;
                        const float inv_cd = fast_rcp(c_d);
                        const float m_d = GA_M_C0 - GA_M_C1 * inv_cd;
                        const float dmd_dd = GA_M_C1 * inv_cd * inv_cd;
                        if (contributor == median_contributor - 1) dL_dz += dL_dmedian;
                        const float dL_dweight = (final_D2 + m_d * m_d * final_A - 2 * m_d * final_D) * dL_dreg;
                        const float dL_dmd = 2.0f * (T * alpha) * (m_d * final_A - final_D) * dL_dreg;
                        dL_dz += dL_dmd * dmd_dd;
                        // v = (colour . dL/dcolour) + depth dL/ddepth + 1 dL/dalpha_acc + (normal . dL/dnormal)
                        const float v = ((nr.w * dpx0 + gb.x * dpx1) + (gb.y * dpx2 + c_d * dL_ddepth)) +
                                        ((nr.x * dn0 + nr.y * dn1) + (nr.z * dn2 + dL_daccum));
                        v_acc = last_alpha * v_last + (1.f - last_alpha) * v_acc;
                        v_last = v;
                        float dL_dalpha = (v - v_acc) + (dL_dweight - last_dL_dT);
                        last_dL_dT = dL_dweight * alpha + (1 - alpha) * last_dL_dT;
                        dL_dalpha *= T;
                        last_alpha = alpha;
                        dL_dalpha += (-T_final * inv1ma) * bg_dot_dpixel;
                        dL_dz += w * dL_ddepth;
                        const int li = sb + bsel;                      // surfel index inside the group
                        const int slot = atomicAdd(&cntp[li], 1);
                        if (slot < cap)
                            sm.list[li * cap + slot] = make_uint4((uint32_t)pix_local, __float_as_uint(dL_dalpha),
                                                                  __float_as_uint(dL_dz), __float_as_uint(w));
                    }
                }
            }
            __syncthreads();
            // ---------------- phase B
            if (threadIdx.x < BWD_MAXG) sm.cnt[parity ^ 1][threadIdx.x] = 0;      // counters of the next group
            if (G == 128) bwd_phase_b<2>(sm, cntp, g0, gcnt, cap, ox, oy, acc_base);
            else if (G == 64) bwd_phase_b<4>(sm, cntp, g0, gcnt, cap, ox, oy, acc_base);
            else if (G == 32) bwd_phase_b<8>(sm, cntp, g0, gcnt, cap, ox, oy, acc_base);
            else bwd_phase_b<16>(sm, cntp, g0, gcnt, cap, ox, oy, acc_base);     // G = 16, and G = 8 with half the threads idle
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------
// K4 split variant (default): the two phases as two kernels, with the per-(tile, surfel) record lists in GLOBAL
// memory (the fused kernel above remains the fallback when the list budget does not cover the scene).
//
// Why: in the fused kernel the lists live in 64 KB of shared memory and both phases share one register budget
// (125 registers, 2 CTAs = 16 warps per SM); its top stall reason is the block barrier between the phases
// (profiles/r02_raster.md: barrier 2.1, wait 1.7 warps per issue at 47 % issue utilisation).  HBM, on the other
// hand, is idle (5 % DRAM utilisation).  So:
//   kernel A (pixel-parallel, back to front)  = phase A; records go to the instance's slice of a global buffer.
//     The slice length is the instance's cull-box area inside the tile -- exact, so there is no capacity rule, no
//     group size G, no phase-B barrier: three block barriers per chunk of 256 surfels instead of seven.
//   kernel B (instance-parallel)              = phase B; TPI lanes walk an instance's records (contiguous 16-byte
//     entries), re-derive the geometry with the same eval_pair() (same bits), reduce-scatter, global atomics.
// Slices are laid out tile by tile: a warp-per-tile pre-pass sums the clipped cull-box areas, one block scans the
// tile totals.  If the total exceeds the buffer, a device flag routes the launch to the fused kernel instead (no
// host synchronisation either way).  Extra traffic: 16 B written + read per record, ~2 x 26 M records on C2.
// ---------------------------------------------------------------------------
// one warp per tile: sum of the clipped cull-box areas of the tile's instances
__global__ void __launch_bounds__(256)
bwd_tile_area_kernel(RasterDims d, RasterWs ws, uint32_t *__restrict__ tile_rec_start)
{
    if (ws.status[1]) return;
    const size_t t = (size_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (t >= (size_t)d.NV * d.T) return;
    const int lane = threadIdx.x & 31;
    const int view = (int)(t / d.T), tile = (int)(t % d.T);
    const int ox = (tile % d.gx) * GA_BLOCK_X, oy = (tile / d.gx) * GA_BLOCK_Y;
    const uint32_t start = ws.tile_start[t], end = ws.tile_start[t + 1];
    const float *rec_base = ws.rec + (size_t)view * d.P * GA_REC_F;
    // 64-bit: up to 256 records per instance, so 2^24 instances of one tile reach 2^32
    unsigned long long sum = 0;
    for (uint32_t i = start + lane; i < end; i += 32) {
        const float4 bb = __ldg(reinterpret_cast<const float4 *>(rec_base + (size_t)ws.ids[i] * GA_REC_F) + 4);
        sum += (unsigned long long)clipped_box_area(bb, ox, oy);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) tile_rec_start[t] = (uint32_t)min(sum, 0xffffffffull);     // saturated: the total saturates too
}

// exclusive scan of the tile totals (one block); sets the fallback flag when the buffer is too small.  The scan runs
// in 64 bits and the total is stored saturated at 0xffffffff, above every capacity (<= 0xfffffff0): a total that
// wrapped at 2^32 could look small enough for the buffer.  The offsets themselves stay 32-bit -- they are only used
// when the total fits the buffer.
__global__ void __launch_bounds__(1024)
bwd_scan_area_kernel(RasterDims d, RasterWs ws, uint32_t *__restrict__ tile_rec_start)
{
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    if (ws.status[1]) return;
    const int n = d.NV * d.T;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const unsigned long long v = i < n ? tile_rec_start[i] : 0u;
        unsigned long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long wv = s_warp[lane];
            unsigned long long wx = wv;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(0xffffffffu, wx, o);
                if (lane >= o) wx += y;
            }
            s_warp[lane] = wx - wv;
        }
        __syncthreads();
        const unsigned long long excl = s_carry + s_warp[warp] + x - v;
        if (i < n) tile_rec_start[i] = (uint32_t)excl;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = excl + v;
        __syncthreads();
    }
    // total records needed; > capacity -> the fused kernel runs instead
    if (threadIdx.x == 0) tile_rec_start[n] = (uint32_t)min(s_carry, 0xffffffffull);
}

// the record buffer of the split backward is too small for this launch: every split kernel exits, the fused one runs
__device__ __forceinline__ bool bwd_lists_overflow(const RasterDims &d, const BwdLists &L)
{
    return L.tile_rec_start[d.NV * d.T] > L.capacity;
}

// LISTS: only the normal / colour records are needed in shared memory (alpha and depth come from the list entries);
// the 16 KB that frees pay for a deeper ring of list rows
template <bool LISTS>
struct BwdASmem {
    float4 rec[LISTS ? 2 : 6][CHUNK];
    uint32_t off[CHUNK];            // start of the instance's slice, relative to the tile's base
    int cnt[CHUNK];
    uint32_t wsum[8];
    int maxc, maxn;
};

#ifndef GA_BWD_A_TMA
#define GA_BWD_A_TMA 1              /* list rows of single-chunk tiles through cp.async.bulk + mbarriers */
#endif
#define BWD_A_RING 9                /* 4 KB list rows in flight per CTA (static shared memory stays below 48 KB) */

// 1-D bulk copy global -> shared with mbarrier completion (SASS: UBLKCP): one 4 KB list row per call
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     sm100::smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(sm100::smem_u32(bar))
                 : "memory");
}

// LISTS = true: the pairs come from the per-pixel contribution lists the forward recorded (RasterWs.lists): every lane
// walks ITS pixel's entries back to front -- {list position, alpha, depth} -- so there is no cull test, no pair
// evaluation and no wasted round on a surfel that does not reach alpha >= 1/255 at this pixel; alpha and depth are
// the forward's own bits.  LISTS = false recomputes (tiles whose lists overflowed, or list_k == 0).
template <bool LISTS>
__global__ void __launch_bounds__(256, BWD_A_CTAS)
render_bwd_a_kernel(RasterDims d, RasterWs ws, BwdLists L, const float *__restrict__ bg,
                    const float *__restrict__ dL_dcolor, const float *__restrict__ dL_dallmap)
{
    __shared__ BwdASmem<LISTS> sm;
    constexpr int REC_NR = LISTS ? 0 : 3, REC_GB = LISTS ? 1 : 5;
    if (ws.status[1] || bwd_lists_overflow(d, L)) return;
    const int view = blockIdx.z;
    const int tile = blockIdx.y * d.gx + blockIdx.x;
    {
        const bool listed = d.list_k > 0 && ws.tile_flag[(size_t)view * d.T + tile] == 0;
        if (listed != LISTS) return;                   // block-uniform: the other instantiation handles this tile
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ox = blockIdx.x * GA_BLOCK_X, oy = blockIdx.y * GA_BLOCK_Y;
    const int lx0 = (warp & 1) * 8, ly0 = (warp >> 1) * 4;
    const int lxi = lx0 + (lane & 7), lyi = ly0 + (lane >> 3);
    const int pxi = ox + lxi, pyi = oy + lyi;
    const int pix_local = lyi * 16 + lxi;
    const bool inside = pxi < d.W && pyi < d.H;
    const float pfx = (float)pxi, pfy = (float)pyi;
    const float bx_lo = (float)(ox + lx0), bx_hi = (float)(ox + lx0 + 7);
    const float by_lo = (float)(oy + ly0), by_hi = (float)(oy + ly0 + 3);

    const size_t gt = (size_t)view * d.T + tile;
    const uint32_t start = ws.tile_start[gt];
    const uint32_t tile_base = L.tile_rec_start[gt];
    const size_t HW = (size_t)d.H * d.W;
    const size_t pix = inside ? (size_t)pyi * d.W + pxi : 0;
    const float *fT = ws.final_T + (size_t)view * 3 * HW;
    const int32_t *nc = ws.n_contrib + (size_t)view * 2 * HW;
    const float *rec_base = ws.rec + (size_t)view * d.P * GA_REC_F;

    const float T_final = inside ? fT[pix] : 0.f;
    float T = T_final;
    const int last_contributor = inside ? nc[pix] : 0;
    const int median_contributor = inside ? nc[pix + HW] : 0;
    float dpx0 = 0, dpx1 = 0, dpx2 = 0, dL_ddepth = 0, dL_daccum = 0, dL_dreg = 0;
    float dn0 = 0, dn1 = 0, dn2 = 0, dL_dmedian = 0;
    if (inside) {
        const float *gc = dL_dcolor + (size_t)view * 3 * HW;
        const float *ga = dL_dallmap + (size_t)view * 7 * HW;
        dpx0 = gc[pix]; dpx1 = gc[pix + HW]; dpx2 = gc[pix + 2 * HW];
        dL_ddepth = ga[pix]; dL_daccum = ga[pix + HW];
        dn0 = ga[pix + 2 * HW]; dn1 = ga[pix + 3 * HW]; dn2 = ga[pix + 4 * HW];
        dL_dmedian = ga[pix + 5 * HW]; dL_dreg = ga[pix + 6 * HW];
    }
    const float final_D = inside ? fT[pix + HW] : 0.f, final_D2 = inside ? fT[pix + 2 * HW] : 0.f;
    const float final_A = 1 - T_final;
    const float bg_dot_dpixel = bg[0] * dpx0 + bg[1] * dpx1 + bg[2] * dpx2;
    float last_alpha = 0, v_last = 0, v_acc = 0, last_dL_dT = 0;        // one scalar suffix recurrence (see the fused kernel)
    // LISTS: this pixel's entries, walked from the last contribution to the first.
    //  * tiles whose surfel list fits one chunk (nearly all): ROW mode.  Row k of the tile's list array is one
    //    contiguous 4 KB block {entry k of the 256 pixels}; thread 0 streams the rows the tile uses, last row first,
    //    through a ring of BWD_A_RING shared-memory slots with cp.async.bulk + full/empty mbarriers (three rows ahead
    //    of the consumers); at row k the lanes whose pixel has more than k contributions take their entry from the slot.
    //  * longer tiles: every lane walks its own list with three entries in flight in registers (`e`, `e1`, `e2`).
    const uint4 *my_list = nullptr;
    const char *tile_rows = nullptr;
    int kk = -1, nl = 0;
    uint4 e = make_uint4(0u, 0u, 0u, 0u), e1 = e, e2 = e;
    __shared__ __align__(128) uint4 s_rows[LISTS ? BWD_A_RING : 1][LISTS ? 256 : 1];
    __shared__ uint64_t s_full[BWD_A_RING], s_empty[BWD_A_RING];
    if (LISTS) {
        const uint4 *tl = ws.lists + ((size_t)view * d.T + tile) * (size_t)d.list_k * 256;
        tile_rows = reinterpret_cast<const char *>(tl);
        my_list = tl + pix_local;
        nl = inside ? ws.n_list[(size_t)view * HW + pix] : 0;
    }

    if (threadIdx.x == 0) {
        sm.maxc = 0;
        sm.maxn = 0;
        if (LISTS) {
#pragma unroll
            for (int i = 0; i < BWD_A_RING; i++) { sm100::mbar_init(&s_full[i], 1); sm100::mbar_init(&s_empty[i], 8); }
            sm100::fence_barrier_init();
        }
    }
    __syncthreads();
    {
        int m = last_contributor, mn = nl;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
            mn = max(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        }
        if (lane == 0) { atomicMax(&sm.maxc, m); atomicMax(&sm.maxn, mn); }
    }
    __syncthreads();
    const int total = sm.maxc;          // list positions [0,total) matter; the rest keep inst_cnt == 0 (memset)
    uint32_t run = 0;                   // records handed out to the chunks staged so far
    const bool rows_mode = LISTS && GA_BWD_A_TMA && total <= CHUNK;          // block-uniform
    const int maxn = sm.maxn;
    auto issue_row = [&](const int j) {                                   // thread 0 only: j-th row in processing order
        const int slot = j % BWD_A_RING, use = j / BWD_A_RING;
        if (use > 0) sm100::mbar_wait(&s_empty[slot], (uint32_t)((use - 1) & 1));      // all 8 warps are done with its last row
        sm100::mbar_expect_tx(&s_full[slot], 4096u);
        bulk_g2s(&s_rows[slot][0], tile_rows + (size_t)(maxn - 1 - j) * 4096, 4096u, &s_full[slot]);
    };
    if (LISTS) {
        if (rows_mode) {
            if (threadIdx.x == 0)
                for (int j = 0; j < min(maxn, BWD_A_RING - 2); j++) issue_row(j);
        } else {
            kk = nl - 1;
            if (kk >= 0) e = __ldg(my_list + (size_t)kk * 256);
            if (kk >= 1) e1 = __ldg(my_list + (size_t)(kk - 1) * 256);
            if (kk >= 2) e2 = __ldg(my_list + (size_t)(kk - 2) * 256);
#pragma unroll
            for (int q = 3; q < 8; q++)
                if (kk >= q) asm volatile("prefetch.global.L2 [%0];" ::"l"(my_list + (size_t)(kk - q) * 256));
        }
    }

    for (int hi = total; hi > 0; hi -= CHUNK) {
        const int lo = max(0, hi - CHUNK);
        const int cnt = hi - lo;
        // stage positions lo..hi-1; slot t holds position hi-1-t (back to front); slice length = clipped box area
        uint32_t area = 0;
        if ((int)threadIdx.x < cnt) {
            const uint32_t id = ws.ids[start + (hi - 1 - threadIdx.x)];
            const float4 *src = reinterpret_cast<const float4 *>(rec_base + (size_t)id * GA_REC_F);
            float4 q4;
            if (LISTS) {
                sm.rec[REC_NR][threadIdx.x] = __ldg(src + 3);
                sm.rec[REC_GB][threadIdx.x] = __ldg(src + 5);
                q4 = __ldg(src + 4);
            } else {
                float4 q[6];
#pragma unroll
                for (int k = 0; k < 6; k++) { q[k] = __ldg(src + k); sm.rec[k][threadIdx.x] = q[k]; }
                q4 = q[4];
            }
            area = (uint32_t)clipped_box_area(q4, ox, oy);
        }
        uint32_t x = area;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) sm.wsum[warp] = x;
        __syncthreads();
        uint32_t wbase = 0, chunk_total = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) { const uint32_t wv = sm.wsum[k]; if (k < warp) wbase += wv; chunk_total += wv; }
        const uint32_t my_off = run + wbase + x - area;
        sm.off[threadIdx.x] = my_off;
        sm.cnt[threadIdx.x] = 0;
        if ((int)threadIdx.x < cnt) L.inst_off[start + (hi - 1 - threadIdx.x)] = tile_base + my_off;
        __syncthreads();

        // one (pixel, surfel) contribution: the compositing recurrences backwards + the 16-byte record for kernel B
        auto contribute = [&](const int jj, const int contributor, const float alpha, const float c_d) {
                    const float4 nr = sm.rec[REC_NR][jj], gb = sm.rec[REC_GB][jj];
                    const float inv1ma = fast_rcp(1.f - alpha);
                    T = T * inv1ma;
                    const float w = alpha * T;
                    float dL_dz = 0.0f;
                    const float inv_cd = fast_rcp(c_d);
                    const float m_d = GA_M_C0 - GA_M_C1 * inv_cd;
                    const float dmd_dd = GA_M_C1 * inv_cd * inv_cd;
                    if (contributor == median_contributor - 1) dL_dz += dL_dmedian;
                    const float dL_dweight = (final_D2 + m_d * m_d * final_A - 2 * m_d * final_D) * dL_dreg;
                    const float dL_dmd = 2.0f * (T * alpha) * (m_d * final_A - final_D) * dL_dreg;
                    dL_dz += dL_dmd * dmd_dd;
                    const float v = ((nr.w * dpx0 + gb.x * dpx1) + (gb.y * dpx2 + c_d * dL_ddepth)) +
                                    ((nr.x * dn0 + nr.y * dn1) + (nr.z * dn2 + dL_daccum));
                    v_acc = last_alpha * v_last + (1.f - last_alpha) * v_acc;
                    v_last = v;
                    float dL_dalpha = (v - v_acc) + (dL_dweight - last_dL_dT);
                    last_dL_dT = dL_dweight * alpha + (1 - alpha) * last_dL_dT;
                    dL_dalpha *= T;
                    last_alpha = alpha;
                    dL_dalpha += (-T_final * inv1ma) * bg_dot_dpixel;
                    dL_dz += w * dL_ddepth;
                    const int slot = atomicAdd(&sm.cnt[jj], 1);          // < the instance's clipped box area by construction
                    L.records[(size_t)tile_base + sm.off[jj] + (uint32_t)slot] =
                        make_uint4((uint32_t)pix_local, __float_as_uint(dL_dalpha), __float_as_uint(dL_dz), __float_as_uint(w));
        };
        if (LISTS && rows_mode) {
            for (int j = 0; j < maxn; j++) {
                const int k = maxn - 1 - j, slot = j % BWD_A_RING;
                if (threadIdx.x == 0 && j + BWD_A_RING - 2 < maxn) issue_row(j + BWD_A_RING - 2);
                sm100::mbar_wait(&s_full[slot], (uint32_t)((j / BWD_A_RING) & 1));
                if (nl > k) {
                    const uint4 cur = s_rows[slot][pix_local];
                    contribute(hi - 1 - (int)cur.x, (int)cur.x, __uint_as_float(cur.y), __uint_as_float(cur.z));
                }
                __syncwarp();
                if (lane == 0) sm100::mbar_arrive(&s_empty[slot]);          // this warp has read row k out of the slot
            }
        } else if (LISTS) {
            while (true) {
                const bool active = kk >= 0 && (int)e.x >= lo;      // entries are in descending list position
                if (!__any_sync(0xffffffffu, active)) break;
                if (active) {
                    const uint4 cur = e;
                    e = e1; e1 = e2;
                    if (kk >= 3) e2 = __ldg(my_list + (size_t)(kk - 3) * 256);   // entries kk-1, kk-2, kk-3 are in flight
                    // ... and the row 8 below is asked into L2 (the list rows stream from HBM exactly once)
                    if (kk >= 8) asm volatile("prefetch.global.L2 [%0];" ::"l"(my_list + (size_t)(kk - 8) * 256));
                    kk--;
                    contribute(hi - 1 - (int)cur.x, (int)cur.x, __uint_as_float(cur.y), __uint_as_float(cur.z));
                }
            }
        } else if constexpr (!LISTS) {
        for (int sb = 0; sb < cnt; sb += 32) {
            bool hit = false;
            if (sb + lane < cnt) {
                const float4 bb = sm.rec[4][sb + lane];
                hit = !(bb.y < bx_lo || bb.x > bx_hi || bb.w < by_lo || bb.z > by_hi);
            }
            unsigned mask = __ballot_sync(0xffffffffu, hit);
            unsigned mine = 0;
            while (mask) {
                const int b = __ffs(mask) - 1;
                mask &= mask - 1;
                const float4 bb = sm.rec[4][sb + b];
                if (pfx >= bb.x && pfx <= bb.y && pfy >= bb.z && pfy <= bb.w && (hi - 1 - (sb + b)) < last_contributor)
                    mine |= 1u << b;
            }
            if (!inside) mine = 0;
            while (__any_sync(0xffffffffu, mine != 0)) {
                const bool active = mine != 0;
                const int bsel = active ? __ffs(mine) - 1 : 0;
                mine &= mine - 1;
                const int jj = sb + bsel;
                const float4 a = sm.rec[0][jj], b = sm.rec[1][jj], c = sm.rec[2][jj];
                PixelGeom pg;
                float k0, k1, k2, l0, l1, l2;
                const bool ok = active && eval_pair(a, b, c, pfx, pfy, pg, k0, k1, k2, l0, l1, l2);
                if (ok) contribute(jj, hi - 1 - jj, pg.alpha, pg.depth);
            }
        }
        }
        __syncthreads();
        if ((int)threadIdx.x < cnt) L.inst_cnt[start + (hi - 1 - threadIdx.x)] = (uint32_t)sm.cnt[threadIdx.x];
        run += chunk_total;
        // sm.rec / off / cnt are rewritten by the next chunk's staging only after every thread passed the barrier above
        // and read its own cnt entry -- the staging below writes rec first, and off/cnt after its own barrier
    }
}

template <int TPI>
__global__ void __launch_bounds__(BWD_B_THREADS, BWD_B_CTAS)
render_bwd_b_kernel(RasterDims d, RasterWs ws, BwdLists L, const float *__restrict__ dL_dcolor,
                    const float *__restrict__ dL_dallmap, float *__restrict__ grad_acc, const int tile_filter)
{
    __shared__ float4 s_up[2][256];
    if (ws.status[1] || bwd_lists_overflow(d, L)) return;
    const int view = blockIdx.z;
    const int tile = blockIdx.y * d.gx + blockIdx.x;
    // tile_filter 1: only tiles whose records came from the list-walking kernel A; 2: only the flagged (recomputed)
    // ones -- the two chains A<true> -> B(1) and A<false> -> B(2) run on two streams; 0: every tile
    if (tile_filter && (ws.tile_flag[(size_t)view * d.T + tile] != 0) != (tile_filter == 2)) return;
    const int ox = blockIdx.x * GA_BLOCK_X, oy = blockIdx.y * GA_BLOCK_Y;
    const size_t gt = (size_t)view * d.T + tile;
    const uint32_t start = ws.tile_start[gt], end = ws.tile_start[gt + 1];
    const int total = (int)(end - start);
    if (total == 0) return;
    {
      for (int px = threadIdx.x; px < 256; px += BWD_B_THREADS) {
        const int lxi = px & 15, lyi = px >> 4;
        const int pxi = ox + lxi, pyi = oy + lyi;
        float4 ua = make_float4(0.f, 0.f, 0.f, 0.f), ub = ua;
        if (pxi < d.W && pyi < d.H) {
            const size_t HW = (size_t)d.H * d.W, pix = (size_t)pyi * d.W + pxi;
            const float *gc = dL_dcolor + (size_t)view * 3 * HW;
            const float *ga = dL_dallmap + (size_t)view * 7 * HW;
            ua = make_float4(gc[pix], gc[pix + HW], gc[pix + 2 * HW], ga[pix + 2 * HW]);
            ub = make_float4(ga[pix + 3 * HW], ga[pix + 4 * HW], 0.f, 0.f);
        }
        s_up[0][px] = ua;              // index = ly * 16 + lx = the records' pixel field
        s_up[1][px] = ub;
      }
    }
    __syncthreads();
    const float *rec_base = ws.rec + (size_t)view * d.P * GA_REC_F;
    float *acc_base = grad_acc + (size_t)view * d.P * GA_GRAD_F;
    const int lane = threadIdx.x & 31;
    const int sub = threadIdx.x % TPI;
    constexpr int IPB = BWD_B_THREADS / TPI;    // instances per pass
    constexpr int NH = 512 / BWD_B_THREADS;     // instances each thread files in the counting sort
    // Instances carry 0 .. ~30 records; a warp's pass lasts as long as its longest instance.  So the tile's instances
    // are handled in super-chunks of 512: a counting sort by record count (descending, empty ones dropped) decides
    // which instance each lane group takes, and every warp gets instances of similar length.
    __shared__ int s_bin[64];
    __shared__ uint16_t s_perm[512];
    __shared__ int s_m;
    // count / surfel id / slice start of the super-chunk's instances, loaded together while the sort runs: a pass then
    // starts with ONE round trip (geometry record + first list records, independent) instead of four dependent ones
    __shared__ uint32_t s_cnt[512], s_id[512], s_off[512];
    for (int c0 = 0; c0 < total; c0 += 512) {
        const int cn = min(512, total - c0);
        if (threadIdx.x < 64) s_bin[threadIdx.x] = 0;
        __syncthreads();
        int myn[NH];
#pragma unroll
        for (int h = 0; h < NH; h++) {
            const int i = h * BWD_B_THREADS + threadIdx.x;
            myn[h] = i < cn ? (int)L.inst_cnt[start + c0 + i] : 0;
            if (i < cn) {
                s_cnt[i] = (uint32_t)myn[h];
                s_id[i] = ws.ids[start + c0 + i];
                s_off[i] = L.inst_off[start + c0 + i];
            }
            if (myn[h] > 0) atomicAdd(&s_bin[min(myn[h], 63)], 1);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            // exclusive prefix over the bins in DESCENDING count order (bin 63 first); bin 0 is unused
            const int hi_bin = 63 - 2 * threadIdx.x, lo_bin = hi_bin - 1;
            const int vh = s_bin[hi_bin], vl = lo_bin >= 1 ? s_bin[lo_bin] : 0;
            int x = vh + vl;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, o);
                if ((int)threadIdx.x >= o) x += y;
            }
            const int excl = x - (vh + vl);
            s_bin[hi_bin] = excl;
            if (lo_bin >= 1) s_bin[lo_bin] = excl + vh;
            if (threadIdx.x == 31) s_m = x;
        }
        __syncthreads();
#pragma unroll
        for (int h = 0; h < NH; h++)
            if (myn[h] > 0) s_perm[atomicAdd(&s_bin[min(myn[h], 63)], 1)] = (uint16_t)(h * BWD_B_THREADS + threadIdx.x);
        __syncthreads();
        const int m = s_m;
    for (int base = 0; base < m; base += IPB) {
        const int slot = base + threadIdx.x / TPI;
        const bool valid = slot < m;
        const int li = valid ? (int)s_perm[slot] : 0;
        const int n = valid ? (int)s_cnt[li] : 0;
        float g[GA_GRAD_F];
#pragma unroll
        for (int f = 0; f < GA_GRAD_F; f++) g[f] = 0.f;
        uint32_t id = 0;
        if (n > 0) {
            id = s_id[li];
            const float4 *src = reinterpret_cast<const float4 *>(rec_base + (size_t)id * GA_REC_F);
            const float4 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
            const float opa = c.w;
            const uint4 *lst = L.records + s_off[li];
            auto process = [&](const uint4 rc) {
                const int pix = (int)rc.x;
                const float dL_dalpha = __uint_as_float(rc.y), dL_dz = __uint_as_float(rc.z), w = __uint_as_float(rc.w);
                const float pfx = (float)(ox + (pix & 15)), pfy = (float)(oy + (pix >> 4));
                PixelGeom pg;
                float k0, k1, k2, l0, l1, l2;
                eval_pair(a, b, c, pfx, pfy, pg, k0, k1, k2, l0, l1, l2);      // same code path as kernel A: same bits
                const float G = pg.G;
                const float dL_dG = opa * dL_dalpha;                           // 0.99 clamp passed through (upstream)
                if (pg.use3d) {
                    const float dL_ds0 = dL_dG * -G * pg.s0 + dL_dz * b.z;
                    const float dL_ds1 = dL_dG * -G * pg.s1 + dL_dz * b.w;
                    const float ip = fast_rcp(pg.p2);
                    const float q0 = dL_ds0 * ip, q1 = dL_ds1 * ip;
                    const float q2 = -(q0 * pg.s0 + q1 * pg.s1);
                    const float dk0 = l1 * q2 - l2 * q1, dk1 = l2 * q0 - l0 * q2, dk2 = l0 * q1 - l1 * q0;
                    const float dl0 = q1 * k2 - q2 * k1, dl1 = q2 * k0 - q0 * k2, dl2 = q0 * k1 - q1 * k0;
                    g[0] -= dk0; g[1] -= dk1; g[2] -= dk2;
                    g[3] -= dl0; g[4] -= dl1; g[5] -= dl2;
                    g[6] += pfx * dk0 + pfy * dl0 + dL_dz * pg.s0;
                    g[7] += pfx * dk1 + pfy * dl1 + dL_dz * pg.s1;
                    g[8] += pfx * dk2 + pfy * dl2 + dL_dz;
                } else {
                    g[9] += dL_dG * (-G * GA_FILTER_INV_SQUARE * pg.dx);
                    g[10] += dL_dG * (-G * GA_FILTER_INV_SQUARE * pg.dy);
                    g[8] += dL_dz;
                }
                g[14] += G * dL_dalpha;
                const float4 ua = s_up[0][pix], ub = s_up[1][pix];
                g[15] += w * ua.x; g[16] += w * ua.y; g[17] += w * ua.z;
                g[11] += w * ua.w; g[12] += w * ub.x; g[13] += w * ub.y;
            };
#if BWD_B_UNROLL == 2
            // two records per iteration: two independent dependency chains per lane (the kernel is latency bound)
            uint4 n0 = sub < n ? __ldg(lst + sub) : make_uint4(0u, 0u, 0u, 0u);
            uint4 n1 = sub + TPI < n ? __ldg(lst + sub + TPI) : n0;
            for (int r = sub; r < n; r += 2 * TPI) {
                const uint4 r0 = n0;
                // no second record: reuse the first one's pixel with zero upstream terms (adds exact zeros), so both
                // bodies run unconditionally and the compiler can interleave them
                const uint4 r1 = (r + TPI < n) ? n1 : make_uint4(n0.x, 0u, 0u, 0u);
                if (r + 2 * TPI < n) n0 = __ldg(lst + r + 2 * TPI);
                if (r + 3 * TPI < n) n1 = __ldg(lst + r + 3 * TPI);
                process(r0);
                process(r1);
            }
#else
            uint4 nxt = sub < n ? __ldg(lst + sub) : make_uint4(0u, 0u, 0u, 0u);
            for (int r = sub; r < n; r += TPI) {
                const uint4 rc = nxt;
                if (r + TPI < n) nxt = __ldg(lst + r + TPI);           // the next record's load overlaps this one's math
                process(rc);
            }
#endif
        }
        if (__any_sync(0xffffffffu, n > 0)) {
            float *dst = acc_base + (size_t)id * GA_GRAD_F;          // lanes without records carry zeros (id 0, adds skipped)
            reduce_scatter18<TPI>(g, lane, dst);
        }
    }
        __syncthreads();                         // s_bin / s_perm are rebuilt for the next super-chunk
    }
}

static int g_bwd_split = -1;

// slice layout of the split backward's record buffer: per-tile sums of the clipped cull-box areas + their scan.
// Called by the forward (list_k > 0) on a side stream, concurrently with the composite, or by the backward.
cudaError_t ga_launch_bwd_slices(const RasterDims &d, const RasterWs &w, uint32_t *tile_rec_start, cudaStream_t s)
{
    const int tiles = d.NV * d.T;
    bwd_tile_area_kernel<<<(tiles + 7) / 8, 256, 0, s>>>(d, w, tile_rec_start);
    bwd_scan_area_kernel<<<1, 1024, 0, s>>>(d, w, tile_rec_start);
    return cudaGetLastError();
}

cudaError_t ga_launch_render_fwd_with_slices(const RasterDims &d, const RasterWs &w, const float *bg, float *out_color,
                                             float *out_allmap, cudaStream_t s)
{
    // the LISTS forward kernel leaves every tile's slice total in tile_rec_start; one small block turns them into offsets
    cudaError_t e = ga_launch_render_fwd(d, w, bg, out_color, out_allmap, s);
    if (e != cudaSuccess) return e;
    bwd_scan_area_kernel<<<1, 1024, 0, s>>>(d, w, w.tile_rec_start);
    return cudaGetLastError();
}

cudaError_t ga_launch_render_bwd(const RasterDims &d, const RasterWs &w, const float *bg,
                                 const float *dL_dcolor, const float *dL_dallmap,
                                 float *grad_acc, const BwdLists &lists_in, cudaStream_t s)
{
    static GaPerDevice attr_set;
    if (ga_first_use_on_device(attr_set)) {
        cudaError_t e = cudaFuncSetAttribute(render_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)sizeof(BwdSmem));
        if (e != cudaSuccess) return e;
    }
    if (g_bwd_split < 0) {
        const char *e = getenv("GA_B200_BWD_SPLIT");        // 0: always the fused kernel (A/B comparisons)
        g_bwd_split = (e && e[0] == '0') ? 0 : 1;
    }
    dim3 grid(d.gx, d.gy, d.NV);
    BwdLists lists = lists_in;
    const bool split = g_bwd_split && lists.records && lists.capacity > 0;
    if (split) {
        cudaError_t e;
        if (d.list_k > 0) {
            lists.tile_rec_start = w.tile_rec_start;                 // laid out by the forward
        } else if ((e = ga_launch_bwd_slices(d, w, lists.tile_rec_start, s)) != cudaSuccess) {
            return e;
        }
        if (d.list_k > 0) {
            // tiles whose per-pixel lists overflowed are few and long: their recompute kernel runs beside the
            // list-walking one instead of after it
            // tiles whose per-pixel lists overflowed are few and long: their chain (recompute kernel A -> kernel B on
            // those tiles) runs on the side stream beside the list-walking chain instead of in front of / behind it
            GaSide *g = ga_side();
            if (g) {
                cudaEventRecord(g->fork, s);
                cudaStreamWaitEvent(g->st, g->fork, 0);
                render_bwd_a_kernel<false><<<grid, 256, 0, g->st>>>(d, w, lists, bg, dL_dcolor, dL_dallmap);
                render_bwd_b_kernel<BWD_B_TPI><<<grid, BWD_B_THREADS, 0, g->st>>>(d, w, lists, dL_dcolor, dL_dallmap, grad_acc, 2);
                cudaEventRecord(g->join, g->st);
                render_bwd_a_kernel<true><<<grid, 256, 0, s>>>(d, w, lists, bg, dL_dcolor, dL_dallmap);
                render_bwd_b_kernel<BWD_B_TPI><<<grid, BWD_B_THREADS, 0, s>>>(d, w, lists, dL_dcolor, dL_dallmap, grad_acc, 1);
                cudaStreamWaitEvent(s, g->join, 0);
            } else {
                render_bwd_a_kernel<true><<<grid, 256, 0, s>>>(d, w, lists, bg, dL_dcolor, dL_dallmap);
                render_bwd_a_kernel<false><<<grid, 256, 0, s>>>(d, w, lists, bg, dL_dcolor, dL_dallmap);
                render_bwd_b_kernel<BWD_B_TPI><<<grid, BWD_B_THREADS, 0, s>>>(d, w, lists, dL_dcolor, dL_dallmap, grad_acc, 0);
            }
        } else {
            render_bwd_a_kernel<false><<<grid, 256, 0, s>>>(d, w, lists, bg, dL_dcolor, dL_dallmap);
            render_bwd_b_kernel<BWD_B_TPI><<<grid, BWD_B_THREADS, 0, s>>>(d, w, lists, dL_dcolor, dL_dallmap, grad_acc, 0);
        }
    }
    // fused kernel: the whole job when the split path is off, a no-op or the fallback (record buffer too small) otherwise
    render_bwd_kernel<<<grid, 256, sizeof(BwdSmem), s>>>(d, w, bg, dL_dcolor, dL_dallmap, grad_acc,
                                                         split ? lists.tile_rec_start + d.NV * d.T : nullptr, lists.capacity);
    return cudaGetLastError();
}
