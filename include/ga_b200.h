/*
 * ga_b200.h -- C ABI of libga_b200.so: B200 (sm_100a) kernels for the two hot
 * paths of GaussianAnything.  Plain pointers and sizes only; no torch types.
 *
 * All pointers are DEVICE pointers unless stated otherwise.  No entry point
 * allocates, frees or synchronises (except the ga_raster_backward_records
 * probe, which returns a device count); everything is enqueued on `stream`
 * (a cudaStream_t passed as void*).  Return value: 0 on success, a negative
 * GA_ERR_* code on a bad argument, or a positive cudaError_t from the launch.
 *
 * ---------------------------------------------------------------------------
 * Part 1: surfel (2D Gaussian) rasteriser.
 * Replaces the native module `diff_surfel_rasterization._C` that the reference
 * binds at /root/reference/nsr/gs_surfel.py:15 and calls at
 * /root/reference/nsr/gs_surfel.py:100-114 (`_C.rasterize_gaussians`,
 * `_C.rasterize_gaussians_backward`), batched over every (batch item, view)
 * of the Python loop at /root/reference/nsr/gs_surfel.py:65,74.
 * ---------------------------------------------------------------------------
 */
#ifndef GA_B200_H
#define GA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GA_ERR_BADARG   (-1)
#define GA_ERR_WORKSPACE (-2)   /* workspace too small for the stated sizes */
#define GA_ERR_SIZE     (-3)    /* image larger than 4080 px or P*views overflow */

#define GA_RASTER_REC_FLOATS 24   /* packed per-(view,surfel) record, 96 bytes */
#define GA_RASTER_GRAD_FLOATS 18  /* per-(view,surfel) gradient accumulator */

/* Byte offsets of the sections inside the forward workspace.  The forward
 * pass fills them; the backward pass reads them (the workspace is the
 * equivalent of upstream's geomBuffer/binningBuffer/imgBuffer). */
typedef struct GaRasterLayout {
    size_t total_bytes;
    size_t status;      /* int32[16]: [0]=instances D, [1]=overflow flag, [2]=tiles sorted out of smem */
    size_t rec;         /* float[NV*P][24]  Tu3 Tv3 Tw3 | xy2 opacity | normal3 | r | bbox x0 x1 y0 y1 | g b - - */
    size_t depth;       /* float[NV*P]      view-space z (0 when culled) */
    size_t rect;        /* uint32[NV*P]     x0 | y0<<8 | x1<<16 | y1<<24 (tile units) */
    size_t tile_count;  /* uint32[NV*T*8]   scratch: per-tile counters, then fill cursors (8 replicas per tile) */
    size_t tile_start;  /* uint32[NV*T+1]   exclusive scan == tile ranges [start,end) */
    size_t keys;        /* uint64[max_instances]  (depth bits<<32 | surfel), sorted per tile */
    size_t ids;         /* uint32[max_instances]  sorted surfel index per instance */
    size_t final_T;     /* float[NV][3][H*W]  T, M1, M2 */
    size_t n_contrib;   /* int32[NV][2][H*W]  last contributor, median contributor */
    size_t inst_off;    /* uint32[max_instances]  backward: start of the instance's record slice */
    size_t inst_cnt;    /* uint32[max_instances]  backward: records in it */
    size_t n_list;      /* int32[NV][H*W]         (list_k > 0) contributions recorded per pixel */
    size_t tile_flag;   /* uint32[NV*T]           (list_k > 0) 1: a pixel of the tile had more than list_k */
    size_t tile_rec_start; /* uint32[NV*T+1]      (list_k > 0) slice layout of the backward's record buffer */
    size_t lists;       /* uint4[NV*T][list_k][256] (list_k > 0) {list position, alpha bits, depth bits, 0} */
} GaRasterLayout;

/* Fills *layout for NV = batch*views images of H x W, P surfels per batch item
 * and room for max_instances (surfel,tile) pairs over all images.
 * Host-only, no CUDA call. */
int ga_raster_layout(int batch, int P, int views, int H, int W,
                     int64_t max_instances, GaRasterLayout *layout);

/* As ga_raster_layout, with room for the per-pixel contribution lists the forward records when list_k > 0
 * (list_k * 4 KB per tile; 32 is the default the Python mirror uses for calls that need gradients). */
int ga_raster_layout_ex(int batch, int P, int views, int H, int W,
                        int64_t max_instances, int list_k, GaRasterLayout *layout);

/*
 * Forward.  gauss13: [batch][P][13] = xyz3 opacity1 scale2 quat4(wxyz) rgb3, the
 * layout of /root/reference/nsr/gs_surfel.py:68-72.  viewmats / projmats:
 * [batch*views][16] exactly as the reference passes `viewmatrix` /
 * `projmatrix` (row-vector convention).  bg: [3].
 * Outputs: out_color [NV][3][H][W], out_allmap [NV][7][H][W] (channel order of
 * /root/reference/nsr/gs_surfel.py:121-142), out_radii int32 [NV][P].
 * If the instance count exceeds max_instances, status[1] is set and the
 * images are undefined (no out-of-bounds access happens); the caller re-runs
 * with a larger workspace.
 */
int ga_raster_forward(const float *gauss13, int batch, int P, int views,
                      const float *viewmats, const float *projmats, const float *bg,
                      int H, int W, float scale_modifier,
                      float *out_color, float *out_allmap, int32_t *out_radii,
                      void *workspace, size_t workspace_bytes, int64_t max_instances,
                      void *stream);

/* ga_raster_forward with per-pixel contribution lists: list_k > 0 makes the composite record, for every pixel, the
 * (list position, alpha, depth) of each surfel that contributed (up to list_k per pixel; a tile with a longer pixel
 * is flagged and its backward recomputes).  ga_raster_backward_ex with the same list_k then walks those lists instead
 * of re-culling and re-evaluating every (pixel, surfel) pair -- what upstream's backward.cu renderCUDA does.
 * status_host / status_event: both NULL, or as in ga_raster_forward_async. */
int ga_raster_forward_ex(const float *gauss13, int batch, int P, int views,
                         const float *viewmats, const float *projmats, const float *bg,
                         int H, int W, float scale_modifier,
                         float *out_color, float *out_allmap, int32_t *out_radii,
                         void *workspace, size_t workspace_bytes, int64_t max_instances, int list_k,
                         int32_t *status_host, void *status_event, void *stream);

/* The same forward in two halves, for callers that want to look at status[0..1] (instance count, overflow) after
 * the binning -- the point where upstream reads `num_rendered` back (rasterizer_impl.cu) -- and only then enqueue
 * the composite: ga_raster_forward_bin = per-surfel stage + binning, ga_raster_forward_render = composite. */
int ga_raster_forward_bin(const float *gauss13, int batch, int P, int views,
                          const float *viewmats, const float *projmats, const float *bg,
                          int H, int W, float scale_modifier,
                          float *out_color, float *out_allmap, int32_t *out_radii,
                          void *workspace, size_t workspace_bytes, int64_t max_instances, void *stream);
int ga_raster_forward_render(const float *gauss13, int batch, int P, int views,
                             const float *viewmats, const float *projmats, const float *bg,
                             int H, int W, float scale_modifier,
                             float *out_color, float *out_allmap, int32_t *out_radii,
                             void *workspace, size_t workspace_bytes, int64_t max_instances, void *stream);

/* The whole forward enqueued at once, with the status read-back overlapped: right after the tile scan (before the
 * scatter, the sort and the composite) status[0..3] = {instance count, overflow flag, tiles sorted in global memory,
 * 0} is copied to `status_host` (pinned host memory, 4 ints) and `status_event` (a cudaEvent_t) is recorded.  The
 * caller synchronises on the event -- the GPU is still busy with the rest of the forward -- and, if the overflow
 * flag is set, re-runs with a larger workspace (the kernels after the scan exit early in that case). */
int ga_raster_forward_async(const float *gauss13, int batch, int P, int views,
                            const float *viewmats, const float *projmats, const float *bg,
                            int H, int W, float scale_modifier,
                            float *out_color, float *out_allmap, int32_t *out_radii,
                            void *workspace, size_t workspace_bytes, int64_t max_instances,
                            int32_t *status_host, void *status_event, void *stream);

/* ga_raster_backward for a workspace laid out and filled with list_k (ga_raster_layout_ex / ga_raster_forward_ex). */
int ga_raster_backward_ex(const float *gauss13, int batch, int P, int views,
                          const float *viewmats, const float *projmats, const float *bg,
                          int H, int W, float scale_modifier,
                          const int32_t *radii,
                          const float *dL_dcolor, const float *dL_dallmap,
                          const void *workspace, size_t workspace_bytes, int64_t max_instances, int list_k,
                          void *scratch, size_t scratch_bytes,
                          float *grad_gauss13, void *stream);

/* Post-processing of /root/reference/nsr/gs_surfel.py:121-163 for all views at once: image = clamp(color,0,1),
 * alpha = allmap[1], depth = nan_to_num(allmap[5], 0, 0), normal[d] = sum_c allmap[2+c] * view[d][c], dist = allmap[6].
 * color [NV,3,H,W], allmap [NV,7,H,W], viewmats [NV,16] (as passed to the rasteriser); outputs contiguous. */
int ga_render_post_forward(const float *color, const float *allmap, const float *viewmats, int num_views,
                           int H, int W, float *image, float *alpha, float *depth, float *normal, float *dist,
                           void *stream);
/* Its backward: any g_* may be NULL (= zero); writes g_color [NV,3,H,W] and g_allmap [NV,7,H,W]. */
int ga_render_post_backward(const float *color, const float *allmap, const float *viewmats, int num_views,
                            int H, int W, const float *g_image, const float *g_alpha, const float *g_depth,
                            const float *g_normal, const float *g_dist, float *g_color, float *g_allmap, void *stream);

/*
 * The two judgement calls of the (parity-unpinned) restatement of upstream's preprocess stage, switchable at run
 * time; the process-wide defaults are the compile-time macros GA_RADIUS_FORMULA / GA_QUAT_NORM_GRAD (both 0):
 *   radius_formula 0: radius = ceil(max(extent.x, extent.y, 3*FilterSize))   1: ceil(3*max(extent.x, extent.y, FilterSize))
 *   quat_norm_grad 0: dL/dquat is the vjp at q/|q|, not chained through the normalisation   1: chained
 * Replaces nothing in the reference (upstream hard-codes its choice); exists so that pinning against
 * github.com/hbb1/diff-surfel-rasterization forward.cu / backward.cu is a one-line flip.  oracle/surfel_oracle.c
 * has the same switch (so_set_variant).  Affects calls made after it returns.
 */
int ga_raster_set_variant(int radius_formula, int quat_norm_grad);
int ga_raster_get_variant(int *radius_formula, int *quat_norm_grad);

/*
 * Scheduling knob of the forward composite (results do not depend on it): lanes per group that walks its own list of
 * hits inside a warp's 8x4 pixel block -- 32 (one surfel per warp round), 16 or 8 (default; env GA_B200_FWD_GROUP).
 * Returns -1 for any other value.
 */
int ga_raster_set_tuning(int fwd_group);

/* Bytes of scratch the backward wants: gradient accumulators [NV*P][18] (mandatory) + the global record lists of
 * the split backward (64 records of 16 bytes per (surfel, view)).  A smaller buffer that still holds the
 * accumulators is accepted: the backward then runs its fused shared-memory kernel. */
size_t ga_raster_backward_scratch_bytes(int batch, int P, int views);

/*
 * Which backward a scratch buffer gets, and the record budget a scene needs.  *total = the number of 16-byte records
 * the split backward would lay out for the forward in `workspace` -- the value it compares with its capacity on the
 * device -- and *capacity = the records `scratch_bytes` of scratch provide (0: the buffer holds no more than the
 * accumulators, tile table and 4 KB, and the fused kernel is chosen on the host).  total <= capacity: the split
 * kernels run; total > capacity: the fused kernel runs instead.  list_k > 0 reads the layout the forward computed;
 * list_k == 0 computes it into `scratch` exactly as ga_raster_backward_ex would (the scratch must then hold at least
 * the accumulators and the tile table).  Unlike every other entry point this one synchronises `stream` and copies
 * the total to the host.  GA_ERR_WORKSPACE when the forward overflowed its workspace.
 */
int ga_raster_backward_records(int batch, int P, int views, int H, int W,
                               const void *workspace, size_t workspace_bytes, int64_t max_instances, int list_k,
                               void *scratch, size_t scratch_bytes, uint64_t *total, uint64_t *capacity,
                               void *stream);

/*
 * Backward.  dL_dcolor [NV][3][H][W], dL_dallmap [NV][7][H][W]; grad_gauss13
 * [batch][P][13] is OVERWRITTEN with the gradient summed over the views of
 * each batch item (same column order as gauss13).  workspace must be the one
 * the matching forward filled.
 */
int ga_raster_backward(const float *gauss13, int batch, int P, int views,
                       const float *viewmats, const float *projmats, const float *bg,
                       int H, int W, float scale_modifier,
                       const int32_t *radii,
                       const float *dL_dcolor, const float *dL_dallmap,
                       const void *workspace, size_t workspace_bytes, int64_t max_instances,
                       void *scratch, size_t scratch_bytes,
                       float *grad_gauss13, void *stream);

/*
 * ---------------------------------------------------------------------------
 * Part 2: DiT denoiser forward (bf16 tensor-core path, fp32 residual stream).
 * Replaces, for DiT_I23D_PCD_PixelArt_noclip[_clay_stage2].forward
 * (/root/reference/dit/dit_i23d.py:511-567,707-750) and its block
 * ImageCondDiTBlockPixelArtRMSNormClayLRM.forward
 * (/root/reference/dit/dit_models_xformers.py:765-787), the cuBLAS nn.Linear
 * calls, xformers.ops.memory_efficient_attention
 * (/root/reference/vit/vision_transformer.py:297,
 * /root/reference/ldm/modules/attention.py:538-546), xformers FusedMLP
 * (/root/reference/dit/dit_models_xformers.py:281-286) and the RMSNorm /
 * modulate / gate / residual elementwise launches around them.
 * ---------------------------------------------------------------------------
 */

/* Epilogues fused into the tcgen05 GEMM  C[M,N] = A[M,K] * W[N,K]^T (+ bias). */
#define GA_EPI_BF16            0   /* out bf16 [M, ld_out]                                   */
#define GA_EPI_GELU_BF16       1   /* out bf16 = gelu_erf(acc + bias)   (FusedMLP first half) */
#define GA_EPI_F32             2   /* out fp32 [M, ld_out]                                   */
#define GA_EPI_RESID_GATE_F32  3   /* out fp32 [M, ld_out] += gate[m / rows_per_batch, n] * (acc + bias)   */
#define GA_EPI_HEADS           4   /* split columns "(K H 64)" into heads: per-head RMSNorm on q/k, write
                                      Q,K [B,H,tok_pitch,64] and V transposed [B,H,64,tok_pitch] (bf16) */

typedef struct GaGemmEpilogue {
    int mode;
    const float *bias;        /* [N] or NULL */
    void *out;                /* modes 0-3 */
    int ld_out;
    const float *gate;        /* mode 3: [batch, gate_ld] (already offset to the gate chunk) or NULL (= 1) */
    int gate_ld;
    int rows_per_batch;       /* tokens per batch item (modes 3, 4) */
    void *q, *k, *vt;         /* mode 4 outputs (any may be NULL when that part is absent) */
    const float *qn_w, *kn_w; /* per-head RMSNorm weights [64] (NULL = no norm) */
    int heads;
    int first_part;           /* mode 4: 0 when columns start with q, 1 when they start with k (cross-attn k|v) */
    int tok_pitch;            /* padded token count of the Q/K rows and Vt columns (multiple of 128) */
    float eps;
} GaGemmEpilogue;

/* A [M, lda] bf16 row-major, W [N, ldw] bf16 row-major (nn.Linear weight), K contiguous in both.
 * block_n = tile width {64, 128, 192, 256} (the 128 x width output tile; 192: not for GA_EPI_HEADS) + 1000 * cluster size {1, 2}: a cluster of
 * CTAs on vertically adjacent tiles shares the W tile through TMA multicast (e.g. 4256 = width 256, cluster 4);
 * 9000 + width {128, 256} = CTA pair (tcgen05 cta_group::2) computing a 256 x width tile.
 * lda, ldw multiples of 8. */
int ga_gemm_bf16_tn(const void *A, int lda, const void *W, int ldw, int M, int N, int K,
                    const GaGemmEpilogue *epi, int block_n, void *stream);

/* softmax(Q K^T * softmax_scale) V, head_dim 64.  Q [B*H, pitch_q, 64], K [B*H, pitch_k, 64],
 * Vt [B*H, 64, pitch_k] (bf16, padding beyond Nk must be finite); out [B, Nq, H*64] bf16.
 * pitch_k must be a multiple of 128. */
int ga_attention_bf16(const void *Q, const void *K, const void *Vt, void *out, int batch, int heads,
                      int Nq, int Nk, int pitch_q, int pitch_k, float softmax_scale, float score_bound,
                      void *stream);
/* score_bound: an upper bound of |q.k| * softmax_scale over all (q, k) pairs, or <= 0 if unknown.  With
 * RMS-normalised q and k (the DiT's qk-norm) it is 64 * max|w_q| * max|w_k| * softmax_scale; when given
 * (and <= 40) the kernel uses it instead of a running row maximum (same result, one pass over the scores). */

/* out_bf16[r,:] = RMSNorm(x[r,:]; eps) * w [* (1 + scale[b,:]) + shift[b,:]], b = r / rows_per_batch;
 * shift/scale both NULL or both set, rows mod_ld apart. */
int ga_rmsnorm_modulate(const float *x, const float *w, const float *shift, const float *scale,
                        int mod_ld, int rows_per_batch, void *out_bf16, int R, int D, float eps, void *stream);

/* y[b,n] (+)= act_out(bias[n] + sum_k act_in(x[b,k]) W[n,k]);  rows <= 16; act: 0 none, 1 SiLU. */
int ga_linear_small(const float *x, const float *W, const float *bias, float *y, int rows, int N, int K,
                    int act_in, int act_out, int accumulate, void *stream);
int ga_timestep_sinusoid(const float *t, float *out, int rows, int dim, void *stream);
int ga_layernorm_rows(const float *x, const float *w, const float *b, float *y, int R, int D, float eps, void *stream);
/* mod[l,b,e] = tables[l,e] + t0[b, e % t0_ld], e in [0, JD) */
int ga_add_tables(const float *tables, const float *t0, float *mod, int L, int rows, int JD, int t0_ld, void *stream);
/* h = gelu_tanh(W1 [xin2 | xin] + b1) -> bf16 [R, D] (token embedder, first layer) */
int ga_embed_fc1(const float *xin, int Cx, const float *xin2, int C2, const float *W1, const float *b1,
                 void *h_bf16, int R, int D, void *stream);
/* NeRF positional encoding of xyz (63 features, padded to 64) -> bf16 [R, 64] */
int ga_xyz_posenc(const float *xyz, void *out_bf16, int R, void *stream);
/* y[r,c] = bias[c] + sum_d (LayerNorm(x[r])[d] (1 + scale[b,d]) + shift[b,d]) W[c,d]; mod [B,2,D]; Cout <= 16 */
int ga_final_layer(const float *x, const float *mod, const float *W, const float *bias, float *y, int R,
                   int D, int Cout, int rows_per_batch, float eps, void *stream);
/* eps [2*half] = (cond | uncond) -> h = u + s (c - u) written to both halves of out */
int ga_cfg_combine(const float *eps, float *out, int64_t half_elems, float cfg_scale, void *stream);
int ga_axpy(float *x, const float *v, float a, int64_t n, void *stream);          /* x += a v */
int ga_f32_to_bf16(const float *x, void *y, int64_t n, void *stream);

/* ---- VAE decode path latent tokens -> surfels (SURVEY 8f row N1; building blocks, see DESIGN.md 6b) -------------
 * Replaces the elementwise / small-matrix torch ops of /root/reference/vit/vit_triplane.py:287-345,991-1064,1289-1313,
 * 1388-1440, /root/reference/dit/dit_decoder.py:15-42 and /root/reference/nsr/srt/layers.py:82-90,146-186. */
/* out_bf16[r] = LayerNorm(x[r]) [* w + bias] [* (1 + scale[b]) + shift[b]], b = r / rows_per_batch (1 = per token);
 * D % 4 == 0, D <= 1024 */
int ga_layernorm_modulate(const float *x, const float *w, const float *bias, const float *shift, const float *scale,
                          int mod_ld, int rows_per_batch, void *out_bf16, int R, int D, float eps, void *stream);
/* y[r, c] = bias[c] + sum_d f(x[r])[d] W[c, d], f = optional LayerNorm (ln_w, ln_b) then optional SiLU; C <= 16 */
int ga_thin_linear(const float *x, const float *ln_w, const float *ln_b, int apply_silu, const float *W,
                   const float *bias, float *y, int R, int D, int C, float eps, void *stream);
/* attention over S sequences of L <= 16 tokens: qkv bf16 [S*L, 3*H*64] ("(K H D)" columns), q/k RMS-normalised per
 * head with weights qn_w / kn_w [64], softmax(q k^T / 8) v -> out bf16 [S*L, H*64] */
int ga_micro_attention_bf16(const void *qkv, const float *qn_w, const float *kn_w, void *out, int S, int L, int H,
                            float eps, void *stream);
/* seq [S, 1+f, D] fp32: row 0 = the parent token (prev_f == 0: parents[s]; else child s % prev_f of sequence
 * s / prev_f of the previous stage's [S/prev_f, 1+prev_f, D] buffer), rows 1..f = queries [f, D] */
int ga_micro_seq_build(const float *parents, int prev_f, const float *queries, float *seq, int64_t S, int f, int D,
                       void *stream);
/* child r of parent r / f: res row = r, or (res_in_sequences) row (r/f)(1+f) + 1 + r%f of the [R/f, 1+f] sequence
 * layout; pre = res[row] + parent_pre[r/f] (parent_pre NULL at the base level); xyz = tanh(res[row][0:3])
 * * offset_scale + parent_pos[(r/f) * parent_pos_stride + 0..2]; other channels from pre: sigmoid | softplus *
 * scale_factor | normalise | 0.5 tanh + 0.5.  out_gauss13 [R,13] is rasteriser input; out_pre [R,13] feeds the next level */
int ga_surfel_cascade_pack(const float *res, int res_in_sequences, const float *parent_pre, const float *parent_pos,
                           int parent_pos_stride,
                           int f, float offset_scale, float scale_factor, float *out_gauss13, float *out_pre,
                           int64_t R, void *stream);
int ga_silu_to_bf16(const float *x, void *y, int64_t n, void *stream);            /* y = bf16(silu(x)) */

/* Measurement aid: when enabled, cudaEvents are recorded around every kernel
 * stage of the next forward/backward; ga_profile_read synchronises on them and
 * returns per-stage milliseconds: [0] preprocess, [1] binning, [2] render fwd,
 * [3] render bwd (+accumulator memset), [4] per-surfel bwd.  Returns the number
 * of stages written (0 if profiling never ran). */
int ga_profile_enable(int on);
int ga_profile_read(float *ms, int n);

/* Library self-description (host only). */
const char *ga_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GA_B200_H */
