/*
 * dss_b200.h -- C ABI of the B200-native surface-splatting rasterizer (libdss_b200.so).
 *
 * This is the drop-in boundary for ONE hot path of yifita/DSS: the elliptical point rasterizer,
 * forward and backward.  Every entry point is `extern "C"`, takes raw DEVICE pointers (unless a
 * parameter is explicitly marked host), sizes, and a cudaStream_t passed as void*; it enqueues
 * work on that stream and returns an int status (DSS_OK or a negative DSS_E_* code, never a C++
 * exception).  dss_last_error() returns a thread-local description of the last failure.
 *
 * The reference interfaces each entry point replaces are cited as <file>:<line> relative to the
 * yifita/DSS checkout (reference commit 8fd8d86).  Reference-side bindings: INTEGRATION.md.
 *
 * Conventions shared with the reference:
 *   - "packed" arrays hold all N views back to back: view n owns rows
 *     [first_idx[n], first_idx[n] + num_points[n]); first_idx / num_points are int64 DEVICE arrays
 *     exactly as DSS._C receives them (DSS/csrc/rasterize_points.h:461-472);
 *   - points are NDC x,y in [-1,1] (+X left, +Y up) and view-space depth z; points with z < 0 are
 *     never rasterized (DSS/csrc/rasterize_points.cu:87-88);
 *   - output pixel (row r, col c) is the NDC pixel (S-1-r, S-1-c) (rasterize_points.cu:577-580);
 *   - idx / zbuf / qvalue are (N,S,S,K), -1 padded; occupancy (N,S,S) is 0/1 float.
 */
#ifndef DSS_B200_H
#define DSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define DSS_API __attribute__((visibility("default")))
#else
#define DSS_API
#endif

#define DSS_OK 0
#define DSS_E_INVALID -1    /* bad argument (null pointer, size out of range, K too large ...) */
#define DSS_E_CUDA -2       /* a CUDA runtime call or kernel launch failed                    */
#define DSS_E_NOMEM -3      /* scratch allocation failed                                      */
#define DSS_E_CAPACITY -4   /* caller-provided output capacity too small (see *_required)     */

#define DSS_MAX_POINTS_PER_PIXEL 64   /* reference allows 150 (rasterization_utils.cuh:18); configs use 5 / 8 */
#define DSS_MAX_SHARED_VIEWS 256      /* views of one shared cloud per render call (checked by forward AND backward) */

typedef struct dss_ctx dss_ctx;   /* owns grow-only device scratch for one device; not thread-safe */

/* ---- library / context ------------------------------------------------------------------- */
DSS_API int dss_version(void);                       /* ABI version, currently 1                        */
DSS_API const char *dss_last_error(void);            /* thread-local message for the last DSS_E_* return */
DSS_API int dss_create(dss_ctx **out);               /* bind to the CURRENT cuda device                  */
DSS_API void dss_destroy(dss_ctx *ctx);
DSS_API size_t dss_scratch_bytes(const dss_ctx *ctx);/* device bytes currently held by the context       */
/* number of kernels the library has launched on this context since creation (bench: gpu_launches) */
DSS_API int64_t dss_launch_count(const dss_ctx *ctx);

/* ---- optional per-stage device timing ------------------------------------------------------
 * When enabled, every stage (preprocess, bin count, scan, scatter, raster, ...) is bracketed by a CUDA
 * event pair on the launch stream.  dss_profile_read synchronises on the recorded events and returns
 * the accumulated milliseconds and number of brackets of one stage since the last reset.  Used by
 * bench.py for the live roofline of the dominant kernel; off by default (zero overhead). */
DSS_API int dss_profile_enable(dss_ctx *ctx, int on);
DSS_API int dss_profile_reset(dss_ctx *ctx);
DSS_API int dss_profile_num_stages(void);
DSS_API const char *dss_profile_stage_name(int stage);
DSS_API int dss_profile_read(dss_ctx *ctx, int stage, double *total_ms, int64_t *brackets);

/* Debug work counters of the depth-sliced rasterizer (off by default; adds global atomics when on):
 * out[0] tile-list entries scanned, [1] survivors of the block-threshold cull, [2] (splat,pixel) tests,
 * [3] accepted fragments queued for insertion, [4] slices skipped by early termination, [5] rasterization passes
 * (queue flushes) executed, [6] tiles rasterized from the records because their list did not fit the id buffer.
 * enable != 0 switches collection on (and zeroes the counters); out may be NULL. Synchronises the device. */
DSS_API int dss_debug_raster_stats(dss_ctx *ctx, int enable, uint64_t out[8]);

/* Total length of the forward's tile lists as the device published it last (mapped pinned word: no synchronisation, may
 * lag one call behind).  Lets a caller that replays a captured CUDA graph notice that the lists have outgrown the buffer
 * the graph was captured with (dss_b200/graph.py). */
DSS_API int64_t dss_debug_tile_total(const dss_ctx *ctx);

/* Testing: cap the forward's tile-list buffer at max_entries (0 = no cap).  Tiles whose list does not fit are then
 * rasterized from the view's records directly -- the path a sudden growth of the lists takes in production, where the
 * buffer is sized from the previous call without the host ever waiting for the device.  Results must not change. */
DSS_API int dss_debug_limit_tile_capacity(dss_ctx *ctx, int64_t max_entries);

/* ---- exclusive prefix sum -----------------------------------------------------------------
 * Replaces prefix_sum.prefix_sum_cuda(grid_cnt, num_grids, grid_off)
 * (external/prefix_sum/prefix_sum.h:6-21, prefix_sum.cu:74-87,135-205): exclusive int32 scan of the
 * first n elements of `in` into `out` (in == out allowed).  Single pass, decoupled look-back; no
 * allocation, no device synchronisation. */
DSS_API int dss_exclusive_scan_i32(dss_ctx *ctx, const int32_t *in, int32_t *out, int64_t n, void *stream);

/* ---- 2-D radius binning (uniform grid) ----------------------------------------------------
 * Replace frnn._C.insert_points_cuda / counting_sort_cuda for D = 2
 * (external/FRNN/frnn/csrc/grid/grid.h:43-50, grid.cu:62-99,144-200;
 *  counting_sort.h:4-11, counting_sort.cu:5-36,72-135).
 * points (N,Pmax,2) f32 padded; lengths (N,) i64; params (N,6) f32 = min_x,min_y,1/cell,res_x,res_y,total;
 * grid_cnt (N,G) i32 must be zero on entry; grid_cell, grid_idx (N,Pmax) i32. */
DSS_API int dss_grid_insert_points_2d(dss_ctx *ctx, const float *points, const int64_t *lengths,
                              const float *params, int32_t *grid_cnt, int32_t *grid_cell,
                              int32_t *grid_idx, int N, int Pmax, int G, void *stream);
DSS_API int dss_grid_counting_sort_2d(dss_ctx *ctx, const float *points, const int64_t *lengths,
                              const int32_t *grid_cell, const int32_t *grid_idx,
                              const int32_t *grid_off, float *sorted_points, int32_t *sorted_idx,
                              int N, int Pmax, int G, void *stream);

/* ---- coarse rasterization (screen-tile binning) -------------------------------------------
 * Replaces _C._rasterize_coarse(points, radii, first_idx, num, image_size, bin_size, M)
 * (DSS/csrc/ext.cpp:11; rasterize_points.h:167-203; rasterize_points.cu:293-500).
 * The reference returns a dense (N,B,B,M) int32 tensor (M = max(1e4,P): 8 GB at 1M points); this
 * returns the same bin membership as CSR: bin_offsets (N*B*B + 1) int32 exclusive offsets and
 * bin_ids, the packed point ids of every bin (order inside a bin unspecified, as in the reference).
 * B = 1 + (S-1)/bin_size; bin (by,bx) of view n is entry (n*B + by)*B + bx, in NDC-index space like
 * the reference.  The overlap predicate is the reference's closed fp32 test (rasterize_points.cu:355-383)
 * evaluated with the identical expression sequence, so membership is bit-exact.
 * If the total exceeds bin_ids_capacity nothing is written to bin_ids, *total_required_host receives
 * the needed size and DSS_E_CAPACITY is returned (call again).  Synchronises the stream once (the
 * total is read back to size the id list, like the reference's host-side `at::full`). */
DSS_API int dss_rasterize_coarse(dss_ctx *ctx, const float *points, const float *radii,
                         const int64_t *first_idx, const int64_t *num_points, int N, int64_t P,
                         int image_size, int bin_size, int32_t *bin_offsets, int32_t *bin_ids,
                         int64_t bin_ids_capacity, int64_t *total_required_host, void *stream);

/* ---- forward rasterization ----------------------------------------------------------------
 * Replaces _C.splat_points(points, ellipse_params, cutoff_thres, radii, first_idx, num_points,
 *                          depth_merging_thres, image_size, points_per_pixel, bin_size, max_points_per_bin)
 * (DSS/csrc/ext.cpp:8; rasterize_points.h:461-525 -> RasterizePointsCoarse + RasterizePointsFine,
 *  rasterize_points.cu:293-432,506-597; CheckPixelInsidePoint :64-124).
 * Per pixel: among points of the view with z >= 0, |dx| <= rx, |dy| <= ry and
 * q = a dx^2 + b dx dy + c dy^2 <= cutoff, keep the K with smallest (z, id), ascending; emit while
 * z_k - z_0 <= depth_merging_thres.  `bin_size` is accepted for signature parity and ignored (tiling
 * is internal); max_points_per_bin does not exist here (lists are exact-size CSR).
 * zbuf / qvalue may be NULL (not written).  All outputs are fully written (no pre-fill needed). */
DSS_API int dss_splat_points(dss_ctx *ctx, const float *points, const float *ellipse_params,
                     const float *cutoff_thres, const float *radii, const int64_t *first_idx,
                     const int64_t *num_points, int N, int64_t P, float depth_merging_thres,
                     int image_size, int points_per_pixel, int bin_size, int32_t *idx, float *zbuf,
                     float *qvalue, float *occupancy, void *stream);

/* ---- backward: visibility, search radius, occupancy / z / colour gradients ------------------ */

/* visible[p] = 1 iff p appears in idx at a pixel whose idx[...,0] >= 0
 * (DSS/core/rasterizer.py:854-860; DSS/utils/__init__.py:320-340 -- replaces two torch.unique calls). */
DSS_API int dss_visibility_from_idx(dss_ctx *ctx, const int32_t *idx, int64_t num_pixels, int K, int64_t P,
                            uint8_t *visible, void *stream);

/* rs[n] = radii_s * lower_median(flattened (rx,ry) of the view's visible points); 0 if none
 * (DSS/core/rasterizer.py:888 -- replaces a per-view host loop with .item() syncs).  Exact radix select. */
DSS_API int dss_search_radius(dss_ctx *ctx, const float *radii, const uint8_t *visible,
                      const int64_t *first_idx, const int64_t *num_points, int N, int64_t P,
                      float radii_s, float *rs, void *stream);

/* Occupancy ("fast") backward.  Replaces the whole fast branch of EllipticalRasterizer.backward
 * (DSS/core/rasterizer.py:845-972): visibility compaction, FRNN grid build, per-view prefix sums,
 * counting sort, _C._splat_points_occ_fast_cuda_backward (rasterize_points_backward.cu:30-212,227-322)
 * and the un-sort / scatter, by one gather kernel: for every visible point of view n,
 *   grad_xy[p] = sum over pixels with g != 0, d2 <= rs[n]^2, not (g > 0 and outside bbox)
 *                of (dx,dy) / eps_denom(d2,1e-10) * g .
 * grad_occ is read as grad_occ[(n*S*S + r*S + c) * pix_stride + pix_offset] so that either a dense
 * (N,S,S) map (stride 1, offset 0) or the alpha channel of an (N,S,S,4) image gradient (4, 3) can be
 * passed.  grad_xy: (P,2), fully written (zeros for invisible points).  Deterministic (no atomics). */
DSS_API int dss_occ_backward(dss_ctx *ctx, const float *points, const float *radii, const uint8_t *visible,
                     const float *rs, const float *grad_occ, int pix_stride, int pix_offset,
                     const int64_t *first_idx, const int64_t *num_points, int N, int64_t P,
                     int image_size, float *grad_xy, void *stream);

/* The reference's "slow" occupancy backward, _C._splat_points_occ_backward (DSS/csrc/ext.cpp:10,16;
 * rasterize_points.cu:673-821) -- disabled in the reference by backward_occ_fast = True (rasterizer.py:816), provided
 * for completeness: every renderable point (z >= 0, |x|,|y| <= 1) of view n gathers
 *   grad_xy[p] = sum over pixels with g != 0, |dx| <= rx*s, |dy| <= ry*s, not (g > 0 and outside the splat's bbox)
 *                of (dx,dy) / eps_denom(dx^2 + dy^2, 1e-10) * g .
 * grad_occ addressing as in dss_occ_backward.  grad_xy (P,2) fully written.  Deterministic (gather, no atomics). */
DSS_API int dss_occ_backward_slow(dss_ctx *ctx, const float *points, const float *radii, const float *grad_occ,
                                  int pix_stride, int pix_offset, const int64_t *first_idx, const int64_t *num_points,
                                  int N, int64_t P, int image_size, float radii_s, float *grad_xy, void *stream);

/* z_grad[idx_k] += grad_zbuf_k until the first idx < 0.  Replaces _C._backward_zbuf
 * (DSS/csrc/ext.cpp:17; rasterize_points.h:388-419; rasterize_points.cu:823-885).  z_grad (P,) in-place. */
DSS_API int dss_zbuf_backward(dss_ctx *ctx, const int32_t *idx, const float *grad_zbuf, int64_t num_pixels,
                      int K, float *z_grad, void *stream);

/* ---- splat-size K-NN (SURVEY.md section 8(f) row 1) -------------------------------------------
 * Replaces frnn.frnn_grid_points(points1, points2, lengths1, lengths2, K, r) (external/FRNN/frnn/frnn.py:15-175;
 * grid.cu:62-99,285-373; counting_sort.cu:5-36), called by DSS with K = 7, r = 0.2 on the world-space cloud to size the
 * splats (DSS/core/rasterizer.py:313-326, 369-388).  For every query of cloud n: the K points of cloud n with the
 * smallest (squared distance, index), squared distance < r^2 (r <= 0: no limit), ascending; missing entries are -1.
 * Semantics and tie rule of the reference's ground truth FRNNBruteForceCPU (bruteforce_cpu.cpp:8-64).
 * Packed layout: cloud n owns rows [first_idx[n], first_idx[n] + num_points[n]) and the clouds are contiguous
 * (first_idx[n] = sum of the earlier num_points); idxs are local to the cloud.  queries == NULL (or == points): the
 * cloud is searched against itself (the self match, distance 0, is returned first, as in the reference).
 * sq_dists (Pq,K) f32, idxs (Pq,K) i32 or NULL.  1 <= K <= 32.  No host synchronisation. */
DSS_API int dss_knn_points(dss_ctx *ctx, const float *queries, const int64_t *query_first_idx,
                           const int64_t *query_num, const float *points, const int64_t *first_idx,
                           const int64_t *num_points, int N, int64_t Pq, int64_t P, int K, float radius,
                           float *sq_dists, int32_t *idxs, void *stream);

/* ---- fused renderer path (what bench.py times) ----------------------------------------------
 * One call per direction for SurfaceSplattingRenderer.forward / its autograd backward
 * (DSS/core/renderer.py:36-82, DSS/core/rasterizer.py:584-664,749-977).  All pointers device. */
typedef struct dss_render_args {
    /* geometry: `shared_cloud` != 0 -> points/normals are (P0,3), every view renders the same P0 points
     * (the `extend`ed cloud of rasterizer.py:236-240) and first_idx/num_points are ignored;
     * otherwise packed (P,3) with first_idx/num_points as above. */
    const float *points_world;     /* (P0,3) or (P,3)                                            */
    const float *normals_world;    /* same shape, unit length                                    */
    const float *colours;          /* (P,3) per (view,point) features, e.g. shaded rgb; (P0,3) if shared_colours */
    const float *proj;             /* (N,4,4) full projection, row-vector convention [x y z 1] M  */
    const float *view;             /* (N,4,4) world-to-view, same convention                      */
    const float *h;                /* (N,) variance scale per view, or (P,) per splat             */
    const int64_t *first_idx;      /* (N,) or NULL when shared_cloud                              */
    const int64_t *num_points;     /* (N,) or NULL when shared_cloud                              */
    int32_t n_views;
    int32_t shared_cloud;
    int64_t P0;                    /* points per view when shared_cloud, else max points per view */
    int64_t P;                     /* packed total (n_views * P0 when shared_cloud)               */
    int32_t h_per_splat;
    int32_t image_size;            /* S                                                           */
    int32_t points_per_pixel;      /* K                                                           */
    int32_t backface_culling;      /* rasterizer.py:148-181                                       */
    float cutoff_threshold;        /* C   (rasterizer.py:522)                                     */
    float depth_merging_threshold;
    float antialiasing_sigma;
    float znear, zfar;             /* depth filter (rasterizer.py:183-217)                        */
    float radii_backward_scaler;   /* radii_s                                                     */
    float clip_pts_grad;           /* <= 0: no clipping (rasterizer.py:667-673,735-736)           */
    /* forward outputs / backward inputs, all caller-allocated */
    float *records;                /* (P,8) packed splat records {x,y,z,rx, ry,a,b,c}: written by the
                                      forward pass, read by the backward pass; 16-byte aligned.  May
                                      be NULL (scratch is used; backward then rebuilds from ndc/radii) */
    float *ndc;                    /* (P,3) x,y NDC, z view depth; z = -1 for filtered points; may be NULL */
    float *ellipse;                /* (P,3) a,b,c; may be NULL                                     */
    float *radii;                  /* (P,2); may be NULL                                           */
    float *scaler;                 /* (P,)                                                         */
    float *image;                  /* (N,S,S,4) rgb + occupancy                                   */
    int32_t *idx;                  /* (N,S,S,K)                                                    */
    float *weights;                /* (N,S,S,K) normalised blend weights w_k / max(sum w, 1e-4)    */
    float *zbuf;                   /* (N,S,S,K) or NULL                                            */
    float *qvalue;                 /* (N,S,S,K) or NULL                                            */
    uint8_t *visible;              /* (P,)                                                         */
    /* backward */
    const float *grad_image;       /* (N,S,S,4)                                                    */
    const float *grad_zbuf;        /* (N,S,S,K) or NULL                                            */
    float *grad_colours;           /* (P,3), or (P0,3) if shared_colours                           */
    float *grad_ndc;               /* (P,3) gradient w.r.t. ndc (after clipping)                   */
    float *grad_points_world;      /* (P0,3) summed over views when shared_cloud, else (P,3)       */
    float *search_radius;          /* (N,) out                                                     */
    /* != 0 (shared_cloud only): `colours` is (P0,3), one feature row per POINT used by every view (view-independent
     * colour, the common host-side input: the reference only materialises the (N*P0,3) tensor on the device, after
     * shading) and `grad_colours` is (P0,3), summed over the views. */
    int32_t shared_colours;
    /* ---- per-point shading fused into the path (SURVEY.md 8(f)3; DSS/core/texture.py:74-127, lighting.py:10-172) ----
     * shade != 0 (shared_cloud only): the per-(view,point) colours are COMPUTED instead of read from `colours`:
     *   shaded = albedo * (ambient + sum_l Cd_l relu(n.d_l)) + sum_l Cs_l (relu(v.r_l) [n.d_l > 0])^shininess,
     *   n = normalize(normal), d_l = normalize(direction_l) or normalize(location_l - p), v = normalize(cam - p),
     *   r_l = -d_l + 2 (n.d_l) n          (all normalisations as F.normalize(eps = 1e-6))
     * in the preprocess kernel (forward), and the backward turns the colour gradient into gradients w.r.t. the albedo,
     * the NORMALS and (view direction, point lights) the positions -- what torch autograd does in the reference after
     * ~40 ATen kernels on (N*P0,3) tensors. */
    int32_t shade;
    int32_t n_lights;              /* L, 1 .. DSS_MAX_LIGHTS                                       */
    int32_t light_type;            /* 0: directional (rows of `lights` start with a direction), 1: point (a location) */
    float shininess;               /* specular exponent (texture.py:76: 64)                        */
    int32_t reserved0;
    const float *albedo;           /* (P0,3) per-point rgb                                         */
    const float *lights;           /* (L,9) {direction | location, diffuse rgb, specular rgb}      */
    const float *ambient;          /* (3,) ambient colour (summed over the lights' ambient terms)  */
    const float *cam_centres;      /* (N,3) camera centres in world space                          */
    float *shaded;                 /* (P,3) shaded colours: written by the forward, the blend reads them */
    /* backward (shade): `grad_colours` is then a (P,3) SCRATCH that receives d L / d shaded; outputs: */
    float *grad_albedo;            /* (P0,3) summed over views                                     */
    float *grad_normals_world;     /* (P0,3) summed over views                                     */
    float *grad_points_shading;    /* (P0,3) position gradient through the shading; dss_render_backward adds it to
                                      grad_points_world when it ran the colour half itself (grad_colours != NULL) */
    /* optional (n_views * OB * OB * 1024,) int32, OB = ceil(S / 32): written by the forward (one count per visible splat in
     * the cell -- pixel of a 32x32 tile -- of its centre; `visible` must then be 4-byte aligned with its capacity rounded
     * up to a multiple of 4), read by the backward, whose binning then skips its counting pass over all P splats.  Give
     * the same tensor to both calls or NULL to both. */
    int32_t *cell_counts;
} dss_render_args;
#define DSS_MAX_LIGHTS 8

/* preprocess -> bin -> rasterize + blend.  Never waits for the device in steady state: the tile-list buffer is sized
 * from the total the PREVIOUS call published; tiles whose list has outgrown it are rasterized from the records on the
 * device (see DESIGN.md "Host side").  Only a context's first call synchronises once to size the buffer. */
DSS_API int dss_render_forward(dss_ctx *ctx, const dss_render_args *args, void *stream);
/* visibility/median radius -> occupancy gather -> colour scatter -> z scatter -> clip -> world chain.
 * grad_colours == NULL skips the colour scatter (see dss_colour_backward). */
DSS_API int dss_render_backward(dss_ctx *ctx, const dss_render_args *args, void *stream);
/* The colour half of the backward alone (norm_weighted_sum backward: grad_colours[idx_k] += g_rgb * w_k), on `stream`.
 * Lets a data-parallel caller start the all-reduce of the colour gradients while dss_render_backward (called with
 * grad_colours == NULL on another stream) is still busy with the occupancy path (dss_b200/parallel.py). */
DSS_API int dss_colour_backward(dss_ctx *ctx, const dss_render_args *args, void *stream);
/* per-(point,view) preprocess only (rasterizer.py:443-565 fused): writes ndc, ellipse, radii, scaler. */
DSS_API int dss_preprocess(dss_ctx *ctx, const dss_render_args *args, void *stream);

/* ---- image objective of a training step (SURVEY.md section 8(f) row 5) ------------------------------
 * Trainer.calc_dr_loss (DSS/training/trainer.py:332-376) with its L1Loss and IouLoss (DSS/training/losses.py:130-137,
 * 498-514), fused and without a host read-back.  With m the GT mask, alpha the rendered occupancy, d = pred - GT per
 * rgb channel and sel = (m != 0) & (alpha != 0):
 *   M      = number of sel pixels over all views
 *   L_rgb  = (1/M) sum_sel sum_c |d_c|, 0 when M == 0
 *   L_mask = mean |m - alpha| over all N*S*S pixels
 *   L_iou  = mean_n (1 - I_n / eps_denom(U_n)),  I_n = sum m alpha,  U_n = sum (m + alpha - m alpha)  (pixels of view n)
 *   L_sil  = iou_weight * L_iou + L_mask
 *   L      = lambda_rgb * L_rgb + lambda_silhouette * L_sil
 * The forward writes terms = {L, L_rgb, L_sil, L_iou} and the per-view sums the backward needs; the backward writes
 * d L / d image as torch autograd gives it for the reference expression (|x|' = 0 at 0, no gradient through U_n where
 * eps_denom clamps it).  Block partials are combined in a fixed order in fp64: bit-reproducible, no atomics, no
 * allocation, no synchronisation (capturable in a CUDA graph). */
#define DSS_DR_LOSS_BLOCKS_PER_VIEW 128
#define DSS_DR_LOSS_NUM_SUMS 5
typedef struct dss_dr_loss_args {
    const float *image;            /* (N,S,S,4) rendered rgb + occupancy alpha, 16-byte aligned                 */
    const float *img;              /* (N,3,S,S) GT colour planes (the data batch's layout: no permute needed)   */
    const float *mask;             /* (N,S,S) GT mask (an (N,1,S,S) tensor has the same layout)                 */
    int32_t n_views;               /* N                                                                         */
    int32_t image_size;            /* S                                                                         */
    float lambda_rgb;
    float lambda_silhouette;
    float iou_weight;              /* 0.01 in the reference (trainer.py:368)                                    */
    int32_t reserved0;
    double *partials;              /* scratch, N * DSS_DR_LOSS_BLOCKS_PER_VIEW * DSS_DR_LOSS_NUM_SUMS doubles      */
    double *sums;                  /* (N+1, DSS_DR_LOSS_NUM_SUMS): row n {M_n, sum |d|, sum |m - alpha|, I_n, U_n} of
                                      view n, row N the totals; written by the forward, read by the backward      */
    float *terms;                  /* (4,) forward output {L, L_rgb, L_sil, L_iou}                               */
    const float *grad_loss;        /* backward: d (objective) / d L, one float in device memory                 */
    float *grad_image;             /* backward output (N,S,S,4), fully written, 16-byte aligned                 */
} dss_dr_loss_args;

DSS_API int dss_dr_loss_forward(dss_ctx *ctx, const dss_dr_loss_args *args, void *stream);
DSS_API int dss_dr_loss_backward(dss_ctx *ctx, const dss_dr_loss_args *args, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DSS_B200_H */
