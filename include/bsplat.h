/*
 * bsplat.h -- C ABI of libbsplat.so, the B200 (sm_100a) backend of the MojoSplat forward path.
 *
 * Plain C: raw device pointers, sizes as runtime integers, a cudaStream_t passed as void*.
 * No torch / C++ types cross this boundary, nothing is allocated inside (the caller owns every
 * buffer and passes workspace), no global mutable state: calls are re-entrant and thread-safe,
 * one stream per call.  Every entry point returns 0 (BSPLAT_OK) or a negative bsplat error /
 * a positive cudaError_t; bsplat_error_string() explains either.
 *
 * Each entry point replaces one reference interface (paths relative to the reference checkout):
 *
 *   bsplat_project_fwd        mojosplat/projection.py:15-48 project_gaussians
 *                             (= MAX op `project_gaussians`, kernels/projection.mojo:260-328,
 *                              destination-passing call at projection.py:438-454; gsplat
 *                              fully_fused_projection call at projection.py:381-397)
 *   bsplat_bin_count_scan     mojosplat/binning.py:139-168   (tile rects, counts, total)
 *   bsplat_bin_emit           mojosplat/binning.py:172-209   (emission loop; gsplat isect_tiles,
 *                              binning.py:73-82)
 *   bsplat_radix_sort_pairs   mojosplat/binning.py:223-231   (argsort depth + stable argsort tile)
 *   bsplat_tile_ranges        mojosplat/binning.py:252-260   (searchsorted -> tile_ranges;
 *                              gsplat isect_offset_encode, binning.py:84-100)
 *   bsplat_bin2_prepare/finish mojosplat/binning.py:108-262 as a whole (two-level sort, default path)
 *   bsplat_rasterize_fwd      mojosplat/rasterization.py:13-57 rasterize_gaussians
 *                             (= MAX op `rasterize_to_pixels_3dgs_fwd`,
 *                              kernels/rasterization.mojo:169-240, call at rasterization.py:167-183)
 *   bsplat_rasterize_fwd_train / bsplat_rasterize_bwd   no reference counterpart (the reference is
 *                             forward-only: render.py:11 @torch.no_grad, README.md:145); derivative of
 *                             kernels/rasterization.mojo:138-162, checked against torch autograd
 *   bsplat_project_bwd / bsplat_sh_bwd   no reference counterpart: backward of the projection and of the SH
 *                             colours (render_gaussians_diff), checked against torch autograd
 *   bsplat_ssim_fwd / bsplat_ssim_bwd   no reference counterpart: the photometric training loss (3DGS's SSIM and
 *                             L1 on one image pair, forward + backward), checked against torch autograd
 *   bsplat_densify_stats / _plan / _apply   no reference counterpart: adaptive density control (3DGS's gradient
 *                             statistics and densify_and_prune), checked against a torch restatement
 *   bsplat_render_fwd         mojosplat/render.py:12-103 render_gaussians (the three stages chained
 *                              on one stream with a single 16-byte read-back)
 *   bsplat_render_enqueue     same without the read-back (device-side M, two-stream overlap, graph capture)
 *   bsplat_render_fwd_host    same, host buffers in / host image out (end-to-end path)
 *
 * Array layouts are the reference's: row-major AoS, fp32 / int32, single camera per launch.
 */
#ifndef BSPLAT_H_
#define BSPLAT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSPLAT_VERSION 1

/* error codes (negative; positive values are cudaError_t) */
#define BSPLAT_OK 0
#define BSPLAT_E_ARG (-1)        /* bad argument (null pointer, negative size, unsupported tile size ...) */
#define BSPLAT_E_WORKSPACE (-2)  /* workspace too small; *needed_bytes tells how much is required */
#define BSPLAT_E_OVERFLOW (-3)   /* more than 2^30-1 intersections */
#define BSPLAT_E_NODEVICE (-4)   /* no CUDA device / wrong architecture */

/* binning / projection rule sets (SURVEY.md H1) */
#define BSPLAT_SEM_TORCH 0   /* reference torch backend: projection.py:199-283, binning.py:139-162 */
#define BSPLAT_SEM_GSPLAT 1  /* gsplat / Mojo rules: projection.mojo:59-87,213-244; isect_tiles */

/* or-ed into the `semantics` argument of the stage-level entry points */
#define BSPLAT_PROJ_ALLOW_FMA 0x100  /* bsplat_project_fwd: let the compiler contract a*b+c into FMAs (A/B build of
                                        the kernel; faster, radii may then differ from the reference by 1 for a few
                                        Gaussians per million -- the default rounds like the eager torch ops) */
#define BSPLAT_PROJ_FAST_MATH 0x200  /* bsplat_project_fwd: MUFU-based exp / reciprocal / square root and free FMA
                                        contraction (third build of the kernel).  Values within 1e-4 + 1e-4 |ref|;
                                        a radius next to an integer boundary may come out one off, so tile lists
                                        can differ from the reference's -- an option for callers that want the
                                        HBM-bound kernel, never the default */
#define BSPLAT_BIN_PACKED 0x100      /* bsplat_bin2_prepare / bsplat_bin2_finish (pass it to both): compact the
                                        Gaussians that own no tile away before the depth sort (gsplat's packed
                                        layout; identical lists) */

/* rasterizer arithmetic */
#define BSPLAT_RASTER_FAST 0      /* folded exp2 form, packed FP32 pairs, sub-tile culling (default) */
#define BSPLAT_RASTER_FAITHFUL 1  /* operation order of kernels/rasterization.mojo:138-157 */
#define BSPLAT_RASTER_FAST_NOCULL 2  /* fast arithmetic without sub-tile culling (exactness A/B) */

/* bsplat_render_fwd `flags`: low byte = rasterizer mode, plus */
#define BSPLAT_FLAG_CAMERA_INDIRECT 0x200   /* bsplat_render_enqueue: the camera pose / intrinsics are read
                                               from `cam` (pinned host memory) when the stream gets there, so a
                                               captured CUDA graph can be replayed with a new pose; width and
                                               height are still read on the host at enqueue time */
#define BSPLAT_FLAG_PACKED 0x400            /* packed (culled-compacted) layout: Gaussians without a tile leave the
                                               frame right after projection (one stable compaction), so the depth
                                               sort, count + scan and the raster records only see the visible ones
                                               (projection.mojo:73-87,213-244; gsplat packed=True).  Same image and
                                               lists.  A no-op under BSPLAT_SEM_TORCH, where every Gaussian owns a tile */
#define BSPLAT_FLAG_NO_BAND_PRETEST 0x1000  /* row-band frames: project every Gaussian instead of only those a
                                             * conservative pre-test cannot rule out of the band (A/B and tests:
                                             * both ways give bit-identical lists and images) */

/* Pinhole camera, world->camera. Mirrors mojosplat/utils.py:5-31 (Camera.view_matrix, Ks, H, W,
 * near, far) as a POD. viewmat is row-major 4x4. */
typedef struct bsplat_camera {
    float viewmat[16];
    float fx, fy, cx, cy;
    int32_t width, height;
    float near_plane, far_plane;
} bsplat_camera;

/* Device-side summary written by bsplat_bin_count_scan (32 bytes). */
typedef struct bsplat_bin_info {
    uint64_t n_isect;        /* M: number of (gaussian, tile) intersections */
    uint32_t min_depth_key;  /* min / max monotone depth key over Gaussians with >= 1 tile */
    uint32_t max_depth_key;
    uint32_t reserved[4];    /* [0]: scratch; [1]: 1 = M exceeded the capacity of a sync-free frame (bsplat_render_enqueue) */
} bsplat_bin_info;

/* Key layout chosen on the host from a bsplat_bin_info. */
typedef struct bsplat_key_layout {
    uint32_t depth_bias;  /* subtracted from every depth key (= min_depth_key) */
    int32_t depth_bits;   /* live depth bits after the bias */
    int32_t tile_bits;    /* ceil(log2(n_tiles)) */
} bsplat_key_layout;

int bsplat_version(void);
const char* bsplat_error_string(int code);
/* 0 when device `device` (or the current one if < 0) is an sm_100 part. */
int bsplat_check_device(int device);

/* ---- stage 1: projection ------------------------------------------------------------------- */
/* Projects N Gaussians through n_cams cameras; outputs are [n_cams, N, ...] contiguous.
 * opacities may be NULL for BSPLAT_SEM_TORCH (the torch backend ignores them). */
int bsplat_project_fwd(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                       const float* opacities, const bsplat_camera* cams_host, int32_t n_cams,
                       float eps2d, int32_t semantics, float* means2d, float* conics, float* depths,
                       int32_t* radii, void* stream);
/* Backward of bsplat_project_fwd for one camera (same eps2d and rule set, no option bits): given the gradients of
 * the forward's outputs, WRITES (does not accumulate) d loss / d means3d [N,3], d / d log_scales [N,3] and
 * d / d quats [N,4]; the quaternion gradient is taken with respect to the raw quaternion, through the forward's
 * normalisation q / max(|q|, 1e-12).  radii is the forward's output: rows with radii == (0, 0) were culled and get
 * exact zeros (the rasterizer never gives them a gradient; a row behind the camera has infinite intermediates, and
 * 0 * inf would otherwise turn into NaN).  Clamps follow torch.clamp: the gradient passes through the x/z, y/z clamp of
 * the Jacobian inside [-lim_neg, lim_pos], bounds included; under BSPLAT_SEM_TORCH no gradient flows through det
 * where it is clamped at 1e-10.  Opacity only decides the BSPLAT_SEM_GSPLAT radius and cull: no gradient.
 * v_depths may be NULL (zero).  The forward is recomputed in fp32 from the inputs; nothing is saved by it. */
int bsplat_project_bwd(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                       const bsplat_camera* cam_host, float eps2d, int32_t semantics, const int32_t* radii,
                       const float* v_means2d, const float* v_conics, const float* v_depths, float* v_means3d,
                       float* v_log_scales, float* v_quats, void* stream);

/* ---- stage 2: binning ---------------------------------------------------------------------- */
size_t bsplat_bin_scan_workspace_bytes(int64_t N);
/* Tile rect per Gaussian -> exclusive prefix sum offsets[N+1] (uint32) and *info (device).
 * radii is int32 [N,2] (projection output) or float [N,2] when radii_is_float != 0
 * (the reference's tests pass float radii, tests/test_binning.py:23).
 * tile_row_begin/end restrict emission to a band of tile rows (row-band multi-GPU split);
 * pass 0 and tiles_h for the whole image. */
int bsplat_bin_count_scan(int64_t N, const float* means2d, const void* radii, int32_t radii_is_float,
                          const float* depths, int32_t width, int32_t height, int32_t tile_size,
                          int32_t tile_row_begin, int32_t tile_row_end, int32_t semantics,
                          uint32_t* offsets, bsplat_bin_info* info, void* workspace,
                          size_t workspace_bytes, void* stream);
/* Host helper: key layout (depth bias / live bits) from a read-back info. */
bsplat_key_layout bsplat_make_key_layout(const bsplat_bin_info* info_host, int32_t width,
                                         int32_t height, int32_t tile_size);
/* Writes keys[M] = (tile_id << depth_bits) | (depth_key - depth_bias) and gaussian ids[M] in
 * emission order (gaussian, tile row, tile column ascending). */
int bsplat_bin_emit(int64_t N, const float* means2d, const void* radii, int32_t radii_is_float,
                    const float* depths, int32_t width, int32_t height, int32_t tile_size,
                    int32_t tile_row_begin, int32_t tile_row_end, int32_t semantics,
                    const uint32_t* offsets, bsplat_key_layout layout, uint64_t* keys, int32_t* ids,
                    void* stream);
size_t bsplat_radix_sort_workspace_bytes(int64_t M, int32_t begin_bit, int32_t end_bit);
/* Stable LSD onesweep radix sort of (uint64 key, int32 value) pairs on key bits
 * [begin_bit, end_bit). Ping-pongs between the two buffer pairs; *result_in_alt tells where the
 * sorted data ended up (0: keys/vals, 1: keys_alt/vals_alt). */
int bsplat_radix_sort_pairs(int64_t M, uint64_t* keys, uint64_t* keys_alt, int32_t* vals,
                            int32_t* vals_alt, int32_t begin_bit, int32_t end_bit, void* workspace,
                            size_t workspace_bytes, int32_t* result_in_alt, void* stream);
/* tile_ranges[n_tiles, 2] int32 = [first, past-last) index of each tile in the sorted keys
 * (searchsorted-left semantics for empty tiles, binning.py:252-260). */
int bsplat_tile_ranges(int64_t M, const uint64_t* sorted_keys, int32_t tile_shift, int32_t n_tiles,
                       int32_t* tile_ranges, void* stream);

/* Two-level binning (default path; same results, ~4x less sort traffic): depth-sort the N
 * Gaussians (4 onesweep passes over uint32 depth keys), count + scan and emit in depth order, then a
 * stable sort by tile id only (ceil(log2 n_tiles) bits in ceil(bits / 8) passes over the M pairs: 2 for up to
 * 65 536 tiles, 3-4 beyond) -- the structure of the reference's argsort(depth) + stable argsort(tile)
 * (binning.py:223-231).  means2d / radii / depths are read by prepare only (finish ignores them).
 * prepare: writes M to *info_out (device); the caller reads it back, sizes sorted_ids[M] and calls
 * finish with the same workspace (>= bsplat_bin2_workspace_bytes(N, M, n_tiles)). The last sort pass
 * also yields the per-tile counts, so tile_ranges (and the rasterizer's tile_order) cost one tiny kernel. */
size_t bsplat_bin2_workspace_bytes(int64_t N, int64_t M_capacity, int64_t n_tiles);
int bsplat_bin2_prepare(int64_t N, const float* means2d, const void* radii, int32_t radii_is_float,
                        const float* depths, int32_t width, int32_t height, int32_t tile_size,
                        int32_t tile_row_begin, int32_t tile_row_end, int32_t semantics, void* workspace,
                        size_t workspace_bytes, bsplat_bin_info* info_out, void* stream);
int bsplat_bin2_finish(int64_t N, int64_t M, const float* means2d, const void* radii,
                       int32_t radii_is_float, int32_t width, int32_t height, int32_t tile_size,
                       int32_t tile_row_begin, int32_t tile_row_end, int32_t semantics, void* workspace,
                       size_t workspace_bytes, int32_t* sorted_ids, int32_t* tile_ranges,
                       int32_t* tile_order /* nullable: [tiles of the band], longest list first */,
                       void* stream);

/* ---- stage 3: rasterization ---------------------------------------------------------------- */
/* tile_order[n_tiles]: tile ids sorted by list length, longest first (scheduling hint for the
 * rasterizer: under the torch binning rules the culled Gaussians pile up in the corner tiles). */
int bsplat_tile_order(int32_t first_tile, int32_t n_tiles, const int32_t* tile_ranges,
                      int32_t* tile_order, void* stream);
/* image[height, width, channels]. opacities are used raw (no sigmoid), like the reference.
 * tile_order may be NULL (row-major tile order). Only tile rows [tile_row_begin, tile_row_end) are
 * rasterized and written (pass 0 and tiles_h for the whole frame; a row band for the multi-GPU split --
 * tile_order, if given, must then list exactly the band's tiles).
 * workspace (optional, bsplat_rasterize_workspace_bytes(N) = 48 B per Gaussian, 16-byte aligned): holds the
 * per-Gaussian raster records, written once per call; with it the fast kernel stages its batches with
 * cp.async one batch ahead (faster, identical results); without it it stages from the raw arrays.
 * mode: BSPLAT_RASTER_FAST / _FAITHFUL / _FAST_NOCULL (anything else: BSPLAT_E_ARG). */
size_t bsplat_rasterize_workspace_bytes(int64_t N);
int bsplat_rasterize_fwd(int64_t N, int32_t channels, const float* means2d, const float* conics,
                         const float* colors, const float* opacities, const float* background,
                         const int32_t* tile_ranges, const int32_t* tile_order,
                         const int32_t* sorted_ids, int64_t M, int32_t width, int32_t height,
                         int32_t tile_size, int32_t tile_row_begin, int32_t tile_row_end, int32_t mode,
                         float* image, void* workspace, size_t workspace_bytes, void* stream);

/* Faithful kernel + counters: stats[0] += evaluated (pixel, Gaussian) pairs, stats[1] += contributing
 * pairs (device uint64[2], caller-zeroed) -- the algorithmic work E_all / E_pass of SURVEY.md 8d. */
int bsplat_rasterize_stats(int64_t N, int32_t channels, const float* means2d, const float* conics,
                           const float* colors, const float* opacities, const float* background,
                           const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                           int32_t width, int32_t height, int32_t tile_size, float* image,
                           uint64_t* stats, void* stream);

/* ---- colours: spherical harmonics (SURVEY.md 8f rank 4; placeholder in the reference, render.py:82-87) -- */
/* colors[N,3] = max(sum_k Y_k(dir) coeffs[n,k,:] + 0.5, 0), dir = normalize(means3d[n] - campos), real SH of
 * `degree` (0..3), coeffs [N, K_stored, 3] with K_stored >= (degree+1)^2 (extra bands ignored).
 * campos_host: camera position in world space, 3 floats on the host. */
int bsplat_sh_eval(int64_t N, int32_t degree, int32_t K_stored, const float* coeffs, const float* means3d,
                   const float* campos_host, float* colors, void* stream);
/* Backward of bsplat_sh_eval: WRITES v_coeffs [N, K_stored, 3] (= Y_k(dir) v_colors; bands above `degree` are
 * zero) and, when v_means3d is not NULL, d loss / d means3d [N,3] through dir = normalize(means3d - campos) (zero for
 * degree 0; the camera gets no gradient).  The clamp max(r + 0.5, 0) passes the gradient like torch.clamp(min=0),
 * where r + 0.5 >= 0. */
int bsplat_sh_bwd(int64_t N, int32_t degree, int32_t K_stored, const float* coeffs, const float* means3d,
                  const float* campos_host, const float* v_colors, float* v_coeffs, float* v_means3d, void* stream);

/* ---- photometric training loss (no reference counterpart) ---------------------------------- */
/* SSIM as 3DGS defines it (11x11 Gaussian window, sigma 1.5, per channel, zero padding 5, C1 = 0.01^2, C2 = 0.03^2,
 * mean over all H*W*C values) and the L1 term mean |img - target|, for fp32 images [H, W, C] with H, W >= 1 and
 * 1 <= C <= 4 (else BSPLAT_E_ARG).  Nothing is read back to the host; both sums are deterministic (per-CTA partials
 * in the workspace, added in a fixed order).
 * fwd: writes out2 (device) = [mean SSIM, mean L1].  maps [3, H, W, C] (NULL when no gradient is wanted) receives the
 * per-pixel factors the backward convolves: dS/dmu_x - 2 mu_x dS/dsigma_x^2 - mu_y dS/dsigma_xy, dS/dsigma_x^2,
 * dS/dsigma_xy.  A workspace shorter than bsplat_ssim_workspace_bytes (8-byte aligned) is BSPLAT_E_WORKSPACE with
 * *needed_bytes (nullable) set. */
size_t bsplat_ssim_workspace_bytes(int32_t H, int32_t W, int32_t C);
int bsplat_ssim_fwd(int32_t H, int32_t W, int32_t C, const float* img, const float* target, float* out2,
                    float* maps, void* workspace, size_t workspace_bytes, size_t* needed_bytes, void* stream);
/* bwd: v_out2 (device) = [dL/d mean SSIM, dL/d mean L1]; WRITES v_img [H, W, C] = d loss / d img (maps from
 * bsplat_ssim_fwd on the same images; the L1 term's derivative is sign(img - target), 0 where they are equal). */
int bsplat_ssim_bwd(int32_t H, int32_t W, int32_t C, const float* img, const float* target, const float* maps,
                    const float* v_out2, float* v_img, void* stream);

/* ---- adaptive density control (no reference counterpart) ----------------------------------- */
/* 3DGS's densify_and_prune.  Thresholds are fp32 values the caller computes in double and rounds once; every
 * decision compares in log space (no exp).  +inf / INT32_MAX (and -inf for min_opacity) disable a prune rule. */
typedef struct bsplat_densify_params {
    float grad_threshold;       /* clone / split when count > 0 and grad2d / count >= this */
    float log_clone_max_scale;  /* log(percent_dense * scene_extent): max log-scale <= this clones, else splits */
    float min_opacity;          /* prune when opacity < this */
    float log_max_world_scale;  /* prune when the row's max log-scale > this (split children: their reduced scale) */
    int32_t max_screen_radius;  /* prune when max_radius > this */
    int32_t reserved;
} bsplat_densify_params;
/* roles of a bsplat_densify_tensor */
#define BSPLAT_DENSIFY_COPY 0        /* every output row copies its parent's row */
#define BSPLAT_DENSIFY_MEANS 1       /* [N, 3] means3d: split children mu + R(q / |q|) (exp(s) * noise[k, c]) */
#define BSPLAT_DENSIFY_LOG_SCALES 2  /* [N, 3] log-scales: split children s - (float)ln 1.6 */
#define BSPLAT_DENSIFY_STATE 3       /* optimizer state: kept rows keep theirs, clone copies and split children get 0 */
typedef struct bsplat_densify_tensor {
    const float* src;  /* [N, width] */
    float* dst;        /* [n_out, width], not src */
    int32_t width;     /* 1..256 floats per row */
    int32_t role;
} bsplat_densify_tensor;
typedef struct bsplat_densify_counts {
    int64_t n_out;     /* output rows: N + n_clone + n_split - n_pruned */
    int64_t n_clone;   /* clone decisions */
    int64_t n_split;   /* split decisions (rows of the noise tensor), pruned ones included */
    int64_t n_pruned;  /* output rows dropped by the prune rules */
} bsplat_densify_counts;

size_t bsplat_densify_workspace_bytes(int64_t N);
/* Adds one view's statistics: for every i with max(radii[i]) > 0, grad2d[i] += |(v.x W / 2, v.y H / 2)| of
 * v = v_means2d[i] (pixels), count[i] += 1, max_radius[i] = max(max_radius[i], max(radii[i])).  Other rows untouched.
 * v_means2d [N, 2] and radii [N, 2] are read as 8-byte vectors (8-byte aligned). */
int bsplat_densify_stats(int64_t N, const float* v_means2d, const int32_t* radii, int32_t width, int32_t height,
                         float* grad2d, int32_t* count, int32_t* max_radius, void* stream);
/* Decides every Gaussian (keep / clone / split, then prune) into the workspace (16-byte aligned, at least
 * bsplat_densify_workspace_bytes(N), else BSPLAT_E_WORKSPACE with *needed_bytes set) and stores the totals into
 * counts_host, a host-visible block the device writes directly: valid once the stream has reached this point. */
int bsplat_densify_plan(int64_t N, const float* grad2d, const int32_t* count, const int32_t* max_radius,
                        const float* log_scales, const float* opacities, const bsplat_densify_params* params,
                        void* workspace, size_t workspace_bytes, size_t* needed_bytes,
                        bsplat_densify_counts* counts_host, void* stream);
/* Writes the n_out rows of every tensor from the plan in the same workspace, in one launch.  Each parent is replaced
 * in place, in index order, by its surviving rows: kept (itself), clone (itself, then a copy), split (two children);
 * child c of the k-th split parent in index order uses noise[k, c, 0..2] ([n_split, 2, 3]; NULL when n_split = 0).  1 to 32
 * tensors, exactly one MEANS (src == means3d) and one LOG_SCALES (src == log_scales) among them; quats [N, 4]. */
int bsplat_densify_apply(int64_t N, const void* workspace, const float* means3d, const float* log_scales,
                         const float* quats, const float* noise, int32_t n_tensors,
                         const bsplat_densify_tensor* tensors, void* stream);

/* ---- stage 3, training side (SURVEY.md 8f rank 1; the reference is forward-only, render.py:11) --------- */
/* Forward with the faithful arithmetic (kernels/rasterization.mojo:138-162) that also stores what the
 * backward pass needs: final_T[height, width] (transmittance left at each pixel) and
 * last_idx[height, width] (index INTO sorted_ids of the last Gaussian composited there, -1 if none).
 * channels in 1..4; any tile size <= 32. */
int bsplat_rasterize_fwd_train(int64_t N, int32_t channels, const float* means2d, const float* conics,
                               const float* colors, const float* opacities, const float* background,
                               const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                               int32_t width, int32_t height, int32_t tile_size, float* image,
                               float* final_T, int32_t* last_idx, void* stream);
/* The same through the fast forward kernel (16x16 tiles, RGB): image bit-identical to bsplat_rasterize_fwd's default
 * mode (within 1e-4 of the faithful arithmetic, like every fast frame); last_idx holds the last list entry the
 * backward pass has to look at (the entry in front of the one that saturated the pixel, or the end of the tile's
 * list). tile_order (optional, bsplat_tile_order): heavy tiles first. workspace (optional,
 * bsplat_rasterize_workspace_bytes(N)): per-Gaussian records + cp.async staging. */
int bsplat_rasterize_fwd_train_fast(int64_t N, const float* means2d, const float* conics, const float* colors,
                                    const float* opacities, const float* background, const int32_t* tile_ranges,
                                    const int32_t* tile_order, const int32_t* sorted_ids, int64_t M, int32_t width,
                                    int32_t height, float* image, float* final_T, int32_t* last_idx,
                                    void* workspace, size_t workspace_bytes, void* stream);
/* Backward of the compositing: ACCUMULATES d loss / d (means2d[N,2], conics[N,3], colors[N,C],
 * opacities[N]) into the caller-zeroed gradient arrays, given grad_image[height, width, C] and the
 * final_T / last_idx of bsplat_rasterize_fwd_train[_fast] on the same inputs. Threshold tests are piecewise
 * constant; no gradient flows through the 0.999 alpha clamp. (d loss / d background =
 * sum_pixels final_T * grad_image is left to the caller.) */
int bsplat_rasterize_bwd(int64_t N, int32_t channels, const float* means2d, const float* conics,
                         const float* colors, const float* opacities, const float* background,
                         const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                         int32_t width, int32_t height, int32_t tile_size, const float* final_T,
                         const int32_t* last_idx, const float* grad_image, float* grad_means2d,
                         float* grad_conics, float* grad_colors, float* grad_opacities, void* stream);

/* ---- fused forward ------------------------------------------------------------------------- */
/* Optional outputs of the fused path (any pointer may be NULL). */
typedef struct bsplat_render_aux {
    float* means2d;        /* [N,2] */
    float* conics;         /* [N,3] */
    float* depths;         /* [N]   */
    int32_t* radii;        /* [N,2] */
    int32_t* tile_ranges;  /* [tiles_h, tiles_w, 2] */
    int32_t* sorted_ids;   /* [sorted_ids_capacity]; filled when M <= capacity */
    int64_t sorted_ids_capacity;
    int64_t n_isect;       /* out: M */
    int32_t timing;        /* in: record per-stage CUDA-event times (adds a final sync) */
    int32_t n_launches;    /* out: kernels launched by this call */
    int32_t sort_passes;   /* out: onesweep passes (= ceil(live key bits / 8)) */
    int32_t key_bits;      /* out: live key bits (depth_bits + tile_bits) */
    float stage_ms[4];     /* out when timing != 0: projection, count+scan+emit, sort+ranges, raster */
} bsplat_render_aux;

size_t bsplat_render_workspace_bytes(int64_t N, int64_t M_capacity, int32_t width, int32_t height,
                                     int32_t tile_size);
/* render.py:63-101 on one stream. Returns BSPLAT_E_WORKSPACE and sets *needed_bytes when the
 * workspace cannot hold the M this frame produced (call again with a larger one).
 * M == 0 gives an all-zero image (render.py:73-76), not the background. */
int bsplat_render_fwd(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                      const float* opacities, const float* colors, int32_t channels,
                      const bsplat_camera* cam_host, const float* background, int32_t tile_size,
                      int32_t semantics, int32_t flags, float* image, void* workspace,
                      size_t workspace_bytes, size_t* needed_bytes, bsplat_render_aux* aux,
                      void* stream);
/* Split-phase frame for pipelined multi-view rendering. begin: projection + depth sort + count/scan
 * and an ASYNC copy of the bin info (M) into pinned host memory -- no sync. The caller waits for the
 * stream (event), reads M, then calls end (emit + tile sort + ranges + raster) with the same workspace,
 * which must hold bsplat_render_workspace_bytes(N, M, ...). Two streams with one workspace each overlap
 * begin(k+1) with end(k). */
int bsplat_render_begin(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                        const float* opacities, const bsplat_camera* cam_host, int32_t tile_size,
                        int32_t semantics, void* workspace, size_t workspace_bytes,
                        bsplat_bin_info* info_host_pinned, void* stream);
int bsplat_render_end(int64_t N, int64_t M, const float* colors, const float* opacities, int32_t channels,
                      const bsplat_camera* cam_host, const float* background, int32_t tile_size,
                      int32_t semantics, int32_t flags, float* image, void* workspace,
                      size_t workspace_bytes, size_t* needed_bytes, void* stream);
/* Sync-free frame (render.py:63-101 without the M read-back): nothing in this call waits for the GPU.
 * The workspace is sized for M_capacity pairs; the real M stays on the device. If a frame produces more
 * pairs than that, info.reserved[1] is set and the image is invalid: the caller inspects
 * *info_host_pinned (copied asynchronously on stream_bin; nullable) after synchronising and re-renders
 * with a larger capacity. stream_raster may be NULL / equal to stream_bin (single stream) or a second,
 * lower-priority stream: event_bin_done (a cudaEvent_t) then orders rasterization behind binning, and
 * binning of the next frame overlaps rasterization of this one. Safe to capture into a CUDA graph. */
int bsplat_render_enqueue(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                          const float* opacities, const float* colors, int32_t channels,
                          const bsplat_camera* cam, const float* background, int32_t tile_size,
                          int32_t semantics, int32_t flags, float* image, void* workspace,
                          size_t workspace_bytes, int64_t M_capacity, size_t* needed_bytes,
                          bsplat_bin_info* info_host_pinned, void* stream_bin, void* stream_raster,
                          void* event_bin_done);
/* The sync-free frame restricted to tile rows [tile_row_begin, tile_row_end) (row-band multi-GPU split):
 * all N Gaussians are projected, only the band is binned / rasterized / written into `image`. */
int bsplat_render_enqueue_band(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                               const float* opacities, const float* colors, int32_t channels,
                               const bsplat_camera* cam, const float* background, int32_t tile_size,
                               int32_t semantics, int32_t flags, int32_t tile_row_begin, int32_t tile_row_end,
                               float* image, void* workspace, size_t workspace_bytes, int64_t M_capacity,
                               size_t* needed_bytes, bsplat_bin_info* info_host_pinned, void* stream_bin,
                               void* stream_raster, void* event_bin_done);
/* ... with the band exchange fused into the rasterizer: every finished tile is also stored (128-bit stores)
 * into the image buffers of the n_peers (<= 7) other ranks -- peer-mapped device pointers of the same layout,
 * e.g. torch symmetric memory over NVLink / NVSwitch. Follow with a cross-device barrier on the stream; no
 * all-gather is needed. 16x16 tiles, RGB, BSPLAT_RASTER_FAST only. */
int bsplat_render_enqueue_band_p2p(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                                   const float* opacities, const float* colors, int32_t channels,
                                   const bsplat_camera* cam, const float* background, int32_t tile_size,
                                   int32_t semantics, int32_t flags, int32_t tile_row_begin,
                                   int32_t tile_row_end, float* image, float* const* peer_images,
                                   int32_t n_peers, void* workspace, size_t workspace_bytes,
                                   int64_t M_capacity, size_t* needed_bytes, bsplat_bin_info* info_host_pinned,
                                   void* stream_bin, void* stream_raster, void* event_bin_done);
/* Same with HOST buffers (pinned or pageable): copies the Gaussians in, renders, copies the
 * image out and synchronises the stream. device_scratch must hold
 * bsplat_render_host_scratch_bytes() in addition to the render workspace (a shorter one is BSPLAT_E_ARG;
 * BSPLAT_E_WORKSPACE / *needed_bytes always refer to `workspace`). */
size_t bsplat_render_host_scratch_bytes(int64_t N, int32_t channels, int32_t width, int32_t height);
int bsplat_render_fwd_host(int64_t N, const float* means3d, const float* log_scales,
                           const float* quats, const float* opacities, const float* colors,
                           int32_t channels, const bsplat_camera* cam_host, const float* background,
                           int32_t tile_size, int32_t semantics, int32_t flags,
                           float* image_host, void* device_scratch, size_t scratch_bytes,
                           void* workspace, size_t workspace_bytes, size_t* needed_bytes,
                           bsplat_render_aux* aux, void* stream);

/* ---- measurement helper (not on the product path) ------------------------------------------ */
/* Issue-rate micro-benchmark: kind 0 = FP32 FFMA chains, kind 1 = MUFU.EX2 chains; blocks x 256
 * threads x 8 x iters operations. Timed by the caller with CUDA events; gives the measured
 * FP32 / SFU denominators of the rasterizer roofline. */
int bsplat_microbench(int32_t kind, int32_t blocks, int32_t iters, float* out, void* stream);

/* The backward pass in the fast kernel's layout (16x16 tiles, RGB; two pixels per lane, packed FP32, MUFU ex2 / rcp):
 * same contract as bsplat_rasterize_bwd; gradients agree with it within float rounding (both are checked against
 * fp64 autograd at 1e-3). workspace: bsplat_rasterize_workspace_bytes(N), 16-byte aligned (the records are rebuilt
 * here); tile_order optional (bsplat_tile_order). */
int bsplat_rasterize_bwd_fast(int64_t N, const float* means2d, const float* conics, const float* colors,
                              const float* opacities, const float* background, const int32_t* tile_ranges,
                              const int32_t* tile_order, const int32_t* sorted_ids, int64_t M, int32_t width,
                              int32_t height, const float* final_T, const int32_t* last_idx,
                              const float* grad_image, float* grad_means2d, float* grad_conics, float* grad_colors,
                              float* grad_opacities, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BSPLAT_H_ */
