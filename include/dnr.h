/*
 * dnr.h — C ABI of libdnr_b200.so: the B200 (sm_100a) depth+normal Gaussian rasterizer that
 * replaces the two gsplat calls (and the torch glue between them) inside
 * DNSplatterModel.get_outputs of maturk/dn-splatter.
 *
 * Reference interfaces replaced (paths relative to /root/reference/):
 *   dnr_project_fwd    gsplat fully_fused_projection + spherical_harmonics + param activations
 *                      (dn_splatter/dn_model.py:495-500 arguments of rasterization();
 *                      :543-560 per-Gaussian normals)
 *   dnr_bin_scan/sort  gsplat isect_tiles + radix sort + isect_offset_encode, shared by the colour and
 *                      the normal pass (dn_model.py:495-516 and the second binning hidden in :564-575)
 *   dnr_raster_fwd     gsplat rasterize_to_pixels (RGB+ED, dn_model.py:495-516) + legacy
 *                      rasterize_gaussians on normals (:564-575) + blend/clamp/normalise (:526-537,:577-578)
 *   dnr_finalize_fwd   depth fill with the global max (dn_model.py:534-537) + normal_from_depth_image
 *                      (dn_splatter/utils/normal_utils.py:25-48, called at dn_model.py:589-603)
 *   dnr_raster_bwd     autograd backward of the two rasterizations and of the glue above
 *   dnr_project_bwd    autograd backward of projection / SH / activations / normals
 *   dnr_loss_*         DNRegularization depth + normal terms (dn_splatter/regularization_strategy.py:146-193,
 *                      dn_splatter/losses.py:155-224,279-295) fused: value + per-pixel gradient
 *
 * Conventions: plain C, POD only, every pointer is a DEVICE pointer unless named *_host, row-major
 * contiguous fp32, images [H,W,C], quaternions wxyz, viewmat = world->camera (OpenCV), pixel centres
 * at +0.5, tile size 16.  The caller owns every buffer (including workspaces sized by the *_bytes
 * queries).  All work is enqueued on the stream passed in (a cudaStream_t cast to void*); the only
 * host synchronisation is the documented n_isects read-back inside dnr_bin_scan.
 * Return value: 0 = ok, <0 = DNR_E_* argument error, >0 = cudaError_t of a failed launch.
 * No global state, re-entrant, never throws, never prints.
 */
#ifndef DNR_H_
#define DNR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DNR_VERSION 100 /* 0.1.0 */

#define DNR_E_NULL (-1)     /* a required pointer is NULL */
#define DNR_E_SIZE (-2)     /* non-positive / inconsistent sizes */
#define DNR_E_OPTION (-3)   /* unsupported option (tile size, sh degree, ...) */
#define DNR_E_OVERFLOW (-4) /* more than 2^31-1 tile intersections */
#define DNR_E_WORKSPACE (-5)/* workspace too small */

/* flags */
#define DNR_FLAG_ACTIVATED 1u   /* scales/opacities are already exp()/sigmoid()-activated (gsplat's signature) */
#define DNR_FLAG_ANTIALIASED 2u /* rasterize_mode == "antialiased": opacity *= compensation */
#define DNR_FLAG_NORMALS 4u     /* predict_normals: render the per-Gaussian normal channels */
#define DNR_FLAG_ACCUMULATE 8u  /* project_bwd adds into the parameter-gradient buffers */
#define DNR_FLAG_COMPACT_BWD 64u /* project_bwd walks the depth-sorted index (validated, but slower than DNR_FLAG_TOUCHED_BWD: kept for A/B)
                                    (a->depth_order), so only visible Gaussians occupy lanes; needs DNR_FLAG_ACCUMULATE */
#define DNR_FLAG_HOST_CAMERA 32u /* camera passed by value in host_cam[] (no device reads, no H2D copy) */
#define DNR_FLAG_EXACT_LISTS 16u /* parity mode: emit gsplat's full bbox intersection lists (no precise-hit cull) */
#define DNR_FLAG_TOUCHED_BWD 128u /* project_bwd processes only Gaussians with touched[g] != 0 (needs DNR_FLAG_ACCUMULATE) */

/* floats per packed per-Gaussian raster record, without / with normals */
#define DNR_REC_FLOATS 12
#define DNR_REC_FLOATS_N 16
/* floats per per-Gaussian raster-gradient record (always) */
#define DNR_GRAD_FLOATS 16

typedef struct DnrArgs {
  /* ---- sizes and options (host scalars) ---- */
  int32_t n_gauss;   /* N */
  int32_t width, height;
  int32_t tile_size; /* must be 16 (dn_model.py:470-472) */
  int32_t sh_degree; /* active degree 0..3 (dn_model.py:487-490) */
  int32_t sh_bases;  /* bases stored per Gaussian: sh_rest is [N, sh_bases-1, 3] */
  uint32_t flags;    /* DNR_FLAG_* */
  int32_t list_shift; /* intersection lists are kept per SUPERTILE of (16 << list_shift)^2 pixels (0..3); every 16x16 tile
                         walks its supertile's list and drops, inside the raster kernels, the entries that cannot reach it.
                         0 = one list per tile (required with DNR_FLAG_EXACT_LISTS: gsplat's lists) */
  float near_plane, far_plane, eps2d, radius_clip;
  float background[3];
  float reserved1;
  int64_t n_isects; /* capacity of flatten_ids / ws_sort in intersections (>= the count dnr_bin_scan reports, or an
                       estimate when running sync-free: see n_isects_dev) */

  /* ---- camera (device) ---- */
  const float* viewmat; /* [4,4] */
  const float* K;       /* [3,3] */
  const float* c2w;     /* [3,4] nerfstudio camera_to_world (OpenGL, un-optimised); normals only */

  /* ---- Gaussian parameters (device, the reference's gauss_params layout, dn_model.py:227-237) ---- */
  const float* means;     /* [N,3] */
  const float* quats;     /* [N,4] */
  const float* scales;    /* [N,3] log-scales (or activated with DNR_FLAG_ACTIVATED) */
  const float* opacities; /* [N]   logits     (or activated) */
  const float* sh_dc;     /* [N,3] */
  const float* sh_rest;   /* [N,sh_bases-1,3] (may be NULL when sh_bases==1) */

  /* ---- projection outputs (info dict of gsplat.rasterization, dn_model.py:517-524) ---- */
  int32_t* radii;           /* [N] */
  float* means2d;           /* [N,2] */
  float* depths;            /* [N] */
  float* conics;            /* [N,3] */
  float* opac_act;          /* [N] activated (x compensation) opacity */
  float* compensations;     /* [N] or NULL */
  float* colors;            /* [N,3] clamp_min(SH+0.5,0) */
  float* normals_world;     /* [N,3] flipped world normals (gauss_params["normals"], dn_model.py:558) or NULL */
  int32_t* tiles_per_gauss; /* [N] */
  uint32_t* depth_keys;     /* [N] bit pattern of depth, 0xFFFFFFFF when culled */
  float* records;           /* [N, DNR_REC_FLOATS(_N)] packed raster records */
  float* cull_lim;          /* [N] ln(255 * sigmoid opacity) + margin: largest sigma that can still reach alpha >= 1/255 */

  /* ---- binning ---- */
  void* ws_scan;         /* dnr_bin_scan_workspace_bytes(N) */
  void* ws_sort;         /* dnr_bin_sort_workspace_bytes(N, I, n_tiles) */
  int32_t* flatten_ids;  /* [I] Gaussian ids sorted by (tile, depth, id) */
  int32_t* tile_offsets; /* [n_tiles+1] */
  int64_t* n_isects_dev; /* [1] device copy of the intersection count (may exceed the capacity: then the render is
                            truncated and the caller must retry with a larger n_isects) */

  /* ---- raster forward outputs / backward state ---- */
  float* out_rgb;      /* [H,W,3] clamp(C + (1-alpha) bg, 0, 1) */
  float* out_depth;    /* [H,W]   D/alpha, then filled by dnr_finalize_fwd */
  float* out_alpha;    /* [H,W] */
  float* out_normal;   /* [H,W,3] (n/|n|+1)/2 or NULL */
  float* out_surface_normal; /* [H,W,3] or NULL */
  int32_t* last_ids;   /* [H,W] */
  float* normal_norm;  /* [H,W] |n_raw| (backward state) or NULL */
  uint8_t* clamp_mask; /* [H,W] bit k set: rgb channel k passes gradient */
  int32_t* depth_max;  /* [1] bit pattern of max expected depth */

  /* ---- raster backward ---- */
  const float* v_rgb;    /* [H,W,3] or NULL */
  const float* v_depth;  /* [H,W]   or NULL */
  const float* v_normal; /* [H,W,3] or NULL */
  const float* v_alpha;  /* [H,W]   or NULL */
  float* grad_records;   /* [N, DNR_GRAD_FLOATS] zeroed by dnr_raster_bwd */

  /* ---- projection backward outputs ---- */
  float* v_means;       /* [N,3] */
  float* v_quats;       /* [N,4] */
  float* v_scales;      /* [N,3] */
  float* v_opacities;   /* [N] */
  float* v_sh_dc;       /* [N,3] */
  float* v_sh_rest;     /* [N,sh_bases-1,3] */
  float* v_means2d;     /* [N,2] or NULL  (info["means2d"].grad) */
  float* v_means2d_abs; /* [N,2] or NULL  (info["means2d"].absgrad) */

  /* ---- fused regularisers (DNRegularization) ---- */
  const float* gt_depth;  /* [H,W] */
  const float* gt_normal; /* [H,W,3] */
  const float* gt_rgb;    /* [H,W,3] */
  float* loss_partials;   /* [12] fp32 accumulators + results, see dnr_loss_fwd */
  const float* v_loss;    /* [1] device scalar: upstream gradient of the regulariser (NULL = 1) */
  float depth_lambda, depth_tolerance;
  int32_t depth_loss_type; /* 0 none, 1 EdgeAwareLogL1, 2 LogL1, 3 L1, 4 MSE */
  int32_t use_normal_loss;
  /* with DNR_FLAG_HOST_CAMERA: [0..15] viewmat, [16..19] fx fy cx cy, [20..31] c2w[3,4]; viewmat/K/c2w pointers unused */
  float host_cam[32];
  const int32_t* depth_order; /* [N] Gaussian ids sorted by depth, visible first (dnr_depth_order_ptr); COMPACT_BWD only */

  /* ---- loss gradients evaluated inside dnr_raster_bwd (BASELINE north_star: regularisers fused into the backward) ----
   * With DNR_LOSS_FUSED_BWD the per-pixel gradients of
   *   *v_l1  * mean|rgb - gt_image|                     (parent photometric L1; term off when v_l1 == NULL)
   *   *v_loss * DNRegularization(depth, normal)         (dnr_loss_fwd's terms; uses gt_depth, gt_normal, gt_rgb /
   *                                                      gt_image, loss_partials, depth_* fields, use_normal_loss)
   * are computed in the kernel's prologue from the rendered maps instead of being read from v_rgb / v_depth / v_normal
   * images; non-NULL v_rgb / v_depth / v_normal / v_alpha are ADDED (e.g. the SSIM gradient). */
  uint32_t loss_flags;   /* DNR_LOSS_* */
  int32_t variant;       /* kernel tuning knob (0 = default); see csrc/raster.cu */
  const void* gt_image;  /* [H,W,3] photometric target: uint8 (DNR_LOSS_IMG_U8, scaled by 1/255) or fp32 */
  const float* v_l1;     /* [1] device scalar */
  uint8_t* touched;      /* [N] or NULL: dnr_raster_bwd sets touched[g] = 1 for every Gaussian that received a gradient
                            (zeroed by the call); dnr_project_bwd then skips the others (DNR_FLAG_TOUCHED_BWD) */
  uint64_t* stats; /* [4] or NULL: += {list entries walked, entries kept by the tile filter} (fwd: [0],[1]; bwd: [2],[3]) */
} DnrArgs;

/* loss_flags */
#define DNR_LOSS_FUSED_BWD 1u  /* dnr_raster_bwd evaluates the loss gradients itself (see above) */
#define DNR_LOSS_IMG_U8 2u     /* gt_image is uint8 */
#define DNR_LOSS_NORMAL_U8 4u  /* gt_normal is uint8 [H,W,3] (value / 255, as get_gt_img does) */
#define DNR_LOSS_EDGE_FROM_IMAGE 8u /* EdgeAwareLogL1 edge weights from gt_image clamped below at 10/255 (dn_model.py:633)
                                       instead of the fp32 gt_rgb map */

int dnr_version(void);
const char* dnr_error_string(int code);

int dnr_project_fwd(const DnrArgs* a, void* stream);

size_t dnr_bin_scan_workspace_bytes(int32_t n_gauss);
/* Sorts visible Gaussians by depth, counts the tiles each one really touches (or its whole bbox with
 * DNR_FLAG_EXACT_LISTS), scans the counts and stores the total in *a->n_isects_dev.  If n_isects_host is not
 * NULL the total is also copied there and the stream is synchronised (the one documented host sync);
 * pass NULL to stay asynchronous and size by capacity. */
int dnr_bin_scan(const DnrArgs* a, void* stream, int64_t* n_isects_host);
size_t dnr_bin_sort_workspace_bytes(int32_t n_gauss, int64_t n_isects, int32_t n_tiles);
/* Device pointer to the depth-sorted Gaussian ids inside a bin_scan workspace (valid after dnr_bin_scan). */
const int32_t* dnr_depth_order_ptr(void* ws_scan, int32_t n_gauss);
int dnr_bin_sort(const DnrArgs* a, void* stream);

int dnr_raster_fwd(const DnrArgs* a, void* stream);
int dnr_finalize_fwd(const DnrArgs* a, void* stream);
/* normal_from_depth_image for an arbitrary depth map: depth in a->out_depth, result (un-flipped,
 * un-remapped, zero border) in a->out_surface_normal; intrinsics from a->K. */
int dnr_normal_from_depth(const DnrArgs* a, void* stream);

int dnr_raster_bwd(const DnrArgs* a, void* stream);
int dnr_project_bwd(const DnrArgs* a, void* stream);

/* DNRegularization depth + normal terms on rendered maps: pred depth in a->out_depth, pred normal in
 * a->out_normal.  loss_partials (zeroed by the call):
 * [0] sum_x  [1] count_x  [2] sum_y  [3] count_y  (depth term; for non edge-aware types only x is used)
 * [4] sum |n - n_gt|   [5] sum |dW n|   [6] sum |dH n|
 * [8] depth term incl. the (1 + depth_lambda) factor  [9] normal L1  [10] normal TV  [11] [8]+[9]+[10].
 * dnr_loss_bwd writes d(loss)/d(depth) [H,W] and d(loss)/d(normal) [H,W,3] (either may be NULL). */
int dnr_loss_fwd(const DnrArgs* a, void* stream);
int dnr_loss_bwd(const DnrArgs* a, float* v_depth_out, float* v_normal_out, void* stream);

/* DNRegularization.get_scale_loss (regularization_strategy.py:195-199): mean_i min_k exp(scales[i,k]).
 * fwd: *loss_out (zeroed by the call) = the mean.  bwd: v_scales[N,3] = v * d(loss)/d(scales) (dense). */
int dnr_scale_loss_fwd(const float* scales, int32_t n_gauss, float* loss_out, void* stream);
int dnr_scale_loss_bwd(const float* scales, int32_t n_gauss, const float* v_loss, float* v_scales, void* stream);

/* Photometric L1 of the parent SplatfactoModel.get_loss_dict [EXT] (dn_splatter/dn_model.py:624-628 calls it):
 * mean |pred - gt| over n floats; gt is fp32, or uint8 (gt_is_u8 != 0, scaled by 1/255 as get_gt_img does).
 * fwd: *loss_out (zeroed by the call) = the mean.  bwd: v_pred[n] = (*v_loss or 1) * sign(pred - gt) / n. */
int dnr_l1_fwd(const float* pred, const void* gt, int64_t n, int32_t gt_is_u8, float* loss_out, void* stream);
int dnr_l1_bwd(const float* pred, const void* gt, int64_t n, int32_t gt_is_u8, const float* v_loss, float* v_pred,
               void* stream);
/* get_gt_img's uint8 -> float conversion in one pass: dst[i] = max(src[i] / divisor, clamp_min). */
int dnr_u8_to_f32(const uint8_t* src, int64_t n, float divisor, float clamp_min, float* dst, void* stream);

/* SSIM term of the same photometric loss: torchmetrics StructuralSimilarityIndexMeasure(data_range=1.0,
 * kernel_size=11) (dn_splatter/dn_model.py:180), i.e. an 11x11 Gaussian window (sigma 1.5), mean over the
 * (H-10)x(W-10) interior.  pred / gt: [H,W,C] fp32.  fwd: *sum_out (zeroed by the call) = SUM of the SSIM map over
 * the interior and all channels (divide by (H-10)(W-10)C for the mean); dmaps [3,H,W,C] keeps the partial
 * derivatives for the backward.  bwd: v_pred[H,W,C] = (*v_mean or 1) * d(mean SSIM)/d(pred).
 * Default since round 2 (DNSplatterModelConfig.fused_ssim). */
int dnr_ssim_fwd(const float* pred, const float* gt, int32_t H, int32_t W, int32_t C, float* dmaps, float* sum_out,
                 void* stream);
int dnr_ssim_bwd(const float* pred, const float* gt, int32_t H, int32_t W, int32_t C, const float* dmaps,
                 const float* v_mean, float* v_pred, void* stream);
/* The same with the target read as stored: gt is uint8 (value / 255, as get_gt_img does) when gt_is_u8 != 0, else fp32. */
int dnr_ssim_fwd_ex(const float* pred, const void* gt, int32_t gt_is_u8, int32_t H, int32_t W, int32_t C, float* dmaps,
                    float* sum_out, void* stream);
int dnr_ssim_bwd_ex(const float* pred, const void* gt, int32_t gt_is_u8, int32_t H, int32_t W, int32_t C, const float* dmaps,
                    const float* v_mean, float* v_pred, void* stream);

/* The whole photometric term of the parent SplatfactoModel.get_loss_dict [EXT] (dn_splatter/dn_model.py:624-628 calls it):
 *   main = (1 - ssim_lambda) * mean|pred - gt| + ssim_lambda * (1 - mean SSIM)
 * in one pass each way (the L1 sum shares the SSIM kernel's loads; its sign gradient is added by the SSIM backward).
 * out (3 floats, zeroed by the call): [0] SSIM sum over the interior, [1] sum |pred - gt|, [2] main.
 * bwd: v_pred[H,W,C] = (*v_main or 1) * d(main)/d(pred). */
int dnr_photometric_fwd(const float* pred, const void* gt, int32_t gt_is_u8, int32_t H, int32_t W, int32_t C,
                        float ssim_lambda, float* dmaps, float* out, void* stream);
int dnr_photometric_bwd(const float* pred, const void* gt, int32_t gt_is_u8, int32_t H, int32_t W, int32_t C,
                        float ssim_lambda, const float* dmaps, const float* v_main, float* v_pred, void* stream);

/* One-launch Adam over all Gaussian parameter groups: replaces the per-group torch.optim.Adam instances of
 * dn_splatter/dn_config.py:29-68 (lr per group, eps 1e-15; betas (0.9, 0.999), no weight decay, no amsgrad).
 * bc1 = 1 - beta1^t and bc2_sqrt = sqrt(1 - beta2^t) are computed by the host for each group's own step count t.
 * Python surface: optim.FusedAdam. */
#define DNR_ADAM_MAX_SEGS 16
typedef struct DnrAdamSeg {
  float* p;       /* [n] parameters, updated in place */
  const float* g; /* [n] gradients */
  float* m;       /* [n] exp_avg, updated in place */
  float* v;       /* [n] exp_avg_sq, updated in place */
  int64_t n;
  double lr, eps, bc1, bc2_sqrt; /* doubles: rounded to fp32 exactly where torch.optim.Adam rounds them */
  int64_t dense; /* dnr_adam_step_reduce only: != 0 -> every rank's rows of this segment are gathered, not just the rows of
                    the ranks that touched the Gaussian (a gradient term that depends on the parameters alone, e.g. the
                    min-scale regulariser, makes the whole segment non-zero on every rank) */
} DnrAdamSeg;
int dnr_adam_step(const DnrAdamSeg* segs /* HOST array */, int32_t n_segs, double beta1, double beta2, void* stream);

/* Multi-GPU: the gradient reduction fused into the Adam pass over NVLink peer memory (replaces the
 * bucket.all_reduce() + optimizer.step() pair that stands in for the reference's DDP wrapper, dn_pipeline.py:123-128).
 * Every rank keeps its flat gradient bucket and its `touched` flags (DnrArgs.touched, written by dnr_raster_bwd) in
 * peer-mapped memory at the same offsets; rows of untouched Gaussians are exactly zero.  For each element the gradient
 * is the sum, in rank order, of the rows of the ranks that touched the Gaussian (read straight from their memory), so
 * all replicas apply bit-identical updates.  segs[i].g must point into THIS rank's bucket (peer_flat[rank]); widths[i] =
 * floats per Gaussian of segment i.  The caller brackets the call with cross-rank barriers (all buckets final before,
 * all reads done before anyone zeroes its bucket again). */
#define DNR_PEER_MAX 8
typedef struct DnrPeerReduce {
  int32_t world, rank;
  int32_t n_gauss, reserved;
  const float* peer_flat[DNR_PEER_MAX];      /* device pointers valid on THIS device: rank k's flat bucket */
  const uint8_t* peer_touched[DNR_PEER_MAX]; /* rank k's touched flags [n_gauss] */
  uint8_t* mask;                             /* [n_gauss] local scratch (bit k: rank k touched the Gaussian) */
} DnrPeerReduce;
int dnr_adam_step_reduce(const DnrAdamSeg* segs /* HOST array */, const int32_t* widths /* HOST array */, int32_t n_segs,
                         double beta1, double beta2, const DnrPeerReduce* peers /* HOST struct */, void* stream);

/* ---- SuGaR-style queries (SURVEY 8f-4; Python surface: dn_splatter_b200.sugar) ----
 * Grid-hash k-NN: replaces sklearn behind dn_splatter/utils/knn.py:29-43 (knn_sk) and nerfstudio's k_nearest_sklearn
 * (dn_model.py:187).  The host chooses the grid; points outside it are clamped into the border cells (still exact). */
typedef struct DnrKnnGrid {
  float lo[3];     /* origin of cell (0,0,0) */
  float cell;      /* cell edge */
  float inv_cell;  /* 1 / cell */
  int32_t dims[3]; /* cells per axis; product <= 2^26 */
} DnrKnnGrid;
int64_t dnr_knn_workspace_bytes(int32_t n_points, const DnrKnnGrid* grid);
int dnr_knn_build(const float* points /* [n,3] */, int32_t n_points, const DnrKnnGrid* grid, void* ws, int64_t ws_bytes,
                  void* stream);
/* out_idx [n_queries,k] int64 (-1 where fewer than k points exist), out_dist [n_queries,k] Euclidean or NULL.
 * skip_first != 0 reproduces knn_sk: search k+1 and drop the nearest (the query itself when it is a data point). */
int dnr_knn_query(int32_t n_points, const DnrKnnGrid* grid, const void* ws, const float* queries /* [m,3] */,
                  int32_t n_queries, int32_t k, int32_t skip_first, int64_t* out_idx, float* out_dist, void* stream);
/* Density of the Gaussian set at samples [n,3] given neighbour lists nbr_idx [n / samples_per_row, k] (int64, -1 =
 * none): get_density (dn_model.py:1077-1135) with clamp_min = 1e-4.  Raw parameters (log-scales, opacity logits,
 * un-normalised wxyz quats). */
int dnr_density(const float* samples, int64_t n_samples, const int64_t* nbr_idx, int32_t k, int32_t samples_per_row,
                const float* means, const float* scales, const float* quats, const float* opacities, int32_t n_gauss,
                float clamp_min, float* out, void* stream);
/* The ray sampling of compute_level_surface_points (dn_model.py:1264-1345): for each point p (a back-projected
 * pixel) 21 samples p + t_j d, t_j = linspace(-range, range, 21) * std(first neighbour), d = normalize(p - cam).
 * out_dens / out_t [n_points,21], out_dirs [n_points,3].  cam_pos_host: 3 floats on the HOST. */
int dnr_ray_densities(const float* points, int64_t n_points, const int64_t* nbr_idx, int32_t k, const float* cam_pos_host,
                      const float* means, const float* scales, const float* quats, const float* opacities,
                      int32_t n_gauss, int32_t n_range, float range_size, float* out_dens, float* out_t, float* out_dirs,
                      void* stream);

/* ---- TSDF mesh extraction (gs-mesh o3dtsdf, export_mesh.py:931-1047; Python surface: dn_splatter_b200.export_mesh) ----
 * Open3D's legacy ScalableTSDFVolume on the device: volume units of 16^3 voxels in an open-addressing hash, allocated
 * from the stride-4 depth point cloud and integrated per view; marching cubes over the allocated units; the connected-
 * cluster filter of the exporter.  Unit coordinates must lie in [-2^20, 2^20) (counters[3] counts points outside). */
typedef struct DnrTsdfVolume {
  double voxel_size;   /* voxel edge (Open3D voxel_length) */
  double sdf_trunc;    /* truncation distance */
  float depth_trunc;   /* depth > depth_trunc is treated as no depth */
  int32_t capacity;    /* volume units in the pool */
  int32_t hash_size;   /* hash slots: a power of two >= capacity */
  int32_t reserved;
  void* hash_keys;     /* uint64[hash_size]: packed unit coordinates, ~0 = empty */
  void* hash_vals;     /* int32[hash_size]: pool slot of the unit, -1 when the pool was full */
  void* hash_stamp;    /* int32[hash_size]: stamp of the last view that touched the unit */
  void* voxels;        /* float[capacity][5][4096]: tsdf, weight, r, g, b (0..255); voxel x + 16 y + 256 z */
  void* touched;       /* int32[hash_size]: hash slots touched by the current view */
  void* counters;      /* int32[4]: units requested (> capacity = overflow), touched this view, hash full, out of range */
} DnrTsdfVolume;
typedef struct DnrTsdfView {
  int32_t width, height;
  int32_t stamp;        /* distinct per view since the last reset, >= 0 */
  int32_t reserved;
  float fx, fy, cx, cy;
  float extrinsic[16];  /* world -> camera (OpenCV), fp32, row-major */
  double pose[16];      /* camera -> world, fp64 (inverse of extrinsic), row-major */
  const float* depth;   /* [H,W] */
  const float* rgb;     /* [H,W,3] in [0,1]; the colour used is (uint8)(rgb * 255) */
  const uint8_t* mask;  /* [H,W] or NULL: 0 = no depth */
} DnrTsdfView;
/* Empties the hash, zeroes the pool and the counters. */
int dnr_tsdf_reset(const DnrTsdfVolume* vol /* HOST struct */, void* stream);
/* Allocation: inserts the units within sdf_trunc of every stride-4 depth point, lists this view's units. */
int dnr_tsdf_allocate(const DnrTsdfVolume* vol, const DnrTsdfView* view /* HOST structs */, void* stream);
/* Integration of the units listed by the last dnr_tsdf_allocate (one CTA per unit, one thread per voxel column). */
int dnr_tsdf_integrate(const DnrTsdfVolume* vol, const DnrTsdfView* view, void* stream);
/* Marching cubes over n_units = counters[0] (no overflow) units, in sorted unit order.  extract_count writes int64
 * {n_vertices, n_triangles} at the start of ws; extract_emit fills vertices / colours [n_vertices,3] f32 and triangles
 * [n_triangles,3] int32. */
int64_t dnr_tsdf_extract_workspace_bytes(int32_t n_units);
int dnr_tsdf_extract_count(const DnrTsdfVolume* vol, int32_t n_units, void* ws, int64_t ws_bytes, void* stream);
int dnr_tsdf_extract_emit(const DnrTsdfVolume* vol, int32_t n_units, void* ws, int64_t ws_bytes, float* vertices,
                          float* colors, int32_t* triangles, void* stream);
/* Cluster filter: triangles sharing an edge are connected; triangles of clusters smaller than
 * max(size of the keep_largest-th largest cluster (0 if fewer), min_triangles) are removed, then unreferenced vertices;
 * order is kept.  cluster_count writes int64 {kept vertices, kept triangles} at the start of ws. */
int64_t dnr_mesh_cluster_workspace_bytes(int32_t n_triangles, int32_t n_vertices);
int dnr_mesh_cluster_count(const int32_t* triangles, int32_t n_triangles, int32_t n_vertices, int32_t keep_largest,
                           int32_t min_triangles, void* ws, int64_t ws_bytes, void* stream);
int dnr_mesh_cluster_emit(const int32_t* triangles, const float* vertices, const float* colors, int32_t n_triangles,
                          int32_t n_vertices, void* ws, int64_t ws_bytes, int32_t* out_triangles, float* out_vertices,
                          float* out_colors, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DNR_H_ */
