/*
 * ddn_b200.h - C ABI of the B200-native DepthDensifier hot path (libddn_b200.so).
 *
 * Drop-in boundary.  The reference (OpsiClear/DepthDensifier) has no FFI: the path sits behind
 * Python calls.  Each entry point below names the reference code it replaces; the Python shim in
 * depthdensifier_b200/ keeps the reference's names (DepthRefiner.refine_depth, project_points,
 * unproject_points, main) and binds these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All data pointers are DEVICE pointers unless the
 *     parameter name ends in _host.  `stream` is a cudaStream_t passed as void*.
 *   - every call returns 0 (DDN_OK) or a negative DDN_ERR_* code; ddn_last_error_string() gives
 *     the thread-local message.  Nothing throws across the boundary.
 *   - the caller owns every buffer (inputs, outputs, workspaces).  A *_workspace_bytes() query
 *     precedes any call that needs scratch.
 *   - calls are stream-ordered and asynchronous: no hidden device synchronisation, no global
 *     mutable state.  Counts are written to device memory; the caller decides when to sync.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef DDN_B200_H_
#define DDN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define DDN_API __attribute__((visibility("default")))
#else
#define DDN_API
#endif

#define DDN_VERSION 200 /* ABI revision 2 (device-resident fusion sessions); the Python package keeps the reference's __version__ 0.1.0 */

enum {
  DDN_OK = 0,
  DDN_ERR_INVALID_ARGUMENT = -1,
  DDN_ERR_CUDA = -2,
  DDN_ERR_WORKSPACE_TOO_SMALL = -3,
  DDN_ERR_UNSUPPORTED = -4
};

DDN_API int ddn_version(void);
DDN_API const char* ddn_last_error_string(void);
/* Number of kernels this library has launched in the calling process (for bench.py gpu_launches). */
DDN_API int64_t ddn_launch_count(void);
/* Diagnostics (single-threaded use): with profiling on, the multi-GPU merge records a CUDA event after each of its
 * kernels; ddn_profile_report synchronises the device and writes "name milliseconds" lines (time since the previous
 * mark on the stream, so the first line of a call also contains whatever ran before it) into buf. */
/* Diagnostic: reads `bytes` from src (local or NVLink peer memory) with mode 0 = ld.global.cv, 1 = plain ld.global,
 * 2 = ld.global.nc; per_thread (1..8) 16-byte loads in flight per thread; out: device [1] u32 scratch. */
DDN_API int ddn_debug_peer_read(const void* src, int64_t bytes, int32_t mode, int32_t per_thread, int32_t ctas, void* out,
                        void* stream);
DDN_API void ddn_profile_enable(int on);
DDN_API int ddn_profile_report(char* buf, int64_t size);

/* ------------------------------------------------------------------------------------------
 * Stage 1 - per-view alignment of monocular depth to projected sparse points.
 * Replaces DepthRefiner.refine_depth, src/depthdensifier/depth_refiner.py:207-328
 * (_project_points :92-115, bounds+grid_sample :247-288, _remove_outliers_fast :117-139,
 *  min-count gate and subsample :296-306, _pchip_interpolate_optimized :141-178,
 *  _apply_transformation incl. 3x3 median :180-205), batched over V views.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t min_correspondences;      /* RefinerConfig.min_correspondences (50)  depth_refiner.py:21 */
  int32_t edge_margin;              /* RefinerConfig.edge_margin (10)          :22 */
  int32_t robust;                   /* RefinerConfig.robust (1)                :23 */
  float outlier_threshold;          /* RefinerConfig.outlier_threshold (2.5)   :24 */
  int32_t skip_smoothing;           /* RefinerConfig.skip_smoothing (0)        :28 */
  int32_t adaptive_correspondences; /* RefinerConfig.adaptive_correspondences (1) :29 */
  int32_t max_pairs;                /* 500, depth_refiner.py:302-306 */
  int32_t mode;                     /* 0 = piecewise-linear LUT (reference); 1 = affine scale/shift LSQ (new) */
  uint32_t subsample_seed;          /* seed of the hash permutation that replaces torch.randperm (:304) */
  int32_t zero_unmasked_passthrough; /* 1: pass-through views are also zeroed outside the mask (scripts/test.py:194) */
  int32_t mask_packed;              /* 1: mask is one BIT per pixel ([V, ceil(H*W/8)] u8, bit g & 7 of byte g >> 3) */
  int32_t use_tma;                  /* 1: the remap kernel loads its depth tile with one TMA tensor copy (needs W % 4 == 0, W >= 132, H >= 34; same bits, measured 6 % slower than the default loads) */
} ddn_align_config;

/* status values in ddn_view_stats */
enum {
  DDN_VIEW_REFINED = 0,
  DDN_VIEW_NO_POINTS_IN_BOUNDS = 1, /* depth_refiner.py:256-259 */
  DDN_VIEW_NO_POSITIVE_SAMPLES = 2, /* :275-285 */
  DDN_VIEW_TOO_FEW = 3,             /* :296-299 */
  DDN_VIEW_DEGENERATE_FIT = 4,      /* affine mode only */
  DDN_VIEW_NO_SPARSE = 5            /* scripts/test.py:136-137: view skipped by the pipeline */
};

typedef struct {
  int32_t status;
  int32_t num_correspondences; /* refine_depth()["num_correspondences"] */
  int32_t outliers_removed;    /* refine_depth()["outliers_removed"] */
  int32_t num_table;           /* knots in the view's lookup table */
  float scale_factor;          /* refine_depth()["scale_factor"]: lower median of z_colmap/(z_depth+1e-6) */
  float affine_scale;          /* mode 1 */
  float affine_shift;          /* mode 1 */
  int32_t reserved;
} ddn_view_stats;

DDN_API void ddn_align_config_default(ddn_align_config* cfg);

DDN_API int ddn_align_workspace_bytes(int64_t n_views, int64_t max_sparse_per_view, int64_t* bytes_out);

/* depth [V,H,W] f32; mask [V,H,W] u8 (or bit-packed, cfg->mask_packed) or NULL (=> depth > 0, depth_refiner.py:238-241);
 * cam_from_world [V,3,4] f64 row-major; kmat [V,3,3] f64 (only the top two rows are used, :112);
 * sparse_xyz [S,3] f64 world, CSR sparse_offsets [V+1] i64; refined [V,H,W] f32 out;
 * stats [V] out.  A view with no sparse points gets status DDN_VIEW_NO_SPARSE and an all-zero map.
 * Views that the reference returns unchanged get a copy of their input depth.
 * Optional bounding-box epilogue (src_table and bbox both non-NULL): bbox [6] (ddn_bbox_init encoding)
 * is extended to enclose the back-projection (src_table [V,16] f32 from ddn_build_pair_tables, the
 * arithmetic of ddn_backproject_filter) of every refined pixel > 0.  It is a tile-wise bound (the 8 corners
 * of each 126x32 pixel tile at its smallest and largest depth), i.e. a superset of the exact box, and makes
 * the voxel grid known BEFORE stages 2+3 run. */
DDN_API int ddn_align_views(const ddn_align_config* cfg, int64_t n_views, int64_t height, int64_t width,
                    const float* depth, const uint8_t* mask, const double* cam_from_world,
                    const double* kmat, const double* sparse_xyz, const int64_t* sparse_offsets,
                    int64_t max_sparse_per_view, float* refined, ddn_view_stats* stats,
                    void* workspace, int64_t workspace_bytes, const float* src_table, float* bbox,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * Stages 2+3 - pixel back-projection fused with the multi-view consistency vote.
 * Replaces scripts/test.py:205-233 (pixel grid, unproject_points :79-90, cam_from_world().inverse())
 * and scripts/test.py:273-330 (project_points :58-76, grazing gate, nearest lookup, floater vote),
 * evaluated against a neighbour table nbr[V,K] instead of all views.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  float depth_threshold;   /* FilteringConfig.depth_threshold (0.7) scripts/test.py:45 */
  float grazing_cos;       /* 0.087, scripts/test.py:295 */
  int32_t sample_mode;     /* 0 = nearest/truncate (reference, :308-309); 1 = bilinear 4-tap (new) */
  float two_sided_tau;     /* <= 0: one-sided z < thr*D (reference, :319-321); > 0: |z-D| > tau*D (new) */
  int32_t stride;          /* ProcessingConfig.downsample_density (scripts/test.py:37); 1 = densest */
  int32_t normals_in_world; /* 0 = reference quirk (camera-frame normal vs world dir, :291, used as given);
                               1 = rotate by R_src^T and divide by (|n| + 1e-8) (visualizer.py:346-376) */
  int32_t pixel_layout;    /* which 4 pixels a thread owns: 0 = 32 apart (default), 1 = adjacent (vector I/O); same results */
} ddn_filter_config;

DDN_API void ddn_filter_config_default(ddn_filter_config* cfg);

#define DDN_PAIR_TABLE_FLOATS 24
/* pair_table [n_src,K,DDN_PAIR_TABLE_FLOATS] f32 and src_table [n_src,16] f32 are computed in float64
 * on the device from the poses (cam_from_world [V,3,4] f64) and PINHOLE intrinsics
 * (intr [V,4] f64: fx, fy, cx, cy - scripts/test.py:81) and rounded once. */
DDN_API int ddn_build_pair_tables(int64_t n_views_total, int64_t src_begin, int64_t n_src, int64_t k_nbr,
                          int64_t height, int64_t width, const double* cam_from_world, const double* intr,
                          const int32_t* nbr, float* pair_table, float* src_table, void* stream);

/* refined_all [V,H,W] f32 (zero outside the mask); normal [n_src,H,W,3] f32 for the source views
 * src_begin..src_begin+n_src - only the normals of vote candidates are read, so this one pointer may
 * also be PINNED HOST memory (unified addressing): the map then never moves to the device; outputs on the strided grid Hs=ceil(H/stride), Ws=ceil(W/stride):
 * xyz [n_src,Hs,Ws,3] f32 world, votes [n_src,Hs,Ws] u8 (255 = pixel has no point, i.e. depth<=0).
 * bbox [6] f32 (optional, may be NULL): running min xyz / max xyz over points with
 * votes < vote_threshold; must be initialised to +inf/-inf by ddn_bbox_init.
 * vote_threshold is clamped to 255: votes saturate at 254 and 255 marks "no point", so a threshold of 255
 * or more keeps every point that exists and never a pixel without one, whatever its count (also 255 or
 * more), so votes[i] < min(vote_threshold, 255) reproduces the kernel's keep and mark exactly.
 * mark (optional, may be NULL): a fusion session opened by ddn_fuse_begin*; the kernel then also sets the
 * occupancy bit of every kept point (the "mark" pass of stage 4 fused into the epilogue, where the point
 * is still in registers) and adds their number to the session's counts[0]. */
struct ddn_fuse_session;
DDN_API int ddn_backproject_filter(const ddn_filter_config* cfg, int64_t n_views_total, int64_t src_begin,
                           int64_t n_src, int64_t height, int64_t width, int64_t k_nbr,
                           const float* refined_all, const float* normal, const int32_t* nbr,
                           const float* pair_table, const float* src_table, int32_t vote_threshold,
                           float* xyz, uint8_t* votes, float* bbox, const struct ddn_fuse_session* mark,
                           void* stream);

/* ddn_backproject_filter with a multi-view support count (new; parity unpinned, DESIGN.md §2).  Neighbour entry t of
 * the table SUPPORTS the point of a pixel when the point projects into t's map in bounds, the sampled depth D
 * (cfg->sample_mode, as for the vote) is > 0, and |z - D| <= support_tau * D, with z the point's depth in view t.  No
 * grazing gate; entries of the source view itself never count.  support [n_src,Hs,Ws] u8 (same grid as votes):
 * min(count, 254), 255 = no point.  A point is kept iff it exists, its vote count is below vote_threshold (as in
 * ddn_backproject_filter) and count >= min_support.  min_support in [0, 1024]; support_tau > 0 and finite.
 *
 * The keep decision is carried in the vote byte, so every fusion call (ddn_fuse_*, ddn_voxel_*) and a host-side
 * keep mask reproduce K4's keep, its bounding box and its occupancy mark (counts[0]) when they are given the
 * threshold min(vote_threshold, 254).  For a point:
 *   votes = 254                  when count < min_support;
 *   votes = min(nvotes, 254)     otherwise, when vote_threshold <= 254;
 *   votes = min(nvotes, 253)     otherwise, when vote_threshold >= 255 (every supported point is kept);
 *   votes = 255                  when the pixel has no point.
 * Then keep == (votes < min(vote_threshold, 254)) at every vote_threshold and min_support.  With min_support = 0 and
 * vote_threshold <= 254, votes, xyz, bbox and the mark are those of ddn_backproject_filter, byte for byte. */
DDN_API int ddn_backproject_filter_support(const ddn_filter_config* cfg, int64_t n_views_total, int64_t src_begin,
                                   int64_t n_src, int64_t height, int64_t width, int64_t k_nbr,
                                   const float* refined_all, const float* normal, const int32_t* nbr,
                                   const float* pair_table, const float* src_table, int32_t vote_threshold,
                                   int32_t min_support, float support_tau, float* xyz, uint8_t* votes,
                                   uint8_t* support, float* bbox, const struct ddn_fuse_session* mark, void* stream);

/* ddn_backproject_filter_support with a forward-backward reprojection check (new; parity unpinned: the reference has
 * no such check).  For the point of source view s at pixel (x, y) with depth d, and neighbour entry t: (u, v, z) is its
 * projection into t and D the sampled depth, both as for ddn_backproject_filter_support.  Back-project t's pixel at the
 * CONTINUOUS coordinates (u, v) at depth D, take that point into s: pixel (x', y'), depth z'.  Continuous in both
 * sampling modes: with bilinear sampling that is MVSNet's check; with nearest, back-projecting the truncated pixel
 * would add up to sqrt(2) px of lookup error by itself, so the continuous point measures only the depth disagreement
 * along the epipolar line.  Entry t SUPPORTS the point iff
 *   the depth test of ddn_backproject_filter_support holds (in bounds, D > 0, |z - D| <= support_tau * D, not the
 *   source view itself)  and  z' > 0  and  |(x', y') - (x, y)|_2 <= reproj_px.
 * Closed form, which the kernel evaluates: with e = K_s (R_s c_t + t_s), t's epipole in s (homogeneous), P = d x,
 * Q = d y and w = (z - D) / z,
 *   z' = d + w (e_z - d),   (x' - x, y' - y) = w (d e_x - P e_z, d e_y - Q e_z) / (d z'),
 * so the test is  z' > 0  and  w^2 [(d e_x - P e_z)^2 + (d e_y - Q e_z)^2] <= reproj_px^2 (d z')^2.
 * reproj_px > 0 and finite.  The support byte, the keep rule and the vote encoding are those of
 * ddn_backproject_filter_support, with "supports" meaning the combined test. */
DDN_API int ddn_backproject_filter_support_reproj(const ddn_filter_config* cfg, int64_t n_views_total,
                                          int64_t src_begin, int64_t n_src, int64_t height, int64_t width,
                                          int64_t k_nbr, const float* refined_all, const float* normal,
                                          const int32_t* nbr, const float* pair_table, const float* src_table,
                                          int32_t vote_threshold, int32_t min_support, float support_tau,
                                          float reproj_px, float* xyz, uint8_t* votes, uint8_t* support,
                                          float* bbox, const struct ddn_fuse_session* mark, void* stream);

DDN_API int ddn_bbox_init(float* bbox, void* stream);

/* ------------------------------------------------------------------------------------------
 * Ragged views: stages 1-3 for V views of DIFFERENT sizes (H_v, W_v) in one pass each, as the reference's
 * per-image loop allows (scripts/test.py:145-173 refines each image at its own size, :275-328 votes with every
 * cached view at that view's size).  Per-pixel buffers (depth, mask, refined, normal) are the concatenation of
 * the views' row-major maps; strided-grid buffers (xyz, votes) the concatenation of their
 * Hs_v x Ws_v = ceil(H_v/stride) x ceil(W_v/stride) grids.  Sizes and offsets travel as a LAYOUT,
 * int64 [V + 1, DDN_LAYOUT_COLS]:
 *   row v < V:  H_v, W_v, pix_off[v], grid_off[v], tile_off[v], chunk_off[v], 0, 0
 *   row V:      stride, V, total pixels, total grid points, total tiles, total chunks, 0, 0
 * with pix_off[v] = sum_{u<v} H_u W_u, grid_off[v] = sum_{u<v} Hs_u Ws_u, tile_off[v] = sum_{u<v} ceil(H_u/32)
 * ceil(W_u/126) (remap tiles) and chunk_off[v] = sum_{u<v} ceil(Hs_u Ws_u / 1024) (consistency CTAs): the kernels
 * run one flat grid over all tiles / chunks and find their view from these prefixes.  Limits: 1 <= V <= 65535,
 * every side below 2^22, fewer than 2^32 pixels in all.  Each ragged call takes the layout twice: `layout` in
 * device memory for the kernels and `layout_host`, the same values on the host, which the call validates (the
 * offsets must be the prefix sums of the sizes) and sizes its launches from, so it never reads the device back.
 * The uniform entry points above are unchanged; uniform views through the ragged path give the same bits.
 * ------------------------------------------------------------------------------------------ */
#define DDN_LAYOUT_COLS 8

/* ddn_align_views over a layout: depth, mask (one byte per pixel, or NULL) and refined are flat [total pixels];
 * workspace from ddn_align_workspace_bytes(V, ...); stats [V]; src_table [V,16] (ddn_build_pair_tables_ragged) and
 * bbox as in ddn_align_views (the box's tiles are the ragged tiles of each view).  Needs H_v, W_v >= 2.
 * cfg->mask_packed and cfg->use_tma are byte-layout options of the uniform call: here they return
 * DDN_ERR_UNSUPPORTED. */
DDN_API int ddn_align_views_ragged(const ddn_align_config* cfg, int64_t n_views, const int64_t* layout,
                           const int64_t* layout_host, const float* depth, const uint8_t* mask,
                           const double* cam_from_world, const double* kmat, const double* sparse_xyz,
                           const int64_t* sparse_offsets, int64_t max_sparse_per_view, float* refined,
                           ddn_view_stats* stats, void* workspace, int64_t workspace_bytes, const float* src_table,
                           float* bbox, void* stream);

/* ddn_build_pair_tables for all V views of a layout (sources 0..V-1).  Entries as in the uniform tables except
 * floats 16-19, which describe the NEIGHBOUR's map: W_t, H_t (int bits), (float)W_t, (float)H_t, and the gather
 * offset (float 21) pix_off[t] - 0x4B000000 (W_t + 1) mod 2^32.  The sizes come from the same layout the
 * consistency kernel reads, so a table cannot disagree with the maps it is used with. */
DDN_API int ddn_build_pair_tables_ragged(int64_t n_views, int64_t k_nbr, const int64_t* layout,
                                 const int64_t* layout_host, const double* cam_from_world, const double* intr,
                                 const int32_t* nbr, float* pair_table, float* src_table, void* stream);

/* ddn_backproject_filter for all V views of a layout: refined_all flat [total pixels] f32; normal flat
 * [total pixels, 3] f32 (device or pinned host memory); pair_table / src_table from ddn_build_pair_tables_ragged;
 * xyz [total grid points, 3] f32 and votes [total grid points] u8 on each view's strided grid.  cfg->stride must
 * equal the layout's stride.  bbox, vote_threshold and mark as in ddn_backproject_filter; a fusion session then
 * finishes with row_len = 0. */
DDN_API int ddn_backproject_filter_ragged(const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr,
                                  const int64_t* layout, const int64_t* layout_host, const float* refined_all,
                                  const float* normal, const float* pair_table, const float* src_table,
                                  int32_t vote_threshold, float* xyz, uint8_t* votes, float* bbox,
                                  const struct ddn_fuse_session* mark, void* stream);

/* ddn_backproject_filter_ragged with the support count, keep rule and vote encoding of
 * ddn_backproject_filter_support; support [total grid points] u8 on the same grids as votes. */
DDN_API int ddn_backproject_filter_support_ragged(const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr,
                                          const int64_t* layout, const int64_t* layout_host,
                                          const float* refined_all, const float* normal, const float* pair_table,
                                          const float* src_table, int32_t vote_threshold, int32_t min_support,
                                          float support_tau, float* xyz, uint8_t* votes, uint8_t* support,
                                          float* bbox, const struct ddn_fuse_session* mark, void* stream);

/* ddn_backproject_filter_support_ragged with the reprojection check of ddn_backproject_filter_support_reproj. */
DDN_API int ddn_backproject_filter_support_reproj_ragged(const ddn_filter_config* cfg, int64_t n_views, int64_t k_nbr,
                                                 const int64_t* layout, const int64_t* layout_host,
                                                 const float* refined_all, const float* normal,
                                                 const float* pair_table, const float* src_table,
                                                 int32_t vote_threshold, int32_t min_support, float support_tau,
                                                 float reproj_px, float* xyz, uint8_t* votes, uint8_t* support,
                                                 float* bbox, const struct ddn_fuse_session* mark, void* stream);

/* Neighbouring per-pixel helpers (SURVEY.md 8(f) rank 4).
 * ddn_gradient_mask: compute_depth_normal_gradient_mask, src/depthdensifier/initilizer.py:236-328 - mask_out [H,W]
 *   u8 = 1 where the Sobel magnitude of the (zero-padded, separable) Gaussian-smoothed depth relative to that depth
 *   exceeds depth_threshold, or the torch.gradient magnitude over the three normal channels exceeds
 *   normal_threshold.  taps_host: the n_taps (odd; 0 = no smoothing) float32 Gaussian taps; depth or normal may be
 *   NULL; workspace >= two float planes + 512 bytes when smoothing.
 * ddn_transform_normals: COLMAPVisualizer._transform_normals, src/depthdensifier/visualizer.py:346-376 -
 *   normal_world [N,3] f64 = normalise(R^T n_cam); cam_from_world_host is a row-major [3,4] or [4,4] HOST matrix
 *   (row_stride 4) or a 3x3 rotation (row_stride 3). */
DDN_API int ddn_gradient_mask(int64_t height, int64_t width, const float* depth, const float* normal,
                      const float* taps_host, int32_t n_taps, float depth_threshold, float normal_threshold,
                      uint8_t* mask_out, void* workspace, int64_t workspace_bytes, void* stream);
DDN_API int ddn_transform_normals(int64_t n_points, const float* normal_cam, const double* cam_from_world_host,
                          int32_t row_stride, double* normal_world, void* stream);

/* Stand-alone helpers with the reference script's own semantics, float64 (device arrays except params4_host):
 * ddn_project_points   = project_points, scripts/test.py:58-76: points3d [N,3], cam_from_world [3,4],
 *                        kmat [3,3] -> points2d [N,2], depths [N] (no validity handling, +1e-8 in the divide);
 * ddn_unproject_points = unproject_points, scripts/test.py:79-90: points2d [N,2], depth [N] f32, PINHOLE
 *                        params (fx, fy, cx, cy) on the HOST -> camera-frame points [N,3]. */
DDN_API int ddn_project_points(int64_t n_points, const double* points3d, const double* cam_from_world,
                       const double* kmat, double* points2d, double* depths, void* stream);
DDN_API int ddn_unproject_points(int64_t n_points, const double* points2d, const float* depth,
                         const double* params4_host, double* points3d_cam, void* stream);

/* ------------------------------------------------------------------------------------------
 * Alternative stage 1: the per-pixel part of FastPCHIPRefiner, src/depthdensifier/fast_pchip_refiner.py
 * (SURVEY.md 8(f) rank 3).  One view per call; the O(C) correspondence logic stays on the host as in the
 * reference.
 *
 * ddn_pchip_edge_mask: _detect_depth_edges :226-273 (gray == NULL) or _detect_image_edges :187-224 (gray =
 *   float64 grey image [H,W]).  gauss_weights_host[0..radius] = the normalised taps of scipy's Gaussian at
 *   distance 0..radius (host array); normal [H,W,3] and mask [H,W] may be NULL.  edge_out [H,W] u8.
 * ddn_pchip_apply: _apply_edge_aware_transformation :550-579 with the cubic-Hermite evaluation :300-366 for the
 *   float32 knots (ascending x); mask and edge [H,W] u8; refined [H,W] f32.
 * ------------------------------------------------------------------------------------------ */
DDN_API int ddn_pchip_workspace_bytes(int64_t height, int64_t width, int64_t* bytes_out);
DDN_API int ddn_pchip_edge_mask(int64_t height, int64_t width, const float* depth, const uint8_t* mask,
                        const float* normal, const double* gray, const double* gauss_weights_host,
                        int32_t radius, float edge_threshold, double image_edge_threshold, uint8_t* edge_out,
                        void* workspace, int64_t workspace_bytes, void* stream);
DDN_API int ddn_pchip_apply(int64_t height, int64_t width, const float* depth, const uint8_t* mask,
                    const uint8_t* edge, const float* knots_x, const float* knots_y, int32_t n_knots,
                    float* refined, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 4 - voxel-grid fusion (new capability; the reference only concatenates,
 * scripts/test.py:353-359).  key = kx | ky<<21 | kz<<42 with k = floor((p - origin)/voxel) in
 * IEEE float32.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  float voxel;
  float origin[3];
  int32_t bits[3]; /* significant bits per axis (from the bounding box); sum <= 63 */
  int32_t dims[3]; /* cells per axis, <= 2^bits (0 => 2^bits); points outside do not participate */
} ddn_voxel_grid;

/* Scratch for ddn_voxel_fuse / ddn_voxel_partials / ddn_voxel_merge on `grid_host` with up to
 * n_points points (or records).  Grids of up to 2^35 cells use a dense occupancy bitmap
 * (cells/8 bytes + 40 B per possible voxel); larger grids (and grid_host == NULL) use the hashed path
 * (ddn_fuse_finish_hashed and its partial and merge forms) on hash buffers carved out of the workspace:
 * 100-124 B per point or record, the most any of the three calls needs. */
DDN_API int ddn_fuse_workspace_bytes(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t* bytes_out);

/* xyz [N,3] f32, rgb [N,3] u8, votes [N] u8 (point i participates iff votes[i] < vote_threshold;
 * votes may be NULL => all).  row_len: 0, or the image width when the points are the pixels of
 * [rows, row_len] depth maps in row-major order (a locality hint: the result does not depend on it).  Outputs sized for the worst case N: out_keys [N] u64 ascending,
 * out_xyz [N,3] f32, out_rgb [N,3] u8, out_count [N] i32; counts_out [2] i64 device:
 * {number of participating points, number of voxels}; the first is -1 if a voxel collected 2^24 or
 * more points (colour sums are 32-bit). */
DDN_API int ddn_voxel_fuse(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t row_len, const float* xyz,
                   const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold,
                   uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb, int32_t* out_count,
                   int64_t* counts_out, void* workspace, int64_t workspace_bytes, void* stream);

/* Multi-GPU form of stage 4.  ddn_voxel_partials fuses the rank's own points into per-voxel PARTIAL
 * records, keys ascending.  A record is DDN_RECORD_WORDS u64:
 *   [0] key   [1..3] sum of (p - voxel centre) * fl(1/voxel) * 2^20 per axis (two's complement)
 *   [4] sum(r) << 32 | sum(g)   [5] sum(b) << 32 | count
 * Integer sums make the final means independent of how points are split over ranks, and because the
 * records are sorted a destination rank's share is one contiguous slice.  ddn_voxel_merge adds the
 * records of equal key (any input order, e.g. the concatenation of the runs received from R ranks)
 * and finalises them.  records: [N, DDN_RECORD_WORDS] u64, 16-byte aligned, sized for the worst case. */
#define DDN_RECORD_WORDS 6
/* Ownership is by TILE: a tile is cells_per_tile consecutive cells of the grid in key order, so a range of
 * tiles is a key range.  *n_tiles = 0 means the grid is too large for the dense path (no tiles: partition by
 * sampled splitter keys instead). */
DDN_API int ddn_fuse_tile_info(const ddn_voxel_grid* grid_host, int64_t* n_tiles, int64_t* cells_per_tile);

/* tile_prefix (optional, dense path only): [n_tiles + 1] u32, tile_prefix[t] = index of the first record of
 * tile t in `records` (the last entry is the record count) - what a rank needs to cut its records at tile
 * boundaries without searching. */
DDN_API int ddn_voxel_partials(const ddn_voxel_grid* grid_host, int64_t n_points, int64_t row_len, const float* xyz,
                       const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold, uint64_t* records,
                       uint32_t* tile_prefix, int64_t* counts_out, void* workspace, int64_t workspace_bytes,
                       void* stream);

/* [tile_begin, tile_end): the tiles this call owns (0, 0 = the whole grid).  Only that slice of the grid is
 * scanned; records of other tiles are ignored. */
DDN_API int ddn_voxel_merge(const ddn_voxel_grid* grid_host, int64_t n_records, const uint64_t* records,
                    int64_t tile_begin, int64_t tile_end, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                    int32_t* out_count, int64_t* counts_out, void* workspace, int64_t workspace_bytes,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 4 without a host round trip: the FUSION SESSION.  The grid is derived ON THE DEVICE from one or
 * more bounding boxes (ddn_bbox_init encoding; with R ranks the R boxes may sit in peer memory) and kept
 * in device memory, launch sizes come from capacities, actual extents are read by the kernels.  A step is
 *   ddn_fuse_begin -> ddn_backproject_filter(..., mark = session) -> ddn_fuse_finish[_partial]
 *   [-> ddn_fuse_merge_peers]
 * and never needs the host to look at a result in between.
 * ------------------------------------------------------------------------------------------ */
enum { DDN_GRID_OK = 0, DDN_GRID_EMPTY = 1, DDN_GRID_TOO_LARGE = 2, DDN_GRID_TOO_MANY_BITS = 3, DDN_GRID_HASHED = 4 };

typedef struct ddn_grid_state { /* 64 bytes of DEVICE memory, written by ddn_fuse_begin* */
  float voxel;
  float origin[3]; /* (floor(box_min / voxel) - 1) * voxel in float32: one cell of slack below the box */
  int32_t bits[3];
  int32_t dims[3];
  int64_t n_units; /* occupancy units in use: ceil(cells / 96); 0 unless status == DDN_GRID_OK */
  int32_t status;  /* DDN_GRID_*: EMPTY = no finite box, TOO_LARGE = more cells than cap_units * 96, HASHED = a
                      TOO_LARGE grid that ddn_fuse_finish_hashed fused (origin, bits and dims are valid) */
  int32_t reserved;
  int64_t cells;
} ddn_grid_state;

#define DDN_MAX_PEERS 16

typedef struct ddn_fuse_session { /* HOST struct of DEVICE pointers, owned by the caller */
  ddn_grid_state* grid;
  void* units;           /* [cap_units] 16-byte units: 96 occupancy bits + the unit's rank prefix */
  int64_t cap_units;
  uint8_t* dirty;        /* [cap_units / 2048 + 1] one flag per 32 KB of units, or NULL.  With flags the
                            session keeps its units clean between steps (ddn_fuse_begin clears only what the
                            previous step touched) and the rank passes skip untouched tiles; without, every
                            step clears and scans the whole grid. */
  uint32_t* tile_sums;   /* [cap_units / 256 + 2] scratch */
  uint32_t* tile_prefix; /* [cap_units / 256 + 2] or NULL: index of the first record of every ownership tile
                            (256 units = 24,576 cells in key order); needed by ddn_fuse_merge_peers */
  int64_t* counts;       /* [2]: participating points, voxels (the true count even when it exceeds a capacity) */
} ddn_fuse_session;

/* Sizes of the session buffers for grids of up to max_cells cells (all outputs in bytes but cap_units). */
DDN_API int ddn_fuse_session_sizes(int64_t max_cells, int64_t* cap_units, int64_t* units_bytes, int64_t* dirty_bytes,
                           int64_t* tile_sums_bytes, int64_t* tile_prefix_bytes);
/* Size of ddn_fuse_merge_peers' scratch for a session of cap_units units, n_ranks ranks and an output capacity of
 * cap_out voxels (= the most records this rank can receive). */
DDN_API int ddn_fuse_merge_scratch_bytes(int64_t cap_units, int32_t n_ranks, int64_t cap_out, int64_t* bytes_out);
/* Once after allocation (and after any error): clears units and flags. */
DDN_API int ddn_fuse_session_reset(const ddn_fuse_session* s, void* stream);
/* Opens a step: grid from the n_boxes (<= DDN_MAX_PEERS) bounding boxes bbox_ptrs_host[i] (HOST array of
 * device pointers to [6] encoded boxes), occupancy cleared, counts zeroed. */
DDN_API int ddn_fuse_begin(const ddn_fuse_session* s, const void* const* bbox_ptrs_host, int32_t n_boxes, float voxel,
                   void* stream);
/* Same with a grid chosen on the host. */
DDN_API int ddn_fuse_begin_grid(const ddn_fuse_session* s, const ddn_voxel_grid* grid_host, void* stream);
/* Stand-alone mark pass for points that did not come out of ddn_backproject_filter(mark = s). */
DDN_API int ddn_fuse_mark_points(const ddn_fuse_session* s, int64_t n_points, const float* xyz, const uint8_t* votes,
                         int32_t vote_threshold, void* stream);
/* N5, sparse-cloud merge with de-duplication (SURVEY.md 8a row N5; the reference only concatenates,
 * scripts/test.py:353-359): clears the occupancy of every cell that holds one of the given points (xyz [N,3]
 * f32, e.g. the COLMAP sparse cloud), so no dense voxel is created there and the points that fell into it do
 * not participate.  Call between the mark and ddn_fuse_finish*. */
DDN_API int ddn_fuse_unmark_points(const ddn_fuse_session* s, int64_t n_points, const float* xyz, void* stream);
/* Rank + accumulate + finalise of the marked points (same xyz / votes / threshold as the mark).  Outputs as
 * ddn_voxel_fuse with capacity cap_out voxels; accum: scratch of cap_out * 40 bytes, 16-byte aligned. */
DDN_API int ddn_fuse_finish(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz,
                    const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold, uint64_t* out_keys,
                    float* out_xyz, uint8_t* out_rgb, int32_t* out_count, int64_t cap_out, void* accum,
                    int64_t accum_bytes, void* stream);
/* Rank + accumulate into partial RECORDS [cap_records, DDN_RECORD_WORDS] (keys ascending) and, when the session
 * has one, the tile prefix. */
DDN_API int ddn_fuse_finish_partial(const ddn_fuse_session* s, int64_t n_points, int64_t row_len, const float* xyz,
                            const uint8_t* rgb, const uint8_t* votes, int32_t vote_threshold, uint64_t* records,
                            int64_t cap_records, void* stream);
/* Owner-side exchange + merge over PEER MEMORY (NVLink loads inside the kernels, no host plan).  Every rank calls
 * it after all ranks finished ddn_fuse_finish_partial on the same grid (the caller provides that barrier).
 * peer_*_host: HOST arrays of n_ranks device pointers - every rank's records and tile_prefix as mapped into this
 * process (entry `rank` = the local buffers).  The ranks split the tiles that hold records into n_ranks contiguous
 * ranges balancing the global record count (each computes the same cuts from the summed prefixes, which it first
 * copies into local memory in one bulk pass); this rank pulls its share of every rank's sorted records ONCE -
 * coalesced 512-byte requests, peers visited in rotated order - into local staging, setting the occupancy bit of
 * every record on the way, then ranks the occupancy of its range, adds the staged records and finalises.
 * plan: device scratch [64] i64 (out: [0],[1] = tile range, [2] = records received); scratch: device,
 * ddn_fuse_merge_scratch_bytes, 16-byte aligned.  drop_xyz [n_drop,3] f32 (optional, n_drop = 0: none): N5 at the
 * owner - the cells of these points (ALL ranks' sparse points) leave the merged occupancy before it is ranked.
 * Outputs as ddn_fuse_finish.  The rank-ordered concatenation of the outputs is globally key-sorted. */
DDN_API int ddn_fuse_merge_peers(const ddn_fuse_session* s, int32_t rank, int32_t n_ranks, const void* const* peer_records_host,
                         const void* const* peer_tile_prefix_host, int64_t* plan, void* scratch, int64_t scratch_bytes,
                         const float* drop_xyz, int64_t n_drop, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                         int32_t* out_count, int64_t cap_out, void* accum, int64_t accum_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 4 for grids too large for the session's occupancy bitmap: the HASHED PATH (one GPU).  Memory is sized by
 * the points of a step, not by the volume of its box.  An open-addressing table of canonical keys gives every
 * occupied cell a dense voxel index while the points are accumulated (one pass); the voxel keys are then radix-sorted
 * with a count read from device memory and finalised in key order.  Outputs are those of ddn_fuse_finish on the same
 * grid, bit for bit.  A step enqueues ddn_fuse_finish and then ddn_fuse_finish_hashed(mode 0) on the same outputs:
 * whichever path the device grid selects runs, the other returns at once, and nothing is read back.
 * ------------------------------------------------------------------------------------------ */
#define DDN_HASH_STATE_BYTES 64

struct ddn_hash_fuse { /* HOST struct of DEVICE pointers, owned by the caller; sizes from ddn_hash_fuse_sizes */
  void* table;           /* [cap_slots] u64 keys (all bits set = empty), then [cap_slots] u32 voxel indices */
  uint32_t* slots;       /* [cap_voxels] the table slot of every voxel, at the index of the point that created it
                            (and of every tombstone, from the top); all bits set = unused */
  void* sort;            /* [2, cap_voxels] u64 compact keys, then (256-byte aligned) [2, cap_voxels] u32 indices */
  uint32_t* hist;        /* radix histograms */
  int64_t* state;        /* DDN_HASH_STATE_BYTES: [0] 1 = the path ran this step, [1] 1 = table overflow (the step's
                            voxels are incomplete), [2] tombstones */
  int64_t cap_slots;     /* table slots: 2 x the next power of two >= cap_voxels, at least 64 */
  int64_t cap_voxels;    /* the most points (+ dedup points) one step may pass */
};

/* Buffer sizes (bytes) for steps of up to cap_voxels points + dedup points; the table then never gets more than half
 * full, so it cannot overflow. */
DDN_API int ddn_hash_fuse_sizes(int64_t cap_voxels, int64_t* cap_slots, int64_t* table_bytes, int64_t* slots_bytes,
                        int64_t* sort_bytes, int64_t* hist_bytes);
/* Once after allocation (and after any error): empties the table and the slot list and clears the state.  Every step
 * leaves them empty again (it clears the entries it used). */
DDN_API int ddn_hash_fuse_reset(const struct ddn_hash_fuse* hash, void* stream);
/* Fusion of the points of a session step through the hash table.  mode 0: runs only when the session's grid is
 * DDN_GRID_TOO_LARGE (which it rewrites to DDN_GRID_HASHED) or HASHED; mode 1: on any grid with valid dims (tests
 * compare it with the dense path on one grid).  When it runs it resets counts and fills them itself: [0] = points
 * that pass the vote and fall inside the grid (what K4's mark counts), [1] = voxels.  dedup_xyz [n_dedup,3] f32
 * (optional): N5 as ddn_fuse_unmark_points - no voxel in the cells of these points, whose points still count in
 * counts[0].  Needs n_points + n_dedup <= hash->cap_voxels.  accum: max(cap_out, n_points) * 40 bytes (a voxel's
 * accumulator is indexed by the point that created it).  Other arguments and outputs as ddn_fuse_finish. */
DDN_API int ddn_fuse_finish_hashed(const ddn_fuse_session* s, const struct ddn_hash_fuse* hash, int32_t mode, int64_t n_points,
                           int64_t row_len, const float* xyz, const uint8_t* rgb, const uint8_t* votes,
                           int32_t vote_threshold, const float* dedup_xyz, int64_t n_dedup, uint64_t* out_keys,
                           float* out_xyz, uint8_t* out_rgb, int32_t* out_count, int64_t cap_out, void* accum,
                           int64_t accum_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * The HASHED PATH on several GPUs (one process per GPU, peer memory as for ddn_fuse_merge_peers).  A step enqueues
 *   ddn_fuse_finish_partial, ddn_fuse_finish_hashed_partial(mode 0) -> barrier -> ddn_fuse_merge_peers,
 *   ddn_fuse_merge_hashed_peers
 * on the same outputs; whichever path the device grid selects runs, the other returns at once.  The rank-ordered
 * concatenation of the owners' outputs equals ddn_fuse_finish_hashed on one GPU over all points, bit for bit.
 * ------------------------------------------------------------------------------------------ */
#define DDN_HASH_SAMPLES 4096
/* Hashed fusion of this rank's points into sorted partial RECORDS (DDN_RECORD_WORDS u64 each, keys ascending, as
 * ddn_voxel_partials) and SAMPLES [DDN_HASH_SAMPLES + 1] u64: the keys of records floor(i M / DDN_HASH_SAMPLES) for
 * i < DDN_HASH_SAMPLES, then the record count M.  Both in peer-visible memory; other ranks read them in their merge
 * (after the caller's barrier) until this rank's next step.  mode, dedup_xyz (N5: applied on every rank, pass ALL
 * ranks' sparse points) and the other point arguments as ddn_fuse_finish_hashed.  counts[0] = the rank's points that
 * pass the vote and fall inside the grid (their sum over the ranks is the one-GPU count), counts[1] = M.  Needs
 * n_points + n_dedup <= hash->cap_voxels; records: cap_records >= n_points, 16-byte aligned; accum: n_points * 40
 * bytes, 16-byte aligned. */
DDN_API int ddn_fuse_finish_hashed_partial(const ddn_fuse_session* s, const struct ddn_hash_fuse* hash, int32_t mode, int64_t n_points,
                                   int64_t row_len, const float* xyz, const uint8_t* rgb, const uint8_t* votes,
                                   int32_t vote_threshold, const float* dedup_xyz, int64_t n_dedup, uint64_t* records,
                                   int64_t cap_records, uint64_t* samples, void* accum, int64_t accum_bytes, void* stream);
/* Size of ddn_fuse_merge_hashed_peers' scratch for n_ranks ranks and an output capacity of cap_out voxels. */
DDN_API int ddn_fuse_merge_hashed_scratch_bytes(int32_t n_ranks, int64_t cap_out, int64_t* bytes_out);
/* Owner-side merge of the hashed partials over PEER MEMORY; runs when this rank's ddn_fuse_finish_hashed_partial ran
 * (same hash buffers), returns at once otherwise.  peer_*_host: HOST arrays of n_ranks device pointers - every rank's
 * records and samples as mapped into this process.  Every rank derives the same n_ranks - 1 splitter keys from all
 * samples (copied into local memory in one bulk pass): an owner's share of T records in all is at most
 * T / n_ranks + 2 (T / DDN_HASH_SAMPLES + n_ranks) records, so cap_out >= n_max + ceil(2 n_ranks n_max /
 * DDN_HASH_SAMPLES) + 2 n_ranks, n_max = the most points of any rank, cannot overflow (a status word reports it
 * anyway: ddn_hash_fuse.state[1]).  This rank pulls its share of every rank's records once - coalesced 512-byte
 * requests, peers in rotated order - adds the copies of every key through its hash table and finalises.  Needs
 * cap_out <= hash->cap_voxels.  plan: device scratch [64] i64 in ddn_fuse_merge_peers' layout, with [0], [1] = the
 * owned key range [begin, end) (end -1: unbounded), [2] = records received, [3] = records of all ranks.  scratch:
 * ddn_fuse_merge_hashed_scratch_bytes, 16-byte aligned.  counts[0] keeps the rank's own points (-1 when a merged
 * voxel holds 2^24 or more points), counts[1] = the voxels of this rank's range.  Outputs as ddn_fuse_finish; the
 * rank-ordered concatenation of the outputs is globally key-sorted. */
DDN_API int ddn_fuse_merge_hashed_peers(const ddn_fuse_session* s, const struct ddn_hash_fuse* hash, int32_t rank, int32_t n_ranks,
                                const void* const* peer_records_host, const void* const* peer_samples_host, int64_t* plan,
                                void* scratch, int64_t scratch_bytes, uint64_t* out_keys, float* out_xyz, uint8_t* out_rgb,
                                int32_t* out_count, int64_t cap_out, void* stream);

/* Stand-alone pieces of stage 4 (used by the multi-GPU path and by tests). */
DDN_API int ddn_voxel_keys(const ddn_voxel_grid* grid_host, int64_t n_points, const float* xyz,
                   uint64_t* keys, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DDN_B200_H_ */
