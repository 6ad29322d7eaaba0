/*
 * g2pc.h — C ABI of libg2pc.so: B200-native (sm_100a) kernels for the 3DGS-to-PC hot path
 * (per-Gaussian point sampling + Mahalanobis cull, per-camera colour / visibility rasterisation).
 *
 * This is the drop-in boundary.  The reference has two native/op boundaries on this path:
 *   - pybind11 module `gaussian_pointcloud_rasterization._C`
 *       (gaussian-pointcloud-rasterization/ext.cpp:15-17, rasterize_points.cu:36-145, rasterize_points.h:18-46)
 *   - pure-torch call chains for the sampler
 *       (gauss_to_pc.py:140-275, gauss_handler.py:26-63)
 * Both are replaced by the plain-C entry points below.  Conventions (all entry points):
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`; the caller owns all memory,
 *     including scratch (sizes come from the *_bytes query functions or are stated in the comment);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); no allocation, no host
 *     synchronisation and no global mutable state inside the library;
 *   - return value: 0 = G2PC_OK, otherwise an error code; g2pc_last_error() gives a thread-local message;
 *   - no C++ exception crosses the ABI.
 */
#ifndef G2PC_H
#define G2PC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G2PC_OK 0
#define G2PC_ERR_INVALID 1   /* bad argument */
#define G2PC_ERR_CUDA 2      /* a CUDA runtime call / launch failed */
#define G2PC_ERR_WORKSPACE 3 /* caller-provided scratch too small */

#define G2PC_F32 0
#define G2PC_F64 1

/* ---- misc ------------------------------------------------------------------------------------ */
int g2pc_version(void);
const char* g2pc_last_error(void);

/* ---- S1: covariance build ------------------------------------------------------------------- */
/* Replaces build_rotation / build_scaling_rotation / build_covariance_from_scaling_rotation
 * (gauss_handler.py:26-63): R(q) without re-normalisation, L = R*diag(exp(mod*s)), Sigma = L*L^T.
 * scales (n,3) log-space and rots (n,4) in `in_dtype` (the ply loader feeds f64, gauss_dataloader.py:66-80;
 * the elements of R and exp(s) are formed in the input precision and then rounded to f32, as the
 * reference's slice-assignments into float tensors do).  cov: (n,3,3) f32 row-major. */
int g2pc_cov_build(const void* scales, const void* rots, int in_dtype, float scale_modifier,
                   int64_t n, float* cov, void* stream);

/* Replaces Gaussians.calculate_normals (gauss_handler.py:89-106): column argmin(scale) of R(q).
 * normals: (n,3) f32. */
int g2pc_normals(const void* scales, const void* rots, int in_dtype, int64_t n, float* normals,
                 void* stream);

/* Replaces torch.linalg.eigvals(covariances).real on the N x 3 x 3 covariance batch
 * (gauss_handler.py:112 non_posdef_covariances, :259 get_gaussian_magnitudes): eigenvalues of the symmetric part,
 * closed form in f64, rounded to f32, ascending.  eigvals: (n,3) f32.  The callers keep the reference's
 * elementwise f32 chains (ellipsoid area, <= epsilon tests) in torch. */
int g2pc_eigvals_sym3(const float* cov, int64_t n, float* eigvals, void* stream);

/* ---- S2: sampling + Mahalanobis cull --------------------------------------------------------- */
/* Replaces sample_from_multivariate_normal + mahalanobis + create_new_gaussian_points +
 * the bin loop of generate_pointcloud (gauss_to_pc.py:92-103,140-371) and
 * torch.distributions.MultivariateNormal (Cholesky + loc + L*eps).
 *
 * Work is described by host-built tables (the reference builds the same bins on the host,
 * gauss_to_pc.py:308-343):
 *   tile  = <=256/lpg consecutive Gaussians (in bin order) of one bin, all drawing k samples per attempt
 *   unit  = one contiguous span of the output, in the reference's output order:
 *           the centre points of a bin, or the samples one tile emits in one attempt.            */
typedef struct {
    int32_t j0;    /* first Gaussian (bin-order index) */
    int32_t count; /* Gaussians in the tile (<= 256/lpg) */
    int32_t k;     /* samples drawn per Gaussian per attempt = bin's points-per-Gaussian - 1 */
    int32_t lpg;   /* threads cooperating on one Gaussian: power of two, 1..256 */
} g2pc_tile_t;

typedef struct {
    int32_t attempt; /* >=0: sample unit of that attempt; -1: centre-point unit */
    int32_t j0;      /* first Gaussian (bin-order index) */
    int32_t count;   /* Gaussians covered */
    int32_t k;       /* samples per Gaussian per attempt (0 for centre units) */
} g2pc_unit_t;

#define G2PC_CULL_EPS_NORM 0 /* accept iff |eps| <= std (exact-arithmetic identity of the reference test) */
#define G2PC_CULL_EXPLICIT 1 /* accept iff sqrt(d^T Sigma^-1 d) <= std, d = mu - x, fp32 (gauss_to_pc.py:92-103) */

/* status words written by g2pc_sample_count (int32 each) */
#define G2PC_ST_OVERFLOW 0  /* !=0: some Gaussian emitted in an attempt >= attempts_stored (re-run with more) */
#define G2PC_ST_CHOLFAIL 1  /* number of Gaussians whose covariance had no Cholesky factor even after +2e-6*I */
#define G2PC_ST_CHOLREG 2   /* number of Gaussians that needed +1e-6*I or +2e-6*I (gauss_to_pc.py:147-155) */
#define G2PC_ST_WORDS 4

/* Pass 1.  For every tile: gather the tile's Gaussians through `perm`, factor Sigma (closed-form
 * Cholesky), write one 64-byte record per Gaussian in bin order, then simulate the attempt loop of
 * create_new_gaussian_points: draw k samples per unfinished Gaussian with Philox4x32-10
 * (key = seed, counter = (gid, sample, attempt, call_id)) + Box-Muller, count the accepted ones,
 * m = min(k - added, count), and write the tile-local exclusive prefix of m
 * (xl[attempt*n + j]) and the tile total (tile_totals[tile*attempts_stored + attempt]).
 *   xyz (N,3) f32 · cov (N,3,3) f32 · colours (N,3) colour_dtype · normals (N,3) f32 or NULL
 *   perm (n,) int32: bin-order index -> row of the input arrays;  the RNG is keyed by the global Gaussian id
 *   gids[row] (uint32 per input row; survives culls and sharding) or, if gids is NULL, row + gid_offset
 *   records: n*64 bytes, 16-byte aligned · xl: attempts_stored*n uint32 · tile_totals: num_tiles*attempts_stored
 *   uint32, MUST be zero-filled by the caller · status: G2PC_ST_WORDS int32, zero-filled by the caller. */
int g2pc_sample_count(const float* xyz, const float* cov, const void* colours, int colour_dtype,
                      const float* normals, const int32_t* perm, const uint32_t* gids, int64_t gid_offset, int64_t n,
                      const g2pc_tile_t* tiles, int32_t num_tiles, int32_t num_attempts,
                      int32_t attempts_stored, float mahalanobis_std, int32_t cull_mode, uint64_t seed,
                      uint32_t call_id, void* records, uint32_t* xl, uint32_t* tile_totals,
                      int32_t* status, void* stream);

/* Pass 2.  Load-balanced expansion over OUTPUT points: point p belongs to unit u (unit_base[u] <= p <
 * unit_base[u+1], unit_base = exclusive prefix sum of the unit lengths, num_units+1 int64 entries, built by the
 * caller from tile_totals); inside a sample unit the Gaussian and sample index come from a search of xl;
 * eps is regenerated from the counter and x = mu + L*eps written ("first m samples of the block",
 * gauss_to_pc.py:247-258).  Outputs: out_xyz (capacity,3) f32; out_rgb / out_nrm (capacity,3) in out_dtype
 * (out_nrm may be NULL).  The launch covers `capacity` points in chunks of C = g2pc_sample_emit_chunk_points();
 * threads beyond unit_base[num_units] exit.  chunk_unit (optional, ceil(capacity/C)+1 int32): index of the unit holding
 * output point c*C (last u with unit_base[u] <= c*C, clamped to num_units - 1) — saves the per-CTA search. */
int g2pc_sample_emit_chunk_points(void); /* output points per CTA of g2pc_sample_emit (chunk size of chunk_unit) */
int g2pc_sample_emit(const void* records, const uint32_t* xl, int64_t n, const g2pc_unit_t* units,
                     const int64_t* unit_base, const int32_t* chunk_unit, int32_t num_units, uint64_t seed,
                     uint32_t call_id,
                     float* out_xyz, void* out_rgb, void* out_nrm, int out_dtype, int64_t capacity,
                     void* stream);

/* The standard-normal draws the sampler uses: eps[s, i, :] for sample s < k of Gaussian gids[i] in `attempt`
 * — the (k, n', 3) tensor torch's MultivariateNormal.rsample would have drawn (gauss_to_pc.py:149).
 * Used to inject the kernel's random stream into the reference/oracle for parity tests. */
int g2pc_dump_eps(const int64_t* gids, int64_t n_gids, int32_t k, int32_t attempt, uint64_t seed,
                  uint32_t call_id, float* eps, void* stream);

/* ---- N4 / N1: culls and point budget (s8_cull.cu) ----------------------------------------------------------------- */
/* Fused cull + compaction.  Replaces the mask chain of gauss_to_pc.py:483-496 and Gaussians.filter_gaussians
 * (gauss_handler.py:171-193: one boolean-index pass and one host sync per array).  keep(i) = lo <= i < hi
 * && max_contrib[i] > vis_threshold && opacity[i] > min_opacity && bbox_min < xyz[i] < bbox_max (open box)
 * && surface_dist[i] < *surface_threshold_dev && extra_mask[i]; every criterion whose array is NULL is skipped
 * (bbox_*_host: 3 host floats or NULL).  index: ascending row numbers of the kept Gaussians (capacity n int32);
 * count: one int64 in device memory.  workspace: g2pc_cull_workspace_bytes(n). */
int64_t g2pc_cull_workspace_bytes(int64_t n);
int g2pc_cull_select(const float* max_contrib, float vis_threshold, const float* opacity, float min_opacity,
                     const float* xyz, const float* bbox_min3_host, const float* bbox_max3_host,
                     const float* surface_dist, const float* surface_threshold_dev, const uint8_t* extra_mask,
                     int64_t lo, int64_t hi, int64_t n, int32_t* index, int64_t* count, void* workspace,
                     int64_t workspace_bytes, void* stream);
/* dsts[a][r, :] = srcs[a][index[r], :] for r < m, rows of row_bytes[a] bytes (multiples of 4); srcs / dsts / row_bytes
 * are HOST arrays of num_arrays entries (device pointers inside). */
int g2pc_gather_rows(const int32_t* index, int64_t m, int32_t num_arrays, const void* const* srcs, void* const* dsts,
                     const int32_t* row_bytes, void* stream);

/* Magnitudes and point budget without a host round trip: magnitudes[i] (float64) = sqrt(ellipsoid area of Sigma_i,
 * p = 1.6075) * contrib[i] (gauss_handler.py:252-279, float32 chain, closed-form eigenvalues), ppg[i] (int32) =
 * round-half-even(magnitude * num_points / sum) with the first min(deficit, #zeros) zero entries raised to 1
 * (gauss_to_pc.py:73-90; the sum is reduced in a fixed order: bit-identical re-runs). */
int64_t g2pc_ppg_workspace_bytes(int64_t n);
int g2pc_points_per_gaussian(const float* cov, const float* contrib, int64_t n, double num_points, double* magnitudes,
                             int32_t* ppg, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- point-cloud cleaning: statistical outlier removal (s9_knn.cu) ------------------------------------------------- */
/* Replaces Open3D's PointCloud.remove_statistical_outlier (mesh_handler.py:89-94, nb_neighbors = k).
 * avg[i] (n float64) = mean Euclidean distance of point i to its k nearest points of the cloud, itself included (all n
 * points when n < k); exact kNN over xyz (n,3) f32 through a Morton-ordered bucket tree, distances recomputed in float64.
 * A point with a non-finite coordinate gets avg = NaN.  1 <= k <= 32, n < 2^31.  workspace: g2pc_knn_workspace_bytes(n,
 * k), 256-byte aligned (0 for invalid arguments). */
int64_t g2pc_knn_workspace_bytes(int64_t n, int32_t k);
int g2pc_knn_mean_distance(const float* xyz, int64_t n, int32_t k, double* avg, void* workspace, int64_t workspace_bytes,
                           void* stream);
/* mean = sum of avg over avg > 0, divided by n; std = sqrt(sum over avg > 0 of (avg - mean)^2 / (n - 1)); threshold =
 * mean + std_ratio * std (fixed-order float64 reductions: bit-identical re-runs).  keep[i] (n uint8) = 0 < avg[i] <
 * threshold.  stats4 (4 float64, device) = {mean, std, threshold, number of non-finite avg}.  std_ratio > 0.
 * Compact with g2pc_cull_select(extra_mask = keep) + g2pc_gather_rows.  workspace: g2pc_outlier_workspace_bytes(n),
 * 8-byte aligned. */
int64_t g2pc_outlier_workspace_bytes(int64_t n);
int g2pc_outlier_mask(const double* avg, int64_t n, double std_ratio, uint8_t* keep, double* stats4, void* workspace,
                      int64_t workspace_bytes, void* stream);

/* ---- S3-S6: colour stage, renderer_type=python semantics (gauss_render.py:101-465) ------------------------------ */
/* Replaces GaussPythonRenderer.__call__/render (gauss_render.py:266-465) and — as the native op boundary — the role
 * of _C.rasterize_gaussians (rasterize_points.cu:36-145) in the per-camera loop of gauss_to_pc.py:437-454.
 * One camera (a "frame") = preprocess -> depth_sort -> build_tree -> multisplit -> blend -> accumulate
 * (-> compose_image).  No call waits for the device: every size the later stages need is read from the device-side
 * frame header; a frame that does not fit the caller's buffers poisons the header (see G2PC_HDR_POISON). */
typedef struct {
    float view[16];  /* world_view_transform, row-vector convention p_view = [p,1] * V (camera_handler.py:46), row-major */
    float proj[16];  /* projection_matrix as stored by Camera (already transposed, camera_handler.py:48), row-major */
    float campos[3]; /* camera centre (SH view directions) */
    float tan_fovx, tan_fovy, focal_x, focal_y;
    int32_t width, height;
} g2pc_camera_t;

typedef struct {
    int32_t r0, c0, w, h;    /* first row / column and size of the leaf tile in pixels */
    int32_t inst_begin;      /* offset of the leaf's list in inst_gid */
    int32_t inst_count;      /* Gaussians whose rect overlaps the leaf */
    int32_t pix_offset;      /* offset of the leaf's pixels in the concatenated leaf-colour buffer */
    int32_t node;            /* index of the quadtree node */
} g2pc_leaf_t;

#define G2PC_MAX_LEVELS 12
/* frame header (int32 words, device memory, written by g2pc_build_tree) */
#define G2PC_HDR_NUM_LEAVES 0
#define G2PC_HDR_TOTAL_INST 1     /* sum of the leaves' instance counts, low word */
#define G2PC_HDR_TOTAL_PIX 2
#define G2PC_HDR_NEED_DEEPER 3    /* a tile at the deepest tabulated level still has to split: tabulate more levels */
#define G2PC_HDR_LEAF_OVERFLOW 4  /* more leaves than max_leaves */
#define G2PC_HDR_CAP_OVERFLOW 5   /* instance / leaf-pixel / multisplit-matrix capacity too small for this frame */
#define G2PC_HDR_POISON 6         /* snapshot of the shared failure word at the end of this frame's build_tree: 0 = no
                                     frame has failed, else 1 + the LOWEST frame number that did not fit */
#define G2PC_HDR_FRAME 7          /* frame number of the header's contents */
#define G2PC_HDR_TOTAL_INST_HI 8
#define G2PC_HDR_WORDS 16
#define G2PC_WORK_COUNTERS 4      /* int32 work-distribution counters cleared by g2pc_build_tree */
/* device-side statistics (uint64 words, accumulated by g2pc_blend when `stats` is not NULL) */
#define G2PC_STAT_WARP_GAUSSIANS 0  /* (warp, Gaussian) iterations executed: x 128 = (pixel, Gaussian) pairs */
#define G2PC_STAT_WORDS 4

/* The failure word `fail` (one uint32 in device memory, shared by the frames in flight, initialised to 0xFFFFFFFF):
 * build_tree lowers it to 1 + frame when the frame does not fit; build_tree, multisplit and blend of frame f do nothing
 * iff f + 1 >= *fail.  Frames may be enqueued on two streams (the front-end of frame f + 1 overlaps the blend of frame
 * f), so a later frame can fail first: earlier frames still complete.  The caller resets the word after growing its
 * buffers and replays from the failed frame. */

/* Quadtree tables (host-built, g2pc/quadtree.py): `tables` = 6 int32 arrays of n1 = 2^num_levels - 1 entries each,
 * concatenated: x start, x end (inclusive), x flags, y start, y end, y flags; level l at offset 2^l - 1.
 * 2-D node index = (4^l - 1)/3 + iy * 2^l + ix.  level_mask: bit l set iff level l has nodes small enough to be
 * leaves.  clean_mask: bit l set iff level l has no dropped / degenerate node on either axis (then the membership of
 * an interval is exactly its looked-up node range and the kernels skip the per-node table checks). */

/* Once per renderer: geom (n x 48 bytes, 16-byte aligned) = {x,y,z,S00} {S01,S02,S11,S12} {S22,log2(opacity),0,0}
 * from xyz (n,3), cov (n,3,3), opacity (n) — the coalesced 16-byte-load form the per-camera kernel reads. */
int g2pc_pack_geometry(const float* xyz, const float* cov, const float* opacity, int64_t n, void* geom, void* stream);

/* S3.  Per Gaussian: projection (projection_ndc, gauss_render.py:151-168), EWA covariance (build_covariance_2d
 * :101-148), radius / rect (:171-193), conic = inverse(cov2d) (:349) pre-scaled by -0.5*log2(e), colour (given, or SH
 * deg <= 3 evaluated towards the camera: eval_sh :43-99 + 0.5, clamped at 0), and tile-membership counting on the
 * leaf-candidate levels.  colours (n,3) f32 or NULL · shs (n,3,sh_stride) f32 channel-major or NULL.
 * proj: n x 48 bytes (3 float4: {mx,my,c00',c01'} {c11',log2(opacity),r,g} {b,depth,radius,valid}).
 * node_cnt: one uint32 per 2-D node, zero on entry (g2pc_build_tree clears it again).  depth_key (n) uint32:
 * bits(-z_view), 0xFFFFFFFF if behind the camera.  val (n) uint64: (node range at the first candidate level, 8 bits per
 * bound: xlo | xhi<<8 | ylo<<16 | yhi<<24) << 32 | Gaussian index.
 * luts (uint16, 4-byte aligned): per level [x lo (W)][x hi+1 (W)][y lo (H)][y hi+1 (H)] — node range of an interval as
 * a lookup over pixel coordinates, lo[floor(min)] .. hi1[ceil(max)] - 1 (g2pc/quadtree.py QuadtreeTables.pixel_luts). */
int g2pc_preprocess(const void* geom, const float* colours, const float* shs, int32_t sh_stride, int32_t sh_degree,
                    int64_t n, const g2pc_camera_t* cam_host, const int32_t* tables, const uint16_t* luts,
                    int32_t num_levels, uint32_t level_mask, uint32_t clean_mask, void* proj, uint32_t* node_cnt,
                    uint32_t* depth_key, uint64_t* val, void* stream);

/* S4a.  val_sorted[k] = val of the k-th nearest Gaussian (stable radix sort of depth_key: ties keep index order, the
 * reference's torch.sort is unstable there, gauss_render.py:340-344).  cub::DeviceRadixSort (library call). */
int64_t g2pc_depth_sort_workspace_bytes(int64_t n);
int g2pc_depth_sort(const uint32_t* depth_key, const uint64_t* val, int64_t n, uint64_t* val_sorted, void* workspace,
                    int64_t workspace_bytes, void* stream);

/* S4b.  Resolve the quadtree (one CTA): node states, node_leaf (int32 per node: leaf id, -1 none, -2 split), leaves in
 * the reference's BFS order with list / pixel offsets, leaf_order (heaviest leaf first, the blend's launch order), the
 * frame header; clears node_cnt and work_counters.  inst_capacity (uint32 ids) / pix_capacity (pixels) /
 * matrix_capacity (uint32 words, >= ms_chunks * leaves): sizes of the caller's buffers, checked here. */
int g2pc_build_tree(const int32_t* tables, int32_t num_levels, int32_t max_gaussians_per_tile, uint32_t* node_cnt,
                    uint8_t* node_state, int32_t* node_leaf, g2pc_leaf_t* leaves, int32_t* leaf_order,
                    int32_t max_leaves, int64_t inst_capacity, int64_t pix_capacity, int64_t matrix_capacity,
                    int32_t ms_chunks, int32_t frame, int32_t* header, uint32_t* fail, int32_t* work_counters,
                    void* stream);

/* S4c.  Stable multisplit of the depth-ordered stream into the leaves' lists: inst_gid[leaf.inst_begin ..
 * + leaf.inst_count) = Gaussian ids overlapping the leaf, nearest first.  Three kernels (count, scan, scatter) over
 * chunks of C = g2pc_multisplit_chunk(leaf_cap) sorted entries; matrix: g2pc_multisplit_rows(n, leaf_cap) x leaves
 * uint32 scratch (pass that row count as ms_chunks to g2pc_build_tree, which checks the capacity).
 * leaf_cap = max_leaves given to g2pc_build_tree. */
int32_t g2pc_multisplit_chunk(int32_t leaf_cap);
int32_t g2pc_multisplit_rows(int64_t n, int32_t leaf_cap); /* rows of `matrix` needed (chunks + one per persistent CTA) */
int g2pc_multisplit(const uint64_t* val_sorted, int64_t n, const void* proj, int32_t width, int32_t height,
                    const int32_t* tables, int32_t num_levels, uint32_t level_mask, uint32_t clean_mask,
                    const int32_t* node_leaf, const g2pc_leaf_t* leaves, const int32_t* header, const uint32_t* fail,
                    int32_t frame,
                    int32_t leaf_cap, uint32_t* matrix, uint32_t* inst_gid, void* stream);

/* S5.  Front-to-back blend of every leaf (gauss_render.py:337-369) + per-Gaussian maximum contribution / arg-max pixel
 * (:371-385) published as cam_best[g] = max((bits(contribution) << 32) | ~leaf_pixel_index).
 * The leaf count comes from `header` (device).  max_leaf_pixels_quads: upper bound of ceil(w/4)*h over the leaves.
 * max_contrib (n) f32: the running maxima of the earlier cameras (read-only here; contributions that cannot beat
 * them skip the bookkeeping).  leaf_colour: (pix_capacity,3) f32.  owner: uint32 per image pixel (zero on entry):
 * 1 + index of the last leaf pixel covering it.  work_counters: cleared by g2pc_build_tree (persistent CTAs pull
 * (leaf, slab) items, heaviest leaf first).
 * t_stop: a warp stops walking its leaf's list once ALL of its 128 pixels have transmittance T < t_stop; every
 * contribution it skips is then < t_stop and their sum per pixel is < t_stop.  t_stop = 0 selects FLT_MIN (only
 * contributions that underflow are dropped: the strict-parity setting); the reference's CUDA back-end stops each pixel
 * at T < 1e-4 (forward.cu:415).  stats: G2PC_STAT_WORDS uint64 or NULL. */
int g2pc_blend(const g2pc_leaf_t* leaves, const int32_t* leaf_order, const int32_t* header, const uint32_t* fail,
               int32_t frame, int32_t max_leaf_pixels_quads, const uint32_t* inst_gid, const void* proj, uint64_t* cam_best,
               const float* max_contrib, float* leaf_colour, uint32_t* owner, int32_t width, int32_t height,
               float background, float t_stop, int32_t* work_counters, uint64_t* stats, void* stream);

/* Pixel-to-thread mapping of g2pc_blend: 1 (default) = a warp owns a compact block of <= 32 quads (e.g. 20 x 6 pixels),
 * 0 = a warp owns a strip of full rows.  Results do not depend on it up to the t_stop tolerance. */
void g2pc_blend_set_compact(int on);

/* S6.  Fold one camera into the per-Gaussian accumulators (gauss_render.py:387-395; the role of
 * GaussianRasterizer.update_max_contributions, gaussian_pointcloud_rasterization/__init__.py:142-152):
 * where the camera's best contribution beats max_contrib[g] (strict >) store it and the blended colour of the winning
 * pixel.  Clears cam_best.  first_frame (n) int32 or NULL: set to `frame` where the maximum was raised (the multi-GPU
 * merge needs the index of the camera that first reached each maximum, g2pc/dist.py). */
int g2pc_accumulate(uint64_t* cam_best, const float* leaf_colour, int64_t n, float* max_contrib, float* colours,
                    int32_t* first_frame, int32_t frame, void* stream);

/* Rendered image (H,W,3) f32, flipped left-right like the reference (gauss_render.py:402); clears `owner`. */
int g2pc_compose_image(uint32_t* owner, const float* leaf_colour, int32_t width, int32_t height, float background,
                       float* image, void* stream);

/* ---- colour stage, renderer_type=cuda semantics: the reference's CUDA rasterizer restated (16x16 tiles) ---------- */
/* Replaces _C.rasterize_gaussians (gaussian-pointcloud-rasterization/ext.cpp:15-17, rasterize_points.cu:36-145 ->
 * CudaRasterizer::Rasterizer::forward, rasterizer_impl.cu:197-352: preprocessCUDA forward.cu:153-271, duplicateWithKeys /
 * radix sort / identifyTileRanges rasterizer_impl.cu:69-137,285-326, renderCUDA forward.cu:303-497) and the accumulator
 * updates of GaussianRasterizer.forward (gaussian_pointcloud_rasterization/__init__.py:126-158).
 * One camera = tiles_preprocess -> depth_sort -> tiles_build -> multisplit_grid -> tiles_blend -> tiles_accumulate.
 * The depth-ordered lists are built per SUPER-TILE of 2x2 tiles (32x32 pixels; grid SW x SH = ceil(ceil(W/16)/2) x
 * ceil(ceil(H/16)/2)); the blend of a tile walks its super-tile's list and skips the entries whose tile rect (packed into
 * the projection record) does not contain the tile, so every tile sees exactly the reference's per-tile list. */
typedef struct {
    float viewmatrix[16];  /* world->view, row-vector convention, z forward (camera_handler.py:75,91), row-major */
    float projmatrix[16];  /* viewmatrix @ projection (camera_handler.py:100), row-major */
    float campos[3];
    float tan_fovx, tan_fovy;
    int32_t width, height;
} g2pc_raster_t;

/* preprocessCUDA: near cull z_view <= 0.2, EWA covariance + 0.3, conic, radius = ceil(3 sqrt(lambda_max)), tile rect
 * (16x16 tiles), colour given or SH deg <= 3 (sh_layout 0: (n,3,stride) channel-major as the loader yields it,
 * gauss_dataloader.py:42-44; 1: (n,stride,3) coefficient-major as forward.cu:31 reads it).  Outputs as g2pc_preprocess
 * (proj records — the last word holds the packed TILE rect; depth_key = bits(z_view); val = packed SUPER-TILE rect << 32 |
 * index; node_cnt (SW*SH, zeroed by the caller / by tiles_build) = Gaussians per super-tile); radii (n) int32 or NULL. */
int g2pc_tiles_preprocess(const void* geom, const float* colours, const float* shs, int32_t sh_stride,
                          int32_t sh_degree, int32_t sh_layout, int64_t n, const g2pc_raster_t* rs_host, void* proj,
                          uint32_t* node_cnt, uint32_t* depth_key, uint64_t* val, int32_t* radii, void* stream);

/* List table: every super-tile of the SW x SH grid is a leaf (leaf index = super-tile index, row-major; max_leaves >=
 * SW*SH); list offsets, launch order, frame header / poison as g2pc_build_tree; clears node_cnt and work_counters. */
int g2pc_tiles_build(uint32_t* node_cnt, int32_t width, int32_t height, g2pc_leaf_t* leaves, int32_t* leaf_order,
                     int32_t max_leaves, int64_t inst_capacity, int64_t matrix_capacity, int32_t ms_rows, int32_t frame,
                     int32_t* header, uint32_t* fail, int32_t* work_counters, void* stream);

/* g2pc_multisplit over a flat grid (grid_w x grid_h = SW x SH here; the packed range is the rect in grid cells). */
int g2pc_multisplit_grid(const uint64_t* val_sorted, int64_t n, int32_t grid_w, int32_t grid_h,
                         const g2pc_leaf_t* leaves, const int32_t* header, const uint32_t* fail, int32_t frame,
                         int32_t leaf_cap, uint32_t* matrix, uint32_t* inst_gid, void* stream);

/* renderCUDA: per pixel front-to-back blend (power > 0 and alpha < 1/255 skipped, the pixel stops before T < 1e-4),
 * out_color (3,H,W) = C + T*bg, out_depth / out_invdepth (H,W) = sum depth*alpha*T / sum alpha*T/depth, written for
 * pixels inside the image whose mask (H*W int32 or NULL) is non-zero; cam_best[g] = max((bits(alpha*T) << 32) |
 * ~pixel_id) (deterministic arg-max: lowest pixel id among equals); cam_dist (n uint32, pre-filled with the bits of
 * FLT_MAX, or NULL): bits of the minimum surface distance (see s7_tiles.cu header). */
int g2pc_tiles_blend(const g2pc_leaf_t* leaves, const int32_t* leaf_order, const int32_t* header, const uint32_t* fail,
                     int32_t frame, const uint32_t* inst_gid, const void* proj, uint64_t* cam_best, uint32_t* cam_dist,
                     const int32_t* mask, float* out_color, float* out_depth, float* out_invdepth, int32_t width,
                     int32_t height, const float* background3_host, int32_t* work_counters, uint64_t* stats,
                     void* stream);

/* Accumulator update of one camera (__init__.py:128-158): where the camera's contribution beats max_contrib (strict >)
 * store it and the FINAL colour of its arg-max pixel; total_contrib += contribution; min_dist = min(min_dist, cam_dist).
 * Clears cam_best / re-arms cam_dist.  Optional per-camera outputs of the op (n each): cam_contrib f32, cam_pixel i32,
 * cam_surface f32. */
int g2pc_tiles_accumulate(uint64_t* cam_best, uint32_t* cam_dist, const float* out_color, int32_t width, int32_t height,
                          int64_t n, float* max_contrib, float* total_contrib, float* colours, float* min_dist,
                          int32_t* first_frame, int32_t frame, float* cam_contrib, int32_t* cam_pixel,
                          float* cam_surface, void* stream);

int g2pc_fill_u32(uint32_t* v, uint32_t value, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* G2PC_H */
