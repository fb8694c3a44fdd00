/*
 * libdropclip - C ABI of the B200-native DROP-CLIP fusion / grounding path.
 *
 * The reference (gtziafas/DROP-CLIP) is pure Python; it has no native boundary of its own.
 * The drop-in boundary for callers is therefore the Python surface in `drop-clip_b200/`
 * (same names and argument meaning as utils/feature_fusion.py, utils/projections.py and
 * models/similarity.py). This header is the boundary *under* that surface: what the host
 * side binds with ctypes, and what a maintainer of the reference would bind from
 * utils/feature_fusion.py directly (INTEGRATION.md shows the stub). Each entry point names
 * the reference lines it replaces (paths relative to the reference root).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its comment says "host";
 *  - all memory is caller-owned; the library never allocates device memory, never
 *    synchronises and only enqueues work on `stream` (a cudaStream_t);
 *  - scene batches are ragged and described by prefix-offset arrays (CSR style), int64, on
 *    the device; extents that size a launch are passed by value;
 *  - return value: 0 on success, a negative dc_status otherwise; dc_last_error() gives a
 *    thread-local message. No C++ exception crosses the boundary;
 *  - built for sm_100a only; there is no CPU path. Calls fail with DC_ERR_CUDA on any other
 *    device.
 */
#ifndef DROPCLIP_H_
#define DROPCLIP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DC_ABI_VERSION 2
#if defined(__GNUC__)
#define DC_API __attribute__((visibility("default")))
#else
#define DC_API
#endif

typedef void* dc_stream_t; /* cudaStream_t */

enum dc_status {
  DC_OK = 0,
  DC_ERR_INVALID = -1,     /* bad argument */
  DC_ERR_CUDA = -2,        /* CUDA runtime / driver error, wrong architecture */
  DC_ERR_UNSUPPORTED = -3, /* shape or dtype outside what the kernels implement */
  DC_ERR_WORKSPACE = -4    /* workspace too small */
};

enum dc_dtype { DC_F16 = 0, DC_F32 = 1, DC_U8 = 2, DC_I32 = 3, DC_I64 = 4, DC_F64 = 5 };

enum dc_sim_kernel { DC_SIM_NONE = 0, DC_SIM_MAX = 1, DC_SIM_MEAN = 2 };

enum dc_ground_mode {
  DC_GROUND_RAW = 0,    /* sims[n, p] = <x_n, t_p>                         models/similarity.py:49,67 */
  DC_GROUND_PAIRED = 1, /* paired softmax of column 0 against the others   models/similarity.py:51-61 */
  DC_GROUND_ARGMAX = 2, /* pos - mean(neg) and (argmax == 0)               models/similarity.py:91-101 */
  DC_GROUND_CLASS = 3   /* raw sims (optional) + index of the row maximum  engine/distil.py:244-246,289-290 */
};

DC_API int dc_abi_version(void);
DC_API const char* dc_last_error(void);
/* host out-params; any may be NULL */
DC_API int dc_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes);
/* Two-stream mode of the object-level step (engine.FusionEngine.fuse_object_level): when on (the default), the
 * instance-histogram pass of the object branch and the visibility filter of the point branch are shaped to share every
 * SM (dc_seg_histogram takes its bulk-copy ring kernel for large int64 batches, and both kernels ask for the same
 * shared-memory carve-out, because an SM cannot change it while CTAs are resident). Off: each kernel is configured for
 * running alone. Results are identical either way. Process-wide; returns the previous setting. */
DC_API int dc_set_stream_overlap(int on);

/* ------------------------------------------------------------------------------------------
 * (1)+(2) Projection, depth-tolerance visibility and instance-mask lookup.
 * Replaces MultiviewFeatureFusion.get_visibility_mask  utils/feature_fusion.py:81-125, the
 * duplicate in aggregate_features :201-229, transform_pointcloud_to_camera_frame
 * utils/transforms.py:52-61 and the `seg[ys, xs]` lookups tools/preprocess_data.py:395-401.
 *
 * For scene s, view v (global view index g = view_off[s] + v) and point i (global index
 * j = point_off[s] + i) it evaluates, in fp64 with the exact operation order of the
 * reference's BLAS calls (k-ascending fused multiply-add chains):
 *     c  = inv_pose[g][:3,:] . [p;1];  c.y = -c.y;  c.z = -c.z;   q = K[s] . c
 *     (u,v) = trunc(q.x / q.z, q.y / q.z)   (0,0) when q.z == 0
 *     visible = 0<=u<W and 0<=v<H and |double(depth[g][v,u]) - q.z| <= threshold
 * and writes mask[mask_off[s] + v*N_s + i] (uint8 or int64, selected by mask_elem_size).
 * Optional outputs (NULL to skip): any_visible[j] = OR over views; point_object[same layout
 * as mask] = seg[g][v,u] for visible points, -1 otherwise (needs `seg`).
 * The inverse pose is an input (16 fp64 per view, row-major) because the reference inverts with
 * LAPACK on the host in the POSE's dtype (np.linalg.inv, utils/transforms.py:54) and np.dot then promotes an
 * fp32 inverse to fp64 exactly; the host side inverts in the caller's dtype and widens, so fp32 and fp64
 * poses both reproduce the reference bit for bit.
 */
DC_API int dc_project_visibility(const double* points, const int64_t* point_off, const int64_t* view_off,
                          const float* depths, const double* inv_poses, const double* intrinsics,
                          const int64_t* mask_off, int n_scenes, int64_t max_points_per_scene,
                          int max_views_per_scene, int height, int width, double threshold,
                          void* mask, int mask_elem_size, uint8_t* any_visible,
                          const void* seg, int seg_dtype, int32_t* point_object, dc_stream_t stream);

/* Same results as dc_project_visibility, organised for throughput on unordered clouds: points are
 * counting-sorted by a coarse Morton cell per scene so that the depth gathers of a warp fall on a
 * few cache lines, visibility is evaluated in sorted order and bit-packed:
 *   records [ceil(max_views/32)][total_points] uint32, bit (v & 31) of word v/32 at the point's
 *           sorted position;  rank [total_points] = sorted position of each point inside its scene.
 * dc_unpack_visibility expands the records into the (V_s, N_s) mask blocks (mask_elem_size 1 or 8);
 * dc_unpack_visibility_compact writes only the points with any_visible != 0 at their compacted
 * rank (new_index / kept_off from dc_compact_scan, out_off = prefix of V_s * N'_s), i.e. the mask
 * fuse_obj_prior returns (utils/feature_fusion.py:277-281) without materialising the full one.
 * The kernel decides each (point, view) pair from an fp32 evaluation with a proven error bound and
 * re-evaluates the undecided ones (~0.2 %) with the literal fp64 sequence, so results stay bit-identical.
 * Limits: at most 819 views per scene, height * width <= 2^23.
 * workspace: dc_visibility_sorted_workspace(total_points, n_scenes, max_views_per_scene) bytes. */
DC_API size_t dc_visibility_sorted_workspace(int64_t total_points, int n_scenes, int max_views_per_scene);
/* number of filter-kernel launches dc_project_visibility_sorted issues for these extents (launch accounting) */
DC_API int dc_visibility_sorted_groups(int n_scenes, int64_t max_points_per_scene, int max_views_per_scene);
DC_API int dc_project_visibility_sorted(const double* points, const int64_t* point_off, const int64_t* view_off,
                                 const float* depths, const double* inv_poses, const double* intrinsics,
                                 int n_scenes, int64_t total_points, int64_t max_points_per_scene,
                                 int max_views_per_scene, int height, int width, double threshold,
                                 uint32_t* records, int64_t* rank, uint8_t* any_visible, void* workspace,
                                 size_t workspace_bytes, dc_stream_t stream);
/* The counting sort by Morton cell on its own: perm[p0 + s] = scene-local index of the point at sorted position s,
 * rank[p0 + i] = sorted position of point i. Used to give point-major kernels spatially coherent warps
 * (dc_pixel_fuse takes `perm`). The order inside a cell is arbitrary; consumers must not depend on it. */
DC_API size_t dc_spatial_sort_workspace(int n_scenes);
DC_API int dc_spatial_sort(const double* points, const int64_t* point_off, int n_scenes, int64_t total_points,
                    int64_t max_points_per_scene, int64_t* perm, int64_t* rank, void* workspace,
                    size_t workspace_bytes, dc_stream_t stream);
DC_API int dc_unpack_visibility(const uint32_t* records, const int64_t* rank, const int64_t* point_off,
                         const int64_t* view_off, const int64_t* mask_off, int n_scenes, int64_t total_points,
                         int64_t max_points_per_scene, void* mask, int mask_elem_size, dc_stream_t stream);
DC_API int dc_unpack_visibility_compact(const uint32_t* records, const int64_t* rank, const int64_t* point_off,
                                 const int64_t* view_off, const uint8_t* any_visible, const int64_t* new_index,
                                 const int64_t* kept_off, const int64_t* out_off, int n_scenes,
                                 int64_t total_points, int64_t max_points_per_scene, void* out,
                                 int out_elem_size, void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* Optional scratch of dc_unpack_visibility_compact (4 bytes per point for 1-byte masks, else 0): with it the 1-byte
 * masks are written four columns per thread with 32-bit stores; without it (NULL) one byte per store. Same bytes. */
DC_API size_t dc_unpack_compact_workspace(int64_t total_points, int out_elem_size);

/* Per-view instance histogram: counts[g*nbins + id] = #pixels of view g with that id (nbins <= 8192; the host
 * side uses max(256, max Q) so that every id the reference can index has a bin). outside[4*g ..]: [0] #pixels with
 * id >= nbins, [1] #pixels with id < 0, [2] smallest negative id (int64, 0 if none), [3] largest negative id
 * + 2^63 (0 if none). Replaces np.unique(seg) utils/feature_fusion.py:307 and (seg == obj).sum() :320.
 * seg_dtype: DC_U8 / DC_I32 / DC_I64. */
DC_API int dc_seg_histogram(const void* seg, int seg_dtype, int64_t total_views, int64_t pixels_per_view,
                     int nbins, uint32_t* counts, uint64_t* outside, dc_stream_t stream);

/* Binds feature rows to object ids the way the reference's loop does (utils/feature_fusion.py
 * :307,315,333): the ids present in a view, ascending, minus the smallest one; row i of the
 * view's feature block belongs to the i-th remaining id.
 *   feat_off   [total_views+1] first feature row of each view
 *   view_scene [total_views]   scene of each view;   view_off / query_off / wobj_off [n_scenes+1]
 * Outputs: row_object[total_rows] (id or -1), object_row[wobj layout: wobj_off[s] + id*V_s + v]
 * (global row or -1), view_status[total_views] bit0: an id the reference's loop would index lies outside
 * [0,Q_s) (IndexError there; a single distinct negative id, e.g. a -1 background, is the dropped smallest id and
 * is fine), bit1: fewer feature rows than ids (IndexError as well). */
DC_API int dc_view_table(const uint32_t* counts, const uint64_t* outside, const int64_t* feat_off,
                  const int32_t* view_scene, const int64_t* view_off, const int64_t* query_off,
                  const int64_t* wobj_off, int64_t total_views, int64_t total_rows, int64_t total_wobj,
                  int nbins, int32_t* row_object, int32_t* object_row, int32_t* view_status,
                  dc_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (3) Semantic view-informativeness score. Replaces utils/feature_fusion.py:311-313:
 *     sims[r, o] = < feat[r] / |feat[r]| , query[query_off[s] + o] >     r in view g of scene s
 * as one batched tcgen05 GEMM (fp16 operand planes, fp32 accumulate in TMEM; fp32 inputs are
 * split into hi+lo fp16 planes so the result keeps fp32-level accuracy).
 * feats: [total_rows, dim] DC_F16 or DC_F32 (rows of all views stacked; dim % 64 == 0).
 * queries: [total_queries, dim] fp32.  sims: [total_rows, sims_ld] fp32, sims_ld >= 16-aligned
 * max Q_s (use dc_view_score_ld()).
 * workspace: dc_view_score_workspace() bytes, 1024-byte aligned.
 */
DC_API int dc_view_score_ld(int max_queries_per_scene);
DC_API size_t dc_view_score_workspace(int64_t total_rows, int64_t total_queries, int dim, int feat_dtype);
DC_API int dc_view_score(const void* feats, int feat_dtype, int64_t total_rows, int dim, const int64_t* feat_off,
                  const int64_t* view_off, const float* queries, const int64_t* query_off,
                  int64_t total_queries, int n_scenes, int max_queries_per_scene, float* sims, int sims_ld,
                  void* workspace, size_t workspace_bytes, dc_stream_t stream);

/* View weights. Replaces utils/feature_fusion.py:313-331 and calculate_sim :65-73: per view a
 * global min-max normalisation of its sims block, then per bound row
 *     w = clip(sn[obj] - max_{o != obj} sn[o], 1e-6)        (DC_SIM_MAX, or mean for DC_SIM_MEAN)
 * use_visibility writes the pixel count of the object instead; DC_SIM_NONE without visibility
 * writes 1. Similarity overrides visibility like the reference (quirk q8).
 * weight_obj: wobj layout, fp32, must be zero-filled by the caller.
 * Exact weights (feats != NULL, sim_kernel != NONE): for rows whose weight from `sims` is below `refine_below` (pass
 * +inf to re-evaluate every row) `sims` only selects - the positive and the negatives within 1e-5 of the arg-max
 * (all of them for DC_SIM_MEAN) are re-evaluated as fp64 dot products of the normalised feature row with the queries
 * and the weight (s_pos - red(s_neg)) / (max - min) is formed in fp64, so weights next to the 1e-6 clip keep a
 * relative accuracy of ~1e-7 instead of the GEMM's absolute 1e-7. feats [total_rows, dim] as given to dc_view_score,
 * queries [total_queries, dim] fp32, scratch: dc_view_weights_scratch(total_views, total_rows) bytes (4-byte aligned;
 * per-view extrema and the queue of rows to re-evaluate), feats_normalized: for fp16 features the fp16 plane of
 * normalised rows dc_view_score left at the start of its workspace (or NULL: normalised here). */
DC_API size_t dc_view_weights_scratch(int64_t total_views, int64_t total_rows);
DC_API int dc_view_weights(const float* sims, int sims_ld, const int64_t* feat_off, const int32_t* view_scene,
                    const int64_t* view_off, const int64_t* query_off, const int64_t* wobj_off,
                    const int32_t* row_object, const uint32_t* counts, int nbins, int64_t total_views,
                    int sim_kernel, int use_visibility, float* weight_obj, const void* feats, int feat_dtype, int dim,
                    const float* queries, int64_t total_rows, void* scratch, const void* feats_normalized,
                    float refine_below, dc_stream_t stream);

/* (4) Object-level segmented weighted mean over views. Replaces the einsum and division at
 * utils/feature_fusion.py:333-335:  fused[query_off[s]+o, :] = sum_v w[o,v] * feat[row(o,v)] / sum_v w[o,v]
 * (0/0 = NaN for objects seen in no view, quirk q10). fused: [total_queries, dim] fp32. */
DC_API int dc_segmented_wmean(const void* feats, int feat_dtype, int dim, const int32_t* object_row,
                       const float* weight_obj, const int64_t* view_off, const int64_t* query_off,
                       const int64_t* wobj_off, int n_scenes, int max_queries_per_scene, float* fused,
                       dc_stream_t stream);

/* (4) Scatter object features back to points. Replaces reconstruct_per_obj_feat
 * utils/feature_fusion.py:127-136 (skip_first = 1: object 0 and unknown labels give zero rows)
 * and the dataset twin feat[label] data/dataset_blender.py:128-130 (skip_first = 0).
 * labels: [total_points] int64; out: [total_points, dim] fp32. */
DC_API int dc_scatter_to_points(const float* fused, const int64_t* query_off, const int64_t* labels,
                         const int64_t* point_off, int n_scenes, int64_t max_points_per_scene, int dim,
                         int skip_first, float* out, dc_stream_t stream);

/* Stream compaction of never-visible points (utils/feature_fusion.py:277-281, :257-264).
 * new_index[j] = rank of point j among the kept points of the whole batch (exclusive scan of
 * any_visible), kept_off[n_scenes+1] = scene prefix of kept counts. workspace:
 * dc_compact_workspace(total_points) bytes. */
DC_API size_t dc_compact_workspace(int64_t total_points);
DC_API int dc_compact_scan(const uint8_t* any_visible, int64_t total_points, const int64_t* point_off,
                    int n_scenes, int64_t* new_index, int64_t* kept_off, void* workspace,
                    size_t workspace_bytes, dc_stream_t stream);
/* out_off[n_scenes + 1] = prefix of V_s * N'_s (layout of the compacted mask blocks) computed on the device, so a
 * device-resident pipeline needs no host round trip between dc_compact_scan and dc_unpack_visibility_compact. */
DC_API int dc_compact_mask_offsets(const int64_t* kept_off, const int64_t* view_off, int n_scenes, int64_t* out_off,
                            dc_stream_t stream);
/* out[new_index[j]] = in[j] for kept rows of `row_bytes` bytes (points, colours, labels, features). */
DC_API int dc_compact_rows(const void* in, int64_t row_bytes, const uint8_t* any_visible, const int64_t* new_index,
                    int64_t total_points, void* out, dc_stream_t stream);
/* Column compaction of the per-scene (V_s, N_s) masks into (V_s, N'_s) blocks at out_off[s]
 * (out_off = prefix of V_s * N'_s, computed by the caller from kept_off). elem_size 1, 4 or 8;
 * elem_size 18 reads a uint8 mask and writes int64 (the dtype the reference returns). */
DC_API int dc_compact_mask(const void* mask, int elem_size, const int64_t* mask_off, const int64_t* point_off,
                    const int64_t* view_off, const uint8_t* any_visible, const int64_t* new_index,
                    const int64_t* kept_off, const int64_t* out_off, int n_scenes,
                    int64_t max_points_per_scene, int max_views_per_scene, void* out, dc_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Pixel-level fusion. Replaces aggregate_features utils/feature_fusion.py:138-250 and the
 * division in fuse_points :266-268 without materialising the 480x640xC bicubic map: for each
 * visible (point, view) it evaluates the 16 bicubic taps (align_corners=False, A=-0.75) of the
 * patch map at the projected pixel, optionally L2-normalises, scores the feature against all
 * queries to obtain the relative-similarity weight of the pixel's instance id, and accumulates
 * point-major over views.
 *   patch_feats [total_views, ph, pw, dim] fp32;  queries as above (sim_kernel != NONE)
 *   visible     [mask layout] uint8 from dc_project_visibility; pixels recomputed internally
 *   out_sum     [total_points, dim] fp32 (sum of weighted features, = sum_features :243)
 *   out_weight  [mask layout] fp32 similarity weights (similarity_mask :238) or NULL
 *   perm        [total_points] from dc_spatial_sort or NULL: processing order of the points inside a scene
 *               (neighbouring warps then share bicubic taps in L1); results do not depend on it
 *   normalize   1: out_sum holds the final features of fuse_points :266-268 (sums divided by sum_v weight, or by the
 *               number of views that see the point without similarity) - saves the separate dc_pixel_normalize pass
 *   workspace   dc_pixel_fuse_workspace(...) bytes (sim_kernel != NONE): the similarity of an interpolated feature
 *               with a query is linear in the 16 taps, so patch-cell . query dots are computed once per view and
 *               interpolated with the same bicubic weights (then divided by |f| under norm_feat)
 */
DC_API int dc_pixel_fuse(const double* points, const int64_t* point_off, const int64_t* view_off,
                  const double* inv_poses, const double* intrinsics, const int64_t* mask_off,
                  const uint8_t* visible, const void* seg, int seg_dtype, const float* patch_feats, int patch_h,
                  int patch_w, int dim, const float* queries, const int64_t* query_off, int sim_kernel,
                  int norm_feat, int n_scenes, int64_t max_points_per_scene, int max_views_per_scene,
                  int height, int width, const int64_t* perm, float* out_sum, float* out_weight, int normalize,
                  int64_t total_views, int max_queries_per_scene, void* workspace, size_t workspace_bytes,
                  dc_stream_t stream);
/* The same computation on the tensor cores (dim 512 / 768 / 1024): the visible (point, view) pairs are counting-sorted by
 * (view, bicubic footprint), every 128 sorted pairs form a tcgen05 tile D[128 x dim] = sum_segments A_g[128 x 16] . B_g[16 x dim]
 * (A = the pairs' 16 tap weights, B = the footprint's 16 taps, fp16 hi/lo planes for fp32 accuracy), a first pass yields
 * |f| per pair (norm_feat), the similarity weights follow from the (patch cell . query) table in fp64, and the second pass
 * scales each row in the TMEM epilogue and adds it to its point's row (red.global.add.v4.f32: the order of the additions
 * over a point's views is not fixed; results differ from the view-ordered sum by fp32 rounding only).
 * `rank` [total_points] from dc_spatial_sort or NULL: with it the pairs are grouped by Morton-contiguous point regions first, so
 * that the output rows being added to stay resident in L2 (without it the accumulate pass misses L2 on most additions).
 * Arguments as dc_pixel_fuse plus total_points and mask_elems (= mask_off[n_scenes]); out_weight is required when
 * sim_kernel != NONE; workspace 256-byte aligned, dc_pixel_fuse_mma_workspace() bytes. */
DC_API size_t dc_pixel_fuse_mma_workspace(int64_t total_views, int64_t mask_elems, int patch_h, int patch_w, int dim,
                                   int max_queries_per_scene);
DC_API int dc_pixel_fuse_mma(const double* points, const int64_t* point_off, const int64_t* view_off,
                      const double* inv_poses, const double* intrinsics, const int64_t* mask_off,
                      const uint8_t* visible, const void* seg, int seg_dtype, const float* patch_feats, int patch_h,
                      int patch_w, int dim, const float* queries, const int64_t* query_off, int sim_kernel,
                      int norm_feat, int n_scenes, int64_t max_points_per_scene, int max_views_per_scene,
                      int height, int width, const int64_t* rank, float* out_sum, float* out_weight, int normalize,
                      int64_t total_views, int64_t total_points, int64_t mask_elems, int max_queries_per_scene,
                      void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* workspace of dc_pixel_fuse when sim_kernel != NONE: the per-view (patch cell x query) dot table (0 bytes otherwise) */
DC_API size_t dc_pixel_fuse_workspace(int64_t total_views, int patch_h, int patch_w, int max_queries_per_scene);
/* generate_view_clip (data/dataset_blender.py:132-171): out[v, i, :] = bicubic(patch_feats[v])[clip(pixel of point i in view v)].
 * Projection in fp64 with the json world_matrix inverted in fp64 by the caller (utils/transforms.py:52-61), y/z flip,
 * truncation toward zero, pixel (0,0) when the projected z is 0, coordinates clipped into the image (:158-159); no
 * visibility test. inv_poses [n_views,16] fp64, intrinsics [9] fp64 (self.K), patch_feats [n_views, ph, pw, dim] fp32,
 * out [n_views, n_points, dim] fp32. */
DC_API int dc_view_clip_gather(const double* points, int64_t n_points, const double* inv_poses, const double* intrinsics,
                        const float* patch_feats, int n_views, int patch_h, int patch_w, int dim, int height, int width,
                        float* out, dc_stream_t stream);
/* feat[j,:] = sum[j,:] / denom[j] with denom = sum_v weight (similarity) or sum_v visible. */
DC_API int dc_pixel_normalize(float* sums, const int64_t* point_off, const int64_t* view_off, const int64_t* mask_off,
                       const uint8_t* visible, const float* weight, int n_scenes, int64_t max_points_per_scene,
                       int dim, dc_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (5) Voxelisation to MinkowskiEngine sparse coordinates. Replaces ME.utils.sparse_quantize as
 * called at data/dataset_blender.py:406-414 / data/dataset.py:164-172, for a batch of samples:
 *   coords = floor(xyz / voxel_size) (fp32 true division) -> int32; unique voxels in order of
 *   first occurrence per sample; inverse map; label collision -> ignore_label.
 *   xyz [total_points,3] fp32, sample_off [n_samples+1], labels int32 or NULL.
 * Outputs: coords [total_points,3] int32 (first n_voxels rows valid per sample block),
 *   unique_map [total_points] int64 (sample-local point index of each voxel), inverse_map
 *   [total_points] int64 (sample-local voxel index of each point), voxel_labels int32 or NULL,
 *   voxel_off [n_samples+1] prefix of voxel counts. Sample blocks in coords/unique_map/
 *   voxel_labels start at sample_off[b] (not compacted across samples; use voxel_off for counts).
 */
DC_API size_t dc_voxelize_workspace(int64_t total_points);
DC_API int dc_voxelize(const float* xyz, const int64_t* sample_off, int n_samples, int64_t total_points,
                float voxel_size, const int32_t* labels, int32_t ignore_label, int32_t* coords,
                int64_t* unique_map, int64_t* inverse_map, int32_t* voxel_labels, int64_t* voxel_off,
                void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* out[b-th sample voxel k, :] = in[sample_off[b] + unique_map[sample_off[b] + k], :] - the
 * features[unique_map] gather of sparse_quantize; rows of `row_bytes` bytes, output compacted
 * with voxel_off. */
DC_API int dc_voxel_gather(const void* in, int64_t row_bytes, const int64_t* sample_off, const int64_t* voxel_off,
                    const int64_t* unique_map, int n_samples, int64_t total_points, void* out,
                    dc_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (6) Text-prompt grounding. Replaces ClipSimilarity.compute_similarity / predict
 * models/similarity.py:28-101 (after the text tower) and _get_similarity engine/distil.py:244-246.
 */
/* In-place row L2 normalisation x /= |x| with torch's per-dtype rounding (fp16: the norm and
 * the quotient are rounded to fp16). models/similarity.py:35,45,77. Optionally also writes
 * fp16 hi/lo operand planes for the GEMM (NULL to skip; lo only meaningful for fp32 input). */
DC_API int dc_row_normalize(void* x, int dtype, int64_t n_rows, int dim, int normalize, void* plane_hi,
                     void* plane_lo, dc_stream_t stream);

/* sims = X . T^T followed by the mode's epilogue, one tcgen05 GEMM per block of 256 prompts.
 *   x_hi/x_lo  [n_points, dim] fp16 planes (x_lo NULL for fp16 features)
 *   t_hi/t_lo  [n_prompts, dim] fp16 planes (t_lo NULL for fp16 prompts), any n_prompts >= 1, prompt 0 is the positive
 *              one. Either lo plane may be NULL while the other is set; the GEMM adds the lo product of each plane given.
 *   DC_GROUND_RAW:    out [n_points, out_ld] fp32 raw similarities
 *   DC_GROUND_PAIRED: out [n_points] fp32
 *   DC_GROUND_ARGMAX: out [n_points] fp32 (pos - mean(neg)), pred [n_points] uint8 (argmax == 0)
 *   DC_GROUND_CLASS:  argmax_idx [n_points] int64 = torch.max(sims, 1)[1]; out as RAW, or NULL to skip the matrix
 *                     (replaces _get_similarity + argmax, engine/distil.py:244-246,289-290,
 *                     tools/validate_upper_bound.py:59-61,101-102)
 *   minmax [4] fp32: min/max of `out` values and min/max of the raw similarities (device,
 *   updated atomically; initialise with dc_ground_init_minmax).
 *   workspace: dc_ground_workspace() bytes (0 up to 256 prompts; per-point partial results beyond).
 *   normalize_fp16_rows != 0 (fp16 features only, x_lo NULL): x_hi is L2-normalised IN PLACE first with torch's fp16
 *   semantics (models/similarity.py:77, quirk q15) - inside the GEMM kernel for dim 512/768/1024 (extra warps normalise the
 *   rows of the coming tiles, the A-operand TMA loads then hit L2), by a separate pass otherwise.
 */
DC_API int dc_ground_init_minmax(float* minmax, dc_stream_t stream);
DC_API size_t dc_ground_workspace(int64_t n_points, int n_prompts, int mode);
DC_API int dc_ground(const void* x_hi, const void* x_lo, int64_t n_points, const void* t_hi, const void* t_lo,
              int n_prompts, int dim, int mode, float softmax_temp, int normalize_fp16_rows, float* out, int out_ld,
              uint8_t* pred, int64_t* argmax_idx, float* minmax, void* workspace, size_t workspace_bytes,
              dc_stream_t stream);
/* ClipSimilarity.predict after the text tower (models/similarity.py:77-101) as ONE call: init of the extrema, operand
 * planes, in-place normalisation of the features (`normalize`), GEMM + epilogue, global min-max and threshold - four to
 * six launches back to back without returning to the host in between.
 *   feats [n_points, dim] fp16/fp32 (normalised in place when `normalize`), text [n_prompts, dim] fp16/fp32 rows already
 *   L2-normalised, prompt 0 positive; mode RAW (no negatives: n_prompts == 1), PAIRED or ARGMAX.
 *   out [n_points] fp32 = the min-max normalised score, pred [n_points] uint8 (score > threshold, or argmax == 0).
 *   *minmax_out (host pointer, optional) receives the device address of the four extrema inside the workspace.
 *   workspace: 256-byte aligned, dc_predict_workspace() bytes. */
DC_API size_t dc_predict_workspace(int64_t n_points, int n_prompts, int dim, int feat_dtype, int text_dtype, int mode);
DC_API int dc_predict(void* feats, int feat_dtype, int64_t n_points, const void* text, int text_dtype, int n_prompts, int dim,
               int mode, float softmax_temp, int normalize, float threshold, float* out, uint8_t* pred,
               float** minmax_out, void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* ClipSimilarity.predict for every text query of a scene in ONE call: the features are normalised (when `normalize`)
 * and multiplied with the prompt rows once, S = X . T^T [n_points, n_prompts] (dc_ground, RAW), then each query is scored
 * from its own columns of S, with its own min-max and threshold. Row q of the result equals dc_predict on the prompt rows
 * [pos[q], neg_cols[neg_off[q]], ..., neg_cols[neg_off[q+1] - 1]].
 *   feats [n_points, dim] fp16/fp32 (normalised in place when `normalize`), text [n_prompts, dim] fp16/fp32 rows already
 *   L2-normalised, each distinct prompt once; n_prompts <= 1536. feats, out and pred may be NULL when n_points == 0.
 *   pos [n_queries], neg_off [n_queries + 1], neg_cols [neg_off[n_queries]] int32 in HOST memory: query q's positive
 *   column and its negative columns (CSR; repeats allowed). Checked on the host (every column in [0, n_prompts); RAW:
 *   no query has negatives; PAIRED / ARGMAX: every query has one at least) and copied into the workspace by
 *   cudaMemcpyAsync, so pageable arrays may be reused when the call returns.
 *   out [n_queries, n_points] fp32 = the min-max normalised scores, pred [n_queries, n_points] uint8 (score > threshold,
 *   or argmax == 0).
 *   workspace: 256-byte aligned, dc_predict_queries_workspace() bytes (S alone is 4 * n_points * n_prompts). */
DC_API size_t dc_predict_queries_workspace(int64_t n_points, int n_prompts, int n_queries, int64_t n_neg_total, int dim,
                                           int feat_dtype, int text_dtype);
DC_API int dc_predict_queries(void* feats, int feat_dtype, int64_t n_points, const void* text, int text_dtype, int n_prompts,
                              int dim, const int32_t* pos, const int32_t* neg_off, const int32_t* neg_cols, int n_queries,
                              int mode, float softmax_temp, int normalize, float threshold, float* out, uint8_t* pred,
                              void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* dc_predict_queries for every scene of a batch in ONE call. Scene s owns the feature rows [point_off[s], point_off[s+1]),
 * the prompt rows [prompt_off[s], prompt_off[s+1]) and the queries [query_off[s], query_off[s+1]); its (Q_s, N_s) block of
 * the result equals what dc_predict_queries returns for that scene alone, bit for bit (same operands, same K order, same
 * epilogue arithmetic).
 *   feats [sum N, dim] fp16/fp32, the rows of the scenes with queries normalised in place when `normalize` (the rows of a
 *   scene without queries are left untouched); text [sum P, dim] fp16/fp32 rows already L2-normalised; P_s <= 1536.
 *   point_off (int64), prompt_off and query_off (int32) [n_scenes + 1] in HOST memory, starting at 0; sum N < 2^31,
 *   sum Q <= 65535.
 *   pos [sum Q], neg_off [sum Q + 1], neg_cols [neg_off[sum Q]] int32 in HOST memory: the columns of query q of scene s,
 *   LOCAL to the scene's prompt block ([0, P_s)). Checked on the host like dc_predict_queries' table, then copied into
 *   the workspace by cudaMemcpyAsync, with the GEMM's tile list and the scoring tables.
 *   out fp32 / pred uint8: scene s's (Q_s, N_s) block starts at sum_{s' < s} Q_s' * N_s'.
 *   One tcgen05 GEMM per block of 256 prompt columns over a tile list (128 rows of one scene x that scene's prompts)
 *   writes S = X . T^T once, at a row stride of ld = max P_s rounded up to 4.
 *   workspace: 256-byte aligned, dc_predict_many_workspace() bytes. S alone is 4 * sum N * ld bytes, so one scene with
 *   many prompts widens S for the whole batch. */
DC_API size_t dc_predict_many_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off,
                                        const int32_t* query_off, int64_t n_neg_total, int dim, int feat_dtype, int text_dtype);
DC_API int dc_predict_many(void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                           const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off, const int32_t* pos,
                           const int32_t* neg_off, const int32_t* neg_cols, int mode, float softmax_temp, int normalize,
                           float threshold, float* out, uint8_t* pred, void* workspace, size_t workspace_bytes,
                           dc_stream_t stream);
/* dc_predict_many scored against per-point ground truth in ONE call, for the grounding evaluation (trainMetricPC
 * utils/misc.py:21-50 after the query loop): the same launches up to the threshold pass, which counts instead of writing
 * the predictions. For query q, inter[q] = |pred_q & gt_q| and uni[q] = |pred_q | gt_q|, where pred_q is row q of
 * dc_predict_many's pred (the same bits) and gt_q[i] = (labels[i] is one of the query's ids) over the query's scene.
 * Neither the scores nor the predictions are returned: they stay in the workspace.
 *   feats, text, the offset tables, pos / neg_off / neg_cols, mode, softmax_temp, normalize, threshold: as in
 *   dc_predict_many, with the same rules and limits (the rows of the scenes with queries are normalised in place).
 *   labels [sum N] int32 (DC_I32) or int64 (DC_I64), device memory, in feature-row order; compared as int64.
 *   gt_off [sum Q + 1] int32 and gt_ids [gt_off[sum Q]] int64 in HOST memory: query q's object ids are
 *   gt_ids[gt_off[q] .. gt_off[q+1]), strictly ascending (an empty list: no point is ground truth). Checked on the host
 *   before any launch (gt_off[0] == 0, gt_off does not decrease, ids ascend), then staged with the other tables.
 *   inter / uni [sum Q] int64, device memory: zeroed first, so a query of an empty scene reports 0 / 0.
 *   workspace: 256-byte aligned, dc_predict_many_iou_workspace() bytes, n_gt_total = gt_off[sum Q]. It holds
 *   dc_predict_many's workspace plus the (sum Q_s * N_s) scores and argmax bytes.
 * The call does not synchronise. */
DC_API size_t dc_predict_many_iou_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off,
                                            const int32_t* query_off, int64_t n_neg_total, int64_t n_gt_total, int dim,
                                            int feat_dtype, int text_dtype);
DC_API int dc_predict_many_iou(void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                               const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off,
                               const int32_t* pos, const int32_t* neg_off, const int32_t* neg_cols, const void* labels,
                               int label_dtype, const int32_t* gt_off, const int64_t* gt_ids, int mode, float softmax_temp,
                               int normalize, float threshold, int64_t* inter, int64_t* uni, void* workspace,
                               size_t workspace_bytes, dc_stream_t stream);
/* dc_predict_many_iou at many thresholds in ONE call, for choosing the threshold or reporting mIoU / Pr@k against it:
 * everything up to the threshold pass runs once. Row t of inter / uni equals, bit for bit, what dc_predict_many_iou
 * returns with threshold = thresholds[t] on the same (unnormalised) inputs. The pass bins each point by how many of the
 * distinct thresholds its normalised score exceeds, so its cost per point does not grow with n_thresholds.
 *   Every argument as in dc_predict_many_iou, with the same rules and limits, except:
 *   thresholds [n_thresholds] fp32 in HOST memory, 1 <= n_thresholds <= 1024, in any order; duplicates, +-inf and NaN
 *   allowed (x > NaN is false: a NaN threshold predicts no point, like +inf). Argmax ignores them: every row is equal.
 *   inter / uni [n_thresholds * sum Q] int64, device memory, row-major by threshold (row t = thresholds[t]), zeroed by
 *   the call.
 *   workspace: 256-byte aligned, dc_predict_many_iou_sweep_workspace() bytes (0 for n_thresholds outside 1..1024):
 *   dc_predict_many_iou's workspace plus two tables of n_thresholds 4-byte entries and 8 * (n_thresholds + 1) bytes
 *   of histograms per query, each region rounded up to 256 bytes.
 * Host-side checks happen before any launch. The call does not synchronise. */
DC_API size_t dc_predict_many_iou_sweep_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off,
                                                  const int32_t* query_off, int64_t n_neg_total, int64_t n_gt_total,
                                                  int n_thresholds, int dim, int feat_dtype, int text_dtype);
DC_API int dc_predict_many_iou_sweep(void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                                     const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off,
                                     const int32_t* pos, const int32_t* neg_off, const int32_t* neg_cols,
                                     const void* labels, int label_dtype, const int32_t* gt_off, const int64_t* gt_ids,
                                     int mode, float softmax_temp, int normalize, const float* thresholds,
                                     int n_thresholds, int64_t* inter, int64_t* uni, void* workspace,
                                     size_t workspace_bytes, dc_stream_t stream);
/* The host table dc_predict_many_iou_sweep stages (pure host code, no device needed): levels[0 .. *n_levels) are the
 * distinct values of thresholds[0 .. n_thresholds) ascending, with NaN taken as +inf and -0 and +0 one level, and rank[t]
 * is the index of entry t's level. levels and rank have room for n_thresholds entries; 1 <= n_thresholds <= 1024. */
DC_API int dc_sweep_levels(const float* thresholds, int n_thresholds, float* levels, int32_t* rank, int* n_levels);

/* Global min-max normalisation + threshold (models/similarity.py:83-88, :95-98):
 * values <- (v - min)/(max - min) (or v / max when the raw extrema coincide), pred = values > thr
 * when pred_from_threshold != 0. */
DC_API int dc_minmax_threshold(float* values, int64_t n, const float* minmax, int use_raw_extrema_for_test,
                        float threshold, int pred_from_threshold, uint8_t* pred, dc_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Geometry helpers of utils/projections.py.
 */
/* depth_to_pointcloud utils/projections.py:67-86 (+ optional axis flips :89-97 and cam->world
 * utils/transforms.py:43-49): out[v, y, x, :] fp64. flip_y bit0 / flip_z negate after back-projection;
 * flip_y bit1 selects Open3D's rounding order (u - cx) * z / fx; poses (fp64 [n_views,16],
 * camera->world, widened from the caller's dtype) may be NULL. */
DC_API int dc_backproject(const float* depths, int n_views, int height, int width, const double* fxfycxcy,
                   int flip_y, int flip_z, const double* poses, double* out, dc_stream_t stream);
/* pointcloud_to_pixel utils/projections.py:59-64: un-truncated fp64 pixel coordinates. */
DC_API int dc_points_to_pixels(const double* cam_points, int64_t n, const double* fxfycxcy, double* pixels,
                        dc_stream_t stream);

/* Rigid transform out[i,:] = (M . [p_i;1])[:3] in fp64 with np.dot's operation order;
 * M: 16 fp64 (host pointer, row-major; an fp32 matrix widens exactly like np.dot's promotion). Replaces transform_pointcloud_to_world_frame /
 * _to_camera_frame utils/transforms.py:43-61 (the caller inverts the pose for the latter). */
DC_API int dc_transform_points(const double* points, int64_t n, const double* matrix_host, double* out,
                        dc_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Sort-based helpers of the REGRAD-style functions in utils/projections.py.
 * workspace for the two calls below: dc_sort_workspace(n) bytes.
 */
DC_API size_t dc_sort_workspace(int64_t n);
/* pool_multiview_features utils/projections.py:245-261: np.unique(points, axis=0) (lexicographic
 * order) + per-unique-row maximum of the features. points (n,3) fp64, feats (n,dim) DC_F32/DC_F64.
 * Outputs hold n rows of capacity; *n_unique (device int64) gives the valid count. */
DC_API int dc_unique_max_pool(const double* points, const void* feats, int feat_dtype, int dim, int64_t n,
                       double* out_points, void* out_feats, int64_t* n_unique, void* workspace,
                       size_t workspace_bytes, dc_stream_t stream);
/* pc_voxel_down utils/geometry.py:350-352 (Open3D voxel_down_sample semantics, parity unpinned):
 * voxel index = floor((p - (min_bound - size/2)) / size), output = mean of the voxel's points summed
 * in point order; voxels ordered by index. first_index[u] = smallest point index of voxel u. */
DC_API int dc_voxel_down_mean(const double* points, int64_t n, double voxel_size, double* out_points,
                       int64_t* first_index, int64_t* n_voxels, void* workspace, size_t workspace_bytes,
                       dc_stream_t stream);
/* voxel_down_sample_and_trace + label majority vote of aggregate_views_blender_new utils/geometry.py:186-201
 * (Open3D semantics, parity unpinned): per voxel the mean position, the mean colour (optional) and the most
 * frequent label (optional; ties: the label met first in point order, like Counter.most_common()[0][0]);
 * counts[u] = members of voxel u, first_index[u] its smallest point index (both optional). Voxels ordered by
 * voxel index. The one-scene, one-size case of dc_aggregate_views' trace. workspace:
 * dc_voxel_down_trace_workspace(n) bytes. */
DC_API size_t dc_voxel_down_trace_workspace(int64_t n);
DC_API int dc_voxel_down_trace(const double* points, const double* colors, const int64_t* labels, int64_t n,
                        double voxel_size, double* out_points, double* out_colors, int64_t* out_labels,
                        int64_t* first_index, int64_t* counts, int64_t* n_voxels, void* workspace,
                        size_t workspace_bytes, dc_stream_t stream);
/* aggregate_views_blender_new utils/geometry.py:120-204 for S scenes at U voxel sizes in one call.
 * Inputs (device): the views' depth maps (fp32), instance maps (DC_U8 / DC_I64) and RGB images (3 channels,
 * DC_U8 / DC_F64), concatenated view after view (scene after scene); view v covers pixels
 * [view_pix_off[v], view_pix_off[v + 1]) as a row-major view_hw[2v] x view_hw[2v + 1] image.
 * Host tables: view_pix_off[V + 1], view_hw[2V], scene_view_off[S + 1], poses[16V] (fp64 world matrices,
 * row-major 4x4), fxfycxcy[4], voxel_sizes[U] (each > 0; depth_trunc must not be NaN when U > 0).
 * Per scene, a pixel is labelled when depth < depth_trunc and kept as a point when 0 < depth < depth_trunc:
 * points / colors / labels receive scene s's rows at [point_off[s], point_off[s + 1]) / [label_off[s], ...)
 * (device int64 [S + 1]); a point is the Open3D back-projection flipped by (1, -1, -1) and moved by the view's
 * world matrix, a colour is rgb / 255.0. Point j of a scene votes with label j of that scene.
 * Voxel outputs: segment (u, s) = scene s at voxel_sizes[u] is rows [vox_off[u S + s], vox_off[u S + s + 1])
 * of vox_points / vox_colors / vox_labels (device int64 vox_off[U S + 1]); see dc_voxel_down_trace.
 * Capacities: n_pixels rows for points / colors / labels, U * n_pixels for the voxel outputs, where
 * n_pixels = view_pix_off[V] and U * n_pixels < 2^31. workspace: dc_aggregate_views_workspace bytes. */
DC_API size_t dc_aggregate_views_workspace(int n_scenes, int n_views, int64_t n_pixels, int n_sizes);
DC_API int dc_aggregate_views(const float* depths, const void* segs, int seg_dtype, const void* rgbs, int rgb_dtype,
                              const int64_t* view_pix_off, const int32_t* view_hw, const int32_t* scene_view_off,
                              const double* poses, const double* fxfycxcy, float depth_trunc, const double* voxel_sizes,
                              int n_scenes, int n_views, int n_sizes, double* points, double* colors, int64_t* labels,
                              int64_t* point_off, int64_t* label_off, double* vox_points, double* vox_colors,
                              int64_t* vox_labels, int64_t* vox_off, void* workspace, size_t workspace_bytes,
                              dc_stream_t stream);
/* find_closest_indices utils/geometry.py:390-401 (cKDTree.query k=1): exact fp64 nearest neighbour
 * of every query point in `ref` (ties: smallest index); out_dist2 (squared distance) may be NULL. */
DC_API int dc_nearest_index(const double* query, int64_t m, const double* ref, int64_t n, int64_t* out_index,
                     double* out_dist2, dc_stream_t stream);

/* ---- metric counts that follow the grounding kernel (SURVEY.md 8f-2) ----
 * dc_binary_iou_counts: trainMetricPC utils/misc.py:21-50 for a ragged batch of instances
 * (inst_off[n_instances + 1]): pred is binarised at `threshold` exactly like `pred[pred < thr] = 0;
 * pred[pred >= thr] = 1` (NaN stays NaN and counts as set), written back in place when
 * binarize_in_place != 0 and no sigmoid is applied (the reference mutates the caller's tensor then);
 * inter / uni [n_instances] int64 = |pred & gt|, |pred | gt|. gt dtype: DC_U8 (bool), DC_I32, DC_I64, DC_F32.
 * dc_class_iou_hist: intersectionAndUnionGPU utils/misc.py:186-199 - output[target == ignore_index] =
 * ignore_index in place, then the K-bin histograms of output[output == target], output and target
 * (torch.histc(bins=K, min=0, max=K-1) maps class c in [0, K-1] to bin c); fp32 results,
 * area_union = area_output + area_target - area_intersection. */
DC_API int dc_binary_iou_counts(float* pred, const void* gt, int gt_dtype, const int64_t* inst_off, int n_instances,
                         int64_t max_points_per_instance, float threshold, int apply_sigmoid, int binarize_in_place,
                         int64_t* inter, int64_t* uni, dc_stream_t stream);
DC_API size_t dc_class_iou_workspace(int n_classes);
DC_API int dc_class_iou_hist(void* output, const void* target, int dtype, int64_t n, int n_classes, int64_t ignore_index,
                      float* area_intersection, float* area_union, float* area_target, void* workspace,
                      size_t workspace_bytes, dc_stream_t stream);

/* ---- training-sample assembly (SURVEY.md 8f-4): MVDistilDataset.__getitem__ data/dataset_blender.py:330-362,400-414
 * for a ragged batch of samples; random choices (views, point indices) are inputs.
 * dc_sample_keep_flags: keep[j] = OR over the sample's view_list of vis_mask[v, j] (vis_mask: per sample a (V_s, N_s)
 *   uint8 block at mask_off[s]); an empty view list keeps every point (use_full_pc).
 * dc_sample_gather: with new_index / kept_off from dc_compact_scan(keep): row r of sample s = kept point number
 *   indices[r]; out_xyz = float(xyz - column mean of the selected rows) (numpy's sequential axis-0 mean, fp64),
 *   out_rgb = float(rgb), out_label = label (through uint8 when label_as_u8, like `.astype(np.uint8)` at :349),
 *   out_feat[r] = per_obj[obj_off[s] + label]  (feat[label], :128-130). Scratch: rows / kept_idx int64
 *   [total_rows] / [total_points], mean [3 * n_samples] fp64. *error: 1 = index out of range, 2 = label without
 *   a per_obj row (numpy raises IndexError in both cases). */
DC_API int dc_sample_keep_flags(const uint8_t* vis_mask, const int64_t* mask_off, const int64_t* point_off,
                         const int32_t* view_list, const int64_t* view_list_off, int n_samples,
                         int64_t max_points_per_sample, uint8_t* keep, dc_stream_t stream);
DC_API int dc_sample_gather(const double* xyz, const double* rgb, const int64_t* label, const float* per_obj,
                     const int64_t* obj_off, const uint8_t* keep, const int64_t* new_index, const int64_t* kept_off,
                     const int64_t* point_off, const int64_t* indices, const int64_t* out_off, int n_samples,
                     int64_t total_points, int64_t total_rows, int64_t max_rows_per_sample, int dim, int label_as_u8,
                     float* out_xyz, float* out_rgb, int32_t* out_label, float* out_feat, int64_t* rows,
                     int64_t* kept_idx, double* mean, int* error, dc_stream_t stream);

/* ---- host-side staging (no device work): used by the Python drop-in to fill pinned upload buffers ----
 * dc_host_gather_copy: dst[i * item_bytes ...] = srcs[i][0 .. item_bytes) for n_items host arrays, on n_threads
 * threads. dc_host_gather_narrow_i64_u8: same for int64 arrays of item_elems elements narrowed to uint8;
 * *out_of_range = 1 if any value lies outside [0, 255] (the caller then ships the int64 maps unchanged, keeping
 * the reference's error behaviour for ids >= Q, utils/feature_fusion.py:317,328-333). */
DC_API int dc_host_gather_copy(const void* const* srcs, int64_t n_items, int64_t item_bytes, void* dst, int n_threads);
DC_API int dc_host_gather_narrow_i64_u8(const int64_t* const* srcs, int64_t n_items, int64_t item_elems, uint8_t* dst,
                                        int n_threads, int* out_of_range);
/* dc_host_masks_to_seg: binary_masks_to_seg utils/image.py:11-15 for n_views views in one pass over the masks:
 * view v has masks masks[mask_off[v] .. mask_off[v + 1]) (bool or uint8, view_pixels[v] bytes each, at least one)
 * with instance ids ids[mask_off[v] ..]; its map, value = max over k of (int64) mask_k * id_k as numpy computes
 * it (a pixel covered by every mask takes the largest product, without the 0), is written at dst + pix_off[v]
 * elements. out_dtype DC_U8 or DC_I64; with DC_U8, *out_of_range = 1 when a value lies outside [0, 255] (the
 * maps are then incomplete; the caller builds them again as DC_I64). */
DC_API int dc_host_masks_to_seg(const uint8_t* const* masks, const int64_t* ids, const int64_t* mask_off, int n_views,
                                const int64_t* view_pixels, const int64_t* pix_off, int out_dtype, void* dst,
                                int n_threads, int* out_of_range);

#ifdef __cplusplus
}
#endif
#endif /* DROPCLIP_H_ */
