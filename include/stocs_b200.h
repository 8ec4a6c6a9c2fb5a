/* stocs_b200.h -- C ABI of libstocs_b200.so: the B200 (sm_100a) implementation of the
 * data-parallel core of StoCS pose estimation (kuwt/model_matching, src/stocs.cpp).
 *
 * The reference has no FFI layer: its boundary is the C++ class stocs::stocs_estimator
 * (include/stocs.hpp:16-180).  This header is what the drop-in shim of that class
 * (model_matching_b200/host/stocs.hpp) binds; each entry point cites the reference code it
 * replaces.  Conventions: plain pointers and sizes only; every function returns an int status
 * (0 = ok, negative = error, text via stocs_b200_last_error); the caller owns every host buffer,
 * the context owns every device buffer and stream; calls on one context must be serialised by
 * the caller (the reference estimator is not thread-safe either, SURVEY.md section 8b); there
 * is NO CPU fallback: without a usable sm_100 device stocs_b200_create fails.
 *
 * Matrices are 16 floats in column-major order (Eigen::Matrix4f memory layout,
 * include/stocs.hpp:9).  Points are tightly packed xyz float triples.  Pixels are (row, col).
 */
#ifndef STOCS_B200_H_
#define STOCS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct stocs_b200_ctx stocs_b200_ctx;

enum {
  STOCS_OK = 0,
  STOCS_E_ARG = -1,        /* bad argument */
  STOCS_E_CUDA = -2,       /* CUDA runtime error (see last_error) */
  STOCS_E_STATE = -3,      /* call order violated (e.g. score before upload_scene) */
  STOCS_E_NODEVICE = -4,   /* no sm_100 device / driver */
  STOCS_E_CAPACITY = -5,   /* caller-provided output capacity too small */
  STOCS_E_NCCL = -6        /* NCCL missing or failed (see last_error) */
};

#define STOCS_B200_ABI_VERSION 2
int stocs_b200_abi_version(void);

/* One context per GPU (one process per GPU in multi-GPU runs).  device = CUDA ordinal. */
int stocs_b200_create(stocs_b200_ctx** out, int device);
void stocs_b200_destroy(stocs_b200_ctx* ctx);
const char* stocs_b200_last_error(stocs_b200_ctx* ctx);

/* Estimator parameters (constructor arguments of stocs::stocs_estimator, include/stocs.hpp:18-30;
 * defaults = src/stocs_match_one_object.cpp:7-10). */
int stocs_b200_set_params(stocs_b200_ctx* ctx, float distance_threshold, int ppf_tr_discretization,
                          int ppf_rot_discretization);

/* ---- a1: depth back-projection (src/rgbd.cpp:208-225) -------------------------------------
 * depth: H*W uint16 row-major; bgr: H*W*3 uint8 (may be NULL); intrinsics order {fx,cx,fy,cy}
 * as in src/stocs_match_one_object.cpp:20.  xyz_out: H*W*3 floats; rgb_out: H*W packed
 * 0x00RRGGBB (may be NULL).  Every pixel is emitted, including depth 0. */
int stocs_b200_backproject(stocs_b200_ctx* ctx, const uint16_t* depth, const uint8_t* bgr, int W,
                           int H, float fx, float cx, float fy, float cy, float depth_scale,
                           float* xyz_out, uint32_t* rgb_out);

/* ---- f1: scene-cloud construction (body of rgbd::load_rgbd_data_sampled, src/rgbd.cpp:190-279) ----
 * back-projection -> voxel-grid centroids (leaf = voxel_size) -> radius outlier removal
 * (r = 2*voxel_size + 0.005, more than 10 neighbours) -> per centroid: 0 < z <= 2, re-projection to
 * (row, col), class probability (uint16 / 10000) >= class_threshold, valid depth normal.
 * class_prob: H*W uint16; edge: H*W uint8 or NULL (treated as 0).  Outputs hold up to cap points
 * (rgb3, edge_p may be NULL); *n_out = number of points (STOCS_E_CAPACITY if > cap).  Entries of
 * the output arrays beyond *n_out (up to cap) may be overwritten: the call fetches its results before
 * it knows their count, with the previous frame's as the estimate. */
int stocs_b200_build_scene_cloud(stocs_b200_ctx* ctx, const uint16_t* depth, const uint8_t* bgr,
                                 const uint16_t* class_prob, const uint8_t* edge, int W, int H, float fx,
                                 float cx, float fy, float cy, float depth_scale, float voxel_size,
                                 float class_threshold, float* pos3, float* nrm3, float* rgb3,
                                 int32_t* pixel_rc, float* class_p, float* edge_p, int64_t cap, int64_t* n_out);

/* The scene clouds of n_objects objects of one frame in one call: the back-projection, voxel grid, outlier
 * removal and depth normals run once, and only the class test runs per object.  class_probs holds
 * n_objects H*W uint16 maps, object after object; class_thresholds one threshold per object.  The
 * outputs are those of build_scene_cloud, concatenated: object k's points are rows
 * [offsets[k], offsets[k+1]) (offsets: n_objects + 1 entries, the CSR of find_congruent), and that slice
 * is bit-identical, in the same order, to build_scene_cloud on (class_probs[k], class_thresholds[k]).
 * rgb3 and edge_p may be NULL.  More than cap points in all: STOCS_E_CAPACITY with offsets filled.
 * STOCS_E_ARG: n_objects outside 1..STOCS_B200_MAX_CLOUD_OBJECTS, class_probs, class_thresholds or
 * offsets NULL, the argument checks of build_scene_cloud, or a required output NULL while points are
 * emitted.  Like build_scene_cloud, the call synchronises once when its read-back estimate (from the
 * previous call) covers the output, twice otherwise.  Device memory per object, held by the context:
 * one 4-byte flag per pixel plus the 2-byte map (1.8 MB at 640x480), besides the output rows. */
#define STOCS_B200_MAX_CLOUD_OBJECTS 32
int stocs_b200_build_scene_clouds(stocs_b200_ctx* ctx, const uint16_t* depth, const uint8_t* bgr,
                                  const uint16_t* class_probs, const float* class_thresholds, int n_objects,
                                  const uint8_t* edge, int W, int H, float fx, float cx, float fy, float cy,
                                  float depth_scale, float voxel_size,
                                  float* pos3, float* nrm3, float* rgb3, int32_t* pixel_rc, float* class_p,
                                  float* edge_p, int64_t cap, int64_t* offsets);

/* The same from a frame already in GPU memory (e.g. a segmentation network's output), with the same stages, output
 * order, CSR offsets (a host array), capacity rule and STOCS_E_CAPACITY with offsets filled.  Every image and output
 * pointer is device memory on the context's device; d_bgr, d_edge, d_rgb3 and d_edge_p may be NULL.  d_class_maps is
 * a host array of n_objects device pointers, each to a row-major W*H map of map_type; entries may repeat, so the
 * channels of a [C,H,W] tensor can be passed in any order without a copy.
 *   STOCS_B200_MAP_U16: uint16, converted as build_scene_clouds does, (float)((double)(float)v * (1.0/10000));
 *   STOCS_B200_MAP_F32: float, used as given; the class test is p == p && !(p < threshold), so a NaN never passes,
 *   and a float map holding the exact uint16 conversion gives bit-identical output.
 * stream (a cudaStream_t of the context's device; NULL is its default stream): the call's work is ordered after
 * what the caller has queued on it so far.  The call synchronises once and reads back only the voxel count and the
 * object ends; on return the outputs are complete, and rows past offsets[n_objects] are not written.  The context's
 * read-back estimate afterwards is what build_scene_clouds leaves.  STOCS_E_ARG, before anything
 * is enqueued: the checks of build_scene_clouds, an unknown map_type, a NULL map entry, or a pointer that is not
 * device memory on the context's device (the message names the argument).  Nothing of the frame or the cloud
 * crosses PCIe. */
enum { STOCS_B200_MAP_U16 = 0, STOCS_B200_MAP_F32 = 1 };
int stocs_b200_build_scene_clouds_device(
    stocs_b200_ctx* ctx, const uint16_t* d_depth, const uint8_t* d_bgr,
    const void* const* d_class_maps, int map_type, const float* class_thresholds, int n_objects,
    const uint8_t* d_edge, int W, int H, float fx, float cx, float fy, float cy,
    float depth_scale, float voxel_size,
    float* d_pos3, float* d_nrm3, float* d_rgb3, int32_t* d_pixel_rc, float* d_class_p, float* d_edge_p,
    int64_t cap, int64_t* offsets, void* stream);

/* ---- a2/a11: model and scene upload --------------------------------------------------------
 * upload_model replaces load_object_info's point part (src/stocs.cpp:86-97) and the model half of
 * centroid_shift (src/stocs.cpp:951-962); it also builds the compact own-bin PPF table that
 * replaces PPFMapType (include/rgbd.hpp:23; src/stocs.cpp:62-78; src/rgbd.cpp:123-154).
 * upload_scene replaces the scene half of centroid_shift (src/stocs.cpp:948-960) and
 * kdtree_initialize (src/stocs.cpp:966-980): the scene is centred with the reference's sequential
 * fp32 centroid and indexed by a voxel grid (+ the reference kd-tree, used only to break exact
 * distance ties the way kdtree.h:416-428 does).  pixel_rc may be NULL.
 * upload_scene returns when the grid index is complete; the kd-tree (host work) is finished on a
 * host thread and collected by the first scoring launch that follows, or by the next upload_scene /
 * destroy.  (upload_scenes_device builds it on the device instead, on the context's copy stream, and
 * the same calls wait for it.)  The input buffers are not referenced after the call returns. */
int stocs_b200_upload_model(stocs_b200_ctx* ctx, const float* pos3, const float* nrm3, int M);
int stocs_b200_upload_scene(stocs_b200_ctx* ctx, const float* pos3, const float* nrm3,
                            const float* class_probability, const int32_t* pixel_rc, int S);
int stocs_b200_get_centroids(stocs_b200_ctx* ctx, float* scene3, float* model3);
/* centred point sets as the estimator holds them after centroid_shift (for visualize_best_pose,
 * include/stocs.hpp:136-149).  Either pointer may be NULL. */
int stocs_b200_get_centred(stocs_b200_ctx* ctx, float* scene_pos3, float* model_pos3);

/* Replace the PPF table that upload_model derived from the points by a preloaded one (the
 * reference's ppf_map_preloaded, src/stocs.cpp:94; src/stocs_match_one_object.cpp:201-203) in the
 * layout of stocs_b200_ppf_export: n entries, keys4 = own-bin key (mm, deg, deg, deg), pairs2 = model
 * ids.  The header values must match the estimator (set_params discretisations, |M| of the uploaded
 * model) and every entry must fit the model: otherwise STOCS_E_ARG with an explanatory message --
 * a table built for something else is never silently ignored. */
int stocs_b200_upload_ppf_table(stocs_b200_ctx* ctx, const int32_t* keys4, const int32_t* pairs2, int64_t n,
                                int tr_discretization, int rot_discretization, int num_model_points);

/* PPF table queries (replace ppf_map.find, src/stocs.cpp:403,780-786).
 * ppf_lookup: number of pairs stored under key4 in the reference's expanded map, -1 if the key is
 * absent; copies up to cap pairs (id1,id2) in the reference's list order. */
int stocs_b200_ppf_num_pairs(stocs_b200_ctx* ctx, int64_t* own_bin_pairs, int64_t* own_bin_keys);
/* number of keys of the reference's expanded map (what `ppf_map.size()` prints, src/stocs.cpp:96) */
int stocs_b200_ppf_num_expanded_keys(stocs_b200_ctx* ctx, int64_t* expanded_keys);
/* the compact table itself, for the `ppf_map` file written by model_preprocess
 * (src/model_preprocess.cpp:28-36): per stored pair its own-bin key (4 ints) and (id1,id2),
 * sorted by (key, id1, id2).  cap = capacity in pairs; *n = number of pairs. */
int stocs_b200_ppf_export(stocs_b200_ctx* ctx, int32_t* keys4, int32_t* pairs2, int64_t cap, int64_t* n);
int stocs_b200_ppf_lookup(stocs_b200_ctx* ctx, const int32_t* key4, int32_t* pairs2, int64_t cap,
                          int64_t* count);

/* ---- a5/a6/a8: probability-weighted base sampling, class mode (src/stocs.cpp:133-268,363-519)
 * Samples n_bases bases numbered first_base_no.. with the counter-based stream keyed by seed.
 * base_idx4: n_bases*4 scene indices (reordered by try_sampled_base); inv2: n_bases*2
 * invariants; valid: n_bases flags (0 = the reference's "return false"). */
int stocs_b200_sample_bases(stocs_b200_ctx* ctx, uint64_t seed, uint32_t first_base_no, int n_bases,
                            int32_t* base_idx4, float* inv2, uint8_t* valid);

/* ---- a7: edge-aware instance sampling (src/stocs.cpp:521-535, 559-751; src/rgbd.cpp:314-367) ----
 * upload_edge_map: the 8-bit edge probability image (H*W, 255 = no edge, as cv::imread(.., CV_8UC1)
 * returns it); resets previous_segment / segmentation_buffer.  W*H must be a multiple of 4.
 * sample_instance_base: ONE base (bases are sequentially coupled in this mode): decays the class
 * prior inside the previous segment by `dispersion` (permanently), prunes edge pixels, draws the
 * base restricted to the flood-filled segment around the first point.  base_num is 1..255 as in
 * the reference driver (i+1) and also keys the random stream.  upload_scene must have been given
 * pixel coordinates.  mask_out (may be NULL): the H*W segmentation mask (255 inside).
 * segment_bits (may be NULL): ceil(S/32) words, bit i set = scene point i is in the reference's
 * `segment` output (survived the first update and lies inside the mask). */
int stocs_b200_upload_edge_map(stocs_b200_ctx* ctx, const uint8_t* edge, int W, int H);
int stocs_b200_sample_instance_base(stocs_b200_ctx* ctx, uint64_t seed, int base_num, float dispersion,
                                    int32_t* base_idx4, float* inv2, uint8_t* valid, uint8_t* mask_out,
                                    uint32_t* segment_bits);
/* current per-point class probability (instance sampling decays it; LCP uses the decayed value,
 * src/stocs.cpp:577,1033) */
int stocs_b200_get_class_probability(stocs_b200_ctx* ctx, float* out);
/* overwrite it (S floats): keeps the replicas of a multi-GPU group consistent after instance
 * sampling changed the prior on one device */
int stocs_b200_set_class_probability(stocs_b200_ctx* ctx, const float* class_probability);

/* ---- a9: congruent-set lookup (src/stocs.cpp:753-869) --------------------------------------
 * For each of n_bases bases returns its quadrilaterals (4 model indices each) in the reference's
 * std::set order; quad_offsets has n_bases+1 entries (CSR).  quads4 holds up to cap quads;
 * returns STOCS_E_CAPACITY (with quad_offsets filled) when more are needed. */
int stocs_b200_find_congruent(stocs_b200_ctx* ctx, int n_bases, const int32_t* base_idx4,
                              const float* inv2, int32_t* quads4, int64_t cap,
                              int64_t* quad_offsets);

/* ---- a10: rigid transform per (base, quad) (src/stocs.cpp:270-361, 871-941) ----------------
 * n items; base_idx4 and quads4 are n*4 each.  T_centred16 = all_transforms entry, T_world16 =
 * PoseCandidate::transform; ok[i] = 0 when the reference would not push a transform. */
int stocs_b200_fit_transforms(stocs_b200_ctx* ctx, int64_t n, const int32_t* base_idx4,
                              const int32_t* quads4, float* T_centred16, float* T_world16,
                              uint8_t* ok);

/* ---- a12: LCP scoring (src/stocs.cpp:1006-1041 + kdtree.h:394-459) -------------------------
 * Scores H centred transforms; lcp[i] is bit-identical to the reference's sequential fp32 sum,
 * inliers[i] the number of model points passing both tests (may be NULL).  Host buffers. */
int stocs_b200_score_lcp(stocs_b200_ctx* ctx, const float* T16, int64_t H, float* lcp,
                         int32_t* inliers);
/* Same, all pointers are device pointers; runs on the context stream (or `stream` if non-NULL,
 * a cudaStream_t) and does not synchronise.  */
int stocs_b200_score_lcp_device(stocs_b200_ctx* ctx, const float* d_T16, int64_t H, float* d_lcp,
                                int32_t* d_inliers, void* stream);

/* ---- a13: best pose / top-K reduction (src/stocs.cpp:982-1004) -----------------------------
 * Over the lcp array of the most recent score call (or an explicit device array for the _device
 * variant): best = first strict maximum (index -1 and lcp 0 when all are 0); top-K ordered by
 * (lcp desc, index asc).  topk arrays hold K entries (unused entries: index -1, lcp 0). */
int stocs_b200_reduce_best(stocs_b200_ctx* ctx, const float* lcp, int64_t H, int K,
                           int64_t* best_index, float* best_lcp, int64_t* topk_index,
                           float* topk_lcp);
int stocs_b200_reduce_best_device(stocs_b200_ctx* ctx, const float* d_lcp, int64_t H, int K,
                                  int64_t index_offset, int64_t* d_topk_index, float* d_topk_lcp,
                                  void* stream);

/* Every hypothesis with lcp > threshold (and > 0), ordered by (lcp descending, index ascending):
 * the filter + sort that opens clustering::greedy_clustering (src/pose_clustering.cpp:93-101).
 * lcp == NULL uses the resident array of the last score call.  STOCS_E_CAPACITY (with *n_out set)
 * when more than cap qualify. */
int stocs_b200_select_above(stocs_b200_ctx* ctx, const float* lcp, int64_t H, float threshold,
                            int64_t* index_out, float* lcp_out, int64_t cap, int64_t* n_out);

/* Point-to-plane ICP refinement: clustering::point_to_plane_icp (src/pose_clustering.cpp:123-141;
 * pcl::IterativeClosestPointWithNormals with setMaximumIterations(5),
 * setMaxCorrespondenceDistance(0.035), source = segment, target = model cloud with normals).
 * Host arrays in, xyz triples.  T16_out: accumulated transform (column-major), identity when the
 * first iteration already fails; aligned_pos3 (optional): the moved source, as the reference leaves
 * it in segment_cloud; pairs_per_iteration (optional): max_iterations entries; *converged = 0 when
 * an iteration found fewer than 3 correspondences or a singular system (PCL's "not converged";
 * the reference then sets offset_transform to identity, src/pose_clustering.cpp:136-139, and so
 * does the host shim clustering::point_to_plane_icp).  Needs no uploaded model or scene. */
int stocs_b200_icp_point_to_plane(stocs_b200_ctx* ctx, const float* src_pos3, int n_src,
                                  const float* tgt_pos3, const float* tgt_nrm3, int n_tgt,
                                  int max_iterations, float max_correspondence_distance,
                                  float* T16_out, float* aligned_pos3, int32_t* pairs_per_iteration,
                                  int32_t* iterations_done, int32_t* converged);

/* ---- fused online pipeline (run_stocs_estimation, src/stocs_match_one_object.cpp:79-165) ----
 * sample n_bases bases -> congruent sets -> at most max_sets transforms per base (when a base has
 * max_sets quads or more: the even spread floor(k * count / max_sets), k = 0..max_sets-1, over its
 * list in set order; see DESIGN.md on quirk 5) -> score -> best.
 * Everything stays on the device and is enqueued without a host round trip -- list lengths, offsets
 * and counts live in device memory, buffers are sized by capacities the context remembers -- and the
 * call synchronises once, on the summary below (a frame whose lists outgrow the capacities is run a
 * second time after growing them; the result is the same). */
typedef struct stocs_b200_pipeline_result {
  int32_t n_valid_bases;
  int64_t n_congruent_sets;
  int64_t n_transforms;
  int64_t best_index;        /* index into the transform list, -1 = no pose */
  float best_lcp;
  int32_t best_base;         /* PoseCandidate::base_index of the winner */
  float best_T_centred[16];
  float best_T_world[16];
} stocs_b200_pipeline_result;
int stocs_b200_run_pipeline(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                            stocs_b200_pipeline_result* result);
/* The same with the instance-mode sampler (edge map uploaded; src/stocs_match_one_object.cpp:89-92):
 * bases 1..n_bases (n_bases <= 255) are sampled in sequence -- each launch sees the prior decay and
 * the cached masks of its predecessors -- but enqueued back to back, without a host round trip per
 * base.  Like n_bases calls of sample_instance_base, it advances the context's instance state. */
int stocs_b200_run_pipeline_instance(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                     float dispersion, stocs_b200_pipeline_result* result);

/* ---- f3: greedy pose clustering (clustering::greedy_clustering, src/pose_clustering.cpp:79-122) ----
 * Keeps the candidates with lcp > acceptable_fraction * best_score (product in binary32), orders them
 * by lcp descending (equal lcps: index ascending, the shim's std::stable_sort), and walks them in that
 * order: a candidate is dropped when some already kept pose c gives get_pose_diff(candidate, c) with
 * rotation < min_angle AND translation < min_distance.  As in the reference the walk stops once MORE
 * than maximum_pose_count poses are kept, so up to maximum_pose_count + 1 come back.  The pose distance
 * is csrc/stocs_pose_math.h, which the host shim's get_pose_diff calls too: both keep the same poses.
 * Runs on the device in one CTA after a device sort; the call synchronises once. */
typedef struct stocs_b200_cluster_params {
  float acceptable_fraction;
  int32_t maximum_pose_count;   /* 0..1023; up to maximum_pose_count + 1 poses are returned (reference break rule) */
  float min_distance;           /* metres, translation of the world poses */
  float min_angle;              /* degrees, max Euler angle after symmetry folding */
  float sym_info[3];            /* per axis: 90, 180, 360 or anything else (no folding), as pose_clustering.cpp:31-48 */
} stocs_b200_cluster_params;

typedef struct stocs_b200_pose {
  int64_t index;       /* rank in the list of pushed transforms: the convention of pipeline_result.best_index */
  float lcp;
  int32_t base;        /* PoseCandidate::base_index, as pipeline_result.best_base */
  float T_centred[16];
  float T_world[16];   /* PoseCandidate::transform: the pose the clustering compares */
} stocs_b200_pose;     /* 144 bytes */

/* greedy_clustering over H host poses (world, column-major) and their LCPs.  Needs no model or scene.
 * index_out receives the kept indices in the order they were kept (index_out[0] is the best candidate
 * when any qualifies), *n_out their number.  STOCS_E_ARG: p or n_out NULL, maximum_pose_count outside
 * 0..1023, cap < maximum_pose_count + 1 (results are never partial), H outside 0 <= H < 2^31. */
int stocs_b200_cluster_poses(stocs_b200_ctx* ctx, const float* T16_world, const float* lcp, int64_t H,
                             float best_score, const stocs_b200_cluster_params* p,
                             int64_t* index_out, int64_t cap, int64_t* n_out);

/* run_pipeline[_instance] + greedy_clustering of its scored list, best_score = the run's best LCP.
 * The candidates are the transforms the fit pushed (a failed fit is never a candidate); poses[k].index
 * is the rank among them, so poses[0] is the result's best pose whenever there is one.  `result` is
 * what the plain call returns; the clustering is enqueued behind it and the call still synchronises
 * once.  cap < maximum_pose_count + 1 is STOCS_E_ARG. */
int stocs_b200_run_pipeline_clustered(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                      const stocs_b200_cluster_params* p, stocs_b200_pipeline_result* result,
                                      stocs_b200_pose* poses, int cap, int* n_poses);
int stocs_b200_run_pipeline_instance_clustered(stocs_b200_ctx* ctx, uint64_t seed, int n_bases, int max_sets,
                                               float dispersion, const stocs_b200_cluster_params* p,
                                               stocs_b200_pipeline_result* result, stocs_b200_pose* poses,
                                               int cap, int* n_poses);

/* ---- a15/f3: several objects of one frame, one context per object ------------------------------
 * A context holds one object's model, PPF table, scene and instance state and shares nothing with other
 * contexts, so a caller who keeps one context per object also keeps every model resident across frames.
 * These two calls give K such contexts a frame's work together: every object's work is enqueued on its
 * own context's stream, stage by stage across the objects, and the host waits once at the end, so the
 * objects' chains of small launches overlap on the device.  Every object's device buffers are grown before
 * any object's work is enqueued (growth frees memory, which waits for the whole device).  Each context's work runs under
 * cudaSetDevice(ctx->device); the contexts may sit on different devices.
 *
 * Equivalence: object k's outcome is bit-identical to the single call on ctxs[k] (upload_scene on its
 * slice; run_pipeline, run_pipeline_instance, run_pipeline_clustered or run_pipeline_instance_clustered
 * with seeds[k] and cluster[k]), and each context ends in the state that single call leaves: centroid,
 * centred points, grid, candidate lists, kd-tree, class-weight bound, pixel range, reset instance state,
 * counters [2], [3] and [6]; instance mode advances each context's prior decay and mask cache.
 *
 * Empty slices (an object that is not visible): upload_scenes leaves that context with no scene (counters
 * [2], [3] and [6] zero) and marks it as holding an empty scene; run_pipelines then returns the no-pose result for it (zeros,
 * best_index and best_base -1, n_poses 0) and enqueues nothing for it.  The single calls are unchanged:
 * upload_scene with S = 0 is STOCS_E_ARG, run_pipeline without a scene STOCS_E_STATE.
 *
 * Validation happens before anything is enqueued on any context, and a rejected call changes no context:
 * n_objects < 1, a NULL entry or one context given twice (STOCS_E_ARG; the objects would share a stream
 * and scratch), NULL required arrays, offsets that do not start at 0 or decrease, a slice over 2^27
 * points, any argument check of the single call, a context without a model or without any scene (never
 * uploaded, or its last upload failed: STOCS_E_STATE), in instance mode an edge map or pixel coordinates
 * missing, in a clustered run a bad parameter record or cap < maximum_pose_count + 1.  The error text
 * ("<call>: object k: ...") names the object and is set on the failing context and on ctxs[0].
 *
 * Errors after validation (a CUDA error, a kernel error, non-finite coordinates found while centring):
 * the first in object order is returned; every other object completes as its single call would, the
 * failing context is left as its single call leaves it, and no stream has work pending on return.
 * An object whose capacities overflow (congruent code/quad buffers, candidate records) is grown and
 * enqueued again on its own, with the same result.  The input buffers are not referenced after return. */

/* Object k's scene = rows [offsets[k], offsets[k+1]) of the arrays stocs_b200_build_scene_clouds writes
 * (pos3, nrm3, class_p as class_probability, pixel_rc or NULL); offsets has n_objects + 1 entries. */
int stocs_b200_upload_scenes(stocs_b200_ctx* const* ctxs, int n_objects, const float* pos3, const float* nrm3,
                             const float* class_probability, const int32_t* pixel_rc, const int64_t* offsets);

/* upload_scenes, word for word, from device arrays, e.g. the outputs of build_scene_clouds_device: the arrays are
 * device memory on any device (a context on another device copies its slice with cudaMemcpyPeerAsync); offsets is a
 * host array.  Nothing scene-sized crosses to the host: the centroid, box, class-weight bound and pixel range of
 * each slice are reduced on the device and come back as one 64-byte record per context (the host lays out the
 * grid from it), the index build returns its two list lengths as upload_scenes does, and the reference kd-tree is
 * built on the device beside the index build and joined by the first scoring launch.  Everything else moves
 * device to device.  d_nrm3, d_class_probability and d_pixel_rc (may be NULL) are on the device of d_pos3; a
 * pointer that is not device memory is STOCS_E_ARG.  stream (a cudaStream_t of that device; NULL is its default
 * stream): the call's work is ordered after what the caller has queued on it so far. */
int stocs_b200_upload_scenes_device(stocs_b200_ctx* const* ctxs, int n_objects, const float* d_pos3,
                                    const float* d_nrm3, const float* d_class_probability, const int32_t* d_pixel_rc,
                                    const int64_t* offsets, void* stream);

/* instance_mode 0 or 1; cluster: NULL (plain run) or n_objects parameter records (sym_info is per
 * object); results: n_objects records; poses: n_objects * cap records, object k's at poses + k * cap, and
 * n_poses: n_objects entries (both used by a clustered run only; n_poses is zeroed when given). */
int stocs_b200_run_pipelines(stocs_b200_ctx* const* ctxs, int n_objects, const uint64_t* seeds, int n_bases,
                             int max_sets, int instance_mode, float dispersion,
                             const stocs_b200_cluster_params* cluster, stocs_b200_pipeline_result* results,
                             stocs_b200_pose* poses, int cap, int* n_poses);

/* ---- e: multi-GPU, hypothesis sharding (SURVEY.md section 8e) -------------------------------
 * The reference scores its hypotheses in one sequential loop (src/stocs.cpp:990-998); they are
 * independent, so the list is split into contiguous blocks, one per GPU.  Every GPU holds a replica
 * of the scene index and model tables (upload_model / upload_scene on each context), scores its
 * block, keeps its K best as 64-byte records, and ONE ncclAllGather (NVLink / NVSwitch) hands every
 * rank all nranks*K records; the merge orders them by (lcp descending, global index ascending), so
 * record 0 is the reference's first strict maximum over the whole list (src/stocs.cpp:994).
 * NCCL is loaded at run time (dlopen of libnccl.so.2, or $STOCS_NCCL_LIB): contexts that never
 * call comm_* do not need it.
 *
 * One process per GPU: rank 0 calls comm_unique_id, the caller distributes the 128 bytes by any
 * transport (MPI, torch.distributed, a file), every rank calls comm_init (collective).
 * One process, several GPUs (what stocs_single uses with STOCS_DEVICES=0,1,..): group_create. */
typedef struct stocs_b200_record {
  float lcp;          /* 0 and index -1: empty slot */
  int32_t inliers;
  int64_t index;      /* position in the GLOBAL hypothesis list */
  float T[12];        /* rows 0..2 of the scored (centred) transform, row-major */
} stocs_b200_record;  /* 64 bytes */

#define STOCS_B200_UNIQUE_ID_BYTES 128
int stocs_b200_comm_unique_id(void* id128);
int stocs_b200_comm_init(stocs_b200_ctx* ctx, const void* id128, int rank, int nranks);
int stocs_b200_comm_destroy(stocs_b200_ctx* ctx);
/* Block [lo, hi) of ceil(H / nranks) hypotheses owned by `rank`. */
void stocs_b200_shard_range(int64_t H, int rank, int nranks, int64_t* lo, int64_t* hi);

/* Score the local block (H_local transforms whose first global index is index_offset), reduce it to
 * the K best (K <= 32), all-gather, merge: d_topk_out receives the K best records of the WHOLE list
 * on every rank.  Device pointers; runs on `stream` (NULL: the context stream) without
 * synchronising.  Without comm_init (or nranks 1) the collective is skipped.  Collective call:
 * every rank must make it, also with H_local == 0. */
int stocs_b200_score_sharded_device(stocs_b200_ctx* ctx, const float* d_T16_local, int64_t H_local,
                                    int64_t index_offset, int K, stocs_b200_record* d_topk_out,
                                    void* stream);
/* Same with host buffers (page-locked transforms are read in place, pageable ones are staged);
 * synchronises.  lcp_local / inliers_local (may be NULL) receive the local block's results. */
int stocs_b200_score_sharded(stocs_b200_ctx* ctx, const float* T16_local, int64_t H_local,
                             int64_t index_offset, int K, stocs_b200_record* topk_out,
                             float* lcp_local, int32_t* inliers_local);

/* Single-process group over n_dev devices (SURVEY.md section 8b: create(device_ids, n_dev)).
 * group_ctx(i) is the context of device i (upload model / scene through group_upload_* or per
 * context).  group_score_best splits the H host transforms across the devices, scores, gathers and
 * merges as above; lcp / inliers (may be NULL) receive the full per-hypothesis results. */
typedef struct stocs_b200_group stocs_b200_group;
int stocs_b200_group_create(stocs_b200_group** out, const int* device_ids, int n_dev);
void stocs_b200_group_destroy(stocs_b200_group* g);
int stocs_b200_group_size(stocs_b200_group* g);
stocs_b200_ctx* stocs_b200_group_ctx(stocs_b200_group* g, int i);
const char* stocs_b200_group_last_error(stocs_b200_group* g);
int stocs_b200_group_set_params(stocs_b200_group* g, float distance_threshold, int ppf_tr_discretization,
                                int ppf_rot_discretization);
int stocs_b200_group_upload_model(stocs_b200_group* g, const float* pos3, const float* nrm3, int M);
int stocs_b200_group_upload_scene(stocs_b200_group* g, const float* pos3, const float* nrm3,
                                  const float* class_probability, const int32_t* pixel_rc, int S);
int stocs_b200_group_score_best(stocs_b200_group* g, const float* T16, int64_t H, int K,
                                stocs_b200_record* topk_out, float* lcp, int32_t* inliers);

/* ---- diagnostics ---------------------------------------------------------------------------
 * [0] score kernels launched and [1] NN queries resolved by the kd-tree tie path, both accumulated
 * over the lifetime of the context; [2] grid cells and [3] replicated candidate records of the
 * current scene index; [4] / [5] hypotheses the device top-K path (score_sharded_device,
 * group_score_best without per-hypothesis outputs) left unscored because they provably cannot
 * enter the top K, rejected on the prefilter count (a launch of more than 300 000 hypotheses: the
 * survivor count on the fine occupancy map; otherwise loop 1's coarse count) / before a queue drain,
 * accumulated over the
 * lifetime of the context; [6] and [7] are internal; [8] hypotheses of the same path rejected
 * after the brick-bit refinement of the coarse survivors, which runs between the two, accumulated
 * likewise. */
int stocs_b200_get_counters(stocs_b200_ctx* ctx, int64_t* counters, int n);
/* Data-dependent work of ONE scoring launch over H device-resident transforms, counted exactly by a
 * counting instantiation of the scoring kernel (results discarded, not for timing).  counters (up
 * to 9): [0] NN queries = H*|M|, [1] queries that survive the shared-memory coarse occupancy test,
 * [2] 16-byte brick records fetched, [3] queries whose grid cell is occupied (queued),
 * [4] candidate records examined (16 B each), [5] queries with a scene point within the distance
 * threshold (one 16-byte attribute fetch each), [6] inliers, [7] queue drains, [8] H.
 * bench.py derives SURVEY.md section 8(d)'s data-dependent byte figure from these. */
int stocs_b200_score_counters(stocs_b200_ctx* ctx, const float* d_T16, int64_t H, int64_t* counters,
                              int n);
/* Test hook: the coarse-survivor count of each of H device-resident transforms, as the device top-K
 * path computes it to order its claims: model points whose block of the coarse occupancy map is
 * occupied (counters[1] of score_counters on that one transform, for a finite transform and |M| a
 * multiple of 32), or |M| for a transform whose grid map is not finite or too large to evaluate
 * without overflow.  counts: H host int32. */
int stocs_b200_debug_survivor_counts(stocs_b200_ctx* ctx, const float* d_T16, int64_t H, int32_t* counts);
/* Test hook: the count a top-K launch of more than 300 000 hypotheses actually orders and stops its claims
 * by: the same test on the scene's fine occupancy map (blocks of 2^fine_shift cells per axis, at most
 * the coarse map's 2^coarse_shift).  For a transform whose grid map is below the overflow limit at both
 * scales it is at most the coarse count and at least the transform's inlier count.  fine_shift (optional):
 * 2 host int32, {fine_shift, coarse_shift} of the current scene. */
int stocs_b200_debug_fine_survivor_counts(stocs_b200_ctx* ctx, const float* d_T16, int64_t H, int32_t* counts,
                                          int32_t* fine_shift);
/* name + average duration (ms, CUDA events on the context stream) of the dominant kernel of the
 * most recent score call; used by bench.py for the roofline line. */
int stocs_b200_last_kernel_ms(stocs_b200_ctx* ctx, float* ms);
/* Mean / max duration (ms) of the scoring kernel over the timed launches since the last reset (at
 * most the 512 most recent), from CUDA event pairs recorded around each launch on the stream it
 * ran on.  Synchronises with those launches.  reset != 0 restarts the window. */
int stocs_b200_kernel_ms_stats(stocs_b200_ctx* ctx, int reset, int32_t* n_launches, float* mean_ms,
                               float* max_ms);
/* Host-only test hook (no context, no GPU): builds the reference kd-tree (kdtree.h:461-538: split at the
 * middle of the longest box side, leaves of <= 64 points, depth <= 32) over n points exactly as
 * upload_scene does for the scoring kernel's tie rule, and returns the original index of every point
 * in leaf order plus the node count.  The build's partition is a branch-free rewrite of the reference's
 * loop; the CPU tests compare its output with the oracle's literal restatement. */
int stocs_b200_host_kdtree_order(const float* pos3, int n, int32_t* leaf_order, int32_t* n_nodes);
/* Test hook: the same kd-tree over n finite host points (taken as given, not centred), built on the context's
 * device as upload_scenes_device builds it (on_device != 0) or on the host as upload_scene builds it.  leaf_order:
 * n original indices in leaf order; n_nodes: node count; nodes_out (may be NULL, 3 * (n + 3) entries): every node
 * in pre-order from the root, first child first, as (leaf, bits of the split value, split axis or leaf size), so
 * that two builds can be compared whatever their node numbering.  The context's scene is not touched. */
int stocs_b200_debug_kdtree(stocs_b200_ctx* ctx, const float* pos3, int n, int on_device, int32_t* leaf_order,
                            int32_t* n_nodes, int32_t* nodes_out);
/* Test hook: the samplers decide the integer part of a PPF angle (int(atan2(y, x) * 180 / M_PI)) and the
 * side of 30 degrees an internal angle lies on from fp32 estimates whenever those are safely away from
 * the deciding thresholds, and by the pinned binary64 evaluation otherwise.  For n pairs (y, x) this
 * returns the estimate, the pinned value, both integer parts, and -- with d = x -- both forms of the
 * 30-degree predicate, so that a test can bound the estimate's error and compare the decisions. */
int stocs_b200_debug_angle_estimates(stocs_b200_ctx* ctx, const float* y, const float* x, int64_t n, float* est_deg,
                                     double* pinned_deg, int32_t* fast_floor, int32_t* pinned_floor,
                                     uint8_t* below30_fast, uint8_t* below30_pinned);

#ifdef __cplusplus
}
#endif
#endif /* STOCS_B200_H_ */
