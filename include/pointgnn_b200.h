/*
 * pointgnn_b200.h - C ABI of libpointgnn_b200.so
 *
 * B200 (sm_100a) implementation of Point-GNN's per-frame message-passing hot
 * path.  Every entry point replaces one piece of the reference's Python/TF path;
 * the reference interface each one stands in for is cited as
 * /root/reference/<file>:<line>.
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless the parameter name ends in _host.
 *  - Row-major, C-contiguous arrays; float = IEEE fp32, indices = int32.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *  - Return value: 0 = ok, <0 = error (PG_ERR_*); pg_last_error() gives the
 *    message of the last failure on the calling thread.  Nothing aborts.
 *  - Kernels never retain caller pointers after the call returns; temporary
 *    buffers come from the stream-ordered allocator (cudaMallocAsync).
 *  - Multi-frame batches follow the reference's batch_data semantics
 *    (/root/reference/train.py:135-171): frames are concatenated, `frame_ptr`
 *    [num_frames+1] gives each frame's row range, and all emitted indices are
 *    GLOBAL (already offset), i.e. exactly what batch_data would produce.
 */
#ifndef POINTGNN_B200_H_
#define POINTGNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PG_API __attribute__((visibility("default")))
#else
#define PG_API
#endif

#define PG_OK 0
#define PG_ERR_INVALID_ARGUMENT (-1)
#define PG_ERR_CUDA (-2)
#define PG_ERR_CAPACITY (-3)   /* caller-provided output buffer too small   */
#define PG_ERR_RANGE (-4)      /* cloud extent / cell index exceeds key bits */
#define PG_ERR_UNSUPPORTED (-5)

/* Library ABI version (bumped on any signature change). */
PG_API int pg_version(void);
/* Message of the last error on this thread ("" if none). */
PG_API const char* pg_last_error(void);
/* 1 if the visible device is sm_100 (B200); the tcgen05 kernels require it. */
PG_API int pg_device_is_sm100(void);
/* 1 if the tcgen05 (precision = 1) kernels are built in AND the device can run them. */
PG_API int pg_tc_available(void);

/* ------------------------------------------------------------------------ *
 * Input stage: the step before the path (SURVEY 8f-2; reference dataset/kitti_dataset.py)
 * ------------------------------------------------------------------------ */

/*
 * KittiDataset.get_cam_points_in_image_with_rgb (kitti_dataset.py:666-689) for a batch of frames:
 * velodyne points -> camera frame (velo_points_to_cam, :998-1006: float32 matmul + float32 offset) ->
 * keep z > 0.1 and a projection strictly inside the image (cam_points_to_image, :1036-1052, float64) ->
 * attributes [reflectance] or, with images, [reflectance, r, g, b] (rgb_to_cam_points, :990-996).
 *   velo_points        [M,4] fp32 (x, y, z, reflectance) = the bytes of the .bin files, 16-byte aligned
 *   frame_ptr          [num_frames+1] int32 over the M points
 *   velo_to_cam_host   (host) [num_frames][4][4] fp32  calib['velo_to_cam'] (kitti_dataset.py:510-511)
 *   cam_to_image_host  (host) [num_frames][3][4] fp64  calib['cam_to_image'] (:501)
 *   image_size_host    (host) [num_frames][2] int32    (width, height) of the frame's image
 *   images / image_offset_host  optional: concatenated [H,W,3] uint8 BGR images (cv2.imread layout) and the
 *                      byte offset of each frame's image; required when attr_channels == 4
 * Output order = input order.  out_xyz [N,3], out_attr [N,attr_channels], out_frame_ptr [num_frames+1];
 * *out_num_points_host = N (one host round trip); PG_ERR_CAPACITY when capacity < N.
 */
PG_API int pg_cam_points_in_image(const float* velo_points, const int32_t* frame_ptr, int32_t num_frames,
                           int64_t num_points, const float* velo_to_cam_host,
                           const double* cam_to_image_host, const int32_t* image_size_host,
                           const uint8_t* images, const int64_t* image_offset_host, float* out_xyz,
                           float* out_attr, int32_t attr_channels, int64_t capacity,
                           int32_t* out_frame_ptr, int64_t* out_num_points_host, void* stream);

/* ------------------------------------------------------------------------ *
 * Graph construction  (reference models/graph_gen.py)
 * ------------------------------------------------------------------------ */

/*
 * Voxel keypoint selection = multi_layer_downsampling (open3d.voxel_down_sample,
 * graph_gen.py:41-45) + the kd-tree 1-NN snap of multi_layer_downsampling_select
 * (graph_gen.py:84-88), for one voxel scale, over a batch of frames.
 *
 *   xyz        [N,3] fp32 points of all frames, concatenated
 *   frame_ptr  [num_frames+1] int32, frame f owns rows frame_ptr[f]..frame_ptr[f+1)
 *   voxel_size [3] (host) fp64 voxel edge per axis (= base_voxel_size*graph_scale)
 *   out_keypoint_idx [capacity] int32: GLOBAL row index of the original point
 *              nearest to each voxel centroid (fp64 distance, ties -> lowest index);
 *              per frame in ascending linear-voxel-key order; duplicates kept.
 *   out_kp_frame_ptr [num_frames+1] int32 keypoint range of each frame
 *   out_num_keypoints_host  (host) total K.  The call synchronises the stream.
 * Returns PG_ERR_CAPACITY (and the needed K in *out_num_keypoints_host) if
 * capacity < K; capacity = N always suffices.
 */
PG_API int pg_voxel_keypoints(const float* xyz, const int32_t* frame_ptr, int32_t num_frames,
                       int64_t num_points, const double* voxel_size_host,
                       int32_t* out_keypoint_idx, int64_t capacity,
                       int32_t* out_kp_frame_ptr, int64_t* out_num_keypoints_host,
                       void* stream);

/*
 * multi_layer_downsampling for ONE scale (graph_gen.py:11-47, Open3D branch :41-45): the fp64 centroid of
 * every occupied voxel of the cloud, per frame in ascending linear-voxel-key order (the oracle's canonical
 * order; Open3D's own order is unspecified).
 *   out_centroids [capacity,3] fp64 (device), out_frame_ptr [num_frames+1], out_num_host (host) = K.
 * Synchronises the stream; PG_ERR_CAPACITY as pg_voxel_keypoints.
 */
PG_API int pg_voxel_centroids(const float* xyz, const int32_t* frame_ptr, int32_t num_frames,
                       int64_t num_points, const double* voxel_size_host, double* out_centroids,
                       int64_t capacity, int32_t* out_frame_ptr, int64_t* out_num_host, void* stream);

/*
 * multi_layer_downsampling_select for a level whose scale differs from the previous level's
 * (graph_gen.py:82-88) in the general case of several distinct scales (graph_gen.py:17-23,76-88): the
 * voxel centroids of the ORIGINAL cloud `xyz` (:41-45), each snapped to the nearest vertex of the
 * PREVIOUS level `base_xyz` [num_base,3] / `base_frame_ptr` (kd_tree 1-NN, :84-87; fp64 distance, ties ->
 * lowest index, same frame only).  out_keypoint_idx [K] are GLOBAL rows of base_xyz.  With base == xyz
 * this equals pg_voxel_keypoints.  Other arguments and errors as pg_voxel_keypoints.
 */
PG_API int pg_voxel_keypoints_select(const float* xyz, const int32_t* frame_ptr, int32_t num_frames,
                              int64_t num_points, const double* voxel_size_host, const float* base_xyz,
                              const int32_t* base_frame_ptr, int64_t num_base, int32_t* out_keypoint_idx,
                              int64_t capacity, int32_t* out_kp_frame_ptr,
                              int64_t* out_num_keypoints_host, void* stream);

/*
 * multi_layer_downsampling / multi_layer_downsampling_select with add_rnd3d=True and the centroid method
 * (graph_gen.py:24-39, 82-88; no shipped config - the training configs use downsample_method 'random'):
 *   voxel index = floor_divide((p - frame_min)[float32] + voxel * shift[frame], voxel) in float64 (:25-28),
 *   shift_host = (host) [num_frames][3] the np.random.random((1,3)) draw of each frame;
 *   one centroid per occupied voxel, per frame in ascending linear-voxel-key order (:30-36) -> out_centroids
 *   [capacity,3] fp64 (optional);  with base_xyz: each centroid snapped to the nearest base vertex (:84-87) ->
 *   out_keypoint_idx [K] rows of base_xyz (base_xyz == NULL <=> out_keypoint_idx == NULL).
 * The reference sums a voxel's points in float32 in argsort order (np.add.reduceat, :36-37; the order among equal
 * keys is numpy's unstable sort); this call sums in fp64 in ascending point order: centroids agree to ~1e-6
 * relative, so a snapped index can differ where two vertices are equidistant within that (two-point voxels).
 */
PG_API int pg_voxel_keypoints_rnd3d(const float* xyz, const int32_t* frame_ptr, int32_t num_frames,
                             int64_t num_points, const double* voxel_size_host, const double* shift_host,
                             const float* base_xyz, const int32_t* base_frame_ptr, int64_t num_base,
                             int32_t* out_keypoint_idx, double* out_centroids, int64_t capacity,
                             int32_t* out_kp_frame_ptr, int64_t* out_num_keypoints_host, void* stream);

/*
 * Radius-neighbour graph = gen_disjointed_rnn_local_graph_v3
 * (graph_gen.py:197-220; ball_tree radius_neighbors, fp64 predicate
 * ((dx*dx+dy*dy)+dz*dz) <= r*r on float32-valued coordinates, inclusive), with
 * num_neighbors <= 0 (no random cap: the inference path, run.py:219-222).
 * Two passes so the caller owns the edge buffer:
 *
 *   pg_radius_graph_count: out_row_ptr [K+1] int32 (CSR by destination/centre),
 *                          *out_num_edges_host = E (synchronises the stream).
 *   pg_radius_graph_fill:  out_src [E] int32 source (point) index of every edge,
 *                          ascending inside a row; out_dst [E] int32 (may be NULL)
 *                          the expanded destination index, so that
 *                          stack([out_src,out_dst],1) == the reference's [E,2]
 *                          `vertices` array after a (dst,src) sort.
 *
 *   points  [P,3] fp32 source set,  point_frame_ptr  [num_frames+1]
 *   centers [K,3] fp32 centre set,  center_frame_ptr [num_frames+1]
 * Edges only connect points and centres of the same frame.
 */
PG_API int pg_radius_graph_count(const float* points, const int32_t* point_frame_ptr,
                          const float* centers, const int32_t* center_frame_ptr,
                          int32_t num_frames, int64_t num_points, int64_t num_centers,
                          double radius, int32_t* out_row_ptr, int64_t* out_num_edges_host,
                          void* stream);
PG_API int pg_radius_graph_fill(const float* points, const int32_t* point_frame_ptr,
                         const float* centers, const int32_t* center_frame_ptr,
                         int32_t num_frames, int64_t num_points, int64_t num_centers,
                         double radius, const int32_t* row_ptr, int64_t num_edges,
                         int32_t* out_src, int32_t* out_dst, void* stream);

/*
 * Single-call variant (one grid build, count -> scan -> fill) writing into a caller buffer of
 * `capacity` edges.  Returns PG_ERR_CAPACITY with the needed E in *out_num_edges_host when
 * the buffer is too small (out_row_ptr is valid in that case).
 */
PG_API int pg_radius_graph(const float* points, const int32_t* point_frame_ptr, const float* centers,
                    const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                    int64_t num_centers, double radius, int32_t* out_row_ptr, int32_t* out_src,
                    int32_t* out_dst, int64_t capacity, int64_t* out_num_edges_host, void* stream);

/*
 * pg_radius_graph with the per-axis `scale` argument of gen_disjointed_rnn_local_graph_v3 (graph_gen.py:203-206:
 * points_xyz / np.array(scale), center_xyz / np.array(scale) - a float64 division of the float32 coordinates - before
 * the ball tree is built).  scale_host = (host) [3] positive divisors, NULL = no scaling (= pg_radius_graph); the
 * division is done in float64 inside the kernels, the predicate is evaluated on the quotients exactly as above.
 */
PG_API int pg_radius_graph_scaled(const float* points, const int32_t* point_frame_ptr, const float* centers,
                           const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                           int64_t num_centers, double radius, const double* scale_host, int32_t* out_row_ptr,
                           int32_t* out_src, int32_t* out_dst, int64_t capacity, int64_t* out_num_edges_host,
                           void* stream);

/*
 * gen_multi_level_local_graph_v3 (graph_gen.py:155-195) for the two-level structure of every shipped
 * config - level 0: original cloud -> keypoints of ONE voxel scale (radius0), level 1: those keypoints
 * -> themselves (radius1; equal consecutive scales, graph_gen.py:76-81) - as ONE call with ONE host
 * round trip.  Keypoint and edge counts stay on the device between the stages; the caller passes
 * over-sized buffers (kp_capacity <= num_points rows, capacity0 / capacity1 edges) and gets
 * out_sizes_host = {K, E0, E1}.  PG_ERR_CAPACITY (sizes filled in) means a buffer was too small and the
 * call must be repeated with larger ones.  Outputs as pg_voxel_keypoints / pg_radius_graph:
 *   out_keypoint_idx [K], out_kp_frame_ptr [num_frames+1], out_kp_xyz [K,3] = xyz[out_keypoint_idx],
 *   out_row_ptr{0,1} [kp_capacity+1] (entries beyond K repeat E), out_src / out_dst [E] per level.
 */
PG_API int pg_multi_level_graph(const float* xyz, const int32_t* frame_ptr, int32_t num_frames,
                         int64_t num_points, const double* voxel_size_host, double radius0, double radius1,
                         int32_t* out_keypoint_idx, int64_t kp_capacity, int32_t* out_kp_frame_ptr,
                         float* out_kp_xyz, int32_t* out_row_ptr0, int32_t* out_src0, int32_t* out_dst0,
                         int64_t capacity0, int32_t* out_row_ptr1, int32_t* out_src1, int32_t* out_dst1,
                         int64_t capacity1, int64_t* out_sizes_host, void* stream);

/*
 * Training-time graph path (train.py:88-90 with configs/*_train_config: downsample_method 'random',
 * add_rnd3d true, num_neighbors 256).  The reference draws from Python / NumPy global generators, so
 * these two calls take their randomness as ARGUMENTS; everything else is reproduced exactly.
 *
 * pg_random_keypoints = multi_layer_downsampling_random for one scale (graph_gen.py:92-153):
 *   xyz / frame_ptr [num_points]: the ORIGINAL cloud, whose per-frame minimum frame_min is the grid origin of every
 *   level (:107-110); base_xyz / base_frame_ptr [num_base]: the points voxelised at this scale, the previous level's
 *   vertices (:115);
 *   voxel index of every base point: floor_divide(p - frame_min, voxel) in float32 (shift_host == NULL, add_rnd3d
 *   false and a scalar voxel size, :123-124) or floor_divide(p - frame_min + voxel * shift, voxel) in float64
 *   (:126-128), shift_host = (host) [num_frames][3] the np.random.random((1,3)) draw of each frame; an all-zero
 *   shift gives the float64 quotient NumPy computes for an array voxel size without add_rnd3d;
 *   one keypoint per occupied voxel, voxels in order of first appearance (the dict order of :133-139);
 *   keypoint o = the floor(uniform[o] * count)-th point (ascending index) of its voxel - uniform [num_base]
 *   device fp32 in [0,1) stands in for random.choice (:143-146).
 * Outputs as pg_voxel_keypoints: out_keypoint_idx [K] rows of base_xyz.
 */
PG_API int pg_random_keypoints(const float* xyz, const int32_t* frame_ptr, int32_t num_frames,
                        int64_t num_points, const double* voxel_size_host, const double* shift_host,
                        const float* base_xyz, const int32_t* base_frame_ptr, int64_t num_base,
                        const float* uniform, int32_t* out_keypoint_idx, int64_t capacity,
                        int32_t* out_kp_frame_ptr, int64_t* out_num_keypoints_host, void* stream);

/*
 * The random neighbour cap of gen_disjointed_rnn_local_graph_v3 (graph_gen.py:210-214) applied to a CSR graph
 * (row_ptr [num_rows+1], src [E], rows ascending as pg_radius_graph emits them): rows with at most
 * num_neighbors entries are copied, longer rows keep exactly num_neighbors distinct entries - those with the
 * smallest hash(seed, row, src) priority, a uniformly random subset for a random seed (np.random.choice(...,
 * replace=False)) - in ascending source order.  *out_num_edges_host = E'.
 */
PG_API int pg_cap_neighbors(const int32_t* row_ptr, const int32_t* src, int64_t num_rows, int32_t num_neighbors,
                     uint32_t seed, int32_t* out_row_ptr, int32_t* out_src, int32_t* out_dst,
                     int64_t capacity, int64_t* out_num_edges_host, void* stream);

/* ------------------------------------------------------------------------ *
 * GNN ops  (reference models/gnn.py)
 * ------------------------------------------------------------------------ */

/*
 * graph_scatter_max_fn (gnn.py:106-109) = tf.math.unsorted_segment_max:
 * out[k,c] = max over edges e with centers[e]==k of features[e,c]; empty segment
 * -> -FLT_MAX (numeric_limits<float>::lowest()).  `centers` may be in any order.
 */
PG_API int pg_scatter_max(const float* features, const int32_t* centers, int64_t num_edges,
                   int32_t num_channels, int64_t num_centers, float* out, void* stream);

/*
 * graph_scatter_sum_fn / graph_scatter_mean_fn (gnn.py:111-119) = tf.math.unsorted_segment_sum / unsorted_segment_mean
 * (the aggregation plug-ins no shipped config selects): out[k,c] = sum (mean) over edges e with centers[e]==k of
 * features[e,c]; an empty segment gives 0 for both (the mean divides by max(count, 1)).  fp32 accumulation, partial sums
 * combined with atomics (order not fixed, as in TF's GPU kernel).  Ids outside [0, num_centers) are dropped, as TF does.
 */
PG_API int pg_scatter_sum(const float* features, const int32_t* centers, int64_t num_edges,
                   int32_t num_channels, int64_t num_centers, float* out, void* stream);
PG_API int pg_scatter_mean(const float* features, const int32_t* centers, int64_t num_edges,
                    int32_t num_channels, int64_t num_centers, float* out, void* stream);

/* tf.gather(params, indices) for [R,C] fp32 rows (gnn.py:256-262,338-348). */
PG_API int pg_gather_rows(const float* params, int64_t num_rows, int32_t num_channels,
                   const int32_t* indices, int64_t num_indices, float* out, void* stream);

/*
 * One slim.fully_connected layer (gnn.py:63-80,93-103), normalizer NONE:
 *   out[M,N] = act(x[M,K] @ w[K,N] + bias[N]) (+ residual[M,N] if not NULL)
 * act: 0 = linear (the is_logits last layer), 1 = ReLU.
 * precision: 0 = fp32 FFMA, 1 = tcgen05 BF16x3 split (fp32-class accuracy).
 */
PG_API int pg_fully_connected(const float* x, int64_t m, int32_t k, const float* w, const float* bias,
                       int32_t n, int32_t act, const float* residual, float* out,
                       int32_t precision, void* stream);

/*
 * Fused per-edge MLP + segment max: the body of PointSetPooling.apply_regular
 * (gnn.py:256-277) and of GraphNetAutoCenter.apply_regular (gnn.py:338-365),
 * never materialising the [E, D] edge tensors.
 *
 *   mode PG_EDGE_POOL : e0 = concat(point_features[src], xyz_src[src] - xyz_dst[kp[dst]])
 *                       (feature first, then relative xyz; gnn.py:264-267)
 *   mode PG_EDGE_GNN  : e0 = concat(vertex_features[src], xyz_src[src] - xyz_dst[dst])
 *                       xyz_src = un-offset coords, xyz_dst = coords + auto-offset
 *                       (gnn.py:338-352; SURVEY fact 4)
 *   then num_layers x relu(. @ W_l + b_l)      (is_logits=False, gnn.py:99-103)
 *   then out[k,:] = max over the edges of destination k   (gnn.py:362-365)
 *
 *   src, dst     [E] int32; dst must be non-decreasing (CSR order, as produced by
 *                pg_radius_graph_fill and by the reference generator).
 *   dst_index    POOL: keypoint_indices [num_dst] int32 (row of xyz_dst per dst);
 *                GNN: NULL (identity)
 *   weights_host / biases_host: (host) arrays of num_layers DEVICE pointers,
 *                W_l is [dims[l], dims[l+1]] row-major, dims[0] = C_in + 3.
 *   dims_host    (host) [num_layers+1]
 *   out          [num_dst, dims[num_layers]]; empty segments get -FLT_MAX.
 *   precision    0 = fp32 FFMA, 1 = tcgen05 BF16x3 for the wide layers; may be OR-ed with
 *                PG_FLAG_TRUSTED_INDICES: the caller guarantees src / dst are in range (they come from
 *                pg_radius_graph, or passed pg_check_edges), so the call skips the device->host
 *                read-back of the range-error flag and does not synchronise the stream.  Out-of-range
 *                indices are still clamped on the device (never dereferenced), just not reported.
 */
#define PG_PRECISION_MASK 0xff
#define PG_FLAG_TRUSTED_INDICES 0x100
#define PG_EDGE_POOL 0
#define PG_EDGE_GNN 1
PG_API int pg_edge_mlp_max(int32_t mode, const float* features, int32_t num_feature_channels,
                    const float* xyz_src, const float* xyz_dst, const int32_t* dst_index,
                    const int32_t* src, const int32_t* dst, int64_t num_edges, int64_t num_src,
                    int64_t num_dst, const float* const* weights_host,
                    const float* const* biases_host, const int32_t* dims_host,
                    int32_t num_layers, float* out, int32_t precision, void* stream);

/*
 * Range check of an edge list: 0 <= src[e] < num_src and 0 <= dst[e] < num_dst for every e (what TF's
 * gather / unsorted_segment_max raise InvalidArgumentError for at sess.run, run.py:260).  Synchronises.
 */
PG_API int pg_check_edges(const int32_t* src, const int32_t* dst, int64_t num_edges, int64_t num_src,
                   int64_t num_dst, void* stream);

/* ------------------------------------------------------------------------ *
 * Prepared layers.  The reference creates its variables once (tf.variable_scope +
 * slim.fully_connected at graph-build time, gnn.py:63-80, models.py:113-163) and
 * restores them once (run.py:192-202); every sess.run then only computes.  The
 * equivalent here: pg_layer_create packs everything that depends on the weights
 * only (BF16 hi / lo tensor-core operand images, padded biases, the hoisted first
 * edge layer, the concatenated predictor heads) into an opaque handle; the
 * pg_layer_* calls below launch compute kernels only.  The handle keeps the
 * caller's weight pointers (the fp32 FFMA paths read them directly): they must
 * outlive it.  Handles are immutable after creation and may be shared by streams.
 *
 *   kind PG_LAYER_MLP        num_layers fully-connected layers (gnn.py:34-104),
 *                            dims_host [num_layers + 1].
 *   kind PG_LAYER_EDGE_POOL  PointSetPooling's point MLP + max (gnn.py:256-277)
 *   kind PG_LAYER_EDGE_GNN   GraphNetAutoCenter's edge MLP + max (gnn.py:338-365)
 *                            dims_host [num_layers + 1], dims[0] = C_in + 3 (as pg_edge_mlp_max).
 *   kind PG_LAYER_PREDICTOR  ClassAwarePredictor (gnn.py:133-163, models.py:60-64):
 *                            dims_host = {D, H, C, box_len}; layers in the order the
 *                            reference creates them: cls fc (D->H), cls fc_1 (H->C), then
 *                            for every class c: loc fc (D->H), fc_1 (H->H), fc_2 (H->box_len);
 *                            num_layers = 2 + 3 C.
 *   precision 0 = fp32 FFMA, 1 = tcgen05 BF16x3 wherever the shapes allow.
 * ------------------------------------------------------------------------ */
typedef struct pg_layer pg_layer;
#define PG_LAYER_MLP 0
#define PG_LAYER_EDGE_POOL 1
#define PG_LAYER_EDGE_GNN 2
#define PG_LAYER_PREDICTOR 3
PG_API int pg_layer_create(int32_t kind, const float* const* weights_host, const float* const* biases_host,
                    const int32_t* dims_host, int32_t num_layers, int32_t precision, void* stream,
                    pg_layer** out_layer);
PG_API int pg_layer_destroy(pg_layer* layer);

/* multi_layer_neural_network_fn / multi_layer_fc_fn (gnn.py:34-104) on a prepared chain:
 * ReLU after every layer except - when last_linear != 0 (is_logits=True) - the last;
 * `residual` [m, dims[last]] (optional) is added to the last layer's output (gnn.py:346, 372). */
PG_API int pg_layer_mlp(const pg_layer* layer, const float* x, int64_t m, int32_t last_linear,
                 const float* residual, float* out, void* stream);

/* pg_edge_mlp_max on a prepared edge layer; flags: 0 or PG_FLAG_TRUSTED_INDICES. */
PG_API int pg_layer_edge_mlp_max(const pg_layer* layer, const float* features, const float* xyz_src,
                          const float* xyz_dst, const int32_t* dst_index, const int32_t* src,
                          const int32_t* dst, int64_t num_edges, int64_t num_src, int64_t num_dst,
                          float* out, int32_t flags, void* stream);

/* ClassAwarePredictor.apply_regular (gnn.py:133-163) + postprocess (models.py:165-168):
 * logits [m, C], boxes [m, C, box_len], probs [m, C] (probs may be NULL). */
PG_API int pg_layer_predictor(const pg_layer* layer, const float* x, int64_t m, float* logits, float* boxes,
                       float* probs, void* stream);

/* Row-wise softmax, MultiLayerFastLocalGraphModelV2.postprocess (models.py:165-168). */
PG_API int pg_softmax_rows(const float* logits, int64_t num_rows, int32_t num_classes, float* out,
                    void* stream);

/* ------------------------------------------------------------------------ *
 * Post-processing: the step after the path (SURVEY 8f-1; reference run.py:265-325)
 * ------------------------------------------------------------------------ */

/*
 * classaware_all_class_box_decoding (models/box_encoding.py:265-299) for every (vertex, class) pair.
 *   class_table_host  (host) [C][4] floats per class label: median l, h, w (box_encoding.py:211-229) and the
 *                     yaw offset (0 for the "horizontal" label, pi/2 for the "vertical" one); l <= 0 marks
 *                     labels that are not decoded (Background, DontCare).
 *   out_boxes [K, C, 7] = (x, y, z, l, h, w, yaw), float32 arithmetic as the reference's NumPy code.
 */
PG_API int pg_decode_boxes(const float* box_encodings, const float* xyz, int64_t num_vertices,
                    int32_t num_classes, const float* class_table_host, float* out_boxes, void* stream);

/*
 * Candidate selection + decoding + NMS for a batch of frames (run.py:265-325):
 *   candidates      class c of vertex v iff 0 < c < C-1 and probs[v,c] > 1/C (run.py:281-284), labels 2/4/6
 *                   folded onto 1/3/5 (run.py:291-293), decoded with pg_decode_boxes' rule;
 *   NMS             nms.nms_boxes_3d_uncertainty (models/nms.py:133-170, 256-270) with
 *                   overlapped_boxes_3d_fast_poly (nms.py:64-88) and top_k = -1: score-sorted greedy
 *                   suppression inside a class; flags bit 0 (PG_NMS_MERGE): the kept box becomes the
 *                   coordinate-wise median of itself and the boxes it suppresses; bit 1 (PG_NMS_RESCORE): its
 *                   score grows by sum_j score_j * IoU(merged box, box_j).  flags 0 / 1 / 2 are nms_boxes_3d's
 *                   siblings (nms.py:172-240).
 *   frame_ptr [num_frames+1] partitions the K vertices; frames are processed independently.
 * Outputs (caller buffers of `capacity` detections, frame by frame, in score order of the candidates):
 *   out_label / out_box [.,7] / out_score / out_index (= flat v*C + c of the kept candidate, i.e.
 *   box_indices[nms_indices] of run.py), out_det_frame_ptr [num_frames+1];
 *   out_cand_index [K*(C-2)] + out_cand_frame_ptr [num_frames+1] (optional): all candidates in ascending
 *   (v, c) order = run.py's box_indices (the KITTI writer's occlusion rescoring needs them, run.py:395-404);
 *   out_sizes_host = {detections, candidates}.
 * max_candidates_per_frame bounds the pairwise bit matrix; PG_ERR_CAPACITY when a frame exceeds it or the
 * detection buffer is too small.  Two host round trips (matrix width, result size).
 */
#define PG_NMS_MERGE 1
#define PG_NMS_RESCORE 2
#define PG_NMS_INT_CORNERS 4   /* pg_nms_boxes_3d only: np.int32(corners * appr_factor), nms.py:114 */
PG_API int pg_postprocess(const float* probs, const float* box_encodings, const float* xyz,
                   const int32_t* frame_ptr, int32_t num_frames, int64_t num_vertices, int32_t num_classes,
                   const float* class_table_host, double overlapped_thres, int32_t flags,
                   int64_t max_candidates_per_frame, int32_t* out_label, float* out_box, float* out_score,
                   int32_t* out_index, int64_t capacity, int32_t* out_det_frame_ptr,
                   int32_t* out_cand_index, int32_t* out_cand_frame_ptr, int64_t* out_sizes_host,
                   void* stream);

/* The NMS stage alone on caller-provided boxes (models/nms.py:243-301's four entry points):
 * class_labels / boxes [B,7] / scores, frame_ptr [num_frames+1] over the B boxes; out_index = position of the
 * kept box in the input (the reference's `attributes=np.arange(B)` convention, run.py:305). */
PG_API int pg_nms_boxes_3d(const int32_t* class_labels, const float* boxes, const float* scores,
                    const int32_t* frame_ptr, int32_t num_frames, int64_t num_boxes, double overlapped_thres,
                    double appr_factor, int32_t flags, int64_t max_candidates_per_frame, int32_t* out_label,
                    float* out_box, float* out_score, int32_t* out_index, int64_t capacity,
                    int32_t* out_det_frame_ptr, int64_t* out_sizes_host, void* stream);

/* tcgen05 kernel launches so far (which: 0 = fused edge MLP + segment max, 1 = dense layer);
 * lets callers and tests verify that the tensor-core path, not the FFMA path, actually ran. */
PG_API int64_t pg_tc_launch_count(int32_t which);

/* Number of kernels this library has launched in the calling process (bench.py). */
PG_API int64_t pg_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* POINTGNN_B200_H_ */
