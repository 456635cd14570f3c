/*
 * pcr_b200.h -- C ABI of the B200-native k-nearest-neighbour engine that replaces the KNN hot
 * path of nahomes-15/pointclouds-rs ("pcrs").  Plain pointers and sizes only; no C++/torch types.
 *
 * What each entry point replaces (reference file:line, relative to the pcrs repository root):
 *
 *   pcr_index_build / pcr_index_free / pcr_index_len
 *       pointclouds_spatial::KdTree::{build,len,is_empty}      crates/spatial/src/kdtree.rs:25-54
 *   pcr_knn                     KdTree::knn / knn_indices       crates/spatial/src/kdtree.rs:64-96
 *   pcr_radius_count / pcr_radius_search
 *       KdTree::radius_search[_unsorted]                        crates/spatial/src/kdtree.rs:105-163
 *   pcr_sor                     statistical_outlier_removal     crates/filters/src/statistical_outlier.rs:4-69
 *   pcr_radius_outlier          radius_outlier_removal          crates/filters/src/radius_outlier.rs:4-18
 *   pcr_estimate_normals        estimate_normals_with_viewpoint crates/normals/src/estimate.rs:19-124,139-238
 *   pcr_find_correspondences    find_correspondences            crates/registration/src/correspondence.rs:16-39
 *   pcr_apply_transform         apply_transform                 crates/registration/src/icp.rs:39-47,77-92
 *   pcr_icp_point_to_point      icp_point_to_point              crates/registration/src/icp.rs:125-282
 *   pcr_icp_point_to_plane      icp_point_to_plane              crates/registration/src/icp_plane.rs:20-97,131-236
 *   pcr_sor_normals_batch       the SOR -> normals chain of the demo pipelines, per frame
 *                               (examples/python/kitti_obstacle_detection.py:99-101)
 *   pcr_voxel_downsample_batch / pcr_estimate_normals_batch / pcr_icp_point_to_*_batch
 *                               voxel_downsample, estimate_normals and ICP of many frames per call
 *   pcr_ransac_plane_samples_batch / pcr_euclidean_cluster_batch
 *                               the plane fit and clustering of the obstacle pipeline, many frames per call
 *                               (examples/python/kitti_obstacle_detection.py:87-122)
 *   pcr_radius_outlier_batch    radius_outlier_removal of many frames per call
 *   pcr_frames_*                a batch of frames kept in HBM between those calls (the batch form of pcr_cloud_*)
 *   pcr_index_build_batch / pcr_knn_batch / pcr_radius_*_batch / pcr_find_correspondences_batch
 *                               the KdTree queries of many frames per call, each frame searched alone
 *   pcr_apply_transform_batch / pcr_frames_apply_transform / pcr_transform_compose / pcr_frames_merge
 *                               apply_transform of many frames per call, RigidTransform::compose
 *                               (crates/registration/src/icp.rs:39-92), and the frames joined into one cloud: the
 *                               map of an odometry chain assembled on the device
 *
 * The reference calls its kd-tree once per point inside serial loops; a per-query C call would be
 * useless on a GPU, so the boundary is BATCHED and sits one level up: it replaces the bodies of the
 * consumer functions and offers a batched form of the KdTree queries.  Results follow the
 * reference on the same inputs: KNN index lists are exact under an ascending (d^2, index) order
 * (kiddo leaves ties unspecified), d^2 = ((dx*dx)+(dy*dy))+(dz*dz) in f32 without FMA.
 *
 * Conventions
 *   - Clouds are SoA: three f32 arrays x/y/z of n elements (PointCloud, crates/core/src/cloud.rs:4-11).
 *   - The caller owns every buffer; pointers need to stay valid only for the duration of the call.
 *     Outputs go to caller-allocated buffers.  The library only allocates the opaque handles.
 *   - Every function returns a pcr_status (0 = ok).  pcr_last_error() gives the message.  No C++
 *     exception and no sticky CUDA error crosses this boundary.  There is NO CPU fallback: without
 *     a usable CUDA device the calls fail with PCR_ERR_NO_DEVICE / PCR_ERR_CUDA.
 *   - Calls are synchronous (they return after the context's stream has drained) unless the name
 *     ends in _async.  A pcr_ctx is single-caller: use one context per host thread.
 *   - *_dev variants take DEVICE pointers (same layouts) and are enqueued on the context's stream
 *     without host<->device copies; pcr_ctx_synchronize() waits for them.
 *   - Non-finite points are left out of the index and are never returned as neighbours; as queries
 *     they give empty results exactly like kdtree.rs:65 / statistical_outlier.rs:22-24.
 */
#ifndef PCR_B200_H
#define PCR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCR_B200_VERSION 122 /* 0.1.1: + voxel, cluster, RANSAC, device-resident clouds; 111/112: + block upload / download, nowait;
                                0.2.0 (120): + query sharding over a communicator, frame-stream hint statistics; 121: + pcr_ctx_comm_kind;
                                122: + pcr_cloud_upload_rows / _download_rows, pcr_sor_normals_batch_rows */

typedef enum pcr_status {
    PCR_OK = 0,
    PCR_ERR_INVALID_ARG = 1,      /* null pointer, bad size, non-finite parameter */
    PCR_ERR_NORMALS_MISMATCH = 2, /* IcpPlaneError::NormalsMismatch, icp_plane.rs:100-107 */
    PCR_ERR_CUDA = 3,
    PCR_ERR_NCCL = 4,
    PCR_ERR_OOM = 5,
    PCR_ERR_NO_DEVICE = 6,
    PCR_ERR_UNSUPPORTED = 7,      /* e.g. k above PCR_MAX_K */
    PCR_ERR_CAPACITY = 8          /* caller buffer too small (radius_search) */
} pcr_status;

#define PCR_MAX_K 1024 /* largest k accepted by the KNN kernels */

typedef struct pcr_ctx pcr_ctx;     /* device, stream, scratch memory, optional NCCL communicator */
typedef struct pcr_index pcr_index; /* uniform-grid index over one cloud, resident in HBM */

/* ---- context ------------------------------------------------------------------------------- */
int pcr_version(void);
/* Number of visible CUDA devices (0 when there is none or the driver is missing). */
int pcr_device_count(void);
int pcr_ctx_create(int device, pcr_ctx **out);
/* Same, but enqueue everything on an existing cudaStream_t (passed as void*), e.g. the current
 * stream of the embedding framework.  The stream must outlive the context. */
int pcr_ctx_create_on_stream(int device, void *cuda_stream, pcr_ctx **out);
void pcr_ctx_destroy(pcr_ctx *ctx);
int pcr_ctx_synchronize(pcr_ctx *ctx);
/* Message of the last failure on this context (ctx == NULL: last failure of a create call on the
 * calling thread).  Never NULL. */
const char *pcr_last_error(const pcr_ctx *ctx);
/* Kernel launches issued by this context since creation (bench.py's gpu_launches). */
uint64_t pcr_ctx_launch_count(const pcr_ctx *ctx);
/* Per-stage device timing for benchmarks: when enabled, every stage is bracketed by a cudaEvent
 * pair on the context's stream.  pcr_ctx_get_timing synchronises, adds the elapsed milliseconds of
 * all spans since the previous call per tag, and resets.  Tags: 0 index build, 1 KNN kernel on grid
 * level 0 (with its fused consumer), 2 deferred queries on coarser levels (their builds included),
 * 3 SOR statistics + mask, 4 ICP step kernel, 5 ICP reduce/solve, 6 KNN + normals kernel on grid
 * level 0, 7 other.  (Tag 1 is the KNN kernel of pcr_knn and of SOR.) */
#define PCR_NUM_TIMING_TAGS 8
int pcr_ctx_set_timing(pcr_ctx *ctx, int enable);
int pcr_ctx_get_timing(pcr_ctx *ctx, double *ms_per_tag /* [PCR_NUM_TIMING_TAGS] */,
                       uint64_t *spans_per_tag /* [PCR_NUM_TIMING_TAGS] or NULL */);
/* While timing is enabled the level-0 KNN kernel counts its work: out = {queries searched, candidate distance evaluations}
 * since the previous call (SURVEY.md 8d: "report candidates/query so the judge can recompute" the FP32 roofline). */
int pcr_ctx_get_knn_counters(pcr_ctx *ctx, uint64_t out[2]);
/* Tuning: force the grid cell size (metres) for subsequent index builds; 0 = automatic. */
int pcr_ctx_set_cell_size(pcr_ctx *ctx, float cell_size);
/* Hint: the clouds this context sees come from one sensor stream (consecutive frames of similar size, extent and
 * density).  The cell size found by one call's occupancy probe is then reused by the next call whose point count
 * and bounding box are within 12.5 % of it, which skips the probe grid and its host round trip.  Results never
 * depend on the cell size; an unrepresentative reuse only costs speed.  The same hint lets voxel_downsample size
 * its table from the previous frame's key box (padded) without measuring the new frame first -- a point outside the
 * box is detected and the frame redone the exact way -- lets the KNN levels queue the next-coarser grid before
 * the count that decides whether it is needed has come back, and lets the fused SOR -> normals call skip the round trip
 * for the number of queries its first grid level left over when that number was zero on the previous frame (it is then
 * read with the call's last round trip; non-zero: the call is redone with the wait).  Off by default. */
int pcr_ctx_set_frame_stream(pcr_ctx *ctx, int enable);
/* How often the frame-stream hints held since the context was created: {cell size reused, cell size probed again,
 * voxel key box guess held, guess missed (frame redone the exact way), coarser KNN level built ahead and needed,
 * built ahead and not needed, deferred counts of the fused SOR pass not awaited and zero, not awaited and non-zero (call
 * redone)}.  bench.py reports them so that the timed steps cannot be a best case by construction. */
#define PCR_NUM_HINT_STATS 8
int pcr_ctx_get_hint_stats(pcr_ctx *ctx, uint64_t out[PCR_NUM_HINT_STATS]);

/* ---- multi-GPU (one process per GPU; the host exchanges the id, e.g. torch.distributed) ------ */
#define PCR_UNIQUE_ID_BYTES 128
int pcr_comm_unique_id(void *out_id /* PCR_UNIQUE_ID_BYTES */);
int pcr_ctx_comm_init(pcr_ctx *ctx, const void *id, int rank, int world_size);
int pcr_ctx_comm_rank(const pcr_ctx *ctx);
int pcr_ctx_comm_size(const pcr_ctx *ctx);
/* How the ICP normal equations (icp_plane.rs:55-79, icp.rs:221-244 summed over a sharded source) are all-reduced on this
 * context: 0 = no exchange (one rank), 1 = ncclAllReduce, 2 = a one-shot all-reduce over NVLink peer memory fused into the
 * reduction kernel (one process per GPU on one node, blocks shared through CUDA IPC; chosen by pcr_ctx_comm_init when
 * every rank could map every peer, PCR_ICP_NCCL=1 forces 1). */
#define PCR_COMM_NONE 0
#define PCR_COMM_NCCL 1
#define PCR_COMM_PEER 2
int pcr_ctx_comm_kind(const pcr_ctx *ctx);
/* Query sharding of ONE cloud over the ranks of the context's communicator (SURVEY.md 8e rows 1-2; the reference's
 * loops this parallelises: crates/normals/src/estimate.rs:42-45, crates/filters/src/statistical_outlier.rs:19-39,
 * crates/filters/src/radius_outlier.rs:8-16).  When enabled (and pcr_ctx_comm_init gave the context more than one
 * rank), pcr_sor[_dev], pcr_estimate_normals[_dev] and pcr_radius_outlier[_dev] must be called by EVERY rank with the
 * SAME full cloud: each rank builds the (replicated) index, searches only its share of the queries -- a contiguous
 * range of the cell-sorted order cut at cell boundaries -- and the per-point results (SOR mean distances, normals,
 * neighbour counts) are merged over NCCL so that every rank returns the complete result.  The SOR statistics are then
 * folded by every rank over all N mean distances in the reference's order: the result is bit-identical to the
 * single-GPU call for any number of ranks.  Off by default; ICP shards its SOURCE cloud instead (see the ICP calls). */
int pcr_ctx_set_query_sharding(pcr_ctx *ctx, int enable);
/* Test hook: give the context a rank and a world size WITHOUT a communicator; the merging collectives become no-ops, so
 * a query-sharded call returns this rank's PARTIAL result (zero / 0-bytes where another rank would have written).  One
 * GPU can then play every rank in turn and the test checks that the parts are disjoint and add up to the unsharded
 * result (tests/test_gpu_parity.py).  Not for production use. */
int pcr_ctx_debug_set_shard(pcr_ctx *ctx, int rank, int world_size);

/* ---- spatial index (KdTree) ------------------------------------------------------------------ */
/* k_hint: the k the index will mostly be queried with (0 = unknown); only steers the cell size. */
int pcr_index_build(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                    size_t k_hint, pcr_index **out);
int pcr_index_build_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n,
                        size_t k_hint, pcr_index **out);
void pcr_index_free(pcr_index *index);
size_t pcr_index_len(const pcr_index *index); /* points of the cloud, kdtree.rs:47-49 */
/* Grid description for diagnostics: cell size, dims[3], indexed (finite) point count. */
int pcr_index_info(const pcr_index *index, float *cell_size, int32_t dims[3], size_t *n_indexed);

/* KdTree::knn for nq queries at once.  idx, dist: row-major nq x k; row q holds counts[q] =
 * min(k, indexed points) valid entries in ascending (distance, index) order (0 for a non-finite
 * query or k == 0 or an empty cloud), the rest is padded with UINT32_MAX / +INF.  dist is the
 * Euclidean distance sqrt(d^2) (kdtree.rs:76).  dist and counts may be NULL (knn_indices). */
int pcr_knn(pcr_index *index, const float *qx, const float *qy, const float *qz, size_t nq,
            size_t k, uint32_t *idx, float *dist, uint32_t *counts);
int pcr_knn_dev(pcr_index *index, const float *d_qx, const float *d_qy, const float *d_qz, size_t nq,
                size_t k, uint32_t *d_idx, float *d_dist, uint32_t *d_counts);

/* radius_search_unsorted(q, r).len() per query (d^2 <= r*r, r*r rounded in f32; 0 if r <= 0,
 * r non-finite or q non-finite, kdtree.rs:106-112). */
int pcr_radius_count(pcr_index *index, const float *qx, const float *qy, const float *qz, size_t nq,
                     float radius, uint32_t *counts);
/* radius_search in CSR form: offsets[nq+1], idx[offsets[q]..offsets[q+1]) ascending by index
 * (kdtree.rs:132).  *total receives offsets[nq]; if it exceeds cap nothing is written to idx and
 * PCR_ERR_CAPACITY is returned (call again with a larger buffer). */
int pcr_radius_search(pcr_index *index, const float *qx, const float *qy, const float *qz, size_t nq,
                      float radius, uint64_t *offsets, uint32_t *idx, size_t cap, size_t *total);

/* Batch index: the KdTree queries of many frames per call.  The index is built over F frames back to back, frame f =
 * points [frame_offsets[f], frame_offsets[f+1]) (HOST, n_frames + 1 entries, as in the other batch calls), and queried
 * with frames of queries back to back, query frame f = queries [query_offsets[f], query_offsets[f+1]) (HOST, the index's
 * n_frames + 1 entries).  Query frame f is searched in index frame f only, and its results are bit for bit what the
 * single call returns for index frame f alone (pcr_index_build on that frame) and the queries of frame f: KNN rows
 * (indices, distances, counts, padding), radius counts, ascending radius CSR rows, correspondences in source order.
 * Indices in and out are FRAME-LOCAL.  Edge cases follow the single calls (k == 0, non-finite queries, r <= 0 or
 * non-finite r, k above a frame's indexed count); an index frame that is empty or holds only non-finite points gives
 * every query of its frame count 0, and a query frame may be empty.
 * Unlike the transient indexes inside the batch consumers, a batch index is persistent: it owns its cell table and its
 * coarser and finer grid levels (a 100-frame table can take hundreds of MB), so other calls on the same context and
 * other batch indexes leave it unchanged.  pcr_index_len returns N; pcr_index_info describes frame 0's grid and the
 * indexed count of all frames.  The single-cloud queries (pcr_knn[_dev], pcr_radius_count, pcr_radius_search,
 * pcr_find_correspondences) on a batch index of more than one frame -> PCR_ERR_INVALID_ARG naming the _batch form; the
 * _batch queries on a single-cloud index are a batch of one.
 * Errors: frame or query offsets not starting at 0 or decreasing, n_frames == 0 at build, a query frame count other
 * than the index's, or a null pointer -> PCR_ERR_INVALID_ARG; N >= 2^31, more than 65535 frames, more than 0xfffffff0
 * queries or k > PCR_MAX_K -> PCR_ERR_UNSUPPORTED.  The batch never shards its queries: on a context with a communicator
 * every rank queries the frames it was given. */
int pcr_index_build_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                          const uint64_t *frame_offsets, size_t n_frames, size_t k_hint, pcr_index **out);
/* _dev: x, y, z are device pointers (e.g. pcr_frames_device_pointers); frame_offsets stays on the host. */
int pcr_index_build_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                              const uint64_t *frame_offsets /* HOST */, size_t n_frames, size_t k_hint, pcr_index **out);
/* pcr_knn per query frame: idx, dist row-major nq x k (nq = query_offsets[n_frames], nq * k in 64 bits), counts nq;
 * dist and counts may be NULL. */
int pcr_knn_batch(pcr_index *index, const float *qx, const float *qy, const float *qz,
                  const uint64_t *query_offsets, size_t n_frames, size_t k, uint32_t *idx, float *dist, uint32_t *counts);
/* _dev: queries and outputs are device pointers, query_offsets stays on the host; enqueued like pcr_knn_dev. */
int pcr_knn_batch_dev(pcr_index *index, const float *d_qx, const float *d_qy, const float *d_qz,
                      const uint64_t *query_offsets /* HOST */, size_t n_frames, size_t k, uint32_t *d_idx,
                      float *d_dist, uint32_t *d_counts);
/* pcr_radius_count per query frame (counts: nq entries). */
int pcr_radius_count_batch(pcr_index *index, const float *qx, const float *qy, const float *qz,
                           const uint64_t *query_offsets, size_t n_frames, float radius, uint32_t *counts);
int pcr_radius_count_batch_dev(pcr_index *index, const float *d_qx, const float *d_qy, const float *d_qz,
                               const uint64_t *query_offsets /* HOST */, size_t n_frames, float radius,
                               uint32_t *d_counts);
/* pcr_radius_search per query frame: offsets[nq + 1] over all queries, row q frame-local and ascending; the
 * PCR_ERR_CAPACITY protocol of pcr_radius_search. */
int pcr_radius_search_batch(pcr_index *index, const float *qx, const float *qy, const float *qz,
                            const uint64_t *query_offsets, size_t n_frames, float radius, uint64_t *offsets,
                            uint32_t *idx, size_t cap, size_t *total);
/* pcr_find_correspondences per query frame: frame f's pairs are [corr_offsets[f], corr_offsets[f+1]) of src_idx,
 * tgt_idx and dist (each sized nq; corr_offsets HOST, n_frames + 1), in source order, both indices frame-local. */
int pcr_find_correspondences_batch(pcr_index *target, const float *sx, const float *sy, const float *sz,
                                   const uint64_t *query_offsets, size_t n_frames, float max_distance,
                                   uint32_t *src_idx, uint32_t *tgt_idx, float *dist, uint64_t *corr_offsets);

/* ---- filters ----------------------------------------------------------------------------------- */
/* statistical_outlier_removal up to (not including) cloud.select(): keep[i] = 1 iff point i
 * survives; *n_kept = number of ones.  mean_d (may be NULL) receives the per-point mean neighbour
 * distance (INF for non-finite points).  stats (may be NULL) receives {global_mean,
 * global_stddev, threshold}.  Empty cloud or k == 0: all zeros (the reference returns an empty
 * cloud); n == 1: keep[0] = 1. */
int pcr_sor(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, size_t k,
            float std_mul, uint8_t *keep, size_t *n_kept, float *mean_d, float *stats);
int pcr_sor_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n,
                size_t k, float std_mul, uint8_t *d_keep, float *d_mean_d /* may be NULL */);
/* radius_outlier_removal: keep[i] = 1 iff #{j : d^2(i,j) <= r^2} >= min_neighbors (self counts). */
int pcr_radius_outlier(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                       float radius, size_t min_neighbors, uint8_t *keep, size_t *n_kept);

int pcr_radius_outlier_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n,
                           float radius, size_t min_neighbors, uint8_t *d_keep);
/* The same for every frame of a batch (frame f = points [frame_offsets[f], frame_offsets[f+1]), HOST offsets): each point
 * counts the points of its own frame only, and frame f's keep bytes are bit for bit pcr_radius_outlier's for the frame
 * alone (radius <= 0 or not finite: every count is 0, a point is kept iff min_neighbors == 0).  n_kept_per_frame (may be
 * NULL): n_frames entries.  Offsets not starting at 0 or decreasing, or a null pointer -> PCR_ERR_INVALID_ARG; N >= 2^31
 * or more than 65535 frames -> PCR_ERR_UNSUPPORTED.  The batch never shards its queries over a communicator. */
int pcr_radius_outlier_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                             size_t n_frames, float radius, size_t min_neighbors, uint8_t *keep, uint64_t *n_kept_per_frame);
/* _dev: x, y, z and keep are device pointers, frame_offsets stays on the host; enqueued on the context's stream. */
int pcr_radius_outlier_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                 size_t n_frames, float radius, size_t min_neighbors, uint8_t *d_keep);

/* ---- normals ----------------------------------------------------------------------------------- */
int pcr_estimate_normals(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                         size_t k, const float viewpoint[3], float *nx, float *ny, float *nz);
int pcr_estimate_normals_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                             size_t n, size_t k, const float viewpoint[3], float *d_nx, float *d_ny,
                             float *d_nz);

/* ---- registration ------------------------------------------------------------------------------ */
typedef struct pcr_icp_params { /* IcpParams, icp.rs:95-109 (defaults 50, 1e-5, INF) */
    uint64_t max_iterations;
    float tolerance;
    float max_correspondence_distance;
} pcr_icp_params;

typedef struct pcr_icp_result { /* IcpResult + RigidTransform, icp.rs:8-11,112-118 */
    float rotation[9];          /* row-major 3x3 */
    float translation[3];
    float fitness;
    float rmse;
    int32_t converged;
    uint64_t num_iterations;
} pcr_icp_result;

/* Outputs sized ns; *count receives the number of correspondences (source order). */
int pcr_find_correspondences(pcr_index *target, const float *sx, const float *sy, const float *sz,
                             size_t ns, float max_distance, uint32_t *src_idx, uint32_t *tgt_idx,
                             float *dist, size_t *count);
int pcr_apply_transform(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                        const float rotation[9], const float translation[3], float *ox, float *oy,
                        float *oz);
/* apply_transform of every frame of a batch: frame f = points [frame_offsets[f], frame_offsets[f+1]) (HOST offsets) is
 * moved by transforms[12f .. 12f+12) (HOST: row-major rotation[9], then translation[3]); frame f's output is bit for bit
 * what pcr_apply_transform returns for frame f alone with that transform.  Offsets that do not start at 0 or decrease, or a
 * NULL pointer -> PCR_ERR_INVALID_ARG; N >= 2^31 or more than 65535 frames -> PCR_ERR_UNSUPPORTED; n_frames == 0 -> PCR_OK.
 * The transform values are not checked, as in pcr_apply_transform.  _dev: device points, host offsets and transforms
 * (free for reuse on return), enqueued on the context's stream. */
int pcr_apply_transform_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                              const uint64_t *frame_offsets, size_t n_frames, const float *transforms,
                              float *ox, float *oy, float *oz);
int pcr_apply_transform_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                  const uint64_t *frame_offsets, size_t n_frames, const float *transforms,
                                  float *d_ox, float *d_oy, float *d_oz);
/* RigidTransform::compose (icp.rs:52-73): apply `first`, then `then`.  R = then.R * first.R,
 * t = then.R * first.t + then.t, f32 in the reference's operation order, no FMA; 12-float layout as above.  Host only:
 * needs no context or device.  out may alias first or then. */
int pcr_transform_compose(const float first[12], const float then[12], float out[12]);
int pcr_icp_point_to_point(pcr_ctx *ctx, const float *sx, const float *sy, const float *sz, size_t ns,
                           const float *tx, const float *ty, const float *tz, size_t nt,
                           const pcr_icp_params *params, pcr_icp_result *result);
/* n_normals != nt -> PCR_ERR_NORMALS_MISMATCH (icp_plane.rs:27-32).  With a communicator
 * (pcr_ctx_comm_init) every rank passes ITS shard of the source and the full target; the 6x6
 * system is all-reduced each iteration and every rank returns the same result. */
int pcr_icp_point_to_plane(pcr_ctx *ctx, const float *sx, const float *sy, const float *sz, size_t ns,
                           const float *tx, const float *ty, const float *tz, size_t nt,
                           const float *nx, const float *ny, const float *nz, size_t n_normals,
                           const pcr_icp_params *params, pcr_icp_result *result);
int pcr_icp_point_to_point_dev(pcr_ctx *ctx, const float *d_sx, const float *d_sy, const float *d_sz,
                               size_t ns, const float *d_tx, const float *d_ty, const float *d_tz,
                               size_t nt, const pcr_icp_params *params, pcr_icp_result *result);
int pcr_icp_point_to_plane_dev(pcr_ctx *ctx, const float *d_sx, const float *d_sy, const float *d_sz,
                               size_t ns, const float *d_tx, const float *d_ty, const float *d_tz,
                               size_t nt, const float *d_nx, const float *d_ny, const float *d_nz,
                               size_t n_normals, const pcr_icp_params *params, pcr_icp_result *result);

/* Batched ICP: many (source, target) pairs of frames in one call.  The frames sit back to back in one buffer, frame f =
 * points [frame_offsets[f], frame_offsets[f+1]) (as in pcr_sor_normals_batch), N = frame_offsets[n_frames].  Pair p
 * registers frame pairs[2p] (the source) onto frame pairs[2p+1] (the target); results[p] is its result.  Independent
 * pairs and a sequence (pairs (i+1, i): frame-to-frame odometry, every frame uploaded and indexed once) are both
 * this form, and a frame may appear in any number of pairs, on either side.
 * Every pair is what the single-pair call on the same two clouds returns: the same parameter checks, the same empty-cloud
 * rules (icp.rs:131-139), max_iterations == 0 computes the metrics only.  A pair's result does not depend on the other
 * pairs of the call, and repeated calls return the same bits; against the single-pair call it agrees within f64
 * rounding of the sums (the single-pair call orders the points inside a grid cell by atomics, the batch by index).
 * Point-to-plane: one normal per point of the buffer (only target frames' entries are read); n_normals != N ->
 * PCR_ERR_NORMALS_MISMATCH.  frame_offsets not starting at 0 or decreasing, a frame id >= n_frames, or a null pointer
 * -> PCR_ERR_INVALID_ARG.  Source frames summed over the pairs reaching 2^31 points, or more than 65535 frames ->
 * PCR_ERR_UNSUPPORTED.
 * The batch never communicates: on a context with a communicator every rank registers the pairs it was given (frames
 * dealt to ranks), with its whole source frames. */
int pcr_icp_point_to_point_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                                 const uint64_t *frame_offsets, size_t n_frames,
                                 const uint32_t *pairs, size_t n_pairs,
                                 const pcr_icp_params *params, pcr_icp_result *results /* n_pairs */);
int pcr_icp_point_to_plane_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                                 const uint64_t *frame_offsets, size_t n_frames,
                                 const float *nx, const float *ny, const float *nz, size_t n_normals,
                                 const uint32_t *pairs, size_t n_pairs,
                                 const pcr_icp_params *params, pcr_icp_result *results);
/* _dev: x .. nz are device pointers; frame_offsets, pairs, params and results stay on the host.  Synchronous. */
int pcr_icp_point_to_point_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                     const uint64_t *frame_offsets, size_t n_frames,
                                     const uint32_t *pairs, size_t n_pairs,
                                     const pcr_icp_params *params, pcr_icp_result *results);
int pcr_icp_point_to_plane_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                     const uint64_t *frame_offsets, size_t n_frames,
                                     const float *d_nx, const float *d_ny, const float *d_nz, size_t n_normals,
                                     const uint32_t *pairs, size_t n_pairs,
                                     const pcr_icp_params *params, pcr_icp_result *results);

/* ---- voxel grid filter (SURVEY 8f-2) ---------------------------------------------------------------
 * voxel_downsample (crates/filters/src/voxel_downsample.rs:12-65): one point per occupied voxel
 * (key = floor(p / voxel_size) as i32), the mean of the voxel's points summed in input order, voxels
 * in ascending key order.  Outputs sized n; *n_out = number of voxels.  voxel_size not finite or <= 0
 * -> PCR_ERR_INVALID_ARG (the reference panics, :13-16; its Python layer raises ValueError). */
int pcr_voxel_downsample(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                         float voxel_size, float *ox, float *oy, float *oz, size_t *n_out);
int pcr_voxel_downsample_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                             size_t n, float voxel_size, float *d_ox, float *d_oy, float *d_oz,
                             size_t *n_out);

/* ---- segmentation (SURVEY 8f-1) ------------------------------------------------------------------
 * euclidean_cluster (crates/segmentation/src/euclidean_cluster.rs:96-101): connected components of
 * "d^2 <= r^2 between points of key-adjacent cells", clusters with min_size <= size <= max_size,
 * size descending then first index ascending, indices ascending inside a cluster.  CSR output:
 * cluster c = indices[offsets[c] .. offsets[c+1]); the caller sizes offsets n + 1 and indices n.
 * Empty cloud, threshold <= 0 or min_size == 0 -> 0 clusters (:102-104).  Non-finite points are
 * singleton components. */
int pcr_euclidean_cluster(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                          float distance_threshold, size_t min_size, size_t max_size,
                          uint32_t *offsets, uint32_t *indices, size_t *n_clusters);
/* Device form: d_labels[i] = smallest index of the component of point i (before the size filter). */
int pcr_cluster_labels_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                           size_t n, float distance_threshold, uint32_t *d_labels);

typedef struct pcr_cloud pcr_cloud; /* device-resident cloud, see the end of this header */

/* ---- plane segmentation (SURVEY 8f-4) -------------------------------------------------------------
 * ransac_plane_seeded (crates/segmentation/src/ransac_plane.rs:56-129) AFTER its sampling step: `samples`
 * holds the m index triples exactly as the reference's sample_three_distinct produced them (StdRng stays on
 * the Rust side).  Fits, inlier counts (m x n distances), the reference's choice rule (sequential with the
 * adaptive early exit, or first-maximum when n >= 10000 and m >= 16) and the inlier list run here.
 * model = {nx, ny, nz, d} (default (0,0,1,0) if n < 3 or no sample is valid); inliers sized n, ascending. */
int pcr_ransac_plane_samples(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n,
                             float distance_threshold, const uint32_t *samples, size_t m, float model[4],
                             uint32_t *inliers, size_t *n_inliers);
int pcr_cloud_ransac_plane_samples(const pcr_cloud *cloud, float distance_threshold, const uint32_t *samples,
                                   size_t m, float model[4], uint32_t *inliers, size_t *n_inliers);

/* Batched plane fit and clustering: the back end of the obstacle pipeline (voxel -> SOR -> ransac_plane -> select_inverse
 * -> euclidean_cluster) for many frames per call.  The frames sit back to back, frame f = points
 * [frame_offsets[f], frame_offsets[f+1]), N = frame_offsets[n_frames]; every frame gets bit for bit what the single call
 * returns for that frame alone.  Indices in and out are FRAME-LOCAL.
 * RANSAC: frame f's triples are samples[3 * sample_offsets[f] .. 3 * sample_offsets[f+1]) (HOST, sample_offsets
 * n_frames + 1 entries; both may be NULL when no frame has triples).  models[4f .. 4f+4) (HOST) and the ascending inlier
 * list inliers[inlier_offsets[f] .. inlier_offsets[f+1]) (inlier_offsets HOST, n_frames + 1; inliers sized N) are what
 * pcr_ransac_plane_samples returns for frame f and its triples: the default model and no inliers below 3 points, the
 * default model when no triple is valid (its inliers are still those of the plane z = 0), and the choice rule applied
 * with the frame's own point and triple counts.  A triple index >= the frame's point count (in a frame of 3 points or
 * more), or sample_offsets not starting at 0 or decreasing -> PCR_ERR_INVALID_ARG.
 * Clustering: frame f's clusters are c in [cluster_offsets[f], cluster_offsets[f+1]) (HOST, n_frames + 1), cluster c is
 * indices[offsets[c] .. offsets[c+1]) (offsets sized N + 1, indices N).  Minus offsets[cluster_offsets[f]], frame f's
 * CSR is pcr_euclidean_cluster's for the frame alone (size descending, then first index ascending, indices ascending).
 * threshold <= 0 or min_size == 0 -> no cluster in any frame and offsets[0] = 0; N >= 2^30 -> PCR_ERR_UNSUPPORTED.
 * Both: frame_offsets not starting at 0 or decreasing, or a null pointer -> PCR_ERR_INVALID_ARG; more than 65535 frames
 * -> PCR_ERR_UNSUPPORTED.  Neither batch communicates: on a context with a communicator every rank processes the frames
 * it was given.  Synchronous, two host round trips each whatever the number of frames.  Measured on an NVIDIA B200 at a
 * 1000 W power limit, 100 frames of 65 K points after voxel 0.15 and SOR: RANSAC with 500 triples per frame 1.88 ms
 * against 23.9 ms for 100 single calls on resident clouds, clustering of their 487 K non-ground points 0.99 ms against
 * 36.4 ms (DESIGN section 6). */
int pcr_ransac_plane_samples_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                                   const uint64_t *frame_offsets, size_t n_frames, float distance_threshold,
                                   const uint32_t *samples, const uint64_t *sample_offsets, float *models,
                                   uint32_t *inliers, uint64_t *inlier_offsets);
/* _dev: x, y, z and inliers are device pointers; everything else stays on the host. */
int pcr_ransac_plane_samples_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                       const uint64_t *frame_offsets /* HOST */, size_t n_frames, float distance_threshold,
                                       const uint32_t *samples /* HOST */, const uint64_t *sample_offsets /* HOST */,
                                       float *models /* HOST */, uint32_t *d_inliers, uint64_t *inlier_offsets /* HOST */);
int pcr_euclidean_cluster_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                                const uint64_t *frame_offsets, size_t n_frames, float distance_threshold,
                                size_t min_size, size_t max_size, uint32_t *offsets, uint32_t *indices,
                                uint64_t *cluster_offsets);
/* _dev: x, y, z, offsets and indices are device pointers; frame_offsets and cluster_offsets stay on the host. */
int pcr_euclidean_cluster_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                    const uint64_t *frame_offsets /* HOST */, size_t n_frames, float distance_threshold,
                                    size_t min_size, size_t max_size, uint32_t *d_offsets, uint32_t *d_indices,
                                    uint64_t *cluster_offsets /* HOST */);
/* d_labels[i] = smallest FRAME-LOCAL index of the component of point i inside its frame (pcr_cluster_labels_dev of each
 * frame alone).  threshold <= 0 -> PCR_ERR_INVALID_ARG.  Enqueued on the context's stream like pcr_cluster_labels_dev. */
int pcr_cluster_labels_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                 const uint64_t *frame_offsets /* HOST */, size_t n_frames, float distance_threshold,
                                 uint32_t *d_labels);

/* ---- multi-frame batch (BASELINE config 5) ------------------------------------------------------
 * Frames are independent clouds stored back to back: frame f = points [frame_offsets[f],
 * frame_offsets[f+1]).  Per frame: SOR(k_sor, std_mul) then normals(k_normals, viewpoint) on the
 * KEPT points (the reference rebuilds its tree on the filtered cloud).  keep: one byte per input
 * point.  nx/ny/nz: one entry per input point; entries of removed points are set to 0. */
int pcr_sor_normals_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                          const uint64_t *frame_offsets, size_t n_frames, size_t k_sor,
                          float std_mul, size_t k_normals, const float viewpoint[3], uint8_t *keep,
                          float *nx, float *ny, float *nz, uint64_t *n_kept_per_frame);
/* The same for the PyO3 surface's layout: `xyz` and `normals` are row-major (N, 3) blocks (see pcr_cloud_upload_rows);
 * one contiguous transfer each way, split / interleaved on the device. */
int pcr_sor_normals_batch_rows(pcr_ctx *ctx, const float *xyz, const uint64_t *frame_offsets, size_t n_frames,
                               size_t k_sor, float std_mul, size_t k_normals, const float viewpoint[3],
                               uint8_t *keep, float *normals, uint64_t *n_kept_per_frame);
int pcr_sor_normals_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                              const uint64_t *frame_offsets /* HOST */, size_t n_frames,
                              size_t k_sor, float std_mul, size_t k_normals,
                              const float viewpoint[3], uint8_t *d_keep, float *d_nx, float *d_ny,
                              float *d_nz);

/* Batched voxel_downsample and estimate_normals: the steps in front of pcr_sor_normals_batch and of the ICP batch, for
 * many frames in one call.  The frames sit back to back as above, N = frame_offsets[n_frames]; every frame is processed
 * as if it were alone.
 * Voxel: frame f's voxels are written to [out_offsets[f], out_offsets[f+1]) of ox/oy/oz (sized N); out_offsets is HOST
 * memory of n_frames + 1 entries, out_offsets[0] = 0, so it can be passed as the frame_offsets of the other batch calls.
 * Those entries are bit for bit what pcr_voxel_downsample returns for frame f alone: the same key order and input-order
 * f32 sums, non-finite points skipped, a frame that is empty or holds no finite point gives 0 voxels, saturated i32 keys
 * merge.  voxel_size not finite or <= 0 -> PCR_ERR_INVALID_ARG.  The batch neither reads nor updates the frame-stream
 * voxel key box of the context (pcr_ctx_set_frame_stream), and leaves pcr_ctx_get_hint_stats unchanged.
 * Normals: one normal per input point, each frame searched only within itself; frame f's entries are bit for bit what
 * pcr_estimate_normals returns for frame f alone.  k == 0 or N == 0 -> PCR_OK and nothing is written; k > PCR_MAX_K ->
 * PCR_ERR_UNSUPPORTED; a null viewpoint -> PCR_ERR_INVALID_ARG.
 * Both: frame_offsets not starting at 0 or decreasing, or a null pointer -> PCR_ERR_INVALID_ARG; N >= 2^31 or more than
 * 65535 frames -> PCR_ERR_UNSUPPORTED.  Neither batch communicates or shards its queries: on a context with a communicator
 * every rank processes the frames it was given. */
int pcr_voxel_downsample_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                               const uint64_t *frame_offsets, size_t n_frames, float voxel_size,
                               float *ox, float *oy, float *oz, uint64_t *out_offsets);
/* _dev: x .. oz are device pointers; frame_offsets and out_offsets stay on the host.  Synchronous. */
int pcr_voxel_downsample_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                   const uint64_t *frame_offsets /* HOST */, size_t n_frames, float voxel_size,
                                   float *d_ox, float *d_oy, float *d_oz, uint64_t *out_offsets /* HOST */);
int pcr_estimate_normals_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z,
                               const uint64_t *frame_offsets, size_t n_frames, size_t k,
                               const float viewpoint[3], float *nx, float *ny, float *nz);
/* _dev: device pointers, frame_offsets on the host; enqueued on the context's stream like pcr_sor_normals_batch_dev. */
int pcr_estimate_normals_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z,
                                   const uint64_t *frame_offsets /* HOST */, size_t n_frames, size_t k,
                                   const float viewpoint[3], float *d_nx, float *d_ny, float *d_nz);

/* ---- device-resident clouds (SURVEY 8f-3) ---------------------------------------------------------
 * PointCloud (crates/core/src/cloud.rs:4-18) kept in HBM between the steps of a pipeline: one upload,
 * one download, `select` (cloud.rs:103-140) as a device compaction that carries the normals along.
 * Every function that returns a cloud allocates a new handle (free it with pcr_cloud_free); inputs
 * are never modified.  Edge cases follow the reference functions named on each line.
 * A cloud belongs to the context that made it: free it before pcr_ctx_destroy, and use it only from
 * the thread that drives that context.  Contexts are independent of one another, so several host
 * threads, each with its own context, can keep several frames in flight on one GPU. */
int pcr_cloud_upload(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, pcr_cloud **out);
void pcr_cloud_free(pcr_cloud *cloud);
size_t pcr_cloud_len(const pcr_cloud *cloud);
int pcr_cloud_has_normals(const pcr_cloud *cloud);
int pcr_cloud_download(const pcr_cloud *cloud, float *x, float *y, float *z);            /* arrays of pcr_cloud_len */
int pcr_cloud_download_normals(const pcr_cloud *cloud, float *nx, float *ny, float *nz);
/* The same for callers that keep their SoA arrays in ONE block, `stride` floats apart (x | y | z [| nx | ny | nz]):
 * a single strided transfer each way instead of three or six. */
int pcr_cloud_upload_block(pcr_ctx *ctx, const float *xyz, size_t stride, size_t n, pcr_cloud **out);
/* The same without waiting for the copy: the steps queued next run right behind it.  `xyz` (pinned memory, or the
 * copy is staged and waits anyway) must stay unchanged until a later call on this context has returned data that
 * depends on the cloud (any filter's result, a download) or pcr_ctx_synchronize has returned. */
int pcr_cloud_upload_block_nowait(pcr_ctx *ctx, const float *xyz, size_t stride, size_t n, pcr_cloud **out);
int pcr_cloud_download_block(const pcr_cloud *cloud, float *dst, size_t stride, int with_normals);
/* The PyO3 surface takes and returns row-major (N, 3) arrays (crates/python/src/cloud.rs:25-53, from_numpy / to_numpy,
 * which copy between that layout and the SoA vectors on the host).  Here the copy crosses PCIe as it is -- one contiguous
 * transfer -- and the (de)interleaving runs on the device: `xyz` is n rows of x, y, z; `normals` (NULL: not wanted) n rows
 * of nx, ny, nz, PCR_ERR_INVALID_ARG if wanted from a cloud without normals. */
int pcr_cloud_upload_rows(pcr_ctx *ctx, const float *xyz, size_t n, pcr_cloud **out);
int pcr_cloud_download_rows(const pcr_cloud *cloud, float *xyz, float *normals);
/* device pointers of the SoA arrays (valid until the cloud is freed; normals NULL if absent) */
int pcr_cloud_device_pointers(const pcr_cloud *cloud, const float **d_x, const float **d_y, const float **d_z,
                              const float **d_nx, const float **d_ny, const float **d_nz);
/* cloud.rs:103-140; an index >= len -> PCR_ERR_INVALID_ARG (the reference panics, :109) */
int pcr_cloud_select(const pcr_cloud *cloud, const uint32_t *indices, size_t m, pcr_cloud **out);
int pcr_cloud_voxel_downsample(const pcr_cloud *cloud, float voxel_size, pcr_cloud **out);           /* voxel_downsample.rs:12 */
int pcr_cloud_statistical_outlier_removal(const pcr_cloud *cloud, size_t k, float std_mul,
                                          pcr_cloud **out);                                           /* statistical_outlier.rs:4 */
int pcr_cloud_radius_outlier_removal(const pcr_cloud *cloud, float radius, size_t min_neighbors,
                                     pcr_cloud **out);                                                /* radius_outlier.rs:4 */
/* estimate.rs:19: a copy of the cloud with normals attached (viewpoint NULL = origin, :13-15) */
int pcr_cloud_estimate_normals(const pcr_cloud *cloud, size_t k, const float viewpoint[3], pcr_cloud **out);
/* statistical_outlier_removal then estimate_normals on the kept points, one index for both (the
 * single-frame form of pcr_sor_normals_batch): the kept points with their normals */
int pcr_cloud_sor_normals(const pcr_cloud *cloud, size_t k_sor, float std_mul, size_t k_normals,
                          const float viewpoint[3], pcr_cloud **out);
int pcr_cloud_euclidean_cluster(const pcr_cloud *cloud, float distance_threshold, size_t min_size,
                                size_t max_size, uint32_t *offsets, uint32_t *indices,
                                size_t *n_clusters);                                                  /* euclidean_cluster.rs:96 */
int pcr_cloud_apply_transform(const pcr_cloud *cloud, const float rotation[9], const float translation[3],
                              pcr_cloud **out);                                                       /* icp.rs:77-92 */
int pcr_cloud_icp_point_to_point(const pcr_cloud *source, const pcr_cloud *target,
                                 const pcr_icp_params *params, pcr_icp_result *result);              /* icp.rs:125 */
/* the target must carry normals (crates/python/src/registration.rs:80-86) */
int pcr_cloud_icp_point_to_plane(const pcr_cloud *source, const pcr_cloud *target,
                                 const pcr_icp_params *params, pcr_icp_result *result);              /* icp_plane.rs:20 */

/* ---- device-resident frame batches ------------------------------------------------------------------
 * F clouds back to back in one device allocation, frame f = points [offsets[f], offsets[f+1]): the batch counterpart of
 * pcr_cloud, so that a pipeline over many frames is one upload, a chain of batch calls and one download.  The rules of
 * pcr_cloud hold: a batch belongs to the context that made it and is freed before pcr_ctx_destroy; every function that
 * returns a batch allocates a new handle and leaves its input unchanged; *out is set on success only (a failed call
 * returns no handle).  Each method runs the core of the matching raw-pointer batch call, so frame f of a result is bit
 * for bit what the pcr_cloud method returns for frame f alone, edge cases included (empty, one-point and non-finite
 * frames).  Indices in and out are FRAME-LOCAL.  A filter ends in one compaction of all frames, which costs one host
 * round trip (all F + 1 new offsets in one copy) on top of the round trips of its batch core.
 * Uploads: n_frames >= 1, frame_offsets starting at 0 and never decreasing, else PCR_ERR_INVALID_ARG; N >= 2^31 or more
 * than 65535 frames -> PCR_ERR_UNSUPPORTED.  `xyz` of the _rows form is N rows of x, y, z (see pcr_cloud_upload_rows). */
typedef struct pcr_frames pcr_frames;
int pcr_frames_upload(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                      pcr_frames **out);
int pcr_frames_upload_rows(pcr_ctx *ctx, const float *xyz, const uint64_t *frame_offsets, size_t n_frames, pcr_frames **out);
void pcr_frames_free(pcr_frames *frames);
size_t pcr_frames_len(const pcr_frames *frames);    /* points of all frames */
size_t pcr_frames_count(const pcr_frames *frames);  /* frames */
int pcr_frames_offsets(const pcr_frames *frames, uint64_t *out /* pcr_frames_count + 1 */);
int pcr_frames_has_normals(const pcr_frames *frames);
int pcr_frames_device_pointers(const pcr_frames *frames, const float **d_x, const float **d_y, const float **d_z,
                               const float **d_nx, const float **d_ny, const float **d_nz);
/* arrays of pcr_frames_len; nx, ny, nz NULL: normals not wanted (PCR_ERR_INVALID_ARG if wanted from a batch without) */
int pcr_frames_download(const pcr_frames *frames, float *x, float *y, float *z, float *nx, float *ny, float *nz);
int pcr_frames_download_rows(const pcr_frames *frames, float *xyz, float *normals);
/* frame f as a new pcr_cloud (a device copy, normals carried), for the single-frame calls; f >= count -> INVALID_ARG */
int pcr_frames_frame(const pcr_frames *frames, size_t f, pcr_cloud **out);
/* all frames as one pcr_cloud, in frame order, normals carried (the map that pcr_cloud_voxel_downsample then thins) */
int pcr_frames_merge(const pcr_frames *frames, pcr_cloud **out);
/* pcr_apply_transform_batch on the batch: frame f moved by transforms[12f .. 12f+12) (HOST, count x 12 floats).  The
 * result holds xyz only (icp.rs:91, as pcr_cloud_apply_transform); the offsets are unchanged. */
int pcr_frames_apply_transform(const pcr_frames *frames, const float *transforms, pcr_frames **out);
/* Per frame, list f = indices[index_offsets[f] .. index_offsets[f+1]) (HOST, index_offsets count + 1 entries).
 * invert = 0: select (cloud.rs:103-140), the listed points in list order, duplicates kept; invert = 1: select_inverse,
 * the unlisted points in their order.  Normals are carried.  An index >= its frame's size -> PCR_ERR_INVALID_ARG naming the
 * frame and the index (the reference panics, cloud.rs:109), before any device work. */
int pcr_frames_select(const pcr_frames *frames, const uint32_t *indices, const uint64_t *index_offsets, int invert, pcr_frames **out);
/* pcr_voxel_downsample_batch: the result has no normals (voxel_downsample.rs:64) */
int pcr_frames_voxel_downsample(const pcr_frames *frames, float voxel_size, pcr_frames **out);
/* statistical_outlier_removal of every frame (the SOR of pcr_sor_normals_batch); k == 0 empties every frame and drops
 * the normals, as pcr_cloud_statistical_outlier_removal does; otherwise normals are carried */
int pcr_frames_statistical_outlier_removal(const pcr_frames *frames, size_t k, float std_mul, pcr_frames **out);
/* pcr_radius_outlier_batch, then the compaction; normals carried */
int pcr_frames_radius_outlier_removal(const pcr_frames *frames, float radius, size_t min_neighbors, pcr_frames **out);
/* pcr_estimate_normals_batch / pcr_sor_normals_batch: the result carries normals (viewpoint NULL = origin; k == 0 or
 * k_normals == 0 -> PCR_ERR_INVALID_ARG, as for pcr_cloud) */
int pcr_frames_estimate_normals(const pcr_frames *frames, size_t k, const float viewpoint[3], pcr_frames **out);
int pcr_frames_sor_normals(const pcr_frames *frames, size_t k_sor, float std_mul, size_t k_normals, const float viewpoint[3],
                           pcr_frames **out);
/* pcr_ransac_plane_samples_batch on the batch (models, inlier_offsets HOST as there; inliers HOST, may be NULL: the
 * lists are not downloaded).  outliers non-NULL: also every frame's select_inverse(inliers), built on the device from
 * the device inlier lists -- the ground removal of the obstacle pipeline. */
int pcr_frames_ransac_plane_samples(const pcr_frames *frames, float distance_threshold, const uint32_t *samples,
                                    const uint64_t *sample_offsets, float *models, uint32_t *inliers, uint64_t *inlier_offsets,
                                    pcr_frames **outliers);
/* pcr_euclidean_cluster_batch on the batch; host CSR as there (offsets sized len + 1, indices len) */
int pcr_frames_euclidean_cluster(const pcr_frames *frames, float distance_threshold, size_t min_size, size_t max_size,
                                 uint32_t *offsets, uint32_t *indices, uint64_t *cluster_offsets);
/* pcr_icp_point_to_*_batch on the batch's frames (pairs of frame ids, HOST).  Point-to-plane reads the batch's normals:
 * a batch without normals -> PCR_ERR_INVALID_ARG (crates/python/src/registration.rs:80-86). */
int pcr_frames_icp_point_to_point(const pcr_frames *frames, const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params,
                                  pcr_icp_result *results);
int pcr_frames_icp_point_to_plane(const pcr_frames *frames, const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params,
                                  pcr_icp_result *results);

#ifdef __cplusplus
}
#endif
#endif /* PCR_B200_H */
