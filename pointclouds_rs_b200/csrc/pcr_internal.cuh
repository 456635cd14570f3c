// pcr_internal.cuh -- shared declarations of the sm_100a KNN engine (not part of the C ABI).
#pragma once
#include <cstdlib>

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <memory>
#include <string>
#include <vector>

#include "../../include/pcr_b200.h"

namespace pcr {

// ------------------------------------------------------------------------------------------------
// Grid description.  One per frame (a plain cloud is one frame).  Axes are PERMUTED so that the
// axis with the most cells is the fastest-varying one: a row of cells along it is one contiguous
// run of points in the cell-sorted array, which is what the query kernels stream.
// ------------------------------------------------------------------------------------------------
struct GridDesc {
    double o[3];         // origin (bbox min) of permuted axis j
    double h, inv_h;     // cell size and its reciprocal (f64: cell coordinates are computed in f64)
    int32_t dims[3];     // cells along permuted axis j (j = 2 is the fastest)
    int32_t ax[3];       // ax[j] = original axis (0 = x, 1 = y, 2 = z) behind permuted axis j
    uint32_t cell_base;  // first entry of this frame in the cell table
    uint32_t n_cells;    // dims[0] * dims[1] * dims[2]
    uint32_t pt_begin;   // [pt_begin, pt_end): this frame's slice of the cell-sorted point array
    uint32_t pt_end;
    uint32_t in_begin;   // [in_begin, in_end): this frame's slice of the input (original order)
    uint32_t in_end;
};

constexpr int kLevelFactor = 6;  // cell-size ratio between consecutive grid levels (knn_search.cuh)

struct DevBuf {  // grow-only device scratch buffer
    void *p = nullptr;
    size_t cap = 0;
};

struct Ctx;

// Exchange block of one rank: data[2 slots][kPeerMaxWorld senders][kPeerWords] f64, then flag[2][kPeerMaxWorld] u64.
constexpr int kPeerMaxWorld = 8;
constexpr int kPeerWords = 32;
constexpr size_t kPeerDataBytes = 2 * kPeerMaxWorld * kPeerWords * sizeof(double);
constexpr size_t kPeerBlockBytes = kPeerDataBytes + 2 * kPeerMaxWorld * sizeof(unsigned long long);
struct PeerComm {
    double *data[kPeerMaxWorld];              // rank p's block as mapped on this device
    unsigned long long *flag[kPeerMaxWorld];
    int rank, world;                          // world == 0: no peer exchange (one rank, or NCCL is used)
};

// Device-resident index over one cloud or a batch of frames.
struct Index {
    Ctx *ctx = nullptr;
    size_t n = 0;          // points of the cloud(s) (incl. non-finite ones)
    size_t n_indexed = 0;  // finite points, i.e. entries of `sorted`
    int n_frames = 1;
    std::vector<GridDesc> grids_h;
    GridDesc *grids = nullptr;       // device copy [n_frames]
    uint32_t *frame_in_off = nullptr;  // device [n_frames + 1] input offsets (nullptr if n_frames == 1)
    float4 *sorted = nullptr;        // [n_indexed] (x, y, z, original index as bits), cell order
    float4 *orig4 = nullptr;         // [n] (x, y, z, -) in original order (gather target)
    uint32_t *cell_start = nullptr;  // [total_cells + 1] exclusive prefix of the per-cell counts
    uint32_t total_cells = 0;
    bool owns_memory = true;
    // bounding boxes (original axis order, 3 doubles per frame: min and extent) and finite counts
    std::vector<double> box_min, box_ext;
    std::vector<uint32_t> box_count;
    const uint8_t *d_mask = nullptr;  // keep-mask the index was built with (caller memory)
    Index *coarser = nullptr;         // next grid level (8x the cell size), built on demand
    Index *finer = nullptr;           // half the cell size: where the dense class of level 0 is searched (knn.cu), built on demand
    bool shares_orig4 = false;        // coarser levels borrow orig4 / grids layout from level 0
    int cell_slot = -1;               // >= 0: cell_start lives in ctx->b_cells[cell_slot] (transient index), not owned
    bool level_bufs_borrowed = false; // sorted and grids live in ctx->b_lsorted / b_lgrids[cell_slot], not owned
    // query shard of this rank (sorted positions; SURVEY 8e): set by index_shard_queries, default = every indexed point
    uint32_t q_begin = 0;
    uint32_t q_count = 0xffffffffu;
};

struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    int sm_count = 148;
    std::string err;
    uint64_t err_seq = 0;  // stamp of `err` (pcr_last_error reports the more recent of this and the calling thread's last failure)
    uint64_t launches = 0;
    float forced_cell = 0.f;
    // cell size chosen by the last single-frame probe, reused for the next cloud of the same shape (a stream of
    // LiDAR frames): skips the probe grid and its host round trip.  Only speed depends on the cell size.
    bool frame_stream = false;  // pcr_ctx_set_frame_stream: enables the reuse below
    struct {
        bool valid = false;
        size_t k_hint = 0;
        uint32_t count = 0;
        double ext[3] = {0, 0, 0};
        double h = 0;
    } cell_cache;
    // voxel key box of the last frame, padded: a frame stream sizes its column table from it without measuring the
    // new frame first (a point outside it raises a flag and the frame is redone the exact way).
    struct {
        bool valid = false;
        float voxel = 0.f;
        int mn[3] = {0, 0, 0}, mx[3] = {0, 0, 0};
        int uses = 0;       // frames since the box was last measured
        int pad_shift = 6;  // pad = extent >> pad_shift on each side; widened after a miss
    } vox_cache;
    // scratch
    DevBuf b_in;       // staged input x|y|z
    DevBuf b_in2;      // second cloud (ICP source)
    DevBuf b_out;      // staged outputs
    DevBuf b_misc;     // per-point scratch (cell ids, ranks, mean distances ...)
    // the finer level is built on a side stream while the coarser one is built on another: own per-point and scan scratch
    DevBuf b_fine_misc, b_fine_scan;
    uint32_t fine_scan_epoch = 0;
    DevBuf b_misc2;
    DevBuf b_small;    // reductions, statistics, ICP state
    DevBuf b_table;    // probe cell table
    struct Piggy {     // a small device->host copy that rides along with the next round trip of run_levels
        void *dst;
        const void *src;
        size_t bytes;
    };
    std::vector<Piggy> piggy;
    bool spec_coarser = false;         // frame stream: the previous frame's level-0 pass deferred queries
    // Frame stream, fused SOR -> normals: when the previous frame's level-0 pass left nothing for the coarser levels, the
    // next frame's deferred counts are copied to a mailbox of their own and NOT awaited; the pipeline goes on, and the
    // counts are checked at the call's last round trip.  Non-zero (rare) = the whole call is redone the careful way.
    bool spec_request = false;   // set by the caller that can redo (batch_core)
    bool spec_pending = false;   // the counts of this call are still unchecked (mailbox: pinned + 128 words)
    bool spec_zero = false;      // the previous frame's counts were all zero
    uint64_t stat_nowait_hits = 0, stat_nowait_misses = 0;
    cudaEvent_t ev_count = nullptr;    // marks the deferred count's copy when work is queued behind it
    // level 0 of the KNN runs three ways at once (knn.cu run_levels): side streams + fork / join events, created on first use
    cudaStream_t side[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    DevBuf b_scan;     // single-pass scan: ticket + one state word per tile (tagged with scan_epoch, never cleared between scans)
    uint32_t scan_epoch = 0;
    DevBuf b_list;     // deferred-query lists of the level loop
    DevBuf b_qoff;     // u32 query offsets of the external queries of a batch index (knn.cu upload_query_offsets)
    // cell tables of TRANSIENT indices (the ones an entry point builds and frees itself), one per grid
    // level.  A 100-frame batch needs a 280 MB table: taking it from the stream-ordered pool on every
    // call cost 4-16 ms (the pool had just carved the freed block up for the smaller arrays).
    DevBuf b_cells[6];
    // ... and, for the levels built on the side streams (coarser / finer), their sorted points and grid descriptors too: a
    // side-stream cudaMallocAsync finds the blocks the main stream freed after the previous call only some of the time
    // (otherwise it carves up a larger block or maps new memory: intermittent 20-700 ms host stalls on the 8 M-point batch)
    DevBuf b_lsorted[6], b_lgrids[6];
    void *pinned = nullptr;  // small pinned host mailbox
    size_t pinned_cap = 0;
    // optional per-stage device timing (cudaEvents on the context's stream; bench.py's roofline)
    bool timing = false;
    struct TimedSpan {
        cudaEvent_t a, b;
        int tag;
    };
    std::vector<TimedSpan> spans;
    unsigned long long *d_knn_stats = nullptr;  // {queries, distance evaluations} of the level-0 selection kernel while timing is on
    std::vector<cudaEvent_t> event_pool;
    // NCCL (loaded lazily with dlopen, see comm.cu)
    void *nccl_comm = nullptr;
    int rank = 0, world = 1;
    // One-shot all-reduce of the ICP sums over NVLink peer memory (comm.cu sets it up, icp.cu's reduce kernel uses it): every
    // rank owns one exchange block (cudaMalloc, shared through CUDA IPC) and holds a pointer into every peer's.
    PeerComm peer = {};
    void *peer_block = nullptr;             // this rank's block
    void *peer_open[kPeerMaxWorld] = {};    // peers' blocks as opened here (cudaIpcOpenMemHandle), nullptr for the own rank
    bool peer_ok = false;                   // all ranks agreed to use it
    unsigned long long peer_seq = 0;        // exchanges issued so far: the value the flags of the next one carry
    // pcr_ctx_set_query_sharding: with a communicator, sor / estimate_normals / radius_outlier_removal of ONE cloud
    // given in full on every rank search only this rank's share of the queries and merge the results over NCCL
    bool shard_queries = false;
    bool fake_comm = false;  // pcr_ctx_debug_set_shard: rank / world without a communicator, collectives are no-ops (partition tests on one GPU)
    // frame-stream bookkeeping for the bench line (pcr_ctx_get_hint_stats)
    uint64_t stat_cell_hits = 0, stat_cell_misses = 0, stat_vox_hits = 0, stat_vox_misses = 0, stat_spec_hits = 0, stat_spec_misses = 0;
};

// ------------------------------------------------------------------------------------------------
// error plumbing: nothing throws across the ABI
// ------------------------------------------------------------------------------------------------
int fail(Ctx *ctx, int code, const char *fmt, ...);
void set_thread_error(const char *msg);

#define PCR_CUDA(ctx, expr)                                                                       \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            cudaGetLastError();                                                                   \
            return pcr::fail((ctx), _e == cudaErrorMemoryAllocation ? PCR_ERR_OOM : PCR_ERR_CUDA, \
                             "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,    \
                             __LINE__);                                                           \
        }                                                                                         \
    } while (0)

#define PCR_TRY(expr)              \
    do {                           \
        int _s = (expr);           \
        if (_s != PCR_OK) return _s; \
    } while (0)

#define PCR_LAUNCH_CHECK(ctx)                                                                   \
    do {                                                                                        \
        (ctx)->launches++;                                                                      \
        cudaError_t _e = cudaGetLastError();                                                    \
        if (_e != cudaSuccess)                                                                  \
            return pcr::fail((ctx), PCR_ERR_CUDA, "kernel launch failed: %s (%s:%d)",           \
                             cudaGetErrorString(_e), __FILE__, __LINE__);                       \
    } while (0)

// stage tags of the timing spans (pcr_ctx_get_timing)
enum TimeTag { kTagBuild = 0, kTagKnn = 1, kTagKnnDeferred = 2, kTagSorStats = 3, kTagIcpStep = 4, kTagIcpSolve = 5, kTagKnnNormals = 6, kTagOther = 7, kNumTags = 8 };

// Host-side trace for latency work (PCR_TRACE=1): time stamps at the marks, the last ones printed when the context
// is destroyed.  Off by default; a mark is then one predictable branch.
extern bool g_trace_on;
void trace_mark(const char *label);
#define PCR_MARK(label)                            \
    do {                                           \
        if (pcr::g_trace_on) pcr::trace_mark(label); \
    } while (0)

struct TimeScope {  // records an event pair around a stage when timing is enabled
    Ctx *c;
    int idx = -1;
    TimeScope(Ctx *ctx, int tag);
    ~TimeScope();
};

int ensure(Ctx *ctx, DevBuf &b, size_t bytes);
int ensure_pinned(Ctx *ctx, size_t bytes);

// A device allocation owned by a scope: cudaMallocAsync in alloc(), cudaFreeAsync on the same stream at scope exit,
// so an error return frees it in stream order after the work already queued.
template <class T = void>
struct StreamAlloc {
    T *p = nullptr;
    cudaStream_t s;
    explicit StreamAlloc(cudaStream_t stream) : s(stream) {}
    StreamAlloc(const StreamAlloc &) = delete;
    StreamAlloc &operator=(const StreamAlloc &) = delete;
    ~StreamAlloc() {
        if (p) cudaFreeAsync(p, s);
    }
    cudaError_t alloc(size_t bytes) {
        const cudaError_t e = cudaMallocAsync((void **)&p, bytes, s);
        if (e != cudaSuccess) p = nullptr;
        return e;
    }
};

// ------------------------------------------------------------------------------------------------
// host entry points implemented across the .cu files (all asynchronous on ctx->stream)
// ------------------------------------------------------------------------------------------------
// Bounding box and finite-point count of one frame, as the index build measures them (order-preserving u32
// encodings of f32).  A step that has just written a cloud can hand them on and save the build a round trip.
struct CloudStats {
    unsigned mn[3], mx[3];
    unsigned count;
    unsigned valid;  // host side: 1 once filled (always 0 on the device)
};

struct BuildOpts {
    const CloudStats *known_stats = nullptr;  // host; single unmasked frame only
    size_t k_hint = 0;
    bool self_knn = false;  // the index serves the self-queries of SOR / normals (cell-tile kernel: larger cells, see occupancy_target)
    int n_frames = 1;
    const uint64_t *frame_offsets = nullptr;  // host, n_frames + 1 (nullptr if n_frames == 1)
    const uint8_t *d_mask = nullptr;          // optional device keep-mask: index only points with mask != 0
    bool transient = false;                   // the caller frees the index before it returns: use the context's cached cell tables
};
int index_build_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n,
                    const BuildOpts &opts, Index **out);
void index_free(Index *ix);
struct IndexFree {
    void operator()(Index *ix) const { index_free(ix); }
};
using IndexPtr = std::unique_ptr<Index, IndexFree>;  // an index owned by a scope
// The next-coarser level of `ix` (cell size x kLevelFactor), built on first use and owned by `ix`.
int index_coarser_level(Index *ix, Index **out);
// The finer level of `ix` (cell size / 2, or as fine as the cell-table cap allows), built on first use and owned by `ix`.
int index_finer_level(Index *ix, Index **out);

// External queries of a batch index (pcr_*_batch): query frame f = queries [offsets[f], offsets[f+1]) (HOST, n_frames + 1
// entries, checked by the caller) is searched in index frame f only, and the indices come back frame-local.
struct QueryFrames {
    const uint64_t *offsets;
    size_t n_frames;
};
// KNN over external queries.  d_idx/d_dist row-major nq x k.  A multi-frame index needs qf (with its frame count); on a
// single-frame index qf is ignored (a batch of one).
int knn_queries_dev(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq,
                    size_t k, uint32_t *d_idx, float *d_dist, uint32_t *d_counts, const QueryFrames *qf = nullptr);
// mean neighbour distance of every point of the indexed cloud(s) (SOR, k+1 neighbours, drop self)
// Neighbour lists a fused SOR -> normals pipeline keeps from its SOR pass (knn.cu): entry j of the query at
// cell-sorted position q is lists[j * stride + q]; cnt[q] = valid entries, 0xff = no list.
struct SorLists {
    size_t K = 0;         // neighbours searched per query (>= k_sor + 1 and >= k_normals + 1, <= 32)
    size_t stride = 0;    // >= n_indexed
    uint32_t *lists = nullptr;
    uint8_t *cnt = nullptr;
    uint32_t *fallback = nullptr;  // stride + 1 entries: query ids without a usable list, then their count
    bool initialised = false;      // cnt (0xff) and the fallback counter (0) were set by the caller, ahead of the kernels
};
int sor_mean_dist_dev(Index *ix, size_t k, float *d_mean_d, const SorLists *keep_lists = nullptr, bool allow_shard = false);
int normals_from_lists_dev(Index *ix, size_t k, const float vp[3], const SorLists &sl, const uint8_t *d_keep, float *d_nx, float *d_ny,
                           float *d_nz,
                           const unsigned long long *d_kept0 = nullptr, unsigned long long *h_kept0 = nullptr, bool early = false);
int normals_early_fork(Ctx *ctx);
int normals_early_from_lists_dev(Index *ix, size_t k, const float vp[3], const SorLists &sl, float *d_nx, float *d_ny, float *d_nz, bool *launched);
// normals of every point of the indexed cloud(s); points not indexed get (0,0,1) (no neighbours)
int normals_dev(Index *ix, size_t k, const float vp[3], float *d_nx, float *d_ny, float *d_nz,
                const uint8_t *d_mask, bool allow_shard = false);
// Query sharding (one cloud, index replicated on every rank of the context's communicator): this rank's share of the
// cell-sorted order, cut at cell boundaries so that every rank derives the same partition from its own copy of the index.
bool query_sharding_active(const Ctx *ctx, const Index *ix);
int index_shard_queries(Index *ix);
// Removes the points with keep[idx] == 0 from every built level of the index IN PLACE (their
// coordinates become NaN) and makes later-built levels skip them: the index of the SOR pass is
// reused for the normals of the kept points without a rebuild.
int index_apply_mask_dev(Index *ix, const uint8_t *d_keep);
// On a multi-frame index without qf the queries must be the indexed points themselves (query i = input point i), each
// counted in its own frame only; with qf they are external queries as in knn_queries_dev (radius_fill_dev needs qf there).
int radius_count_dev(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq,
                     float radius, uint32_t *d_counts, const QueryFrames *qf = nullptr);
int radius_fill_dev(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq,
                    float radius, const uint64_t *d_offsets, uint32_t *d_idx, const QueryFrames *qf = nullptr);

// SOR statistics + mask (statistical_outlier.rs:43-66), one segment per frame.  d_stats receives
// per frame {mean, stddev, threshold, n_finite(as float bits)}; d_kept per-frame kept counts.
int sor_threshold_mask_dev(Ctx *ctx, const float *d_mean_d, const uint32_t *d_frame_off /*dev, n_frames+1*/,
                           int n_frames, size_t n, float std_mul, uint8_t *d_keep, float *d_stats,
                           unsigned long long *d_kept, bool kept_zeroed = false /* the caller zeroed d_kept earlier in the stream */);

int exclusive_scan_u32_dev(Ctx *ctx, uint32_t *d_data, size_t n_plus_1);
int exclusive_scan_u64_from_u32_dev(Ctx *ctx, const uint32_t *d_in, uint64_t *d_out, size_t n);

struct IcpArgs {
    const float *d_sx, *d_sy, *d_sz;
    size_t ns;
    const float *d_tx, *d_ty, *d_tz;
    size_t nt;
    const float *d_nx, *d_ny, *d_nz;  // nullptr for point-to-point
    pcr_icp_params params;
    const float *init = nullptr;  // host, 12 floats (row-major R, then t): the loop's start; nullptr = identity
};
int icp_dev(Ctx *ctx, const IcpArgs &a, pcr_icp_result *result);
// Pairs of frames of one buffer (pcr_icp_point_to_*_batch, arguments checked by the caller, results preset to each pair's start).
struct IcpBatchArgs {
    const float *d_x, *d_y, *d_z;  // every frame, back to back
    size_t n;
    const uint64_t *frame_offsets;  // host, n_frames + 1
    size_t n_frames;
    const float *d_nx, *d_ny, *d_nz;  // one normal per point; nullptr for point-to-point
    const uint32_t *pairs;            // host: pair p = (source frame, target frame)
    size_t n_pairs;
    pcr_icp_params params;
    const float *inits = nullptr;  // host, 12 floats per pair (row-major R, then t): each pair's start; nullptr = identity
};
int icp_batch_dev(Ctx *ctx, const IcpBatchArgs &a, pcr_icp_result *results);
int find_correspondences_dev(Index *target, const float *dsx, const float *dsy, const float *dsz,
                             size_t ns, float max_distance, uint32_t *d_tgt, float *d_dist, const QueryFrames *qf = nullptr);
int apply_transform_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n,
                        const float R[9], const float t[3], float *ox, float *oy, float *oz);
// every frame of a batch (pcr_apply_transform_batch, arguments checked by the caller): frame f = points [frame_offsets[f],
// frame_offsets[f+1]) (host) moved by transforms[12f .. 12f+12) (host: row-major R, then t).  d_frame_off: the same offsets
// as u32 on the device if the caller holds them (a pcr_frames batch), else nullptr and they are uploaded with the transforms.
int apply_transform_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                              const uint32_t *d_frame_off, const float *transforms, float *ox, float *oy, float *oz);

// euclidean_cluster (cluster.cu): labels[i] = smallest index of the component of point i
// (d_frame_off: device frame offsets of a batch, no component crosses a frame; labels stay global indices)
int cluster_labels_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, float threshold, uint32_t *d_labels,
                       const uint32_t *d_frame_off = nullptr, int n_frames = 1);
size_t clusters_from_labels(const uint32_t *labels, size_t n, size_t min_size, size_t max_size, uint32_t *offsets, uint32_t *indices,
                            std::vector<uint32_t> &scratch);
// every frame of a batch (pcr_cluster_labels_batch_dev / pcr_euclidean_cluster_batch, arguments checked by the caller):
// frame-local labels, and the CSR of every frame in the single call's order (frame f's clusters are
// [cluster_offsets[f], cluster_offsets[f+1]), host; *total = clustered points)
int cluster_labels_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                             float threshold, uint32_t *d_labels);
int euclidean_cluster_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                                float threshold, size_t min_size, size_t max_size, uint32_t *d_offsets, uint32_t *d_indices,
                                uint64_t *cluster_offsets, size_t *total);

// voxel_downsample + the stable radix sort it uses (voxel.cu)
int voxel_downsample_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, float voxel, float *d_ox, float *d_oy,
                         float *d_oz, size_t *n_out, CloudStats *stats_out = nullptr /* host; filled (valid = 1) when it comes for free */,
                         bool allow_guess = true /* frame streams: size the table from the previous frame's key box */);
// every frame of a batch in one call (pcr_voxel_downsample_batch, arguments checked by the caller); out_offsets: host,
// n_frames + 1, frame f's voxels are [out_offsets[f], out_offsets[f+1]) of the outputs (sized frame_offsets[n_frames])
int voxel_downsample_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets,
                               size_t n_frames, float voxel, float *d_ox, float *d_oy, float *d_oz, uint64_t *out_offsets);
int radix_sort_pairs_dev(Ctx *ctx, unsigned long long **keys, uint32_t **vals, unsigned long long **keys_alt, uint32_t **vals_alt,
                         size_t n, int bits, uint32_t *d_hist);
size_t radix_sort_hist_words(size_t n);  // u32 words of radix_sort_pairs_dev's d_hist for n pairs
int bits_for(uint64_t range);            // smallest b with 2^b >= range

// ransac_plane_seeded for given samples (ransac.cu); h_samples: HOST array of m index triples
int ransac_plane_samples_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, float threshold,
                             const uint32_t *h_samples, size_t m, float model_out[4], uint32_t *d_inliers, size_t *n_inliers);
// every frame of a batch (pcr_ransac_plane_samples_batch, frame and sample offsets checked by the caller): h_samples holds
// frame-LOCAL triples, frame f's are [sample_offsets[f], sample_offsets[f+1]); models_out 4 per frame (host), frame f's
// ascending frame-local inliers at [inlier_offsets[f], inlier_offsets[f+1]) of d_inliers (inlier_offsets: host)
int ransac_plane_samples_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets,
                                   size_t n_frames, float threshold, const uint32_t *h_samples, const uint64_t *sample_offsets,
                                   float *models_out, uint32_t *d_inliers, uint64_t *inlier_offsets);

// NCCL plumbing (comm.cu)
int comm_unique_id(void *out);
int comm_init(Ctx *ctx, const void *id, int rank, int world);
void comm_destroy(Ctx *ctx);
int comm_allreduce_f64(Ctx *ctx, double *d_buf, size_t count);
int comm_allgather_bytes(Ctx *ctx, const void *d_send, void *d_recv, size_t bytes);
// in-place sum of u32 words: merges result arrays in which every element was written by exactly one rank (zero elsewhere), bit for bit
int comm_allreduce_u32(Ctx *ctx, uint32_t *d_buf, size_t count);

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
}  // namespace pcr

// the opaque handles of the C ABI
struct pcr_ctx {
    pcr::Ctx c;
};
struct pcr_index {
    pcr::Index *ix;
    pcr_ctx *owner;
};

namespace pcr {

#ifdef __CUDACC__

// Programmatic dependent launch (sm_90+): a kernel launched with launch_chained() may be scheduled while its predecessor in
// the stream is still draining; it must call PCR_GRID_DEP_SYNC() before it touches anything the predecessor wrote (here:
// as its first statement).  The predecessors never trigger early, so the wait returns when they have completed and
// flushed: what overlaps is the launch itself -- 2-4 us per kernel boundary, and the step is a chain of ~28 small kernels.
// A kernel WITHOUT the wait must never be launched this way.  PCR_NO_PDL=1 turns the attribute off (A/B hook).
// Measured and dropped: an explicit cudaTriggerProgrammaticLaunchCompletion() after the wait (no gain: 0.487 vs 0.486 ms per
// step); before the wait it lets a successor start while the predecessor's predecessor still runs and gave wrong voxel counts.
#define PCR_GRID_DEP_SYNC() cudaGridDependencySynchronize()

template <class... KArgs, class... Args>
inline cudaError_t launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    static const bool off = getenv("PCR_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = off ? 0 : 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

#define PCR_FULL 0xffffffffu
// "no entry" sentinel: just above every real key (d^2 bits <= 0x7f800000 = +inf).  A candidate whose
// d^2 is NaN -- a tombstoned point, see tombstone_kernel -- has a key >= the sentinel and can
// therefore never pass `key < threshold`, even while a list is not full yet.
#define PCR_EMPTY_KEY 0x7f80000100000000ull

// kiddo SquaredEuclidean on f32: ((dx*dx)+(dy*dy))+(dz*dz), every operation rounded, no FMA
// (call sites crates/spatial/src/kdtree.rs:70,93,121-123).
__device__ __forceinline__ float dist2_exact(float ax, float ay, float az, float bx, float by, float bz) {
    float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    float s = __fmul_rn(dx, dx);
    s = __fadd_rn(s, __fmul_rn(dy, dy));
    s = __fadd_rn(s, __fmul_rn(dz, dz));
    return s;
}

// (d^2, index) total order in one u64: d^2 >= 0, so its bit pattern is monotone.
__device__ __forceinline__ unsigned long long make_key(float d2, uint32_t idx) {
    return ((unsigned long long)__float_as_uint(d2) << 32) | idx;
}
__device__ __forceinline__ float key_d2(unsigned long long k) { return __uint_as_float((uint32_t)(k >> 32)); }
__device__ __forceinline__ uint32_t key_idx(unsigned long long k) { return (uint32_t)k; }

__device__ __forceinline__ bool finite3(float a, float b, float c) { return isfinite(a) && isfinite(b) && isfinite(c); }
// order-preserving map f32 -> u32 (so min / max of floats are integer atomics)
__device__ __forceinline__ unsigned f32_ordered(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float pick_axis(int ax, float x, float y, float z) { return ax == 0 ? x : (ax == 1 ? y : z); }

// Cell coordinate along permuted axis j and the fractional position inside that cell.  f64 on
// purpose: the error of the cell assignment then is ~1e-16 relative, which the 1e-6 slack of the
// ring-termination test (knn.cuh) covers with a wide margin.
__device__ __forceinline__ int cell_coord(const GridDesc &g, int j, float v, double *frac) {
    double t = ((double)v - g.o[j]) * g.inv_h;
    double f = floor(t);
    f = fmin(fmax(f, 0.0), (double)(g.dims[j] - 1));
    if (frac) *frac = t - f;  // < 0 or > 1 for a query outside the grid (clamped cell)
    return (int)f;
}

__device__ __forceinline__ uint32_t cell_linear(const GridDesc &g, int c0, int c1, int c2) {
    return g.cell_base + ((uint32_t)c0 * (uint32_t)g.dims[1] + (uint32_t)c1) * (uint32_t)g.dims[2] + (uint32_t)c2;
}

// frame of input point i (binary search over the frame offsets); n_frames == 1 -> 0
__device__ __forceinline__ int frame_of(const uint32_t *__restrict__ off, int n_frames, uint32_t i) {
    if (n_frames <= 1) return 0;
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

#endif  // __CUDACC__

}  // namespace pcr
