// knn.cu -- batched KNN and the consumers fused onto it.
//
//   knn_queries_kernel   KdTree::knn / knn_indices for a batch of queries   kdtree.rs:64-96
//   sor_mean_kernel      per-point mean neighbour distance                  statistical_outlier.rs:19-39
//   normals_kernel       covariance + Cardano eigenvector + orientation     estimate.rs:42-109,139-238
//   radius_*_kernel      radius_search[_unsorted]                           kdtree.rs:105-163
//
// Work layout: one warp per query for the search (lanes stream candidates, the top-k lives in
// registers, one entry per lane); every warp takes 32 consecutive queries of the CELL-SORTED order
// (neighbouring queries touch the same cells, so the runs they stream stay in L1), parks the 32
// results in shared memory transposed, and then runs the per-query epilogue with one THREAD per
// query -- the epilogues are sequential f32 folds in neighbour order (that order is part of the
// reference's arithmetic), which would waste 31 lanes if done warp-wide.
#include "knn_search.cuh"
#include "knn_tile.cuh"

#include <algorithm>
#include <vector>
#include <type_traits>

namespace pcr {

namespace {

constexpr int kWarps = 4;              // warps per block
constexpr int kThreads = kWarps * 32;
constexpr int kQPW0 = 32;              // queries per warp on level 0 (consecutive in cell order)
constexpr int kQPWL = 1;               // queries per warp on the deferred lists (few, long queries)
constexpr int kQPWS = 4;               // queries per warp on level 0 when a warp takes one query at a time (warp_select_cube)

// One pass over one level of the grid.  Level 0 takes every query; level l > 0 takes the queries
// the previous level deferred (qlist) and searches the 8x coarser grid of that level.
struct LevelArgs {
    const GridDesc *grids;
    int n_frames;
    const uint32_t *cell_start;
    const float4 *pts;         // this level's cell-sorted points
    const float4 *qpts;        // level-0 sorted points: where self-queries are read from
    const uint32_t *qlist;     // nullptr on level 0 (query id == position)
    const uint32_t *qlist2;    // tile kernel: a second list that is taken FIRST (its length in *nq2_dev), then qlist
    const uint32_t *nq2_dev;
    uint32_t nq;
    uint32_t q_offset;         // level 0 without a list: query id = q_offset + slot (this rank's query shard)
    const uint32_t *nq_dev;    // optional: the real count, still on the device (nq is then the launch capacity)
    uint32_t *defer_list;      // queries this pass could not finish within max_rings shells
    uint32_t *defer_count;
    int max_rings;
    int last_level;
    // selection kernels (knn_sel_kernel): the first pass stops after the 27 cells and queues the queries the ring
    // rule cannot confirm yet; a second launch of the same kernel takes them from cont_list through the shells
    int first_only;  // shells the first pass walks (0: this is not a first pass)
    uint32_t *cont_list;
    uint32_t *cont_count;
    int follow_up;  // this launch takes cont_list of the first pass (warp per query, same grid level)
    // cell-tile kernel (knn_tile_kernel): queries it hands back to the thread-per-query selection kernel
    uint32_t *ovf_list;
    uint32_t *ovf_count;
    int no_tile;    // this launch is the dense class / the overflow list: thread per query
    unsigned long long *prof;  // PCR_TILE_PROF: per-warp cycle counters of the tile kernel (8 words per warp)
    unsigned long long *stats;  // optional {queries, distance evaluations} counters of the selection kernel (timing on)
};

__device__ __forceinline__ void defer_query(const LevelArgs &a, uint32_t qid, int lane) {
    if (lane == 0) a.defer_list[atomicAdd(a.defer_count, 1u)] = qid;
}

__device__ __forceinline__ int frame_of_sorted(const GridDesc *__restrict__ grids, int n_frames, uint32_t pos) {
    if (n_frames <= 1) return 0;
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (grids[mid].pt_begin <= pos) lo = mid;
        else hi = mid - 1;
    }
    // skip empty frames that share pt_begin
    while (lo + 1 < n_frames && grids[lo].pt_end <= pos) lo++;
    return lo;
}

// ---- external queries -----------------------------------------------------------------------------
// base: subtracted from every emitted index (a batch index: the query's frame's first input point -> frame-local indices)
template <class TopK>
__device__ __forceinline__ void emit_row(const TopK &tk, int cnt, size_t k, size_t qi, uint32_t *__restrict__ idx,
                                         float *__restrict__ dist, uint32_t base);

template <>
__device__ __forceinline__ void emit_row<RegTopK>(const RegTopK &tk, int cnt, size_t k, size_t qi,
                                                  uint32_t *__restrict__ idx, float *__restrict__ dist, uint32_t base) {
    if ((size_t)tk.lane < k) {
        bool v = tk.lane < cnt;
        idx[qi * k + tk.lane] = v ? key_idx(tk.K) - base : 0xffffffffu;
        if (dist) dist[qi * k + tk.lane] = v ? __fsqrt_rn(key_d2(tk.K)) : INFINITY;  // kdtree.rs:76
    }
}
template <>
__device__ __forceinline__ void emit_row<SmemTopK>(const SmemTopK &tk, int cnt, size_t k, size_t qi,
                                                   uint32_t *__restrict__ idx, float *__restrict__ dist, uint32_t base) {
    for (size_t j = tk.lane; j < k; j += 32) {
        bool v = j < (size_t)cnt;
        unsigned long long key = v ? tk.s[j] : 0ull;
        idx[qi * k + j] = v ? key_idx(key) - base : 0xffffffffu;
        if (dist) dist[qi * k + j] = v ? __fsqrt_rn(key_d2(key)) : INFINITY;
    }
}

// kQFrames (batch index): query qi belongs to query frame f = frame_of(qoff, a.n_frames, qi) and is searched in grid f of
// the level only; indices come back frame-local.  The single-frame calls pass no qoff.
// (kQFrames, warp per query: the frame's grid stays live through the search; 7 blocks per SM instead of 8 keep its spills below
// the single-frame form's)
template <bool kSmem, int QPW, bool kQFrames = false>
__global__ void __launch_bounds__(kThreads, (!kSmem && QPW == kQPWS) ? (kQFrames ? 7 : 8) : 1) knn_queries_kernel(LevelArgs a, const float *__restrict__ qx,
                                                               const float *__restrict__ qy, const float *__restrict__ qz,
                                                               int kk, uint32_t *__restrict__ idx, float *__restrict__ dist,
                                                               uint32_t *__restrict__ counts, const uint32_t *__restrict__ qoff = nullptr) {
    extern __shared__ unsigned long long smem_keys[];
    __shared__ WarpSelScratch s_sel[kWarps];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    GridDesc g = a.grids[0];
    typename std::conditional<kSmem, SmemTopK, RegTopK>::type tk;
    tk.kk = kk;
    tk.lane = lane;
    if constexpr (kSmem) tk.s = smem_keys + (size_t)w * kk;
    const uint32_t nq = a.nq_dev ? min(a.nq, *a.nq_dev) : a.nq;  // (a launch for a capacity strides over the real count)
    for (uint32_t q0 = (blockIdx.x * kWarps + w) * QPW; q0 < nq; q0 += gridDim.x * kWarps * QPW)
    for (int t = 0; t < QPW; t++) {
        if (q0 + t >= nq) break;
        const uint32_t qi = a.qlist ? a.qlist[q0 + t] : a.q_offset + q0 + t;
        float x = __ldg(&qx[qi]), y = __ldg(&qy[qi]), z = __ldg(&qz[qi]);
        int cnt = 0;
        tk.reset(PCR_EMPTY_KEY);
        bool searchable = finite3(x, y, z);  // kdtree.rs:65
        if constexpr (kQFrames) {
            g = a.grids[frame_of(qoff, a.n_frames, qi)];
            searchable = searchable && g.pt_end > g.pt_begin;  // (an empty index frame: no neighbours)
        }
        if (searchable) {
            if (!warp_knn_search(tk, g, a.cell_start, a.pts, x, y, z, a.max_rings, a.last_level != 0, PCR_EMPTY_KEY, (QPW == kQPWS || a.no_tile) ? &s_sel[w] : nullptr)) {
                defer_query(a, qi, lane);
                continue;
            }
            cnt = tk.count();
        }
        emit_row(tk, cnt, (size_t)kk, (size_t)qi, idx, dist, kQFrames ? g.in_begin : 0u);
        if (counts && lane == 0) counts[qi] = (uint32_t)cnt;
        if constexpr (kSmem) __syncwarp();
    }
}

// ---- SOR: mean distance to the k nearest neighbours (k+1 searched, self dropped) ----------------
// smem per warp: dist[(kk)][33] f32 (transposed: neighbour-major) + cnt[32]
// `lists` (optional, register path only): the fused SOR -> normals pipeline keeps the kk >= kk_sor neighbours
// of every query (SorLists layout); the statistic then uses the first kk_sor entries.
template <bool kSmem, int QPW>
__global__ void __launch_bounds__(kThreads, (!kSmem && QPW == kQPWS) ? 8 : 1) sor_mean_kernel(LevelArgs a, int kk, float *__restrict__ mean_d, uint32_t *__restrict__ lists,
                                                            uint8_t *__restrict__ list_cnt, size_t list_stride, int kk_sor) {
    PCR_GRID_DEP_SYNC();
    extern __shared__ unsigned long long smem_raw[];
    __shared__ WarpSelScratch s_sel[kWarps];
    constexpr int kCol = QPW + 1;  // column stride of the parked results (conflict-free transposed reads)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t nq = a.nq_dev ? min(a.nq, *a.nq_dev) : a.nq;  // (a launch for a capacity strides over the real count)
    for (uint32_t q0 = (blockIdx.x * kWarps + w) * QPW; q0 < nq; q0 += gridDim.x * kWarps * QPW) {
    if constexpr (!kSmem) {
        float *sd = reinterpret_cast<float *>(smem_raw) + (size_t)w * (kk * kCol + 64);
        int *scnt = reinterpret_cast<int *>(sd + kk * kCol);
        uint32_t *spos = reinterpret_cast<uint32_t *>(scnt + 32);
        RegTopK tk;
        tk.kk = kk;
        tk.lane = lane;
        int f = -1;
        GridDesc g;
        for (int t = 0; t < QPW; t++) {
            if (q0 + t >= nq) break;
            const uint32_t pos = a.qlist ? a.qlist[q0 + t] : a.q_offset + q0 + t;
            if (f < 0 || pos >= g.pt_end || pos < g.pt_begin) {
                f = frame_of_sorted(a.grids, a.n_frames, pos);
                g = a.grids[f];
            }
            float4 q = __ldg(&a.qpts[pos]);
            if (q.x != q.x) {  // tombstoned point: not a query
                if (lane == 0) scnt[t] = -1;
                continue;
            }
            bool done = warp_knn_search(tk, g, a.cell_start, a.pts, q.x, q.y, q.z, a.max_rings, a.last_level != 0, PCR_EMPTY_KEY, (QPW == kQPWS || a.no_tile) ? &s_sel[w] : nullptr);
            int cnt = tk.count();
            if (!done) {
                defer_query(a, pos, lane);
                cnt = -1;
            } else if (lane < kk) {
                sd[lane * kCol + t] = __fsqrt_rn(key_d2(tk.K));  // kdtree.rs:76
                if (lists) lists[(size_t)lane * list_stride + pos] = lane < cnt ? key_idx(tk.K) : 0xffffffffu;
            }
            if (lane == 0) {
                scnt[t] = cnt;
                spos[t] = pos;
                if (lists && done) list_cnt[pos] = (uint8_t)cnt;
            }
        }
        __syncwarp();
        if (lane < QPW && q0 + lane < nq) {
            int cnt = scnt[lane];
            if (cnt >= 0) {
                // statistical_outlier.rs:28-37: drop the first (self) if there is more than one
                // result, sequential f32 sum in ascending-distance order, divide by the count
                if (cnt > kk_sor) cnt = kk_sor;  // (the top-kk list starts with the top-kk_sor list)
                int first = cnt > 1 ? 1 : 0;
                float sum = 0.0f;
                for (int j = first; j < cnt; j++) sum = __fadd_rn(sum, sd[j * kCol + lane]);
                int m = cnt - first;
                float md = m > 0 ? __fdiv_rn(sum, (float)m) : INFINITY;
                mean_d[__float_as_uint(__ldg(&a.qpts[spos[lane]]).w)] = md;
            }
        }
        __syncwarp();
    } else {
        SmemTopK tk;
        tk.kk = kk;
        tk.lane = lane;
        tk.s = smem_raw + (size_t)w * kk;
        for (int t = 0; t < QPW; t++) {
            if (q0 + t >= nq) break;
            const uint32_t pos = a.qlist ? a.qlist[q0 + t] : a.q_offset + q0 + t;
            const GridDesc g = a.grids[frame_of_sorted(a.grids, a.n_frames, pos)];
            float4 q = __ldg(&a.qpts[pos]);
            if (q.x != q.x) continue;  // tombstoned point: not a query
            bool done = warp_knn_search(tk, g, a.cell_start, a.pts, q.x, q.y, q.z, a.max_rings, a.last_level != 0);
            __syncwarp();
            if (!done) {
                defer_query(a, pos, lane);
            } else if (lane == 0) {
                int cnt = tk.count();
                int first = cnt > 1 ? 1 : 0;
                float sum = 0.0f;
                for (int j = first; j < cnt; j++) sum = __fadd_rn(sum, __fsqrt_rn(key_d2(tk.s[j])));
                int m = cnt - first;
                mean_d[__float_as_uint(q.w)] = m > 0 ? __fdiv_rn(sum, (float)m) : INFINITY;
            }
            __syncwarp();
        }
    }
    }
}

// ---- normals ----------------------------------------------------------------------------------------
// estimate.rs:139-238, f64 internally (compiled with -fmad=false: like the reference, no fusing)
__device__ __forceinline__ void smallest_eigenvector_3x3(float fa00, float fa01, float fa02, float fa11, float fa12,
                                                         float fa22, float &ox, float &oy, float &oz) {
    const double a00 = fa00, a01 = fa01, a02 = fa02, a11 = fa11, a12 = fa12, a22 = fa22;
    const double m = (a00 + a11 + a22) / 3.0;
    const double b00 = a00 - m, b11 = a11 - m, b22 = a22 - m;
    const double q = (b00 * (b11 * b22 - a12 * a12) - a01 * (a01 * b22 - a12 * a02) + a02 * (a01 * a12 - b11 * a02)) / 2.0;
    const double p = (b00 * b00 + b11 * b11 + b22 * b22 + 2.0 * (a01 * a01 + a02 * a02 + a12 * a12)) / 6.0;
    const double pp = p > 0.0 ? p : 0.0;  // f64::max(0.0): NaN -> 0.0
    ox = 0.f; oy = 0.f; oz = 1.f;
    if (pp < 1e-30) return;
    const double sqrt_p = sqrt(pp);
    double det_ratio = q / (pp * sqrt_p);
    det_ratio = det_ratio < -1.0 ? -1.0 : (det_ratio > 1.0 ? 1.0 : det_ratio);
    const double phi = acos(det_ratio) / 3.0;
    const double FRAC_PI_3 = 1.04719755119659774615421446109316763;
    const double eig0 = m + 2.0 * sqrt_p * cos(phi + 2.0 * FRAC_PI_3);
    const double eig2 = m + 2.0 * sqrt_p * cos(phi);
    const double eig1 = 3.0 * m - eig0 - eig2;
    double lambda;
    if (fabs(eig0) <= fabs(eig1) && fabs(eig0) <= fabs(eig2)) lambda = eig0;
    else if (fabs(eig1) <= fabs(eig2)) lambda = eig1;
    else lambda = eig2;
    const double r00 = a00 - lambda, r11 = a11 - lambda, r22 = a22 - lambda;
    double ex = a01 * a12 - r11 * a02, ey = a02 * a01 - a12 * r00, ez = r00 * r11 - a01 * a01;
    double len2 = ex * ex + ey * ey + ez * ez;
    if (len2 < 1e-30) {
        ex = a01 * r22 - a12 * a02; ey = a02 * a02 - r22 * r00; ez = r00 * a12 - a01 * a02;
        len2 = ex * ex + ey * ey + ez * ez;
        if (len2 < 1e-30) {
            ex = r11 * r22 - a12 * a12; ey = a12 * a02 - r22 * a01; ez = a01 * a12 - r11 * a02;
            len2 = ex * ex + ey * ey + ez * ez;
            if (len2 < 1e-30) return;
        }
    }
    const double inv = 1.0 / sqrt(len2);
    ox = (float)(ex * inv);
    oy = (float)(ey * inv);
    oz = (float)(ez * inv);
}

// estimate.rs:47-109 for one point whose neighbours' coordinates are read through `nb(j, c)`
template <class NB>
__device__ __forceinline__ void normal_from_neighbours(int cnt, NB nb, float px, float py, float pz, float vx_, float vy_,
                                                       float vz_, float &nx, float &ny, float &nz) {
    if (cnt < 1) {
        nx = 0.f; ny = 0.f; nz = 1.f;
        return;
    }
    const float count = (float)cnt;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    for (int j = 0; j < cnt; j++) {
        cx = __fadd_rn(cx, nb(j, 0));
        cy = __fadd_rn(cy, nb(j, 1));
        cz = __fadd_rn(cz, nb(j, 2));
    }
    cx = __fdiv_rn(cx, count);
    cy = __fdiv_rn(cy, count);
    cz = __fdiv_rn(cz, count);
    float c00 = 0.f, c01 = 0.f, c02 = 0.f, c11 = 0.f, c12 = 0.f, c22 = 0.f;
    for (int j = 0; j < cnt; j++) {
        float dx = __fsub_rn(nb(j, 0), cx), dy = __fsub_rn(nb(j, 1), cy), dz = __fsub_rn(nb(j, 2), cz);
        c00 = __fadd_rn(c00, __fmul_rn(dx, dx));
        c01 = __fadd_rn(c01, __fmul_rn(dx, dy));
        c02 = __fadd_rn(c02, __fmul_rn(dx, dz));
        c11 = __fadd_rn(c11, __fmul_rn(dy, dy));
        c12 = __fadd_rn(c12, __fmul_rn(dy, dz));
        c22 = __fadd_rn(c22, __fmul_rn(dz, dz));
    }
    float ex, ey, ez;
    smallest_eigenvector_3x3(c00, c01, c02, c11, c12, c22, ex, ey, ez);
    float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez)));
    if (len > 1e-10f) {
        ex = __fdiv_rn(ex, len);
        ey = __fdiv_rn(ey, len);
        ez = __fdiv_rn(ez, len);
    }
    float vx = __fsub_rn(vx_, px), vy = __fsub_rn(vy_, py), vz = __fsub_rn(vz_, pz);
    float dot = __fadd_rn(__fadd_rn(__fmul_rn(ex, vx), __fmul_rn(ey, vy)), __fmul_rn(ez, vz));
    if (dot < 0.0f) {
        ex = -ex; ey = -ey; ez = -ez;
    }
    nx = ex; ny = ey; nz = ez;
}

// smem per warp (register path): coords[(kk*3)][33] f32 + cnt[32] + pos[32]
template <bool kSmem, int QPW>
__global__ void __launch_bounds__(kThreads, (!kSmem && QPW == kQPWS) ? 8 : 1) normals_kernel(LevelArgs a, const float4 *__restrict__ orig4, int kk, float vx,
                                                           float vy, float vz, float *__restrict__ nx, float *__restrict__ ny,
                                                           float *__restrict__ nz) {
    extern __shared__ unsigned long long smem_raw[];
    __shared__ WarpSelScratch s_sel[kWarps];
    constexpr int kCol = QPW + 1;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t nq = a.nq_dev ? min(a.nq, *a.nq_dev) : a.nq;  // (a launch for a capacity strides over the real count)
    for (uint32_t q0 = (blockIdx.x * kWarps + w) * QPW; q0 < nq; q0 += gridDim.x * kWarps * QPW) {
    if constexpr (!kSmem) {
        float *sc = reinterpret_cast<float *>(smem_raw) + (size_t)w * (kk * 3 * kCol + 64);
        int *scnt = reinterpret_cast<int *>(sc + kk * 3 * kCol);
        uint32_t *spos = reinterpret_cast<uint32_t *>(scnt + 32);
        RegTopK tk;
        tk.kk = kk;
        tk.lane = lane;
        int f = -1;
        GridDesc g;
        for (int t = 0; t < QPW; t++) {
            if (q0 + t >= nq) break;
            const uint32_t pos = a.qlist ? a.qlist[q0 + t] : a.q_offset + q0 + t;
            if (f < 0 || pos >= g.pt_end || pos < g.pt_begin) {
                f = frame_of_sorted(a.grids, a.n_frames, pos);
                g = a.grids[f];
            }
            float4 q = __ldg(&a.qpts[pos]);
            if (q.x != q.x) {  // tombstoned point: not a query
                if (lane == 0) scnt[t] = -1;
                continue;
            }
            bool done = warp_knn_search(tk, g, a.cell_start, a.pts, q.x, q.y, q.z, a.max_rings, a.last_level != 0, PCR_EMPTY_KEY, (QPW == kQPWS || a.no_tile) ? &s_sel[w] : nullptr);
            int cnt = tk.count();
            if (!done) {
                defer_query(a, pos, lane);
                cnt = -1;
            } else if (lane < cnt) {  // gather the neighbour's coordinates once (one 16 B load per lane)
                float4 p = __ldg(&orig4[key_idx(tk.K)]);
                sc[(lane * 3 + 0) * kCol + t] = p.x;
                sc[(lane * 3 + 1) * kCol + t] = p.y;
                sc[(lane * 3 + 2) * kCol + t] = p.z;
            }
            if (lane == 0) {
                scnt[t] = cnt;
                spos[t] = pos;
            }
        }
        __syncwarp();
        if (lane < QPW && q0 + lane < nq && scnt[lane] >= 0) {
            float4 q = __ldg(&a.qpts[spos[lane]]);
            float ox, oy, oz;
            normal_from_neighbours(scnt[lane], [&](int j, int c) { return sc[(j * 3 + c) * kCol + lane]; }, q.x, q.y, q.z, vx, vy,
                                   vz, ox, oy, oz);
            uint32_t oi = __float_as_uint(q.w);
            nx[oi] = ox;
            ny[oi] = oy;
            nz[oi] = oz;
        }
        __syncwarp();
    } else {
        SmemTopK tk;
        tk.kk = kk;
        tk.lane = lane;
        tk.s = smem_raw + (size_t)w * kk;
        for (int t = 0; t < QPW; t++) {
            if (q0 + t >= nq) break;
            const uint32_t pos = a.qlist ? a.qlist[q0 + t] : a.q_offset + q0 + t;
            const GridDesc g = a.grids[frame_of_sorted(a.grids, a.n_frames, pos)];
            float4 q = __ldg(&a.qpts[pos]);
            if (q.x != q.x) continue;  // tombstoned point: not a query
            bool done = warp_knn_search(tk, g, a.cell_start, a.pts, q.x, q.y, q.z, a.max_rings, a.last_level != 0);
            __syncwarp();
            if (!done) {
                defer_query(a, pos, lane);
            } else if (lane == 0) {
                float ox, oy, oz;
                const unsigned long long *s = tk.s;
                normal_from_neighbours(tk.count(),
                                       [&](int j, int c) {
                                           float4 p = __ldg(&orig4[key_idx(s[j])]);
                                           return c == 0 ? p.x : (c == 1 ? p.y : p.z);
                                       },
                                       q.x, q.y, q.z, vx, vy, vz, ox, oy, oz);
                uint32_t oi = __float_as_uint(q.w);
                nx[oi] = ox;
                ny[oi] = oy;
                nz[oi] = oz;
            }
            __syncwarp();
        }
    }
    }
}

// ---- level 0, k <= 32: one THREAD per query, top-k in registers -----------------------------------
struct ThreadArgs {
    // MODE 0: external queries
    const float *qx, *qy, *qz;
    uint32_t *idx;
    float *dist;
    uint32_t *counts;
    // MODE 1: SOR
    float *mean_d;
    // MODE 2: normals
    const float4 *orig4;
    float vx, vy, vz;
    float *nx, *ny, *nz;
    int kk;
    // MODE 3: SOR whose neighbour lists are kept for the normals of the same pipeline
    uint32_t *lists;     // [kk][list_stride]: entry j of the query at cell-sorted position q at lists[j * list_stride + q]
    uint8_t *list_cnt;   // [list_stride]: valid entries (0xff = no list: the query was deferred)
    size_t list_stride;
    int kk_sor;          // k_sor + 1 <= kk: the SOR statistic uses the first kk_sor entries
    // MODE 0 on a batch index (kQFrames): device query offsets [n_frames + 1], query frame f searched in index frame f only
    const uint32_t *qoff;
};

constexpr int kTQThreads = 128;

// estimate.rs:47-109 with the neighbour list in registers (static indexing: no local memory)
template <int KC>
__device__ __forceinline__ void normal_from_topk(const ThreadTopK<KC> &acc, int cnt, const float4 *__restrict__ orig4, float px,
                                                 float py, float pz, float vx_, float vy_, float vz_, float &nx, float &ny,
                                                 float &nz) {
    if (cnt < 1) {
        nx = 0.f; ny = 0.f; nz = 1.f;
        return;
    }
    const float count = (float)cnt;
    float cx = 0.f, cy = 0.f, cz = 0.f;
#pragma unroll
    for (int j = 0; j < KC; j++)
        if (j < cnt) {
            float4 p = __ldg(&orig4[key_idx(acc.K[j])]);
            cx = __fadd_rn(cx, p.x);
            cy = __fadd_rn(cy, p.y);
            cz = __fadd_rn(cz, p.z);
        }
    cx = __fdiv_rn(cx, count);
    cy = __fdiv_rn(cy, count);
    cz = __fdiv_rn(cz, count);
    float c00 = 0.f, c01 = 0.f, c02 = 0.f, c11 = 0.f, c12 = 0.f, c22 = 0.f;
#pragma unroll
    for (int j = 0; j < KC; j++)
        if (j < cnt) {
            float4 p = __ldg(&orig4[key_idx(acc.K[j])]);  // second pass: L1 hits
            float dx = __fsub_rn(p.x, cx), dy = __fsub_rn(p.y, cy), dz = __fsub_rn(p.z, cz);
            c00 = __fadd_rn(c00, __fmul_rn(dx, dx));
            c01 = __fadd_rn(c01, __fmul_rn(dx, dy));
            c02 = __fadd_rn(c02, __fmul_rn(dx, dz));
            c11 = __fadd_rn(c11, __fmul_rn(dy, dy));
            c12 = __fadd_rn(c12, __fmul_rn(dy, dz));
            c22 = __fadd_rn(c22, __fmul_rn(dz, dz));
        }
    float ex, ey, ez;
    smallest_eigenvector_3x3(c00, c01, c02, c11, c12, c22, ex, ey, ez);
    float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez)));
    if (len > 1e-10f) {
        ex = __fdiv_rn(ex, len);
        ey = __fdiv_rn(ey, len);
        ez = __fdiv_rn(ez, len);
    }
    float vx = __fsub_rn(vx_, px), vy = __fsub_rn(vy_, py), vz = __fsub_rn(vz_, pz);
    float dot = __fadd_rn(__fadd_rn(__fmul_rn(ex, vx), __fmul_rn(ey, vy)), __fmul_rn(ez, vz));
    if (dot < 0.0f) {
        ex = -ex; ey = -ey; ez = -ez;
    }
    nx = ex; ny = ey; nz = ez;
}

template <int KC, int MODE, bool kQFrames = false>
__global__ void __launch_bounds__(kTQThreads) knn_thread_kernel(LevelArgs a, ThreadArgs t) {
    const uint32_t q = a.q_offset + blockIdx.x * kTQThreads + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool active = q - a.q_offset < a.nq;
    ThreadTopK<KC> acc;
    acc.kk = t.kk;
    bool resolved = true, skip = false;
    float px = 0.f, py = 0.f, pz = 0.f;
    uint32_t out = q;
    int cnt = 0;
    if (active) {
        bool searchable = true;
        int f = 0;
        if (MODE == 0) {
            px = __ldg(&t.qx[q]);
            py = __ldg(&t.qy[q]);
            pz = __ldg(&t.qz[q]);
            searchable = finite3(px, py, pz);  // kdtree.rs:65
            if constexpr (kQFrames) {
                f = frame_of(t.qoff, a.n_frames, q);
                searchable = searchable && a.grids[f].pt_end > a.grids[f].pt_begin;  // (an empty index frame: no neighbours)
            }
        } else {
            float4 p = __ldg(&a.qpts[q]);
            px = p.x; py = p.y; pz = p.z;
            out = __float_as_uint(p.w);
            f = frame_of_sorted(a.grids, a.n_frames, q);
            searchable = px == px;  // a tombstoned point (index_apply_mask_dev) is not a query either
            skip = !searchable;
        }
        acc.reset();
        if (searchable) {
            const GridDesc g = a.grids[f];
            // short lists tighten quickly, so skipping the rows / cells beyond the current k-th best pays
            // (SOR k = 10 on the 122 K frame: 153 -> 112 us); for k = 20 the extra per-row arithmetic and the
            // more ragged trip counts cost more than the skipped candidates save (212 -> 225 us, measured)
            if constexpr (KC <= 12)
                resolved = thread_grid_search_pruned(acc, g, a.cell_start, a.pts, px, py, pz, t.kk, a.max_rings, a.last_level != 0);
            else
                resolved = thread_grid_search(acc, g, a.cell_start, a.pts, px, py, pz, t.kk, a.max_rings, a.last_level != 0);
            cnt = acc.count();
        }
    }
    // deferred queries: one atomic per warp
    const unsigned dmask = __ballot_sync(PCR_FULL, active && !resolved);
    if (dmask) {
        uint32_t base = 0;
        if (lane == __ffs(dmask) - 1) base = atomicAdd(a.defer_count, (uint32_t)__popc(dmask));
        base = __shfl_sync(PCR_FULL, base, __ffs(dmask) - 1);
        if (active && !resolved) a.defer_list[base + __popc(dmask & ((1u << lane) - 1u))] = q;
    }
    if (!active || !resolved || skip) return;
    if (MODE == 0) {
        uint32_t *ri = t.idx + (size_t)q * t.kk;
        float *rd = t.dist ? t.dist + (size_t)q * t.kk : nullptr;
        // (frame-local indices; the frame is looked up again rather than kept live through the search)
        const uint32_t base = kQFrames ? a.grids[frame_of(t.qoff, a.n_frames, q)].in_begin : 0u;
#pragma unroll
        for (int j = 0; j < KC; j++)
            if (j < t.kk) {
                bool v = j < cnt;
                ri[j] = v ? key_idx(acc.K[j]) - base : 0xffffffffu;
                if (rd) rd[j] = v ? __fsqrt_rn(key_d2(acc.K[j])) : INFINITY;  // kdtree.rs:76
            }
        if (t.counts) t.counts[q] = (uint32_t)cnt;
    } else if (MODE == 3) {
        // SOR on the first kk_sor entries of the list (the top-kk list starts with the top-kk_sor list), and
        // the whole list kept for normals_from_lists_kernel
        const int cs = cnt < t.kk_sor ? cnt : t.kk_sor;
        const int first = cs > 1 ? 1 : 0;
        float sum = 0.0f;
#pragma unroll
        for (int j = 0; j < KC; j++)
            if (j >= first && j < cs) sum = __fadd_rn(sum, __fsqrt_rn(key_d2(acc.K[j])));
        const int m = cs - first;
        t.mean_d[out] = m > 0 ? __fdiv_rn(sum, (float)m) : INFINITY;
#pragma unroll
        for (int j = 0; j < KC; j++)
            if (j < t.kk) t.lists[(size_t)j * t.list_stride + q] = j < cnt ? key_idx(acc.K[j]) : 0xffffffffu;
        t.list_cnt[q] = (uint8_t)cnt;
    } else if (MODE == 1) {
        // statistical_outlier.rs:28-37: drop the first (self) if there is more than one result,
        // sequential f32 sum in ascending-distance order, divide by the count
        const int first = cnt > 1 ? 1 : 0;
        float sum = 0.0f;
#pragma unroll
        for (int j = 0; j < KC; j++)
            if (j >= first && j < cnt) sum = __fadd_rn(sum, __fsqrt_rn(key_d2(acc.K[j])));
        const int m = cnt - first;
        t.mean_d[out] = m > 0 ? __fdiv_rn(sum, (float)m) : INFINITY;
    } else {
        float ox, oy, oz;
        normal_from_topk<KC>(acc, cnt, t.orig4, px, py, pz, t.vx, t.vy, t.vz, ox, oy, oz);
        t.nx[out] = ox;
        t.ny[out] = oy;
        t.nz[out] = oz;
    }
}

template <int MODE, bool kQFrames = false>
int launch_sel_kernel(Ctx *ctx, const LevelArgs &a, const ThreadArgs &t);
inline bool use_select(int kk);
template <class Kern>
int set_smem(Ctx *ctx, Kern kern, size_t bytes);

template <int MODE, bool kQFrames = false>
int launch_thread_kernel(Ctx *ctx, const LevelArgs &a, const ThreadArgs &t) {
    if (use_select(t.kk)) return launch_sel_kernel<MODE, kQFrames>(ctx, a, t);
    const unsigned blocks = (a.nq + kTQThreads - 1) / kTQThreads;
    const int kk = t.kk;
#define PCR_TQ(KC)                                                                          \
    if (kk <= KC) {                                                                         \
        knn_thread_kernel<KC, MODE, kQFrames><<<blocks, kTQThreads, 0, ctx->stream>>>(a, t); \
        PCR_LAUNCH_CHECK(ctx);                                                              \
        return PCR_OK;                                                                      \
    }
    PCR_TQ(2) PCR_TQ(4) PCR_TQ(8) PCR_TQ(11) PCR_TQ(12) PCR_TQ(16) PCR_TQ(20) PCR_TQ(21) PCR_TQ(24) PCR_TQ(32)
#undef PCR_TQ
    return fail(ctx, PCR_ERR_UNSUPPORTED, "thread kernel: k too large");
}

// ---- level 0, k <= kSelMaxK: one thread per query, selection instead of insertion (knn_search.cuh) ----
// The k best keys of a thread end up sorted in its column of the block's shared buffer; the epilogues are
// the ones of knn_thread_kernel, reading the list from there.
__device__ __forceinline__ void push_list(bool mine, uint32_t *__restrict__ list, uint32_t *__restrict__ count, uint32_t q, int lane) {
    const unsigned mask = __ballot_sync(PCR_FULL, mine);
    if (!mask) return;
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(count, (uint32_t)__popc(mask));
    base = __shfl_sync(PCR_FULL, base, leader);
    if (mine) list[base + __popc(mask & ((1u << lane) - 1u))] = q;
}

// (kQFrames: the query's grid pointer stays live through the search; 5 blocks per SM instead of 6 keep it free of spills)
template <int MODE, bool kQFrames = false>
__global__ void __launch_bounds__(kTQThreads, kQFrames ? 5 : 6) knn_sel_kernel(LevelArgs a, ThreadArgs t) {
    static_assert(kTQThreads == kSelStride, "one buffer column per thread");
    const uint32_t nq = a.nq_dev ? min(a.nq, *a.nq_dev) : a.nq;
    if (blockIdx.x * kTQThreads >= nq) return;  // (block-uniform: the follow-up pass is launched for a capacity)
    const uint32_t slot = blockIdx.x * kTQThreads + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool active = slot < nq;
    const uint32_t q = active ? (a.qlist ? a.qlist[slot] : a.q_offset + slot) : 0u;
    ThreadSel acc;
    acc.kk = t.kk;
    bool searchable = false, skip = false;
    float px = 0.f, py = 0.f, pz = 0.f;
    uint32_t out = q;
    int f = 0;
    if (active) {
        if (MODE == 0) {
            px = __ldg(&t.qx[q]);
            py = __ldg(&t.qy[q]);
            pz = __ldg(&t.qz[q]);
            searchable = finite3(px, py, pz);  // kdtree.rs:65
            if constexpr (kQFrames) {
                f = frame_of(t.qoff, a.n_frames, q);
                searchable = searchable && a.grids[f].pt_end > a.grids[f].pt_begin;  // (an empty index frame: no neighbours)
            }
        } else {
            const float4 p = __ldg(&a.qpts[q]);
            px = p.x; py = p.y; pz = p.z;
            out = __float_as_uint(p.w);
            f = frame_of_sorted(a.grids, a.n_frames, q);
            searchable = px == px;  // a tombstoned point (index_apply_mask_dev) is not a query either
            skip = !searchable;
        }
    }
    const int outcome = ws_grid_search(acc, searchable, a.grids + f, a.cell_start, a.pts, px, py, pz, a.max_rings, a.last_level != 0, a.first_only);
    push_list(outcome == kSelDefer, a.defer_list, a.defer_count, q, lane);
    if (a.cont_list) push_list(outcome == kSelContinue, a.cont_list, a.cont_count, q, lane);
    if (a.stats) {  // (bench.py: candidates per query of the dominant kernel)
        const unsigned evals = __reduce_add_sync(PCR_FULL, acc.n_eval), nqw = __popc(__ballot_sync(PCR_FULL, searchable));
        if (lane == 0) {
            atomicAdd(&a.stats[0], (unsigned long long)nqw);
            atomicAdd(&a.stats[1], (unsigned long long)evals);
        }
    }
    if (!active || outcome != kSelDone || skip) return;
    const int cnt = acc.count();
    // (the list is read through acc.ord[j], j a literal: the ranking stays in registers)
    if (MODE == 0) {
        uint32_t *ri = t.idx + (size_t)q * t.kk;
        float *rd = t.dist ? t.dist + (size_t)q * t.kk : nullptr;
        // (frame-local indices; the frame is looked up again rather than kept live through the search)
        const uint32_t base = kQFrames ? a.grids[frame_of(t.qoff, a.n_frames, q)].in_begin : 0u;
#pragma unroll
        for (int j = 0; j < kSelMaxK; j++)
            if (j < t.kk) {
                const bool v = j < cnt;
                const unsigned long long key = v ? acc.key_at(acc.ord[j]) : 0ull;
                ri[j] = v ? key_idx(key) - base : 0xffffffffu;
                if (rd) rd[j] = v ? __fsqrt_rn(key_d2(key)) : INFINITY;  // kdtree.rs:76
            }
        if (t.counts) t.counts[q] = (uint32_t)cnt;
    } else if (MODE == 1 || MODE == 3) {
        // statistical_outlier.rs:28-37: drop the first (self) if there is more than one result, sequential f32 sum in
        // ascending-distance order, divide by the count.  MODE 3 searched kk >= kk_sor neighbours (the top-kk list
        // starts with the top-kk_sor list) and keeps the whole list for normals_from_lists_kernel.
        const int cs = MODE == 3 ? (cnt < t.kk_sor ? cnt : t.kk_sor) : cnt;
        const int first = cs > 1 ? 1 : 0;
        float sum = 0.0f;
#pragma unroll
        for (int j = 0; j < kSelMaxK; j++) {
            const bool v = j < cnt;
            const unsigned long long key = v ? acc.key_at(acc.ord[j]) : 0ull;
            if (j >= first && j < cs) sum = __fadd_rn(sum, __fsqrt_rn(key_d2(key)));
            if (MODE == 3 && j < t.kk) t.lists[(size_t)j * t.list_stride + q] = v ? key_idx(key) : 0xffffffffu;
        }
        const int m = cs - first;
        t.mean_d[out] = m > 0 ? __fdiv_rn(sum, (float)m) : INFINITY;
        if (MODE == 3) t.list_cnt[q] = (uint8_t)cnt;
    } else {
        // estimate.rs:47-109 (normal_from_neighbours with the list read through the ranking)
        float ox = 0.f, oy = 0.f, oz = 1.f;
        if (cnt >= 1) {
            const float count = (float)cnt;
            float cx = 0.f, cy = 0.f, cz = 0.f;
#pragma unroll
            for (int j = 0; j < kSelMaxK; j++)
                if (j < cnt) {
                    const float4 p = __ldg(&t.orig4[key_idx(acc.key_at(acc.ord[j]))]);
                    cx = __fadd_rn(cx, p.x);
                    cy = __fadd_rn(cy, p.y);
                    cz = __fadd_rn(cz, p.z);
                }
            cx = __fdiv_rn(cx, count);
            cy = __fdiv_rn(cy, count);
            cz = __fdiv_rn(cz, count);
            float c00 = 0.f, c01 = 0.f, c02 = 0.f, c11 = 0.f, c12 = 0.f, c22 = 0.f;
#pragma unroll
            for (int j = 0; j < kSelMaxK; j++)
                if (j < cnt) {
                    const float4 p = __ldg(&t.orig4[key_idx(acc.key_at(acc.ord[j]))]);  // second pass: L1 hits
                    const float dx = __fsub_rn(p.x, cx), dy = __fsub_rn(p.y, cy), dz = __fsub_rn(p.z, cz);
                    c00 = __fadd_rn(c00, __fmul_rn(dx, dx));
                    c01 = __fadd_rn(c01, __fmul_rn(dx, dy));
                    c02 = __fadd_rn(c02, __fmul_rn(dx, dz));
                    c11 = __fadd_rn(c11, __fmul_rn(dy, dy));
                    c12 = __fadd_rn(c12, __fmul_rn(dy, dz));
                    c22 = __fadd_rn(c22, __fmul_rn(dz, dz));
                }
            float ex, ey, ez;
            smallest_eigenvector_3x3(c00, c01, c02, c11, c12, c22, ex, ey, ez);
            const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez)));
            if (len > 1e-10f) {
                ex = __fdiv_rn(ex, len);
                ey = __fdiv_rn(ey, len);
                ez = __fdiv_rn(ez, len);
            }
            const float vx = __fsub_rn(t.vx, px), vy = __fsub_rn(t.vy, py), vz = __fsub_rn(t.vz, pz);
            const float dot = __fadd_rn(__fadd_rn(__fmul_rn(ex, vx), __fmul_rn(ey, vy)), __fmul_rn(ez, vz));
            if (dot < 0.0f) {
                ex = -ex; ey = -ey; ez = -ez;
            }
            ox = ex; oy = ey; oz = ez;
        }
        t.nx[out] = ox;
        t.ny[out] = oy;
        t.nz[out] = oz;
    }
}


// ---- level 0 as a cell-tile program (knn_tile.cuh): MODE 1 SOR, 2 normals, 3 SOR + lists kept ------------------------
enum TileOutcome { kTileDone = 0, kTileDefer = 1, kTileContinue = 2, kTileDense = 3, kTileSkip = 4 };

template <int MODE>
__global__ void __launch_bounds__(kTileThreads, 16 / kTileWarps) knn_tile_kernel(LevelArgs a, ThreadArgs t) {
    PCR_GRID_DEP_SYNC();
    extern __shared__ __align__(16) unsigned char tile_raw[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    TileWarp &S = reinterpret_cast<TileWarp *>(tile_raw)[w];
    const uint32_t n2 = a.nq2_dev ? *a.nq2_dev : 0u;  // (the heavy queries lead)
    const uint32_t nq = a.nq_dev ? min(a.nq, *a.nq_dev + n2) : a.nq;
    const uint32_t slot = blockIdx.x * kTileThreads + threadIdx.x;
    if ((slot & ~31u) >= nq) return;  // (warp-uniform: the launch is for a capacity)
    const bool active = slot < nq;
    const uint32_t q = active ? (slot < n2 ? a.qlist2[slot] : (a.qlist ? a.qlist[slot - n2] : a.q_offset + slot)) : 0u;
    const int kk = t.kk;
    if (lane == 0) mbar_init(&S.bar, 1);
    fence_mbar_init();
    __syncwarp();
    float4 qp = make_float4(__int_as_float(0x7fc00000), 0.f, 0.f, 0.f);
    if (active) qp = __ldg(&a.qpts[q]);
    const float px = qp.x, py = qp.y, pz = qp.z;
    const uint32_t out = __float_as_uint(qp.w);
    const int f = active ? frame_of_sorted(a.grids, a.n_frames, q) : 0;
    bool pending = active && px == px;  // a tombstoned point (index_apply_mask_dev) is not a query
    int outcome = pending ? kTileDone : kTileSkip;
    int c0 = 0, c1 = 0, c2 = 0;
    float ff0 = 0.f, ff1 = 0.f, ff2 = 0.f;
    if (pending) {
        const GridDesc g = a.grids[f];
        const uint32_t m = g.pt_end - g.pt_begin;
        if (m <= kBruteFrame || m <= (uint32_t)kk) {  // tiny frame: the follow-up pass scans it whole
            outcome = kTileContinue;
            pending = false;
        } else {
            double f0, f1, f2;
            c0 = cell_coord(g, 0, pick_axis(g.ax[0], px, py, pz), &f0);
            c1 = cell_coord(g, 1, pick_axis(g.ax[1], px, py, pz), &f1);
            c2 = cell_coord(g, 2, pick_axis(g.ax[2], px, py, pz), &f2);
            ff0 = (float)f0;
            ff1 = (float)f1;
            ff2 = (float)f2;
        }
    }
    uint32_t phase = 0, n_eval = 0;
    long long pt0 = clock64(), pt_stage = 0, pt_collect = 0, pt_rank = 0, pt_epi = 0, pt_mark = 0;
    unsigned n_sub = 0, n_max = 0;
#define PCR_PROF_MARK(acc)                \
    if (a.prof) {                         \
        const long long now_ = clock64(); \
        acc += now_ - pt_mark;            \
        pt_mark = now_;                   \
    }
    while (true) {
        const unsigned pm = __ballot_sync(PCR_FULL, pending);
        if (!pm) break;
        n_sub++;
        pt_mark = clock64();
        // ---- the sub-tile: pending queries of the first pending query's layer, up to kTileRowSpan rows from its row and
        // kTileZReach cells from its cell; if that is too much for the buffer its row alone, then its cell alone ---------
        const int leader = __ffs(pm) - 1;
        const int Lf = __shfl_sync(PCR_FULL, f, leader), L0 = __shfl_sync(PCR_FULL, c0, leader), L1 = __shfl_sync(PCR_FULL, c1, leader),
                  L2 = __shfl_sync(PCR_FULL, c2, leader);
        const GridDesc *lg = a.grids + Lf;
        const int d0n = lg->dims[0], d1n = lg->dims[1], d2n = lg->dims[2];
        const uint32_t cell_base = lg->cell_base;
        bool member = false;
        int W = 3;  // staged rows per layer: the members' rows and one on either side
        uint32_t lin = 0, gb = 0, n = 0, inc = 0, Nu = 0;
#pragma unroll 1
        for (int attempt = 0; attempt < 3; attempt++) {
            member = pending && f == Lf && c0 == L0 &&
                     (attempt == 0 ? ((unsigned)(c1 - L1) < (unsigned)kTileRowSpan && abs(c2 - L2) <= kTileZReach)
                                   : (c1 == L1 && (attempt == 1 ? abs(c2 - L2) <= kTileZReach : c2 == L2)));
            const int a1hi = __reduce_max_sync(PCR_FULL, member ? c1 : L1);
            const int zlo = __reduce_min_sync(PCR_FULL, member ? c2 : 0x7fffffff), zhi = __reduce_max_sync(PCR_FULL, member ? c2 : -1);
            W = a1hi - L1 + 3;
            // lanes 0 .. 3 W - 1: rows (L0 - 1 .. L0 + 1) x (L1 - 1 .. a1hi + 1), cells [zlo - 1, zhi + 1]
            const int a0 = L0 + lane / W - 1, a1 = L1 - 1 + lane % W;
            const bool rvalid = lane < 3 * W && a0 >= 0 && a0 < d0n && a1 >= 0 && a1 < d1n;
            lin = rvalid ? cell_base + ((uint32_t)a0 * (uint32_t)d1n + (uint32_t)a1) * (uint32_t)d2n : 0u;
            const int zb = max(zlo - 1, 0), ze = min(zhi + 1, d2n - 1);
            uint32_t ge = 0;
            gb = 0;
            if (rvalid) {
                gb = __ldg(&a.cell_start[lin + (uint32_t)zb]);
                ge = __ldg(&a.cell_start[lin + (uint32_t)ze + 1u]);
            }
            n = ge - gb;
            inc = n;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t up = __shfl_up_sync(PCR_FULL, inc, d);
                if (lane >= d) inc += up;
            }
            Nu = __shfl_sync(PCR_FULL, inc, 31);
            if (Nu <= (uint32_t)kTileCap) break;
        }
        if (Nu > (uint32_t)kTileCap) {  // (warp-uniform) a dense object: not a tile's job
            if (member) {
                outcome = kTileDense;
                pending = false;
            }
            continue;
        }
        __syncwarp();  // every lane is done with the previous sub-tile
        if (lane < 3 * W) S.row[lane] = make_int4((int)lin, (int)gb, (int)(inc - n), (int)n);
        fence_proxy_async();  // generic reads / writes of the staging buffer before the async proxy overwrites it
        __syncwarp();
        if (lane == 0) mbar_expect_tx(&S.bar, Nu * 16u);
        __syncwarp();
        if (n) bulk_g2s(&S.stage[inc - n], a.pts + gb, n * 16u, &S.bar);
        // while the copies fly: every member's window in each staged row
        uint32_t N = 0;
        if (member) {
            const int z0 = max(c2 - 1, 0), z1 = min(c2 + 1, d2n - 1);
#pragma unroll
            for (int r = 0; r < 9; r++) {
                const int4 R = S.row[(r / 3) * W + (c1 - L1) + r % 3];
                uint32_t b = 0, e = 0;
                if (R.w) {
                    const uint32_t wb = __ldg(&a.cell_start[(uint32_t)R.x + (uint32_t)z0]), we = __ldg(&a.cell_start[(uint32_t)R.x + (uint32_t)z1 + 1u]);
                    b = (uint32_t)R.z + (wb - (uint32_t)R.y);
                    e = (uint32_t)R.z + (we - (uint32_t)R.y);
                }
                S.seg[r][lane] = b | (e << 16);
                N += e - b;
            }
        }
        mbar_wait(&S.bar, phase);
        phase ^= 1u;
        PCR_PROF_MARK(pt_stage)
        n_max = max(n_max, __reduce_max_sync(PCR_FULL, N));

        const float h2 = (float)(lg->h * lg->h);
        // ---- the 27 cells: threshold, collection, ranking --------------------------------------------------------
        bool live = member;
        int cnt = 0;
        if (live) {
            cnt = tile_collect(S, lane, kk, N, px, py, pz, h2, n_eval);
            if (cnt > kTileSlots || cnt < 0) {  // more than the slots hold below the threshold: exact ties
                outcome = kTileDense;
                live = false;
            }
        }
        if (!live) cnt = 0;
        PCR_PROF_MARK(pt_collect)
        const int m = cnt < kk ? cnt : kk;
        {
            uint32_t k[kTileSlots];
            tile_rank(S, lane, cnt, k);
            if (live) tile_fix(S, lane, cnt, m, k, px, py, pz);
            // the ranked list back into the slots: the k-th and the epilogue read it from there (a select chain over k[]
            // makes the compiler index a local-memory copy of it)
#pragma unroll
            for (int j = 0; j < kTileMaxK; j++)
                if (j < m) S.slot[j][lane] = k[j];
        }
        bool fin = false;
        if (live) {
            // ---- is the list final?  (the ring rule of every search in this library, shell 1) -----------------------
            unsigned long long kth_key = PCR_EMPTY_KEY;
            if (m == kk) kth_key = tile_full_key(S, S.slot[kk - 1][lane], px, py, pz);
            const GridDesc g = *lg;
            double f0, f1, f2, bound2;
            cell_coord(g, 0, pick_axis(g.ax[0], px, py, pz), &f0);
            cell_coord(g, 1, pick_axis(g.ax[1], px, py, pz), &f1);
            cell_coord(g, 2, pick_axis(g.ax[2], px, py, pz), &f2);
            if (!ring_bound2(g, c0, c1, c2, f0, f1, f2, 1, bound2)) {
                fin = true;  // the whole grid has been scanned
            } else if (kth_key != PCR_EMPTY_KEY && (double)key_d2(kth_key) < bound2 * (1.0 - 1e-6)) {
                fin = true;
            } else if (!a.last_level && (1 >= a.max_rings || m * 4 < kk)) {
                outcome = kTileDefer;  // same rule as every level-0 search: a sparse neighbourhood belongs to the coarser grid
            } else {
                // a second shell: rows read from global memory, trimmed to the k-th distance.  One thread doing that costs
                // 20 K cycles of dependent loads (measured, in-tile variant of round 2) and stalls its 31 neighbours: the
                // follow-up pass gives such a query a whole warp.  The cell size keeps them rare (occupancy_target).
                outcome = kTileContinue;
            }
        }
        PCR_PROF_MARK(pt_rank)
        if (fin) {
            // ---- epilogue: the list is slot[0 .. m), ascending by (d^2, index) -------------------------------------
            if (MODE == 1 || MODE == 3) {
                // statistical_outlier.rs:28-37: drop the first (self) if there is more than one result, sequential f32 sum
                // in ascending-distance order, divide by the count.  MODE 3 searched kk >= kk_sor neighbours and keeps the list.
                const int cs = MODE == 3 ? (m < t.kk_sor ? m : t.kk_sor) : m;
                const int first = cs > 1 ? 1 : 0;
                float sum = 0.0f;
#pragma unroll 4
                for (int j = 0; j < kk; j++) {
                    float4 p = make_float4(0.f, 0.f, 0.f, __uint_as_float(0xffffffffu));
                    if (j < m) p = S.stage[S.slot[j][lane] & kTilePos];
                    if (j >= first && j < cs) sum = __fadd_rn(sum, __fsqrt_rn(dist2_exact(px, py, pz, p.x, p.y, p.z)));  // kdtree.rs:76
                    if (MODE == 3) t.lists[(size_t)j * t.list_stride + q] = __float_as_uint(p.w);
                }
                const int mm = cs - first;
                t.mean_d[out] = mm > 0 ? __fdiv_rn(sum, (float)mm) : INFINITY;
                if (MODE == 3) t.list_cnt[q] = (uint8_t)m;
            } else {
                // estimate.rs:47-109; the neighbours' coordinates are the staged points themselves
                float ox, oy, oz;
                normal_from_neighbours(
                    m,
                    [&](int j, int c) {
                        const float4 p = S.stage[S.slot[j][lane] & kTilePos];
                        return c == 0 ? p.x : (c == 1 ? p.y : p.z);
                    },
                    px, py, pz, t.vx, t.vy, t.vz, ox, oy, oz);
                t.nx[out] = ox;
                t.ny[out] = oy;
                t.nz[out] = oz;
            }
        }
        PCR_PROF_MARK(pt_epi)
        pending = pending && !member;
    }
    if (a.prof && lane == 0) {
        unsigned long long *pr = a.prof + (size_t)(slot >> 5) * 8;
        pr[0] = (unsigned long long)(clock64() - pt0);
        pr[1] = (unsigned long long)pt_stage;
        pr[2] = (unsigned long long)pt_collect;
        pr[3] = (unsigned long long)pt_rank;
        pr[4] = 0ull;
        pr[5] = (unsigned long long)pt_epi;
        pr[6] = ((unsigned long long)n_sub << 32) | n_max;
        pr[7] = q;
    }
#undef PCR_PROF_MARK
    push_list(outcome == kTileDefer, a.defer_list, a.defer_count, q, lane);
    push_list(outcome == kTileContinue, a.cont_list, a.cont_count, q, lane);
    push_list(outcome == kTileDense, a.ovf_list, a.ovf_count, q, lane);
    if (a.stats) {
        const unsigned evals = __reduce_add_sync(PCR_FULL, n_eval), nqw = __popc(__ballot_sync(PCR_FULL, outcome != kTileSkip && outcome != kTileDense));
        if (lane == 0) {
            atomicAdd(&a.stats[0], (unsigned long long)nqw);
            atomicAdd(&a.stats[1], (unsigned long long)evals);
        }
    }
}

enum KnnImpl { kImplInsert = 0, kImplSelect = 1, kImplWarp = 2 };
inline int knn_impl() {  // A/B hook: PCR_KNN_IMPL = insert (round-1 insertion kernels) | select (thread per query, selection) | warp
    static const int impl = [] {
        const char *e = getenv("PCR_KNN_IMPL");
        if (e && !strcmp(e, "insert")) return (int)kImplInsert;
        if (e && !strcmp(e, "warp")) return (int)kImplWarp;
        return (int)kImplSelect;
    }();
    return impl;
}
inline bool use_select(int kk) { return kk <= kSelMaxK && knn_impl() == kImplSelect; }
// level 0 with a warp per query (warp_select_cube front-end), kQPWS consecutive queries per warp
inline bool use_warp(int kk) { return kk > 0 && kk <= 32 && knn_impl() == kImplWarp; }
// shells the thread-per-query pass walks before it hands a query to the follow-up pass (tuning hook PCR_FIRST_SHELLS)
inline int first_shells() {
    static const int n = [] {
        const char *e = getenv("PCR_FIRST_SHELLS");
        const int v = e ? atoi(e) : 2;
        return v < 1 ? 1 : (v > kLevelRings ? kLevelRings : v);
    }();
    return n;
}

// level 0 as a cell-tile program (A/B hook: PCR_KNN_TILE=0 keeps the thread-per-query selection kernel for everything)
inline bool use_tile(int kk) {
    static const bool on = [] {
        const char *e = getenv("PCR_KNN_TILE");
        return !(e && !strcmp(e, "0"));
    }();
    return on && kk > 0 && kk <= kTileMaxK;
}

template <int MODE, bool kQFrames>
int launch_sel_kernel(Ctx *ctx, const LevelArgs &a, const ThreadArgs &t) {
    const unsigned blocks = (a.nq + kTQThreads - 1) / kTQThreads;
    if constexpr (MODE != 0) {
        if (use_tile(t.kk) && !a.no_tile && a.ovf_list && a.cont_list) {
            // (tuning hook PCR_TILE_PAD_SMEM: extra bytes per block = fewer resident tile blocks per SM, room for the other classes)
            static const size_t pad = getenv("PCR_TILE_PAD_SMEM") ? (size_t)atoi(getenv("PCR_TILE_PAD_SMEM")) : 0;
            const size_t smem = sizeof(TileWarp) * kTileWarps + pad;
            static bool attr_set = false;  // (one device per process)
            if (!attr_set) {
                PCR_TRY(set_smem(ctx, knn_tile_kernel<MODE>, smem));
                attr_set = true;
            }
            static const bool prof = getenv("PCR_TILE_PROF") != nullptr;  // debug: per-warp cycle counters, ten slowest warps printed
            if (prof) {
                LevelArgs ap = a;
                const size_t nw = (a.nq + 31) / 32;
                unsigned long long *d = nullptr;
                PCR_CUDA(ctx, cudaMalloc(&d, nw * 64));
                PCR_CUDA(ctx, cudaMemset(d, 0, nw * 64));
                ap.prof = d;
                knn_tile_kernel<MODE><<<(a.nq + kTileThreads - 1) / kTileThreads, kTileThreads, smem, ctx->stream>>>(ap, t);
                PCR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                std::vector<unsigned long long> h(nw * 8);
                PCR_CUDA(ctx, cudaMemcpy(h.data(), d, nw * 64, cudaMemcpyDeviceToHost));
                cudaFree(d);
                std::vector<size_t> order(nw);
                for (size_t i = 0; i < nw; i++) order[i] = i;
                std::sort(order.begin(), order.end(), [&](size_t x, size_t y) { return h[x * 8] > h[y * 8]; });
                unsigned long long tot[6] = {0, 0, 0, 0, 0, 0}, subs = 0;
                for (size_t i = 0; i < nw; i++) {
                    for (int j = 0; j < 6; j++) tot[j] += h[i * 8 + j];
                    subs += h[i * 8 + 6] >> 32;
                }
                fprintf(stderr, "[pcr] tile profile: %zu warps, %.2f sub-tiles / warp; mean cycles total %.0f = stage %.0f + collect %.0f + rank %.0f + shell2 %.0f + epilogue %.0f\n",
                        nw, (double)subs / nw, (double)tot[0] / nw, (double)tot[1] / nw, (double)tot[2] / nw, (double)tot[3] / nw, (double)tot[4] / nw,
                        (double)tot[5] / nw);
                for (size_t r = 0; r < 10 && r < nw; r++) {
                    const unsigned long long *e = &h[order[r] * 8];
                    fprintf(stderr, "[pcr]   warp %zu (q %llu): total %llu = stage %llu + collect %llu + rank %llu + shell2 %llu + epilogue %llu; %llu sub-tiles, max N %llu\n",
                            order[r], e[7], e[0], e[1], e[2], e[3], e[4], e[5], e[6] >> 32, e[6] & 0xffffffffull);
                }
                return PCR_OK;
            }
            PCR_CUDA(ctx, launch_chained(knn_tile_kernel<MODE>, dim3((a.nq + kTileThreads - 1) / kTileThreads), dim3(kTileThreads), smem, ctx->stream, a, t));
            ctx->launches++;
            return PCR_OK;  // (run_levels launches a warp-per-query pass over what the tiles handed back)
        }
    }
    knn_sel_kernel<MODE, kQFrames><<<blocks, kTQThreads, 0, ctx->stream>>>(a, t);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

// value for points that are not in the index: non-finite points have no neighbours -> (0,0,1)
// (estimate.rs:49-51); points removed by a mask (batch pipeline) -> 0.
__global__ void fill_unindexed_normals_kernel(const float4 *__restrict__ orig4, const uint8_t *__restrict__ mask, size_t n,
                                              float *__restrict__ nx, float *__restrict__ ny, float *__restrict__ nz) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 p = orig4[i];
    bool removed = mask && !mask[i];
    if (removed) {
        nx[i] = 0.f; ny[i] = 0.f; nz[i] = 0.f;
    } else if (!finite3(p.x, p.y, p.z)) {
        nx[i] = 0.f; ny[i] = 0.f; nz[i] = 1.f;
    }
}

__global__ void fill_f32_kernel(float *__restrict__ p, size_t n, float v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---- radius search (thread per query) ------------------------------------------------------------
// d^2 <= r*r with r*r rounded in f32 (kdtree.rs:114,127).  Cells are taken from the box
// [q - r', q + r'] with r' = sqrt(r2) * (1 + 1e-6): a point that passes the f32 test is at most a
// few ulp further than sqrt(r2) on any axis.
// kFrames (batch): query i belongs to frame frame_of(frame_in_off, n_frames, i) and is searched only in the grid of that frame
// -- the input points of a multi-frame index themselves (frame_in_off = its input offsets), or the external queries of a
// batch (frame_in_off = the query offsets; the filled indices are then frame-local).  The single-frame calls leave
// frame_in_off / n_frames unset.
template <bool kFill, bool kFrames = false>
__global__ void __launch_bounds__(256) radius_kernel(const GridDesc *__restrict__ grids,
                                                     const uint32_t *__restrict__ cell_start,
                                                     const float4 *__restrict__ sorted, const float *__restrict__ qx,
                                                     const float *__restrict__ qy, const float *__restrict__ qz, size_t nq,
                                                     float radius, uint32_t *__restrict__ counts,
                                                     const uint64_t *__restrict__ offsets, uint32_t *__restrict__ out_idx,
                                                     const uint32_t *__restrict__ frame_in_off = nullptr, int n_frames = 1) {
    size_t qi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    const GridDesc g = grids[kFrames ? frame_of(frame_in_off, n_frames, (uint32_t)qi) : 0];
    float x = qx[qi], y = qy[qi], z = qz[qi];
    uint32_t cnt = 0;
    uint32_t *dst = kFill ? out_idx + offsets[qi] : nullptr;
    // kdtree.rs:106-112
    if (g.pt_end > g.pt_begin && radius > 0.0f && isfinite(radius) && finite3(x, y, z)) {
        const float r2 = __fmul_rn(radius, radius);
        const double rr = sqrt((double)r2) * (1.0 + 1e-6) + 1e-300;
        int lo[3], hi[3];
        bool any = true;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            double v = (double)pick_axis(g.ax[j], x, y, z);
            double tl = floor((v - rr - g.o[j]) * g.inv_h), th = floor((v + rr - g.o[j]) * g.inv_h);
            if (th < 0.0 || tl > (double)(g.dims[j] - 1)) any = false;
            lo[j] = (int)fmin(fmax(tl, 0.0), (double)(g.dims[j] - 1));
            hi[j] = (int)fmin(fmax(th, 0.0), (double)(g.dims[j] - 1));
        }
        if (any) {
            for (int a0 = lo[0]; a0 <= hi[0]; a0++)
                for (int a1 = lo[1]; a1 <= hi[1]; a1++) {
                    uint32_t lin = cell_linear(g, a0, a1, lo[2]);
                    uint32_t b = __ldg(&cell_start[lin]), e = __ldg(&cell_start[lin + (uint32_t)(hi[2] - lo[2]) + 1u]);
                    for (uint32_t i = b; i < e; i++) {
                        float4 p = __ldg(&sorted[i]);
                        if (dist2_exact(x, y, z, p.x, p.y, p.z) <= r2) {
                            if (kFill) dst[cnt] = __float_as_uint(p.w) - (kFrames ? g.in_begin : 0u);
                            cnt++;
                        }
                    }
                }
        }
    }
    if (!kFill) {
        counts[qi] = cnt;
    } else if (cnt > 1) {
        // ascending index order (kdtree.rs:132): in-place heapsort of this query's slice
        for (uint32_t start = cnt / 2; start-- > 0;) {
            uint32_t root = start;
            for (;;) {
                uint32_t c = 2 * root + 1;
                if (c >= cnt) break;
                if (c + 1 < cnt && dst[c] < dst[c + 1]) c++;
                if (dst[root] >= dst[c]) break;
                uint32_t tmp = dst[root]; dst[root] = dst[c]; dst[c] = tmp;
                root = c;
            }
        }
        for (uint32_t end = cnt - 1; end > 0; end--) {
            uint32_t tmp = dst[0]; dst[0] = dst[end]; dst[end] = tmp;
            uint32_t root = 0;
            for (;;) {
                uint32_t c = 2 * root + 1;
                if (c >= end) break;
                if (c + 1 < end && dst[c] < dst[c + 1]) c++;
                if (dst[root] >= dst[c]) break;
                uint32_t t2 = dst[root]; dst[root] = dst[c]; dst[c] = t2;
                root = c;
            }
        }
    }
}

template <class Kern>
int set_smem(Ctx *ctx, Kern kern, size_t bytes) {
    if (bytes > 48 * 1024) {
        if (bytes > 200 * 1024) return fail(ctx, PCR_ERR_UNSUPPORTED, "k too large for shared memory");
        PCR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    }
    return PCR_OK;
}

// Runs `launch(args, qpw)` level by level until no query is left deferred.  Reading the deferred
// count costs one small D2H + sync per level that is actually needed (clouds without far outliers
// finish on level 0 and pay exactly one).
// ---- classification of the level-0 queries ---------------------------------------------------------------------
// A frame mixes three kinds of query, and one launch over all of them is as slow as its slowest kind (ncu, round 2:
// the warps inside a dense object ran five times longer than the rest and WERE the kernel's duration; the ~2 % of
// isolated outliers cost a grid level, a launch and a round trip after it).  One cheap kernel therefore sorts the
// queries by the number of points in their 27 cells into three lists, and the three kinds run AT THE SAME TIME:
//   sparse  (fewer than kk / 4 candidates: the first shell would end with "deferred")   -> the next-coarser level
//           is built and searched on a side stream while level 0 is still running,
//   dense   (more than kSelHistMaxN candidates: a volume, not a surface)                -> own launch, side stream,
//   normal  everything else                                                             -> the main launch.
// The lists keep the cell-sorted order inside every block of 256 queries (one atomic per block and class), so
// neighbouring threads still hold neighbouring queries.  Every path is exact; the classes only decide where a query runs.
constexpr int kClsThreads = 256;
struct ClassArgs {
    uint32_t *list[4];       // normal, dense, sparse, heavy normal (tile kernel: the queries with many candidates start first)
    uint32_t *count[4];
    const float *qx, *qy, *qz;  // external queries (nullptr: the indexed points themselves)
    int kk;
    // tile kernel in use: a query with fewer than kk candidates in its 27 cells goes straight to the follow-up pass (warp
    // per query, all shells): inside a tile it is a sub-tile of its own whose second shell has no threshold to trim it
    uint32_t *thin;
    uint32_t *thin_count;
    uint32_t dense_n;  // more candidates than this in the 27 cells: the dense class
    uint32_t heavy_n;  // more than this: heavy normal (0: no such class)
};

// kQFrames: external queries of a batch index, qoff their device offsets (frame f searched in grid f).  (qoff is a parameter
// of its own: the kernel copies ClassArgs to local memory, and a longer struct would change the single-frame SASS.)
template <bool kQFrames = false>
__global__ void __launch_bounds__(kClsThreads) classify_kernel(LevelArgs a, ClassArgs c, const uint32_t *__restrict__ qoff) {
    PCR_GRID_DEP_SYNC();
    const uint32_t slot = blockIdx.x * kClsThreads + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t q = a.q_offset + slot;
    int cls = 7;  // no query in this slot
    if (slot < a.nq) {
        float px, py, pz;
        int f = 0;
        bool searchable;
        if (c.qx) {
            px = __ldg(&c.qx[q]);
            py = __ldg(&c.qy[q]);
            pz = __ldg(&c.qz[q]);
            searchable = finite3(px, py, pz);
            if constexpr (kQFrames) f = frame_of(qoff, a.n_frames, q);
        } else {
            const float4 p = __ldg(&a.qpts[q]);
            px = p.x; py = p.y; pz = p.z;
            f = frame_of_sorted(a.grids, a.n_frames, q);
            searchable = px == px;
        }
        cls = 0;  // (queries that are not searched still produce their empty result in the main launch)
        if (searchable) {
            const GridDesc *gp = a.grids + f;
            const uint32_t m = gp->pt_end - gp->pt_begin;
            if (m > kBruteFrame && m > (uint32_t)c.kk) {
                // (fewer than kk in the cube: the search needs more shells whatever happens -- a warp's job, see thin)
                // and so does a query with at most one neighbour in the three cells of its own row: an off-surface point, a
                // sub-tile of its own wherever it sits in the order)
                uint32_t n_row = 0;
                const uint32_t n27 = count_27_cells(gp, a.cell_start, px, py, pz, &n_row);
                cls = n27 * 4u < (uint32_t)c.kk ? 2 : (n27 > c.dense_n ? 1 : (c.thin && (n27 < (uint32_t)c.kk || n_row <= 2u) ? 4 : 0));
                if (cls == 0 && c.heavy_n && n27 > c.heavy_n) cls = 3;
            }
        }
    }
    __shared__ uint32_t s_warp[4][kClsThreads / 32];
    __shared__ uint32_t s_base[4];
    uint32_t my_rank = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const unsigned mask = __ballot_sync(PCR_FULL, cls == k);
        if (lane == 0) s_warp[k][w] = __popc(mask);
        if (cls == k) my_rank = __popc(mask & ((1u << lane) - 1u));
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        uint32_t tot = 0;
        for (int i = 0; i < kClsThreads / 32; i++) tot += s_warp[threadIdx.x][i];
        s_base[threadIdx.x] = tot ? atomicAdd(c.count[threadIdx.x], tot) : 0u;
    }
    __syncthreads();
    if (cls < 4) {
        uint32_t off = s_base[cls] + my_rank;
        for (int i = 0; i < w; i++) off += s_warp[cls][i];
        c.list[cls][off] = q;
    }
    push_list(cls == 4, c.thin, c.thin_count, q, lane);
}

struct StreamSwap {  // the library's helpers launch on ctx->stream: run a few of them on a side stream
    Ctx *c;
    cudaStream_t saved;
    StreamSwap(Ctx *ctx, cudaStream_t s) : c(ctx), saved(ctx->stream) { c->stream = s; }
    ~StreamSwap() { c->stream = saved; }
};

int ensure_side_streams(Ctx *ctx) {
    if (ctx->side[0]) return PCR_OK;
    for (int i = 0; i < 2; i++) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);  // (lo = the numerically greatest = the least urgent)
        static const bool flat = getenv("PCR_SIDE_FIRST") != nullptr;
        PCR_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->side[i], cudaStreamNonBlocking, flat ? hi : lo));
        PCR_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming));
    }
    PCR_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    return PCR_OK;
}

template <class Launch>
int run_levels(Index *ix, uint32_t nq, int tag0, Launch launch, const uint32_t *init_list = nullptr, const uint32_t *nq_dev = nullptr,
               int sel_kk = 0 /* > 0: level 0 is a thread-per-query launch for this many neighbours */,
               uint32_t q_offset = 0 /* level 0 takes the queries q_offset .. q_offset + nq (a rank's shard) */,
               const float *eqx = nullptr, const float *eqy = nullptr, const float *eqz = nullptr /* external queries (device) */,
               bool tile_ok = false /* level 0 may run as the cell-tile kernel (self-queries with a fused consumer) */,
               const uint32_t *eq_off = nullptr /* external queries of a batch index: device query offsets [n_frames + 1] */) {
    // init_list: level 0 runs over these nq query ids only (warp kernels) instead of over all queries
    // nq_dev:    the length of init_list is still on the device; nq is the capacity level 0 is launched for
    Ctx *ctx = ix->ctx;
    if (nq == 0) return PCR_OK;
    // Selection kernels (two_pass): level 0 = classification, then three concurrent launches (see classify_kernel); the
    // thread-per-query launches walk first_shells() shells and queue what needs more for a warp-per-query follow-up.
    const bool two_pass = !init_list && sel_kk > 0 && use_select(sel_kk);
    static const bool no_split = getenv("PCR_NO_CLASS_SPLIT") != nullptr;  // A/B hook: one launch over all queries
    static const bool dense_warp = getenv("PCR_DENSE_THREAD") == nullptr;   // A/B hook: the dense class thread per query
    static const bool dense_fine = getenv("PCR_DENSE_NO_FINE") == nullptr;  // A/B hook: the dense class on level 0, warp per query
    static const int dense_qpw = getenv("PCR_DENSE_QPW1") ? kQPWL : kQPWS;  // A/B hook: one query per warp and grid step (85 vs 97 us alone on
                                                                            // the 122 K frame, but 14.9 vs 12.5 ms on the 8 M batch)
    const bool split = two_pass && !no_split;
    PCR_TRY(ensure(ctx, ctx->b_list, (size_t)nq * (two_pass ? 8 : 2) * sizeof(uint32_t) + 256));
    // counters: [0], [1] deferred counts of even / odd levels, [2] follow-up count, [3..5] normal / dense / sparse counts
    uint32_t *counters = (uint32_t *)ctx->b_list.p;
    uint32_t *lists[2] = {counters + 64, counters + 64 + nq};
    uint32_t *cont = counters + 64 + 2 * (size_t)nq;
    uint32_t *cls_list[3] = {cont + nq, cont + 2 * (size_t)nq, cont + 3 * (size_t)nq};
    uint32_t *ovf = cont + 4 * (size_t)nq;    // counters[6]: queries the tile kernel hands back
    uint32_t *heavy = cont + 5 * (size_t)nq;  // counters[7]: normal queries with many candidates (they lead the tile launch)
    Index *cur = ix;
    const uint32_t *qlist = init_list;
    uint32_t n_cur = nq;
    bool join_pending = false;  // the side streams of the class split have not been joined yet
    bool pre_level1 = false;  // the sparse queries have already been searched on level 1 (their own deferrals sit in lists[1])
    static const bool dbg = getenv("PCR_DEBUG") != nullptr;
    for (int level = 0;; level++) {
        const bool last = level == kMaxLevels - 1;
        uint32_t *cnt = counters + (level & 1);
        if (level == 0) PCR_CUDA(ctx, cudaMemsetAsync(counters, 0, 16 * sizeof(uint32_t), ctx->stream));
        else if (!(level == 1 && pre_level1)) PCR_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(uint32_t), ctx->stream));
        LevelArgs a;
        a.grids = cur->grids;
        a.n_frames = cur->n_frames;
        a.cell_start = cur->cell_start;
        a.pts = cur->sorted;
        a.qpts = ix->sorted;
        a.qlist = qlist;
        a.qlist2 = nullptr;
        a.nq2_dev = nullptr;
        a.q_offset = (level == 0 && !init_list) ? q_offset : 0u;
        a.nq = n_cur;
        a.nq_dev = level == 0 ? nq_dev : nullptr;
        a.defer_list = lists[level & 1];
        a.defer_count = cnt;
        a.max_rings = last ? kMaxRings : kLevelRings;
        a.last_level = last ? 1 : 0;
        const bool first_of_two = two_pass && level == 0;
        a.follow_up = 0;
        a.stats = (ctx->timing && first_of_two) ? ctx->d_knn_stats : nullptr;
        a.first_only = first_of_two ? first_shells() : 0;
        a.cont_list = first_of_two ? cont : nullptr;
        a.cont_count = first_of_two ? counters + 2 : nullptr;
        a.ovf_list = first_of_two && tile_ok && use_tile(sel_kk) ? ovf : nullptr;
        a.ovf_count = counters + 6;
        a.no_tile = 0;
        a.prof = nullptr;
        // what the tile kernel hands back (exact ties, a dense cell in a non-split launch): a warp per query
        auto launch_ovf = [&]() -> int {
            LevelArgs o = a;
            o.qlist = ovf;
            o.q_offset = 0;
            o.nq_dev = counters + 6;
            o.no_tile = 1;
            o.stats = nullptr;
            TimeScope ts(ctx, kTagKnnDeferred);
            return launch(o, kQPWS);
        };
        if (first_of_two && split) {
            PCR_TRY(ensure_side_streams(ctx));
            ClassArgs ca;
            for (int k = 0; k < 3; k++) {
                ca.list[k] = cls_list[k];
                ca.count[k] = counters + 3 + k;
            }
            ca.list[3] = heavy;
            ca.count[3] = counters + 7;
            ca.qx = eqx; ca.qy = eqy; ca.qz = eqz;
            ca.kk = sel_kk;
            ca.thin = a.ovf_list ? cont : nullptr;
            ca.thin_count = counters + 2;
            // (a tile's warp is as slow as its heaviest query: with tiles the dense class starts lower)
            static const uint32_t tile_dense_n = getenv("PCR_TILE_DENSE_N") ? (uint32_t)atoi(getenv("PCR_TILE_DENSE_N")) : kTileDenseN;
            ca.dense_n = a.ovf_list ? tile_dense_n : kSelHistMaxN;
            // (heavy-first order measured WORSE, 123 -> 144 us: pulling the many-candidate cells out of the cell order leaves
            // both lists with gaps, i.e. more sub-tiles per warp; PCR_TILE_HEAVY_N re-enables the split for experiments)
            static const uint32_t heavy_n = getenv("PCR_TILE_HEAVY_N") ? (uint32_t)atoi(getenv("PCR_TILE_HEAVY_N")) : 0u;
            ca.heavy_n = a.ovf_list ? heavy_n : 0u;
            {
                TimeScope ts(ctx, kTagKnnDeferred);
                PCR_CUDA(ctx, launch_chained(eq_off ? classify_kernel<true> : classify_kernel<false>, dim3((n_cur + kClsThreads - 1) / kClsThreads),
                                             dim3(kClsThreads), 0, ctx->stream, a, ca, eq_off));
                ctx->launches++;
            }
            PCR_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
            for (int i = 0; i < 2; i++) PCR_CUDA(ctx, cudaStreamWaitEvent(ctx->side[i], ctx->ev_fork, 0));
            // The main launch goes first and the side streams have the lowest priority: the tile kernel's blocks take every
            // SM's shared memory (15 x 14 KB), so whichever kernel starts first runs alone -- and the tile kernel is the one
            // with the long tail (its SMs are busy half of its duration) that the two small classes can fill.
            auto launch_main = [&]() -> int {
                LevelArgs m = a;
                m.qlist = cls_list[0];
                m.q_offset = 0;
                m.nq_dev = counters + 3;
                if (a.ovf_list) {
                    m.qlist2 = heavy;
                    m.nq2_dev = counters + 7;
                }
                {
                    TimeScope ts(ctx, tag0);
                    PCR_TRY(launch(m, kQPW0));
                }
                if (a.ovf_list) PCR_TRY(launch_ovf());
                return PCR_OK;
            };
            static const bool side_first = getenv("PCR_SIDE_FIRST") != nullptr;  // A/B hook: the round-2a order
            PCR_MARK("levels: classes queued");
            if (!side_first) PCR_TRY(launch_main());
            PCR_MARK("levels: main launch queued");
            // side 0: the sparse queries on the next-coarser level (built here, behind the fork, while level 0 runs)
            if (!last) {
                StreamSwap sw(ctx, ctx->side[0]);
                TimeScope ts(ctx, kTagKnnDeferred);
                Index *next = nullptr;
                PCR_TRY(index_coarser_level(cur, &next));
                PCR_MARK("levels: coarser level queued");
                LevelArgs s1 = a;
                s1.grids = next->grids;
                s1.cell_start = next->cell_start;
                s1.pts = next->sorted;
                s1.qlist = cls_list[2];
                s1.q_offset = 0;
                s1.nq_dev = counters + 5;
                s1.defer_list = lists[1];
                s1.defer_count = counters + 1;
                const bool last1 = kMaxLevels - 1 == 1;
                s1.max_rings = last1 ? kMaxRings : kLevelRings;
                s1.last_level = last1 ? 1 : 0;
                s1.first_only = 0;
                s1.cont_list = nullptr;
                s1.cont_count = nullptr;
                s1.stats = nullptr;
                // (the selection front-end is NOT used here: measured 58 -> 137 us -- the 27 coarse cells of a point above the
                // ground hold thousands of candidates, and the insertion walk trims most rows by the k-th distance instead)
                PCR_TRY(launch(s1, kQPWL));
                pre_level1 = true;
            }
            if (pre_level1) PCR_CUDA(ctx, cudaEventRecord(ctx->ev_join[0], ctx->side[0]));
            {  // side 1: the dense queries
                StreamSwap sw(ctx, ctx->side[1]);
                LevelArgs d = a;
                d.qlist = cls_list[1];
                d.q_offset = 0;
                d.nq_dev = counters + 4;
                d.no_tile = 1;
                TimeScope ts(ctx, kTagKnnDeferred);
                if (a.ovf_list && dense_fine) {
                    // Dense means "too many points per cell", so these queries get smaller cells: the FINER level (cell / 2,
                    // built here on this side stream), same warp-per-query kernel -- an eighth of the candidates.  A dense query
                    // on level 0 costs 15 ns of the whole GPU (1 900 candidates, two passes) against 0.4 ns for a tile query:
                    // 2.9 of the 8 M batch's 11.7 ms for 2.4 % of its queries.  (Measured and dropped: the fine level under the
                    // TILE kernel -- 165 us for 11 K queries: 240 candidates per thread is a long serial chain, and only 350
                    // warps carry it; its leftovers then need lists of their own for the level-0 warp kernels.)
                    Index *fine = nullptr;
                    PCR_MARK("levels: sparse class queued");
                    PCR_TRY(index_finer_level(cur, &fine));
                    PCR_MARK("levels: finer level queued");
                    d.grids = fine->grids;
                    d.cell_start = fine->cell_start;
                    d.pts = fine->sorted;
                    d.stats = nullptr;
                    PCR_TRY(launch(d, dense_qpw));
                } else {
                    // (a warp per query: a dense query reads thousands of candidates, 32 at a time instead of one thread's
                    // serial walk -- the thread-per-query launch of this class took 0.34 ms and bounded the step)
                    PCR_TRY(launch(d, dense_warp ? dense_qpw : kQPW0));
                }
                PCR_CUDA(ctx, cudaEventRecord(ctx->ev_join[1], ctx->stream));
            }
            if (side_first) PCR_TRY(launch_main());
            join_pending = true;  // (after the follow-up pass: it only needs the main launch's list, and runs beside the side streams' tails)
        } else {
            {
                TimeScope ts(ctx, level == 0 ? tag0 : kTagKnnDeferred);
                PCR_TRY(launch(a, level == 0 && !init_list ? (use_warp(sel_kk) ? kQPWS : kQPW0) : kQPWL));
            }
            if (a.ovf_list) PCR_TRY(launch_ovf());
        }
        if (first_of_two) {
            // the queries that need more than the first pass's shells: warp per query over the shells of the same level
            // (they are few and far apart in the list: a thread-per-query launch would leave most of the GPU idle)
            LevelArgs b = a;
            b.first_only = 0;
            b.cont_list = nullptr;
            b.cont_count = nullptr;
            b.stats = nullptr;
            b.qlist = cont;
            b.q_offset = 0;
            b.nq_dev = counters + 2;
            b.follow_up = 1;
            TimeScope ts(ctx, kTagKnnDeferred);
            PCR_TRY(launch(b, kQPWL));
        }
        if (join_pending) {
            for (int i = pre_level1 ? 0 : 1; i < 2; i++) PCR_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join[i], 0));
            join_pending = false;
        }
        if (last) break;
        // (see Ctx::spec_request: a frame stream does not wait for counts that were zero on the previous frame)
        static const bool no_nowait = getenv("PCR_WAIT_COUNTS") != nullptr;  // A/B hook
        const bool nowait = level == 0 && !init_list && split && pre_level1 && ctx->spec_request && ctx->frame_stream && ctx->spec_zero && !no_nowait;
        uint32_t *mail = (uint32_t *)ctx->pinned + (nowait ? 128 : 32);
        PCR_CUDA(ctx, cudaMemcpyAsync(mail, counters, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));  // (words 32 .. 47 of the block)
        for (const auto &pg : ctx->piggy)  // small results other steps want from the same round trip
            PCR_CUDA(ctx, cudaMemcpyAsync(pg.dst, pg.src, pg.bytes, cudaMemcpyDeviceToHost, ctx->stream));
        ctx->piggy.clear();
        if (nowait) {
            ctx->spec_pending = true;
            PCR_MARK("levels: deferred count left for the last round trip");
            return PCR_OK;
        }
        // A frame stream whose previous frame needed the next level will need it again: queue its build behind the
        // count's copy and wait on an event, so the GPU builds while the host wakes up and reads the count.
        const bool speculate = level == 0 && !init_list && ctx->frame_stream && ctx->spec_coarser && !cur->coarser;
        PCR_MARK("levels: wait for deferred count");
        if (speculate) {
            if (!ctx->ev_count) PCR_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_count, cudaEventDisableTiming));
            PCR_CUDA(ctx, cudaEventRecord(ctx->ev_count, ctx->stream));
            Index *pre = nullptr;
            {
                TimeScope ts(ctx, kTagKnnDeferred);
                PCR_TRY(index_coarser_level(cur, &pre));
            }
            PCR_CUDA(ctx, cudaEventSynchronize(ctx->ev_count));
        } else {
            PCR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        PCR_MARK("levels: got deferred count");
        n_cur = mail[level & 1];
        if (speculate) (n_cur > 0 ? ctx->stat_spec_hits : ctx->stat_spec_misses)++;
        if (level == 0 && !init_list && !split) ctx->spec_coarser = n_cur > 0;
        if (level == 0 && !init_list && split && pre_level1) ctx->spec_zero = mail[0] == 0 && mail[1] == 0;
        if (dbg) fprintf(stderr, "[pcr] level %d: %u of %u queries deferred (cell %.4g)\n", level, n_cur, a.nq, cur->grids_h[0].h);
        if (dbg && first_of_two)
            fprintf(stderr, "[pcr] level 0: %u normal / %u dense / %u sparse queries, %u needed more than the first pass's shells, %u of the sparse deferred again, %u handed back by the tiles\n",
                    mail[3] + mail[7], mail[4], mail[5], mail[2], mail[1], mail[6]);
        if (level == 0 && pre_level1) (mail[5] > 0 ? ctx->stat_spec_hits : ctx->stat_spec_misses)++;  // was the level built ahead needed?
        if (level == 0 && pre_level1) {
            // the sparse queries are done on level 1; what they deferred there sits in lists[1] (count mail[1]).  Level 0's own
            // leftovers (n_cur) go through level 1 next and append to the same list.
            if (n_cur == 0) {
                if (mail[1] == 0 || kMaxLevels < 3) break;
                // nothing for level 1: continue with level 2 over the sparse pass's leftovers
                Index *l2 = nullptr;
                {
                    TimeScope ts(ctx, kTagKnnDeferred);
                    PCR_TRY(index_coarser_level(cur->coarser, &l2));
                }
                cur = l2;
                qlist = lists[1];
                n_cur = mail[1];
                level = 1;
                continue;
            }
        } else if (n_cur == 0) {
            break;
        }
        Index *next = nullptr;
        {
            TimeScope ts(ctx, kTagKnnDeferred);
            PCR_TRY(index_coarser_level(cur, &next));
        }
        cur = next;
        qlist = lists[level & 1];
    }
    return PCR_OK;
}

inline unsigned blocks_for(uint32_t nq, int qpw) { return (nq + kWarps * qpw - 1) / (kWarps * qpw); }
// a launch whose real length is still on the device (a.nq is its capacity) strides over the list with a bounded grid
inline unsigned blocks_for(Ctx *ctx, const LevelArgs &a, int qpw) {
    const unsigned b = blocks_for(a.nq, qpw);
    return a.nq_dev ? std::min<unsigned>(b, (unsigned)ctx->sm_count * 16u) : b;
}

}  // namespace

// ---- query sharding over the ranks of a communicator (SURVEY 8e: KNN / normals / SOR of ONE cloud) -------------
// Every rank holds the whole cloud and builds the same index (cell membership and the cell table are deterministic;
// the order of the points INSIDE a cell is not: it comes from atomics).  The queries are therefore split at CELL
// boundaries of the cell-sorted order -- rank r takes the cells whose first point lies in [r n / G, (r + 1) n / G) --
// so every rank derives the same partition of the points from its own copy.  Results are written at original
// indices into zero-initialised arrays and merged with an integer sum over NCCL: every element is written by
// exactly one rank, so the sum reproduces its bits (including -0.0 and inf), and every rank ends up with the
// full result.  Points outside the index (non-finite) belong to rank 0.
namespace {
__global__ void shard_bounds_kernel(const uint32_t *__restrict__ cell_start, uint32_t total_cells, uint32_t n_indexed, int rank, int world,
                                    uint32_t *__restrict__ out) {
    const int t = threadIdx.x;  // 0: begin of this rank, 1: begin of the next
    if (t > 1) return;
    const uint32_t target = (uint32_t)(((unsigned long long)n_indexed * (unsigned)(rank + t)) / (unsigned)world);
    uint32_t lo = 0, hi = total_cells;  // smallest cell c with cell_start[c] >= target (cell_start[total_cells] = n_indexed)
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (cell_start[mid] >= target) hi = mid;
        else lo = mid + 1;
    }
    out[t] = cell_start[lo];
}

// SOR: non-finite points have mean distance INF (statistical_outlier.rs:22-24); only they are written here
__global__ void fill_nonfinite_f32_kernel(const float4 *__restrict__ orig4, size_t n, float *__restrict__ p, float v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 q = orig4[i];
    if (!finite3(q.x, q.y, q.z)) p[i] = v;
}
}  // namespace

bool query_sharding_active(const Ctx *ctx, const Index *ix) { return ctx->shard_queries && ctx->world > 1 && ix->n_frames == 1; }

int index_shard_queries(Index *ix) {
    Ctx *ctx = ix->ctx;
    ix->q_begin = 0;
    ix->q_count = (uint32_t)ix->n_indexed;
    if (!query_sharding_active(ctx, ix) || ix->n_indexed == 0) return PCR_OK;
    PCR_TRY(ensure(ctx, ctx->b_small, 4096));
    uint32_t *d_out = (uint32_t *)((char *)ctx->b_small.p + 2048);
    shard_bounds_kernel<<<1, 32, 0, ctx->stream>>>(ix->cell_start, ix->total_cells, (uint32_t)ix->n_indexed, ctx->rank, ctx->world, d_out);
    PCR_LAUNCH_CHECK(ctx);
    uint32_t *mail = (uint32_t *)ctx->pinned + 48;
    PCR_CUDA(ctx, cudaMemcpyAsync(mail, d_out, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PCR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ix->q_begin = mail[0];
    ix->q_count = mail[1] - mail[0];
    return PCR_OK;
}

namespace {
// Device u32 copy of the query offsets of a batch (in ctx->b_qoff, valid until the next batch query on the context).
int upload_query_offsets(Ctx *ctx, const QueryFrames &qf, const uint32_t **d_off) {
    std::vector<uint32_t> h(qf.n_frames + 1);
    for (size_t f = 0; f <= qf.n_frames; f++) h[f] = (uint32_t)qf.offsets[f];
    PCR_TRY(ensure(ctx, ctx->b_qoff, sizeof(uint32_t) * h.size()));
    PCR_CUDA(ctx, cudaMemcpyAsync(ctx->b_qoff.p, h.data(), sizeof(uint32_t) * h.size(), cudaMemcpyHostToDevice, ctx->stream));
    *d_off = (const uint32_t *)ctx->b_qoff.p;
    return PCR_OK;
}

// kQFrames: the queries of a batch index, d_qoff their device offsets (see knn_queries_kernel)
template <bool kQFrames>
int knn_queries_run(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq, size_t k, uint32_t *d_idx,
                    float *d_dist, uint32_t *d_counts, const uint32_t *d_qoff) {
    Ctx *ctx = ix->ctx;
    const int kk = (int)k;
    if (k > 32) PCR_TRY(set_smem(ctx, knn_queries_kernel<true, kQPW0, kQFrames>, sizeof(unsigned long long) * k * kWarps));
    if (k > 32) PCR_TRY(set_smem(ctx, knn_queries_kernel<true, kQPWL, kQFrames>, sizeof(unsigned long long) * k * kWarps));
    ThreadArgs ta = {};
    ta.qx = dqx; ta.qy = dqy; ta.qz = dqz;
    ta.idx = d_idx; ta.dist = d_dist; ta.counts = d_counts;
    ta.kk = kk;
    ta.qoff = d_qoff;
    return run_levels(ix, (uint32_t)nq, kTagKnn, [&](const LevelArgs &a, int qpw) -> int {
        if (qpw == kQPW0 && k <= 32) return launch_thread_kernel<0, kQFrames>(ctx, a, ta);
        unsigned blocks = blocks_for(ctx, a, qpw);
        if (qpw == kQPWS) {
            knn_queries_kernel<false, kQPWS, kQFrames><<<blocks, kThreads, 0, ctx->stream>>>(a, dqx, dqy, dqz, kk, d_idx, d_dist, d_counts, d_qoff);
            PCR_LAUNCH_CHECK(ctx);
            return PCR_OK;
        }
        size_t smem = k <= 32 ? 0 : sizeof(unsigned long long) * k * kWarps;
        if (k <= 32) {
            if (qpw == kQPW0) knn_queries_kernel<false, kQPW0, kQFrames><<<blocks, kThreads, 0, ctx->stream>>>(a, dqx, dqy, dqz, kk, d_idx, d_dist, d_counts, d_qoff);
            else knn_queries_kernel<false, kQPWL, kQFrames><<<blocks, kThreads, 0, ctx->stream>>>(a, dqx, dqy, dqz, kk, d_idx, d_dist, d_counts, d_qoff);
        } else {
            if (qpw == kQPW0) knn_queries_kernel<true, kQPW0, kQFrames><<<blocks, kThreads, smem, ctx->stream>>>(a, dqx, dqy, dqz, kk, d_idx, d_dist, d_counts, d_qoff);
            else knn_queries_kernel<true, kQPWL, kQFrames><<<blocks, kThreads, smem, ctx->stream>>>(a, dqx, dqy, dqz, kk, d_idx, d_dist, d_counts, d_qoff);
        }
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    }, nullptr, nullptr, k <= 32 ? kk : 0, 0, dqx, dqy, dqz, false, d_qoff);
}
}  // namespace

int knn_queries_dev(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq, size_t k, uint32_t *d_idx,
                    float *d_dist, uint32_t *d_counts, const QueryFrames *qf) {
    Ctx *ctx = ix->ctx;
    if (nq == 0 || k == 0) return PCR_OK;
    if (k > PCR_MAX_K) return fail(ctx, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    if (nq > 0xfffffff0ull) return fail(ctx, PCR_ERR_UNSUPPORTED, "too many queries");
    if (ix->n_frames == 1) return knn_queries_run<false>(ix, dqx, dqy, dqz, nq, k, d_idx, d_dist, d_counts, nullptr);  // (a batch of one)
    if (!qf || qf->n_frames != (size_t)ix->n_frames)
        return fail(ctx, PCR_ERR_INVALID_ARG, "queries on a batch index of %d frames need query offsets of as many frames (pcr_knn_batch)", ix->n_frames);
    const uint32_t *d_qoff = nullptr;
    PCR_TRY(upload_query_offsets(ctx, *qf, &d_qoff));
    return knn_queries_run<true>(ix, dqx, dqy, dqz, nq, k, d_idx, d_dist, d_counts, d_qoff);
}

int sor_mean_dist_dev(Index *ix, size_t k, float *d_mean_d, const SorLists *keep_lists, bool allow_shard) {
    Ctx *ctx = ix->ctx;
    if (ix->n == 0) return PCR_OK;
    const size_t kk = k + 1;  // statistical_outlier.rs:25
    if (kk > PCR_MAX_K) return fail(ctx, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K - 1", k);
    // a rank of a query-sharded call searches its share of the cloud; the mean distances are merged at the end, so
    // that every rank folds the same N values in the same order and gets the same statistics and mask (SURVEY 8e)
    const bool shard = allow_shard && !keep_lists && query_sharding_active(ctx, ix);
    uint32_t q_begin = 0, q_count = (uint32_t)ix->n_indexed;
    if (shard) {
        PCR_TRY(index_shard_queries(ix));
        q_begin = ix->q_begin;
        q_count = ix->q_count;
        PCR_CUDA(ctx, cudaMemsetAsync(d_mean_d, 0, sizeof(float) * ix->n, ctx->stream));
        if (ix->n_indexed < ix->n && ctx->rank == 0) {
            fill_nonfinite_f32_kernel<<<(unsigned)((ix->n + 255) / 256), 256, 0, ctx->stream>>>(ix->orig4, ix->n, d_mean_d, INFINITY);
            PCR_LAUNCH_CHECK(ctx);
        }
    } else if (ix->n_indexed < ix->n) {  // statistical_outlier.rs:22-24: non-finite points -> INF
        fill_f32_kernel<<<(unsigned)((ix->n + 255) / 256), 256, 0, ctx->stream>>>(d_mean_d, ix->n, INFINITY);
        PCR_LAUNCH_CHECK(ctx);
    }
    if (ix->n_indexed == 0) return PCR_OK;
    const size_t smem = kk <= 32 ? (kk * 33 + 64) * sizeof(float) * kWarps : sizeof(unsigned long long) * kk * kWarps;
    if (kk > 32) {
        PCR_TRY(set_smem(ctx, sor_mean_kernel<true, kQPW0>, smem));
        PCR_TRY(set_smem(ctx, sor_mean_kernel<true, kQPWL>, smem));
    }
    ThreadArgs ta = {};
    ta.mean_d = d_mean_d;
    ta.kk = (int)kk;
    if (keep_lists) {  // search K >= kk neighbours on level 0 and keep the lists (deferred queries get none)
        ta.kk = (int)keep_lists->K;
        ta.kk_sor = (int)kk;
        ta.lists = keep_lists->lists;
        ta.list_cnt = keep_lists->cnt;
        ta.list_stride = keep_lists->stride;
        if (!keep_lists->initialised) PCR_CUDA(ctx, cudaMemsetAsync(keep_lists->cnt, 0xff, keep_lists->stride, ctx->stream));
    }
    const int rc = run_levels(ix, q_count, kTagKnn, [&](const LevelArgs &a, int qpw) -> int {
        if (qpw == kQPW0 && keep_lists) return launch_thread_kernel<3>(ctx, a, ta);
        if (qpw == kQPW0 && kk <= 32) return launch_thread_kernel<1>(ctx, a, ta);
        unsigned blocks = blocks_for(ctx, a, qpw);
        if (qpw == kQPWS) {  // level 0, a warp per query
            const int kw = keep_lists ? ta.kk : (int)kk;
            const size_t smem_w = ((size_t)kw * (kQPWS + 1) + 64) * sizeof(float) * kWarps;
            if (keep_lists)
                PCR_CUDA(ctx, launch_chained(sor_mean_kernel<false, kQPWS>, dim3(blocks), dim3(kThreads), smem_w, ctx->stream, a, kw, d_mean_d, ta.lists,
                                             ta.list_cnt, ta.list_stride, ta.kk_sor));
            else
                PCR_CUDA(ctx, launch_chained(sor_mean_kernel<false, kQPWS>, dim3(blocks), dim3(kThreads), smem_w, ctx->stream, a, kw, d_mean_d,
                                             (uint32_t *)nullptr, (uint8_t *)nullptr, (size_t)0, kw));
            ctx->launches++;
            return PCR_OK;
        }
        if ((a.follow_up || a.no_tile) && keep_lists) {  // the first pass's leftovers / the dense class on the same level: K neighbours, lists kept
            const size_t smem_k = ((size_t)ta.kk * (kQPWL + 1) + 64) * sizeof(float) * kWarps;
            PCR_CUDA(ctx, launch_chained(sor_mean_kernel<false, kQPWL>, dim3(blocks), dim3(kThreads), smem_k, ctx->stream, a, ta.kk, d_mean_d, ta.lists,
                                         ta.list_cnt, ta.list_stride, ta.kk_sor));
        } else if (kk <= 32) {
            if (qpw == kQPW0) sor_mean_kernel<false, kQPW0><<<blocks, kThreads, smem, ctx->stream>>>(a, (int)kk, d_mean_d, nullptr, nullptr, 0, (int)kk);
            else sor_mean_kernel<false, kQPWL><<<blocks, kThreads, smem, ctx->stream>>>(a, (int)kk, d_mean_d, nullptr, nullptr, 0, (int)kk);
        } else {
            if (qpw == kQPW0) sor_mean_kernel<true, kQPW0><<<blocks, kThreads, smem, ctx->stream>>>(a, (int)kk, d_mean_d, nullptr, nullptr, 0, (int)kk);
            else sor_mean_kernel<true, kQPWL><<<blocks, kThreads, smem, ctx->stream>>>(a, (int)kk, d_mean_d, nullptr, nullptr, 0, (int)kk);
        }
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    }, nullptr, nullptr, keep_lists ? ta.kk : (kk <= 32 ? (int)kk : 0), q_begin, nullptr, nullptr, nullptr, true);
    PCR_TRY(rc);
    if (shard) PCR_TRY(comm_allreduce_u32(ctx, reinterpret_cast<uint32_t *>(d_mean_d), ix->n));
    return PCR_OK;
}

int normals_dev(Index *ix, size_t k, const float vp[3], float *d_nx, float *d_ny, float *d_nz, const uint8_t *d_mask, bool allow_shard) {
    Ctx *ctx = ix->ctx;
    if (ix->n == 0 || k == 0) return PCR_OK;
    if (k > PCR_MAX_K) return fail(ctx, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    const bool shard = allow_shard && query_sharding_active(ctx, ix);  // (see index_shard_queries)
    uint32_t q_begin = 0, q_count = (uint32_t)ix->n_indexed;
    if (shard) {
        PCR_TRY(index_shard_queries(ix));
        q_begin = ix->q_begin;
        q_count = ix->q_count;
        for (float *p : {d_nx, d_ny, d_nz}) PCR_CUDA(ctx, cudaMemsetAsync(p, 0, sizeof(float) * ix->n, ctx->stream));
    }
    if ((d_mask || ix->n_indexed < ix->n) && (!shard || ctx->rank == 0)) {
        fill_unindexed_normals_kernel<<<(unsigned)((ix->n + 255) / 256), 256, 0, ctx->stream>>>(ix->orig4, d_mask, ix->n, d_nx,
                                                                                                d_ny, d_nz);
        PCR_LAUNCH_CHECK(ctx);
    }
    if (ix->n_indexed == 0) return PCR_OK;
    const size_t smem = k <= 32 ? (k * 3 * 33 + 64) * sizeof(float) * kWarps : sizeof(unsigned long long) * k * kWarps;
    if (k <= 32) {
        PCR_TRY(set_smem(ctx, normals_kernel<false, kQPW0>, smem));
        PCR_TRY(set_smem(ctx, normals_kernel<false, kQPWL>, smem));
    } else {
        PCR_TRY(set_smem(ctx, normals_kernel<true, kQPW0>, smem));
        PCR_TRY(set_smem(ctx, normals_kernel<true, kQPWL>, smem));
    }
    const float v0 = vp[0], v1 = vp[1], v2 = vp[2];
    ThreadArgs ta = {};
    ta.orig4 = ix->orig4;
    ta.vx = v0; ta.vy = v1; ta.vz = v2;
    ta.nx = d_nx; ta.ny = d_ny; ta.nz = d_nz;
    ta.kk = (int)k;
    const int rc = run_levels(ix, q_count, kTagKnnNormals, [&](const LevelArgs &a, int qpw) -> int {
        if (qpw == kQPW0 && k <= 32) return launch_thread_kernel<2>(ctx, a, ta);
        unsigned blocks = blocks_for(ctx, a, qpw);
        if (qpw == kQPWS) {  // level 0, a warp per query
            const size_t smem_w = ((size_t)k * 3 * (kQPWS + 1) + 64) * sizeof(float) * kWarps;
            normals_kernel<false, kQPWS><<<blocks, kThreads, smem_w, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
            PCR_LAUNCH_CHECK(ctx);
            return PCR_OK;
        }
        if (k <= 32) {
            if (qpw == kQPW0) normals_kernel<false, kQPW0><<<blocks, kThreads, smem, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
            else normals_kernel<false, kQPWL><<<blocks, kThreads, smem, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
        } else {
            if (qpw == kQPW0) normals_kernel<true, kQPW0><<<blocks, kThreads, smem, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
            else normals_kernel<true, kQPWL><<<blocks, kThreads, smem, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
        }
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    }, nullptr, nullptr, k <= 32 ? (int)k : 0, q_begin, nullptr, nullptr, nullptr, true);
    PCR_TRY(rc);
    if (shard)
        for (float *p : {d_nx, d_ny, d_nz}) PCR_TRY(comm_allreduce_u32(ctx, reinterpret_cast<uint32_t *>(p), ix->n));
    return PCR_OK;
}

// ---- normals of the kept points from the SOR pass's neighbour lists -------------------------------
// The K nearest of a point among ALL points, filtered by the keep mask, are its nearest among the KEPT
// points, in the same (d^2, index) order -- as long as k of them survive (or the list is complete).
// Queries without a usable list go to `fallback` and are searched again on the tombstoned index.
namespace {
// MODE 0: every query, filtered by the keep mask (the plain form).
// MODE 1: EARLY pass, launched before the mask exists (it overlaps the exact fold, which occupies 16 SMs): every query as if
//         nothing were removed -- its first min(c, k) list entries.  Never falls back (a list shorter than k is complete).
// MODE 2: FIX-UP pass after the mask: removed queries get 0; a query none of whose first min(c, k) entries was removed keeps
//         the early result (the filtered walk would take exactly those entries); the others are gathered per CTA and
//         recomputed by its first threads, so that a warp does not pay a full evaluation for one lane in thirty.
template <bool kFilter>
__device__ __forceinline__ void normal_from_list(uint32_t q, float4 p, int c, const uint32_t *__restrict__ lists, size_t stride, int K, int k,
                                                 const uint8_t *__restrict__ keep, const float4 *__restrict__ orig4, float vx_, float vy_,
                                                 float vz_, float *__restrict__ nx, float *__restrict__ ny, float *__restrict__ nz,
                                                 uint32_t *__restrict__ fallback, uint32_t *__restrict__ fallback_count) {
    // The list is walked eight entries at a time: the indices, then the keep flags, then the points are independent loads
    // (one entry after the other was three dependent L2 round trips per neighbour); only the additions are a chain.
    bool ok = c != 0xff;
    int taken = 0;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    uint32_t used = 0;  // bit j: list entry j is one of the (at most k) neighbours taken
    if (ok) {
        for (int j0 = 0; j0 < c && taken < k; j0 += 8) {  // estimate.rs:54-65, neighbour order
            uint32_t id[8];
            bool kp[8];
            float4 t[8];
#pragma unroll
            for (int u = 0; u < 8; u++) id[u] = __ldg(&lists[(size_t)min(j0 + u, c - 1) * stride + q]);
#pragma unroll
            for (int u = 0; u < 8; u++) kp[u] = j0 + u < c && (!kFilter || keep[id[u]] != 0);
#pragma unroll
            for (int u = 0; u < 8; u++) t[u] = kp[u] ? __ldg(&orig4[id[u]]) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 8; u++) {
                if (kp[u] && taken < k) {
                    cx = __fadd_rn(cx, t[u].x);
                    cy = __fadd_rn(cy, t[u].y);
                    cz = __fadd_rn(cz, t[u].z);
                    taken++;
                    used |= 1u << (j0 + u);
                }
            }
        }
        ok = taken == k || c < K;  // a truncated list with fewer than k survivors cannot be trusted
    }
    if (!ok) {
        if (kFilter) fallback[atomicAdd(fallback_count, 1u)] = q;
        return;  // (early pass: a query without a list is left to the fix-up pass)
    }
    float ox = 0.f, oy = 0.f, oz = 1.f;
    if (taken >= 1) {
        const float count = (float)taken;
        cx = __fdiv_rn(cx, count);
        cy = __fdiv_rn(cy, count);
        cz = __fdiv_rn(cz, count);
        float c00 = 0.f, c01 = 0.f, c02 = 0.f, c11 = 0.f, c12 = 0.f, c22 = 0.f;
        for (int j0 = 0; j0 < 32 && (used >> j0) != 0u; j0 += 8) {  // estimate.rs:68-84
            float4 t[8];
#pragma unroll
            for (int u = 0; u < 8; u++)
                t[u] = ((used >> (j0 + u)) & 1u) ? __ldg(&orig4[__ldg(&lists[(size_t)(j0 + u) * stride + q])]) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 8; u++) {
                if ((used >> (j0 + u)) & 1u) {
                    const float dx = __fsub_rn(t[u].x, cx), dy = __fsub_rn(t[u].y, cy), dz = __fsub_rn(t[u].z, cz);
                    c00 = __fadd_rn(c00, __fmul_rn(dx, dx));
                    c01 = __fadd_rn(c01, __fmul_rn(dx, dy));
                    c02 = __fadd_rn(c02, __fmul_rn(dx, dz));
                    c11 = __fadd_rn(c11, __fmul_rn(dy, dy));
                    c12 = __fadd_rn(c12, __fmul_rn(dy, dz));
                    c22 = __fadd_rn(c22, __fmul_rn(dz, dz));
                }
            }
        }
        float ex, ey, ez;
        smallest_eigenvector_3x3(c00, c01, c02, c11, c12, c22, ex, ey, ez);
        const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez)));
        if (len > 1e-10f) {
            ex = __fdiv_rn(ex, len);
            ey = __fdiv_rn(ey, len);
            ez = __fdiv_rn(ez, len);
        }
        const float vx = __fsub_rn(vx_, p.x), vy = __fsub_rn(vy_, p.y), vz = __fsub_rn(vz_, p.z);
        const float dot = __fadd_rn(__fadd_rn(__fmul_rn(ex, vx), __fmul_rn(ey, vy)), __fmul_rn(ez, vz));
        if (dot < 0.0f) {
            ex = -ex; ey = -ey; ez = -ez;
        }
        ox = ex; oy = ey; oz = ez;
    }
    const uint32_t oi = __float_as_uint(p.w);
    nx[oi] = ox;
    ny[oi] = oy;
    nz[oi] = oz;
}

constexpr int kNflThreads = 128;
template <int MODE>
__global__ void __launch_bounds__(kNflThreads) normals_from_lists_kernel(const float4 *__restrict__ qpts, uint32_t nq,
                                                                 const uint32_t *__restrict__ lists, const uint8_t *__restrict__ list_cnt,
                                                                 size_t stride, int K, int k, const uint8_t *__restrict__ keep,
                                                                 const float4 *__restrict__ orig4, float vx_, float vy_, float vz_,
                                                                 float *__restrict__ nx, float *__restrict__ ny, float *__restrict__ nz,
                                                                 uint32_t *__restrict__ fallback, uint32_t *__restrict__ fallback_count) {
    PCR_GRID_DEP_SYNC();
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (MODE == 1) {
        if (q >= nq) return;
        normal_from_list<false>(q, __ldg(&qpts[q]), list_cnt[q], lists, stride, K, k, nullptr, orig4, vx_, vy_, vz_, nx, ny, nz, nullptr, nullptr);
        return;
    }
    __shared__ uint32_t s_redo[kNflThreads];
    __shared__ int s_n;
    if (MODE == 2) {
        if (threadIdx.x == 0) s_n = 0;
        __syncthreads();
    }
    bool work = q < nq;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (work) {
        p = __ldg(&qpts[q]);
        if (p.x != p.x) {  // removed by SOR (tombstoned): not a point of the kept cloud -> 0 (like the unindexed fill)
            const uint32_t oi = __float_as_uint(p.w);
            nx[oi] = 0.f;
            ny[oi] = 0.f;
            nz[oi] = 0.f;
            work = false;
        }
    }
    if (MODE == 2) {
        if (work) {
            const int c = list_cnt[q];
            bool redo = c == 0xff;
            if (!redo) {
                const int m = min(c, k);
                for (int j0 = 0; j0 < m; j0 += 8) {  // (eight independent index loads, then eight independent flag loads)
                    uint32_t id[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) id[u] = __ldg(&lists[(size_t)min(j0 + u, m - 1) * stride + q]);
#pragma unroll
                    for (int u = 0; u < 8; u++) redo |= keep[id[u]] == 0;
                }
            }
            if (redo) s_redo[atomicAdd(&s_n, 1)] = q;
        }
        __syncthreads();
        work = (int)threadIdx.x < s_n;
        if (work) {
            q = s_redo[threadIdx.x];
            p = __ldg(&qpts[q]);
        }
    }
    if (!work) return;
    normal_from_list<true>(q, p, list_cnt[q], lists, stride, K, k, keep, orig4, vx_, vy_, vz_, nx, ny, nz, fallback, fallback_count);
}
}  // namespace

// normals of the kept points of `ix` (already tombstoned with d_keep) from the lists of the SOR pass;
// the few queries without a usable list are searched again (warp kernels on the tombstoned levels)
// The early pass (MODE 1 above) on a side stream, forked from the main stream's current position (the searches are done, the
// lists complete); `ev_join[0]` marks its end.  The caller makes the main stream wait for that event before the index is
// tombstoned and the fix-up pass runs (normals_from_lists_dev with early = true).
// (the fork: where in the main stream the side stream's pass may start -- recorded BEFORE the fold is launched, the pass
// itself queued AFTER it, so that the fold's cluster, which needs 16 empty SMs, is first in line.  Measured: no difference
// on the single frame -- the fold reads 65 us beside the pass either way, 58 us without it -- 10.8 -> 10.7 ms on the batch.)
int normals_early_fork(Ctx *ctx) {
    PCR_TRY(ensure_side_streams(ctx));
    PCR_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
    return PCR_OK;
}

int normals_early_from_lists_dev(Index *ix, size_t k, const float vp[3], const SorLists &sl, float *d_nx, float *d_ny, float *d_nz, bool *launched) {
    Ctx *ctx = ix->ctx;
    *launched = false;
    static const bool off = getenv("PCR_NO_EARLY_NORMALS") != nullptr;  // A/B hook
    const uint32_t nq = (uint32_t)ix->n_indexed;
    if (off || ix->n == 0 || k == 0 || nq == 0) return PCR_OK;
    PCR_CUDA(ctx, cudaStreamWaitEvent(ctx->side[0], ctx->ev_fork, 0));  // (normals_early_fork)
    {
        StreamSwap sw(ctx, ctx->side[0]);
        TimeScope ts(ctx, kTagKnnNormals);
        normals_from_lists_kernel<1><<<(nq + kNflThreads - 1) / kNflThreads, kNflThreads, 0, ctx->stream>>>(
            ix->sorted, nq, sl.lists, sl.cnt, sl.stride, (int)sl.K, (int)k, nullptr, ix->orig4, vp[0], vp[1], vp[2], d_nx, d_ny, d_nz, nullptr, nullptr);
        PCR_LAUNCH_CHECK(ctx);
    }
    PCR_CUDA(ctx, cudaEventRecord(ctx->ev_join[0], ctx->side[0]));
    *launched = true;
    return PCR_OK;
}

int normals_from_lists_dev(Index *ix, size_t k, const float vp[3], const SorLists &sl, const uint8_t *d_keep, float *d_nx, float *d_ny,
                           float *d_nz, const unsigned long long *d_kept0, unsigned long long *h_kept0, bool early) {
    Ctx *ctx = ix->ctx;
    if (ix->n == 0 || k == 0) return PCR_OK;
    if (ix->n_indexed < ix->n) {  // points outside the index (non-finite); the removed indexed ones are zeroed by the kernel below
        fill_unindexed_normals_kernel<<<(unsigned)((ix->n + 255) / 256), 256, 0, ctx->stream>>>(ix->orig4, d_keep, ix->n, d_nx, d_ny, d_nz);
        PCR_LAUNCH_CHECK(ctx);
    }
    const uint32_t nq = (uint32_t)ix->n_indexed;
    if (nq == 0) return PCR_OK;
    uint32_t *d_fb_count = sl.fallback + sl.stride;  // one counter behind the list
    if (!sl.initialised) PCR_CUDA(ctx, cudaMemsetAsync(d_fb_count, 0, sizeof(uint32_t), ctx->stream));
    {
        TimeScope ts(ctx, kTagKnnNormals);
        PCR_CUDA(ctx, launch_chained(early ? normals_from_lists_kernel<2> : normals_from_lists_kernel<0>, dim3((nq + kNflThreads - 1) / kNflThreads),
                                     dim3(kNflThreads), 0, ctx->stream, ix->sorted, nq, sl.lists, sl.cnt, sl.stride, (int)sl.K, (int)k, d_keep, ix->orig4,
                                     vp[0], vp[1], vp[2], d_nx, d_ny, d_nz, sl.fallback, d_fb_count));
        ctx->launches++;
    }
    // The queries that fall back are few, and their count is still on the device: launch their level-0 pass now for a
    // fixed capacity (the kernel reads the count itself) and let the count, the kept count the caller's compaction
    // wants and the pass's own deferred count come back in ONE round trip.
    uint32_t *mail = (uint32_t *)ctx->pinned + 40;
    unsigned long long *mail_kept = (unsigned long long *)((uint32_t *)ctx->pinned + 42);
    ctx->piggy.clear();
    ctx->piggy.push_back({mail, d_fb_count, sizeof(uint32_t)});
    if (d_kept0 && h_kept0) ctx->piggy.push_back({mail_kept, d_kept0, sizeof(unsigned long long)});
    const size_t smem = k <= 32 ? (k * 3 * 33 + 64) * sizeof(float) * kWarps : sizeof(unsigned long long) * k * kWarps;
    if (k <= 32) PCR_TRY(set_smem(ctx, normals_kernel<false, kQPWL>, smem));
    else PCR_TRY(set_smem(ctx, normals_kernel<true, kQPWL>, smem));
    const float v0 = vp[0], v1 = vp[1], v2 = vp[2];
    auto launch = [&](const LevelArgs &a, int qpw) -> int {
        const unsigned blocks = blocks_for(ctx, a, qpw);
        if (k <= 32) normals_kernel<false, kQPWL><<<blocks, kThreads, smem, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
        else normals_kernel<true, kQPWL><<<blocks, kThreads, smem, ctx->stream>>>(a, ix->orig4, (int)k, v0, v1, v2, d_nx, d_ny, d_nz);
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    };
    uint32_t cap = std::min<uint32_t>(nq, 2048u);
    if (const char *e = getenv("PCR_FALLBACK_CAP")) cap = std::max(1u, std::min<uint32_t>(nq, (uint32_t)atoi(e)));  // test hook
    PCR_MARK("normals: fallback pass queued blind");
    const int rc = run_levels(ix, cap, kTagKnnDeferred, launch, sl.fallback, d_fb_count);
    ctx->piggy.clear();
    PCR_TRY(rc);
    PCR_MARK("normals: fallback pass done");
    const uint32_t n_fb = *mail;
    if (d_kept0 && h_kept0) *h_kept0 = *mail_kept;
    if (getenv("PCR_DEBUG")) fprintf(stderr, "[pcr] normals from SOR lists: %u of %u queries fall back to a search\n", n_fb, nq);
    if (n_fb <= cap) return PCR_OK;
    return run_levels(ix, n_fb - cap, kTagKnnDeferred, launch, sl.fallback + cap);  // more than the blind pass covered
}

int radius_count_dev(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq, float radius,
                     uint32_t *d_counts, const QueryFrames *qf) {
    Ctx *ctx = ix->ctx;
    if (nq == 0) return PCR_OK;
    if (ix->n_frames != 1 && qf) {  // external queries of a batch: query frame f counts in index frame f
        if (qf->n_frames != (size_t)ix->n_frames)
            return fail(ctx, PCR_ERR_INVALID_ARG, "queries on a batch index of %d frames need query offsets of as many frames", ix->n_frames);
        const uint32_t *d_qoff = nullptr;
        PCR_TRY(upload_query_offsets(ctx, *qf, &d_qoff));
        radius_kernel<false, true><<<(unsigned)((nq + 255) / 256), 256, 0, ctx->stream>>>(ix->grids, ix->cell_start, ix->sorted, dqx, dqy, dqz, nq,
                                                                                          radius, d_counts, nullptr, nullptr, d_qoff, ix->n_frames);
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    }
    if (ix->n_frames != 1) {  // a batch: every indexed point counts its neighbours inside its own frame
        if (nq != ix->n) return fail(ctx, PCR_ERR_UNSUPPORTED, "radius queries on a multi-frame index must be its own points");
        radius_kernel<false, true><<<(unsigned)((nq + 255) / 256), 256, 0, ctx->stream>>>(ix->grids, ix->cell_start, ix->sorted, dqx, dqy, dqz, nq,
                                                                                          radius, d_counts, nullptr, nullptr, ix->frame_in_off,
                                                                                          ix->n_frames);
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    }
    radius_kernel<false><<<(unsigned)((nq + 255) / 256), 256, 0, ctx->stream>>>(ix->grids, ix->cell_start, ix->sorted, dqx, dqy,
                                                                                dqz, nq, radius, d_counts, nullptr, nullptr);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

int radius_fill_dev(Index *ix, const float *dqx, const float *dqy, const float *dqz, size_t nq, float radius,
                    const uint64_t *d_offsets, uint32_t *d_idx, const QueryFrames *qf) {
    Ctx *ctx = ix->ctx;
    if (nq == 0) return PCR_OK;
    if (ix->n_frames != 1) {  // external queries of a batch: frame-local indices
        if (!qf || qf->n_frames != (size_t)ix->n_frames)
            return fail(ctx, PCR_ERR_INVALID_ARG, "queries on a batch index of %d frames need query offsets of as many frames", ix->n_frames);
        const uint32_t *d_qoff = nullptr;
        PCR_TRY(upload_query_offsets(ctx, *qf, &d_qoff));
        radius_kernel<true, true><<<(unsigned)((nq + 255) / 256), 256, 0, ctx->stream>>>(ix->grids, ix->cell_start, ix->sorted, dqx, dqy, dqz, nq,
                                                                                         radius, nullptr, d_offsets, d_idx, d_qoff, ix->n_frames);
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    }
    radius_kernel<true><<<(unsigned)((nq + 255) / 256), 256, 0, ctx->stream>>>(ix->grids, ix->cell_start, ix->sorted, dqx, dqy,
                                                                               dqz, nq, radius, nullptr, d_offsets, d_idx);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

}  // namespace pcr
