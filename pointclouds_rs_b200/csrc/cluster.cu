// cluster.cu -- euclidean_cluster (crates/segmentation/src/euclidean_cluster.rs:96-187) on the GPU.
//
// The reference bins the finite points into cells of size r keyed by floor(x * (1/r)) as i32
// (:55-61), tests every pair of points that share a cell or sit in key-adjacent cells with
// dx*dx + dy*dy + dz*dz <= r*r (f32, :147-151) and takes the connected components of that graph.
// The components do not depend on the order the pairs are visited in, so the GPU version may test
// them in any order -- but it has to test exactly the SAME pair set, which is why the cells here are
// keyed by the reference's own f32 expression and not by the KNN grid's f64 cell coordinates (a pair
// closer than r whose keys differ by 2 through f32 rounding is missed by the reference, and must be
// missed here too).
//
//   insert_kernel    open-addressing hash table of cells (one representative point per slot); the
//                    return value of the per-cell counter atomic is the point's rank     12 B/pt + table
//   (scan)           exclusive scan of the table's counters -> cell start offsets
//   scatter_kernel   cell-ordered float4 copy (x, y, z, original index)                  28 B/pt
//   union_kernel     one thread per point: own cell (later positions only) + the 13 forward
//                    neighbour cells (:65-82); hits are queued per warp and united together by a
//                    lock-free union-find over cell-sorted positions with randomised linking
//   roots / labels   roots compressed, per root the smallest original index -> label[i]
// The host side of the entry point turns the labels into the reference's output order (size
// descending, then first index ascending, indices ascending): one counting pass over n labels.
// A batch (frames back to back) runs the insert and union kernels with a frame axis and builds the same order on the
// device with two stable radix sorts (euclidean_cluster_batch_dev, at the end of this file).
#include "pcr_internal.cuh"

#include <algorithm>

namespace pcr {

namespace {

constexpr uint32_t kEmptySlot = 0xffffffffu;

// euclidean_cluster.rs:55-61: (v * inv_r).floor() as i32 -- cvt.rmi.s32.f32 rounds down, saturates and
// maps NaN to 0, exactly like Rust's `as i32` after floor()
__device__ __forceinline__ int ref_cell(float v, float inv_r) { return __float2int_rd(__fmul_rn(v, inv_r)); }

// kFrames (batch): the cell key is (frame, kx, ky, kz).  The frames of a drive share their geometry, so without the frame
// the copies of one cell in 100 frames would all land on one probe chain.
template <bool kFrames>
__device__ __forceinline__ uint32_t hash_cell(int kx, int ky, int kz, uint32_t frame, uint32_t mask) {
    unsigned long long k = ((unsigned long long)(uint32_t)kx << 32) | (uint32_t)ky;
    k ^= (unsigned long long)(uint32_t)kz * 0x9e3779b97f4a7c15ull;
    if (kFrames) k ^= (unsigned long long)frame * 0xd6e8feb86659fd93ull;
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return (uint32_t)k & mask;
}

// The hash table stores, per occupied slot, the index of ONE point of that cell (its representative):
// a full i32 x 3 key does not fit a single CAS word, the representative does, and the key is
// recomputed from its coordinates whenever two cells have to be told apart.  No spinning, exact for
// every key the reference can form (including the saturated keys of far-away points).
// kFrames (batch): frame f = points [frame_off[f], frame_off[f+1]); a representative of another frame is another cell.
// The single call leaves frame_off / n_frames unset.
template <bool kFrames>
__global__ void __launch_bounds__(256) cluster_insert_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                             const float *__restrict__ z, size_t n, float inv_r,
                                                             uint32_t *__restrict__ rep, uint32_t mask, uint32_t *__restrict__ count,
                                                             uint32_t *__restrict__ slot_of, uint32_t *__restrict__ rank_of,
                                                             const uint32_t *__restrict__ frame_off, int n_frames) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float px = x[i], py = y[i], pz = z[i];
    if (!finite3(px, py, pz)) {  // :114-116
        slot_of[i] = kEmptySlot;
        return;
    }
    uint32_t f = 0, fb = 0, fe = 0;
    if (kFrames) {
        f = (uint32_t)frame_of(frame_off, n_frames, (uint32_t)i);
        fb = frame_off[f];
        fe = frame_off[f + 1];
    }
    const int kx = ref_cell(px, inv_r), ky = ref_cell(py, inv_r), kz = ref_cell(pz, inv_r);
    uint32_t h = hash_cell<kFrames>(kx, ky, kz, f, mask);
    for (;;) {
        const uint32_t old = atomicCAS(&rep[h], kEmptySlot, (uint32_t)i);
        if (old == kEmptySlot) break;  // this point now represents the cell
        if ((!kFrames || (old >= fb && old < fe)) && ref_cell(x[old], inv_r) == kx && ref_cell(y[old], inv_r) == ky &&
            ref_cell(z[old], inv_r) == kz)
            break;
        h = (h + 1) & mask;
    }
    slot_of[i] = h;
    rank_of[i] = atomicAdd(&count[h], 1u);
}

__global__ void __launch_bounds__(256) cluster_scatter_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                              const float *__restrict__ z, size_t n,
                                                              const uint32_t *__restrict__ start, const uint32_t *__restrict__ slot_of,
                                                              const uint32_t *__restrict__ rank_of, float4 *__restrict__ cpts,
                                                              uint32_t *__restrict__ cslot) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = slot_of[i];
    if (s == kEmptySlot) return;
    const uint32_t pos = start[s] + rank_of[i];
    cpts[pos] = make_float4(x[i], y[i], z[i], __uint_as_float((uint32_t)i));
    cslot[pos] = s;
}

// Lock-free union-find over the CELL-SORTED positions (neighbours in space are neighbours in the
// parent array, so the walks stay in L1/L2 lines the pair loop has just touched); the root
// with the smaller PRIORITY wins.  Priorities only ever decrease along a walk, so neither the racy path-halving store nor
// a stale cached read can close a cycle or leave the component: a stale parent is still a member of
// the same tree.  Only the CAS decides a link, and it sees the true value.
__device__ __forceinline__ uint32_t uf_find(volatile uint32_t *parent, uint32_t v) {
    for (;;) {
        const uint32_t p = parent[v];
        if (p == v) return v;
        const uint32_t gp = parent[p];
        if (gp != p) parent[v] = gp;
        v = p;
    }
}

// Link order: a pseudo-random priority of the position, not the position itself.  Positions are in
// cell order, so "smaller position wins" builds chains as long as a row of cells (measured: 9.5 ms for
// the union kernel); with random priorities the expected depth is logarithmic, as in randomised linking.
__device__ __forceinline__ uint32_t uf_prio(uint32_t v) {
    v *= 0x9e3779b1u;
    v ^= v >> 15;
    v *= 0x85ebca77u;
    v ^= v >> 13;
    return v;
}
__device__ __forceinline__ bool uf_before(uint32_t a, uint32_t b) {  // a becomes (stays) the root when linked with b
    const uint32_t pa = uf_prio(a), pb = uf_prio(b);
    return pa != pb ? pa < pb : a < b;
}

// one edge: link the trees of positions a and b (exact walks with halving, CAS decides)
__device__ __forceinline__ void uf_unite(uint32_t *parent, uint32_t a, uint32_t b) {
    if (parent[a] == parent[b]) return;  // already hanging under the same node: the common case once components have formed
    uint32_t ra = uf_find(parent, a), rb = uf_find(parent, b);
    while (ra != rb) {
        const bool a_first = uf_before(ra, rb);
        const uint32_t lo = a_first ? ra : rb, hi = a_first ? rb : ra;
        if (atomicCAS(&parent[hi], hi, lo) == hi) return;  // hi was still a root: linked under the one that comes first
        ra = uf_find(parent, ra);
        rb = uf_find(parent, rb);
    }
}

__constant__ int kHalfOff[13][3] = {{1, 0, 0},  {1, 1, 0},   {1, -1, 0}, {1, 0, 1}, {1, 0, -1}, {1, 1, 1}, {1, 1, -1},
                                    {1, -1, 1}, {1, -1, -1}, {0, 1, 0},  {0, 1, 1}, {0, 1, -1}, {0, 0, 1}};  // :65-82

constexpr int kUnionWarps = 4;

// One thread per point walks its own cell (later positions only, :145) and the 13 forward neighbour
// cells.  The pair test is cheap and regular; the union that follows a hit is a serial pointer walk that
// different lanes reach at different times -- executed in place it ran with 3.5 of 32 lanes active
// (ncu, 191 M warp instructions, 2.8 ms on the 122 K frame).  So hits are only QUEUED (warp-aggregated
// push into shared memory) and the warp drains the queue together, one edge per lane.
// kFrames (batch): the neighbour cells are looked up in the point's own frame (as in cluster_insert_kernel).  A cell
// never spans two frames, so no pair crosses frames and the union-find is the single call's.
template <bool kFrames>
__global__ void __launch_bounds__(32 * kUnionWarps) cluster_union_kernel(const float4 *__restrict__ cpts, const uint32_t *__restrict__ cslot,
                                                                         uint32_t m_bound, const float *__restrict__ x,
                                                                         const float *__restrict__ y, const float *__restrict__ z,
                                                                         const uint32_t *__restrict__ rep, uint32_t mask,
                                                                         const uint32_t *__restrict__ start, float inv_r, float r2,
                                                                         uint32_t *parent /* by position */,
                                                                         const uint32_t *__restrict__ frame_off, int n_frames) {
    __shared__ uint2 queue[kUnionWarps][64];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m = min(m_bound, start[mask + 1]);  // start[T] = number of finite points
    const bool live = t < m;
    if (!__any_sync(PCR_FULL, live)) return;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t s = 0;
    if (live) {
        a = cpts[t];
        s = cslot[t];
    }
    int qn = 0;  // entries in this warp's queue (warp-uniform)
    auto drain = [&](int keep_below) {
        while (qn > keep_below) {
            const int take = min(qn, 32);
            uint2 e = make_uint2(0, 0);
            if (lane < take) e = queue[w][qn - take + lane];
            __syncwarp();
            if (lane < take) uf_unite(parent, e.x, e.y);
            qn -= take;
            __syncwarp();
        }
    };
    auto scan = [&](uint32_t b, uint32_t e) {  // warp-uniform loop, per-lane ranges; the pair test of :147-151
        for (uint32_t j = b;; j++) {
            const bool act = j < e;
            if (!__any_sync(PCR_FULL, act)) break;
            bool hit = false;
            if (act) {
                const float4 p = __ldg(&cpts[j]);
                hit = dist2_exact(a.x, a.y, a.z, p.x, p.y, p.z) <= r2;
            }
            const unsigned hm = __ballot_sync(PCR_FULL, hit);
            if (hm) {
                if (hit) queue[w][qn + __popc(hm & ((1u << lane) - 1u))] = make_uint2(t, j);
                qn += __popc(hm);
                __syncwarp();
                if (qn >= 32) drain(31);
            }
        }
    };
    scan(live ? t + 1 : 0, live ? start[s + 1] : 0);  // own cell: every unordered pair once (:145)
    const int kx = ref_cell(a.x, inv_r), ky = ref_cell(a.y, inv_r), kz = ref_cell(a.z, inv_r);
    uint32_t f = 0, fb = 0, fe = 0;
    if (kFrames && live) {
        f = (uint32_t)frame_of(frame_off, n_frames, __float_as_uint(a.w));
        fb = frame_off[f];
        fe = frame_off[f + 1];
    }
#pragma unroll 1
    for (int o = 0; o < 13; o++) {
        uint32_t b = 0, e = 0;
        if (live) {
            // cx + dx on i32 (wrapping, as in a release build of the reference; only saturated keys get there)
            const int nx = (int)((uint32_t)kx + (uint32_t)kHalfOff[o][0]), ny = (int)((uint32_t)ky + (uint32_t)kHalfOff[o][1]);
            const int nz = (int)((uint32_t)kz + (uint32_t)kHalfOff[o][2]);
            uint32_t h = hash_cell<kFrames>(nx, ny, nz, f, mask);
            for (;;) {
                const uint32_t r = __ldg(&rep[h]);
                if (r == kEmptySlot) break;
                if ((!kFrames || (r >= fb && r < fe)) && ref_cell(__ldg(&x[r]), inv_r) == nx && ref_cell(__ldg(&y[r]), inv_r) == ny &&
                    ref_cell(__ldg(&z[r]), inv_r) == nz) {
                    b = start[h];
                    e = start[h + 1];
                    break;
                }
                h = (h + 1) & mask;
            }
        }
        scan(b, e);
    }
    drain(0);
}

__global__ void __launch_bounds__(256) cluster_init_parent_kernel(uint32_t *__restrict__ parent, uint32_t *__restrict__ min_idx, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    parent[i] = (uint32_t)i;
    min_idx[i] = 0xffffffffu;
}

// root position of every finite point (parents fully compressed), and per root the smallest ORIGINAL index
__global__ void __launch_bounds__(256) cluster_roots_kernel(uint32_t *__restrict__ parent, const float4 *__restrict__ cpts, uint32_t m_bound,
                                                            const uint32_t *__restrict__ start, uint32_t mask, uint32_t *__restrict__ min_idx) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < m_bound && t < start[mask + 1];
    const unsigned lm = __ballot_sync(PCR_FULL, live);
    if (!live) return;
    const uint32_t r = uf_find(parent, t);
    parent[t] = r;
    // one atomic per distinct root in the warp (a 108 K-point ground plane is ONE root: 79 us of
    // same-address atomics without this)
    const unsigned peers = __match_any_sync(lm, r);
    const uint32_t mn = __reduce_min_sync(peers, __float_as_uint(cpts[t].w));
    if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicMin(&min_idx[r], mn);
}

__global__ void __launch_bounds__(256) cluster_labels_kernel(const uint32_t *__restrict__ parent, const uint32_t *__restrict__ min_idx,
                                                             const uint32_t *__restrict__ start, const uint32_t *__restrict__ slot_of,
                                                             const uint32_t *__restrict__ rank_of, size_t n, uint32_t *__restrict__ labels) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = slot_of[i];
    if (s == kEmptySlot) {  // non-finite point: its own component (:164-168)
        labels[i] = (uint32_t)i;
        return;
    }
    const uint32_t pos = start[s] + rank_of[i];
    labels[i] = min_idx[parent[parent[pos]]];  // parent[pos] is a root after cluster_roots_kernel (or one step from it)
}

}  // namespace

// labels[i] = smallest index of the connected component of point i (non-finite points: i itself).
// Preconditions (checked by the callers): n > 0, threshold > 0 or NaN.  No host round trip.
// d_frame_off (batch, device, n_frames + 1): the points are frames back to back and no component crosses a frame;
// labels stay global indices.
int cluster_labels_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, float threshold, uint32_t *d_labels,
                       const uint32_t *d_frame_off, int n_frames) {
    if (n > 0x3fffffffull) return fail(ctx, PCR_ERR_UNSUPPORTED, "euclidean_cluster: clouds above 2^30 points are not supported");
    cudaStream_t st = ctx->stream;
    TimeScope ts(ctx, kTagOther);
    const float inv_r = 1.0f / threshold;    // :107
    const float r2 = threshold * threshold;  // :108
    uint32_t T = 256;
    while (T < 2u * (uint32_t)n) T <<= 1;
    // scratch: cpts[n] | rep[T] | count[T+1] | slot_of[n] | rank_of[n] | cslot[n] | parent[n] | min_idx[n]
    const size_t need = sizeof(float4) * n + sizeof(uint32_t) * (2 * (size_t)T + 1 + 5 * n) + 256;
    PCR_TRY(ensure(ctx, ctx->b_table, need));  // (b_misc2 is the scan's own scratch)
    char *p = (char *)ctx->b_table.p;
    float4 *cpts = (float4 *)p;
    p += sizeof(float4) * n;
    uint32_t *rep = (uint32_t *)p;
    p += sizeof(uint32_t) * T;
    uint32_t *count = (uint32_t *)p;
    p += sizeof(uint32_t) * ((size_t)T + 1);
    uint32_t *slot_of = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *rank_of = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *cslot = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *parent = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *min_idx = (uint32_t *)p;
    PCR_CUDA(ctx, cudaMemsetAsync(rep, 0xff, sizeof(uint32_t) * T, st));
    PCR_CUDA(ctx, cudaMemsetAsync(count, 0, sizeof(uint32_t) * ((size_t)T + 1), st));
    const unsigned nb = (unsigned)((n + 255) / 256);
    cluster_init_parent_kernel<<<nb, 256, 0, st>>>(parent, min_idx, n);
    PCR_LAUNCH_CHECK(ctx);
    if (d_frame_off)
        cluster_insert_kernel<true><<<nb, 256, 0, st>>>(dx, dy, dz, n, inv_r, rep, T - 1, count, slot_of, rank_of, d_frame_off, n_frames);
    else
        cluster_insert_kernel<false><<<nb, 256, 0, st>>>(dx, dy, dz, n, inv_r, rep, T - 1, count, slot_of, rank_of, nullptr, 1);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(exclusive_scan_u32_dev(ctx, count, (size_t)T + 1));
    cluster_scatter_kernel<<<nb, 256, 0, st>>>(dx, dy, dz, n, count, slot_of, rank_of, cpts, cslot);
    PCR_LAUNCH_CHECK(ctx);
    const unsigned nbu = (unsigned)((n + 32 * kUnionWarps - 1) / (32 * kUnionWarps));
    if (d_frame_off)
        cluster_union_kernel<true><<<nbu, 32 * kUnionWarps, 0, st>>>(cpts, cslot, (uint32_t)n, dx, dy, dz, rep, T - 1, count, inv_r, r2, parent,
                                                                     d_frame_off, n_frames);
    else
        cluster_union_kernel<false><<<nbu, 32 * kUnionWarps, 0, st>>>(cpts, cslot, (uint32_t)n, dx, dy, dz, rep, T - 1, count, inv_r, r2, parent,
                                                                      nullptr, 1);
    PCR_LAUNCH_CHECK(ctx);
    cluster_roots_kernel<<<nb, 256, 0, st>>>(parent, cpts, (uint32_t)n, count, T - 1, min_idx);
    PCR_LAUNCH_CHECK(ctx);
    cluster_labels_kernel<<<nb, 256, 0, st>>>(parent, min_idx, count, slot_of, rank_of, n, d_labels);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

// Labels (root = smallest index of the component) -> the reference's output (:164-186): clusters
// with min_size <= size <= max_size, size descending then first index ascending, indices ascending.
size_t clusters_from_labels(const uint32_t *labels, size_t n, size_t min_size, size_t max_size, uint32_t *offsets, uint32_t *indices,
                            std::vector<uint32_t> &scratch) {
    scratch.assign(2 * n, 0);
    uint32_t *size = scratch.data(), *slot = scratch.data() + n;
    for (size_t i = 0; i < n; i++) size[labels[i]]++;
    std::vector<std::pair<uint32_t, uint32_t>> comps;  // (size, root); root == first index
    for (size_t r = 0; r < n; r++)
        if (size[r] && size[r] >= min_size && size[r] <= max_size) comps.emplace_back(size[r], (uint32_t)r);
    std::sort(comps.begin(), comps.end(), [](const std::pair<uint32_t, uint32_t> &a, const std::pair<uint32_t, uint32_t> &b) {
        return a.first != b.first ? a.first > b.first : a.second < b.second;
    });
    for (size_t r = 0; r < n; r++) slot[r] = 0xffffffffu;
    offsets[0] = 0;
    for (size_t c = 0; c < comps.size(); c++) {
        slot[comps[c].second] = offsets[c];
        offsets[c + 1] = offsets[c] + comps[c].first;
    }
    for (size_t i = 0; i < n; i++)
        if (slot[labels[i]] != 0xffffffffu) indices[slot[labels[i]]++] = (uint32_t)i;
    return comps.size();
}

// ---- batch: the reference's output order, built on the device ---------------------------------------------------
namespace {

// size[r] = points of the component whose smallest index is r (0 where r is not a root); one atomic per root and warp
__global__ void __launch_bounds__(256) cluster_sizes_kernel(const uint32_t *__restrict__ labels, size_t n, uint32_t *__restrict__ size) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;
    const unsigned lm = __ballot_sync(PCR_FULL, live);
    if (!live) return;
    const uint32_t r = labels[i];
    const unsigned peers = __match_any_sync(lm, r);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&size[r], (uint32_t)__popc(peers));
}

// flag[r] = 1 iff component r is kept (lo >= 1, so a non-root never is); flag[n] = 0 is the slot of the total
__global__ void __launch_bounds__(256) cluster_keep_kernel(const uint32_t *__restrict__ size, size_t n, uint32_t lo, uint32_t hi,
                                                           uint32_t *__restrict__ flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    flag[i] = (i < n && size[i] >= lo && size[i] <= hi) ? 1u : 0u;
}

// kept component r (cid = exclusive scan of the flags, so kept components are numbered in first-index order, which is
// frame order) -> sort pair ((frame << size_bits) | (cap - size), r): one stable sort gives size descending, then first
// index ascending, inside every frame
__global__ void __launch_bounds__(256) cluster_comp_keys_kernel(const uint32_t *__restrict__ size, const uint32_t *__restrict__ cid, size_t n,
                                                                const uint32_t *__restrict__ frame_off, int n_frames, int size_bits,
                                                                uint32_t cap, unsigned long long *__restrict__ keys,
                                                                uint32_t *__restrict__ vals) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || cid[i + 1] == cid[i]) return;
    const unsigned long long f = (unsigned long long)frame_of(frame_off, n_frames, (uint32_t)i);
    keys[cid[i]] = (f << size_bits) | (unsigned long long)(cap - size[i]);
    vals[cid[i]] = (uint32_t)i;
}

// sorted cluster c: its size into offsets[c] (scanned into the CSR offsets next; offsets[k] = 0 becomes the total) and
// crank[root] = c
__global__ void __launch_bounds__(256) cluster_rank_kernel(const uint32_t *__restrict__ roots, uint32_t k, const uint32_t *__restrict__ size,
                                                           uint32_t *__restrict__ offsets, uint32_t *__restrict__ crank) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > k) return;
    if (c == k) {
        offsets[k] = 0;
        return;
    }
    const uint32_t r = roots[c];
    offsets[c] = size[r];
    crank[r] = c;
}

// point i -> sort pair (rank of its cluster, i); points of components that were filtered out get k and sort last
__global__ void __launch_bounds__(256) cluster_point_keys_kernel(const uint32_t *__restrict__ labels, const uint32_t *__restrict__ cid,
                                                                 const uint32_t *__restrict__ crank, size_t n, uint32_t k,
                                                                 unsigned long long *__restrict__ keys, uint32_t *__restrict__ vals) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = labels[i];
    keys[i] = cid[r + 1] != cid[r] ? crank[r] : k;
    vals[i] = (uint32_t)i;
}

// indices[j] = frame-local index of the j-th point in cluster order, j < offsets[k] (the number of clustered points)
__global__ void __launch_bounds__(256) cluster_emit_kernel(const uint32_t *__restrict__ sorted, const uint32_t *__restrict__ total, size_t n,
                                                           const uint32_t *__restrict__ frame_off, int n_frames, uint32_t *__restrict__ indices) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n || j >= *total) return;
    const uint32_t v = sorted[j];
    indices[j] = v - frame_off[frame_of(frame_off, n_frames, v)];
}

// cluster_offsets[f] = first cluster of frame f in sorted order, [n_frames] = k: thread c writes the entries of the
// frames that start between sorted clusters c - 1 and c (frames without a cluster included)
__global__ void __launch_bounds__(256) cluster_frame_starts_kernel(const unsigned long long *__restrict__ keys, uint32_t k, int size_bits,
                                                                   int n_frames, uint32_t *__restrict__ out) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > k) return;
    const int hi = c < k ? (int)(keys[c] >> size_bits) : n_frames;
    const int lo = c > 0 ? (int)(keys[c - 1] >> size_bits) : -1;
    for (int f = lo + 1; f <= hi; f++) out[f] = c;
}

// global smallest index -> index inside the point's frame
__global__ void __launch_bounds__(256) cluster_local_labels_kernel(uint32_t *__restrict__ labels, size_t n, const uint32_t *__restrict__ frame_off,
                                                                   int n_frames) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    labels[i] -= frame_off[frame_of(frame_off, n_frames, (uint32_t)i)];
}

// Global labels of every frame into *labels (nullptr: into b_misc).  Scratch of a batch (b_misc): frame offsets
// u32[F + 1] | cluster offsets u32[F + 1] [| labels u32[n]]
int batch_labels(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, int F, float threshold,
                 uint32_t **labels, uint32_t **d_off, uint32_t **d_cofs) {
    const size_t n = (size_t)frame_offsets[F];
    PCR_TRY(ensure(ctx, ctx->b_misc, sizeof(uint32_t) * (2 * ((size_t)F + 1) + (*labels ? 0 : n))));
    *d_off = (uint32_t *)ctx->b_misc.p;
    *d_cofs = *d_off + F + 1;
    if (!*labels) *labels = *d_cofs + F + 1;
    std::vector<uint32_t> h_off(F + 1);
    for (int f = 0; f <= F; f++) h_off[f] = (uint32_t)frame_offsets[f];
    // (pageable source: the copy has taken the bytes when it returns)
    PCR_CUDA(ctx, cudaMemcpyAsync(*d_off, h_off.data(), sizeof(uint32_t) * (F + 1), cudaMemcpyHostToDevice, ctx->stream));
    return cluster_labels_dev(ctx, dx, dy, dz, n, threshold, *labels, *d_off, F);
}

}  // namespace

// pcr_cluster_labels_batch_dev: frame-local labels (arguments checked by the caller, n > 0)
int cluster_labels_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                             float threshold, uint32_t *d_labels) {
    const int F = (int)n_frames;
    const size_t n = (size_t)frame_offsets[F];
    uint32_t *d_off, *d_cofs;
    PCR_TRY(batch_labels(ctx, dx, dy, dz, frame_offsets, F, threshold, &d_labels, &d_off, &d_cofs));
    cluster_local_labels_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_labels, n, d_off, F);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

// euclidean_cluster of every frame of a batch (arguments checked by the caller: n > 0, threshold > 0 or NaN, min_size > 0).
// d_offsets (n + 1) and d_indices (n) receive the CSR of all frames, frame f's clusters being
// [cluster_offsets[f], cluster_offsets[f+1]) (host, n_frames + 1), indices frame-local.  The order inside a frame is
// clusters_from_labels' (size descending, then first index ascending, indices ascending), built with two stable sorts
// and no host pass over the points.  Two host round trips: the number of kept components, then the frame starts with
// the number of clustered points (*total).
int euclidean_cluster_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                                float threshold, size_t min_size, size_t max_size, uint32_t *d_offsets, uint32_t *d_indices,
                                uint64_t *cluster_offsets, size_t *total) {
    const int F = (int)n_frames;
    const size_t n = (size_t)frame_offsets[F];
    cudaStream_t st = ctx->stream;
    for (int f = 0; f <= F; f++) cluster_offsets[f] = 0;
    *total = 0;
    uint32_t *labels = nullptr, *d_off, *d_cofs;
    PCR_TRY(batch_labels(ctx, dx, dy, dz, frame_offsets, F, threshold, &labels, &d_off, &d_cofs));
    TimeScope ts(ctx, kTagOther);
    // scratch (b_table, free again once the labels are written): keys A/B u64[n] | size u32[n] | cid u32[n + 1] |
    // crank u32[n] | vals A/B u32[n] | hist
    const size_t hist_words = radix_sort_hist_words(n);
    PCR_TRY(ensure(ctx, ctx->b_table, sizeof(unsigned long long) * 2 * n + sizeof(uint32_t) * (6 * n + 1 + hist_words) + 256));
    char *p = (char *)ctx->b_table.p;
    unsigned long long *kA = (unsigned long long *)p, *kB = kA + n;
    uint32_t *size = (uint32_t *)(kB + n), *cid = size + n, *crank = cid + n + 1, *vA = crank + n, *vB = vA + n, *hist = vB + n;
    PCR_TRY(ensure_pinned(ctx, std::max<size_t>(4096, sizeof(uint32_t) * ((size_t)F + 2))));
    uint32_t *mail = (uint32_t *)ctx->pinned;
    const unsigned nb = (unsigned)((n + 255) / 256);
    PCR_CUDA(ctx, cudaMemsetAsync(size, 0, sizeof(uint32_t) * n, st));
    cluster_sizes_kernel<<<nb, 256, 0, st>>>(labels, n, size);
    PCR_LAUNCH_CHECK(ctx);
    // sizes are <= n < 2^30: clamping the bounds there keeps the filter exact
    const uint32_t lo = (uint32_t)std::min<size_t>(min_size, 0x7fffffffu), hi = (uint32_t)std::min<size_t>(max_size, 0x7fffffffu);
    cluster_keep_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(size, n, lo, hi, cid);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(exclusive_scan_u32_dev(ctx, cid, n + 1));
    PCR_CUDA(ctx, cudaMemcpyAsync(mail, cid + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PCR_MARK("cluster batch: wait for the number of clusters");
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t k = *mail;
    if (k == 0) {
        PCR_CUDA(ctx, cudaMemsetAsync(d_offsets, 0, sizeof(uint32_t), st));
        PCR_CUDA(ctx, cudaStreamSynchronize(st));
        return PCR_OK;
    }
    // clusters: (frame, size descending) stably over first-index order
    const uint32_t cap = std::min<uint32_t>(hi, (uint32_t)n);
    const int size_bits = bits_for((uint64_t)cap), frame_bits = bits_for((uint64_t)F);
    cluster_comp_keys_kernel<<<nb, 256, 0, st>>>(size, cid, n, d_off, F, size_bits, cap, kA, vA);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, k, frame_bits + size_bits, hist));
    cluster_rank_kernel<<<(k + 1 + 255) / 256, 256, 0, st>>>(vA, k, size, d_offsets, crank);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(exclusive_scan_u32_dev(ctx, d_offsets, (size_t)k + 1));
    cluster_frame_starts_kernel<<<(k + 1 + 255) / 256, 256, 0, st>>>(kA, k, size_bits, F, d_cofs);
    PCR_LAUNCH_CHECK(ctx);
    // points: stably by cluster rank over index order -> ascending indices inside every cluster (the pair buffers are
    // free again: the two kernels above are the last readers of the cluster sort)
    kA = (unsigned long long *)p;
    kB = kA + n;
    vA = crank + n;
    vB = vA + n;
    cluster_point_keys_kernel<<<nb, 256, 0, st>>>(labels, cid, crank, n, k, kA, vA);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, n, bits_for((uint64_t)k + 1), hist));
    cluster_emit_kernel<<<nb, 256, 0, st>>>(vA, d_offsets + k, n, d_off, F, d_indices);
    PCR_LAUNCH_CHECK(ctx);
    PCR_CUDA(ctx, cudaMemcpyAsync(mail, d_cofs, sizeof(uint32_t) * (F + 1), cudaMemcpyDeviceToHost, st));
    PCR_CUDA(ctx, cudaMemcpyAsync(mail + F + 1, d_offsets + k, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PCR_MARK("cluster batch: wait for the frame starts");
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    for (int f = 0; f <= F; f++) cluster_offsets[f] = mail[f];
    *total = mail[F + 1];
    return PCR_OK;
}

}  // namespace pcr
