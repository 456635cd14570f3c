// voxel.cu -- voxel_downsample (crates/filters/src/voxel_downsample.rs:12-65) on the GPU, and the
// stable LSD radix sort it is built on.
//
// The reference accumulates, per voxel key (floor(p / voxel) as i32, :32-36), the f32 sums of x, y, z
// in INPUT order (:38-42: sequential f32 additions, so the order is part of the result), divides by the
// count and emits the voxels in ascending key order (:49-50).  One stable sort of (packed key, index)
// pairs gives both orders at once: equal keys keep their input order, and the runs come out in key
// order.
//
//   vox_range_kernel   key range of the finite points (warp redux + atomics)             12 B/pt
//   vox_pack_kernel    packed u64 key per point (non-finite points sort last)            12 + 12 B/pt
//   radix passes       8 bits per pass over the significant bits only (KITTI frame at 5 cm: 29 bits,
//                      4 passes); one WARP owns a tile of 256 consecutive pairs and walks it in order,
//                      __match_any_sync ranks equal digits inside a round of 32, running per-digit
//                      offsets in shared memory carry the order across rounds: stable by construction
//   vox_heads_kernel   run heads -> voxel ids (exclusive scan) -> run starts
//   vox_mean_kernel    one thread per voxel: the reference's sequential f32 sums, then / count
// If the key box needs more than 63 bits (a far outlier with a tiny voxel) the same sort runs three
// times on 32-bit axis keys (z, then y, then x): stable LSD over the axes.
// Fast path (the usual case): when the (kx, ky) rectangle fits a dense table, ONE counting sort by column and a
// per-column sort by (kz, index) replace the radix passes (vox_col_* kernels below).
#include "pcr_internal.cuh"

#include <algorithm>

namespace pcr {

namespace {

constexpr int kSortRounds = 8;                   // rounds of 32 pairs per warp tile (more tiles = more warps in flight)
constexpr int kSortTile = 32 * kSortRounds;      // 256 pairs
constexpr int kSortWarps = 4;                    // warps (tiles) per block

// Head of the column path's scratch block: zeroed together with the column counters by ONE memset, read back by ONE
// copy.  The box is kept as maxima only (mn_c = complement of the ordered encoding), so that zero is its identity.
struct VoxHeader {
    unsigned mn_c[3], mx[3];  // bounding box of the cloud written (f32_ordered encodings)
    unsigned count;           // finite points written
    unsigned outside;         // a point fell outside a guessed key box
    unsigned total;           // voxels written
    unsigned tall;            // a column holds more members than one thread should sort: the caller takes the radix path
    unsigned pad[6];
};
// Members one thread sorts in place.  A coarse voxel, a wall or a dense small-footprint cloud can put 10^5..10^7 points
// into one column; a serial sort of that in global memory would take seconds, the radix path sorts it in 4 passes.
constexpr uint32_t kTallColumn = 256;
constexpr uint32_t kLocalColumn = 32;  // columns up to this many members are sorted in local memory
static_assert(sizeof(VoxHeader) == 64, "header layout");

struct VoxRange {
    int mn[3];
    int mx[3];
    unsigned finite;
};

// voxel_downsample.rs:32-36: (p / voxel).floor() as i32 -- IEEE division, round down, saturate, NaN -> 0
__device__ __forceinline__ int vox_cell(float v, float voxel) { return __float2int_rd(__fdiv_rn(v, voxel)); }

__global__ void vox_init_kernel(VoxRange *r, int n_ranges) {
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < n_ranges; f += gridDim.x * blockDim.x) {
        for (int a = 0; a < 3; a++) {
            r[f].mn[a] = 2147483647;
            r[f].mx[a] = -2147483647 - 1;
        }
        r[f].finite = 0;
    }
}

// frame_off == nullptr: the range of the n points.  Otherwise (batch) frame blockIdx.y = points [frame_off[y],
// frame_off[y + 1]) and its range goes to r[y]: a block never crosses a frame, so the reductions below stay per frame.
__global__ void __launch_bounds__(256) vox_range_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                        const float *__restrict__ z, const uint32_t *__restrict__ frame_off,
                                                        size_t n, float voxel, VoxRange *r) {
    int mn[3] = {2147483647, 2147483647, 2147483647}, mx[3] = {-2147483647 - 1, -2147483647 - 1, -2147483647 - 1};
    unsigned cnt = 0;
    size_t b = 0, e = n;
    if (frame_off) {
        b = frame_off[blockIdx.y];
        e = frame_off[blockIdx.y + 1];
        r += blockIdx.y;
    }
    for (size_t i = b + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < e; i += (size_t)gridDim.x * blockDim.x) {
        const float px = x[i], py = y[i], pz = z[i];
        if (!finite3(px, py, pz)) continue;  // :28-30
        const int k[3] = {vox_cell(px, voxel), vox_cell(py, voxel), vox_cell(pz, voxel)};
        for (int a = 0; a < 3; a++) {
            mn[a] = min(mn[a], k[a]);
            mx[a] = max(mx[a], k[a]);
        }
        cnt++;
    }
    for (int a = 0; a < 3; a++) {
        mn[a] = __reduce_min_sync(PCR_FULL, mn[a]);
        mx[a] = __reduce_max_sync(PCR_FULL, mx[a]);
    }
    cnt = __reduce_add_sync(PCR_FULL, cnt);
    // block-level combine first: seven same-address atomics per WARP cost 20 us on the 122 K frame
    __shared__ int smn[3][8], smx[3][8];
    __shared__ unsigned scnt[8];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        for (int a = 0; a < 3; a++) {
            smn[a][w] = mn[a];
            smx[a][w] = mx[a];
        }
        scnt[w] = cnt;
    }
    __syncthreads();
    if (w == 0) {
        const bool in = lane < (int)(blockDim.x >> 5);
        for (int a = 0; a < 3; a++) {
            mn[a] = __reduce_min_sync(PCR_FULL, in ? smn[a][lane] : 2147483647);
            mx[a] = __reduce_max_sync(PCR_FULL, in ? smx[a][lane] : -2147483647 - 1);
        }
        cnt = __reduce_add_sync(PCR_FULL, in ? scnt[lane] : 0u);
        if (lane == 0 && cnt) {
            for (int a = 0; a < 3; a++) {
                atomicMin(&r->mn[a], mn[a]);
                atomicMax(&r->mx[a], mx[a]);
            }
            atomicAdd(&r->finite, cnt);
        }
    }
}

// axis < 0: packed key ((kx - mn0) << s0) | ((ky - mn1) << s1) | (kz - mn2); axis 0..2: that axis alone
// (biased to unsigned).  Non-finite points get `last`, above every real key.
// Batch (fr != nullptr): the point's frame f (frame_of over frame_off) takes the biases from its own range fr[f] and
// leads the packed key, (f << fshift) | ...; axis 3 is the frame id alone.
__global__ void __launch_bounds__(256) vox_pack_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                       const float *__restrict__ z, const uint32_t *order, size_t n,
                                                       float voxel, int axis, int mn0, int mn1, int mn2, int s0, int s1,
                                                       unsigned long long last, unsigned long long *__restrict__ keys,
                                                       uint32_t *vals /* may alias order */, const uint32_t *__restrict__ frame_off,
                                                       int n_frames, const VoxRange *__restrict__ fr, int fshift) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint32_t i = order ? order[t] : (uint32_t)t;
    const float px = x[i], py = y[i], pz = z[i];
    unsigned long long key = last;
    if (finite3(px, py, pz)) {
        const int kx = vox_cell(px, voxel), ky = vox_cell(py, voxel), kz = vox_cell(pz, voxel);
        if (axis < 0) {
            unsigned long long head = 0;
            if (fr) {
                const int f = frame_of(frame_off, n_frames, i);
                mn0 = fr[f].mn[0];
                mn1 = fr[f].mn[1];
                mn2 = fr[f].mn[2];
                head = (unsigned long long)f << fshift;
            }
            key = head | ((unsigned long long)(uint32_t)(kx - mn0) << s0) | ((unsigned long long)(uint32_t)(ky - mn1) << s1) |
                  (unsigned long long)(uint32_t)(kz - mn2);
        } else if (axis == 3) {
            key = (unsigned long long)frame_of(frame_off, n_frames, i);
        } else {
            key = (unsigned long long)((uint32_t)(axis == 0 ? kx : (axis == 1 ? ky : kz)) ^ 0x80000000u);
        }
    }
    keys[t] = key;
    vals[t] = i;
}

// ---- stable LSD radix sort, 8 bits per pass -----------------------------------------------------------
// hist[digit * n_tiles + tile] = number of pairs of `tile` with that digit
__global__ void __launch_bounds__(32 * kSortWarps) sort_hist_kernel(const unsigned long long *__restrict__ keys, size_t n, int shift,
                                                                    uint32_t n_tiles, uint32_t *__restrict__ hist) {
    __shared__ uint32_t cnt[kSortWarps][256];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t tile = blockIdx.x * kSortWarps + w;
    for (int d = lane; d < 256; d += 32) cnt[w][d] = 0;
    __syncwarp();
    if (tile < n_tiles) {
        const size_t base = (size_t)tile * kSortTile;
        for (int r = 0; r < kSortRounds; r++) {
            const size_t i = base + (size_t)r * 32 + lane;
            const bool valid = i < n;
            const unsigned vmask = __ballot_sync(PCR_FULL, valid);
            if (valid) {
                const unsigned d = (unsigned)(keys[i] >> shift) & 255u;
                const unsigned peers = __match_any_sync(vmask, d);
                if (lane == __ffs(peers) - 1) cnt[w][d] += __popc(peers);
            }
            __syncwarp();
        }
        for (int d = lane; d < 256; d += 32) hist[(size_t)d * n_tiles + tile] = cnt[w][d];
    }
}

__global__ void __launch_bounds__(32 * kSortWarps) sort_scatter_kernel(const unsigned long long *__restrict__ keys,
                                                                       const uint32_t *__restrict__ vals, size_t n, int shift,
                                                                       uint32_t n_tiles, const uint32_t *__restrict__ offs,
                                                                       unsigned long long *__restrict__ keys_out,
                                                                       uint32_t *__restrict__ vals_out) {
    __shared__ uint32_t pos[kSortWarps][256];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t tile = blockIdx.x * kSortWarps + w;
    if (tile >= n_tiles) return;
    for (int d = lane; d < 256; d += 32) pos[w][d] = offs[(size_t)d * n_tiles + tile];
    __syncwarp();
    const size_t base = (size_t)tile * kSortTile;
    for (int r = 0; r < kSortRounds; r++) {
        const size_t i = base + (size_t)r * 32 + lane;
        const bool valid = i < n;
        const unsigned vmask = __ballot_sync(PCR_FULL, valid);
        unsigned long long key = 0;
        uint32_t val = 0, dst = 0;
        unsigned d = 0, peers = 0;
        if (valid) {
            key = keys[i];
            val = vals[i];
            d = (unsigned)(key >> shift) & 255u;
            peers = __match_any_sync(vmask, d);
            dst = pos[w][d] + __popc(peers & ((1u << lane) - 1u));  // earlier lanes = earlier input positions
        }
        __syncwarp();
        if (valid && lane == __ffs(peers) - 1) pos[w][d] += __popc(peers);
        __syncwarp();
        if (valid) {
            keys_out[dst] = key;
            vals_out[dst] = val;
        }
    }
}

// ---- runs -> voxels -----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) vox_heads_kernel(const unsigned long long *__restrict__ keys, uint32_t m, uint32_t *__restrict__ flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > m) return;
    flag[i] = (i < m && (i == 0 || keys[i] != keys[i - 1])) ? 1u : 0u;  // flag[m] = 0: slot of the total
}

// the three-pass (z, y, x) fallback has no packed key: heads are compared on the recomputed triple (and, in a batch,
// on the frame: the same voxel of two frames is two voxels)
__global__ void __launch_bounds__(256) vox_heads_triple_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                               const float *__restrict__ z, const uint32_t *__restrict__ vals, uint32_t m,
                                                               float voxel, const uint32_t *__restrict__ frame_off, int n_frames,
                                                               uint32_t *__restrict__ flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > m) return;
    uint32_t f = 0;
    if (i < m) {
        f = 1;
        if (i > 0) {
            const uint32_t a = vals[i], b = vals[i - 1];
            f = (vox_cell(x[a], voxel) != vox_cell(x[b], voxel) || vox_cell(y[a], voxel) != vox_cell(y[b], voxel) ||
                 vox_cell(z[a], voxel) != vox_cell(z[b], voxel) || frame_of(frame_off, n_frames, a) != frame_of(frame_off, n_frames, b))
                    ? 1u
                    : 0u;
        }
    }
    flag[i] = f;
}

// vid = exclusive scan of the head flags (m + 1 entries, vid[m] = number of voxels): position i is a
// head iff vid[i + 1] != vid[i], and then it starts voxel vid[i]
__global__ void __launch_bounds__(256) vox_starts_kernel(const uint32_t *__restrict__ vid, uint32_t m, uint32_t *__restrict__ start) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > m) return;
    if (i == m) {
        start[vid[m]] = m;  // end sentinel of the last voxel
        return;
    }
    if (vid[i + 1] != vid[i]) start[vid[i]] = i;
}

__global__ void __launch_bounds__(128) vox_mean_kernel(const float *__restrict__ x, const float *__restrict__ y, const float *__restrict__ z,
                                                       const uint32_t *__restrict__ vals, const uint32_t *__restrict__ start,
                                                       const uint32_t *__restrict__ n_vox_dev, float *__restrict__ ox,
                                                       float *__restrict__ oy, float *__restrict__ oz) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= *n_vox_dev) return;
    const uint32_t b = start[v], e = start[v + 1];
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (uint32_t i = b; i < e; i++) {  // :38-42, input order (the sort is stable)
        const uint32_t p = vals[i];
        sx = __fadd_rn(sx, x[p]);
        sy = __fadd_rn(sy, y[p]);
        sz = __fadd_rn(sz, z[p]);
    }
    const float denom = (float)(e - b);  // :56
    ox[v] = __fdiv_rn(sx, denom);
    oy[v] = __fdiv_rn(sy, denom);
    oz[v] = __fdiv_rn(sz, denom);
}

// ---- column path: dense (kx, ky) table + per-column sort by (kz, index) -----------------------------------
// When the (kx, ky) key rectangle is small enough for a dense table (the usual case: a 70 m x 50 m frame at
// 5 cm is 1.4 M columns), one counting sort puts every point into its column -- a single pass instead of the
// four radix passes -- and a column rarely holds more than a handful of points, which one thread orders by
// (kz, index) in place.  Columns in table order and kz inside a column give the reference's key order (:49-50);
// index order inside a voxel gives its summation order (:38-42).
__global__ void __launch_bounds__(256) vox_col_count_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                            const float *__restrict__ z, size_t n, float voxel, int mn0, int mn1,
                                                            int mn2, unsigned long long nx, unsigned long long ny,
                                                            unsigned long long nz, uint32_t nyc, int ys, uint32_t *__restrict__ count,
                                                            uint32_t *__restrict__ col_of, uint32_t *__restrict__ rank_of,
                                                            uint32_t *__restrict__ outside) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float px = x[i], py = y[i], pz = z[i];
    if (!finite3(px, py, pz)) {
        col_of[i] = 0xffffffffu;
        return;
    }
    const int kx = vox_cell(px, voxel), ky = vox_cell(py, voxel), kz = vox_cell(pz, voxel);
    // the key box may be a guess (the previous frame's, padded): a point outside it voids the pass
    if ((unsigned long long)((long long)kx - mn0) >= nx || (unsigned long long)((long long)ky - mn1) >= ny ||
        (unsigned long long)((long long)kz - mn2) >= nz) {
        col_of[i] = 0xffffffffu;
        *outside = 1u;
        return;
    }
    const uint32_t col = (uint32_t)(kx - mn0) * nyc + ((uint32_t)(ky - mn1) >> ys);
    col_of[i] = col;
    rank_of[i] = atomicAdd(&count[col], 1u);
}

// member key = (ky mod 2^ys, kz, index): a column spans 2^ys voxels along y, so the y remainder leads
__global__ void __launch_bounds__(256) vox_col_scatter_kernel(const float *__restrict__ y, const float *__restrict__ z, size_t n,
                                                              float voxel, int mn1, int mn2, int ys,
                                                              const uint32_t *__restrict__ start, const uint32_t *__restrict__ col_of,
                                                              const uint32_t *__restrict__ rank_of, unsigned long long *__restrict__ members) {
    PCR_GRID_DEP_SYNC();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t col = col_of[i];
    if (col == 0xffffffffu) return;
    const uint32_t ylo = (uint32_t)(vox_cell(y[i], voxel) - mn1) & ((1u << ys) - 1u);
    const uint32_t hi = (ys ? ylo << (32 - ys) : 0u) | (uint32_t)(vox_cell(z[i], voxel) - mn2);  // kz - mn2 < 2^(32 - ys), checked by the host
    members[start[col] + rank_of[i]] = ((unsigned long long)hi << 32) | (uint32_t)i;
}

// One thread per NON-EMPTY column -- the thread of the point that arrived first in it (rank 0): a 5 cm table over a
// LiDAR frame is more than 90 % empty, so walking the points instead of the table leaves a tenth of the threads and
// none of the table reads.  Orders the column's members by (y remainder, kz, index) and counts its voxels.  The count
// goes to nvox[start of the column in the member array], NOT to a second table over the columns: the member array is
// ordered by column, so an exclusive scan over its n + 1 slots (zeroed with the counters; 0.5 MB) gives the same output
// offsets as a scan over the 1.4 M-entry table did (15.8 -> 6.6 us).
__global__ void __launch_bounds__(256) vox_col_sort_kernel(const uint32_t *__restrict__ col_of, const uint32_t *__restrict__ rank_of,
                                                           size_t n, const uint32_t *__restrict__ start,
                                                           unsigned long long *__restrict__ members, uint32_t *__restrict__ nvox,
                                                           unsigned *__restrict__ tall) {
    PCR_GRID_DEP_SYNC();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t c = col_of[i];
    if (c == 0xffffffffu || rank_of[i] != 0u) return;
    const uint32_t b = start[c], e = start[c + 1], m = e - b;
    if (m > kTallColumn) {  // not a job for one thread: flag it, the host redoes the cloud on the radix path
        *tall = 1u;
        return;
    }
    unsigned long long *a = members + b;
    if (m == 1) {  // (nine columns in ten of a LiDAR frame)
        nvox[b] = 1u;
        return;
    }
    if (m <= kLocalColumn) {
        // A wall or a pedestrian puts 10-30 points in a column.  Sorted in place in global memory every compare of the
        // insertion sort was a dependent L2 round trip (the kernel took as long as its slowest column: 29 us); the column
        // is copied to local memory instead (eight independent loads in flight), sorted there and written back.
        unsigned long long loc[kLocalColumn];
        for (uint32_t j0 = 0; j0 < m; j0 += 8) {
            unsigned long long t[8];
#pragma unroll
            for (int u = 0; u < 8; u++) t[u] = a[min(j0 + u, m - 1)];
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (j0 + u < m) loc[j0 + u] = t[u];
        }
        for (uint32_t i = 1; i < m; i++) {  // insertion sort
            const unsigned long long v = loc[i];
            uint32_t j = i;
            while (j > 0 && loc[j - 1] > v) {
                loc[j] = loc[j - 1];
                j--;
            }
            loc[j] = v;
        }
        uint32_t nv = 1;
        a[0] = loc[0];
        for (uint32_t i = 1; i < m; i++) {
            a[i] = loc[i];
            nv += (uint32_t)(loc[i] >> 32) != (uint32_t)(loc[i - 1] >> 32) ? 1u : 0u;
        }
        nvox[b] = nv;
        return;
    } else {  // heapsort: O(m log m) for the rare tall column (a wall, a whole cloud in one column)
        for (uint32_t s0 = m / 2; s0-- > 0;) {
            uint32_t root = s0;
            for (;;) {
                uint32_t ch = 2 * root + 1;
                if (ch >= m) break;
                if (ch + 1 < m && a[ch] < a[ch + 1]) ch++;
                if (a[root] >= a[ch]) break;
                const unsigned long long t = a[root]; a[root] = a[ch]; a[ch] = t;
                root = ch;
            }
        }
        for (uint32_t end = m - 1; end > 0; end--) {
            const unsigned long long t0 = a[0]; a[0] = a[end]; a[end] = t0;
            uint32_t root = 0;
            for (;;) {
                uint32_t ch = 2 * root + 1;
                if (ch >= end) break;
                if (ch + 1 < end && a[ch] < a[ch + 1]) ch++;
                if (a[root] >= a[ch]) break;
                const unsigned long long t = a[root]; a[root] = a[ch]; a[ch] = t;
                root = ch;
            }
        }
    }
    uint32_t nv = 1;
    for (uint32_t i = 1; i < m; i++) nv += (uint32_t)(a[i] >> 32) != (uint32_t)(a[i - 1] >> 32) ? 1u : 0u;
    nvox[b] = nv;
}

__global__ void __launch_bounds__(256) vox_col_emit_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                           const float *__restrict__ z, const uint32_t *__restrict__ col_of,
                                                           const uint32_t *__restrict__ rank_of, size_t n,
                                                           const uint32_t *__restrict__ start, const uint32_t *__restrict__ vstart,
                                                           const unsigned long long *__restrict__ members, float *__restrict__ ox,
                                                           float *__restrict__ oy, float *__restrict__ oz) {
    PCR_GRID_DEP_SYNC();
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // again the thread of the column's first arrival
    if (t >= n) return;
    const uint32_t c = col_of[t];
    if (c == 0xffffffffu || rank_of[t] != 0u) return;
    const uint32_t b = start[c], e = start[c + 1];
    if (e - b > kTallColumn) return;  // flagged by vox_col_sort_kernel: this pass is void
    // Eight members at a time: their keys, then their coordinates, are independent loads; only the additions are a chain
    // (one member after the other was two dependent L2 round trips per member: 15 us for the tallest column).
    uint32_t v = vstart[b];  // (indexed by the column's first member slot, see vox_col_sort_kernel)
    uint32_t cur = (uint32_t)(members[b] >> 32);
    float sx = 0.f, sy = 0.f, sz = 0.f;
    uint32_t cnt = 0;
    for (uint32_t i = b; i < e; i += 8) {
        unsigned long long mm[8];
#pragma unroll
        for (int u = 0; u < 8; u++) mm[u] = members[min(i + u, e - 1)];
        float X[8], Y[8], Z[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const uint32_t p = (uint32_t)mm[u];
            X[u] = x[p];
            Y[u] = y[p];
            Z[u] = z[p];
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            if (i + u >= e) break;
            const uint32_t kz = (uint32_t)(mm[u] >> 32);
            if (kz != cur) {
                const float denom = (float)cnt;  // :56
                ox[v] = __fdiv_rn(sx, denom);
                oy[v] = __fdiv_rn(sy, denom);
                oz[v] = __fdiv_rn(sz, denom);
                v++;
                sx = sy = sz = 0.f;
                cnt = 0;
                cur = kz;
            }
            sx = __fadd_rn(sx, X[u]);  // :38-42, input order
            sy = __fadd_rn(sy, Y[u]);
            sz = __fadd_rn(sz, Z[u]);
            cnt++;
        }
    }
    const float denom = (float)cnt;  // :56
    ox[v] = __fdiv_rn(sx, denom);
    oy[v] = __fdiv_rn(sy, denom);
    oz[v] = __fdiv_rn(sz, denom);
}

// Bounding box and finite count of the cloud just written, its length still on the device: what the index
// build of the next step would otherwise measure with a kernel and a round trip of its own.
__global__ void __launch_bounds__(256) vox_out_stats_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                            const float *__restrict__ z, const uint32_t *__restrict__ d_n,
                                                            VoxHeader *hdr) {
    PCR_GRID_DEP_SYNC();
    const uint32_t n = *d_n;
    if (blockIdx.x == 0 && threadIdx.x == 0) hdr->total = n;
    unsigned mn_c[3] = {0u, 0u, 0u}, mx[3] = {0u, 0u, 0u}, cnt = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float px = x[i], py = y[i], pz = z[i];
        if (!finite3(px, py, pz)) continue;
        const unsigned u[3] = {f32_ordered(px), f32_ordered(py), f32_ordered(pz)};
        for (int a = 0; a < 3; a++) {
            mn_c[a] = max(mn_c[a], ~u[a]);
            mx[a] = max(mx[a], u[a]);
        }
        cnt++;
    }
    for (int a = 0; a < 3; a++) {
        mn_c[a] = __reduce_max_sync(PCR_FULL, mn_c[a]);
        mx[a] = __reduce_max_sync(PCR_FULL, mx[a]);
    }
    cnt = __reduce_add_sync(PCR_FULL, cnt);
    __shared__ unsigned s_mn[3], s_mx[3], s_cnt;
    if (threadIdx.x == 0) {
        s_mn[0] = s_mn[1] = s_mn[2] = 0u;
        s_mx[0] = s_mx[1] = s_mx[2] = 0u;
        s_cnt = 0;
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && cnt) {
        for (int a = 0; a < 3; a++) {
            atomicMax(&s_mn[a], mn_c[a]);
            atomicMax(&s_mx[a], mx[a]);
        }
        atomicAdd(&s_cnt, cnt);
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_cnt) {
        for (int a = 0; a < 3; a++) {
            atomicMax(&hdr->mn_c[a], s_mn[a]);
            atomicMax(&hdr->mx[a], s_mx[a]);
        }
        atomicAdd(&hdr->count, s_cnt);
    }
}

// Batch: out_off[f] = first voxel of frame f, out_off[n_frames] = number of voxels.  The m finite points are sorted by
// frame first, so thread i in [0, m] writes the entries of the frames that start between sorted positions i - 1 and i
// (empty frames and frames without a finite point included): all of them start at voxel vid[i].
__global__ void __launch_bounds__(256) vox_frame_starts_kernel(const unsigned long long *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                               uint32_t m, int fshift /* < 0: no frame in the key */,
                                                               const uint32_t *__restrict__ frame_off, int n_frames,
                                                               const uint32_t *__restrict__ vid, uint32_t *__restrict__ out_off) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > m) return;
    auto frame = [&](uint32_t j) { return fshift >= 0 ? (int)(keys[j] >> fshift) : frame_of(frame_off, n_frames, vals[j]); };
    const int hi = i < m ? frame(i) : n_frames;
    const int lo = i > 0 ? frame(i - 1) : -1;
    for (int f = lo + 1; f <= hi; f++) out_off[f] = vid[i];
}

}  // namespace

int bits_for(uint64_t range) {  // smallest b with 2^b >= range
    int b = 0;
    while (b < 64 && (1ull << b) < range) b++;
    return b;
}

size_t radix_sort_hist_words(size_t n) { return (size_t)256 * ((n + kSortTile - 1) / kSortTile) + 1; }

// Sorts the n (key, val) pairs by the low `bits` bits of the key, stably.  The result is in
// (*keys, *vals): the pointers are swapped with the alternate buffers after every pass.
int radix_sort_pairs_dev(Ctx *ctx, unsigned long long **keys, uint32_t **vals, unsigned long long **keys_alt, uint32_t **vals_alt,
                         size_t n, int bits, uint32_t *d_hist /* 256 * n_tiles + 1 */) {
    if (n == 0) return PCR_OK;
    const uint32_t n_tiles = (uint32_t)((n + kSortTile - 1) / kSortTile);
    const unsigned blocks = (n_tiles + kSortWarps - 1) / kSortWarps;
    for (int shift = 0; shift < bits; shift += 8) {
        sort_hist_kernel<<<blocks, 32 * kSortWarps, 0, ctx->stream>>>(*keys, n, shift, n_tiles, d_hist);
        PCR_LAUNCH_CHECK(ctx);
        PCR_TRY(exclusive_scan_u32_dev(ctx, d_hist, (size_t)256 * n_tiles + 1));
        sort_scatter_kernel<<<blocks, 32 * kSortWarps, 0, ctx->stream>>>(*keys, *vals, n, shift, n_tiles, d_hist, *keys_alt, *vals_alt);
        PCR_LAUNCH_CHECK(ctx);
        std::swap(*keys, *keys_alt);
        std::swap(*vals, *vals_alt);
    }
    return PCR_OK;
}

// voxel_downsample on device arrays.  Outputs sized n; *n_out = number of voxels.  One host round trip
// (key range), one more for the count.
int voxel_downsample_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, float voxel, float *d_ox, float *d_oy,
                         float *d_oz, size_t *n_out, CloudStats *stats_out, bool allow_guess) {
    *n_out = 0;
    if (stats_out) stats_out->valid = 0;
    if (n == 0) return PCR_OK;  // :18-20
    if (n > 0x7fffffffull) return fail(ctx, PCR_ERR_UNSUPPORTED, "clouds above 2^31 points are not supported");
    cudaStream_t st = ctx->stream;
    TimeScope ts(ctx, kTagOther);
    PCR_TRY(ensure(ctx, ctx->b_small, 4096));
    PCR_TRY(ensure_pinned(ctx, 4096));
    VoxRange *d_range = (VoxRange *)ctx->b_small.p;
    uint32_t *d_nvox = (uint32_t *)((char *)ctx->b_small.p + 256);
    VoxRange *h_range = (VoxRange *)ctx->pinned;
    // A frame stream sizes the table from the previous frame's key box (padded) and skips the measuring pass and its
    // round trip; every 32nd frame is measured again so that the box follows the scene.
    auto &vc = ctx->vox_cache;
    static const bool no_guess = getenv("PCR_NO_VOXEL_GUESS") != nullptr;  // A/B hook
    const bool guessed = allow_guess && !no_guess && ctx->frame_stream && vc.valid && vc.voxel == voxel && vc.uses < 32;
    uint32_t m;
    if (guessed) {
        vc.uses++;
        for (int a = 0; a < 3; a++) {
            h_range->mn[a] = vc.mn[a];
            h_range->mx[a] = vc.mx[a];
        }
        m = (uint32_t)n;  // (an upper bound is all the sizing below needs)
    } else {
        vox_init_kernel<<<1, 1, 0, st>>>(d_range, 1);
        PCR_LAUNCH_CHECK(ctx);
        const unsigned bx = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 2);
        vox_range_kernel<<<bx, 256, 0, st>>>(dx, dy, dz, nullptr, n, voxel, d_range);
        PCR_LAUNCH_CHECK(ctx);
        PCR_CUDA(ctx, cudaMemcpyAsync(h_range, d_range, sizeof(VoxRange), cudaMemcpyDeviceToHost, st));
        PCR_MARK("voxel: wait for range");
        PCR_CUDA(ctx, cudaStreamSynchronize(st));
        PCR_MARK("voxel: got range");
        m = h_range->finite;
        if (m == 0) return PCR_OK;  // :45-47
        vc.valid = false;
        if (ctx->frame_stream) {  // remember the box, padded, for the next frames
            bool ok = true;
            for (int a = 0; a < 3; a++) {
                const long long ext = (long long)h_range->mx[a] - (long long)h_range->mn[a] + 1;
                const long long pad = std::max<long long>(2, ext >> vc.pad_shift);
                const long long lo = (long long)h_range->mn[a] - pad, hi = (long long)h_range->mx[a] + pad;
                if (lo < -2147483647ll || hi > 2147483646ll) ok = false;
                vc.mn[a] = (int)lo;
                vc.mx[a] = (int)hi;
            }
            vc.valid = ok;
            vc.voxel = voxel;
            vc.uses = 0;
        }
    }
    // ---- column path ------------------------------------------------------------------------------------
    {
        const uint64_t nx = (uint64_t)((int64_t)h_range->mx[0] - (int64_t)h_range->mn[0]) + 1;
        const uint64_t ny = (uint64_t)((int64_t)h_range->mx[1] - (int64_t)h_range->mn[1]) + 1;
        const uint64_t nz = (uint64_t)((int64_t)h_range->mx[2] - (int64_t)h_range->mn[2]) + 1;
        // A column may span 2^ys voxels along y (the MINOR of the two table axes, so table order stays the key order),
        // which shrinks the table.  Measured on the 122 K frame: the cheaper scans do not pay for the fuller columns
        // (more contended counters, longer per-thread sorts): 0.123 ms at ys = 0, 0.145 at 2, 0.179 at 3.  Off by default;
        // the hook stays for clouds whose (kx, ky) rectangle is too large for a one-voxel-wide table.
        int ys = 0;
        static const int ys_max = getenv("PCR_VOXEL_YS") ? atoi(getenv("PCR_VOXEL_YS")) : 0;  // tuning hook
        while (ys < ys_max && nz < (1ull << (32 - (ys + 1))) && nx * ((ny + (2ull << ys) - 1) >> (ys + 1)) >= (uint64_t)m) ys++;
        // ... and widened automatically when a one-voxel-wide table would not fit
        while (ys < 4 && nz < (1ull << (32 - (ys + 1))) && nx * ((ny + (1ull << ys) - 1) >> ys) > (1ull << 24)) ys++;
        const uint64_t nyc64 = (ny + (1ull << ys) - 1) >> ys;
        const uint64_t n_cols64 = nx * nyc64;  // (both < 2^32: no overflow)
        static const bool no_cols = getenv("PCR_VOXEL_RADIX") != nullptr;  // A/B hook: force the radix path
        if (!no_cols && nx < (1ull << 31) && ny < (1ull << 31) && nz < (1ull << (32 - ys)) && n_cols64 <= (1ull << 24) &&
            n_cols64 <= 64ull * m + 65536ull) {
            const uint32_t n_cols = (uint32_t)n_cols64;
            // scratch (b_table): header 64 B | count u32[n_cols + 1] | nvox u32[n + 1] | col_of u32[n] | rank_of u32[n] | members u64[n]
            const size_t tab = (sizeof(uint32_t) * ((size_t)n_cols + 1) + 15) & ~(size_t)15;  // (16 B-aligned tables: the scan's vector path)
            const size_t tab_v = (sizeof(uint32_t) * ((size_t)n + 1) + 15) & ~(size_t)15;
            const size_t o_count = sizeof(VoxHeader), o_nvox = o_count + tab;
            const size_t o_col = (o_nvox + tab_v + 15) & ~(size_t)15;
            const size_t o_rank = o_col + sizeof(uint32_t) * n;
            const size_t o_mem = (o_rank + sizeof(uint32_t) * n + 15) & ~(size_t)15;
            PCR_TRY(ensure(ctx, ctx->b_table, o_mem + sizeof(unsigned long long) * n));
            char *base = (char *)ctx->b_table.p;
            VoxHeader *d_hdr = (VoxHeader *)base;
            uint32_t *count = (uint32_t *)(base + o_count), *nvox = (uint32_t *)(base + o_nvox);
            uint32_t *col_of = (uint32_t *)(base + o_col), *rank_of = (uint32_t *)(base + o_rank);
            unsigned long long *members = (unsigned long long *)(base + o_mem);
            PCR_CUDA(ctx, cudaMemsetAsync(base, 0, o_nvox + tab_v, st));  // header, counters and nvox in one go
            const unsigned nbp = (unsigned)((n + 255) / 256);
            vox_col_count_kernel<<<nbp, 256, 0, st>>>(dx, dy, dz, n, voxel, h_range->mn[0], h_range->mn[1], h_range->mn[2], nx, ny, nz,
                                                      (uint32_t)nyc64, ys, count, col_of, rank_of, &d_hdr->outside);
            PCR_LAUNCH_CHECK(ctx);
            PCR_TRY(exclusive_scan_u32_dev(ctx, count, (size_t)n_cols + 1));
            // (a chain of small kernels: programmatic dependent launches, see launch_chained)
            PCR_CUDA(ctx, launch_chained(vox_col_scatter_kernel, dim3(nbp), dim3(256), 0, st, dy, dz, n, voxel, h_range->mn[1], h_range->mn[2], ys,
                                         count, col_of, rank_of, members));
            PCR_CUDA(ctx, launch_chained(vox_col_sort_kernel, dim3(nbp), dim3(256), 0, st, col_of, rank_of, n, count, members, nvox, &d_hdr->tall));
            ctx->launches += 2;
            PCR_TRY(exclusive_scan_u32_dev(ctx, nvox, n + 1));
            PCR_CUDA(ctx, launch_chained(vox_col_emit_kernel, dim3(nbp), dim3(256), 0, st, dx, dy, dz, col_of, rank_of, n, count, nvox, members, d_ox,
                                         d_oy, d_oz));
            ctx->launches++;
            // the box and count of what was written (the next step's index build wants them), the voxel count and the
            // outside flag come back together
            PCR_CUDA(ctx, launch_chained(vox_out_stats_kernel, dim3((unsigned)ctx->sm_count), dim3(256), 0, st, d_ox, d_oy, d_oz, nvox + n, d_hdr));
            ctx->launches++;
            VoxHeader *mail = (VoxHeader *)((uint32_t *)ctx->pinned + 64);
            PCR_CUDA(ctx, cudaMemcpyAsync(mail, d_hdr, sizeof(VoxHeader), cudaMemcpyDeviceToHost, st));
            PCR_MARK("voxel: wait for count");
            PCR_CUDA(ctx, cudaStreamSynchronize(st));
            PCR_MARK("voxel: got count");
            if (guessed) (mail->outside ? ctx->stat_vox_misses : ctx->stat_vox_hits)++;
            if (guessed && mail->outside) {  // a point fell outside the guessed box: measure, with a wider pad from now on
                vc.valid = false;
                vc.pad_shift = std::max(2, vc.pad_shift - 1);
                return voxel_downsample_dev(ctx, dx, dy, dz, n, voxel, d_ox, d_oy, d_oz, n_out, stats_out, false);
            }
            const bool tall = mail->tall != 0;
            if (tall && guessed) {  // (the guessed box is not what the radix path below wants: measure first)
                vc.valid = false;
                return voxel_downsample_dev(ctx, dx, dy, dz, n, voxel, d_ox, d_oy, d_oz, n_out, stats_out, false);
            }
            if (!tall) *n_out = mail->total;
            if (!tall && stats_out) {
                for (int a = 0; a < 3; a++) {
                    stats_out->mn[a] = ~mail->mn_c[a];
                    stats_out->mx[a] = mail->mx[a];
                }
                stats_out->count = mail->count;
                stats_out->valid = 1;
            }
            if (!tall) return PCR_OK;
            // a tall column: fall through to the radix path (h_range is measured here: `guessed` was handled above)
        }
    }
    if (guessed) {  // the padded box does not suit the column path: measure
        vc.valid = false;
        return voxel_downsample_dev(ctx, dx, dy, dz, n, voxel, d_ox, d_oy, d_oz, n_out, stats_out, false);
    }
    // ---- radix path -------------------------------------------------------------------------------------
    int bits[3];
    for (int a = 0; a < 3; a++) bits[a] = bits_for((uint64_t)((int64_t)h_range->mx[a] - (int64_t)h_range->mn[a]) + 1);
    const int total_bits = bits[0] + bits[1] + bits[2];
    const bool packed = total_bits <= 63;

    // scratch (b_table): keys A/B u64[n] | vals A/B u32[n] | hist u32[256 * tiles + 1] | flag/vid u32[n + 1] | start u32[n + 1]
    const size_t n_tiles = (n + kSortTile - 1) / kSortTile;
    const size_t need = 2 * sizeof(unsigned long long) * n + sizeof(uint32_t) * (2 * n + 256 * n_tiles + 1 + 2 * (n + 1)) + 1024;
    PCR_TRY(ensure(ctx, ctx->b_table, need));
    char *p = (char *)ctx->b_table.p;
    unsigned long long *kA = (unsigned long long *)p;
    p += sizeof(unsigned long long) * n;
    unsigned long long *kB = (unsigned long long *)p;
    p += sizeof(unsigned long long) * n;
    uint32_t *vA = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *vB = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *hist = (uint32_t *)p;
    p += sizeof(uint32_t) * (256 * n_tiles + 1);
    uint32_t *vid = (uint32_t *)p;
    p += sizeof(uint32_t) * (n + 1);
    uint32_t *start = (uint32_t *)p;
    const unsigned nb = (unsigned)((n + 255) / 256);
    if (packed) {
        const unsigned long long last = 1ull << total_bits;  // non-finite points: above every real key
        vox_pack_kernel<<<nb, 256, 0, st>>>(dx, dy, dz, nullptr, n, voxel, -1, h_range->mn[0], h_range->mn[1], h_range->mn[2],
                                            bits[1] + bits[2], bits[2], last, kA, vA, nullptr, 1, nullptr, 0);
        PCR_LAUNCH_CHECK(ctx);
        PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, n, total_bits + 1, hist));
        vox_heads_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(kA, m, vid);
        PCR_LAUNCH_CHECK(ctx);
    } else {
        const unsigned long long last = 1ull << 32;
        for (int axis = 2; axis >= 0; axis--) {  // LSD over the axes: z, y, x
            // after the first pass vA holds the order so far; the pack kernel reads and rewrites it in place
            vox_pack_kernel<<<nb, 256, 0, st>>>(dx, dy, dz, axis == 2 ? nullptr : vA, n, voxel, axis, 0, 0, 0, 0, 0, last, kA, vA, nullptr, 1,
                                                nullptr, 0);
            PCR_LAUNCH_CHECK(ctx);
            PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, n, 33, hist));
        }
        vox_heads_triple_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(dx, dy, dz, vA, m, voxel, nullptr, 1, vid);
        PCR_LAUNCH_CHECK(ctx);
    }
    PCR_TRY(exclusive_scan_u32_dev(ctx, vid, (size_t)m + 1));  // vid[m] = number of voxels
    vox_starts_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(vid, m, start);
    PCR_LAUNCH_CHECK(ctx);
    PCR_CUDA(ctx, cudaMemcpyAsync(d_nvox, vid + m, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    vox_mean_kernel<<<(m + 127) / 128, 128, 0, st>>>(dx, dy, dz, vA, start, d_nvox, d_ox, d_oy, d_oz);
    PCR_LAUNCH_CHECK(ctx);
    uint32_t *mail = (uint32_t *)ctx->pinned + 64;
    PCR_CUDA(ctx, cudaMemcpyAsync(mail, d_nvox, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    *n_out = *mail;
    return PCR_OK;
}

// voxel_downsample of every frame of a batch (frame f = points [frame_offsets[f], frame_offsets[f+1]), offsets on the
// host, checked by the caller) in one set of launches: the radix path above with the frame as the most significant
// part of the key.  Frame f's voxels go to [out_offsets[f], out_offsets[f+1]) of the outputs (sized n), bit for bit
// what voxel_downsample_dev returns for the frame alone: the same key order and the same input-order sums, since the
// sort is stable and a frame's points keep their order.  Two host round trips: the per-frame key ranges, and the
// per-frame voxel counts.  The frame-stream key box (ctx->vox_cache) is neither read nor written.
int voxel_downsample_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets,
                               size_t n_frames, float voxel, float *d_ox, float *d_oy, float *d_oz, uint64_t *out_offsets) {
    const int F = (int)n_frames;
    for (int f = 0; f <= F; f++) out_offsets[f] = 0;
    const size_t n = F ? (size_t)frame_offsets[F] : 0;
    if (n == 0) return PCR_OK;
    cudaStream_t st = ctx->stream;
    TimeScope ts(ctx, kTagOther);
    // scratch (b_table): keys A/B u64[n] | vals A/B u32[n] | hist u32[256 * tiles + 1] | flag/vid u32[n + 1] | start u32[n + 1]
    //                    | frame offsets u32[F + 1] | out offsets u32[F + 1] | ranges VoxRange[F]
    const size_t n_tiles = (n + kSortTile - 1) / kSortTile;
    const size_t need = 2 * sizeof(unsigned long long) * n + sizeof(uint32_t) * (2 * n + 256 * n_tiles + 1 + 2 * (n + 1)) +
                        sizeof(uint32_t) * 2 * (F + 1) + sizeof(VoxRange) * F + 1024;
    PCR_TRY(ensure(ctx, ctx->b_table, need));
    PCR_TRY(ensure_pinned(ctx, std::max<size_t>(4096, std::max(sizeof(VoxRange) * F, sizeof(uint32_t) * (F + 1)))));
    char *p = (char *)ctx->b_table.p;
    unsigned long long *kA = (unsigned long long *)p;
    p += sizeof(unsigned long long) * n;
    unsigned long long *kB = (unsigned long long *)p;
    p += sizeof(unsigned long long) * n;
    uint32_t *vA = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *vB = (uint32_t *)p;
    p += sizeof(uint32_t) * n;
    uint32_t *hist = (uint32_t *)p;
    p += sizeof(uint32_t) * (256 * n_tiles + 1);
    uint32_t *vid = (uint32_t *)p;
    p += sizeof(uint32_t) * (n + 1);
    uint32_t *start = (uint32_t *)p;
    p += sizeof(uint32_t) * (n + 1);
    uint32_t *d_off = (uint32_t *)p;
    p += sizeof(uint32_t) * (F + 1);
    uint32_t *d_out_off = (uint32_t *)p;
    p += sizeof(uint32_t) * (F + 1);
    VoxRange *d_range = (VoxRange *)p;

    // per-frame key ranges, ONE round trip for all of them
    std::vector<uint32_t> h_off(F + 1);
    size_t longest = 0;
    for (int f = 0; f <= F; f++) h_off[f] = (uint32_t)frame_offsets[f];
    for (int f = 0; f < F; f++) longest = std::max<size_t>(longest, h_off[f + 1] - h_off[f]);
    // (pageable source: the copy has taken the bytes when it returns)
    PCR_CUDA(ctx, cudaMemcpyAsync(d_off, h_off.data(), sizeof(uint32_t) * (F + 1), cudaMemcpyHostToDevice, st));
    vox_init_kernel<<<(F + 255) / 256, 256, 0, st>>>(d_range, F);
    PCR_LAUNCH_CHECK(ctx);
    const unsigned bx = (unsigned)std::max<size_t>(1, std::min<size_t>((longest + 255) / 256, (size_t)ctx->sm_count * 8 / F));
    vox_range_kernel<<<dim3(bx, F), 256, 0, st>>>(dx, dy, dz, d_off, n, voxel, d_range);
    PCR_LAUNCH_CHECK(ctx);
    VoxRange *h_range = (VoxRange *)ctx->pinned;
    PCR_CUDA(ctx, cudaMemcpyAsync(h_range, d_range, sizeof(VoxRange) * F, cudaMemcpyDeviceToHost, st));
    PCR_MARK("voxel batch: wait for ranges");
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    uint64_t m64 = 0;
    int bits[3] = {0, 0, 0};  // per axis, the widest frame's
    for (int f = 0; f < F; f++) {
        if (!h_range[f].finite) continue;
        m64 += h_range[f].finite;
        for (int a = 0; a < 3; a++)
            bits[a] = std::max(bits[a], bits_for((uint64_t)((int64_t)h_range[f].mx[a] - (int64_t)h_range[f].mn[a]) + 1));
    }
    if (m64 == 0) return PCR_OK;  // :45-47, in every frame
    const uint32_t m = (uint32_t)m64;
    const int fbits = bits_for((uint64_t)F), key_bits = bits[0] + bits[1] + bits[2];
    const bool packed = fbits + key_bits <= 63;

    // one stable sort of all frames: (frame, key, index) order
    const unsigned nb = (unsigned)((n + 255) / 256);
    if (packed) {
        const unsigned long long last = 1ull << (fbits + key_bits);  // non-finite points: above every real key of every frame
        vox_pack_kernel<<<nb, 256, 0, st>>>(dx, dy, dz, nullptr, n, voxel, -1, 0, 0, 0, bits[1] + bits[2], bits[2], last, kA, vA, d_off, F,
                                            d_range, key_bits);
        PCR_LAUNCH_CHECK(ctx);
        PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, n, fbits + key_bits + 1, hist));
        vox_heads_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(kA, m, vid);
        PCR_LAUNCH_CHECK(ctx);
    } else {  // LSD over z, y, x as in the single call, then one more stable pass on the frame id
        for (int axis = 2; axis >= 0; axis--) {
            vox_pack_kernel<<<nb, 256, 0, st>>>(dx, dy, dz, axis == 2 ? nullptr : vA, n, voxel, axis, 0, 0, 0, 0, 0, 1ull << 32, kA, vA, nullptr, 1,
                                                nullptr, 0);
            PCR_LAUNCH_CHECK(ctx);
            PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, n, 33, hist));
        }
        if (F > 1) {
            vox_pack_kernel<<<nb, 256, 0, st>>>(dx, dy, dz, vA, n, voxel, 3, 0, 0, 0, 0, 0, (unsigned long long)F, kA, vA, d_off, F, nullptr, 0);
            PCR_LAUNCH_CHECK(ctx);
            PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, n, bits_for((uint64_t)F + 1), hist));
        }
        vox_heads_triple_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(dx, dy, dz, vA, m, voxel, d_off, F, vid);
        PCR_LAUNCH_CHECK(ctx);
    }
    PCR_TRY(exclusive_scan_u32_dev(ctx, vid, (size_t)m + 1));  // vid[m] = number of voxels
    vox_starts_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(vid, m, start);
    PCR_LAUNCH_CHECK(ctx);
    vox_mean_kernel<<<(m + 127) / 128, 128, 0, st>>>(dx, dy, dz, vA, start, vid + m, d_ox, d_oy, d_oz);
    PCR_LAUNCH_CHECK(ctx);
    vox_frame_starts_kernel<<<(m + 1 + 255) / 256, 256, 0, st>>>(kA, vA, m, packed ? key_bits : -1, d_off, F, vid, d_out_off);
    PCR_LAUNCH_CHECK(ctx);
    uint32_t *h_out = (uint32_t *)ctx->pinned;
    PCR_CUDA(ctx, cudaMemcpyAsync(h_out, d_out_off, sizeof(uint32_t) * (F + 1), cudaMemcpyDeviceToHost, st));
    PCR_MARK("voxel batch: wait for counts");
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    for (int f = 0; f <= F; f++) out_offsets[f] = h_out[f];
    return PCR_OK;
}

}  // namespace pcr
