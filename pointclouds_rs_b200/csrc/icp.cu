// icp.cu -- ICP registration on the grid index.
//
//   correspondences      find_correspondences          crates/registration/src/correspondence.rs:16-39
//   loop + convergence   icp_point_to_point / _plane   icp.rs:125-206, icp_plane.rs:20-97
//   p2p solve            compute_rigid_transform_svd   icp.rs:210-270
//   p2plane solve        solve_point_to_plane          icp_plane.rs:131-236
//   transform            apply_to_point / compose      icp.rs:39-73
//
// Per iteration ONE streaming kernel does: apply the previous incremental transform to the working
// copy of the source (in place, f32, the reference's operation order), 1-NN search of every source
// point in the target grid, the max-distance test, and the accumulation of the normal equations
// (f64, like icp_plane.rs:145-180) as per-block partials.  A single-block kernel then folds the
// partials in a fixed order, (multi-GPU: ncclAllReduce of the 30 doubles in between), tests
// convergence, solves the 6x6 / 3x3 system and composes the transforms -- all on the device, so the
// host never waits inside the loop; it only polls a flag in pinned memory to stop enqueueing.
// The source is binned by TARGET cell once up front so that neighbouring threads search
// neighbouring cells.
#include "knn_search.cuh"

#include <algorithm>

namespace pcr {

namespace {

constexpr int NP = 30;  // doubles per partial
// plane : [0,21) upper triangle of A^T A, [21,27) A^T b
// p2p   : [0,3) sum s, [3,6) sum t, [6,15) sum s t^T (row-major)
constexpr int kSumSq = 27, kCount = 28, kSrcN = 29;
constexpr int kIcpThreads = 256;

struct IcpState {
    float inc_R[9], inc_t[3];
    float cum_R[9], cum_t[3];
    float prev_rmse, last_rmse, last_fitness;
    int has_inc, converged, done;
    unsigned long long num_iterations;
    double sums[NP];
};

__device__ __forceinline__ void apply_point(const float *R, const float *t, float x, float y, float z, float &ox, float &oy,
                                            float &oz) {
    // icp.rs:42-46: r0*x + r1*y + r2*z + t, left to right, every op rounded
    ox = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[0], x), __fmul_rn(R[1], y)), __fmul_rn(R[2], z)), t[0]);
    oy = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[3], x), __fmul_rn(R[4], y)), __fmul_rn(R[5], z)), t[1]);
    oz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[6], x), __fmul_rn(R[7], y)), __fmul_rn(R[8], z)), t[2]);
}

__global__ void apply_transform_kernel(const float *__restrict__ x, const float *__restrict__ y, const float *__restrict__ z,
                                       size_t n, const float *__restrict__ Rt /* 9 + 3 */, float *__restrict__ ox,
                                       float *__restrict__ oy, float *__restrict__ oz) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float R[9], t[3];
#pragma unroll
    for (int j = 0; j < 9; j++) R[j] = Rt[j];
#pragma unroll
    for (int j = 0; j < 3; j++) t[j] = Rt[9 + j];
    float a, b, c;
    apply_point(R, t, x[i], y[i], z[i], a, b, c);
    ox[i] = a;
    oy[i] = b;
    oz[i] = c;
}

// Every frame of a batch by its own transform: one thread per point over all N points, so the grid does not depend on
// how uneven the frames are; point i finds its frame in the u32 offsets and reads that frame's 12 floats.
__global__ void apply_transform_batch_kernel(const float *__restrict__ x, const float *__restrict__ y, const float *__restrict__ z,
                                             size_t n, const float *__restrict__ Rt /* 12 per frame */,
                                             const uint32_t *__restrict__ frame_off, int n_frames, float *__restrict__ ox,
                                             float *__restrict__ oy, float *__restrict__ oz) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *rt = Rt + 12 * frame_of(frame_off, n_frames, (uint32_t)i);
    float R[9], t[3];
#pragma unroll
    for (int j = 0; j < 9; j++) R[j] = rt[j];
#pragma unroll
    for (int j = 0; j < 3; j++) t[j] = rt[9 + j];
    float a, b, c;
    apply_point(R, t, x[i], y[i], z[i], a, b, c);
    ox[i] = a;
    oy[i] = b;
    oz[i] = c;
}

// ---- plain correspondences (C ABI pcr_find_correspondences): k = 1 KNN + the distance test ------
__global__ void correspond_filter_kernel(size_t ns, float max_distance, uint32_t *__restrict__ tgt, float *__restrict__ dist,
                                         const uint32_t *__restrict__ counts) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    bool ok = counts[i] > 0 && dist[i] <= max_distance;  // correspondence.rs:27-28
    if (!ok) {
        tgt[i] = 0xffffffffu;
        dist[i] = INFINITY;
    }
}

// ---- binning of the source by target cell ---------------------------------------------------------
// kInit: the loop starts from a guess, and the working copy holds apply_point(init, p) from the start.  The moved point
// is what the first pass searches, so it is also what gets binned: binning the unmoved source would scatter the
// threads of one target cell over the whole source when the guess moves it by metres.
struct Xform {
    float R[9], t[3];  // row-major R, then t (the 12 floats of pcr_apply_transform_batch)
};

template <bool kInit>
__global__ void __launch_bounds__(256) src_count_kernel(const float *__restrict__ sx, const float *__restrict__ sy,
                                                        const float *__restrict__ sz, size_t ns,
                                                        const GridDesc *__restrict__ grids, uint32_t *__restrict__ table,
                                                        uint32_t *__restrict__ cell_id, uint32_t *__restrict__ rank, Xform init) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const GridDesc g = grids[0];
    float x = sx[i], y = sy[i], z = sz[i];
    if (kInit) apply_point(init.R, init.t, x, y, z, x, y, z);
    uint32_t cid = 0;
    if (finite3(x, y, z) && g.n_cells > 0) {
        int c0 = cell_coord(g, 0, pick_axis(g.ax[0], x, y, z), nullptr);
        int c1 = cell_coord(g, 1, pick_axis(g.ax[1], x, y, z), nullptr);
        int c2 = cell_coord(g, 2, pick_axis(g.ax[2], x, y, z), nullptr);
        cid = cell_linear(g, c0, c1, c2) - g.cell_base;
    }
    cell_id[i] = cid;
    rank[i] = atomicAdd(&table[cid], 1u);
}

template <bool kInit>
__global__ void __launch_bounds__(256) src_scatter_kernel(const float *__restrict__ sx, const float *__restrict__ sy,
                                                          const float *__restrict__ sz, size_t ns,
                                                          const uint32_t *__restrict__ table,
                                                          const uint32_t *__restrict__ cell_id,
                                                          const uint32_t *__restrict__ rank, float4 *__restrict__ cur, Xform init) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    float x = sx[i], y = sy[i], z = sz[i];
    if (kInit) apply_point(init.R, init.t, x, y, z, x, y, z);
    cur[table[cell_id[i]] + rank[i]] = make_float4(x, y, z, __uint_as_float((uint32_t)i));
}

// ---- per-iteration kernels ---------------------------------------------------------------------------
// (A) transform + 1-NN on grid level 0, one thread per source point.  A point whose 27 cells are
//     empty (a source that pokes out of the target, e.g. two scans that only partly overlap) is
//     deferred to the coarser levels instead of walking shells of empty fine cells.
//     (The body is shared with the batch kernel: one working-copy point i searched in target grid g.)
__device__ __forceinline__ void icp_search_point(const GridDesc &g, const uint32_t *__restrict__ cell_start,
                                                 const float4 *__restrict__ sorted, const float4 *__restrict__ tgt4,
                                                 float4 *__restrict__ cur, size_t i, const IcpState *__restrict__ state,
                                                 unsigned long long *__restrict__ nn, uint32_t *__restrict__ defer_list,
                                                 uint32_t *__restrict__ defer_count, int last_level) {
    float4 p = cur[i];
    if (state->has_inc) {  // icp.rs:186 / icp_plane.rs:78: current = apply_transform(current, incremental)
        float a, b, c;
        apply_point(state->inc_R, state->inc_t, p.x, p.y, p.z, a, b, c);
        p.x = a; p.y = b; p.z = c;
        cur[i] = p;
    }
    unsigned long long best = PCR_EMPTY_KEY;
    if (finite3(p.x, p.y, p.z)) {  // kdtree.rs:65: a non-finite query has no neighbour
        ThreadBest1 acc;
        acc.reset();
        // Warm start: the neighbour found in the previous iteration is still a point of the target, so its
        // distance r0 to the moved source point bounds the search (the minimum over the target cannot change by
        // looking at one of its points first).  Worth it only if the seed is CLOSE: within 1.5 cells the ball
        // scan reads a handful of cells and usually just confirms the seed; a far seed (early iterations move
        // the source by metres) would make the ball larger than the 27 cells the plain walk needs.
        unsigned long long seed = PCR_EMPTY_KEY;
        if (state->has_inc) {
            const unsigned long long prev = nn[i];
            if (prev != PCR_EMPTY_KEY) {
                const float4 t = __ldg(&tgt4[key_idx(prev)]);
                seed = make_key(dist2_exact(p.x, p.y, p.z, t.x, t.y, t.z), key_idx(prev));
            }
        }
        bool ok = false;
        if (seed != PCR_EMPTY_KEY && (double)key_d2(seed) < 2.25 * g.h * g.h) {
            acc.offer(seed);
            ok = thread_ball_search(acc, g, cell_start, sorted, p.x, p.y, p.z, 3);
        }
        if (!ok) ok = thread_grid_search_pruned(acc, g, cell_start, sorted, p.x, p.y, p.z, 1, last_level ? kMaxRings : kLevelRings, last_level != 0, 0);
        if (ok) {
            best = acc.best;
        } else {
            best = seed;  // the seed (if any) travels to the deferred passes through nn[i]
            defer_list[atomicAdd(defer_count, 1u)] = (uint32_t)i;
        }
    }
    nn[i] = best;
}

__global__ void __launch_bounds__(kIcpThreads) icp_search_kernel(const GridDesc *__restrict__ grids,
                                                                 const uint32_t *__restrict__ cell_start,
                                                                 const float4 *__restrict__ sorted, const float4 *__restrict__ tgt4,
                                                                 float4 *__restrict__ cur, size_t ns,
                                                                 const IcpState *__restrict__ state, unsigned long long *__restrict__ nn,
                                                                 uint32_t *__restrict__ defer_list,
                                                                 uint32_t *__restrict__ defer_count, int last_level) {
    if (state->done) return;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const GridDesc g = grids[0];
    icp_search_point(g, cell_start, sorted, tgt4, cur, i, state, nn, defer_list, defer_count, last_level);
}

// (A') deferred source points on a coarser level, persistent over the device-side list: one warp per point
//      (a coarse cell holds ~70 points, so the lanes are busy).  nn[i] carries the warm-start candidate the
//      search kernel left there (or EMPTY); the warp search inserts it first and prunes with it.
__device__ __forceinline__ void icp_deferred_point(RegTopK &tk, const GridDesc &g, const uint32_t *__restrict__ cell_start,
                                                   const float4 *__restrict__ pts, const float4 *__restrict__ cur, uint32_t i,
                                                   unsigned long long *__restrict__ nn, uint32_t *__restrict__ out_list,
                                                   uint32_t *__restrict__ out_count, int last_level) {
    const float4 p = cur[i];
    const unsigned long long seed = nn[i];
    if (warp_knn_search(tk, g, cell_start, pts, p.x, p.y, p.z, last_level ? kMaxRings : kLevelRings, last_level != 0, seed)) {
        unsigned long long best = __shfl_sync(PCR_FULL, tk.K, 0);
        if (tk.lane == 0) nn[i] = best;
    } else if (tk.lane == 0) {
        out_list[atomicAdd(out_count, 1u)] = i;
    }
}

__global__ void __launch_bounds__(128) icp_deferred_kernel(const GridDesc *__restrict__ grids, const uint32_t *__restrict__ cell_start,
                                                           const float4 *__restrict__ pts, const float4 *__restrict__ cur,
                                                           const IcpState *__restrict__ state, const uint32_t *__restrict__ in_list,
                                                           const uint32_t *__restrict__ in_count, unsigned long long *__restrict__ nn,
                                                           uint32_t *__restrict__ out_list, uint32_t *__restrict__ out_count,
                                                           int last_level) {
    if (state->done) return;
    const uint32_t n = *in_count;
    const GridDesc g = grids[0];
    const int lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    RegTopK tk;
    tk.kk = 1;
    tk.lane = lane;
    for (uint32_t j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < n; j += warps)
        icp_deferred_point(tk, g, cell_start, pts, cur, in_list[j], nn, out_list, out_count, last_level);
}

// (B) residuals and normal equations from the correspondences, per-block partials in a fixed order.
//     icp_accum_point adds source point i's terms to acc; icp_block_partials folds acc over the block.
template <bool kPlane>
__device__ __forceinline__ void icp_accum_point(double (&acc)[NP], const float4 *__restrict__ tgt4, const float4 *__restrict__ nrm4,
                                                const float4 *__restrict__ cur, const unsigned long long *__restrict__ nn, size_t i,
                                                float max_distance) {
    const unsigned long long best = nn[i];
    if (best == PCR_EMPTY_KEY) return;
    const float d = __fsqrt_rn(key_d2(best));
    if (!(d <= max_distance)) return;  // correspondence.rs:28
    const float4 p = cur[i];
    const float4 t = __ldg(&tgt4[key_idx(best)]);
    acc[kSumSq] += (double)__fmul_rn(d, d);  // icp.rs:279
    acc[kCount] += 1.0;
    if (kPlane) {  // icp_plane.rs:152-179
        const float4 nn4 = __ldg(&nrm4[key_idx(best)]);
        const double sx = p.x, sy = p.y, sz = p.z, n0 = nn4.x, n1 = nn4.y, n2 = nn4.z;
        double a[6] = {sy * n2 - sz * n1, sz * n0 - sx * n2, sx * n1 - sy * n0, n0, n1, n2};
        const double b = ((double)t.x - sx) * n0 + ((double)t.y - sy) * n1 + ((double)t.z - sz) * n2;
        int o = 0;
#pragma unroll
        for (int r = 0; r < 6; r++)
#pragma unroll
            for (int c = r; c < 6; c++) acc[o++] += a[r] * a[c];
#pragma unroll
        for (int r = 0; r < 6; r++) acc[21 + r] += a[r] * b;
    } else {  // icp.rs:221-244 (sums; centring is done in the solve)
        const double s[3] = {p.x, p.y, p.z}, tt[3] = {t.x, t.y, t.z};
#pragma unroll
        for (int r = 0; r < 3; r++) {
            acc[r] += s[r];
            acc[3 + r] += tt[r];
#pragma unroll
            for (int c = 0; c < 3; c++) acc[6 + r * 3 + c] += s[r] * tt[c];
        }
    }
}

// block reduction in a fixed order: shuffle tree inside the warp, then warps in order (every thread of the block calls it)
__device__ __forceinline__ void icp_block_partials(const double (&acc)[NP], double *__restrict__ out /* NP */) {
    __shared__ double sh[kIcpThreads / 32][NP];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < NP; j++) {
        double v = acc[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(PCR_FULL, v, o);
        if (lane == 0) sh[w][j] = v;
    }
    __syncthreads();
    if (threadIdx.x < NP) {
        double v = 0.0;
#pragma unroll
        for (int ww = 0; ww < kIcpThreads / 32; ww++) v += sh[ww][threadIdx.x];
        out[threadIdx.x] = v;
    }
}

template <bool kPlane>
__global__ void __launch_bounds__(kIcpThreads) icp_accum_kernel(const float4 *__restrict__ tgt4, const float4 *__restrict__ nrm4,
                                                                const float4 *__restrict__ cur,
                                                                const unsigned long long *__restrict__ nn, size_t ns,
                                                                float max_distance, const IcpState *__restrict__ state,
                                                                double *__restrict__ partials) {
    if (state->done) return;
    double acc[NP];
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += (size_t)gridDim.x * blockDim.x)
        icp_accum_point<kPlane>(acc, tgt4, nrm4, cur, nn, i, max_distance);
    icp_block_partials(acc, partials + (size_t)blockIdx.x * NP);
}

// Folds the per-block partials in a fixed order: 32 lanes per value take strided subsets, then a
// shuffle tree -- deterministic for a given launch configuration.
//
// Sharded source, pc.world > 1: the reduction is followed IN THE SAME KERNEL by a one-shot all-reduce over NVLink peer
// memory instead of an ncclAllReduce launch (whose span -- small-message latency plus launch -- was 0.13 ms of a 0.19 ms
// iteration at 8 GPUs).  Every rank owns an exchange block that all peers have mapped (comm.cu: CUDA IPC):
//   1. warp j, lane p < world, stores this rank's sum j into peer p's block at [slot][this rank][j]   (NVLink stores)
//   2. __threadfence_system + block barrier, then thread p publishes flag[slot][this rank] = seq in peer p's block (release)
//   3. thread p waits for flag[slot][p] == seq in the OWN block (acquire), block barrier
//   4. warp j adds the world's contributions in RANK order: every rank computes the same bits, as after ncclAllReduce.
// slot = seq & 1: a rank can be at most one exchange ahead of the slowest (it needs everybody's flag of exchange n to leave
// it), so exchange n + 2 never overwrites data somebody still reads.  All ranks skip the same exchanges (state->done is
// computed from the all-reduced sums, and the host queues passes in lock step), and seq counts the queued ones on every rank.
// A peer that never arrives (a crashed rank) must not hang this GPU: after ~2e7 polls the kernel gives up and marks the
// state as failed (rmse NaN, done), which the host reports.
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// sum j of n_blocks partials, in the fixed order above (one warp per value; every lane returns the sum)
__device__ __forceinline__ double icp_fold_partials(const double *__restrict__ partials, int n_blocks, int j, int lane) {
    double v = 0.0;
    for (int b = lane; b < n_blocks; b += 32) v += partials[(size_t)b * NP + j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(PCR_FULL, v, o);
    return v;
}

__global__ void __launch_bounds__(NP * 32) icp_reduce_kernel(const double *__restrict__ partials, int n_blocks, size_t ns_local,
                                                             IcpState *state, PeerComm pc, unsigned long long seq) {
    if (state->done) return;
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double v = icp_fold_partials(partials, n_blocks, j, lane);
    v = j == kSrcN ? (double)ns_local : v;  // (every lane holds the sum)
    if (pc.world <= 1) {
        if (lane == 0) state->sums[j] = v;
        return;
    }
    const int slot = (int)(seq & 1ull);
    if (lane < pc.world) pc.data[lane][((size_t)slot * kPeerMaxWorld + pc.rank) * kPeerWords + j] = v;
    __threadfence_system();
    __syncthreads();
    __shared__ int s_failed;
    if (threadIdx.x == 0) s_failed = 0;
    if (threadIdx.x < pc.world) st_release_sys_u64(&pc.flag[threadIdx.x][slot * kPeerMaxWorld + pc.rank], seq);
    __syncthreads();
    if (threadIdx.x < pc.world) {
        const unsigned long long *f = &pc.flag[pc.rank][slot * kPeerMaxWorld + threadIdx.x];
        unsigned polls = 0;
        while (ld_acquire_sys_u64(f) != seq)
            if (++polls > 20000000u) {
                s_failed = 1;
                break;
            }
    }
    __syncthreads();
    if (s_failed) {
        if (threadIdx.x == 0) {
            state->last_rmse = __int_as_float(0x7fc00000);
            state->converged = 0;
            state->done = 1;
        }
        return;
    }
    if (lane == 0) {
        const volatile double *mine = pc.data[pc.rank] + (size_t)slot * kPeerMaxWorld * kPeerWords;
        double t = 0.0;
        for (int p = 0; p < pc.world; p++) t += mine[(size_t)p * kPeerWords + j];
        state->sums[j] = t;
    }
}

// ---- device-side solves ----------------------------------------------------------------------------
__device__ void mat3_mul_f32(const float *a, const float *b, float *o) {
    float r[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++)
            r[i * 3 + j] = __fadd_rn(__fadd_rn(__fmul_rn(a[i * 3 + 0], b[0 * 3 + j]), __fmul_rn(a[i * 3 + 1], b[1 * 3 + j])),
                                     __fmul_rn(a[i * 3 + 2], b[2 * 3 + j]));
    for (int i = 0; i < 9; i++) o[i] = r[i];
}

// 3x3 SVD a = U diag(s) V^T (s descending) by cyclic Jacobi on a^T a, f64.
__device__ void svd3(const double *a, double *U, double *s, double *V) {
    double ata[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double t = 0;
            for (int k = 0; k < 3; k++) t += a[k * 3 + i] * a[k * 3 + j];
            ata[i * 3 + j] = t;
        }
    double v[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int sweep = 0; sweep < 60; sweep++) {
        double off = fabs(ata[1]) + fabs(ata[2]) + fabs(ata[5]);
        double diag = fabs(ata[0]) + fabs(ata[4]) + fabs(ata[8]);
        if (off <= 1e-300 || off <= 1e-18 * diag) break;
        for (int p = 0; p < 2; p++)
            for (int q = p + 1; q < 3; q++) {
                double apq = ata[p * 3 + q];
                if (fabs(apq) < 1e-300) continue;
                double app = ata[p * 3 + p], aqq = ata[q * 3 + q];
                double theta = (aqq - app) / (2.0 * apq);
                double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
                for (int k = 0; k < 3; k++) {
                    double akp = ata[k * 3 + p], akq = ata[k * 3 + q];
                    ata[k * 3 + p] = c * akp - sn * akq;
                    ata[k * 3 + q] = sn * akp + c * akq;
                }
                for (int k = 0; k < 3; k++) {
                    double apk = ata[p * 3 + k], aqk = ata[q * 3 + k];
                    ata[p * 3 + k] = c * apk - sn * aqk;
                    ata[q * 3 + k] = sn * apk + c * aqk;
                }
                for (int k = 0; k < 3; k++) {
                    double vkp = v[k * 3 + p], vkq = v[k * 3 + q];
                    v[k * 3 + p] = c * vkp - sn * vkq;
                    v[k * 3 + q] = sn * vkp + c * vkq;
                }
            }
    }
    int ord[3] = {0, 1, 2};
    double ev[3] = {ata[0], ata[4], ata[8]};
    for (int i = 0; i < 2; i++)
        for (int j = i + 1; j < 3; j++)
            if (ev[ord[j]] > ev[ord[i]]) {
                int t = ord[i];
                ord[i] = ord[j];
                ord[j] = t;
            }
    for (int c = 0; c < 3; c++) {
        s[c] = sqrt(ev[ord[c]] > 0 ? ev[ord[c]] : 0);
        for (int r = 0; r < 3; r++) V[r * 3 + c] = v[r * 3 + ord[c]];
    }
    double u[3][3];
    int have[3] = {0, 0, 0};
    for (int c = 0; c < 3; c++) {
        double col[3];
        for (int r = 0; r < 3; r++) col[r] = a[r * 3 + 0] * V[0 * 3 + c] + a[r * 3 + 1] * V[1 * 3 + c] + a[r * 3 + 2] * V[2 * 3 + c];
        double nrm = sqrt(col[0] * col[0] + col[1] * col[1] + col[2] * col[2]);
        if (s[0] > 0 && nrm > 1e-12 * s[0] && nrm > 1e-300) {
            for (int r = 0; r < 3; r++) u[c][r] = col[r] / nrm;
            have[c] = 1;
        }
    }
    for (int c = 0; c < 3; c++) {
        if (have[c]) continue;
        int c1 = (c + 1) % 3, c2 = (c + 2) % 3;
        double wv[3];
        if (have[c1] && have[c2]) {
            wv[0] = u[c1][1] * u[c2][2] - u[c1][2] * u[c2][1];
            wv[1] = u[c1][2] * u[c2][0] - u[c1][0] * u[c2][2];
            wv[2] = u[c1][0] * u[c2][1] - u[c1][1] * u[c2][0];
        } else {
            double best = -1;
            wv[0] = wv[1] = wv[2] = 0;
            for (int e = 0; e < 3; e++) {
                double cand[3] = {0, 0, 0};
                cand[e] = 1;
                for (int o = 0; o < 3; o++)
                    if (have[o]) {
                        double d = cand[0] * u[o][0] + cand[1] * u[o][1] + cand[2] * u[o][2];
                        for (int r = 0; r < 3; r++) cand[r] -= d * u[o][r];
                    }
                double n2 = cand[0] * cand[0] + cand[1] * cand[1] + cand[2] * cand[2];
                if (n2 > best) {
                    best = n2;
                    wv[0] = cand[0]; wv[1] = cand[1]; wv[2] = cand[2];
                }
            }
        }
        double n = sqrt(wv[0] * wv[0] + wv[1] * wv[1] + wv[2] * wv[2]);
        for (int r = 0; r < 3; r++) u[c][r] = wv[r] / n;
        have[c] = 1;
    }
    for (int c = 0; c < 3; c++)
        for (int r = 0; r < 3; r++) U[r * 3 + c] = u[c][r];
}

// icp.rs:210-270 from the f64 sums (centroids and H formed here)
__device__ void solve_p2p(const double *sums, double m, float *R, float *t) {
    double sc[3], tc[3], H[9];
    for (int a = 0; a < 3; a++) {
        sc[a] = sums[a] / m;
        tc[a] = sums[3 + a] / m;
    }
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) H[r * 3 + c] = sums[6 + r * 3 + c] - m * sc[r] * tc[c];
    float hf[9];
    for (int i = 0; i < 9; i++) hf[i] = (float)H[i];  // the reference's H is f32
    double hd[9], U[9], S[3], V[9];
    for (int i = 0; i < 9; i++) hd[i] = hf[i];
    svd3(hd, U, S, V);
    float u[9], vt[9], v[9], ut[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            u[i * 3 + j] = (float)U[i * 3 + j];
            vt[i * 3 + j] = (float)V[j * 3 + i];
        }
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            v[i * 3 + j] = vt[j * 3 + i];
            ut[i * 3 + j] = u[j * 3 + i];
        }
    float vut[9];
    mat3_mul_f32(v, ut, vut);
    float det = vut[0] * (vut[4] * vut[8] - vut[5] * vut[7]) - vut[1] * (vut[3] * vut[8] - vut[5] * vut[6]) +
                vut[2] * (vut[3] * vut[7] - vut[4] * vut[6]);
    if (det < 0.0f) {  // icp.rs:253-261
        vt[6] = -vt[6]; vt[7] = -vt[7]; vt[8] = -vt[8];
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) v[i * 3 + j] = vt[j * 3 + i];
    }
    mat3_mul_f32(v, ut, R);
    float scf[3] = {(float)sc[0], (float)sc[1], (float)sc[2]}, tcf[3] = {(float)tc[0], (float)tc[1], (float)tc[2]};
    for (int i = 0; i < 3; i++)  // icp.rs:264
        t[i] = __fsub_rn(tcf[i], __fadd_rn(__fadd_rn(__fmul_rn(R[i * 3 + 0], scf[0]), __fmul_rn(R[i * 3 + 1], scf[1])),
                                           __fmul_rn(R[i * 3 + 2], scf[2])));
}

// icp_plane.rs:183-236 from the accumulated normal equations
__device__ void solve_p2plane(const double *sums, float *R, float *t) {
    double ata[36], atb[6];
    int o = 0;
    for (int r = 0; r < 6; r++)
        for (int c = r; c < 6; c++) {
            ata[r * 6 + c] = sums[o];
            ata[c * 6 + r] = sums[o];
            o++;
        }
    for (int r = 0; r < 6; r++) atb[r] = sums[21 + r];
    double diag_max = 0.0;
    for (int i = 0; i < 6; i++) diag_max = fmax(diag_max, fabs(ata[i * 6 + i]));
    const double lambda = 1e-6 * fmax(diag_max, 1e-12);
    for (int i = 0; i < 6; i++) ata[i * 6 + i] += lambda;
    for (int i = 0; i < 9; i++) R[i] = (i % 4 == 0) ? 1.f : 0.f;
    t[0] = t[1] = t[2] = 0.f;
    double xs[6];
    bool solved = false;
    {
        double L[36];
        for (int i = 0; i < 36; i++) L[i] = 0.0;
        bool ok = true;
        for (int j = 0; j < 6 && ok; j++) {
            double d = ata[j * 6 + j];
            for (int k = 0; k < j; k++) d -= L[j * 6 + k] * L[j * 6 + k];
            if (!(d > 0.0)) {
                ok = false;
                break;
            }
            L[j * 6 + j] = sqrt(d);
            for (int i = j + 1; i < 6; i++) {
                double v = ata[i * 6 + j];
                for (int k = 0; k < j; k++) v -= L[i * 6 + k] * L[j * 6 + k];
                L[i * 6 + j] = v / L[j * 6 + j];
            }
        }
        if (ok) {
            double yv[6];
            for (int i = 0; i < 6; i++) {
                double v = atb[i];
                for (int k = 0; k < i; k++) v -= L[i * 6 + k] * yv[k];
                yv[i] = v / L[i * 6 + i];
            }
            for (int i = 5; i >= 0; i--) {
                double v = yv[i];
                for (int k = i + 1; k < 6; k++) v -= L[k * 6 + i] * xs[k];
                xs[i] = v / L[i * 6 + i];
            }
            solved = true;
        }
    }
    if (!solved) {  // LU with partial pivoting
        double A[36], b[6];
        for (int i = 0; i < 36; i++) A[i] = ata[i];
        for (int i = 0; i < 6; i++) b[i] = atb[i];
        bool ok = true;
        for (int c = 0; c < 6 && ok; c++) {
            int piv = c;
            for (int r = c + 1; r < 6; r++)
                if (fabs(A[r * 6 + c]) > fabs(A[piv * 6 + c])) piv = r;
            if (A[piv * 6 + c] == 0.0 || !isfinite(A[piv * 6 + c])) {
                ok = false;
                break;
            }
            if (piv != c) {
                for (int k = 0; k < 6; k++) {
                    double tmp = A[c * 6 + k];
                    A[c * 6 + k] = A[piv * 6 + k];
                    A[piv * 6 + k] = tmp;
                }
                double tmp = b[c];
                b[c] = b[piv];
                b[piv] = tmp;
            }
            for (int r = c + 1; r < 6; r++) {
                double f = A[r * 6 + c] / A[c * 6 + c];
                for (int k = c; k < 6; k++) A[r * 6 + k] -= f * A[c * 6 + k];
                b[r] -= f * b[c];
            }
        }
        if (!ok) return;  // identity
        for (int i = 5; i >= 0; i--) {
            double v = b[i];
            for (int k = i + 1; k < 6; k++) v -= A[i * 6 + k] * xs[k];
            xs[i] = v / A[i * 6 + i];
        }
    }
    const float alpha = (float)xs[0], beta = (float)xs[1], gamma = (float)xs[2];
    const float angle = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(alpha, alpha), __fmul_rn(beta, beta)), __fmul_rn(gamma, gamma)));
    if (angle < 1e-10f) {
        R[0] = 1.0f; R[1] = -gamma; R[2] = beta;
        R[3] = gamma; R[4] = 1.0f; R[5] = -alpha;
        R[6] = -beta; R[7] = alpha; R[8] = 1.0f;
    } else {
        const float ax = __fdiv_rn(alpha, angle), ay = __fdiv_rn(beta, angle), az = __fdiv_rn(gamma, angle);
        const float c = cosf(angle), s = sinf(angle), tt = __fsub_rn(1.0f, c);
        // t*ax*ax + c etc., left to right
        auto m3 = [](float a, float b, float cc) { return __fmul_rn(__fmul_rn(a, b), cc); };
        R[0] = __fadd_rn(m3(tt, ax, ax), c);
        R[1] = __fsub_rn(m3(tt, ax, ay), __fmul_rn(s, az));
        R[2] = __fadd_rn(m3(tt, ax, az), __fmul_rn(s, ay));
        R[3] = __fadd_rn(m3(tt, ax, ay), __fmul_rn(s, az));
        R[4] = __fadd_rn(m3(tt, ay, ay), c);
        R[5] = __fsub_rn(m3(tt, ay, az), __fmul_rn(s, ax));
        R[6] = __fsub_rn(m3(tt, ax, az), __fmul_rn(s, ay));
        R[7] = __fadd_rn(m3(tt, ay, az), __fmul_rn(s, ax));
        R[8] = __fadd_rn(m3(tt, az, az), c);
    }
    t[0] = (float)xs[3];
    t[1] = (float)xs[4];
    t[2] = (float)xs[5];
}

// Convergence test, solve, compose (icp.rs:154-187 / icp_plane.rs:55-79) of one registration, on one thread.
// Returns true when this step finished it (state->done was just set).
template <bool kPlane>
__device__ __forceinline__ bool icp_step(IcpState *state, int metrics_only, float tolerance) {
    if (state->done) return false;
    const double m = state->sums[kCount];
    const double ns = state->sums[kSrcN];
    if (metrics_only) {  // max_iterations == 0: icp.rs:190-197
        if (m > 0.0) {
            state->last_rmse = __fsqrt_rn(__fdiv_rn((float)state->sums[kSumSq], (float)m));
            state->last_fitness = __fdiv_rn((float)m, (float)ns);
        }
        state->done = 1;
        return true;
    }
    state->num_iterations += 1;
    if (!(m > 0.0)) {  // no correspondences: break
        state->done = 1;
        return true;
    }
    const float rmse = __fsqrt_rn(__fdiv_rn((float)state->sums[kSumSq], (float)m));
    state->last_rmse = rmse;
    state->last_fitness = __fdiv_rn((float)m, (float)ns);
    if (fabsf(__fsub_rn(state->prev_rmse, rmse)) < tolerance) {
        state->converged = 1;
        state->done = 1;
        return true;
    }
    state->prev_rmse = rmse;
    float R[9], t[3];
    if (kPlane) solve_p2plane(state->sums, R, t);
    else solve_p2p(state->sums, m, R, t);
    // cumulative = cumulative.compose(incremental): R = R_inc * R_cum, t = R_inc * t_cum + t_inc
    float cr[9], ct[3];
    for (int i = 0; i < 9; i++) cr[i] = state->cum_R[i];
    for (int i = 0; i < 3; i++) ct[i] = state->cum_t[i];
    float nr[9], nt[3];
    mat3_mul_f32(R, cr, nr);
    for (int i = 0; i < 3; i++)
        nt[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(R[i * 3 + 0], ct[0]), __fmul_rn(R[i * 3 + 1], ct[1])),
                                    __fmul_rn(R[i * 3 + 2], ct[2])),
                          t[i]);
    for (int i = 0; i < 9; i++) {
        state->cum_R[i] = nr[i];
        state->inc_R[i] = R[i];
    }
    for (int i = 0; i < 3; i++) {
        state->cum_t[i] = nt[i];
        state->inc_t[i] = t[i];
    }
    state->has_inc = 1;
    return false;
}

template <bool kPlane>
__global__ void icp_solve_kernel(IcpState *state, int metrics_only, float tolerance, int *host_done_) {
    volatile int *host_done = host_done_;
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (icp_step<kPlane>(state, metrics_only, tolerance)) *host_done = 1;
}

__device__ __forceinline__ void icp_init_state(IcpState *s) {
    for (int i = 0; i < 9; i++) {
        s->inc_R[i] = s->cum_R[i] = (i % 4 == 0) ? 1.f : 0.f;
    }
    for (int i = 0; i < 3; i++) s->inc_t[i] = s->cum_t[i] = 0.f;
    s->prev_rmse = INFINITY;
    s->last_rmse = INFINITY;
    s->last_fitness = 0.f;
    s->has_inc = 0;
    s->converged = 0;
    s->done = 0;
    s->num_iterations = 0;
    for (int i = 0; i < NP; i++) s->sums[i] = 0.0;
}

// kInit: cumulative = init, no increment pending (the working copy was moved by init when it was binned)
__device__ __forceinline__ void icp_seed_state(IcpState *s, const float *R, const float *t) {
    for (int i = 0; i < 9; i++) s->cum_R[i] = R[i];
    for (int i = 0; i < 3; i++) s->cum_t[i] = t[i];
}

template <bool kInit>
__global__ void icp_init_state_kernel(IcpState *s, Xform init) {
    if (threadIdx.x != 0) return;
    icp_init_state(s);
    if (kInit) icp_seed_state(s, init.R, init.t);
}

__global__ void pack_normals_kernel(const float *__restrict__ nx, const float *__restrict__ ny, const float *__restrict__ nz,
                                    size_t n, float4 *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_float4(nx[i], ny[i], nz[i], 0.f);
}

// ---- batch of (source, target) frame pairs ----------------------------------------------------------------
// All pairs of one call run through the same launches.  Pair q (of the pairs with a non-empty source and target) owns
//   - the working-copy range [cur_off[q], cur_off[q+1]): its source frame, binned by the cells of its target frame;
//   - the accumulation blocks [blk_off[q], blk_off[q+1]): min(ceil(ns / 256), 4 SMs) of them, as in icp_dev, so its
//     partition (and with it every bit of its result) does not depend on the other pairs of the call;
//   - states[q], and grid tgt_frame[q] in every level of the multi-frame target index.
// Threads resolve their pair by a binary search over cur_off (blocks: over blk_off).
struct IcpBatchPairs {
    const uint32_t *cur_off;    // [n_pairs + 1]
    const uint32_t *blk_off;    // [n_pairs + 1]
    const uint32_t *tgt_frame;  // [n_pairs]
    const uint32_t *src_begin;  // [n_pairs]: first input point of the source frame
    int n_pairs;
};

// Binning, deterministic: key (pair, target cell) for every working-copy point, in working-copy order, then the stable
// radix sort; a cell's points end up in source order.  Non-finite points go to cell 0, as in src_count_kernel.
// kInit: pair q's points are moved by inits[12q .. 12q + 12) before they are binned and stored (see src_count_kernel).
template <bool kInit>
__global__ void __launch_bounds__(256) icp_batch_bin_key_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                const float *__restrict__ z, IcpBatchPairs bp, uint32_t total,
                                                                const GridDesc *__restrict__ grids, int cell_bits,
                                                                unsigned long long *__restrict__ keys, uint32_t *__restrict__ vals,
                                                                const float *__restrict__ inits) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int q = frame_of(bp.cur_off, bp.n_pairs, i);
    const uint32_t gi = bp.src_begin[q] + (i - bp.cur_off[q]);
    const GridDesc g = grids[bp.tgt_frame[q]];
    float px = x[gi], py = y[gi], pz = z[gi];
    if (kInit) apply_point(inits + 12 * q, inits + 12 * q + 9, px, py, pz, px, py, pz);
    uint32_t cid = 0;
    if (finite3(px, py, pz) && g.n_cells > 0) {
        const int c0 = cell_coord(g, 0, pick_axis(g.ax[0], px, py, pz), nullptr);
        const int c1 = cell_coord(g, 1, pick_axis(g.ax[1], px, py, pz), nullptr);
        const int c2 = cell_coord(g, 2, pick_axis(g.ax[2], px, py, pz), nullptr);
        cid = cell_linear(g, c0, c1, c2) - g.cell_base;
    }
    keys[i] = ((unsigned long long)q << cell_bits) | cid;
    vals[i] = gi;
}

template <bool kInit>
__global__ void __launch_bounds__(256) icp_batch_bin_gather_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                   const float *__restrict__ z, IcpBatchPairs bp, uint32_t total,
                                                                   int cell_bits, const unsigned long long *__restrict__ keys,
                                                                   const uint32_t *__restrict__ vals, float4 *__restrict__ cur,
                                                                   const float *__restrict__ inits) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint32_t q = (uint32_t)(keys[i] >> cell_bits), gi = vals[i];
    float px = x[gi], py = y[gi], pz = z[gi];
    if (kInit) apply_point(inits + 12 * q, inits + 12 * q + 9, px, py, pz, px, py, pz);
    cur[i] = make_float4(px, py, pz, __uint_as_float(gi - bp.src_begin[q]));
}

template <bool kInit>
__global__ void icp_batch_init_kernel(IcpState *states, int n_pairs, unsigned *active, const float *__restrict__ inits) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n_pairs) {
        icp_init_state(states + q);
        if (kInit) icp_seed_state(states + q, inits + 12 * q, inits + 12 * q + 9);
    }
    if (q == 0) *active = (unsigned)n_pairs;
}

__global__ void __launch_bounds__(kIcpThreads) icp_batch_search_kernel(const GridDesc *__restrict__ grids,
                                                                       const uint32_t *__restrict__ cell_start,
                                                                       const float4 *__restrict__ sorted,
                                                                       const float4 *__restrict__ tgt4, float4 *__restrict__ cur,
                                                                       uint32_t total, IcpBatchPairs bp,
                                                                       const IcpState *__restrict__ states,
                                                                       unsigned long long *__restrict__ nn,
                                                                       uint32_t *__restrict__ defer_list,
                                                                       uint32_t *__restrict__ defer_count, int last_level) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int q = frame_of(bp.cur_off, bp.n_pairs, i);
    const IcpState *state = states + q;
    if (state->done) return;  // a finished pair
    const GridDesc g = grids[bp.tgt_frame[q]];
    icp_search_point(g, cell_start, sorted, tgt4, cur, i, state, nn, defer_list, defer_count, last_level);
}

// the deferred lists hold points of unfinished pairs only (the search kernel skips the finished ones)
__global__ void __launch_bounds__(128) icp_batch_deferred_kernel(const GridDesc *__restrict__ grids,
                                                                 const uint32_t *__restrict__ cell_start,
                                                                 const float4 *__restrict__ pts, const float4 *__restrict__ cur,
                                                                 IcpBatchPairs bp, const uint32_t *__restrict__ in_list,
                                                                 const uint32_t *__restrict__ in_count,
                                                                 unsigned long long *__restrict__ nn, uint32_t *__restrict__ out_list,
                                                                 uint32_t *__restrict__ out_count, int last_level) {
    const uint32_t n = *in_count;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    RegTopK tk;
    tk.kk = 1;
    tk.lane = threadIdx.x & 31;
    for (uint32_t j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < n; j += warps) {
        const uint32_t i = in_list[j];
        const GridDesc g = grids[bp.tgt_frame[frame_of(bp.cur_off, bp.n_pairs, i)]];
        icp_deferred_point(tk, g, cell_start, pts, cur, i, nn, out_list, out_count, last_level);
    }
}

template <bool kPlane>
__global__ void __launch_bounds__(kIcpThreads) icp_batch_accum_kernel(const float4 *__restrict__ tgt4, const float4 *__restrict__ nrm4,
                                                                      const float4 *__restrict__ cur,
                                                                      const unsigned long long *__restrict__ nn, IcpBatchPairs bp,
                                                                      float max_distance, const IcpState *__restrict__ states,
                                                                      double *__restrict__ partials) {
    const int q = frame_of(bp.blk_off, bp.n_pairs, blockIdx.x);
    if (states[q].done) return;
    const uint32_t b0 = bp.cur_off[q], ns = bp.cur_off[q + 1] - b0;
    const uint32_t nb = bp.blk_off[q + 1] - bp.blk_off[q], lb = blockIdx.x - bp.blk_off[q];
    double acc[NP];
#pragma unroll
    for (int j = 0; j < NP; j++) acc[j] = 0.0;
    for (size_t i = (size_t)lb * blockDim.x + threadIdx.x; i < ns; i += (size_t)nb * blockDim.x)
        icp_accum_point<kPlane>(acc, tgt4, nrm4, cur + b0, nn + b0, i, max_distance);
    icp_block_partials(acc, partials + (size_t)blockIdx.x * NP);
}

// one block per pair: its partials folded exactly as icp_reduce_kernel folds them for one GPU
__global__ void __launch_bounds__(NP * 32) icp_batch_reduce_kernel(const double *__restrict__ partials, IcpBatchPairs bp,
                                                                   IcpState *states) {
    const int q = blockIdx.x;
    IcpState *state = states + q;
    if (state->done) return;
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t b0 = bp.blk_off[q];
    double v = icp_fold_partials(partials + (size_t)b0 * NP, (int)(bp.blk_off[q + 1] - b0), j, lane);
    v = j == kSrcN ? (double)(bp.cur_off[q + 1] - bp.cur_off[q]) : v;
    if (lane == 0) state->sums[j] = v;
}

// one thread per pair; the pair that finishes last raises the host flag
template <bool kPlane>
__global__ void icp_batch_solve_kernel(IcpState *states, int n_pairs, int metrics_only, float tolerance, unsigned *active,
                                       int *host_done_) {
    volatile int *host_done = host_done_;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_pairs) return;
    if (icp_step<kPlane>(states + q, metrics_only, tolerance) && atomicSub(active, 1u) == 1u) *host_done = 1;
}

}  // namespace

int apply_transform_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, const float R[9],
                        const float t[3], float *ox, float *oy, float *oz) {
    if (n == 0) return PCR_OK;
    PCR_TRY(ensure(ctx, ctx->b_small, 4096));
    float h[12];
    memcpy(h, R, sizeof(float) * 9);
    memcpy(h + 9, t, sizeof(float) * 3);
    float *d_rt = (float *)((char *)ctx->b_small.p + 2048);
    PCR_TRY(ensure_pinned(ctx, 4096));
    memcpy((char *)ctx->pinned + 2048, h, sizeof(h));
    PCR_CUDA(ctx, cudaMemcpyAsync(d_rt, (char *)ctx->pinned + 2048, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    apply_transform_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dx, dy, dz, n, d_rt, ox, oy, oz);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

int apply_transform_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                              const uint32_t *d_frame_off, const float *transforms, float *ox, float *oy, float *oz) {
    const size_t n = (size_t)frame_offsets[n_frames];
    if (n == 0) return PCR_OK;
    // transforms (12 f32 per frame), then the u32 offsets unless the caller has them on the device: one pageable staging
    // copy, so the caller's arrays are free again when the call returns
    std::vector<uint32_t> h(12 * n_frames + (d_frame_off ? 0 : n_frames + 1));
    memcpy(h.data(), transforms, sizeof(float) * 12 * n_frames);
    if (!d_frame_off)
        for (size_t f = 0; f <= n_frames; f++) h[12 * n_frames + f] = (uint32_t)frame_offsets[f];
    StreamAlloc<uint32_t> mem(ctx->stream);
    PCR_CUDA(ctx, mem.alloc(sizeof(uint32_t) * h.size()));
    PCR_CUDA(ctx, cudaMemcpyAsync(mem.p, h.data(), sizeof(uint32_t) * h.size(), cudaMemcpyHostToDevice, ctx->stream));
    const float *d_rt = (const float *)mem.p;
    const uint32_t *d_off = d_frame_off ? d_frame_off : mem.p + 12 * n_frames;
    apply_transform_batch_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dx, dy, dz, n, d_rt, d_off, (int)n_frames, ox, oy, oz);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

int find_correspondences_dev(Index *target, const float *dsx, const float *dsy, const float *dsz, size_t ns,
                             float max_distance, uint32_t *d_tgt, float *d_dist, const QueryFrames *qf) {
    Ctx *ctx = target->ctx;
    if (ns == 0) return PCR_OK;
    PCR_TRY(ensure(ctx, ctx->b_misc2, ns * sizeof(uint32_t)));
    uint32_t *d_cnt = (uint32_t *)ctx->b_misc2.p;
    PCR_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, ns * sizeof(uint32_t), ctx->stream));
    PCR_TRY(knn_queries_dev(target, dsx, dsy, dsz, ns, 1, d_tgt, d_dist, d_cnt, qf));  // correspondence.rs:25
    correspond_filter_kernel<<<(unsigned)((ns + 255) / 256), 256, 0, ctx->stream>>>(ns, max_distance, d_tgt, d_dist, d_cnt);
    PCR_LAUNCH_CHECK(ctx);
    return PCR_OK;
}

int icp_dev(Ctx *ctx, const IcpArgs &a, pcr_icp_result *result) {
    cudaStream_t st = ctx->stream;
    const bool plane = a.d_nx != nullptr;
    // the start (identity or init) and the empty cases are handled by the caller (api.cu); here nt > 0
    Index *tgt = nullptr;
    BuildOpts bo;
    bo.k_hint = 1;
    bo.transient = true;
    PCR_TRY(index_build_dev(ctx, a.d_tx, a.d_ty, a.d_tz, a.nt, bo, &tgt));
    const IndexPtr guard(tgt);

    const size_t ns = a.ns;
    Xform init = {};
    if (a.init) memcpy(&init, a.init, sizeof(init));
    // working copy of the source (moved by init), binned by target cell
    StreamAlloc<float4> cur_mem(st), nrm4_mem(st);
    PCR_CUDA(ctx, cur_mem.alloc(sizeof(float4) * std::max<size_t>(ns, 1)));
    float4 *cur = cur_mem.p, *nrm4 = nullptr;
    if (plane) {
        PCR_CUDA(ctx, nrm4_mem.alloc(sizeof(float4) * a.nt));
        nrm4 = nrm4_mem.p;
        pack_normals_kernel<<<(unsigned)((a.nt + 255) / 256), 256, 0, st>>>(a.d_nx, a.d_ny, a.d_nz, a.nt, nrm4);
        PCR_LAUNCH_CHECK(ctx);
    }
    if (ns > 0) {
        const size_t cells = (size_t)tgt->total_cells + 1;
        PCR_TRY(ensure(ctx, ctx->b_table, sizeof(uint32_t) * cells));
        PCR_TRY(ensure(ctx, ctx->b_misc, sizeof(uint32_t) * 2 * ns));
        uint32_t *table = (uint32_t *)ctx->b_table.p;
        uint32_t *cid = (uint32_t *)ctx->b_misc.p, *rank = cid + ns;
        PCR_CUDA(ctx, cudaMemsetAsync(table, 0, sizeof(uint32_t) * cells, st));
        (a.init ? src_count_kernel<true> : src_count_kernel<false>)<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(
            a.d_sx, a.d_sy, a.d_sz, ns, tgt->grids, table, cid, rank, init);
        PCR_LAUNCH_CHECK(ctx);
        PCR_TRY(exclusive_scan_u32_dev(ctx, table, cells));
        (a.init ? src_scatter_kernel<true> : src_scatter_kernel<false>)<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(
            a.d_sx, a.d_sy, a.d_sz, ns, table, cid, rank, cur, init);
        PCR_LAUNCH_CHECK(ctx);
    }

    // coarser levels of the target grid for deferred source points (built once, reused every iteration)
    Index *levels[kMaxLevels] = {tgt, nullptr, nullptr, nullptr};
    for (int l = 1; l < kMaxLevels; l++) PCR_TRY(index_coarser_level(levels[l - 1], &levels[l]));
    StreamAlloc<unsigned long long> nn_mem(st);
    PCR_CUDA(ctx, nn_mem.alloc(sizeof(unsigned long long) * std::max<size_t>(ns, 1)));
    StreamAlloc<uint32_t> dlist_mem(st);  // 2 ping-pong lists of ns entries + counters
    PCR_CUDA(ctx, dlist_mem.alloc(sizeof(uint32_t) * (2 * std::max<size_t>(ns, 1) + 64)));
    unsigned long long *nn = nn_mem.p;
    uint32_t *dlist = dlist_mem.p;
    uint32_t *dcount = dlist;  // [kMaxLevels]
    uint32_t *dl[2] = {dlist + 64, dlist + 64 + std::max<size_t>(ns, 1)};

    const int n_blocks = (int)std::max<size_t>(1, std::min<size_t>((ns + kIcpThreads - 1) / kIcpThreads, (size_t)ctx->sm_count * 4));
    PCR_TRY(ensure(ctx, ctx->b_small, 8192 + sizeof(IcpState)));
    PCR_TRY(ensure(ctx, ctx->b_misc2, sizeof(double) * NP * (size_t)n_blocks));
    PCR_TRY(ensure_pinned(ctx, 8192 + sizeof(IcpState)));
    IcpState *d_state = (IcpState *)((char *)ctx->b_small.p + 8192);
    IcpState *h_state = (IcpState *)((char *)ctx->pinned + 8192);
    volatile int *h_done = (volatile int *)ctx->pinned;  // device-visible through UVA
    *h_done = 0;
    double *partials = (double *)ctx->b_misc2.p;
    (a.init ? icp_init_state_kernel<true> : icp_init_state_kernel<false>)<<<1, 32, 0, st>>>(d_state, init);
    PCR_LAUNCH_CHECK(ctx);

    auto one_pass = [&](int metrics_only) -> int {
        {
            TimeScope ts(ctx, kTagIcpStep);
            PCR_CUDA(ctx, cudaMemsetAsync(dcount, 0, sizeof(uint32_t) * kMaxLevels, st));
            if (ns > 0) {
                icp_search_kernel<<<(unsigned)((ns + kIcpThreads - 1) / kIcpThreads), kIcpThreads, 0, st>>>(
                    tgt->grids, tgt->cell_start, tgt->sorted, tgt->orig4, cur, ns, d_state, nn, dl[0], dcount + 0, 0);
                PCR_LAUNCH_CHECK(ctx);
                // deferred points on the coarser levels, warp per point (no host round trip: the list lengths stay on
                // the device).  The warp search is seeded with nn[i] and skips rows / cells beyond the current best.
                // (Measured and dropped: thread-per-point on the coarse levels, 1.8x slower; a seeded thread-per-point
                // ball scan on the fine grid before the coarse levels, 0.43 -> 0.47-0.52 ms per iteration.)
                for (int l = 1; l < kMaxLevels; l++) {
                    const bool last = l == kMaxLevels - 1;
                    // level 1 may hold 10-20 % of a badly aligned source: give it more resident warps
                    icp_deferred_kernel<<<ctx->sm_count * (l == 1 ? 8 : 2), 128, 0, st>>>(
                        levels[l]->grids, levels[l]->cell_start, levels[l]->sorted, cur, d_state, dl[(l - 1) & 1], dcount + (l - 1), nn,
                        dl[l & 1], dcount + l, last ? 1 : 0);
                    PCR_LAUNCH_CHECK(ctx);
                }
            }
            if (plane)
                icp_accum_kernel<true><<<n_blocks, kIcpThreads, 0, st>>>(tgt->orig4, nrm4, cur, nn, ns,
                                                                         a.params.max_correspondence_distance, d_state, partials);
            else
                icp_accum_kernel<false><<<n_blocks, kIcpThreads, 0, st>>>(tgt->orig4, nullptr, cur, nn, ns,
                                                                          a.params.max_correspondence_distance, d_state, partials);
            PCR_LAUNCH_CHECK(ctx);
        }
        if (getenv("PCR_DEBUG")) {
            uint32_t hc[kMaxLevels];
            cudaMemcpyAsync(hc, dcount, sizeof(hc), cudaMemcpyDeviceToHost, st);
            cudaStreamSynchronize(st);
            fprintf(stderr, "[pcr] icp pass: deferred per level %u %u %u %u of %zu (cells %.3g / %.3g)\n", hc[0], hc[1], hc[2], hc[3], ns,
                    levels[0]->grids_h[0].h, levels[1]->grids_h[0].h);
        }
        TimeScope ts2(ctx, kTagIcpSolve);
        const bool peer = ctx->world > 1 && ctx->peer_ok;
        PeerComm pc = {};
        if (peer) pc = ctx->peer;
        icp_reduce_kernel<<<1, NP * 32, 0, st>>>(partials, n_blocks, ns, d_state, pc, peer ? ++ctx->peer_seq : 0ull);
        PCR_LAUNCH_CHECK(ctx);
        if (ctx->world > 1 && !peer) PCR_TRY(comm_allreduce_f64(ctx, d_state->sums, NP));
        if (plane) icp_solve_kernel<true><<<1, 32, 0, st>>>(d_state, metrics_only, a.params.tolerance, (int *)h_done);
        else icp_solve_kernel<false><<<1, 32, 0, st>>>(d_state, metrics_only, a.params.tolerance, (int *)h_done);
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    };

    if (a.params.max_iterations == 0) {
        PCR_TRY(one_pass(1));
    } else {
        // Sharded: every rank must enqueue the same number of all-reduces, so the ranks decide in lock step -- but only
        // every kSyncEvery passes: after the all-reduce every rank solves the same system and raises its flag in the
        // same pass, so at a pass boundary all ranks read the same value; the passes queued after convergence are no-ops
        // on the device (at most kSyncEvery - 1 of them).  One sync per pass left the GPU idle for ~0.2 ms per iteration.
        constexpr uint64_t kSyncEvery = 4;
        for (uint64_t it = 0; it < a.params.max_iterations; it++) {
            if (ctx->world > 1) {
                if (it && it % kSyncEvery == 0) {
                    PCR_CUDA(ctx, cudaStreamSynchronize(st));
                    if (*h_done) break;
                }
            } else if (*h_done) {
                break;  // the device has finished; later passes would be no-ops
            }
            PCR_TRY(one_pass(0));
            if (ctx->world == 1 && (it & 3) == 3) cudaStreamQuery(st);  // flush, so the flag is seen soon after convergence
        }
    }
    PCR_CUDA(ctx, cudaMemcpyAsync(h_state, d_state, sizeof(IcpState), cudaMemcpyDeviceToHost, st));
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    memcpy(result->rotation, h_state->cum_R, sizeof(float) * 9);
    memcpy(result->translation, h_state->cum_t, sizeof(float) * 3);
    result->fitness = h_state->last_fitness;
    result->rmse = h_state->last_rmse;
    result->converged = h_state->converged;
    result->num_iterations = h_state->num_iterations;
    return PCR_OK;
}

// Many (source frame, target frame) pairs in one device-resident loop: one multi-frame index (and its coarser levels)
// over every frame, one working copy per pair, and per pass the same seven launches as icp_dev for all pairs together.
// The host waits only for the index build and the results.  No communication: each rank registers its own pairs.
int icp_batch_dev(Ctx *ctx, const IcpBatchArgs &a, pcr_icp_result *results) {
    cudaStream_t st = ctx->stream;
    const bool plane = a.d_nx != nullptr;
    const uint64_t *off = a.frame_offsets;
    // pairs with an empty side are answered here (icp.rs:131-139: the guess the caller stored, 0 iterations); the
    // others are numbered q = 0 .. Q - 1
    std::vector<uint32_t> act, cur_off(1, 0), blk_off(1, 0), tgt_frame, src_begin;
    const uint64_t blk_cap = (uint64_t)ctx->sm_count * 4;
    for (size_t p = 0; p < a.n_pairs; p++) {
        const uint32_t s = a.pairs[2 * p], t = a.pairs[2 * p + 1];
        const uint64_t ns = off[s + 1] - off[s], nt = off[t + 1] - off[t];
        if (ns == 0 || nt == 0) {
            results[p].converged = (ns == 0 && nt == 0) ? 1 : 0;
            continue;
        }
        act.push_back((uint32_t)p);
        cur_off.push_back(cur_off.back() + (uint32_t)ns);  // (the caller checked that the sum stays below 2^31)
        blk_off.push_back(blk_off.back() + (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((ns + kIcpThreads - 1) / kIcpThreads, blk_cap)));
        tgt_frame.push_back(t);
        src_begin.push_back((uint32_t)off[s]);
    }
    const int Q = (int)act.size();
    if (Q == 0) return PCR_OK;
    const uint32_t total = cur_off.back(), n_blocks = blk_off.back();

    Index *tgt = nullptr;
    BuildOpts bo;
    bo.k_hint = 1;
    bo.transient = true;
    bo.n_frames = (int)a.n_frames;
    bo.frame_offsets = a.frame_offsets;
    PCR_TRY(index_build_dev(ctx, a.d_x, a.d_y, a.d_z, a.n, bo, &tgt));
    const IndexPtr guard(tgt);
    Index *levels[kMaxLevels] = {tgt, nullptr, nullptr, nullptr};
    for (int l = 1; l < kMaxLevels; l++) PCR_TRY(index_coarser_level(levels[l - 1], &levels[l]));

    // one allocation: working copy | nn | deferred lists (counters, active-pair counter, 2 lists) | partials | states |
    // pair table | packed normals
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o_nn = up(sizeof(float4) * total);
    const size_t o_dl = o_nn + up(sizeof(unsigned long long) * total);
    const size_t o_part = o_dl + up(sizeof(uint32_t) * (64 + 2 * (size_t)total));
    const size_t o_state = o_part + up(sizeof(double) * NP * (size_t)n_blocks);
    const size_t o_tab = o_state + up(sizeof(IcpState) * Q);
    const size_t tab_words = 4 * (size_t)Q + 2 + (a.inits ? 12 * (size_t)Q : 0);  // (+ the guesses of the pairs)
    const size_t o_nrm = o_tab + up(sizeof(uint32_t) * tab_words);
    const size_t bytes = o_nrm + (plane ? sizeof(float4) * a.n : 0);
    StreamAlloc<char> mem_alloc(st);
    PCR_CUDA(ctx, mem_alloc.alloc(bytes));
    char *mem = mem_alloc.p;
    float4 *cur = (float4 *)mem;
    unsigned long long *nn = (unsigned long long *)(mem + o_nn);
    uint32_t *dcount = (uint32_t *)(mem + o_dl);  // [kMaxLevels]
    unsigned *active = dcount + 32;
    uint32_t *dl[2] = {dcount + 64, dcount + 64 + total};
    double *partials = (double *)(mem + o_part);
    IcpState *d_states = (IcpState *)(mem + o_state);
    uint32_t *d_tab = (uint32_t *)(mem + o_tab);
    float4 *nrm4 = plane ? (float4 *)(mem + o_nrm) : nullptr;

    // the pair table goes up through the pinned mailbox (word 0 is the host flag, the table starts at byte 256)
    const size_t state_bytes = sizeof(IcpState) * Q;
    PCR_TRY(ensure_pinned(ctx, 256 + std::max(sizeof(uint32_t) * tab_words, state_bytes)));
    volatile int *h_done = (volatile int *)ctx->pinned;
    *h_done = 0;
    uint32_t *h_tab = (uint32_t *)((char *)ctx->pinned + 256);
    memcpy(h_tab, cur_off.data(), sizeof(uint32_t) * (Q + 1));
    memcpy(h_tab + Q + 1, blk_off.data(), sizeof(uint32_t) * (Q + 1));
    memcpy(h_tab + 2 * Q + 2, tgt_frame.data(), sizeof(uint32_t) * Q);
    memcpy(h_tab + 3 * Q + 2, src_begin.data(), sizeof(uint32_t) * Q);
    if (a.inits)
        for (int q = 0; q < Q; q++) memcpy(h_tab + 4 * Q + 2 + 12 * q, a.inits + 12 * (size_t)act[q], sizeof(float) * 12);
    PCR_CUDA(ctx, cudaMemcpyAsync(d_tab, h_tab, sizeof(uint32_t) * tab_words, cudaMemcpyHostToDevice, st));
    IcpBatchPairs bp;
    bp.cur_off = d_tab;
    bp.blk_off = d_tab + Q + 1;
    bp.tgt_frame = d_tab + 2 * Q + 2;
    bp.src_begin = d_tab + 3 * Q + 2;
    bp.n_pairs = Q;
    const float *d_inits = a.inits ? (const float *)(d_tab + 4 * Q + 2) : nullptr;

    if (plane) {
        pack_normals_kernel<<<(unsigned)((a.n + 255) / 256), 256, 0, st>>>(a.d_nx, a.d_ny, a.d_nz, a.n, nrm4);
        PCR_LAUNCH_CHECK(ctx);
    }
    {  // working copies, binned by target cell in a deterministic order
        TimeScope ts(ctx, kTagOther);
        uint32_t max_cells = 1;
        for (int q = 0; q < Q; q++) max_cells = std::max(max_cells, tgt->grids_h[tgt_frame[q]].n_cells);
        const int cell_bits = bits_for(max_cells);
        const int key_bits = cell_bits + bits_for((uint64_t)Q);
        const size_t hist_words = radix_sort_hist_words(total);
        StreamAlloc<char> sm_alloc(st);
        PCR_CUDA(ctx, sm_alloc.alloc(up(2 * sizeof(unsigned long long) * total) + up(2 * sizeof(uint32_t) * total) + sizeof(uint32_t) * hist_words));
        char *sm = sm_alloc.p;
        unsigned long long *kA = (unsigned long long *)sm, *kB = kA + total;
        uint32_t *vA = (uint32_t *)(sm + up(2 * sizeof(unsigned long long) * total)), *vB = vA + total;
        uint32_t *hist = (uint32_t *)((char *)vA + up(2 * sizeof(uint32_t) * total));
        const unsigned nb = (total + 255) / 256;
        (a.inits ? icp_batch_bin_key_kernel<true> : icp_batch_bin_key_kernel<false>)<<<nb, 256, 0, st>>>(
            a.d_x, a.d_y, a.d_z, bp, total, tgt->grids, cell_bits, kA, vA, d_inits);
        PCR_LAUNCH_CHECK(ctx);
        PCR_TRY(radix_sort_pairs_dev(ctx, &kA, &vA, &kB, &vB, total, key_bits, hist));
        (a.inits ? icp_batch_bin_gather_kernel<true> : icp_batch_bin_gather_kernel<false>)<<<nb, 256, 0, st>>>(
            a.d_x, a.d_y, a.d_z, bp, total, cell_bits, kA, vA, cur, d_inits);
        PCR_LAUNCH_CHECK(ctx);
    }
    (a.inits ? icp_batch_init_kernel<true> : icp_batch_init_kernel<false>)<<<(Q + 127) / 128, 128, 0, st>>>(d_states, Q, active, d_inits);
    PCR_LAUNCH_CHECK(ctx);

    auto one_pass = [&](int metrics_only) -> int {
        {
            TimeScope ts(ctx, kTagIcpStep);
            PCR_CUDA(ctx, cudaMemsetAsync(dcount, 0, sizeof(uint32_t) * kMaxLevels, st));
            icp_batch_search_kernel<<<(total + kIcpThreads - 1) / kIcpThreads, kIcpThreads, 0, st>>>(
                tgt->grids, tgt->cell_start, tgt->sorted, tgt->orig4, cur, total, bp, d_states, nn, dl[0], dcount + 0, 0);
            PCR_LAUNCH_CHECK(ctx);
            for (int l = 1; l < kMaxLevels; l++) {  // (launch sizes as in icp_dev)
                const bool last = l == kMaxLevels - 1;
                icp_batch_deferred_kernel<<<ctx->sm_count * (l == 1 ? 8 : 2), 128, 0, st>>>(
                    levels[l]->grids, levels[l]->cell_start, levels[l]->sorted, cur, bp, dl[(l - 1) & 1], dcount + (l - 1), nn, dl[l & 1],
                    dcount + l, last ? 1 : 0);
                PCR_LAUNCH_CHECK(ctx);
            }
            if (plane)
                icp_batch_accum_kernel<true><<<n_blocks, kIcpThreads, 0, st>>>(tgt->orig4, nrm4, cur, nn, bp,
                                                                               a.params.max_correspondence_distance, d_states, partials);
            else
                icp_batch_accum_kernel<false><<<n_blocks, kIcpThreads, 0, st>>>(tgt->orig4, nullptr, cur, nn, bp,
                                                                                a.params.max_correspondence_distance, d_states, partials);
            PCR_LAUNCH_CHECK(ctx);
        }
        TimeScope ts2(ctx, kTagIcpSolve);
        icp_batch_reduce_kernel<<<Q, NP * 32, 0, st>>>(partials, bp, d_states);
        PCR_LAUNCH_CHECK(ctx);
        if (plane)
            icp_batch_solve_kernel<true><<<(Q + 31) / 32, 32, 0, st>>>(d_states, Q, metrics_only, a.params.tolerance, active, (int *)h_done);
        else
            icp_batch_solve_kernel<false><<<(Q + 31) / 32, 32, 0, st>>>(d_states, Q, metrics_only, a.params.tolerance, active, (int *)h_done);
        PCR_LAUNCH_CHECK(ctx);
        return PCR_OK;
    };

    if (a.params.max_iterations == 0) {
        PCR_TRY(one_pass(1));
    } else {
        for (uint64_t it = 0; it < a.params.max_iterations; it++) {
            if (*h_done) break;  // every pair has finished; later passes would be no-ops
            PCR_TRY(one_pass(0));
            if ((it & 3) == 3) cudaStreamQuery(st);  // flush, so the flag is seen soon after the last pair finishes
        }
    }
    IcpState *h_states = (IcpState *)((char *)ctx->pinned + 256);
    PCR_CUDA(ctx, cudaMemcpyAsync(h_states, d_states, state_bytes, cudaMemcpyDeviceToHost, st));
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    for (int q = 0; q < Q; q++) {
        const IcpState &s = h_states[q];
        pcr_icp_result &r = results[act[q]];
        memcpy(r.rotation, s.cum_R, sizeof(float) * 9);
        memcpy(r.translation, s.cum_t, sizeof(float) * 3);
        r.fitness = s.last_fitness;
        r.rmse = s.last_rmse;
        r.converged = s.converged;
        r.num_iterations = s.num_iterations;
    }
    return PCR_OK;
}

}  // namespace pcr
