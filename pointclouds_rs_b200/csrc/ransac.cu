// ransac.cu -- ransac_plane_seeded (crates/segmentation/src/ransac_plane.rs:56-129) for GIVEN samples.
//
// The reference draws all index triples up front (StdRng, :75-78), fits a plane through each (:166-190)
// and counts its inliers over the whole cloud (:132-137): m x n point-plane distances, the only heavy
// part.  The sampling stays with the caller (ChaCha12 cannot be reproduced here; the Rust wrapper keeps
// its `sample_three_distinct`), everything after it runs on the device and is bit-exact:
//
//   ransac_fit_kernel     one thread per sample: the plane through its three points, or "collinear"
//   ransac_count_kernel   every block holds 1024 points in registers (4 per thread) and streams the
//                         models through shared memory; per-model counts: warp redux -> shared atomics
//                         -> one global atomic per model and block                  12 B/pt + 16 B/model
//   (host)                the reference's choice rule on the m counts: sequential with its adaptive
//                         early exit (:95-121), or first-maximum for the parallel path (:82-93)
//   ransac_inlier_kernel  inlier flags of the winner -> exclusive scan -> ascending index list (:123-126)
// f32 arithmetic is the reference's, operation by operation (no FMA: the library is built -fmad=false).
// A batch (frames back to back) fits all frames' triples in one launch, counts with blocks that never cross a frame
// against that frame's models only, and writes every frame's inliers with one scan (ransac_plane_samples_batch_dev).
#include "pcr_internal.cuh"

#include <algorithm>
#include <cmath>

namespace pcr {

namespace {

constexpr int kRansacThreads = 256;
constexpr int kRansacItems = 4;
constexpr int kModelChunk = 512;

// ransac_plane.rs:17-20
__device__ __forceinline__ float plane_dist(float4 m, float x, float y, float z) {
    return fabsf(__fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m.x, x), __fmul_rn(m.y, y)), __fmul_rn(m.z, z)), m.w));
}

__global__ void __launch_bounds__(256) ransac_fit_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                         const float *__restrict__ z, const uint32_t *__restrict__ samples, size_t m,
                                                         float4 *__restrict__ models, uint32_t *__restrict__ counts) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const uint32_t i0 = samples[3 * t], i1 = samples[3 * t + 1], i2 = samples[3 * t + 2];
    const float p0x = x[i0], p0y = y[i0], p0z = z[i0];
    const float v1x = __fsub_rn(x[i1], p0x), v1y = __fsub_rn(y[i1], p0y), v1z = __fsub_rn(z[i1], p0z);
    const float v2x = __fsub_rn(x[i2], p0x), v2y = __fsub_rn(y[i2], p0y), v2z = __fsub_rn(z[i2], p0z);
    const float nx = __fsub_rn(__fmul_rn(v1y, v2z), __fmul_rn(v1z, v2y));  // :171-174
    const float ny = __fsub_rn(__fmul_rn(v1z, v2x), __fmul_rn(v1x, v2z));
    const float nz = __fsub_rn(__fmul_rn(v1x, v2y), __fmul_rn(v1y, v2x));
    const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz)));
    float4 mdl;
    if (len < 1e-10f) {  // :178-181 collinear (a NaN length is NOT caught, as in the reference)
        mdl = make_float4(__int_as_float(0x7fc00000), 0.f, 0.f, 0.f);
        counts[t] = 0xffffffffu;  // "no model"
    } else {
        mdl.x = __fdiv_rn(nx, len);
        mdl.y = __fdiv_rn(ny, len);
        mdl.z = __fdiv_rn(nz, len);
        mdl.w = -__fadd_rn(__fadd_rn(__fmul_rn(mdl.x, p0x), __fmul_rn(mdl.y, p0y)), __fmul_rn(mdl.z, p0z));  // :186
        counts[t] = 0;
    }
    models[t] = mdl;
}

// one block's share of the counts: points base + j * kRansacThreads (j < kRansacItems) below n, against the m models
__device__ __forceinline__ void ransac_count_block(const float *__restrict__ x, const float *__restrict__ y, const float *__restrict__ z,
                                                   size_t base, size_t n, float threshold, const float4 *__restrict__ models, size_t m,
                                                   uint32_t *__restrict__ counts) {
    __shared__ float4 smodel[kModelChunk];
    __shared__ uint32_t scount[kModelChunk];
    float px[kRansacItems], py[kRansacItems], pz[kRansacItems];
#pragma unroll
    for (int j = 0; j < kRansacItems; j++) {
        const size_t i = base + (size_t)j * kRansacThreads;
        const bool in = i < n;
        // a point past the end never counts: NaN fails every `<=`
        px[j] = in ? x[i] : __int_as_float(0x7fc00000);
        py[j] = in ? y[i] : 0.f;
        pz[j] = in ? z[i] : 0.f;
    }
    for (size_t c0 = 0; c0 < m; c0 += kModelChunk) {
        const int cm = (int)min((size_t)kModelChunk, m - c0);
        for (int t = threadIdx.x; t < cm; t += kRansacThreads) {
            smodel[t] = models[c0 + t];
            scount[t] = 0;
        }
        __syncthreads();
        for (int t = 0; t < cm; t++) {
            const float4 mdl = smodel[t];  // broadcast
            unsigned c = 0;
#pragma unroll
            for (int j = 0; j < kRansacItems; j++) c += plane_dist(mdl, px[j], py[j], pz[j]) <= threshold ? 1u : 0u;  // :135
            c = __reduce_add_sync(PCR_FULL, c);
            if ((threadIdx.x & 31) == 0 && c) atomicAdd(&scount[t], c);
        }
        __syncthreads();
        for (int t = threadIdx.x; t < cm; t += kRansacThreads)
            if (scount[t] && counts[c0 + t] != 0xffffffffu) atomicAdd(&counts[c0 + t], scount[t]);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kRansacThreads) ransac_count_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                      const float *__restrict__ z, size_t n, float threshold,
                                                                      const float4 *__restrict__ models, size_t m,
                                                                      uint32_t *__restrict__ counts) {
    ransac_count_block(x, y, z, (size_t)blockIdx.x * (kRansacThreads * kRansacItems) + threadIdx.x, n, threshold, models, m, counts);
}

// Batch: every block holds kRansacThreads * kRansacItems points of ONE frame (blocks[b] = {frame, first point}) and
// streams only that frame's models, [model_off[f], model_off[f+1]).
__global__ void __launch_bounds__(kRansacThreads) ransac_count_batch_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                            const float *__restrict__ z, const uint2 *__restrict__ blocks,
                                                                            const uint32_t *__restrict__ frame_off,
                                                                            const uint32_t *__restrict__ model_off, float threshold,
                                                                            const float4 *__restrict__ models, uint32_t *__restrict__ counts) {
    const uint2 b = blocks[blockIdx.x];
    const uint32_t m0 = model_off[b.x];
    ransac_count_block(x, y, z, (size_t)b.y + threadIdx.x, frame_off[b.x + 1], threshold, models + m0, model_off[b.x + 1] - m0, counts + m0);
}

__global__ void __launch_bounds__(256) ransac_inlier_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                            const float *__restrict__ z, size_t n, float4 model, float threshold,
                                                            uint32_t *__restrict__ flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    flag[i] = (i < n && plane_dist(model, x[i], y[i], z[i]) <= threshold) ? 1u : 0u;  // :123-126
}

__global__ void __launch_bounds__(256) ransac_emit_kernel(const uint32_t *__restrict__ pos, size_t n, uint32_t *__restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (pos[i + 1] != pos[i]) out[pos[i]] = (uint32_t)i;
}

// Batch: the inlier flags of every point against its frame's winner (a frame of fewer than 3 points has none, :64-66) ...
__global__ void __launch_bounds__(256) ransac_inlier_batch_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                  const float *__restrict__ z, size_t n, const uint32_t *__restrict__ frame_off,
                                                                  int n_frames, const float4 *__restrict__ best, float threshold,
                                                                  uint32_t *__restrict__ flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    uint32_t v = 0;
    if (i < n) {
        const int f = frame_of(frame_off, n_frames, (uint32_t)i);
        v = (frame_off[f + 1] - frame_off[f] >= 3 && plane_dist(best[f], x[i], y[i], z[i]) <= threshold) ? 1u : 0u;
    }
    flag[i] = v;
}

// ... the frame-local index of every inlier at its scanned position ...
__global__ void __launch_bounds__(256) ransac_emit_batch_kernel(const uint32_t *__restrict__ pos, size_t n, const uint32_t *__restrict__ frame_off,
                                                                int n_frames, uint32_t *__restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || pos[i + 1] == pos[i]) return;
    out[pos[i]] = (uint32_t)i - frame_off[frame_of(frame_off, n_frames, (uint32_t)i)];
}

// ... and the first inlier of every frame (entry n_frames: the total)
__global__ void ransac_frame_starts_kernel(const uint32_t *__restrict__ pos, const uint32_t *__restrict__ frame_off, int n_frames,
                                           uint32_t *__restrict__ out) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f <= n_frames) out[f] = pos[frame_off[f]];
}

// the reference's choice rule (:80-121), replayed on the counts of one cloud's m hypotheses (0xffffffff: collinear sample)
float4 ransac_choose(const uint32_t *counts, const float4 *models, size_t m, size_t n) {
    float4 best = make_float4(0.f, 0.f, 1.f, 0.f);
    const bool parallel = n >= 10000 && m >= 16;  // :80
    size_t best_count = 0;
    bool have = false;
    for (size_t it = 0; it < m; it++) {
        if (counts[it] == 0xffffffffu) continue;  // collinear sample (:86 / :98-101)
        const size_t cnt = counts[it];
        if (parallel) {  // :84-93: first hypothesis with the largest count
            if (!have || cnt > best_count) {
                have = true;
                best_count = cnt;
                best = models[it];
            }
        } else if (cnt > best_count) {  // :106
            best_count = cnt;
            best = models[it];
            const double w = (double)best_count / (double)n;  // :110-117
            if (w > 0.5) {
                const double needed = std::log(1.0 - 0.999) / std::log(1.0 - w * w * w);
                if ((double)it > needed) break;
            }
        }
    }
    return best;
}

}  // namespace

// model_out = {nx, ny, nz, d}; d_inliers (device, n entries) receives the ascending inlier indices.
int ransac_plane_samples_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, size_t n, float threshold,
                             const uint32_t *h_samples, size_t m, float model_out[4], uint32_t *d_inliers, size_t *n_inliers) {
    model_out[0] = 0.f; model_out[1] = 0.f; model_out[2] = 1.f; model_out[3] = 0.f;  // PlaneModel::default(), :23-30
    *n_inliers = 0;
    if (n < 3) return PCR_OK;  // :64-66
    if (n > 0x7fffffffull) return fail(ctx, PCR_ERR_UNSUPPORTED, "clouds above 2^31 points are not supported");
    for (size_t t = 0; t < 3 * m; t++)
        if (h_samples[t] >= n) return fail(ctx, PCR_ERR_INVALID_ARG, "sample index %u out of bounds for cloud with %zu points", h_samples[t], n);
    cudaStream_t st = ctx->stream;
    TimeScope ts(ctx, kTagOther);
    // scratch (b_table): samples u32[3m] | models float4[m] | counts u32[m] | pos u32[n + 1]
    const size_t off_models = (sizeof(uint32_t) * 3 * m + 255) & ~(size_t)255;
    const size_t off_counts = off_models + sizeof(float4) * std::max<size_t>(m, 1);
    const size_t off_pos = (off_counts + sizeof(uint32_t) * std::max<size_t>(m, 1) + 255) & ~(size_t)255;
    PCR_TRY(ensure(ctx, ctx->b_table, off_pos + sizeof(uint32_t) * (n + 1)));
    char *base = (char *)ctx->b_table.p;
    uint32_t *d_samples = (uint32_t *)base;
    float4 *d_models = (float4 *)(base + off_models);
    uint32_t *d_counts = (uint32_t *)(base + off_counts);
    uint32_t *d_pos = (uint32_t *)(base + off_pos);
    float4 best = make_float4(0.f, 0.f, 1.f, 0.f);
    if (m > 0) {
        PCR_CUDA(ctx, cudaMemcpyAsync(d_samples, h_samples, sizeof(uint32_t) * 3 * m, cudaMemcpyHostToDevice, st));
        ransac_fit_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(dx, dy, dz, d_samples, m, d_models, d_counts);
        PCR_LAUNCH_CHECK(ctx);
        const size_t per_block = (size_t)kRansacThreads * kRansacItems;
        ransac_count_kernel<<<(unsigned)((n + per_block - 1) / per_block), kRansacThreads, 0, st>>>(dx, dy, dz, n, threshold, d_models, m,
                                                                                                    d_counts);
        PCR_LAUNCH_CHECK(ctx);
        std::vector<uint32_t> counts(m);
        std::vector<float4> models(m);
        PCR_CUDA(ctx, cudaMemcpyAsync(counts.data(), d_counts, sizeof(uint32_t) * m, cudaMemcpyDeviceToHost, st));
        PCR_CUDA(ctx, cudaMemcpyAsync(models.data(), d_models, sizeof(float4) * m, cudaMemcpyDeviceToHost, st));
        PCR_CUDA(ctx, cudaStreamSynchronize(st));
        best = ransac_choose(counts.data(), models.data(), m, n);
    }
    model_out[0] = best.x; model_out[1] = best.y; model_out[2] = best.z; model_out[3] = best.w;
    ransac_inlier_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(dx, dy, dz, n, best, threshold, d_pos);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(exclusive_scan_u32_dev(ctx, d_pos, n + 1));
    ransac_emit_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_pos, n, d_inliers);
    PCR_LAUNCH_CHECK(ctx);
    uint32_t *mail = (uint32_t *)ctx->pinned + 112;
    PCR_CUDA(ctx, cudaMemcpyAsync(mail, d_pos + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    *n_inliers = *mail;
    return PCR_OK;
}

// Every frame of a batch in one set of launches; frame f gets what ransac_plane_samples_dev returns for it alone with its
// own triples (its own n and m in the choice rule).  The triples are turned into global indices while they are staged,
// so the fit is the single call's kernel over all M triples.  Two host round trips: all counts and models, then the
// per-frame inlier offsets.
int ransac_plane_samples_batch_dev(Ctx *ctx, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets,
                                   size_t n_frames, float threshold, const uint32_t *h_samples, const uint64_t *sample_offsets,
                                   float *models_out, uint32_t *d_inliers, uint64_t *inlier_offsets) {
    const int F = (int)n_frames;
    for (int f = 0; f < F; f++) {
        float *mo = models_out + 4 * f;
        mo[0] = 0.f; mo[1] = 0.f; mo[2] = 1.f; mo[3] = 0.f;  // PlaneModel::default(), :23-30
    }
    for (int f = 0; f <= F; f++) inlier_offsets[f] = 0;
    const size_t n = F ? (size_t)frame_offsets[F] : 0;
    if (n == 0) return PCR_OK;
    // host staging, ONE copy: triples u32[3M] (global indices) | frame offsets u32[F + 1] | model offsets u32[F + 1] |
    // count blocks uint2[B].  A frame below 3 points keeps none of its triples (the single call returns before it
    // reads them, :64-66).
    const size_t per_block = (size_t)kRansacThreads * kRansacItems;
    std::vector<uint32_t> moff(F + 1, 0);
    size_t n_blocks = 0;
    for (int f = 0; f < F; f++) {
        const uint64_t b = frame_offsets[f], nf = frame_offsets[f + 1] - b;
        const uint64_t mf = sample_offsets ? sample_offsets[f + 1] - sample_offsets[f] : 0;
        moff[f + 1] = moff[f];
        if (nf < 3 || mf == 0) continue;
        const uint32_t *t = h_samples + 3 * sample_offsets[f];
        for (uint64_t j = 0; j < 3 * mf; j++)
            if (t[j] >= nf)
                return fail(ctx, PCR_ERR_INVALID_ARG, "frame %d: sample index %u out of bounds for a frame with %llu points", f, t[j],
                            (unsigned long long)nf);
        moff[f + 1] += (uint32_t)mf;
        n_blocks += (nf + per_block - 1) / per_block;
    }
    const size_t M = moff[F];
    const size_t o_foff = (3 * M + 3) & ~(size_t)3, o_moff = (o_foff + F + 1 + 3) & ~(size_t)3, o_blk = (o_moff + F + 1 + 3) & ~(size_t)3;
    std::vector<uint32_t> stage(o_blk + 2 * n_blocks);
    for (int f = 0; f < F; f++) {
        const uint32_t b = (uint32_t)frame_offsets[f], nf = (uint32_t)(frame_offsets[f + 1] - b);
        stage[o_foff + f] = b;
        stage[o_moff + f] = moff[f];
        const uint32_t mf = moff[f + 1] - moff[f];
        if (!mf) continue;
        const uint32_t *t = h_samples + 3 * sample_offsets[f];
        for (uint32_t j = 0; j < 3 * mf; j++) stage[3 * (size_t)moff[f] + j] = t[j] + b;
    }
    stage[o_foff + F] = (uint32_t)n;
    stage[o_moff + F] = (uint32_t)M;
    for (int f = 0, blk = 0; f < F; f++) {
        if (moff[f + 1] == moff[f]) continue;
        for (uint64_t p = frame_offsets[f]; p < frame_offsets[f + 1]; p += per_block, blk++) {
            stage[o_blk + 2 * (size_t)blk] = (uint32_t)f;
            stage[o_blk + 2 * (size_t)blk + 1] = (uint32_t)p;
        }
    }
    cudaStream_t st = ctx->stream;
    TimeScope ts(ctx, kTagOther);
    // scratch (b_table): staging | models float4[M] | counts u32[M] | pos u32[n + 1] | winners float4[F] | inlier offsets u32[F + 1]
    const size_t off_models = (sizeof(uint32_t) * stage.size() + 255) & ~(size_t)255;
    const size_t off_counts = off_models + sizeof(float4) * std::max<size_t>(M, 1);
    const size_t off_pos = (off_counts + sizeof(uint32_t) * std::max<size_t>(M, 1) + 255) & ~(size_t)255;
    const size_t off_best = (off_pos + sizeof(uint32_t) * (n + 1) + 255) & ~(size_t)255;
    const size_t off_inl = off_best + sizeof(float4) * F;
    PCR_TRY(ensure(ctx, ctx->b_table, off_inl + sizeof(uint32_t) * (F + 1)));
    PCR_TRY(ensure_pinned(ctx, std::max<size_t>(4096, sizeof(uint32_t) * (F + 1))));
    char *base = (char *)ctx->b_table.p;
    const uint32_t *d_stage = (const uint32_t *)base;
    const uint32_t *d_foff = d_stage + o_foff, *d_moff = d_stage + o_moff;
    float4 *d_models = (float4 *)(base + off_models);
    uint32_t *d_counts = (uint32_t *)(base + off_counts);
    uint32_t *d_pos = (uint32_t *)(base + off_pos);
    float4 *d_best = (float4 *)(base + off_best);
    uint32_t *d_inl_off = (uint32_t *)(base + off_inl);
    // (pageable source: the copy has taken the bytes when it returns)
    PCR_CUDA(ctx, cudaMemcpyAsync(base, stage.data(), sizeof(uint32_t) * stage.size(), cudaMemcpyHostToDevice, st));
    std::vector<float4> best(F, make_float4(0.f, 0.f, 1.f, 0.f));
    if (M > 0) {
        ransac_fit_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(dx, dy, dz, d_stage, M, d_models, d_counts);
        PCR_LAUNCH_CHECK(ctx);
        ransac_count_batch_kernel<<<(unsigned)n_blocks, kRansacThreads, 0, st>>>(dx, dy, dz, (const uint2 *)(d_stage + o_blk), d_foff, d_moff,
                                                                                 threshold, d_models, d_counts);
        PCR_LAUNCH_CHECK(ctx);
        std::vector<uint32_t> counts(M);
        std::vector<float4> models(M);
        PCR_CUDA(ctx, cudaMemcpyAsync(counts.data(), d_counts, sizeof(uint32_t) * M, cudaMemcpyDeviceToHost, st));
        PCR_CUDA(ctx, cudaMemcpyAsync(models.data(), d_models, sizeof(float4) * M, cudaMemcpyDeviceToHost, st));
        PCR_MARK("ransac batch: wait for counts");
        PCR_CUDA(ctx, cudaStreamSynchronize(st));
        for (int f = 0; f < F; f++) {
            const size_t mf = moff[f + 1] - moff[f];
            if (mf) best[f] = ransac_choose(counts.data() + moff[f], models.data() + moff[f], mf, frame_offsets[f + 1] - frame_offsets[f]);
        }
    }
    for (int f = 0; f < F; f++) {
        float *mo = models_out + 4 * f;
        mo[0] = best[f].x; mo[1] = best[f].y; mo[2] = best[f].z; mo[3] = best[f].w;
    }
    PCR_CUDA(ctx, cudaMemcpyAsync(d_best, best.data(), sizeof(float4) * F, cudaMemcpyHostToDevice, st));
    ransac_inlier_batch_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(dx, dy, dz, n, d_foff, F, d_best, threshold, d_pos);
    PCR_LAUNCH_CHECK(ctx);
    PCR_TRY(exclusive_scan_u32_dev(ctx, d_pos, n + 1));
    ransac_emit_batch_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_pos, n, d_foff, F, d_inliers);
    PCR_LAUNCH_CHECK(ctx);
    ransac_frame_starts_kernel<<<(F + 1 + 255) / 256, 256, 0, st>>>(d_pos, d_foff, F, d_inl_off);
    PCR_LAUNCH_CHECK(ctx);
    uint32_t *mail = (uint32_t *)ctx->pinned;
    PCR_CUDA(ctx, cudaMemcpyAsync(mail, d_inl_off, sizeof(uint32_t) * (F + 1), cudaMemcpyDeviceToHost, st));
    PCR_MARK("ransac batch: wait for inlier offsets");
    PCR_CUDA(ctx, cudaStreamSynchronize(st));
    for (int f = 0; f <= F; f++) inlier_offsets[f] = mail[f];
    return PCR_OK;
}

}  // namespace pcr
