// Frame-to-frame motion from feature-point matches: per pair of consecutive frames (f, f + 1), a 2-D affine map
// [y1, x1] = T[:, :2] @ [y0, x0] + T[:, 2] in frame pixels, found by a seeded RANSAC over the correspondences the matcher
// left (row i of frame f with next[i] >= 0), then refined by one least-squares step on the inliers of the best
// hypothesis. Three launches, all programmatic dependent launches that read the count and frame_offsets on the device:
//  - motion_compact_kernel: one CTA per pair. A block scan over frame f's rows writes the pair's correspondences, in row
//    order, to the workspace from base frame_offsets[f] (the rows of frame f bound their number M_f, so no global scan
//    is needed); writes matched[f], zeroes the pair's winner word and the inlier flags;
//  - motion_score_kernel: grid (pair, hypothesis chunk), one thread per hypothesis. Correspondence tiles are staged in
//    shared memory and read as broadcasts; each CTA sends one 64-bit atomicMax of (count << 32) | ~h per pair, so the
//    winner (most inliers, ties to the smaller h) does not depend on the order the CTAs finish in;
//  - motion_refine_kernel: one CTA per pair. Rebuilds the winner from h, forms the normal-equation sums over its
//    inliers in a fixed order, solves, rescores and writes T, the inlier count and the flags.
// Every decision is a function of the inputs alone: no atomics order, grid size or warp schedule changes a result.
#include <algorithm>

#include "common.cuh"

namespace silent {

constexpr int kMotionThreads = 256;   // compaction and refinement: 8 warps per pair
constexpr int kScoreThreads = 128;    // scoring: one hypothesis per thread, tiles of 128 correspondences

__device__ __forceinline__ long long clamp_rows(long long v, long long lo, long long hi)
{
    return v < lo ? lo : (v > hi ? hi : v);
}

// rows of frame f: [lo, hi) = clamp(frame_offsets[f], 0, rows), clamp(frame_offsets[f + 1], lo, rows)
__device__ __forceinline__ void frame_rows(const long long *offsets, int f, long long rows, long long &lo, long long &hi)
{
    lo = clamp_rows(__ldg(offsets + f), 0, rows);
    hi = clamp_rows(__ldg(offsets + f + 1), lo, rows);
}

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long z)
{
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// correspondence index of draw d (0, 1, 2) of hypothesis h of pair f: mulhi64(u, M),
// u = splitmix64(seed ^ splitmix64((f << 32) | (h << 2) | d))
__device__ __forceinline__ long long motion_draw(unsigned long long seed, int f, int h, int d, long long m)
{
    const unsigned long long key = ((unsigned long long)(unsigned)f << 32) | ((unsigned long long)h << 2) | d;
    return (long long)__umul64hi(splitmix64(seed ^ splitmix64(key)), (unsigned long long)m);
}

// hypothesis h of pair f over its m correspondences c[k] = (y0, x0, y1, x1): false when degenerate (a repeated draw, or
// !(|D| >= 1) with D twice the signed area of the three source points). Otherwise t = (a, b, c, d, e, g) with
// y1 = a y0 + b x0 + c, x1 = d y0 + e x0 + g through the three points, in float64 and this order of operations (the
// library builds with -fmad=false, so nothing below is fused); k0 is the first draw
__device__ __forceinline__ bool motion_hypothesis(const float4 *__restrict__ c, long long m, unsigned long long seed,
                                                  int f, int h, double t[6], long long &k0)
{
    k0 = motion_draw(seed, f, h, 0, m);
    const long long k1 = motion_draw(seed, f, h, 1, m), k2 = motion_draw(seed, f, h, 2, m);
    if (k0 == k1 || k0 == k2 || k1 == k2) return false;
    const float4 p0 = c[k0], p1 = c[k1], p2 = c[k2];
    const double y0 = p0.x, x0 = p0.y;
    const double dy1 = (double)p1.x - y0, dx1 = (double)p1.y - x0;
    const double dy2 = (double)p2.x - y0, dx2 = (double)p2.y - x0;
    const double det = dy1 * dx2 - dx1 * dy2;
    if (!(fabs(det) >= 1.0)) return false;
    const double u0[2] = {p0.z, p0.w}, u1[2] = {p1.z, p1.w}, u2[2] = {p2.z, p2.w};
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const double du1 = u1[r] - u0[r], du2 = u2[r] - u0[r];
        const double a = (du1 * dx2 - dx1 * du2) / det;
        const double b = (dy1 * du2 - du1 * dy2) / det;
        t[3 * r] = a;
        t[3 * r + 1] = b;
        t[3 * r + 2] = u0[r] - (a * y0 + b * x0);
    }
    return true;
}

// float32 residual test of one correspondence against a model rounded to float32 once: every operation rounded
__device__ __forceinline__ bool motion_inlier(const float m[6], float4 c, float thr2)
{
    const float ey = __fsub_rn(c.z, __fadd_rn(__fadd_rn(__fmul_rn(m[0], c.x), __fmul_rn(m[1], c.y)), m[2]));
    const float ex = __fsub_rn(c.w, __fadd_rn(__fadd_rn(__fmul_rn(m[3], c.x), __fmul_rn(m[4], c.y)), m[5]));
    return __fadd_rn(__fmul_rn(ey, ey), __fmul_rn(ex, ex)) <= thr2;
}

__device__ __forceinline__ void round_model(const double t[6], float m[6])
{
#pragma unroll
    for (int i = 0; i < 6; ++i) m[i] = __double2float_rn(t[i]);
}

__device__ __forceinline__ long long used_rows(const long long *count, long long capacity)
{
    const long long total = __ldg(count);
    return total < 0 ? 0 : (total < capacity ? total : capacity);
}

// correspondences of pair f = blockIdx.x, in row order, to corr / corr_row from the frame's first row; matched[f];
// winner[f] = 0; inlier = 0 over the whole capacity (grid-strided across the pairs)
__global__ void __launch_bounds__(kMotionThreads) motion_compact_kernel(const long long *__restrict__ offsets,
                                                                        const float2 *__restrict__ frame_yx,
                                                                        const long long *__restrict__ next,
                                                                        const long long *__restrict__ count,
                                                                        long long capacity, float4 *__restrict__ corr,
                                                                        long long *__restrict__ corr_row,
                                                                        long long *__restrict__ matched,
                                                                        unsigned long long *__restrict__ winner,
                                                                        unsigned char *__restrict__ inlier)
{
    pdl_enter();
    __shared__ int warp_n[kMotionThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (long long i = (long long)blockIdx.x * kMotionThreads + tid; i < capacity;
         i += (long long)gridDim.x * kMotionThreads)
        inlier[i] = 0;
    const long long rows = used_rows(count, capacity);
    const int f = blockIdx.x;
    long long lo, hi;
    frame_rows(offsets, f, rows, lo, hi);
    long long m = 0;
    for (long long base = lo; base < hi; base += kMotionThreads) {
        const long long i = base + tid;
        bool ok = false;
        float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < hi) {
            const long long j = __ldg(next + i);
            if (j >= 0 && j < rows) {
                const float2 a = frame_yx[i], b = frame_yx[j];
                c = make_float4(a.x, a.y, b.x, b.y);
                ok = isfinite(a.x) && isfinite(a.y) && isfinite(b.x) && isfinite(b.y);
            }
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) warp_n[warp] = __popc(ballot);
        __syncthreads();
        int before = 0, all = 0;
#pragma unroll
        for (int w = 0; w < kMotionThreads / 32; ++w) {
            before += w < warp ? warp_n[w] : 0;
            all += warp_n[w];
        }
        if (ok) {
            const long long k = lo + m + before + __popc(ballot & ((1u << lane) - 1u));
            corr[k] = c;
            corr_row[k] = i;
        }
        m += all;
        __syncthreads();   // warp_n is rewritten by the next run of rows
    }
    if (tid == 0) {
        matched[f] = m;
        winner[f] = 0;
    }
}

// winner[f] = max over the live hypotheses h of pair f = blockIdx.x of (inliers << 32) | ~h (0: none is live)
__global__ void __launch_bounds__(kScoreThreads) motion_score_kernel(const long long *__restrict__ offsets,
                                                                     const long long *__restrict__ count,
                                                                     long long capacity,
                                                                     const float4 *__restrict__ corr,
                                                                     const long long *__restrict__ matched,
                                                                     int hypotheses, float thr2,
                                                                     unsigned long long seed,
                                                                     unsigned long long *__restrict__ winner)
{
    pdl_enter();
    __shared__ float4 tile[kScoreThreads];
    __shared__ unsigned long long warp_best[kScoreThreads / 32];
    const int f = blockIdx.x, tid = threadIdx.x;
    const long long m = matched[f];
    if (m < 3) return;   // the same in the whole CTA
    long long lo, hi;
    frame_rows(offsets, f, used_rows(count, capacity), lo, hi);
    const float4 *c = corr + lo;
    const int h = blockIdx.y * kScoreThreads + tid;
    double t[6];
    long long k0;
    const bool live = h < hypotheses && motion_hypothesis(c, m, seed, f, h, t, k0);
    float model[6];
    round_model(t, model);   // unused when not live
    unsigned n = 0;
    for (long long base = 0; base < m; base += kScoreThreads) {
        if (base + tid < m) tile[tid] = c[base + tid];
        __syncthreads();
        const int len = m - base < kScoreThreads ? (int)(m - base) : kScoreThreads;
        if (live) {
#pragma unroll 8
            for (int k = 0; k < len; ++k) n += motion_inlier(model, tile[k], thr2);
        }
        __syncthreads();
    }
    unsigned long long word = live ? ((unsigned long long)n << 32) | (unsigned)~h : 0ull;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) word = max(word, __shfl_xor_sync(0xffffffffu, word, s));
    if ((tid & 31) == 0) warp_best[tid >> 5] = word;
    __syncthreads();
    if (tid == 0) {
#pragma unroll
        for (int w = 1; w < kScoreThreads / 32; ++w) word = max(word, warp_best[w]);
        if (word) atomicMax(winner + f, word);
    }
}

// block sum of one int per thread (exact: any order)
__device__ __forceinline__ long long block_count(unsigned n, int *scratch)
{
    n = __reduce_add_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = (int)n;
    __syncthreads();
    long long s = 0;
#pragma unroll
    for (int w = 0; w < kMotionThreads / 32; ++w) s += scratch[w];
    __syncthreads();
    return s;
}

constexpr int kSums = 11;   // Y, X, YY, YX, XX, U, YU, XU, V, YV, XV

// T, inlier_count and flags of pair f = blockIdx.x from its winner word (which shares inlier_count's storage)
__global__ void __launch_bounds__(kMotionThreads) motion_refine_kernel(const long long *__restrict__ offsets,
                                                                       const long long *__restrict__ count,
                                                                       long long capacity,
                                                                       const float4 *__restrict__ corr,
                                                                       const long long *__restrict__ corr_row,
                                                                       const long long *__restrict__ matched,
                                                                       float thr2, unsigned long long seed,
                                                                       double *__restrict__ transform,
                                                                       unsigned long long *winner,
                                                                       unsigned char *__restrict__ inlier)
{
    pdl_enter();
    __shared__ double warp_sum[kMotionThreads / 32][kSums];
    __shared__ double refit[6];
    __shared__ int scratch[kMotionThreads / 32];
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long word = winner[f];
    __syncthreads();   // every thread has read the word before thread 0 overwrites it with the count
    double *out = transform + 6 * (long long)f;
    long long *out_count = reinterpret_cast<long long *>(winner) + f;
    if (word == 0) {
        if (tid < 6) out[tid] = NAN;
        if (tid == 0) *out_count = 0;
        return;
    }
    const long long m = matched[f];
    long long lo, hi;
    frame_rows(offsets, f, used_rows(count, capacity), lo, hi);
    const float4 *c = corr + lo;
    double t[6];
    long long k0;
    motion_hypothesis(c, m, seed, f, (int)~(unsigned)word, t, k0);   // live: it won
    float model[6];
    round_model(t, model);
    // sums over the inliers, coordinates relative to the first draw (py, px) -> (qy, qx)
    const float4 p = c[k0];
    const double py = p.x, px = p.y, qy = p.z, qx = p.w;
    double s[kSums];
#pragma unroll
    for (int q = 0; q < kSums; ++q) s[q] = 0.0;
    unsigned n = 0;
    for (long long k = tid; k < m; k += kMotionThreads) {
        const float4 v = c[k];
        if (!motion_inlier(model, v, thr2)) continue;
        ++n;
        const double Y = (double)v.x - py, X = (double)v.y - px, U = (double)v.z - qy, V = (double)v.w - qx;
        s[0] += Y;
        s[1] += X;
        s[2] += Y * Y;
        s[3] += Y * X;
        s[4] += X * X;
        s[5] += U;
        s[6] += Y * U;
        s[7] += X * U;
        s[8] += V;
        s[9] += Y * V;
        s[10] += X * V;
    }
#pragma unroll
    for (int q = 0; q < kSums; ++q) {
#pragma unroll
        for (int b = 16; b >= 1; b >>= 1) s[q] += __shfl_xor_sync(0xffffffffu, s[q], b);
        if (lane == 0) warp_sum[warp][q] = s[q];
    }
    const long long inliers = block_count(n, scratch);   // also orders warp_sum's writes before the reads below
    if (tid == 0) {
        double S[kSums];
#pragma unroll
        for (int q = 0; q < kSums; ++q) {
            S[q] = warp_sum[0][q];
#pragma unroll
            for (int w = 1; w < kMotionThreads / 32; ++w) S[q] = S[q] + warp_sum[w][q];
        }
        const double nn = (double)inliers;
        const double Sy = S[0], Sx = S[1], Syy = S[2], Syx = S[3], Sxx = S[4];
        const double c00 = Sxx * nn - Sx * Sx, c01 = Sx * Sy - Syx * nn, c02 = Syx * Sx - Sxx * Sy;
        const double c11 = Syy * nn - Sy * Sy, c12 = Syx * Sy - Syy * Sx, c22 = Syy * Sxx - Syx * Syx;
        const double det = (Syy * c00 + Syx * c01) + Sy * c02;
        const double r[2][3] = {{S[6], S[7], S[5]}, {S[9], S[10], S[8]}}, q0[2] = {qy, qx};
#pragma unroll
        for (int o = 0; o < 2; ++o) {
            const double a = ((c00 * r[o][0] + c01 * r[o][1]) + c02 * r[o][2]) / det;
            const double b = ((c01 * r[o][0] + c11 * r[o][1]) + c12 * r[o][2]) / det;
            const double cc = ((c02 * r[o][0] + c12 * r[o][1]) + c22 * r[o][2]) / det;
            refit[3 * o] = a;
            refit[3 * o + 1] = b;
            refit[3 * o + 2] = (q0[o] + cc) - (a * py + b * px);
        }
    }
    __syncthreads();
    double t2[6];
    bool finite = true;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        t2[i] = refit[i];
        finite = finite && isfinite(t2[i]);
    }
    float model2[6];
    round_model(t2, model2);
    unsigned n2 = 0;
    if (finite)
        for (long long k = tid; k < m; k += kMotionThreads) n2 += motion_inlier(model2, c[k], thr2);
    const long long inliers2 = block_count(n2, scratch);
    const bool keep = finite && inliers2 >= inliers;   // the same in every thread
    float fm[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) fm[i] = keep ? model2[i] : model[i];
    for (long long k = tid; k < m; k += kMotionThreads) inlier[corr_row[lo + k]] = motion_inlier(fm, c[k], thr2);
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 6; ++i) out[i] = keep ? t2[i] : t[i];
        *out_count = keep ? inliers2 : inliers;
    }
}

}  // namespace silent

using namespace silent;

extern "C" {

size_t silent_motion_workspace_bytes(int64_t capacity)
{
    return capacity > 0 ? (size_t)capacity * (sizeof(float4) + sizeof(long long)) : 0;
}

int silent_estimate_motion(const int64_t *frame_offsets_dev, const float *frame_yx_dev, const int64_t *next_dev,
                           const int64_t *count_dev, int64_t capacity, int batch, int hypotheses, float threshold,
                           uint64_t seed, void *workspace_dev, size_t workspace_bytes, double *transform_dev,
                           int64_t *inlier_count_dev, int64_t *matched_dev, uint8_t *inlier_dev, silent_stream stream)
{
    if (capacity < 0) return fail(SILENT_E_INVAL, "silent_estimate_motion: capacity must be >= 0");
    if (batch < 1) return fail(SILENT_E_INVAL, "silent_estimate_motion: batch must be >= 1, got %d", batch);
    if (capacity > 0 && (!frame_offsets_dev || !frame_yx_dev || !next_dev || !count_dev || !workspace_dev ||
                         !inlier_dev || (batch > 1 && (!transform_dev || !inlier_count_dev || !matched_dev))))
        return fail(SILENT_E_INVAL, "silent_estimate_motion: null input, workspace or output with capacity %lld",
                    (long long)capacity);
    if (!(threshold > 0.0f) || !isfinite(threshold))   // NaN fails the first
        return fail(SILENT_E_INVAL, "silent_estimate_motion: threshold must be finite and > 0, got %g",
                    (double)threshold);
    if (hypotheses < 1 || hypotheses > SILENT_MOTION_HYPOTHESES_MAX)
        return fail(SILENT_E_SHAPE, "silent_estimate_motion: hypotheses must be in [1, %d], got %d",
                    SILENT_MOTION_HYPOTHESES_MAX, hypotheses);
    const size_t need = silent_motion_workspace_bytes(capacity);
    if (workspace_bytes < need)
        return fail(SILENT_E_CAPACITY, "silent_estimate_motion: workspace of %zu bytes, need %zu", workspace_bytes,
                    need);
    if (capacity > 0 && ((uintptr_t)workspace_dev & 15))
        return fail(SILENT_E_INVAL, "silent_estimate_motion: workspace must be 16-byte aligned");
    if (capacity == 0 || batch == 1) return SILENT_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(SILENT_E_CUDA, "silent_estimate_motion: no CUDA device; no CPU fallback exists");
    const cudaStream_t s = (cudaStream_t)stream;
    const unsigned pairs = (unsigned)(batch - 1);
    float4 *corr = (float4 *)workspace_dev;
    long long *corr_row = (long long *)((char *)workspace_dev + (size_t)capacity * sizeof(float4));
    unsigned long long *winner = (unsigned long long *)inlier_count_dev;
    const float thr2 = threshold * threshold;   // float32, rounded once
    SILENT_CUDA(launch_dependent(motion_compact_kernel, dim3(pairs), dim3(kMotionThreads), 0, s,
                                 (const long long *)frame_offsets_dev, (const float2 *)frame_yx_dev,
                                 (const long long *)next_dev, (const long long *)count_dev, (long long)capacity, corr,
                                 corr_row, (long long *)matched_dev, winner, (unsigned char *)inlier_dev));
    SILENT_LAUNCH_CHECK("motion_compact_kernel");
    const dim3 score_grid(pairs, (unsigned)((hypotheses + kScoreThreads - 1) / kScoreThreads));
    SILENT_CUDA(launch_dependent(motion_score_kernel, score_grid, dim3(kScoreThreads), 0, s,
                                 (const long long *)frame_offsets_dev, (const long long *)count_dev,
                                 (long long)capacity, (const float4 *)corr, (const long long *)matched_dev, hypotheses,
                                 thr2, (unsigned long long)seed, winner));
    SILENT_LAUNCH_CHECK("motion_score_kernel");
    SILENT_CUDA(launch_dependent(motion_refine_kernel, dim3(pairs), dim3(kMotionThreads), 0, s,
                                 (const long long *)frame_offsets_dev, (const long long *)count_dev,
                                 (long long)capacity, (const float4 *)corr, (const long long *)corr_row,
                                 (const long long *)matched_dev, thr2, (unsigned long long)seed, transform_dev, winner,
                                 (unsigned char *)inlier_dev));
    SILENT_LAUNCH_CHECK("motion_refine_kernel");
    return SILENT_OK;
}

}  // extern "C"
