// Feature-point matches between consecutive frames of one batch: for every record row i (level n = frame * L + l, y, x)
// the row j of level n + L within the search window |y_j - y_i| <= R, |x_j - x_i| <= R whose descriptor is nearest
// (float32 SSD, a fixed lane-strided order), accepted when it passes the ratio test and i is in turn j's nearest in the
// previous frame. Two launches, both programmatic dependent launches that read the emit's count on the device:
//  - match_search_kernel: one warp per (row, direction), lanes on descriptor elements. The window's first row comes
//    from a binary search on (level, y) over the used rows; the warp then reads 32 rows at a time, keeps those of the
//    target level with y in the window and x within R, and computes the SSD of each with all 32 lanes. It writes the raw
//    forward link to next, the raw backward link to prev and the forward d1 to distance;
//  - match_finalise_kernel: keeps only the mutual links, in place.
// Rows are sorted by (level, y, x) as every emit writes them; the order is not checked, but no read leaves [0, rows).
#include <algorithm>

#include "common.cuh"

namespace silent {

constexpr int kMatchThreads = 256;   // 8 warps per CTA

// SSD of the E-float rows a and b, identical in every lane: lane k sums (a_e - b_e)^2 over e = k, k + 32, ... in that
// order, then the lanes' sums are added by an xor butterfly over m = 16, 8, 4, 2, 1. Every product and sum is rounded
// on its own (the library builds with -fmad=false; the intrinsics say so here as well). The SSD of (a, b) and of (b, a)
// have the same bits: d and -d square alike.
__device__ __forceinline__ float warp_ssd(const float *__restrict__ a, const float *__restrict__ b, long long elems,
                                          int lane)
{
    float s = 0.0f;
    for (long long e = lane; e < elems; e += 32) {
        const float d = __fsub_rn(__ldg(a + e), __ldg(b + e));
        s = __fadd_rn(s, __fmul_rn(d, d));
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, m));
    return s;
}

// raw links of the first rows = clamp(*count, 0, capacity) rows in both directions; -1 / -1 / NaN at and past rows
__global__ void __launch_bounds__(kMatchThreads) match_search_kernel(const long long *__restrict__ points,
                                                                     const long long *__restrict__ count,
                                                                     long long capacity, const float *__restrict__ values,
                                                                     long long elems, int levels, int radius,
                                                                     float ratio, long long *__restrict__ next,
                                                                     long long *__restrict__ prev,
                                                                     float *__restrict__ distance)
{
    pdl_enter();
    const long long total = __ldg(count);
    const long long rows = total < 0 ? 0 : (total < capacity ? total : capacity);
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (kMatchThreads / 32);
    // task = 2 * row + direction (0: the next frame, 1: the previous one): both directions of a row in adjacent warps
    for (long long task = ((long long)blockIdx.x * kMatchThreads + threadIdx.x) / 32; task < 2 * capacity;
         task += warps) {
        const long long i = task >> 1;
        const bool forward = (task & 1) == 0;
        long long best = -1;
        float d1 = INFINITY;
        if (i < rows) {
            const long long n = __ldg(points + 4 * i), y = __ldg(points + 4 * i + 1), x = __ldg(points + 4 * i + 2);
            const long long target = forward ? n + levels : n - levels;
            const long long y_lo = y - radius, y_hi = y + radius;
            // first row with (level, y) >= (target, y - R), the same in every lane
            long long lo = 0, hi = rows;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                const long long ln = __ldg(points + 4 * mid), ly = __ldg(points + 4 * mid + 1);
                if (ln < target || (ln == target && ly < y_lo)) lo = mid + 1;
                else hi = mid;
            }
            const float *a = values + i * elems;
            float d2 = INFINITY;
            for (long long base = lo; base < rows; base += 32) {
                const long long j = base + lane;
                bool band = false, near = false;
                if (j < rows) {
                    const long long jn = __ldg(points + 4 * j), jy = __ldg(points + 4 * j + 1);
                    band = jn == target && jy <= y_hi;
                    if (band) {
                        const long long dx = __ldg(points + 4 * j + 2) - x;
                        near = dx >= -radius && dx <= radius;
                    }
                }
                unsigned cand = __ballot_sync(0xffffffffu, near);
                while (cand) {   // in row order: the first of equal SSDs stays the best
                    const int b = __ffs(cand) - 1;
                    cand &= cand - 1;
                    const long long k = base + b;
                    const float s = warp_ssd(a, values + k * elems, elems, lane);
                    if (s != s) continue;   // NaN: not a candidate
                    if (best < 0 || s < d1) {
                        d2 = d1;
                        d1 = s;
                        best = k;
                    } else if (s < d2) {
                        d2 = s;
                    }
                }
                if (__ballot_sync(0xffffffffu, band) != 0xffffffffu) break;   // the window ended in this run of rows
            }
            if (best >= 0 && !(d1 <= __fmul_rn(ratio, d2))) best = -1;
        }
        if (lane == 0) {
            if (forward) {
                next[i] = best;
                distance[i] = best >= 0 ? d1 : NAN;
            } else {
                prev[i] = best;
            }
        }
    }
}

// next[i] = j stays iff prev[j] == i, prev[j] = i stays iff next[i] == j; distance NaN where next ends at -1. In place:
// a thread writes only its own row and only ever lowers a link to -1, and only a link that is not mutual. A link of a
// mutual pair is never lowered, so whichever value a racing read sees (the raw link or the -1 written over it), a
// mutual pair reads back its partner and any other link reads something that is not the row itself: the same decision
__global__ void __launch_bounds__(kMatchThreads) match_finalise_kernel(const long long *__restrict__ count,
                                                                       long long capacity, long long *next,
                                                                       long long *prev, float *distance)
{
    pdl_enter();
    const long long total = *count;
    const long long rows = total < 0 ? 0 : (total < capacity ? total : capacity);
    const long long stride = (long long)gridDim.x * kMatchThreads;
    for (long long i = (long long)blockIdx.x * kMatchThreads + threadIdx.x; i < rows; i += stride) {
        const long long j = next[i], k = prev[i];
        const bool keep_next = j >= 0 && j < rows && prev[j] == i;
        const bool keep_prev = k >= 0 && k < rows && next[k] == i;
        if (!keep_next) {
            next[i] = -1;
            distance[i] = NAN;
        }
        if (!keep_prev) prev[i] = -1;
    }
}

}  // namespace silent

using namespace silent;

extern "C" {

int silent_match_points(const int64_t *points_dev, const int64_t *count_dev, int64_t capacity, const float *values_dev,
                        int64_t row_elems, int levels, int search_radius, float max_ratio, int64_t *next_dev,
                        int64_t *prev_dev, float *distance_dev, silent_stream stream)
{
    if (!count_dev) return fail(SILENT_E_INVAL, "silent_match_points: null count");
    if (capacity < 0) return fail(SILENT_E_INVAL, "silent_match_points: capacity must be >= 0");
    if (capacity > 0 && (!points_dev || !values_dev || !next_dev || !prev_dev || !distance_dev))
        return fail(SILENT_E_INVAL, "silent_match_points: null points, values or output with capacity %lld",
                    (long long)capacity);
    if (!(max_ratio > 0.0f && max_ratio <= 1.0f))   // NaN fails both
        return fail(SILENT_E_INVAL, "silent_match_points: max_ratio must be in (0, 1], got %g", (double)max_ratio);
    if (row_elems < 1) return fail(SILENT_E_SHAPE, "silent_match_points: row_elems must be >= 1, got %lld",
                                   (long long)row_elems);
    if (levels < 1) return fail(SILENT_E_SHAPE, "silent_match_points: levels must be >= 1, got %d", levels);
    if (search_radius < 0)
        return fail(SILENT_E_SHAPE, "silent_match_points: search_radius must be >= 0, got %d", search_radius);
    if (capacity == 0) return SILENT_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(SILENT_E_CUDA, "silent_match_points: no CUDA device; no CPU fallback exists");
    const cudaStream_t s = (cudaStream_t)stream;
    const int64_t waves = 148 * 8;   // at most a few waves of CTAs; the loops stride beyond that
    const dim3 search_grid((unsigned)std::min<int64_t>((2 * capacity + kMatchThreads / 32 - 1) / (kMatchThreads / 32),
                                                       waves));
    SILENT_CUDA(launch_dependent(match_search_kernel, search_grid, dim3(kMatchThreads), 0, s,
                                 (const long long *)points_dev, (const long long *)count_dev, (long long)capacity,
                                 values_dev, (long long)row_elems, levels, search_radius, max_ratio,
                                 (long long *)next_dev, (long long *)prev_dev, distance_dev));
    SILENT_LAUNCH_CHECK("match_search_kernel");
    const dim3 final_grid((unsigned)std::min<int64_t>((capacity + kMatchThreads - 1) / kMatchThreads, waves));
    SILENT_CUDA(launch_dependent(match_finalise_kernel, final_grid, dim3(kMatchThreads), 0, s,
                                 (const long long *)count_dev, (long long)capacity, (long long *)next_dev,
                                 (long long *)prev_dev, distance_dev));
    SILENT_LAUNCH_CHECK("match_finalise_kernel");
    return SILENT_OK;
}

}  // extern "C"
