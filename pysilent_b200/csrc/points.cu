// Feature-point records: for each emitted row (level, y, x, 0) its position in the frame and the responses there
// (gray, orient[C], padded_line_end[C]), gathered on the device from the emit's own rows and count, so that a caller who
// wants points never has to fetch the whole output tensors. A record may carry the square patch of side P = 2r + 1
// around the point instead of its one pixel (r = 0). One launch: a grid-stride loop over the (row, patch pixel) pairs of
// the written rows, and a binary search per frame for frame_offsets (rows are sorted by level, levels by frame).
#include <algorithm>

#include <cuda_fp16.h>

#include "plan.h"

namespace silent {

__device__ __forceinline__ float widen(const float *p, size_t i) { return __ldg(p + i); }
__device__ __forceinline__ float widen(const __half *p, size_t i) { return __half2float(p[i]); }   // exact

// records of the first min(*count, capacity) rows of points [.][4]: coords [.][2] = (frame_y, frame_x) from the plan's
// per-level coordinate tables, values [.][P][P][1 + 2C] = (gray, orient[C], line_end[C]) at (level, y + dy, x + dx) for
// dy, dx in [-radius, radius], at [radius + dy][radius + dx]; +0.0 (what SAME zero padding reads) where that pixel
// leaves the level. One thread per (row, patch pixel), so radius 0 is one thread per row. A row outside the call's
// [images, h, w] (no emit writes one) gets NaN everywhere instead of a read out of bounds.
template <int C, typename T>
__global__ void __launch_bounds__(256) point_records_kernel(const long long *__restrict__ points,
                                                            const long long *__restrict__ count, long long capacity,
                                                            int batch, int levels, int h, int w, int radius,
                                                            const float *__restrict__ coord_y,
                                                            const float *__restrict__ coord_x, const T *__restrict__ orient,
                                                            const T *__restrict__ line_end, const float *__restrict__ gray,
                                                            long long *__restrict__ frame_offsets,
                                                            float *__restrict__ coords, float *__restrict__ values)
{
    pdl_enter();
    constexpr int kV = 1 + 2 * C;
    const int side = 2 * radius + 1, area = side * side;
    const long long total = __ldg(count);
    const long long rows = total < 0 ? 0 : (total < capacity ? total : capacity);
    const long long images = (long long)batch * levels;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long k = first; k < rows * area; k += stride) {
        const long long i = area == 1 ? k : k / area;
        const int p = (int)(k - i * area), dy = p / side - radius, dx = p % side - radius;
        const long long n = __ldg(points + 4 * i), y = __ldg(points + 4 * i + 1), x = __ldg(points + 4 * i + 2);
        const bool valid = n >= 0 && n < images && y >= 0 && y < h && x >= 0 && x < w;
        float v[kV];
        if (valid && y + dy >= 0 && y + dy < h && x + dx >= 0 && x + dx < w) {
            const size_t pix = ((size_t)n * h + y + dy) * w + x + dx;
            v[0] = __ldg(gray + pix);
#pragma unroll
            for (int c = 0; c < C; ++c) v[1 + c] = widen(orient, pix * C + c), v[1 + C + c] = widen(line_end, pix * C + c);
        } else {
#pragma unroll
            for (int c = 0; c < kV; ++c) v[c] = valid ? 0.0f : NAN;
        }
        if (p == 0) {   // one thread per row writes its coordinates
            float fy = NAN, fx = NAN;
            if (valid) {
                const int l = (int)(n % levels);
                fy = __ldg(coord_y + (size_t)l * h + y);
                fx = __ldg(coord_x + (size_t)l * w + x);
            }
            reinterpret_cast<float2 *>(coords)[i] = make_float2(fy, fx);
        }
        float *dst = values + k * kV;
#pragma unroll
        for (int c = 0; c < kV; ++c) dst[c] = v[c];
    }
    // frame_offsets[f] = the first written row of a level >= f * levels (f = batch: rows)
    for (long long f = first; f <= batch; f += stride) {
        const long long key = f * levels;
        long long lo = 0, hi = rows;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (__ldg(points + 4 * mid) < key) lo = mid + 1;
            else hi = mid;
        }
        frame_offsets[f] = lo;
    }
}

template <int C>
static cudaError_t launch_records(bool half, dim3 grid, cudaStream_t s, const int64_t *points, const int64_t *count,
                                  int64_t capacity, int batch, const silent_plan *plan, int radius, const void *orient,
                                  const void *line_end, const float *gray, int64_t *frame_offsets, float *coords,
                                  float *values)
{
    if (half)
        return launch_dependent(point_records_kernel<C, __half>, grid, dim3(256), 0, s, (const long long *)points,
                                (const long long *)count, (long long)capacity, batch, plan->levels, plan->h, plan->w,
                                radius, (const float *)plan->d_coord_y, (const float *)plan->d_coord_x,
                                (const __half *)orient, (const __half *)line_end, gray, (long long *)frame_offsets,
                                coords, values);
    return launch_dependent(point_records_kernel<C, float>, grid, dim3(256), 0, s, (const long long *)points,
                            (const long long *)count, (long long)capacity, batch, plan->levels, plan->h, plan->w, radius,
                            (const float *)plan->d_coord_y, (const float *)plan->d_coord_x, (const float *)orient,
                            (const float *)line_end, gray, (long long *)frame_offsets, coords, values);
}

// silent_point_records / silent_point_patches: `name` prefixes the error messages
static int point_gather(const char *name, const silent_plan *plan, int batch, const int64_t *points_dev,
                        const int64_t *count_dev, int64_t capacity, const void *orient_dev, const void *line_end_dev,
                        int channels, int half, const float *gray_dev, int radius, int64_t *frame_offsets_dev,
                        float *coords_dev, float *values_dev, silent_stream stream)
{
    if (!plan || !count_dev || !orient_dev || !line_end_dev || !frame_offsets_dev)
        return fail(SILENT_E_INVAL, "%s: null argument", name);
    if (capacity < 0) return fail(SILENT_E_INVAL, "%s: capacity must be >= 0", name);
    if (capacity > 0 && (!points_dev || !coords_dev || !values_dev))
        return fail(SILENT_E_INVAL, "%s: null points, coords or values with capacity %lld", name, (long long)capacity);
    if (channels != 3 && channels != 4 && channels != 8 && channels != 12 && channels != 16)
        return fail(SILENT_E_SHAPE, "%s: channels must be 3, 4, 8, 12 or 16, got %d", name, channels);
    if (radius < 0 || radius > SILENT_PATCH_RADIUS_MAX)
        return fail(SILENT_E_SHAPE, "%s: radius must be in [0, %d], got %d", name, SILENT_PATCH_RADIUS_MAX, radius);
    if (half != 0 && half != 1) return fail(SILENT_E_INVAL, "%s: half must be 0 or 1, got %d", name, half);
    if (batch <= 0) return fail(SILENT_E_INVAL, "%s: batch must be positive", name);
    if (plan->levels == 0) return fail(SILENT_E_SHAPE, "frame is not larger than the pyramid centre: 0 levels");
    if ((int64_t)batch * plan->levels > INT32_MAX)
        return fail(SILENT_E_SHAPE, "%s: batch * levels = %lld is too large", name, (long long)batch * plan->levels);
    if (!gray_dev && batch > plan->ws.batch)
        return fail(SILENT_E_CAPACITY, "%s: the plan's gray holds %d frames (silent_plan_reserve), need %d", name,
                    plan->ws.batch, batch);
    if (!plan->on_device) return fail(SILENT_E_CUDA, "plan was created without a CUDA device; no CPU fallback exists");
    const float *gray = gray_dev ? gray_dev : plan->ws.d_gray;
    // enough threads for the (row, patch pixel) pairs and for the batch + 1 searches, at most a few waves (the loops
    // stride beyond that)
    const int64_t side = 2 * radius + 1, waves = 148 * 8;
    const int64_t work = std::max<int64_t>(std::min<int64_t>(capacity, waves * 256) * side * side, (int64_t)batch + 1);
    const dim3 grid((unsigned)std::min<int64_t>((work + 255) / 256, waves));
    const cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    switch (channels) {
        case 3: e = launch_records<3>(half, grid, s, points_dev, count_dev, capacity, batch, plan, radius, orient_dev, line_end_dev, gray, frame_offsets_dev, coords_dev, values_dev); break;
        case 4: e = launch_records<4>(half, grid, s, points_dev, count_dev, capacity, batch, plan, radius, orient_dev, line_end_dev, gray, frame_offsets_dev, coords_dev, values_dev); break;
        case 8: e = launch_records<8>(half, grid, s, points_dev, count_dev, capacity, batch, plan, radius, orient_dev, line_end_dev, gray, frame_offsets_dev, coords_dev, values_dev); break;
        case 12: e = launch_records<12>(half, grid, s, points_dev, count_dev, capacity, batch, plan, radius, orient_dev, line_end_dev, gray, frame_offsets_dev, coords_dev, values_dev); break;
        default: e = launch_records<16>(half, grid, s, points_dev, count_dev, capacity, batch, plan, radius, orient_dev, line_end_dev, gray, frame_offsets_dev, coords_dev, values_dev); break;
    }
    SILENT_CUDA(e);
    SILENT_LAUNCH_CHECK("point_records_kernel");
    return SILENT_OK;
}

}  // namespace silent

using namespace silent;

extern "C" {

int silent_point_records(const silent_plan *plan, int batch, const int64_t *points_dev, const int64_t *count_dev,
                         int64_t capacity, const void *orient_dev, const void *line_end_dev, int channels, int half,
                         const float *gray_dev, int64_t *frame_offsets_dev, float *coords_dev, float *values_dev,
                         silent_stream stream)
{
    return point_gather("silent_point_records", plan, batch, points_dev, count_dev, capacity, orient_dev, line_end_dev,
                        channels, half, gray_dev, 0, frame_offsets_dev, coords_dev, values_dev, stream);
}

int silent_point_patches(const silent_plan *plan, int batch, const int64_t *points_dev, const int64_t *count_dev,
                         int64_t capacity, const void *orient_dev, const void *line_end_dev, int channels, int half,
                         const float *gray_dev, int radius, int64_t *frame_offsets_dev, float *coords_dev,
                         float *values_dev, silent_stream stream)
{
    return point_gather("silent_point_patches", plan, batch, points_dev, count_dev, capacity, orient_dev, line_end_dev,
                        channels, half, gray_dev, radius, frame_offsets_dev, coords_dev, values_dev, stream);
}

}  // extern "C"
