// NV12 -> BGR: cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12) on the GPU, bit for bit (BT.601 limited range in OpenCV's
// 20-bit fixed point; include/silent_b200.h states the formula). It runs in front of the pyramid of an NV12 plan, which
// then reads uint8 BGR exactly as from a BGR caller, and behind silent_nv12_to_bgr.
//
// One thread converts 2 rows x 16 pixels: the two rows share their 8 (U, V) pairs, so the fast variant reads two 128-bit
// words of Y and one of UV and writes six 128-bit words of BGR (48 bytes per row). A pixel costs three int32 IMADs and
// three clamps. Converting inside the pyramid's phase V instead would repeat the conversion on every fetch of a frame
// word (up to levels x 6 tap rows).
#include "plan.h"
#include "stack.h"

namespace silent {

struct Nv12Args {
    const uint8_t *src;   // frame 0 of the NV12 batch
    size_t src_stride;    // bytes per NV12 frame (H * W * 3 / 2)
    int H, W;
    uint8_t *dst;         // frame 0 of the BGR batch
    size_t dst_stride;    // bytes per BGR frame
    int dst_pitch;        // bytes per BGR row
    int y0, x0, x1;       // first row (even), first column (multiple of 16), column end of the converted region
    int runs, tasks;      // 16-pixel runs per row pair, runs x row pairs per frame
};

__device__ __forceinline__ int sat8(int v) { return min(max(v, 0), 255); }

// VEC: every Y and UV word is 16-byte aligned (W % 16 == 0 and an aligned source), so a run is three 128-bit loads.
// Otherwise bytes are loaded one by one, and only the pixels before x1 are stored.
template <bool VEC>
__global__ void __launch_bounds__(128) nv12_to_bgr_kernel(const __grid_constant__ Nv12Args A)
{
    pdl_enter();
    const int task = blockIdx.x * blockDim.x + threadIdx.x;
    if (task >= A.tasks) return;
    const int pair = task / A.runs, run = task - pair * A.runs;
    const int y = A.y0 + 2 * pair, x = A.x0 + 16 * run;
    const uint8_t *frame = A.src + (size_t)blockIdx.y * A.src_stride;
    const uint8_t *yrow = frame + (size_t)y * A.W + x;
    const uint8_t *uvrow = frame + (size_t)(A.H + (y >> 1)) * A.W + 2 * (x >> 1);   // absolute chroma coordinates
    const int n = VEC ? 16 : min(16, A.x1 - x);
    uint32_t yw[2][4], uvw[4];
    if constexpr (VEC) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(yrow));
        const uint4 b = __ldg(reinterpret_cast<const uint4 *>(yrow + A.W));
        const uint4 c = __ldg(reinterpret_cast<const uint4 *>(uvrow));
        yw[0][0] = a.x, yw[0][1] = a.y, yw[0][2] = a.z, yw[0][3] = a.w;
        yw[1][0] = b.x, yw[1][1] = b.y, yw[1][2] = b.z, yw[1][3] = b.w;
        uvw[0] = c.x, uvw[1] = c.y, uvw[2] = c.z, uvw[3] = c.w;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) yw[0][k] = yw[1][k] = uvw[k] = 0u;
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (i < n) {
                yw[0][i >> 2] |= (uint32_t)__ldg(yrow + i) << (8 * (i & 3));
                yw[1][i >> 2] |= (uint32_t)__ldg(yrow + A.W + i) << (8 * (i & 3));
                uvw[i >> 2] |= (uint32_t)__ldg(uvrow + i) << (8 * (i & 3));
            }
    }
    uint32_t ow[2][12];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int k = 0; k < 12; ++k) ow[r][k] = 0u;
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        const int u = (int)((uvw[p >> 1] >> (16 * (p & 1))) & 0xff) - 128;
        const int v = (int)((uvw[p >> 1] >> (16 * (p & 1) + 8)) & 0xff) - 128;
        const int cb = (1 << 19) + 2116026 * u;
        const int cg = (1 << 19) - 852492 * v - 409993 * u;
        const int cr = (1 << 19) + 1673527 * v;
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int i = 2 * p + k;   // pixel of the run; its bytes are 3i .. 3i + 2
                const int yy = max(0, (int)((yw[r][i >> 2] >> (8 * (i & 3))) & 0xff) - 16) * 1220542;
                const int bgr[3] = {sat8((yy + cb) >> 20), sat8((yy + cg) >> 20), sat8((yy + cr) >> 20)};
#pragma unroll
                for (int c = 0; c < 3; ++c) ow[r][(3 * i + c) >> 2] |= (uint32_t)bgr[c] << (8 * ((3 * i + c) & 3));
            }
    }
    uint8_t *out = A.dst + (size_t)blockIdx.y * A.dst_stride + (size_t)y * A.dst_pitch + (size_t)x * 3;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        uint8_t *o = out + (size_t)r * A.dst_pitch;
        if (VEC || (n == 16 && ((uintptr_t)o & 15) == 0)) {
            uint4 *o4 = reinterpret_cast<uint4 *>(o);
#pragma unroll
            for (int k = 0; k < 3; ++k) o4[k] = make_uint4(ow[r][4 * k], ow[r][4 * k + 1], ow[r][4 * k + 2], ow[r][4 * k + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < 48; ++j)
                if (j < 3 * n) o[j] = (uint8_t)(ow[r][j >> 2] >> (8 * (j & 3)));
        }
    }
}

// rows [y0, y1) (even bounds) x columns [x0, x1) (x0 a multiple of 16) of `batch` NV12 frames -> BGR frames at
// dst_pitch / dst_stride. Host-side shape checks are the callers'.
static int launch_nv12(const uint8_t *src, int batch, int H, int W, uint8_t *dst, size_t dst_stride, int dst_pitch,
                       int y0, int y1, int x0, int x1, cudaStream_t stream)
{
    if (y1 <= y0 || x1 <= x0) return SILENT_OK;
    Nv12Args A;
    A.src = src, A.src_stride = (size_t)H * W * 3 / 2, A.H = H, A.W = W;
    A.dst = dst, A.dst_stride = dst_stride, A.dst_pitch = dst_pitch;
    A.y0 = y0, A.x0 = x0, A.x1 = x1;
    A.runs = ceil_div(x1 - x0, 16);
    const int64_t tasks = (int64_t)A.runs * ((y1 - y0) / 2);
    if (tasks > INT32_MAX - 128) return fail(SILENT_E_SHAPE, "NV12 frame of %dx%d is too large", H, W);
    if (batch > 65535) return fail(SILENT_E_SHAPE, "at most 65535 NV12 frames per conversion, got %d", batch);
    A.tasks = (int)tasks;
    const bool vec = W % 16 == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0 && dst_pitch % 16 == 0 &&
                     dst_stride % 16 == 0 && (x1 - x0) % 16 == 0;
    const dim3 grid(ceil_div(A.tasks, 128), batch);
    SILENT_CUDA(launch_dependent(vec ? nv12_to_bgr_kernel<true> : nv12_to_bgr_kernel<false>, grid, dim3(128), 0, stream, A));
    SILENT_LAUNCH_CHECK("nv12_to_bgr_kernel");
    return SILENT_OK;
}

int nv12_convert(const silent_plan *plan, const void *nv12_dev, int frame0, int nb, cudaStream_t stream)
{
    const silent_params &p = plan->params;
    const size_t src_frame = (size_t)p.frame_h * p.frame_w * 3 / 2;
    return launch_nv12((const uint8_t *)nv12_dev + src_frame * frame0, nb, p.frame_h, p.frame_w,
                       plan->ws.d_bgr + (size_t)plan->frame_stride * frame0, (size_t)plan->frame_stride,
                       (int)plan->frame_pitch, plan->nv12_y0, plan->nv12_y1, plan->nv12_x0, plan->nv12_x1, stream);
}

}  // namespace silent

extern "C" int silent_nv12_to_bgr(const uint8_t *nv12_dev, int batch, int h, int w, uint8_t *bgr_dev,
                                  silent_stream stream)
{
    using namespace silent;
    if (!nv12_dev || !bgr_dev) return fail(SILENT_E_INVAL, "silent_nv12_to_bgr: null argument");
    if (batch <= 0) return fail(SILENT_E_INVAL, "silent_nv12_to_bgr: batch must be positive, got %d", batch);
    if (h <= 0 || w <= 0) return fail(SILENT_E_INVAL, "silent_nv12_to_bgr: frame size must be positive, got %dx%d", h, w);
    if (h % 2 || w % 2) return fail(SILENT_E_SHAPE, "silent_nv12_to_bgr: NV12 frames need even height and width, got %dx%d", h, w);
    if ((int64_t)w * 3 > INT32_MAX) return fail(SILENT_E_SHAPE, "silent_nv12_to_bgr: frame width %d is too large", w);
    return launch_nv12(nv12_dev, batch, h, w, bgr_dev, (size_t)h * w * 3, w * 3, 0, h, 0, w, (cudaStream_t)stream);
}
