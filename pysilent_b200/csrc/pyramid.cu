// K1: foveated pyramid build = zoom.from_image (reference util/zoom/from_image.py:48-64) for a batch of frames:
// per level, a centred crop resampled to h x w with the order-5 spline of scipy.ndimage.zoom(prefilter=False).
//
// Canonical order (oracle/silent_oracle.c:so_pyramid): separable, VERTICAL pass first -- for each of the 6 source
// columns an fmaf chain over the 6 y-taps -- then the fmaf chain over the 6 x-taps.
//
// Two kernels:
//  * pyramid_kernel      one thread per output pixel, NHWC float32 output: the stand-alone from_image operator, any
//                        channel count / frame dtype. Frames are read at the plan's row pitch and frame stride.
//  * pyramid_pair_kernel the pipeline's producer. One CTA = one tile of one level for TWO frames in lockstep (float2
//                        lanes, like the stack kernels). Phase V walks ALIGNED 128-bit words of the uint8 frame down the
//                        6 tap rows (coalesced, 16 byte-columns per load), converts with PRMT + FADD2 (the I2F pipe is
//                        16/clk/SM on B200: measured 2.4x slower), accumulates with FFMA2 and parks the column sums in
//                        shared memory; phase H gathers 6 of them per output sample. ~10x fewer instructions than the
//                        per-pixel kernel (which re-converts every tap for every pixel). Output is the pair-interleaved
//                        planar layout xpair[pair][c][y][x] = (frame A, frame B) that stack_a_kernel loads verbatim.
//                        One launch covers every level, coarsest first (it pulls a frame pair through L2 once; finer
//                        levels re-read their crops from L2) and bulk-prefetches the next pair's rows into L2. Tile
//                        width (72 columns for 288-wide levels) and height are chosen per plan (plan.cu). The frame
//                        words and the phase-H table entries arrive through the TEXTURE path (tex1Dfetch on linear
//                        textures, SASS TLD.LZ): the kernel is bound by the LSU's L1 data pipe, which the texture
//                        unit's own write-back bypasses. The first CTA of every pair also zeroes the buffers that the
//                        kernels AFTER this one expect clean (PairClear), so the step has no memset of its own.
#include <algorithm>

#include "plan.h"
#include "stack.h"

namespace silent {

template <typename T>
__device__ __forceinline__ float load_sample(const T *p);
template <>
__device__ __forceinline__ float load_sample<uint8_t>(const uint8_t *p) { return (float)__ldg(p); }
template <>
__device__ __forceinline__ float load_sample<float>(const float *p) { return __ldg(p); }

template <typename T, int NC>
__global__ void __launch_bounds__(256) pyramid_kernel(const T *__restrict__ frames, float *__restrict__ out,
                                                      const int32_t *__restrict__ idx_y, const float *__restrict__ w_y,
                                                      const int32_t *__restrict__ idx_x, const float *__restrict__ w_x,
                                                      int L, int h, int w, size_t frame_stride, int row_pitch, int FC)
{
    const int ox = blockIdx.x * blockDim.x + threadIdx.x;
    const int oy = blockIdx.y * blockDim.y + threadIdx.y;
    const int n = blockIdx.z;   // frame * L + level
    if (ox >= w || oy >= h) return;
    const int s = n % L, b = n / L;
    const int32_t *ty = idx_y + ((size_t)s * h + oy) * kTaps;
    const int32_t *tx = idx_x + ((size_t)s * w + ox) * kTaps;
    const float *gy = w_y + ((size_t)s * h + oy) * kTaps;
    const float *gx = w_x + ((size_t)s * w + ox) * kTaps;
    float *dst = out + (((size_t)n * h + oy) * w + ox) * NC;

    float acc[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] = 0.0f;

    if (__ldg(ty) >= 0 && __ldg(tx) >= 0) {
        const T *frame = frames + (size_t)b * frame_stride;
        size_t row_off[kTaps];
        float wy[kTaps];
#pragma unroll
        for (int j = 0; j < kTaps; ++j) {
            row_off[j] = (size_t)__ldg(ty + j) * row_pitch;
            wy[j] = __ldg(gy + j);
        }
#pragma unroll
        for (int i = 0; i < kTaps; ++i) {
            const int col = __ldg(tx + i) * FC;
            const float wxi = __ldg(gx + i);
            float t[NC];
#pragma unroll
            for (int c = 0; c < NC; ++c) t[c] = 0.0f;
#pragma unroll
            for (int j = 0; j < kTaps; ++j) {
#pragma unroll
                for (int c = 0; c < NC; ++c) t[c] = fmaf(wy[j], load_sample<T>(frame + row_off[j] + col + c), t[c]);
            }
#pragma unroll
            for (int c = 0; c < NC; ++c) acc[c] = fmaf(wxi, t[c], acc[c]);
        }
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) dst[c] = acc[c];
}

template <typename T>
static int launch_pyramid(const silent_plan *plan, const T *frames, int batch, float *out, cudaStream_t stream)
{
    const int L = plan->levels, h = plan->h, w = plan->w;
    const silent_params &p = plan->params;
    dim3 block(32, 8);
    dim3 grid(ceil_div(w, 32), ceil_div(h, 8), batch * L);
#define SILENT_PYR_CASE(NC)                                                                                           \
    case NC:                                                                                                          \
        pyramid_kernel<T, NC><<<grid, block, 0, stream>>>(frames, out, plan->d_idx_y, plan->d_w_y, plan->d_idx_x,     \
                                                          plan->d_w_x, L, h, w, (size_t)plan->frame_stride,           \
                                                          (int)plan->frame_pitch, p.frame_c);                         \
        break;
    switch (p.num_colors) {
        SILENT_PYR_CASE(1)
        SILENT_PYR_CASE(2)
        SILENT_PYR_CASE(3)
        SILENT_PYR_CASE(4)
        SILENT_PYR_CASE(5)
        SILENT_PYR_CASE(6)
        SILENT_PYR_CASE(7)
        SILENT_PYR_CASE(8)
        default:
            return fail(SILENT_E_SHAPE, "num_colors=%d not supported (1..8)", p.num_colors);
    }
#undef SILENT_PYR_CASE
    SILENT_LAUNCH_CHECK("pyramid_kernel");
    return SILENT_OK;
}

int pyramid_build(const silent_plan *plan, const void *frames_dev, int batch, float *pyramid_dev, cudaStream_t stream)
{
    if (!plan || !frames_dev || !pyramid_dev) return fail(SILENT_E_INVAL, "silent_pyramid_build: null argument");
    if (batch <= 0) return fail(SILENT_E_INVAL, "batch must be positive, got %d", batch);
    if (plan->levels == 0) return SILENT_OK;
    if (!plan->on_device) return fail(SILENT_E_CUDA, "plan was created without a CUDA device; no CPU fallback exists");
    if ((long long)batch * plan->levels > 65535) return fail(SILENT_E_SHAPE, "batch * levels must be <= 65535");
    if (plan->params.frame_dtype != SILENT_F32)   // uint8 BGR frames, or NV12 frames converted to them
        return launch_pyramid<uint8_t>(plan, (const uint8_t *)frames_dev, batch, pyramid_dev, stream);
    return launch_pyramid<float>(plan, (const float *)frames_dev, batch, pyramid_dev, stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// frame-pair kernel
// ---------------------------------------------------------------------------------------------------------------------

typedef float2 f2;
constexpr int kVGroup = kPairVGroup;   // float2 slots per group of 16 byte-columns in the column-sum buffer (plan.h)

struct PairParams {
    const uint8_t *frames;
    cudaTextureObject_t frames_tex;   // TEX variant: the same frames as a linear texture of 128-bit texels
    cudaTextureObject_t htab_tex;     // TEX variant: htab as a texture of int4 texels
    f2 *xpair;
    const int4 *ytab;     // [L][h][3]: phase-V table (first tap row's byte offset, step, six weights | other offsets; plan.cu)
    const int4 *words;    // [L][kPairMaxTiles]: (first 32-bit word of a frame row, word count, 2^32 / groups + 1, 0) per x tile
    const int4 *htab;     // [L][w][3][3]: phase-H tap offsets in the tile's column-sum row + six weights (plan.cu)
    size_t frame_bytes;
    int h, w, L, B, tile_w;
    uint4 *clear_a;       // zeroed by the first CTA of every pair (PairClear, stack.h): n16 128-bit words ...
    uint32_t *clear_b;    // ... and n32 32-bit words
    unsigned clear_n16, clear_n32;
    // ONE launch covers every level: blockIdx.x is the x tile, blockIdx.y enumerates the tile rows of a frame pair with
    // the COARSEST level first (it pulls the whole frame through L2; the finer levels, whose crops are subsets, then hit
    // L2), blockIdx.z the pair.
    int th[kPairMaxLevels];            // output rows per tile
    int vpitch[kPairMaxLevels];        // float2 per row of the column-sum buffer
    int row_start[kPairMaxLevels + 1];   // first blockIdx.y by order position k (level = L - 1 - k)
};

// byte k of `word` as an exact float: PRMT builds the bit pattern of 2^23 + byte, the caller subtracts 2^23 (FADD2)
__device__ __forceinline__ float magic_byte(uint32_t word, uint32_t selector)
{
    return __uint_as_float(__byte_perm(word, 0x4B000000u, selector));
}

// TEX: phase V fetches the frame rows as 128-bit texels (tex1Dfetch, SASS TLD.LZ) instead of LDG.128. The kernel is
// bound by the L1 data pipe of the LSU (86 % busy with LDG; a 512-byte LDG.128 costs 8 of its wavefronts -- the row loads
// were 28 % of the kernel's total, the table loads another 14 %): the texture path returns its data through the TEX
// pipe's own write-back and leaves the LSU pipe to the shared-memory traffic of both phases (measured: 0.262 -> 0.250 ms
// with the rows, 0.245 ms with the phase-H table entries too; the phase-V table entries gain nothing -- their latency
// sits in front of every task's row loads, so they always take LDG). Same bits either way: TEX = false is the variant for
// frame buffers the texture unit cannot address.
template <bool TEX>
__global__ void __launch_bounds__(kPairThreads, 768 / kPairThreads) pyramid_pair_kernel(const __grid_constant__ PairParams P)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    f2 *sV = reinterpret_cast<f2 *>(smem_raw);                          // [th][vpitch] column sums (frame A, frame B)
    pdl_enter();

    const int tid = threadIdx.x;
    if (blockIdx.x == 0 && blockIdx.y == 0) {   // (after the wait: the previous step's kernels have read these buffers)
        const unsigned stride = gridDim.z * kPairThreads;
        for (unsigned i = blockIdx.z * kPairThreads + tid; i < P.clear_n16; i += stride) P.clear_a[i] = make_uint4(0, 0, 0, 0);
        for (unsigned i = blockIdx.z * kPairThreads + tid; i < P.clear_n32; i += stride) P.clear_b[i] = 0u;
    }
    int k = 0;
    while (k + 1 < P.L && (int)blockIdx.y >= P.row_start[k + 1]) ++k;
    const int level = P.L - 1 - k, bx = blockIdx.x, by = blockIdx.y - P.row_start[k], q = blockIdx.z;
    const int th = P.th[level], vpitch = P.vpitch[level], h = P.h, w = P.w;
    const int oy0 = by * th;
    const int rows = min(th, h - oy0);
    // (first word, word count, reciprocal of the group count) of this x tile; nothing is staged in shared memory before
    // phase V: every task reads its row's tap offsets and weights straight from the (L1-resident) table
    const int4 span = __ldg(P.words + (size_t)level * kPairMaxTiles + bx);
    const int4 *ytab = P.ytab + ((size_t)level * h + oy0) * 3;
    const uint8_t *frameA = P.frames + (size_t)(2 * q) * P.frame_bytes + (size_t)span.x * 4;
    const uint8_t *frameB = (2 * q + 1 < P.B) ? frameA + P.frame_bytes : frameA;
    const int nq = span.y >> 2;
    const uint32_t magic = (uint32_t)span.z;
    // texel (16-byte) index of this tile's first word in frames A and B (every term is a multiple of 16 bytes)
    const int texA = (int)(((size_t)(2 * q) * P.frame_bytes + (size_t)span.x * 4) >> 4);
    const int texB = (2 * q + 1 < P.B) ? texA + (int)(P.frame_bytes >> 4) : texA;

    // ---- the coarsest level is the first reader of a frame pair (finer levels then hit L2): ask L2 for the same tile of
    //      the NEXT pair now, one bulk prefetch per (tap row, frame), so that CTA finds its rows in L2 instead of HBM --
    if (level == P.L - 1 && 2 * (q + 1) < P.B && nq > 0) {
        const int32_t *yt = reinterpret_cast<const int32_t *>(ytab);
        for (int i = tid; i < 2 * rows * kTaps; i += kPairThreads) {
            const int e = i >> 1, f = 2 + (i & 1), r = e / kTaps, j = e - kTaps * r;
            const int off0 = __ldg(yt + 12 * r), step = __ldg(yt + 12 * r + 1);
            const int off = step > 0 ? off0 + j * step : j == 0 ? off0 : j == 5 ? -step - 1 : __ldg(yt + 12 * r + 7 + j);
            if (off0 >= 0 && 2 * q + f < P.B) {
                const uint8_t *src = frameA + (size_t)f * P.frame_bytes + off;
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(span.y * 4) : "memory");
            }
        }
    }

    // ---- phase V: column sums over the 6 y-taps, 16 byte-columns (one aligned 128-bit load per tap row and frame) per
    //      task: 12 independent 16-byte loads in flight per thread cover the HBM/L2 latency ---------------------------
    const f2 bias = make_float2(-8388608.0f, -8388608.0f);
    for (int t = tid; t < rows * nq; t += kPairThreads) {
        const int r = nq > 1 ? (int)__umulhi((uint32_t)t, magic) : t, qi = t - r * nq;
        // the row's table entry: two 128-bit words (first offset, step, six weights); a third one only for the few rows
        // whose tap rows are not consecutive (mirrored at the crop's edge)
        const int4 y0 = __ldg(ytab + 3 * r), y1 = __ldg(ytab + 3 * r + 1);
        f2 acc[16];
        if (y0.x < 0) {
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = make_float2(0.0f, 0.0f);
        } else {
            int yoff[kTaps];
            if (y0.y > 0) {
#pragma unroll
                for (int j = 0; j < kTaps; ++j) yoff[j] = y0.x + j * y0.y;
            } else {
                const int4 y2 = __ldg(ytab + 3 * r + 2);
                yoff[0] = y0.x, yoff[1] = y2.x, yoff[2] = y2.y, yoff[3] = y2.z, yoff[4] = y2.w, yoff[5] = -y0.y - 1;
            }
            const float wyv[kTaps] = {__int_as_float(y0.z), __int_as_float(y0.w), __int_as_float(y1.x),
                                      __int_as_float(y1.y), __int_as_float(y1.z), __int_as_float(y1.w)};
            uint4 qa[kTaps], qb[kTaps];
#pragma unroll
            for (int j = 0; j < kTaps; ++j) {
                if constexpr (TEX) {
                    qa[j] = tex1Dfetch<uint4>(P.frames_tex, texA + (yoff[j] >> 4) + qi);
                    qb[j] = tex1Dfetch<uint4>(P.frames_tex, texB + (yoff[j] >> 4) + qi);
                } else {
                    qa[j] = __ldg(reinterpret_cast<const uint4 *>(frameA + yoff[j]) + qi);
                    qb[j] = __ldg(reinterpret_cast<const uint4 *>(frameB + yoff[j]) + qi);
                }
            }
            // The first tap is a plain product: fma(w, v, +0) and w * v differ only when the product is -0 (a negative
            // weight on a zero byte), and a -0 column sum cannot change any output bit (phase H adds every term to +0).
#pragma unroll
            for (int j = 0; j < kTaps; ++j) {
                const f2 wy2 = make_float2(wyv[j], wyv[j]);
                const uint32_t wa[4] = {qa[j].x, qa[j].y, qa[j].z, qa[j].w}, wb[4] = {qb[j].x, qb[j].y, qb[j].z, qb[j].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const f2 v = __fadd2_rn(make_float2(magic_byte(wa[k], 0x7440 + b), magic_byte(wb[k], 0x7440 + b)), bias);
                        acc[4 * k + b] = j == 0 ? __fmul2_rn(wy2, v) : __ffma2_rn(wy2, v, acc[4 * k + b]);
                    }
                }
            }
        }
        // 16 columns = 128 B per task: padded to 144 B so consecutive lanes start in consecutive 16-byte bank groups
        float4 *dst = reinterpret_cast<float4 *>(sV + (size_t)r * vpitch + kVGroup * qi);
#pragma unroll
        for (int k = 0; k < 8; ++k) dst[k] = make_float4(acc[2 * k].x, acc[2 * k].y, acc[2 * k + 1].x, acc[2 * k + 1].y);
    }
    if (nq == 0 && tid < rows) sV[(size_t)tid * vpitch] = make_float2(0.0f, 0.0f);   // a tile without any defined column:
    __syncthreads();                                                                  // phase H reads slot 0 with weight 0

    // ---- phase H: chain over the 6 x-taps. A thread owns one (output column, channel) and walks all rows of the tile:
    //      its six column-sum offsets and weights come from a host-built table (three 128-bit loads, no arithmetic), each
    //      row then costs 6 LDS.64 + 6 FFMA2 + 1 store.
    // Lanes interleave (column, channel): three consecutive lanes read three consecutive column sums (the B, G, R bytes
    // of one source pixel), so a warp's gather touches a third of the 128-byte lines it would with one channel per warp.
    const size_t plane = (size_t)h * w;
    for (int item = tid; item < 3 * P.tile_w; item += kPairThreads) {   // one pass when the CTA has >= 3 * tile_w threads
        const int c = item % 3;
        const int ox = bx * P.tile_w + item / 3;
        if (ox >= w) break;
        int4 t0, t1, t2;
        if constexpr (TEX) {
            const int ht = (level * w + ox) * 9 + 3 * c;
            t0 = tex1Dfetch<int4>(P.htab_tex, ht), t1 = tex1Dfetch<int4>(P.htab_tex, ht + 1), t2 = tex1Dfetch<int4>(P.htab_tex, ht + 2);
        } else {
            const int4 *tab = P.htab + ((size_t)level * w + ox) * 9 + 3 * c;
            t0 = __ldg(tab), t1 = __ldg(tab + 1), t2 = __ldg(tab + 2);
        }
        const int off[kTaps] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y};
        const float wv[kTaps] = {__int_as_float(t1.z), __int_as_float(t1.w), __int_as_float(t2.x),
                                 __int_as_float(t2.y), __int_as_float(t2.z), __int_as_float(t2.w)};
        f2 wx[kTaps];
#pragma unroll
        for (int i = 0; i < kTaps; ++i) wx[i] = make_float2(wv[i], wv[i]);
        f2 *out = P.xpair + (((size_t)q * P.L + level) * 3 + c) * plane + (size_t)oy0 * w + ox;
        for (int r = 0; r < rows; ++r) {
            const f2 *row = sV + (size_t)r * vpitch;
            f2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
            for (int i = 0; i < kTaps; ++i) acc = __ffma2_rn(wx[i], row[off[i]], acc);   // zero weights for undefined columns
            out[(size_t)r * w] = acc;
        }
    }
}

// Can the pair kernel serve this plan? (uint8 frames, or NV12 frames converted to them, 3 colours, 16-byte aligned rows,
// table of tiles fits)
bool pyramid_pair_supported(const silent_plan *plan)
{
    const silent_params &p = plan->params;
    return plan->on_device && (p.frame_dtype == SILENT_U8 || p.frame_dtype == SILENT_NV12) && p.num_colors == 3 &&
           plan->frame_pitch % 16 == 0 && plan->pair_ok;
}

size_t pyramid_pair_bytes(const silent_plan *plan, int batch)
{
    return (size_t)((batch + 1) / 2) * plan->levels * 3 * plan->h * plan->w * sizeof(f2);
}

int pyramid_pair_build(const silent_plan *plan, const void *frames_dev, int batch, void *xpair_dev, cudaStream_t stream,
                       const PairClear *clear)
{
    if (!pyramid_pair_supported(plan)) return fail(SILENT_E_SHAPE, "frame-pair pyramid kernel does not support this plan");
    if (((uintptr_t)frames_dev & 15) != 0) return fail(SILENT_E_INVAL, "frames must be 16-byte aligned");
    const int pairs = (batch + 1) / 2;
    if (pairs > 65535) return fail(SILENT_E_SHAPE, "at most 131070 frames per call");
    // frames as a texture of 128-bit texels (cached per plan: same pointer and size -> same object). The texture variant
    // needs a pointer at the device's texture alignment (CUDA requires it of a linear texture's devPtr), fewer than 2^27
    // texels (1-D linear textures; the texel index is a 32-bit int) and the phase-H table's texture; any other buffer
    // takes the LDG variant, which computes the same bits
    const size_t total_bytes = (size_t)batch * plan->frame_stride;
    bool use_tex = plan->texture_alignment > 0 && (uintptr_t)frames_dev % (uintptr_t)plan->texture_alignment == 0 &&
                   (total_bytes >> 4) < ((size_t)1 << 27) && plan->htab_tex != 0;
    cudaTextureObject_t tex = 0;
    if (use_tex) {
        silent_plan *mp = const_cast<silent_plan *>(plan);   // (the cache is plan-owned scratch, like the workspace)
        for (const silent_plan::FrameTexture &ft : mp->frame_textures)
            if (ft.ptr == frames_dev && ft.bytes == total_bytes) tex = ft.tex;
        if (tex == 0) {
            constexpr size_t kMaxFrameTextures = 64;
            if (mp->frame_textures.size() >= kMaxFrameTextures) {   // rare: drop them all, once nothing can be reading them
                SILENT_CUDA(cudaDeviceSynchronize());
                for (silent_plan::FrameTexture &ft : mp->frame_textures) cudaDestroyTextureObject(ft.tex);
                mp->frame_textures.clear();
            }
            cudaResourceDesc rd = {};
            rd.resType = cudaResourceTypeLinear;
            rd.res.linear.devPtr = const_cast<void *>(frames_dev);
            rd.res.linear.desc = cudaCreateChannelDesc<uint4>();
            rd.res.linear.sizeInBytes = total_bytes;
            cudaTextureDesc td = {};
            td.readMode = cudaReadModeElementType;
            cudaTextureObject_t obj = 0;
            if (cudaCreateTextureObject(&obj, &rd, &td, nullptr) == cudaSuccess) {
                silent_plan::FrameTexture ft;
                ft.ptr = frames_dev, ft.bytes = total_bytes, ft.tex = obj;
                mp->frame_textures.push_back(ft);
                tex = obj;
            } else {
                (void)cudaGetLastError();   // the LDG variant computes the same bits
                use_tex = false;
            }
        }
    }
    const auto kernel = use_tex ? pyramid_pair_kernel<true> : pyramid_pair_kernel<false>;
    // per launch, not once per process: the attribute belongs to the CURRENT device's context, and one process may
    // drive several GPUs (one LineEndPipeline per camera thread and device)
    SILENT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    PairParams P;
    P.frames = (const uint8_t *)frames_dev;
    P.frames_tex = tex;
    P.htab_tex = plan->htab_tex;
    P.xpair = (f2 *)xpair_dev;
    P.ytab = reinterpret_cast<const int4 *>(plan->d_pair_ytab);
    P.words = reinterpret_cast<const int4 *>(plan->d_pair_words);
    P.htab = reinterpret_cast<const int4 *>(plan->d_pair_htab);
    P.frame_bytes = (size_t)plan->frame_stride;
    P.h = plan->h, P.w = plan->w, P.L = plan->levels, P.B = batch;
    P.tile_w = plan->pair_tile_w;
    P.clear_a = clear ? (uint4 *)clear->a : nullptr, P.clear_n16 = clear && clear->a ? (unsigned)(clear->a_bytes / 16) : 0u;
    P.clear_b = clear ? (uint32_t *)clear->b : nullptr, P.clear_n32 = clear && clear->b ? (unsigned)(clear->b_bytes / 4) : 0u;
    size_t smem = 0;
    int tile_rows = 0;
    for (int k = 0; k < plan->levels; ++k) {   // coarsest level first
        const int s = plan->levels - 1 - k;
        const PairLevel &pl = plan->pair[s];
        P.th[s] = pl.th;
        P.vpitch[s] = pl.vpitch;
        P.row_start[k] = tile_rows;
        tile_rows += ceil_div(plan->h, pl.th);
        smem = std::max(smem, std::max((size_t)16, (size_t)pl.th * pl.vpitch * sizeof(f2)));
    }
    P.row_start[plan->levels] = tile_rows;
    if (tile_rows > 65535) return fail(SILENT_E_SHAPE, "too many tile rows for one launch (%d)", tile_rows);
    SILENT_CUDA(launch_dependent(kernel, dim3(plan->pair[0].ntx, tile_rows, pairs), dim3(kPairThreads), smem,
                                 stream, P));
    SILENT_LAUNCH_CHECK("pyramid_pair_kernel");
    return SILENT_OK;
}

}  // namespace silent

extern "C" int silent_pyramid_build(const silent_plan *plan, const void *frames_dev, int batch, float *pyramid_dev,
                                    silent_stream stream)
{
    using namespace silent;
    // NV12 frames are converted into the plan's buffer first; pyramid_build reads them there
    if (plan && frames_dev && pyramid_dev && batch > 0 && plan->levels > 0 && plan->params.frame_dtype == SILENT_NV12) {
        if (!plan->on_device) return fail(SILENT_E_CUDA, "plan was created without a CUDA device; no CPU fallback exists");
        if (plan->ws.batch < batch)
            return fail(SILENT_E_CAPACITY, "NV12 plan holds converted frames for %d frames, need %d: call silent_plan_reserve",
                        plan->ws.batch, batch);
        const int rc = nv12_convert(plan, frames_dev, 0, batch, (cudaStream_t)stream);
        if (rc != SILENT_OK) return rc;
        frames_dev = plan->ws.d_bgr;
    }
    return pyramid_build(plan, frames_dev, batch, pyramid_dev, (cudaStream_t)stream);
}
