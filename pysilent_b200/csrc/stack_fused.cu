// K2: the fused stack S1-S7 of LineEndDisplayer.compile (reference recognition_testing.py:69-77):
//   rgc 3x3 + relu -> rgby 3x3 + relu -> stripe 3x3 + relu -> 7x7 blur regulator -> end 3x3 + relu + clip ->
//   border mask -> channel mean (+ per-region maxima for the feature-point emit).
//
// B200 design (measured: v1, one thread per pixel reading shared memory per tap, was instruction-issue bound at ~1400
// thread-instructions per pixel against ~240 useful FMAs):
//  * TWO IMAGES IN LOCKSTEP. Every value in shared memory and registers is a float2 (image A, image B) of the same
//    pixel/channel of two pyramid levels, so every tap is an aligned pair: all arithmetic is FFMA2/FADD2/FMUL2
//    (sm_100 packed fp32: one issue slot for two FMAs), every shared-memory access is a 128-bit LDS/STS of two pixels,
//    and the weights ride in uniform registers as (w, w) pairs straight from the kernel-parameter constant bank.
//  * REGISTER BLOCKING. A thread owns a run of 8 pixels of one row; for each (ky, ci) it loads the 10 (14 for the blur)
//    input columns once with 128-bit loads and feeds all kx taps / outputs from registers: ~13 FMAs per load.
//    Lanes of a warp walk ROWS and the row pitch is an odd multiple of 16 B, so the 128-bit accesses are conflict-free.
//  * TWO KERNELS, CUT AT THE ONE-CHANNEL TENSOR. stack_a: x -> rgc -> rgby -> channel sum b (1 channel, written as
//    interleaved pairs); stack_b: b -> stripe -> regulator -> end -> outputs. The stripe filter only needs the channel
//    sum of b, so the cut costs 2 x 1/6 of the output traffic but shrinks halos (2 and 5 instead of 7), which keeps
//    the redundant halo arithmetic at ~15 % with 32 x 48 tiles (288-wide levels: 6 tiles, no ragged edge).
//  * zero weights cost nothing: rgc is depthwise and rgby has 28 structural zeros; both patterns are verified on the
//    host and compiled out (dense variants exist for arbitrary weights).
//  * TILES IN BY TMA, ROWS OUT BY BULK STORES. Inputs arrive as one cp.async.bulk.tensor box (zero fill = SAME padding);
//    outputs are staged in shared memory in NHWC order and leave as one cp.async.bulk store per row, issued by a few
//    lanes of every warp; in stack_b the warps that have no S5 task restage and store `orient` behind a named barrier
//    while the others run the end filter. Kernels of one step are chained by programmatic dependent launch.
// Evaluation order = canonical order of oracle/silent_oracle.c (chains in (ky, ci, kx) order), so results are
// bit-identical to it. Tensor cores do not apply (3-channel fp32 stencils); measured, the path is bound by packed-fp32
// issue and shared-memory bandwidth rather than HBM (DESIGN.md section 4).
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <mutex>
#include <vector>

#include "plan.h"
#include "stack.h"

namespace silent {

typedef float2 f2;

__device__ __forceinline__ f2 fma2(f2 w, f2 v, f2 a) { return __ffma2_rn(w, v, a); }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ f2 zero2() { return make_float2(0.0f, 0.0f); }

// relu / clip that propagate NaN (canon_relu / canon_clip_hi on every reachable value; -0 never occurs, see DESIGN.md)
__device__ __forceinline__ float relu_nan(float v)
{
    float r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float clip_nan(float v, float hi)
{
    float r;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "f"(hi));
    return r;
}
__device__ __forceinline__ f2 relu2_finite(f2 v) { return make_float2(relu_nan(v.x), relu_nan(v.y)); }
__device__ __noinline__ float slow_gain(float m, float value, float root) { return canon_gain(m, value, root); }

constexpr int kPX = 8;   // pixels per thread run

// ---- TMA (cp.async.bulk.tensor) tile loads: one elected thread issues a 3-D box copy global -> shared; the hardware
//      zero-fills everything outside the tensor, which is exactly the SAME padding of the first convolution of a kernel.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_box3(void *dst, const CUtensorMap *map, int c0, int c1, int c2, uint64_t *bar,
                                              uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
            "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}

// ---- bulk stores (cp.async.bulk shared -> global): one instruction moves a whole staged row; the TMA unit does the
//      address arithmetic that a per-float4 copy loop spent ~30 instructions on
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#ifndef SILENT_ABLATE
#define SILENT_ABLATE 0   // experiments only: 1 no output stores, 2 no S5 arithmetic, 4 no S3 arithmetic (bit mask)
#endif
__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, uint32_t bytes)
{
    if (SILENT_ABLATE & 1) return;
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes)
                 : "memory");
}
// ---- TMA tile stores: ONE cp.async.bulk.tensor moves a whole staged tile (kTileStoreRows rows of one image) shared ->
//      global. The output tensor is described as [image][row][tile column][floats of one tile row] and the box is FOUR
//      floats wider than a tile row: the box then reads the staging buffer at its padded row pitch (an odd multiple of
//      16 bytes, what keeps the staging writes conflict-free) and the hardware clips the extra floats, like the rows of a
//      ragged last tile, as out of bounds. (A first version with 16-byte chunks as the inner dimension was 20 % SLOWER
//      than one bulk copy per row: the TMA unit works row by row of the inner dimension.)
struct StoreMaps {
    CUtensorMap orient, line_end, gray;
};
__device__ __forceinline__ void tma_store_tile(const CUtensorMap *map, const void *ssrc, int tile_x, int y, int img)
{
    if (SILENT_ABLATE & 1) return;
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
                 "r"(smem_u32(ssrc)), "r"(0), "r"(tile_x), "r"(y), "r"(img)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// smallest pitch (in float2) >= n whose byte stride is an odd multiple of 16: conflict-free 128-bit row-strided access
constexpr int round_pitch(int n) { return n + ((2 - n % 4) + 4) % 4; }

template <int NQ>
__device__ __forceinline__ void load_cols(const f2 *__restrict__ src, f2 (&v)[2 * NQ])
{
    const float4 *p = reinterpret_cast<const float4 *>(src);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const float4 t = p[q];
        v[2 * q] = make_float2(t.x, t.y);
        v[2 * q + 1] = make_float2(t.z, t.w);
    }
}

// 8 pixels x 3 channels of one lane of the pair as NHWC floats: six 128-bit stores (96 contiguous bytes)
template <int LANE>
__device__ __forceinline__ void store_nhwc8(float *__restrict__ dst, const f2 (&v)[kPX][3], bool vec_ok, int valid_px)
{
    float vals[kPX * 3];
#pragma unroll
    for (int p = 0; p < kPX; ++p)
#pragma unroll
        for (int co = 0; co < 3; ++co) vals[3 * p + co] = LANE ? v[p][co].y : v[p][co].x;
    if (vec_ok) {
#pragma unroll
        for (int q = 0; q < kPX * 3 / 4; ++q)
            reinterpret_cast<float4 *>(dst)[q] = make_float4(vals[4 * q], vals[4 * q + 1], vals[4 * q + 2], vals[4 * q + 3]);
    } else {
#pragma unroll
        for (int e = 0; e < kPX * 3; ++e)
            if (e / 3 < valid_px) dst[e] = vals[e];
    }
}

// Write a staged tile ([2 images][TH][TW*3 (+4 pad)] floats, NHWC) to global memory with coalesced 128-bit stores.
template <int TH, int TW, int NT>
__device__ __forceinline__ void copy_out_tile(const float *__restrict__ stage, float *__restrict__ out, int img0, int img1,
                                              bool has_b, int ty0, int tx0, int h, int w, int tid)
{
    if (!out) return;
    constexpr int QUADS = TW * 3 / 4, PITCH = TW * 3 + 4;
    const int valid_floats = min(TW, w - tx0) * 3;
    const bool vec_ok = (w % 4) == 0;
    for (int i = tid; i < 2 * TH * QUADS; i += NT) {
        const int q = i % QUADS, rest = i / QUADS;
        const int r = rest % TH, lane = rest / TH;
        const int gy = ty0 + r;
        if (gy >= h || (lane == 1 && !has_b) || 4 * q >= valid_floats) continue;
        const float4 v = *reinterpret_cast<const float4 *>(stage + (size_t)(lane * TH + r) * PITCH + 4 * q);
        float *dst = out + (((size_t)(lane ? img1 : img0) * h + gy) * w + tx0) * 3 + 4 * q;
        if (vec_ok && 4 * q + 4 <= valid_floats) {
            *reinterpret_cast<float4 *>(dst) = v;
        } else {
            const float vals[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (4 * q + e < valid_floats) dst[e] = vals[e];
        }
    }
}

// Same tile through the TMA unit: ONE bulk store per staged row (needs 16-byte aligned rows). The `rows` staged rows
// (2 * TH: image A's rows, then image B's) are dealt in contiguous blocks to the warps [warp0, warp0 + nwarps); lane 0 of
// each warp issues its block in a loop whose trip count and addresses are warp-uniform (a per-lane deal made the compiler
// serialise the lanes around the uniform-operand UBLKCP: ~20 instructions per store). row_floats: floats per global row
// of one image (w * channels); tile_floats: floats this tile covers of a row. The caller fences + barriers before; the
// issuing lane commits its group and must bulk_wait_read() before the staging buffer is reused.
template <int TH>
__device__ __forceinline__ bool bulk_rows(const float *__restrict__ stage, int stage_pitch, float *__restrict__ out,
                                          int img0, int img1, bool has_b, int ty0, int h, size_t row_floats, size_t col0,
                                          uint32_t tile_floats, int warp, int warp0, int nwarps, bool leader)
{
    const int wi = warp - warp0;
    if (wi < 0 || wi >= nwarps) return false;
    const int per_warp = (2 * TH + nwarps - 1) / nwarps;
    const int first = wi * per_warp, last = min(first + per_warp, 2 * TH);
    const uint32_t bytes = tile_floats * (uint32_t)sizeof(float);
#pragma unroll
    for (int lane = 0; lane < 2; ++lane) {   // this warp's rows of image A, then of image B: pointers step by one row
        const int r0 = max(first, lane * TH) - lane * TH;
        const int r1 = min(min(last, (lane + 1) * TH) - lane * TH, h - ty0);
        if (r0 >= r1 || (lane == 1 && !has_b)) continue;
        float *dst = out + ((size_t)(lane ? img1 : img0) * h + ty0 + r0) * row_floats + col0;
        const float *src = stage + (size_t)(lane * TH + r0) * stage_pitch;
#pragma unroll 1
        for (int r = r0; r < r1; ++r, dst += row_floats, src += stage_pitch)
            if (leader) bulk_store(dst, src, bytes);
    }
    if (leader) bulk_commit();
    return leader;
}

// the staged rows of a tile ([2][TH][pitch] floats: image A's rows, then image B's) as TMA tile stores of kTileStoreRows rows
constexpr int kTileStoreRows = 16;
template <int TH>
__device__ __forceinline__ void tile_store_images(const CUtensorMap *map, const float *stage, int pitch, int bx, int ty0, int h,
                                                  int img0, int img1, bool has_b)
{
    static_assert(TH % kTileStoreRows == 0, "tiles are whole multiples of the store box");
#pragma unroll
    for (int part = 0; part < TH / kTileStoreRows; ++part) {
        const int y = ty0 + part * kTileStoreRows;
        if (y >= h) break;
        tma_store_tile(map, stage + (size_t)part * kTileStoreRows * pitch, bx, y, img0);
        if (has_b) tma_store_tile(map, stage + (size_t)(TH + part * kTileStoreRows) * pitch, bx, y, img1);
    }
}

__device__ __forceinline__ void store_cols8(f2 *__restrict__ dst, const f2 (&v)[kPX])
{
    float4 *p = reinterpret_cast<float4 *>(dst);
#pragma unroll
    for (int q = 0; q < kPX / 2; ++q) p[q] = make_float4(v[2 * q].x, v[2 * q].y, v[2 * q + 1].x, v[2 * q + 1].y);
}

// ---------------------------------------------------------------------------------------------------------------------
// kernel A: x (pyramid, NHWC) -> rgc -> rgby -> channel sum, written as pairs bsum2[pair][y][x] = (imgA, imgB)
// ---------------------------------------------------------------------------------------------------------------------

struct ParamsA {
    f2 w1[9][3][3];   // rgc  [tap][ci][co] as (w, w)
    f2 w2[9][3][3];   // rgby
    f2 s2s[9];        // S2 mode 2: the shared surround kernel S (centre tap unused)
    f2 s2c[6];        // S2 mode 2: centre taps d0, d1, d2 (ci -> ci), e12 (1 -> 2), e21 (2 -> 1), and the constant 2
    int h, w, n;      // level shape, number of images
    unsigned long long pair_levels;  // image pairing: pair p holds images (a, a + levels), packed by pack_pair_levels()
    int use_tma;      // PAIRED_IN only: load the tile with one TMA box copy
    int prefetch_pairs;   // L2 prefetch distance in image pairs (0: off)
};

// Which two images ride in the float2 lanes of pair p. With pair_levels = 1 these are images (2p, 2p + 1); the
// pipeline pairs the SAME level of two consecutive frames (pair_levels = levels per frame), which lets the pyramid
// kernel share its tap tables between the lanes. Lane B mirrors lane A (and is never stored) when it has no image.
// levels is packed with its reciprocal: pair_levels = levels | (2^32 / levels + 1) << 32 (pack_pair_levels), exact for
// p < 2^32 / levels -- one multiply-high instead of a 20-instruction integer division in every thread
__host__ __device__ inline unsigned long long pack_pair_levels(int levels)
{
    const unsigned long long magic = levels > 1 ? (1ull << 32) / (unsigned)levels + 1 : 0ull;
    return (unsigned)levels | (magic << 32);
}
__device__ __forceinline__ void pair_images(int p, unsigned long long packed, int n, int &a, int &b, bool &has_b)
{
    const int levels = (int)(unsigned)packed;
    const unsigned magic = (unsigned)(packed >> 32);
    const int frame_pair = levels > 1 ? (int)__umulhi((unsigned)p, magic) : p, s = p - frame_pair * levels;
    a = frame_pair * 2 * levels + s;
    b = a + levels;
    has_b = b < n;
    if (!has_b) b = a;
}

// Shared-memory bank groups (16 bytes, 8 per 128-byte line) of S1's accesses: task (row triple rt, channel c, run k) reads
// x at (3 rt + i) * X_PITCH + c * X_PLANE + 8 k (+ 2 q) float2 and writes a at the same expression with the A constants.
// With odd pitches (in 16-byte units) and PLANE strides == 1 (mod 8 units) both map a task to the group
// (s * rt + c + 4 k) mod 8 (s = 3 * pitch units, odd), so ONE deal of tasks to lanes (s1_deal, built on the host) makes
// the eight lanes of almost every quarter-warp hit eight different groups for loads and stores alike. The x planes get
// there with one extra (unused) row in the TMA box, the a planes with 14 float2 of padding.
constexpr int plane_rows_for_unit_stride(int rows, int pitch)
{
    for (int extra = 0; extra < 8; ++extra)
        if (((rows + extra) * (pitch / 2)) % 8 == 1) return rows + extra;
    return rows;
}
constexpr int plane_size_for_unit_stride(int size)
{
    for (int extra = 0; extra < 16; extra += 2)
        if (((size + extra) / 2) % 8 == 1) return size + extra;
    return size;
}

template <int TH, int TW>
struct TileA {
    static constexpr int A_ROWS = TH + 2;                       // a: halo 1 (origin -1)
    static constexpr int A_RUNS = (TW + 2 + kPX - 1) / kPX;     // S1 runs start at column -1
    static constexpr int B_RUNS = TW / kPX;
    static constexpr int X_PITCH = round_pitch(kPX * (A_RUNS - 1) + 10 > TW + 4 ? kPX * (A_RUNS - 1) + 10 : TW + 4);
    static constexpr int A_PITCH = round_pitch(kPX * A_RUNS > kPX * (B_RUNS - 1) + 10 ? kPX * A_RUNS : kPX * (B_RUNS - 1) + 10);
    static constexpr int X_ROWS = plane_rows_for_unit_stride(TH + 4, X_PITCH);   // x: halo 2 (origin -2) + bank padding rows
    static constexpr int X_PLANE = X_ROWS * X_PITCH, A_PLANE = plane_size_for_unit_stride(A_ROWS * A_PITCH);
    static constexpr bool kDealOk = (X_PLANE / 2) % 8 == 1 && (A_PLANE / 2) % 8 == 1 && ((3 * X_PITCH / 2) % 8) == ((3 * A_PITCH / 2) % 8);
    static constexpr int kBankStep = (3 * X_PITCH / 2) % 8;    // bank groups per row triple (odd)
    static constexpr int O_PITCH = round_pitch(TW);   // staged output rows (overlaid on the x planes)
    static_assert(TH * O_PITCH <= 3 * X_PLANE, "output staging must fit in the x planes");
    static constexpr size_t kSmemBytes = (size_t)(3 * X_PLANE + 3 * A_PLANE) * sizeof(f2);
    static_assert(TW % kPX == 0 && TW % 4 == 0, "tile width must be a multiple of the run length");
};

// rgby_3 structure (SURVEY Appendix A): off-centre taps couple only DIFFERENT channels; the centre tap couples each
// channel with itself and channels 1 <-> 2. Anything else is structurally zero (28 of 81 weights).
__host__ __device__ constexpr bool rgby_nonzero(int tap, int ci, int co)
{
    return tap == 4 ? (ci == co || (ci == 1 && co == 2) || (ci == 2 && co == 1)) : (ci != co);
}

// PAIRED_IN: the input is xpair[pair][c][y][x] float2 written by pyramid_pair_kernel (a verbatim 128-bit copy into the
// planes); otherwise it is an NHWC float32 pyramid [n][h][w][3] (stand-alone silent_stack_fused).
// S2 modes: 0 dense; 1 rgby_3 zero pattern (28 structural zeros skipped, 53 FFMA2 per pixel pair); 2 rgby_3 SHARED
// surround (SURVEY Appendix A): off-centre taps couple every channel pair (i != j) through ONE kernel S, doubled for the
// pair (1, 2), and the centre tap carries d_i on the diagonal plus e between channels 1 and 2. Then
//   T_i = S * a_i  (8 taps each),   u0 = d0 a0 + (T1 + T2),   u1 = d1 a1 + (e21 a2 + (2 T2 + T0)),   u2 likewise:
// 24 + 8 FFMA2/FADD2 instead of 53. Part of the canonical FUSED order (oracle/silent_oracle.c: so_rgby_shared).
template <int TH, int TW, int NT, bool S1_DEPTHWISE, int S2_MODE, bool PAIRED_IN>
__global__ void __launch_bounds__(NT) stack_a_kernel(const void *__restrict__ input, const __grid_constant__ ParamsA P,
                                                     const __grid_constant__ CUtensorMap tmap, f2 *__restrict__ bsum2,
                                                     const unsigned char *__restrict__ s1_deal)
{
    using T = TileA<TH, TW>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t tma_bar;
    pdl_enter();
    f2 *sX = reinterpret_cast<f2 *>(smem_raw);   // [3][X_ROWS][X_PITCH]
    f2 *sA = sX + 3 * T::X_PLANE;                // [3][A_ROWS][A_PITCH]
    f2 *sOut = sX;                               // [TH][O_PITCH] channel sums of the tile, valid after the S1 barrier

    const int tid = threadIdx.x;
    const int pair = blockIdx.z;
    const int ty0 = blockIdx.y * TH, tx0 = blockIdx.x * TW;
    const int h = P.h, w = P.w;
    int img0, img1;
    bool has_b;
    pair_images(pair, P.pair_levels, P.n, img0, img1, has_b);

    if (PAIRED_IN && P.use_tma) {
        // ---- load x: the planes are already pair-interleaved; one TMA box [3 planes][X_ROWS][X_PITCH] -------------------
        if (tid == 0) {   // requested before the barrier that publishes the mbarrier to the other threads
            mbar_init(&tma_bar, 1);
            tma_load_box3(sX, &tmap, 2 * (tx0 - 2), ty0 - 2, 3 * pair, &tma_bar, (uint32_t)(3 * T::X_PLANE * sizeof(f2)));
            // the same tile of a pair that is scheduled a few waves from now: pull it from HBM into L2 meanwhile
            const int kPrefetchPairs = P.prefetch_pairs;
            if (kPrefetchPairs > 0 && pair + kPrefetchPairs < (int)gridDim.z)
                asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(&tmap),
                             "r"(2 * (tx0 - 2)), "r"(ty0 - 2), "r"(3 * (pair + kPrefetchPairs))
                             : "memory");
        }
        __syncthreads();
        mbar_wait(&tma_bar, 0);
    } else if (PAIRED_IN) {
        // ---- same tile with plain 128-bit loads (= 2 pixels x 2 frames), zero outside the level ------------------------
        constexpr int QUADS = T::X_PITCH / 2;
        const f2 *src = reinterpret_cast<const f2 *>(input) + (size_t)pair * 3 * h * w;
        const bool vec_ok = (w % 2) == 0;
        for (int i = tid; i < 3 * T::X_ROWS * QUADS; i += NT) {
            const int q = i % QUADS, rest = i / QUADS;
            const int r = rest % T::X_ROWS, c = rest / T::X_ROWS;
            const int gy = ty0 - 2 + r, x0 = tx0 - 2 + 2 * q, x1 = x0 + 1;
            float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (gy >= 0 && gy < h) {
                const f2 *row = src + ((size_t)c * h + gy) * w;
                if (vec_ok && x0 >= 0 && x1 < w) {
                    v = __ldg(reinterpret_cast<const float4 *>(row + x0));
                } else {
                    if (x0 >= 0 && x0 < w) {
                        const f2 a = __ldg(row + x0);
                        v.x = a.x, v.y = a.y;
                    }
                    if (x1 >= 0 && x1 < w) {
                        const f2 b = __ldg(row + x1);
                        v.z = b.x, v.w = b.y;
                    }
                }
            }
            reinterpret_cast<float4 *>(sX + c * T::X_PLANE + r * T::X_PITCH)[q] = v;
        }
    } else {
        // ---- load x: 4-pixel groups (3 x 128-bit) of each image row, scattered into the pair-interleaved planes -------
        const float *pyr = reinterpret_cast<const float *>(input);
        constexpr int GROUPS = (TW + 8) / 4;   // columns tx0-4 .. tx0+TW+4
        float *sXf = reinterpret_cast<float *>(sX);
        const bool vec_ok = (w % 4) == 0;
        for (int i = tid; i < 2 * T::X_ROWS * GROUPS; i += NT) {
            const int g = i % GROUPS, rest = i / GROUPS;
            const int r = rest % T::X_ROWS, lane = rest / T::X_ROWS;
            const int gy = ty0 - 2 + r, gx = tx0 - 4 + 4 * g;
            float vals[12];
            const bool row_ok = gy >= 0 && gy < h;
            const float *src = pyr + (((size_t)(lane ? img1 : img0) * h + (row_ok ? gy : 0)) * w) * 3;
            if (row_ok && vec_ok && gx >= 0 && gx + 4 <= w) {
                const float4 *p4 = reinterpret_cast<const float4 *>(src + (size_t)gx * 3);
                const float4 a = __ldg(p4), b = __ldg(p4 + 1), c = __ldg(p4 + 2);
                vals[0] = a.x, vals[1] = a.y, vals[2] = a.z, vals[3] = a.w, vals[4] = b.x, vals[5] = b.y;
                vals[6] = b.z, vals[7] = b.w, vals[8] = c.x, vals[9] = c.y, vals[10] = c.z, vals[11] = c.w;
            } else {
#pragma unroll
                for (int e = 0; e < 12; ++e) {
                    const int x = gx + e / 3;
                    vals[e] = (row_ok && x >= 0 && x < w) ? __ldg(src + (size_t)x * 3 + e % 3) : 0.0f;
                }
            }
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const int idx = 4 * g - 2 + p;   // column index in the x planes (origin -2)
                if (idx >= 0 && idx < T::X_PITCH) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) sXf[2 * (c * T::X_PLANE + r * T::X_PITCH + idx) + lane] = vals[3 * p + c];
                }
            }
        }
        // columns the loader never touches but the last S1 run over-reads
        constexpr int LOADED = 4 * GROUPS - 2;
        if (LOADED < T::X_PITCH) {
            for (int i = tid; i < 3 * T::X_ROWS * (T::X_PITCH - LOADED); i += NT) {
                const int c = i % (T::X_PITCH - LOADED), rest = i / (T::X_PITCH - LOADED);
                sX[(rest / T::X_ROWS) * T::X_PLANE + (rest % T::X_ROWS) * T::X_PITCH + LOADED + c] = zero2();
            }
        }
    }
    __syncthreads();

    // ---- S1: a = relu(conv3x3(x, rgc))   rows -1..TH, runs of 8 columns from -1               filters/rgc.py:13-16
    if constexpr (S1_DEPTHWISE) {
        // depthwise weights (midget_rgc): a task is ONE channel of THREE output rows x 8 columns. Its five input rows are
        // loaded once (25 LDS.128 for 216 FFMA2, against 45 for a one-row three-channel task: this kernel is bound by
        // shared-memory bandwidth). Input rows are visited in ascending order, so every output still sees its taps in
        // the canonical (ky, kx) order.
        static_assert(T::A_ROWS % 3 == 0, "S1 row triples");
        constexpr int TRIPLES = T::A_ROWS / 3;
        static_assert(3 * TRIPLES * T::A_RUNS <= NT || !T::kDealOk, "the dealt form of S1 is one task per thread");
        for (int t = tid; t < (s1_deal ? NT : 3 * TRIPLES * T::A_RUNS); t += NT) {   // (dealt: any lane may hold a task)
            int rt = t % TRIPLES, c = (t / TRIPLES) % 3, k = t / (3 * TRIPLES);
            if (s1_deal) {   // bank-conflict-free deal of the tasks to the lanes (see TileA)
                const int packed = __ldg(s1_deal + tid);
                if (packed == 255) break;
                rt = packed & 7, c = (packed >> 3) & 3, k = packed >> 5;
            }
            const int r0 = 3 * rt, gx0 = tx0 - 1 + kPX * k;
            f2 wt[9];
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) wt[tap] = P.w1[tap][c][c];
            f2 acc[3][kPX];
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
                for (int p = 0; p < kPX; ++p) acc[j][p] = zero2();
#pragma unroll
            for (int i = 0; i < 5; ++i) {
                f2 v[10];
                load_cols<5>(sX + c * T::X_PLANE + (r0 + i) * T::X_PITCH + kPX * k, v);
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    const int j = i - ky;
                    if (j < 0 || j > 2) continue;
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int p = 0; p < kPX; ++p) acc[j][p] = fma2(wt[ky * 3 + kx], v[p + kx], acc[j][p]);
                }
            }
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int gy = ty0 - 1 + r0 + j;
                const bool row_ok = gy >= 0 && gy < h;
                f2 out[kPX];
                if (row_ok && gx0 >= 0 && gx0 + kPX <= w) {   // the common case: the whole run lies inside the level
#pragma unroll
                    for (int p = 0; p < kPX; ++p) out[p] = relu2_finite(acc[j][p]);
                } else {
#pragma unroll
                    for (int p = 0; p < kPX; ++p) {
                        const int gx = gx0 + p;
                        out[p] = (row_ok && gx >= 0 && gx < w) ? relu2_finite(acc[j][p]) : zero2();   // SAME padding of S2
                    }
                }
                store_cols8(sA + c * T::A_PLANE + (r0 + j) * T::A_PITCH + kPX * k, out);
            }
        }
    } else {
    for (int t = tid; t < T::A_ROWS * T::A_RUNS; t += NT) {
            const int r = t % T::A_ROWS, k = t / T::A_ROWS;
            const int gy = ty0 - 1 + r, gx0 = tx0 - 1 + kPX * k;
            f2 acc[kPX][3];
#pragma unroll
            for (int p = 0; p < kPX; ++p) acc[p][0] = acc[p][1] = acc[p][2] = zero2();
            if (gy >= 0 && gy < h) {
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                    for (int ci = 0; ci < 3; ++ci) {
                        f2 v[10];
                        load_cols<5>(sX + ci * T::X_PLANE + (r + ky) * T::X_PITCH + kPX * k, v);
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                            for (int p = 0; p < kPX; ++p)
#pragma unroll
                                for (int co = 0; co < 3; ++co)
                                    if (!S1_DEPTHWISE || ci == co)
                                        acc[p][co] = fma2(P.w1[ky * 3 + kx][ci][co], v[p + kx], acc[p][co]);
                    }
                }
            }
#pragma unroll
            for (int co = 0; co < 3; ++co) {
                f2 out[kPX];
#pragma unroll
                for (int p = 0; p < kPX; ++p) {
                    const int gx = gx0 + p;
                    out[p] = (gx >= 0 && gx < w) ? relu2_finite(acc[p][co]) : zero2();   // SAME padding of the next conv
                }
                store_cols8(sA + co * T::A_PLANE + r * T::A_PITCH + kPX * k, out);
            }
        }
    }
    __syncthreads();

    // ---- S2: b = relu(conv3x3(a, rgby)); only (b0 + b1) + b2 is needed downstream              filters/rgby.py:11-12
    for (int t = tid; t < TH * T::B_RUNS; t += NT) {
        const int r = t % TH, k = t / TH;
        const int gy = ty0 + r, gx0 = tx0 + kPX * k;
        if (gy >= h || gx0 >= w) continue;
        f2 s[kPX];
        if constexpr (S2_MODE == 2) {
            f2 T[3][kPX], ctr[3][kPX];
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
#pragma unroll
                for (int p = 0; p < kPX; ++p) T[ci][p] = zero2();
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    f2 v[10];
                    load_cols<5>(sA + ci * T::A_PLANE + (r + ky) * T::A_PITCH + kPX * k, v);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        if (ky == 1 && kx == 1) {
#pragma unroll
                            for (int p = 0; p < kPX; ++p) ctr[ci][p] = v[p + 1];
                        } else {
#pragma unroll
                            for (int p = 0; p < kPX; ++p) T[ci][p] = fma2(P.s2s[ky * 3 + kx], v[p + kx], T[ci][p]);
                        }
                    }
                }
            }
#pragma unroll
            for (int p = 0; p < kPX; ++p) {
                const f2 u0 = fma2(P.s2c[0], ctr[0][p], add2(T[1][p], T[2][p]));
                const f2 u1 = fma2(P.s2c[1], ctr[1][p], fma2(P.s2c[4], ctr[2][p], fma2(P.s2c[5], T[2][p], T[0][p])));
                const f2 u2 = fma2(P.s2c[2], ctr[2][p], fma2(P.s2c[3], ctr[1][p], fma2(P.s2c[5], T[1][p], T[0][p])));
                s[p] = add2(add2(relu2_finite(u0), relu2_finite(u1)), relu2_finite(u2));
            }
        } else {
            f2 acc[kPX][3];
#pragma unroll
            for (int p = 0; p < kPX; ++p) acc[p][0] = acc[p][1] = acc[p][2] = zero2();
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int ci = 0; ci < 3; ++ci) {
                    f2 v[10];
                    load_cols<5>(sA + ci * T::A_PLANE + (r + ky) * T::A_PITCH + kPX * k, v);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int p = 0; p < kPX; ++p)
#pragma unroll
                            for (int co = 0; co < 3; ++co)
                                if (S2_MODE == 0 || rgby_nonzero(ky * 3 + kx, ci, co))
                                    acc[p][co] = fma2(P.w2[ky * 3 + kx][ci][co], v[p + kx], acc[p][co]);
                }
            }
#pragma unroll
            for (int p = 0; p < kPX; ++p)
                s[p] = add2(add2(relu2_finite(acc[p][0]), relu2_finite(acc[p][1])), relu2_finite(acc[p][2]));
        }
        // staged in shared memory (over the x planes, dead since S1) and written out row-contiguously below: a run is
        // 64 B of ONE row, so storing it from here would touch 32 different rows per instruction
        store_cols8(sOut + r * T::O_PITCH + kPX * k, s);
    }
    __syncthreads();
    // rows of bsum2 are w + 2 wide: pixel x lives in column x + 1 between two zero columns, so that stack_b's tile
    // origin (x - 5) is an even column = a 16-byte aligned TMA box start (and these stores are 8-byte, not 16-byte)
    constexpr int ROWS_PER_PASS = NT / TW;   // a thread keeps its column and steps down the rows: no index arithmetic
    static_assert(ROWS_PER_PASS >= 1, "stack_a needs at least TW threads");
    const int x = tid % TW, r0 = tid / TW;
    if (r0 < ROWS_PER_PASS && tx0 + x < w) {
        const bool first = tx0 + x == 0, last = tx0 + x == w - 1;
        const int rows = min(TH, h - ty0);
        f2 *dst = bsum2 + ((size_t)pair * h + ty0 + r0) * (w + 2) + tx0 + 1 + x;
        const f2 *src = sOut + r0 * T::O_PITCH + x;
        for (int r = r0; r < rows; r += ROWS_PER_PASS) {
            *dst = *src;
            if (first) dst[-1] = zero2();
            if (last) dst[1] = zero2();
            dst += (size_t)ROWS_PER_PASS * (w + 2);
            src += ROWS_PER_PASS * T::O_PITCH;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// kernel B: bsum2 -> stripe -> regulator -> end filter -> orient, padded_line_end, gray, per-region maxima
// ---------------------------------------------------------------------------------------------------------------------

struct ParamsB {
    f2 w3[9][3];      // stripe [tap][co]  (identical over ci); SYM3: taps 0..4 = the five distinct weights, see S3
    f2 wb[49];        // blur   [tap]      (identical over ci, co)
    f2 w5[9][3][3];   // end    [tap][ci][co]; OWNOTH: [tap][ci][0] = ci -> ci, [tap][ci][1] = ci -> each other channel
    float reg_value, reg_root, clip_max;
    float quick_thr;  // S4 early-out: a channel sum >= quick_thr under ANY blur tap proves m >= 1 (0: early-out disabled)
    int border;
    int h, w, n;
    unsigned long long pair_levels;  // see pair_images() / pack_pair_levels()
    int use_tma;      // load the channel-sum tile with one TMA box copy
    int tma_store;    // outputs leave as TMA tile stores (StoreMaps valid) instead of one bulk copy per staged row
    int prefetch_pairs, pairs;   // quick variant: L2 prefetch distance in image pairs (0: off), number of pairs
    WindowGeom win;   // fused region maxima (stack.h)
};

// LITE: the quick variant of stack_b. The 7x7 blur only matters where it falls below 1, and the early-out test
// (see S4) decides that from sums over the stripe responses the tile computes anyway -- so the quick variant keeps no
// 7x7 halo at all: the stripe stage covers the tile + 1 (what the end filter needs), the blur is never evaluated, and a
// tile in which ANY run fails the test is left untouched and flagged for the full variant (launched right after on the
// flagged tiles only). Less shared memory (68 KB instead of 92 KB for 24-row tiles: 3 CTAs per SM) and a third of the
// halo arithmetic.
template <int TH, int TW, bool LITE>
struct TileB {
    static constexpr int HALO_C = LITE ? 1 : 4;                   // rows of stripe output around the tile
    static constexpr int C_RUNS = (TW + 8) / kPX;                 // S3 runs start at column -4 (TW % 8 == 0)
    static constexpr int D_RUNS = (TW + 2 + kPX - 1) / kPX;       // S4 runs start at column -1
    static constexpr int E_RUNS = TW / kPX;
    static constexpr int CS_ROWS = TH + 2 * HALO_C, B_ROWS = CS_ROWS + 2, CD_ROWS = TH + 2;
    static constexpr int B_PITCH = round_pitch(kPX * (C_RUNS - 1) + 10);                     // origin -5
    static constexpr int CS_PITCH = round_pitch(kPX * (D_RUNS - 1) + 14 > kPX * C_RUNS ? kPX * (D_RUNS - 1) + 14
                                                                                       : kPX * C_RUNS);   // origin -4
    static constexpr int CD_PITCH = round_pitch(kPX * D_RUNS > kPX * (E_RUNS - 1) + 10 ? kPX * D_RUNS
                                                                                       : kPX * (E_RUNS - 1) + 10);  // -1
    static constexpr int B_PLANE = B_ROWS * B_PITCH, CS_PLANE = LITE ? 0 : CS_ROWS * CS_PITCH, CD_PLANE = CD_ROWS * CD_PITCH;
    // output staging (NHWC rows of one tile for both images), overlaid on sB + sCs once S4 is done. The row pitch is
    // an odd multiple of 16 B: the run-per-lane 128-bit stores AND the linear copy-out loads are conflict-free.
    static constexpr int ST_PITCH = TW * 3 + 4;                       // floats per staged row
    static constexpr int STAGE_F2 = 2 * TH * ST_PITCH / 2;            // float2 slots
    static constexpr int G_PITCH = TW + 4;                            // floats per staged gray row (odd multiple of 16 B)
    static constexpr int FRONT_F2 = B_PLANE + CS_PLANE > STAGE_F2 ? B_PLANE + CS_PLANE : STAGE_F2;
    // sums of the stripe channel sum over aligned groups of 4 columns ("quads", origin -4): the S4 early-out reads
    // 7 rows x 3 quads instead of 7 x 14 values. Two spare quads per row (never computed, always "large").
    static constexpr int Q_PITCH = round_pitch(2 * C_RUNS + 2);
    static constexpr int Q_PLANE = CS_ROWS * Q_PITCH;
    // the quad sums die with S4, before the staging buffer is first written: they live in the part of the front region
    // the input planes leave free when there is room (quick variant, 16-row tiles: 44 KB per CTA, 5 CTAs per SM)
    static constexpr bool Q_IN_FRONT = B_PLANE + CS_PLANE + Q_PLANE <= FRONT_F2;
    static constexpr int Q_OFFSET = Q_IN_FRONT ? B_PLANE + CS_PLANE : FRONT_F2 + 3 * CD_PLANE;
    static constexpr size_t kSmemBytes = (size_t)(FRONT_F2 + 3 * CD_PLANE + (Q_IN_FRONT ? 0 : Q_PLANE) + 8) * sizeof(f2) + 64;
    static_assert(TW % kPX == 0, "tile width must be a multiple of the run length");
};

// SYM3: every stripe kernel is symmetric under a 180-degree rotation (K[ky][kx] == K[2-ky][2-kx], true for
// rgb_2d_stripe_tensors): opposite taps are added first, 4 FADD2 + 15 FFMA2 per pixel pair instead of 27 FFMA2.
// OWNOTH: an input channel of the end filter feeds the two OTHER output channels with one and the same 3x3 kernel (true
// for rgb_2d_end_tensors): per input channel one "own" and one "other" chain, 54 FFMA2 + 6 FADD2 instead of 81 FFMA2.
// Both orders are part of the canonical FUSED evaluation order (oracle/silent_oracle.c: so_line_end_stack_fused).
// tile_flag [pairs][tile rows][tile cols] bytes: the LITE variant sets the flag of a tile it could not finish; the
// full variant, given the flags, only works on flagged tiles (null: every tile).
// One tile (bx, by) of image pair bz in a grid of nbx x nby tiles per pair.
template <int TH, int TW, int NT, bool SYM3, bool OWNOTH, bool LITE>
__device__ __forceinline__ void stack_b_tile(const int bx, const int by, const int bz, const int nbx, const int nby,
                                             const f2 *__restrict__ bsum2, const ParamsB &P, const CUtensorMap &tmap,
                                             const StoreMaps &M, float *__restrict__ orient, float *__restrict__ line_end,
                                             float *__restrict__ gray, int *__restrict__ winmax, int *__restrict__ tilemax,
                                             unsigned char *__restrict__ tile_flag, const int tm_split)
{
    using T = TileB<TH, TW, LITE>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t tma_bar;
    const size_t tile_id = ((size_t)bz * nby + by) * nbx + bx;
    f2 *sB = reinterpret_cast<f2 *>(smem_raw);   // [B_ROWS][B_PITCH]       rgby channel sum, origin (-5, -5)
    f2 *sCs = sB + T::B_PLANE;                   // [CS_ROWS][CS_PITCH]     stripe channel sum, origin (-4, -4)
    f2 *sCD = sB + T::FRONT_F2;                  // [3][CD_ROWS][CD_PITCH]  stripe, regulated in place, origin (-1, -1)
    f2 *sQ = sB + T::Q_OFFSET;                   // [CS_ROWS][Q_PITCH]      quad sums of the stripe sum, origin (-4, -4)
    float *sStage = reinterpret_cast<float *>(sB);   // [2][TH][ST_PITCH] NHWC staging, valid after the S4 barrier
    int *sWin = reinterpret_cast<int *>(sB + T::FRONT_F2 + 3 * T::CD_PLANE + (T::Q_IN_FRONT ? 0 : T::Q_PLANE));   // 10 ints
    float *sGray = reinterpret_cast<float *>(sCD);                // [2][TH][G_PITCH] gray staging, valid after the S5 barrier

    const int tid = threadIdx.x;
    const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp index the compiler can see is warp-uniform
    const bool leader = (tid & 31) == 0;
    const int pair = bz;
    const int ty0 = by * TH, tx0 = bx * TW;
    int h = P.h, w = P.w, border = P.border;
    float clip_max = P.clip_max;
    // pin the epilogue's parameters in registers now: re-reading them from the constant bank after the long S5 loop
    // showed up as ~10 % long-scoreboard stalls
    asm volatile("" : "+r"(h), "+r"(w), "+r"(border), "+f"(clip_max), "+l"(orient), "+l"(line_end), "+l"(gray));
    int img0, img1;
    bool has_b;
    pair_images(pair, P.pair_levels, P.n, img0, img1, has_b);

    if (tid < 10) sWin[tid] = 0;

    // ---- load the channel-sum tile (pairs are already interleaved): one TMA box [B_ROWS][B_PITCH], zero outside -------
    if (P.use_tma) {
        if (tid == 0) {   // the copy is requested before the barrier that publishes the mbarrier to the other threads
            mbar_init(&tma_bar, 1);
            tma_load_box3(sB, &tmap, 2 * (tx0 - 4), ty0 - T::HALO_C - 1, pair, &tma_bar, (uint32_t)(T::B_PLANE * sizeof(f2)));
            // the same tile of a pair a few waves ahead: pull it from HBM into L2 meanwhile (like stack_a does)
            if (LITE && P.prefetch_pairs > 0 && pair + P.prefetch_pairs < P.pairs)
                asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(&tmap),
                             "r"(2 * (tx0 - 4)), "r"(ty0 - T::HALO_C - 1), "r"(pair + P.prefetch_pairs)
                             : "memory");
        }
        __syncthreads();
        mbar_wait(&tma_bar, 0);
    } else {
        constexpr int QUADS = T::B_PITCH / 2;
        const f2 *src = bsum2 + (size_t)pair * h * (w + 2) + 1;   // pixel x is stored in column x + 1
        const bool vec_ok = (w % 2) == 0;
        for (int i = tid; i < T::B_ROWS * QUADS; i += NT) {
            const int q = i % QUADS, r = i / QUADS;
            const int gy = ty0 - T::HALO_C - 1 + r;
            float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            const int x0 = tx0 - 5 + 2 * q, x1 = x0 + 1;   // plane column 2q <-> level column tx0 - 5 + 2q
            if (gy >= 0 && gy < h) {
                const f2 *row = src + (size_t)gy * (w + 2);
                if (vec_ok && x0 >= 0 && x1 < w) {   // x0 is odd, so column x0 + 1 is even: 16-byte aligned
                    v = __ldg(reinterpret_cast<const float4 *>(row + x0));
                } else {
                    if (x0 >= 0 && x0 < w) {
                        const f2 a = __ldg(row + x0);
                        v.x = a.x, v.y = a.y;
                    }
                    if (x1 >= 0 && x1 < w) {
                        const f2 b = __ldg(row + x1);
                        v.z = b.x, v.w = b.y;
                    }
                }
            }
            reinterpret_cast<float4 *>(sB + r * T::B_PITCH)[q] = v;
        }
    }
    __syncthreads();
    if (!LITE && P.use_tma && tid == 0)   // every thread has seen the phase flip: a later tile of this CTA starts afresh
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(&tma_bar)) : "memory");

    // ---- S3: c = relu(conv3x3(b, stripe)) on the channel sum; rows -4..TH+3, runs from column -4   orientation.py:24-29
    for (int t = tid; t < T::CS_ROWS * T::C_RUNS; t += NT) {
        const int r = t % T::CS_ROWS, k = t / T::CS_ROWS;
        const int gy = ty0 - T::HALO_C + r, gx0 = tx0 - 4 + kPX * k;
        f2 acc[kPX][3];
#pragma unroll
        for (int p = 0; p < kPX; ++p) acc[p][0] = acc[p][1] = acc[p][2] = zero2();
        if ((SILENT_ABLATE & 4) && gy >= 0 && gy < h) {
#pragma unroll
            for (int p = 0; p < kPX; ++p) acc[p][0] = acc[p][1] = acc[p][2] = sB[(r + 1) * T::B_PITCH + kPX * k + p + 1];
        } else if (gy >= 0 && gy < h) {
            if constexpr (SYM3) {
                // chain over (b[-1,-1] + b[1,1]), (b[-1,0] + b[1,0]), (b[-1,1] + b[1,-1]), (b[0,-1] + b[0,1]), b[0,0]
                {
                    f2 v0[10], v2[10];
                    load_cols<5>(sB + r * T::B_PITCH + kPX * k, v0);
                    load_cols<5>(sB + (r + 2) * T::B_PITCH + kPX * k, v2);
#pragma unroll
                    for (int p = 0; p < kPX; ++p) {
                        const f2 p1 = add2(v0[p], v2[p + 2]), p2 = add2(v0[p + 1], v2[p + 1]), p3 = add2(v0[p + 2], v2[p]);
#pragma unroll
                        for (int co = 0; co < 3; ++co) {
                            acc[p][co] = fma2(P.w3[0][co], p1, acc[p][co]);
                            acc[p][co] = fma2(P.w3[1][co], p2, acc[p][co]);
                            acc[p][co] = fma2(P.w3[2][co], p3, acc[p][co]);
                        }
                    }
                }
                f2 v1[10];
                load_cols<5>(sB + (r + 1) * T::B_PITCH + kPX * k, v1);
#pragma unroll
                for (int p = 0; p < kPX; ++p) {
                    const f2 p4 = add2(v1[p], v1[p + 2]);
#pragma unroll
                    for (int co = 0; co < 3; ++co) {
                        acc[p][co] = fma2(P.w3[3][co], p4, acc[p][co]);
                        acc[p][co] = fma2(P.w3[4][co], v1[p + 1], acc[p][co]);
                    }
                }
            } else {
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    f2 v[10];
                    load_cols<5>(sB + (r + ky) * T::B_PITCH + kPX * k, v);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int p = 0; p < kPX; ++p)
#pragma unroll
                            for (int co = 0; co < 3; ++co) acc[p][co] = fma2(P.w3[ky * 3 + kx][co], v[p + kx], acc[p][co]);
                }
            }
        }
        f2 cs[kPX];
        if (gx0 >= 0 && gx0 + kPX <= w) {   // the common case: the whole run lies inside the level
#pragma unroll
            for (int p = 0; p < kPX; ++p) {
#pragma unroll
                for (int co = 0; co < 3; ++co) acc[p][co] = relu2_finite(acc[p][co]);
                cs[p] = add2(add2(acc[p][0], acc[p][1]), acc[p][2]);
            }
        } else {
#pragma unroll
            for (int p = 0; p < kPX; ++p) {
                const int gx = gx0 + p;
                const bool inside = gx >= 0 && gx < w;
#pragma unroll
                for (int co = 0; co < 3; ++co) acc[p][co] = inside ? relu2_finite(acc[p][co]) : zero2();
                cs[p] = add2(add2(acc[p][0], acc[p][1]), acc[p][2]);
            }
        }
        if constexpr (!LITE) store_cols8(sCs + r * T::CS_PITCH + kPX * k, cs);
        {   // quad sums for the S4 early-out; a quad that lies wholly outside the level can only serve pixels outside
            // the level (whose d is 0 whatever m is): it reads "large" so that it never forces the slow path
            const float big = 1.0e30f;
            f2 q0 = add2(add2(cs[0], cs[1]), add2(cs[2], cs[3]));
            f2 q1 = add2(add2(cs[4], cs[5]), add2(cs[6], cs[7]));
            if (gx0 + 3 < 0 || gx0 >= w) q0 = make_float2(big, big);
            if (gx0 + 7 < 0 || gx0 + 4 >= w) q1 = make_float2(big, big);
            float4 *qd = reinterpret_cast<float4 *>(sQ + r * T::Q_PITCH + 2 * k);
            qd[0] = make_float4(q0.x, q0.y, q1.x, q1.y);
            if (k == T::C_RUNS - 1) qd[1] = make_float4(big, big, big, big);   // the two spare quads of this row
        }
        const int rd = r - (T::HALO_C - 1);   // row in the CD planes (origin -1)
        if (rd >= 0 && rd < T::CD_ROWS) {
            // column -4 + 8k + p sits at idx = 8k - 3 + p of the CD planes (origin -1): odd p starts an aligned pair
            const int base = kPX * k - 3;
#pragma unroll
            for (int co = 0; co < 3; ++co) {
                f2 *row = sCD + co * T::CD_PLANE + rd * T::CD_PITCH;
                if (base >= 0 && base < T::CD_PITCH) row[base] = acc[0][co];
#pragma unroll
                for (int p = 1; p + 1 < kPX; p += 2)
                    if (base + p >= 0 && base + p + 1 < T::CD_PITCH)
                        *reinterpret_cast<float4 *>(row + base + p) =
                            make_float4(acc[p][co].x, acc[p][co].y, acc[p + 1][co].x, acc[p + 1][co].y);
                if (base + kPX - 1 < T::CD_PITCH) row[base + kPX - 1] = acc[kPX - 1][co];
            }
        }
    }
    __syncthreads();

    // ---- S4: d = c * (value / pow(min(blur7x7(csum), 1), root)), in place          gaussian_regulator_tensor.py:34-36
    // Early-out. Every blur weight is positive and every stripe response is >= 0 and finite here, so with u = 2^-24 the
    // 49-step fmaf chain m satisfies m >= (1-u)^49 * sum(w c) >= (1 - 3e-6) * w_min * S for the sum S of ANY subset of
    // the window. A pixel's aligned quad of columns lies inside its window for every window row, so S = the quad sums of
    // the window rows at hand, summed in float (27 roundings: S >= S_float * (1 - 2e-6)). quick_thr is chosen on the host
    // with w_min * quick_thr >= 1.0001, hence S_float >= quick_thr proves m > 1, where the gain is exactly reg_value
    // (gaussian_regulator_tensor.py:35: min(m, 1)) -- bit-identical to evaluating the blur.
    bool task_failed = false;
    for (int t = tid; t < T::CD_ROWS * T::D_RUNS; t += NT) {
        const int r = t % T::CD_ROWS, k = t / T::CD_ROWS;
        const int gy = ty0 - 1 + r, gx0 = tx0 - 1 + kPX * k;
        if (gy < 0 || gy >= h) {   // outside the level: zero padding of the end convolution
            f2 z[kPX];
#pragma unroll
            for (int p = 0; p < kPX; ++p) z[p] = zero2();
#pragma unroll
            for (int co = 0; co < 3; ++co) store_cols8(sCD + co * T::CD_PLANE + r * T::CD_PITCH + kPX * k, z);
            continue;
        }
        if (LITE || P.quick_thr > 0.0f) {
            f2 qa = zero2(), qb = zero2(), qc = zero2();
            const int rs = r + T::HALO_C - 1;   // this row in the stripe-stage rows
#pragma unroll
            for (int dy = -3; dy <= 3; ++dy) {
                if (LITE && (rs + dy < 0 || rs + dy >= T::CS_ROWS)) continue;   // (the full variant has all 7 rows)
                const f2 *qrow = sQ + (rs + dy) * T::Q_PITCH + 2 * k;
                const float4 ab = *reinterpret_cast<const float4 *>(qrow);
                qa = add2(qa, make_float2(ab.x, ab.y));
                qb = add2(qb, make_float2(ab.z, ab.w));
                qc = add2(qc, qrow[2]);
            }
            const float thr = P.quick_thr;
            float lo = fminf(fminf(qa.x, qa.y), fminf(qb.x, qb.y));
            if (kPX * k + 4 <= TW) lo = fminf(lo, fminf(qc.x, qc.y));   // columns 8k+4.. are needed only if inside tile + 1
            if (lo >= thr) {
                if (P.reg_value != 1.0f) {   // d = c * reg_value; with the reference's value of 1 the planes already hold d
                    const f2 gain = make_float2(P.reg_value, P.reg_value);
#pragma unroll
                    for (int co = 0; co < 3; ++co) {
                        float4 *cd = reinterpret_cast<float4 *>(sCD + co * T::CD_PLANE + r * T::CD_PITCH + kPX * k);
#pragma unroll
                        for (int q = 0; q < kPX / 2; ++q) {
                            const float4 tq = cd[q];
                            const f2 a = mul2(make_float2(tq.x, tq.y), gain), b = mul2(make_float2(tq.z, tq.w), gain);
                            cd[q] = make_float4(a.x, a.y, b.x, b.y);
                        }
                    }
                }
                continue;
            }
        }
        if constexpr (LITE) {
            task_failed = true;   // this tile needs the blur itself: left to the full variant
        } else {
            f2 m[kPX];
#pragma unroll
            for (int p = 0; p < kPX; ++p) m[p] = zero2();
#pragma unroll
            for (int ky = 0; ky < 7; ++ky) {
                f2 v[14];
                load_cols<7>(sCs + (r + ky) * T::CS_PITCH + kPX * k, v);
#pragma unroll
                for (int kx = 0; kx < 7; ++kx)
#pragma unroll
                    for (int p = 0; p < kPX; ++p) m[p] = fma2(P.wb[ky * 7 + kx], v[p + kx], m[p]);
            }
            bool all_unity = true;   // m >= 1 everywhere: the gain is exactly reg_value
#pragma unroll
            for (int p = 0; p < kPX; ++p) {
                if (kPX * k + p - 1 > TW) m[p] = make_float2(1.0f, 1.0f);   // over-computed columns of the last run
                all_unity = all_unity && (m[p].x >= 1.0f) && (m[p].y >= 1.0f);
            }
            f2 gain[kPX];
            if (all_unity) {
#pragma unroll
                for (int p = 0; p < kPX; ++p) gain[p] = make_float2(P.reg_value, P.reg_value);
            } else {
#pragma unroll
                for (int p = 0; p < kPX; ++p)   // rare path (flat / dark regions): one out-of-line copy of the pow code
                    gain[p] = make_float2(slow_gain(m[p].x, P.reg_value, P.reg_root), slow_gain(m[p].y, P.reg_value, P.reg_root));
            }
#pragma unroll
            for (int co = 0; co < 3; ++co) {
                f2 *cd = sCD + co * T::CD_PLANE + r * T::CD_PITCH + kPX * k;
                f2 c[kPX];
                {
                    const float4 *p4 = reinterpret_cast<const float4 *>(cd);
#pragma unroll
                    for (int q = 0; q < kPX / 2; ++q) {
                        const float4 tq = p4[q];
                        c[2 * q] = make_float2(tq.x, tq.y);
                        c[2 * q + 1] = make_float2(tq.z, tq.w);
                    }
                }
                if (gx0 >= 0 && gx0 + kPX <= w) {   // (rows outside the level never get here)
#pragma unroll
                    for (int p = 0; p < kPX; ++p) c[p] = mul2(c[p], gain[p]);
                } else {
#pragma unroll
                    for (int p = 0; p < kPX; ++p) {
                        const int gx = gx0 + p;
                        c[p] = (gx >= 0 && gx < w) ? mul2(c[p], gain[p]) : zero2();   // SAME padding of the end conv
                    }
                }
                store_cols8(cd, c);
            }
        }
    }
    if constexpr (LITE) {
        if (__syncthreads_or(task_failed)) {   // nothing of this tile has been written yet
            if (tid == 0) {
                tile_flag[tile_id] = 1;
                atomicAdd(reinterpret_cast<int *>(tile_flag - 4), 1);   // the fix-up pass's "anything to do?" counter
            }
            return;
        }
    } else {
        __syncthreads();
    }

    // ---- orient = d: restage the centre rows of the CD planes in NHWC order (same run-per-lane mapping as S5) and hand
    //      the rows to the TMA unit. When the CTA has at least two warps WITHOUT an S5 task (S5 has the fewest tasks of
    //      the three phases) they do all of this on their own, synchronised by a named barrier, while the S5 warps start
    //      the end filter at once; the copy drains while S5 computes ---------------------------------------------
    const bool bulk_ok = (w % 4) == 0;   // staged rows start and end on 16-byte boundaries of the global tensors
    // TMA tile stores need 128-byte aligned shared-memory sources: every 16-row part of the staging buffers must be one
    constexpr bool kStageTileStore = (kTileStoreRows * T::ST_PITCH * 4) % 128 == 0;
    constexpr bool kGrayTileStore = ((size_t)T::FRONT_F2 * sizeof(f2)) % 128 == 0 && (kTileStoreRows * T::G_PITCH * 4) % 128 == 0;
    const bool tile_store = kStageTileStore && P.tma_store != 0;   // (the host checked w % TW == 0 and built the maps)
    constexpr int kS5Warps = (TH * T::E_RUNS + 31) / 32, kIdleWarps = NT / 32 - kS5Warps;
    constexpr bool kSideRestage = kIdleWarps >= 1;   // (16-row tiles: 3 warps run S5, the 4th restages and stores orient)
    constexpr int kRestageFirst = kSideRestage ? 32 * kS5Warps : 0, kRestageThreads = kSideRestage ? 32 * kIdleWarps : NT;
    bool issued_orient = false, issued_line_end = false;
    if (orient && tid >= kRestageFirst) {
        for (int t = tid - kRestageFirst; t < TH * T::E_RUNS; t += kRestageThreads) {
            const int r = t % TH, k = t / TH;
            f2 d[kPX][3];
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
                f2 v[10];
                load_cols<5>(sCD + ci * T::CD_PLANE + (r + 1) * T::CD_PITCH + kPX * k, v);
#pragma unroll
                for (int p = 0; p < kPX; ++p) d[p][ci] = v[p + 1];
            }
            store_nhwc8<0>(sStage + (size_t)r * T::ST_PITCH + 3 * kPX * k, d, true, kPX);
            store_nhwc8<1>(sStage + (size_t)(TH + r) * T::ST_PITCH + 3 * kPX * k, d, true, kPX);
        }
        fence_async_smem();
        if (kSideRestage) {
            asm volatile("bar.sync 1, %0;" ::"n"(kRestageThreads) : "memory");   // only the restaging warps
        } else {
            __syncthreads();
        }
        if (tile_store) {
            if (tid == kRestageFirst) {   // two tile stores per 16 rows (one per image) instead of a bulk copy per row
                tile_store_images<TH>(&M.orient, sStage, T::ST_PITCH, bx, ty0, h, img0, img1, has_b);
                bulk_commit();
                issued_orient = true;
            }
        } else if (bulk_ok) {
            issued_orient = bulk_rows<TH>(sStage, T::ST_PITCH, orient, img0, img1, has_b, ty0, h, (size_t)w * 3, (size_t)tx0 * 3,
                                          (uint32_t)(min(TW, w - tx0) * 3), warp_u, kRestageFirst / 32, kRestageThreads / 32,
                                          leader);
        } else {
            copy_out_tile<TH, TW, kRestageThreads>(sStage, orient, img0, img1, has_b, ty0, tx0, h, w, tid - kRestageFirst);
        }
    }

    // ---- S5-S7: e = clip(relu(conv3x3(d, end))); p = mask * e; g = mean(p)                 recognition_testing.py:73-77
    static_assert(NT >= TH * T::E_RUNS, "one S5 task per thread");
    const int r5 = tid % TH, k5 = tid / TH;
    const int gy = ty0 + r5, gx0 = tx0 + kPX * k5;
    const bool active = tid < TH * T::E_RUNS && gy < h && gx0 < w;
    f2 acc[kPX][3];
    if ((SILENT_ABLATE & 2) && active) {
#pragma unroll
        for (int p = 0; p < kPX; ++p) acc[p][0] = acc[p][1] = acc[p][2] = sCD[(r5 + p) * T::CD_PITCH + kPX * k5];
    } else if (active) {
        if constexpr (OWNOTH) {
            // per input channel: own = its kernel into its own output channel, oth = the ONE kernel it feeds both other
            // output channels with; e_co = (t_0 + t_1) + t_2 with t_ci = (ci == co ? own_ci : oth_ci)
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
                f2 own[kPX], oth[kPX];
#pragma unroll
                for (int p = 0; p < kPX; ++p) own[p] = oth[p] = zero2();
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    f2 v[10];
                    load_cols<5>(sCD + ci * T::CD_PLANE + (r5 + ky) * T::CD_PITCH + kPX * k5, v);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int p = 0; p < kPX; ++p) {
                            own[p] = fma2(P.w5[ky * 3 + kx][ci][0], v[p + kx], own[p]);
                            oth[p] = fma2(P.w5[ky * 3 + kx][ci][1], v[p + kx], oth[p]);
                        }
                }
#pragma unroll
                for (int p = 0; p < kPX; ++p)
#pragma unroll
                    for (int co = 0; co < 3; ++co) {
                        const f2 t = co == ci ? own[p] : oth[p];
                        acc[p][co] = ci == 0 ? t : add2(acc[p][co], t);
                    }
            }
        } else {
#pragma unroll
            for (int p = 0; p < kPX; ++p) acc[p][0] = acc[p][1] = acc[p][2] = zero2();
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int ci = 0; ci < 3; ++ci) {
                    f2 v[10];
                    load_cols<5>(sCD + ci * T::CD_PLANE + (r5 + ky) * T::CD_PITCH + kPX * k5, v);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int p = 0; p < kPX; ++p)
#pragma unroll
                            for (int co = 0; co < 3; ++co)
                                acc[p][co] = fma2(P.w5[ky * 3 + kx][ci][co], v[p + kx], acc[p][co]);
                }
            }
        }
    }
    // the staging buffer is free again once the orient rows have been read out
    // every S5 warp is done reading the CD planes (the gray staging below overwrites them), and the orient rows have left
    // the staging buffer
    if (issued_orient) bulk_wait_read();
    __syncthreads();
    int best0 = 0, best1 = 0;
    if (active) {
        const bool row_in = gy >= border && gy < h - border;
        const bool all_keep = row_in && gx0 >= border && gx0 + kPX <= w - border;   // run clear of the border mask
        const float third = __fdiv_rn(1.0f, 3.0f);
        f2 g[kPX];
#pragma unroll
        for (int p = 0; p < kPX; ++p)
#pragma unroll
            for (int co = 0; co < 3; ++co)
                acc[p][co] = make_float2(clip_nan(relu_nan(acc[p][co].x), clip_max), clip_nan(relu_nan(acc[p][co].y), clip_max));
        if (!all_keep) {
#pragma unroll
            for (int p = 0; p < kPX; ++p) {
                const int gx = gx0 + p;
                if (row_in && gx >= border && gx < w - border) continue;
#pragma unroll
                for (int co = 0; co < 3; ++co) {   // pad_inwards multiplies by 0: NaN stays NaN
                    const float a = acc[p][co].x, b = acc[p][co].y;
                    acc[p][co] = make_float2(a != a ? a : 0.0f * a, b != b ? b : 0.0f * b);
                }
            }
        }
#pragma unroll
        for (int p = 0; p < kPX; ++p)
            g[p] = mul2(add2(add2(acc[p][0], acc[p][1]), acc[p][2]), make_float2(third, third));
        const size_t pix_a = ((size_t)img0 * h + gy) * w + gx0, pix_b = ((size_t)img1 * h + gy) * w + gx0;
        // stage padded_line_end in NHWC order: 96 contiguous bytes per image and run; written out row by row below
        store_nhwc8<0>(sStage + (size_t)r5 * T::ST_PITCH + 3 * kPX * k5, acc, true, kPX);
        store_nhwc8<1>(sStage + (size_t)(TH + r5) * T::ST_PITCH + 3 * kPX * k5, acc, true, kPX);
        if (gray) {
            if (bulk_ok) {   // staged over the (now dead) CD planes: rows of TW floats, written by bulk stores below
                float4 *ga = reinterpret_cast<float4 *>(sGray + (size_t)r5 * T::G_PITCH + kPX * k5);
                float4 *gb = reinterpret_cast<float4 *>(sGray + (size_t)(TH + r5) * T::G_PITCH + kPX * k5);
                ga[0] = make_float4(g[0].x, g[1].x, g[2].x, g[3].x);
                ga[1] = make_float4(g[4].x, g[5].x, g[6].x, g[7].x);
                gb[0] = make_float4(g[0].y, g[1].y, g[2].y, g[3].y);
                gb[1] = make_float4(g[4].y, g[5].y, g[6].y, g[7].y);
            } else {
#pragma unroll
                for (int lane = 0; lane < 2; ++lane) {
                    if (lane == 1 && !has_b) break;
                    float *dst = gray + (lane ? pix_b : pix_a);
#pragma unroll
                    for (int p = 0; p < kPX; ++p)
                        if (gx0 + p < w) dst[p] = lane ? g[p].y : g[p].x;
                }
            }
        }
        // run maximum per image as ordered ints: values are >= 0, NaN maps to 0x7fc00000 which beats everything
#pragma unroll
        for (int p = 0; p < kPX; ++p) {
            if (gx0 + p < w) {
                const int a = g[p].x != g[p].x ? 0x7fc00000 : __float_as_int(g[p].x);
                const int b = g[p].y != g[p].y ? 0x7fc00000 : __float_as_int(g[p].y);
                best0 = max(best0, a);
                best1 = max(best1, b);
            }
        }
    }
    if (tilemax && tid < (TH * T::E_RUNS + 31) / 32 * 32) {   // maximum of gray over the whole tile (emit skips most tiles)
        const int m0 = __reduce_max_sync(0xffffffffu, active ? best0 : 0);
        const int m1 = __reduce_max_sync(0xffffffffu, active ? best1 : 0);
        if ((tid & 31) == 0) {
            if (m0) atomicMax(&sWin[8], m0);
            if (m1) atomicMax(&sWin[9], m1);
        }
    }
    if (P.win.count && tid < (TH * T::E_RUNS + 31) / 32 * 32) {   // whole warps: the reduction needs every lane
        // lanes of a warp hold consecutive rows of one run: reduce per window across the warp (0 is the identity and
        // what inactive lanes carry), then one shared atomic per warp instead of one 32-way serialised atomic
        const int nwy = P.win.count / P.win.ow;
        for (int i = 0; i < nwy; ++i) {
            const bool row_in_win = active && gy >= P.win.y0[i] && gy < P.win.y1[i];
            for (int j = 0; j < P.win.ow; ++j) {
                const bool in_win = row_in_win && gx0 >= P.win.x0[j] && gx0 < P.win.x1[j];   // bounds: multiples of 8
                const int m0 = __reduce_max_sync(0xffffffffu, in_win ? best0 : 0);
                const int m1 = __reduce_max_sync(0xffffffffu, in_win ? best1 : 0);
                if ((tid & 31) == 0) {
                    if (m0) atomicMax(&sWin[i * P.win.ow + j], m0);
                    if (m1) atomicMax(&sWin[4 + i * P.win.ow + j], m1);
                }
            }
        }
    }
    // ---- copy-out: staged rows -> global NHWC, one bulk store per row ---------------------------------------------------
    fence_async_smem();
    __syncthreads();
    if (gray && tile_store && kGrayTileStore) {
        if (tid == 32) {
            tile_store_images<TH>(&M.gray, sGray, T::G_PITCH, bx, ty0, h, img0, img1, has_b);
            bulk_commit();
            issued_line_end = true;
        }
    } else if (gray && bulk_ok)   // 2 * TH rows of TW floats, dealt like the line_end rows
        issued_line_end |= bulk_rows<TH>(sGray, T::G_PITCH, gray, img0, img1, has_b, ty0, h, (size_t)w, (size_t)tx0,
                                         (uint32_t)min(TW, w - tx0), warp_u, 0, NT / 32, leader);
    if (line_end) {
        if (tile_store) {
            if (tid == 0) {
                tile_store_images<TH>(&M.line_end, sStage, T::ST_PITCH, bx, ty0, h, img0, img1, has_b);
                bulk_commit();
                issued_line_end = true;
            }
        } else if (bulk_ok) {
            issued_line_end |= bulk_rows<TH>(sStage, T::ST_PITCH, line_end, img0, img1, has_b, ty0, h, (size_t)w * 3,
                                             (size_t)tx0 * 3, (uint32_t)(min(TW, w - tx0) * 3), warp_u, 0, NT / 32, leader);
        } else {
            copy_out_tile<TH, TW, NT>(sStage, line_end, img0, img1, has_b, ty0, tx0, h, w, tid);
        }
    }
    if (P.win.count) {
        if (tid < 8) {
            const int lane = tid >> 2, win = tid & 3;
            const int v = sWin[tid];
            if (win < P.win.count && (lane == 0 || has_b) && v != 0)
                atomicMax(&winmax[(size_t)(lane ? img1 : img0) * P.win.count + win], v);
        }
    }
    if (tilemax && tid >= 32 && tid < 34) {   // [image][tile row][tile column], ordered-int encoding like winmax
        const int lane = tid - 32;
        // the emit's grid has rows of TH / tm_split: a taller tile (one-wave launches) reports its maximum for each of them
        if (lane == 0 || has_b)
            for (int part = 0; part < tm_split; ++part)
                tilemax[((size_t)(lane ? img1 : img0) * nby * tm_split + by * tm_split + part) * nbx + bx] = sWin[8 + lane];
    }
    if (issued_line_end) bulk_wait_read();   // the CTA's shared memory must outlive the reads
}

// tile_flag [pairs][tile rows][tile cols] bytes. The LITE variant (one CTA per tile) sets the flag of a tile it could not
// finish. The full variant without flags works on every tile (one CTA per tile); WITH flags it is the fix-up pass: a
// small 1-D grid of CTAs walks the tile list and redoes the flagged tiles (none on textured input: the pass then costs
// a few microseconds instead of a full grid of early exits).
template <int TH, int TW, int NT, bool SYM3, bool OWNOTH, bool LITE>
__global__ void __launch_bounds__(NT, LITE ? (TH <= 16 ? 5 : 3) : 2)
stack_b_kernel(const f2 *__restrict__ bsum2, const __grid_constant__ ParamsB P, const __grid_constant__ CUtensorMap tmap,
               const __grid_constant__ StoreMaps M, float *__restrict__ orient, float *__restrict__ line_end, float *__restrict__ gray, int *__restrict__ winmax,
               int *__restrict__ tilemax, unsigned char *__restrict__ tile_flag, int nbx, int nby, int pairs, int tm_split)
{
    pdl_enter();
    if (!LITE && tile_flag) {
        // tile_flag[-4 .. -1] counts the tiles the quick pass flagged: on textured input it is 0 and the pass ends here
        if (*reinterpret_cast<const volatile int *>(tile_flag - 4) == 0) return;
        const int per_pair = nbx * nby, total = per_pair * pairs;
        __shared__ unsigned s_mask;
        bool again = false;
        // this CTA's tiles are t = blockIdx.x + j * gridDim.x; 32 of them are tested at a time (one per lane of warp 0)
        for (int j0 = 0; blockIdx.x + (long long)j0 * gridDim.x < total; j0 += 32) {
            if (again) __syncthreads();   // s_mask of the previous batch has been consumed
            if (threadIdx.x < 32) {
                const long long t = blockIdx.x + (long long)(j0 + threadIdx.x) * gridDim.x;
                bool flagged = false;
                if (t < total) {
                    const int bz = (int)(t / per_pair), rest = (int)(t - (long long)bz * per_pair);
                    // the flags live on the quick pass's grid (tiles of TH / tm_split rows): a taller fix-up tile is redone
                    // when any of the quick tiles it covers is flagged (the others just get the same bits written again)
                    for (int part = 0; part < tm_split; ++part)
                        flagged |= tile_flag[((size_t)bz * nby * tm_split + (rest / nbx) * tm_split + part) * nbx + rest % nbx] != 0;
                }
                const unsigned mask = __ballot_sync(0xffffffffu, flagged);
                if (threadIdx.x == 0) s_mask = mask;
            }
            __syncthreads();
            unsigned mask = s_mask;
            while (mask) {
                const int bit = __ffs(mask) - 1;
                mask &= mask - 1;
                const int t = blockIdx.x + (j0 + bit) * gridDim.x;
                const int bz = t / per_pair, rest = t - bz * per_pair;
                if (again) __syncthreads();   // every thread is done with the previous tile's shared memory
                again = true;
                stack_b_tile<TH, TW, NT, SYM3, OWNOTH, LITE>(rest % nbx, rest / nbx, bz, nbx, nby, bsum2, P, tmap, M, orient,
                                                             line_end, gray, winmax, tilemax, tile_flag, tm_split);
            }
            again = true;
        }
    } else {
        stack_b_tile<TH, TW, NT, SYM3, OWNOTH, LITE>(blockIdx.x, blockIdx.y, blockIdx.z, gridDim.x, gridDim.y, bsum2, P, tmap,
                                                     M, orient, line_end, gray, winmax, tilemax, tile_flag, tm_split);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// kernel BANK: stack_b for an orientation BANK of NB = 4, 8, 12 or 16 orientations (BASELINE config C4: 8 orientations)
// through the reference's per-vector generators, stripe_tensor.py:21-70 / oriented_end_detector.py:13-55 /
// gaussian_blur.py:13-54:
//   bsum2 -> stripe bank 1 -> NB (identical over the rgby channels, so it runs on the channel sum like S3) -> regulator
//   (one 7x7 blur of the NB-channel sum, all NB x NB slices identical) -> end bank, DEPTHWISE (orientation k only feeds
//   orientation k) + relu + clip -> border mask -> mean. Outputs orient / padded_line_end [n, h, w, NB], gray [n, h, w].
// Same building blocks as stack_b_kernel (frame pairs in float2 lanes, lanes walk rows over odd-multiple-of-16-byte
// pitches, staged NHWC rows leaving through bulk stores, the quad-sum early-out of the blur) with runs of 4 pixels, so
// that 4 orientations x 4 pixels of results fit in registers at a time. Chains run in the canonical (ky, kx) order of
// the per-operator kernels: skipping the end bank's exact-zero cross-orientation weights is a no-op for finite data.
// Orientations are handled in groups of 4 (one float4 per pixel in the NHWC restage, NB / 4 groups in S5), hence NB % 4 == 0.
// ---------------------------------------------------------------------------------------------------------------------

constexpr int kRun = 4;  // pixels per run

template <int NB>
struct ParamsBank {
    static_assert(NB % 4 == 0, "orientations are processed in groups of four");
    f2 w3[9][NB];   // stripe [tap][orientation]
    f2 wb[49];       // blur
    f2 w5[9][NB];   // end, depthwise [tap][orientation]
    float reg_value, reg_root, clip_max, quick_thr;
    int border, h, w, n;
    unsigned long long pair_levels;   // pack_pair_levels()
    int tma_store;   // orient / line_end leave as TMA tile stores (StoreMaps valid)
};

template <int NB, int TH, int TW>
struct TileBank {
    static constexpr int C_RUNS = (TW + 9 + kRun - 1) / kRun;   // stripe runs start at column -5 (need -4 .. TW + 3)
    static constexpr int D_RUNS = (TW + 2 + kRun - 1) / kRun;   // regulator runs start at column -1
    static constexpr int E_RUNS = TW / kRun;
    static constexpr int B_ROWS = TH + 10, CS_ROWS = TH + 8, CD_ROWS = TH + 2;   // row origins -5, -4, -1
    static constexpr int B_PITCH = round_pitch(kRun * (C_RUNS - 1) + 6);          // column origin -6
    static constexpr int CS_PITCH = round_pitch(kRun * (D_RUNS - 1) + 12 > kRun * C_RUNS ? kRun * (D_RUNS - 1) + 12
                                                                                         : kRun * C_RUNS);   // origin -5
    static constexpr int CD_PITCH = round_pitch(kRun * D_RUNS > kRun * (E_RUNS - 1) + 6 ? kRun * D_RUNS
                                                                                       : kRun * (E_RUNS - 1) + 6);   // -1
    static constexpr int Q_PITCH = C_RUNS | 1;                                     // one quad sum per stripe run
    static constexpr int B_PLANE = B_ROWS * B_PITCH, CS_PLANE = CS_ROWS * CS_PITCH, CD_PLANE = CD_ROWS * CD_PITCH;
    static constexpr int ST_PITCH = TW * NB + 4;                    // floats per staged NHWC row (odd multiple of 16 B)
    static constexpr int STAGE_F2 = 2 * TH * ST_PITCH / 2;
    static constexpr int FRONT_F2 = B_PLANE + CS_PLANE > STAGE_F2 ? B_PLANE + CS_PLANE : STAGE_F2;
    static constexpr size_t kSmemBytes = (size_t)(FRONT_F2 + NB * CD_PLANE + CS_ROWS * Q_PITCH) * sizeof(f2) + 64;
    static_assert(TW % kRun == 0 && TW % 4 == 0, "tile width must be a multiple of the run length");
};

__device__ __forceinline__ void store_cols4(f2 *__restrict__ dst, const f2 (&v)[kRun])
{
    float4 *p = reinterpret_cast<float4 *>(dst);
    p[0] = make_float4(v[0].x, v[0].y, v[1].x, v[1].y);
    p[1] = make_float4(v[2].x, v[2].y, v[3].x, v[3].y);
}

template <int NB, int TH, int TW, int NT>
__global__ void __launch_bounds__(NT, 2) stack_bank_kernel(const f2 *__restrict__ bsum2, const __grid_constant__ ParamsBank<NB> P,
                                                           const __grid_constant__ StoreMaps M, float *__restrict__ orient, float *__restrict__ line_end,
                                                           float *__restrict__ gray)
{
    using T = TileBank<NB, TH, TW>;
    // loops over the orientations, unrolled whole up to 8 orientations. Wider banks walk them in chunks (4 orientations
    // in S3 / S4, one group of 4 in the restage and S5) that are not unrolled into each other: unrolled whole, the
    // compiler hoists every orientation's weights into registers and spills.
    constexpr int kChunkO = NB <= 8 ? NB : 4, kChunkG = NB <= 8 ? NB / 4 : 1;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    pdl_enter();
    f2 *sB = reinterpret_cast<f2 *>(smem_raw);   // [B_ROWS][B_PITCH]      rgby channel sum, origin (-5, -6)
    f2 *sCs = sB + T::B_PLANE;                   // [CS_ROWS][CS_PITCH]    sum of the stripe bank, origin (-4, -5)
    f2 *sCD = sB + T::FRONT_F2;                  // [NB][CD_ROWS][CD_PITCH] stripe bank, regulated in place, origin (-1, -1)
    f2 *sQ = sCD + NB * T::CD_PLANE;            // [CS_ROWS][Q_PITCH]     quad sums of sCs
    float *sStage = reinterpret_cast<float *>(sB);   // [2][TH][ST_PITCH] NHWC staging, valid after the S4 barrier

    const int tid = threadIdx.x;
    const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const bool leader = (tid & 31) == 0;
    const int pair = blockIdx.z, ty0 = blockIdx.y * TH, tx0 = blockIdx.x * TW;
    const int h = P.h, w = P.w;
    int img0, img1;
    bool has_b;
    pair_images(pair, P.pair_levels, P.n, img0, img1, has_b);

    // ---- channel-sum tile (pixel x lives in column x + 1 of the (w + 2)-wide rows), zero outside the level -----------
    {
        const f2 *src = bsum2 + (size_t)pair * h * (w + 2) + 1;
        for (int i = tid; i < T::B_ROWS * T::B_PITCH; i += NT) {
            const int c = i % T::B_PITCH, r = i / T::B_PITCH;
            const int gy = ty0 - 5 + r, gx = tx0 - 6 + c;
            sB[i] = (gy >= 0 && gy < h && gx >= 0 && gx < w) ? __ldg(src + (size_t)gy * (w + 2) + gx) : zero2();
        }
    }
    __syncthreads();

    // ---- S3: stripe bank on the channel sum; rows -4 .. TH+3, runs of 4 columns from -5 ------------------------------
    for (int t = tid; t < T::CS_ROWS * T::C_RUNS; t += NT) {
        const int r = t % T::CS_ROWS, k = t / T::CS_ROWS;
        const int gy = ty0 - 4 + r, gx0 = tx0 - 5 + kRun * k;
        const bool row_ok = gy >= 0 && gy < h;
        f2 v[3][6];
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) load_cols<3>(sB + (r + ky) * T::B_PITCH + kRun * k, v[ky]);
        f2 cs[kRun];
#pragma unroll
        for (int p = 0; p < kRun; ++p) cs[p] = zero2();
        const int rd = r - 3;   // row in the CD planes
#pragma unroll 1
        for (int o0 = 0; o0 < NB; o0 += kChunkO)
#pragma unroll
        for (int o = o0; o < o0 + kChunkO; ++o) {
            f2 acc[kRun];
#pragma unroll
            for (int p = 0; p < kRun; ++p) acc[p] = zero2();
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                    for (int p = 0; p < kRun; ++p) acc[p] = fma2(P.w3[ky * 3 + kx][o], v[ky][p + kx], acc[p]);
#pragma unroll
            for (int p = 0; p < kRun; ++p) {
                const int gx = gx0 + p;
                acc[p] = (row_ok && gx >= 0 && gx < w) ? relu2_finite(acc[p]) : zero2();   // SAME padding downstream
                cs[p] = o == 0 ? acc[p] : add2(cs[p], acc[p]);                             // ((c0 + c1) + c2) + ...
            }
            if (rd >= 0 && rd < T::CD_ROWS && k >= 1 && kRun * (k - 1) + kRun <= T::CD_PITCH)
                store_cols4(sCD + o * T::CD_PLANE + rd * T::CD_PITCH + kRun * (k - 1), acc);
        }
        store_cols4(sCs + r * T::CS_PITCH + kRun * k, cs);
        f2 q = add2(add2(cs[0], cs[1]), add2(cs[2], cs[3]));
        if (gx0 + kRun - 1 < 0 || gx0 >= w) q = make_float2(1.0e30f, 1.0e30f);   // wholly outside: never forces the blur
        sQ[r * T::Q_PITCH + k] = q;
    }
    __syncthreads();

    // ---- S4: regulator, in place; rows -1 .. TH, runs of 4 from column -1 (quad of run j = stripe run j + 1) -----------
    for (int t = tid; t < T::CD_ROWS * T::D_RUNS; t += NT) {
        const int r = t % T::CD_ROWS, j = t / T::CD_ROWS;
        const int gy = ty0 - 1 + r, gx0 = tx0 - 1 + kRun * j;
        if (gy < 0 || gy >= h) continue;   // the planes already hold zeros there
        bool unity = false;
        if (P.quick_thr > 0.0f) {   // see stack_b_kernel S4: quad sums of the 7 window rows prove m >= 1
            f2 qs = zero2();
#pragma unroll
            for (int ky = 0; ky < 7; ++ky) qs = add2(qs, sQ[(r + ky) * T::Q_PITCH + j + 1]);
            unity = fminf(qs.x, qs.y) >= P.quick_thr;
        }
        f2 gain[kRun];
        if (unity) {
            if (P.reg_value == 1.0f) continue;
#pragma unroll
            for (int p = 0; p < kRun; ++p) gain[p] = make_float2(P.reg_value, P.reg_value);
        } else {
            f2 m[kRun];
#pragma unroll
            for (int p = 0; p < kRun; ++p) m[p] = zero2();
#pragma unroll
            for (int ky = 0; ky < 7; ++ky) {
                f2 cv[12];   // Cs columns 4j .. 4j+11 (level columns gx0 - 4 .. gx0 + 7); pixel p uses 1 + p .. 7 + p
                load_cols<6>(sCs + (r + ky) * T::CS_PITCH + kRun * j, cv);
#pragma unroll
                for (int kx = 0; kx < 7; ++kx)
#pragma unroll
                    for (int p = 0; p < kRun; ++p) m[p] = fma2(P.wb[ky * 7 + kx], cv[1 + p + kx], m[p]);
            }
#pragma unroll
            for (int p = 0; p < kRun; ++p)
                gain[p] = make_float2(slow_gain(m[p].x, P.reg_value, P.reg_root), slow_gain(m[p].y, P.reg_value, P.reg_root));
        }
#pragma unroll 1
        for (int o0 = 0; o0 < NB; o0 += kChunkO)
#pragma unroll
        for (int o = o0; o < o0 + kChunkO; ++o) {
            f2 *cd = sCD + o * T::CD_PLANE + r * T::CD_PITCH + kRun * j;
            f2 c[4];
            load_cols<2>(cd, c);
#pragma unroll
            for (int p = 0; p < kRun; ++p) {
                const int gx = gx0 + p;
                c[p] = (gx >= 0 && gx < w) ? mul2(c[p], gain[p]) : zero2();
            }
            store_cols4(cd, c);
        }
    }
    __syncthreads();

    // ---- orient = d: centre rows of the planes, restaged NHWC (4 orientations = one 128-bit chunk per pixel and image) --
    const bool bulk_ok = (w % 4) == 0;
    constexpr bool kStageTileStore = (kTileStoreRows * T::ST_PITCH * 4) % 128 == 0;
    const bool tile_store = kStageTileStore && P.tma_store != 0;
    bool issued = false;
    if (orient) {
        for (int t = tid; t < TH * T::E_RUNS; t += NT) {
            const int r = t % TH, k = t / TH;
#pragma unroll 1
            for (int g0 = 0; g0 < NB / 4; g0 += kChunkG)
#pragma unroll
            for (int g = g0; g < g0 + kChunkG; ++g) {
                f2 d[4][6];
#pragma unroll
                for (int oo = 0; oo < 4; ++oo) load_cols<3>(sCD + (4 * g + oo) * T::CD_PLANE + (r + 1) * T::CD_PITCH + kRun * k, d[oo]);
#pragma unroll
                for (int p = 0; p < kRun; ++p) {
                    float *a = sStage + (size_t)r * T::ST_PITCH + (kRun * k + p) * NB + 4 * g;
                    float *b = sStage + (size_t)(TH + r) * T::ST_PITCH + (kRun * k + p) * NB + 4 * g;
                    *reinterpret_cast<float4 *>(a) = make_float4(d[0][p + 1].x, d[1][p + 1].x, d[2][p + 1].x, d[3][p + 1].x);
                    *reinterpret_cast<float4 *>(b) = make_float4(d[0][p + 1].y, d[1][p + 1].y, d[2][p + 1].y, d[3][p + 1].y);
                }
            }
        }
        fence_async_smem();
        __syncthreads();
        if (tile_store) {
            if (tid == 0) {
                tile_store_images<TH>(&M.orient, sStage, T::ST_PITCH, blockIdx.x, ty0, h, img0, img1, has_b);
                bulk_commit();
                issued = true;
            }
        } else if (bulk_ok) {
            issued = bulk_rows<TH>(sStage, T::ST_PITCH, orient, img0, img1, has_b, ty0, h, (size_t)w * NB, (size_t)tx0 * NB,
                                   (uint32_t)(min(TW, w - tx0) * NB), warp_u, 0, NT / 32, leader);
        } else {
            for (int i = tid; i < 2 * TH * TW * NB; i += NT) {
                const int e = i % (TW * NB), row = i / (TW * NB), lane = row / TH, gy = ty0 + row % TH;
                if (gy < h && tx0 + e / NB < w && (lane == 0 || has_b))
                    orient[(((size_t)(lane ? img1 : img0) * h + gy) * w + tx0) * NB + e] = sStage[(size_t)row * T::ST_PITCH + e];
            }
        }
        if (issued) bulk_wait_read();
        __syncthreads();   // the staging buffer is free again
    }

    // ---- S5-S7: depthwise end bank + relu + clip, border mask, mean over the orientations --------------------------------
    const float inv_nb = __fdiv_rn(1.0f, (float)NB);
    for (int t = tid; t < TH * T::E_RUNS; t += NT) {
        const int r = t % TH, k = t / TH;
        const int gy = ty0 + r, gx0 = tx0 + kRun * k;
        const bool row_in = gy >= P.border && gy < h - P.border;
        f2 g[kRun];
#pragma unroll 1
        for (int gq0 = 0; gq0 < NB / 4; gq0 += kChunkG)
#pragma unroll
        for (int gq = gq0; gq < gq0 + kChunkG; ++gq) {
            f2 e[4][kRun];
#pragma unroll
            for (int oo = 0; oo < 4; ++oo) {
                const int o = 4 * gq + oo;
#pragma unroll
                for (int p = 0; p < kRun; ++p) e[oo][p] = zero2();
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    f2 v[6];
                    load_cols<3>(sCD + o * T::CD_PLANE + (r + ky) * T::CD_PITCH + kRun * k, v);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int p = 0; p < kRun; ++p) e[oo][p] = fma2(P.w5[ky * 3 + kx][o], v[p + kx], e[oo][p]);
                }
#pragma unroll
                for (int p = 0; p < kRun; ++p) {
                    f2 x = make_float2(clip_nan(relu_nan(e[oo][p].x), P.clip_max), clip_nan(relu_nan(e[oo][p].y), P.clip_max));
                    const int gx = gx0 + p;
                    if (!(row_in && gx >= P.border && gx < w - P.border))   // pad_inwards multiplies by 0: NaN stays NaN
                        x = make_float2(x.x != x.x ? x.x : 0.0f * x.x, x.y != x.y ? x.y : 0.0f * x.y);
                    e[oo][p] = x;
                    g[p] = o == 0 ? x : add2(g[p], x);
                }
            }
#pragma unroll
            for (int p = 0; p < kRun; ++p) {
                float *a = sStage + (size_t)r * T::ST_PITCH + (kRun * k + p) * NB + 4 * gq;
                float *b = sStage + (size_t)(TH + r) * T::ST_PITCH + (kRun * k + p) * NB + 4 * gq;
                *reinterpret_cast<float4 *>(a) = make_float4(e[0][p].x, e[1][p].x, e[2][p].x, e[3][p].x);
                *reinterpret_cast<float4 *>(b) = make_float4(e[0][p].y, e[1][p].y, e[2][p].y, e[3][p].y);
            }
        }
#pragma unroll
        for (int p = 0; p < kRun; ++p) g[p] = mul2(g[p], make_float2(inv_nb, inv_nb));
        if (gray) {   // few bytes: written straight from registers (4 consecutive floats per image)
            if (bulk_ok && gx0 + kRun <= w && gy < h) {
                *reinterpret_cast<float4 *>(gray + ((size_t)img0 * h + gy) * w + gx0) = make_float4(g[0].x, g[1].x, g[2].x, g[3].x);
                if (has_b)
                    *reinterpret_cast<float4 *>(gray + ((size_t)img1 * h + gy) * w + gx0) = make_float4(g[0].y, g[1].y, g[2].y, g[3].y);
            } else if (gy < h) {
#pragma unroll
                for (int p = 0; p < kRun; ++p)
                    if (gx0 + p < w) {
                        gray[((size_t)img0 * h + gy) * w + gx0 + p] = g[p].x;
                        if (has_b) gray[((size_t)img1 * h + gy) * w + gx0 + p] = g[p].y;
                    }
            }
        }
    }
    fence_async_smem();
    __syncthreads();
    issued = false;
    if (line_end) {
        if (tile_store) {
            if (tid == 0) {
                tile_store_images<TH>(&M.line_end, sStage, T::ST_PITCH, blockIdx.x, ty0, h, img0, img1, has_b);
                bulk_commit();
                issued = true;
            }
        } else if (bulk_ok) {
            issued = bulk_rows<TH>(sStage, T::ST_PITCH, line_end, img0, img1, has_b, ty0, h, (size_t)w * NB, (size_t)tx0 * NB,
                                   (uint32_t)(min(TW, w - tx0) * NB), warp_u, 0, NT / 32, leader);
        } else {
            for (int i = tid; i < 2 * TH * TW * NB; i += NT) {
                const int e = i % (TW * NB), row = i / (TW * NB), lane = row / TH, gy = ty0 + row % TH;
                if (gy < h && tx0 + e / NB < w && (lane == 0 || has_b))
                    line_end[(((size_t)(lane ? img1 : img0) * h + gy) * w + tx0) * NB + e] = sStage[(size_t)row * T::ST_PITCH + e];
            }
        }
    }
    if (issued) bulk_wait_read();
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------

static bool bits_equal(float a, float b) { return std::memcmp(&a, &b, 4) == 0; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// float32 view [planes][rows][2 * w] of a pair-interleaved tensor, boxes of [bp][br][2 * pitch]. False if TMA cannot be used.
static bool make_pair_map(CUtensorMap *map, const void *base, int w, int rows, long long planes, int pitch, int box_rows,
                          int box_planes)
{
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
            (void)cudaGetLastError();
            return false;
        }
        encode = (EncodeTiledFn)fn;
    }
    if ((w % 2) != 0 || 2 * pitch > 256 || box_rows > 256 || ((uintptr_t)base & 15) != 0) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)2 * w, (cuuint64_t)rows, (cuuint64_t)planes};
    const cuuint64_t strides[2] = {(cuuint64_t)2 * w * 4, (cuuint64_t)2 * w * 4 * rows};
    const cuuint32_t box[3] = {(cuuint32_t)(2 * pitch), (cuuint32_t)box_rows, (cuuint32_t)box_planes};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// Store view of an NHWC float32 output [n][h][w][ch] for TMA tile stores (see tma_store_tile): dims (floats of a tile row,
// tiles per row, rows, images), box (tile row + pad, 1, box_rows, 1). False if the geometry does not allow it.
static bool make_tile_store_map(CUtensorMap *map, const void *base, int n, int h, int w, int ch, int tw, int pad, int box_rows,
                                int elem_floats = 1)   // 2: 8-byte elements (tile rows of more than 252 floats: boxes hold <= 256 elements)
{
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
            (void)cudaGetLastError();
            return false;
        }
        encode = (EncodeTiledFn)fn;
    }
    const int tile_floats = tw * ch;
    if (!base || ((uintptr_t)base & 15) != 0 || w % tw != 0 || tile_floats % 4 != 0 || (tile_floats + pad) % 4 != 0 ||
        (tile_floats + pad) / elem_floats > 256 || box_rows > 256)
        return false;
    const cuuint64_t row_bytes = (cuuint64_t)w * ch * 4;
    const cuuint64_t dims[4] = {(cuuint64_t)(tile_floats / elem_floats), (cuuint64_t)(w / tw), (cuuint64_t)h, (cuuint64_t)n};
    const cuuint64_t strides[3] = {(cuuint64_t)tile_floats * 4, row_bytes, row_bytes * h};
    const cuuint32_t box[4] = {(cuuint32_t)((tile_floats + pad) / elem_floats), 1, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return encode(map, elem_floats == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static f2 dup(float v) { return make_float2(v, v); }

struct StackPlanHost {
    ParamsA a;
    ParamsB b;
    bool s1_depthwise, s2_rgby;
    bool s2_shared;           // rgby_3's shared-surround structure (stack_a_kernel, S2 mode 2)
    bool s3_sym, s5_ownoth;   // structure of the stripe / end filters (see stack_b_kernel)
};

// Validate the structure the fused kernels rely on and repack the HWIO filters as (w, w) pairs.
int pack_stack_params(const silent_stack_weights *W, int n, int h, int w, StackPlanHost *S)
{
    if (!W) return fail(SILENT_E_INVAL, "null weights");
    if (W->border < 0) return fail(SILENT_E_INVAL, "border must be >= 0");
    S->s1_depthwise = S->s2_rgby = true;
    for (int t = 0; t < 9; ++t)
        for (int ci = 0; ci < 3; ++ci)
            for (int co = 0; co < 3; ++co) {
                const int i = (t * 3 + ci) * 3 + co;
                S->a.w1[t][ci][co] = dup(W->rgc[i]);
                S->a.w2[t][ci][co] = dup(W->rgby[i]);
                S->b.w5[t][ci][co] = dup(W->end[i]);
                if (ci != co && W->rgc[i] != 0.0f) S->s1_depthwise = false;
                if (!rgby_nonzero(t, ci, co) && W->rgby[i] != 0.0f) S->s2_rgby = false;
                if (!bits_equal(W->stripe[i], W->stripe[(t * 3) * 3 + co]))
                    return fail(SILENT_E_STRUCTURE, "stripe filter differs across input channels at tap %d; the fused "
                                                    "stack needs identical input slices (use the per-operator calls)", t);
                S->b.w3[t][co] = dup(W->stripe[(t * 3) * 3 + co]);
            }
    {   // rgby_3 shared-surround structure (all comparisons bitwise; 2 * S is exact in float32)
        const float *R = W->rgby;
        auto at = [&](int t, int ci, int co) { return R[(t * 3 + ci) * 3 + co]; };
        bool ok = bits_equal(at(4, 0, 1), 0.0f);
        for (int t = 0; t < 9 && ok; ++t) {
            const float sv = at(t, 0, 1);
            ok = bits_equal(at(t, 0, 2), sv) && bits_equal(at(t, 1, 0), sv) && bits_equal(at(t, 2, 0), sv);
            if (t != 4)
                ok = ok && bits_equal(at(t, 1, 2), 2.0f * sv) && bits_equal(at(t, 2, 1), 2.0f * sv) &&
                     bits_equal(at(t, 0, 0), 0.0f) && bits_equal(at(t, 1, 1), 0.0f) && bits_equal(at(t, 2, 2), 0.0f);
            S->a.s2s[t] = dup(sv);
        }
        S->s2_shared = ok && S->s2_rgby;
        S->a.s2c[0] = dup(at(4, 0, 0)), S->a.s2c[1] = dup(at(4, 1, 1)), S->a.s2c[2] = dup(at(4, 2, 2));
        S->a.s2c[3] = dup(at(4, 1, 2)), S->a.s2c[4] = dup(at(4, 2, 1)), S->a.s2c[5] = dup(2.0f);
    }
    float blur_min = INFINITY;
    for (int t = 0; t < 49; ++t) {
        for (int s = 0; s < 9; ++s)
            if (!bits_equal(W->blur[t * 9 + s], W->blur[t * 9]))
                return fail(SILENT_E_STRUCTURE, "blur filter slices differ at tap %d; the fused stack needs one 7x7 "
                                                "kernel in every slice (use the per-operator calls)", t);
        S->b.wb[t] = dup(W->blur[t * 9]);
        blur_min = W->blur[t * 9] < blur_min ? W->blur[t * 9] : blur_min;   // (a NaN weight leaves blur_min alone ...)
        if (!(W->blur[t * 9] > 0.0f) || std::isinf(W->blur[t * 9])) blur_min = -1.0f;   // ... and lands here
    }
    // S4 early-out threshold: the smallest float T with rn(w_min * T) >= 1 (only when every blur weight is positive)
    S->b.quick_thr = 0.0f;
    if (blur_min > 0.0f && blur_min < INFINITY) {   // w_min * T >= 1.0001 in exact arithmetic (see S4 in stack_b_kernel)
        float T = (float)(1.0001 / (double)blur_min);
        for (int guard = 0; guard < 8 && !((double)blur_min * (double)T >= 1.0001); ++guard) T = std::nextafterf(T, INFINITY);
        if ((double)blur_min * (double)T >= 1.0001 && T < 1.0e20f) S->b.quick_thr = T;
    }
    // stripe kernels symmetric under a 180-degree rotation: w3[0..4] already are the five distinct taps
    S->s3_sym = true;
    for (int t = 0; t < 4; ++t)
        for (int co = 0; co < 3; ++co)
            if (!bits_equal(W->stripe[(t * 3) * 3 + co], W->stripe[((8 - t) * 3) * 3 + co])) S->s3_sym = false;
    // end filter: input channel ci feeds both other output channels with the same kernel
    S->s5_ownoth = true;
    for (int t = 0; t < 9; ++t)
        for (int ci = 0; ci < 3; ++ci) {
            const int o1 = (ci + 1) % 3, o2 = (ci + 2) % 3;
            if (!bits_equal(W->end[(t * 3 + ci) * 3 + o1], W->end[(t * 3 + ci) * 3 + o2])) S->s5_ownoth = false;
        }
    if (!(S->s3_sym && S->s5_ownoth)) S->s3_sym = S->s5_ownoth = false;   // two kernel variants: structured or dense
    if (S->s5_ownoth)
        for (int t = 0; t < 9; ++t)
            for (int ci = 0; ci < 3; ++ci) {
                S->b.w5[t][ci][0] = dup(W->end[(t * 3 + ci) * 3 + ci]);
                S->b.w5[t][ci][1] = dup(W->end[(t * 3 + ci) * 3 + (ci + 1) % 3]);
                S->b.w5[t][ci][2] = dup(0.0f);
            }
    S->a.h = S->b.h = h;
    S->a.w = S->b.w = w;
    S->a.n = S->b.n = n;
    S->b.reg_value = W->regulation_value;
    S->b.reg_root = W->regulation_root;
    S->b.clip_max = W->clip_max;
    S->b.border = W->border;
    S->b.win = WindowGeom();
    S->b.prefetch_pairs = 0, S->b.pairs = 0;
    return SILENT_OK;
}

#ifndef SILENT_TILE_HB
#define SILENT_TILE_HB 16
#endif
#ifndef SILENT_TILE_HA
#define SILENT_TILE_HA 16
#endif
// stack_a tile rows: TH + 2 must be a multiple of 3 (S1 row triples); with 22 the 8 triples of a tile fill a quarter-warp
constexpr int kTileHA = SILENT_TILE_HA, kTileHB = SILENT_TILE_HB;   // stack_b tile rows (quick and full variant share the tile grid)

// Tile width: the candidate that wastes the fewest columns of the last tile (288-wide levels: 6 x 48 instead of 4.5 x 64).
static int pick_tile_w(int w) { return ceil_div(w, 48) * 48 < ceil_div(w, 64) * 64 ? 48 : 64; }
// threads of stack_a: one warp-rounded round of S1 (its widest phase)
template <int TW>
struct ThreadsA {
    static constexpr int value = (TileA<kTileHA, TW>::A_ROWS * TileA<kTileHA, TW>::A_RUNS + 31) / 32 * 32;
};
// threads of stack_b: one warp-rounded round of its widest phase (S3), which also covers one S5 task per thread
template <int TH, int TW, bool LITE>
struct ThreadsB {
    static constexpr int value = (TileB<TH, TW, LITE>::CS_ROWS * TileB<TH, TW, LITE>::C_RUNS + 31) / 32 * 32;
};

// S1's deal of tasks (row triple, channel, run) to the lanes of stack_a (see TileA): octets of tasks whose bank groups
// (step * rt + c + 4 k) mod 8 are all different, as many full ones as the class sizes allow; the left-over tasks fill the
// remaining octets so that no group repeats more than it must. One table per tile shape and device, built on first use.
template <int TW>
static const unsigned char *s1_deal_table()
{
    using T = TileA<kTileHA, TW>;
    constexpr int NT = ThreadsA<TW>::value, TRIPLES = T::A_ROWS / 3, TASKS = 3 * TRIPLES * T::A_RUNS;
    if (!T::kDealOk || TASKS > NT || TRIPLES > 8 || T::A_RUNS > 8) return nullptr;
    static std::mutex lock;
    static unsigned char *tables[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> guard(lock);
    if (tables[dev]) return tables[dev];
    std::vector<int> by_unit[8];
    for (int k = 0; k < T::A_RUNS; ++k)
        for (int c = 0; c < 3; ++c)
            for (int rt = 0; rt < TRIPLES; ++rt) by_unit[(T::kBankStep * rt + c + 4 * k) % 8].push_back(rt | (c << 3) | (k << 5));
    std::vector<unsigned char> deal(NT, 255);
    const int octets = NT / 8;
    std::vector<int> used(octets * 8, 0);   // [octet][unit]: tasks of that unit already in the octet
    int next = 0;
    // pass 1: full octets (one task of every unit) while every class still has a task; pass 2: the rest, each task into the
    // octet where its unit is rarest (lanes of an octet are consecutive, so an octet is a quarter-warp of 128-bit accesses)
    std::vector<int> fill(octets, 0);
    for (; next < octets; ++next) {
        bool all = true;
        for (int u = 0; u < 8; ++u) all = all && !by_unit[u].empty();
        if (!all) break;
        for (int u = 0; u < 8; ++u) {
            deal[next * 8 + fill[next]++] = (unsigned char)by_unit[u].back();
            by_unit[u].pop_back();
            used[next * 8 + u] = 1;
        }
    }
    for (int u = 0; u < 8; ++u)
        while (!by_unit[u].empty()) {
            int best = -1;
            for (int o = next; o < octets; ++o)
                if (fill[o] < 8 && (best < 0 || used[o * 8 + u] < used[best * 8 + u] ||
                                    (used[o * 8 + u] == used[best * 8 + u] && fill[o] < fill[best])))
                    best = o;
            if (best < 0) return nullptr;   // cannot happen: TASKS <= NT
            deal[best * 8 + fill[best]++] = (unsigned char)by_unit[u].back();
            by_unit[u].pop_back();
            ++used[best * 8 + u];
        }
    unsigned char *d = nullptr;
    if (cudaMalloc(&d, NT) != cudaSuccess || cudaMemcpy(d, deal.data(), NT, cudaMemcpyHostToDevice) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    tables[dev] = d;
    return d;
}

template <int TW, bool DW, int RGBY, bool PAIRED>
static int launch_a(const void *pyr, const ParamsA &P, const CUtensorMap &tmap, f2 *bsum2, int pairs, cudaStream_t stream)
{
    using T = TileA<kTileHA, TW>;
    constexpr int kThreadsA = ThreadsA<TW>::value;
    auto kern = stack_a_kernel<kTileHA, TW, kThreadsA, DW, RGBY, PAIRED>;
    SILENT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::kSmemBytes));
    const dim3 grid(ceil_div(P.w, TW), ceil_div(P.h, kTileHA), pairs);
    const unsigned char *deal = DW ? s1_deal_table<TW>() : nullptr;
    SILENT_CUDA(launch_dependent(kern, grid, dim3(kThreadsA), T::kSmemBytes, stream, pyr, P, tmap, bsum2, deal));
    SILENT_LAUNCH_CHECK("stack_a_kernel");
    return SILENT_OK;
}

// room for one float2 plane per image pair (n images pair up into at most (n + levels) / 2 pairs for any pairing)
// ... plus one flag byte per (pair, stack_b tile)
static size_t stack_flag_bytes(int n, int h, int w)
{
    return ((size_t)(n / 2 + 8) * ceil_div(h, kTileHB) * ceil_div(w, 48) + 16 + 255) / 256 * 256;
}
static size_t stack_plane_bytes(int n, int h, int w) { return ((size_t)(n / 2 + 8) * h * (w + 2) * sizeof(f2) + 255) / 256 * 256; }
size_t stack_workspace_bytes(int n, int h, int w) { return stack_plane_bytes(n, h, w) + stack_flag_bytes(n, h, w) + 256; }

// three variants: the reference's filters (depthwise rgc + shared-surround rgby), their zero patterns only, dense
template <int TW, bool PAIRED>
static int dispatch_a(bool dw, bool rgby, bool shared, const void *in, const ParamsA &P, const CUtensorMap &tmap, f2 *bsum2,
                      int pairs, cudaStream_t stream)
{
    if (dw && shared) return launch_a<TW, true, 2, PAIRED>(in, P, tmap, bsum2, pairs, stream);
    if (dw && rgby) return launch_a<TW, true, 1, PAIRED>(in, P, tmap, bsum2, pairs, stream);
    return launch_a<TW, false, 0, PAIRED>(in, P, tmap, bsum2, pairs, stream);
}

template <int TH, int TW, bool STRUCTURED, bool LITE>
static int launch_b(StackPlanHost &S, int pairs, f2 *bsum2, float *orient, float *line_end, float *gray, int *winmax,
                    int *tilemax, unsigned char *tile_flag, cudaStream_t stream)
{
    const int h = S.b.h, w = S.b.w;
    CUtensorMap map_b;
    std::memset(&map_b, 0, sizeof(map_b));
    using TB = TileB<TH, TW, LITE>;
    constexpr int NT = ThreadsB<TH, TW, LITE>::value;
    auto kern = stack_b_kernel<TH, TW, NT, STRUCTURED, STRUCTURED, LITE>;
    SILENT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TB::kSmemBytes));
    S.b.use_tma = (w % 2) == 0 && make_pair_map(&map_b, bsum2, w + 2, h, pairs, TB::B_PITCH, TB::B_ROWS, 1);
    // outputs as TMA tile stores (one per 16 rows and image instead of one bulk copy per row) when every tile is whole in x
    StoreMaps maps;
    std::memset(&maps, 0, sizeof(maps));
    S.b.tma_store = (!orient || make_tile_store_map(&maps.orient, orient, S.b.n, h, w, 3, TW, TB::ST_PITCH - 3 * TW, kTileStoreRows)) &&
                    (!line_end || make_tile_store_map(&maps.line_end, line_end, S.b.n, h, w, 3, TW, TB::ST_PITCH - 3 * TW, kTileStoreRows)) &&
                    (!gray || make_tile_store_map(&maps.gray, gray, S.b.n, h, w, 1, TW, TB::G_PITCH - TW, kTileStoreRows));
    if (const char *e = std::getenv("SILENT_B_TILE_STORE")) S.b.tma_store = S.b.tma_store && std::atoi(e) != 0;   // tuning knob
    S.b.pairs = pairs;
    S.b.prefetch_pairs = 4;   // measured: 2 / 4 / 8 alike (-5 % on the quick pass), 0 = off
    if (const char *e = std::getenv("SILENT_B_PREFETCH")) S.b.prefetch_pairs = std::atoi(e);   // tuning knob
    const int nbx = ceil_div(w, TW), nby = ceil_div(h, TH);
    dim3 grid(nbx, nby, pairs);
    if (!LITE && tile_flag) {   // fix-up pass: two CTAs per SM walk the flagged tiles
        int dev = 0, sms = 148;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        grid = dim3((unsigned)std::min<long long>((long long)nbx * nby * pairs, 2LL * sms));
    }
    static_assert(TH % kTileHB == 0, "a launch's tiles are whole multiples of the emit grid's tile rows");
    SILENT_CUDA(launch_dependent(kern, grid, dim3(NT), TB::kSmemBytes, stream, (const f2 *)bsum2, S.b, map_b, maps, orient, line_end,
                                 gray, winmax, tilemax, tile_flag, nbx, nby, pairs, TH / kTileHB));
    SILENT_LAUNCH_CHECK("stack_b_kernel");
    return SILENT_OK;
}

template <int TWA>
static int launch_stack_a(const void *pyr, StackPlanHost &S, bool paired_in, int pairs, f2 *bsum2, cudaStream_t stream)
{
    const int h = S.a.h, w = S.a.w;
    CUtensorMap map_x;
    std::memset(&map_x, 0, sizeof(map_x));
    using TA = TileA<kTileHA, TWA>;
    S.a.prefetch_pairs = 8;   // ~ the image pairs whose tiles are resident on the chip at once
    if (const char *e = std::getenv("SILENT_A_PREFETCH")) S.a.prefetch_pairs = std::atoi(e);   // tuning knob
    S.a.use_tma = paired_in && make_pair_map(&map_x, pyr, w, h, 3LL * pairs, TA::X_PITCH, TA::X_ROWS, 3);
    return paired_in ? dispatch_a<TWA, true>(S.s1_depthwise, S.s2_rgby, S.s2_shared, pyr, S.a, map_x, bsum2, pairs, stream)
                     : dispatch_a<TWA, false>(S.s1_depthwise, S.s2_rgby, S.s2_shared, pyr, S.a, map_x, bsum2, pairs, stream);
}

template <int TW>
static int launch_stack(const void *pyr, StackPlanHost &S, bool paired_in, int pairs, f2 *bsum2, float *orient,
                        float *line_end, float *gray, int *winmax, int *tilemax, unsigned char *tile_flag, bool flags_clean,
                        cudaStream_t stream, cudaEvent_t between_kernels)
{
    int rc = launch_stack_a<TW>(pyr, S, paired_in, pairs, bsum2, stream);   // (96-wide stack_a tiles: measured 8 % slower)
    if (rc != SILENT_OK) return rc;
    if (between_kernels) SILENT_CUDA(cudaEventRecord(between_kernels, stream));   // stage timing hook
    if (!(S.s3_sym && S.s5_ownoth))
        return launch_b<kTileHB, TW, false, false>(S, pairs, bsum2, orient, line_end, gray, winmax, tilemax, nullptr, stream);
    // a grid that fits the device in about one wave (single frames, config C2) gains nothing from the quick variant's
    // higher occupancy and would pay for a second launch: the full variant does it alone
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (long long)pairs * ceil_div(S.b.h, kTileHB) * ceil_div(S.b.w, TW);
    if (tiles <= 3LL * sms && (S.b.h % (2 * kTileHB)) == 0)   // ... on tiles twice as tall (half as many CTAs, one wave)
        return launch_b<2 * kTileHB, TW, true, false>(S, pairs, bsum2, orient, line_end, gray, winmax, tilemax, nullptr, stream);
    if (!(S.b.quick_thr > 0.0f && tile_flag) || tiles <= 3LL * sms)
        return launch_b<kTileHB, TW, true, false>(S, pairs, bsum2, orient, line_end, gray, winmax, tilemax, nullptr, stream);
    // quick variant on every tile, then the full variant on the tiles it flagged (none on textured input)
    if (!flags_clean) {   // (the pipeline clears them before the pyramid launch, so that no memset sits between kernels)
        const size_t flags = (size_t)pairs * ceil_div(S.b.h, kTileHB) * ceil_div(S.b.w, TW);
        SILENT_CUDA(cudaMemsetAsync(tile_flag - 16, 0, flags + 16, stream));   // flags and the counter in front of them
    }
    rc = launch_b<kTileHB, TW, true, true>(S, pairs, bsum2, orient, line_end, gray, winmax, tilemax, tile_flag, stream);
    if (rc != SILENT_OK) return rc;
    if ((S.b.h % (2 * kTileHB)) == 0)   // fix-up on tiles twice as tall: a third less halo arithmetic per redone row
        return launch_b<2 * kTileHB, TW, true, false>(S, pairs, bsum2, orient, line_end, gray, winmax, tilemax, tile_flag, stream);
    return launch_b<kTileHB, TW, true, false>(S, pairs, bsum2, orient, line_end, gray, winmax, tilemax, tile_flag, stream);
}

// Tile grid of stack_b for a level shape (the emit stage reads the per-tile maxima it writes).
void stack_tile_grid(int h, int w, int *tile_h, int *tile_w, int *nty, int *ntx)
{
    *tile_h = kTileHB;
    *tile_w = pick_tile_w(w);
    *nty = ceil_div(h, *tile_h);
    *ntx = ceil_div(w, *tile_w);
}

// pyr: NHWC float32 [n][h][w][3] when pair_levels == 0 (images paired (2p, 2p+1)), else the pair-interleaved planar
// tensor of pyramid_pair_kernel with `pair_levels` levels per frame (images paired across consecutive frames).
// winmax: optional int[n * windows] (zeroed by the caller) receiving the per-region maxima of gray; geometry in *geo.
// Zeroes the tile flags (and the counter in front of them) stack_fused will use for n images; the pipeline calls this
// ahead of the pyramid launch and then passes flags_clean = true.
void stack_flag_region(void *workspace, int n, int h, int w, void **ptr, size_t *bytes)
{
    unsigned char *base = reinterpret_cast<unsigned char *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    *ptr = base + stack_plane_bytes(n, h, w);
    *bytes = stack_flag_bytes(n, h, w);
}

int stack_clear_flags(void *workspace, int n, int h, int w, cudaStream_t stream)
{
    unsigned char *base = reinterpret_cast<unsigned char *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    SILENT_CUDA(cudaMemsetAsync(base + stack_plane_bytes(n, h, w), 0, stack_flag_bytes(n, h, w), stream));
    return SILENT_OK;
}

int stack_fused(const void *pyr, int n, int h, int w, int pair_levels, const silent_stack_weights *W, float *orient,
                float *line_end, float *gray, void *workspace, size_t workspace_bytes, const WindowGeom *geo,
                int *winmax, int *tilemax, cudaStream_t stream, cudaEvent_t between_kernels, bool flags_clean)
{
    if (!pyr) return fail(SILENT_E_INVAL, "silent_stack_fused: null pyramid");
    if (n <= 0 || h <= 0 || w <= 0) return fail(SILENT_E_INVAL, "silent_stack_fused: bad shape %dx%dx%d", n, h, w);
    const bool paired_in = pair_levels > 0;
    const int levels = paired_in ? pair_levels : 1;
    if (n % levels != 0) return fail(SILENT_E_INVAL, "silent_stack_fused: n must be a multiple of the levels per frame");
    const int pairs = ((n / levels + 1) / 2) * levels;
    if (pairs > 65535) return fail(SILENT_E_SHAPE, "silent_stack_fused: at most 65535 image pairs per call");
    if (!workspace || workspace_bytes < stack_workspace_bytes(n, h, w))
        return fail(SILENT_E_CAPACITY, "silent_stack_fused: workspace too small (%zu < %zu bytes)", workspace_bytes,
                    stack_workspace_bytes(n, h, w));
    for (const void *p : {(const void *)pyr, (const void *)orient, (const void *)line_end, (const void *)gray})
        if (((uintptr_t)p & 15) != 0) return fail(SILENT_E_INVAL, "silent_stack_fused: tensors must be 16-byte aligned");
    StackPlanHost S;
    int rc = pack_stack_params(W, n, h, w, &S);
    if (rc != SILENT_OK) return rc;
    if (geo && winmax) S.b.win = *geo;
    S.a.pair_levels = S.b.pair_levels = pack_pair_levels(levels);
    f2 *bsum2 = reinterpret_cast<f2 *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    unsigned char *tile_flag = reinterpret_cast<unsigned char *>(bsum2) + stack_plane_bytes(n, h, w) + 16;   // [-4]: counter
    if (pick_tile_w(w) == 48)
        return launch_stack<48>(pyr, S, paired_in, pairs, bsum2, orient, line_end, gray, winmax, tilemax, tile_flag,
                                flags_clean, stream, between_kernels);
    return launch_stack<64>(pyr, S, paired_in, pairs, bsum2, orient, line_end, gray, winmax, tilemax, tile_flag, flags_clean,
                            stream, between_kernels);
}


// ---- orientation banks (config C4 and its 4-, 12- and 16-wide variants): S1-S2 through stack_a, then stack_bank_kernel ---

// Tile per width, 16 rows x 32 columns up to 8 orientations, 16 x 16 beyond: wider banks on 32 columns fit one CTA per SM
// (115 / 152 KB of shared memory) and, at NB = 16, a tile row outgrows the 256-element TMA store box; on 16 columns
// they run 2 CTAs/SM with tile stores, 15 % (NB = 12) and 18 % (NB = 16) faster on C4 frames (DESIGN §4).
template <int NB>
struct BankTile {
    static constexpr int TH = 16;
    static constexpr int TW = NB <= 8 ? 32 : 16;
    using T = TileBank<NB, TH, TW>;
    static constexpr int NT = (T::CS_ROWS * T::C_RUNS + 31) / 32 * 32;   // one warp-rounded round of S3
};

static bool bank_width_supported(int nb) { return nb == 4 || nb == 8 || nb == 12 || nb == 16; }

int check_bank(const silent_orientation_bank *W, const char *who)
{
    if (!W) return fail(SILENT_E_INVAL, "%s: null bank", who);
    const int nb = W->orientations;
    if (!bank_width_supported(nb))
        return fail(SILENT_E_SHAPE, "%s: %d orientations; the fused bank supports 4, 8, 12 or 16", who, nb);
    // structure the kernel relies on (what the reference's per-vector generators produce, SURVEY 8(d) config C4); runs
    // on every call, so the bitwise comparisons go by memcmp over contiguous runs
    for (int t = 0; t < 9; ++t) {
        const float *s0 = W->stripe + t * 3 * nb;
        if (std::memcmp(s0 + nb, s0, nb * sizeof(float)) != 0 || std::memcmp(s0 + 2 * nb, s0, nb * sizeof(float)) != 0)
            return fail(SILENT_E_STRUCTURE, "stripe bank differs across input channels at tap %d", t);
        for (int ci = 0; ci < nb; ++ci)
            for (int o = 0; o < nb; ++o)
                if (ci != o && W->end[(t * nb + ci) * nb + o] != 0.0f)
                    return fail(SILENT_E_STRUCTURE, "end bank couples orientations %d -> %d (needs a depthwise bank)", ci, o);
    }
    for (int t = 0; t < 49; ++t) {   // all nb * nb slices equal <=> every element equals its successor
        const float *b = W->blur + t * nb * nb;
        if (std::memcmp(b + 1, b, (nb * nb - 1) * sizeof(float)) != 0)
            return fail(SILENT_E_STRUCTURE, "blur bank slices differ at tap %d", t);
    }
    return SILENT_OK;
}

template <int NB>
static int launch_bank(const silent_orientation_bank *W, int n, int h, int w, int levels, int pairs, const f2 *bsum2,
                       float *orient, float *line_end, float *gray, cudaStream_t stream)
{
    ParamsBank<NB> B;
    float blur_min = INFINITY;
    for (int t = 0; t < 49; ++t) {
        const float b = W->blur[t * NB * NB];
        B.wb[t] = dup(b);
        blur_min = b < blur_min ? b : blur_min;
        if (!(b > 0.0f) || std::isinf(b)) blur_min = -1.0f;
    }
    for (int t = 0; t < 9; ++t)
        for (int o = 0; o < NB; ++o) {
            B.w3[t][o] = dup(W->stripe[(t * 3) * NB + o]);
            B.w5[t][o] = dup(W->end[(t * NB + o) * NB + o]);
        }
    B.quick_thr = 0.0f;
    if (blur_min > 0.0f && blur_min < INFINITY) {
        float T = (float)(1.0001 / (double)blur_min);
        for (int guard = 0; guard < 8 && !((double)blur_min * (double)T >= 1.0001); ++guard) T = std::nextafterf(T, INFINITY);
        if ((double)blur_min * (double)T >= 1.0001 && T < 1.0e20f) B.quick_thr = T;
    }
    B.reg_value = W->regulation_value, B.reg_root = W->regulation_root, B.clip_max = W->clip_max, B.border = W->border;
    B.h = h, B.w = w, B.n = n, B.pair_levels = pack_pair_levels(levels);

    using Tile = BankTile<NB>;
    using T = typename Tile::T;
    auto kern = stack_bank_kernel<NB, Tile::TH, Tile::TW, Tile::NT>;
    SILENT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::kSmemBytes));
    const dim3 grid(ceil_div(w, Tile::TW), ceil_div(h, Tile::TH), pairs);
    StoreMaps maps;   // tile rows of up to 388 floats: described in 8-byte elements (a box holds at most 256 of them)
    std::memset(&maps, 0, sizeof(maps));
    const int pad = T::ST_PITCH - NB * Tile::TW;
    B.tma_store = (!orient || make_tile_store_map(&maps.orient, orient, n, h, w, NB, Tile::TW, pad, kTileStoreRows, 2)) &&
                  (!line_end || make_tile_store_map(&maps.line_end, line_end, n, h, w, NB, Tile::TW, pad, kTileStoreRows, 2));
    if (const char *e = std::getenv("SILENT_B_TILE_STORE")) B.tma_store = B.tma_store && std::atoi(e) != 0;   // tuning knob
    SILENT_CUDA(launch_dependent(kern, grid, dim3(Tile::NT), T::kSmemBytes, stream, bsum2, B, maps, orient, line_end, gray));
    SILENT_LAUNCH_CHECK("stack_bank_kernel");
    return SILENT_OK;
}

int stack_bank(const void *pyr, int n, int h, int w, int pair_levels, const silent_orientation_bank *W, float *orient,
               float *line_end, float *gray, void *workspace, size_t workspace_bytes, cudaStream_t stream,
               cudaEvent_t between_kernels)
{
    if (!pyr || !W) return fail(SILENT_E_INVAL, "bank stack: null argument");
    if (n <= 0 || h <= 0 || w <= 0) return fail(SILENT_E_INVAL, "bank stack: bad shape %dx%dx%d", n, h, w);
    const bool paired_in = pair_levels > 0;
    const int levels = paired_in ? pair_levels : 1;
    if (n % levels != 0) return fail(SILENT_E_INVAL, "bank stack: n must be whole frames");
    const int pairs = ((n / levels + 1) / 2) * levels;
    if (pairs > 65535) return fail(SILENT_E_SHAPE, "bank stack: at most 65535 image pairs per call");
    if (!workspace || workspace_bytes < stack_workspace_bytes(n, h, w))
        return fail(SILENT_E_CAPACITY, "bank stack: workspace too small (%zu < %zu bytes)", workspace_bytes,
                    stack_workspace_bytes(n, h, w));
    for (const void *p : {(const void *)pyr, (const void *)orient, (const void *)line_end, (const void *)gray})
        if (((uintptr_t)p & 15) != 0) return fail(SILENT_E_INVAL, "bank stack: tensors must be 16-byte aligned");

    // S1 + S2 -> channel sum, exactly as in the three-orientation stack
    silent_stack_weights tmp;
    std::memset(&tmp, 0, sizeof(tmp));
    std::memcpy(tmp.rgc, W->rgc, sizeof(tmp.rgc));
    std::memcpy(tmp.rgby, W->rgby, sizeof(tmp.rgby));
    for (float &b : tmp.blur) b = 1.0f;
    tmp.regulation_value = 1.0f, tmp.regulation_root = 0.1f, tmp.clip_max = W->clip_max, tmp.border = W->border;
    StackPlanHost S;
    int rc = pack_stack_params(&tmp, n, h, w, &S);
    if (rc != SILENT_OK) return rc;
    S.a.pair_levels = pack_pair_levels(levels);
    f2 *bsum2 = reinterpret_cast<f2 *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    rc = pick_tile_w(w) == 48 ? launch_stack_a<48>(pyr, S, paired_in, pairs, bsum2, stream)
                              : launch_stack_a<64>(pyr, S, paired_in, pairs, bsum2, stream);
    if (rc != SILENT_OK) return rc;
    if (between_kernels) SILENT_CUDA(cudaEventRecord(between_kernels, stream));   // stage timing hook
    switch (W->orientations) {
    case 4: return launch_bank<4>(W, n, h, w, levels, pairs, bsum2, orient, line_end, gray, stream);
    case 8: return launch_bank<8>(W, n, h, w, levels, pairs, bsum2, orient, line_end, gray, stream);
    case 12: return launch_bank<12>(W, n, h, w, levels, pairs, bsum2, orient, line_end, gray, stream);
    default: return launch_bank<16>(W, n, h, w, levels, pairs, bsum2, orient, line_end, gray, stream);
    }
}

}  // namespace silent

extern "C" {

size_t silent_stack_workspace_bytes(int n, int h, int w)
{
    if (n <= 0 || h <= 0 || w <= 0) return 0;
    return silent::stack_workspace_bytes(n, h, w);
}

int silent_stack_fused(const float *pyramid_dev, int n, int h, int w, const silent_stack_weights *weights_host,
                       float *orient_dev, float *line_end_dev, float *gray_dev, void *workspace_dev,
                       size_t workspace_bytes, silent_stream stream)
{
    return silent::stack_fused(pyramid_dev, n, h, w, 0, weights_host, orient_dev, line_end_dev, gray_dev, workspace_dev,
                               workspace_bytes, nullptr, nullptr, nullptr, (cudaStream_t)stream, nullptr, false);
}

int silent_stack_bank(const float *pyramid_dev, int n, int h, int w, const silent_orientation_bank *bank_host,
                      float *orient_dev, float *line_end_dev, float *gray_dev, void *workspace_dev, size_t workspace_bytes,
                      silent_stream stream)
{
    const int rc = silent::check_bank(bank_host, "silent_stack_bank");
    if (rc != SILENT_OK) return rc;
    return silent::stack_bank(pyramid_dev, n, h, w, 0, bank_host, orient_dev, line_end_dev, gray_dev, workspace_dev,
                              workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
