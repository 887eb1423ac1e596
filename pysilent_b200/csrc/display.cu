// The display tensors that follow gray_line_end_tensor in LineEndDisplayer.compile (reference
// recognition_testing.py:79-100): block centroids (util/centroids.py:21-71), nearest-neighbour resize, the stateful
// boosting non-max (util/energy/boosting.py:10-42, recovery.py:4-22) and the scalar display arithmetic.
//
// All of them are tiny against the filter stack (a 3 x 3 block pool of a one-channel level, 64 x 96 per level for the
// boosting state): one thread per output element, coalesced one-channel reads, no shared memory. Arithmetic follows the
// canonical order of oracle/silent_oracle.c ("next rows" section), so results are bit-identical to it.
//
// display_sequence_kernel is the exception: it walks the boosting recurrence of a whole clip with the state of a level
// held on chip, one thread-block cluster per level, the CTAs of a cluster sharing the non-max halo rows through
// distributed shared memory.
#include <cooperative_groups.h>
#include <limits.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace silent {

__host__ __device__ inline void same_geometry(int n, int k, int s, int *out, int *before)
{
    *out = (n + s - 1) / s;
    int total = (*out - 1) * s + k - n;
    if (total < 0) total = 0;
    *before = total / 2;
}

// tf.image.resize_nearest_neighbor, align_corners = False: min(floor(dst * float32(in / out)), in - 1)
__device__ __forceinline__ int nearest_src(int dst, int n_in, float scale)
{
    const int s = (int)floorf(__fmul_rn((float)dst, scale));
    return s < n_in - 1 ? s : n_in - 1;
}
static float nearest_scale(int n_in, int n_out) { return (float)((double)n_in / (double)n_out); }

// one thread per (image, block): value-weighted index sums over the region window, centroid = sum / total
__global__ void __launch_bounds__(256) centroid_blocks_kernel(const float *__restrict__ value, int n, int h, int w, int rh,
                                                              int rw, int oh, int ow, int pt, int pl,
                                                              float *__restrict__ corrected, float *__restrict__ total)
{
    const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= (size_t)n * oh * ow) return;
    const int j = (int)(o % ow), i = (int)((o / ow) % oh), img = (int)(o / ((size_t)ow * oh));
    const float *v = value + (size_t)img * h * w;
    float sx = 0.0f, sy = 0.0f, st = 0.0f;
    for (int ky = 0; ky < rh; ++ky) {
        const int y = i * rh - pt + ky;
        if (y < 0 || y >= h) continue;
        for (int kx = 0; kx < rw; ++kx) {
            const int x = j * rw - pl + kx;
            if (x < 0 || x >= w) continue;
            const float val = __ldg(v + (size_t)y * w + x);
            sx = __fadd_rn(sx, __fmul_rn((float)x, val));
            sy = __fadd_rn(sy, __fmul_rn((float)y, val));
            st = __fadd_rn(st, val);
        }
    }
    corrected[2 * o] = __fdiv_rn(sx, st);       // 0 / 0 = NaN on an empty block, like the reference graph
    corrected[2 * o + 1] = __fdiv_rn(sy, st);
    total[o] = st;
}

// one thread per pixel: L1 distance to the centroid of its (nearest-upsampled) block
__global__ void __launch_bounds__(256) centroid_distance_kernel(const float *__restrict__ corrected, int n, int h, int w,
                                                                int oh, int ow, float sy_scale, float sx_scale,
                                                                float *__restrict__ out)
{
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (size_t)n * h * w) return;
    const int x = (int)(p % w), y = (int)((p / w) % h), img = (int)(p / ((size_t)w * h));
    const int i = nearest_src(y, oh, sy_scale), j = nearest_src(x, ow, sx_scale);
    const float2 c = __ldg(reinterpret_cast<const float2 *>(corrected) + ((size_t)img * oh + i) * ow + j);
    out[p] = __fadd_rn(fabsf(__fsub_rn(c.x, (float)x)), fabsf(__fsub_rn(c.y, (float)y)));
}

__global__ void __launch_bounds__(256) resize_nearest_kernel(const float *__restrict__ x, int n, int h, int w, int c, int oh,
                                                             int ow, float sy_scale, float sx_scale,
                                                             float *__restrict__ out)
{
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)n * oh * ow * c) return;
    const int ch = (int)(e % c);
    const size_t p = e / c;
    const int xx = (int)(p % ow), yy = (int)((p / ow) % oh), img = (int)(p / ((size_t)ow * oh));
    const int sy = nearest_src(yy, h, sy_scale), sx = nearest_src(xx, w, sx_scale);
    out[e] = __ldg(x + (((size_t)img * h + sy) * w + sx) * c + ch);
}

__global__ void __launch_bounds__(256) boosting_bias_kernel(const float *__restrict__ inp, const float *__restrict__ energy,
                                                            size_t count, float *__restrict__ biased)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) biased[i] = canon_pow(inp[i], energy[i]);   // input ** exhaustion_tensor.value()  boosting.py:17
}

__device__ __forceinline__ float nan_max(float a, float b) { return (a != a) ? a : ((b != b) ? b : (a > b ? a : b)); }

// the 3 x 3 max-pool (SAME, NaN propagating) of the reference's non-max at (y, x) of an h x w grid; load(yy, xx) reads
// one value. Both boosting display kernels take their window through here, so they visit it in the same order.
template <class Load>
__device__ __forceinline__ float window_max3(Load load, int y, int x, int h, int w)
{
    bool first = true;
    float m = 0.0f;
    for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
            const int yy = y + dy, xx = x + dx;
            if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
            const float v = load(yy, xx);
            m = first ? v : nan_max(m, v);
            first = false;
        }
    return m;
}

// one cell of get_boosting(for_visualizing=True) after the non-max: `own` is the cell's importance ** energy and m its
// window maximum. Writes the two 3-channel display values of cell o and returns the updated energy.
__device__ __forceinline__ float display_cell(float own, float m, float inp, float energy, float exhaustion_max,
                                              float excitation_max, int recovery_mode, float normer, float centerer,
                                              size_t o, float *__restrict__ fired_disp, float *__restrict__ update_disp)
{
    const float f = (own == m) ? 1.0f : 0.0f;                                      // boosting.py:20-22
    const float strength = __fmul_rn(f, inp);                                      // :24
    const float exhaustion = __fmul_rn(f, 255.0f);                                 // :26
    float recovery = 10.0f;                                                        // recovery.py:4-5
    if (recovery_mode == 2) recovery = __fmul_rn(strength, 0.8f);                  // recovery.py:8-9
    if (recovery_mode == 3) recovery = nan_max(__fmul_rn(strength, 0.8f), 10.0f);  // recovery.py:19
    float t = __fmul_rn(energy, 255.0f);                                           // boosting.py:30-33
    t = __fsub_rn(t, exhaustion);
    t = __fadd_rn(t, recovery);
    t = __fdiv_rn(t, 255.0f);
    t = t < -exhaustion_max ? -exhaustion_max : t;
    t = t > excitation_max ? excitation_max : t;
    const float fd = __fmul_rn(strength, 255.0f);                                  // (has_fired * input) * 255
    const float ud = __fadd_rn(__fmul_rn(t, normer), centerer);                    // update_energy * normer + centerer
    fired_disp[3 * o] = fired_disp[3 * o + 1] = fired_disp[3 * o + 2] = fd;
    update_disp[3 * o] = update_disp[3 * o + 1] = update_disp[3 * o + 2] = ud;
    return t;
}

// 3 x 3 max-pool equality test (the reference's non-max), fire strength, exhaustion / recovery, state update
__global__ void __launch_bounds__(256) boosting_update_kernel(const float *__restrict__ inp, const float *__restrict__ biased,
                                                              float *__restrict__ energy, int n, int h, int w,
                                                              float exhaustion_max, float excitation_max, int recovery_mode,
                                                              float *__restrict__ fired)
{
    const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= (size_t)n * h * w) return;
    const int x = (int)(o % w), y = (int)((o / w) % h);
    const float *b = biased + (o - (size_t)y * w - x);
    bool first = true;
    float m = 0.0f;
    for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
            const int yy = y + dy, xx = x + dx;
            if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
            const float v = __ldg(b + (size_t)yy * w + xx);
            m = first ? v : nan_max(m, v);
            first = false;
        }
    const float f = (__ldg(b + (size_t)y * w + x) == m) ? 1.0f : 0.0f;                 // boosting.py:20-22
    const float strength = __fmul_rn(f, inp[o]);                                       // :24
    const float exhaustion = __fmul_rn(f, 255.0f);                                     // :26
    float recovery = 10.0f;                                                            // recovery.py:4-5
    if (recovery_mode == 2) recovery = __fmul_rn(strength, 0.8f);                      // recovery.py:8-9
    if (recovery_mode == 3) recovery = nan_max(__fmul_rn(strength, 0.8f), 10.0f);      // recovery.py:19
    float t = __fmul_rn(energy[o], 255.0f);                                            // boosting.py:30-33
    t = __fsub_rn(t, exhaustion);
    t = __fadd_rn(t, recovery);
    t = __fdiv_rn(t, 255.0f);
    t = t < -exhaustion_max ? -exhaustion_max : t;
    t = t > excitation_max ? excitation_max : t;
    fired[o] = f;
    energy[o] = t;
}

__global__ void __launch_bounds__(256) pointwise_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                        size_t count, int kind, float *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const float v = x[i];
    float r;
    switch (kind) {
        case SILENT_PW_DIV255: r = __fdiv_rn(v, 255.0f); break;
        case SILENT_PW_INVERT255: r = __fsub_rn(255.0f, __fmul_rn(v, 255.0f)); break;
        case SILENT_PW_IMPORTANCE: {
            float t = __fmul_rn(v, 63.75f);
            t = t < 1.0f ? 1.0f : t;
            t = t > 256.0f ? 256.0f : t;
            r = __fsub_rn(t, 1.0f);
        } break;
        case SILENT_PW_MUL255: r = __fmul_rn(v, 255.0f); break;
        case SILENT_PW_ENERGY_DISPLAY: r = __fadd_rn(__fmul_rn(v, 127.5f), 127.5f); break;
        default: r = __fmul_rn(v, y[i]); break;
    }
    out[i] = r;
}

// rows [0, capacity) = the rank's points with the level id rebased to the global frame order (rows beyond the count are
// zeroed), row `capacity` = (count, 0, 0, 0): ONE buffer, so the exchange is a single all-gather
__global__ void __launch_bounds__(256) pack_points_kernel(const long long *__restrict__ points,
                                                          const long long *__restrict__ count, long long capacity,
                                                          long long level_offset, long long *__restrict__ packed)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > capacity) return;
    const long long n = *count < capacity ? *count : capacity;
    longlong2 a = make_longlong2(0, 0), b = make_longlong2(0, 0);
    if (i == capacity) {
        a.x = *count;
    } else if (i < n) {
        a = reinterpret_cast<const longlong2 *>(points)[2 * i];
        b = reinterpret_cast<const longlong2 *>(points)[2 * i + 1];
        a.x += level_offset;
    }
    reinterpret_cast<longlong2 *>(packed)[2 * i] = a;
    reinterpret_cast<longlong2 *>(packed)[2 * i + 1] = b;
}

// ---------------------------------------------------------------------------------------------------------------------
// The whole display chain of LineEndDisplayer.compile (reference recognition_testing.py:79-100) in TWO launches instead of
// seventeen. The operators above stay as the stand-alone API; these kernels apply the same roundings in the same order,
// so their results are bit-identical to the chain of operators (tests/test_gpu_parity.py compares both).
// ---------------------------------------------------------------------------------------------------------------------
struct DisplayGeom {
    int n, h, w;                 // gray levels
    int rh, rw;                  // centroid region
    int oh, ow, pt, pl;          // block grid of the full image (SAME geometry) ...
    float by, bx;                // ... and the nearest-neighbour scales that map a pixel to its block
    int h2, w2;                  // the e^-0.5 resize of gray (recognition_testing.py:82-83)
    float ry, rx;                // nearest-neighbour scales gray -> im2
    int oh2, ow2, pt2, pl2;      // block grid of im2
    float by2, bx2;
};

// value-weighted index sums of block (i, j); HALF reads gray through the nearest-neighbour map of im2. value = gray / 255.
template <bool HALF>
__device__ __forceinline__ void block_sums(const float *__restrict__ gray, const DisplayGeom &G, int i, int j, float &sx,
                                           float &sy, float &st)
{
    const int hh = HALF ? G.h2 : G.h, ww = HALF ? G.w2 : G.w, pt = HALF ? G.pt2 : G.pt, pl = HALF ? G.pl2 : G.pl;
    sx = sy = st = 0.0f;
    for (int ky = 0; ky < G.rh; ++ky) {
        const int y = i * G.rh - pt + ky;
        if (y < 0 || y >= hh) continue;
        const int gy = HALF ? nearest_src(y, G.h, G.ry) : y;
        for (int kx = 0; kx < G.rw; ++kx) {
            const int x = j * G.rw - pl + kx;
            if (x < 0 || x >= ww) continue;
            const int gx = HALF ? nearest_src(x, G.w, G.rx) : x;
            const float val = __fdiv_rn(__ldg(gray + (size_t)gy * G.w + gx), 255.0f);
            sx = __fadd_rn(sx, __fmul_rn((float)x, val));
            sy = __fadd_rn(sy, __fmul_rn((float)y, val));
            st = __fadd_rn(st, val);
        }
    }
}

// threads [0, n*h*w): 255 - centroids * 255; then [.., + n*h2*w2): the same on im2; then [.., + n*oh*ow): block importance
// and (BIASED) importance ** energy for the non-max of the second launch. A pixel recomputes the sums of its own block (9
// cached loads) instead of waiting for a block pass: no dependency between threads, one launch. A clip runs it without
// BIASED (energy and biased unused): there the bias of step t needs the energy of step t - 1.
template <bool BIASED>
__global__ void __launch_bounds__(256) display_centroids_kernel(const float *__restrict__ gray, const DisplayGeom G,
                                                                const float *__restrict__ energy,
                                                                float *__restrict__ cent_disp, float *__restrict__ cent2_disp,
                                                                float *__restrict__ importance, float *__restrict__ biased)
{
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t full = (size_t)G.n * G.h * G.w, half = (size_t)G.n * G.h2 * G.w2, blocks = (size_t)G.n * G.oh * G.ow;
    float sx, sy, st;
    if (t < full) {
        const int x = (int)(t % G.w), y = (int)((t / G.w) % G.h), img = (int)(t / ((size_t)G.w * G.h));
        block_sums<false>(gray + (size_t)img * G.h * G.w, G, nearest_src(y, G.oh, G.by), nearest_src(x, G.ow, G.bx), sx, sy, st);
        const float d = __fadd_rn(fabsf(__fsub_rn(__fdiv_rn(sx, st), (float)x)), fabsf(__fsub_rn(__fdiv_rn(sy, st), (float)y)));
        cent_disp[t] = __fsub_rn(255.0f, __fmul_rn(d, 255.0f));
        return;
    }
    t -= full;
    if (t < half) {
        const int x = (int)(t % G.w2), y = (int)((t / G.w2) % G.h2), img = (int)(t / ((size_t)G.w2 * G.h2));
        block_sums<true>(gray + (size_t)img * G.h * G.w, G, nearest_src(y, G.oh2, G.by2), nearest_src(x, G.ow2, G.bx2), sx, sy, st);
        const float d = __fadd_rn(fabsf(__fsub_rn(__fdiv_rn(sx, st), (float)x)), fabsf(__fsub_rn(__fdiv_rn(sy, st), (float)y)));
        cent2_disp[t] = __fsub_rn(255.0f, __fmul_rn(d, 255.0f));
        return;
    }
    t -= half;
    if (t < blocks) {
        const int j = (int)(t % G.ow), i = (int)((t / G.ow) % G.oh), img = (int)(t / ((size_t)G.ow * G.oh));
        block_sums<false>(gray + (size_t)img * G.h * G.w, G, i, j, sx, sy, st);
        float v = __fmul_rn(st, 63.75f);                       // clip(importances * (255 / 4), 1, 256) - 1  (:81)
        v = v < 1.0f ? 1.0f : v;
        v = v > 256.0f ? 256.0f : v;
        v = __fsub_rn(v, 1.0f);
        importance[t] = v;
        if (BIASED) biased[t] = canon_pow(v, energy[t]);       // boosting.py:17
    }
}

// the non-max / exhaustion / recovery update of boosting_update_kernel plus the two display tensors made from it
// (boosting.py:35-40 with for_visualizing, recognition_testing.py:98-100): three equal channels each
__global__ void __launch_bounds__(256) display_boosting_kernel(const float *__restrict__ inp, const float *__restrict__ biased,
                                                               float *__restrict__ energy, int n, int h, int w,
                                                               float exhaustion_max, float excitation_max, int recovery_mode,
                                                               float normer, float centerer, float *__restrict__ fired_disp,
                                                               float *__restrict__ update_disp)
{
    const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= (size_t)n * h * w) return;
    const int x = (int)(o % w), y = (int)((o / w) % h);
    const float *b = biased + (o - (size_t)y * w - x);
    const float m = window_max3([&](int yy, int xx) { return __ldg(b + (size_t)yy * w + xx); }, y, x, h, w);
    energy[o] = display_cell(__ldg(b + (size_t)y * w + x), m, inp[o], energy[o], exhaustion_max, excitation_max,
                             recovery_mode, normer, centerer, o, fired_disp, update_disp);
}

// The boosting recurrence of a whole clip: steps x n level images, time-major (image t * n + e is step t of energy slice
// e). One cluster of C CTAs per slice e; CTA r owns block rows [r * band, r * band + rows) and each thread a fixed set of
// up to CPT cells of that band, so the cell's energy lives in a register from the first step to the last. Per step a
// CTA writes importance ** energy of its band into one of two shared buffers, the cluster meets at one barrier, and the
// non-max reads the row above and below the band from the neighbours' buffers (distributed shared memory). Alternating
// the buffers makes one barrier per step enough: a CTA writes a buffer again two steps later, after a barrier that every
// reader of its previous contents has passed. importance_{t+1} is loaded while step t waits at its barrier.
template <int CPT>
__global__ void __launch_bounds__(1024) display_sequence_kernel(const float *__restrict__ importance, int steps, int n, int oh,
                                                                int ow, int band, float *__restrict__ energy,
                                                                float exhaustion_max, float excitation_max, int recovery_mode,
                                                                float normer, float centerer, float *__restrict__ fired_disp,
                                                                float *__restrict__ update_disp)
{
    extern __shared__ float biased_bufs[];   // [2][band * ow]
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank(), C = (int)cluster.num_blocks();
    const int e = (int)blockIdx.x / C, y0 = rank * band;
    const int rows = max(0, min(band, oh - y0)), cells = rows * ow;
    const size_t plane = (size_t)oh * ow, band_off = (size_t)y0 * ow;
    // the rows just outside the band: the last row of rank - 1's band and the first of rank + 1's, in both buffers
    const size_t buf = (size_t)band * ow;
    const float *above = rank > 0 ? cluster.map_shared_rank(biased_bufs, rank - 1) + buf - ow : nullptr;
    const float *below = rank + 1 < C ? cluster.map_shared_rank(biased_bufs, rank + 1) : nullptr;
    float en[CPT], imp[CPT];
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int c = (int)threadIdx.x + k * (int)blockDim.x;
        if (c < cells) {
            en[k] = energy[(size_t)e * plane + band_off + c];
            imp[k] = __ldg(importance + (size_t)e * plane + band_off + c);
        }
    }
    for (int t = 0; t < steps; ++t) {
        const size_t odd = (t & 1) ? buf : 0;
        float *B = biased_bufs + odd;
        const size_t img = (size_t)t * n + e;
        float cur[CPT];
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const int c = (int)threadIdx.x + k * (int)blockDim.x;
            if (c < cells) {
                cur[k] = imp[k];
                B[c] = canon_pow(cur[k], en[k]);                                   // boosting.py:17
                if (t + 1 < steps) imp[k] = __ldg(importance + (img + n) * plane + band_off + c);
            }
        }
        cluster.sync();
        const float *up = above + odd, *down = below + odd;
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const int c = (int)threadIdx.x + k * (int)blockDim.x;
            if (c < cells) {
                const int ly = c / ow, x = c - ly * ow;
                const float m = window_max3(
                    [&](int yy, int xx) {
                        const int r = yy - y0;
                        return (r < 0 ? up[xx] : (r >= rows ? down[xx] : B[r * ow + xx]));
                    },
                    y0 + ly, x, oh, ow);
                en[k] = display_cell(B[c], m, cur[k], en[k], exhaustion_max, excitation_max, recovery_mode, normer,
                                     centerer, img * plane + band_off + c, fired_disp, update_disp);
            }
        }
    }
    cluster.sync();   // no CTA leaves while a neighbour may still read its shared memory
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int c = (int)threadIdx.x + k * (int)blockDim.x;
        if (c < cells) energy[(size_t)e * plane + band_off + c] = en[k];
    }
}

static unsigned blocks_for(size_t count) { return (unsigned)((count + 255) / 256); }

static DisplayGeom display_geom(int n, int h, int w, int region_h, int region_w, int half_h, int half_w)
{
    DisplayGeom G;
    G.n = n, G.h = h, G.w = w, G.rh = region_h, G.rw = region_w, G.h2 = half_h, G.w2 = half_w;
    same_geometry(h, region_h, region_h, &G.oh, &G.pt);
    same_geometry(w, region_w, region_w, &G.ow, &G.pl);
    same_geometry(half_h, region_h, region_h, &G.oh2, &G.pt2);
    same_geometry(half_w, region_w, region_w, &G.ow2, &G.pl2);
    G.by = nearest_scale(G.oh, h), G.bx = nearest_scale(G.ow, w);
    G.by2 = nearest_scale(G.oh2, half_h), G.bx2 = nearest_scale(G.ow2, half_w);
    G.ry = nearest_scale(h, half_h), G.rx = nearest_scale(w, half_w);
    return G;
}

// launch shape of display_sequence_kernel: C CTAs per slice of `band` block rows each, `threads` threads of CPT cells
struct SequenceShape {
    int C, band, cpt, threads;
    size_t smem;
    void (*kernel)(const float *, int, int, int, int, int, float *, float, float, int, float, float, float *, float *);
};

// a CTA holds at most kSeqMaxThreads * kSeqMaxCpt cells of its band: 2 x 32 KB of biased buffers, 8 energies per thread
constexpr int kSeqMaxThreads = 1024, kSeqMaxCpt = 8, kSeqMaxCluster = 16;

static bool sequence_shape(int C, int oh, int ow, SequenceShape *S)
{
    S->C = C;
    S->band = ceil_div(oh, C);
    const long long cells = (long long)S->band * ow;
    if (cells > (long long)kSeqMaxCpt * kSeqMaxThreads) return false;
    S->cpt = 1;
    while (cells > (long long)S->cpt * kSeqMaxThreads) S->cpt *= 2;
    S->threads = (ceil_div((int)cells, S->cpt) + 31) / 32 * 32;
    S->smem = (size_t)2 * cells * sizeof(float);
    S->kernel = S->cpt == 1 ? display_sequence_kernel<1>
                : S->cpt == 2 ? display_sequence_kernel<2>
                : S->cpt == 4 ? display_sequence_kernel<4>
                              : display_sequence_kernel<8>;
    return true;
}

static cudaLaunchConfig_t sequence_config(const SequenceShape &S, int n, cudaStream_t stream, cudaLaunchAttribute *attr)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n * S.C));
    cfg.blockDim = dim3((unsigned)S.threads);
    cfg.dynamicSmemBytes = S.smem;
    cfg.stream = stream;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S.C;
    attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

// The cluster size of a clip of n slices on an oh x ow grid, 0 when no cluster holds a slice (the per-step fallback).
// Among the sizes whose band fits a CTA (1 ... 16, at most one CTA per block row) it takes the largest that keeps the n
// clusters within one CTA per SM, so a few slices still spread over many SMs and many slices do not queue in waves; the
// recurrence is a chain of dependent steps, and a smaller band is a shorter step. Sizes above 8 are non-portable, and a
// size the device cannot co-schedule (cudaOccupancyMaxActiveClusters = 0) gives way to the next smaller one.
static int choose_sequence_shape(int n, int oh, int ow, cudaStream_t stream, SequenceShape *out)
{
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return -1;
    int smallest = 0, chosen = 0;
    for (int C = 1; C <= kSeqMaxCluster && C <= oh; C *= 2) {
        SequenceShape S;
        if (!sequence_shape(C, oh, ow, &S)) continue;
        if (!smallest) smallest = C;
        if ((long long)n * C <= sms) chosen = C;
    }
    if (!smallest) return 0;
    if (!chosen) chosen = smallest;
    for (int C = chosen; C >= smallest; C /= 2) {
        SequenceShape S;
        if (!sequence_shape(C, oh, ow, &S)) break;
        if (cudaFuncSetAttribute(S.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.smem) != cudaSuccess ||
            cudaFuncSetAttribute(S.kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess)
            return -1;
        cudaLaunchAttribute attr[1];
        cudaLaunchConfig_t cfg = sequence_config(S, n, stream, attr);
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, S.kernel, &cfg) != cudaSuccess) {
            (void)cudaGetLastError();   // a size the device rejects outright: try the next smaller one
            continue;
        }
        if (clusters > 0) {
            *out = S;
            return C;
        }
    }
    return 0;
}

}  // namespace silent

using namespace silent;

extern "C" {

int silent_get_centroids(const float *value_dev, int n, int h, int w, int region_h, int region_w, float *corrected_dev,
                         float *total_dev, float *centroids_dev, silent_stream stream)
{
    if (!value_dev || !corrected_dev || !total_dev) return fail(SILENT_E_INVAL, "silent_get_centroids: null argument");
    if (n <= 0 || h <= 0 || w <= 0 || region_h <= 0 || region_w <= 0)
        return fail(SILENT_E_INVAL, "silent_get_centroids: bad shape %dx%dx%d region %dx%d", n, h, w, region_h, region_w);
    int oh, ow, pt, pl;
    same_geometry(h, region_h, region_h, &oh, &pt);
    same_geometry(w, region_w, region_w, &ow, &pl);
    cudaStream_t s = (cudaStream_t)stream;
    centroid_blocks_kernel<<<blocks_for((size_t)n * oh * ow), 256, 0, s>>>(value_dev, n, h, w, region_h, region_w, oh, ow,
                                                                           pt, pl, corrected_dev, total_dev);
    SILENT_LAUNCH_CHECK("centroid_blocks_kernel");
    if (centroids_dev) {
        centroid_distance_kernel<<<blocks_for((size_t)n * h * w), 256, 0, s>>>(corrected_dev, n, h, w, oh, ow,
                                                                              nearest_scale(oh, h), nearest_scale(ow, w),
                                                                              centroids_dev);
        SILENT_LAUNCH_CHECK("centroid_distance_kernel");
    }
    return SILENT_OK;
}

int silent_resize_nearest(const float *x_dev, int n, int h, int w, int c, int out_h, int out_w, float *out_dev,
                          silent_stream stream)
{
    if (!x_dev || !out_dev) return fail(SILENT_E_INVAL, "silent_resize_nearest: null argument");
    if (n <= 0 || h <= 0 || w <= 0 || c <= 0 || out_h <= 0 || out_w <= 0)
        return fail(SILENT_E_INVAL, "silent_resize_nearest: bad shape");
    resize_nearest_kernel<<<blocks_for((size_t)n * out_h * out_w * c), 256, 0, (cudaStream_t)stream>>>(
        x_dev, n, h, w, c, out_h, out_w, nearest_scale(h, out_h), nearest_scale(w, out_w), out_dev);
    SILENT_LAUNCH_CHECK("resize_nearest_kernel");
    return SILENT_OK;
}

int silent_get_boosting(const float *input_dev, float *energy_dev, int n, int h, int w, float exhaustion_max,
                        float excitation_max, int recovery_mode, float *fired_dev, float *scratch_dev,
                        silent_stream stream)
{
    if (!input_dev || !energy_dev || !fired_dev || !scratch_dev)
        return fail(SILENT_E_INVAL, "silent_get_boosting: null argument");
    if (n <= 0 || h <= 0 || w <= 0) return fail(SILENT_E_INVAL, "silent_get_boosting: bad shape %dx%dx%d", n, h, w);
    if (recovery_mode < 1 || recovery_mode > 3)
        return fail(SILENT_E_INVAL, "You must choose a type of recovery");   /* recovery.py:21 */
    const size_t count = (size_t)n * h * w;
    cudaStream_t s = (cudaStream_t)stream;
    boosting_bias_kernel<<<blocks_for(count), 256, 0, s>>>(input_dev, energy_dev, count, scratch_dev);
    SILENT_LAUNCH_CHECK("boosting_bias_kernel");
    boosting_update_kernel<<<blocks_for(count), 256, 0, s>>>(input_dev, scratch_dev, energy_dev, n, h, w, exhaustion_max,
                                                            excitation_max, recovery_mode, fired_dev);
    SILENT_LAUNCH_CHECK("boosting_update_kernel");
    return SILENT_OK;
}

int silent_display_tensors(const float *gray_dev, int n, int h, int w, int region_h, int region_w, int half_h, int half_w,
                           float *energy_dev, float exhaustion_max, float excitation_max, int recovery_mode, float normer,
                           float centerer, float *centroids_disp_dev, float *centroids2_disp_dev, float *fired_disp_dev,
                           float *update_disp_dev, float *scratch_dev, silent_stream stream)
{
    if (!gray_dev || !energy_dev || !centroids_disp_dev || !centroids2_disp_dev || !fired_disp_dev || !update_disp_dev ||
        !scratch_dev)
        return fail(SILENT_E_INVAL, "silent_display_tensors: null argument");
    if (n <= 0 || h <= 0 || w <= 0 || region_h <= 0 || region_w <= 0 || half_h <= 0 || half_w <= 0)
        return fail(SILENT_E_INVAL, "silent_display_tensors: bad shape %dx%dx%d region %dx%d half %dx%d", n, h, w, region_h,
                    region_w, half_h, half_w);
    if (recovery_mode < 1 || recovery_mode > 3)
        return fail(SILENT_E_INVAL, "You must choose a type of recovery");   /* recovery.py:21 */
    const DisplayGeom G = display_geom(n, h, w, region_h, region_w, half_h, half_w);
    const size_t blocks = (size_t)n * G.oh * G.ow;
    float *importance = scratch_dev, *biased = scratch_dev + blocks;
    cudaStream_t s = (cudaStream_t)stream;
    display_centroids_kernel<true><<<blocks_for((size_t)n * h * w + (size_t)n * half_h * half_w + blocks), 256, 0, s>>>(
        gray_dev, G, energy_dev, centroids_disp_dev, centroids2_disp_dev, importance, biased);
    SILENT_LAUNCH_CHECK("display_centroids_kernel");
    display_boosting_kernel<<<blocks_for(blocks), 256, 0, s>>>(importance, biased, energy_dev, n, G.oh, G.ow, exhaustion_max,
                                                               excitation_max, recovery_mode, normer, centerer,
                                                               fired_disp_dev, update_disp_dev);
    SILENT_LAUNCH_CHECK("display_boosting_kernel");
    return SILENT_OK;
}

size_t silent_display_sequence_scratch_bytes(int steps, int n, int h, int w, int region_h, int region_w)
{
    if (steps <= 0 || n <= 0 || h <= 0 || w <= 0 || region_h <= 0 || region_w <= 0) return 0;
    const size_t plane = (size_t)ceil_div(h, region_h) * ceil_div(w, region_w);
    return ((size_t)steps * n + n) * plane * sizeof(float);   // importance of every step + one step of the fallback's bias
}

int silent_display_sequence(const float *gray_dev, int steps, int n, int h, int w, int region_h, int region_w,
                            int half_h, int half_w, float *energy_dev, float exhaustion_max, float excitation_max,
                            int recovery_mode, float normer, float centerer, float *centroids_disp_dev,
                            float *centroids2_disp_dev, float *fired_disp_dev, float *update_disp_dev, void *scratch_dev,
                            size_t scratch_bytes, silent_stream stream)
{
    if (!gray_dev || !energy_dev || !centroids_disp_dev || !centroids2_disp_dev || !fired_disp_dev || !update_disp_dev ||
        !scratch_dev)
        return fail(SILENT_E_INVAL, "silent_display_sequence: null argument");
    if (steps <= 0 || n <= 0 || h <= 0 || w <= 0 || region_h <= 0 || region_w <= 0 || half_h <= 0 || half_w <= 0)
        return fail(SILENT_E_INVAL, "silent_display_sequence: bad shape %d steps of %dx%dx%d region %dx%d half %dx%d",
                    steps, n, h, w, region_h, region_w, half_h, half_w);
    if ((long long)steps * n > INT_MAX)
        return fail(SILENT_E_INVAL, "silent_display_sequence: %d steps of %d images is too many", steps, n);
    const size_t need = silent_display_sequence_scratch_bytes(steps, n, h, w, region_h, region_w);
    if (scratch_bytes < need)
        return fail(SILENT_E_INVAL, "silent_display_sequence: scratch of %zu bytes, needs %zu", scratch_bytes, need);
    if (recovery_mode < 1 || recovery_mode > 3)
        return fail(SILENT_E_INVAL, "You must choose a type of recovery");   /* recovery.py:21 */
    const DisplayGeom G = display_geom(steps * n, h, w, region_h, region_w, half_h, half_w);
    const size_t plane = (size_t)G.oh * G.ow, blocks = (size_t)steps * n * plane;
    float *importance = static_cast<float *>(scratch_dev), *biased = importance + blocks;
    cudaStream_t s = (cudaStream_t)stream;
    // every step's centroid images and importance at once: they depend on gray only
    display_centroids_kernel<false><<<blocks_for((size_t)G.n * h * w + (size_t)G.n * half_h * half_w + blocks), 256, 0, s>>>(
        gray_dev, G, nullptr, centroids_disp_dev, centroids2_disp_dev, importance, nullptr);
    SILENT_LAUNCH_CHECK("display_centroids_kernel");
    SequenceShape S;
    const int C = choose_sequence_shape(n, G.oh, G.ow, s, &S);
    if (C < 0)
        return fail(SILENT_E_CUDA, "silent_display_sequence: cluster set-up failed: %s",
                    cudaGetErrorString(cudaGetLastError()));
    if (C > 0) {
        cudaLaunchAttribute attr[1];
        const cudaLaunchConfig_t cfg = sequence_config(S, n, s, attr);
        SILENT_CUDA(cudaLaunchKernelEx(&cfg, S.kernel, (const float *)importance, steps, n, G.oh, G.ow, S.band, energy_dev,
                                       exhaustion_max, excitation_max, recovery_mode, normer, centerer, fired_disp_dev,
                                       update_disp_dev));
        SILENT_LAUNCH_CHECK("display_sequence_kernel");
        return SILENT_OK;
    }
    // no cluster holds a slice of this grid: the two launches of silent_display_tensors' boosting half, step by step
    const size_t count = (size_t)n * plane;
    for (int t = 0; t < steps; ++t) {
        const float *imp = importance + (size_t)t * count;
        boosting_bias_kernel<<<blocks_for(count), 256, 0, s>>>(imp, energy_dev, count, biased);
        SILENT_LAUNCH_CHECK("boosting_bias_kernel");
        display_boosting_kernel<<<blocks_for(count), 256, 0, s>>>(imp, biased, energy_dev, n, G.oh, G.ow, exhaustion_max,
                                                                  excitation_max, recovery_mode, normer, centerer,
                                                                  fired_disp_dev + 3 * (size_t)t * count,
                                                                  update_disp_dev + 3 * (size_t)t * count);
        SILENT_LAUNCH_CHECK("display_boosting_kernel");
    }
    return SILENT_OK;
}

int silent_pack_points(const int64_t *points_dev, const int64_t *count_dev, int64_t capacity, int64_t level_offset,
                       int64_t *packed_dev, silent_stream stream)
{
    if (!points_dev || !count_dev || !packed_dev) return fail(SILENT_E_INVAL, "silent_pack_points: null argument");
    if (capacity <= 0) return fail(SILENT_E_INVAL, "silent_pack_points: capacity must be positive");
    pack_points_kernel<<<blocks_for((size_t)capacity + 1), 256, 0, (cudaStream_t)stream>>>(
        (const long long *)points_dev, (const long long *)count_dev, (long long)capacity, (long long)level_offset,
        (long long *)packed_dev);
    SILENT_LAUNCH_CHECK("pack_points_kernel");
    return SILENT_OK;
}

int silent_pointwise(const float *x_dev, const float *y_dev, size_t count, int kind, float *out_dev, silent_stream stream)
{
    if (!x_dev || !out_dev) return fail(SILENT_E_INVAL, "silent_pointwise: null argument");
    if (kind < SILENT_PW_DIV255 || kind > SILENT_PW_PRODUCT) return fail(SILENT_E_INVAL, "silent_pointwise: bad kind %d", kind);
    if (kind == SILENT_PW_PRODUCT && !y_dev) return fail(SILENT_E_INVAL, "silent_pointwise: product needs two inputs");
    if (count == 0) return SILENT_OK;
    pointwise_kernel<<<blocks_for(count), 256, 0, (cudaStream_t)stream>>>(x_dev, y_dev, count, kind, out_dev);
    SILENT_LAUNCH_CHECK("pointwise_kernel");
    return SILENT_OK;
}

}  // extern "C"
