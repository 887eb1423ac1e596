// K3: feature-point emit = max_value_indices_region (reference util/selection/top_value_points.py:32-45) and the
// top-percent mask top_value_points (:8-29).
//
// max_value_indices_region: max-pool with ksize = whole level and stride = region (SAME) -> NN-upsample -> value >= up
// -> tf.where. Here: (1) per-window maxima (NaN-propagating; reduced inside stack_b on the fused path), (2) per-row hit
// counts, (3) exclusive scan over the rows of each level, (4) ordered warp-ballot compaction (a hit row adds up the
// totals of the levels before it), so the int64 rows (level, y, x, 0) come out in tf.where's row-major order.
#include "plan.h"
#include "stack.h"

namespace silent {

struct PoolGeom {
    int oh, ow;          // pooled grid
    int pt, pl;          // SAME pad before
    float sy, sx;        // float32(in / out) of the NN upsample, in = pooled, out = level
};

static PoolGeom pool_geometry(int h, int w, int region_h, int region_w)
{
    PoolGeom g;
    g.oh = ceil_div(h, region_h);
    g.ow = ceil_div(w, region_w);
    int total_h = (g.oh - 1) * region_h + h - h, total_w = (g.ow - 1) * region_w + w - w;   // ksize = (h, w)
    g.pt = (total_h > 0 ? total_h : 0) / 2;
    g.pl = (total_w > 0 ? total_w : 0) / 2;
    g.sy = (float)((double)g.oh / (double)h);
    g.sx = (float)((double)g.ow / (double)w);
    return g;
}

__device__ __forceinline__ int nearest_src(int dst, float scale, int n_in)
{
    const int src = (int)floorf((float)dst * scale);
    return src < n_in - 1 ? src : n_in - 1;
}

constexpr float kNegInf = -INFINITY;

// grid (oh*ow, n, row slices): a CTA reduces one slice of the rows of one window of one level (the windows of the
// reference's max_pool span the WHOLE level, so one CTA per window walked 55 k pixels on its own: 62 us for a 1080p frame).
// Warps take rows, lanes take columns: independent loads, no index division. The slices meet in `pooled` (preset to
// 0xffffffff, which loses against every float below) through an order-independent NaN-propagating float maximum: signed
// atomicMax for values >= +0, unsigned atomicMin for negative ones, and NaN (0x7fc00000, above every finite or infinite
// pattern in both orders) through the signed atomicMax.
__global__ void __launch_bounds__(256) window_max_kernel(const float *__restrict__ value, int h, int w, int region_h,
                                                         int region_w, PoolGeom g, float *__restrict__ pooled)
{
    const int win = blockIdx.x, n = blockIdx.y;
    const int i = win / g.ow, j = win % g.ow;
    int ya = i * region_h - g.pt, yb = ya + h, xa = j * region_w - g.pl, xb = xa + w;
    ya = max(ya, 0), xa = max(xa, 0), yb = min(yb, h), xb = min(xb, w);
    const int per = ((yb - ya) + (int)gridDim.z - 1) / (int)gridDim.z;
    const int y0 = ya + (int)blockIdx.z * per, y1 = min(yb, y0 + per);
    const float *v = value + (size_t)n * h * w;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float best = kNegInf;
    int seen_nan = 0, seen_any = 0;
    for (int y = y0 + warp; y < y1; y += 8) {
        const float *row = v + (size_t)y * w;
#pragma unroll 4
        for (int x = xa + lane; x < xb; x += 32) {
            const float f = __ldg(row + x);
            seen_any = 1;
            if (f != f) seen_nan = 1;
            else if (f > best) best = f;
        }
    }
    __shared__ float s_best[8];
    __shared__ int s_nan[8], s_any[8];
    for (int o = 16; o > 0; o >>= 1) {
        best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));   // no NaN reaches here
        seen_nan |= __shfl_xor_sync(0xffffffffu, seen_nan, o);
        seen_any |= __shfl_xor_sync(0xffffffffu, seen_any, o);
    }
    if (lane == 0) s_best[warp] = best, s_nan[warp] = seen_nan, s_any[warp] = seen_any;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < (int)(blockDim.x >> 5); ++k) best = fmaxf(best, s_best[k]), seen_nan |= s_nan[k], seen_any |= s_any[k];
        if (!seen_any) return;   // an empty slice
        int *dst = reinterpret_cast<int *>(pooled + (size_t)n * g.oh * g.ow + win);
        if (seen_nan) atomicMax(dst, 0x7fc00000);
        else if (!(__float_as_int(best) < 0)) atomicMax(dst, __float_as_int(best));
        else atomicMin(reinterpret_cast<unsigned int *>(dst), __float_as_uint(best));
    }
}

// One warp per row (level, y). Pass 0 counts hits, pass 1 writes them at row_offset in x order.
// COUNT pass: one warp per row (level, y); 128-bit loads when the row length and the tensor's address allow (a contiguous
// caller tensor may start 4 bytes past a 16-byte boundary); writes the row's hit count.
__global__ void __launch_bounds__(256) count_rows_kernel(const float *__restrict__ value, int rows, int h, int w, PoolGeom g,
                                                         const float *__restrict__ pooled, int *__restrict__ row_count)
{
    pdl_enter();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const int n = row / h, y = row - n * h;
    const float *v = value + (size_t)row * w;
    const float *pool_row = pooled + ((size_t)n * g.oh + nearest_src(y, g.sy, g.oh)) * g.ow;
    int hits = 0;
    if ((w & 3) == 0 && (reinterpret_cast<uintptr_t>(value) & 15) == 0) {
        for (int q = lane; q < (w >> 2); q += 32) {
            const float4 f = __ldg(reinterpret_cast<const float4 *>(v) + q);
            const int x = 4 * q;
            hits += (f.x >= __ldg(pool_row + nearest_src(x, g.sx, g.ow))) + (f.y >= __ldg(pool_row + nearest_src(x + 1, g.sx, g.ow))) +
                    (f.z >= __ldg(pool_row + nearest_src(x + 2, g.sx, g.ow))) + (f.w >= __ldg(pool_row + nearest_src(x + 3, g.sx, g.ow)));
        }
    } else {
        for (int x = lane; x < w; x += 32) hits += __ldg(v + x) >= __ldg(pool_row + nearest_src(x, g.sx, g.ow));
    }
    hits = __reduce_add_sync(0xffffffffu, hits);
    if (lane == 0) row_count[row] = hits;
}

// One CTA per level: exclusive scan of the level's row counts -> row_offset (within the level, in place) + level_total.
__global__ void __launch_bounds__(256) scan_level_kernel(int *__restrict__ row_count, int h, int *__restrict__ level_total)
{
    pdl_enter();
    __shared__ int s_warp[8];
    __shared__ int s_carry;
    int *rows = row_count + (size_t)blockIdx.x * h;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < h; base += 256) {
        const int i = base + threadIdx.x;
        const int mine = i < h ? rows[i] : 0;
        int incl = mine;
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int before = s_carry + incl - mine;
        for (int k = 0; k < warp; ++k) before += s_warp[k];
        if (i < h) rows[i] = before | (mine ? 0x40000000 : 0);   // bit 30 flags rows that have hits (counts < 2^30)
        __syncthreads();
        if (threadIdx.x == 255) s_carry = before + mine;
        __syncthreads();
    }
    if (threadIdx.x == 0) level_total[blockIdx.x] = s_carry;
}

// WRITE pass: one warp per row; rows without hits (the vast majority) return at once. A row WITH hits first adds up the
// totals of the levels before its own (a warp-wide sum of at most a few hundred ints: cheaper than a separate scan
// launch) and then writes its hits in x order at that base + row_offset[row], i.e. in tf.where's row-major order.
// Warp 0 of block 0 also publishes the grand total.
__global__ void __launch_bounds__(256) write_rows_kernel(const float *__restrict__ value, int rows, int h, int w, PoolGeom g,
                                                         const float *__restrict__ pooled, const int *__restrict__ row_offset,
                                                         const int *__restrict__ level_total, int levels,
                                                         long long *__restrict__ points, long long capacity,
                                                         long long *__restrict__ total)
{
    pdl_enter();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row == 0) {
        long long sum = 0;
        for (int k = lane; k < levels; k += 32) sum += __ldg(level_total + k);
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) *total = sum;
    }
    if (row >= rows || capacity <= 0) return;
    const int packed = __ldg(row_offset + row);
    if (!(packed & 0x40000000)) return;
    const int n = row / h, y = row - n * h;
    long long before = 0;
    for (int k = lane; k < n; k += 32) before += __ldg(level_total + k);
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    const float *v = value + (size_t)row * w;
    const float *pool_row = pooled + ((size_t)n * g.oh + nearest_src(y, g.sy, g.oh)) * g.ow;
    long long base = before + (packed & 0x3fffffff);
    for (int x0 = 0; x0 < w; x0 += 32) {
        const int x = x0 + lane;
        bool hit = false;
        if (x < w) hit = __ldg(v + x) >= __ldg(pool_row + nearest_src(x, g.sx, g.ow));
        const unsigned ballot = __ballot_sync(0xffffffffu, hit);
        if (hit) {
            const long long slot = base + __popc(ballot & ((1u << lane) - 1u));
            if (slot < capacity) {
                longlong2 a = make_longlong2(n, y), b = make_longlong2(x, 0);
                reinterpret_cast<longlong2 *>(points)[slot * 2] = a;
                reinterpret_cast<longlong2 *>(points)[slot * 2 + 1] = b;
            }
        }
        base += __popc(ballot);
    }
}

// ---- fused path: per-tile maxima are available (stack_b_kernel), so a level is ONE CTA --------------------------------
// Only tiles whose maximum reaches the region maximum they are compared with can hold a hit (a handful per level on
// generic input; every tile of an all-zero level). emit_count_kernel flags those tiles, scans each flagged tile with the
// whole CTA (one 128-bit load per thread and round, all independent: a level costs about two memory round trips) and
// scans the row counts; emit_write_kernel adds up the totals of the levels before its own and lets one warp per row
// WITH hits write them in x order, so the int64 rows (level, y, x, 0) come out in tf.where's row-major order. Two
// launches of n CTAs instead of three launches of n * h / 8.
constexpr int kEmitMaxTiles = 1024;   // tiles per level the one-CTA path handles (else the row kernels run)
constexpr int kEmitMaxRows = 2048;    // rows per level (shared-memory row counters)

__device__ __forceinline__ bool tile_is_candidate(const TileMaxima &tm, const int *__restrict__ level_tiles, int ty, int tx,
                                                  int h, int w, const PoolGeom &g, const float *__restrict__ level_pool)
{
    const int x0 = tx * tm.tile_w, x1 = min(w, x0 + tm.tile_w) - 1;
    const int y0 = ty * tm.tile_h, y1 = min(h, y0 + tm.tile_h) - 1;
    const int best = __ldg(level_tiles + ty * tm.ntx + tx);
    bool cand = best == 0x7fc00000;   // a NaN somewhere in the tile: let the exact comparison decide
    const float bf = __int_as_float(best);
    for (int i = nearest_src(y0, g.sy, g.oh); i <= nearest_src(y1, g.sy, g.oh); ++i)
        for (int j = nearest_src(x0, g.sx, g.ow); j <= nearest_src(x1, g.sx, g.ow); ++j)
            cand |= bf >= __ldg(level_pool + i * g.ow + j);
    return cand;
}

constexpr int kEmitCompact = 64;   // a level with at most this many hits hands their coordinates to emit_write_kernel

__global__ void __launch_bounds__(256) emit_count_kernel(const float *__restrict__ value, int h, int w, PoolGeom g,
                                                         const float *__restrict__ pooled, TileMaxima tm,
                                                         int *__restrict__ row_offset, int *__restrict__ level_total,
                                                         int *__restrict__ level_hits, int *__restrict__ level_compact)
{
    pdl_enter();
    __shared__ int s_rows[kEmitMaxRows];
    __shared__ unsigned char s_flag[kEmitMaxTiles];
    __shared__ int s_warp[8];
    __shared__ int s_carry;
    const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *v = value + (size_t)n * h * w;
    const float *level_pool = pooled + (size_t)n * g.oh * g.ow;
    const int *level_tiles = tm.data + (size_t)n * tm.nty * tm.ntx;
    const int ntiles = tm.nty * tm.ntx;
    for (int y = tid; y < h; y += 256) s_rows[y] = 0;
    if (tid == 0) s_carry = 0;
    for (int t = tid; t < ntiles; t += 256)
        s_flag[t] = tile_is_candidate(tm, level_tiles, t / tm.ntx, t % tm.ntx, h, w, g, level_pool);
    __syncthreads();
    // compact list of the flagged tiles (order is irrelevant for counting), then ONE flat loop over (flagged tile, quad):
    // a thread's loads are independent of each other, so the level costs about one memory round trip however many tiles
    // are flagged (a loop per tile cost one round trip per flagged tile)
    __shared__ int s_list[kEmitMaxTiles];
    __shared__ int s_nflag;
    // The hits themselves, (y << 16 | x), while there are at most kEmitCompact of them: sorted below and left for
    // emit_write_kernel, which then needs neither the tile flags nor a second look at the pixels (two memory round trips)
    __shared__ int s_hit[kEmitCompact], s_nhit;
    const bool keep_hits = level_hits && w <= 65535;
    if (tid == 0) s_nflag = 0, s_nhit = 0;
    __syncthreads();
    for (int t = tid; t < ntiles; t += 256)
        if (s_flag[t]) s_list[atomicAdd(&s_nflag, 1)] = t;
    __syncthreads();
    const int quads = (tm.tile_w + 3) >> 2;
    const bool vec_ok = (w & 3) == 0 && (tm.tile_w & 3) == 0;
    const int per_tile = tm.tile_h * quads, items = s_nflag * per_tile;
    for (int i0 = tid; i0 < items; i0 += 4 * 256) {
        float4 q[4];
        int xs[4], ys[4], xe[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {   // up to four independent 128-bit loads in flight per thread
            const int i = i0 + u * 256;
            ys[u] = -1;
            if (i >= items) continue;
            const int t = s_list[i / per_tile], rest = i % per_tile;
            const int ty = t / tm.ntx, tx = t - ty * tm.ntx;
            const int r = rest / quads, x = tx * tm.tile_w + 4 * (rest - r * quads), y = ty * tm.tile_h + r;
            if (y >= h || x >= w) continue;
            ys[u] = y, xs[u] = x, xe[u] = min(w, tx * tm.tile_w + tm.tile_w);
            const float *src = v + (size_t)y * w + x;
            if (vec_ok && x + 4 <= w) {
                q[u] = __ldg(reinterpret_cast<const float4 *>(src));
            } else {
                q[u].x = __ldg(src);
                q[u].y = x + 1 < xe[u] ? __ldg(src + 1) : -1.0f;
                q[u].z = x + 2 < xe[u] ? __ldg(src + 2) : -1.0f;
                q[u].w = x + 3 < xe[u] ? __ldg(src + 3) : -1.0f;
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (ys[u] < 0) continue;
            const float *pool_row = level_pool + nearest_src(ys[u], g.sy, g.oh) * g.ow;
            const float f[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
            int hits = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (xs[u] + e < xe[u] && f[e] >= __ldg(pool_row + nearest_src(xs[u] + e, g.sx, g.ow))) {
                    ++hits;
                    if (keep_hits) {
                        const int at = atomicAdd(&s_nhit, 1);
                        if (at < kEmitCompact) s_hit[at] = (ys[u] << 16) | (xs[u] + e);
                    }
                }
            if (hits) atomicAdd(&s_rows[ys[u]], hits);
        }
    }
    __syncthreads();
    for (int base = 0; base < h; base += 256) {
        const int y = base + tid;
        const int mine = y < h ? s_rows[y] : 0;
        int incl = mine;
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int before = s_carry + incl - mine;
        for (int k = 0; k < warp; ++k) before += s_warp[k];
        if (y < h) row_offset[(size_t)n * h + y] = before | (mine ? 0x40000000 : 0);   // bit 30: the row has hits
        __syncthreads();
        if (tid == 255) s_carry = before + mine;
        __syncthreads();
    }
    if (tid == 0) level_total[n] = s_carry;
    if (level_compact) {   // (s_nhit is final since the barrier behind the scan loop)
        const int cnt = s_nhit;
        const bool compact = keep_hits && cnt <= kEmitCompact;
        if (tid == 0) level_compact[n] = compact ? 1 : 0;
        if (compact && tid < cnt) {   // rank sort: the keys are distinct, row-major order = key order
            const int mine = s_hit[tid];
            int rank = 0;
            for (int k = 0; k < cnt; ++k) rank += s_hit[k] < mine;
            level_hits[(size_t)n * kEmitCompact + rank] = mine;
        }
    }
}

__global__ void __launch_bounds__(256) emit_write_kernel(const float *__restrict__ value, int h, int w, PoolGeom g,
                                                         const float *__restrict__ pooled, TileMaxima tm,
                                                         const int *__restrict__ row_offset,
                                                         const int *__restrict__ level_total, int levels,
                                                         long long *__restrict__ points, long long capacity,
                                                         long long *__restrict__ total, const int *__restrict__ level_hits,
                                                         const int *__restrict__ level_compact)
{
    pdl_enter();
    __shared__ long long s_sum[8];
    const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool last = n == levels - 1;
    if (level_compact && __ldg(level_compact + n)) {
        // emit_count_kernel left this level's (few) hits sorted: the totals of the levels before, the own count and the
        // hit list are independent loads, one memory round trip, then the rows are written
        const int cnt = __ldg(level_total + n);
        const int key = tid < cnt ? __ldg(level_hits + (size_t)n * kEmitCompact + tid) : 0;
        if (cnt == 0 && !last) return;
        long long part = 0;
        for (int k = tid; k < n; k += 256) part += __ldg(level_total + k);
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane == 0) s_sum[warp] = part;
        __syncthreads();
        long long base = 0;
        for (int k = 0; k < 8; ++k) base += s_sum[k];
        if (last && tid == 0) *total = base + cnt;
        const long long at = base + tid;
        if (tid < cnt && at < capacity) {
            reinterpret_cast<longlong2 *>(points)[at * 2] = make_longlong2(n, key >> 16);
            reinterpret_cast<longlong2 *>(points)[at * 2 + 1] = make_longlong2(key & 0xffff, 0);
        }
        return;
    }
    // points of the levels before this one (the last level also publishes the grand total); these loads and the row
    // flags below are independent, so they share one memory round trip
    long long sum = 0;
    for (int k = tid; k < n; k += 256) sum += __ldg(level_total + k);
    // the rows of this level that have hits, as a compact list (a warp that walked all rows to find them paid one memory
    // round trip per row: 24 in a row for a 192-row level)
    __shared__ int s_hit_y[kEmitMaxRows], s_hit_off[kEmitMaxRows];
    __shared__ int s_nhit;
    if (tid == 0) s_nhit = 0;
    __syncthreads();
    for (int y = tid; y < h; y += 256) {
        const int packed = __ldg(row_offset + (size_t)n * h + y);
        if (packed & 0x40000000) {
            const int i = atomicAdd(&s_nhit, 1);
            s_hit_y[i] = y, s_hit_off[i] = packed & 0x3fffffff;
        }
    }
    __syncthreads();
    const bool any = s_nhit > 0 && capacity > 0;
    if (!any && !last) return;
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) s_sum[warp] = sum;
    __syncthreads();
    long long before = 0;
    for (int k = 0; k < 8; ++k) before += s_sum[k];
    if (last && tid == 0) *total = before + __ldg(level_total + n);
    if (!any) return;
    const float *level_pool = pooled + (size_t)n * g.oh * g.ow;
    const int *level_tiles = tm.data + (size_t)n * tm.nty * tm.ntx;
    for (int i = warp; i < s_nhit; i += 8) {   // one warp per row with hits
        const int y = s_hit_y[i];
        const float *v = value + ((size_t)n * h + y) * w;
        const float *pool_row = level_pool + nearest_src(y, g.sy, g.oh) * g.ow;
        long long slot = before + s_hit_off[i];
        // the row's tiles are tested by one lane each (their loads overlap), then only flagged tiles are walked in x order
        unsigned flagged = 0;
        for (int t0 = 0; t0 < tm.ntx; t0 += 32) {   // (levels wider than 32 tiles: the walk below re-tests beyond bit 31)
            const int tx = t0 + lane;
            const bool cand = tx < tm.ntx && tile_is_candidate(tm, level_tiles, y / tm.tile_h, tx, h, w, g, level_pool);
            const unsigned b = __ballot_sync(0xffffffffu, cand);
            if (t0 == 0) flagged = b;
        }
        for (int tx = 0; tx < tm.ntx; ++tx) {
            if (tx < 32 ? !((flagged >> tx) & 1u) : !tile_is_candidate(tm, level_tiles, y / tm.tile_h, tx, h, w, g, level_pool))
                continue;
            const int x1 = min(w, (tx + 1) * tm.tile_w);
            for (int xb = tx * tm.tile_w; xb < x1; xb += 32) {
                const int x = xb + lane;
                const bool hit = x < x1 && __ldg(v + x) >= __ldg(pool_row + nearest_src(x, g.sx, g.ow));
                const unsigned ballot = __ballot_sync(0xffffffffu, hit);
                if (hit) {
                    const long long at = slot + __popc(ballot & ((1u << lane) - 1u));
                    if (at < capacity) {
                        reinterpret_cast<longlong2 *>(points)[at * 2] = make_longlong2(n, y);
                        reinterpret_cast<longlong2 *>(points)[at * 2 + 1] = make_longlong2(x, 0);
                    }
                }
                slot += __popc(ballot);
            }
        }
    }
}

// top_value_points: per-level threshold (1-p)*max + p*min with min = -1 * max(-v); NaN in a level poisons its threshold.
__global__ void __launch_bounds__(256) level_threshold_kernel(const float *__restrict__ value, int hw, float keep_max,
                                                              float keep_min, float *__restrict__ thr)
{
    const float *v = value + (size_t)blockIdx.x * hw;
    float mx = kNegInf, mneg = kNegInf;
    int seen_nan = 0;
    for (int t = threadIdx.x; t < hw; t += blockDim.x) {
        const float f = __ldg(v + t);
        if (f != f) seen_nan = 1;
        else {
            if (f > mx) mx = f;
            if (-f > mneg) mneg = -f;
        }
    }
    __shared__ float s_mx[8], s_mn[8];
    __shared__ int s_nan[8];
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mneg = fmaxf(mneg, __shfl_xor_sync(0xffffffffu, mneg, o));
        seen_nan |= __shfl_xor_sync(0xffffffffu, seen_nan, o);
    }
    if ((threadIdx.x & 31) == 0) s_mx[threadIdx.x >> 5] = mx, s_mn[threadIdx.x >> 5] = mneg, s_nan[threadIdx.x >> 5] = seen_nan;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < (int)(blockDim.x >> 5); ++k)
            mx = fmaxf(mx, s_mx[k]), mneg = fmaxf(mneg, s_mn[k]), seen_nan |= s_nan[k];
        const float mn = -1.0f * mneg;
        thr[blockIdx.x] = seen_nan ? __int_as_float(0x7fc00000) : keep_max * mx + keep_min * mn;
    }
}

__global__ void apply_threshold_kernel(const float *__restrict__ color, const float *__restrict__ value,
                                       const float *__restrict__ thr, size_t total, int hw, int c, float *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const size_t pix = i / c;
    const float keep = value[pix] >= thr[pix / hw] ? 1.0f : 0.0f;
    out[i] = color[i] * keep;
}

// ---- peak emit: every 3x3 local maximum of a level above its top-percent threshold -------------------------------------
// Pixel (y, x) of level v fires iff v > 0, v >= thr (level_threshold_kernel) and v >= the NaN-propagating maximum of the
// 3x3 window around it (TF max_pool SAME: neighbours outside the level are ignored). Rows of (level, y, x, 0) in row-major
// order: peak_count_kernel counts each row's hits, scan_level_kernel turns the counts into offsets within the level,
// peak_base_kernel scans the level totals into each level's first row (and the grand total), peak_write_kernel writes
// each row's hits in x order at its level base + row offset. The hit test reads rows y - 1, y and y + 1.

__device__ __forceinline__ float max_nan(float a, float b)
{
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

// V = 4: the run of pixels x .. x + 3 as one 128-bit load (the row length is a multiple of 4 and the tensor 16-byte
// aligned); V = 1: pixel x. Out of the level (row null, or x >= w): -inf, which every comparison below ignores.
template <int V>
__device__ __forceinline__ void load_run(const float *row, int x, int w, float (&f)[V])
{
    if (V == 4) {
        float4 q = make_float4(kNegInf, kNegInf, kNegInf, kNegInf);
        if (row && x < w) q = __ldg(reinterpret_cast<const float4 *>(row + x));
        f[0] = q.x, f[1] = q.y, f[2] = q.z, f[3] = q.w;
    } else {
        f[0] = row && x < w ? __ldg(row + x) : kNegInf;
    }
}

__device__ __forceinline__ float column_max(const float *up, const float *mid, const float *down, int x)
{
    const float a = up ? __ldg(up + x) : kNegInf, c = down ? __ldg(down + x) : kNegInf;
    return max_nan(max_nan(a, __ldg(mid + x)), c);
}

// Hit mask (bit i: pixel x + i) of the lane's run in row `mid`; every lane of the warp calls it (the columns next to the
// run come from the neighbouring lanes; lanes 0 and 31 read theirs). x >= w: no hits.
template <int V>
__device__ __forceinline__ unsigned peak_bits(const float *up, const float *mid, const float *down, int x, int w,
                                              float thr, int lane)
{
    float a[V], v[V], c[V], col[V];
    load_run<V>(up, x, w, a);
    load_run<V>(mid, x, w, v);
    load_run<V>(down, x, w, c);
#pragma unroll
    for (int i = 0; i < V; ++i) col[i] = max_nan(max_nan(a[i], v[i]), c[i]);
    float left = __shfl_up_sync(0xffffffffu, col[V - 1], 1);
    float right = __shfl_down_sync(0xffffffffu, col[0], 1);
    if (lane == 0) left = x > 0 && x < w ? column_max(up, mid, down, x - 1) : kNegInf;
    if (x + V >= w) right = kNegInf;
    else if (lane == 31) right = column_max(up, mid, down, x + V);
    unsigned bits = 0;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const float m = max_nan(max_nan(i == 0 ? left : col[i - 1], col[i]), i == V - 1 ? right : col[i + 1]);
        if (x + i < w && v[i] > 0.0f && v[i] >= thr && v[i] >= m) bits |= 1u << i;
    }
    return bits;
}

struct PeakRow {
    const float *up, *mid, *down;
    float thr;
};

__device__ __forceinline__ PeakRow peak_row(const float *value, int row, int h, int w, const float *thr)
{
    const int n = row / h, y = row - n * h;
    const float *mid = value + (size_t)row * w;
    return PeakRow{y > 0 ? mid - w : nullptr, mid, y + 1 < h ? mid + w : nullptr, __ldg(thr + n)};
}

// COUNT pass: one warp per row (level, y); 128-bit loads under count_rows_kernel's condition; writes the row's hit count.
__global__ void __launch_bounds__(256) peak_count_kernel(const float *__restrict__ value, int rows, int h, int w,
                                                         const float *__restrict__ thr, int *__restrict__ row_count)
{
    pdl_enter();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const PeakRow r = peak_row(value, row, h, w, thr);
    int hits = 0;
    if ((w & 3) == 0 && (reinterpret_cast<uintptr_t>(value) & 15) == 0) {
        for (int x0 = 0; x0 < w; x0 += 128) hits += __popc(peak_bits<4>(r.up, r.mid, r.down, x0 + 4 * lane, w, r.thr, lane));
    } else {
        for (int x0 = 0; x0 < w; x0 += 32) hits += __popc(peak_bits<1>(r.up, r.mid, r.down, x0 + lane, w, r.thr, lane));
    }
    hits = __reduce_add_sync(0xffffffffu, hits);
    if (lane == 0) row_count[row] = hits;
}

// One CTA: exclusive scan of the level totals -> level_base (the first row of each level), and the grand total. Replaces
// write_rows_kernel's per-row sum over the levels before, which dense output (most rows with hits) would pay per row.
__global__ void __launch_bounds__(1024) peak_base_kernel(const int *__restrict__ level_total, int levels,
                                                         long long *__restrict__ level_base, long long *__restrict__ total)
{
    pdl_enter();
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < levels; base += 1024) {
        const int i = base + threadIdx.x;
        const long long mine = i < levels ? __ldg(level_total + i) : 0;
        long long incl = mine;
        for (int o = 1; o < 32; o <<= 1) {
            const long long up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        long long before = s_carry + incl - mine;
        for (int k = 0; k < warp; ++k) before += s_warp[k];
        if (i < levels) level_base[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + mine;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}

// WRITE pass: one warp per row with hits; each lane's hits go at the row's slot + the hits of the lanes before it (a warp
// scan of the per-lane counts), so the rows come out in x order without a pass per hit.
template <int V>
__device__ __forceinline__ void write_peak_row(const PeakRow &r, int n, int y, int w, long long slot, int lane,
                                               long long *__restrict__ points, long long capacity)
{
    for (int x0 = 0; x0 < w; x0 += 32 * V) {
        const int x = x0 + V * lane;
        unsigned bits = peak_bits<V>(r.up, r.mid, r.down, x, w, r.thr, lane);
        const int mine = __popc(bits);
        int incl = mine;
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        long long at = slot + incl - mine;
        while (bits) {
            const int i = __ffs(bits) - 1;
            bits &= bits - 1;
            if (at < capacity) {
                reinterpret_cast<longlong2 *>(points)[at * 2] = make_longlong2(n, y);
                reinterpret_cast<longlong2 *>(points)[at * 2 + 1] = make_longlong2(x + i, 0);
            }
            ++at;
        }
        slot += __shfl_sync(0xffffffffu, incl, 31);
    }
}

__global__ void __launch_bounds__(256) peak_write_kernel(const float *__restrict__ value, int rows, int h, int w,
                                                         const float *__restrict__ thr,
                                                         const int *__restrict__ row_offset,
                                                         const long long *__restrict__ level_base,
                                                         long long *__restrict__ points, long long capacity)
{
    pdl_enter();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows || capacity <= 0) return;
    const int packed = __ldg(row_offset + row);
    if (!(packed & 0x40000000)) return;
    const int n = row / h, y = row - n * h;
    const long long slot = __ldg(level_base + n) + (packed & 0x3fffffff);
    if (slot >= capacity) return;
    const PeakRow r = peak_row(value, row, h, w, thr);
    if ((w & 3) == 0 && (reinterpret_cast<uintptr_t>(value) & 15) == 0) write_peak_row<4>(r, n, y, w, slot, lane, points, capacity);
    else write_peak_row<1>(r, n, y, w, slot, lane, points, capacity);
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

size_t selection_bytes(int n, int h, int w)
{
    const size_t rows = (size_t)n * h;
    (void)w;
    return align_up((size_t)n * 4096 * sizeof(float), 256) + align_up(rows * sizeof(int), 256) +
           align_up((size_t)n * sizeof(long long), 256) + align_up((size_t)n * sizeof(int), 256) + 256;
}

// True when the pooling windows of max_value_indices_region can be reduced inside stack_b_kernel.
bool window_geometry(int h, int w, int region_h, int region_w, WindowGeom *geo)
{
    if (region_h <= 0 || region_w <= 0) return false;
    const PoolGeom g = pool_geometry(h, w, region_h, region_w);
    if (g.oh > 2 || g.ow > 2) return false;
    geo->count = g.oh * g.ow;
    geo->ow = g.ow;
    for (int i = 0; i < g.oh; ++i) {
        const int ya = i * region_h - g.pt;
        geo->y0[i] = ya > 0 ? ya : 0;
        geo->y1[i] = ya + h < h ? ya + h : h;
    }
    for (int j = 0; j < g.ow; ++j) {
        const int xa = j * region_w - g.pl;
        geo->x0[j] = xa > 0 ? xa : 0;
        geo->x1[j] = xa + w < w ? xa + w : w;
        if ((geo->x0[j] % 8) != 0 || (geo->x1[j] % 8 != 0 && geo->x1[j] != w)) return false;
    }
    return true;
}

int max_value_indices_region(const float *value, int n, int h, int w, int region_h, int region_w, int64_t *points,
                             int64_t capacity, int64_t *count, void *workspace, size_t workspace_bytes,
                             const int *fused_winmax, const TileMaxima *tiles, cudaStream_t stream)
{
    if (!value || !count || !workspace || (!points && capacity > 0))
        return fail(SILENT_E_INVAL, "silent_max_value_indices_region: null argument");
    if (n <= 0 || h <= 0 || w <= 0) return fail(SILENT_E_INVAL, "silent_max_value_indices_region: bad shape");
    if (region_h <= 0 || region_w <= 0) return fail(SILENT_E_INVAL, "region shape must be positive");
    if (capacity < 0) return fail(SILENT_E_INVAL, "capacity must be >= 0");
    if (n > 65535) return fail(SILENT_E_SHAPE, "at most 65535 levels per call");
    const PoolGeom g = pool_geometry(h, w, region_h, region_w);
    if (g.oh * g.ow > 4096) return fail(SILENT_E_SHAPE, "too many regions per level (%d x %d)", g.oh, g.ow);
    if (workspace_bytes < selection_bytes(n, h, w))
        return fail(SILENT_E_CAPACITY, "selection workspace too small: %zu < %zu", workspace_bytes,
                    selection_bytes(n, h, w));
    const int rows = n * h;
    char *ws = (char *)workspace;
    float *pooled = (float *)ws;
    ws += align_up((size_t)n * 4096 * sizeof(float), 256);
    int *row_offset = (int *)ws;            // offset of each row within its level
    ws += align_up((size_t)rows * sizeof(int), 256);
    ws += align_up((size_t)n * sizeof(long long), 256);   // (reserved)
    int *level_total = (int *)ws;

    if (fused_winmax) {
        // the stack kernel already reduced the per-region maxima (ordered-int encoding == float bits, NaN = 0x7fc00000)
        pooled = reinterpret_cast<float *>(const_cast<int *>(fused_winmax));
    } else {
        const int slices = std::max(1, std::min(h / 8, 16));   // row slices per window: enough CTAs for one frame's levels
        SILENT_CUDA(cudaMemsetAsync(pooled, 0xff, (size_t)n * g.oh * g.ow * sizeof(float), stream));
        window_max_kernel<<<dim3(g.oh * g.ow, n, slices), 256, 0, stream>>>(value, h, w, region_h, region_w, g, pooled);
        SILENT_LAUNCH_CHECK("window_max_kernel");
    }
    if ((long long)h * w >= (1 << 30)) return fail(SILENT_E_SHAPE, "levels of 2^30 pixels or more are not supported");
    if (tiles && tiles->data && tiles->nty * tiles->ntx <= kEmitMaxTiles && h <= kEmitMaxRows) {
        // fused path: one CTA per level, only the tiles that can hold a hit are scanned
        // the compact hit lists live in the workspace's window-maxima area when the stack kernel delivered the maxima
        // (fused_winmax: that area is unused then), the per-level "compact" marks in the reserved words before level_total
        int *level_hits = fused_winmax ? (int *)workspace : nullptr;
        int *level_compact = fused_winmax ? (int *)((char *)level_total - align_up((size_t)n * sizeof(long long), 256)) : nullptr;
        SILENT_CUDA(launch_dependent(emit_count_kernel, dim3(n), dim3(256), 0, stream, value, h, w, g, (const float *)pooled,
                                     *tiles, row_offset, level_total, level_hits, level_compact));
        SILENT_LAUNCH_CHECK("emit_count_kernel");
        SILENT_CUDA(launch_dependent(emit_write_kernel, dim3(n), dim3(256), 0, stream, value, h, w, g, (const float *)pooled,
                                     *tiles, (const int *)row_offset, (const int *)level_total, n, (long long *)points,
                                     (long long)capacity, (long long *)count, (const int *)level_hits,
                                     (const int *)level_compact));
        SILENT_LAUNCH_CHECK("emit_write_kernel");
        return SILENT_OK;
    }
    const unsigned blocks = (unsigned)ceil_div(rows, 8);
    SILENT_CUDA(launch_dependent(count_rows_kernel, dim3(blocks), dim3(256), 0, stream, value, rows, h, w, g,
                                 (const float *)pooled, row_offset));
    SILENT_LAUNCH_CHECK("count_rows_kernel");
    SILENT_CUDA(launch_dependent(scan_level_kernel, dim3(n), dim3(256), 0, stream, row_offset, h, level_total));
    SILENT_LAUNCH_CHECK("scan_level_kernel");
    // (also when capacity == 0: the kernel publishes the total)
    SILENT_CUDA(launch_dependent(write_rows_kernel, dim3(blocks), dim3(256), 0, stream, value, rows, h, w, g,
                                 (const float *)pooled, (const int *)row_offset, (const int *)level_total, n,
                                 (long long *)points, (long long)capacity, (long long *)count));
    SILENT_LAUNCH_CHECK("write_rows_kernel");
    return SILENT_OK;
}

// Host-side checks of the peak emit's shape and top_percent (`who` prefixes the messages); SILENT_OK or the status.
static int check_peaks(const char *who, int64_t n, int h, int w, double top_percent, int64_t capacity)
{
    if (n <= 0 || h <= 0 || w <= 0) return fail(SILENT_E_INVAL, "%s: bad shape", who);
    if (capacity < 0) return fail(SILENT_E_INVAL, "%s: capacity must be >= 0", who);
    if (!(top_percent >= 0.0 && top_percent <= 1.0))   // (NaN fails both)
        return fail(SILENT_E_INVAL, "%s: top_percent must be in [0, 1], got %g", who, top_percent);
    if (n > 65535) return fail(SILENT_E_SHAPE, "%s: at most 65535 levels per call, got %lld", who, (long long)n);
    if ((long long)h * w >= (1 << 30)) return fail(SILENT_E_SHAPE, "%s: levels of 2^30 pixels or more are not supported", who);
    if (n * h > INT32_MAX - 255) return fail(SILENT_E_SHAPE, "%s: %lld rows are too many for one call", who, (long long)(n * h));
    return SILENT_OK;
}

// The peak emit on checked arguments: level_threshold_kernel, then the four row kernels (programmatic dependent
// launches). Workspace: thr in the window-maxima area, level_base in the reserved words, row_offset and level_total as
// for max_value_indices_region.
static int peak_points(const float *value, int n, int h, int w, double top_percent, int64_t *points, int64_t capacity,
                       int64_t *count, void *workspace, cudaStream_t stream)
{
    const int rows = n * h;
    char *ws = (char *)workspace;
    float *thr = (float *)ws;
    ws += align_up((size_t)n * 4096 * sizeof(float), 256);
    int *row_offset = (int *)ws;
    ws += align_up((size_t)rows * sizeof(int), 256);
    long long *level_base = (long long *)ws;
    ws += align_up((size_t)n * sizeof(long long), 256);
    int *level_total = (int *)ws;
    // the constants of silent_top_value_points: (1.0 - p) and p rounded to float32
    const float keep_max = (float)(1.0 - top_percent), keep_min = (float)top_percent;
    level_threshold_kernel<<<n, 256, 0, stream>>>(value, h * w, keep_max, keep_min, thr);
    SILENT_LAUNCH_CHECK("level_threshold_kernel");
    const unsigned blocks = (unsigned)ceil_div(rows, 8);
    SILENT_CUDA(launch_dependent(peak_count_kernel, dim3(blocks), dim3(256), 0, stream, value, rows, h, w,
                                 (const float *)thr, row_offset));
    SILENT_LAUNCH_CHECK("peak_count_kernel");
    SILENT_CUDA(launch_dependent(scan_level_kernel, dim3(n), dim3(256), 0, stream, row_offset, h, level_total));
    SILENT_LAUNCH_CHECK("scan_level_kernel");
    SILENT_CUDA(launch_dependent(peak_base_kernel, dim3(1), dim3(1024), 0, stream, (const int *)level_total, n, level_base,
                                 (long long *)count));
    SILENT_LAUNCH_CHECK("peak_base_kernel");
    SILENT_CUDA(launch_dependent(peak_write_kernel, dim3(blocks), dim3(256), 0, stream, value, rows, h, w,
                                 (const float *)thr, (const int *)row_offset, (const long long *)level_base,
                                 (long long *)points, (long long)capacity));
    SILENT_LAUNCH_CHECK("peak_write_kernel");
    return SILENT_OK;
}

}  // namespace silent

using namespace silent;

extern "C" {

size_t silent_selection_workspace_bytes(int n, int h, int w)
{
    if (n <= 0 || h <= 0 || w <= 0) return 0;
    return selection_bytes(n, h, w);
}

int silent_max_value_indices_region(const float *value_dev, int n, int h, int w, int region_h, int region_w,
                                    int64_t *points_dev, int64_t capacity, int64_t *count_dev, void *workspace_dev,
                                    size_t workspace_bytes, silent_stream stream)
{
    return max_value_indices_region(value_dev, n, h, w, region_h, region_w, points_dev, capacity, count_dev,
                                    workspace_dev, workspace_bytes, nullptr, nullptr, (cudaStream_t)stream);
}

int silent_peak_points(const float *value_dev, int n, int h, int w, double top_percent, int64_t *points_dev,
                       int64_t capacity, int64_t *count_dev, void *workspace_dev, size_t workspace_bytes,
                       silent_stream stream)
{
    if (!value_dev || !count_dev || !workspace_dev || (!points_dev && capacity > 0))
        return fail(SILENT_E_INVAL, "silent_peak_points: null argument");
    const int rc = check_peaks("silent_peak_points", n, h, w, top_percent, capacity);
    if (rc != SILENT_OK) return rc;
    if (workspace_bytes < selection_bytes(n, h, w))
        return fail(SILENT_E_CAPACITY, "silent_peak_points: selection workspace too small: %zu < %zu", workspace_bytes,
                    selection_bytes(n, h, w));
    return peak_points(value_dev, n, h, w, top_percent, points_dev, capacity, count_dev, workspace_dev,
                       (cudaStream_t)stream);
}

int silent_plan_peak_points(silent_plan *plan, int batch, double top_percent, int64_t *points_dev, int64_t capacity,
                            int64_t *count_dev, silent_stream stream)
{
    if (!plan || !count_dev || (!points_dev && capacity > 0))
        return fail(SILENT_E_INVAL, "silent_plan_peak_points: null argument");
    if (batch <= 0) return fail(SILENT_E_INVAL, "silent_plan_peak_points: batch must be positive");
    if (plan->levels == 0) return fail(SILENT_E_SHAPE, "frame is not larger than the pyramid centre: 0 levels");
    const int rc = check_peaks("silent_plan_peak_points", (int64_t)batch * plan->levels, plan->h, plan->w, top_percent,
                               capacity);
    if (rc != SILENT_OK) return rc;
    if (batch > plan->ws.batch)
        return fail(SILENT_E_CAPACITY, "silent_plan_peak_points: the plan's gray holds %d frames (silent_plan_reserve), "
                    "need %d", plan->ws.batch, batch);
    if (!plan->on_device) return fail(SILENT_E_CUDA, "plan was created without a CUDA device; no CPU fallback exists");
    return peak_points(plan->ws.d_gray, batch * plan->levels, plan->h, plan->w, top_percent, points_dev, capacity,
                       count_dev, plan->ws.d_select, (cudaStream_t)stream);
}

int silent_top_value_points(const float *color_dev, const float *value_dev, int n, int h, int w, int c,
                            double top_percent, float *out_dev, void *workspace_dev, size_t workspace_bytes,
                            silent_stream stream)
{
    if (!color_dev || !value_dev || !out_dev || !workspace_dev)
        return fail(SILENT_E_INVAL, "silent_top_value_points: null argument");
    if (n <= 0 || h <= 0 || w <= 0 || c <= 0) return fail(SILENT_E_INVAL, "silent_top_value_points: bad shape");
    if (workspace_bytes < (size_t)n * sizeof(float)) return fail(SILENT_E_CAPACITY, "selection workspace too small");
    float *thr = (float *)workspace_dev;
    // (1.0 - top_percent) and top_percent are Python floats converted to float32 constants by TF (top_value_points.py:22)
    const float keep_max = (float)(1.0 - top_percent), keep_min = (float)top_percent;
    cudaStream_t s = (cudaStream_t)stream;
    level_threshold_kernel<<<n, 256, 0, s>>>(value_dev, h * w, keep_max, keep_min, thr);
    SILENT_LAUNCH_CHECK("level_threshold_kernel");
    const size_t total = (size_t)n * h * w * c;
    apply_threshold_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(color_dev, value_dev, thr, total, h * w, c,
                                                                            out_dev);
    SILENT_LAUNCH_CHECK("apply_threshold_kernel");
    return SILENT_OK;
}

}  // extern "C"
