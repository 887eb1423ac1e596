// Plan: the geometry of zoom.from_image (reference util/zoom/from_image.py:43-51) and the order-5 spline tap tables
// of scipy.ndimage.zoom(prefilter=False, mode='constant'), computed once on the host in float64 and uploaded.
#include <stdarg.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "plan.h"

namespace silent {

static thread_local char g_error[512] = "";
static std::atomic<long long> g_launches{0};

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int fail(int status, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
    return status;
}

// Quintic cardinal B-spline, evaluated with the same expression tree as oracle/silent_oracle.py:bspline5.
static double bspline5(double x)
{
    x = std::fabs(x);
    const double x2 = x * x;
    if (x < 1.0) return (66 - 60 * x2 + 30 * x2 * x2 - 10 * x2 * x2 * x) / 120.0;
    if (x < 2.0) return (51 + 75 * x - 210 * x2 + 150 * x2 * x - 45 * x2 * x2 + 5 * x2 * x2 * x) / 120.0;
    if (x < 3.0) {
        const double t = 3 - x;
        return t * t * t * t * t / 120.0;
    }
    return 0.0;
}

// One axis of scipy's zoom: cc = o * (n_in - 1) / (n_out - 1); taps floor(cc)-2 .. +3, mirror-reflected; cc outside
// [0, n_in - 1] -> the output sample is cval = 0 (idx[0] = -1 marks it). coord[o] = the sample's frame position
// offset + cc, rounded once to float32 (left NaN where the sample is 0).
static void axis_table(int n_in, int n_out, int n_keep, int offset, int32_t *idx, float *wts, float *coord)
{
    const double factor = n_out > 1 ? (double)(n_in - 1) / (double)(n_out - 1) : 1.0;
    for (int o = 0; o < n_keep; ++o) {
        const double cc = (double)o * factor;
        if (cc < 0 || cc > n_in - 1) continue;
        coord[o] = (float)((double)offset + cc);
        const int base = (int)std::floor(cc) - 2;
        for (int t = 0; t < kTaps; ++t) {
            int src = base + t;
            wts[o * kTaps + t] = (float)bspline5(cc - src);
            if (n_in == 1) {
                src = 0;
            } else {
                const int period = 2 * n_in - 2;
                src %= period;
                if (src < 0) src += period;
                if (src >= n_in) src = period - src;
            }
            idx[o * kTaps + t] = src + offset;
        }
    }
}

static int python_int(double v) { return (int)v; }  // truncation toward zero, like int(float)

}  // namespace silent

using namespace silent;

extern "C" {

int silent_abi_version(void) { return SILENT_ABI_VERSION; }

const char *silent_last_error(void) { return g_error; }

int64_t silent_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int silent_device_count(void)
{
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess) return fail(SILENT_E_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(err));
    return n;
}

int silent_plan_create(const silent_params *p, silent_plan **out_plan)
{
    if (!p || !out_plan) return fail(SILENT_E_INVAL, "silent_plan_create: null argument");
    *out_plan = nullptr;
    if (!(p->scale > 1.0)) return fail(SILENT_E_INVAL, "Scale must be greater than one.");
    if (p->num_colors <= 0) return fail(SILENT_E_INVAL, "Number of colors must be greater than zero.");
    if (p->center_w <= 0 || p->center_h <= 0) return fail(SILENT_E_INVAL, "Each dimension must be larger than zero.");
    if (p->frame_h <= 0 || p->frame_w <= 0 || p->frame_c <= 0)
        return fail(SILENT_E_INVAL, "frame shape must be positive, got %dx%dx%d", p->frame_h, p->frame_w, p->frame_c);
    if (p->num_colors > p->frame_c || p->num_colors > kMaxChannels)
        return fail(SILENT_E_SHAPE, "num_colors=%d must be <= frame channels (%d) and <= %d", p->num_colors, p->frame_c,
                    kMaxChannels);
    if (p->frame_dtype != SILENT_U8 && p->frame_dtype != SILENT_F32 && p->frame_dtype != SILENT_NV12)
        return fail(SILENT_E_INVAL, "frame_dtype must be SILENT_U8, SILENT_F32 or SILENT_NV12");
    const bool nv12 = p->frame_dtype == SILENT_NV12;
    if (nv12 && (p->frame_c != 3 || p->num_colors != 3))
        return fail(SILENT_E_SHAPE, "NV12 frames convert to 3 colours: frame_c and num_colors must be 3, got %d and %d",
                    p->frame_c, p->num_colors);
    if (nv12 && (p->frame_h % 2 || p->frame_w % 2))
        return fail(SILENT_E_SHAPE, "NV12 frames need even height and width, got %dx%d", p->frame_h, p->frame_w);

    silent_plan *plan = new (std::nothrow) silent_plan();
    if (!plan) return fail(SILENT_E_CAPACITY, "out of host memory");
    plan->params = *p;
    plan->h = p->center_h;
    plan->w = p->center_w;
    plan->frame_pitch = nv12 ? ((int64_t)p->frame_w * 3 + 15) / 16 * 16 : (int64_t)p->frame_w * p->frame_c;
    const int dims_img[2] = {p->frame_h, p->frame_w};
    const int dims_ctr[2] = {p->center_h, p->center_w};

    // num_scales = ceil(max_i log_scale(img_i / center_i))                                   from_image.py:45-46
    double most = -INFINITY;
    for (int a = 0; a < 2; ++a)
        most = std::max(most, std::log((double)dims_img[a] / (double)dims_ctr[a]) / std::log(p->scale));
    const int levels = (int)std::ceil(most);
    plan->levels = levels > 0 ? levels : 0;

    const int L = plan->levels, h = plan->h, w = plan->w;
    plan->info.resize(L);
    plan->idx_y.assign((size_t)L * h * kTaps, -1);
    plan->w_y.assign((size_t)L * h * kTaps, 0.0f);
    plan->idx_x.assign((size_t)L * w * kTaps, -1);
    plan->w_x.assign((size_t)L * w * kTaps, 0.0f);
    plan->coord_y.assign((size_t)L * h, NAN);
    plan->coord_x.assign((size_t)L * w, NAN);
    plan->union_h = plan->union_w = 0;
    for (int s = 0; s < L; ++s) {
        const double grow = std::pow(p->scale, (double)s);    // scale ** s
        LevelInfo &li = plan->info[s];
        int lo[2], hi[2];
        for (int a = 0; a < 2; ++a) {
            const double c = dims_ctr[a] * grow;                                              // from_image.py:49
            lo[a] = python_int(std::max((dims_img[a] - c) / 2, 0.0));                        // from_image.py:50
            hi[a] = python_int((dims_img[a] + c) / 2);
            lo[a] = std::min(lo[a], dims_img[a]);
            hi[a] = std::min(std::max(hi[a], 0), dims_img[a]);
            if (hi[a] < lo[a]) hi[a] = lo[a];
        }
        li.y0 = lo[0], li.y1 = hi[0], li.x0 = lo[1], li.x1 = hi[1];
        const double factor = 1.0 / grow;                                                     // from_image.py:59
        const int out_h = (int)std::nearbyint((li.y1 - li.y0) * factor);   // scipy: int(round(in * zoom)), half-even
        const int out_w = (int)std::nearbyint((li.x1 - li.x0) * factor);
        li.valid_h = std::min(h, std::max(out_h, 0));                                         // from_image.py:61-62
        li.valid_w = std::min(w, std::max(out_w, 0));
        if (li.y1 > li.y0 && li.x1 > li.x0) {
            axis_table(li.y1 - li.y0, out_h, li.valid_h, li.y0, &plan->idx_y[(size_t)s * h * kTaps],
                       &plan->w_y[(size_t)s * h * kTaps], &plan->coord_y[(size_t)s * h]);
            axis_table(li.x1 - li.x0, out_w, li.valid_w, li.x0, &plan->idx_x[(size_t)s * w * kTaps],
                       &plan->w_x[(size_t)s * w * kTaps], &plan->coord_x[(size_t)s * w]);
        } else {
            li.valid_h = li.valid_w = 0;
        }
        plan->union_h = std::max(plan->union_h, li.y1 - li.y0);
        plan->union_w = std::max(plan->union_w, li.x1 - li.x0);
    }

    // NV12: the frame rows and columns any tap reads, rounded out to row pairs and 16-pixel runs (the converter's unit)
    if (nv12) {
        int y0 = p->frame_h, y1 = 0, x0 = p->frame_w, x1 = 0;
        for (size_t o = 0; o < plan->idx_y.size(); o += kTaps)
            if (plan->idx_y[o] >= 0)
                for (int t = 0; t < kTaps; ++t) y0 = std::min(y0, plan->idx_y[o + t]), y1 = std::max(y1, plan->idx_y[o + t] + 1);
        for (size_t o = 0; o < plan->idx_x.size(); o += kTaps)
            if (plan->idx_x[o] >= 0)
                for (int t = 0; t < kTaps; ++t) x0 = std::min(x0, plan->idx_x[o + t]), x1 = std::max(x1, plan->idx_x[o + t] + 1);
        if (y1 > y0 && x1 > x0) {
            plan->nv12_y0 = y0 & ~1, plan->nv12_y1 = std::min(p->frame_h, (y1 + 1) & ~1);
            plan->nv12_x0 = x0 & ~15, plan->nv12_x1 = std::min(p->frame_w, (x1 + 15) & ~15);
        }
    }

    // geometry of the frame-pair pyramid kernel: per level and x tile, the span of frame-row words its x-taps touch
    plan->pair.assign(L, PairLevel());
    // tile width: the widest one (<= 85 columns = 255 phase-H threads) that wastes the fewest columns of the last tile
    // (288-wide levels: 4 x 72 instead of 4.5 x 64, measured -3.5 %)
    int kPairTileW = 64, best_waste = 1 << 30;
    for (int tw = 48; tw <= kPairTileWMax; ++tw) {
        const int waste = ceil_div(w, tw) * tw - w;
        if (waste <= best_waste) best_waste = waste, kPairTileW = tw;
    }
    plan->pair_tile_w = kPairTileW;
    plan->pair_ok = L > 0 && L <= kPairMaxLevels && ceil_div(w, kPairTileW) <= kPairMaxTiles && p->frame_c >= 3 &&
                    (int64_t)p->frame_h * plan->frame_pitch < INT32_MAX;   // row offsets inside a frame are 32-bit
    for (int s = 0; s < L && plan->pair_ok; ++s) {
        PairLevel &pl = plan->pair[s];
        pl.ntx = ceil_div(w, kPairTileW);
        int widest = 1;
        for (int t = 0; t < pl.ntx; ++t) {
            int lo = INT32_MAX, hi = -1;
            for (int ox = t * kPairTileW; ox < std::min(w, (t + 1) * kPairTileW); ++ox) {
                const int32_t *tx = &plan->idx_x[((size_t)s * w + ox) * kTaps];
                if (tx[0] < 0) continue;
                for (int i = 0; i < kTaps; ++i) lo = std::min(lo, tx[i]), hi = std::max(hi, tx[i]);
            }
            if (hi < 0) {
                pl.word_lo[t] = pl.nwords[t] = 0;
                continue;
            }
            const int byte_lo = lo * p->frame_c, byte_hi = (hi + 1) * p->frame_c;
            pl.word_lo[t] = (byte_lo / 16) * 4;                       // 128-bit aligned span, in 32-bit words
            pl.nwords[t] = ((byte_hi + 15) / 16) * 4 - pl.word_lo[t];
            widest = std::max(widest, pl.nwords[t]);
        }
        pl.vpitch = (widest / 4) * 18;   // 16 byte-columns + 2 padding slots per 128-bit group (pyramid.cu: kVGroup)
        // rows per tile: fit the column-sum buffer in ~72 KB (3 CTAs per SM) and make the phase-V task count
        // (rows x 128-bit groups) fill whole rounds of the CTA's threads -- a 1.09-round tile idles the CTA at the barrier
        const int groups = widest / 4;
        double best = -1.0;
        pl.th = 1;
        for (int th = 1; th <= 48; ++th) {   // (16 was measured 3 % slower: taller tiles amortise the per-tile set-up)
            if ((size_t)th * pl.vpitch * 8 > (size_t)72 * 1024 * kPairThreads / 256 && th > 1) break;   // 768 threads per SM
            const int tasks = th * groups, rounds = ceil_div(tasks, kPairThreads);
            const double fill = (double)tasks / ((double)kPairThreads * rounds) + 0.002 * th;   // prefer taller tiles on ties
            if (fill > best) best = fill, pl.th = th;
        }
        if ((size_t)pl.th * pl.vpitch * 8 > 190 * 1024) plan->pair_ok = false;
    }

    if (L > 0) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
            (void)cudaGetLastError();
            plan->on_device = false;   // geometry-only plan (host queries still work; compute calls fail loudly)
        } else {
            const size_t by = plan->idx_y.size(), bx = plan->idx_x.size();
            const size_t cy = plan->coord_y.size(), cx = plan->coord_x.size();
            cudaError_t e = cudaMalloc(&plan->d_tables, (by + bx) * (sizeof(int32_t) + sizeof(float)) + (cy + cx) * sizeof(float));
            if (e != cudaSuccess) {
                delete plan;
                return fail(SILENT_E_CUDA, "cudaMalloc(tap tables) failed: %s", cudaGetErrorString(e));
            }
            char *base = (char *)plan->d_tables;
            plan->d_idx_y = (int32_t *)base;
            plan->d_idx_x = plan->d_idx_y + by;
            plan->d_w_y = (float *)(plan->d_idx_x + bx);
            plan->d_w_x = plan->d_w_y + by;
            plan->d_coord_y = plan->d_w_x + bx;
            plan->d_coord_x = plan->d_coord_y + cy;
            e = cudaMemcpy(plan->d_idx_y, plan->idx_y.data(), by * 4, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(plan->d_idx_x, plan->idx_x.data(), bx * 4, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(plan->d_w_y, plan->w_y.data(), by * 4, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(plan->d_w_x, plan->w_x.data(), bx * 4, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(plan->d_coord_y, plan->coord_y.data(), cy * 4, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(plan->d_coord_x, plan->coord_x.data(), cx * 4, cudaMemcpyHostToDevice);
            if (e != cudaSuccess) {
                delete plan;
                return fail(SILENT_E_CUDA, "upload of tap tables failed: %s", cudaGetErrorString(e));
            }
            if (plan->pair_ok) {   // per-level / per-tile word spans of the frame-pair pyramid kernel
                // (word_lo, nwords, M, 0): M = 2^32 / groups + 1 turns the kernel's task -> (row, group) division into one
                // multiply-high (exact for task < 2^32 / groups; groups = 1 is special-cased there)
                std::vector<int> words((size_t)L * kPairMaxTiles * 4, 0);
                for (int s = 0; s < L; ++s)
                    for (int t = 0; t < plan->pair[s].ntx; ++t) {
                        int *e4 = &words[((size_t)s * kPairMaxTiles + t) * 4];
                        e4[0] = plan->pair[s].word_lo[t];
                        e4[1] = plan->pair[s].nwords[t];
                        const uint32_t groups = (uint32_t)plan->pair[s].nwords[t] / 4;
                        const uint32_t magic = groups > 1 ? (uint32_t)((1ull << 32) / groups + 1) : 0u;
                        std::memcpy(&e4[2], &magic, 4);
                    }
                e = cudaMalloc(&plan->d_pair_words, words.size() * sizeof(int));
                if (e == cudaSuccess)
                    e = cudaMemcpy(plan->d_pair_words, words.data(), words.size() * sizeof(int), cudaMemcpyHostToDevice);
                // phase-H table: per (level, output column, channel) the six offsets of its taps in the padded column-sum
                // row of ITS tile and the six weights (offset 0 / weight 0 for columns the reference leaves undefined).
                // position(B) = B + 2 * (B >> 4) for the absolute byte column B = tap * frame_c + channel; tiles start at
                // multiples of 16 bytes, so the shift distributes and the tile origin is 4 * word_lo + 2 * (word_lo >> 2).
                std::vector<int32_t> htab((size_t)L * w * 3 * 12, 0);
                for (int s = 0; s < L; ++s)
                    for (int ox = 0; ox < w; ++ox) {
                        const int32_t *tx = &plan->idx_x[((size_t)s * w + ox) * kTaps];
                        const float *gx = &plan->w_x[((size_t)s * w + ox) * kTaps];
                        const int wlo = plan->pair[s].word_lo[ox / kPairTileW];
                        const int origin = 4 * wlo + (kPairVGroup - 16) * (wlo >> 2);
                        for (int c = 0; c < 3; ++c) {
                            int32_t *row = &htab[(((size_t)s * w + ox) * 3 + c) * 12];
                            for (int i = 0; i < kTaps; ++i) {
                                const int B = tx[0] >= 0 ? tx[i] * p->frame_c + c : -1;
                                row[i] = B >= 0 ? B + (kPairVGroup - 16) * (B >> 4) - origin : 0;
                                const float wv = tx[0] >= 0 ? gx[i] : 0.0f;
                                std::memcpy(&row[6 + i], &wv, 4);
                            }
                        }
                    }
                if (e == cudaSuccess) e = cudaMalloc(&plan->d_pair_htab, htab.size() * sizeof(int32_t));
                if (e == cudaSuccess)
                    e = cudaMemcpy(plan->d_pair_htab, htab.data(), htab.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
                // phase-V table: per (level, output row) 12 words = (offset of tap row 0 in a frame or -1 for a row the
                // reference leaves undefined, STEP, six weights, offsets of tap rows 1..4). When the six tap rows are
                // consecutive frame rows (every row but the few whose taps are mirrored at the crop's edge) STEP is the
                // frame's row pitch in bytes and a task needs the first TWO 128-bit words only; else STEP = -(offset of
                // tap row 5) - 1 and the third word holds the other four offsets.
                std::vector<int32_t> ytab((size_t)L * h * 12, 0);
                const int64_t row_bytes = plan->frame_pitch;
                for (int s = 0; s < L; ++s)
                    for (int oy = 0; oy < h; ++oy) {
                        const int32_t *ty = &plan->idx_y[((size_t)s * h + oy) * kTaps];
                        const float *gy = &plan->w_y[((size_t)s * h + oy) * kTaps];
                        int32_t *row = &ytab[((size_t)s * h + oy) * 12];
                        if (ty[0] < 0) {
                            row[0] = -1, row[1] = (int32_t)row_bytes;   // (weights and offsets stay 0)
                            continue;
                        }
                        bool regular = true;
                        for (int j = 1; j < kTaps; ++j) regular = regular && ty[j] == ty[0] + j;
                        row[0] = (int32_t)(ty[0] * row_bytes);
                        row[1] = regular ? (int32_t)row_bytes : -(int32_t)(ty[5] * row_bytes) - 1;
                        std::memcpy(&row[2], gy, kTaps * sizeof(float));
                        for (int j = 1; j <= 4; ++j) row[7 + j] = (int32_t)(ty[j] * row_bytes);
                    }
                if (e == cudaSuccess) e = cudaMalloc(&plan->d_pair_ytab, ytab.size() * sizeof(int32_t));
                if (e == cudaSuccess)
                    e = cudaMemcpy(plan->d_pair_ytab, ytab.data(), ytab.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
                if (e == cudaSuccess) {   // the phase-H table as a linear texture of int4 texels, and the alignment a
                    // linear texture's devPtr needs (either failing only keeps the frame-pair kernel on its LDG variant)
                    cudaResourceDesc rd = {};
                    rd.resType = cudaResourceTypeLinear;
                    rd.res.linear.devPtr = plan->d_pair_htab;
                    rd.res.linear.desc = cudaCreateChannelDesc<int4>();
                    rd.res.linear.sizeInBytes = htab.size() * sizeof(int32_t);
                    cudaTextureDesc td = {};
                    td.readMode = cudaReadModeElementType;
                    if (cudaCreateTextureObject(&plan->htab_tex, &rd, &td, nullptr) != cudaSuccess) {
                        (void)cudaGetLastError();
                        plan->htab_tex = 0;
                    }
                    int dev = 0;
                    if (cudaGetDevice(&dev) != cudaSuccess ||
                        cudaDeviceGetAttribute(&plan->texture_alignment, cudaDevAttrTextureAlignment, dev) != cudaSuccess) {
                        (void)cudaGetLastError();
                        plan->texture_alignment = 0;
                    }
                }
                if (e != cudaSuccess) {
                    delete plan;
                    return fail(SILENT_E_CUDA, "upload of pyramid tile spans failed: %s", cudaGetErrorString(e));
                }
            }
            plan->on_device = true;
        }
    }
    // NV12: converted frames start at the texture alignment (512 B on B200), so every frame pair and every chunk of the
    // host-buffer path can take the frame-pair kernel's texture route
    const int64_t frame_align = nv12 ? std::max(plan->texture_alignment, 512) : 1;
    plan->frame_stride = ((int64_t)p->frame_h * plan->frame_pitch + frame_align - 1) / frame_align * frame_align;
    *out_plan = plan;
    return SILENT_OK;
}

void silent_plan_destroy(silent_plan *plan) { delete plan; }

int silent_plan_levels(const silent_plan *plan) { return plan ? plan->levels : fail(SILENT_E_INVAL, "null plan"); }

int silent_plan_level_hw(const silent_plan *plan, int *h, int *w)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (h) *h = plan->h;
    if (w) *w = plan->w;
    return SILENT_OK;
}

int silent_plan_level_info(const silent_plan *plan, int level, int *y0, int *y1, int *x0, int *x1, int *valid_h,
                           int *valid_w)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (level < 0 || level >= plan->levels) return fail(SILENT_E_INVAL, "level %d out of range [0,%d)", level, plan->levels);
    const LevelInfo &li = plan->info[level];
    if (y0) *y0 = li.y0;
    if (y1) *y1 = li.y1;
    if (x0) *x0 = li.x0;
    if (x1) *x1 = li.x1;
    if (valid_h) *valid_h = li.valid_h;
    if (valid_w) *valid_w = li.valid_w;
    return SILENT_OK;
}

int silent_plan_level_tables(const silent_plan *plan, int level, int32_t *idx_y, float *w_y, int32_t *idx_x, float *w_x)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (level < 0 || level >= plan->levels) return fail(SILENT_E_INVAL, "level %d out of range [0,%d)", level, plan->levels);
    const size_t ny = (size_t)plan->h * kTaps, nx = (size_t)plan->w * kTaps;
    if (idx_y) std::memcpy(idx_y, &plan->idx_y[level * ny], ny * 4);
    if (w_y) std::memcpy(w_y, &plan->w_y[level * ny], ny * 4);
    if (idx_x) std::memcpy(idx_x, &plan->idx_x[level * nx], nx * 4);
    if (w_x) std::memcpy(w_x, &plan->w_x[level * nx], nx * 4);
    return SILENT_OK;
}

int silent_plan_level_coords(const silent_plan *plan, int level, float *frame_y, float *frame_x)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (level < 0 || level >= plan->levels) return fail(SILENT_E_INVAL, "level %d out of range [0,%d)", level, plan->levels);
    if (frame_y) std::memcpy(frame_y, &plan->coord_y[(size_t)level * plan->h], (size_t)plan->h * sizeof(float));
    if (frame_x) std::memcpy(frame_x, &plan->coord_x[(size_t)level * plan->w], (size_t)plan->w * sizeof(float));
    return SILENT_OK;
}

int64_t silent_plan_algorithmic_bytes(const silent_plan *plan)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    const int64_t px = (int64_t)plan->union_h * plan->union_w;
    const int dtype = plan->params.frame_dtype;
    const int64_t in_bytes = dtype == SILENT_NV12 ? px * 3 / 2 : px * plan->params.frame_c * (dtype == SILENT_U8 ? 1 : 4);
    const int64_t out_bytes = 2LL * plan->levels * plan->h * plan->w * plan->params.num_colors * 4;
    return in_bytes + out_bytes;
}

}  // extern "C"
