// The whole hot path behind one call: frames -> pyramid (K1) -> fused stack (K2) -> feature points (K3).
// silent_pipeline_run works on buffers resident in HBM; silent_pipeline_run_host is the drop-in for
// LineEndDisplayer.callback (reference recognition_testing.py:136-144) with host buffers on both sides.
#include <algorithm>
#include <cstring>
#include <memory>

#include <nvtx3/nvToolsExt.h>

#include "plan.h"
#include "stack.h"

namespace silent {

// NVTX range over a stage's launches (free when no profiler is attached; shows the stage next to its kernels in nsys)
struct StageRange {
    explicit StageRange(const char *name) { nvtxRangePushA(name); }
    ~StageRange() { nvtxRangePop(); }
};

static void release(Workspace &ws)
{
    cudaFree(ws.d_frames);
    cudaFree(ws.d_pyramid);
    cudaFree(ws.d_orient);
    cudaFree(ws.d_line_end);
    cudaFree(ws.d_gray);
    cudaFree(ws.d_select);
    cudaFree(ws.d_stack);
    cudaFree(ws.d_winmax);
    cudaFree(ws.d_tilemax);
    cudaFree(ws.d_points);
    cudaFree(ws.d_count);
    cudaFreeHost(ws.h_frames);
    cudaFreeHost(ws.h_orient);
    cudaFreeHost(ws.h_line_end);
    cudaFreeHost(ws.h_points);
    cudaFreeHost(ws.h_count);
    for (cudaEvent_t e : ws.ev_in)
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ws.ev_done)
        if (e) cudaEventDestroy(e);
    if (ws.s_in) cudaStreamDestroy(ws.s_in);
    if (ws.s_out) cudaStreamDestroy(ws.s_out);
    ws = Workspace();
}

// Page-locked host memory (cudaMallocHost / cudaHostRegister / torch pin_memory) can be copied asynchronously in place;
// pageable memory is staged through the plan's pinned mirrors.
static bool is_pinned_at(const void *p)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}
// both ends of the range: a buffer that only STARTS in a page-locked allocation is staged like pageable memory
static bool is_pinned(const void *p, size_t bytes)
{
    return p && bytes > 0 && is_pinned_at(p) && is_pinned_at((const char *)p + bytes - 1);
}

static size_t frame_bytes(const silent_plan *plan)
{
    const silent_params &p = plan->params;
    return (size_t)p.frame_h * p.frame_w * p.frame_c * (p.frame_dtype == SILENT_U8 ? 1 : 4);
}

}  // namespace silent

using namespace silent;

silent_plan::~silent_plan()
{
    for (cudaEvent_t e : ev)
        if (e) cudaEventDestroy(e);
    if (ev_mid) cudaEventDestroy(ev_mid);
    release(ws);
    if (d_tables) cudaFree(d_tables);
    if (d_pair_words) cudaFree(d_pair_words);
    if (d_pair_htab) cudaFree(d_pair_htab);
    if (d_pair_ytab) cudaFree(d_pair_ytab);
    for (FrameTexture &ft : frame_textures)
        if (ft.tex) cudaDestroyTextureObject(ft.tex);
    if (ytab_tex) cudaDestroyTextureObject(ytab_tex);
    if (htab_tex) cudaDestroyTextureObject(htab_tex);
}

extern "C" {

int silent_plan_reserve(silent_plan *plan, int max_batch)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (max_batch <= 0) return fail(SILENT_E_INVAL, "max_batch must be positive");
    if (!plan->on_device && plan->levels > 0)
        return fail(SILENT_E_CUDA, "plan was created without a CUDA device; no CPU fallback exists");
    Workspace &ws = plan->ws;
    if (ws.batch >= max_batch) return SILENT_OK;
    release(ws);
    const size_t n = (size_t)max_batch * (plan->levels > 0 ? plan->levels : 1);
    const size_t level_elems = (size_t)plan->h * plan->w;
    const size_t tensor_bytes = n * level_elems * 3 * sizeof(float);
    size_t pyr_bytes = n * level_elems * plan->params.num_colors * sizeof(float);
    if (pyramid_pair_supported(plan)) pyr_bytes = std::max(pyr_bytes, pyramid_pair_bytes(plan, max_batch));
    ws.select_bytes = silent_selection_workspace_bytes((int)n, plan->h, plan->w);
    ws.points_capacity = (int64_t)n * 64;
    SILENT_CUDA(cudaMalloc(&ws.d_frames, frame_bytes(plan) * max_batch));
    SILENT_CUDA(cudaMalloc(&ws.d_pyramid, pyr_bytes));
    SILENT_CUDA(cudaMalloc(&ws.d_orient, tensor_bytes));
    SILENT_CUDA(cudaMalloc(&ws.d_line_end, tensor_bytes));
    SILENT_CUDA(cudaMalloc(&ws.d_gray, n * level_elems * sizeof(float)));
    SILENT_CUDA(cudaMalloc(&ws.d_select, ws.select_bytes));
    ws.stack_bytes = stack_workspace_bytes((int)n, plan->h, plan->w);
    SILENT_CUDA(cudaMalloc(&ws.d_stack, ws.stack_bytes));
    SILENT_CUDA(cudaMalloc(&ws.d_winmax, n * 4 * sizeof(int)));
    {
        int th, tw, nty, ntx;
        stack_tile_grid(plan->h, plan->w, &th, &tw, &nty, &ntx);
        SILENT_CUDA(cudaMalloc(&ws.d_tilemax, n * nty * ntx * sizeof(int)));
    }
    SILENT_CUDA(cudaMalloc(&ws.d_points, ws.points_capacity * 4 * sizeof(int64_t)));
    SILENT_CUDA(cudaMalloc(&ws.d_count, sizeof(int64_t)));
    // h_frames / h_orient / h_line_end (pinned mirrors for PAGEABLE caller buffers) are allocated on first need
    SILENT_CUDA(cudaMallocHost(&ws.h_points, ws.points_capacity * 4 * sizeof(int64_t)));
    SILENT_CUDA(cudaMallocHost(&ws.h_count, sizeof(int64_t)));
    ws.batch = max_batch;
    return SILENT_OK;
}

// the per-tile maxima of gray that stack_b_kernel writes for the whole batch (read by the emit stage)
static TileMaxima tile_maxima(const silent_plan *plan)
{
    TileMaxima tm;
    stack_tile_grid(plan->h, plan->w, &tm.tile_h, &tm.tile_w, &tm.nty, &tm.ntx);
    tm.data = plan->ws.d_tilemax;
    return tm;
}

// K1 + K2 for frames [frame0, frame0 + nb) of a batch: the outputs, gray and the region maxima of these frames land at
// their place in the whole-batch tensors, so that the emit stage can run once over the batch afterwards. frame0 must be
// even on the frame-pair path (pairs never straddle a chunk).
static int run_stack_stages(silent_plan *plan, const silent_stack_weights *W, const void *frames_dev, int frame0, int nb,
                            float *pyramid_dev, float *orient_dev, float *line_end_dev, const WindowGeom *geo,
                            cudaStream_t s, const PairClear *also_clear = nullptr)
{
    Workspace &ws = plan->ws;
    const bool pair_path = pyramid_pair_supported(plan);
    const size_t level_elems = (size_t)plan->h * plan->w;
    const size_t img0 = (size_t)frame0 * plan->levels;
    const int n = nb * plan->levels;
    const unsigned char *frames = (const unsigned char *)frames_dev + frame_bytes(plan) * frame0;
    // stack_b's tile flags must be zero before it runs: the frame-pair pyramid kernel clears them on its way (and what
    // the caller adds in also_clear), so that no memset sits between the previous step's last kernel and this launch;
    // without that kernel a memset ahead of the launches does it
    int rc = SILENT_OK;
    PairClear clear;
    if (pair_path) {
        stack_flag_region(ws.d_stack, n, plan->h, plan->w, &clear.a, &clear.a_bytes);
        if (also_clear) clear.b = also_clear->b, clear.b_bytes = also_clear->b_bytes;
    } else {
        rc = stack_clear_flags(ws.d_stack, n, plan->h, plan->w, s);
        if (rc != SILENT_OK) return rc;
        if (also_clear && also_clear->b) SILENT_CUDA(cudaMemsetAsync(also_clear->b, 0, also_clear->b_bytes, s));
    }
    // Fast path: the frame-pair pyramid kernel feeds the stack in its own pair-interleaved layout. The NHWC pyramid is
    // only materialised when the caller asks for it (pyramid_dev) or the plan does not qualify (float frames, ...).
    {
        StageRange range("silent:pyramid");
        if (pyramid_dev || !pair_path) {
            float *dst = pyramid_dev ? pyramid_dev + img0 * level_elems * plan->params.num_colors : ws.d_pyramid;
            rc = pyramid_build(plan, frames, nb, dst, s);
            if (rc != SILENT_OK) return rc;
        }
        if (pair_path) {
            rc = pyramid_pair_build(plan, frames, nb, ws.d_pyramid, s, &clear);
            if (rc != SILENT_OK) return rc;
        }
    }
    StageRange range("silent:stack");
    const void *pyr = pair_path ? (const void *)ws.d_pyramid
                                : (const void *)(pyramid_dev ? pyramid_dev + img0 * level_elems * 3 : ws.d_pyramid);
    if (plan->timing) SILENT_CUDA(cudaEventRecord(plan->ev[1], s));
    const TileMaxima tm = tile_maxima(plan);
    return stack_fused(pyr, n, plan->h, plan->w, pair_path ? plan->levels : 0, W,
                       orient_dev ? orient_dev + img0 * level_elems * 3 : nullptr,
                       line_end_dev ? line_end_dev + img0 * level_elems * 3 : nullptr, ws.d_gray + img0 * level_elems,
                       ws.d_stack, ws.stack_bytes, geo, geo ? ws.d_winmax + img0 * geo->count : nullptr,
                       ws.d_tilemax + img0 * tm.nty * tm.ntx, s, plan->timing ? plan->ev_mid : nullptr, true);
}

static int check_pipeline_args(const silent_plan *plan, const silent_stack_weights *W, const void *frames, int batch)
{
    if (!plan || !W || !frames) return fail(SILENT_E_INVAL, "silent_pipeline_run: null argument");
    if (batch <= 0) return fail(SILENT_E_INVAL, "batch must be positive");
    if (plan->params.num_colors != 3) return fail(SILENT_E_SHAPE, "the fused stack needs num_colors == 3");
    if (plan->levels == 0) return fail(SILENT_E_SHAPE, "frame is not larger than the pyramid centre: 0 levels");
    if ((plan->h % 2) || (plan->w % 2))
        return fail(SILENT_E_SHAPE, "Ambiguous dimension: region shape (h/2, w/2) must be integral (h=%d, w=%d)", plan->h,
                    plan->w);
    return SILENT_OK;
}

int silent_pipeline_run(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_dev, int batch,
                        float *pyramid_dev, float *orient_dev, float *line_end_dev, int64_t *points_dev,
                        int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    int rc = check_pipeline_args(plan, weights_host, frames_dev, batch);
    if (rc != SILENT_OK) return rc;
    Workspace &ws = plan->ws;
    if (ws.batch < batch)
        return fail(SILENT_E_CAPACITY, "plan workspace holds %d frames, need %d: call silent_plan_reserve", ws.batch, batch);
    cudaStream_t s = (cudaStream_t)stream;
    const int n = batch * plan->levels;
    const bool timing = plan->timing;
    if (timing) SILENT_CUDA(cudaEventRecord(plan->ev[0], s));
    WindowGeom geo;
    const bool fuse_windows = count_dev && window_geometry(plan->h, plan->w, plan->h / 2, plan->w / 2, &geo);
    PairClear winmax_clear;   // the region maxima start at 0: cleared together with the tile flags (see run_stack_stages)
    if (fuse_windows) winmax_clear.b = ws.d_winmax, winmax_clear.b_bytes = (size_t)n * geo.count * sizeof(int);
    rc = run_stack_stages(plan, weights_host, frames_dev, 0, batch, pyramid_dev, orient_dev, line_end_dev,
                          fuse_windows ? &geo : nullptr, s, &winmax_clear);
    if (rc != SILENT_OK) return rc;
    if (timing) SILENT_CUDA(cudaEventRecord(plan->ev[2], s));
    if (count_dev) {
        StageRange range("silent:emit");
        const TileMaxima tm = tile_maxima(plan);
        rc = max_value_indices_region(ws.d_gray, n, plan->h, plan->w, plan->h / 2, plan->w / 2, points_dev, capacity,
                                      count_dev, ws.d_select, ws.select_bytes, fuse_windows ? ws.d_winmax : nullptr, &tm, s);
    }
    if (timing) SILENT_CUDA(cudaEventRecord(plan->ev[3], s));
    return rc;
}

int silent_pipeline_run_orientations(silent_plan *plan, const silent_orientation_bank *bank_host, const void *frames_dev,
                                     int batch, float *orient_dev, float *line_end_dev, int64_t *points_dev,
                                     int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    int rc = check_bank(bank_host, "silent_pipeline_run_orientations");
    if (rc != SILENT_OK) return rc;
    if (!plan || !frames_dev) return fail(SILENT_E_INVAL, "silent_pipeline_run_orientations: null argument");
    if (batch <= 0) return fail(SILENT_E_INVAL, "batch must be positive");
    if (plan->levels == 0) return fail(SILENT_E_SHAPE, "frame is not larger than the pyramid centre: 0 levels");
    if (!pyramid_pair_supported(plan))
        return fail(SILENT_E_SHAPE, "the fused orientation bank needs uint8 frames with 3 colours (frame-pair pyramid path)");
    if ((plan->h % 2) || (plan->w % 2))
        return fail(SILENT_E_SHAPE, "Ambiguous dimension: region shape (h/2, w/2) must be integral (h=%d, w=%d)", plan->h,
                    plan->w);
    Workspace &ws = plan->ws;
    if (ws.batch < batch)
        return fail(SILENT_E_CAPACITY, "plan workspace holds %d frames, need %d: call silent_plan_reserve", ws.batch, batch);
    cudaStream_t s = (cudaStream_t)stream;
    const int n = batch * plan->levels;
    if (plan->timing) SILENT_CUDA(cudaEventRecord(plan->ev[0], s));
    rc = pyramid_pair_build(plan, frames_dev, batch, ws.d_pyramid, s);
    if (rc != SILENT_OK) return rc;
    if (plan->timing) SILENT_CUDA(cudaEventRecord(plan->ev[1], s));
    rc = stack_bank(ws.d_pyramid, n, plan->h, plan->w, plan->levels, bank_host, orient_dev, line_end_dev, ws.d_gray,
                    ws.d_stack, ws.stack_bytes, s, plan->timing ? plan->ev_mid : nullptr);
    if (rc != SILENT_OK) return rc;
    if (plan->timing) SILENT_CUDA(cudaEventRecord(plan->ev[2], s));
    if (count_dev)
        rc = max_value_indices_region(ws.d_gray, n, plan->h, plan->w, plan->h / 2, plan->w / 2, points_dev, capacity,
                                      count_dev, ws.d_select, ws.select_bytes, nullptr, nullptr, s);
    if (plan->timing) SILENT_CUDA(cudaEventRecord(plan->ev[3], s));
    return rc;
}

int silent_pipeline_run_bank(silent_plan *plan, const silent_bank_weights *weights_host, const void *frames_dev, int batch,
                             float *orient_dev, float *line_end_dev, int64_t *points_dev, int64_t capacity,
                             int64_t *count_dev, silent_stream stream)
{
    if (!weights_host) return fail(SILENT_E_INVAL, "silent_pipeline_run_bank: null argument");
    std::unique_ptr<silent_orientation_bank> bank(new silent_orientation_bank());
    const silent_bank_weights &W = *weights_host;
    bank->orientations = SILENT_BANK;
    std::memcpy(bank->rgc, W.rgc, sizeof(W.rgc));
    std::memcpy(bank->rgby, W.rgby, sizeof(W.rgby));
    std::memcpy(bank->stripe, W.stripe, sizeof(W.stripe));
    std::memcpy(bank->blur, W.blur, sizeof(W.blur));
    std::memcpy(bank->end, W.end, sizeof(W.end));
    bank->regulation_value = W.regulation_value, bank->regulation_root = W.regulation_root, bank->clip_max = W.clip_max;
    bank->border = W.border;
    return silent_pipeline_run_orientations(plan, bank.get(), frames_dev, batch, orient_dev, line_end_dev, points_dev,
                                            capacity, count_dev, stream);
}

int silent_plan_enable_timing(silent_plan *plan, int enable)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (enable)
        for (cudaEvent_t &e : plan->ev)
            if (!e) SILENT_CUDA(cudaEventCreate(&e));
    if (enable && !plan->ev_mid) SILENT_CUDA(cudaEventCreate(&plan->ev_mid));
    plan->timing = enable != 0;
    return SILENT_OK;
}

int silent_plan_stage_ms(silent_plan *plan, float *pyramid_ms, float *stack_ms, float *emit_ms)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (!plan->timing || !plan->ev[3]) return fail(SILENT_E_INVAL, "timing is not enabled on this plan");
    SILENT_CUDA(cudaEventSynchronize(plan->ev[3]));
    float *dst[3] = {pyramid_ms, stack_ms, emit_ms};
    for (int i = 0; i < 3; ++i)
        if (dst[i]) SILENT_CUDA(cudaEventElapsedTime(dst[i], plan->ev[i], plan->ev[i + 1]));
    return SILENT_OK;
}

// Frames per chunk of the host-buffer pipeline: even (frame pairs), at most kMaxChunks chunks per call.
static int host_chunk_frames(int batch)
{
    int per = (batch + kMaxChunks - 1) / kMaxChunks;   // small chunks: the first download starts early
    per = std::max(per, 2);
    per += per & 1;
    while ((batch + per - 1) / per > kMaxChunks) per += 2;
    return per;
}

int silent_plan_stack_split_ms(silent_plan *plan, float *stack_a_ms, float *stack_b_ms)
{
    if (!plan) return fail(SILENT_E_INVAL, "null plan");
    if (!plan->timing || !plan->ev[3] || !plan->ev_mid) return fail(SILENT_E_INVAL, "timing is not enabled on this plan");
    SILENT_CUDA(cudaEventSynchronize(plan->ev[3]));
    if (stack_a_ms) SILENT_CUDA(cudaEventElapsedTime(stack_a_ms, plan->ev[1], plan->ev_mid));
    if (stack_b_ms) SILENT_CUDA(cudaEventElapsedTime(stack_b_ms, plan->ev_mid, plan->ev[2]));
    return SILENT_OK;
}

int silent_pipeline_run_host(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_host,
                             int batch, float *orient_host, float *line_end_host, int64_t *points_host,
                             int64_t capacity, int64_t *count_host, silent_stream stream)
{
    int rc = check_pipeline_args(plan, weights_host, frames_host, batch);
    if (rc != SILENT_OK) return rc;
    if (capacity < 0) return fail(SILENT_E_INVAL, "capacity must be >= 0");
    rc = silent_plan_reserve(plan, batch);
    if (rc != SILENT_OK) return rc;
    Workspace &ws = plan->ws;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t fbytes = frame_bytes(plan);
    const size_t n = (size_t)batch * plan->levels;
    const size_t image_bytes = (size_t)plan->h * plan->w * 3 * sizeof(float);
    const size_t cap_tensor_bytes = (size_t)ws.batch * plan->levels * image_bytes;

    // Three queues: s_in (host -> HBM), the caller's stream (kernels), s_out (HBM -> host). The batch is cut into chunks
    // of whole frame pairs; chunk c + 1 uploads while chunk c computes and chunk c - 1 downloads, so on a full-duplex
    // PCIe link the call costs about max(upload, download) instead of their sum.
    if (!ws.s_in) SILENT_CUDA(cudaStreamCreateWithFlags(&ws.s_in, cudaStreamNonBlocking));
    if (!ws.s_out) SILENT_CUDA(cudaStreamCreateWithFlags(&ws.s_out, cudaStreamNonBlocking));
    for (int i = 0; i < kMaxChunks; ++i) {
        if (!ws.ev_in[i]) SILENT_CUDA(cudaEventCreateWithFlags(&ws.ev_in[i], cudaEventDisableTiming));
        if (!ws.ev_done[i]) SILENT_CUDA(cudaEventCreateWithFlags(&ws.ev_done[i], cudaEventDisableTiming));
    }
    const bool frames_direct = is_pinned(frames_host, fbytes * batch);
    const bool orient_direct = orient_host && is_pinned(orient_host, n * image_bytes);
    const bool line_end_direct = line_end_host && is_pinned(line_end_host, n * image_bytes);
    if (!frames_direct && !ws.h_frames) SILENT_CUDA(cudaMallocHost(&ws.h_frames, fbytes * ws.batch));
    if (orient_host && !orient_direct && !ws.h_orient) SILENT_CUDA(cudaMallocHost(&ws.h_orient, cap_tensor_bytes));
    if (line_end_host && !line_end_direct && !ws.h_line_end)
        SILENT_CUDA(cudaMallocHost(&ws.h_line_end, cap_tensor_bytes));
    char *orient_dst = (char *)(orient_direct ? orient_host : ws.h_orient);
    char *line_end_dst = (char *)(line_end_direct ? line_end_host : ws.h_line_end);

    WindowGeom geo;
    const bool fuse_windows = window_geometry(plan->h, plan->w, plan->h / 2, plan->w / 2, &geo);
    // work queued on the caller's stream before this call stays ordered before anything we overwrite
    SILENT_CUDA(cudaEventRecord(ws.ev_done[0], s));
    SILENT_CUDA(cudaStreamWaitEvent(ws.s_in, ws.ev_done[0], 0));
    SILENT_CUDA(cudaStreamWaitEvent(ws.s_out, ws.ev_done[0], 0));
    if (fuse_windows) SILENT_CUDA(cudaMemsetAsync(ws.d_winmax, 0, n * geo.count * sizeof(int), s));
    // Everything below queues asynchronous work against the caller's buffers and the plan's staging buffers: whatever
    // goes wrong, ALL three queues are drained before the call returns (run_chunks never returns early past a copy).
    auto drain = [&]() {
        cudaStreamSynchronize(ws.s_in);
        cudaStreamSynchronize(s);
        cudaStreamSynchronize(ws.s_out);
    };
    if (points_host && capacity > ws.points_capacity) {   // a caller retrying after *count_host > capacity (an all-zero
        cudaFree(ws.d_points);                             // level emits every pixel): grow the plan's point buffers
        cudaFreeHost(ws.h_points);
        ws.d_points = nullptr, ws.h_points = nullptr, ws.points_capacity = 0;
        SILENT_CUDA(cudaMalloc(&ws.d_points, capacity * 4 * sizeof(int64_t)));
        SILENT_CUDA(cudaMallocHost(&ws.h_points, capacity * 4 * sizeof(int64_t)));
        ws.points_capacity = capacity;
    }
    const int64_t cap = capacity < ws.points_capacity ? capacity : ws.points_capacity;
    auto run_chunks = [&]() -> int {
        const int per = host_chunk_frames(batch);
        int chunk = 0;
        for (int f0 = 0; f0 < batch; f0 += per, ++chunk) {
            const int nb = std::min(per, batch - f0);
            const char *src = (const char *)frames_host + fbytes * f0;
            if (!frames_direct) {
                std::memcpy((char *)ws.h_frames + fbytes * f0, src, fbytes * nb);
                src = (const char *)ws.h_frames + fbytes * f0;
            }
            SILENT_CUDA(cudaMemcpyAsync((char *)ws.d_frames + fbytes * f0, src, fbytes * nb, cudaMemcpyHostToDevice, ws.s_in));
            SILENT_CUDA(cudaEventRecord(ws.ev_in[chunk], ws.s_in));
            SILENT_CUDA(cudaStreamWaitEvent(s, ws.ev_in[chunk], 0));
            const int rcs = run_stack_stages(plan, weights_host, ws.d_frames, f0, nb, nullptr,
                                             orient_host ? ws.d_orient : nullptr, line_end_host ? ws.d_line_end : nullptr,
                                             fuse_windows ? &geo : nullptr, s);
            if (rcs != SILENT_OK) return rcs;
            SILENT_CUDA(cudaEventRecord(ws.ev_done[chunk], s));
            SILENT_CUDA(cudaStreamWaitEvent(ws.s_out, ws.ev_done[chunk], 0));
            const size_t off = (size_t)f0 * plan->levels * image_bytes, bytes = (size_t)nb * plan->levels * image_bytes;
            if (orient_host)
                SILENT_CUDA(cudaMemcpyAsync(orient_dst + off, (char *)ws.d_orient + off, bytes, cudaMemcpyDeviceToHost, ws.s_out));
            if (line_end_host)
                SILENT_CUDA(cudaMemcpyAsync(line_end_dst + off, (char *)ws.d_line_end + off, bytes, cudaMemcpyDeviceToHost,
                                            ws.s_out));
        }
        const TileMaxima tm = tile_maxima(plan);
        const int rce = max_value_indices_region(ws.d_gray, (int)n, plan->h, plan->w, plan->h / 2, plan->w / 2, ws.d_points,
                                                 cap, ws.d_count, ws.d_select, ws.select_bytes,
                                                 fuse_windows ? ws.d_winmax : nullptr, &tm, s);
        if (rce != SILENT_OK) return rce;
        SILENT_CUDA(cudaMemcpyAsync(ws.h_count, ws.d_count, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        if (points_host && cap > 0)
            SILENT_CUDA(cudaMemcpyAsync(ws.h_points, ws.d_points, cap * 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        return SILENT_OK;
    };
    rc = run_chunks();
    drain();
    if (rc != SILENT_OK) return rc;
    {
        const cudaError_t late = cudaGetLastError();   // an asynchronous failure surfaces at the synchronisation
        if (late != cudaSuccess) return fail(SILENT_E_CUDA, "silent_pipeline_run_host: %s", cudaGetErrorString(late));
    }
    const size_t tensor_bytes = n * image_bytes;
    if (orient_host && !orient_direct) std::memcpy(orient_host, ws.h_orient, tensor_bytes);
    if (line_end_host && !line_end_direct) std::memcpy(line_end_host, ws.h_line_end, tensor_bytes);
    const int64_t total = *ws.h_count;
    if (count_host) *count_host = total;
    if (points_host && cap > 0) {
        const int64_t rows = total < cap ? total : cap;
        std::memcpy(points_host, ws.h_points, rows * 4 * sizeof(int64_t));
    }
    return SILENT_OK;
}

}  // extern "C"
