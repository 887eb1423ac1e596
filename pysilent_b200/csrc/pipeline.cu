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
    cudaFree(ws.d_bgr);
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

// bytes of one frame as the caller passes it
static size_t frame_bytes(const silent_plan *plan)
{
    const silent_params &p = plan->params;
    if (p.frame_dtype == SILENT_NV12) return (size_t)p.frame_h * p.frame_w * 3 / 2;
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
    if (plan->params.frame_dtype == SILENT_NV12) SILENT_CUDA(cudaMalloc(&ws.d_bgr, (size_t)plan->frame_stride * max_batch));
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
// even on the frame-pair path (pairs never straddle a chunk). K2 is the three-orientation stack (W) or, when bank is set,
// the orientation bank's stack (frame-pair path only; no tile flags, geo must be null). orient_dev / line_end_dev hold
// float32, or binary16 when half_out. NV12 frames are converted into ws.d_bgr first (these frames only), and the pyramid
// reads them there.
static int run_stack_stages(silent_plan *plan, const silent_stack_weights *W, const silent_orientation_bank *bank,
                            const void *frames_dev, int frame0, int nb, float *pyramid_dev, void *orient_dev,
                            void *line_end_dev, bool half_out, const WindowGeom *geo, cudaStream_t s,
                            const PairClear *also_clear = nullptr)
{
    Workspace &ws = plan->ws;
    const bool pair_path = pyramid_pair_supported(plan);
    const size_t level_elems = (size_t)plan->h * plan->w;
    const size_t img0 = (size_t)frame0 * plan->levels;
    const int n = nb * plan->levels;
    const unsigned char *frames = (const unsigned char *)frames_dev + frame_bytes(plan) * frame0;
    int rc = SILENT_OK;
    if (plan->params.frame_dtype == SILENT_NV12) {
        StageRange range("silent:nv12");
        rc = nv12_convert(plan, frames_dev, frame0, nb, s);
        if (rc != SILENT_OK) return rc;
        frames = ws.d_bgr + (size_t)plan->frame_stride * frame0;
    }
    // stack_b's tile flags must be zero before it runs: the frame-pair pyramid kernel clears them on its way (and what
    // the caller adds in also_clear), so that no memset sits between the previous step's last kernel and this launch;
    // without that kernel a memset ahead of the launches does it
    PairClear clear;   // (the bank's kernel keeps no tile flags: nothing to clear)
    if (!bank && pair_path) {
        stack_flag_region(ws.d_stack, n, plan->h, plan->w, &clear.a, &clear.a_bytes);
        if (also_clear) clear.b = also_clear->b, clear.b_bytes = also_clear->b_bytes;
    } else if (!bank) {
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
    const size_t ch = bank ? bank->orientations : 3;
    const size_t out_offset = img0 * level_elems * ch * (half_out ? 2 : sizeof(float));   // bytes
    void *orient = orient_dev ? (char *)orient_dev + out_offset : nullptr;
    void *line_end = line_end_dev ? (char *)line_end_dev + out_offset : nullptr;
    cudaEvent_t mid = plan->timing ? plan->ev_mid : nullptr;
    if (bank)
        return stack_bank(pyr, n, plan->h, plan->w, plan->levels, bank, orient, line_end, half_out,
                          ws.d_gray + img0 * level_elems, ws.d_stack, ws.stack_bytes, s, mid);
    const TileMaxima tm = tile_maxima(plan);
    return stack_fused(pyr, n, plan->h, plan->w, pair_path ? plan->levels : 0, W, orient, line_end, half_out,
                       ws.d_gray + img0 * level_elems, ws.d_stack, ws.stack_bytes, geo,
                       geo ? ws.d_winmax + img0 * geo->count : nullptr, ws.d_tilemax + img0 * tm.nty * tm.ntx, s, mid, true);
}

// checks shared by the pipeline entry points (`who` names the entry point); weights: the entry point's weight struct
static int check_pipeline_args(const char *who, const silent_plan *plan, const void *weights, const void *frames, int batch)
{
    if (!plan || !weights || !frames) return fail(SILENT_E_INVAL, "%s: null argument", who);
    if (batch <= 0) return fail(SILENT_E_INVAL, "batch must be positive");
    if (plan->params.num_colors != 3) return fail(SILENT_E_SHAPE, "the fused stack needs num_colors == 3");
    if (plan->levels == 0) return fail(SILENT_E_SHAPE, "frame is not larger than the pyramid centre: 0 levels");
    if ((plan->h % 2) || (plan->w % 2))
        return fail(SILENT_E_SHAPE, "Ambiguous dimension: region shape (h/2, w/2) must be integral (h=%d, w=%d)", plan->h,
                    plan->w);
    return SILENT_OK;
}

// pyramid -> stack -> emit of a batch resident in HBM, with the three-orientation stack (W) or an orientation bank
// (bank). The bank's kernel reduces neither region nor tile maxima: its emit scans gray on its own. Outputs in float32,
// or binary16 when half_out.
static int run_pipeline(silent_plan *plan, const silent_stack_weights *W, const silent_orientation_bank *bank,
                        const void *frames_dev, int batch, float *pyramid_dev, void *orient_dev, void *line_end_dev,
                        bool half_out, int64_t *points_dev, int64_t capacity, int64_t *count_dev, cudaStream_t s)
{
    Workspace &ws = plan->ws;
    if (ws.batch < batch)
        return fail(SILENT_E_CAPACITY, "plan workspace holds %d frames, need %d: call silent_plan_reserve", ws.batch, batch);
    const int n = batch * plan->levels;
    const bool timing = plan->timing;
    if (timing) SILENT_CUDA(cudaEventRecord(plan->ev[0], s));
    WindowGeom geo;
    const bool fuse_windows = !bank && count_dev && window_geometry(plan->h, plan->w, plan->h / 2, plan->w / 2, &geo);
    PairClear winmax_clear;   // the region maxima start at 0: cleared together with the tile flags (see run_stack_stages)
    if (fuse_windows) winmax_clear.b = ws.d_winmax, winmax_clear.b_bytes = (size_t)n * geo.count * sizeof(int);
    int rc = run_stack_stages(plan, W, bank, frames_dev, 0, batch, pyramid_dev, orient_dev, line_end_dev, half_out,
                              fuse_windows ? &geo : nullptr, s, &winmax_clear);
    if (rc != SILENT_OK) return rc;
    if (timing) SILENT_CUDA(cudaEventRecord(plan->ev[2], s));
    if (count_dev) {
        StageRange range("silent:emit");
        const TileMaxima tm = tile_maxima(plan);
        rc = max_value_indices_region(ws.d_gray, n, plan->h, plan->w, plan->h / 2, plan->w / 2, points_dev, capacity,
                                      count_dev, ws.d_select, ws.select_bytes, fuse_windows ? ws.d_winmax : nullptr,
                                      bank ? nullptr : &tm, s);
    }
    if (timing) SILENT_CUDA(cudaEventRecord(plan->ev[3], s));
    return rc;
}

// shared body of silent_pipeline_run and silent_pipeline_run_f16
static int pipeline_run_entry(const char *who, silent_plan *plan, const silent_stack_weights *weights_host,
                              const void *frames_dev, int batch, float *pyramid_dev, void *orient_dev, void *line_end_dev,
                              bool half_out, int64_t *points_dev, int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    const int rc = check_pipeline_args(who, plan, weights_host, frames_dev, batch);
    if (rc != SILENT_OK) return rc;
    return run_pipeline(plan, weights_host, nullptr, frames_dev, batch, pyramid_dev, orient_dev, line_end_dev, half_out,
                        points_dev, capacity, count_dev, (cudaStream_t)stream);
}

int silent_pipeline_run(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_dev, int batch,
                        float *pyramid_dev, float *orient_dev, float *line_end_dev, int64_t *points_dev,
                        int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    return pipeline_run_entry("silent_pipeline_run", plan, weights_host, frames_dev, batch, pyramid_dev, orient_dev,
                              line_end_dev, false, points_dev, capacity, count_dev, stream);
}

int silent_pipeline_run_f16(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_dev, int batch,
                            float *pyramid_dev, uint16_t *orient_dev, uint16_t *line_end_dev, int64_t *points_dev,
                            int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    return pipeline_run_entry("silent_pipeline_run_f16", plan, weights_host, frames_dev, batch, pyramid_dev, orient_dev,
                              line_end_dev, true, points_dev, capacity, count_dev, stream);
}

// shared body of silent_pipeline_run_orientations and silent_pipeline_run_orientations_f16
static int pipeline_run_orientations_entry(const char *who, silent_plan *plan, const silent_orientation_bank *bank_host,
                                           const void *frames_dev, int batch, void *orient_dev, void *line_end_dev,
                                           bool half_out, int64_t *points_dev, int64_t capacity, int64_t *count_dev,
                                           silent_stream stream)
{
    int rc = check_bank(bank_host, who);
    if (rc == SILENT_OK) rc = check_pipeline_args(who, plan, bank_host, frames_dev, batch);
    if (rc != SILENT_OK) return rc;
    if (!pyramid_pair_supported(plan))
        return fail(SILENT_E_SHAPE, "the fused orientation bank needs uint8 frames with 3 colours (frame-pair pyramid path)");
    return run_pipeline(plan, nullptr, bank_host, frames_dev, batch, nullptr, orient_dev, line_end_dev, half_out, points_dev,
                        capacity, count_dev, (cudaStream_t)stream);
}

int silent_pipeline_run_orientations(silent_plan *plan, const silent_orientation_bank *bank_host, const void *frames_dev,
                                     int batch, float *orient_dev, float *line_end_dev, int64_t *points_dev,
                                     int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    return pipeline_run_orientations_entry("silent_pipeline_run_orientations", plan, bank_host, frames_dev, batch,
                                           orient_dev, line_end_dev, false, points_dev, capacity, count_dev, stream);
}

int silent_pipeline_run_orientations_f16(silent_plan *plan, const silent_orientation_bank *bank_host,
                                         const void *frames_dev, int batch, uint16_t *orient_dev, uint16_t *line_end_dev,
                                         int64_t *points_dev, int64_t capacity, int64_t *count_dev, silent_stream stream)
{
    return pipeline_run_orientations_entry("silent_pipeline_run_orientations_f16", plan, bank_host, frames_dev, batch,
                                           orient_dev, line_end_dev, true, points_dev, capacity, count_dev, stream);
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

// shared body of silent_pipeline_run_host and silent_pipeline_run_host_f16: outputs of float32, or binary16 when half_out
static int pipeline_run_host(const char *who, silent_plan *plan, const silent_stack_weights *weights_host,
                             const void *frames_host, int batch, void *orient_host, void *line_end_host, bool half_out,
                             int64_t *points_host, int64_t capacity, int64_t *count_host, silent_stream stream)
{
    int rc = check_pipeline_args(who, plan, weights_host, frames_host, batch);
    if (rc != SILENT_OK) return rc;
    if (capacity < 0) return fail(SILENT_E_INVAL, "capacity must be >= 0");
    rc = silent_plan_reserve(plan, batch);
    if (rc != SILENT_OK) return rc;
    Workspace &ws = plan->ws;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t fbytes = frame_bytes(plan);
    const size_t n = (size_t)batch * plan->levels;
    const size_t image_bytes = (size_t)plan->h * plan->w * 3 * (half_out ? 2 : sizeof(float));   // one output level
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
    // the mirrors are sized for this call's element type; a later call with wider elements replaces them (nothing is
    // in flight on them between calls: every call drains its queues before it returns)
    auto mirror = [&](void *&buf, size_t &bytes) -> int {
        if (buf && bytes >= cap_tensor_bytes) return SILENT_OK;
        cudaFreeHost(buf);
        buf = nullptr, bytes = 0;
        SILENT_CUDA(cudaMallocHost(&buf, cap_tensor_bytes));
        bytes = cap_tensor_bytes;
        return SILENT_OK;
    };
    if (orient_host && !orient_direct) rc = mirror(ws.h_orient, ws.h_orient_bytes);
    if (rc == SILENT_OK && line_end_host && !line_end_direct) rc = mirror(ws.h_line_end, ws.h_line_end_bytes);
    if (rc != SILENT_OK) return rc;
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
            const int rcs = run_stack_stages(plan, weights_host, nullptr, ws.d_frames, f0, nb, nullptr,
                                             orient_host ? ws.d_orient : nullptr, line_end_host ? ws.d_line_end : nullptr,
                                             half_out, fuse_windows ? &geo : nullptr, s);
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
        if (late != cudaSuccess) return fail(SILENT_E_CUDA, "%s: %s", who, cudaGetErrorString(late));
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

int silent_pipeline_run_host(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_host,
                             int batch, float *orient_host, float *line_end_host, int64_t *points_host,
                             int64_t capacity, int64_t *count_host, silent_stream stream)
{
    return pipeline_run_host("silent_pipeline_run_host", plan, weights_host, frames_host, batch, orient_host, line_end_host,
                             false, points_host, capacity, count_host, stream);
}

int silent_pipeline_run_host_f16(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_host,
                                 int batch, uint16_t *orient_host, uint16_t *line_end_host, int64_t *points_host,
                                 int64_t capacity, int64_t *count_host, silent_stream stream)
{
    return pipeline_run_host("silent_pipeline_run_host_f16", plan, weights_host, frames_host, batch, orient_host,
                             line_end_host, true, points_host, capacity, count_host, stream);
}

}  // extern "C"
