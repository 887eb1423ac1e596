// Internal definition of the opaque silent_plan.
#pragma once

#include <vector>

#include "common.cuh"

namespace silent {

struct LevelInfo {
    int y0, y1, x0, x1;     // crop of this level in the frame (from_image.py:49-51)
    int valid_h, valid_w;   // rows / cols the reference actually writes (from_image.py:61-62)
};

// Launch geometry of pyramid_pair_kernel for one level: x tiles of kPairTileW output columns; per tile the span of
// aligned 32-bit words of a frame row that its x-taps touch.
constexpr int kPairTileWMax = 85;   // phase H deals the (column, channel) items of a tile over the CTA's threads
constexpr int kPairMaxTiles = 64, kPairMaxLevels = 16;
constexpr int kPairVGroup = 18;   // float2 slots per group of 16 byte-columns in the column-sum buffer (16 + 2 of padding)
constexpr int kPairThreads = 128;   // threads per CTA of pyramid_pair_kernel (measured: 64 / 96 / 192 / 256 slower)
struct PairLevel {
    int ntx = 0, th = 0, vpitch = 0;
    int word_lo[kPairMaxTiles], nwords[kPairMaxTiles];
};

constexpr int kMaxChunks = 16;   // chunks per silent_pipeline_run_host call

// Plan-owned device scratch, sized by silent_plan_reserve(max_batch).
struct Workspace {
    int batch = 0;
    void *d_frames = nullptr;      // [B,H,W,FC] staging for *_host calls ([B,H*3/2,W] on an NV12 plan)
    uint8_t *d_bgr = nullptr;      // NV12 plans only: the converted frames the pyramid reads, [B][frame_stride] bytes
    float *d_pyramid = nullptr;    // [B*L,h,w,C] (NHWC path) or [ceil(B/2)*L][3][h][w] float2 (frame-pair path)
    float *d_orient = nullptr;     // [B*L,h,w,3] staging for *_host calls
    float *d_line_end = nullptr;
    float *d_gray = nullptr;       // [B*L,h,w]
    void *d_select = nullptr;      // selection workspace
    size_t select_bytes = 0;
    void *d_stack = nullptr;       // fused-stack workspace (paired channel-sum tensor)
    size_t stack_bytes = 0;
    int *d_winmax = nullptr;       // [B*L][<=4] per-region maxima reduced inside the stack kernel
    int *d_tilemax = nullptr;      // [B*L][tile rows][tile cols] per-tile maxima of gray (stack_b -> emit)
    int64_t *d_points = nullptr;   // [points_capacity][4]
    int64_t points_capacity = 0;
    int64_t *d_count = nullptr;
    void *h_frames = nullptr;      // pinned mirrors
    void *h_orient = nullptr;      // ... of h_orient_bytes / h_line_end_bytes (sized by the output element type)
    void *h_line_end = nullptr;
    size_t h_orient_bytes = 0, h_line_end_bytes = 0;
    int64_t *h_points = nullptr;
    int64_t *h_count = nullptr;
    // silent_pipeline_run_host: upload / download queues and per-chunk events (chunked, overlapped transfers)
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[kMaxChunks] = {}, ev_done[kMaxChunks] = {};
};

}  // namespace silent

struct silent_plan {
    silent_params params;
    int levels = 0, h = 0, w = 0;
    int union_h = 0, union_w = 0;
    bool on_device = false;
    // the frames the pyramid kernels read: row pitch and frame stride in bytes (frame elements for SILENT_F32). BGR and
    // float frames are read in place (W * FC and H * W * FC). NV12 frames are converted first into ws.d_bgr, whose rows
    // are padded to 16 bytes and whose frames to the texture alignment, so every frame takes the frame-pair path
    int64_t frame_pitch = 0, frame_stride = 0;
    int nv12_y0 = 0, nv12_y1 = 0, nv12_x0 = 0, nv12_x1 = 0;   // NV12: rows / columns converted (all tap rows / columns)
    std::vector<silent::LevelInfo> info;
    std::vector<int32_t> idx_y, idx_x;   // [L][h|w][6], absolute frame row / column, idx[.][0] = -1 => sample is 0
    std::vector<float> w_y, w_x;
    // [L][h|w]: frame row / column of each level row / column, float32(offset + o * (n_in - 1) / (n_out - 1)) from the
    // float64 of axis_table; NaN where idx[.][0] < 0 (the sample is defined as 0). Read by point_records_kernel
    std::vector<float> coord_y, coord_x;
    std::vector<silent::PairLevel> pair;   // per level
    bool pair_ok = false;
    int pair_tile_w = 64;                  // output columns per tile of the frame-pair pyramid kernel (see plan.cu)
    int *d_pair_words = nullptr;           // [L][kPairMaxTiles][4]: (word_lo, nwords, 2^32 / groups + 1, 0) per level and x tile
    int32_t *d_pair_htab = nullptr;        // [L][w][3][12]: phase-H tap offsets in the tile's column-sum row (6 ints) and weights (6 floats)
    int32_t *d_pair_ytab = nullptr;        // [L][h][12]: phase-V table: first tap row's byte offset ([0] < 0: zero row), step, six weights, other offsets (plan.cu)
    cudaTextureObject_t htab_tex = 0;      // d_pair_htab as a linear texture of int4 texels
    int texture_alignment = 0;             // cudaDevAttrTextureAlignment of the plan's device (0: unknown, no textures)
    // linear textures over the callers' frame buffers, keyed by (pointer, bytes). An object may still be read by a
    // kernel in flight, so none is destroyed while the plan lives unless the table is full (then after a device
    // synchronisation): the host-buffer path cycles through its <= kMaxChunks staging slices, callers through a few buffers
    struct FrameTexture {
        const void *ptr = nullptr;
        size_t bytes = 0;
        cudaTextureObject_t tex = 0;
    };
    std::vector<FrameTexture> frame_textures;
    void *d_tables = nullptr;
    int32_t *d_idx_y = nullptr, *d_idx_x = nullptr;
    float *d_w_y = nullptr, *d_w_x = nullptr;
    float *d_coord_y = nullptr, *d_coord_x = nullptr;   // coord_y / coord_x, in the d_tables allocation
    silent::Workspace ws;
    bool timing = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // before pyramid / stack / emit, after emit
    cudaEvent_t ev_mid = nullptr;                               // between the two stack kernels

    ~silent_plan();
};
