// Internal interface between the fused stack (stack_fused.cu), the emit kernels (emit.cu) and the pipeline.
#pragma once

#include "common.cuh"

namespace silent {

// Geometry of max_value_indices_region's pooling windows when they can be reduced inside the stack kernel:
// at most 2 x 2 windows per level and column bounds that are multiples of the 8-pixel run length.
struct WindowGeom {
    int count = 0;   // windows per level (0: not fused, the stand-alone window_max kernel is used instead)
    int ow = 1;      // windows per row of the pooled grid
    int y0[2] = {0, 0}, y1[2] = {0, 0}, x0[2] = {0, 0}, x1[2] = {0, 0};
};

size_t stack_workspace_bytes(int n, int h, int w);
int stack_fused(const void *pyr, int n, int h, int w, int pair_levels, const silent_stack_weights *W, float *orient,
                float *line_end, float *gray, void *workspace, size_t workspace_bytes, const WindowGeom *geo,
                int *winmax, int *tilemax, cudaStream_t stream, cudaEvent_t between_kernels = nullptr,
                bool flags_clean = false);
int stack_clear_flags(void *workspace, int n, int h, int w, cudaStream_t stream);
// the region stack_clear_flags zeroes (256-byte aligned, a multiple of 256 bytes): the pipeline lets the pyramid kernel clear it
void stack_flag_region(void *workspace, int n, int h, int w, void **ptr, size_t *bytes);
// tile grid of stack_b_kernel; tilemax is int [n][nty][ntx] (ordered-int maxima of gray per tile, NaN = 0x7fc00000)
void stack_tile_grid(int h, int w, int *tile_h, int *tile_w, int *nty, int *ntx);
struct TileMaxima {
    const int *data = nullptr;   // null: every tile is scanned
    int tile_h = 0, tile_w = 0, nty = 0, ntx = 0;
};

// orientation bank of W->orientations = 4, 8, 12 or 16 (config C4: 8): pyr -> orient / line_end [n,h,w,nb], gray [n,h,w].
// pyr as in stack_fused: NHWC [n][h][w][3] when pair_levels == 0, else the pyramid_pair_kernel layout. between_kernels
// (optional) is recorded between stack_a and stack_bank_kernel. The caller has passed W through check_bank.
int stack_bank(const void *pyr, int n, int h, int w, int pair_levels, const silent_orientation_bank *W, float *orient,
               float *line_end, float *gray, void *workspace, size_t workspace_bytes, cudaStream_t stream,
               cudaEvent_t between_kernels = nullptr);
// width (SILENT_E_SHAPE) and structure (SILENT_E_STRUCTURE) checks of a bank; host only, no CUDA call
int check_bank(const silent_orientation_bank *W, const char *who);

// pyramid.cu
int pyramid_build(const silent_plan *plan, const void *frames_dev, int batch, float *pyramid_dev, cudaStream_t stream);
bool pyramid_pair_supported(const silent_plan *plan);
size_t pyramid_pair_bytes(const silent_plan *plan, int batch);
// Buffers the frame-pair pyramid kernel zeroes on its way (consumed by the kernels AFTER it: stack_b's tile flags and
// region maxima): a memset in front of the pyramid launch would sit between the previous step's last kernel and this one
// as a stream operation of its own. a: 16-byte aligned, bytes a multiple of 16; b: 4-byte words.
struct PairClear {
    void *a = nullptr;
    size_t a_bytes = 0;
    void *b = nullptr;
    size_t b_bytes = 0;
};
int pyramid_pair_build(const silent_plan *plan, const void *frames_dev, int batch, void *xpair_dev, cudaStream_t stream,
                       const PairClear *clear = nullptr);

// emit.cu
bool window_geometry(int h, int w, int region_h, int region_w, WindowGeom *geo);
int max_value_indices_region(const float *value, int n, int h, int w, int region_h, int region_w, int64_t *points,
                             int64_t capacity, int64_t *count, void *workspace, size_t workspace_bytes,
                             const int *fused_winmax, const TileMaxima *tiles, cudaStream_t stream);
size_t selection_bytes(int n, int h, int w);

}  // namespace silent
