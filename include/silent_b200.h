/*
 * silent_b200.h -- C ABI of libsilent_b200.so: pySILEnT's slam_recognition filter pipeline on B200 (sm_100a).
 *
 * The reference (SimLeek/pySILEnT) has no native code: its hot path is Python that builds a TensorFlow-1 graph plus a
 * scipy pyramid builder. Each entry point below cites the reference interface it replaces (paths relative to
 * /root/reference/slam_recognition); INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *  - every function returns 0 (SILENT_OK) or a negative silent_status; silent_last_error() returns a thread-local
 *    message for the last failure on the calling thread.
 *  - the caller owns every buffer. Pointers named *_dev are device pointers on the current CUDA device, *_host are
 *    host pointers. Nothing is allocated inside a call except by silent_plan_create / silent_plan_reserve (plan-owned
 *    tap tables, workspace and staging buffers, freed by silent_plan_destroy).
 *  - every launch is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream) unless the
 *    function name ends in _host, which synchronises before returning.
 *  - tensors are NHWC float32, contiguous: [levels, h, w, C] exactly as the reference feeds its placeholder
 *    (recognition_testing.py:62,130). Filters are HWIO float32 [k, k, Cin, Cout] (constant_convolutions/).
 *  - there is no CPU fallback: without a CUDA device every compute entry point returns SILENT_E_CUDA.
 */
#ifndef SILENT_B200_H
#define SILENT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SILENT_ABI_VERSION 1

typedef enum silent_status {
    SILENT_OK = 0,
    SILENT_E_INVAL = -1,    /* bad argument (null pointer, non-positive size, scale <= 1, ...) */
    SILENT_E_SHAPE = -2,    /* shape / channel count / filter size not supported by this entry point */
    SILENT_E_CAPACITY = -3, /* plan workspace or caller buffer too small */
    SILENT_E_CUDA = -4,     /* CUDA runtime error (message has the cudaError string) */
    SILENT_E_STRUCTURE = -5, /* weights lack the structure the fused stack needs; use the per-operator calls */
    SILENT_E_NCCL = -6       /* NCCL could not be loaded, or reported an error (also asynchronously) */
} silent_status;

typedef enum silent_dtype { SILENT_U8 = 0, SILENT_F32 = 1 } silent_dtype;

typedef void *silent_stream; /* cudaStream_t */
typedef struct silent_plan silent_plan;

/* Geometry of the pyramid build: the arguments of zoom.from_image(image, num_colors, center_dimensions, scale)
 * (util/zoom/from_image.py:10-14) plus the frame shape/dtype the reference reads from the ndarray. */
typedef struct silent_params {
    int32_t frame_h, frame_w, frame_c; /* input frames are [H, W, frame_c], channel-interleaved */
    int32_t num_colors;                /* channels 0..num_colors-1 go into the pyramid (from_image.py:54) */
    int32_t center_w, center_h;        /* center_dimensions, (w, h) order as the reference passes it (from_image.py:44) */
    double scale;                      /* zoom_ratio > 1 (from_image.py:38) */
    int32_t frame_dtype;               /* silent_dtype of the frames: SILENT_U8 (camera) or SILENT_F32 */
    int32_t reserved;
} silent_params;

/* Weights and constants of the fused stack = the graph LineEndDisplayer.compile builds (recognition_testing.py:69-77).
 * All filters HWIO float32. */
typedef struct silent_stack_weights {
    float rgc[3 * 3 * 3 * 3];    /* midget_rgc(2),            filters/rgc.py:9-11 */
    float rgby[3 * 3 * 3 * 3];   /* rgby_3(2),                filters/rgby.py:9-10 */
    float stripe[3 * 3 * 3 * 3]; /* rgb_2d_stripe_tensors(),  filters/orientation.py:19-22 */
    float blur[7 * 7 * 3 * 3];   /* blur_tensor(2, 7),        filters/orientation.py:20,31 */
    float end[3 * 3 * 3 * 3];    /* rgb_2d_end_tensors(),     recognition_testing.py:29 */
    float regulation_value;      /* 1.0,   filters/orientation.py:33 */
    float regulation_root;       /* 0.1,   filters/orientation.py:33 */
    float clip_max;              /* 255,   recognition_testing.py:74 */
    int32_t border;              /* 2,     recognition_testing.py:75 */
} silent_stack_weights;

/* Orientation BANK of BASELINE config C4 (SURVEY 8(d)): 8 orientations built with the reference's per-vector generators
 * stripe_tensor (edge_orientation_detector/stripe_tensor.py:21-70, [3,3,8,8] sliced to its first 3 input channels),
 * blur_tensor(2, 7, 8, 8) (gaussian_blur/gaussian_blur.py:13-54) and end_tensor (oriented_end_detector.py:13-55). */
#define SILENT_BANK 8
typedef struct silent_bank_weights {
    float rgc[3 * 3 * 3 * 3];
    float rgby[3 * 3 * 3 * 3];
    float stripe[3 * 3 * 3 * SILENT_BANK];          /* identical over the 3 input channels */
    float blur[7 * 7 * SILENT_BANK * SILENT_BANK];  /* every slice identical */
    float end[3 * 3 * SILENT_BANK * SILENT_BANK];   /* depthwise: orientation k only feeds orientation k */
    float regulation_value, regulation_root, clip_max;
    int32_t border;
} silent_bank_weights;

/* Orientation bank of any fused width: `orientations` = 4, 8, 12 or 16 (SILENT_E_SHAPE otherwise), n below. Each HWIO
 * array is sized for SILENT_BANK_MAX and holds the n-wide filter packed densely at its front ([3,3,3,n] for the stripe
 * bank, [7,7,n,n] blur, [3,3,n,n] end); the rest is ignored. orientation_bank_filters(n) (pipeline.py) builds them with
 * the generators named at silent_bank_weights. Same structure requirements as silent_bank_weights (SILENT_E_STRUCTURE). */
#define SILENT_BANK_MAX 16
typedef struct silent_orientation_bank {
    int32_t orientations;
    float rgc[3 * 3 * 3 * 3];
    float rgby[3 * 3 * 3 * 3];
    float stripe[3 * 3 * 3 * SILENT_BANK_MAX];                  /* identical over the 3 input channels */
    float blur[7 * 7 * SILENT_BANK_MAX * SILENT_BANK_MAX];      /* every slice identical */
    float end[3 * 3 * SILENT_BANK_MAX * SILENT_BANK_MAX];       /* depthwise */
    float regulation_value, regulation_root, clip_max;
    int32_t border;
} silent_orientation_bank;

int silent_abi_version(void);
const char *silent_last_error(void);
/* Number of CUDA kernels this library has launched in this process so far (bench.py reports the delta per step). */
int64_t silent_launch_count(void);
/* Number of CUDA devices visible, or a negative status. */
int silent_device_count(void);

/* ---- plan ------------------------------------------------------------------------------------------------------ */

/* Replaces the per-call geometry code of image_to_zoom_tensor (from_image.py:43-51): level count, crop bounds and the
 * order-5 spline tap tables of scipy.ndimage.zoom(prefilter=False), computed once in float64 on the host. */
int silent_plan_create(const silent_params *params, silent_plan **out_plan);
void silent_plan_destroy(silent_plan *plan);
/* Pre-size the plan-owned workspace / pinned staging buffers for up to max_batch frames (needed by *_host calls and
 * silent_pipeline_run). May be called again with a larger batch. */
int silent_plan_reserve(silent_plan *plan, int max_batch);

int silent_plan_levels(const silent_plan *plan);                 /* num_scales, from_image.py:45-46 */
int silent_plan_level_hw(const silent_plan *plan, int *h, int *w); /* reversed center_dimensions */
/* Crop [y0,y1) x [x0,x1) of `level` in the frame (from_image.py:49-51) and the rows/cols actually written (:61-62). */
int silent_plan_level_info(const silent_plan *plan, int level, int *y0, int *y1, int *x0, int *x1, int *valid_h,
                           int *valid_w);
/* Test hook: copy the host tap tables of one level. idx_y/w_y: [h][6], idx_x/w_x: [w][6]; idx[.][0] < 0 marks an
 * output row/column that is defined as 0. */
int silent_plan_level_tables(const silent_plan *plan, int level, int32_t *idx_y, float *w_y, int32_t *idx_x,
                             float *w_x);
/* Algorithmic HBM bytes of one frame through silent_pipeline_run (SURVEY.md 8(d)): union crop read + two output
 * tensors; feature points excluded. */
int64_t silent_plan_algorithmic_bytes(const silent_plan *plan);

/* ---- per-operator entry points ----------------------------------------------------------------------------------- */

/* zoom.from_image (util/zoom/from_image.py:10-69) for a batch: frames_dev [batch, H, W, frame_c] of params.frame_dtype
 * -> pyramid_dev [batch * L, h, w, num_colors] float32. Rows/columns the reference leaves uninitialised are 0. */
int silent_pyramid_build(const silent_plan *plan, const void *frames_dev, int batch, float *pyramid_dev,
                         silent_stream stream);

/* tf.nn.conv2d(x, filter, [1,1,1,1], 'SAME') as used by apply_filter (util/apply_filter.py:4-7), optionally followed by
 * tf.maximum(., [0]) (post = 1; filters/rgc.py:13-16, rgby.py:11-12, orientation.py:24-29) and tf.clip_by_value(., 0,
 * clip_max) (post = 2; recognition_testing.py:73-74). cin, cout <= 8; k odd, <= 7. */
int silent_conv2d(const float *x_dev, int n, int h, int w, int cin, const float *filter_hwio_dev, int k, int cout,
                  int post, float clip_max, float *out_dev, silent_stream stream);

/* regulate_tensor(input, blur, regulation_value, regulation_root) (util/regulator/gaussian_regulator_tensor.py:10-36):
 * out = x * (value / pow(min(conv2d(x, blur), 1), root)). blur is [k, k, c, c]. */
int silent_regulate(const float *x_dev, int n, int h, int w, int c, const float *blur_hwio_dev, int k, float value,
                    float root, float *out_dev, silent_stream stream);

/* pad_inwards(tensor, [[0,0],[top,bottom],[left,right],[0,0]]) (util/selection/isolate_rectangle.py:19-23). */
int silent_pad_inwards(const float *x_dev, int n, int h, int w, int c, int top, int bottom, int left, int right,
                       float *out_dev, silent_stream stream);

/* get_value_from_color (util/color/get_value.py:6-12): [n,h,w,c] -> [n,h,w,1]. */
int silent_value_from_color(const float *x_dev, int n, int h, int w, int c, float *out_dev, silent_stream stream);

/* Workspace bytes for the two selection calls below. */
size_t silent_selection_workspace_bytes(int n, int h, int w);

/* max_value_indices_region(color, region_shape, value) (util/selection/top_value_points.py:32-45): writes int64 rows
 * (level, y, x, 0) in row-major order to points_dev[capacity][4] and the TOTAL number of qualifying pixels to
 * *count_dev (it can exceed capacity; only the first `capacity` rows are written). value_dev is [n,h,w,1]. */
int silent_max_value_indices_region(const float *value_dev, int n, int h, int w, int region_h, int region_w,
                                    int64_t *points_dev, int64_t capacity, int64_t *count_dev, void *workspace_dev,
                                    size_t workspace_bytes, silent_stream stream);

/* top_value_points(color, top_percent, value) (util/selection/top_value_points.py:8-29). */
int silent_top_value_points(const float *color_dev, const float *value_dev, int n, int h, int w, int c,
                            double top_percent, float *out_dev, void *workspace_dev, size_t workspace_bytes,
                            silent_stream stream);

/* ---- display tensors that follow gray_line_end_tensor (recognition_testing.py:79-100) --------------------------------- */

/* get_centroids(value_tensor, region_shape) / get_centroids_array (util/centroids.py:21-71): per region_h x region_w
 * block (stride = region, SAME) the value-weighted mean index (x, y) -> corrected_dev [n,oh,ow,2] and the block totals
 * -> total_dev [n,oh,ow,1], oh = ceil(h / region_h); then, if centroids_dev is not NULL, the L1 distance of every pixel
 * to the centroid of its (nearest-upsampled) block -> centroids_dev [n,h,w,1]. value_dev is [n,h,w,1]. */
int silent_get_centroids(const float *value_dev, int n, int h, int w, int region_h, int region_w, float *corrected_dev,
                         float *total_dev, float *centroids_dev, silent_stream stream);

/* tf.image.resize_nearest_neighbor(x, (out_h, out_w)) (align_corners False; recognition_testing.py:83). */
int silent_resize_nearest(const float *x_dev, int n, int h, int w, int c, int out_h, int out_w, float *out_dev,
                          silent_stream stream);

/* get_boosting(input, exhaustion_tensor, exhaustion_max, excitation_max, ...) (util/energy/boosting.py:10-42): 3 x 3
 * max-pool equality on input ** energy -> fired_dev [n,h,w,1] (1 / 0); energy_dev [n,h,w,1] (the tf.Variable) is
 * updated in place: clip((energy * 255 - fired * 255 + recovery) / 255, -exhaustion_max, excitation_max).
 * recovery_mode (util/energy/recovery.py:12-22): 1 constant, 2 input based, 3 both. scratch_dev: [n,h,w] floats. */
int silent_get_boosting(const float *input_dev, float *energy_dev, int n, int h, int w, float exhaustion_max,
                        float excitation_max, int recovery_mode, float *fired_dev, float *scratch_dev,
                        silent_stream stream);

/* The scalar arithmetic between those operators (recognition_testing.py:79-100, boosting.py:36-39), one rounding per
 * written operation. y_dev is only read by SILENT_PW_PRODUCT. */
enum {
    SILENT_PW_DIV255 = 0,          /* x / 255.0                       gray / 255.0, :79 */
    SILENT_PW_INVERT255 = 1,       /* 255 - x * 255                   255 - centroids * 255, :98 */
    SILENT_PW_IMPORTANCE = 2,      /* clip(x * (255 / 4.0), 1, 256) - 1                      :81 */
    SILENT_PW_MUL255 = 3,          /* x * 255                         fired_importants * 255, :98 */
    SILENT_PW_ENERGY_DISPLAY = 4,  /* x * 127.5 + 127.5               boosting.py:37-39 with both maxima 1 */
    SILENT_PW_PRODUCT = 5          /* x * y                           has_fired * input, boosting.py:36 */
};
int silent_pointwise(const float *x_dev, const float *y_dev, size_t count, int kind, float *out_dev,
                     silent_stream stream);

/* Everything LineEndDisplayer.compile builds after gray_line_end_tensor (recognition_testing.py:79-100) in two launches:
 * centroids_disp_dev [n,h,w,1] = 255 - get_centroids(gray / 255)[0] * 255, centroids2_disp_dev [n,half_h,half_w,1] = the
 * same on resize_nearest(gray, (half_h, half_w)), and from importance = clip(total_pool * (255 / 4), 1, 256) - 1 the
 * boosting pair of get_boosting(for_visualizing=True): fired_disp_dev [n,oh,ow,3] = has_fired * importance * 255 and
 * update_disp_dev [n,oh,ow,3] = energy * normer + centerer (normer = 255 / (exhaustion_max + excitation_max), centerer =
 * excitation_max / (exhaustion_max + excitation_max) * 255, boosting.py:37-39); energy_dev [n,oh,ow,1] is updated in place
 * as by silent_get_boosting. oh = ceil(h / region_h), ow = ceil(w / region_w); scratch_dev: 2 * n * oh * ow floats.
 * Bit-identical to the chain silent_pointwise / silent_get_centroids / silent_resize_nearest / silent_get_boosting. */
int silent_display_tensors(const float *gray_dev, int n, int h, int w, int region_h, int region_w, int half_h, int half_w,
                           float *energy_dev, float exhaustion_max, float excitation_max, int recovery_mode, float normer,
                           float centerer, float *centroids_disp_dev, float *centroids2_disp_dev, float *fired_disp_dev,
                           float *update_disp_dev, float *scratch_dev, silent_stream stream);

/* ---- multi-GPU: the path's only exchange is the feature-point gather (SURVEY 8(e)) ------------------------------------- */

/* Packs one rank's points for a single fixed-size all-gather: packed_dev [capacity + 1][4] int64 = the first
 * min(*count_dev, capacity) rows of points_dev with level_offset added to column 0 (level ids in global frame order),
 * zero rows up to capacity, and the row (count, 0, 0, 0) last. points_dev must hold >= capacity rows. No reference
 * counterpart (the reference is single-device, recognition_testing.py:64). */
int silent_pack_points(const int64_t *points_dev, const int64_t *count_dev, int64_t capacity, int64_t level_offset,
                       int64_t *packed_dev, silent_stream stream);

/* The gather itself, over NCCL/NVLink: every rank passes its packed block of `rows` (= capacity + 1) int64x4 rows;
 * packed_recv_dev [nranks][rows][4] receives all blocks in rank order (= global frame order when ranks own contiguous
 * frame blocks). One ncclAllGather on `stream` (asynchronous; use a side stream to overlap the next batch's kernels).
 * NCCL is bound at run time (dlopen of the libnccl.so.2 already loaded in the process, e.g. PyTorch's, else the system's).
 * Communicator set-up is the usual NCCL pattern: rank 0 calls silent_comm_unique_id (128 bytes), the host ships the id
 * to every rank (any channel: torch.distributed, MPI, a file), every rank calls silent_comm_create on its own device.
 * silent_gather_points and silent_comm_check report asynchronous NCCL errors of earlier collectives (SILENT_E_NCCL). */
typedef struct silent_comm silent_comm;
int silent_comm_unique_id(void *id_out_128_bytes);
int silent_comm_create(const void *id_128_bytes, int nranks, int rank, silent_comm **out_comm);
void silent_comm_destroy(silent_comm *comm);
int silent_comm_check(silent_comm *comm);
int silent_gather_points(silent_comm *comm, const int64_t *packed_send_dev, int64_t rows, int64_t *packed_recv_dev,
                         silent_stream stream);

/* ---- fused path ---------------------------------------------------------------------------------------------------- */

/* S1-S7 of LineEndDisplayer.compile (recognition_testing.py:69-77) fused into two kernels (cut at the one-channel
 * rgby channel sum, which lives in workspace_dev: silent_stack_workspace_bytes(n, h, w)): pyramid_dev [n,h,w,3] ->
 * orient_dev (orient_tensor), line_end_dev (padded_line_end_tensor), both [n,h,w,3], and gray_dev [n,h,w,1]
 * (gray_line_end_tensor). Any output pointer may be NULL to skip its store. Returns SILENT_E_STRUCTURE when the weights
 * are not (stripe: identical input-channel slices; blur: all slices identical), which the reference's generators
 * always produce.
 * PRECONDITION: every input value is finite with magnitude <= 1e30. The fused kernels skip exact-zero weights, share
 * sub-kernels between output channels (rgby_3's surround, the end filter's "other channel" kernel, the stripe filter's
 * point symmetry -- each detected bitwise on the weights) and leave the 7x7 blur out where it is provably >= 1; all of
 * that is exact for finite data, but NaN / Inf inputs would not propagate the way the reference graph propagates them
 * (0 * inf = NaN). Callers with such data use the per-operator entry points (silent_conv2d, silent_regulate, ...), as
 * LineEndPipeline.run does. uint8 frames (silent_pipeline_run*) always satisfy the precondition. */
size_t silent_stack_workspace_bytes(int n, int h, int w);
int silent_stack_fused(const float *pyramid_dev, int n, int h, int w, const silent_stack_weights *weights_host,
                       float *orient_dev, float *line_end_dev, float *gray_dev, void *workspace_dev,
                       size_t workspace_bytes, silent_stream stream);

/* The orientation bank's stack on an NHWC pyramid: pyramid_dev [n,h,w,3] -> rgc -> rgby -> stripe bank -> regulator ->
 * end bank -> mask -> mean, orient_dev / line_end_dev [n,h,w,nb], gray_dev [n,h,w,1] (nb = bank_host->orientations; any
 * output may be NULL). Two kernels: stack_a (as in silent_stack_fused) and stack_bank_kernel. Workspace size and the
 * finite-input PRECONDITION as for silent_stack_fused. The width and structure checks (SILENT_E_SHAPE,
 * SILENT_E_STRUCTURE) run on the host before any CUDA call. */
int silent_stack_bank(const float *pyramid_dev, int n, int h, int w, const silent_orientation_bank *bank_host,
                      float *orient_dev, float *line_end_dev, float *gray_dev, void *workspace_dev, size_t workspace_bytes,
                      silent_stream stream);

/* The whole hot path for a batch resident in HBM: frames -> pyramid -> S1-S7 -> feature points (S8, region =
 * (h/2, w/2), recognition_testing.py:40,90-91). Uses the plan workspace (silent_plan_reserve(batch) first).
 * Outputs as in silent_stack_fused / silent_max_value_indices_region; pyramid_dev may be NULL (plan scratch is used). */
int silent_pipeline_run(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_dev, int batch,
                        float *pyramid_dev, float *orient_dev, float *line_end_dev, int64_t *points_dev,
                        int64_t capacity, int64_t *count_dev, silent_stream stream);

/* The same path with the 8-orientation bank (config C4): frames -> pyramid -> rgc -> rgby -> stripe bank -> regulator ->
 * end bank -> mask -> mean -> feature points; orient_dev / line_end_dev are [batch*L, h, w, 8]. uint8 frames with 3 colours
 * only; SILENT_E_STRUCTURE when the bank lacks the generators' structure (use the per-operator calls then). Equal to
 * silent_pipeline_run_orientations with the same 8-wide bank. */
int silent_pipeline_run_bank(silent_plan *plan, const silent_bank_weights *weights_host, const void *frames_dev, int batch,
                             float *orient_dev, float *line_end_dev, int64_t *points_dev, int64_t capacity,
                             int64_t *count_dev, silent_stream stream);

/* The same path for a bank of 4, 8, 12 or 16 orientations: orient_dev / line_end_dev are [batch*L, h, w, nb]. Same
 * preconditions as silent_pipeline_run_bank (uint8 frames, 3 colours, frame-pair pyramid path). The bank's width and
 * structure are checked on the host before any CUDA call (SILENT_E_SHAPE, SILENT_E_STRUCTURE). */
int silent_pipeline_run_orientations(silent_plan *plan, const silent_orientation_bank *bank_host, const void *frames_dev,
                                     int batch, float *orient_dev, float *line_end_dev, int64_t *points_dev,
                                     int64_t capacity, int64_t *count_dev, silent_stream stream);

/* Measurement hook: when enabled, silent_pipeline_run (and the two bank entries above) brackets its stages with CUDA
 * events on the launching stream.
 * silent_plan_stage_ms synchronises those events and returns the device time of the LAST run's pyramid, fused-stack and
 * emit stages in milliseconds. */
int silent_plan_enable_timing(silent_plan *plan, int enable);
int silent_plan_stage_ms(silent_plan *plan, float *pyramid_ms, float *stack_ms, float *emit_ms);
/* the fused stack's two kernels separately: x -> channel sum (stack_a) and channel sum -> outputs (stack_b, or
 * stack_bank_kernel on the bank entries) */
int silent_plan_stack_split_ms(silent_plan *plan, float *stack_a_ms, float *stack_b_ms);

/* Same, with HOST buffers on both sides: the drop-in for LineEndDisplayer.callback (recognition_testing.py:136-144):
 * frames_host [batch,H,W,frame_c] -> orient_host, line_end_host [batch*L,h,w,3], points_host [capacity][4], *count_host.
 * Copies go through plan-owned pinned staging buffers; synchronises `stream` before returning. Output pointers may be
 * NULL to skip the corresponding device->host copy. */
int silent_pipeline_run_host(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_host,
                             int batch, float *orient_host, float *line_end_host, int64_t *points_host,
                             int64_t capacity, int64_t *count_host, silent_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SILENT_B200_H */
