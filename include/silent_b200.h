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

/* SILENT_NV12: 4:2:0 frames as video decoders (NVDEC) and cv2 lay them out, one contiguous [H * 3 / 2, W] uint8 array per
 * frame: H rows of Y, then H / 2 rows of interleaved (U, V) pairs, one pair per 2 x 2 block, U first. A plan of this
 * dtype needs frame_c = num_colors = 3 and even H and W. Every entry point that accepts it computes exactly what it
 * computes on the BGR frame cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12) returns (BT.601 limited range, see
 * silent_nv12_to_bgr): the frames are converted on the GPU first, into a plan-owned buffer, and then take the uint8
 * BGR path. The plan's geometry (levels, level info, tap tables) is the BGR plan's for the same H x W. */
typedef enum silent_dtype { SILENT_U8 = 0, SILENT_F32 = 1, SILENT_NV12 = 2 } silent_dtype;

typedef void *silent_stream; /* cudaStream_t */
typedef struct silent_plan silent_plan;

/* Geometry of the pyramid build: the arguments of zoom.from_image(image, num_colors, center_dimensions, scale)
 * (util/zoom/from_image.py:10-14) plus the frame shape/dtype the reference reads from the ndarray. */
typedef struct silent_params {
    int32_t frame_h, frame_w, frame_c; /* input frames are [H, W, frame_c], channel-interleaved */
    int32_t num_colors;                /* channels 0..num_colors-1 go into the pyramid (from_image.py:54) */
    int32_t center_w, center_h;        /* center_dimensions, (w, h) order as the reference passes it (from_image.py:44) */
    double scale;                      /* zoom_ratio > 1 (from_image.py:38) */
    int32_t frame_dtype;               /* silent_dtype of the frames: SILENT_U8 (camera), SILENT_F32 or SILENT_NV12 */
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
 * silent_pipeline_run, and by silent_pyramid_build on an SILENT_NV12 plan, whose converted frames live in it). May be
 * called again with a larger batch. */
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
/* Frame position of every row and column of `level`: frame_y [h], frame_x [w] (either may be NULL). Along each axis the
 * value is offset + o * (n_in - 1) / (n_out - 1) (scipy.ndimage.zoom's sample position; the factor is 1 when n_out <= 1),
 * computed in float64 when the plan is created and rounded once to float32; offset is the crop's y0 / x0, n_in its
 * height / width and n_out the zoomed size. NaN where silent_plan_level_tables marks the row / column as 0 (o >= valid_h /
 * valid_w, or the position outside [0, n_in - 1]). These are the tables silent_point_records reads. */
int silent_plan_level_coords(const silent_plan *plan, int level, float *frame_y, float *frame_x);
/* Algorithmic HBM bytes of one frame through silent_pipeline_run (SURVEY.md 8(d)): union crop read (1.5 bytes per pixel
 * for SILENT_NV12) + two output tensors; feature points excluded. */
int64_t silent_plan_algorithmic_bytes(const silent_plan *plan);

/* ---- per-operator entry points ----------------------------------------------------------------------------------- */

/* zoom.from_image (util/zoom/from_image.py:10-69) for a batch: frames_dev [batch, H, W, frame_c] of params.frame_dtype
 * -> pyramid_dev [batch * L, h, w, num_colors] float32. Rows/columns the reference leaves uninitialised are 0.
 * SILENT_NV12 plans take frames_dev [batch, H * 3 / 2, W] and need silent_plan_reserve(plan, batch) first. */
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

/* Peak feature points: every 3 x 3 local maximum of a level above its top-percent threshold. This project's composition
 * of two reference operators, not a reference function: the per-level threshold of top_value_points (above) and the 3 x 3
 * max-pool equality get_boosting uses as its non-max (util/energy/boosting.py:18-22). For each level v of value_dev
 * [n,h,w,1] and p = top_percent in [0, 1]:
 *   thr = float32(1 - p) * max(v) + float32(p) * min(v), in float32 without FMA (as silent_top_value_points; a NaN
 *     anywhere in the level makes thr NaN);
 *   pixel (y, x) fires iff v[y,x] > 0 and v[y,x] >= thr and v[y,x] >= the NaN-propagating maximum of the 3 x 3 window
 *     around it, the pixel included and neighbours outside the level ignored (tf.nn.max_pool SAME).
 * So a plateau fires on every one of its pixels (equality, as in the reference's non-max), a level holding a NaN emits
 * nothing, and an all-zero level emits nothing (the v > 0 term: pad_inwards's zero border and the rows a level defines
 * as 0 would otherwise fire wherever thr is 0, e.g. at p = 1). Output and capacity contract as for
 * silent_max_value_indices_region: int64 rows (level, y, x, 0) in row-major order to points_dev[capacity][4], the TOTAL
 * in *count_dev, only the first min(total, capacity) rows written, nothing past capacity. The rows feed
 * silent_point_records / silent_point_patches and silent_pack_points unchanged. Workspace: silent_selection_workspace_bytes.
 * Five kernels on `stream` (the threshold, then four programmatic dependent launches). Argument checks (all on the host,
 * before any CUDA call): null pointers (points_dev may be NULL when capacity is 0), n, h or w <= 0, capacity < 0, or
 * top_percent NaN or outside [0, 1] -> SILENT_E_INVAL; more than 65535 levels or levels of 2^30 pixels or more ->
 * SILENT_E_SHAPE; a short workspace -> SILENT_E_CAPACITY. */
int silent_peak_points(const float *value_dev, int n, int h, int w, double top_percent, int64_t *points_dev,
                       int64_t capacity, int64_t *count_dev, void *workspace_dev, size_t workspace_bytes,
                       silent_stream stream);

/* silent_peak_points on the plan's own gray, [batch * L, h, w], with the plan's own workspace: the gray of the latest
 * silent_pipeline_run* / silent_pipeline_run_host* call on this plan, with the validity and stream rules of gray_dev =
 * NULL in silent_point_records. A caller runs silent_pipeline_run* with count_dev = NULL (no region emit) and then this,
 * and when *count_dev exceeds the capacity redoes only this call with a larger buffer. Argument checks (all on the host,
 * before any CUDA call): those of silent_peak_points (batch <= 0 -> SILENT_E_INVAL; a plan of 0 levels or more than 65535
 * levels in batch * L -> SILENT_E_SHAPE), and batch above the plan's reserve -> SILENT_E_CAPACITY. */
int silent_plan_peak_points(silent_plan *plan, int batch, double top_percent, int64_t *points_dev, int64_t capacity,
                            int64_t *count_dev, silent_stream stream);

/* cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12) for a batch on the GPU: nv12_dev [batch, h * 3 / 2, w] uint8 (layout at
 * SILENT_NV12) -> bgr_dev [batch, h, w, 3] uint8, both contiguous. h and w even. BT.601 limited range in 20-bit fixed
 * point, bit-identical to OpenCV's integer code: with u = U - 128, v = V - 128 of the pixel's 2 x 2 block and
 * y = max(0, Y - 16) * 1220542,
 *   B = sat8((y + 2^19 + 2116026 u) >> 20), G = sat8((y + 2^19 - 852492 v - 409993 u) >> 20),
 *   R = sat8((y + 2^19 + 1673527 v) >> 20)   (arithmetic shift; every sum fits in int32).
 * The same device routine converts the frames of a SILENT_NV12 plan. Argument checks run before any CUDA call. */
int silent_nv12_to_bgr(const uint8_t *nv12_dev, int batch, int h, int w, uint8_t *bgr_dev, silent_stream stream);

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

/* silent_display_tensors over a clip: `steps` consecutive time steps of n images each, time-major (gray_dev
 * [steps*n,h,w,1], image t*n + e is step t of energy slice e). energy_dev [n,oh,ow,1] is updated in place and the four
 * outputs hold steps*n images each, shaped as in silent_display_tensors: the result equals `steps` calls of
 * silent_display_tensors on the consecutive slices of n images, bit for bit. Two launches: the centroid images and block
 * importance of every step at once, then the boosting recurrence of the whole clip in one thread-block cluster per
 * energy slice, its state on chip. A grid no cluster can hold (a band of more than 8192 cells on 16 CTAs: levels far
 * beyond a megapixel at 3 x 3 blocks) takes 2 launches per step instead. scratch_dev: at least
 * silent_display_sequence_scratch_bytes(steps, n, h, w, region_h, region_w) bytes (0 for a non-positive argument). */
size_t silent_display_sequence_scratch_bytes(int steps, int n, int h, int w, int region_h, int region_w);
int silent_display_sequence(const float *gray_dev, int steps, int n, int h, int w, int region_h, int region_w,
                            int half_h, int half_w, float *energy_dev, float exhaustion_max, float excitation_max,
                            int recovery_mode, float normer, float centerer, float *centroids_disp_dev,
                            float *centroids2_disp_dev, float *fired_disp_dev, float *update_disp_dev, void *scratch_dev,
                            size_t scratch_bytes, silent_stream stream);

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
 * frames_host [batch,H,W,frame_c] ([batch,H*3/2,W] on a SILENT_NV12 plan: half the upload of BGR) -> orient_host,
 * line_end_host [batch*L,h,w,3], points_host [capacity][4], *count_host.
 * Copies go through plan-owned pinned staging buffers; synchronises `stream` before returning. Output pointers may be
 * NULL to skip the corresponding device->host copy. */
int silent_pipeline_run_host(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_host,
                             int batch, float *orient_host, float *line_end_host, int64_t *points_host,
                             int64_t capacity, int64_t *count_host, silent_stream stream);

/* ---- binary16 outputs ---------------------------------------------------------------------------------------------
 * The five calls below are their float32 counterparts above with orient and line_end stored as IEEE binary16: each
 * output holds the bit patterns (uint16_t) of the float32 value the counterpart computes, rounded once to nearest even
 * (subnormals kept, overflow to +-inf, NaN stays NaN with an unspecified payload) -- what torch's Tensor.half() does to
 * the float32 result. Everything else is computed from the float32 values exactly as by the counterpart: gray (still
 * float32), the regulator's early-out, and the feature points, which are bit-identical to the counterpart's. Output
 * bytes halve. Arguments, checks (all on the host, before any CUDA call) and status codes are those of the counterpart.
 * uint8 frames through the three-orientation stack stay far inside binary16's range (orient <= ~5.7e3, line_end <= 255),
 * with 11 significant bits (steps of 0.125 just below 255). */
int silent_stack_fused_f16(const float *pyramid_dev, int n, int h, int w, const silent_stack_weights *weights_host,
                           uint16_t *orient_dev, uint16_t *line_end_dev, float *gray_dev, void *workspace_dev,
                           size_t workspace_bytes, silent_stream stream);
int silent_stack_bank_f16(const float *pyramid_dev, int n, int h, int w, const silent_orientation_bank *bank_host,
                          uint16_t *orient_dev, uint16_t *line_end_dev, float *gray_dev, void *workspace_dev,
                          size_t workspace_bytes, silent_stream stream);
int silent_pipeline_run_f16(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_dev, int batch,
                            float *pyramid_dev, uint16_t *orient_dev, uint16_t *line_end_dev, int64_t *points_dev,
                            int64_t capacity, int64_t *count_dev, silent_stream stream);
int silent_pipeline_run_orientations_f16(silent_plan *plan, const silent_orientation_bank *bank_host,
                                         const void *frames_dev, int batch, uint16_t *orient_dev, uint16_t *line_end_dev,
                                         int64_t *points_dev, int64_t capacity, int64_t *count_dev, silent_stream stream);
/* The host-buffer call with binary16 outputs: its pinned staging mirrors and its device-to-host copies are half the
 * bytes of silent_pipeline_run_host's. */
int silent_pipeline_run_host_f16(silent_plan *plan, const silent_stack_weights *weights_host, const void *frames_host,
                                 int batch, uint16_t *orient_host, uint16_t *line_end_host, int64_t *points_host,
                                 int64_t capacity, int64_t *count_host, silent_stream stream);

/* ---- feature-point records ---------------------------------------------------------------------------------------------
 * One record per emitted point, gathered on the device, so that a caller who wants points and what fired there needs
 * neither the host round trip for the count nor the whole output tensors. Reads the first min(*count_dev, capacity) rows
 * (level, y, x, 0) of points_dev (as written by silent_pipeline_run* / silent_max_value_indices_region, level =
 * frame * L + l) and writes, for row i:
 *   coords_dev [capacity][2]: (frame_y, frame_x) of the point, from silent_plan_level_coords (NaN on an axis whose row /
 *     column the level defines as 0);
 *   values_dev [capacity][1 + 2 * channels]: gray, orient[channels], line_end[channels] at (level, y, x), as float32.
 *     orient_dev / line_end_dev are [batch * L, h, w, channels], float32, or binary16 (uint16_t bits) when half = 1,
 *     widened exactly; channels is 3 or an orientation bank's width (4, 8, 12, 16). gray_dev is [batch * L, h, w].
 *   frame_offsets_dev [batch + 1]: int64, the rows of frame b are [frame_offsets[b], frame_offsets[b + 1]) among the
 *     written rows (frame_offsets[batch] = min(count, capacity)).
 * Nothing is written past row `capacity`; *count_dev may exceed it (the emit's total), the records then stop at capacity.
 * gray_dev = NULL reads the plan's own gray: that of the latest silent_pipeline_run* / silent_pipeline_run_host* call on
 * this plan, valid until the next such call on it, or a silent_plan_reserve that grows it (or silent_plan_destroy), and
 * ordered by `stream` (pass the stream of that call, or order the two yourself); batch must not exceed the batch
 * reserved. A row whose (level, y, x) lies outside [batch * L, h, w] gets NaN records. One kernel, launched as a
 * programmatic dependent launch on `stream`: it may start while the emit drains. Argument checks (all on the host,
 * before any CUDA call): null pointers (points, coords and values may be NULL when capacity is 0) or capacity < 0 or half
 * not 0 / 1 or batch <= 0 -> SILENT_E_INVAL; channels not 3, 4, 8, 12, 16 or a plan of 0 levels -> SILENT_E_SHAPE;
 * gray_dev = NULL with batch above the plan's reserve -> SILENT_E_CAPACITY. */
int silent_point_records(const silent_plan *plan, int batch, const int64_t *points_dev, const int64_t *count_dev,
                         int64_t capacity, const void *orient_dev, const void *line_end_dev, int channels, int half,
                         const float *gray_dev, int64_t *frame_offsets_dev, float *coords_dev, float *values_dev,
                         silent_stream stream);

/* ---- feature-point patches ---------------------------------------------------------------------------------------------
 * silent_point_records with the square neighbourhood of side P = 2 * radius + 1 around each point instead of its one
 * pixel, for descriptors, sub-pixel refinement or orientation histograms built from the raw responses. Everything is as
 * for silent_point_records (the rows read, coords_dev, frame_offsets_dev, gray_dev = NULL, the capacity and the launch)
 * except values_dev, which is [capacity][P][P][1 + 2 * channels] float32: pixel (y + dy, x + dx) of the point's level,
 * dy, dx in [-radius, radius], at [radius + dy][radius + dx], holding gray, orient[channels], line_end[channels] there.
 * A patch pixel outside the level's [0, h) x [0, w) is +0.0 in every value (what the stack's SAME zero padding reads
 * there); a row outside [batch * L, h, w] gets NaN in its whole patch. radius = 0 is silent_point_records, bit for bit.
 * Argument checks (all on the host, before any CUDA call): those of silent_point_records, and radius < 0 or radius >
 * SILENT_PATCH_RADIUS_MAX -> SILENT_E_SHAPE. */
#define SILENT_PATCH_RADIUS_MAX 31
int silent_point_patches(const silent_plan *plan, int batch, const int64_t *points_dev, const int64_t *count_dev,
                         int64_t capacity, const void *orient_dev, const void *line_end_dev, int channels, int half,
                         const float *gray_dev, int radius, int64_t *frame_offsets_dev, float *coords_dev,
                         float *values_dev, silent_stream stream);

/* ---- feature-point matches ---------------------------------------------------------------------------------------------
 * Links between the points of consecutive frames of one batch, computed on the device from the records, so that a
 * tracker needs a few bytes per point instead of the patches. Reads the first rows = clamp(*count_dev, 0, capacity) rows
 * (level, y, x, 0) of points_dev [capacity][4] (level = frame * levels + l, sorted by (level, y, x) as every emit writes
 * them; the order is not checked, but nothing outside [0, rows) is read) and their descriptors values_dev
 * [capacity][row_elems] float32 (a record's values, P * P * (1 + 2C) with a patch). Level n of frame f pairs with level
 * n + levels of frame f + 1:
 *   candidates of row i in the next frame: rows j of level_i + levels with |y_j - y_i| <= search_radius and
 *     |x_j - x_i| <= search_radius (level pixels); in the previous frame the same with level_i - levels;
 *   SSD(i, j): for k = 0..31, s_k = +0.0, then for e = k, k + 32, ... < row_elems: d = a_e - b_e, s_k = s_k + d * d;
 *     then for m = 16, 8, 4, 2, 1: s_k = s_k + s_(k xor m); SSD = s_0. Float32, every operation rounded to nearest, no
 *     fused products. Symmetric in i and j bit for bit. A candidate whose SSD is NaN is ignored;
 *   raw link of i in one direction: the candidate of smallest SSD d1 (ties to the smaller row), kept iff
 *     d1 <= float32(max_ratio) * d2 (rounded), d2 the smallest SSD over the other candidates (+inf without any);
 *     max_ratio = 1 turns the test off, and it applies to SSD (Lowe's 0.8 on distances is 0.64 here);
 *   accepted match i -> j: j is i's raw link in the next frame and i is j's raw link in the previous frame.
 * Outputs, over the whole capacity: next_dev [capacity] int64, j or -1; prev_dev [capacity] int64, i for the j above or
 * -1; distance_dev [capacity] float32, SSD(i, next[i]) or NaN where next is -1. Rows at or past `rows` get -1 / -1 / NaN.
 * Matches never span calls: a stream processed in batches keeps one frame of overlap. No plan and no workspace. Two
 * kernels, launched as programmatic dependent launches on `stream`; capacity 0 launches nothing. Argument checks (all
 * on the host, before any CUDA call): a null count_dev, capacity < 0, a null points, values or output pointer with
 * capacity > 0, or max_ratio NaN, <= 0 or > 1 -> SILENT_E_INVAL; row_elems < 1, levels < 1 or search_radius < 0 ->
 * SILENT_E_SHAPE; no CUDA device -> SILENT_E_CUDA. */
int silent_match_points(const int64_t *points_dev, const int64_t *count_dev, int64_t capacity, const float *values_dev,
                        int64_t row_elems, int levels, int search_radius, float max_ratio, int64_t *next_dev,
                        int64_t *prev_dev, float *distance_dev, silent_stream stream);

/* ---- frame-to-frame motion ---------------------------------------------------------------------------------------------
 * How the camera moved between consecutive frames of one batch, and which matches agree with that motion: a 2-D affine
 * map per frame pair, found by a seeded RANSAC on the device from the records and matches, so that only 48 bytes per
 * pair and one byte per point come back. Reads the first rows = clamp(*count_dev, 0, capacity) rows, the batch + 1
 * entries of frame_offsets_dev (the rows of frame f are [lo, hi) = [clamp(frame_offsets[f], 0, rows),
 * clamp(frame_offsets[f + 1], lo, rows)), as silent_point_records writes them), frame_yx_dev [capacity][2] float32 (a
 * record's frame coordinates, 8-byte aligned) and next_dev [capacity] int64 (silent_match_points' links). For each pair
 * f = 0 .. batch - 2:
 *   correspondences: the rows i of frame f, in row order, with 0 <= next[i] < rows and frame_yx[i], frame_yx[next[i]]
 *     all finite (a level that defines an axis as 0 has NaN coordinates, so its rows never take part); M_f of them,
 *     c_k = (y0, x0, y1, x1), k = 0 .. M_f - 1;
 *   model: [y1, x1] = T[:, :2] @ [y0, x0] + T[:, 2] in frame pixels, T float64 [2][3] = (a, b, c; d, e, g);
 *   hypothesis h = 0 .. hypotheses - 1: draws k_d = mulhi64(u_d, M_f) (the high 64 bits of the 128-bit product), d = 0,
 *     1, 2, u_d = splitmix64(seed ^ splitmix64((f << 32) | (h << 2) | d)), splitmix64(z): z += 0x9e3779b97f4a7c15,
 *     z = (z ^ z >> 30) * 0xbf58476d1ce4e5b9, z = (z ^ z >> 27) * 0x94d049bb133111eb, z ^ z >> 31 (64-bit wrapping).
 *     Degenerate if two draws are equal. Otherwise, in float64 and this order: with (y0, x0) = c_k0's source and
 *     dyj = yj - y0, dxj = xj - x0 for the sources of c_k1 (j = 1) and c_k2 (j = 2), D = dy1 * dx2 - dx1 * dy2;
 *     degenerate if !(|D| >= 1) (NaN too). Then per target u (y1, then x1): du1 = u_k1 - u_k0, du2 = u_k2 - u_k0,
 *     a = (du1 * dx2 - dx1 * du2) / D, b = (dy1 * du2 - du1 * dy2) / D, c = u_k0 - (a * y0 + b * x0);
 *   score of a model T: with m = float32(T) (rounded once) and t2 = float32(threshold) * float32(threshold) (rounded),
 *     c_k is an inlier iff e_y * e_y + e_x * e_x <= t2, e_y = y1 - ((m_a * y0 + m_b * x0) + m_c), e_x likewise with
 *     (m_d, m_e, m_g); float32, every operation rounded to nearest, no fused products. A NaN residual is no inlier;
 *   best hypothesis: the most inliers over the hypotheses that are not degenerate, ties to the smaller h;
 *   refit: over the inliers of the best hypothesis, with (py, px, qy, qx) = c_k0 of that hypothesis and, in float64,
 *     Y = y0 - py, X = x0 - px, U = y1 - qy, V = x1 - qx, the 11 sums S of Y, X, YY, YX, XX, U, YU, XU, V, YV, XV (in
 *     that order of the products' factors). Each sum in a fixed order: thread t = 0..255 adds its terms over k = t,
 *     t + 256, ... in order from +0.0 (a correspondence that is no inlier adds nothing); then within each warp of 32
 *     threads s_t = s_t + s_(t xor b) for b = 16, 8, 4, 2, 1; then the warps' lane-0 sums w_0 .. w_7 are added as
 *     ((w_0 + w_1) + w_2) + ... + w_7. With n the inlier count, c00 = Sxx*n - Sx*Sx, c01 = Sx*Sy - Syx*n,
 *     c02 = Syx*Sx - Sxx*Sy, c11 = Syy*n - Sy*Sy, c12 = Syx*Sy - Syy*Sx, c22 = Syy*Sxx - Syx*Syx,
 *     det = (Syy*c00 + Syx*c01) + Sy*c02, and per target (r0, r1, r2, q) = (SYU, SXU, SU, qy), then (SYV, SXV, SV, qx):
 *     a = ((c00*r0 + c01*r1) + c02*r2) / det, b = ((c01*r0 + c11*r1) + c12*r2) / det,
 *     c' = ((c02*r0 + c12*r1) + c22*r2) / det, c = (q + c') - (a * py + b * px);
 *   final model: the refit if its six values are finite and it scores at least as many inliers, else the best
 *     hypothesis's T.
 * Outputs: transform_dev [batch - 1][2][3] float64, the final T, all NaN when M_f < 3 or every hypothesis is degenerate;
 * inlier_count_dev [batch - 1] int64, its inliers (0 then); matched_dev [batch - 1] int64, M_f; inlier_dev [capacity]
 * uint8, 1 iff the row is a correspondence of its pair and an inlier of the final model, 0 elsewhere (every row of the
 * last frame, and at and past `rows`). inlier_count_dev also holds each pair's winner between the kernels. No result
 * depends on the order of atomics, the grid or the warp schedule.
 * workspace_dev: silent_motion_workspace_bytes(capacity) bytes, 16-byte aligned. Matches never span calls, so motion
 * never does either. Three kernels, launched as programmatic dependent launches on `stream`; capacity 0 or batch 1
 * launches nothing and writes nothing (every pair then has M_f = 0). Argument checks (all on the host, before any CUDA
 * call): capacity < 0, batch < 1, a null input, workspace, inlier or (with batch > 1) pair output with capacity > 0, a
 * workspace that is not 16-byte aligned, or threshold NaN, infinite or <= 0 -> SILENT_E_INVAL; hypotheses outside
 * [1, SILENT_MOTION_HYPOTHESES_MAX] -> SILENT_E_SHAPE; workspace_bytes short -> SILENT_E_CAPACITY; no CUDA device ->
 * SILENT_E_CUDA. */
#define SILENT_MOTION_HYPOTHESES_MAX 4096
size_t silent_motion_workspace_bytes(int64_t capacity);
int silent_estimate_motion(const int64_t *frame_offsets_dev, const float *frame_yx_dev, const int64_t *next_dev,
                           const int64_t *count_dev, int64_t capacity, int batch, int hypotheses, float threshold,
                           uint64_t seed, void *workspace_dev, size_t workspace_bytes, double *transform_dev,
                           int64_t *inlier_count_dev, int64_t *matched_dev, uint8_t *inlier_dev, silent_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SILENT_B200_H */
