/*
 * mavd.h — C ABI of the B200-native mav-detection hot path (libmavd.so).
 *
 * The reference (evroon/mav-detection) has no FFI layer: its boundary is a set of Python call
 * signatures (SURVEY.md §8b).  Every entry point below names the reference interface it replaces;
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *  - plain pointers and sizes only; `stream` is a cudaStream_t passed as void* (NULL = default stream)
 *  - every function returns an int status (MAVD_OK == 0); nothing throws across this boundary;
 *    mavd_last_error() returns a thread-local message for the last non-zero status
 *  - pointers prefixed d_ are DEVICE pointers, h_ are HOST pointers
 *  - all device entry points are stream-ordered and never retain caller pointers past the call (small host
 *    arrays such as the imu are copied into library-owned pinned staging before the call returns)
 *  - a handle owns ONE set of scratch buffers: drive it from one stream at a time (calls on the same stream, or
 *    calls separated by a synchronisation); use one handle per concurrent stream
 *  - entry points that take a handle switch to the handle's device for the duration of the call and restore the
 *    caller's current device before returning; the handle-less entry points run on the CURRENT device, which
 *    must be the one `stream` and the buffers belong to
 *  - frames are dense row-major (H, W) uint8; flow is dense (H, W, 2) float32, x displacement first
 *    (the layout cv2.calcOpticalFlowFarneback / Dataset.get_flow_uv return)
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    MAVD_ERR_CUDA
 */
#ifndef MAVD_H_
#define MAVD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAVD_ABI_VERSION 3

enum {
    MAVD_OK = 0,
    MAVD_ERR_INVALID = 1,      /* bad shape / parameter / null pointer  -> ValueError   */
    MAVD_ERR_CUDA = 2,         /* CUDA runtime failure                  -> RuntimeError */
    MAVD_ERR_UNSUPPORTED = 3,  /* parameter outside the supported range -> ValueError   */
    MAVD_ERR_NOMEM = 4         /* device allocation failed              -> MemoryError  */
};

/* cv2 flag values accepted in mavd_farneback_params.flags */
#define MAVD_FARNEBACK_GAUSSIAN 256 /* cv2.OPTFLOW_FARNEBACK_GAUSSIAN */

#define MAVD_N_SAMPLE_PAIRS 1000  /* focus_of_expansion.py:65 (N) */
#define MAVD_SAMPLES_PER_FRAME (4 * MAVD_N_SAMPLE_PAIRS) /* 2000 row draws then 2000 column draws */
#define MAVD_MAX_BOXES 32         /* component boxes kept per frame record */
#define MAVD_HOST_SLOTS 3         /* batches that may be in flight through mavd_submit_host */
#define MAVD_MAX_DETECTIONS 256   /* largest max_det of a detection table */

/* Arguments of cv2.calcOpticalFlowFarneback as called at src/farneback.py:76-80. */
typedef struct mavd_farneback_params {
    double pyr_scale;   /* < 1 */
    int32_t levels;     /* N -> up to N+1 pyramid images, capped at 32 px */
    int32_t winsize;    /* 2 <= winsize <= 63 */
    int32_t iterations; /* >= 1 */
    int32_t poly_n;     /* 1 <= poly_n <= 8 */
    double poly_sigma;
    int32_t flags;      /* 0 or MAVD_FARNEBACK_GAUSSIAN */
} mavd_farneback_params;

typedef struct mavd_config {
    int32_t device;     /* CUDA device ordinal */
    int32_t width;      /* frame width  W */
    int32_t height;     /* frame height H */
    int32_t max_pairs;  /* largest batch (frame pairs) one call may carry */
    mavd_farneback_params farneback;
} mavd_config;

/* Per-frame IMU input of Detector.derotate (src/detector.py:70-117):
 * ang = Dataset.get_angular_difference(i-1, i), dt = Dataset.get_delta_time(i).
 * derotate == 0 reproduces the `current_frame_index < 1` pass-through (flow stays float32). */
typedef struct mavd_imu {
    double ang[3];
    double dt;
    int32_t derotate;
    int32_t _pad;
} mavd_imu;

/* Tunables that are public attributes of FocusOfExpansion (src/focus_of_expansion.py:22-23)
 * and the hard-coded mask constants of src/processor.py:333-341. */
typedef struct mavd_detect_params {
    double magnitude_threshold; /* 2.5  */
    double ransac_threshold;    /* 30.0 */
    double dyn_offset;          /* 0.25 */
    double dyn_base;            /* 0.5  */
    double dyn_gain;            /* 8.0  */
    double dyn_min_mag;         /* 0.5  */
    double fixed_min_mag;       /* 1.0  */
    double fixed_angle;         /* 15.0 */
} mavd_detect_params;

/* Launch-shape choices that never change results.  Each default is the form that measured fastest on the B200; each
 * other position selects a path that production still runs for some inputs, so tests use it as the bit-identity
 * reference of the default.  Set once after mavd_create with mavd_set_tuning while the handle is idle;
 * tools/gpu_ab.sh A/Bs them through bench.py --tune. */
typedef struct mavd_tuning {
    int32_t mat_coord;    /* level-entry matrices: 0 = recompute resize coordinates (float32 when exact), 1 = read
                             the host tables, 2 = always recompute in float64 (default 0) */
    int32_t pyr_staged;   /* pyramid: horizontal pass of the coarse levels through shared memory (default 1) */
    int32_t use_graph;    /* replay the per-batch launch sequence from a CUDA graph keyed by (n_pairs, pair_stride,
                             outputs requested) instead of launching kernel by kernel (default 1) */
    int32_t polyexp_tma;  /* polynomial expansion: tile staged by one TMA box (default 1) */
    int32_t iter_small_tiles; /* fused iteration: 64 x 16 tiles for launches too small to fill the GPU with 64 x 32
                                 ones (single pairs, coarse levels; default 1) */
    int32_t use_pdl;      /* programmatic dependent launch: every kernel of the batch is set up while its predecessor
                             on the stream drains and waits for it with griddepcontrol.wait, so launch latency and
                             the ramp of the first wave leave the critical path (default 1) */
    int32_t pyr_sweep;    /* pyramid: exact power-of-two levels (pyr_scale 0.5) through the sweep / vectorised kernels;
                             0 = off, 1 = on with an automatic band count (default), n >= 2 = on with n bands */
    int32_t reserved[1];
} mavd_tuning;

/* Optional per-frame inputs of the detection stages.  All pointers are DEVICE pointers for the d_ entry points and
 * HOST pointers for the _host entry points; every member may be NULL.
 * sky / seg: (H, W) uint8 per frame, stride in bytes between frames (0 = one image shared by all frames; H*W = one per
 * frame), or 1 bit per pixel when the MAVD_HOST_*_PACKED flag of the host call says so.
 * gt_flow: (n, H, W, 2) float32 ground-truth flow, Dataset.get_gt_of (src/processor.py:309-310): derotated like the
 * estimated flow and summed over segmentation > 127 into stats.gt_flow_sum (drone_flow_avg_gt, processor.py:344). */
typedef struct mavd_aux_inputs {
    const uint8_t* sky; int64_t sky_stride;
    const uint8_t* seg; int64_t seg_stride;
    const float* gt_flow;
} mavd_aux_inputs;

/* flags of mavd_submit_host_ex / mavd_detect_host_ex */
#define MAVD_HOST_BGR 1           /* h_frames are (H, W, 3) BGR frames, converted to gray on the device */
#define MAVD_HOST_SEG_PACKED 2    /* aux.seg is 1 bit per pixel (bit set = 255), mavd_packed_mask_bytes per frame */
#define MAVD_HOST_SKY_PACKED 4    /* aux.sky is 1 bit per pixel (bit set = sky) */
#define MAVD_HOST_FIXED_PACKED 8  /* h_fixed_out receives 1 bit per pixel, mavd_packed_mask_bytes per frame */
#define MAVD_HOST_COPY_ONLY 16    /* move the bytes (and pack / unpack) but skip the compute: the host-feed ceiling */

/* Integer reductions behind FrameResult (src/frame_result.py:4-17, src/processor.py:343-362). */
typedef struct mavd_frame_stats {
    double max_phi;          /* FocusOfExpansion.max_flow (focus_of_expansion.py:179) */
    int64_t n_total;         /* pixels set in total_mask      */
    int64_t n_fixed;         /* pixels set in estimate_fixed  */
    int64_t positives;       /* calculate_tpr_fpr: sum(gt > 127)            (im_helpers.py:245) */
    int64_t negatives;       /* sum(255 - gt > 127)                           (im_helpers.py:246) */
    int64_t tp_total, fp_total; /* against 255*total_mask                     (processor.py:351) */
    int64_t tp_fixed, fp_fixed; /* against 255*estimate_fixed                 (processor.py:350) */
    int32_t seg_bbox[4];     /* get_simple_bounding_box(segmentation): x0,y0,x1,y1 or -1 (im_helpers.py:55-84) */
    double seg_flow_sum[2];  /* sum of derotated flow over segmentation > 127 (processor.py:343) */
    double gt_flow_sum[2];   /* the same sum for the derotated GROUND-TRUTH flow (processor.py:309-310,344); 0 when no
                                ground-truth flow was given */
} mavd_frame_stats;

typedef struct mavd_frame_record {
    double foe[2];            /* FrameResult.foe_dense */
    int32_t n_intersections;  /* K of focus_of_expansion.py:85 */
    int32_t n_labels;         /* components of estimate_fixed (may exceed MAVD_MAX_BOXES) */
    mavd_frame_stats stats;
    int32_t boxes[MAVD_MAX_BOXES][5]; /* left, top, width, height, area; raster first-appearance order */
} mavd_frame_record;

/* One entry of a frame's detection table: an 8-connected component of estimate_fixed (or of the mask given to
 * mavd_detections).  A table lists the max_det largest components of a frame, ordered by area descending, then label
 * ascending; entries past min(n_labels, max_det) are all zero.  Every frame's table depends on that frame alone. */
typedef struct mavd_detection {
    int32_t label;        /* canonical label as mavd_ccl numbers it (raster first appearance); 0 = unused entry */
    int32_t box[4];       /* left, top, width, height */
    int32_t area;
    int64_t sum_x, sum_y; /* sums of column and row indices over the pixels: centroid = sum / area, exact */
    double flow_sum[2];   /* sum over the pixels of the derotated flow (mavd_derotate's float64 values; the float32
                             flow widened when imu.derotate == 0).  Summed with float64 atomics: reproducible to the
                             rounding of the summation order, not bit for bit */
} mavd_detection;        /* 56 bytes */

/* Arguments of cv2.goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, mask, blockSize, gradientSize)
 * (Shi-Tomasi corners; the Harris detector is not supported). */
typedef struct mavd_gftt_params {
    int32_t max_corners;     /* corners written per frame (>= 0); the count returned is never limited */
    double quality_level;    /* > 0 */
    double min_distance;     /* >= 0 */
    int32_t block_size;      /* 1..31 */
    int32_t gradient_size;   /* 3 */
} mavd_gftt_params;

/* cv2 flag and termination-criteria values of mavd_lk_params */
#define MAVD_LK_GET_MIN_EIGENVALS 8 /* cv2.OPTFLOW_LK_GET_MIN_EIGENVALS: err = the window's minimum eigenvalue */
#define MAVD_LK_MAX_LEVEL 16        /* largest max_level accepted (levels smaller than the window are never used) */
#define MAVD_TERM_COUNT 1           /* cv2.TERM_CRITERIA_COUNT */
#define MAVD_TERM_EPS 2             /* cv2.TERM_CRITERIA_EPS */

/* Arguments of cv2.calcOpticalFlowPyrLK(prev, next, prevPts, None, winSize, maxLevel, criteria, flags,
 * minEigThreshold).  OPTFLOW_USE_INITIAL_FLOW is not supported. */
typedef struct mavd_lk_params {
    int32_t win_w, win_h;     /* 3..63 each */
    int32_t max_level;        /* 0..MAVD_LK_MAX_LEVEL */
    int32_t criteria_type;    /* MAVD_TERM_COUNT | MAVD_TERM_EPS bits: without COUNT 30 iterations, without EPS 0.01 */
    int32_t criteria_count;   /* clamped to 0..100 */
    double criteria_eps;      /* clamped to 0..10 */
    int32_t flags;            /* 0 or MAVD_LK_GET_MIN_EIGENVALS */
    double min_eig_threshold;
} mavd_lk_params;

typedef struct mavd_handle_s* mavd_handle;

/* ---- library ---- */
int mavd_abi_version(void);
const char* mavd_last_error(void);
void mavd_default_detect_params(mavd_detect_params* out);

/* ---- lifecycle: one handle per (device, W, H, Farneback parameters).  Owns all workspace. ---- */
int mavd_create(const mavd_config* cfg, mavd_handle* out);
int mavd_destroy(mavd_handle h);
int mavd_workspace_bytes(mavd_handle h, size_t* out);
void mavd_default_tuning(mavd_tuning* out);
int mavd_set_tuning(mavd_handle h, const mavd_tuning* t); /* the handle must be idle; invalidates captured graphs */
int mavd_get_tuning(mavd_handle h, mavd_tuning* out);
/* Pyramid geometry actually used: n_images = capped levels + 1; arrays sized >= 16, finest first. */
int mavd_level_info(mavd_handle h, int32_t* n_images, int32_t* widths, int32_t* heights);

/* ---- stage 0 (next-row f1): cv2.cvtColor(img, COLOR_BGR2GRAY) at src/farneback.py:74 ---- */
int mavd_bgr2gray(const uint8_t* d_bgr, uint8_t* d_gray, int64_t n_pixels, void* stream);

/* ---- stage 1: cv2.calcOpticalFlowFarneback(prev, next, None, ...) — src/farneback.py:76-80 ----
 * d_frames holds dense (H, W) uint8 frames; pair p uses frames p*pair_stride and p*pair_stride+1.
 * pair_stride 1: a sequence of n_pairs+1 frames (each frame's pyramid + polynomial expansion is
 * computed once and shared by its two pairs); pair_stride 2: n_pairs independent (prev, next) pairs.
 * d_flow receives n_pairs dense (H, W, 2) float32 fields. */
int mavd_farneback(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride,
                   float* d_flow, void* stream);

/* Test tap: copy an internal buffer of the LAST mavd_farneback call out as a dense array.
 * kind 0: pyramid image (h_l, w_l); 1: polynomial expansion R (h_l, w_l, 5), index = frame;
 * 2: matrices M after the last update (h_l, w_l, 5), index = pair; 3: level flow (h_l, w_l, 2). */
int mavd_farneback_tap(mavd_handle h, int32_t kind, int32_t level, int32_t index, float* d_out,
                       void* stream);

/* ---- stage 1.5: Detector.derotate — src/detector.py:70-117.  d_out is (H, W, 2) float64. ---- */
int mavd_derotate(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, double* d_out,
                  void* stream);
/* The same for a flow that is already float64 (NumPy promotes nothing then: flow - derotation, src/detector.py:117). */
int mavd_derotate_f64(mavd_handle h, const double* d_flow, int32_t n, const mavd_imu* h_imu, double* d_out,
                      void* stream);

/* ---- stage 2: FocusOfExpansion.get_FOE_dense + ransac — src/focus_of_expansion.py:32-86 ----
 * d_samples: per frame MAVD_SAMPLES_PER_FRAME int32 laid out [ry(2000) | rx(2000)], the two
 * np.random.randint draws of focus_of_expansion.py:69-71 made by the host in frame order.
 * Derotation is applied inline to the sampled vectors.  d_foe: n x 2 float64 (x, y); (0,0) = none. */
int mavd_foe(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu,
             const mavd_detect_params* prm, const int32_t* d_samples, double* d_foe,
             int32_t* d_n_intersections, void* stream);

/* FocusOfExpansion.get_FOE_dense(flow_uv) taken literally (src/focus_of_expansion.py:56-86): the flow is
 * used as given — float32 (flow_is_f64 == 0) or float64 (an already derotated field) — no IMU. */
int mavd_foe_dense(mavd_handle h, const void* d_flow, int32_t flow_is_f64, int32_t n,
                   const mavd_detect_params* prm, const int32_t* d_samples, double* d_foe,
                   int32_t* d_n_intersections, void* stream);

/* FocusOfExpansion.ransac(estimates) (src/focus_of_expansion.py:32-54): d_estimates is (k, 2) float64;
 * d_foe receives the winning estimate, (0, 0) when no estimate has another one within the threshold. */
int mavd_ransac(mavd_handle h, const double* d_estimates, int32_t k, double ransac_threshold, double* d_foe,
                void* stream);

/* FocusOfExpansion.get_phi(flow, FoE) (src/focus_of_expansion.py:150-184) on the flow as given: d_phi has
 * the flow's dtype, (n, H, W) dense.  d_max_phi (nullable, n float64) is the max_flow side effect (:179). */
int mavd_get_phi(mavd_handle h, const void* d_flow, int32_t flow_is_f64, int32_t n, const double* d_foe,
                 void* d_phi, double* d_max_phi, void* stream);

/* ---- stage 3: FocusOfExpansion.get_phi + mask block — focus_of_expansion.py:150-184,
 *      processor.py:307,333-341 (+ the reductions of processor.py:343-362 when d_seg is given) ----
 * d_sky / d_seg: (H, W) uint8 per frame (stride 0 = one image shared by all frames), nullable.
 * d_phi: nullable; float64 (H, W) per frame when imu.derotate != 0, float32 otherwise (the dtype
 * the reference returns); the buffer is always n * H * W * 8 bytes, float32 results use the front.
 * d_total / d_fixed: (H, W) uint8 0/1 masks (total_mask, estimate_fixed); either may be NULL.
 * When d_phi is NULL the masks are pre-decided from a float32 estimate with guard bands and only
 * borderline pixels take the float64 path (results stay bit-exact); stats.max_phi is then -1 for the
 * derotated frames (not evaluated). */
int mavd_residual_masks(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu,
                        const mavd_detect_params* prm, const double* d_foe,
                        const uint8_t* d_sky, int64_t sky_stride, const uint8_t* d_seg, int64_t seg_stride,
                        void* d_phi, uint8_t* d_total, uint8_t* d_fixed, mavd_frame_stats* d_stats,
                        void* stream);

/* ---- stand-alone im_helpers seams (no handle needed) ----
 * im_helpers.get_magnitude (src/im_helpers.py:150-159): np.linalg.norm(flow, axis=-1) in the flow's dtype. */
int mavd_magnitude(const void* d_flow, int32_t flow_is_f64, int64_t n_pixels, void* d_out, void* stream);
/* im_helpers.get_simple_bounding_box (src/im_helpers.py:55-84) of a uint8 (H, W, C) image: d_out5 receives
 * {start_x, start_y, end_x, end_y, max(img)}; all four coordinates are -1 when no element exceeds 0.1*max. */
int mavd_simple_bbox(const uint8_t* d_img, int32_t width, int32_t height, int32_t channels, int32_t* d_out5,
                     void* stream);
/* im_helpers.calculate_tpr_fpr (src/im_helpers.py:244-252) integer part: d_counts4 = {positives, negatives,
 * true_positives, false_positives} for a uint8 ground truth and an int64 image (255 * mask at processor.py:350). */
int mavd_tpr_fpr_counts(const uint8_t* d_gt, const int64_t* d_img, int64_t n, int64_t* d_counts4, void* stream);

/* ---- next-row f4: the visualisation Farneback.process() returns (src/farneback.py:83-99) ----
 * cartToPolar -> hue / value bytes (value = 2 * min-max normalised magnitude, wrapping like the NumPy uint8
 * store) -> pixels with value 0 become (127, 255, 255) -> HSV2BGR.  d_bgr: n_pixels x 3 uint8.
 * d_scratch3: 3 uint32 of device scratch; on return [2] = number of pixels with a non-zero value byte
 * (0 = the reference's `invalid_frame`). */
int mavd_flow_vis(const float* d_flow, int64_t n_pixels, uint8_t* d_bgr, uint32_t* d_scratch3, void* stream);

/* ---- next-row f4: the image payloads Processor.run_detection writes (src/processor.py:324,364-376,385-392) ----
 * mavd_phi_colormap: im_helpers.apply_colormap(im_helpers.to_rgb(phi, max_value)) (src/im_helpers.py:112-135,162-201):
 * v = uint8(around(|phi| * 255 / max_value)) evaluated in phi's own dtype (float32 phi stays float32), then OpenCV's JET
 * table.  d_gray_rgb (nullable) receives to_rgb's (n_pixels, 3) image, d_bgr (nullable) the colour-mapped one. */
int mavd_phi_colormap(const void* d_phi, int32_t phi_is_f64, int64_t n_pixels, double max_value, uint8_t* d_gray_rgb,
                      uint8_t* d_bgr, void* stream);
/* mavd_mask_overlay: mask_rgb = frame with (150, 0, 150) where estimate_fixed is set; cv2.addWeighted(frame, 0.2,
 * mask_rgb, 0.8, 0) (src/processor.py:385-392).  d_frame is (n_pixels, channels) uint8 with channels 3 (BGR, as
 * Dataset.get_frame delivers) or 1 (gray, replicated); d_out (n_pixels, 3).  d_mask_rgb (nullable) receives
 * im_helpers.to_rgb(255 * estimate_fixed) (src/processor.py:364). */
int mavd_mask_overlay(const uint8_t* d_frame, int32_t channels, const uint8_t* d_mask, int64_t n_pixels, uint8_t* d_out,
                      uint8_t* d_mask_rgb, void* stream);

/* ---- stage 4 (not in the reference, SURVEY D3/a17): 8-connected components of a mask ----
 * Labels are numbered 1..n by first appearance in a raster scan (0 = background).
 * d_boxes: n x max_boxes x 5 int32 [left, top, width, height, area]; d_n_labels: n int32 (true count).
 * d_labels may be NULL when only the count and the boxes are wanted. */
int mavd_ccl(mavd_handle h, const uint8_t* d_mask, int32_t n, int32_t* d_labels, int32_t* d_boxes,
             int32_t max_boxes, int32_t* d_n_labels, void* stream);

/* Detection tables of n masks (H, W) uint8, non-zero = foreground: d_det receives n x max_det mavd_detection,
 * 1 <= max_det <= MAVD_MAX_DETECTIONS.  d_flow (nullable) is (n, H, W, 2) float32 and then needs h_imu (n entries): each
 * flow_sum adds mavd_derotate's value of every pixel; without a flow flow_sum is 0.  The first call that asks a handle
 * for a table allocates (max_pairs x (ceil(W/2) * ceil(H/2) + 1)) int32 of per-label workspace. */
int mavd_detections(mavd_handle h, const uint8_t* d_mask, int32_t n, const float* d_flow, const mavd_imu* h_imu,
                    int32_t max_det, mavd_detection* d_det, void* stream);

/* ---- detection from a given flow field, device buffers: derotate -> FoE -> phi/masks -> components ----
 * One iteration of Processor.run_detection (src/processor.py:305-362) per frame, starting from the
 * flow that Dataset.get_flow_uv returns (src/datasets/dataset.py:205-212).  d_total_out / d_fixed_out
 * nullable.  d_records: n mavd_frame_record. */
int mavd_detect(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu,
                const mavd_detect_params* prm, const int32_t* d_samples, const uint8_t* d_sky, int64_t sky_stride,
                const uint8_t* d_seg, int64_t seg_stride, uint8_t* d_total_out, uint8_t* d_fixed_out,
                mavd_frame_record* d_records, void* stream);

/* ---- whole path, device buffers: flow -> derotate -> FoE -> phi/masks -> components ----
 * mavd_farneback followed by mavd_detect.  d_flow_out / d_fixed_out / d_total_out nullable. */
int mavd_process(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride,
                 const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* d_samples,
                 const uint8_t* d_sky, int64_t sky_stride, const uint8_t* d_seg, int64_t seg_stride,
                 float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out,
                 mavd_frame_record* d_records, void* stream);

/* ---- whole path, HOST buffers (the end-to-end call): copies frames/samples/sky/seg in, runs
 * mavd_process, copies the records (and, when non-NULL, estimate_fixed masks and flow) back.
 * Host buffers should be pinned for the copies to be asynchronous; the call returns after the
 * results have landed (it synchronises). */
int mavd_process_host(mavd_handle h, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                      const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                      const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride,
                      float* h_flow_out, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream);

/* The same, split into an asynchronous submit and a wait so that a caller can keep up to
 * MAVD_HOST_SLOTS batches in flight: batch k+1's host->device copies run on a copy stream while batch k
 * computes on `stream` and batch k-1's results return on a third stream.  `slot` in [0, MAVD_HOST_SLOTS)
 * names the staging buffers used; a slot must be waited on before it is submitted again.  All host
 * buffers of a submit must stay valid (and unmodified) until its wait returns. */
int mavd_submit_host(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                     const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                     const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride,
                     float* h_flow_out, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream);
int mavd_wait_host(mavd_handle h, int32_t slot);
/* The same with (H, W, 3) uint8 BGR frames as cv2.VideoCapture.read() / Dataset.get_frame() deliver them
 * (src/farneback.py:73, src/datasets/dataset.py:223-230): the frames are copied as they are and converted to gray on
 * the device on the copy-in stream (mavd_bgr2gray == cv2.cvtColor(COLOR_BGR2GRAY), src/farneback.py:74). */
int mavd_submit_host_bgr(mavd_handle h, int32_t slot, const uint8_t* h_bgr_frames, int32_t n_pairs, int32_t pair_stride,
                         const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                         const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride,
                         float* h_flow_out, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream);

/* Detection from a HOST flow field (n x H x W x 2 float32), the Dataset.get_flow_uv seam end to end. */
int mavd_detect_host(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu,
                     const mavd_detect_params* prm, const int32_t* h_samples, const uint8_t* h_sky,
                     int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride, uint8_t* h_fixed_out,
                     mavd_frame_record* h_records, void* stream);

/* ---- the same calls with every optional per-frame input in one struct (ground-truth flow included) ----
 * mavd_detect / mavd_process / mavd_submit_host / mavd_detect_host forward to these.  One device call per batch also
 * for datasets that carry a ground-truth flow (SimData: src/processor.py:309-310,344,359). */
int mavd_detect_ex(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
                   const int32_t* d_samples, const mavd_aux_inputs* d_aux, uint8_t* d_total_out, uint8_t* d_fixed_out,
                   mavd_frame_record* d_records, void* stream);
int mavd_process_ex(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_imu* h_imu,
                    const mavd_detect_params* prm, const int32_t* d_samples, const mavd_aux_inputs* d_aux,
                    float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                    void* stream);
/* flags: MAVD_HOST_* above.  With MAVD_HOST_SEG_PACKED / MAVD_HOST_SKY_PACKED the segmentation / sky masks cross the
 * bus at 1 bit per pixel and are expanded on the device on the copy-in stream; with MAVD_HOST_FIXED_PACKED the
 * estimate_fixed masks are packed on the copy-out stream and return at 1 bit per pixel (numpy.packbits(mask.ravel(),
 * bitorder='little') per frame, padded to mavd_packed_mask_bytes).  Sample indices are range-checked on the host. */
int mavd_submit_host_ex(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                        const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                        const mavd_aux_inputs* h_aux, int32_t flags, float* h_flow_out, uint8_t* h_fixed_out,
                        mavd_frame_record* h_records, void* stream);
int mavd_detect_host_ex(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu,
                        const mavd_detect_params* prm, const int32_t* h_samples, const mavd_aux_inputs* h_aux,
                        int32_t flags, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream);

/* ---- the _ex calls plus each frame's detection table (mavd_detection) of estimate_fixed ----
 * The _ex calls forward to these with det = NULL.  det: n x max_det entries, a DEVICE pointer for mavd_detect_det /
 * mavd_process_det and a HOST pointer for mavd_submit_host_det / mavd_detect_host_det (valid after the wait, like the
 * records); 1 <= max_det <= MAVD_MAX_DETECTIONS when det is non-NULL.  The table comes from the same labelling as
 * record.boxes (an entry with label <= MAVD_MAX_BOXES has the box and area of boxes[label - 1]); flow_sum sums the
 * derotated flow of the call (the caller's flow, or the Farneback flow of the pair). */
int mavd_detect_det(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
                    const int32_t* d_samples, const mavd_aux_inputs* d_aux, uint8_t* d_total_out, uint8_t* d_fixed_out,
                    mavd_frame_record* d_records, int32_t max_det, mavd_detection* d_det, void* stream);
int mavd_process_det(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_imu* h_imu,
                     const mavd_detect_params* prm, const int32_t* d_samples, const mavd_aux_inputs* d_aux,
                     float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                     int32_t max_det, mavd_detection* d_det, void* stream);
int mavd_submit_host_det(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                         const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                         const mavd_aux_inputs* h_aux, int32_t flags, float* h_flow_out, uint8_t* h_fixed_out,
                         mavd_frame_record* h_records, int32_t max_det, mavd_detection* h_det, void* stream);
int mavd_detect_host_det(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu,
                         const mavd_detect_params* prm, const int32_t* h_samples, const mavd_aux_inputs* h_aux,
                         int32_t flags, uint8_t* h_fixed_out, mavd_frame_record* h_records, int32_t max_det,
                         mavd_detection* h_det, void* stream);

/* ---- sparse features: cv2.goodFeaturesToTrack and cv2.calcOpticalFlowPyrLK (the LucasKanade class's calls) ----
 * mavd_good_features_to_track: Shi-Tomasi corners of n_frames dense (H, W) uint8 frames (n_frames <= 2 * max_pairs).
 * d_corners: n_frames x max_corners x 2 float32 (x, y) in cv2's order; d_count[i] is frame i's corner count WITHOUT a
 * limit, and min(count, max_corners) entries are written (the rest of the row is zero).  d_mask (nullable): (H, W) uint8,
 * mask_stride bytes between frames (0 = one mask for every frame).  d_eig (nullable): n_frames x (H, W) float32
 * cv2.cornerMinEigenVal images, bit for bit.  d_corners may be NULL when max_corners is 0.
 * The first call allocates the corner workspace: about 50 bytes per pixel for 16 frames. */
int mavd_good_features_to_track(mavd_handle h, const uint8_t* d_frames, int32_t n_frames, const mavd_gftt_params* prm,
                                const uint8_t* d_mask, int64_t mask_stride, float* d_corners, int32_t* d_count,
                                float* d_eig, void* stream);
/* mavd_pyr_lk: pair p tracks d_prev_pts[p] (n_points x 2 float32) from frame p*pair_stride to frame p*pair_stride+1
 * (pair_stride 1 or 2, as in mavd_farneback).  d_n_points (nullable): n_pairs int32 counts, points past a pair's count
 * are not tracked (next (0, 0), status 0, err 0); mavd_good_features_to_track's d_count feeds it directly.
 * d_next_pts: n_pairs x n_points x 2 float32, d_status: uint8, d_err: float32 (cv2's err; 0 where cv2 leaves it
 * unset).  Non-finite points get status 0 and err 0.  The first call allocates the pyramid workspace: about 6 bytes per
 * pixel per frame (2 * max_pairs frames). */
int mavd_pyr_lk(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_lk_params* prm,
                const float* d_prev_pts, int32_t n_points, const int32_t* d_n_points, float* d_next_pts,
                uint8_t* d_status, float* d_err, void* stream);

/* ---- 1-bit-per-pixel masks on the wire (ground-truth segmentation in, estimate_fixed out) ----
 * Bytes one packed (H, W) mask occupies: ceil(H*W / 8) rounded up to a multiple of 4.  Bit k of byte j is pixel
 * 8*j + k of the flattened frame (numpy bitorder='little'). */
int64_t mavd_packed_mask_bytes(int32_t width, int32_t height);
/* d_mask (n, H*W) uint8, any non-zero byte -> bit set; d_bits (n, mavd_packed_mask_bytes) */
int mavd_pack_mask(const uint8_t* d_mask, int32_t n, int64_t n_pixels, uint8_t* d_bits, void* stream);
/* the inverse: set bits become `value` (255 for a segmentation image, 1 for a 0/1 mask), clear bits 0 */
int mavd_unpack_mask(const uint8_t* d_bits, int32_t n, int64_t n_pixels, uint8_t value, uint8_t* d_mask, void* stream);

/* ---- optional per-kernel-class device timing (CUDA events on the launching stream) ---- */
enum {
    MAVD_PROF_PYRAMID = 0,       /* pyramid blur+resize passes                       */
    MAVD_PROF_POLYEXP = 1,       /* polynomial expansion                             */
    MAVD_PROF_MATRICES = 2,      /* level-entry UpdateMatrices (+ flow upsample)     */
    MAVD_PROF_ITER_FULL = 3,     /* fused iteration, finest level, not the last one  */
    MAVD_PROF_ITER_FULL_LAST = 4,/* finest level, last iteration (blur + solve only) */
    MAVD_PROF_ITER_COARSE = 5,   /* fused iterations on all coarser levels           */
    MAVD_PROF_FOE = 6,
    MAVD_PROF_RESIDUAL = 7,
    MAVD_PROF_CCL = 8,
    MAVD_PROF_CLASSES = 12
};
typedef struct mavd_profile {
    double ms[MAVD_PROF_CLASSES];        /* summed device time per class since enable */
    int64_t launches[MAVD_PROF_CLASSES]; /* timed launch groups per class             */
} mavd_profile;
int mavd_profile_enable(mavd_handle h, int32_t on); /* also clears the counters */
int mavd_profile_read(mavd_handle h, mavd_profile* out); /* waits for the recorded events */
/* Start / end of every timed launch group recorded since enable, relative to the first one, as (class, start ms,
 * end ms) triples in launch order (does not clear the records).  For timeline views of the two-stream schedule. */
int mavd_profile_timeline(mavd_handle h, double* out, int32_t max_records, int32_t* n_out);

/* Tests: route the Farneback iterations through the generic (non-TMA) kernel, which production uses only
 * for winsize/2 outside 5..8. */
int mavd_debug_force_generic_iteration(mavd_handle h, int32_t on);

/* Tests: evaluate every pixel of the residual stage in float64 even when phi is not requested. */
int mavd_debug_force_exact_residual(mavd_handle h, int32_t on);

/* Number of kernel launches issued by this library since process start (bench.py's gpu_launches). */
int64_t mavd_launch_count(void);

/* Captured launch sequences the handle holds (tuning.use_graph): how many replay as a CUDA graph and how many could
 * not be captured or instantiated and run kernel by kernel instead (expected 0; a diagnostic, results are the same). */
int mavd_graph_stats(mavd_handle h, int32_t* n_captured, int32_t* n_direct);

#ifdef __cplusplus
}
#endif
#endif /* MAVD_H_ */
