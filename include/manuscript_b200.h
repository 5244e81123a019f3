/*
 * manuscript_b200.h -- C ABI of the B200-native (sm_100a) EAST post-processing -> TRBA batch path.
 *
 * Drop-in boundary for the detector->recognizer hot path of olegiy/manuscript-ocr v0.1.8.
 * Each entry point names the reference interface it replaces (paths relative to the reference
 * root).  The reference has no FFI of its own (it is pure Python, SURVEY 8b): these are the
 * functions its numpy-level seam would bind -- see INTEGRATION.md for the ctypes stubs.
 *
 * Conventions
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as void* (NULL = default).
 *   - *_host entry points take HOST buffers, copy in/out themselves and synchronise before return.
 *   - device entry points take DEVICE pointers, are stream-ordered and never synchronise; data-
 *     dependent sizes stay on the device (counts arrays), so a whole page batch runs without a
 *     host round trip.  Per-page outputs are "page-strided": page p owns rows
 *     [p*cap_per_page, p*cap_per_page + counts[p]).
 *   - a context owns ONE scratch arena: use it from one thread and one stream at a time (one context per GPU
 *     worker); calls on the same stream may follow each other without synchronisation.
 *   - return value: MS_OK or a negative MS_ERR_*; ms_last_error() gives a message.  No exceptions
 *     cross the boundary.  There is NO CPU fallback: without a CUDA device every call fails.
 *   - quads are rows of 9 float32: x0,y0,x1,y1,x2,y2,x3,y3,score (the reference's (N,9) layout).
 *   - tie rule: where the reference uses numpy's unstable argsort (lanms.py:138,167; infer.py:199)
 *     ties are broken by original index (numpy kind="stable"), see DESIGN.md.
 */
#ifndef MANUSCRIPT_B200_H
#define MANUSCRIPT_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define MS_API __attribute__((visibility("default")))
#else
#define MS_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MS_OK 0
#define MS_ERR_INVALID (-1)  /* bad argument                                                  */
#define MS_ERR_CUDA (-2)     /* CUDA runtime error (message in ms_last_error)                  */
#define MS_ERR_CAPACITY (-3) /* an output or internal capacity was exceeded                    */
#define MS_ERR_INDEX (-4)    /* quantised pixel outside the map: reference raises IndexError   */
#define MS_ERR_NO_DEVICE (-5)

/* per-page status bits written by the device entry points into `flags` (int32 per page) */
#define MS_FLAG_CAND_OVERFLOW 1 /* more candidates than cap_per_page            */
#define MS_FLAG_INDEX_ERROR 2   /* utils.py:370 would raise IndexError          */
#define MS_FLAG_EDGE_OVERFLOW 4 /* NMS suppression-edge buffer exceeded         */
#define MS_FLAG_ORDER_OVERFLOW 8 /* reading order not computed on the device for this page (more than
                                    max(65536, 16 cap) intersecting box pairs): its boxes and crops are in detection order */

/* element type of the recogniser batch written by the *_ex crop entry points (`batch_dtype`).  The 16-bit batches are
 * an EXTENSION (not a reference behaviour): every value is the float32 batch value ((v - 127.5) * (1/127.5), computed in
 * float32) rounded to nearest-even, bit for bit what torch's batch_f32.to(torch.float16 / torch.bfloat16) gives -- half
 * the bytes written, and no cast for a recogniser that runs in 16 bits.  An unknown code is MS_ERR_INVALID. */
#define MS_DTYPE_F32 0
#define MS_DTYPE_F16 1
#define MS_DTYPE_BF16 2

typedef struct ms_ctx ms_ctx;

/* EAST constructor parameters that shape the path (infer.py:28-43). */
typedef struct ms_east_params {
    float score_thresh;          /* 0.6  */
    double scale;                /* 1/score_geo_scale = 4.0 */
    int quantization;            /* 2    */
    double iou_threshold;        /* 0.2  */
    double expand_ratio_w;       /* 0.9  */
    double expand_ratio_h;       /* 0.9  */
    int target_size;             /* 1280 */
    int axis_aligned_output;     /* 1    */
    int remove_area_anomalies;   /* 1    */
    double anomaly_sigma_threshold; /* 5.0 */
    int anomaly_min_box_count;   /* 30   */
    int sort_reading_order;      /* 0: EAST.predict(sort_reading_order=False) default, infer.py:240;
                                    1: what Pipeline.predict always does, _pipeline.py:105-123 */
} ms_east_params;

MS_API const char *ms_version(void);
MS_API const char *ms_last_error(void);
MS_API void ms_east_params_default(ms_east_params *p);

/* context = device + scratch arena (grown on demand, reused across calls) */
MS_API int ms_create(int device, ms_ctx **out);
MS_API void ms_destroy(ms_ctx *ctx);
MS_API int ms_device_count(void);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
MS_API int64_t ms_launch_count(const ms_ctx *ctx);

/* NMS neighbour-pair capacity per candidate box (default 16).  The *_host entry points grow it (x4, up to 4096) and
 * run again when a page overflows it; callers of the device entry points see MS_FLAG_EDGE_OVERFLOW in `flags` and
 * raise it here before re-running. */
MS_API int ms_set_edge_factor(ms_ctx *ctx, int pairs_per_candidate);
MS_API int ms_get_edge_factor(const ms_ctx *ctx);

/* Per-stage device timing of ms_page_batch (CUDA events recorded on the launch stream between the
 * stages; used by bench.py for the live roofline numbers).  Stages: 0 decode, 1 lanms, 2 expand+filters,
 * 3 word rects, 4 crop/resize/pad.  ms_stage_times waits for the recorded batches, writes the SUM of
 * each stage's milliseconds over the batches recorded since the last read into ms[0..MS_N_STAGES) and
 * returns the number of batches (<= 256 are retained), or a negative error. */
#define MS_N_STAGES 5
MS_API int ms_stage_timing(ms_ctx *ctx, int enable);
MS_API int ms_stage_times(ms_ctx *ctx, double *ms);

/* ---------------------------------------------------------------------------------------------
 * HOST-buffer entry points: one page, the reference's function-level seam.
 * ------------------------------------------------------------------------------------------- */

/* replaces decode_quads_from_maps, detectors/_east/utils.py:328 (called infer.py:319).
 * score (map_h,map_w) f32; geo (8,map_h,map_w) f32 planar (the memory behind infer.py:321's
 * transposed view).  Writes up to `cap` rows, *n_out = N (rows in (y,x) order). */
MS_API int ms_decode_quads_host(ms_ctx *ctx, const float *score, const float *geo, int map_h, int map_w,
                         float score_thresh, double scale, int quantization, float *quads_out,
                         int64_t cap, int64_t *n_out);

/* north_star's RBOX geometry decode -- NOT a reference behaviour (the reference's head is QUAD only: detectors/_east/
 * east.py:99-100, utils.py:368-376; SURVEY 0), "parity unpinned".  Same thresholding, quantisation and row order as
 * ms_decode_quads_host; geo5 (5,map_h,map_w) f32 = distances to the top, right, bottom, left edge of the rotated word
 * rectangle (map units) and its angle (radians); rows are the rectangle's corners TL,TR,BR,BL + score, by the closed
 * form of the public EAST implementations (restore_rectangle_rbox) in float64. */
MS_API int ms_decode_rbox_host(ms_ctx *ctx, const float *score, const float *geo5, int map_h, int map_w,
                        float score_thresh, double scale, int quantization, float *quads_out, int64_t cap,
                        int64_t *n_out);

/* replaces locality_aware_nms, detectors/_east/lanms.py:156 (called infer.py:332).
 * boxes (n,9) f32 -> out (<=n,9) f32 in descending-score order. */
MS_API int ms_lanms_host(ms_ctx *ctx, const float *boxes, int64_t n, double iou_threshold, float *out,
                  int64_t *m_out);

/* replaces standard_nms, detectors/_east/lanms.py:133.  polys (n,4,2) f64, scores (n) f64 ->
 * keep_idx (<=n) int64 indices in kept order. */
MS_API int ms_standard_nms_host(ms_ctx *ctx, const double *polys, const double *scores, int64_t n,
                         double iou_threshold, int64_t *keep_idx, int64_t *k_out);

/* replaces polygon_iou / should_merge, lanms.py:80-96, evaluated on the device for n pairs:
 * subj,clip (n,4,2) f64 -> iou (n) f64. */
MS_API int ms_polygon_iou_host(ms_ctx *ctx, const double *subj, const double *clip, int64_t n, double *iou);

/* TEST-ONLY (not a reference interface): the device predicates that let the NMS skip the float64 clip of lanms.py:80-96
 * for a pair of quads.  out[i] bit 0 = both quads "regular" (convex, positively oriented, well conditioned); bit 1 =
 * regular and IoU(subj, clip) > thr PROVEN by the shrink-and-contain bound (DESIGN 4.1).  tests/ assert that bit 1
 * never contradicts the float64 IoU of the oracle. */
MS_API int ms_test_iou_proved_host(ms_ctx *ctx, const double *subj, const double *clip, int64_t n, double thr,
                            uint8_t *out);

/* TEST-ONLY (not a reference interface): the device functions that size a crop and build its cv2.resize coefficient
 * tables, evaluated on the device.  wh (n_plans,2) int32 (w, h) -> plans_out (n_plans,8) int32: nw, nh, y0, interp
 * (0 copy, 1 INTER_LINEAR, 2 INTER_AREA integer ratio, 3 INTER_AREA general), isx, isy, 1 if the plan alone admits
 * the persistent crop kernel (INTER_AREA general with shrink factors below 2.999, or exactly 2 x 2), 0 -- of the
 * ResizeAndPadA plan at an out_h x out_w canvas.  axes (n_axes,3) int32 (ssize, dsize, mode) -> entries_out, 8 int32
 * words per destination index, the axes one after another (at most entries_cap entries): mode 0 / 1 the INTER_AREA
 * x tables / y records of the persistent kernel (x: word d = s0 | n << 16 and word (1 + k) * dsize + d = weight of
 * tap k, within the axis' 8 * dsize words; y: word 8d = s0 | n << 16, words 8d + 4.. = the tap weights), mode 2 the
 * INTER_AREA entry of the generic kernel {s0, n, nfirst, nmid, first, middle and last weight (f32), 0}, mode 3 / 4
 * the INTER_LINEAR x / y entry {s0, edge flag (x) or second row (y), 11-bit coefficients c0, c1, 0, 0, 0, 0}. */
MS_API int ms_test_resize_tables_host(ms_ctx *ctx, int out_h, int out_w, const int32_t *wh, int64_t n_plans,
                               int32_t *plans_out, const int32_t *axes, int64_t n_axes, int32_t *entries_out,
                               int64_t entries_cap);

/* replaces expand_boxes, detectors/_east/utils.py:384 (called infer.py:340). */
MS_API int ms_expand_boxes_host(ms_ctx *ctx, const float *quads, int64_t n, double expand_w, double expand_h,
                         float *out);

/* replaces EAST._scale_boxes_to_original/_remove_fully_contained_boxes/_remove_area_anomalies/
 * _convert_to_axis_aligned, infer.py:134-233, applied after expand_boxes exactly as
 * infer.py:340-356 does.  quads (n,9) post-NMS -> out (<=n,9). */
MS_API int ms_east_boxes_host(ms_ctx *ctx, const float *quads, int64_t n, const ms_east_params *p, int orig_h,
                       int orig_w, float *out, int64_t *m_out);

/* replaces the crop loop of Pipeline.predict + Pipeline._extract_word_image, _pipeline.py:125-137,
 * 204-221: polys (n,8) f32 -> rects (n,4) int32 [x1,y1,x2,y2) and valid (n) u8. */
MS_API int ms_word_rects_host(ms_ctx *ctx, const float *polys8, int64_t n, int img_h, int img_w,
                       int min_text_size, int32_t *rects, uint8_t *valid);

/* replaces sort_boxes_reading_order_with_resolutions, detectors/_east/utils.py:610-644 (default y_tol_ratio /
 * x_gap_ratio), and the word re-matching of Pipeline.predict, _pipeline.py:105-123 (== infer.py:365-385):
 * polys (n,8) f32 -> order (n) int32, order[r] = index of the word at reading position r (the reference's quirks
 * with duplicate boxes included).  Pages of up to 4096 boxes and 28672 intersecting pairs run in one shared-memory kernel, larger ones in
 * a global-memory kernel; beyond max(65536, 16 n) intersecting pairs (or 2^20 boxes) the call
 * returns MS_ERR_CAPACITY (the Python host side then runs its exact restatement of the reference's host logic). */
MS_API int ms_reading_order_host(ms_ctx *ctx, const float *polys8, int64_t n, int32_t *order);

/* replaces ResizeAndPadA.apply + get_val_transform + the torch.stack of TRBA.predict,
 * recognizers/_trba/data/transforms.py:85-120,185-193 and recognizers/_trba/__init__.py:264-288,
 * 382-390: page (img_h,img_w,3) u8 + rects (n,4) -> batch (n,3,out_h,out_w) f32 normalised
 * (and/or the uint8 canvases (n,out_h,out_w,3); either output may be NULL). */
MS_API int ms_crop_resize_pad_host(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const int32_t *rects,
                            int64_t n, int out_h, int out_w, float *batch_f32, uint8_t *canvas_u8);

/* DIAGNOSTIC (tests, bench): how the quads of this context's LAST ms_quad_crop_resize_pad* call were served --
 * counts[0] quads taken by the staged (TMA window) kernel, counts[1] quads served by the generic kernel (not
 * stageable, or handed back by the staged kernel).  Waits for the call's stream work. */
MS_API int ms_quad_crop_last_counts(ms_ctx *ctx, int32_t *counts);

/* DIAGNOSTIC (tests): how the crops of this context's LAST axis-aligned crop call (ms_crop_resize_pad*, or the crop
 * stage of a page batch) were served -- counts[0] crops listed for the persistent TMA kernel, counts[1] crops listed
 * for the generic kernel (not stageable, another interpolation, invalid, or handed back by the persistent kernel).
 * Waits for the call's stream work. */
MS_API int ms_crop_last_counts(ms_ctx *ctx, int32_t *counts);

/* ms_quad_crop_resize_pad for one page with HOST buffers: quads (n,8) f32, sizes_out (n,2) int32 or NULL. */
MS_API int ms_quad_crop_resize_pad_host(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const float *quads,
                                 int64_t n, int min_text_size, int border_mode, int border_value, int out_h,
                                 int out_w, float *batch_f32, uint8_t *canvas_u8, int32_t *sizes_out);
/* The rectified patch of one quad alone (h x w x 3 u8, row-major) -- the cv2.warpPerspective call above.  *w,*h get
 * the patch size ((0,0): no patch); MS_ERR_CAPACITY (with *w,*h set) when it does not fit patch_cap bytes. */
MS_API int ms_warp_quad_host(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const float *quad, int border_mode,
                      int border_value, uint8_t *patch_out, int64_t patch_cap, int *w, int *h);


/* ---------------------------------------------------------------------------------------------
 * DEVICE entry points: a batch of pages, stream-ordered, no host synchronisation.
 * ------------------------------------------------------------------------------------------- */

/* replaces the input preparation of EAST.predict, detectors/_east/infer.py:301-305: cv2.resize(img, (T, T))
 * [INTER_LINEAR on uint8, aspect not preserved] -> ToTensor (x / 255) -> Normalize(0.5, 0.5).  page (img_h,img_w,3)
 * u8 RGB on the device -> out_f32 (3,target_h,target_w) f32 (the network input) and/or out_u8 (target_h,target_w,3)
 * (the resized image itself; either may be NULL).  With it the page crosses PCIe once: the original is uploaded,
 * the detector input is made on the device, and the crops are cut from the same upload. */
MS_API int ms_detector_input(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, int target_h, int target_w,
                      float *out_f32, uint8_t *out_u8, void *stream);

/* infer.py:301-305 (as ms_detector_input) for n_pages pages of their own sizes in one call: page_ptrs (n_pages) device
 * pointers to (h_i,w_i,3) u8 RGB images and page_hw (n_pages,2) int32 on the device -- the tables ms_page_batch_ragged
 * takes -> out (n_pages,3,target_h,target_w) in out_dtype (MS_DTYPE_*).  Every page is bit for bit what
 * ms_detector_input makes of it.  MS_DTYPE_F16 / MS_DTYPE_BF16 (an EXTENSION) are that float32 value rounded to
 * nearest-even, bit for bit out_f32.to(torch.float16 / torch.bfloat16); nothing is normalised in 16 bits.  Page sizes
 * are device data: a page with h <= 0, w <= 0 or a NULL pointer is not read and its input is written as zeros.  NULL
 * tables or output, n_pages <= 0, a non-positive target or an unknown dtype is MS_ERR_INVALID. */
MS_API int ms_detector_input_batch(ms_ctx *ctx, const uint8_t *const *page_ptrs, const int32_t *page_hw, int n_pages,
                                   int target_h, int target_w, void *out, int out_dtype, void *stream);

/* utils.py:328 for n_pages maps.  score (n_pages,map_h,map_w), geo (n_pages,8,map_h,map_w).
 * quads_out (n_pages*cap_per_page,9); counts (n_pages) int32; flags (n_pages) int32 (OR-ed). */
MS_API int ms_decode_quads(ms_ctx *ctx, const float *score, const float *geo, int n_pages, int map_h, int map_w,
                    float score_thresh, double scale, int quantization, float *quads_out,
                    int cap_per_page, int32_t *counts, int32_t *flags, void *stream);

/* ms_decode_rbox_host for n_pages maps on the device: geo5 (n_pages,5,map_h,map_w). */
MS_API int ms_decode_rbox(ms_ctx *ctx, const float *score, const float *geo5, int n_pages, int map_h, int map_w,
                   float score_thresh, double scale, int quantization, float *quads_out, int cap_per_page,
                   int32_t *counts, int32_t *flags, void *stream);

/* lanms.py:156 for n_pages candidate lists (page-strided in, page-strided out). */
MS_API int ms_lanms(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
             double iou_threshold, float *quads_out, int32_t *counts_out, int32_t *flags, void *stream);

/* utils.py:384 + infer.py:134-233 for n_pages NMS outputs.  orig_hw (n_pages,2) int32 on the
 * device, or NULL for (target_size,target_size). */
MS_API int ms_east_boxes(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                  const ms_east_params *p, const int32_t *orig_hw, float *quads_out, int32_t *counts_out,
                  void *stream);

/* utils.py:610-644 + _pipeline.py:105-123 for n_pages box lists (page-strided): order (n_pages*cap_per_page) int32 and,
 * if quads_out != NULL (must not alias quads), the rows in reading order.  A page beyond the device capacity (more than
 * max(65536, 16 cap_per_page) intersecting pairs) keeps its detection order and gets MS_FLAG_ORDER_OVERFLOW in `flags`. */
MS_API int ms_reading_order(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                     int32_t *order, float *quads_out, int32_t *flags, void *stream);

/* _pipeline.py:125-137,204-221 for n_pages box lists: compacts the valid crops of all pages, in
 * (page, box) order, into crops_out rows of 5 int32 [page,x1,y1,x2,y2]; *n_crops (device int32). */
MS_API int ms_word_rects(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                  const int32_t *img_hw, int img_h, int img_w, int min_text_size, int32_t *crops_out,
                  int64_t crops_cap, int32_t *n_crops, void *stream);

/* transforms.py:85-120,185-193 for a crop list over a batch of equally sized pages
 * pages (n_pages,img_h,img_w,3) u8.  crops (<=crops_cap,5) int32 and n_crops on the device.
 * batch_f32 (crops_cap,3,out_h,out_w) and/or canvas_u8 (crops_cap,out_h,out_w,3). */
MS_API int ms_crop_resize_pad(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                       const int32_t *crops, const int32_t *n_crops, int64_t crops_cap, int out_h,
                       int out_w, float *batch_f32, uint8_t *canvas_u8, void *stream);
/* ms_crop_resize_pad with the batch (crops_cap,3,out_h,out_w) in batch_dtype (MS_DTYPE_*); batch may be NULL. */
MS_API int ms_crop_resize_pad_ex(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                          const int32_t *crops, const int32_t *n_crops, int64_t crops_cap, int out_h, int out_w,
                          void *batch, int batch_dtype, uint8_t *canvas_u8, void *stream);

/* SURVEY 8f-4, an EXTENSION (the reference crops axis-aligned rectangles only, _pipeline.py:204-221; todo.md:1):
 * rectified crops of rotated quads.  For every quad (rows of quad_stride >= 8 floats x0,y0..x3,y3 in the order
 * top-left, top-right, bottom-right, bottom-left):
 *   w,h   = round-half-even of the longer of each pair of opposite edges; no patch when a side is < max(2,
 *           min_text_size) or > 32767, a coordinate is not finite or the 4-point system is singular
 *   patch = cv2.warpPerspective(page, cv2.getPerspectiveTransform(rect(w,h), quad), (w,h),
 *                               INTER_LINEAR | WARP_INVERSE_MAP, border)        (bit-exact, see quadcrop.cu)
 * then the ResizeAndPadA + normalise of ms_crop_resize_pad.  Output row i belongs to quad i; a quad without a patch
 * gives an all-padding canvas and sizes_out (w,h) = (0,0).  border_mode 0 = BORDER_CONSTANT with border_value on all
 * channels, 1 = BORDER_REPLICATE.  Pages at most 32767 pixels on a side.  page_of (n) int32 or NULL (all page 0). */
MS_API int ms_quad_crop_resize_pad(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                            const float *quads, int quad_stride, const int32_t *page_of, int64_t n,
                            int min_text_size, int border_mode, int border_value, int out_h, int out_w,
                            float *batch_f32, uint8_t *canvas_u8, int32_t *sizes_out, void *stream);
/* ms_quad_crop_resize_pad with the batch (n,3,out_h,out_w) in batch_dtype (MS_DTYPE_*); batch may be NULL. */
MS_API int ms_quad_crop_resize_pad_ex(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                               const float *quads, int quad_stride, const int32_t *page_of, int64_t n,
                               int min_text_size, int border_mode, int border_value, int out_h, int out_w,
                               void *batch, int batch_dtype, uint8_t *canvas_u8, int32_t *sizes_out, void *stream);

/* north_star's "TPS rectification grid_sample" -- NOT a reference behaviour (the reference's TRBAModel has no
 * transformation stage, recognizers/_trba/model/model.py:338-393; SURVEY 0), "parity unpinned"; specified as the
 * TPS-STN of the TRBA literature and checked against torch.nn.functional.grid_sample.  All pointers on the device:
 * input (batch,chans,in_h,in_w) f32, c_prime (batch,n_fid,2) f32 predicted fiducial points in [-1,1],
 * inv_delta_c (n_fid+3,n_fid+3) f32 and p_hat_t (n_fid+3, out_h*out_w) f32 (the TRANSPOSED P_hat) as
 * manuscript_b200.tps.TPSGrid computes them; out (batch,chans,out_h,out_w) f32 =
 * grid_sample(input, P_hat @ inv_delta_c @ [c_prime; 0], bilinear, padding_mode="border", align_corners=True). */
MS_API int ms_tps_rectify(ms_ctx *ctx, const float *input, const float *c_prime, const float *inv_delta_c,
                   const float *p_hat_t, int batch, int n_fid, int chans, int in_h, int in_w, int out_h, int out_w,
                   float *out, void *stream);

/* decode -> LANMS -> expand/filters -> word rects -> crop batch in one call (device buffers).
 * boxes_out (n_pages*cap_boxes,9), box_counts (n_pages); crops_out/n_crops/batch as above. */
MS_API int ms_page_batch(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages, int n_pages,
                  int map_h, int map_w, int img_h, int img_w, const ms_east_params *p, int min_text_size,
                  int out_h, int out_w, int cap_boxes, float *boxes_out, int32_t *box_counts,
                  int32_t *crops_out, int64_t crops_cap, int32_t *n_crops, float *batch_f32,
                  uint8_t *canvas_u8, int32_t *flags, void *stream);
/* ms_page_batch with the crop batch in batch_dtype (MS_DTYPE_*).  The dtype is part of the call's identity for the
 * CUDA-graph cache: the same buffers with another dtype are a different call. */
MS_API int ms_page_batch_ex(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages, int n_pages,
                     int map_h, int map_w, int img_h, int img_w, const ms_east_params *p, int min_text_size,
                     int out_h, int out_w, int cap_boxes, float *boxes_out, int32_t *box_counts,
                     int32_t *crops_out, int64_t crops_cap, int32_t *n_crops, void *batch, int batch_dtype,
                     uint8_t *canvas_u8, int32_t *flags, void *stream);

/* ms_page_batch for page images of their OWN sizes (a batch of originals: EAST.predict resizes each to target_size,
 * so the maps are uniform while the images are not).  page_ptrs (n_pages) device pointers to (h_i, w_i, 3) u8
 * images, page_hw (n_pages,2) int32 on the device.  Boxes are scaled to each page's size (infer.py:134-147) and the
 * crops cut from its pixels.  Images whose base address is 16-byte aligned use the TMA path. */
MS_API int ms_page_batch_ragged(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *const *page_ptrs,
                         const int32_t *page_hw, int n_pages, int map_h, int map_w, const ms_east_params *p,
                         int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                         int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                         float *batch_f32, uint8_t *canvas_u8, int32_t *flags, void *stream);
/* ms_page_batch_ragged with the crop batch in batch_dtype (MS_DTYPE_*). */
MS_API int ms_page_batch_ragged_ex(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *const *page_ptrs,
                            const int32_t *page_hw, int n_pages, int map_h, int map_w, const ms_east_params *p,
                            int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                            int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                            void *batch, int batch_dtype, uint8_t *canvas_u8, int32_t *flags, void *stream);

/* Same path with HOST buffers (pinned or pageable; `score` / `geo` may also be DEVICE pointers of this context's
 * device -- maps a detector left on the GPU are used in place and only the page images cross PCIe): H2D of maps + pages, the batch, D2H of boxes,
 * counts, crop list and (optionally, if batch_f32_host != NULL) the crop batch.  Of boxes_out (n_pages*cap_boxes,9)
 * only rows [0, box_counts[p]) of each page p are defined.  When
 * batch_dev_out != NULL the crop batch stays on the device (as the reference leaves it on `self.device`,
 * recognizers/_trba/__init__.py:288):
 *   *batch_dev_out != NULL on entry  -> a CALLER-OWNED device buffer of crops_cap crops; the batch is written there;
 *   *batch_dev_out == NULL on entry  -> the batch is written to library-owned staging memory and its address is
 *                                       returned; it is valid only until the NEXT call on this context (which may
 *                                       overwrite or free it).  Prefer the caller-owned form. */
MS_API int ms_page_batch_host(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages,
                       int n_pages, int map_h, int map_w, int img_h, int img_w, const ms_east_params *p,
                       int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                       int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                       float *batch_f32_host, float **batch_dev_out, int32_t *flags);
/* ms_page_batch_host with the crop batch in batch_dtype (MS_DTYPE_*): the host copy (batch_host), a caller-owned
 * device buffer (*batch_dev_out) and the library-owned device batch are all of that element type. */
MS_API int ms_page_batch_host_ex(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages,
                          int n_pages, int map_h, int map_w, int img_h, int img_w, const ms_east_params *p,
                          int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                          int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                          void *batch_host, int batch_dtype, void **batch_dev_out, int32_t *flags);

/* ms_page_batch_ragged with HOST buffers: pages (n_pages) host pointers, page_hw (n_pages,2) int32 on the host;
 * outputs as ms_page_batch_host (of boxes_out, only rows [0, box_counts[p]) of each page p are defined). */
MS_API int ms_page_batch_ragged_host(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *const *pages,
                              const int32_t *page_hw, int n_pages, int map_h, int map_w, const ms_east_params *p,
                              int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                              int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                              float *batch_f32_host, float **batch_dev_out, int32_t *flags);
/* ms_page_batch_ragged_host with the crop batch in batch_dtype (MS_DTYPE_*), as ms_page_batch_host_ex. */
MS_API int ms_page_batch_ragged_host_ex(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *const *pages,
                                 const int32_t *page_hw, int n_pages, int map_h, int map_w, const ms_east_params *p,
                                 int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                                 int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                                 void *batch_host, int batch_dtype, void **batch_dev_out, int32_t *flags);

#ifdef __cplusplus
}
#endif
#endif /* MANUSCRIPT_B200_H */
