// Internal declarations shared by the sm_100a kernels and the C-ABI layer.
// Everything here is compiled with --fmad=false: the reference's numpy / numba arithmetic never
// fuses a*b+c, and keep/suppress decisions must be bit-identical (SURVEY 7, "hard parts").
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/manuscript_b200.h"

#define MS_NUM_SMS_B200 148

// Everything that defines one page-batch call (api.cu).  Per-page arrays point at the call's page 0 and are
// page-strided: the maps (n_pages, map_h, map_w) and (n_pages, 8, map_h / q or map_h, map_w) at their element strides
// and element type, boxes_out (n_pages,
// cap_boxes, 9), box_counts / flags (n_pages), page_hw (n_pages, 2).  pages (n_pages, img_h, img_w, 3) u8 or, for
// images of their own sizes, page_ptrs + page_hw.  The host entry points describe the caller's host buffers in one
// pb_call and the device staging in a copy of it.
struct pb_call {
    ms_maps maps;  // copied field by field (pb_set_maps): no padding bytes of the caller's struct
    const uint8_t *pages;
    const uint8_t *const *page_ptrs;
    const int32_t *page_hw;
    int n_pages, map_h, map_w, img_h, img_w, min_text_size, out_h, out_w, cap_boxes;
    int64_t crops_cap;
    ms_east_params params;
    float *boxes_out;
    int32_t *box_counts, *crops_out, *n_crops;
    void *batch;
    int batch_dtype;
    uint8_t *canvas_u8;
    int32_t *flags;
    int geo_compact;  // geo holds only the rows the decode reads, y % q == q / 2 (q = params.quantization)
    // the crop stage: 0 = axis-aligned rectangles [page, x1, y1, x2, y2); 1 = rectified quads [page, box, w, h, 0]
    // with the border of the perspective warp (0 = constant border_value, 1 = replicate)
    int crop_quads, border_mode, border_value;
};
// A recorded ms_page_batch call and what its launches point into or were sized by; compared bytewise.
struct ms_pb_key {
    pb_call call;
    const char *arena;
    size_t arena_bytes;
    int edge_factor;
};
// ... and, from its second occurrence on, the CUDA graph of its launches.
struct ms_graph_entry {
    ms_pb_key key;
    int used, failed;
    cudaGraphExec_t exec;
    int64_t launches;  // kernels per replay (for ms_launch_count)
};
#define MS_GRAPH_SLOTS 4

// The kernels launched with more dynamic shared memory than the default 48 KB allows (ms_allow_smem); the crop kernels
// once per output instantiation, in groups of seven (batch_slot, crop_common.cuh): u8 canvas only, then each batch
// element type (f32, f16, bf16) without and with the u8 canvas.
enum ms_smem_slot {
    MS_SMEM_CROP_U8,
    MS_SMEM_CROP_F32,
    MS_SMEM_CROP_F32_U8,
    MS_SMEM_CROP_F16,
    MS_SMEM_CROP_F16_U8,
    MS_SMEM_CROP_BF16,
    MS_SMEM_CROP_BF16_U8,
    MS_SMEM_QUAD_U8,
    MS_SMEM_QUAD_F32,
    MS_SMEM_QUAD_F32_U8,
    MS_SMEM_QUAD_F16,
    MS_SMEM_QUAD_F16_U8,
    MS_SMEM_QUAD_BF16,
    MS_SMEM_QUAD_BF16_U8,
    MS_SMEM_QUAD_STAGED_U8,
    MS_SMEM_QUAD_STAGED_F32,
    MS_SMEM_QUAD_STAGED_F32_U8,
    MS_SMEM_QUAD_STAGED_F16,
    MS_SMEM_QUAD_STAGED_F16_U8,
    MS_SMEM_QUAD_STAGED_BF16,
    MS_SMEM_QUAD_STAGED_BF16_U8,
    MS_SMEM_READING_ORDER,
    MS_SMEM_READING_ORDER_LARGE,
    MS_SMEM_SLOTS
};

struct ms_ctx {
    int device;
    int num_sms;
    char *arena;          // device scratch
    size_t arena_bytes;
    char *pinned;         // small pinned host staging (counts / flags read-back)
    size_t pinned_bytes;
    cudaStream_t own_stream;
    int64_t launches;
    // host-API device staging, grown on demand
    char *stage;
    size_t stage_bytes;
    // ms_stage_timing: ring of per-batch event sets
    int edge_factor;              // NMS neighbour-pair capacity per candidate (grown by the host entry points)
    int smem_granted[MS_SMEM_SLOTS];  // largest dynamic shared-memory size already granted to each kernel
    cudaStream_t copy_stream;     // H2D stream of the pipelined host entry point
    cudaEvent_t chunk_ev[2];
    cudaStream_t aux_stream;      // second half of a batch's front stages (page_batch_impl)
    cudaEvent_t split_ev[2];      // fork / join of that half
    int split_front;              // 0 with MS_B200_NO_SPLIT=1
    int timing;
    int timing_n;                 // batches recorded since the last read (<= MS_TIMING_RING)
    cudaEvent_t *timing_ev;       // MS_TIMING_RING * (MS_N_STAGES + 1) events, created lazily
    // A batch is ~50 short launches: a repeated ms_page_batch call (same buffers, sizes and parameters -- a serving
    // loop) is captured into a CUDA graph at its second occurrence and replayed afterwards.
    int graphs_enabled;           // 0 with MS_B200_NO_GRAPHS=1 in the environment
    int graph_clock;
    ms_graph_entry graphs[MS_GRAPH_SLOTS];
    const int32_t *quad_cnt;      // device counters of the last rotated-crop call (ms_quad_crop_last_counts)
    cudaStream_t quad_stream;
    const int32_t *crop_cnt;      // device counters of the last axis-crop call (ms_crop_last_counts)
    cudaStream_t crop_stream;
    int quad_no_stage;            // MS_B200_QUAD_NO_STAGE=1: rotated crops by the generic kernel only (A/B runs, tests)
    int ro_force_large;           // MS_B200_RO_FORCE_LARGE=1: every page takes the large-page reading-order kernel (tests)
    char *jpeg_pinned;            // pinned staging of ms_jpeg_decode_batch (descriptors + entropy-coded bytes), grown
    size_t jpeg_pinned_bytes;     // on demand; jpeg_ev marks the end of the last copy out of it
    cudaEvent_t jpeg_ev;
    int jpeg_pending;
    int busy;                     // 1 while a thread is inside an entry point (atomic test-and-set): a context owns ONE
                                  // scratch arena, so a second thread entering gets MS_ERR_INVALID instead of corrupting it
};
#define MS_TIMING_RING 256

struct ms_bump {
    char *base;
    size_t off, cap;
    template <typename T>
    T *take(size_t n)
    {
        size_t a = (off + 255) & ~size_t(255);
        size_t end = a + n * sizeof(T);
        if (end > cap) {
            off = end;  // remember the demand so a sizing pass can read it back
            return nullptr;
        }
        off = end;
        return reinterpret_cast<T *>(base + a);
    }
};

void ms_set_error(const char *fmt, ...);
// bytes of one batch element of an MS_DTYPE_* code; 0 for an unknown code
inline size_t ms_dtype_bytes(int dtype)
{
    return dtype == MS_DTYPE_F32 ? 4 : (dtype == MS_DTYPE_F16 || dtype == MS_DTYPE_BF16) ? 2 : 0;
}
int ms_check_cuda(cudaError_t e, const char *what);
// bump allocator over ctx->arena; ms_arena_reserve grows it (synchronises the device when it does)
int ms_arena_reserve(ms_ctx *ctx, size_t bytes);
int ms_stage_reserve(ms_ctx *ctx, size_t bytes);


#define MS_CUDA(call)                                                  \
    do {                                                               \
        int _rc = ms_check_cuda((call), #call);                        \
        if (_rc != MS_OK) return _rc;                                  \
    } while (0)

#define MS_TRY(expr)                 \
    do {                             \
        int _r = (expr);             \
        if (_r != MS_OK) return _r;  \
    } while (0)

// Lets `kernel` (slot `slot`) be launched with `bytes` of dynamic shared memory.  cudaFuncSetAttribute is a synchronous
// driver call (milliseconds): it is made once per context and kernel, and again only for a larger size.
template <typename Kernel>
inline int ms_allow_smem(ms_ctx *ctx, ms_smem_slot slot, Kernel kernel, int bytes)
{
    if (bytes > ctx->smem_granted[slot]) {
        MS_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        ctx->smem_granted[slot] = bytes;
    }
    return MS_OK;
}

// ---- programmatic dependent launch --------------------------------------------------------------------------------
// The front stages are ~50 short kernels, each depending on the one before it: the gap between two of them (the next
// kernel's CTAs are only scheduled after the previous grid has completed and flushed) is a few microseconds per edge,
// direct or as a graph.  Kernels launched through ms_launch carry cudaLaunchAttributeProgrammaticStreamSerialization, so
// their CTAs are scheduled while the previous kernel's last CTAs drain; EVERY such kernel executes ms_pdl_wait()
// (griddepcontrol.wait: returns when the preceding grid has completed and its writes are visible) before it touches
// memory, which makes the chain transitive and the results those of plain stream order.  MS_B200_NO_PDL=1: plain launches.
#if defined(__CUDACC__)
__device__ __forceinline__ void ms_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

inline bool ms_pdl_enabled()
{
    static const bool on = getenv("MS_B200_NO_PDL") == nullptr;
    return on;
}

template <typename... KArgs, typename... Args>
inline void ms_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = ms_pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);  // errors surface through MS_LAUNCH_CHECK (cudaGetLastError)
}
#endif

#define MS_LAUNCH_CHECK(ctx)                                           \
    do {                                                               \
        (ctx)->launches++;                                             \
        int _rc = ms_check_cuda(cudaGetLastError(), "kernel launch");  \
        if (_rc != MS_OK) return _rc;                                  \
    } while (0)

// ---- stage launchers (device pointers, stream-ordered) -------------------------------------------
// Every launcher takes its scratch as an ms_bump BY VALUE (stage-local; stages of one stream may
// reuse the same bytes) sized by the matching msk_*_scratch().
// decode.cu
// Maps at their strides (geo_compact: the geometry strides are those of the compact (P, 8, H / q, W) tensor).
int msk_decode(ms_ctx *ctx, const ms_maps &m, int n_pages, int H, int W, float thr, double scale, int q,
               float *quads_out, int cap_per_page, int32_t *counts, int32_t *flags, ms_bump bump, cudaStream_t st,
               int geo_compact = 0, int rbox = 0);  // rbox: geo is (P,5,H,W) float32
// dense float32 maps: score (P, H, W), geo (P, chans, geo_rows, W)
inline ms_maps ms_dense_maps(const float *score, const float *geo, int H, int W, int geo_rows, int chans)
{
    ms_maps m;
    memset(&m, 0, sizeof(m));
    m.score = score;
    m.geo = geo;
    m.dtype = MS_DTYPE_F32;
    m.score_strides[0] = (int64_t)H * W;
    m.score_strides[1] = W;
    m.score_strides[2] = 1;
    m.geo_strides[0] = (int64_t)chans * geo_rows * W;
    m.geo_strides[1] = (int64_t)geo_rows * W;
    m.geo_strides[2] = W;
    m.geo_strides[3] = 1;
    return m;
}
size_t msk_decode_scratch(int n_pages, int H, int W, int q);
// sort.cu : stable LSD radix sort, per-page segments [page_off[p], page_off[p+1]) of (u32 key, u32 value), 4 passes
int msk_sort_pages(ms_ctx *ctx, uint32_t *keys, uint32_t *vals, uint32_t *keys_tmp, uint32_t *vals_tmp,
                   const int32_t *page_off, const int32_t *seg_len, int skip_le, int n_pages, int cap_per_page,
                   ms_bump bump, cudaStream_t st);
size_t msk_sort_pages_scratch(int n_pages, int cap_per_page);
// lanms.cu
int msk_lanms(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
              double thr, float *quads_out, int32_t *counts_out, int32_t *flags, ms_bump bump, cudaStream_t st);
size_t msk_lanms_scratch(int n_pages, int cap_per_page, int ef);
int msk_standard_nms(ms_ctx *ctx, const double *polys, const double *scores, int n, double thr,
                     int32_t *keep_idx, int32_t *k_out, int32_t *flags, ms_bump bump, cudaStream_t st);
size_t msk_standard_nms_scratch(int n, int ef);
int msk_polygon_iou(ms_ctx *ctx, const double *subj, const double *clip, int64_t n, double *iou, cudaStream_t st);
int msk_iou_proved(ms_ctx *ctx, const double *subj, const double *clip, int64_t n, double thr, uint8_t *out,
                   cudaStream_t st);
// boxes.cu
int msk_expand(ms_ctx *ctx, const float *quads, int64_t n, double ew, double eh, float *out, cudaStream_t st);
int msk_east_boxes(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                   const ms_east_params *p, const int32_t *orig_hw, float *quads_out, int out_cap,
                   int32_t *counts_out, int32_t *flags, ms_bump bump, cudaStream_t st, int orig_h = 0,
                   int orig_w = 0);  // orig_hw == NULL: every page is (orig_h, orig_w), or target_size when <= 0
size_t msk_east_boxes_scratch(int n_pages, int cap_per_page);
// np_sum_test.cu, test-only (ms_test_np_sum_host): the numpy pairwise sums of east_finish_kernel, one CTA per vector
int msk_test_np_sum(ms_ctx *ctx, const float *values, const int64_t *offsets, const int32_t *lengths, int n_vec,
                    float *out_serial, float *out_cta, cudaStream_t st);
int msk_word_rects(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                   const int32_t *img_hw, int img_h, int img_w, int min_text_size, int32_t *crops_out,
                   int64_t crops_cap, int32_t *n_crops, int page_base, int append, int32_t *range, ms_bump bump,
                   cudaStream_t st);
size_t msk_word_rects_scratch(int n_pages);
int msk_word_rects_flat(ms_ctx *ctx, const float *polys8, int64_t n, int img_h, int img_w, int min_text_size,
                        int32_t *rects, uint8_t *valid, cudaStream_t st);
// reading_order.cu
int msk_reading_order(ms_ctx *ctx, const float *boxes8, int row_stride, const int32_t *counts, int n_pages,
                      int cap_per_page, int32_t *order, float *reordered, int32_t *flags, ms_bump bump, cudaStream_t st);
size_t msk_reading_order_scratch(int n_pages, int cap_per_page);
// crop.cu
// batch: (crops_cap, 3, out_h, out_w) of batch_dtype (MS_DTYPE_*), or NULL
int msk_crop(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w, const int32_t *crops,
             const int32_t *n_crops, const int32_t *range, int64_t crops_cap, int out_h, int out_w, void *batch,
             int batch_dtype, uint8_t *canvas_u8, ms_bump bump, cudaStream_t st, const uint8_t *const *page_ptrs = nullptr,
             const int32_t *page_hw = nullptr);  // page_ptrs / page_hw (device): pages of their own sizes
// test-only (ms_test_resize_tables_host): the resize plan and coefficient-table device functions on device buffers
int msk_test_resize_tables(ms_ctx *ctx, int out_h, int out_w, const int32_t *wh, int64_t n_plans, int32_t *plans_out,
                           const int32_t *axes, int64_t n_axes, int32_t *entries_out, cudaStream_t st);
// tps.cu
int msk_tps_rectify(ms_ctx *ctx, const float *input, const float *c_prime, const float *inv_delta_c, const float *p_hat_t,
                    int batch, int n_fid, int chans, int in_h, int in_w, int out_h, int out_w, float *out, cudaStream_t st);
// detector input of n_pages pages: page_ptrs / page_hw (device tables) or, when they are NULL, the one page `one`
// (one_h, one_w).  out (n_pages, 3, target_h, target_w) of out_dtype and / or out_u8 (n_pages, target_h, target_w, 3)
int msk_detector_input(ms_ctx *ctx, const uint8_t *const *page_ptrs, const int32_t *page_hw, const uint8_t *one,
                       int one_h, int one_w, int n_pages, int target_h, int target_w, void *out, int out_dtype,
                       uint8_t *out_u8, ms_bump bump, cudaStream_t st);
size_t msk_detector_input_scratch(int n_pages, int target_h, int target_w);
size_t msk_crop_scratch(int64_t crops_cap, int n_pages);
// quadcrop.cu
int msk_quad_crop(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w, const float *quads,
                  int quad_stride, const int32_t *page_of, int64_t n, int min_text_size, int border_mode,
                  int border_value, int out_h, int out_w, void *batch, int batch_dtype, uint8_t *canvas_u8,
                  int32_t *sizes_out, ms_bump bump, cudaStream_t st);
size_t msk_quad_crop_scratch(int64_t n);
// the crop stage of a quad page batch over the final boxes (n_pages, cap_boxes, 9) / counts; pages (n_pages, img_h,
// img_w, 3) or page_ptrs / page_hw.  msk_quad_list: crops_out rows [page, box, w, h, 0] of the boxes that have a
// patch, in (page, box) order, and *n_crops = min(listed, crops_cap), all on the device.  msk_quad_crop_rows: the crop
// of every listed row (batch row i = list row i; rows past *n_crops are not written).
int msk_quad_list(ms_ctx *ctx, const float *boxes, const int32_t *counts, int n_pages, int cap_boxes,
                  const uint8_t *pages, int img_h, int img_w, const uint8_t *const *page_ptrs, const int32_t *page_hw,
                  int min_text_size, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops, ms_bump bump,
                  cudaStream_t st);
size_t msk_quad_list_scratch(int n_pages, int cap_boxes);
int msk_quad_crop_rows(ms_ctx *ctx, const float *boxes, int cap_boxes, int n_pages, const uint8_t *pages, int img_h,
                       int img_w, const uint8_t *const *page_ptrs, const int32_t *page_hw, const int32_t *crops,
                       const int32_t *n_crops, int64_t crops_cap, int min_text_size, int border_mode, int border_value,
                       int out_h, int out_w, void *batch, int batch_dtype, uint8_t *canvas_u8, ms_bump bump,
                       cudaStream_t st);
int msk_quad_warp(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const float *quad_dev, int border_mode,
                  int border_value, uint8_t *patch_dev, size_t patch_cap, int *w, int *h, ms_bump bump, cudaStream_t st);

// jpeg.cu: ms_jpeg_decode_batch without the entry guard
int ms_jpeg_decode_batch_impl(ms_ctx *ctx, const uint8_t *const *files, const int64_t *sizes, int n,
                              uint8_t *const *out_pages, int32_t *out_status, cudaStream_t st);

// ---- device geometry: lanms.py:7-130 in float64, no fused multiply-add ------------------------------
#define MS_MAXV 20  // lanms.py:34

struct quad64 {
    double v[8];
};

__device__ __forceinline__ double ms_shoelace(const double *p, int n)
{
    // lanms.py:7-14: sequential accumulation from 0.0, |.|/2
    double acc = 0.0;
    for (int i = 0; i < n; i++) {
        int j = (i + 1 == n) ? 0 : i + 1;
        acc = acc + (p[2 * i] * p[2 * j + 1] - p[2 * j] * p[2 * i + 1]);
    }
    return fabs(acc) / 2.0;
}

__device__ __forceinline__ bool ms_left_of(double ax, double ay, double bx, double by, double px, double py)
{
    // lanms.py:40-45
    return (bx - ax) * (py - ay) - (by - ay) * (px - ax) >= 0;
}

__device__ __forceinline__ void ms_line_hit(double p1x, double p1y, double p2x, double p2y, double ax,
                                            double ay, double bx, double by, double &ox, double &oy)
{
    // lanms.py:17-29
    double ex = p2x - p1x, ey = p2y - p1y;
    double lx = bx - ax, ly = by - ay;
    double den = ex * ly - ey * lx;
    double cx = ax - p1x, cy = ay - p1y;
    if (den == 0) {
        ox = p1x;
        oy = p1y;
        return;
    }
    double t = (cx * ly - cy * lx) / den;
    ox = p1x + t * ex;
    oy = p1y + t * ey;
}

// lanms.py:80-91 polygon_iou(subject, clip) for two quads.  `buf` is 4*MS_MAXV doubles of scratch
// private to the calling thread (local or shared memory).
static __device__ __noinline__ double ms_quad_iou(const double *s, const double *c, double *buf)
{
    double *cur = buf, *nxt = buf + 2 * MS_MAXV;
    int n = 4;
#pragma unroll
    for (int k = 0; k < 8; k++) cur[k] = s[k];
    for (int e = 0; e < 4; e++) {
        double ax = c[2 * e], ay = c[2 * e + 1];
        int e1 = (e + 1) & 3;
        double bx = c[2 * e1], by = c[2 * e1 + 1];
        int cnt = 0;
        double px = cur[2 * (n - 1)], py = cur[2 * (n - 1) + 1];
        bool pin = ms_left_of(ax, ay, bx, by, px, py);
        for (int i = 0; i < n; i++) {
            double qx = cur[2 * i], qy = cur[2 * i + 1];
            bool cin = ms_left_of(ax, ay, bx, by, qx, qy);
            if (cin) {
                if (!pin) {
                    ms_line_hit(px, py, qx, qy, ax, ay, bx, by, nxt[2 * cnt], nxt[2 * cnt + 1]);
                    cnt++;
                }
                nxt[2 * cnt] = qx;
                nxt[2 * cnt + 1] = qy;
                cnt++;
            } else if (pin) {
                ms_line_hit(px, py, qx, qy, ax, ay, bx, by, nxt[2 * cnt], nxt[2 * cnt + 1]);
                cnt++;
            }
            px = qx;
            py = qy;
            pin = cin;
        }
        double *t = cur;
        cur = nxt;
        nxt = t;
        n = cnt;
        if (n == 0) break;
    }
    double ia = 0.0;
    if (n > 2) ia = ms_shoelace(cur, n);
    double a1 = ms_shoelace(s, 4);
    double a2 = ms_shoelace(c, 4);
    double uni = a1 + a2 - ia;
    if (uni <= 0) return 0.0;
    return ia / uni;
}

// lanms.py:99-130 normalize_polygon(ref, poly) -> out
__device__ __forceinline__ void ms_align_vertices(const double *ref, const double *poly, double *out)
{
    int best_dir = 0, best_start = 0;
    double best = 1e20;
    for (int s = 0; s < 4; s++) {
        double d = 0.0;
        for (int i = 0; i < 4; i++) {
            int k = (s + i) & 3;
            double dx = ref[2 * i] - poly[2 * k];
            double dy = ref[2 * i + 1] - poly[2 * k + 1];
            d = d + (dx * dx + dy * dy);
        }
        if (d < best) {
            best = d;
            best_start = s;
            best_dir = 0;
        }
    }
    for (int s = 0; s < 4; s++) {
        double d = 0.0;
        for (int i = 0; i < 4; i++) {
            int k = (s - i) & 3;
            double dx = ref[2 * i] - poly[2 * k];
            double dy = ref[2 * i + 1] - poly[2 * k + 1];
            d = d + (dx * dx + dy * dy);
        }
        if (d < best) {
            best = d;
            best_start = s;
            best_dir = 1;
        }
    }
    for (int i = 0; i < 4; i++) {
        int k = best_dir == 0 ? (best_start + i) & 3 : (best_start - i) & 3;
        out[2 * i] = poly[2 * k];
        out[2 * i + 1] = poly[2 * k + 1];
    }
}

// monotone u32 image of a float for radix sorting; numpy sort order (NaN last, -0 == +0)
__device__ __forceinline__ uint32_t ms_orderable_f32(float f)
{
    if (f != f) return 0xFFFFFFFFu;
    if (f == 0.0f) f = 0.0f;  // fold -0 onto +0
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
