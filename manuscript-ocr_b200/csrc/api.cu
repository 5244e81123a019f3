// C-ABI layer of libmanuscript_b200.so: context, scratch arenas, the host-buffer entry points (one
// page, the reference's function-level seam) and the device-buffer entry points (page batches,
// stream-ordered).  Declarations and the reference interface each entry replaces: include/manuscript_b200.h.
//
// There is no CPU path in this library: every entry point launches the sm_100a kernels of
// decode.cu / sort.cu / lanms.cu / boxes.cu / crop.cu or fails.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "ms_internal.cuh"

// ---- errors ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void ms_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int ms_check_cuda(cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return MS_OK;
    ms_set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
    return MS_ERR_CUDA;
}

extern "C" const char *ms_last_error(void) { return g_err; }
extern "C" const char *ms_version(void) { return "manuscript_b200 0.1 (sm_100a)"; }

extern "C" void ms_east_params_default(ms_east_params *p)
{
    // EAST.__init__ defaults, infer.py:28-43
    if (!p) return;
    p->score_thresh = 0.6f;
    p->scale = 1.0 / 0.25;
    p->quantization = 2;
    p->iou_threshold = 0.2;
    p->expand_ratio_w = 0.9;
    p->expand_ratio_h = 0.9;
    p->target_size = 1280;
    p->axis_aligned_output = 1;
    p->remove_area_anomalies = 1;
    p->anomaly_sigma_threshold = 5.0;
    p->anomaly_min_box_count = 30;
    p->sort_reading_order = 0;
}

extern "C" int ms_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---- context --------------------------------------------------------------------------------------------
extern "C" int ms_create(int device, ms_ctx **out)
{
    if (!out) {
        ms_set_error("ms_create: out is NULL");
        return MS_ERR_INVALID;
    }
    *out = nullptr;
    int n = ms_device_count();
    if (n <= 0) {
        ms_set_error("ms_create: no CUDA device (this library has no CPU path)");
        return MS_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) {
        ms_set_error("ms_create: device %d out of range [0,%d)", device, n);
        return MS_ERR_INVALID;
    }
    MS_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MS_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        ms_set_error("ms_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                     prop.minor);
        return MS_ERR_NO_DEVICE;
    }
    ms_ctx *c = new (std::nothrow) ms_ctx();
    if (!c) {
        ms_set_error("ms_create: out of host memory");
        return MS_ERR_INVALID;
    }
    memset(c, 0, sizeof(*c));
    c->device = device;
    c->num_sms = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : MS_NUM_SMS_B200;
    c->edge_factor = 16;
    c->graphs_enabled = getenv("MS_B200_NO_GRAPHS") ? 0 : 1;
    c->ro_force_large = getenv("MS_B200_RO_FORCE_LARGE") ? 1 : 0;
    c->split_front = getenv("MS_B200_NO_SPLIT") ? 0 : 1;
    c->quad_no_stage = getenv("MS_B200_QUAD_NO_STAGE") ? 1 : 0;
    int rc = ms_check_cuda(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    if (rc == MS_OK) rc = ms_check_cuda(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    if (rc == MS_OK) rc = ms_check_cuda(cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    for (int i = 0; i < 2 && rc == MS_OK; i++)
        rc = ms_check_cuda(cudaEventCreateWithFlags(&c->split_ev[i], cudaEventDisableTiming), "cudaEventCreate");
    for (int i = 0; i < 2 && rc == MS_OK; i++)
        rc = ms_check_cuda(cudaEventCreateWithFlags(&c->chunk_ev[i], cudaEventDisableTiming), "cudaEventCreate");
    if (rc == MS_OK)
        rc = ms_check_cuda(cudaEventCreateWithFlags(&c->jpeg_ev, cudaEventDisableTiming), "cudaEventCreate");
    if (rc == MS_OK) {
        c->pinned_bytes = 1 << 20;
        rc = ms_check_cuda(cudaMallocHost((void **)&c->pinned, c->pinned_bytes), "cudaMallocHost");
    }
    if (rc != MS_OK) {
        ms_destroy(c);
        return rc;
    }
    *out = c;
    return MS_OK;
}

extern "C" void ms_destroy(ms_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) {
        cudaStreamSynchronize(ctx->own_stream);
        cudaStreamDestroy(ctx->own_stream);
    }
    if (ctx->aux_stream) {
        cudaStreamSynchronize(ctx->aux_stream);
        cudaStreamDestroy(ctx->aux_stream);
    }
    for (int i = 0; i < 2; i++)
        if (ctx->split_ev[i]) cudaEventDestroy(ctx->split_ev[i]);
    if (ctx->copy_stream) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamDestroy(ctx->copy_stream);
    }
    for (int i = 0; i < 2; i++)
        if (ctx->chunk_ev[i]) cudaEventDestroy(ctx->chunk_ev[i]);
    if (ctx->timing_ev) {
        for (int i = 0; i < MS_TIMING_RING * (MS_N_STAGES + 1); i++) cudaEventDestroy(ctx->timing_ev[i]);
        free(ctx->timing_ev);
    }
    for (int i = 0; i < MS_GRAPH_SLOTS; i++)
        if (ctx->graphs[i].exec) cudaGraphExecDestroy(ctx->graphs[i].exec);
    if (ctx->arena) cudaFree(ctx->arena);
    if (ctx->stage) cudaFree(ctx->stage);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->jpeg_ev) {
        cudaEventSynchronize(ctx->jpeg_ev);
        cudaEventDestroy(ctx->jpeg_ev);
    }
    if (ctx->jpeg_pinned) cudaFreeHost(ctx->jpeg_pinned);
    delete ctx;
}

extern "C" int64_t ms_launch_count(const ms_ctx *ctx) { return ctx ? ctx->launches : 0; }

extern "C" int ms_set_edge_factor(ms_ctx *ctx, int pairs_per_candidate)
{
    if (!ctx || pairs_per_candidate < 1 || pairs_per_candidate > 4096) {
        ms_set_error("ms_set_edge_factor: bad arguments");
        return MS_ERR_INVALID;
    }
    ctx->edge_factor = pairs_per_candidate;
    return MS_OK;
}

extern "C" int ms_get_edge_factor(const ms_ctx *ctx) { return ctx ? ctx->edge_factor : 0; }

// dense candidates can exceed the NMS neighbour-pair capacity: the host entry points grow it and run again
static bool grow_edge_factor(ms_ctx *ctx, int32_t flags)
{
    if (!(flags & MS_FLAG_EDGE_OVERFLOW) || (flags & (MS_FLAG_INDEX_ERROR | MS_FLAG_CAND_OVERFLOW))) return false;
    if (ctx->edge_factor >= 4096) return false;
    ctx->edge_factor *= 4;
    return true;
}

extern "C" int ms_stage_timing(ms_ctx *ctx, int enable)
{
    if (!ctx) return MS_ERR_INVALID;
    MS_CUDA(cudaSetDevice(ctx->device));
    if (enable && !ctx->timing_ev) {
        const int n = MS_TIMING_RING * (MS_N_STAGES + 1);
        ctx->timing_ev = (cudaEvent_t *)calloc(n, sizeof(cudaEvent_t));
        if (!ctx->timing_ev) return MS_ERR_INVALID;
        for (int i = 0; i < n; i++) MS_CUDA(cudaEventCreate(&ctx->timing_ev[i]));
    }
    ctx->timing = enable ? 1 : 0;
    ctx->timing_n = 0;
    return MS_OK;
}

extern "C" int ms_stage_times(ms_ctx *ctx, double *ms)
{
    if (!ctx || !ms) return MS_ERR_INVALID;
    MS_CUDA(cudaSetDevice(ctx->device));
    for (int s = 0; s < MS_N_STAGES; s++) ms[s] = 0.0;
    const int n = ctx->timing_n;
    for (int b = 0; b < n; b++) {
        cudaEvent_t *ev = ctx->timing_ev + (size_t)b * (MS_N_STAGES + 1);
        MS_CUDA(cudaEventSynchronize(ev[MS_N_STAGES]));
        for (int s = 0; s < MS_N_STAGES; s++) {
            float t = 0.f;
            MS_CUDA(cudaEventElapsedTime(&t, ev[s], ev[s + 1]));
            ms[s] += (double)t;
        }
    }
    ctx->timing_n = 0;
    return n;
}

// records the boundary event `idx` of the current batch when stage timing is on
static int timing_mark(ms_ctx *ctx, int idx, cudaStream_t st)
{
    if (!ctx->timing || !ctx->timing_ev || ctx->timing_n >= MS_TIMING_RING) return MS_OK;
    MS_CUDA(cudaEventRecord(ctx->timing_ev[(size_t)ctx->timing_n * (MS_N_STAGES + 1) + idx], st));
    if (idx == MS_N_STAGES) ctx->timing_n++;
    return MS_OK;
}

static int grow(char **buf, size_t *have, size_t want, const char *what)
{
    if (want <= *have) return MS_OK;
    // growing frees memory that queued work may still use: drain the device first
    MS_CUDA(cudaDeviceSynchronize());
    if (*buf) MS_CUDA(cudaFree(*buf));
    *buf = nullptr;
    *have = 0;
    size_t sz = want + want / 4 + (1 << 20);
    cudaError_t e = cudaMalloc((void **)buf, sz);
    if (e != cudaSuccess) {
        cudaGetLastError();
        sz = want;
        e = cudaMalloc((void **)buf, sz);
    }
    if (e != cudaSuccess) {
        ms_set_error("%s: cudaMalloc(%zu) failed: %s", what, sz, cudaGetErrorString(e));
        return MS_ERR_CUDA;
    }
    *have = sz;
    return MS_OK;
}

int ms_arena_reserve(ms_ctx *ctx, size_t bytes)
{
    if (bytes > ctx->arena_bytes) {  // the counters of the last rotated- and axis-crop calls go with the old arena
        ctx->quad_cnt = nullptr;
        ctx->crop_cnt = nullptr;
    }
    return grow(&ctx->arena, &ctx->arena_bytes, bytes, "arena");
}
int ms_stage_reserve(ms_ctx *ctx, size_t bytes) { return grow(&ctx->stage, &ctx->stage_bytes, bytes, "stage"); }

// the whole scratch arena as `bump`, grown to at least `bytes` first
static int arena_bump(ms_ctx *ctx, size_t bytes, ms_bump &bump)
{
    MS_TRY(ms_arena_reserve(ctx, bytes));
    bump = ms_bump{ctx->arena, 0, ctx->arena_bytes};
    return MS_OK;
}

// The device staging of a host entry point: carve(ms_bump &) takes the call's buffers from the bump.  A first pass
// over an empty bump measures them, the stage grows to that size, and a second pass hands them out.
template <typename Carve>
static int stage_carve(ms_ctx *ctx, const char *who, Carve &&carve)
{
    ms_bump probe{nullptr, 0, 0};
    carve(probe);
    MS_TRY(ms_stage_reserve(ctx, probe.off));
    ms_bump sb{ctx->stage, 0, ctx->stage_bytes};
    carve(sb);
    if (sb.off > sb.cap) {
        ms_set_error("%s: staging too small", who);
        return MS_ERR_CAPACITY;
    }
    return MS_OK;
}

static inline size_t al256(size_t b) { return (b + 255) & ~size_t(255); }

// Entry guard: a context is single-threaded by contract (one scratch arena); the guard turns a violation into an error.
struct ms_ctx_guard {
    ms_ctx *c = nullptr;
    int enter(ms_ctx *ctx, const char *fn)
    {
        if (__atomic_exchange_n(&ctx->busy, 1, __ATOMIC_ACQUIRE) != 0) {
            ms_set_error("%s: this ms_ctx is in use by another thread (one context per thread)", fn);
            return MS_ERR_INVALID;
        }
        c = ctx;
        return MS_OK;
    }
    ~ms_ctx_guard()
    {
        if (c) __atomic_store_n(&c->busy, 0, __ATOMIC_RELEASE);
    }
};

#define MS_CTX(ctx)                                          \
    if (!(ctx)) {                                            \
        ms_set_error("%s: ctx is NULL", __func__);           \
        return MS_ERR_INVALID;                               \
    }                                                        \
    ms_ctx_guard _ms_guard;                                  \
    {                                                        \
        int _grc = _ms_guard.enter((ctx), __func__);         \
        if (_grc != MS_OK) return _grc;                      \
    }                                                        \
    MS_CUDA(cudaSetDevice((ctx)->device))

static int flags_to_rc(int32_t f, const char *where)
{
    if (f & MS_FLAG_INDEX_ERROR) {
        ms_set_error("%s: quantised pixel index outside the map (the reference raises IndexError, utils.py:370); "
                     "map sides must be multiples of the quantisation step",
                     where);
        return MS_ERR_INDEX;
    }
    if (f & MS_FLAG_CAND_OVERFLOW) {
        ms_set_error("%s: more candidates than the output capacity", where);
        return MS_ERR_CAPACITY;
    }
    if (f & MS_FLAG_EDGE_OVERFLOW) {
        ms_set_error("%s: NMS suppression-edge buffer exceeded", where);
        return MS_ERR_CAPACITY;
    }
    if (f & MS_FLAG_ORDER_OVERFLOW) {
        ms_set_error("%s: a page exceeds the device reading-order capacity (max(65536, 16 cap_boxes) intersecting box "
                     "pairs); run with sort_reading_order = 0 and order the boxes on the host", where);
        return MS_ERR_CAPACITY;
    }
    return MS_OK;
}

// =========================================================================================================
// device entry points
// =========================================================================================================
// An ms_maps descriptor: what can be checked before the page count (a NULL descriptor, an unknown dtype, a negative
// stride), then, for a call with pages, its map pointers.
static int maps_desc_ok(const ms_maps *m, const char *who)
{
    if (!m) {
        ms_set_error("%s: maps is NULL", who);
        return MS_ERR_INVALID;
    }
    if (ms_dtype_bytes(m->dtype) == 0) {
        ms_set_error("%s: unknown map dtype %d", who, (int)m->dtype);
        return MS_ERR_INVALID;
    }
    for (int i = 0; i < 3; i++)
        if (m->score_strides[i] < 0) {
            ms_set_error("%s: negative score stride", who);
            return MS_ERR_INVALID;
        }
    for (int i = 0; i < 4; i++)
        if (m->geo_strides[i] < 0) {
            ms_set_error("%s: negative geometry stride", who);
            return MS_ERR_INVALID;
        }
    return MS_OK;
}

extern "C" int ms_decode_quads_maps(ms_ctx *ctx, const ms_maps *maps, int n_pages, int map_h, int map_w,
                                    float score_thresh, double scale, int quantization, float *quads_out,
                                    int cap_per_page, int32_t *counts, int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(maps_desc_ok(maps, "ms_decode_quads"));
    if (n_pages <= 0) return MS_OK;
    if (!maps->score || !maps->geo || !quads_out || !counts || !flags) {
        ms_set_error("ms_decode_quads: NULL pointer");
        return MS_ERR_INVALID;
    }
    if (quantization < 1) quantization = 1;  // utils.py:347 only quantises when > 1
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_decode_scratch(n_pages, map_h, map_w, quantization), bump));
    return msk_decode(ctx, *maps, n_pages, map_h, map_w, score_thresh, scale, quantization, quads_out, cap_per_page,
                      counts, flags, bump, (cudaStream_t)stream);
}

extern "C" int ms_decode_quads(ms_ctx *ctx, const float *score, const float *geo, int n_pages, int map_h, int map_w,
                               float score_thresh, double scale, int quantization, float *quads_out, int cap_per_page,
                               int32_t *counts, int32_t *flags, void *stream)
{
    const ms_maps m = ms_dense_maps(score, geo, map_h, map_w, map_h, 8);
    return ms_decode_quads_maps(ctx, &m, n_pages, map_h, map_w, score_thresh, scale, quantization, quads_out,
                                cap_per_page, counts, flags, stream);
}

extern "C" int ms_decode_rbox(ms_ctx *ctx, const float *score, const float *geo5, int n_pages, int map_h, int map_w,
                              float score_thresh, double scale, int quantization, float *quads_out, int cap_per_page,
                              int32_t *counts, int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    if (n_pages <= 0) return MS_OK;
    if (!score || !geo5 || !quads_out || !counts || !flags) {
        ms_set_error("ms_decode_rbox: NULL pointer");
        return MS_ERR_INVALID;
    }
    if (quantization < 1) quantization = 1;
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_decode_scratch(n_pages, map_h, map_w, quantization), bump));
    return msk_decode(ctx, ms_dense_maps(score, geo5, map_h, map_w, map_h, 5), n_pages, map_h, map_w, score_thresh,
                      scale, quantization, quads_out, cap_per_page, counts, flags, bump, (cudaStream_t)stream, 0, 1);
}

extern "C" int ms_lanms(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                        double iou_threshold, float *quads_out, int32_t *counts_out, int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    if (n_pages <= 0) return MS_OK;
    if (!quads || !counts || !quads_out || !counts_out || !flags || cap_per_page <= 0) {
        ms_set_error("ms_lanms: bad arguments");
        return MS_ERR_INVALID;
    }
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_lanms_scratch(n_pages, cap_per_page, ctx->edge_factor), bump));
    return msk_lanms(ctx, quads, counts, n_pages, cap_per_page, iou_threshold, quads_out, counts_out, flags, bump,
                     (cudaStream_t)stream);
}

extern "C" int ms_east_boxes(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                             const ms_east_params *p, const int32_t *orig_hw, float *quads_out, int32_t *counts_out,
                             void *stream)
{
    MS_CTX(ctx);
    if (n_pages <= 0) return MS_OK;
    if (!quads || !counts || !quads_out || !counts_out || !p || cap_per_page <= 0) {
        ms_set_error("ms_east_boxes: bad arguments");
        return MS_ERR_INVALID;
    }
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_east_boxes_scratch(n_pages, cap_per_page), bump));
    return msk_east_boxes(ctx, quads, counts, n_pages, cap_per_page, p, orig_hw, quads_out, cap_per_page, counts_out,
                          nullptr, bump, (cudaStream_t)stream);
}

extern "C" int ms_reading_order(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                                int32_t *order, float *quads_out, int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    if (n_pages <= 0) return MS_OK;
    if (!quads || !counts || !order || !flags || cap_per_page <= 0 || quads_out == quads) {
        ms_set_error("ms_reading_order: bad arguments");
        return MS_ERR_INVALID;
    }
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_reading_order_scratch(n_pages, cap_per_page), bump));
    return msk_reading_order(ctx, quads, 9, counts, n_pages, cap_per_page, order, quads_out, flags, bump,
                             (cudaStream_t)stream);
}

extern "C" int ms_reading_order_host(ms_ctx *ctx, const float *polys8, int64_t n, int32_t *order)
{
    MS_CTX(ctx);
    if (n < 0 || (n > 0 && (!polys8 || !order))) {
        ms_set_error("ms_reading_order_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    if (n > (1 << 20)) {
        ms_set_error("ms_reading_order_host: more than 2^20 boxes on the page (got %lld)", (long long)n);
        return MS_ERR_CAPACITY;
    }
    const int cap = (int)n;
    float *d_p;
    int32_t *d_o, *d_i;
    MS_TRY(stage_carve(ctx, "ms_reading_order_host", [&](ms_bump &sb) {
        d_p = sb.take<float>((size_t)n * 8);
        d_o = sb.take<int32_t>((size_t)n);
        d_i = sb.take<int32_t>(2);
    }));
    cudaStream_t st = ctx->own_stream;
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    h[0] = cap;
    h[1] = 0;
    MS_CUDA(cudaMemcpyAsync(d_i, h, 2 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_p, polys8, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_reading_order_scratch(1, cap), bump));
    MS_TRY(msk_reading_order(ctx, d_p, 8, d_i, 1, cap, d_o, nullptr, d_i + 1, bump, st));
    MS_CUDA(cudaMemcpyAsync(order, d_o, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaMemcpyAsync(h + 4, d_i + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    if (h[4] & MS_FLAG_ORDER_OVERFLOW) {
        ms_set_error("ms_reading_order_host: more intersecting box pairs on the page than the device kernels hold "
                     "(max(65536, 16 n))");
        return MS_ERR_CAPACITY;
    }
    return MS_OK;
}

static size_t word_rects_scratch_full(int n_pages, int cap_per_page)
{
    return msk_word_rects_scratch(n_pages) + al256((size_t)n_pages * cap_per_page * 4 * sizeof(int32_t)) + 1024;
}

extern "C" int ms_word_rects(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                             const int32_t *img_hw, int img_h, int img_w, int min_text_size, int32_t *crops_out,
                             int64_t crops_cap, int32_t *n_crops, void *stream)
{
    MS_CTX(ctx);
    if (n_pages <= 0) return MS_OK;
    if (!quads || !counts || !crops_out || !n_crops || cap_per_page <= 0 || crops_cap < 0) {
        ms_set_error("ms_word_rects: bad arguments");
        return MS_ERR_INVALID;
    }
    ms_bump bump;
    MS_TRY(arena_bump(ctx, word_rects_scratch_full(n_pages, cap_per_page), bump));
    return msk_word_rects(ctx, quads, counts, n_pages, cap_per_page, img_hw, img_h, img_w, min_text_size, crops_out,
                          crops_cap, n_crops, 0, 0, nullptr, bump, (cudaStream_t)stream);
}

// the batch_dtype argument of an *_ex entry point
static int dtype_ok(int batch_dtype, const char *who)
{
    if (ms_dtype_bytes(batch_dtype) == 0) {
        ms_set_error("%s: unknown batch dtype %d (MS_DTYPE_F32, MS_DTYPE_F16 or MS_DTYPE_BF16)", who, batch_dtype);
        return MS_ERR_INVALID;
    }
    return MS_OK;
}

extern "C" int ms_crop_resize_pad_ex(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                                     const int32_t *crops, const int32_t *n_crops, int64_t crops_cap, int out_h,
                                     int out_w, void *batch, int batch_dtype, uint8_t *canvas_u8, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(batch_dtype, "ms_crop_resize_pad"));
    if (!pages || !crops || !n_crops) {
        ms_set_error("ms_crop_resize_pad: NULL pointer");
        return MS_ERR_INVALID;
    }
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_crop_scratch(crops_cap, n_pages), bump));
    return msk_crop(ctx, pages, n_pages, img_h, img_w, crops, n_crops, nullptr, crops_cap, out_h, out_w, batch,
                    batch_dtype, canvas_u8, bump, (cudaStream_t)stream);
}

extern "C" int ms_crop_resize_pad(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                                  const int32_t *crops, const int32_t *n_crops, int64_t crops_cap, int out_h, int out_w,
                                  float *batch_f32, uint8_t *canvas_u8, void *stream)
{
    return ms_crop_resize_pad_ex(ctx, pages, n_pages, img_h, img_w, crops, n_crops, crops_cap, out_h, out_w, batch_f32,
                                 MS_DTYPE_F32, canvas_u8, stream);
}

extern "C" int ms_detector_input(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, int target_h, int target_w,
                                 float *out_f32, uint8_t *out_u8, void *stream)
{
    MS_CTX(ctx);
    ms_bump bump;  // the arguments are checked by msk_detector_input
    MS_TRY(arena_bump(ctx, msk_detector_input_scratch(1, target_h, target_w), bump));
    return msk_detector_input(ctx, nullptr, nullptr, page, img_h, img_w, 1, target_h, target_w, out_f32, MS_DTYPE_F32,
                              out_u8, bump, (cudaStream_t)stream);
}

extern "C" int ms_detector_input_batch(ms_ctx *ctx, const uint8_t *const *page_ptrs, const int32_t *page_hw,
                                       int n_pages, int target_h, int target_w, void *out, int out_dtype, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(out_dtype, "ms_detector_input_batch"));
    if (!page_ptrs || !page_hw || !out) {
        ms_set_error("ms_detector_input_batch: NULL tables or output");
        return MS_ERR_INVALID;
    }
    ms_bump bump;  // the sizes are checked by msk_detector_input
    MS_TRY(arena_bump(ctx, msk_detector_input_scratch(n_pages, target_h, target_w), bump));
    return msk_detector_input(ctx, page_ptrs, page_hw, nullptr, 0, 0, n_pages, target_h, target_w, out, out_dtype,
                              nullptr, bump, (cudaStream_t)stream);
}

extern "C" int ms_tps_rectify(ms_ctx *ctx, const float *input, const float *c_prime, const float *inv_delta_c,
                              const float *p_hat_t, int batch, int n_fid, int chans, int in_h, int in_w, int out_h,
                              int out_w, float *out, void *stream)
{
    MS_CTX(ctx);
    return msk_tps_rectify(ctx, input, c_prime, inv_delta_c, p_hat_t, batch, n_fid, chans, in_h, in_w, out_h, out_w, out,
                           (cudaStream_t)stream);
}

// candidate capacity per page that can never overflow: one row per quantisation cell (utils.py:347-356)
static int cand_cap(int map_h, int map_w, int q)
{
    if (q < 1) q = 1;
    long long c = (long long)((map_h + q - 1) / q) * ((map_w + q - 1) / q);
    return (int)(c > 0x7fffffffLL ? 0x7fffffff : c);
}

// Scratch of the front stages (decode -> LANMS -> box filters -> reading order) for n_pages pages: the candidate / NMS
// buffers that live through all of them + the largest stage scratch.
static size_t front_scratch(int n_pages, int map_h, int map_w, int q, int cap_c, int ef, int cap_boxes)
{
    size_t fixed = 2 * al256((size_t)n_pages * cap_c * 9 * sizeof(float)) + 2 * al256((size_t)n_pages * sizeof(int32_t));
    size_t stage = msk_decode_scratch(n_pages, map_h, map_w, q);
    size_t s2 = msk_lanms_scratch(n_pages, cap_c, ef);
    if (s2 > stage) stage = s2;
    s2 = msk_east_boxes_scratch(n_pages, cap_c);
    if (s2 > stage) stage = s2;
    s2 = msk_reading_order_scratch(n_pages, cap_boxes);
    if (s2 > stage) stage = s2;
    // reading order keeps the unsorted boxes and the order next to the candidates for the rest of the call
    fixed += al256((size_t)n_pages * cap_boxes * 36) + al256((size_t)n_pages * cap_boxes * 4) + 512;
    return al256(fixed + stage + 4096);
}

// ... and of the tail (crop rectangles, crops; or the quad list, quad crops), which runs after the front stages and may
// reuse their bytes
static size_t tail_scratch(int n_pages, int cap_c, int64_t crops_cap, int total_pages, bool quads, int cap_boxes)
{
    size_t stage = quads ? msk_quad_list_scratch(n_pages, cap_boxes) : word_rects_scratch_full(n_pages, cap_c);
    const size_t s2 = quads ? msk_quad_crop_scratch(crops_cap) : msk_crop_scratch(crops_cap, total_pages);
    if (s2 > stage) stage = s2;
    return al256(stage + 4096);
}

// Pages below this count run their front stages as one sequence; from it on as two concurrent halves (see below).
#define MS_SPLIT_MIN_PAGES 16

static int pb_quant(const pb_call &c) { return c.params.quantization < 1 ? 1 : c.params.quantization; }

// A call with parameters *p and every other field zero.  The parameters are copied field by field: the caller's struct
// may carry indeterminate padding bytes, and a call is compared bytewise as a graph key (page_batch_cached).
static void pb_init(pb_call &c, const ms_east_params *p)
{
    memset(&c, 0, sizeof(c));
    c.params.score_thresh = p->score_thresh;
    c.params.scale = p->scale;
    c.params.quantization = p->quantization;
    c.params.iou_threshold = p->iou_threshold;
    c.params.expand_ratio_w = p->expand_ratio_w;
    c.params.expand_ratio_h = p->expand_ratio_h;
    c.params.target_size = p->target_size;
    c.params.axis_aligned_output = p->axis_aligned_output;
    c.params.remove_area_anomalies = p->remove_area_anomalies;
    c.params.anomaly_sigma_threshold = p->anomaly_sigma_threshold;
    c.params.anomaly_min_box_count = p->anomaly_min_box_count;
    c.params.sort_reading_order = p->sort_reading_order;
}

// The maps of a call, field by field for the same reason.
static void pb_set_maps(pb_call &c, const ms_maps *m)
{
    c.maps.score = m->score;
    c.maps.geo = m->geo;
    c.maps.dtype = m->dtype;
    for (int i = 0; i < 3; i++) c.maps.score_strides[i] = m->score_strides[i];
    for (int i = 0; i < 4; i++) c.maps.geo_strides[i] = m->geo_strides[i];
}

// the per-page arrays of a call from page `base` on
struct pb_pages {
    ms_maps maps;
    const int32_t *hw;
    float *boxes;
    int32_t *counts, *flags;
};
static pb_pages pb_at(const pb_call &c, int base)
{
    ms_maps m = c.maps;
    const int64_t es = (int64_t)ms_dtype_bytes(m.dtype);
    m.score = static_cast<const char *>(m.score) + base * m.score_strides[0] * es;
    m.geo = static_cast<const char *>(m.geo) + base * m.geo_strides[0] * es;
    return {m, c.page_hw ? c.page_hw + 2 * (size_t)base : nullptr, c.boxes_out + (size_t)base * c.cap_boxes * 9,
            c.box_counts + base, c.flags + base};
}

// decode -> LANMS -> expand + EAST filters (-> reading order) of pages [base, base + n) of call c on stream st, boxes
// into the call's boxes_out / box_counts.  marks: record the stage-timing events (the half that runs on the caller's
// stream does).
static int front_half(ms_ctx *ctx, const pb_call &c, int base, int n, ms_bump bump, cudaStream_t st, bool marks)
{
    const ms_east_params *p = &c.params;
    const int q = pb_quant(c), cap_c = cand_cap(c.map_h, c.map_w, q);
    const pb_pages pg = pb_at(c, base);
    float *qa = bump.take<float>((size_t)n * cap_c * 9);  // candidates
    float *qb = bump.take<float>((size_t)n * cap_c * 9);  // NMS output
    int32_t *ca = bump.take<int32_t>(n);
    int32_t *cb = bump.take<int32_t>(n);
    if (!cb) {
        ms_set_error("ms_page_batch: arena too small");
        return MS_ERR_CAPACITY;
    }
    MS_TRY(msk_decode(ctx, pg.maps, n, c.map_h, c.map_w, p->score_thresh, p->scale, q, qa, cap_c, ca, pg.flags, bump,
                      st, c.geo_compact));
    if (marks) MS_TRY(timing_mark(ctx, 1, st));
    MS_TRY(msk_lanms(ctx, qa, ca, n, cap_c, p->iou_threshold, qb, cb, pg.flags, bump, st));
    // expand + EAST filters; boxes are scaled to the page images' size (infer.py:134-147: the original image), or target_size
    if (marks) MS_TRY(timing_mark(ctx, 2, st));
    if (p->sort_reading_order) {
        // filtered boxes -> scratch, then into boxes_out in reading order (the order the crops are produced in)
        float *tmp = bump.take<float>((size_t)n * c.cap_boxes * 9);
        int32_t *ord = bump.take<int32_t>((size_t)n * c.cap_boxes);
        if (!ord) {
            ms_set_error("ms_page_batch: arena too small");
            return MS_ERR_CAPACITY;
        }
        MS_TRY(msk_east_boxes(ctx, qb, cb, n, cap_c, p, pg.hw, tmp, c.cap_boxes, pg.counts, pg.flags, bump, st, c.img_h,
                              c.img_w));
        MS_TRY(msk_reading_order(ctx, tmp, 9, pg.counts, n, c.cap_boxes, ord, pg.boxes, pg.flags, bump, st));
    } else {
        MS_TRY(msk_east_boxes(ctx, qb, cb, n, cap_c, p, pg.hw, pg.boxes, c.cap_boxes, pg.counts, pg.flags, bump, st,
                              c.img_h, c.img_w));
    }
    return MS_OK;
}

// Pages [page_base, page_base + n_pages) of call c through the whole path; the crop rows index all c.n_pages pages of
// the call (c.pages, or c.page_ptrs / c.page_hw: device images of their own sizes).  append != 0 adds this chunk's
// crops after the *n_crops rows already listed.
//
// The front stages of a batch of MS_SPLIT_MIN_PAGES pages or more run as TWO CONCURRENT HALVES (pages are independent):
// the first on the caller's stream, the second on the context's auxiliary stream, forked and joined with events (under
// stream capture they become two parallel branches of the graph).  Most front kernels are bound by latency -- one CTA
// (or one cluster) per page walking a serial recurrence, or lanes waiting on dependent loads -- and leave most of the
// SMs' issue slots free; the other half's kernels fill them.  The crop rectangles and the crop kernel then run once
// over all pages.  MS_B200_NO_SPLIT=1 keeps one sequence.
static int page_batch_impl(ms_ctx *ctx, const pb_call &c, int page_base, int n_pages, int append, cudaStream_t st)
{
    const bool ragged = c.page_ptrs != nullptr && c.page_hw != nullptr;
    const bool want_crops = (c.pages != nullptr || ragged) && c.crops_out != nullptr && c.n_crops != nullptr && c.crops_cap > 0;
    const int q = pb_quant(c);
    const int cap_c = cand_cap(c.map_h, c.map_w, q);
    const bool split = ctx->split_front && n_pages >= MS_SPLIT_MIN_PAGES && st != ctx->aux_stream;
    const int nA = split ? n_pages / 2 : n_pages, nB = n_pages - nA;
    const size_t szA = front_scratch(nA, c.map_h, c.map_w, q, cap_c, ctx->edge_factor, c.cap_boxes);
    const size_t szB = split ? front_scratch(nB, c.map_h, c.map_w, q, cap_c, ctx->edge_factor, c.cap_boxes) : 0;
    const size_t szT = tail_scratch(n_pages, cap_c, want_crops ? c.crops_cap : 0, c.n_pages, c.crop_quads != 0,
                                    c.cap_boxes);
    // (one sequence: the tail reuses the front stages' scratch; two halves: A | B | tail side by side)
    MS_TRY(ms_arena_reserve(ctx, split ? szA + szB + szT + 1024 : (szA > szT ? szA : szT) + 1024));
    ms_bump bumpA{ctx->arena, 0, split ? szA : ctx->arena_bytes};
    ms_bump bumpT{split ? ctx->arena + szA + szB : ctx->arena, 0, split ? ctx->arena_bytes - szA - szB : ctx->arena_bytes};
    const pb_pages pg = pb_at(c, page_base);
    MS_CUDA(cudaMemsetAsync(pg.flags, 0, (size_t)n_pages * sizeof(int32_t), st));
    MS_TRY(timing_mark(ctx, 0, st));
    if (split) {
        ms_bump bumpB{ctx->arena + szA, 0, szB};
        MS_CUDA(cudaEventRecord(ctx->split_ev[0], st));
        MS_CUDA(cudaStreamWaitEvent(ctx->aux_stream, ctx->split_ev[0], 0));
        int rc = front_half(ctx, c, page_base, nA, bumpA, st, true);
        if (rc == MS_OK) rc = front_half(ctx, c, page_base + nA, nB, bumpB, ctx->aux_stream, false);
        // always join (a capture must not end with the auxiliary stream still forked)
        const int rj = ms_check_cuda(cudaEventRecord(ctx->split_ev[1], ctx->aux_stream), "cudaEventRecord");
        const int rw = ms_check_cuda(cudaStreamWaitEvent(st, ctx->split_ev[1], 0), "cudaStreamWaitEvent");
        if (rc != MS_OK) return rc;
        if (rj != MS_OK) return rj;
        if (rw != MS_OK) return rw;
    } else {
        MS_TRY(front_half(ctx, c, page_base, n_pages, bumpA, st, true));
    }
    MS_TRY(timing_mark(ctx, 3, st));
    int32_t *range = bumpT.take<int32_t>(2);
    if (!range) {
        ms_set_error("ms_page_batch: arena too small");
        return MS_ERR_CAPACITY;
    }
    if (want_crops && c.crop_quads) {  // (page_base == 0, append == 0: the device entry points)
        MS_TRY(msk_quad_list(ctx, pg.boxes, pg.counts, n_pages, c.cap_boxes, c.pages, c.img_h, c.img_w, c.page_ptrs,
                             c.page_hw, c.min_text_size, c.crops_out, c.crops_cap, c.n_crops, bumpT, st));
        MS_TRY(timing_mark(ctx, 4, st));
        if (c.batch || c.canvas_u8)
            MS_TRY(msk_quad_crop_rows(ctx, pg.boxes, c.cap_boxes, n_pages, c.pages, c.img_h, c.img_w, c.page_ptrs,
                                      c.page_hw, c.crops_out, c.n_crops, c.crops_cap, c.min_text_size, c.border_mode,
                                      c.border_value, c.out_h, c.out_w, c.batch, c.batch_dtype, c.canvas_u8, bumpT, st));
    } else if (want_crops) {
        MS_TRY(msk_word_rects(ctx, pg.boxes, pg.counts, n_pages, c.cap_boxes, pg.hw, c.img_h, c.img_w, c.min_text_size,
                              c.crops_out, c.crops_cap, c.n_crops, page_base, append, range, bumpT, st));
        MS_TRY(timing_mark(ctx, 4, st));
        if (c.batch || c.canvas_u8)
            MS_TRY(msk_crop(ctx, c.pages, c.n_pages, c.img_h, c.img_w, c.crops_out, c.n_crops, range, c.crops_cap,
                            c.out_h, c.out_w, c.batch, c.batch_dtype, c.canvas_u8, bumpT, st, c.page_ptrs, c.page_hw));
    } else {
        MS_TRY(timing_mark(ctx, 4, st));
    }
    MS_TRY(timing_mark(ctx, MS_N_STAGES, st));
    return MS_OK;
}

// ms_page_batch / ms_page_batch_ragged: direct launches the first time a call is seen, graph capture (on the
// context's own stream, nothing executes) at its second occurrence, replay on the caller's stream from then on.
// Stage timing needs the events between the stages, so it always launches directly.
static int page_batch_cached(ms_ctx *ctx, const pb_call &c, cudaStream_t st)
{
    auto direct = [&](cudaStream_t s) { return page_batch_impl(ctx, c, 0, c.n_pages, 0, s); };
    if (!ctx->graphs_enabled || ctx->timing) return direct(st);
    // the stream is not part of the key: a graph is replayed on the caller's stream
    ms_pb_key key;
    memset(&key, 0, sizeof(key));
    memcpy(&key.call, &c, sizeof(c));
    key.arena = ctx->arena;
    key.arena_bytes = ctx->arena_bytes;
    key.edge_factor = ctx->edge_factor;
    ms_graph_entry *e = nullptr;
    for (int i = 0; i < MS_GRAPH_SLOTS; i++)
        if (ctx->graphs[i].used && memcmp(&ctx->graphs[i].key, &key, sizeof(key)) == 0) e = &ctx->graphs[i];
    if (e && e->exec) {
        e->used = ++ctx->graph_clock;
        MS_CUDA(cudaGraphLaunch(e->exec, st));
        ctx->launches += e->launches;
        return MS_OK;
    }
    if (e && !e->failed) {  // second occurrence: the arenas and kernel attributes were settled by the first
        e->used = ++ctx->graph_clock;
        const int64_t l0 = ctx->launches;
        cudaStream_t cap = ctx->own_stream;
        if (cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int rc = direct(cap);
            cudaGraph_t g = nullptr;
            const cudaError_t ce = cudaStreamEndCapture(cap, &g);
            const bool same_arena = ctx->arena == key.arena && ctx->arena_bytes == key.arena_bytes;
            if (rc == MS_OK && ce == cudaSuccess && g && same_arena &&
                cudaGraphInstantiate(&e->exec, g, 0) == cudaSuccess) {
                e->launches = ctx->launches - l0;
                ctx->launches = l0;
                cudaGraphDestroy(g);
                MS_CUDA(cudaGraphLaunch(e->exec, st));
                ctx->launches += e->launches;
                return MS_OK;
            }
            if (g) cudaGraphDestroy(g);
            e->exec = nullptr;
        }
        cudaGetLastError();  // a failed capture is not an error of the call: launch directly from now on
        ctx->launches = l0;
        e->failed = 1;
        return direct(st);
    }
    if (!e) {  // first occurrence: remember it (least recently used slot)
        int slot = 0;
        for (int i = 1; i < MS_GRAPH_SLOTS; i++)
            if (ctx->graphs[i].used < ctx->graphs[slot].used) slot = i;
        if (ctx->graphs[slot].exec) cudaGraphExecDestroy(ctx->graphs[slot].exec);
        memset(&ctx->graphs[slot], 0, sizeof(ms_graph_entry));
        ctx->graphs[slot].key = key;
        ctx->graphs[slot].used = ++ctx->graph_clock;
    }
    const int rc = direct(st);
    // the first run may have grown the arena: the remembered key then never matches again and is simply evicted
    return rc;
}

extern "C" int ms_page_batch_maps(ms_ctx *ctx, const ms_maps *maps, const uint8_t *pages, int n_pages, int map_h,
                                  int map_w, int img_h, int img_w, const ms_east_params *p, int min_text_size, int out_h,
                                  int out_w, int cap_boxes, float *boxes_out, int32_t *box_counts, int32_t *crops_out,
                                  int64_t crops_cap, int32_t *n_crops, void *batch, int batch_dtype, uint8_t *canvas_u8,
                                  int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(batch_dtype, "ms_page_batch"));
    MS_TRY(maps_desc_ok(maps, "ms_page_batch"));
    if (n_pages <= 0) return MS_OK;
    if (!maps->score || !maps->geo || !p || !boxes_out || !box_counts || !flags || cap_boxes <= 0) {
        ms_set_error("ms_page_batch: bad arguments");
        return MS_ERR_INVALID;
    }
    pb_call c;
    pb_init(c, p);
    pb_set_maps(c, maps);
    c.pages = pages;
    c.n_pages = n_pages; c.map_h = map_h; c.map_w = map_w; c.img_h = img_h; c.img_w = img_w;
    c.min_text_size = min_text_size; c.out_h = out_h; c.out_w = out_w; c.cap_boxes = cap_boxes; c.crops_cap = crops_cap;
    c.boxes_out = boxes_out; c.box_counts = box_counts; c.crops_out = crops_out; c.n_crops = n_crops;
    c.batch = batch; c.batch_dtype = batch_dtype; c.canvas_u8 = canvas_u8; c.flags = flags;
    return page_batch_cached(ctx, c, (cudaStream_t)stream);
}

extern "C" int ms_page_batch_ex(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages, int n_pages,
                                int map_h, int map_w, int img_h, int img_w, const ms_east_params *p, int min_text_size,
                                int out_h, int out_w, int cap_boxes, float *boxes_out, int32_t *box_counts,
                                int32_t *crops_out, int64_t crops_cap, int32_t *n_crops, void *batch, int batch_dtype,
                                uint8_t *canvas_u8, int32_t *flags, void *stream)
{
    const ms_maps m = ms_dense_maps(score, geo, map_h, map_w, map_h, 8);
    return ms_page_batch_maps(ctx, &m, pages, n_pages, map_h, map_w, img_h, img_w, p, min_text_size, out_h, out_w,
                              cap_boxes, boxes_out, box_counts, crops_out, crops_cap, n_crops, batch, batch_dtype,
                              canvas_u8, flags, stream);
}

extern "C" int ms_page_batch(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages, int n_pages,
                             int map_h, int map_w, int img_h, int img_w, const ms_east_params *p, int min_text_size,
                             int out_h, int out_w, int cap_boxes, float *boxes_out, int32_t *box_counts,
                             int32_t *crops_out, int64_t crops_cap, int32_t *n_crops, float *batch_f32,
                             uint8_t *canvas_u8, int32_t *flags, void *stream)
{
    return ms_page_batch_ex(ctx, score, geo, pages, n_pages, map_h, map_w, img_h, img_w, p, min_text_size, out_h, out_w,
                            cap_boxes, boxes_out, box_counts, crops_out, crops_cap, n_crops, batch_f32, MS_DTYPE_F32,
                            canvas_u8, flags, stream);
}

// =========================================================================================================
// host entry points (one page; copy in, run, copy out, synchronise)
// =========================================================================================================
static int decode_host_impl(ms_ctx *ctx, const float *score, const float *geo, int map_h, int map_w, float score_thresh,
                            double scale, int quantization, float *quads_out, int64_t cap, int64_t *n_out, int rbox);

extern "C" int ms_decode_quads_host(ms_ctx *ctx, const float *score, const float *geo, int map_h, int map_w,
                                    float score_thresh, double scale, int quantization, float *quads_out, int64_t cap,
                                    int64_t *n_out)
{
    return decode_host_impl(ctx, score, geo, map_h, map_w, score_thresh, scale, quantization, quads_out, cap, n_out, 0);
}

extern "C" int ms_decode_rbox_host(ms_ctx *ctx, const float *score, const float *geo5, int map_h, int map_w,
                                   float score_thresh, double scale, int quantization, float *quads_out, int64_t cap,
                                   int64_t *n_out)
{
    return decode_host_impl(ctx, score, geo5, map_h, map_w, score_thresh, scale, quantization, quads_out, cap, n_out, 1);
}

static int decode_host_impl(ms_ctx *ctx, const float *score, const float *geo, int map_h, int map_w, float score_thresh,
                            double scale, int quantization, float *quads_out, int64_t cap, int64_t *n_out, int rbox)
{
    MS_CTX(ctx);
    const int planes = rbox ? 5 : 8;
    if (!score || !geo || !n_out || map_h <= 0 || map_w <= 0 || cap < 0 || (cap > 0 && !quads_out)) {
        ms_set_error("ms_decode_quads_host: bad arguments");
        return MS_ERR_INVALID;
    }
    *n_out = 0;
    if (quantization < 1) quantization = 1;
    const size_t plane = (size_t)map_h * map_w;
    int capd = cand_cap(map_h, map_w, quantization);
    if (cap < capd) capd = (int)cap;
    if (capd < 1) capd = 1;
    float *d_score, *d_geo, *d_out;
    int32_t *d_cnt;
    MS_TRY(stage_carve(ctx, "ms_decode_quads_host", [&](ms_bump &sb) {
        d_score = sb.take<float>(plane);
        d_geo = sb.take<float>(plane * planes);
        d_out = sb.take<float>((size_t)capd * 9);
        d_cnt = sb.take<int32_t>(2);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_score, score, plane * 4, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_geo, geo, plane * 4 * planes, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(int32_t), st));
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_decode_scratch(1, map_h, map_w, quantization), bump));
    MS_TRY(msk_decode(ctx, ms_dense_maps(d_score, d_geo, map_h, map_w, map_h, planes), 1, map_h, map_w, score_thresh,
                      scale, quantization, d_out, capd, d_cnt, d_cnt + 1, bump, st, 0, rbox));
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    MS_CUDA(cudaMemcpyAsync(h, d_cnt, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    MS_TRY(flags_to_rc(h[1], "decode_quads"));
    const int n = h[0];
    if (n > 0) {
        MS_CUDA(cudaMemcpyAsync(quads_out, d_out, (size_t)n * 36, cudaMemcpyDeviceToHost, st));
        MS_CUDA(cudaStreamSynchronize(st));
    }
    *n_out = n;
    return MS_OK;
}

extern "C" int ms_lanms_host(ms_ctx *ctx, const float *boxes, int64_t n, double iou_threshold, float *out,
                             int64_t *m_out)
{
    MS_CTX(ctx);
    if (!m_out || n < 0 || (n > 0 && (!boxes || !out))) {
        ms_set_error("ms_lanms_host: bad arguments");
        return MS_ERR_INVALID;
    }
    *m_out = 0;
    if (n == 0) return MS_OK;  // lanms.py:163-164
    if (n >= (int64_t)1 << 30) {
        ms_set_error("ms_lanms_host: n too large");
        return MS_ERR_INVALID;
    }
    const int cap = (int)n;
    float *d_in, *d_out;
    int32_t *d_cnt;
    MS_TRY(stage_carve(ctx, "ms_lanms_host", [&](ms_bump &sb) {
        d_in = sb.take<float>((size_t)n * 9);
        d_out = sb.take<float>((size_t)n * 9);
        d_cnt = sb.take<int32_t>(3);
    }));
    cudaStream_t st = ctx->own_stream;
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    do {
        h[0] = cap;
        h[1] = 0;
        h[2] = 0;
        MS_CUDA(cudaMemcpyAsync(d_cnt, h, 3 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemcpyAsync(d_in, boxes, (size_t)n * 36, cudaMemcpyHostToDevice, st));
        ms_bump bump;
        MS_TRY(arena_bump(ctx, msk_lanms_scratch(1, cap, ctx->edge_factor), bump));
        MS_TRY(msk_lanms(ctx, d_in, d_cnt, 1, cap, iou_threshold, d_out, d_cnt + 1, d_cnt + 2, bump, st));
        MS_CUDA(cudaMemcpyAsync(h + 4, d_cnt, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MS_CUDA(cudaStreamSynchronize(st));
    } while (grow_edge_factor(ctx, h[6]));
    MS_TRY(flags_to_rc(h[6], "locality_aware_nms"));
    const int m = h[5];
    if (m > 0) {
        MS_CUDA(cudaMemcpyAsync(out, d_out, (size_t)m * 36, cudaMemcpyDeviceToHost, st));
        MS_CUDA(cudaStreamSynchronize(st));
    }
    *m_out = m;
    return MS_OK;
}

extern "C" int ms_standard_nms_host(ms_ctx *ctx, const double *polys, const double *scores, int64_t n,
                                    double iou_threshold, int64_t *keep_idx, int64_t *k_out)
{
    MS_CTX(ctx);
    if (!k_out || n < 0 || (n > 0 && (!polys || !scores || !keep_idx))) {
        ms_set_error("ms_standard_nms_host: bad arguments");
        return MS_ERR_INVALID;
    }
    *k_out = 0;
    if (n == 0) return MS_OK;
    if (n >= (int64_t)1 << 27) {
        ms_set_error("ms_standard_nms_host: n too large");
        return MS_ERR_INVALID;
    }
    double *d_p, *d_s;
    int32_t *d_keep, *d_cnt;
    MS_TRY(stage_carve(ctx, "ms_standard_nms_host", [&](ms_bump &sb) {
        d_p = sb.take<double>((size_t)n * 8);
        d_s = sb.take<double>((size_t)n);
        d_keep = sb.take<int32_t>((size_t)n);
        d_cnt = sb.take<int32_t>(2);
    }));
    cudaStream_t st = ctx->own_stream;
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    do {
        MS_CUDA(cudaMemcpyAsync(d_p, polys, (size_t)n * 64, cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemcpyAsync(d_s, scores, (size_t)n * 8, cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(int32_t), st));
        ms_bump bump;
        MS_TRY(arena_bump(ctx, msk_standard_nms_scratch((int)n, ctx->edge_factor), bump));
        MS_TRY(msk_standard_nms(ctx, d_p, d_s, (int)n, iou_threshold, d_keep, d_cnt, d_cnt + 1, bump, st));
        MS_CUDA(cudaMemcpyAsync(h, d_cnt, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MS_CUDA(cudaStreamSynchronize(st));
    } while (grow_edge_factor(ctx, h[1]));
    MS_TRY(flags_to_rc(h[1], "standard_nms"));
    const int k = h[0];
    if (k > 0) {
        // int32 on the device -> int64 for the caller, staged through a temporary host copy
        int32_t *tmp = (int32_t *)malloc((size_t)k * sizeof(int32_t));
        if (!tmp) {
            ms_set_error("ms_standard_nms_host: out of host memory");
            return MS_ERR_INVALID;
        }
        cudaError_t e = cudaMemcpyAsync(tmp, d_keep, (size_t)k * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            free(tmp);
            return ms_check_cuda(e, "standard_nms read-back");
        }
        for (int i = 0; i < k; i++) keep_idx[i] = tmp[i];
        free(tmp);
    }
    *k_out = k;
    return MS_OK;
}

extern "C" int ms_polygon_iou_host(ms_ctx *ctx, const double *subj, const double *clip, int64_t n, double *iou)
{
    MS_CTX(ctx);
    if (n < 0 || (n > 0 && (!subj || !clip || !iou))) {
        ms_set_error("ms_polygon_iou_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    double *d_a, *d_b, *d_o;
    MS_TRY(stage_carve(ctx, "ms_polygon_iou_host", [&](ms_bump &sb) {
        d_a = sb.take<double>((size_t)n * 8);
        d_b = sb.take<double>((size_t)n * 8);
        d_o = sb.take<double>((size_t)n);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_a, subj, (size_t)n * 64, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_b, clip, (size_t)n * 64, cudaMemcpyHostToDevice, st));
    MS_TRY(msk_polygon_iou(ctx, d_a, d_b, n, d_o, st));
    MS_CUDA(cudaMemcpyAsync(iou, d_o, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_test_iou_proved_host(ms_ctx *ctx, const double *subj, const double *clip, int64_t n, double thr,
                                       uint8_t *out)
{
    MS_CTX(ctx);
    if (n < 0 || (n > 0 && (!subj || !clip || !out))) {
        ms_set_error("ms_test_iou_proved_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    double *d_a, *d_b;
    uint8_t *d_o;
    MS_TRY(stage_carve(ctx, "ms_test_iou_proved_host", [&](ms_bump &sb) {
        d_a = sb.take<double>((size_t)n * 8);
        d_b = sb.take<double>((size_t)n * 8);
        d_o = sb.take<uint8_t>((size_t)n);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_a, subj, (size_t)n * 64, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_b, clip, (size_t)n * 64, cudaMemcpyHostToDevice, st));
    MS_TRY(msk_iou_proved(ctx, d_a, d_b, n, thr, d_o, st));
    MS_CUDA(cudaMemcpyAsync(out, d_o, (size_t)n, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_test_resize_tables_host(ms_ctx *ctx, int out_h, int out_w, const int32_t *wh, int64_t n_plans,
                                          int32_t *plans_out, const int32_t *axes, int64_t n_axes, int32_t *entries_out,
                                          int64_t entries_cap)
{
    MS_CTX(ctx);
    if (n_plans < 0 || n_axes < 0 || entries_cap < 0 || (n_plans > 0 && (!wh || !plans_out || out_h <= 0 || out_w <= 0)) ||
        (n_axes > 0 && (!axes || !entries_out))) {
        ms_set_error("ms_test_resize_tables_host: bad arguments");
        return MS_ERR_INVALID;
    }
    for (int64_t i = 0; i < n_plans; i++)
        if (wh[2 * i] <= 0 || wh[2 * i + 1] <= 0) {
            ms_set_error("ms_test_resize_tables_host: crop %lld is %d x %d", (long long)i, wh[2 * i], wh[2 * i + 1]);
            return MS_ERR_INVALID;
        }
    // the axes with the index of their first entry
    std::vector<int32_t> ax((size_t)n_axes * 4);
    int64_t total = 0;
    for (int64_t a = 0; a < n_axes; a++) {
        const int32_t ssize = axes[3 * a], dsize = axes[3 * a + 1], mode = axes[3 * a + 2];
        if (ssize <= 0 || dsize <= 0 || mode < 0 || mode > 4 || ssize >= 65536) {
            ms_set_error("ms_test_resize_tables_host: axis %lld (%d -> %d, mode %d)", (long long)a, ssize, dsize, mode);
            return MS_ERR_INVALID;
        }
        ax[4 * a] = ssize, ax[4 * a + 1] = dsize, ax[4 * a + 2] = mode, ax[4 * a + 3] = (int32_t)total;
        total += dsize;
        if (total > entries_cap || total >= ((int64_t)1 << 31)) {
            ms_set_error("ms_test_resize_tables_host: the axes have more than %lld entries", (long long)entries_cap);
            return MS_ERR_CAPACITY;
        }
    }
    if (n_plans == 0 && n_axes == 0) return MS_OK;
    int32_t *d_wh, *d_plans, *d_axes, *d_ent;
    MS_TRY(stage_carve(ctx, "ms_test_resize_tables_host", [&](ms_bump &sb) {
        d_wh = sb.take<int32_t>((size_t)n_plans * 2);
        d_plans = sb.take<int32_t>((size_t)n_plans * 8);
        d_axes = sb.take<int32_t>((size_t)n_axes * 4);
        d_ent = sb.take<int32_t>((size_t)total * 8);
    }));
    cudaStream_t st = ctx->own_stream;
    if (n_plans > 0) MS_CUDA(cudaMemcpyAsync(d_wh, wh, (size_t)n_plans * 8, cudaMemcpyHostToDevice, st));
    if (n_axes > 0) {
        MS_CUDA(cudaMemcpyAsync(d_axes, ax.data(), (size_t)n_axes * 16, cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemsetAsync(d_ent, 0, (size_t)total * 32, st));
    }
    MS_TRY(msk_test_resize_tables(ctx, out_h, out_w, d_wh, n_plans, d_plans, d_axes, n_axes, d_ent, st));
    if (n_plans > 0) MS_CUDA(cudaMemcpyAsync(plans_out, d_plans, (size_t)n_plans * 32, cudaMemcpyDeviceToHost, st));
    if (n_axes > 0) MS_CUDA(cudaMemcpyAsync(entries_out, d_ent, (size_t)total * 32, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_test_np_sum_host(ms_ctx *ctx, const float *values, const int64_t *offsets, const int32_t *lengths,
                                   int n_vec, float *out_serial, float *out_cta)
{
    MS_CTX(ctx);
    if (n_vec < 0 || (n_vec > 0 && (!values || !offsets || !lengths || !out_serial || !out_cta))) {
        ms_set_error("ms_test_np_sum_host: bad arguments");
        return MS_ERR_INVALID;
    }
    // the values span [0, max(offsets[v] + lengths[v])); every vector holds at least one value
    int64_t n_values = 0;
    for (int v = 0; v < n_vec; v++) {
        if (offsets[v] < 0 || lengths[v] <= 0) {
            ms_set_error("ms_test_np_sum_host: vector %d at %lld has %d values", v, (long long)offsets[v], lengths[v]);
            return MS_ERR_INVALID;
        }
        if (offsets[v] + lengths[v] > n_values) n_values = offsets[v] + lengths[v];
    }
    if (n_vec == 0) return MS_OK;
    float *d_val, *d_out;
    int64_t *d_off;
    int32_t *d_len;
    MS_TRY(stage_carve(ctx, "ms_test_np_sum_host", [&](ms_bump &sb) {
        d_val = sb.take<float>((size_t)n_values);
        d_off = sb.take<int64_t>((size_t)n_vec);
        d_len = sb.take<int32_t>((size_t)n_vec);
        d_out = sb.take<float>((size_t)n_vec * 2);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_val, values, (size_t)n_values * 4, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_off, offsets, (size_t)n_vec * 8, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_len, lengths, (size_t)n_vec * 4, cudaMemcpyHostToDevice, st));
    MS_TRY(msk_test_np_sum(ctx, d_val, d_off, d_len, n_vec, d_out, d_out + n_vec, st));
    MS_CUDA(cudaMemcpyAsync(out_serial, d_out, (size_t)n_vec * 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaMemcpyAsync(out_cta, d_out + n_vec, (size_t)n_vec * 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_expand_boxes_host(ms_ctx *ctx, const float *quads, int64_t n, double expand_w, double expand_h,
                                    float *out)
{
    MS_CTX(ctx);
    if (n < 0 || (n > 0 && (!quads || !out))) {
        ms_set_error("ms_expand_boxes_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    float *d_in, *d_out;
    MS_TRY(stage_carve(ctx, "ms_expand_boxes_host", [&](ms_bump &sb) {
        d_in = sb.take<float>((size_t)n * 9);
        d_out = sb.take<float>((size_t)n * 9);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_in, quads, (size_t)n * 36, cudaMemcpyHostToDevice, st));
    MS_TRY(msk_expand(ctx, d_in, n, expand_w, expand_h, d_out, st));
    MS_CUDA(cudaMemcpyAsync(out, d_out, (size_t)n * 36, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_east_boxes_host(ms_ctx *ctx, const float *quads, int64_t n, const ms_east_params *p, int orig_h,
                                  int orig_w, float *out, int64_t *m_out)
{
    MS_CTX(ctx);
    if (!m_out || !p || n < 0 || (n > 0 && (!quads || !out))) {
        ms_set_error("ms_east_boxes_host: bad arguments");
        return MS_ERR_INVALID;
    }
    *m_out = 0;
    if (n == 0) return MS_OK;
    if (n >= (int64_t)1 << 30) {
        ms_set_error("ms_east_boxes_host: n too large");
        return MS_ERR_INVALID;
    }
    const int cap = (int)n;
    float *d_in, *d_out;
    int32_t *d_i;
    MS_TRY(stage_carve(ctx, "ms_east_boxes_host", [&](ms_bump &sb) {
        d_in = sb.take<float>((size_t)n * 9);
        d_out = sb.take<float>((size_t)n * 9);
        d_i = sb.take<int32_t>(4);
    }));
    cudaStream_t st = ctx->own_stream;
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    h[0] = cap;
    h[1] = 0;
    h[2] = orig_h;
    h[3] = orig_w;
    MS_CUDA(cudaMemcpyAsync(d_i, h, 4 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_in, quads, (size_t)n * 36, cudaMemcpyHostToDevice, st));
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_east_boxes_scratch(1, cap), bump));
    MS_TRY(msk_east_boxes(ctx, d_in, d_i, 1, cap, p, d_i + 2, d_out, cap, d_i + 1, nullptr, bump, st));
    MS_CUDA(cudaMemcpyAsync(h + 8, d_i + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    const int m = h[8];
    if (m > 0) {
        MS_CUDA(cudaMemcpyAsync(out, d_out, (size_t)m * 36, cudaMemcpyDeviceToHost, st));
        MS_CUDA(cudaStreamSynchronize(st));
    }
    *m_out = m;
    return MS_OK;
}

extern "C" int ms_word_rects_host(ms_ctx *ctx, const float *polys8, int64_t n, int img_h, int img_w, int min_text_size,
                                  int32_t *rects, uint8_t *valid)
{
    MS_CTX(ctx);
    if (n < 0 || (n > 0 && (!polys8 || !rects || !valid))) {
        ms_set_error("ms_word_rects_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    float *d_p;
    int32_t *d_r;
    uint8_t *d_v;
    MS_TRY(stage_carve(ctx, "ms_word_rects_host", [&](ms_bump &sb) {
        d_p = sb.take<float>((size_t)n * 8);
        d_r = sb.take<int32_t>((size_t)n * 4);
        d_v = sb.take<uint8_t>((size_t)n);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_p, polys8, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    MS_TRY(msk_word_rects_flat(ctx, d_p, n, img_h, img_w, min_text_size, d_r, d_v, st));
    MS_CUDA(cudaMemcpyAsync(rects, d_r, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaMemcpyAsync(valid, d_v, (size_t)n, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

__global__ void ms_rects_to_crops_kernel(const int32_t *__restrict__ rects, int64_t n, int32_t *__restrict__ crops,
                                         int32_t *__restrict__ n_crops)
{
    ms_pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        crops[i * 5] = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) crops[i * 5 + 1 + k] = rects[i * 4 + k];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_crops = (int32_t)n;
}

extern "C" int ms_crop_resize_pad_host(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const int32_t *rects,
                                       int64_t n, int out_h, int out_w, float *batch_f32, uint8_t *canvas_u8)
{
    MS_CTX(ctx);
    if (n < 0 || img_h <= 0 || img_w <= 0 || out_h <= 0 || out_w <= 0 || (n > 0 && (!page || !rects)) ||
        (!batch_f32 && !canvas_u8)) {
        ms_set_error("ms_crop_resize_pad_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    if (n >= (int64_t)1 << 30) {
        ms_set_error("ms_crop_resize_pad_host: n too large");
        return MS_ERR_INVALID;
    }
    const size_t page_bytes = (size_t)img_h * img_w * 3;
    const size_t one_f = (size_t)3 * out_h * out_w * sizeof(float), one_u = (size_t)3 * out_h * out_w;
    uint8_t *d_page, *d_u;
    int32_t *d_rects, *d_crops, *d_n;
    float *d_f;
    MS_TRY(stage_carve(ctx, "ms_crop_resize_pad_host", [&](ms_bump &sb) {
        d_page = sb.take<uint8_t>(page_bytes);
        d_rects = sb.take<int32_t>((size_t)n * 4);
        d_crops = sb.take<int32_t>((size_t)n * 5);
        d_n = sb.take<int32_t>(1);
        d_f = batch_f32 ? sb.take<float>((size_t)n * 3 * out_h * out_w) : nullptr;
        d_u = canvas_u8 ? sb.take<uint8_t>((size_t)n * one_u) : nullptr;
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_page, page, page_bytes, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_rects, rects, (size_t)n * 16, cudaMemcpyHostToDevice, st));
    {
        int grid = (int)((n + 255) / 256);
        if (grid > ctx->num_sms * 4) grid = ctx->num_sms * 4;
        ms_launch(ms_rects_to_crops_kernel, grid, 256, 0, st, d_rects, n, d_crops, d_n);
        MS_LAUNCH_CHECK(ctx);
    }
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_crop_scratch(n, 1), bump));
    MS_TRY(msk_crop(ctx, d_page, 1, img_h, img_w, d_crops, d_n, nullptr, n, out_h, out_w, d_f, MS_DTYPE_F32, d_u, bump,
                    st));
    if (batch_f32) MS_CUDA(cudaMemcpyAsync(batch_f32, d_f, (size_t)n * one_f, cudaMemcpyDeviceToHost, st));
    if (canvas_u8) MS_CUDA(cudaMemcpyAsync(canvas_u8, d_u, (size_t)n * one_u, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_page_batch_ragged_maps(ms_ctx *ctx, const ms_maps *maps, const uint8_t *const *page_ptrs,
                                         const int32_t *page_hw, int n_pages, int map_h, int map_w,
                                         const ms_east_params *p, int min_text_size, int out_h, int out_w, int cap_boxes,
                                         float *boxes_out, int32_t *box_counts, int32_t *crops_out, int64_t crops_cap,
                                         int32_t *n_crops, void *batch, int batch_dtype, uint8_t *canvas_u8,
                                         int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(batch_dtype, "ms_page_batch_ragged"));
    MS_TRY(maps_desc_ok(maps, "ms_page_batch_ragged"));
    if (n_pages <= 0) return MS_OK;
    if (!maps->score || !maps->geo || !p || !page_ptrs || !page_hw || !boxes_out || !box_counts || !flags ||
        cap_boxes <= 0) {
        ms_set_error("ms_page_batch_ragged: bad arguments");
        return MS_ERR_INVALID;
    }
    pb_call c;
    pb_init(c, p);
    pb_set_maps(c, maps);
    c.page_ptrs = page_ptrs; c.page_hw = page_hw;
    c.n_pages = n_pages; c.map_h = map_h; c.map_w = map_w;
    c.min_text_size = min_text_size; c.out_h = out_h; c.out_w = out_w; c.cap_boxes = cap_boxes; c.crops_cap = crops_cap;
    c.boxes_out = boxes_out; c.box_counts = box_counts; c.crops_out = crops_out; c.n_crops = n_crops;
    c.batch = batch; c.batch_dtype = batch_dtype; c.canvas_u8 = canvas_u8; c.flags = flags;
    return page_batch_cached(ctx, c, (cudaStream_t)stream);
}

extern "C" int ms_page_batch_ragged_ex(ms_ctx *ctx, const float *score, const float *geo,
                                       const uint8_t *const *page_ptrs, const int32_t *page_hw, int n_pages, int map_h,
                                       int map_w, const ms_east_params *p, int min_text_size, int out_h, int out_w,
                                       int cap_boxes, float *boxes_out, int32_t *box_counts, int32_t *crops_out,
                                       int64_t crops_cap, int32_t *n_crops, void *batch, int batch_dtype,
                                       uint8_t *canvas_u8, int32_t *flags, void *stream)
{
    const ms_maps m = ms_dense_maps(score, geo, map_h, map_w, map_h, 8);
    return ms_page_batch_ragged_maps(ctx, &m, page_ptrs, page_hw, n_pages, map_h, map_w, p, min_text_size, out_h,
                                     out_w, cap_boxes, boxes_out, box_counts, crops_out, crops_cap, n_crops, batch,
                                     batch_dtype, canvas_u8, flags, stream);
}

extern "C" int ms_page_batch_ragged(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *const *page_ptrs,
                                    const int32_t *page_hw, int n_pages, int map_h, int map_w, const ms_east_params *p,
                                    int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                                    int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                                    float *batch_f32, uint8_t *canvas_u8, int32_t *flags, void *stream)
{
    return ms_page_batch_ragged_ex(ctx, score, geo, page_ptrs, page_hw, n_pages, map_h, map_w, p, min_text_size, out_h,
                                   out_w, cap_boxes, boxes_out, box_counts, crops_out, crops_cap, n_crops, batch_f32,
                                   MS_DTYPE_F32, canvas_u8, flags, stream);
}

// ---- EXTENSION -- not a reference behaviour: page batches whose crop stage is the rectified crop of every final quad --
static int quad_batch_args_ok(int batch_dtype, int border_mode, int border_value, const char *who)
{
    MS_TRY(dtype_ok(batch_dtype, who));
    if (border_mode < 0 || border_mode > 1 || border_value < 0 || border_value > 255) {
        ms_set_error("%s: border_mode must be 0 (constant) or 1 (replicate), border_value 0..255", who);
        return MS_ERR_INVALID;
    }
    return MS_OK;
}

extern "C" int ms_page_batch_quads_maps(ms_ctx *ctx, const ms_maps *maps, const uint8_t *pages, int n_pages,
                                        int map_h, int map_w, int img_h, int img_w, const ms_east_params *p,
                                        int min_text_size, int border_mode, int border_value, int out_h, int out_w,
                                        int cap_boxes, float *boxes_out, int32_t *box_counts, int32_t *crops_out,
                                        int64_t crops_cap, int32_t *n_crops, void *batch, int batch_dtype,
                                        uint8_t *canvas_u8, int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(quad_batch_args_ok(batch_dtype, border_mode, border_value, "ms_page_batch_quads"));
    MS_TRY(maps_desc_ok(maps, "ms_page_batch_quads"));
    if (n_pages <= 0) return MS_OK;
    if (!maps->score || !maps->geo || !p || !boxes_out || !box_counts || !flags || cap_boxes <= 0) {
        ms_set_error("ms_page_batch_quads: bad arguments");
        return MS_ERR_INVALID;
    }
    if (pages && (img_h <= 0 || img_w <= 0 || img_h > 32767 || img_w > 32767)) {
        ms_set_error("ms_page_batch_quads: pages must be 1..32767 pixels on a side (16-bit remap coordinates), got %dx%d",
                     img_h, img_w);
        return MS_ERR_INVALID;
    }
    pb_call c;
    pb_init(c, p);
    pb_set_maps(c, maps);
    c.pages = pages;
    c.n_pages = n_pages; c.map_h = map_h; c.map_w = map_w; c.img_h = img_h; c.img_w = img_w;
    c.min_text_size = min_text_size; c.out_h = out_h; c.out_w = out_w; c.cap_boxes = cap_boxes; c.crops_cap = crops_cap;
    c.boxes_out = boxes_out; c.box_counts = box_counts; c.crops_out = crops_out; c.n_crops = n_crops;
    c.batch = batch; c.batch_dtype = batch_dtype; c.canvas_u8 = canvas_u8; c.flags = flags;
    c.crop_quads = 1; c.border_mode = border_mode; c.border_value = border_value;
    return page_batch_cached(ctx, c, (cudaStream_t)stream);
}

extern "C" int ms_page_batch_quads(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages, int n_pages,
                                   int map_h, int map_w, int img_h, int img_w, const ms_east_params *p,
                                   int min_text_size, int border_mode, int border_value, int out_h, int out_w,
                                   int cap_boxes, float *boxes_out, int32_t *box_counts, int32_t *crops_out,
                                   int64_t crops_cap, int32_t *n_crops, void *batch, int batch_dtype,
                                   uint8_t *canvas_u8, int32_t *flags, void *stream)
{
    const ms_maps m = ms_dense_maps(score, geo, map_h, map_w, map_h, 8);
    return ms_page_batch_quads_maps(ctx, &m, pages, n_pages, map_h, map_w, img_h, img_w, p, min_text_size, border_mode,
                                    border_value, out_h, out_w, cap_boxes, boxes_out, box_counts, crops_out, crops_cap,
                                    n_crops, batch, batch_dtype, canvas_u8, flags, stream);
}

extern "C" int ms_page_batch_ragged_quads_maps(ms_ctx *ctx, const ms_maps *maps, const uint8_t *const *page_ptrs,
                                               const int32_t *page_hw, int n_pages, int map_h, int map_w,
                                               const ms_east_params *p, int min_text_size, int border_mode,
                                               int border_value, int out_h, int out_w, int cap_boxes, float *boxes_out,
                                               int32_t *box_counts, int32_t *crops_out, int64_t crops_cap,
                                               int32_t *n_crops, void *batch, int batch_dtype, uint8_t *canvas_u8,
                                               int32_t *flags, void *stream)
{
    MS_CTX(ctx);
    MS_TRY(quad_batch_args_ok(batch_dtype, border_mode, border_value, "ms_page_batch_ragged_quads"));
    MS_TRY(maps_desc_ok(maps, "ms_page_batch_ragged_quads"));
    if (n_pages <= 0) return MS_OK;
    if (!maps->score || !maps->geo || !p || !page_ptrs || !page_hw || !boxes_out || !box_counts || !flags ||
        cap_boxes <= 0) {
        ms_set_error("ms_page_batch_ragged_quads: bad arguments");
        return MS_ERR_INVALID;
    }
    // (the page sizes are device data: quads of a page above 32767 pixels on a side get no patch)
    pb_call c;
    pb_init(c, p);
    pb_set_maps(c, maps);
    c.page_ptrs = page_ptrs; c.page_hw = page_hw;
    c.n_pages = n_pages; c.map_h = map_h; c.map_w = map_w;
    c.min_text_size = min_text_size; c.out_h = out_h; c.out_w = out_w; c.cap_boxes = cap_boxes; c.crops_cap = crops_cap;
    c.boxes_out = boxes_out; c.box_counts = box_counts; c.crops_out = crops_out; c.n_crops = n_crops;
    c.batch = batch; c.batch_dtype = batch_dtype; c.canvas_u8 = canvas_u8; c.flags = flags;
    c.crop_quads = 1; c.border_mode = border_mode; c.border_value = border_value;
    return page_batch_cached(ctx, c, (cudaStream_t)stream);
}

extern "C" int ms_page_batch_ragged_quads(ms_ctx *ctx, const float *score, const float *geo,
                                          const uint8_t *const *page_ptrs, const int32_t *page_hw, int n_pages,
                                          int map_h, int map_w, const ms_east_params *p, int min_text_size,
                                          int border_mode, int border_value, int out_h, int out_w, int cap_boxes,
                                          float *boxes_out, int32_t *box_counts, int32_t *crops_out, int64_t crops_cap,
                                          int32_t *n_crops, void *batch, int batch_dtype, uint8_t *canvas_u8,
                                          int32_t *flags, void *stream)
{
    const ms_maps m = ms_dense_maps(score, geo, map_h, map_w, map_h, 8);
    return ms_page_batch_ragged_quads_maps(ctx, &m, page_ptrs, page_hw, n_pages, map_h, map_w, p, min_text_size,
                                           border_mode, border_value, out_h, out_w, cap_boxes, boxes_out, box_counts,
                                           crops_out, crops_cap, n_crops, batch, batch_dtype, canvas_u8, flags, stream);
}

// Read-back of a host page batch queued on the context's own stream, from device call d to the caller's buffers in h.
// *again: a page overflowed the NMS pair capacity, which has grown, and the batch has to run again.  Otherwise the
// boxes come back (per page, the rows up to the largest count) and, when every page is clean, the crop list and batch.
static int pb_host_read_back(ms_ctx *ctx, const pb_call &h, const pb_call &d, void **batch_dev_out, const char *who,
                             bool *again)
{
    cudaStream_t st = ctx->own_stream;
    const int n_pages = d.n_pages;
    MS_CUDA(cudaMemcpyAsync(h.box_counts, d.box_counts, (size_t)n_pages * 4, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaMemcpyAsync(h.flags, d.flags, (size_t)n_pages * 4, cudaMemcpyDeviceToHost, st));
    if (d.n_crops) MS_CUDA(cudaMemcpyAsync(h.n_crops, d.n_crops, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    int32_t all = 0;
    int max_cnt = 0;
    for (int i = 0; i < n_pages; i++) {
        all |= h.flags[i];
        max_cnt = h.box_counts[i] > max_cnt ? h.box_counts[i] : max_cnt;
    }
    *again = grow_edge_factor(ctx, all);
    if (*again) return MS_OK;
    // 36 bytes per box instead of cap_boxes rows per page; a page's copy runs up to the following pages' rows when they
    // are adjacent anyway
    if (max_cnt > d.cap_boxes) max_cnt = d.cap_boxes;
    const size_t pitch = (size_t)d.cap_boxes * 36;
    if (max_cnt > 0)
        MS_CUDA(cudaMemcpy2DAsync(h.boxes_out, pitch, d.boxes_out, pitch, (size_t)max_cnt * 36, (size_t)n_pages,
                                  cudaMemcpyDeviceToHost, st));
    const int rc = flags_to_rc(all, who);
    const int64_t nc = d.n_crops ? (*h.n_crops < d.crops_cap ? *h.n_crops : d.crops_cap) : 0;
    if (rc == MS_OK && nc > 0) {
        MS_CUDA(cudaMemcpyAsync(h.crops_out, d.crops_out, (size_t)nc * 20, cudaMemcpyDeviceToHost, st));
        if (h.batch) {
            const size_t one = (size_t)3 * d.out_h * d.out_w * ms_dtype_bytes(d.batch_dtype);  // bytes of one crop
            MS_CUDA(cudaMemcpyAsync(h.batch, d.batch, (size_t)nc * one, cudaMemcpyDeviceToHost, st));
        }
    }
    MS_CUDA(cudaStreamSynchronize(st));
    if (rc != MS_OK) return rc;
    if (batch_dev_out) *batch_dev_out = d.batch;
    return MS_OK;
}

extern "C" int ms_page_batch_host_ex(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages,
                                     int n_pages, int map_h, int map_w, int img_h, int img_w, const ms_east_params *p,
                                     int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                                     int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                                     void *batch_host, int batch_dtype, void **batch_dev_out, int32_t *flags)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(batch_dtype, "ms_page_batch_host"));
    if (n_pages <= 0) return MS_OK;
    if (!score || !geo || !p || !boxes_out || !box_counts || !flags || cap_boxes <= 0 || map_h <= 0 || map_w <= 0) {
        ms_set_error("ms_page_batch_host: bad arguments");
        return MS_ERR_INVALID;
    }
    pb_call c;  // the caller's buffers
    pb_init(c, p);
    c.pages = pages;
    c.n_pages = n_pages; c.map_h = map_h; c.map_w = map_w; c.img_h = img_h; c.img_w = img_w;
    c.min_text_size = min_text_size; c.out_h = out_h; c.out_w = out_w; c.cap_boxes = cap_boxes; c.crops_cap = crops_cap;
    c.boxes_out = boxes_out; c.box_counts = box_counts; c.crops_out = crops_out; c.n_crops = n_crops;
    c.batch = batch_host; c.batch_dtype = batch_dtype; c.flags = flags;
    const bool want_crops = pages != nullptr && crops_out != nullptr && n_crops != nullptr && crops_cap > 0;
    const bool want_batch = want_crops && (batch_host || batch_dev_out);
    // *batch_dev_out != NULL on entry: a caller-owned device buffer of crops_cap crops that receives the batch
    void *caller_batch = (want_batch && batch_dev_out) ? *batch_dev_out : nullptr;
    const size_t plane = (size_t)map_h * map_w;
    const size_t page_bytes = (size_t)img_h * img_w * 3;
    const size_t one_f = (size_t)3 * out_h * out_w * ms_dtype_bytes(batch_dtype);  // bytes of one crop of the batch
    // The decode reads the geometry only at the candidate cells (a few per cent of the tensor).  When the caller's
    // geometry lives in pinned host memory the kernel gathers it straight from there over PCIe (zero copy) instead
    // of uploading the tensor; pageable buffers are uploaded.
    const float *geo_mapped = nullptr;
    const float *score_dev = nullptr;  // maps that already live on this device (the detector ran here) are used in place
    {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, geo) == cudaSuccess) {
            if (at.type == cudaMemoryTypeDevice && at.device == ctx->device)
                geo_mapped = geo;
            else if (at.type == cudaMemoryTypeHost && at.devicePointer && !getenv("MS_B200_NO_ZEROCOPY"))
                geo_mapped = static_cast<const float *>(at.devicePointer);
        } else
            cudaGetLastError();
        if (cudaPointerGetAttributes(&at, score) == cudaSuccess) {
            if (at.type == cudaMemoryTypeDevice && at.device == ctx->device) score_dev = score;
        } else
            cudaGetLastError();
    }
    // With quantisation q > 1 the decode reads geometry only at rows y % q == q / 2 (utils.py:347-376), so only those
    // rows cross PCIe: one strided 2-D DMA per chunk into a compact (P, 8, H / q, W) tensor.
    const int q = pb_quant(c);
    pb_call d = c;  // the same call on device staging
    d.geo_compact = (!geo_mapped && q > 1 && map_h % q == 0) ? 1 : 0;
    const size_t gplane = d.geo_compact ? (size_t)(map_h / q) * map_w : plane;
    float *d_score, *d_geo;
    uint8_t *d_pages;
    MS_TRY(stage_carve(ctx, "ms_page_batch_host", [&](ms_bump &sb) {
        d_score = score_dev ? const_cast<float *>(score_dev) : sb.take<float>(n_pages * plane);
        d_geo = geo_mapped ? nullptr : sb.take<float>(n_pages * plane * 8);
        d.boxes_out = sb.take<float>((size_t)n_pages * cap_boxes * 9);
        d.box_counts = sb.take<int32_t>(n_pages);
        d.flags = sb.take<int32_t>(n_pages);
        d_pages = want_crops ? sb.take<uint8_t>(n_pages * page_bytes) : nullptr;
        d.crops_out = want_crops ? sb.take<int32_t>((size_t)crops_cap * 5) : nullptr;
        d.n_crops = want_crops ? sb.take<int32_t>(1) : nullptr;
        d.batch = !want_batch ? nullptr : caller_batch ? caller_batch : sb.take<char>((size_t)crops_cap * one_f);
    }));
    d.maps = ms_dense_maps(d_score, geo_mapped ? geo_mapped : d_geo, map_h, map_w, d.geo_compact ? map_h / q : map_h, 8);
    d.pages = d_pages;
    // Pipeline: pages are independent, so the batch is cut into chunks; the copy stream uploads chunk c+1 (maps +
    // page images) while the compute stream runs chunk c.  PCIe is the floor of this entry point: 22 MB per
    // 2048x2048 page against a few tens of microseconds of kernels.
    cudaStream_t st = ctx->own_stream, cs = ctx->copy_stream;
    int chunk = (n_pages + 7) / 8;
    if (chunk < 1) chunk = 1;
    if (chunk > 8) chunk = 8;
    for (bool again = true; again;) {
        if (want_crops) MS_CUDA(cudaMemsetAsync(d.n_crops, 0, sizeof(int32_t), st));
        int k = 0;
        for (int p0 = 0; p0 < n_pages; p0 += chunk, k++) {
            const int np = n_pages - p0 < chunk ? n_pages - p0 : chunk;
            cudaEvent_t ev = ctx->chunk_ev[k & 1];
            // the event of chunk k-2 was consumed by the compute stream before chunk k-1 was queued; reuse is safe
            if (!score_dev)
                MS_CUDA(cudaMemcpyAsync(d_score + (size_t)p0 * plane, score + (size_t)p0 * plane, np * plane * 4,
                                        cudaMemcpyHostToDevice, cs));
            if (geo_mapped) {
                // nothing to upload
            } else if (d.geo_compact)
                MS_CUDA(cudaMemcpy2DAsync(d_geo + (size_t)p0 * gplane * 8, (size_t)map_w * 4,
                                          geo + (size_t)p0 * plane * 8 + (size_t)(q / 2) * map_w, (size_t)q * map_w * 4,
                                          (size_t)map_w * 4, (size_t)np * 8 * (map_h / q), cudaMemcpyHostToDevice, cs));
            else
                MS_CUDA(cudaMemcpyAsync(d_geo + (size_t)p0 * plane * 8, geo + (size_t)p0 * plane * 8, np * plane * 32,
                                        cudaMemcpyHostToDevice, cs));
            if (want_crops)
                MS_CUDA(cudaMemcpyAsync(d_pages + (size_t)p0 * page_bytes, pages + (size_t)p0 * page_bytes,
                                        np * page_bytes, cudaMemcpyHostToDevice, cs));
            MS_CUDA(cudaEventRecord(ev, cs));
            MS_CUDA(cudaStreamWaitEvent(st, ev, 0));
            MS_TRY(page_batch_impl(ctx, d, p0, np, 1, st));
        }
        MS_TRY(pb_host_read_back(ctx, c, d, batch_dev_out, "page_batch", &again));
    }
    return MS_OK;
}

extern "C" int ms_page_batch_host(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *pages, int n_pages,
                                  int map_h, int map_w, int img_h, int img_w, const ms_east_params *p,
                                  int min_text_size, int out_h, int out_w, int cap_boxes, float *boxes_out,
                                  int32_t *box_counts, int32_t *crops_out, int64_t crops_cap, int32_t *n_crops,
                                  float *batch_f32_host, float **batch_dev_out, int32_t *flags)
{
    return ms_page_batch_host_ex(ctx, score, geo, pages, n_pages, map_h, map_w, img_h, img_w, p, min_text_size, out_h,
                                 out_w, cap_boxes, boxes_out, box_counts, crops_out, crops_cap, n_crops, batch_f32_host,
                                 MS_DTYPE_F32, reinterpret_cast<void **>(batch_dev_out), flags);
}

// ---- SURVEY 8f-4: rectified crops of rotated quads (an extension; see quadcrop.cu) ------------------------------------
extern "C" int ms_quad_crop_resize_pad_ex(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                                          const float *quads, int quad_stride, const int32_t *page_of, int64_t n,
                                          int min_text_size, int border_mode, int border_value, int out_h, int out_w,
                                          void *batch, int batch_dtype, uint8_t *canvas_u8, int32_t *sizes_out,
                                          void *stream)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(batch_dtype, "ms_quad_crop_resize_pad"));
    if (n < 0 || (n > 0 && (!pages || !quads))) {
        ms_set_error("ms_quad_crop_resize_pad: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_quad_crop_scratch(n), bump));
    return msk_quad_crop(ctx, pages, n_pages, img_h, img_w, quads, quad_stride, page_of, n, min_text_size, border_mode,
                         border_value, out_h, out_w, batch, batch_dtype, canvas_u8, sizes_out, bump, (cudaStream_t)stream);
}

extern "C" int ms_quad_crop_resize_pad(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w,
                                       const float *quads, int quad_stride, const int32_t *page_of, int64_t n,
                                       int min_text_size, int border_mode, int border_value, int out_h, int out_w,
                                       float *batch_f32, uint8_t *canvas_u8, int32_t *sizes_out, void *stream)
{
    return ms_quad_crop_resize_pad_ex(ctx, pages, n_pages, img_h, img_w, quads, quad_stride, page_of, n, min_text_size,
                                      border_mode, border_value, out_h, out_w, batch_f32, MS_DTYPE_F32, canvas_u8,
                                      sizes_out, stream);
}

extern "C" int ms_quad_crop_last_counts(ms_ctx *ctx, int32_t *counts)
{
    MS_CTX(ctx);
    if (!counts || !ctx->quad_cnt) {
        ms_set_error("ms_quad_crop_last_counts: no rotated-crop call on this context yet");
        return MS_ERR_INVALID;
    }
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    MS_CUDA(cudaMemcpyAsync(h, ctx->quad_cnt, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->quad_stream));
    MS_CUDA(cudaStreamSynchronize(ctx->quad_stream));
    counts[0] = h[0];
    counts[1] = h[2];
    return MS_OK;
}

extern "C" int ms_crop_last_counts(ms_ctx *ctx, int32_t *counts)
{
    MS_CTX(ctx);
    if (!counts || !ctx->crop_cnt) {
        ms_set_error("ms_crop_last_counts: no axis-crop call on this context yet");
        return MS_ERR_INVALID;
    }
    int32_t *h = reinterpret_cast<int32_t *>(ctx->pinned);
    MS_CUDA(cudaMemcpyAsync(h, ctx->crop_cnt, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->crop_stream));
    MS_CUDA(cudaStreamSynchronize(ctx->crop_stream));
    counts[0] = h[1];  // crops listed for the persistent kernel
    counts[1] = h[0];  // crops listed for the generic kernel (including those handed back)
    return MS_OK;
}

extern "C" int ms_quad_crop_resize_pad_host(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const float *quads,
                                            int64_t n, int min_text_size, int border_mode, int border_value, int out_h,
                                            int out_w, float *batch_f32, uint8_t *canvas_u8, int32_t *sizes_out)
{
    MS_CTX(ctx);
    if (n < 0 || img_h <= 0 || img_w <= 0 || out_h <= 0 || out_w <= 0 || (n > 0 && (!page || !quads)) ||
        (!batch_f32 && !canvas_u8) || n >= (int64_t)1 << 30) {
        ms_set_error("ms_quad_crop_resize_pad_host: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    const size_t page_bytes = (size_t)img_h * img_w * 3;
    const size_t one_f = (size_t)3 * out_h * out_w * sizeof(float), one_u = (size_t)3 * out_h * out_w;
    uint8_t *d_page, *d_u;
    float *d_quads, *d_f;
    int32_t *d_sizes;
    MS_TRY(stage_carve(ctx, "ms_quad_crop_resize_pad_host", [&](ms_bump &sb) {
        d_page = sb.take<uint8_t>(page_bytes);
        d_quads = sb.take<float>((size_t)n * 8);
        d_sizes = sb.take<int32_t>((size_t)n * 2);
        d_f = batch_f32 ? sb.take<float>((size_t)n * 3 * out_h * out_w) : nullptr;
        d_u = canvas_u8 ? sb.take<uint8_t>((size_t)n * one_u) : nullptr;
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_page, page, page_bytes, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_quads, quads, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    ms_bump bump;
    MS_TRY(arena_bump(ctx, msk_quad_crop_scratch(n), bump));
    MS_TRY(msk_quad_crop(ctx, d_page, 1, img_h, img_w, d_quads, 8, nullptr, n, min_text_size, border_mode, border_value,
                         out_h, out_w, d_f, MS_DTYPE_F32, d_u, d_sizes, bump, st));
    if (batch_f32) MS_CUDA(cudaMemcpyAsync(batch_f32, d_f, (size_t)n * one_f, cudaMemcpyDeviceToHost, st));
    if (canvas_u8) MS_CUDA(cudaMemcpyAsync(canvas_u8, d_u, (size_t)n * one_u, cudaMemcpyDeviceToHost, st));
    if (sizes_out) MS_CUDA(cudaMemcpyAsync(sizes_out, d_sizes, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

extern "C" int ms_warp_quad_host(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const float *quad,
                                 int border_mode, int border_value, uint8_t *patch_out, int64_t patch_cap, int *w, int *h)
{
    MS_CTX(ctx);
    if (!page || !quad || !w || !h || img_h <= 0 || img_w <= 0 || patch_cap < 0 || (patch_cap > 0 && !patch_out)) {
        ms_set_error("ms_warp_quad_host: bad arguments");
        return MS_ERR_INVALID;
    }
    const size_t page_bytes = (size_t)img_h * img_w * 3;
    uint8_t *d_page, *d_patch;
    float *d_quad;
    MS_TRY(stage_carve(ctx, "ms_warp_quad_host", [&](ms_bump &sb) {
        d_page = sb.take<uint8_t>(page_bytes);
        d_quad = sb.take<float>(8);
        d_patch = sb.take<uint8_t>((size_t)patch_cap + 1);
    }));
    cudaStream_t st = ctx->own_stream;
    MS_CUDA(cudaMemcpyAsync(d_page, page, page_bytes, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaMemcpyAsync(d_quad, quad, 32, cudaMemcpyHostToDevice, st));
    ms_bump bump;
    MS_TRY(arena_bump(ctx, 8192, bump));
    MS_TRY(msk_quad_warp(ctx, d_page, img_h, img_w, d_quad, border_mode, border_value, d_patch, (size_t)patch_cap, w, h,
                         bump, st));
    const size_t bytes = (size_t)(*w) * (*h) * 3;
    if (bytes) MS_CUDA(cudaMemcpyAsync(patch_out, d_patch, bytes, cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    return MS_OK;
}

// ---- page images of their own sizes (a batch of originals, as EAST.predict + Pipeline.predict see them) ------------------
// Host buffers: pages[i] -> (page_hw[2i], page_hw[2i+1], 3) u8.  Maps are uploaded whole, the images one by one into a
// packed staging buffer (256-byte aligned starts); one pass, no chunk pipelining.
extern "C" int ms_page_batch_ragged_host_ex(ms_ctx *ctx, const float *score, const float *geo,
                                            const uint8_t *const *pages, const int32_t *page_hw, int n_pages, int map_h,
                                            int map_w, const ms_east_params *p, int min_text_size, int out_h, int out_w,
                                            int cap_boxes, float *boxes_out, int32_t *box_counts, int32_t *crops_out,
                                            int64_t crops_cap, int32_t *n_crops, void *batch_host, int batch_dtype,
                                            void **batch_dev_out, int32_t *flags)
{
    MS_CTX(ctx);
    MS_TRY(dtype_ok(batch_dtype, "ms_page_batch_ragged_host"));
    if (n_pages <= 0) return MS_OK;
    if (!score || !geo || !p || !pages || !page_hw || !boxes_out || !box_counts || !flags || !crops_out || !n_crops ||
        cap_boxes <= 0 || map_h <= 0 || map_w <= 0 || crops_cap <= 0) {
        ms_set_error("ms_page_batch_ragged_host: bad arguments");
        return MS_ERR_INVALID;
    }
    size_t img_total = 0;
    for (int i = 0; i < n_pages; i++) {
        if (!pages[i] || page_hw[2 * i] <= 0 || page_hw[2 * i + 1] <= 0) {
            ms_set_error("ms_page_batch_ragged_host: page %d is empty", i);
            return MS_ERR_INVALID;
        }
        img_total += al256((size_t)page_hw[2 * i] * page_hw[2 * i + 1] * 3);
    }
    pb_call c;  // the caller's buffers
    pb_init(c, p);
    c.page_ptrs = pages; c.page_hw = page_hw;
    c.n_pages = n_pages; c.map_h = map_h; c.map_w = map_w;
    c.min_text_size = min_text_size; c.out_h = out_h; c.out_w = out_w; c.cap_boxes = cap_boxes; c.crops_cap = crops_cap;
    c.boxes_out = boxes_out; c.box_counts = box_counts; c.crops_out = crops_out; c.n_crops = n_crops;
    c.batch = batch_host; c.batch_dtype = batch_dtype; c.flags = flags;
    const bool want_batch = batch_host || batch_dev_out;
    void *caller_batch = batch_dev_out ? *batch_dev_out : nullptr;  // caller-owned device buffer (see ms_page_batch_host)
    const size_t plane = (size_t)map_h * map_w;
    const size_t one_f = (size_t)3 * out_h * out_w * ms_dtype_bytes(batch_dtype);  // bytes of one crop of the batch
    pb_call d = c;  // the same call on device staging
    float *d_score, *d_geo;
    const uint8_t **d_ptrs;
    int32_t *d_hw;
    uint8_t *d_img;
    MS_TRY(stage_carve(ctx, "ms_page_batch_ragged_host", [&](ms_bump &sb) {
        d_score = sb.take<float>(n_pages * plane);
        d_geo = sb.take<float>(n_pages * plane * 8);
        d.boxes_out = sb.take<float>((size_t)n_pages * cap_boxes * 9);
        d.box_counts = sb.take<int32_t>(n_pages);
        d.flags = sb.take<int32_t>(n_pages);
        d_ptrs = sb.take<const uint8_t *>(n_pages);
        d_hw = sb.take<int32_t>((size_t)n_pages * 2);
        d.crops_out = sb.take<int32_t>((size_t)crops_cap * 5);
        d.n_crops = sb.take<int32_t>(1);
        d.batch = !want_batch ? nullptr : caller_batch ? caller_batch : sb.take<char>((size_t)crops_cap * one_f);
        d_img = sb.take<uint8_t>(img_total);
    }));
    d.maps = ms_dense_maps(d_score, d_geo, map_h, map_w, map_h, 8);
    d.page_ptrs = d_ptrs;
    d.page_hw = d_hw;
    cudaStream_t st = ctx->own_stream;
    std::vector<const uint8_t *> h_ptrs(n_pages);
    for (bool again = true; again;) {
        size_t off = 0;
        for (int i = 0; i < n_pages; i++) {
            const size_t bytes = (size_t)page_hw[2 * i] * page_hw[2 * i + 1] * 3;
            h_ptrs[i] = d_img + off;
            MS_CUDA(cudaMemcpyAsync(d_img + off, pages[i], bytes, cudaMemcpyHostToDevice, st));
            off += al256(bytes);
        }
        MS_CUDA(cudaMemcpyAsync(d_ptrs, h_ptrs.data(), (size_t)n_pages * sizeof(void *), cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemcpyAsync(d_hw, page_hw, (size_t)n_pages * 8, cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemcpyAsync(d_score, score, n_pages * plane * 4, cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaMemcpyAsync(d_geo, geo, n_pages * plane * 32, cudaMemcpyHostToDevice, st));
        MS_CUDA(cudaStreamSynchronize(st));  // h_ptrs is pageable host memory on this frame
        MS_TRY(page_batch_impl(ctx, d, 0, n_pages, 0, st));
        MS_TRY(pb_host_read_back(ctx, c, d, batch_dev_out, "page_batch_ragged", &again));
    }
    return MS_OK;
}

extern "C" int ms_page_batch_ragged_host(ms_ctx *ctx, const float *score, const float *geo, const uint8_t *const *pages,
                                         const int32_t *page_hw, int n_pages, int map_h, int map_w,
                                         const ms_east_params *p, int min_text_size, int out_h, int out_w, int cap_boxes,
                                         float *boxes_out, int32_t *box_counts, int32_t *crops_out, int64_t crops_cap,
                                         int32_t *n_crops, float *batch_f32_host, float **batch_dev_out, int32_t *flags)
{
    return ms_page_batch_ragged_host_ex(ctx, score, geo, pages, page_hw, n_pages, map_h, map_w, p, min_text_size, out_h,
                                        out_w, cap_boxes, boxes_out, box_counts, crops_out, crops_cap, n_crops,
                                        batch_f32_host, MS_DTYPE_F32, reinterpret_cast<void **>(batch_dev_out), flags);
}

// ---- baseline-JPEG decode (jpeg.cu) ---------------------------------------------------------------------------------
extern "C" int ms_jpeg_decode_batch(ms_ctx *ctx, const uint8_t *const *files, const int64_t *sizes, int n,
                                    uint8_t *const *out_pages, int32_t *out_status, void *stream)
{
    MS_CTX(ctx);
    if (n < 0 || (n > 0 && (!files || !sizes || !out_pages || !out_status))) {
        ms_set_error("ms_jpeg_decode_batch: bad arguments");
        return MS_ERR_INVALID;
    }
    if (n == 0) return MS_OK;
    for (int i = 0; i < n; i++)
        if (sizes[i] < 0) {
            ms_set_error("ms_jpeg_decode_batch: negative size of file %d", i);
            return MS_ERR_INVALID;
        }
    return ms_jpeg_decode_batch_impl(ctx, files, sizes, n, out_pages, out_status, (cudaStream_t)stream);
}
