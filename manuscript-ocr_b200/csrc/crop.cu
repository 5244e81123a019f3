// Crop -> resize-and-pad -> normalise -> CHW float32 batch, written directly as the TRBA input.
// Replaces Pipeline._extract_word_image (reference _pipeline.py:204-221), ResizeAndPadA.apply and
// get_val_transform (recognizers/_trba/data/transforms.py:62-120, 185-193) and the per-image
// `.to(device)` + torch.stack of TRBA.predict (recognizers/_trba/__init__.py:264-288, 382-390).
//
// cv2.resize arithmetic restated bit-exactly for uint8 x 3 channels (OpenCV imgproc/resize.cpp,
// validated against cv2 4.13 through the oracle):
//   INTER_LINEAR  (neither side shrinks): 11-bit fixed-point coefficients, vertical pass
//                 ((b0*(r0>>4))>>16 + (b1*(r1>>4))>>16 + 2) >> 2
//   INTER_AREA    (a side shrinks): integer-ratio fast path (2x2: (s+2)>>2, else round(sum*(1/area)))
//                 or the float decimation-table path, accumulated in OpenCV's order
//   same size:    copy
// then paste at (x0=0, y0=(ih-new_h)//2) on a 255 canvas, (v - 127.5) * (1/127.5) in f32, HWC -> CHW.
// The batch is float32, or (an extension) float16 / bfloat16: the same f32 value rounded to nearest-even.
//
// HBM roofline: per crop 3*w*h source bytes read + 3*ih*iw*sizeof(element) bytes written (49 152 B at 32x128 in
// float32, 24 576 B in 16 bits): the kernel is write dominated.
//
// Kernels:
//   crop_plan_kernel        thread per crop: the float64 sizing arithmetic of transforms.py:91-98, interpolation mode,
//                           staging decision -> Plan
//   crop_resize_pad_kernel  the crops with Plan::fast (INTER_AREA with shrink factors below 3 -- what shrinking a
//                           word box to a 32- or 64-pixel-high canvas gives): persistent, warp specialised, 4 CTAs
//                           of 7 warps per SM.  Warp 0 is the staging-ring copy warp of crop_common.cuh (the crop's
//                           source rows by TMA bulk copies); warp 1 (table warp) builds OpenCV's coefficient tables in
//                           shared memory (structure of arrays) and writes the 255-padding as constant 16-byte
//                           streaming stores; warps 2..6 (consumers) resample column strips out of shared memory
//                           (aligned 32-bit loads + funnel shift + PRMT u8->f32, 3 or 4 taps) and store normalised
//                           pixels straight into the CHW batch.
//   crop_generic_kernel     every other crop (copy, INTER_LINEAR upscale, integer-ratio or long-table INTER_AREA,
//                           rows too long for the stage): one CTA per crop from global memory, same arithmetic.
#include "crop_common.cuh"

namespace {

// CTA shape of the persistent kernel: copy warp + table/padding warp + 5 consumer warps, 4 CTAs per SM (224 threads,
// 72 registers).
constexpr int kThreads = 224;
constexpr int kCtasPerSm = 4;
constexpr int kSlots = 3;  // crops in flight per CTA (ring slots: metadata + tables per slot, bytes from the ring)
constexpr int kSrcBuf = 40 * 1024;  // largest staged crop (bytes); the staging ring of a CTA holds at least one
constexpr int kBandsY = 64, kCellsX = 8;  // work-list buckets per page: (row band, x cell)

// Pages are either one (n_pages, img_h, img_w, 3) tensor, or -- page_ptrs != NULL -- separate images of their own
// sizes: page_ptrs[p] -> (page_hw[2p], page_hw[2p+1], 3) bytes.
__device__ __forceinline__ void make_plan(const int32_t *cr, int n_pages, int img_h, int img_w, int ih, int iw,
                                          const uint8_t *pages, const uint8_t *const *page_ptrs,
                                          const int32_t *page_hw, Plan &p)
{
    plan_reset(p);
    p.page = cr[0];
    p.x1 = cr[1];
    p.y1 = cr[2];
    p.w = cr[3] - cr[1];
    p.h = cr[4] - cr[2];
    p.ok = p.page >= 0 && p.page < n_pages;
    if (!p.ok) return;
    const int H = page_ptrs ? page_hw[2 * p.page] : img_h, W = page_ptrs ? page_hw[2 * p.page + 1] : img_w;
    const uint8_t *page0 = page_ptrs ? page_ptrs[p.page] : pages + (size_t)p.page * img_h * (size_t)img_w * 3;
    p.ok = page0 != nullptr && H > 0 && W > 0 && p.w > 0 && p.h > 0 && p.x1 >= 0 && p.y1 >= 0 && cr[3] <= W && cr[4] <= H;
    if (!p.ok) return;
    const int w = p.w, h = p.h;
    plan_resize(w, h, ih, iw, p);
    // staging: every row is copied as the 16-byte-aligned span that covers it; the pitch is exactly that span (the
    // 4-tap reads may run up to 16 bytes past a row -- into the next row, or into the slack kept after the last one).
    // When the page stride is a multiple of 16 every row has the same misalignment, otherwise assume the worst (15).
    const size_t stride = (size_t)W * 3;
    p.stride = (int)stride;
    p.src = page0 + (size_t)p.y1 * stride + (size_t)p.x1 * 3;
    const uintptr_t first = reinterpret_cast<uintptr_t>(p.src);
    const uintptr_t last_end = first + (size_t)(h - 1) * stride + (size_t)w * 3;
    // the copies may not leave the memory that holds the pages: the whole tensor, or this page's own image
    const uintptr_t lo = reinterpret_cast<uintptr_t>(page_ptrs ? page0 : pages);
    const uintptr_t hi = page_ptrs ? lo + (size_t)H * stride : lo + (size_t)n_pages * img_h * (size_t)img_w * 3;
    const int mis = (stride & 15) == 0 ? (int)(first & 15) : 15;
    const int pitch = (mis + w * 3 + 15) & ~15;
    const bool fits = (size_t)pitch * h + 16 <= (size_t)kSrcBuf;
    const bool tail_ok = ((last_end + 15) & ~(uintptr_t)15) <= hi;
    if (fits && tail_ok && (lo & 15) == 0) {
        p.staged = 1;
        p.pitch = pitch;
    }
    p.fast = p.staged && p.w < 65536 && p.h < 65536 && plan_fast_shape(p);
}

// plans for all crops (thread per crop): the float64 sizing arithmetic of transforms.py:91-98 runs here, off the
// critical path of the persistent resampling kernel.  Fast crops are also counted into their work-list bucket
// (page, row band, x cell): the persistent kernel walks the crops in bucket order, so that overlapping word boxes are
// resampled within microseconds of each other and their shared source rows come out of L2 instead of DRAM.
__device__ __forceinline__ int crop_bucket(const Plan &p, const int32_t *page_hw, int img_h, int img_w, int n_pages)
{
    const int H = page_hw ? page_hw[2 * p.page] : img_h, W = page_hw ? page_hw[2 * p.page + 1] : img_w;
    const int by = min(kBandsY - 1, (int)(((int64_t)p.y1 * kBandsY) / max(H, 1)));
    const int bx = min(kCellsX - 1, (int)(((int64_t)p.x1 * kCellsX) / max(W, 1)));
    return (min(p.page, n_pages - 1) * kBandsY + by) * kCellsX + bx;
}

__global__ void __launch_bounds__(256) crop_plan_kernel(const uint8_t *__restrict__ pages,
                                                        const uint8_t *const *__restrict__ page_ptrs,
                                                        const int32_t *__restrict__ page_hw, int n_pages, int img_h,
                                                        int img_w, const int32_t *__restrict__ crops,
                                                        const int32_t *__restrict__ n_crops_dev,
                                                        const int32_t *__restrict__ range, int64_t crops_cap, int ih,
                                                        int iw, Plan *__restrict__ plans, int32_t *__restrict__ hist)
{
    ms_pdl_wait();
    int64_t begin = range ? range[0] : 0;
    int64_t n_crops = range ? range[1] : *n_crops_dev;
    if (n_crops > crops_cap) n_crops = crops_cap;
    for (int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_crops;
         i += (int64_t)gridDim.x * blockDim.x) {
        Plan p;
        make_plan(crops + i * 5, n_pages, img_h, img_w, ih, iw, pages, page_ptrs, page_hw, p);
        plans[i] = p;
        if (p.fast) atomicAdd(&hist[crop_bucket(p, page_ptrs ? page_hw : nullptr, img_h, img_w, n_pages)], 1);
    }
}

// exclusive scan of the bucket counts (one CTA); hist becomes the buckets' write cursors, *n_work the number of fast
// crops.  A thread owns 32 consecutive counts, fetched with eight independent 16-byte loads (the first version walked
// them one dependent load at a time: 57 us for 32 768 buckets); tiles of 32 768 counts are chained by a carry.
__global__ void __launch_bounds__(1024) crop_bucket_scan_kernel(int32_t *__restrict__ hist, int n_buckets,
                                                                int32_t *__restrict__ n_work)
{
    ms_pdl_wait();
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int tile = 0; tile < n_buckets; tile += 32 * 1024) {
        const int lo = tile + (int)threadIdx.x * 32;
        int v[32];
        if (lo + 32 <= n_buckets) {  // n_buckets is a multiple of 4 and hist is 256-byte aligned
            const int4 *q = reinterpret_cast<const int4 *>(hist + lo);
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int4 x = q[i];
                v[4 * i] = x.x, v[4 * i + 1] = x.y, v[4 * i + 2] = x.z, v[4 * i + 3] = x.w;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 32; i++) v[i] = lo + i < n_buckets ? hist[lo + i] : 0;
        }
        int sum = 0;
#pragma unroll
        for (int i = 0; i < 32; i++) {
            const int c = v[i];
            v[i] = sum;
            sum += c;
        }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        const int carry = s_carry;
        if (warp == 0) {
            const int w = s_warp[lane];
            int wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += u;
            }
            s_warp[lane] = wi - w;
            if (lane == 31) s_carry = carry + wi;
        }
        __syncthreads();
        const int base = carry + s_warp[warp] + incl - sum;
        if (lo + 32 <= n_buckets) {
            int4 *q = reinterpret_cast<int4 *>(hist + lo);
#pragma unroll
            for (int i = 0; i < 8; i++) q[i] = make_int4(base + v[4 * i], base + v[4 * i + 1], base + v[4 * i + 2], base + v[4 * i + 3]);
        } else {
#pragma unroll
            for (int i = 0; i < 32; i++)
                if (lo + i < n_buckets) hist[lo + i] = base + v[i];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_work = s_carry;
}

// work[cursor of the crop's bucket ++] = the crop's staging descriptor (order inside a bucket is arbitrary: it only
// shapes the schedule)
__global__ void __launch_bounds__(256) crop_bucket_scatter_kernel(const Plan *__restrict__ plans,
                                                                  const int32_t *__restrict__ page_hw, int n_pages,
                                                                  int img_h, int img_w,
                                                                  const int32_t *__restrict__ n_crops_dev,
                                                                  const int32_t *__restrict__ range, int64_t crops_cap,
                                                                  int32_t *__restrict__ cursors, StageDesc *__restrict__ work)
{
    ms_pdl_wait();
    int64_t begin = range ? range[0] : 0;
    int64_t n_crops = range ? range[1] : *n_crops_dev;
    if (n_crops > crops_cap) n_crops = crops_cap;
    for (int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_crops;
         i += (int64_t)gridDim.x * blockDim.x) {
        const Plan p = plans[i];
        if (p.fast) {
            StageDesc d;
            d.src = p.src;
            d.stride = p.stride;
            d.pitch = p.pitch;
            d.row_bytes = 3 * p.w;
            d.rows = p.h;
            d.ci = (int)i;
            work[atomicAdd(&cursors[crop_bucket(p, page_hw, img_h, img_w, n_pages)], 1)] = d;
        }
    }
}

// Warp-specialised persistent kernel for the crops with Plan::fast, fed by the staging ring of crop_common.cuh.  Warp 0
// is its copy warp; warp 1 (table warp) builds the crop's axis tables, signals, and then writes the crop's padding
// (which nobody waits for); warps 2..6 (consumers) resample the pasted rectangle straight into the CHW batch.
// Each consumer thread resamples a column strip (one destination column, G consecutive destination rows): with a
// shrink factor near 2 neighbouring destination rows share their boundary source row, so a strip needs ~(2G + 1)
// horizontal row sums instead of 3G; per-pixel arithmetic and its order are unchanged.
constexpr int kProducerWarps = 2;
constexpr int kConsumerWarps = kThreads / 32 - kProducerWarps;

template <class T, bool kWriteU8>
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
    crop_resize_pad_kernel(const Plan *__restrict__ plans, const StageDesc *__restrict__ work,
                           const int32_t *__restrict__ n_work_dev, int32_t *__restrict__ ticket, int ring_bytes, int ih,
                           int iw, T *__restrict__ batch, uint8_t *__restrict__ canvas_out, int vec_ok,
                           uint8_t *__restrict__ redo)
{
    ms_pdl_wait();
    extern __shared__ __align__(128) unsigned char smem[];  // [ring_bytes] staging ring, then kSlots table sets
    const int tab_n = area_tab_words(ih, iw);  // words of one slot's table set
    uint32_t *tabs = reinterpret_cast<uint32_t *>(smem + ring_bytes);  // [kSlots][tab_n]
    __shared__ StageSlots<kSlots> s_stage;
    // per slot: what the consumers need of the crop's plan, so that they never touch the plan array in global memory
    __shared__ int s_meta[kSlots][8];  // nw, nh, y0, pitch, misalignment of row 0, its change per row, <= 3 x taps, strip height

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int plane = ih * iw;
    stage_init(s_stage, kConsumerWarps);

    if (warp == 0) {
        stage_copy_warp(s_stage, smem, ring_bytes, work, *n_work_dev, ticket);
        return;
    }
    if (warp == 1) {
        // ---------------- table warp: OpenCV's axis tables, then all of the padding ----------------
        for (int k = 0;; k++) {
            const int s = k % kSlots;
            const int ci = stage_wait_tick(s_stage, k);
            if (ci < 0) break;
            const Plan p = plans[ci];
            const bool two = p.interp == 2;  // exact 2 x 2 ratio: no tables
            const bool x3 = two || __all_sync(0xffffffffu, build_tables(p, tabs + (size_t)s * tab_n, tab_n, iw, lane));
            if (lane == 0) {
                s_meta[s][0] = p.nw;
                s_meta[s][1] = p.nh;
                s_meta[s][2] = p.y0;
                s_meta[s][3] = p.pitch;
                s_meta[s][4] = (int)(reinterpret_cast<uintptr_t>(p.src) & 15);
                s_meta[s][5] = p.stride & 15;  // per-row change of the 16-byte misalignment
                s_meta[s][6] = two ? 2 : (x3 ? 1 : 0);
                s_meta[s][7] = strip_height<kConsumerWarps * 32>(p.nw, p.nh);
            }
            __syncwarp();  // every lane's table stores are ordered before lane 0's releasing arrive
            if (lane == 0) mbar_arrive(&s_stage.full[s]);
            write_padding<T, kWriteU8>(p.nw, p.nh, p.y0, ih, iw, kHasBatch<T> ? batch + (size_t)ci * 3 * plane : nullptr,
                                               kWriteU8 ? canvas_out + (size_t)ci * 3 * plane : nullptr, vec_ok, lane, 32);
        }
        return;
    }

    // ---------------- consumers ----------------
    const int ct = (warp - kProducerWarps) * 32 + lane;
    constexpr int kCT = kConsumerWarps * 32;
    for (int k = 0;; k++) {
        const int s = k % kSlots;
        const int64_t ci = stage_wait_full(s_stage, k);
        if (ci < 0) break;
        const int nw = s_meta[s][0], nh = s_meta[s][1], y0 = s_meta[s][2];
        const uint32_t pitch = (uint32_t)s_meta[s][3], a0 = (uint32_t)s_meta[s][4], sstep = (uint32_t)s_meta[s][5];
        const int G = s_meta[s][7];
        const uint32_t stage_off = (uint32_t)s_stage.off[s];
        T *dstf = kHasBatch<T> ? batch + (size_t)ci * 3 * plane : nullptr;
        uint8_t *dstu = kWriteU8 ? canvas_out + (size_t)ci * 3 * plane : nullptr;
        const uint32_t *tab = tabs + (size_t)s * tab_n;
        // three x taps at most (shrink factor below 2, most word boxes): a quarter of the horizontal work less; a page
        // stride that is a multiple of 16 bytes (sstep == 0): no per-row misalignment arithmetic
        bool bad = false;
        if (s_meta[s][6] == 2)
            area2x2_pixels<T, kWriteU8, kCT>(smem, stage_off, pitch, a0, sstep, ih, iw, nw, nh, y0, dstf, dstu, ct);
        else if (sstep == 0)
            bad = s_meta[s][6] == 1 ? area4_strips<T, kWriteU8, kCT, 3, true>(smem, stage_off, pitch, a0, 0u, tab, tab_n, ih,
                                                                                 iw, nw, nh, y0, dstf, dstu, ct, G)
                               : area4_strips<T, kWriteU8, kCT, 4, true>(smem, stage_off, pitch, a0, 0u, tab, tab_n, ih,
                                                                                 iw, nw, nh, y0, dstf, dstu, ct, G);
        else
            bad = s_meta[s][6] == 1 ? area4_strips<T, kWriteU8, kCT, 3>(smem, stage_off, pitch, a0, sstep, tab, tab_n, ih, iw,
                                                                           nw, nh, y0, dstf, dstu, ct, G)
                               : area4_strips<T, kWriteU8, kCT, 4>(smem, stage_off, pitch, a0, sstep, tab, tab_n, ih, iw,
                                                                           nw, nh, y0, dstf, dstu, ct, G);
        if (bad) redo[ci] = 1;  // a table entry with more than 4 taps: the generic kernel redoes the crop
        stage_release(s_stage, s);
    }
}

// Crops the persistent kernel does not take (same size copy, INTER_LINEAR upscale, integer-ratio INTER_AREA, shrink
// factors >= 3, rows too long for the stage, invalid rectangles, crops flagged `redo`) are listed first ...
__global__ void __launch_bounds__(256) crop_generic_list_kernel(const Plan *__restrict__ plans,
                                                                const int32_t *__restrict__ n_crops_dev,
                                                                const int32_t *__restrict__ range, int64_t crops_cap,
                                                                const uint8_t *__restrict__ redo,
                                                                int32_t *__restrict__ list, int32_t *__restrict__ list_n)
{
    ms_pdl_wait();
    const int64_t begin = range ? range[0] : 0;
    int64_t n_crops = range ? range[1] : *n_crops_dev;
    if (n_crops > crops_cap) n_crops = crops_cap;
    for (int64_t ci = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ci < n_crops;
         ci += (int64_t)gridDim.x * blockDim.x)
        if (!plans[ci].fast || redo[ci]) list[atomicAdd(list_n, 1)] = (int32_t)ci;
}

// ... and resampled one CTA per crop from global memory with the same arithmetic: the CTA builds the crop's
// coefficient tables in shared memory, then one thread per destination pixel.
constexpr int kGenericMaxTab = 1024;  // table entries kept in shared memory (longer axes recompute per pixel)

template <class T, bool kWriteU8>
__global__ void __launch_bounds__(256) crop_generic_kernel(const Plan *__restrict__ plans,
                                                           const int32_t *__restrict__ list,
                                                           const int32_t *__restrict__ list_n, int ih, int iw,
                                                           T *__restrict__ batch,
                                                           uint8_t *__restrict__ canvas_out, int vec_ok)
{
    ms_pdl_wait();
    __shared__ AxisEnt s_tab[kGenericMaxTab];
    const int plane = ih * iw;
    const int todo = *list_n;
    for (int li = blockIdx.x; li < todo; li += gridDim.x) {
        const int64_t ci = list[li];
        Plan p = plans[ci];
        if (!p.ok) p.nw = p.nh = 0;  // an invalid rectangle pastes nothing: the canvas is all padding
        T *dstf = kHasBatch<T> ? batch + (size_t)ci * 3 * plane : nullptr;
        uint8_t *dstu = kWriteU8 ? canvas_out + (size_t)ci * 3 * plane : nullptr;
        write_padding<T, kWriteU8>(p, ih, iw, dstf, dstu, vec_ok, threadIdx.x, blockDim.x);
        const bool need_tab = p.ok && (p.interp == 1 || p.interp == 3);
        const bool tab_ok = need_tab && p.nw + p.nh <= kGenericMaxTab;
        __syncthreads();  // the previous crop's table is no longer read
        if (tab_ok) fill_axis_table(p, s_tab);
        __syncthreads();
        resample_canvas<T, kWriteU8>(p, PitchedSrc{p.src, (size_t)p.stride}, s_tab, tab_ok, need_tab, ih, iw, dstf,
                                             dstu);
    }
}

// ---- test-only (ms_test_resize_tables_host): the plan and table device functions, evaluated as the kernels call them ----
// plans_out[i] (8 words) = nw, nh, y0, interp, isx, isy, plan_fast_shape, 0 of plan_resize(wh[i]) at an out_h x out_w
// canvas.  Axis a = axes[4a..4a+3] = ssize, dsize, mode, first entry; its dsize entries are 8 words each from word
// 8 * first of entries_out, in the layout of the mode:
//   0  build_tables' x tables (INTER_AREA, crop_resize_pad_kernel): the axis as a crop of width ssize, table stride iw =
//      dsize -- word d packed s0 | n << 16, word (1 + k) * dsize + d tap weight k (the rest of the axis' words untouched)
//   1  build_tables' y records: word 8d packed s0 | n << 16, words 8d + 4 .. 8d + 7 the tap weights
//   2  area_entry as fill_axis_table calls it (crop_generic_kernel): the AxisEnt
//   3  linear_entry_x, 4  linear_entry_y: the AxisEnt
static_assert(sizeof(AxisEnt) == 32, "an AxisEnt is one 8-word entry");
__global__ void __launch_bounds__(128) resize_tables_test_kernel(int out_h, int out_w, const int32_t *__restrict__ wh,
                                                                 int64_t n_plans, int32_t *__restrict__ plans_out,
                                                                 const int32_t *__restrict__ axes, int64_t n_axes,
                                                                 int32_t *__restrict__ entries_out)
{
    ms_pdl_wait();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_plans; i += stride) {
        Plan p;
        plan_reset(p);
        plan_resize(wh[2 * i], wh[2 * i + 1], out_h, out_w, p);
        int32_t *o = plans_out + 8 * i;
        o[0] = p.nw, o[1] = p.nh, o[2] = p.y0, o[3] = p.interp, o[4] = p.isx, o[5] = p.isy;
        o[6] = plan_fast_shape(p) ? 1 : 0;
        o[7] = 0;
    }
    for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_axes; a += stride) {
        const int ssize = axes[4 * a], dsize = axes[4 * a + 1], mode = axes[4 * a + 2];
        int32_t *out = entries_out + 8 * (int64_t)axes[4 * a + 3];
        const double scale = 1.0 / ((double)dsize / (double)ssize);  // plan_resize's scale_x / scale_y
        if (mode <= 1) {
            Plan p;
            plan_reset(p);
            p.w = p.h = ssize;
            p.scale_x = p.scale_y = scale;
            (mode == 0 ? p.nw : p.nh) = dsize;
            build_tables(p, reinterpret_cast<uint32_t *>(out), 0, mode == 0 ? dsize : 0, 0, 1);
            continue;
        }
        for (int d = 0; d < dsize; d++) {
            const AxisEnt e = mode == 2 ? area_entry(d, scale, ssize)
                                        : (mode == 3 ? linear_entry_x(d, scale, ssize) : linear_entry_y(d, scale, ssize));
            *reinterpret_cast<AxisEnt *>(out + 8 * d) = e;
        }
    }
}

// ---- detector input (the caller side of the path, EAST.predict infer.py:301-305) ---------------------------------
// cv2.resize(img, (T, T)) -- INTER_LINEAR on uint8 (11-bit fixed-point coefficients, aspect NOT preserved), then
// torchvision ToTensor (x / 255) and Normalize(0.5, 0.5) ((x - 0.5) / 0.5), written as the (P, 3, th, tw) network input
// in float32, or that float32 value rounded to nearest-even in 16 bits.  Same arithmetic as resample_px's linear branch
// (the oracle's orc_resize_linear_u8c3, pinned to cv2 for shrinking and enlarging).  This is what lets a page cross
// PCIe once: the original image is uploaded, the resized detector input is made on the device.
//
// HBM roofline: per page the distinct source rows the y table names (3 * w bytes each) read, 3 * th * tw * element size
// written.  64 scans of ~2500 x 3500 at T = 1280: ~1.5 GB read, 1.26 GB written in float32.
//
// Kernels:
//   detector_input_plan_kernel  thread per axis entry: every page's source, size and OpenCV x / y tables, once per page
//   detector_input_batch_kernel a warp per chunk of an output row: lanes resample consecutive pixels (the source rows
//                               read through L1), then each thread stores 4 (float32) or 8 (16-bit) consecutive pixels
//                               of every plane as one 16-byte vector
struct DetPage {
    const uint8_t *src;
    int h, w;  // 0 x 0: the page is not read and its input is all zeros
    int same;  // the page already has the target size: cv2.resize returns a copy
};

// The page is table entry p, or -- page_ptrs == NULL -- the one page passed by value (ms_detector_input).
__global__ void __launch_bounds__(256) detector_input_plan_kernel(const uint8_t *const *__restrict__ page_ptrs,
                                                                  const int32_t *__restrict__ page_hw,
                                                                  const uint8_t *one, int one_h, int one_w,
                                                                  int n_pages, int th, int tw, DetPage *__restrict__ pages,
                                                                  AxisEnt *__restrict__ tabs)
{
    ms_pdl_wait();
    const int per = tw + th;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)n_pages * per;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int p = (int)(i / per), t = (int)(i - (int64_t)p * per);
        const uint8_t *src = page_ptrs ? page_ptrs[p] : one;
        int H = page_ptrs ? page_hw[2 * p] : one_h, W = page_ptrs ? page_hw[2 * p + 1] : one_w;
        if (!src || H <= 0 || W <= 0) H = W = 0;
        const bool same = H == th && W == tw;
        if (t == 0) pages[p] = DetPage{src, H, W, same ? 1 : 0};
        if (H == 0) continue;
        AxisEnt e = {};
        if (same) {  // the copy reads destination row d from source row d
            if (t >= tw) e.s0 = e.n = t - tw;
        } else if (t < tw)
            e = linear_entry_x(t, 1.0 / ((double)tw / (double)W), W);
        else
            e = linear_entry_y(t - tw, 1.0 / ((double)th / (double)H), H);
        tabs[i] = e;
    }
}

constexpr int kDetThreads = 256;

// A warp makes chunks of 32 * kV consecutive pixels of an output row: lane l resamples pixels l, l + 32, ... (neighbouring
// lanes read neighbouring source bytes, through L1), the values go through the warp's slice of shared memory, and lane l
// stores pixels [l * kV, l * kV + kV) of each plane as one 16-byte vector.
template <class T, bool kWriteU8>
__global__ void __launch_bounds__(kDetThreads) detector_input_batch_kernel(const DetPage *__restrict__ pages,
                                                                           const AxisEnt *__restrict__ tabs, int n_pages,
                                                                           int th, int tw, T *__restrict__ out,
                                                                           uint8_t *__restrict__ out_u8, int vec_ok)
{
    ms_pdl_wait();
    constexpr int kV = kBatchVec<T>, kChunk = 32 * kV, kWarps = kDetThreads / 32;
    constexpr int kElt = kHasBatch<T> ? (int)sizeof(T) : 1;
    __shared__ __align__(16) unsigned char s_tr[kWarps][3][kChunk * kElt];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per = tw + th, chunks = (tw + kChunk - 1) / kChunk;
    const size_t plane = (size_t)th * tw;
    // (page, row, chunk) tasks, fewer than 2^31 (the host checks), dealt out warp by warp over the grid (1-8 % faster
    // on a B200 than a contiguous run of rows per CTA, which keeps more of a page's x table in L1; profiles/README.md)
    const int tasks = n_pages * th * chunks;
    for (int task = blockIdx.x * kWarps + warp; task < tasks; task += gridDim.x * kWarps) {
        const int item = task / chunks;
        const int p = item / th, dy = item - p * th;
        const int x0 = (task - item * chunks) * kChunk;
        const DetPage pg = pages[p];
        const AxisEnt *xt = tabs + (size_t)p * per;
        T *orow = kHasBatch<T> ? out + (size_t)p * 3 * plane + (size_t)dy * tw : nullptr;
        uint8_t *urow = kWriteU8 ? out_u8 + ((size_t)p * plane + (size_t)dy * tw) * 3 : nullptr;
        // the row's two source rows as rows 0 and 1 of one pitched source
        PitchedSrc src{nullptr, 0};
        AxisEnt ey = {};
        if (pg.h > 0) {
            ey = xt[tw + dy];
            const size_t stride = (size_t)pg.w * 3;
            src = PitchedSrc{pg.src + (size_t)ey.s0 * stride, (size_t)(ey.n - ey.s0) * stride};
            ey.s0 = 0;
            ey.n = 1;
        }
        Plan pl;
        pl.interp = pg.same ? 0 : 1;
        pl.isx = pl.isy = 0;
        T *tr = kHasBatch<T> ? reinterpret_cast<T *>(&s_tr[warp][0][0]) : nullptr;
#pragma unroll 1  // rolled: 48 registers, 5 CTAs per SM (unrolled, 60: bfloat16 9 % slower, profiles/README.md)
        for (int k = 0; k < kV; k++) {
            const int dx = x0 + k * 32 + lane;
            unsigned char o0 = 0, o1 = 0, o2 = 0;
            if (dx < tw && pg.h > 0) {
                AxisEnt ex = {};
                if (!pg.same) {
                    const int4 q = __ldg(reinterpret_cast<const int4 *>(xt + dx));  // s0, n, nfirst, nmid
                    ex.s0 = q.x;
                    ex.n = q.y;
                    ex.nfirst = q.z;
                    ex.nmid = q.w;
                }
                resample_px(pl, dx, 0, src, ex, ey, o0, o1, o2);
            }
            if constexpr (kHasBatch<T>) {
                const float f[3] = {pg.h > 0 ? ((float)o0 / 255.0f - 0.5f) / 0.5f : 0.f,
                                    pg.h > 0 ? ((float)o1 / 255.0f - 0.5f) / 0.5f : 0.f,
                                    pg.h > 0 ? ((float)o2 / 255.0f - 0.5f) / 0.5f : 0.f};
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    if (vec_ok)
                        tr[c * kChunk + k * 32 + lane] = to_batch<T>(f[c]);
                    else if (dx < tw)
                        orow[c * plane + dx] = to_batch<T>(f[c]);
                }
            }
            if (kWriteU8 && dx < tw) {
                urow[(size_t)dx * 3] = o0;
                urow[(size_t)dx * 3 + 1] = o1;
                urow[(size_t)dx * 3 + 2] = o2;
            }
        }
        if constexpr (kHasBatch<T>) {
            if (vec_ok) {  // tw % kV == 0 and a 16-byte-aligned output: every lane's kV pixels are whole and aligned
                __syncwarp();
                if (x0 + lane * kV < tw)
#pragma unroll
                    for (int c = 0; c < 3; c++)
                        __stcs(reinterpret_cast<float4 *>(orow + c * plane + x0 + lane * kV),
                               *reinterpret_cast<const float4 *>(&s_tr[warp][c][lane * kV * kElt]));
                __syncwarp();  // the slice is reused by the warp's next chunk
            }
        }
    }
}

}  // namespace

// 0 for sizes msk_detector_input rejects.  The one-page ms_detector_input uses the context's scratch arena as well (the
// first call, or a larger target, grows it: one cudaMalloc after a device synchronisation).
size_t msk_detector_input_scratch(int n_pages, int target_h, int target_w)
{
    if (n_pages <= 0 || target_h <= 0 || target_w <= 0 || (int64_t)target_h + target_w >= ((int64_t)1 << 30)) return 0;
    return (size_t)n_pages * sizeof(DetPage) + (size_t)n_pages * (size_t)(target_h + target_w) * sizeof(AxisEnt) + 1024;
}

int msk_detector_input(ms_ctx *ctx, const uint8_t *const *page_ptrs, const int32_t *page_hw, const uint8_t *one,
                       int one_h, int one_w, int n_pages, int target_h, int target_w, void *out, int out_dtype,
                       uint8_t *out_u8, ms_bump bump, cudaStream_t st)
{
    const bool tables = page_ptrs != nullptr && page_hw != nullptr;
    if (n_pages <= 0 || target_h <= 0 || target_w <= 0 || (!out && !out_u8) ||
        (!tables && (!one || one_h <= 0 || one_w <= 0 || n_pages != 1))) {
        ms_set_error("detector_input: bad arguments");
        return MS_ERR_INVALID;
    }
    // the kernel counts (page, row, column chunk) tasks in 32 bits; its chunks are at least 32 pixels wide, so this
    // bounds the task count
    if ((int64_t)n_pages * target_h * ((target_w + 31) / 32) >= ((int64_t)1 << 31) ||
        (int64_t)target_h + target_w >= ((int64_t)1 << 30)) {
        ms_set_error("detector_input: %d pages of %d x %d are too many pixels for one call", n_pages, target_h, target_w);
        return MS_ERR_INVALID;
    }
    DetPage *pages = bump.take<DetPage>((size_t)n_pages);
    AxisEnt *tabs = bump.take<AxisEnt>((size_t)n_pages * (target_h + target_w));
    if (!pages || !tabs) {
        ms_set_error("detector_input: scratch too small");
        return MS_ERR_CAPACITY;
    }
    const int64_t entries = (int64_t)n_pages * (target_h + target_w);
    int64_t pgrid = (entries + 255) / 256;
    if (pgrid > (int64_t)ctx->num_sms * 8) pgrid = (int64_t)ctx->num_sms * 8;
    ms_launch(detector_input_plan_kernel, (int)pgrid, 256, 0, st, tables ? page_ptrs : nullptr, page_hw, one, one_h,
              one_w, n_pages, target_h, target_w, pages, tabs);
    MS_LAUNCH_CHECK(ctx);
    return launch_for_outputs(out, out_dtype, out_u8, [&](auto bt, auto u8) {
        using T = typename decltype(bt)::type;
        constexpr bool kU8 = decltype(u8)::value;
        // one wave of CTAs (the kernel loops over its tasks)
        int per_sm = 1;
        MS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, detector_input_batch_kernel<T, kU8>, kDetThreads, 0));
        const int64_t wave = (int64_t)ctx->num_sms * (per_sm > 0 ? per_sm : 1);
        const int64_t grid = (int64_t)n_pages * target_h < wave ? (int64_t)n_pages * target_h : wave;
        ms_launch(detector_input_batch_kernel<T, kU8>, (int)grid, kDetThreads, 0, st, pages, tabs, n_pages, target_h,
                  target_w, static_cast<T *>(out), out_u8, batch_vec_ok<T>(out, target_w));
        MS_LAUNCH_CHECK(ctx);
        return MS_OK;
    });
}

// scratch that depends on the page count as well: the work-list buckets
static size_t crop_bucket_count(int n_pages)
{
    size_t b = (size_t)(n_pages > 0 ? n_pages : 1) * kBandsY * kCellsX;
    return b > ((size_t)1 << 22) ? ((size_t)1 << 22) : b;
}

size_t msk_crop_scratch(int64_t crops_cap, int n_pages)
{
    const size_t n = (size_t)(crops_cap > 0 ? crops_cap : 0);
    return n * sizeof(Plan) + n + n * sizeof(int32_t) + n * sizeof(StageDesc) + crop_bucket_count(n_pages) * sizeof(int32_t) + 8192;
}

int msk_crop(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w, const int32_t *crops,
             const int32_t *n_crops, const int32_t *range, int64_t crops_cap, int out_h, int out_w, void *batch,
             int batch_dtype, uint8_t *canvas_u8, ms_bump bump, cudaStream_t st, const uint8_t *const *page_ptrs, const int32_t *page_hw)
{
    if (crops_cap <= 0 || n_pages <= 0) return MS_OK;
    const bool ragged = page_ptrs != nullptr && page_hw != nullptr;
    if (out_h <= 0 || out_w <= 0 || (!ragged && (img_h <= 0 || img_w <= 0 || !pages)) || (!batch && !canvas_u8)) {
        ms_set_error("crop: bad arguments");
        return MS_ERR_INVALID;
    }
    if ((int64_t)out_h * out_w > (1 << 20)) {
        ms_set_error("crop: canvas %dx%d too large", out_h, out_w);
        return MS_ERR_INVALID;
    }
    // shared memory of the persistent kernel: kSlots table sets + the staging ring, which gets what is left of an SM's
    // 227 KB split over the CTAs per SM (1 KB per CTA is reserved by the system, ~0.5 KB is static)
    const size_t tab_bytes = (size_t)kSlots * (size_t)area_tab_words(out_h, out_w) * sizeof(uint32_t);
    const size_t min_ring = (size_t)kSrcBuf + 128;
    int per_sm = kCtasPerSm;
    while (per_sm > 1 && (227 * 1024) / per_sm < (int)(tab_bytes + min_ring + 1024 + 512)) per_sm--;
    if ((227 * 1024) / per_sm < (int)(tab_bytes + min_ring + 1024 + 512)) {
        ms_set_error("crop: canvas %dx%d needs %zu bytes of shared memory", out_h, out_w, tab_bytes + min_ring);
        return MS_ERR_INVALID;
    }
    size_t ring = ((size_t)(227 * 1024) / per_sm - 1024 - 512 - tab_bytes) & ~(size_t)127;
    if (ring > 96 * 1024) ring = 96 * 1024;
    const size_t smem = ring + tab_bytes;
    const int n_buckets = (int)crop_bucket_count(n_pages);
    Plan *plans = bump.take<Plan>((size_t)crops_cap);
    uint8_t *redo = bump.take<uint8_t>((size_t)crops_cap);
    int32_t *glist = bump.take<int32_t>((size_t)crops_cap);
    StageDesc *work = bump.take<StageDesc>((size_t)crops_cap);
    int32_t *hist = bump.take<int32_t>((size_t)n_buckets);
    int32_t *cnt = bump.take<int32_t>(4);  // generic-list length, fast-crop count, ticket counter
    if (!plans || !redo || !cnt) {
        ms_set_error("crop: scratch too small");
        return MS_ERR_CAPACITY;
    }
    int32_t *glist_n = cnt, *n_work = cnt + 1, *ticket = cnt + 2;
    ctx->crop_cnt = cnt;  // ms_crop_last_counts
    ctx->crop_stream = st;
    MS_CUDA(cudaMemsetAsync(redo, 0, (size_t)crops_cap, st));
    MS_CUDA(cudaMemsetAsync(hist, 0, (size_t)n_buckets * sizeof(int32_t), st));
    MS_CUDA(cudaMemsetAsync(cnt, 0, 4 * sizeof(int32_t), st));
    int64_t lgrid = (crops_cap + 255) / 256;
    if (lgrid > (int64_t)ctx->num_sms * 8) lgrid = (int64_t)ctx->num_sms * 8;
    ms_launch(crop_plan_kernel, (int)lgrid, 256, 0, st, pages, ragged ? page_ptrs : nullptr, page_hw, n_pages, img_h, img_w, crops,
                                                 n_crops, range, crops_cap, out_h, out_w, plans, hist);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(crop_bucket_scan_kernel, 1, 1024, 0, st, hist, n_buckets, n_work);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(crop_bucket_scatter_kernel, (int)lgrid, 256, 0, st, plans, ragged ? page_hw : nullptr, n_pages, img_h, img_w, n_crops,
                                                           range, crops_cap, hist, work);
    MS_LAUNCH_CHECK(ctx);
    int64_t grid = (int64_t)ctx->num_sms * per_sm;
    if (grid > crops_cap) grid = crops_cap;
    // one CTA per listed crop, many in flight: a generic crop reads global memory byte by byte and is latency bound
    int64_t ggrid = (int64_t)ctx->num_sms * 8;
    if (ggrid > crops_cap) ggrid = crops_cap;
    return launch_for_outputs(batch, batch_dtype, canvas_u8, [&](auto bt, auto u8) {
        using T = typename decltype(bt)::type;
        constexpr bool kU8 = decltype(u8)::value;
        T *out = static_cast<T *>(batch);
        const int vec_ok = batch_vec_ok<T>(batch, out_w);
        MS_TRY(ms_allow_smem(ctx, batch_slot<T, kU8>(MS_SMEM_CROP_U8), crop_resize_pad_kernel<T, kU8>, (int)smem));
        ms_launch(crop_resize_pad_kernel<T, kU8>, (int)grid, kThreads, smem, st, plans, work, n_work, ticket, (int)ring,
                  out_h, out_w, out, canvas_u8, vec_ok, redo);
        MS_LAUNCH_CHECK(ctx);
        ms_launch(crop_generic_list_kernel, (int)lgrid, 256, 0, st, plans, n_crops, range, crops_cap, redo, glist, glist_n);
        MS_LAUNCH_CHECK(ctx);
        ms_launch(crop_generic_kernel<T, kU8>, (int)ggrid, 256, 0, st, plans, glist, glist_n, out_h, out_w, out,
                  canvas_u8, vec_ok);
        MS_LAUNCH_CHECK(ctx);
        return MS_OK;
    });
}

int msk_test_resize_tables(ms_ctx *ctx, int out_h, int out_w, const int32_t *wh, int64_t n_plans, int32_t *plans_out,
                           const int32_t *axes, int64_t n_axes, int32_t *entries_out, cudaStream_t st)
{
    const int64_t n = n_plans > n_axes ? n_plans : n_axes;
    if (n <= 0) return MS_OK;
    int64_t grid = (n + 127) / 128;
    if (grid > (int64_t)ctx->num_sms * 16) grid = (int64_t)ctx->num_sms * 16;
    ms_launch(resize_tables_test_kernel, (int)grid, 128, 0, st, out_h, out_w, wh, n_plans, plans_out, axes, n_axes,
              entries_out);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}
