// Shared by crop.cu and quadcrop.cu: the staging ring that feeds their warp-specialised kernels, the resize-and-pad plan
// of one crop, OpenCV's coefficient-table entries and the per-pixel resampling arithmetic (cv2.resize restated, see
// crop.cu), and the 255-padding writer.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "ms_internal.cuh"

namespace {

// ---- batch element types -----------------------------------------------------------------------------------------
// The crop kernels are instantiated for the element type of the network-input batch they write: float, __half,
// __nv_bfloat16, or NoBatch (only the u8 canvas is written).  Every value is normalised in float32 and then converted
// with round-to-nearest-even, so a 16-bit batch is bit for bit the float32 batch cast with torch's .to(dtype).
struct NoBatch {};
template <class T>
constexpr bool kHasBatch = !std::is_same<T, NoBatch>::value;

template <class T>
__device__ __forceinline__ T to_batch(float v);
template <>
__device__ __forceinline__ float to_batch<float>(float v) { return v; }
template <>
__device__ __forceinline__ __half to_batch<__half>(float v) { return __float2half_rn(v); }
template <>
__device__ __forceinline__ __nv_bfloat16 to_batch<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ uint32_t batch_bits(__half v) { return __half_as_ushort(v); }
__device__ __forceinline__ uint32_t batch_bits(__nv_bfloat16 v) { return __bfloat16_as_ushort(v); }

// one normalised batch value ((v - 127.5) / 127.5 as the reference's f32 expression), streaming store
template <class T>
__device__ __forceinline__ void store_norm(T *p, float v)
{
    __stcs(p, to_batch<T>((v - 127.5f) * (1.0f / 127.5f)));
}

// ---- mbarrier + TMA bulk copy (sm_90+ PTX; SASS: SYNCS / UBLKCP) ----------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    // A failed try sleeps (100 ns) before the next one: a waiting warp that retries every few tens of cycles takes issue
    // slots from the warps that do the arithmetic (r2c capture: a quarter of all executed instructions were retries).
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "WAIT_%=:\n"
        "nanosleep.u32 %2;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity), "r"(100u)
        : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- staging ring: the producer of crop_resize_pad_kernel (crop.cu) and quad_crop_staged_kernel (quadcrop.cu) -------
// Both kernels are persistent and warp specialised, with no CTA-wide barrier in their loop.  Warp 0 (copy warp,
// stage_copy_warp) takes the next work item from a global ticket counter (a CTA that drew narrow words simply draws more
// of them), reserves the item's rows in the CTA's staging RING, tells warp 1 (table warp) which item the slot holds and
// issues one TMA bulk copy per row.  The table warp builds the item's tables and metadata and arrives on `full`; the
// consumer warps wait on `full`, work out of shared memory and release the slot on `empty`.  Up to kSlots items are in
// flight per CTA; a slot owns its metadata and tables, its rows take exactly the bytes they need from the ring (a narrow
// word does not hold a 24 KB stage), so the producers can be several items ahead of the consumers and the differences
// between items average out.  History (profiles/README.md): with two fixed 24 KB stages the consumers waited on `full`
// 24 % of their time and the copy warp on `empty` 33 % of its -- producer and consumer periods are equal on average, so
// a two-deep pipeline stalls on every fluctuation.

// What the copy warp needs of one work item (32 bytes: two 16-byte loads).  Row r is copied as the 16-byte-aligned span
// that covers [src + r * stride, + row_bytes), to byte r * pitch of the item's ring space.
struct __align__(16) StageDesc {
    const uint8_t *src;  // first byte of row 0
    int stride;          // bytes between source rows
    int pitch;           // bytes between staged rows (at least the widest span)
    int row_bytes;       // bytes of one source row
    int rows;
    int ci;              // item index (output slot)
};
static_assert(sizeof(StageDesc) == 32, "the copy warp loads a descriptor as two uint4");

// Per slot: `tick` completes when the copy warp has filled the slot, `full` when its bytes have landed and the table
// warp has arrived, `empty` when every consumer warp has released it (and with it its ring bytes).
template <int kSlots>
struct StageSlots {
    uint64_t full[kSlots], empty[kSlots], tick[kSlots];
    int ci[kSlots];     // item of the slot, -1: no more work (copy warp -> table warp and consumers)
    int off[kSlots];    // ring offset of the item's row 0
    int pitch[kSlots];  // bytes between its staged rows
};

// sequence number k -> slot k % kSlots, which it uses for the (k / kSlots)-th time: the parity of that phase
template <int kSlots>
__device__ __forceinline__ uint32_t stage_parity(int k)
{
    return (uint32_t)((k / kSlots) & 1);
}

// called by every thread of the CTA (it ends in __syncthreads)
template <int kSlots>
__device__ __forceinline__ void stage_init(StageSlots<kSlots> &ss, int consumer_warps)
{
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < kSlots; i++) {
            mbar_init(&ss.full[i], 2);  // the copy warp (with the byte count) and the table warp
            mbar_init(&ss.empty[i], consumer_warps);
            mbar_init(&ss.tick[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
}

// The copy warp: fills slots until the work list is exhausted, then posts the end-of-work sentinel (ci = -1).
// Software pipeline: while item k is being copied, the descriptor of item k+1 and the ticket of item k+2 are in flight,
// so neither the atomic nor the descriptor load is on the warp's critical path.  Ring space is allocated first fit at
// the end of the newest item, else at 0, else after the oldest item in flight has been released.
template <int kSlots>
__device__ __forceinline__ void stage_copy_warp(StageSlots<kSlots> &ss, unsigned char *ring, int ring_bytes,
                                                const StageDesc *__restrict__ work, int n_work, int32_t *ticket)
{
    const int lane = threadIdx.x & 31;
    int q_off[kSlots], q_len[kSlots];  // ring intervals of the slots (len 0: free)
#pragma unroll
    for (int i = 0; i < kSlots; i++) q_off[i] = q_len[i] = 0;
    int head = 0;    // where the newest item ended
    int oldest = 0;  // first item (sequence number) whose slot has not been seen released
    auto release_oldest = [&]() {
        mbar_wait(&ss.empty[oldest % kSlots], stage_parity<kSlots>(oldest));
        q_len[oldest % kSlots] = 0;
        oldest++;
    };
    auto load_desc = [&](int t) {
        StageDesc d;
        if (t < n_work) {
            const uint4 *q = reinterpret_cast<const uint4 *>(work + t);
            const uint4 a = q[0], b = q[1];
            d.src = reinterpret_cast<const uint8_t *>(((uint64_t)a.y << 32) | a.x);
            d.stride = (int)a.z;
            d.pitch = (int)a.w;
            d.row_bytes = (int)b.x;
            d.rows = (int)b.y;
            d.ci = (int)b.z;
        } else {
            d.src = nullptr;
            d.stride = d.pitch = d.row_bytes = d.rows = 0;
            d.ci = -1;
        }
        return d;
    };
    int t1 = 0;
    if (lane == 0) t1 = atomicAdd(ticket, 1);
    StageDesc cur = load_desc(__shfl_sync(0xffffffffu, t1, 0));
    if (lane == 0) t1 = atomicAdd(ticket, 1);  // ticket of item 1
    for (int k = 0;; k++) {
        const int s = k % kSlots;
        const StageDesc nxt = load_desc(__shfl_sync(0xffffffffu, t1, 0));  // item k+1: lands during this item's copies
        if (lane == 0 && cur.ci >= 0) t1 = atomicAdd(ticket, 1);            // ticket of item k+2
        // the slot's previous item (k - kSlots) must be done before its metadata / tables are reused
        while (oldest + kSlots <= k) release_oldest();
        if (cur.ci < 0) {  // no more work: tell the table warp, which tells the consumers
            if (lane == 0) {
                ss.ci[s] = -1;
                mbar_arrive(&ss.tick[s]);
                mbar_arrive(&ss.full[s]);
            }
            return;
        }
        // 16 bytes of slack after the last row: the consumers' aligned 32-bit reads may run past a row's end
        const int need = (cur.pitch * cur.rows + 16 + 127) & ~127;
        int off;
        for (;;) {
            auto free_at = [&](int c) {
                bool ok = c + need <= ring_bytes;
#pragma unroll
                for (int i = 0; i < kSlots; i++) ok = ok && (q_len[i] == 0 || c + need <= q_off[i] || q_off[i] + q_len[i] <= c);
                return ok;
            };
            if (free_at(head)) {
                off = head;
                break;
            }
            if (free_at(0)) {
                off = 0;
                break;
            }
            // oldest < k here: with nothing in flight the whole ring is free and `need` fits by construction
            release_oldest();
        }
        q_off[s] = off;
        q_len[s] = need;
        head = off + need;
        if (lane == 0) {
            ss.ci[s] = cur.ci;
            ss.off[s] = off;
            ss.pitch[s] = cur.pitch;
            mbar_arrive(&ss.tick[s]);  // release: the table warp and (through full) the consumers see all three
        }
        uint32_t bytes = 0;
        {
            const size_t stride = (size_t)cur.stride;
            unsigned char *buf = ring + off;
            for (int r = lane; r < cur.rows; r += 32) {
                const uint8_t *g = cur.src + (size_t)r * stride;
                const uint32_t a = (uint32_t)(reinterpret_cast<uintptr_t>(g) & 15);
                const uint32_t sz = (a + (uint32_t)cur.row_bytes + 15) & ~15u;
                tma_bulk_g2s(buf + (size_t)r * cur.pitch, g - a, sz, &ss.full[s]);
                bytes += sz;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) bytes += __shfl_xor_sync(0xffffffffu, bytes, o);
        }
        if (lane == 0) mbar_expect_tx(&ss.full[s], bytes);
        cur = nxt;
    }
}

// The table warp: waits until the copy warp has filled slot k % kSlots and returns its item -- or -1, after passing the
// end-of-work sentinel on to the consumers.  For an item, the table warp arrives on `full` itself when its part is done.
template <int kSlots>
__device__ __forceinline__ int stage_wait_tick(StageSlots<kSlots> &ss, int k)
{
    const int s = k % kSlots;
    mbar_wait(&ss.tick[s], stage_parity<kSlots>(k));
    const int ci = ss.ci[s];
    if (ci < 0 && (threadIdx.x & 31) == 0) mbar_arrive(&ss.full[s]);
    return ci;
}

// A consumer warp: waits until slot k % kSlots is full and returns its item (-1: no more work) ...
template <int kSlots>
__device__ __forceinline__ int stage_wait_full(StageSlots<kSlots> &ss, int k)
{
    mbar_wait(&ss.full[k % kSlots], stage_parity<kSlots>(k));
    return ss.ci[k % kSlots];
}

// ... and hands slot s back when it is done with it
template <int kSlots>
__device__ __forceinline__ void stage_release(StageSlots<kSlots> &ss, int s)
{
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&ss.empty[s]);
}

struct Plan {
    int page, x1, y1, w, h;
    int nw, nh, y0;
    int interp;  // 0 copy, 1 linear, 2 area integer-ratio, 3 area general
    int isx, isy;
    int ok;
    int staged;  // source rows can be staged through TMA into shared memory
    int fast;    // handled by the persistent TMA kernel (INTER_AREA, shrink factors < 3, staged); else generic kernel
    int pitch;   // shared-memory row pitch (bytes) when staged
    int stride;  // bytes between source rows (3 * width of the crop's page)
    const uint8_t *src;  // first source byte of the crop (row y1, column x1 of its page)
    double scale_x, scale_y;
};

// the plan of no crop: not ok, nothing pasted (all padding)
__device__ __forceinline__ void plan_reset(Plan &p)
{
    p.page = p.x1 = p.y1 = p.w = p.h = 0;
    p.nw = p.nh = p.y0 = p.interp = p.isx = p.isy = 0;
    p.ok = p.staged = p.fast = p.pitch = p.stride = 0;
    p.src = nullptr;
    p.scale_x = p.scale_y = 1.0;
}

// one destination index of one axis: the OpenCV coefficient table entry
struct AxisEnt {
    int s0;      // area: first source index; linear: left/top source index
    int n;       // area: number of taps;     linear x: edge flag;  linear y: bottom source index
    int nfirst;  // area: 1 if a partial first tap exists; linear: coefficient 0 (a0 / b0)
    int nmid;    // area: number of full-weight taps;      linear: coefficient 1 (a1 / b1)
    float af, am, al;
    int pad;
};

__device__ __forceinline__ int cv_round(float v) { return __float2int_rn(v); }
__device__ __forceinline__ unsigned char sat_u8(int v) { return (unsigned char)min(max(v, 0), 255); }

// transforms.py:80-98 for a (w, h) source: destination size, interpolation mode and cv2.resize's scale factors
__device__ __forceinline__ void plan_resize(int w, int h, int ih, int iw, Plan &p)
{
    // transforms.py:91-95
    double s1 = (double)ih / (double)max(h, 1), s2 = (double)iw / (double)max(w, 1);
    double sc = fmin(s1, s2);
    p.nw = max(1, (int)rint(w * sc));  // python round(): half to even
    p.nh = max(1, (int)rint(h * sc));
    p.nw = min(p.nw, iw);
    p.nh = min(p.nh, ih);
    int shrink = (p.nh < h || p.nw < w);  // transforms.py:80-83
    p.y0 = (ih - p.nh) / 2;
    p.y0 = max(0, min(p.y0, ih - p.nh));
    p.scale_x = 1.0 / ((double)p.nw / (double)w);
    p.scale_y = 1.0 / ((double)p.nh / (double)h);
    p.isx = (int)rint(p.scale_x);
    p.isy = (int)rint(p.scale_y);
    if (p.nw == w && p.nh == h)
        p.interp = 0;
    else if (!shrink)
        p.interp = 1;
    else {
        bool fast = fabs(p.scale_x - p.isx) < 2.220446049250313e-16 && fabs(p.scale_y - p.isy) < 2.220446049250313e-16;
        p.interp = fast ? 2 : 3;
    }
}

// The part of Plan::fast that depends on the resize plan alone: INTER_AREA general with shrink factors below 3 (a
// decimation window shorter than 3 source pixels touches at most 4 of them: every table entry has <= 4 taps), or the
// exact 2 x 2 integer ratio, which has its own staged routine.
__device__ __forceinline__ bool plan_fast_shape(const Plan &p)
{
    return (p.interp == 3 && p.scale_x < 2.999 && p.scale_y < 2.999) || (p.interp == 2 && p.isx == 2 && p.isy == 2);
}

// (float)(num / den) for 0 <= num <= den, given inv = 1.0 / den (correctly rounded): num * inv is within two double
// ulps of the quotient, so it rounds to the same float unless it sits that close to the midpoint between two floats
// (the 29 bits below float precision near 100...0) -- then, and for tiny values, the division itself is evaluated.
__device__ __noinline__ float div_to_float_slow(double num, double den) { return (float)(num / den); }
__device__ __forceinline__ float div_to_float(double num, double den, double inv)
{
    const double q = num * inv;
    const unsigned lo = (unsigned)__double2loint(q) & 0x1fffffffu;
    if (num == 0.0) return 0.f;  // exact, and common (a window that starts or ends on a pixel boundary)
    if (lo - 0x0ffffff0u <= 0x20u || !(q > 1e-30)) return div_to_float_slow(num, den);
    return (float)q;
}

// OpenCV computeResizeAreaTab for destination index d.  inv_scale = 1.0 / scale, computed once per axis: every entry
// but a clipped last one divides by `scale`, and the three quotients of an entry come out of one reciprocal.
__device__ __forceinline__ AxisEnt area_entry(int d, double scale, int ssize, double inv_scale)
{
    AxisEnt t;
    double f1 = d * scale, f2 = f1 + scale;
    double cell = fmin(scale, (double)ssize - f1);
    int s1 = (int)ceil(f1), s2 = (int)floor(f2);
    s2 = min(s2, ssize - 1);
    s1 = min(s1, s2);
    const bool has_first = (s1 - f1) > 1e-3;
    const bool has_last = (f2 - s2) > 1e-3;
    const double n_first = s1 - f1, n_last = fmin(fmin(f2 - s2, 1.0), cell);
    if (cell == scale && n_first >= 0.0 && n_last >= 0.0) {
        t.af = div_to_float(n_first, cell, inv_scale);
        t.am = (float)inv_scale;
        t.al = div_to_float(n_last, cell, inv_scale);
    } else {  // the clipped last entry of an axis
        t.af = div_to_float_slow(n_first, cell);
        t.am = div_to_float_slow(1.0, cell);
        t.al = div_to_float_slow(n_last, cell);
    }
    t.nfirst = has_first ? 1 : 0;
    t.nmid = s2 > s1 ? s2 - s1 : 0;
    t.s0 = has_first ? s1 - 1 : s1;
    t.n = t.nfirst + t.nmid + (has_last ? 1 : 0);
    t.pad = 0;
    return t;
}
__device__ __forceinline__ AxisEnt area_entry(int d, double scale, int ssize) { return area_entry(d, scale, ssize, 1.0 / scale); }

__device__ __forceinline__ float area_weight(const AxisEnt &t, int e)
{
    return e < t.nfirst ? t.af : (e < t.nfirst + t.nmid ? t.am : t.al);
}

__device__ __forceinline__ AxisEnt linear_entry_x(int dx, double scale, int w)
{
    AxisEnt t;
    float fx = (float)((dx + 0.5) * scale - 0.5);
    int sx = (int)floorf(fx);
    fx -= sx;
    if (sx < 0) {
        fx = 0;
        sx = 0;
    }
    const bool edge = sx + 1 >= w;
    if (edge) {
        fx = 0;
        sx = w - 1;
    }
    t.s0 = sx;
    t.n = edge ? 1 : 0;
    t.nfirst = (short)cv_round((1.f - fx) * 2048.f);
    t.nmid = (short)cv_round(fx * 2048.f);
    t.af = t.am = t.al = 0.f;
    t.pad = 0;
    return t;
}

__device__ __forceinline__ AxisEnt linear_entry_y(int dy, double scale, int h)
{
    AxisEnt t;
    float fy = (float)((dy + 0.5) * scale - 0.5);
    int sy = (int)floorf(fy);
    fy -= sy;
    t.s0 = min(max(sy, 0), h - 1);
    t.n = min(max(sy + 1, 0), h - 1);
    t.nfirst = (short)cv_round((1.f - fy) * 2048.f);
    t.nmid = (short)cv_round(fy * 2048.f);
    t.af = t.am = t.al = 0.f;
    t.pad = 0;
    return t;
}

// Any interpolation mode, any tap count, source read from global memory; ex / ey are the pixel's coefficient-table
// entries (INTER_LINEAR or INTER_AREA general).  Used by crop_generic_kernel for every crop the persistent TMA kernel
// does not take.
// `Src::at(sy, b)` = byte b (3 * column + channel) of source row sy.
struct PitchedSrc {  // rows `stride` bytes apart in global or shared memory
    const uint8_t *base;
    size_t stride;
    __device__ __forceinline__ int at(int sy, int b) const { return base[(size_t)sy * stride + b]; }
};

template <class Src>
__device__ __forceinline__ void resample_px(const Plan &p, int dx, int dy, const Src &src, const AxisEnt &ex,
                                            const AxisEnt &ey, unsigned char &o0, unsigned char &o1, unsigned char &o2)
{
    if (p.interp == 0) {
        o0 = (unsigned char)src.at(dy, dx * 3);
        o1 = (unsigned char)src.at(dy, dx * 3 + 1);
        o2 = (unsigned char)src.at(dy, dx * 3 + 2);
    } else if (p.interp == 1) {
        const int xb = ex.s0 * 3;
        const int a0 = ex.nfirst, a1 = ex.nmid, b0 = ey.nfirst, b1 = ey.nmid;
        unsigned char o[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            int r0, r1;
            if (ex.n) {
                r0 = src.at(ey.s0, xb + c) * 2048;
                r1 = src.at(ey.n, xb + c) * 2048;
            } else {
                r0 = src.at(ey.s0, xb + c) * a0 + src.at(ey.s0, xb + c + 3) * a1;
                r1 = src.at(ey.n, xb + c) * a0 + src.at(ey.n, xb + c + 3) * a1;
            }
            o[c] = (unsigned char)((((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2);
        }
        o0 = o[0];
        o1 = o[1];
        o2 = o[2];
    } else if (p.interp == 2) {
        int s0 = 0, s1 = 0, s2 = 0;
        for (int yy = 0; yy < p.isy; yy++) {
            const int sy = dy * p.isy + yy, xb = dx * p.isx * 3;
            for (int xx = 0; xx < p.isx; xx++) {
                s0 += src.at(sy, xb + xx * 3);
                s1 += src.at(sy, xb + xx * 3 + 1);
                s2 += src.at(sy, xb + xx * 3 + 2);
            }
        }
        if (p.isx == 2 && p.isy == 2) {
            o0 = (unsigned char)((s0 + 2) >> 2);
            o1 = (unsigned char)((s1 + 2) >> 2);
            o2 = (unsigned char)((s2 + 2) >> 2);
        } else {
            const float inv = 1.f / (float)(p.isx * p.isy);
            o0 = sat_u8(cv_round((float)s0 * inv));
            o1 = sat_u8(cv_round((float)s1 * inv));
            o2 = sat_u8(cv_round((float)s2 * inv));
        }
    } else {
        float sum0 = 0.f, sum1 = 0.f, sum2 = 0.f;
        for (int j = 0; j < ey.n; j++) {
            const float beta = area_weight(ey, j);
            const int sy = ey.s0 + j, xb = ex.s0 * 3;
            float b0 = 0.f, b1 = 0.f, b2 = 0.f;
            for (int e = 0; e < ex.n; e++) {
                const float a = area_weight(ex, e);
                b0 = b0 + (float)src.at(sy, xb + e * 3) * a;
                b1 = b1 + (float)src.at(sy, xb + e * 3 + 1) * a;
                b2 = b2 + (float)src.at(sy, xb + e * 3 + 2) * a;
            }
            if (j == 0) {
                sum0 = beta * b0;
                sum1 = beta * b1;
                sum2 = beta * b2;
            } else {
                sum0 += beta * b0;
                sum1 += beta * b1;
                sum2 += beta * b2;
            }
        }
        o0 = sat_u8(cv_round(sum0));
        o1 = sat_u8(cv_round(sum1));
        o2 = sat_u8(cv_round(sum2));
    }
}

// The generic per-pixel path, one CTA per crop.  First the crop's coefficient-table entries in shared memory: tab[t] for
// destination column t < nw, tab[nw + d] for destination row d (INTER_LINEAR or INTER_AREA general) ...
__device__ __forceinline__ void fill_axis_table(const Plan &p, AxisEnt *tab)
{
    for (int t = threadIdx.x; t < p.nw + p.nh; t += blockDim.x) {
        const bool isx = t < p.nw;
        const int d = isx ? t : t - p.nw;
        tab[t] = p.interp == 3 ? (isx ? area_entry(d, p.scale_x, p.w) : area_entry(d, p.scale_y, p.h))
                               : (isx ? linear_entry_x(d, p.scale_x, p.w) : linear_entry_y(d, p.scale_y, p.h));
    }
}

// ... then a thread per pasted pixel, batch (element type T) and / or u8 stores.  tab_ok: the entries are in s_tab;
// otherwise, when the mode needs entries (need_tab), every pixel computes its own.
template <class T, bool kWriteU8, class Src>
__device__ __forceinline__ void resample_canvas(const Plan &p, const Src &src, const AxisEnt *s_tab, bool tab_ok,
                                                bool need_tab, int ih, int iw, T *dstf, uint8_t *dstu)
{
    const int plane = ih * iw;
    const float inv = 1.0f / 127.5f;
    const int nw = p.nw, nh = p.nh, npx = nw * nh;
    for (int t = threadIdx.x; t < npx; t += blockDim.x) {
        const int dy = t / nw, dx = t - dy * nw;
        AxisEnt ex = {}, ey = {};
        if (tab_ok) {
            ex = s_tab[dx];
            ey = s_tab[nw + dy];
        } else if (need_tab) {
            ex = p.interp == 3 ? area_entry(dx, p.scale_x, p.w) : linear_entry_x(dx, p.scale_x, p.w);
            ey = p.interp == 3 ? area_entry(dy, p.scale_y, p.h) : linear_entry_y(dy, p.scale_y, p.h);
        }
        unsigned char o0, o1, o2;
        resample_px(p, dx, dy, src, ex, ey, o0, o1, o2);
        const int at = (p.y0 + dy) * iw + dx;
        if constexpr (kHasBatch<T>) {
            dstf[at] = to_batch<T>(((float)o0 - 127.5f) * inv);
            dstf[plane + at] = to_batch<T>(((float)o1 - 127.5f) * inv);
            dstf[2 * plane + at] = to_batch<T>(((float)o2 - 127.5f) * inv);
        }
        if (kWriteU8) {
            dstu[(size_t)at * 3] = o0;
            dstu[(size_t)at * 3 + 1] = o1;
            dstu[(size_t)at * 3 + 2] = o2;
        }
    }
}

// Batch elements per 16-byte vector store: 4 float, 8 __half / __nv_bfloat16.  The padding writer's vector path needs
// out_w to be a multiple of it and a 16-byte-aligned batch (the host's vec_ok).
template <class T>
constexpr int kBatchVec = sizeof(T) == 2 ? 8 : 4;

// Everything outside the pasted rectangle is the 255 canvas (transforms.py:100), 1.0f after normalisation; written
// as constant 16-byte streaming stores by `nthreads` cooperating threads.
template <class T, bool kWriteU8>
__device__ __forceinline__ void write_padding(int nw, int nh, int y0, int ih, int iw, T *dstf, uint8_t *dstu,
                                              int vec_ok, int tid, int nthreads)
{
    const int plane = ih * iw;
    if constexpr (kHasBatch<T>) {
        constexpr int kV = kBatchVec<T>;
        const T one = to_batch<T>((255.0f - 127.5f) * (1.0f / 127.5f));
        if (vec_ok) {
            // kV copies of `one` in 16 bytes
            float4 one4;
            if constexpr (sizeof(T) == 4) {
                one4 = make_float4(one, one, one, one);
            } else {
                const uint32_t b = batch_bits(one);
                const float v2 = __uint_as_float(b | (b << 16));
                one4 = make_float4(v2, v2, v2, v2);
            }
            const int nw4 = (nw + kV - 1) & ~(kV - 1);
            const int top4 = y0 * iw / kV, bot4 = (ih - y0 - nh) * iw / kV, tail4 = (iw - nw4) / kV;
            const int fr = nw4 - nw;  // scalar fringe [nw, nw4)
            // the pasted rectangle sits at the same place in every channel: one index computation, a store per channel
            float4 *top = reinterpret_cast<float4 *>(dstf);
            float4 *bot = reinterpret_cast<float4 *>(dstf + (size_t)(y0 + nh) * iw);
            const int plane4 = plane / kV;
            for (int i = tid; i < top4; i += nthreads)
                for (int c = 0; c < 3; c++) __stcs(top + (size_t)c * plane4 + i, one4);
            for (int i = tid; i < bot4; i += nthreads)
                for (int c = 0; c < 3; c++) __stcs(bot + (size_t)c * plane4 + i, one4);
            if (tail4 > 0) {
                // right of the pasted rectangle: a thread owns one 16-byte column (and, when the tail is narrower than
                // the thread count, one of `split` row phases) and walks down the rows -- per row one pointer
                // increment and a store per channel, no index arithmetic (a lone warp runs at its dependent-issue
                // latency: the previous per-element division made this loop 5 600 cycles per crop)
                const int split = max(1, nthreads / tail4);
                const int col = tid % tail4, phase = tid / tail4;
                if (phase < split) {
                    float4 *at = reinterpret_cast<float4 *>(dstf + (size_t)(y0 + phase) * iw + nw4) + col;
                    const size_t step = (size_t)split * iw / kV;
                    for (int k = col; k < tail4; k += nthreads) {  // (tails wider than the thread count: several columns)
                        float4 *p4 = at + (k - col);
                        for (int r = phase; r < nh; r += split, p4 += step)
                            for (int c = 0; c < 3; c++) __stcs(p4 + (size_t)c * plane4, one4);
                    }
                }
            }
            if (fr > 0) {
                for (int i = tid; i < nh * fr; i += nthreads) {
                    const int r = i / fr, k = i - r * fr;
                    T *at = dstf + (size_t)(y0 + r) * iw + nw + k;
                    for (int c = 0; c < 3; c++) __stcs(at + (size_t)c * plane, one);
                }
            }
        } else {
            for (int e = tid; e < 3 * plane; e += nthreads) {
                int c = e / plane, rem = e - c * plane;
                int y = rem / iw, x = rem - y * iw;
                if (!(y >= y0 && y < y0 + nh && x < nw)) dstf[e] = one;
            }
        }
    }
    if (kWriteU8) {
        for (int e = tid; e < plane; e += nthreads) {
            int y = e / iw, x = e - y * iw;
            if (!(y >= y0 && y < y0 + nh && x < nw)) {
                dstu[(size_t)e * 3] = 255;
                dstu[(size_t)e * 3 + 1] = 255;
                dstu[(size_t)e * 3 + 2] = 255;
            }
        }
    }
}

template <class T, bool kWriteU8>
__device__ __forceinline__ void write_padding(const Plan &p, int ih, int iw, T *dstf, uint8_t *dstu, int vec_ok,
                                              int tid, int nthreads)
{
    write_padding<T, kWriteU8>(p.ok ? p.nw : 0, p.ok ? p.nh : 0, p.ok ? p.y0 : 0, ih, iw, dstf, dstu, vec_ok, tid,
                               nthreads);
}

// u8 -> f32 without the conversion pipe: byte k of `v` is spliced under the exponent of 2^23, then 2^23 is
// subtracted (exact for 0..255)
__device__ __forceinline__ float byte_f32(uint32_t v, uint32_t sel)
{
    return __uint_as_float(__byte_perm(v, 0x4B000000u, sel)) - 8388608.0f;
}

// Horizontal pass of the INTER_AREA general path for one (source row, destination column) whose table has <= 4 taps,
// out of the staged rows: 12 contiguous bytes (4 taps x RGB) fetched as aligned 32-bit shared-memory words; taps
// beyond n carry weight 0 (x + 0*y == x exactly, every term is >= 0).  Same products and the same summation order as
// resample_px's general branch.  `o` = shared-memory byte offset of the row's first tap.
// kTaps = 3: every x entry of the crop has at most 3 taps (always the case for a shrink factor below 2), so the fourth
// tap -- weight 0, an exact no-op -- and the word that only it needs are not touched.
// Packed float32 pairs (sm_100 FADD2 / FMUL2): two IEEE round-to-nearest operations per issue slot, same results as
// two scalar instructions.  Only conversions and PRODUCTS are packed: ptxas contracts mul.f32x2 + add.f32x2 into FFMA2
// even with --fmad=false, which would change the rounding, so every sum stays a scalar FADD on one half of a pair.
__device__ __forceinline__ void f2_unpack(unsigned long long v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long f2_pack_bits(uint32_t lo, uint32_t hi)
{
    unsigned long long v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "r"(lo), "r"(hi));
    return v;
}
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi)
{
    unsigned long long v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
__device__ __forceinline__ unsigned long long f2_add(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long f2_mul(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// bytes k0 and k1 of `va` / `vb` as two floats: (2^23 + byte) spliced by PRMT, then one packed subtraction of 2^23
__device__ __forceinline__ unsigned long long bytes2_f32(uint32_t va, uint32_t sa, uint32_t vb, uint32_t sb)
{
    const unsigned long long magic = f2_pack(-8388608.0f, -8388608.0f);
    return f2_add(f2_pack_bits(__byte_perm(va, 0x4B000000u, sa), __byte_perm(vb, 0x4B000000u, sb)), magic);
}

template <int kTaps>
__device__ __forceinline__ void hrow_area4(const unsigned char *smem_base, uint32_t o, const float4 wx, float &b0,
                                           float &b1, float &b2)
{
    const uint32_t *smem32 = reinterpret_cast<const uint32_t *>(smem_base);
    const uint32_t wi = o >> 2, sh = (o & 3u) * 8u;
    const uint32_t q0 = smem32[wi], q1 = smem32[wi + 1], q2 = smem32[wi + 2];
    const uint32_t q3 = kTaps > 3 ? smem32[wi + 3] : 0u;
    const uint32_t u0 = __funnelshift_r(q0, q1, sh), u1 = __funnelshift_r(q1, q2, sh), u2 = __funnelshift_r(q2, q3, sh);
    // bytes: tap0 = u0.b0..b2, tap1 = u0.b3 u1.b0 u1.b1, tap2 = u1.b2 u1.b3 u2.b0, tap3 = u2.b1..b3
    float p00, p01, p02, p10, p11, p12, p20, p21, p22;
    f2_unpack(f2_mul(bytes2_f32(u0, 0x7650, u0, 0x7651), f2_pack(wx.x, wx.x)), p00, p01);  // tap 0: channels 0, 1
    f2_unpack(f2_mul(bytes2_f32(u0, 0x7652, u0, 0x7653), f2_pack(wx.x, wx.y)), p02, p10);  // tap 0 ch 2, tap 1 ch 0
    f2_unpack(f2_mul(bytes2_f32(u1, 0x7650, u1, 0x7651), f2_pack(wx.y, wx.y)), p11, p12);  // tap 1: channels 1, 2
    f2_unpack(f2_mul(bytes2_f32(u1, 0x7652, u1, 0x7653), f2_pack(wx.z, wx.z)), p20, p21);  // tap 2: channels 0, 1
    if (kTaps > 3) {
        float p30, p31, p32;
        f2_unpack(f2_mul(bytes2_f32(u2, 0x7650, u2, 0x7651), f2_pack(wx.z, wx.w)), p22, p30);  // tap 2 ch 2, tap 3 ch 0
        f2_unpack(f2_mul(bytes2_f32(u2, 0x7652, u2, 0x7653), f2_pack(wx.w, wx.w)), p31, p32);  // tap 3: channels 1, 2
        b0 = ((p00 + p10) + p20) + p30;
        b1 = ((p01 + p11) + p21) + p31;
        b2 = ((p02 + p12) + p22) + p32;
    } else {
        p22 = byte_f32(u2, 0x7650) * wx.z;
        b0 = (p00 + p10) + p20;
        b1 = (p01 + p11) + p21;
        b2 = (p02 + p12) + p22;
    }
}

// words of one crop's table set: x entries as five arrays of iw words, y entries as ih records of 8 words
__host__ __device__ inline int area_tab_ybase(int iw) { return (5 * iw + 3) & ~3; }  // 16-byte aligned records
__host__ __device__ inline int area_tab_words(int ih, int iw) { return area_tab_ybase(iw) + 8 * ih; }

// The INTER_AREA coefficient tables of one crop for the 4-tap path.  x entries, structure of arrays (a warp's lanes read
// consecutive columns): tab[0][i] = s0 | n << 16, tab[1..4][i] = tap weights (0 beyond n), i in [0, iw).  y entries,
// array of 8-word records after them (a thread walks down the rows: one 16-byte load for the four weights):
// ytab[d] = {s0 | n << 16, -, -, -, w0, w1, w2, w3} at word area_tab_ybase(iw) + 8 * d (weights 16-byte aligned).
// Plan::fast guarantees n <= 4; an entry that violates it is stored with n = 0xffff and makes the consumers hand the
// crop to the generic kernel.
// Returns whether every x entry built by this thread has at most 3 taps (the caller combines the threads' answers).
__device__ __forceinline__ bool build_tables(const Plan &p, uint32_t *tab, int tab_n, int iw, int tid,
                                             int nthreads = 32)
{
    float *tw = reinterpret_cast<float *>(tab);
    bool x3 = true;
    const double inv_x = 1.0 / p.scale_x, inv_y = 1.0 / p.scale_y;
    for (int t = tid; t < p.nw + p.nh; t += nthreads) {
        const bool isx = t < p.nw;
        const int d = isx ? t : t - p.nw;
        const AxisEnt e = isx ? area_entry(d, p.scale_x, p.w, inv_x) : area_entry(d, p.scale_y, p.h, inv_y);
        const bool fits = e.n <= 4 && e.s0 >= 0 && e.s0 < 65536;
        x3 = x3 && !(isx && e.n > 3);
        const uint32_t packed = fits ? ((uint32_t)e.s0 | ((uint32_t)e.n << 16)) : 0xffff0000u;
        if (isx) {
            tab[d] = packed;
#pragma unroll
            for (int k = 0; k < 4; k++) tw[(size_t)(1 + k) * iw + d] = k < e.n ? area_weight(e, k) : 0.f;
        } else {
            uint32_t *rec = tab + area_tab_ybase(iw) + 8 * d;
            rec[0] = packed;
#pragma unroll
            for (int k = 0; k < 4; k++) reinterpret_cast<float *>(rec)[4 + k] = k < e.n ? area_weight(e, k) : 0.f;
        }
    }
    return x3;
}

// INTER_AREA general path for a crop whose axis tables have <= 4 taps per entry (shrink factors below 3), source
// rows in shared memory `pitch` bytes apart starting at byte `stage_off` (+ the 16-byte misalignment a0, which
// advances by sstep per row), SoA tables from build_tables.  kCT cooperating threads (index ct) each resample column
// strips (one destination column, G consecutive destination rows): with a shrink factor near 2 neighbouring
// destination rows share their boundary source row, so a strip needs ~(2G + 1) horizontal row sums instead of 3G;
// per-pixel arithmetic and its order are those of resample_px's general branch.  Returns true when a table entry
// had more than 4 taps (the caller redoes the crop with resample_px).
// strip height (destination rows per thread item) that keeps kCT threads evenly loaded
template <int kCT>
__device__ __forceinline__ int strip_height(int nw, int nh)
{
    int G = 1, best = 0x7fffffff;
    for (int g = 8; g >= 1; g >>= 1) {
        const int items = ((nh + g - 1) / g) * nw;
        const int cost = ((items + kCT - 1) / kCT) * (2 * g + 1);
        if (cost < best) {
            best = cost;
            G = g;
        }
    }
    return G;
}

// INTER_AREA with both scale factors exactly 2 (cv2's integer fast path: (sum of the 2 x 2 block + 2) >> 2), source rows
// staged like area4_strips'; a thread per destination pixel.  A word box exactly twice the canvas height is common
// (2.5 % of the benchmark's crops), and its rounding differs from the float-table path, so it has its own routine.
template <class T, bool kWriteU8, int kCT>
__device__ __forceinline__ void area2x2_pixels(const unsigned char *smem, uint32_t stage_off, uint32_t pitch, uint32_t a0,
                                               uint32_t sstep, int ih, int iw, int nw, int nh, int y0, T *dstf,
                                               uint8_t *dstu, int ct)
{
    const int plane = ih * iw;
    const uint32_t magic = 0xFFFFFFFFu / (uint32_t)nw + 1u;
    for (int t = ct; t < nw * nh; t += kCT) {
        const int dy = nw == 1 ? t : (int)__umulhi((uint32_t)t, magic), dx = t - dy * nw;
        int s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
        for (int yy = 0; yy < 2; yy++) {
            const uint32_t r = (uint32_t)(2 * dy + yy);
            const unsigned char *row = smem + stage_off + r * pitch + ((a0 + r * sstep) & 15u) + 6u * (uint32_t)dx;
            s0 += row[0] + row[3];
            s1 += row[1] + row[4];
            s2 += row[2] + row[5];
        }
        const int o0 = (s0 + 2) >> 2, o1 = (s1 + 2) >> 2, o2 = (s2 + 2) >> 2;
        const int at = (y0 + dy) * iw + dx;
        if constexpr (kHasBatch<T>) {
            store_norm(dstf + at, (float)o0);
            store_norm(dstf + plane + at, (float)o1);
            store_norm(dstf + 2 * plane + at, (float)o2);
        }
        if (kWriteU8) {
            dstu[(size_t)at * 3] = (unsigned char)o0;
            dstu[(size_t)at * 3 + 1] = (unsigned char)o1;
            dstu[(size_t)at * 3 + 2] = (unsigned char)o2;
        }
    }
}

// kAligned: the caller guarantees sstep == 0 (source row stride a multiple of 16 bytes: every staged row has the same
// misalignment a0), so the per-row misalignment arithmetic disappears.
template <class T, bool kWriteU8, int kCT, int kTaps, bool kAligned = false>
__device__ __forceinline__ bool area4_strips(const unsigned char *smem, uint32_t stage_off, uint32_t pitch, uint32_t a0,
                                             uint32_t sstep, const uint32_t *tab, int tab_n, int ih, int iw, int nw,
                                             int nh, int y0, T *dstf, uint8_t *dstu, int ct, int G_in = 0,
                                             int dy_lo = 0, int dy_hi = -1)
{
    // [dy_lo, dy_hi): the destination rows to produce (default: all nh of them); the staged rows are addressed by
    // their absolute source row either way
    const int plane = ih * iw;
    const int G = G_in > 0 ? G_in : strip_height<kCT>(nw, nh);
    if (dy_hi < 0) dy_hi = nh;
    const int nitems = ((dy_hi - dy_lo + G - 1) / G) * nw;
    const uint32_t magic = 0xFFFFFFFFu / (uint32_t)nw + 1u;  // t / nw for t < 2^32 / nw
    const float *tw = reinterpret_cast<const float *>(tab);
    bool bad = false;
    for (int t = ct; t < nitems; t += kCT) {
        const int grp = nw == 1 ? t : (int)__umulhi((uint32_t)t, magic), dx = t - grp * nw;
        const uint32_t px = tab[dx];
        bad = bad || (px >> 16) > 4u;
        const float4 wx = make_float4(tw[iw + dx], tw[2 * iw + dx], tw[3 * iw + dx], tw[4 * iw + dx]);
        const uint32_t xoff = stage_off + (px & 0xffffu) * 3u;
        int last_r = -1;
        float b0 = 0.f, b1 = 0.f, b2 = 0.f;
        const int dy_first = dy_lo + grp * G, dy_end = min(dy_hi, dy_first + G);
        T *orow = kHasBatch<T> ? dstf + (size_t)(y0 + dy_first) * iw + dx : nullptr;  // walks down the strip's rows
        for (int dy = dy_first; dy < dy_end; dy++) {
            const uint32_t *yrec = tab + area_tab_ybase(iw) + 8 * dy;
            const uint32_t py = yrec[0];
            bad = bad || (py >> 16) > 4u;
            const int ys0 = (int)(py & 0xffffu), yn = min((int)(py >> 16), 4);
            const float4 wy4 = *reinterpret_cast<const float4 *>(yrec + 4);
            const float wyv[4] = {wy4.x, wy4.y, wy4.z, wy4.w};
            // row 0 is the previous destination row's last source row when the two share it (uniform branch);
            // the other rows are independent horizontal passes
            const uint32_t rbase = xoff + (uint32_t)ys0 * pitch;
            if (ys0 != last_r) {
                const uint32_t mis = (kAligned || sstep == 0) ? a0 : ((a0 + (uint32_t)ys0 * sstep) & 15u);
                hrow_area4<kTaps>(smem, rbase + mis, wx, b0, b1, b2);
            }
            float sum0 = wyv[0] * b0, sum1 = wyv[0] * b1, sum2 = wyv[0] * b2;
#pragma unroll
            for (int j = 1; j < 4; j++) {
                if (j < yn) {
                    const uint32_t r = (uint32_t)(ys0 + j);
                    const uint32_t mis = (kAligned || sstep == 0) ? a0 : ((a0 + r * sstep) & 15u);
                    hrow_area4<kTaps>(smem, rbase + (uint32_t)j * pitch + mis, wx, b0, b1, b2);
                    sum0 += wyv[j] * b0;
                    sum1 += wyv[j] * b1;
                    sum2 += wyv[j] * b2;
                }
            }
            last_r = ys0 + yn - 1;  // b0..b2 hold that row's horizontal sums
            // cvRound (half to even), kept as floats: the weights sum to 1 within rounding -> [0, 255]
            const float f0 = rintf(sum0), f1 = rintf(sum1), f2 = rintf(sum2);
            const int at = (y0 + dy) * iw + dx;
            if constexpr (kHasBatch<T>) {
                store_norm(orow, f0);
                store_norm(orow + plane, f1);
                store_norm(orow + 2 * plane, f2);
                orow += iw;
            }
            if (kWriteU8) {
                dstu[(size_t)at * 3] = sat_u8((int)f0);
                dstu[(size_t)at * 3 + 1] = sat_u8((int)f1);
                dstu[(size_t)at * 3 + 2] = sat_u8((int)f2);
            }
        }
    }
    return bad;
}

// The crop kernels are instantiated for the outputs they write: <T, kWriteU8> with T the batch element type (float,
// __half, __nv_bfloat16) with or without the u8 canvas, or <NoBatch, true>.  Calls
// launch(BatchType<T>{}, std::bool_constant<kWriteU8>{}) for the outputs present; an unknown batch_dtype is
// MS_ERR_INVALID.
template <class T>
struct BatchType {
    using type = T;
};

template <class Launch>
int launch_for_outputs(const void *batch, int batch_dtype, const uint8_t *canvas_u8, Launch &&launch)
{
    if (!batch) return launch(BatchType<NoBatch>{}, std::true_type{});
    switch (batch_dtype) {
    case MS_DTYPE_F32:
        return canvas_u8 ? launch(BatchType<float>{}, std::true_type{}) : launch(BatchType<float>{}, std::false_type{});
    case MS_DTYPE_F16:
        return canvas_u8 ? launch(BatchType<__half>{}, std::true_type{}) : launch(BatchType<__half>{}, std::false_type{});
    case MS_DTYPE_BF16:
        return canvas_u8 ? launch(BatchType<__nv_bfloat16>{}, std::true_type{})
                         : launch(BatchType<__nv_bfloat16>{}, std::false_type{});
    }
    ms_set_error("crop: unknown batch dtype %d", batch_dtype);
    return MS_ERR_INVALID;
}

// The shared-memory slot of one output instantiation, in the order of a slot group of ms_smem_slot (`first` = the
// group's u8-only slot): u8, f32, f32 + u8, f16, f16 + u8, bf16, bf16 + u8.
template <class T, bool kWriteU8>
constexpr ms_smem_slot batch_slot(ms_smem_slot first)
{
    const int t = std::is_same<T, float>::value ? 0 : std::is_same<T, __half>::value ? 1 : 2;
    return (ms_smem_slot)(first + (kHasBatch<T> ? 1 + 2 * t + (kWriteU8 ? 1 : 0) : 0));
}

// vec_ok of write_padding for a batch of element type T
template <class T>
int batch_vec_ok(const void *batch, int out_w)
{
    return (out_w % kBatchVec<T> == 0 && (reinterpret_cast<uintptr_t>(batch) & 15) == 0) ? 1 : 0;
}

}  // namespace
