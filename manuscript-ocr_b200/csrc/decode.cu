// EAST score-map thresholding + QUAD geometry decode with ordered stream compaction.
// Replaces decode_quads_from_maps (reference detectors/_east/utils.py:328-381).
//
// Reference semantics reproduced bit-exactly (SURVEY 8a-1):
//   * candidate pixels: score > f32(thr), strict (utils.py:340, numpy compares in float32)
//   * quantisation q>1: pixel -> cell (y//q, x//q); one row per cell that holds any candidate,
//     read at the cell's centre pixel (y//q*q + q//2, ...) (utils.py:347-356) -- the centre may be
//     below threshold; rows come out in (y,x) order because np.unique sorts them
//   * v = x*scale [f64] + f32(d*f32(scale)) -> f64 sum -> f32 (utils.py:368-381, NEP-50 promotion)
//   * a centre outside the map raises IndexError in the reference -> MS_FLAG_INDEX_ERROR here
//
// Data layout: score (P,H,W), geo (P,8,H,W) at any element strides (ms_maps), in float32, float16 or bfloat16; every
// value is widened to float32 at its load (exact) and the arithmetic after it is the float32 path's.  Out page-strided
// (P*cap,9) f32.
// HBM traffic (algorithmic): H*W score elements read + 8*N gathered geometry elements + 36*N bytes written per page.
//
// Three launches: mark (ballot bitmasks + per-tile counts), scan (per page), emit (gather + staged,
// coalesced row writes).  One cell per lane; a warp's 32 cells are 32 consecutive cells of a row, so
// score loads are coalesced (one 2-element vector per lane for q=2 where the layout allows it).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "ms_internal.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWordsPerWarp = 8;                      // 8 x 32 cells per warp
constexpr int kWarps = kThreads / 32;
constexpr int kTileWords = kWarps * kWordsPerWarp;    // 64 mask words
// (2048 cells per CTA)

struct DecodeGeom {
    int H, W, q, CH, CW;
    int cells;         // CH*CW
    int words;         // ceil(cells/32)
    int tiles;         // ceil(words/kTileWords)
};

__host__ __device__ inline DecodeGeom make_geom(int H, int W, int q)
{
    DecodeGeom g;
    g.H = H;
    g.W = W;
    g.q = q < 1 ? 1 : q;
    g.CH = (H + g.q - 1) / g.q;
    g.CW = (W + g.q - 1) / g.q;
    g.cells = g.CH * g.CW;
    g.words = (g.cells + 31) / 32;
    g.tiles = (g.words + kTileWords - 1) / kTileWords;
    return g;
}

// Element strides of the two maps (ms_maps) and the load paths the host chose from them and the pointers' alignment.
struct MapLayout {
    int64_t s_page, s_row, s_col;          // score
    int64_t g_page, g_ch, g_row, g_col;    // geometry
    int score_pairs;  // q = 2: the two pixels of a cell row are adjacent and 2-element aligned -> one vector load
};

// a map value widened to float32: the conversions torch's .float() makes on the device
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__device__ __forceinline__ float ld_map(const T *p)
{
    return to_f32(__ldg(p));
}
// two adjacent values, the first aligned to twice the element size: one 8-byte (float32) or 4-byte (16 bits) load
__device__ __forceinline__ float2 ld_map2(const float *p) { return __ldg(reinterpret_cast<const float2 *>(p)); }
template <typename T>
__device__ __forceinline__ float2 ld_map2(const T *p)
{
    const unsigned int u = __ldg(reinterpret_cast<const unsigned int *>(p));
    const T *v = reinterpret_cast<const T *>(&u);
    return make_float2(to_f32(v[0]), to_f32(v[1]));
}
// the 8 geometry values of a pixel, adjacent and 16-byte aligned: two 16-byte loads (float32) or one (16 bits)
__device__ __forceinline__ void ld_geo8(const float *p, float *d)
{
    const float4 a = __ldg(reinterpret_cast<const float4 *>(p)), b = __ldg(reinterpret_cast<const float4 *>(p) + 1);
    d[0] = a.x, d[1] = a.y, d[2] = a.z, d[3] = a.w, d[4] = b.x, d[5] = b.y, d[6] = b.z, d[7] = b.w;
}
template <typename T>
__device__ __forceinline__ void ld_geo8(const T *p, float *d)
{
    const uint4 u = __ldg(reinterpret_cast<const uint4 *>(p));
    const T *v = reinterpret_cast<const T *>(&u);
#pragma unroll
    for (int i = 0; i < 8; i++) d[i] = to_f32(v[i]);
}

template <typename T>
__device__ __forceinline__ bool cell_hit(const T *__restrict__ score, const DecodeGeom &g, const MapLayout &L, int cell,
                                         float thr)
{
    if (cell >= g.cells) return false;
    int cy = cell / g.CW, cx = cell - cy * g.CW;
    if (g.q == 1) return ld_map(score + cy * L.s_row + cx * L.s_col) > thr;
    if (g.q == 2 && L.score_pairs) {
        // both pixels of a row of the cell are in range when W is even (score_pairs implies it)
        int y = 2 * cy;
        const T *r0 = score + y * L.s_row + 2 * cx;
        float2 a = ld_map2(r0);
        bool hit = a.x > thr || a.y > thr;
        if (y + 1 < g.H) {
            float2 b = ld_map2(r0 + L.s_row);
            hit = hit || b.x > thr || b.y > thr;
        }
        return hit;
    }
    bool hit = false;
    for (int dy = 0; dy < g.q; dy++) {
        int y = cy * g.q + dy;
        if (y >= g.H) break;
        for (int dx = 0; dx < g.q; dx++) {
            int x = cx * g.q + dx;
            if (x >= g.W) break;
            hit = hit || (ld_map(score + y * L.s_row + x * L.s_col) > thr);
        }
    }
    return hit;
}

// mark: one lane per cell, ballot -> mask words + per-tile candidate counts
template <typename T>
__global__ void __launch_bounds__(kThreads) decode_mark_kernel(const T *__restrict__ score, DecodeGeom g, MapLayout L,
                                                               float thr, uint32_t *__restrict__ masks,
                                                               int32_t *__restrict__ tile_counts,
                                                               int32_t *__restrict__ flags)
{
    ms_pdl_wait();
    const int page = blockIdx.y, tile = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T *sc = score + page * L.s_page;
    __shared__ int s_cnt[kWarps];
    int cnt = 0;
    bool bad = false;
#pragma unroll
    for (int k = 0; k < kWordsPerWarp; k++) {
        int word = tile * kTileWords + warp * kWordsPerWarp + k;
        int cell = word * 32 + lane;
        bool hit = word < g.words && cell_hit(sc, g, L, cell, thr);
        if (hit && g.q > 1) {
            int cy = cell / g.CW, cx = cell - cy * g.CW;
            if (cy * g.q + g.q / 2 >= g.H || cx * g.q + g.q / 2 >= g.W) {  // utils.py:370 IndexError
                bad = true;
                hit = false;
            }
        }
        uint32_t m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0 && word < g.words) masks[(size_t)page * g.words + word] = m;
        cnt += __popc(m);
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flags + page, MS_FLAG_INDEX_ERROR);
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kWarps; w++) t += s_cnt[w];
        tile_counts[(size_t)page * g.tiles + tile] = t;
    }
}

// scan: one CTA per page, exclusive prefix over its tile counts
__global__ void __launch_bounds__(256) decode_scan_kernel(const int32_t *__restrict__ tile_counts, int tiles,
                                                          int cap, int32_t *__restrict__ tile_base,
                                                          int32_t *__restrict__ counts, int32_t *__restrict__ flags)
{
    ms_pdl_wait();
    const int page = blockIdx.x;
    __shared__ int s_part[256];
    __shared__ int s_run;
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    for (int base = 0; base < tiles; base += 256) {
        int i = base + threadIdx.x;
        int v = i < tiles ? tile_counts[(size_t)page * tiles + i] : 0;
        s_part[threadIdx.x] = v;
        __syncthreads();
        // Hillis-Steele inclusive scan over 256 entries
        for (int off = 1; off < 256; off <<= 1) {
            int t = threadIdx.x >= off ? s_part[threadIdx.x - off] : 0;
            __syncthreads();
            s_part[threadIdx.x] += t;
            __syncthreads();
        }
        int run = s_run;
        if (i < tiles) tile_base[(size_t)page * tiles + i] = run + s_part[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 255) s_run = run + s_part[255];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int total = s_run;
        if (total > cap) {
            atomicOr(flags + page, MS_FLAG_CAND_OVERFLOW);
            total = cap;
        }
        counts[page] = total;
    }
}

// RBOX geometry (EAST, Zhou et al. 2017: four distances to the edges of the rotated word rectangle -- top, right,
// bottom, left -- and its angle) -> the rectangle's corners TL, TR, BR, BL.  NOT a reference behaviour (the reference's
// head is QUAD only, SURVEY 0); the closed form is the one of the public EAST implementations (restore_rectangle_rbox):
// lay the rectangle out with the pixel at (d_left, -d_bottom) from its bottom-left corner (angle >= 0) or at
// (-d_right, -d_bottom) from its bottom-right corner (angle < 0), rotate by the angle, translate the pixel back onto
// (x, y).  float64 throughout; distances are map units times `scale`.
__device__ __forceinline__ void rbox_to_quad(double ox, double oy, double dt, double dr, double db, double dl, double ang,
                                             float *r)
{
    double px[4], py[4], qx, qy, c, s;
    if (ang >= 0.0) {
        px[0] = 0.0, py[0] = -dt - db;
        px[1] = dr + dl, py[1] = -dt - db;
        px[2] = dr + dl, py[2] = 0.0;
        px[3] = 0.0, py[3] = 0.0;
        qx = dl, qy = -db;
        c = cos(ang), s = sin(ang);
    } else {
        px[0] = -dr - dl, py[0] = -dt - db;
        px[1] = 0.0, py[1] = -dt - db;
        px[2] = 0.0, py[2] = 0.0;
        px[3] = -dr - dl, py[3] = 0.0;
        qx = -dr, qy = -db;
        c = cos(-ang), s = -sin(-ang);
    }
    // rotated point = (c * x + s * y, -s * x + c * y)
    const double tx = ox - (c * qx + s * qy), ty = oy - (-s * qx + c * qy);
#pragma unroll
    for (int v = 0; v < 4; v++) {
        r[2 * v] = (float)(c * px[v] + s * py[v] + tx);
        r[2 * v + 1] = (float)(-s * px[v] + c * py[v] + ty);
    }
}

// emit: rank candidates inside the tile, gather geometry at the cell centre, write rows in order.  kGeo8: a pixel's 8
// QUAD geometry values are adjacent and 16-byte aligned (channels-last geometry), gathered by ld_geo8.
template <typename T, bool kRbox, bool kGeo8>
__global__ void __launch_bounds__(kThreads) decode_emit_kernel(const T *__restrict__ score, const T *__restrict__ geo,
                                                               DecodeGeom g, MapLayout L, double scale,
                                                               const uint32_t *__restrict__ masks,
                                                               const int32_t *__restrict__ tile_base, int cap,
                                                               float *__restrict__ out, int geo_compact)
{
    ms_pdl_wait();
    const int page = blockIdx.y, tile = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __shared__ int s_word_base[kTileWords];
    __shared__ float s_rows[kWarps][32 * 9];
    const T *sc = score + page * L.s_page;
    const T *ge = geo + page * L.g_page;
    const uint32_t *mk = masks + (size_t)page * g.words;

    // exclusive prefix over the tile's 64 mask-word popcounts (two warps worth of data)
    if (threadIdx.x < kTileWords) {
        int word = tile * kTileWords + threadIdx.x;
        s_word_base[threadIdx.x] = word < g.words ? __popc(mk[word]) : 0;
    }
    __syncthreads();
    if (warp == 0) {
        int a = s_word_base[lane], b = s_word_base[lane + 32];
        int ia = a, ib = b;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            int ta = __shfl_up_sync(0xffffffffu, ia, off);
            int tb = __shfl_up_sync(0xffffffffu, ib, off);
            if (lane >= off) {
                ia += ta;
                ib += tb;
            }
        }
        int tot_a = __shfl_sync(0xffffffffu, ia, 31);
        s_word_base[lane] = ia - a;
        s_word_base[lane + 32] = tot_a + ib - b;
    }
    __syncthreads();

    const int tbase = tile_base[(size_t)page * g.tiles + tile];
    const float sc32 = (float)scale;
    float *stage = s_rows[warp];
#pragma unroll 1
    for (int k = 0; k < kWordsPerWarp; k++) {
        int wl = warp * kWordsPerWarp + k;
        int word = tile * kTileWords + wl;
        if (word >= g.words) break;
        uint32_t m = mk[word];
        if (m == 0) continue;
        int cnt = __popc(m);
        int row0 = tbase + s_word_base[wl];
        if (row0 >= cap) break;
        if (row0 + cnt > cap) cnt = cap - row0;
        bool mine = (m >> lane) & 1u;
        int rank = __popc(m & ((1u << lane) - 1u));
        if (mine && rank < cnt) {
            int cell = word * 32 + lane;
            int cy = cell / g.CW, cx = cell - cy * g.CW;
            int y = g.q > 1 ? cy * g.q + g.q / 2 : cy;
            int x = g.q > 1 ? cx * g.q + g.q / 2 : cx;
            // geo_compact: the geometry tensor holds only the rows a quantised read can touch (y % q == q / 2), i.e.
            // (P, 8, H / q, W) -- what ms_page_batch_host uploads -- and L's geometry strides are that tensor's
            const T *gp = ge + (geo_compact ? cy : y) * L.g_row + x * L.g_col;
            // the score and geometry loads go out before the arithmetic that uses them: one memory latency per
            // candidate instead of nine dependent ones
            const float score_v = ld_map(sc + y * L.s_row + x * L.s_col);
            double xs = __dmul_rn((double)x, scale);
            double ys = __dmul_rn((double)y, scale);
            float *r = stage + rank * 9;
            if (kRbox) {
                double d[5];
#pragma unroll
                for (int v = 0; v < 5; v++, gp += L.g_ch) d[v] = (double)ld_map(gp);
                rbox_to_quad(xs, ys, d[0] * scale, d[1] * scale, d[2] * scale, d[3] * scale, d[4], r);
            } else {
                float d[8];
                if (kGeo8)
                    ld_geo8(gp, d);
                else
#pragma unroll
                    for (int v = 0; v < 8; v++, gp += L.g_ch) d[v] = ld_map(gp);
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    r[2 * v] = (float)__dadd_rn(xs, (double)__fmul_rn(d[2 * v], sc32));
                    r[2 * v + 1] = (float)__dadd_rn(ys, (double)__fmul_rn(d[2 * v + 1], sc32));
                }
            }
            r[8] = score_v;
        }
        __syncwarp();
        float *dst = out + ((size_t)page * cap + row0) * 9;
        for (int i = lane; i < cnt * 9; i += 32) dst[i] = stage[i];
        __syncwarp();
    }
}

}  // namespace

size_t msk_decode_scratch(int n_pages, int H, int W, int q)
{
    DecodeGeom g = make_geom(H, W, q);
    size_t b = 0;
    b += ((size_t)n_pages * g.words * 4 + 255) & ~size_t(255);
    b += 2 * (((size_t)n_pages * g.tiles * 4 + 255) & ~size_t(255));
    return b + 1024;
}

// the launches of one map element type
template <typename T>
static int decode_launch(ms_ctx *ctx, const T *score, const T *geo, const DecodeGeom &g, const MapLayout &L, bool geo8,
                         float thr, double scale, float *quads_out, int cap_per_page, int32_t *counts, int32_t *flags,
                         uint32_t *masks, int32_t *tile_counts, int32_t *tile_base, int n_pages, cudaStream_t st,
                         int geo_compact, int rbox)
{
    dim3 grid(g.tiles, n_pages);
    ms_launch(decode_mark_kernel<T>, grid, kThreads, 0, st, score, g, L, thr, masks, tile_counts, flags);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(decode_scan_kernel, n_pages, 256, 0, st, tile_counts, g.tiles, cap_per_page, tile_base, counts, flags);
    MS_LAUNCH_CHECK(ctx);
    if constexpr (std::is_same<T, float>::value) {
        if (rbox) {
            ms_launch(decode_emit_kernel<float, true, false>, grid, kThreads, 0, st, score, geo, g, L, scale, masks,
                      tile_base, cap_per_page, quads_out, geo_compact);
            MS_LAUNCH_CHECK(ctx);
            return MS_OK;
        }
    }
    if (geo8)
        ms_launch(decode_emit_kernel<T, false, true>, grid, kThreads, 0, st, score, geo, g, L, scale, masks, tile_base,
                  cap_per_page, quads_out, geo_compact);
    else
        ms_launch(decode_emit_kernel<T, false, false>, grid, kThreads, 0, st, score, geo, g, L, scale, masks, tile_base,
                  cap_per_page, quads_out, geo_compact);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}

int msk_decode(ms_ctx *ctx, const ms_maps &m, int n_pages, int H, int W, float thr, double scale, int q,
               float *quads_out, int cap_per_page, int32_t *counts, int32_t *flags, ms_bump bump, cudaStream_t st,
               int geo_compact, int rbox)
{
    if (n_pages <= 0) return MS_OK;
    if (geo_compact && (q < 2 || H % q != 0)) {
        ms_set_error("decode: compact geometry needs q > 1 and H %% q == 0");
        return MS_ERR_INVALID;
    }
    if (H <= 0 || W <= 0 || q < 1 || cap_per_page <= 0) {
        ms_set_error("decode: bad shape H=%d W=%d q=%d cap=%d", H, W, q, cap_per_page);
        return MS_ERR_INVALID;
    }
    if (rbox && m.dtype != MS_DTYPE_F32) {
        ms_set_error("decode: RBOX maps are float32");
        return MS_ERR_INVALID;
    }
    DecodeGeom g = make_geom(H, W, q);
    uint32_t *masks = bump.take<uint32_t>((size_t)n_pages * g.words);
    int32_t *tile_counts = bump.take<int32_t>((size_t)n_pages * g.tiles);
    int32_t *tile_base = bump.take<int32_t>((size_t)n_pages * g.tiles);
    if (!tile_base) {
        ms_set_error("decode: scratch too small");
        return MS_ERR_CAPACITY;
    }
    // the vector loads: chosen from the strides and the pointers' alignment, else one load per element at the strides
    const int64_t es = (int64_t)ms_dtype_bytes(m.dtype);
    const int64_t *ss = m.score_strides, *gs = m.geo_strides;
    MapLayout L = {ss[0], ss[1], ss[2], gs[0], gs[1], gs[2], gs[3], 0};
    L.score_pairs = g.q == 2 && W % 2 == 0 && ss[2] == 1 && ss[1] % 2 == 0 && (n_pages == 1 || ss[0] % 2 == 0) &&
                    (uintptr_t)m.score % (2 * es) == 0;
    const bool geo8 = !rbox && gs[1] == 1 && gs[3] == 8 && (gs[2] * es) % 16 == 0 &&
                      (n_pages == 1 || (gs[0] * es) % 16 == 0) && (uintptr_t)m.geo % 16 == 0;
    switch (m.dtype) {
    case MS_DTYPE_F32:
        return decode_launch(ctx, (const float *)m.score, (const float *)m.geo, g, L, geo8, thr, scale, quads_out,
                             cap_per_page, counts, flags, masks, tile_counts, tile_base, n_pages, st, geo_compact, rbox);
    case MS_DTYPE_F16:
        return decode_launch(ctx, (const __half *)m.score, (const __half *)m.geo, g, L, geo8, thr, scale, quads_out,
                             cap_per_page, counts, flags, masks, tile_counts, tile_base, n_pages, st, geo_compact, rbox);
    case MS_DTYPE_BF16:
        return decode_launch(ctx, (const __nv_bfloat16 *)m.score, (const __nv_bfloat16 *)m.geo, g, L, geo8, thr, scale,
                             quads_out, cap_per_page, counts, flags, masks, tile_counts, tile_base, n_pages, st,
                             geo_compact, rbox);
    }
    ms_set_error("decode: unknown map dtype %d", m.dtype);
    return MS_ERR_INVALID;
}
