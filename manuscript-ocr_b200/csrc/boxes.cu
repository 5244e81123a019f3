// Box post-processing between NMS and the crop batch, float32, bit-exact with the reference's numpy.
// Replaces expand_boxes (reference detectors/_east/utils.py:384-422), the EAST box filters
// (detectors/_east/infer.py:134-233: _scale_boxes_to_original, _remove_fully_contained_boxes,
// _remove_area_anomalies, _convert_to_axis_aligned) and the crop-rectangle logic of
// Pipeline.predict / _extract_word_image (_pipeline.py:125-137, 204-221).
//
// These stages touch K ~ 10^3 boxes per page (36 B each): they are latency bound, not HBM bound.
// One CTA per page; every reduction follows numpy's summation order so thresholds compare equal.
#include "ms_internal.cuh"

namespace {

// ---- utils.py:384-422 expand_boxes, one quad ---------------------------------------------------------
__device__ __forceinline__ void expand_quad(const float *p, float sx, float sy, float *o)
{
    const float eps = (float)1e-6;
    float t[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int j = (i + 1) & 3;
        t[i] = p[2 * i] * p[2 * j + 1] - p[2 * j] * p[2 * i + 1];
    }
    float area = ((t[0] + t[1]) + t[2]) + t[3];  // np.sum over the 4-long axis: left to right
    float sign = area > 0 ? 1.0f : (area < 0 ? -1.0f : 1.0f);
    if (area != area) sign = area;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int ip = (i + 3) & 3, in = (i + 1) & 3;
        float e1x = p[2 * i] - p[2 * ip], e1y = p[2 * i + 1] - p[2 * ip + 1];
        float e2x = p[2 * in] - p[2 * i], e2y = p[2 * in + 1] - p[2 * i + 1];
        float l1 = sqrtf(e1x * e1x + e1y * e1y);
        float l2 = sqrtf(e2x * e2x + e2y * e2y);
        float n1x = sign * e1y / (l1 + eps), n1y = sign * (-e1x) / (l1 + eps);
        float n2x = sign * e2y / (l2 + eps), n2y = sign * (-e2x) / (l2 + eps);
        float ax = n1x + n2x, ay = n1y + n2y;
        float nn = sqrtf(ax * ax + ay * ay);
        if (nn > 0) {
            ax = ax / nn;
            ay = ay / nn;
        } else {
            ax = 0.0f;
            ay = 0.0f;
        }
        float off = l1 < l2 ? l1 : l2;
        if (l1 != l1 || l2 != l2) off = NAN;
        o[2 * i] = p[2 * i] + (sx * off) * ax;
        o[2 * i + 1] = p[2 * i + 1] + (sy * off) * ay;
    }
    o[8] = p[8];
}

__global__ void expand_kernel(const float *__restrict__ quads, int64_t n, double ew, double eh, float *__restrict__ out)
{
    ms_pdl_wait();
    const bool ident = (ew == 0 && eh == 0);  // utils.py:388 returns the input unchanged
    const float sx = (float)(1.0 + ew) - 1.0f, sy = (float)(1.0 + eh) - 1.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float p[9], o[9];
#pragma unroll
        for (int k = 0; k < 9; k++) p[k] = quads[i * 9 + k];
        if (ident) {
#pragma unroll
            for (int k = 0; k < 9; k++) o[k] = p[k];
        } else {
            expand_quad(p, sx, sy, o);
        }
#pragma unroll
        for (int k = 0; k < 9; k++) out[i * 9 + k] = o[k];
    }
}

// infer.py:174-183
__device__ __forceinline__ float quad_area_f32(const float *p)
{
    float t[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int j = (i + 1) & 3;
        t[i] = p[2 * i] * p[2 * j + 1] - p[2 * i + 1] * p[2 * j];
    }
    float s = ((t[0] + t[1]) + t[2]) + t[3];
    return 0.5f * fabsf(s);
}

// cv2.pointPolygonTest(contour f32 (4 pts), pt, measureDist=False), called from infer.py:185-192
__device__ __forceinline__ int point_in_quad(const float *cnt, float px, float py)
{
    int counter = 0;
    float vx = cnt[6], vy = cnt[7];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float v0x = vx, v0y = vy;
        vx = cnt[2 * i];
        vy = cnt[2 * i + 1];
        if ((v0y <= py && vy <= py) || (v0y > py && vy > py) || (v0x < px && vx < px)) {
            if (py == vy && (px == vx || (py == v0y && ((v0x <= px && px <= vx) || (vx <= px && px <= v0x))))) return 0;
            continue;
        }
        double dist = (double)(py - v0y) * (double)(vx - v0x) - (double)(px - v0x) * (double)(vy - v0y);
        if (dist == 0) return 0;
        if (vy < v0y) dist = -dist;
        counter += dist > 0;
    }
    return (counter & 1) ? 1 : -1;
}

__device__ __forceinline__ bool quad_inside(const float *inner, const float *outer)
{
#pragma unroll
    for (int v = 0; v < 4; v++)
        if (point_in_quad(outer, inner[2 * v], inner[2 * v + 1]) < 0) return false;
    return true;
}

#include "np_sum.cuh"

__device__ __forceinline__ bool area_before(float aa, int ia, float ab, int ib)
{
    // position in np.argsort(areas, kind="stable"): ascending, NaN last, ties by index
    bool an = aa != aa, bn = ab != ab;
    if (an || bn) {
        if (an != bn) return bn;
        return ia < ib;
    }
    if (aa < ab) return true;
    if (aa > ab) return false;
    return ia < ib;
}

struct EastScratch {
    float *work;      // (P*cap, 9) expanded + scaled quads
    float *area;      // P*cap
    float4 *bbox;     // P*cap: vertex bounding box (exact min / max of the f32 coordinates)
    uint8_t *removed; // P*cap
    uint8_t *needseq; // P*cap
    int32_t *seq;     // P*cap: the (rare) boxes resolved sequentially, in area-rank order
    float *karea;     // P*cap compacted areas / deviations
    float *kdev;
    int32_t *kidx;    // P*cap compacted indices
    // uniform grid over the boxes' min corners for the containment search
    float *ext;       // P*8: min x / y of the min corners, cells per unit x / y, max box width / height, margin
    int32_t *dense;   // P: 1 = the page holds a non-finite box -> all-pairs kernel
    int32_t *cell_cnt, *cell_off, *cell_cur;  // P*kCells (+1)
    int32_t *cell_of; // P*cap
    float4 *sb_bbox;  // P*cap, cell order: bbox inflated by the prefilter margin
    float *sb_area;   // P*cap
    int32_t *sb_id;   // P*cap
};

constexpr int kEGrid = 32;
constexpr int kECells = kEGrid * kEGrid;

__device__ __forceinline__ int east_cell(float v, float origin, float scale)
{
    const float f = (v - origin) * scale;  // monotone in v: the same function maps corners and search bounds
    return f > 0.f ? (f < (float)(kEGrid - 1) ? (int)f : kEGrid - 1) : 0;
}

__device__ __forceinline__ float4 east_inflate(const float4 b)
{
    const float mx = 1e-4f * fmaxf(fabsf(b.x), fabsf(b.z)) + 1e-3f;
    const float my = 1e-4f * fmaxf(fabsf(b.y), fabsf(b.w)) + 1e-3f;
    return make_float4(b.x - mx, b.y - my, b.z + mx, b.w + my);
}

__device__ __forceinline__ int block_excl_scan(int v, int *s_warp, int &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += t;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = lane < nw ? s_warp[lane] : 0;
        int winc = w;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, winc, off);
            if (lane >= off) winc += t;
        }
        s_warp[lane] = winc - w;
        if (lane == 31) s_warp[32] = winc;
    }
    __syncthreads();
    total = s_warp[32];
    return s_warp[warp] + inc - v;
}

// 1) expand (utils.py:384) + scale to the original image (infer.py:134-147) + area + bbox, all boxes of all pages
__global__ void __launch_bounds__(256) east_prep_kernel(const float *__restrict__ quads,
                                                        const int32_t *__restrict__ counts, int n_pages, int cap,
                                                        ms_east_params P, const int32_t *__restrict__ orig_hw,
                                                        int orig_h, int orig_w, EastScratch S)
{
    ms_pdl_wait();
    const bool ident = (P.expand_ratio_w == 0 && P.expand_ratio_h == 0);
    const float ex = (float)(1.0 + P.expand_ratio_w) - 1.0f, ey = (float)(1.0 + P.expand_ratio_h) - 1.0f;
    const int page = blockIdx.y;
    const int K = counts[page];
    int oh = orig_h > 0 ? orig_h : P.target_size, ow = orig_w > 0 ? orig_w : P.target_size;
    if (orig_hw) {
        oh = orig_hw[2 * page];
        ow = orig_hw[2 * page + 1];
    }
    const float sx = (float)((double)ow / (double)P.target_size);
    const float sy = (float)((double)oh / (double)P.target_size);
    const size_t pb = (size_t)page * cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < K; i += gridDim.x * blockDim.x) {
        float p[9], o[9];
#pragma unroll
        for (int k = 0; k < 9; k++) p[k] = quads[(pb + i) * 9 + k];
        if (ident) {
#pragma unroll
            for (int k = 0; k < 9; k++) o[k] = p[k];
        } else {
            expand_quad(p, ex, ey, o);
        }
        float x0 = INFINITY, x1 = -INFINITY, y0 = INFINITY, y1 = -INFINITY;
        bool fin = true;
#pragma unroll
        for (int v = 0; v < 4; v++) {
            o[2 * v] = o[2 * v] * sx;
            o[2 * v + 1] = o[2 * v + 1] * sy;
            x0 = fminf(x0, o[2 * v]);
            x1 = fmaxf(x1, o[2 * v]);
            y0 = fminf(y0, o[2 * v + 1]);
            y1 = fmaxf(y1, o[2 * v + 1]);
            fin = fin && (fabsf(o[2 * v]) < 1e30f) && (fabsf(o[2 * v + 1]) < 1e30f);
        }
#pragma unroll
        for (int k = 0; k < 9; k++) S.work[(pb + i) * 9 + k] = o[k];
        S.area[pb + i] = quad_area_f32(o);
        // non-finite boxes get an "everything" box so the prefilter never rejects them
        S.bbox[pb + i] = fin ? make_float4(x0, y0, x1, y1) : make_float4(-INFINITY, -INFINITY, INFINITY, INFINITY);
        S.removed[pb + i] = 0;
        S.needseq[pb + i] = 0;
    }
}

// 1b) page extents + grid geometry (one CTA per page); pages with a non-finite box use the all-pairs kernel
__global__ void __launch_bounds__(256) east_ext_kernel(const int32_t *__restrict__ counts, int cap, EastScratch S)
{
    ms_pdl_wait();
    const int page = blockIdx.x;
    const int K = counts[page];
    const size_t pb = (size_t)page * cap;
    float minx = INFINITY, miny = INFINITY, maxx = -INFINITY, maxy = -INFINITY, mw = 0.f, mh = 0.f, mabs = 0.f;
    int bad = 0;
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        const float4 b = S.bbox[pb + i];
        if (!(b.x > -INFINITY && b.z < INFINITY && b.y > -INFINITY && b.w < INFINITY)) {
            bad = 1;
            continue;
        }
        minx = fminf(minx, b.x);
        miny = fminf(miny, b.y);
        maxx = fmaxf(maxx, b.x);
        maxy = fmaxf(maxy, b.y);
        mw = fmaxf(mw, b.z - b.x);
        mh = fmaxf(mh, b.w - b.y);
        mabs = fmaxf(mabs, fmaxf(fmaxf(fabsf(b.x), fabsf(b.z)), fmaxf(fabsf(b.y), fabsf(b.w))));
    }
    __shared__ float s_r[8][7];
    __shared__ int s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    if (bad) s_bad = 1;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        minx = fminf(minx, __shfl_xor_sync(0xffffffffu, minx, off));
        miny = fminf(miny, __shfl_xor_sync(0xffffffffu, miny, off));
        maxx = fmaxf(maxx, __shfl_xor_sync(0xffffffffu, maxx, off));
        maxy = fmaxf(maxy, __shfl_xor_sync(0xffffffffu, maxy, off));
        mw = fmaxf(mw, __shfl_xor_sync(0xffffffffu, mw, off));
        mh = fmaxf(mh, __shfl_xor_sync(0xffffffffu, mh, off));
        mabs = fmaxf(mabs, __shfl_xor_sync(0xffffffffu, mabs, off));
    }
    if ((threadIdx.x & 31) == 0) {
        float *r = s_r[threadIdx.x >> 5];
        r[0] = minx; r[1] = miny; r[2] = maxx; r[3] = maxy; r[4] = mw; r[5] = mh; r[6] = mabs;
    }
    for (int c = threadIdx.x; c < kECells; c += blockDim.x) S.cell_cnt[(size_t)page * kECells + c] = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) {
            s_r[0][0] = fminf(s_r[0][0], s_r[w][0]);
            s_r[0][1] = fminf(s_r[0][1], s_r[w][1]);
            s_r[0][2] = fmaxf(s_r[0][2], s_r[w][2]);
            s_r[0][3] = fmaxf(s_r[0][3], s_r[w][3]);
            s_r[0][4] = fmaxf(s_r[0][4], s_r[w][4]);
            s_r[0][5] = fmaxf(s_r[0][5], s_r[w][5]);
            s_r[0][6] = fmaxf(s_r[0][6], s_r[w][6]);
        }
        float *e = S.ext + (size_t)page * 8;
        const bool any = s_r[0][2] >= s_r[0][0];
        e[0] = any ? s_r[0][0] : 0.f;
        e[1] = any ? s_r[0][1] : 0.f;
        e[2] = (float)kEGrid / (any ? fmaxf(s_r[0][2] - s_r[0][0], 1e-3f) : 1.f);
        e[3] = (float)kEGrid / (any ? fmaxf(s_r[0][3] - s_r[0][1], 1e-3f) : 1.f);
        e[4] = s_r[0][4];
        e[5] = s_r[0][5];
        e[6] = 2e-4f * s_r[0][6] + 2e-3f;  // >= twice the largest per-box prefilter margin of the page
        S.dense[page] = s_bad;
    }
}

__global__ void __launch_bounds__(256) east_bin_count_kernel(const int32_t *__restrict__ counts, int cap, EastScratch S)
{
    ms_pdl_wait();
    const int page = blockIdx.y;
    if (S.dense[page]) return;
    const int K = counts[page];
    const size_t pb = (size_t)page * cap;
    const float *e = S.ext + (size_t)page * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < K; i += gridDim.x * blockDim.x) {
        const float4 b = S.bbox[pb + i];
        const int cell = east_cell(b.y, e[1], e[3]) * kEGrid + east_cell(b.x, e[0], e[2]);
        S.cell_of[pb + i] = cell;
        atomicAdd(S.cell_cnt + (size_t)page * kECells + cell, 1);
    }
}

__global__ void __launch_bounds__(kECells) east_bin_scan_kernel(EastScratch S)
{
    ms_pdl_wait();
    const int page = blockIdx.x;
    __shared__ int s_warp[33];
    const int v = S.cell_cnt[(size_t)page * kECells + threadIdx.x];
    int total;
    const int off = block_excl_scan(v, s_warp, total);
    S.cell_off[(size_t)page * (kECells + 1) + threadIdx.x] = off;
    S.cell_cur[(size_t)page * kECells + threadIdx.x] = off;
    if (threadIdx.x == 0) S.cell_off[(size_t)page * (kECells + 1) + kECells] = total;
}

__global__ void __launch_bounds__(256) east_bin_scatter_kernel(const int32_t *__restrict__ counts, int cap, EastScratch S)
{
    ms_pdl_wait();
    const int page = blockIdx.y;
    if (S.dense[page]) return;
    const int K = counts[page];
    const size_t pb = (size_t)page * cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < K; i += gridDim.x * blockDim.x) {
        const int pos = atomicAdd(S.cell_cur + (size_t)page * kECells + S.cell_of[pb + i], 1);
        S.sb_bbox[pb + pos] = east_inflate(S.bbox[pb + i]);
        S.sb_area[pb + pos] = S.area[pb + i];
        S.sb_id[pb + pos] = i;
    }
}

// 2a) contained-box removal through the grid: box i can only lie inside a box j whose min corner is at most one box
//     size (+ margin) up / left of i's; same classification as the all-pairs kernel below.
__global__ void __launch_bounds__(256) east_contain_binned_kernel(const int32_t *__restrict__ counts, int cap,
                                                                  EastScratch S)
{
    ms_pdl_wait();
    const int page = blockIdx.y;
    if (S.dense[page]) return;
    const int K = counts[page];
    if (K <= 1) return;
    const size_t pb = (size_t)page * cap;
    const float *work = S.work + pb * 9;
    const float *e = S.ext + (size_t)page * 8;
    const int32_t *coff = S.cell_off + (size_t)page * (kECells + 1);
    const float ox = e[0], oy = e[1], sx = e[2], sy = e[3], mw = e[4], mh = e[5], marg = e[6];
    const float eps = (float)1e-6;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < K; i += gridDim.x * blockDim.x) {
        float qi[8];
#pragma unroll
        for (int k = 0; k < 8; k++) qi[k] = work[(size_t)i * 9 + k];
        const float ai = S.area[pb + i];
        const float4 bi = S.bbox[pb + i];
        const int cx0 = east_cell(bi.x - mw - marg, ox, sx), cx1 = east_cell(bi.x + marg, ox, sx);
        const int cy0 = east_cell(bi.y - mh - marg, oy, sy), cy1 = east_cell(bi.y + marg, oy, sy);
        bool later_hit = false, earlier_hit = false;
        for (int cy = cy0; cy <= cy1 && !later_hit; cy++) {
            const int pos1 = coff[cy * kEGrid + cx1 + 1];
            for (int pos = coff[cy * kEGrid + cx0]; pos < pos1; pos++) {
                const float aj = S.sb_area[pb + pos];
                const float4 bj = S.sb_bbox[pb + pos];
                if ((aj + eps < ai) || !(bi.x >= bj.x && bi.y >= bj.y && bi.z <= bj.z && bi.w <= bj.w)) continue;
                const int j = S.sb_id[pb + pos];
                if (j == i) continue;
                float qj[8];
#pragma unroll
                for (int k = 0; k < 8; k++) qj[k] = work[(size_t)j * 9 + k];
                if (!quad_inside(qi, qj)) continue;
                if (area_before(ai, i, aj, j)) {  // j is visited after i: still kept when i is visited
                    later_hit = true;
                    break;
                }
                earlier_hit = true;  // j's own fate decides
            }
        }
        S.removed[pb + i] = later_hit ? 1 : 0;
        S.needseq[pb + i] = (!later_hit && earlier_hit) ? 1 : 0;
    }
}

// 2) infer.py:194-214 contained-box removal, the pairwise part.  Box i is visited in ascending-area order
//    (stable ties); a container j that comes LATER in that order is still kept when i is visited, so it
//    removes i outright; a container that comes EARLIER only counts if it survived itself -> needseq.
//    cv2.pointPolygonTest >= 0 implies the point lies inside the contour's vertex bounding box (the ray
//    cast skips every edge otherwise), so bbox containment is an exact prefilter; the tiny margin only
//    guards the sign of its double-precision cross product next to a vertex.
constexpr int kContainThreads = 256;

__global__ void __launch_bounds__(kContainThreads) east_contain_kernel(const int32_t *__restrict__ counts, int cap,
                                                                       EastScratch S)
{
    ms_pdl_wait();
    const int page = blockIdx.y;
    if (!S.dense[page]) return;  // the grid search handled this page
    const int K = counts[page];
    if (K <= 1) return;
    const size_t pb = (size_t)page * cap;
    const float *work = S.work + pb * 9;
    const float *area = S.area + pb;
    const float4 *bbox = S.bbox + pb;
    __shared__ float4 s_bb[kContainThreads];
    __shared__ float s_ar[kContainThreads];
    const float eps = (float)1e-6;
    for (int base_i = blockIdx.x * kContainThreads; base_i < K; base_i += gridDim.x * kContainThreads) {
        const int i = base_i + threadIdx.x;
        const bool live = i < K;
        float qi[8];
        float ai = 0.f;
        float4 bi = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live) {
#pragma unroll
            for (int k = 0; k < 8; k++) qi[k] = work[(size_t)i * 9 + k];
            ai = area[i];
            bi = bbox[i];
        }
        bool later_hit = false, earlier_hit = false;
        for (int base_j = 0; base_j < K; base_j += kContainThreads) {
            __syncthreads();
            const int jj = base_j + threadIdx.x;
            if (jj < K) {
                s_bb[threadIdx.x] = east_inflate(bbox[jj]);
                s_ar[threadIdx.x] = area[jj];
            }
            __syncthreads();
            if (!live || later_hit) continue;
            const int nj = min(kContainThreads, K - base_j);
            // branch-free prefilter, 4 candidates per trip; the exact test runs only for the rare survivors
#pragma unroll 4
            for (int t = 0; t < nj; t++) {
                const float aj = s_ar[t];
                const float4 bj = s_bb[t];
                const bool cand = !(aj + eps < ai) &&  // infer.py:208
                                  bi.x >= bj.x && bi.y >= bj.y && bi.z <= bj.z && bi.w <= bj.w;
                if (cand) {
                    const int j = base_j + t;
                    if (j != i && !later_hit) {
                        float qj[8];
#pragma unroll
                        for (int k = 0; k < 8; k++) qj[k] = work[(size_t)j * 9 + k];
                        if (quad_inside(qi, qj)) {
                            if (area_before(ai, i, aj, j))
                                later_hit = true;  // j is visited after i: still kept when i is visited
                            else
                                earlier_hit = true;  // j's own fate decides
                        }
                    }
                }
            }
        }
        if (live) {
            S.removed[pb + i] = later_hit ? 1 : 0;
            S.needseq[pb + i] = (!later_hit && earlier_hit) ? 1 : 0;
        }
    }
}

// 3) one CTA per page: the rare sequential leftovers, then anomaly removal -> axis align -> write.
__global__ void __launch_bounds__(1024) east_finish_kernel(const int32_t *__restrict__ counts, int cap,
                                                          ms_east_params P, EastScratch S, float *__restrict__ out,
                                                          int out_cap, int32_t *__restrict__ counts_out,
                                                          int32_t *__restrict__ flags)
{
    ms_pdl_wait();
    const int page = blockIdx.x;
    const int K = counts[page];
    const size_t pb = (size_t)page * cap;
    const float *work = S.work + pb * 9;
    const float *area = S.area + pb;
    int32_t *kidx = S.kidx + pb, *seq = S.seq + pb;
    uint8_t *removed = S.removed + pb;
    const uint8_t *needseq = S.needseq + pb;
    float *karea = S.karea + pb, *kdev = S.kdev + pb;
    __shared__ int s_warp[33];
    __shared__ int s_flag;
    __shared__ float s_thr;
    __shared__ int s_apply;
    const float eps = (float)1e-6;

    // boxes whose only containers precede them in the scan (near-equal areas, duplicates): gather them,
    // order them by area rank and resolve each one cooperatively
    int NS = 0;
    for (int base = 0; base < K; base += blockDim.x) {
        int i = base + threadIdx.x;
        int k = (i < K && needseq[i]) ? 1 : 0;
        int total;
        int pos = block_excl_scan(k, s_warp, total);
        if (k) kidx[NS + pos] = i;
        NS += total;
    }
    __syncthreads();
    if (NS > 0) {
        for (int t = threadIdx.x; t < NS; t += blockDim.x) {
            const int i = kidx[t];
            const float ai = area[i];
            int r = 0;
            for (int u = 0; u < NS; u++) {
                const int j = kidx[u];
                r += (j != i && area_before(area[j], j, ai, i)) ? 1 : 0;
            }
            seq[r] = i;
        }
        __syncthreads();
        for (int r = 0; r < NS; r++) {
            const int i = seq[r];
            if (threadIdx.x == 0) s_flag = 0;
            __syncthreads();
            float qi[8];
#pragma unroll
            for (int k = 0; k < 8; k++) qi[k] = work[(size_t)i * 9 + k];
            const float ai = area[i];
            bool hit = false;
            for (int j = threadIdx.x; j < K && !hit; j += blockDim.x) {
                if (j == i || removed[j]) continue;
                const float aj = area[j];
                if (!area_before(aj, j, ai, i)) continue;  // later boxes were handled by the pairwise pass
                if (aj + eps < ai) continue;
                float qj[8];
#pragma unroll
                for (int k = 0; k < 8; k++) qj[k] = work[(size_t)j * 9 + k];
                hit = quad_inside(qi, qj);
            }
            if (hit) s_flag = 1;
            __syncthreads();
            if (threadIdx.x == 0) removed[i] = s_flag ? 1 : 0;
            __syncthreads();
        }
    }

    // compaction 1 (original order)
    int K1 = 0;
    for (int base = 0; base < K; base += blockDim.x) {
        int i = base + threadIdx.x;
        int k = (i < K && !removed[i]) ? 1 : 0;
        int total;
        int pos = block_excl_scan(k, s_warp, total);
        if (k) {
            kidx[K1 + pos] = i;
            karea[K1 + pos] = area[i];
        }
        K1 += total;
    }
    __syncthreads();

    // infer.py:216-233 area anomalies: numpy f32 mean / std (pairwise sums), threshold in f32
    if (threadIdx.x == 0) s_apply = 0;
    __syncthreads();
    if (P.remove_area_anomalies && K1 > 0 && K1 > P.anomaly_min_box_count) {
        __shared__ int s_loff[kPwLeafCap], s_llen[kPwLeafCap], s_pwcnt;
        __shared__ float s_lsum[kPwLeafCap], s_pwout;
        const float mean32 = np_pairwise_f32_cta(karea, K1, s_loff, s_llen, s_lsum, &s_pwcnt, &s_pwout) / (float)K1;
        for (int i = threadIdx.x; i < K1; i += blockDim.x) {
            float d = karea[i] - mean32;
            kdev[i] = d * d;
        }
        __syncthreads();
        const float var32 = np_pairwise_f32_cta(kdev, K1, s_loff, s_llen, s_lsum, &s_pwcnt, &s_pwout) / (float)K1;
        if (threadIdx.x == 0) {
            float std32 = sqrtf(var32);
            double stdv = (double)std32;
            if (stdv != 0.0) {
                double thr = (double)mean32 + P.anomaly_sigma_threshold * stdv;
                s_thr = (float)thr;
                s_apply = 1;
            }
        }
        __syncthreads();
        if (s_apply) {
            // `if not np.any(keep): return quads`
            if (threadIdx.x == 0) s_flag = 0;
            __syncthreads();
            bool any = false;
            for (int i = threadIdx.x; i < K1; i += blockDim.x) any = any || (karea[i] <= s_thr);
            if (any) s_flag = 1;
            __syncthreads();
            if (threadIdx.x == 0 && !s_flag) s_apply = 0;
            __syncthreads();
        }
    }
    const bool apply = s_apply != 0;
    const float athr = s_thr;

    // compaction 2 + infer.py:149-172 axis alignment, write (rows beyond out_cap are dropped and flagged)
    int K2 = 0;
    for (int base = 0; base < K1; base += blockDim.x) {
        int t = base + threadIdx.x;
        int k = (t < K1 && (!apply || karea[t] <= athr)) ? 1 : 0;
        int total;
        int pos = block_excl_scan(k, s_warp, total);
        if (k && K2 + pos < out_cap) {
            const float *q = work + (size_t)kidx[t] * 9;
            float *o = out + ((size_t)page * out_cap + K2 + pos) * 9;
            if (P.axis_aligned_output) {
                float x0 = q[0], x1 = q[0], y0 = q[1], y1 = q[1];
#pragma unroll
                for (int v = 1; v < 4; v++) {
                    x0 = q[2 * v] < x0 ? q[2 * v] : x0;
                    x1 = q[2 * v] > x1 ? q[2 * v] : x1;
                    y0 = q[2 * v + 1] < y0 ? q[2 * v + 1] : y0;
                    y1 = q[2 * v + 1] > y1 ? q[2 * v + 1] : y1;
                }
                o[0] = x0; o[1] = y0; o[2] = x1; o[3] = y0;
                o[4] = x1; o[5] = y1; o[6] = x0; o[7] = y1;
            } else {
#pragma unroll
                for (int k2 = 0; k2 < 8; k2++) o[k2] = q[k2];
            }
            o[8] = q[8];
        }
        K2 += total;
    }
    if (threadIdx.x == 0) {
        if (K2 > out_cap) {
            if (flags) atomicOr(flags + page, MS_FLAG_CAND_OVERFLOW);
            K2 = out_cap;
        }
        counts_out[page] = K2;
    }
}

// ---- _pipeline.py:125-137, 204-221 ---------------------------------------------------------------------
__device__ __forceinline__ int py_slice(int start, int stop, int dim, int &s_out)
{
    if (start < 0) {
        start += dim;
        if (start < 0) start = 0;
    } else if (start > dim)
        start = dim;
    if (stop < 0) {
        stop += dim;
        if (stop < 0) stop = 0;
    } else if (stop > dim)
        stop = dim;
    s_out = start;
    return stop > start ? stop - start : 0;
}

__device__ __forceinline__ int f2i_trunc(float v)
{
    // np.array(list of python floats, dtype=int32): C cast; out-of-range / NaN is undefined there --
    // x86 yields INT_MIN, reproduced here
    if (!(v > -2147483904.0f && v < 2147483648.0f)) return INT_MIN;
    return (int)v;
}

__device__ __forceinline__ bool word_rect(const float *q, int img_h, int img_w, int min_text, int *rect)
{
    int xmin, xmax, ymin, ymax;
    xmin = xmax = f2i_trunc(q[0]);
    ymin = ymax = f2i_trunc(q[1]);
#pragma unroll
    for (int v = 1; v < 4; v++) {
        int x = f2i_trunc(q[2 * v]), y = f2i_trunc(q[2 * v + 1]);
        xmin = min(xmin, x);
        xmax = max(xmax, x);
        ymin = min(ymin, y);
        ymax = max(ymax, y);
    }
    rect[0] = rect[1] = rect[2] = rect[3] = 0;
    // numpy int32 subtraction wraps; widths here are far from overflow on every supported input
    if (!((long long)xmax - xmin >= min_text && (long long)ymax - ymin >= min_text)) return false;
    int x1 = max(0, xmin), y1 = max(0, ymin);
    int x2 = min(img_w, xmax), y2 = min(img_h, ymax);
    int sx, sy;
    int w = py_slice(x1, x2, img_w, sx);
    int h = py_slice(y1, y2, img_h, sy);
    if (w <= 0 || h <= 0) return false;
    rect[0] = sx;
    rect[1] = sy;
    rect[2] = sx + w;
    rect[3] = sy + h;
    return true;
}

__global__ void word_rects_flat_kernel(const float *__restrict__ polys8, int64_t n, int img_h, int img_w, int min_text,
                                       int32_t *__restrict__ rects, uint8_t *__restrict__ valid)
{
    ms_pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float q[8];
#pragma unroll
        for (int k = 0; k < 8; k++) q[k] = polys8[i * 8 + k];
        int r[4];
        bool ok = word_rect(q, img_h, img_w, min_text, r);
#pragma unroll
        for (int k = 0; k < 4; k++) rects[i * 4 + k] = r[k];
        valid[i] = ok ? 1 : 0;
    }
}

// one CTA per page: ordered compaction of valid crops into a page-strided temp list
__global__ void __launch_bounds__(1024) word_rects_page_kernel(const float *__restrict__ quads,
                                                              const int32_t *__restrict__ counts, int cap,
                                                              const int32_t *__restrict__ img_hw, int img_h, int img_w,
                                                              int min_text, int32_t *__restrict__ tmp,
                                                              int32_t *__restrict__ page_n)
{
    ms_pdl_wait();
    const int page = blockIdx.x;
    const int K = counts[page];
    const size_t pb = (size_t)page * cap;
    if (img_hw) {
        img_h = img_hw[2 * page];
        img_w = img_hw[2 * page + 1];
    }
    __shared__ int s_warp[33];
    int run = 0;
    for (int base = 0; base < K; base += blockDim.x) {
        int i = base + threadIdx.x;
        int r[4] = {0, 0, 0, 0};
        int ok = 0;
        if (i < K) {
            float q[8];
#pragma unroll
            for (int k = 0; k < 8; k++) q[k] = quads[(pb + i) * 9 + k];
            ok = word_rect(q, img_h, img_w, min_text, r) ? 1 : 0;
        }
        int total;
        int pos = block_excl_scan(ok, s_warp, total);
        if (ok) {
            int32_t *d = tmp + (pb + run + pos) * 4;
            d[0] = r[0]; d[1] = r[1]; d[2] = r[2]; d[3] = r[3];
        }
        run += total;
    }
    if (threadIdx.x == 0) page_n[page] = run;
}

// append != 0: this call's crops go after the *n_crops rows already in the list (page chunks of one batch);
// range[0..1] receives the [begin, end) rows this call produced (input of the crop kernels)
__global__ void word_rects_offsets_kernel(const int32_t *__restrict__ page_n, int n_pages, int32_t *page_off,
                                          int64_t crops_cap, int32_t *n_crops, int append, int32_t *range)
{
    ms_pdl_wait();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        long long run = append ? *n_crops : 0;
        const long long begin = run > crops_cap ? crops_cap : run;
        for (int p = 0; p < n_pages; p++) {
            page_off[p] = (int32_t)run;
            run += page_n[p];
        }
        page_off[n_pages] = (int32_t)run;
        const long long end = run > crops_cap ? crops_cap : run;
        *n_crops = (int32_t)end;
        if (range) {
            range[0] = (int32_t)begin;
            range[1] = (int32_t)end;
        }
    }
}

__global__ void word_rects_pack_kernel(const int32_t *__restrict__ tmp, const int32_t *__restrict__ page_n,
                                       const int32_t *__restrict__ page_off, int n_pages, int cap, int64_t crops_cap,
                                       int page_base, int32_t *__restrict__ crops)
{
    ms_pdl_wait();
    size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int p = (int)(g / cap), i = (int)(g % cap);
    if (p >= n_pages || i >= page_n[p]) return;
    int64_t dst = (int64_t)page_off[p] + i;
    if (dst >= crops_cap) return;
    const int32_t *s = tmp + ((size_t)p * cap + i) * 4;
    int32_t *d = crops + dst * 5;
    d[0] = page_base + p; d[1] = s[0]; d[2] = s[1]; d[3] = s[2]; d[4] = s[3];
}

void carve_east(ms_bump &bump, EastScratch &S, size_t n)
{
    S.work = bump.take<float>(n * 9);
    S.area = bump.take<float>(n);
    S.bbox = bump.take<float4>(n);
    S.removed = bump.take<uint8_t>(n);
    S.needseq = bump.take<uint8_t>(n);
    S.seq = bump.take<int32_t>(n);
    S.karea = bump.take<float>(n);
    S.kdev = bump.take<float>(n);
    S.kidx = bump.take<int32_t>(n);
    S.cell_of = bump.take<int32_t>(n);
    S.sb_bbox = bump.take<float4>(n);
    S.sb_area = bump.take<float>(n);
    S.sb_id = bump.take<int32_t>(n);
}

void carve_east_pages(ms_bump &bump, EastScratch &S, int n_pages)
{
    S.ext = bump.take<float>((size_t)n_pages * 8);
    S.dense = bump.take<int32_t>(n_pages);
    S.cell_cnt = bump.take<int32_t>((size_t)n_pages * kECells);
    S.cell_off = bump.take<int32_t>((size_t)n_pages * (kECells + 1));
    S.cell_cur = bump.take<int32_t>((size_t)n_pages * kECells);
}

}  // namespace

int msk_expand(ms_ctx *ctx, const float *quads, int64_t n, double ew, double eh, float *out, cudaStream_t st)
{
    if (n <= 0) return MS_OK;
    int grid = (int)((n + 127) / 128);
    if (grid > ctx->num_sms * 8) grid = ctx->num_sms * 8;
    ms_launch(expand_kernel, grid, 128, 0, st, quads, n, ew, eh, out);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}

size_t msk_east_boxes_scratch(int n_pages, int cap_per_page)
{
    ms_bump probe{nullptr, 0, 0};
    EastScratch S;
    carve_east(probe, S, (size_t)n_pages * cap_per_page);
    carve_east_pages(probe, S, n_pages);
    return probe.off + 4096;
}

int msk_east_boxes(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                   const ms_east_params *p, const int32_t *orig_hw, float *quads_out, int out_cap, int32_t *counts_out,
                   int32_t *flags, ms_bump bump, cudaStream_t st, int orig_h, int orig_w)
{
    if (n_pages <= 0) return MS_OK;
    if (!p || p->target_size <= 0 || out_cap <= 0) {
        ms_set_error("east_boxes: bad params");
        return MS_ERR_INVALID;
    }
    EastScratch S;
    carve_east(bump, S, (size_t)n_pages * cap_per_page);
    carve_east_pages(bump, S, n_pages);
    if (!S.sb_id || !S.cell_cur) {
        ms_set_error("east_boxes: scratch too small");
        return MS_ERR_CAPACITY;
    }
    // counts live on the device: grids are sized for a few thousand boxes per page and stride beyond that
    int gx = (cap_per_page + 255) / 256;
    if (gx > 16) gx = 16;
    ms_launch(east_prep_kernel, dim3(gx, n_pages), 256, 0, st, quads, counts, n_pages, cap_per_page, *p, orig_hw, orig_h, orig_w, S);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(east_ext_kernel, n_pages, 256, 0, st, counts, cap_per_page, S);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(east_bin_count_kernel, dim3(gx, n_pages), 256, 0, st, counts, cap_per_page, S);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(east_bin_scan_kernel, n_pages, kECells, 0, st, S);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(east_bin_scatter_kernel, dim3(gx, n_pages), 256, 0, st, counts, cap_per_page, S);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(east_contain_binned_kernel, dim3(gx * 2, n_pages), 256, 0, st, counts, cap_per_page, S);
    MS_LAUNCH_CHECK(ctx);
    gx = (cap_per_page + kContainThreads - 1) / kContainThreads;
    if (gx > 32) gx = 32;
    ms_launch(east_contain_kernel, dim3(gx, n_pages), kContainThreads, 0, st, counts, cap_per_page, S);  // dense pages only
    MS_LAUNCH_CHECK(ctx);
    // device recursion in np_pairwise_f32: depth <= log2(cap/128) + 1 frames of a few dozen bytes
    ms_launch(east_finish_kernel, n_pages, 1024, 0, st, counts, cap_per_page, *p, S, quads_out, out_cap, counts_out, flags);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}

size_t msk_word_rects_scratch(int n_pages) { return (size_t)(2 * n_pages + 2) * sizeof(int32_t) + 1024; }

// NOTE: the page-strided temp list (n_pages*cap*4 int32) is taken from the bump as well.
int msk_word_rects(ms_ctx *ctx, const float *quads, const int32_t *counts, int n_pages, int cap_per_page,
                   const int32_t *img_hw, int img_h, int img_w, int min_text_size, int32_t *crops_out,
                   int64_t crops_cap, int32_t *n_crops, int page_base, int append, int32_t *range, ms_bump bump,
                   cudaStream_t st)
{
    if (n_pages <= 0) return MS_OK;
    int32_t *page_n = bump.take<int32_t>(n_pages);
    int32_t *page_off = bump.take<int32_t>(n_pages + 1);
    int32_t *tmp = bump.take<int32_t>((size_t)n_pages * cap_per_page * 4);
    if (!tmp) {
        ms_set_error("word_rects: scratch too small");
        return MS_ERR_CAPACITY;
    }
    ms_launch(word_rects_page_kernel, n_pages, 1024, 0, st, quads, counts, cap_per_page, img_hw, img_h, img_w, min_text_size,
                                                    tmp, page_n);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(word_rects_offsets_kernel, 1, 32, 0, st, page_n, n_pages, page_off, crops_cap, n_crops, append, range);
    MS_LAUNCH_CHECK(ctx);
    size_t threads = (size_t)n_pages * cap_per_page;
    ms_launch(word_rects_pack_kernel, (int)((threads + 255) / 256), 256, 0, st, tmp, page_n, page_off, n_pages, cap_per_page,
                                                                         crops_cap, page_base, crops_out);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}

int msk_word_rects_flat(ms_ctx *ctx, const float *polys8, int64_t n, int img_h, int img_w, int min_text_size,
                        int32_t *rects, uint8_t *valid, cudaStream_t st)
{
    if (n <= 0) return MS_OK;
    int grid = (int)((n + 127) / 128);
    if (grid > ctx->num_sms * 8) grid = ctx->num_sms * 8;
    ms_launch(word_rects_flat_kernel, grid, 128, 0, st, polys8, n, img_h, img_w, min_text_size, rects, valid);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}
