// Reading-order sort of a page's word boxes on the device -- the host logic that sits between NMS and the crop
// loop in the reference (SURVEY 8f-1): resolve_intersections / sort_boxes_reading_order /
// sort_boxes_reading_order_with_resolutions (reference detectors/_east/utils.py:500-644) and the word re-matching
// of Pipeline.predict (_pipeline.py:105-123).  Result for result identical, including the quirks (the dict that
// keeps the LAST box of equal compressed coordinates, the re-match that picks the FIRST word of equal integer box).
//
// The reference's shrink loop is a sequential recurrence over (i, j) pairs in index order.  Two facts make it cheap
// without changing a single step: boxes only ever shrink towards their top-left corner, so a pair that does not
// intersect initially never does (the sweeps visit only the initially intersecting pairs, in the reference's order,
// and drop pairs that stopped intersecting); box centres are multiples of 0.5, so per-line means are exact integer
// sums divided once.  Within a sweep two pairs commute unless they share a box: every pair gets a dependency level
// (1 + the level of the latest earlier pair touching either of its boxes) and the pairs of one level are applied in
// parallel -- any order that respects the levels reproduces the sequential sweep.
//
// One CTA (1024 threads) orders a page in phases: A integer boxes; B the initially intersecting pairs from a grid over
// the page; C levels by parallel relaxation, sweeps over level buckets (one thread sweeps chains deeper than the level
// limit); D line assignment 32 boxes at a time (only the newest line can match -- see D3) and two bitonic sorts; E the
// dict / first-match quirks, behind a hash-table check that two boxes coincide at all.  The phases are written once
// (ro_* below) and run in two storage configurations:
//   RoSmemCfg    reading_order_kernel, one CTA per page of up to 4096 boxes and 28 672 intersecting pairs: 16-bit
//                indices, boxes / pairs / levels in shared memory (the sort and line arrays of D and E overlay the
//                pair region), the transposed pair list and the level buckets in per-page global scratch.  0.39 ms per
//                64 pages of 2000 boxes on a B200 (2.4 ms before these restructurings).
//   RoGlobalCfg  reading_order_large_kernel, for the pages beyond that: 32-bit indices, every array in a global scratch
//                slot (L2-resident: a 10 000-box page needs ~3 MB), shared memory holding whichever of the boxes (B),
//                levels (C) and sort keys (D) fits.  ~2 ms for a 10 000-box page instead of ~100 ms of host Python.
#include "ms_internal.cuh"

namespace {

constexpr int kRoThreads = 1024;
constexpr int kRoMaxBoxes = 4096;   // boxes per page held in shared memory
constexpr int kRoMaxPairs = 28672;  // initially intersecting pairs per page
constexpr int kRoGridCap = 12288;   // (box, cell) registrations of the pair-generation grid (24 KB of shared memory)

// the shared-memory kernel's page
struct RoSmemCfg {
    using Idx = uint16_t;   // box and pair indices
    using Pair = uint32_t;  // (i << 16) | j
    using Level = uint8_t;
    static constexpr Idx kNone = 0xffffu;
    static constexpr int kCells = 32;          // pair-generation grid: cells per axis
    static constexpr int kGridMinBoxes = 256;  // fewer boxes: all pairs are tested
    static constexpr int kMaxLevels = 255;     // dependency levels of the parallel sweeps
    static constexpr int kKeyBits = 12;        // box index bits of the sort keys
    static constexpr bool kPrevI = false;      // relaxation finds a pair's predecessor on its first box inline
    static __device__ __forceinline__ Pair pair(int i, int j) { return ((uint32_t)i << 16) | (uint32_t)j; }
    static __device__ __forceinline__ int first(Pair p) { return (int)(p >> 16); }
    static __device__ __forceinline__ int second(Pair p) { return (int)(p & 0xffffu); }
};

// the global-memory kernel's page
struct RoGlobalCfg {
    using Idx = uint32_t;
    using Pair = uint2;
    using Level = uint16_t;
    static constexpr Idx kNone = 0xffffffffu;
    static constexpr int kCells = 64;
    static constexpr int kGridMinBoxes = 0;
    static constexpr int kMaxLevels = 4095;
    static constexpr int kKeyBits = 20;
    static constexpr bool kPrevI = true;  // relaxation reads a precomputed predecessor list, four pairs per thread in flight
    static __device__ __forceinline__ Pair pair(int i, int j) { return make_uint2((uint32_t)i, (uint32_t)j); }
    static __device__ __forceinline__ int first(Pair p) { return (int)p.x; }
    static __device__ __forceinline__ int second(Pair p) { return (int)p.y; }
};

// scalars of the page routine shared by the CTA
struct RoShared {
    int warp[33];
    int g[4];  // hull of all boxes
    int np, lines, avg_pos, changed, maxl, dup;
    long long hsum;
    double ytol;
};

// the page's arrays; each kernel places them (several share storage in phases where they are not live)
template <class Cfg>
struct RoArrays {
    using Idx = typename Cfg::Idx;
    int4 *box;         // A-E: the boxes, shrunk by the sweeps
    const int4 *bxs;   // B: the boxes the pair generation reads (box, or a copy in faster memory)
    typename Cfg::Pair *pairs;
    typename Cfg::Level *lv;  // C: dependency level per pair (0: dropped)
    Idx *row_cnt, *row_start;  // B: pairs per first box, first pair of each row
    int *ccnt;                 // B: cell counters / fill cursors
    Idx *cstart, *centry;      // B: cell starts, box indices per cell
    Idx *T, *prevJ, *lastJ;    // C: pair list transposed (then bucketed by level), predecessor on the second box
    int *bcnt, *bstart;        // C: transposed bucket sizes / fill cursors, bucket starts
    int *lend;                 // C: pairs per level, then level bucket ends (fill cursors while the buckets fill)
    long long *line_sum;       // D: per line, sum of y0 + y1
    double *line_cy;           // D: per line, mean centre
    int *line_cnt;             // D: per line, members
    Idx *line_rank, *line_of, *seq_of;
    uint32_t *htab;            // E
    int pair_cap, grid_cap;
};

__device__ __forceinline__ int ro_trunc(float v)
{
    // np.array(polygon, dtype=np.int32): C cast of a double; out of range / NaN -> INT_MIN as on x86
    if (!(v > -2147483904.0f && v < 2147483648.0f)) return INT_MIN;
    return (int)v;
}

__device__ __forceinline__ bool ro_intersect(const int4 a, const int4 b)
{
    // utils.py:516-519
    return !(a.z <= b.x || b.z <= a.x || a.w <= b.y || b.w <= a.y);
}

__device__ __forceinline__ int ro_shrink(int lo, int hi)
{
    // int(x1 - (x1 - x0) * 0.1) in Python floats (utils.py:531-542)
    return (int)((double)hi - (double)(hi - lo) * 0.1);
}

__device__ __forceinline__ bool ro_equal(const int4 a, const int4 b) { return a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w; }

// one step of the shrink loop on pair (i, j) (utils.py:521-545); false when the boxes no longer intersect
__device__ __forceinline__ bool ro_shrink_pair(int4 *box, int i, int j)
{
    int4 a = box[i], c = box[j];
    if (!ro_intersect(a, c)) return false;
    a.z = ro_shrink(a.x, a.z);
    a.w = ro_shrink(a.y, a.w);
    c.z = ro_shrink(c.x, c.z);
    c.w = ro_shrink(c.y, c.w);
    box[i] = a;
    box[j] = c;
    return true;
}

__device__ __forceinline__ int ro_block_scan(int v, int *s_warp, int &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
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
        int w = s_warp[lane];
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

// exclusive scan of in[0..n) into out[0..n) (in == out allowed), each start clamped to `clamp`; returns the total
template <class In, class Out>
__device__ __forceinline__ long long ro_scan(const In *in, Out *out, int n, int *s_warp, long long clamp = LLONG_MAX)
{
    long long run = 0;
    for (int base = 0; base < n; base += kRoThreads) {
        const int i = base + threadIdx.x;
        const int c = i < n ? (int)in[i] : 0;
        int total;
        const int off = ro_block_scan(c, s_warp, total);
        if (i < n) out[i] = (Out)min(run + off, clamp);
        run += total;
    }
    __syncthreads();
    return run;
}

__device__ __forceinline__ void ro_bitonic(uint64_t *keys, int n)
{
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += kRoThreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint64_t a = keys[i], b = keys[ixj];
                    if ((a > b) == ((i & k) == 0)) {
                        keys[i] = b;
                        keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
}

// bitonic sort of (k1, k2) tuples, ascending
__device__ __forceinline__ void ro_bitonic2(uint64_t *k1, uint32_t *k2, int n)
{
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += kRoThreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint64_t a1 = k1[i], b1 = k1[ixj];
                    const uint32_t a2 = k2[i], b2 = k2[ixj];
                    const bool gt = a1 > b1 || (a1 == b1 && a2 > b2);
                    if (gt == ((i & k) == 0)) {
                        k1[i] = b1;
                        k1[ixj] = a1;
                        k2[i] = b2;
                        k2[ixj] = a2;
                    }
                }
            }
            __syncthreads();
        }
    }
}

// orderable image of a double (ascending), NaN last
__device__ __forceinline__ uint64_t ro_orderable(double d)
{
    if (d != d) return ~0ull;
    if (d == 0.0) d = 0.0;
    uint64_t u = (uint64_t)__double_as_longlong(d);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// A. integer boxes (_pipeline.py:105-109) into box and obox, and into `copy` unless that is box
__device__ __forceinline__ void ro_int_boxes(const float *__restrict__ boxes8, int row_stride, int K, size_t pb, int4 *box,
                                             int4 *obox, int4 *copy)
{
    for (int k = threadIdx.x; k < K; k += kRoThreads) {
        const float *q = boxes8 + (pb + k) * row_stride;
        int xmin, xmax, ymin, ymax;
        xmin = xmax = ro_trunc(q[0]);
        ymin = ymax = ro_trunc(q[1]);
#pragma unroll
        for (int v = 1; v < 4; v++) {
            const int x = ro_trunc(q[2 * v]), y = ro_trunc(q[2 * v + 1]);
            xmin = min(xmin, x);
            xmax = max(xmax, x);
            ymin = min(ymin, y);
            ymax = max(ymax, y);
        }
        const int4 b = make_int4(xmin, ymin, xmax, ymax);
        box[k] = b;
        obox[k] = b;
        if (copy != box) copy[k] = b;
    }
    __syncthreads();
}

// B. initially intersecting pairs (i < j) in (i, j) order: count, scan, fill.
//    Candidates come from a kCells x kCells grid over the page (power-of-two cells): every box is registered in the
//    cells its hull touches, row i tests only the boxes registered in its cells, and a pair found in several cells is
//    taken in the one that holds (max x0, max y0) -- a point of both hulls whenever the two boxes intersect.  Rows come
//    out in cell order and are sorted by j afterwards.  Pages with fewer than kGridMinBoxes boxes, a box over more than
//    64 cells (page-sized boxes) or more registrations than grid_cap test all pairs instead.
//    Returns false, uniformly over the CTA, when the page has more than pair_cap pairs.
template <class Cfg>
__device__ __forceinline__ bool ro_pairs(const RoArrays<Cfg> &A, RoShared &S, int K)
{
    using Idx = typename Cfg::Idx;
    constexpr int kCells = Cfg::kCells, NC = kCells * kCells;
    const int4 *bxs = A.bxs;
    bool grid = K >= Cfg::kGridMinBoxes;
    int gx0 = 0, gy0 = 0, shx = 0, shy = 0;
    if (grid) {
        if (threadIdx.x == 0) {
            S.g[0] = S.g[1] = INT_MAX;
            S.g[2] = S.g[3] = INT_MIN;
        }
        for (int t = threadIdx.x; t < NC; t += kRoThreads) A.ccnt[t] = 0;
        __syncthreads();
        int mnx = INT_MAX, mny = INT_MAX, mxx = INT_MIN, mxy = INT_MIN;
        for (int i = threadIdx.x; i < K; i += kRoThreads) {
            const int4 b = bxs[i];
            mnx = min(mnx, min(b.x, b.z));
            mxx = max(mxx, max(b.x, b.z));
            mny = min(mny, min(b.y, b.w));
            mxy = max(mxy, max(b.y, b.w));
        }
        mnx = __reduce_min_sync(0xffffffffu, mnx);
        mny = __reduce_min_sync(0xffffffffu, mny);
        mxx = __reduce_max_sync(0xffffffffu, mxx);
        mxy = __reduce_max_sync(0xffffffffu, mxy);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&S.g[0], mnx);
            atomicMin(&S.g[1], mny);
            atomicMax(&S.g[2], mxx);
            atomicMax(&S.g[3], mxy);
        }
        __syncthreads();
        gx0 = S.g[0];
        gy0 = S.g[1];
        const uint32_t ex = (uint32_t)S.g[2] - (uint32_t)gx0, ey = (uint32_t)S.g[3] - (uint32_t)gy0;
        while ((ex >> shx) >= (uint32_t)kCells) shx++;
        while ((ey >> shy) >= (uint32_t)kCells) shy++;
    }
    auto cell_x = [&](int x) { return (int)(((uint32_t)x - (uint32_t)gx0) >> shx); };
    auto cell_y = [&](int y) { return (int)(((uint32_t)y - (uint32_t)gy0) >> shy); };
    if (grid) {
        int mine = 0, big = 0;
        for (int i = threadIdx.x; i < K; i += kRoThreads) {
            const int4 b = bxs[i];
            const int cx0 = cell_x(min(b.x, b.z)), cx1 = cell_x(max(b.x, b.z));
            const int cy0 = cell_y(min(b.y, b.w)), cy1 = cell_y(max(b.y, b.w));
            const int nc = (cx1 - cx0 + 1) * (cy1 - cy0 + 1);
            if (nc <= 64) {
                mine += nc;
                for (int cy = cy0; cy <= cy1; cy++)
                    for (int cx = cx0; cx <= cx1; cx++) atomicAdd(&A.ccnt[cy * kCells + cx], 1);
            } else {
                big = 1;  // a box over more than 64 cells: not worth a grid
            }
        }
        int total_e;
        ro_block_scan(mine, S.warp, total_e);
        grid = !__syncthreads_or(big) && total_e <= A.grid_cap;
        if (grid) {
            const int total_c = (int)ro_scan(A.ccnt, A.cstart, NC, S.warp);
            if (threadIdx.x == 0) A.cstart[NC] = (Idx)total_c;
            for (int t = threadIdx.x; t < NC; t += kRoThreads) A.ccnt[t] = 0;
            __syncthreads();
            for (int i = threadIdx.x; i < K; i += kRoThreads) {
                const int4 b = bxs[i];
                const int cx0 = cell_x(min(b.x, b.z)), cx1 = cell_x(max(b.x, b.z));
                const int cy0 = cell_y(min(b.y, b.w)), cy1 = cell_y(max(b.y, b.w));
                for (int cy = cy0; cy <= cy1; cy++)
                    for (int cx = cx0; cx <= cx1; cx++) {
                        const int c = cy * kCells + cx;
                        A.centry[(int)A.cstart[c] + atomicAdd(&A.ccnt[c], 1)] = (Idx)i;
                    }
            }
            __syncthreads();
        }
    }
    // one pass over row i's candidates: counts them, or writes them from `off` on
    auto row_pass = [&](int i, int off, bool write) -> int {
        const int4 bi = bxs[i];
        int cnt = 0;
        if (grid) {
            const int cx0 = cell_x(min(bi.x, bi.z)), cx1 = cell_x(max(bi.x, bi.z));
            const int cy0 = cell_y(min(bi.y, bi.w)), cy1 = cell_y(max(bi.y, bi.w));
            for (int cy = cy0; cy <= cy1; cy++)
                for (int cx = cx0; cx <= cx1; cx++) {
                    const int c = cy * kCells + cx;
                    const int e1 = A.cstart[c + 1];
                    for (int e = A.cstart[c]; e < e1; e++) {
                        const int j = (int)A.centry[e];
                        if (j <= i) continue;
                        const int4 bj = bxs[j];
                        if (!ro_intersect(bi, bj)) continue;
                        if (cell_y(max(bi.y, bj.y)) * kCells + cell_x(max(bi.x, bj.x)) != c) continue;  // another cell's
                        if (write && off + cnt < A.pair_cap) A.pairs[off + cnt] = Cfg::pair(i, j);
                        cnt++;
                    }
                }
        } else {
            for (int j = i + 1; j < K; j++) {
                if (!ro_intersect(bi, bxs[j])) continue;
                if (write && off + cnt < A.pair_cap) A.pairs[off + cnt] = Cfg::pair(i, j);
                cnt++;
            }
        }
        return cnt;
    };
    // all pairs: row i tests K - 1 - i boxes, so a thread takes rows t and K - 1 - t (equal work); grid: any order
    const int half = (K + 1) / 2;
    for (int t = threadIdx.x; t < half; t += kRoThreads) {
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const int i = side == 0 ? t : K - 1 - t;
            if (side == 1 && i == t) break;
            A.row_cnt[i] = (Idx)min(row_pass(i, 0, false), A.pair_cap + 1);
        }
    }
    __syncthreads();
    // (each row count is at most pair_cap + 1, so a block's sum fits 32 bits for cap <= 2^16)
    const long long np = ro_scan(A.row_cnt, A.row_start, K, S.warp, A.pair_cap);
    if (np > A.pair_cap) return false;
    for (int t = threadIdx.x; t < half; t += kRoThreads) {
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const int i = side == 0 ? t : K - 1 - t;
            if (side == 1 && i == t) break;
            if (A.row_cnt[i] == 0) continue;
            const int s0 = A.row_start[i];
            row_pass(i, s0, true);
            if (grid) {  // cell order -> ascending j (insertion sort of a short row)
                const int e0 = s0 + (int)A.row_cnt[i];
                for (int a = s0 + 1; a < e0; a++) {
                    const typename Cfg::Pair v = A.pairs[a];
                    int bpos = a - 1;
                    while (bpos >= s0 && Cfg::second(A.pairs[bpos]) > Cfg::second(v)) {
                        A.pairs[bpos + 1] = A.pairs[bpos];
                        bpos--;
                    }
                    A.pairs[bpos + 1] = v;
                }
            }
        }
    }
    if (threadIdx.x == 0) {
        S.np = (int)np;
        A.row_start[K] = (Idx)np;
    }
    __syncthreads();
    return true;
}

// C1. dependency levels (one sequential pass over the pair list in the reference).  The pair before p = (i, j) that
//     touches box i is p - 1 inside row i, else the last pair (a, i) of the earlier rows; the one that touches box j is
//     the pair (a, j) with the largest a < i.  Both come from the pair list transposed (bucketed by second box, each
//     bucket ascending); then the levels l(p) = 1 + max(l(prev_i), l(prev_j)) are relaxed in parallel until a pass
//     changes nothing (monotone, at most max-level passes).  S.maxl: the deepest level, -1 beyond kMaxLevels.
template <class Cfg>
__device__ __forceinline__ void ro_levels(const RoArrays<Cfg> &A, RoShared &S, int K)
{
    using Idx = typename Cfg::Idx;
    constexpr int kMaxLevels = Cfg::kMaxLevels;
    const int np = S.np;
    for (int k = threadIdx.x; k <= K; k += kRoThreads) A.bcnt[k] = 0;
    __syncthreads();
    for (int p = threadIdx.x; p < np; p += kRoThreads) atomicAdd(&A.bcnt[Cfg::second(A.pairs[p])], 1);
    __syncthreads();
    const int run = (int)ro_scan(A.bcnt, A.bstart, K, S.warp);
    for (int k = threadIdx.x; k < K; k += kRoThreads) A.bcnt[k] = 0;
    if (threadIdx.x == 0) {
        A.bstart[K] = run;
        S.maxl = 0;
    }
    __syncthreads();
    for (int p = threadIdx.x; p < np; p += kRoThreads) {
        const int j = Cfg::second(A.pairs[p]);
        A.T[A.bstart[j] + atomicAdd(&A.bcnt[j], 1)] = (Idx)p;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < K; j += kRoThreads) {
        const int s0 = A.bstart[j], e0 = A.bstart[j + 1];
        for (int a = s0 + 1; a < e0; a++) {  // insertion sort of a short bucket
            const Idx v = A.T[a];
            int b = a - 1;
            while (b >= s0 && A.T[b] > v) {
                A.T[b + 1] = A.T[b];
                b--;
            }
            A.T[b + 1] = v;
        }
        for (int a = s0; a < e0; a++) A.prevJ[A.T[a]] = a > s0 ? A.T[a - 1] : Cfg::kNone;
        A.lastJ[j] = e0 > s0 ? A.T[e0 - 1] : Cfg::kNone;
    }
    typename Cfg::Level *lv = A.lv;
    if constexpr (Cfg::kPrevI) {
        __syncthreads();  // the buckets in T have been read: T now holds every pair's predecessor on its first box
        Idx *prevI = A.T;
        for (int p = threadIdx.x; p < np; p += kRoThreads) {
            const int i = Cfg::first(A.pairs[p]);
            prevI[p] = p > (int)A.row_start[i] ? (Idx)(p - 1) : A.lastJ[i];
            lv[p] = 1;
        }
        __syncthreads();
        // a pass walks the pairs four per thread with all index loads, then all level loads, in flight together: the
        // arrays live in L2 and a pass is bound by the latency of those dependent loads
        for (int pass = 0; pass < kMaxLevels + 2; pass++) {
            int changed = 0;
            for (int base = 0; base < np; base += 4 * kRoThreads) {
                Idx pi[4], pj[4];
                int cur[4], a[4], b[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int p = base + u * kRoThreads + (int)threadIdx.x;
                    pi[u] = pj[u] = Cfg::kNone;
                    cur[u] = 0;
                    if (p < np) {
                        pi[u] = prevI[p];
                        pj[u] = A.prevJ[p];
                        cur[u] = (int)lv[p];
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    a[u] = pi[u] == Cfg::kNone ? 0 : (int)lv[pi[u]];
                    b[u] = pj[u] == Cfg::kNone ? 0 : (int)lv[pj[u]];
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int p = base + u * kRoThreads + (int)threadIdx.x;
                    if (p < np) {
                        const int l = 1 + max(a[u], b[u]);
                        if (l > kMaxLevels) {
                            S.maxl = -1;  // too deep for the level buckets: sequential sweeps
                        } else if (l != cur[u]) {
                            lv[p] = (typename Cfg::Level)l;
                            changed = 1;
                        }
                    }
                }
            }
            if (!__syncthreads_or(changed) || S.maxl < 0) break;
        }
    } else {
        for (int p = threadIdx.x; p < np; p += kRoThreads) lv[p] = 1;
        __syncthreads();
        for (int pass = 0; pass < kMaxLevels + 2; pass++) {
            int changed = 0;
            for (int p = threadIdx.x; p < np; p += kRoThreads) {
                const int i = Cfg::first(A.pairs[p]);
                const Idx pi = p > (int)A.row_start[i] ? (Idx)(p - 1) : A.lastJ[i];
                const Idx pj = A.prevJ[p];
                const int a = pi == Cfg::kNone ? 0 : (int)lv[pi], b = pj == Cfg::kNone ? 0 : (int)lv[pj];
                const int l = 1 + max(a, b);
                if (l > kMaxLevels) {
                    S.maxl = -1;  // too deep for the level buckets: sequential sweeps
                } else if (l != (int)lv[p]) {
                    lv[p] = (typename Cfg::Level)l;
                    changed = 1;
                }
            }
            if (!__syncthreads_or(changed) || S.maxl < 0) break;
        }
    }
    if (S.maxl >= 0) {
        int m = 0;
        for (int p = threadIdx.x; p < np; p += kRoThreads) m = max(m, (int)lv[p]);
        m = __reduce_max_sync(0xffffffffu, m);
        if ((threadIdx.x & 31) == 0) atomicMax(&S.maxl, m);
    }
    __syncthreads();
}

// C2. up to 50 shrink sweeps (utils.py:521-545), each level's pairs in parallel.  The pairs are bucketed by level first
//     (in T: the transposed list is no longer needed) so that a level touches only its own pairs; a pair that stopped
//     intersecting is dropped (level 0).  Chains deeper than kMaxLevels are swept by one thread.
template <class Cfg>
__device__ __forceinline__ void ro_sweeps(const RoArrays<Cfg> &A, RoShared &S)
{
    using Idx = typename Cfg::Idx;
    constexpr int kMaxLevels = Cfg::kMaxLevels;
    const int np = S.np, maxl = S.maxl;
    typename Cfg::Level *lv = A.lv;
    if (maxl >= 0) {
        Idx *byl = A.T;
        for (int t = threadIdx.x; t <= kMaxLevels; t += kRoThreads) A.lend[t] = 0;
        __syncthreads();
        for (int p = threadIdx.x; p < np; p += kRoThreads) atomicAdd(&A.lend[lv[p]], 1);
        __syncthreads();
        ro_scan(A.lend, A.lend, kMaxLevels + 1, S.warp);
        for (int p = threadIdx.x; p < np; p += kRoThreads) byl[atomicAdd(&A.lend[lv[p]], 1)] = (Idx)p;
        __syncthreads();
        for (int sweep = 0; sweep < 50; sweep++) {
            if (threadIdx.x == 0) S.changed = 0;
            __syncthreads();
            for (int l = 1; l <= maxl; l++) {
                const int e0 = A.lend[l];
                for (int t = A.lend[l - 1] + threadIdx.x; t < e0; t += kRoThreads) {
                    const int p = (int)byl[t];
                    if (lv[p] == 0) continue;
                    const typename Cfg::Pair pr = A.pairs[p];
                    if (ro_shrink_pair(A.box, Cfg::first(pr), Cfg::second(pr)))
                        S.changed = 1;
                    else
                        lv[p] = 0;
                }
                __syncthreads();
            }
            const int changed = S.changed;
            __syncthreads();
            if (!changed) break;
        }
    } else if (threadIdx.x == 0) {
        int n = np;
        for (int sweep = 0; sweep < 50; sweep++) {
            bool changed = false;
            int w = 0;
            for (int p = 0; p < n; p++) {
                const typename Cfg::Pair pr = A.pairs[p];
                if (ro_shrink_pair(A.box, Cfg::first(pr), Cfg::second(pr))) {
                    changed = true;
                    A.pairs[w++] = pr;
                }
            }
            n = w;
            if (!changed) break;
        }
    }
    __syncthreads();
}

// D1. avg_h (utils.py:581) and the vertical tolerance
__device__ __forceinline__ void ro_avg_h(const int4 *box, int K, RoShared &S)
{
    long long hs = 0;
    for (int k = threadIdx.x; k < K; k += kRoThreads) hs += (long long)box[k].w - (long long)box[k].y;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) hs += __shfl_xor_sync(0xffffffffu, hs, off);
    if (threadIdx.x == 0) S.hsum = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(reinterpret_cast<unsigned long long *>(&S.hsum), (unsigned long long)hs);
    __syncthreads();
    if (threadIdx.x == 0) {
        const double avg = K > 0 ? (double)S.hsum / (double)K : 0.0;
        S.ytol = avg * 0.6;
        S.avg_pos = avg > 0.0 ? 1 : 0;  // (b[0] - last_x1) <= avg_h * inf: true iff avg_h > 0 (0 * inf is NaN)
        S.lines = 0;
    }
    __syncthreads();
}

// D2. stable order by centre y (utils.py:584): key = y0 + y1 (cy = key / 2), ties by index; n2 keys, K of them boxes
template <class Cfg>
__device__ __forceinline__ void ro_sort_by_cy(const int4 *box, int K, int n2, uint64_t *keys)
{
    for (int i = threadIdx.x; i < n2; i += kRoThreads) {
        uint64_t key = ~0ull;
        if (i < K) {
            const long long s2 = (long long)box[i].y + (long long)box[i].w;
            key = ((uint64_t)(s2 + (1ll << 33)) << Cfg::kKeyBits) | (uint64_t)i;
        }
        keys[i] = key;
    }
    __syncthreads();
    ro_bitonic(keys, n2);
}

// D3. line assignment (utils.py:584-603) by warp 0, over the boxes in `keys` order.  The reference gives each box, in
//     ascending centre order, to the first line whose mean centre is within the tolerance, else opens a new line.  A
//     line's mean is at most the centre of the box under test (its members came earlier), so a line that fails the
//     test lies more than the tolerance below it -- and below every later box, and its mean no longer changes: when a
//     new line is opened every older line is out of reach for good.  Only the newest line can ever match, and the loop
//     is: join the newest line if |cy - mean| <= tol, else open a line.
//     That recurrence is run 32 boxes at a time: lane t assumes boxes 0..t-1 of the batch joined the newest line
//     (prefix sums give the line's exact state before box t under that assumption) and tests its own box; the boxes
//     before the first failing lane are committed together, the failing box opens the next line.
//     A line keeps the exact integer sum of its members' y0 + y1 and their number; mean = sum / (2 cnt).  The test is
//     decided without the division, from N = s2 * cnt - sum = 2 cnt (cy - mean) (exact integers) against cnt * 2 tol
//     in 2^-16 fixed point, whenever N is outside the slack in which the reference's rounded float64 expression could
//     come out differently; inside the slack the reference's own expression is evaluated.
//     Then D4: line means (np.mean of the members' centres: exact sum, one division) and line ranks by mean
//     (utils.py:605, stable).
template <class Cfg>
__device__ __forceinline__ void ro_lines(const RoArrays<Cfg> &A, RoShared &S, int K, const uint64_t *keys)
{
    using Idx = typename Cfg::Idx;
    constexpr uint64_t kIndex = (1ull << Cfg::kKeyBits) - 1;
    const int4 *box = A.box;
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        const double ytol = S.ytol;
        // 2 tol as a 2^-16 fixed-point integer when it is small enough for 64-bit products (it is an average box height)
        const bool tol_int = ytol >= 0.0 && ytol < 1.0e6;
        const long long tolq = tol_int ? __double2ll_rn(2.0 * ytol * 65536.0) : 0;
        const bool xgap_ok = S.avg_pos != 0;
        auto line_ok = [&](long long s2, long long sum, long long cnt) -> bool {
            const long long N = s2 * cnt - sum;  // |N| < 2^46 for 32-bit coordinates
            const long long aN = N < 0 ? -N : N, asum = sum < 0 ? -sum : sum;
            // cnt/2 units for the rounding of tolq, 2^-13 (|sum| + |N|) units for the rounding of the reference's
            // float64 expression (which is bounded by 2^-52 of those terms, 2^-36 units)
            const long long lhs = aN << 16, rhs = cnt * tolq;
            const long long slack = cnt + ((asum + aN) >> 13) + 2;
            if (tol_int && lhs <= rhs - slack) return true;
            if (tol_int && lhs >= rhs + slack) return false;
            const double d = (double)s2 / 2.0 - ((double)sum * 0.5) / (double)cnt;
            return fabs(d) <= ytol;
        };
        int L = 0;
        long long cur_sum = 0;
        int cur_cnt = 0;  // the newest line (index L - 1) when L > 0
        if (!xgap_ok) {  // avg_h <= 0: the reference's horizontal condition is never true, every box is its own line
            for (int r = lane; r < K; r += 32) {
                const int k = (int)(keys[r] & kIndex);
                A.line_sum[r] = (long long)box[k].y + (long long)box[k].w;
                A.line_cnt[r] = 1;
                A.line_of[k] = (Idx)r;
                A.seq_of[k] = (Idx)r;
            }
            L = K;
        }
        for (int r = xgap_ok ? 0 : K; r < K;) {
            const int n = min(32, K - r);
            int k = 0;
            long long s2 = 0;
            if (lane < n) {
                k = (int)(keys[r + lane] & kIndex);
                const int4 b = box[k];
                s2 = (long long)b.y + (long long)b.w;
            }
            long long pre = s2;  // inclusive prefix sum of s2 over the batch
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, pre, off);
                if (lane >= off) pre += t;
            }
            bool ok = false;
            if (lane < n && xgap_ok && L > 0) ok = line_ok(s2, cur_sum + pre - s2, (long long)cur_cnt + lane);
            const uint32_t fail = __ballot_sync(0xffffffffu, !ok);  // lanes >= n fail
            const int f = __ffs(fail) - 1;                          // 0..n (fail has bit n set when n < 32) or -1
            const int joined = f < 0 ? 32 : f;
            if (lane < joined) {
                A.line_of[k] = (Idx)(L - 1);
                A.seq_of[k] = (Idx)(r + lane);
            }
            if (joined > 0) {
                cur_sum += __shfl_sync(0xffffffffu, pre, joined - 1);
                cur_cnt += joined;
            }
            if (joined < n) {  // box `joined` opens line L
                if (lane == 0 && L > 0) {
                    A.line_sum[L - 1] = cur_sum;
                    A.line_cnt[L - 1] = cur_cnt;
                }
                cur_sum = __shfl_sync(0xffffffffu, s2, joined);
                cur_cnt = 1;
                if (lane == joined) {
                    A.line_of[k] = (Idx)L;
                    A.seq_of[k] = (Idx)(r + lane);
                }
                L++;
                r += joined + 1;
            } else {
                r += joined;
            }
        }
        if (lane == 0) {
            if (L > 0 && xgap_ok) {
                A.line_sum[L - 1] = cur_sum;
                A.line_cnt[L - 1] = cur_cnt;
            }
            S.lines = L;
        }
    }
    __syncthreads();
    const int L = S.lines;
    for (int l = threadIdx.x; l < L; l += kRoThreads) A.line_cy[l] = ((double)A.line_sum[l] * 0.5) / (double)A.line_cnt[l];
    __syncthreads();
    for (int l = threadIdx.x; l < L; l += kRoThreads) {
        const uint64_t key = ro_orderable(A.line_cy[l]);
        int rank = 0;
        for (int m = 0; m < L; m++) {
            const uint64_t km = ro_orderable(A.line_cy[m]);
            rank += (km < key || (km == key && m < l)) ? 1 : 0;
        }
        A.line_rank[l] = (Idx)rank;
    }
    __syncthreads();
}

// E. utils.py:639 (dict: the LAST box with equal compressed coordinates wins) and _pipeline.py:113-123 (the FIRST word
//    with the same integer box is taken).  Both searches only matter when two boxes coincide, which a hash table of
//    hmask + 1 > K slots detects first (compressed boxes `box`, then original boxes `obox`); without a coincidence
//    position r holds box box_at(r).  Writes order[r] and, when `reordered` is set, its rows.
template <class BoxAt>
__device__ __forceinline__ void ro_emit(const int4 *box, const int4 *obox, uint32_t *htab, uint32_t hmask, int K,
                                        RoShared &S, BoxAt box_at, const float *__restrict__ boxes8, int row_stride,
                                        int32_t *__restrict__ order, float *__restrict__ reordered)
{
    if (threadIdx.x == 0) S.dup = 0;
    for (int pass = 0; pass < 2; pass++) {
        const int4 *arr = pass == 0 ? box : obox;
        for (uint32_t t = threadIdx.x; t <= hmask; t += kRoThreads) htab[t] = 0xffffffffu;
        __syncthreads();
        for (int k = threadIdx.x; k < K; k += kRoThreads) {
            const int4 v = arr[k];
            uint32_t h = (uint32_t)v.x * 0x9E3779B1u ^ (uint32_t)v.y * 0x85EBCA77u ^ (uint32_t)v.z * 0xC2B2AE3Du ^
                         (uint32_t)v.w * 0x27D4EB2Fu;
            h ^= h >> 15;
            for (uint32_t slot = h & hmask;; slot = (slot + 1) & hmask) {  // K < hmask + 1 slots: a free slot exists
                const uint32_t old = atomicCAS(&htab[slot], 0xffffffffu, (uint32_t)k);
                if (old == 0xffffffffu) break;
                if (ro_equal(arr[old], v)) {
                    S.dup = 1;
                    break;
                }
            }
        }
        __syncthreads();
    }
    const bool any_dup = S.dup != 0;
    for (int r = threadIdx.x; r < K; r += kRoThreads) {
        const int k = box_at(r);
        int first = k;
        if (any_dup) {
            const int4 ck = box[k];
            int last = k;
            for (int m = K - 1; m > k; m--) {
                if (ro_equal(box[m], ck)) {
                    last = m;
                    break;
                }
            }
            const int4 ob = obox[last];
            first = last;
            for (int w = 0; w < last; w++) {
                if (ro_equal(obox[w], ob)) {
                    first = w;
                    break;
                }
            }
        }
        order[r] = first;
        if (reordered) {
            const float *src = boxes8 + (size_t)first * row_stride;
            float *dst = reordered + (size_t)r * row_stride;
            for (int c = 0; c < row_stride; c++) dst[c] = src[c];
        }
    }
}

// boxes8: rows of `row_stride` floats whose first 8 are x0,y0..x3,y3 (page-strided with `cap` rows per page)
__global__ void __launch_bounds__(kRoThreads) reading_order_kernel(const float *__restrict__ boxes8, int row_stride,
                                                                   const int32_t *__restrict__ counts, int cap,
                                                                   int4 *__restrict__ obox_g, int32_t *__restrict__ order,
                                                                   float *__restrict__ reordered, int32_t *__restrict__ flags,
                                                                   uint16_t *__restrict__ gpairs16, int32_t *__restrict__ gbox32,
                                                                   int32_t *__restrict__ need_large,
                                                                   int32_t *__restrict__ ticket, int force_large)
{
    using Cfg = RoSmemCfg;
    ms_pdl_wait();
    extern __shared__ __align__(16) unsigned char ro_smem[];
    __shared__ RoShared S;
    __shared__ int s_lend[Cfg::kMaxLevels + 1];

    const int page = blockIdx.x;
    const int K = counts[page];
    const size_t pb = (size_t)page * cap;
    if (threadIdx.x == 0 && need_large) {
        need_large[page] = 0;
        if (page == 0) *ticket = 0;  // the large-page kernel's work counter (it is launched after this kernel)
    }
    // beyond the capacity of this kernel the page is written in detection order and handed to reading_order_large_kernel
    // (or, without one, flagged: the host side orders it)
    auto keep_detection_order = [&]() {
        if (threadIdx.x == 0) {
            if (need_large)
                need_large[page] = 1;
            else
                atomicOr(flags + page, MS_FLAG_ORDER_OVERFLOW);
        }
        for (int k = threadIdx.x; k < K; k += kRoThreads) {
            order[pb + k] = k;
            if (reordered)
                for (int c = 0; c < row_stride; c++) reordered[(pb + k) * row_stride + c] = boxes8[(pb + k) * row_stride + c];
        }
    };
    if (K > kRoMaxBoxes || force_large) {
        keep_detection_order();
        return;
    }

    // dynamic shared memory: boxes, pairs, levels, one u16 per box (row counts in B, then the last pair per second
    // box in C), row starts; B's grid tables live in the pair and level regions before the pairs are written, and
    // after the sweeps the pair + level region (148 KB) holds the arrays of D and E
    int4 *box = reinterpret_cast<int4 *>(ro_smem);                               // kRoMaxBoxes
    uint32_t *pairs = reinterpret_cast<uint32_t *>(ro_smem + kRoMaxBoxes * 16);  // kRoMaxPairs
    uint8_t *lv = reinterpret_cast<uint8_t *>(pairs + kRoMaxPairs);              // kRoMaxPairs
    uint16_t *per_box = reinterpret_cast<uint16_t *>(lv + kRoMaxPairs);         // kRoMaxBoxes
    unsigned char *R = reinterpret_cast<unsigned char *>(pairs);
    uint64_t *keys = reinterpret_cast<uint64_t *>(R);                   // kRoMaxBoxes u64          @   0 K
    int4 *obox_s = reinterpret_cast<int4 *>(R + 32 * 1024);             // E: original boxes        @  32 K
    RoArrays<Cfg> A;
    A.box = box;
    A.bxs = box;
    A.pairs = pairs;
    A.lv = lv;
    A.row_cnt = per_box;
    A.row_start = per_box + kRoMaxBoxes;                                // kRoMaxBoxes + 1
    A.ccnt = reinterpret_cast<int *>(pairs);                            // 1024 cells
    A.cstart = reinterpret_cast<uint16_t *>(lv);                        // 1025
    A.centry = A.cstart + 1026;                                         // kRoGridCap
    A.T = gpairs16 + (size_t)page * 2 * kRoMaxPairs;
    A.prevJ = A.T + kRoMaxPairs;
    A.lastJ = per_box;
    A.bcnt = gbox32 + (size_t)page * 2 * (kRoMaxBoxes + 1);
    A.bstart = A.bcnt + (kRoMaxBoxes + 1);
    A.lend = s_lend;
    A.line_sum = reinterpret_cast<long long *>(R + 32 * 1024);          // per line                 @  32 K
    A.line_cy = reinterpret_cast<double *>(R + 64 * 1024);              // per line                 @  64 K
    A.line_cnt = reinterpret_cast<int *>(R + 96 * 1024);                // per line                 @  96 K
    A.line_rank = reinterpret_cast<uint16_t *>(R + 112 * 1024);         // per line                 @ 112 K
    A.line_of = reinterpret_cast<uint16_t *>(R + 120 * 1024);           // per box                  @ 120 K
    A.seq_of = reinterpret_cast<uint16_t *>(R + 128 * 1024);            // per box                  @ 128 K
    A.htab = reinterpret_cast<uint32_t *>(R + 112 * 1024);              // E: 8192 slots            @ 112 K
    A.pair_cap = kRoMaxPairs;
    A.grid_cap = kRoGridCap;

    ro_int_boxes(boxes8, row_stride, K, pb, box, obox_g + pb, box);
    if (!ro_pairs(A, S, K)) {
        keep_detection_order();
        return;
    }
    ro_levels(A, S, K);
    ro_sweeps(A, S);
    ro_avg_h(box, K, S);
    int n2 = 1;
    while (n2 < K) n2 <<= 1;
    ro_sort_by_cy<Cfg>(box, K, n2, keys);
    ro_lines(A, S, K, keys);

    // D5. boxes by (line, x0, insertion order) (utils.py:606-609): one u64 key
    {
        uint64_t mine[kRoMaxBoxes / kRoThreads];
        int cnt = 0;
        for (int i = threadIdx.x; i < n2; i += kRoThreads, cnt++) {
            uint64_t key = ~0ull;
            if (i < K) {
                const uint64_t lr = (uint64_t)A.line_rank[A.line_of[i]];
                const uint64_t x0 = (uint64_t)((long long)box[i].x + (1ll << 31));
                key = (lr << 44) | (x0 << 12) | (uint64_t)A.seq_of[i];
            }
            mine[cnt] = key;
        }
        __syncthreads();  // every thread has read line_rank / line_of / seq_of (they do not alias keys, but keep order)
        cnt = 0;
        for (int i = threadIdx.x; i < n2; i += kRoThreads, cnt++) keys[i] = mine[cnt];
    }
    __syncthreads();
    ro_bitonic(keys, n2);
    // position r holds the box with insertion order seq: map seq -> box index through the first sort's result.
    // seq_of[] is indexed by box; invert it into line_cnt[] (free now)
    int *box_of_seq = A.line_cnt;
    for (int k = threadIdx.x; k < K; k += kRoThreads) {
        box_of_seq[A.seq_of[k]] = k;
        obox_s[k] = obox_g[pb + k];  // line_sum / line_cy are dead
    }
    __syncthreads();
    ro_emit(box, obox_s, A.htab, 8191u, K, S, [&](int r) { return box_of_seq[(int)(keys[r] & 0xfffu)]; }, boxes8 + pb * row_stride,
            row_stride, order + pb, reordered ? reordered + pb * row_stride : nullptr);
}


// =====================================================================================================================
// Pages beyond the shared-memory kernel's capacity (more than 4096 boxes, or more than 28 672 initially intersecting
// pairs): one CTA per such page, at most kRlSlots pages in flight (one scratch slot each); the CTAs draw the marked
// pages from a ticket counter.  Limits: kRlPairFactor * cap intersecting pairs per page (beyond that the page keeps
// its detection order and is flagged) and 4095 dependency levels for the parallel sweeps (deeper chains are swept by
// one thread).
// =====================================================================================================================
constexpr int kRlCells = RoGlobalCfg::kCells;
constexpr int kRlSlots = 8;
constexpr int kRlPairFactor = 16;
constexpr int kRlSmemKeys = 16384;     // sort keys held in dynamic shared memory (8 + 4 bytes each)
constexpr int kRlSmemBytes = kRlSmemKeys * 12;

__host__ __device__ inline int rl_pair_cap(int cap) { return cap * kRlPairFactor < 65536 ? 65536 : cap * kRlPairFactor; }
__host__ __device__ inline int rl_grid_cap(int cap) { return 8 * cap + 4096; }
__host__ __device__ inline int rl_pow2(int n)
{
    int p = 1;
    while (p < n) p <<= 1;
    return p;
}

// byte offsets of one slot's arrays (the same function sizes the scratch on the host and carves it in the kernel)
struct RlLayout {
    size_t box, pairs, lv, T, prevJ, bcnt, bstart, lastJ, row_cnt, row_start, centry, keys, keys2, line_sum, line_cy, line_cnt,
        line_rank, line_of, seq_of, inv_seq, htab, obox, total;
};
__host__ __device__ inline RlLayout rl_layout(int cap)
{
    RlLayout L;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o = (o + bytes + 255) & ~size_t(255);
        return at;
    };
    const size_t pc = (size_t)rl_pair_cap(cap), n2 = (size_t)rl_pow2(cap), c1 = (size_t)cap + 1;
    L.box = take(c1 * 16);
    L.obox = take(c1 * 16);
    L.pairs = take(pc * 8);
    L.lv = take(pc * 2);
    L.T = take(pc * 4);       // transposed pair list, then the pairs bucketed by level
    L.prevJ = take(pc * 4);
    L.bcnt = take(c1 * 4);
    L.bstart = take(c1 * 4);
    L.lastJ = take(c1 * 4);
    L.row_cnt = take(c1 * 4);
    L.row_start = take(c1 * 4);
    L.centry = take((size_t)rl_grid_cap(cap) * 4);
    L.keys = take(n2 * 8);
    L.keys2 = take(n2 * 4);
    L.line_sum = take(c1 * 8);
    L.line_cy = take(c1 * 8);
    L.line_cnt = take(c1 * 4);
    L.line_rank = take(c1 * 4);
    L.line_of = take(c1 * 4);
    L.seq_of = take(c1 * 4);
    L.inv_seq = take(c1 * 4);
    L.htab = take(n2 * 2 * 4);
    L.total = o;
    return L;
}

struct RlShared {
    RoShared s;
    int page;
    // B: cell counters / cell starts; C: level bucket ends in a
    int a[kRlCells * kRlCells + 2];
    int b[kRlCells * kRlCells + 2];
};

// returns false when the page exceeds this kernel's pair capacity (the caller flags it)
__device__ bool rl_order_page(RlShared &SS, const float *__restrict__ boxes8, int row_stride, int K, size_t pb, int cap,
                              int32_t *__restrict__ order, float *__restrict__ reordered, unsigned char *slot)
{
    using Cfg = RoGlobalCfg;
    RoShared &S = SS.s;
    const RlLayout Lo = rl_layout(cap);
    auto at = [&](size_t off) { return reinterpret_cast<void *>(slot + off); };
    // The 192 KB of dynamic shared memory serve three phases in turn: a copy of the boxes while the pairs are generated
    // (B: every candidate test is a random box read), the pairs' levels during the relaxation and the sweeps (C: random
    // level reads), the sort keys (D).  A page too large for one of them uses the global array for that phase.
    extern __shared__ __align__(16) unsigned char rl_dyn[];
    RoArrays<Cfg> A;
    A.box = static_cast<int4 *>(at(Lo.box));
    int4 *bxs = K <= kRlSmemBytes / 16 ? reinterpret_cast<int4 *>(rl_dyn) : A.box;
    A.bxs = bxs;
    A.pairs = static_cast<uint2 *>(at(Lo.pairs));
    A.row_cnt = static_cast<uint32_t *>(at(Lo.row_cnt));
    A.row_start = static_cast<uint32_t *>(at(Lo.row_start));
    A.ccnt = SS.a;
    A.cstart = reinterpret_cast<uint32_t *>(SS.b);
    A.centry = static_cast<uint32_t *>(at(Lo.centry));
    A.T = static_cast<uint32_t *>(at(Lo.T));
    A.prevJ = static_cast<uint32_t *>(at(Lo.prevJ));
    A.lastJ = static_cast<uint32_t *>(at(Lo.lastJ));
    A.bcnt = static_cast<int *>(at(Lo.bcnt));
    A.bstart = static_cast<int *>(at(Lo.bstart));
    A.lend = SS.a;  // the grid tables are dead by then
    A.line_sum = static_cast<long long *>(at(Lo.line_sum));
    A.line_cy = static_cast<double *>(at(Lo.line_cy));
    A.line_cnt = static_cast<int *>(at(Lo.line_cnt));
    A.line_rank = static_cast<uint32_t *>(at(Lo.line_rank));
    A.line_of = static_cast<uint32_t *>(at(Lo.line_of));
    A.seq_of = static_cast<uint32_t *>(at(Lo.seq_of));
    A.htab = static_cast<uint32_t *>(at(Lo.htab));
    A.pair_cap = rl_pair_cap(cap);
    A.grid_cap = rl_grid_cap(cap);
    int4 *obox = static_cast<int4 *>(at(Lo.obox));
    int *inv_seq = static_cast<int *>(at(Lo.inv_seq));

    ro_int_boxes(boxes8, row_stride, K, pb, A.box, obox, bxs);
    if (!ro_pairs(A, S, K)) return false;
    // levels in shared memory when they fit (the box copy is dead)
    A.lv = S.np <= kRlSmemBytes / 2 ? reinterpret_cast<uint16_t *>(rl_dyn) : static_cast<uint16_t *>(at(Lo.lv));
    ro_levels(A, S, K);
    ro_sweeps(A, S);
    ro_avg_h(A.box, K, S);
    // the two sorts run in shared memory when the page has at most 16 384 boxes (192 KB of keys), else in the slot
    const int n2 = rl_pow2(K);
    uint64_t *K1 = n2 <= kRlSmemKeys ? reinterpret_cast<uint64_t *>(rl_dyn) : static_cast<uint64_t *>(at(Lo.keys));
    uint32_t *K2 = n2 <= kRlSmemKeys ? reinterpret_cast<uint32_t *>(rl_dyn + (size_t)kRlSmemKeys * 8)
                                     : static_cast<uint32_t *>(at(Lo.keys2));
    ro_sort_by_cy<Cfg>(A.box, K, n2, K1);
    ro_lines(A, S, K, K1);

    // D5. boxes by (line, x0, insertion order) (utils.py:606-609): a (u64, u32) key
    for (int i = threadIdx.x; i < n2; i += kRoThreads) {
        uint64_t k1 = ~0ull;
        uint32_t k2 = ~0u;
        if (i < K) {
            k1 = ((uint64_t)A.line_rank[A.line_of[i]] << 32) | (uint64_t)(uint32_t)((long long)A.box[i].x + (1ll << 31));
            k2 = A.seq_of[i];
        }
        K1[i] = k1;
        K2[i] = k2;
    }
    for (int k = threadIdx.x; k < K; k += kRoThreads) inv_seq[A.seq_of[k]] = k;
    __syncthreads();
    ro_bitonic2(K1, K2, n2);
    ro_emit(A.box, obox, A.htab, (uint32_t)(2 * n2 - 1), K, S, [&](int r) { return inv_seq[K2[r]]; },
            boxes8 + pb * row_stride, row_stride, order + pb, reordered ? reordered + pb * row_stride : nullptr);
    return true;
}

__global__ void __launch_bounds__(kRoThreads) reading_order_large_kernel(const float *__restrict__ boxes8, int row_stride,
                                                                         const int32_t *__restrict__ counts, int cap,
                                                                         int n_pages, int32_t *__restrict__ order,
                                                                         float *__restrict__ reordered,
                                                                         int32_t *__restrict__ flags,
                                                                         const int32_t *__restrict__ need_large,
                                                                         int32_t *__restrict__ ticket,
                                                                         unsigned char *__restrict__ slots,
                                                                         size_t slot_bytes)
{
    ms_pdl_wait();
    __shared__ RlShared S;
    for (;;) {
        __syncthreads();  // the previous page's shared state is no longer read
        if (threadIdx.x == 0) {
            int p;
            do {
                p = atomicAdd(ticket, 1);
            } while (p < n_pages && need_large[p] == 0);
            S.page = p;
        }
        __syncthreads();
        const int page = S.page;
        if (page >= n_pages) return;
        const bool ok = rl_order_page(S, boxes8, row_stride, counts[page], (size_t)page * cap, cap, order, reordered,
                                      slots + (size_t)blockIdx.x * slot_bytes);
        // beyond this kernel's capacity too: the page keeps the detection order the first kernel wrote, and is flagged
        if (!ok && threadIdx.x == 0) atomicOr(flags + page, MS_FLAG_ORDER_OVERFLOW);
    }
}

}  // namespace

static int rl_slots(int n_pages, int cap_per_page)
{
    if (cap_per_page > (1 << 20)) return 0;  // 20-bit box indices in the sort keys
    return n_pages < kRlSlots ? n_pages : kRlSlots;
}

size_t msk_reading_order_scratch(int n_pages, int cap_per_page)
{
    return (size_t)n_pages * cap_per_page * sizeof(int4) + (size_t)n_pages * 2 * kRoMaxPairs * sizeof(uint16_t) +
           (size_t)n_pages * 2 * (kRoMaxBoxes + 1) * sizeof(int32_t) + (size_t)(n_pages + 1) * sizeof(int32_t) +
           (size_t)rl_slots(n_pages, cap_per_page) * rl_layout(cap_per_page).total + 8192;
}

// order (n_pages*cap) int32: order[p*cap + r] = index of the word at reading position r; `reordered` (may be NULL)
// receives the rows of boxes8 in that order (it must not alias boxes8).
int msk_reading_order(ms_ctx *ctx, const float *boxes8, int row_stride, const int32_t *counts, int n_pages,
                      int cap_per_page, int32_t *order, float *reordered, int32_t *flags, ms_bump bump, cudaStream_t st)
{
    if (n_pages <= 0) return MS_OK;
    int4 *obox = bump.take<int4>((size_t)n_pages * cap_per_page);
    uint16_t *gpairs16 = bump.take<uint16_t>((size_t)n_pages * 2 * kRoMaxPairs);
    int32_t *gbox32 = bump.take<int32_t>((size_t)n_pages * 2 * (kRoMaxBoxes + 1));
    const int slots = rl_slots(n_pages, cap_per_page);
    const size_t slot_bytes = rl_layout(cap_per_page).total;
    int32_t *need_large = slots ? bump.take<int32_t>((size_t)n_pages + 1) : nullptr;  // [n_pages]: ticket counter
    unsigned char *slot_mem = slots ? bump.take<unsigned char>((size_t)slots * slot_bytes) : nullptr;
    if (!obox || !gpairs16 || !gbox32 || (slots && (!need_large || !slot_mem))) {
        ms_set_error("reading_order: scratch too small");
        return MS_ERR_CAPACITY;
    }
    const size_t smem = (size_t)kRoMaxBoxes * 16 + (size_t)kRoMaxPairs * 5 + (size_t)kRoMaxBoxes * 2 +
                        (size_t)(kRoMaxBoxes + 2) * 2;
    static_assert(kRoMaxPairs * 5 + kRoMaxBoxes * 2 >= 144 * 1024 && kRoMaxBoxes == 4096,
                  "pair + level region must hold the sort / line arrays laid out in the kernel");
    MS_TRY(ms_allow_smem(ctx, MS_SMEM_READING_ORDER, reading_order_kernel, (int)smem));
    ms_launch(reading_order_kernel, n_pages, kRoThreads, smem, st, boxes8, row_stride, counts, cap_per_page, obox, order,
                                                           reordered, flags, gpairs16, gbox32, need_large,
                                                           need_large ? need_large + n_pages : nullptr,
                                                           slots ? ctx->ro_force_large : 0);
    MS_LAUNCH_CHECK(ctx);
    if (slots) {  // pages the first kernel could not hold (none, usually: the CTAs find no ticket and leave)
        const int smem_l = kRlSmemKeys * 12;
        MS_TRY(ms_allow_smem(ctx, MS_SMEM_READING_ORDER_LARGE, reading_order_large_kernel, smem_l));
        ms_launch(reading_order_large_kernel, slots, kRoThreads, smem_l, st, boxes8, row_stride, counts, cap_per_page, n_pages, order,
                                                                reordered, flags, need_large, need_large + n_pages,
                                                                slot_mem, slot_bytes);
        MS_LAUNCH_CHECK(ctx);
    }
    return MS_OK;
}
