// Rectified crops of rotated word quads -> resize-and-pad -> normalise -> CHW float32 / float16 / bfloat16 batch
// (SURVEY 8f-4).
//
// NOT a reference behaviour: the reference crops the axis-aligned bounding rectangle of every polygon
// (_pipeline.py:204-221) and lists the rotated crop as future work (todo.md:1).  The operation is defined through the
// OpenCV calls a maintainer would write,
//     w, h  = round-half-even of the longer of each pair of opposite quad edges (float64); no patch if a side is < 2
//             or > 32767
//     Minv  = cv2.getPerspectiveTransform([[0,0],[w-1,0],[w-1,h-1],[0,h-1]], quad)
//     patch = cv2.warpPerspective(page, Minv, (w, h), INTER_LINEAR | WARP_INVERSE_MAP, borderMode, borderValue)
// followed by exactly the ResizeAndPadA + normalise of crop.cu, and restated bit for bit from OpenCV's
// imgproc/imgwarp.cpp + core/matrix_decomp.cpp (checked against cv2 4.13 via tests/golden/quad_warp.npz):
//   * the 8x8 system with float32 products in columns 6-7, LU with partial pivoting in float64 (eps = 100 ulp)
//   * destination coordinates evaluated in blocks of bw0 columns: X0 = M0*bx + M1*y + M2, then (X0 + M0*x1) * (32/W),
//     rounded half-to-even to 5 fractional bits
//   * 15-bit bilinear weights (32-ay)(32-ax)*32 ..., with the integer-position entry {32767, 0, 0, 1};
//     (sum + 2^14) >> 15; BORDER_CONSTANT substitutes the value per tap, BORDER_REPLICATE clamps the tap.
//
// Kernels: quad_plan_kernel (thread per quad: size, homography, resize plan) and quad_crop_kernel (CTA per quad:
// warp the patch into shared memory -- or evaluate it on the fly when it is larger than the stage -- then the same
// per-pixel resampling as crop_generic_kernel).  HBM traffic per quad: the touched page pixels + 3*ih*iw*4 bytes out.
#include "crop_common.cuh"

namespace {

constexpr int kQcThreads = 256;
constexpr int kQcPatchBytes = 40 * 1024;  // shared-memory patch stage (e.g. 260 x 52 pixels)
constexpr int kQcMaxTab = 384;            // AxisEnt entries (nw + nh of a 64 x 256 canvas is 320)

struct QuadPlan {
    double m[9];  // patch (x, y, 1) -> page (X, Y, W)
    int page, w, h, bw0;
    int ok, staged;       // staged: taken by quad_crop_staged_kernel (source window copied into shared memory by TMA)
    int wx0, wy0, ww, wh;  // the window: columns [wx0, wx0 + ww), rows [wy0, wy0 + wh) of the page hold every tap
    int mis, pad0;         // 16-byte misalignment of the window's first byte (the same in every row)
};

// ---- the staged kernel's shape (see quad_crop_staged_kernel) ----
constexpr int kQsThreads = 320;          // copy warp, table / padding warp, 8 consumer warps
constexpr int kQsCW = 8;                 // consumer warps
constexpr int kQsSlots = 3;              // quads in flight per CTA
constexpr int kQsG = 4;                  // destination rows per band (a band is one consumer warp's unit of work)
constexpr int kQsBandBytes = 4096;       // one consumer warp's patch rows (+ 64 bytes of slack)
constexpr int kQsBandPitch = kQsBandBytes + 64;
constexpr int kQsWinMax = 40 * 1024;     // largest staged source window
constexpr int kQsRing = 64 * 1024;       // window ring of a CTA

// oracle quad_patch_size: edge lengths in float64 from the float32 vertices
__device__ __forceinline__ bool quad_patch_size(const float *q, int &w, int &h)
{
    double x[4], y[4];
#pragma unroll
    for (int v = 0; v < 4; v++) {
        x[v] = (double)q[2 * v];
        y[v] = (double)q[2 * v + 1];
    }
    auto edge = [&](int a, int b) {
        const double dx = x[b] - x[a], dy = y[b] - y[a];
        return sqrt(dx * dx + dy * dy);
    };
    const double e01 = edge(0, 1), e32 = edge(3, 2), e03 = edge(0, 3), e12 = edge(1, 2);
    const double ew = e32 > e01 ? e32 : e01, eh = e12 > e03 ? e12 : e03;  // Python max(a, b)
    w = h = 0;
    if (!(isfinite(e01) && isfinite(e32) && isfinite(e03) && isfinite(e12))) return false;
    if (ew > 32767.0 || eh > 32767.0) return false;  // beyond the 16-bit coordinates of the remap
    w = (int)rint(ew);
    h = (int)rint(eh);
    return w >= 2 && h >= 2;
}

// cv2.getPerspectiveTransform(rect(w,h), quad): imgwarp.cpp builds the system, matrix_decomp.cpp LUImpl solves it
__device__ bool perspective_from_rect(const float *q, int w, int h, double *m)
{
    const float sx[4] = {0.f, (float)(w - 1), (float)(w - 1), 0.f};
    const float sy[4] = {0.f, 0.f, (float)(h - 1), (float)(h - 1)};
    double a[8][8], b[8];
    for (int i = 0; i < 4; i++) {
        const float dx = q[2 * i], dy = q[2 * i + 1];
        a[i][0] = a[i + 4][3] = sx[i];
        a[i][1] = a[i + 4][4] = sy[i];
        a[i][2] = a[i + 4][5] = 1.0;
        a[i][3] = a[i][4] = a[i][5] = a[i + 4][0] = a[i + 4][1] = a[i + 4][2] = 0.0;
        a[i][6] = (double)(-sx[i] * dx);  // float32 products (Point2f arithmetic)
        a[i][7] = (double)(-sy[i] * dx);
        a[i + 4][6] = (double)(-sx[i] * dy);
        a[i + 4][7] = (double)(-sy[i] * dy);
        b[i] = dx;
        b[i + 4] = dy;
    }
    const double eps = 2.220446049250313e-16 * 100;
    for (int i = 0; i < 8; i++) {
        int k = i;
        for (int j = i + 1; j < 8; j++)
            if (fabs(a[j][i]) > fabs(a[k][i])) k = j;
        if (fabs(a[k][i]) < eps) return false;
        if (k != i) {
            for (int j = i; j < 8; j++) {
                const double t = a[i][j];
                a[i][j] = a[k][j];
                a[k][j] = t;
            }
            const double t = b[i];
            b[i] = b[k];
            b[k] = t;
        }
        const double d = -1 / a[i][i];
        for (int j = i + 1; j < 8; j++) {
            const double alpha = a[j][i] * d;
            for (int c = i + 1; c < 8; c++) a[j][c] += alpha * a[i][c];
            b[j] += alpha * b[i];
        }
    }
    for (int i = 7; i >= 0; i--) {
        double s = b[i];
        for (int c = i + 1; c < 8; c++) s -= a[i][c] * b[c];
        b[i] = s / a[i][i];
    }
    for (int i = 0; i < 8; i++) m[i] = b[i];
    m[8] = 1.0;
    return true;
}

__global__ void __launch_bounds__(128) quad_plan_kernel(const float *__restrict__ quads, int quad_stride,
                                                        const int32_t *__restrict__ page_of, int64_t n, int n_pages,
                                                        int min_text_size, int ih, int iw, QuadPlan *__restrict__ qplans,
                                                        Plan *__restrict__ plans, int32_t *__restrict__ sizes_out,
                                                        const uint8_t *__restrict__ pages, int img_h, int img_w,
                                                        int stage_ok, StageDesc *__restrict__ work,
                                                        int32_t *__restrict__ n_work)
{
    ms_pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float *q = quads + i * quad_stride;
        QuadPlan qp;
        Plan p;
        plan_reset(p);
        qp.page = page_of ? page_of[i] : 0;
        qp.ok = qp.staged = 0;
        qp.wx0 = qp.wy0 = qp.ww = qp.wh = qp.mis = qp.pad0 = 0;
        qp.bw0 = 1;
#pragma unroll
        for (int k = 0; k < 9; k++) qp.m[k] = 0.0;
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = q[k];
        bool ok = qp.page >= 0 && qp.page < n_pages && quad_patch_size(v, qp.w, qp.h);
        ok = ok && qp.w >= min_text_size && qp.h >= min_text_size;  // _pipeline.py:130-133 applied to the patch
        ok = ok && perspective_from_rect(v, qp.w, qp.h, qp.m);
        if (ok) {
            // WarpPerspectiveInvoker's block width for a (w, h) destination
            const int bh0 = min(16, qp.h);
            qp.bw0 = min(1024 / bh0, qp.w);
            qp.ok = 1;
            p.w = qp.w;
            p.h = qp.h;
            p.ok = 1;
            plan_resize(qp.w, qp.h, ih, iw, p);
            p.staged = (size_t)qp.w * qp.h * 3 <= (size_t)kQcPatchBytes;  // the patch fits the shared-memory stage
            // The staged kernel takes the quad when (i) the resize is the 4-tap INTER_AREA case, (ii) a band of kQsG
            // destination rows needs no more patch rows than a consumer warp's buffer holds, (iii) the coordinate
            // blocks are at most 64 columns wide (patch height >= 16), (iv) the denominator W is positive and away from
            // zero at the four patch corners -- W is linear in (x, y), so it is at least that everywhere on the patch,
            // every coordinate is finite, and the projective image of the patch rectangle is the convex hull of the
            // corner images -- and (v) the window that holds every tap (that hull, plus the bilinear neighbour and a
            // pixel of slack for the 1/32-pixel rounding and the float64 rounding of the per-pixel evaluation, both far
            // below a pixel) is inside the page (no border handling) and fits the ring.
            bool corners_ok = stage_ok && work && p.interp == 3 && p.scale_x < 2.999 && p.scale_y < 2.999 && qp.h >= 16 &&
                              qp.w < 32768;
            double mnx = 1e300, mxx = -1e300, mny = 1e300, mxy = -1e300;
            if (corners_ok) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const double cx = (k & 1) ? (double)(qp.w - 1) : 0.0, cy = (k & 2) ? (double)(qp.h - 1) : 0.0;
                    const double Wc = qp.m[6] * cx + qp.m[7] * cy + qp.m[8];
                    const double Xc = (qp.m[0] * cx + qp.m[1] * cy + qp.m[2]) / Wc;
                    const double Yc = (qp.m[3] * cx + qp.m[4] * cy + qp.m[5]) / Wc;
                    corners_ok = corners_ok && Wc > 1e-3 && Wc < 1e6 && fabs(Xc) < 1e6 && fabs(Yc) < 1e6;
                    mnx = fmin(mnx, Xc);
                    mxx = fmax(mxx, Xc);
                    mny = fmin(mny, Yc);
                    mxy = fmax(mxy, Yc);
                }
            }
            if (corners_ok) {
                const int wx0 = (int)floor(mnx) - 1, wx1 = (int)floor(mxx) + 2;
                const int wy0 = (int)floor(mny) - 1, wy1 = (int)floor(mxy) + 2;
                const int band_rows = (int)ceil(kQsG * p.scale_y) + 2;
                if (wx0 >= 0 && wy0 >= 0 && wx1 < img_w && wy1 < img_h &&
                    (size_t)band_rows * qp.w * 3 <= (size_t)kQsBandBytes) {
                    const size_t stride = (size_t)img_w * 3;
                    const uint8_t *first = pages + (size_t)qp.page * img_h * stride + (size_t)wy0 * stride + (size_t)wx0 * 3;
                    const int a = (int)(reinterpret_cast<uintptr_t>(first) & 15);
                    const int ww = wx1 - wx0 + 1, wh = wy1 - wy0 + 1;
                    const int pitch = (a + ww * 3 + 15) & ~15;
                    const uint8_t *end = pages + (size_t)n_pages * img_h * stride;
                    if ((size_t)pitch * wh + 16 <= (size_t)kQsWinMax &&
                        first - a + (size_t)(wh - 1) * stride + pitch <= end) {
                        qp.staged = 1;
                        qp.wx0 = wx0;
                        qp.wy0 = wy0;
                        qp.ww = ww;
                        qp.wh = wh;
                        qp.mis = a;
                        // the window's rows start 16-byte aligned (the page stride is a multiple of 16): each one is
                        // copied as exactly `pitch` bytes
                        StageDesc d;
                        d.src = first - a;
                        d.stride = (int)stride;
                        d.pitch = pitch;
                        d.row_bytes = pitch;
                        d.rows = wh;
                        d.ci = (int)i;
                        work[atomicAdd(n_work, 1)] = d;
                    }
                }
            }
        } else {
            qp.w = qp.h = 0;
        }
        qplans[i] = qp;
        plans[i] = p;
        if (sizes_out) {
            sizes_out[2 * i] = qp.w;
            sizes_out[2 * i + 1] = qp.h;
        }
    }
}

struct PageView {
    const uint8_t *px;  // (img_h, img_w, 3)
    int img_h, img_w, replicate, bval;
};

// remapBilinear's fixed-point interpolation at the 5-fractional-bit position (X, Y)
__device__ __forceinline__ void sample_px(const PageView &pg, int X, int Y, int &c0, int &c1, int &c2)
{
    const int sx = min(max(X >> 5, -32768), 32767), sy = min(max(Y >> 5, -32768), 32767);
    const int ax = X & 31, ay = Y & 31;
    int w00 = (32 - ay) * (32 - ax) * 32, w01 = (32 - ay) * ax * 32, w10 = ay * (32 - ax) * 32, w11 = ay * ax * 32;
    if ((ax | ay) == 0) {  // initInterTab2D: saturate_cast<short>(32768) = 32767, the missing unit goes to tap (1,1)
        w00 = 32767;
        w11 = 1;
    }
    const int H = pg.img_h, Wd = pg.img_w;
    int t0[3], t1[3], t2[3], t3[3];
    if (sx >= 0 && sy >= 0 && sx + 1 < Wd && sy + 1 < H) {  // all four taps inside: two 6-byte runs
        // a page is at most 32767 x 32767 x 3 bytes: the offset fits 32 bits
        const uint8_t *s = pg.px + ((uint32_t)sy * (uint32_t)Wd + (uint32_t)sx) * 3u;
        const uint8_t *r = s + (uint32_t)Wd * 3u;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            t0[c] = s[c];
            t1[c] = s[3 + c];
            t2[c] = r[c];
            t3[c] = r[3 + c];
        }
    } else {
        auto tap = [&](int yy, int xx, int *t) {
            const bool inside = yy >= 0 && yy < H && xx >= 0 && xx < Wd;
            if (inside || pg.replicate) {
                yy = min(max(yy, 0), H - 1);
                xx = min(max(xx, 0), Wd - 1);
                const uint8_t *s = pg.px + ((uint32_t)yy * (uint32_t)Wd + (uint32_t)xx) * 3u;
                t[0] = s[0];
                t[1] = s[1];
                t[2] = s[2];
            } else {
                t[0] = t[1] = t[2] = pg.bval;
            }
        };
        tap(sy, sx, t0);
        tap(sy, sx + 1, t1);
        tap(sy + 1, sx, t2);
        tap(sy + 1, sx + 1, t3);
    }
    auto mix = [&](int c) { return (t0[c] * w00 + t1[c] * w01 + t2[c] * w10 + t3[c] * w11 + (1 << 14)) >> 15; };
    // the weights are non-negative and sum to 2^15: the result is already within [0, 255]
    c0 = mix(0);
    c1 = mix(1);
    c2 = mix(2);
}

// WarpPerspectiveInvoker's destination -> source coordinates: (X0, Y0, W0) are the terms of the block start
// (bx, y), x1 the column inside the block
__device__ __forceinline__ void warp_xy(const QuadPlan &qp, double X0, double Y0, double W0, int x1, int &X, int &Y)
{
    double W = W0 + qp.m[6] * x1;
    W = W != 0.0 ? 32.0 / W : 0.0;
    const double fX = (X0 + qp.m[0] * x1) * W, fY = (Y0 + qp.m[3] * x1) * W;
    // saturate_cast<int>(std::max((double)INT_MIN, std::min((double)INT_MAX, v))): the conversion instruction already
    // saturates to [INT_MIN, INT_MAX] (round half to even, as cvRound); a NaN comes out of the min/max as INT_MAX
    X = fX != fX ? INT_MAX : __double2int_rn(fX);
    Y = fY != fY ? INT_MAX : __double2int_rn(fY);
}

__device__ __forceinline__ void block_terms(const QuadPlan &qp, int bx, int y, double &X0, double &Y0, double &W0)
{
    X0 = (qp.m[0] * bx + qp.m[1] * y) + qp.m[2];
    Y0 = (qp.m[3] * bx + qp.m[4] * y) + qp.m[5];
    W0 = (qp.m[6] * bx + qp.m[7] * y) + qp.m[8];
}

// one patch pixel at (x, y)
__device__ __forceinline__ void warp_px(const QuadPlan &qp, const PageView &pg, int x, int y, int &c0, int &c1, int &c2)
{
    const int bx = (x / qp.bw0) * qp.bw0;
    double X0, Y0, W0;
    block_terms(qp, bx, y, X0, Y0, W0);
    int X, Y;
    warp_xy(qp, X0, Y0, W0, x - bx, X, Y);
    sample_px(pg, X, Y, c0, c1, c2);
}

// rows [row0, row0 + step, ...) of the patch by one warp each, lanes along x inside every coordinate block: no
// integer division, the block terms are evaluated once per (row, block)
__device__ __forceinline__ void warp_rows(const QuadPlan &qp, const PageView &pg, unsigned char *patch, size_t pitch,
                                          int row0, int row_step, int lane)
{
    for (int y = row0; y < qp.h; y += row_step) {
        unsigned char *dst = patch + (size_t)y * pitch;
        for (int bx = 0; bx < qp.w; bx += qp.bw0) {
            double X0, Y0, W0;
            block_terms(qp, bx, y, X0, Y0, W0);
            const int bw = min(qp.bw0, qp.w - bx);
            for (int x1 = lane; x1 < bw; x1 += 32) {
                int X, Y, c0, c1, c2;
                warp_xy(qp, X0, Y0, W0, x1, X, Y);
                sample_px(pg, X, Y, c0, c1, c2);
                unsigned char *d = dst + (size_t)(bx + x1) * 3;
                d[0] = (unsigned char)c0;
                d[1] = (unsigned char)c1;
                d[2] = (unsigned char)c2;
            }
        }
    }
}

// patch too large for the stage: every tap is evaluated where it is used
struct WarpSrc {
    const QuadPlan *qp;
    PageView pg;
    __device__ __forceinline__ int at(int sy, int b) const
    {
        const int x = b / 3, c = b - 3 * x;
        int c0, c1, c2;
        warp_px(*qp, pg, x, sy, c0, c1, c2);
        return c == 0 ? c0 : (c == 1 ? c1 : c2);
    }
};

template <class T, bool kWriteU8>
__global__ void __launch_bounds__(kQcThreads, 4) quad_crop_kernel(const uint8_t *__restrict__ pages, int img_h,
                                                                  int img_w, const QuadPlan *__restrict__ qplans,
                                                                  const Plan *__restrict__ plans, int64_t n,
                                                                  int replicate, int bval, int ih, int iw,
                                                                  T *__restrict__ batch,
                                                                  uint8_t *__restrict__ canvas_out, int vec_ok,
                                                                  const int32_t *__restrict__ list,
                                                                  const int32_t *__restrict__ list_n)
{
    ms_pdl_wait();
    // `list` != NULL: only the quads it names (those the staged kernel did not take, or handed back)
    // [patch stage kQcPatchBytes + 16][tables: AxisEnt[kQcMaxTab] for resample_px, or the SoA tables of area4_strips]
    extern __shared__ __align__(16) unsigned char qc_smem[];
    unsigned char *qc_patch = qc_smem;
    AxisEnt *s_tab = reinterpret_cast<AxisEnt *>(qc_smem + kQcPatchBytes + 16);
    uint32_t *soa = reinterpret_cast<uint32_t *>(s_tab);
    __shared__ QuadPlan s_qp;
    const int plane = ih * iw, tab_n = area_tab_words(ih, iw);
    const bool soa_fits = (size_t)tab_n * sizeof(uint32_t) <= (size_t)kQcMaxTab * sizeof(AxisEnt);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n_items = list ? (int64_t)*list_n : n;
    for (int64_t li = blockIdx.x; li < n_items; li += gridDim.x) {
        const int64_t ci = list ? (int64_t)list[li] : li;
        __syncthreads();  // the previous quad's plan, patch and tables are no longer read
        if (threadIdx.x == 0) s_qp = qplans[ci];
        const Plan p = plans[ci];
        T *dstf = kHasBatch<T> ? batch + (size_t)ci * 3 * plane : nullptr;
        uint8_t *dstu = kWriteU8 ? canvas_out + (size_t)ci * 3 * plane : nullptr;
        write_padding<T, kWriteU8>(p, ih, iw, dstf, dstu, vec_ok, threadIdx.x, blockDim.x);
        if (!p.ok) continue;  // uniform across the CTA
        // crop.cu's 4-tap INTER_AREA path applies to a staged patch shrunk by factors below 3
        const bool strips = p.staged && soa_fits && p.interp == 3 && p.scale_x < 2.999 && p.scale_y < 2.999;
        const bool need_tab = p.interp == 1 || p.interp == 3;
        const bool tab_ok = need_tab && p.nw + p.nh <= kQcMaxTab;
        bool x3_mine = true;
        if (strips) {
            x3_mine = build_tables(p, soa, tab_n, iw, threadIdx.x, kQcThreads);
        } else if (tab_ok) {
            fill_axis_table(p, s_tab);
        }
        const bool x3 = __syncthreads_and(x3_mine) != 0;  // also the barrier after the tables
        const QuadPlan &qp = s_qp;
        const PageView pg{pages + (size_t)qp.page * img_h * (size_t)img_w * 3, img_h, img_w, replicate, bval};
        if (p.staged) {
            const size_t pitch = (size_t)qp.w * 3;
            warp_rows(qp, pg, qc_patch, pitch, warp, kQcThreads / 32, lane);
            __syncthreads();
            bool redo = !strips;
            if (strips)
                redo = __syncthreads_or(
                    x3 ? area4_strips<T, kWriteU8, kQcThreads, 3>(qc_smem, 0u, (uint32_t)pitch, 0u, 0u, soa, tab_n, ih,
                                                                          iw, p.nw, p.nh, p.y0, dstf, dstu, threadIdx.x)
                       : area4_strips<T, kWriteU8, kQcThreads, 4>(qc_smem, 0u, (uint32_t)pitch, 0u, 0u, soa, tab_n, ih,
                                                                          iw, p.nw, p.nh, p.y0, dstf, dstu, threadIdx.x));
            if (redo) {
                if (strips) {  // an entry with more than 4 taps after all: per-pixel entries, no table
                    resample_canvas<T, kWriteU8>(p, PitchedSrc{qc_patch, pitch}, s_tab, false, need_tab, ih, iw,
                                                         dstf, dstu);
                } else {
                    resample_canvas<T, kWriteU8>(p, PitchedSrc{qc_patch, pitch}, s_tab, tab_ok, need_tab, ih,
                                                         iw, dstf, dstu);
                }
            }
        } else {
            const WarpSrc src{&qp, pg};
            resample_canvas<T, kWriteU8>(p, src, s_tab, tab_ok, need_tab, ih, iw, dstf, dstu);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// The staged kernel: persistent, warp-specialised, fed by the staging ring of crop_common.cuh, like
// crop_resize_pad_kernel.
//   warp 0 (copy warp)    the ring's copy warp: each quad's source window, one TMA bulk copy per window row
//   warp 1 (table warp)   the resize tables of the quad, its homography and window into the slot's metadata, then all
//                         of the canvas padding
//   warps 2..9 (consumers) a quad's destination rows are cut into BANDS of kQsG rows; consumer warp c takes bands c,
//                         c + 8, ...  For a band the warp (i) warps the patch rows the band's taps need out of the staged
//                         window into its own 4 KB buffer -- lanes along x inside OpenCV's 64-column coordinate blocks,
//                         every tap pair fetched as aligned 32-bit shared-memory words, the horizontal blend of a row as
//                         byte dot products (dp4a), then (ii) resamples the band with the 4-tap strip routine of the
//                         axis-aligned kernel.  Nothing but __syncwarp between the two: bands are independent, so the
//                         warps of a CTA drift apart by up to kQsSlots quads and no one waits for the slowest.
// Bit-exactness: coordinates are evaluated exactly as in warp_xy (same float64 operations in the same order; the products
// m*x1 of a lane's two columns are hoisted, which changes no rounding); the blend (sum w_i t_i + 2^14) >> 15 with
// w = 32 (32-ay)(32-ax) ... equals (S + 512) >> 10 for S = sum (32-ay|ay)(32-ax|ax) t_i, integer for integer, and the
// special table entry {32767, 0, 0, 1} at ax = ay = 0 gives t0 either way (|t3 - t0| < 2^14).
// ---------------------------------------------------------------------------------------------------------------------
struct QsMeta {
    double m[9];
    int w, h, bw0, x3;
    int nw, nh, y0;
    int wx0, wy0, umaxx, umaxy;  // window origin; largest window-relative tap origin (ww - 2, wh - 2)
    int pitch, base;             // staged row pitch; ring offset + misalignment of the window's first byte
};

template <class T, bool kWriteU8>
__global__ void __launch_bounds__(kQsThreads, 2)
    quad_crop_staged_kernel(const QuadPlan *__restrict__ qplans, const Plan *__restrict__ plans,
                            const StageDesc *__restrict__ work, const int32_t *__restrict__ n_work_dev,
                            int32_t *__restrict__ ticket, int ih, int iw, T *__restrict__ batch,
                            uint8_t *__restrict__ canvas_out, int vec_ok, uint8_t *__restrict__ redo)
{
    ms_pdl_wait();
    extern __shared__ __align__(128) unsigned char smem[];  // [kQsRing + 64][kQsCW band buffers][kQsSlots table sets]
    const int tab_n = area_tab_words(ih, iw);
    unsigned char *bands = smem + kQsRing + 64;
    uint32_t *tabs = reinterpret_cast<uint32_t *>(bands + kQsCW * kQsBandPitch);
    __shared__ StageSlots<kQsSlots> s_stage;
    __shared__ __align__(16) QsMeta s_meta[kQsSlots];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int plane = ih * iw;
    stage_init(s_stage, kQsCW);

    if (warp == 0) {
        stage_copy_warp(s_stage, smem, kQsRing, work, *n_work_dev, ticket);
        return;
    }
    if (warp == 1) {
        // ---------------- table warp: resize tables + slot metadata, then the padding ----------------
        for (int k = 0;; k++) {
            const int s = k % kQsSlots;
            const int ci = stage_wait_tick(s_stage, k);
            if (ci < 0) break;
            const Plan p = plans[ci];
            const bool x3 = __all_sync(0xffffffffu, build_tables(p, tabs + (size_t)s * tab_n, tab_n, iw, lane));
            if (lane < 9) s_meta[s].m[lane] = qplans[ci].m[lane];
            if (lane == 0) {
                const QuadPlan *qp = qplans + ci;
                QsMeta &me = s_meta[s];
                const int wx0 = qp->wx0, wy0 = qp->wy0;
                me.w = qp->w;
                me.h = qp->h;
                me.bw0 = qp->bw0;
                me.nw = p.nw;
                me.nh = p.nh;
                me.y0 = p.y0;
                me.x3 = x3 ? 1 : 0;
                me.wx0 = wx0;
                me.wy0 = wy0;
                me.umaxx = qp->ww - 2;
                me.umaxy = qp->wh - 2;
                me.pitch = s_stage.pitch[s];
                // the page stride is a multiple of 16: every row has this misalignment
                me.base = s_stage.off[s] + qp->mis;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&s_stage.full[s]);
            write_padding<T, kWriteU8>(p.nw, p.nh, p.y0, ih, iw, kHasBatch<T> ? batch + (size_t)ci * 3 * plane : nullptr,
                                               kWriteU8 ? canvas_out + (size_t)ci * 3 * plane : nullptr, vec_ok, lane, 32);
        }
        return;
    }

    // ---------------- consumers ----------------
    const int cw = warp - 2;
    unsigned char *band = bands + cw * kQsBandPitch;
    const uint32_t band_off = (uint32_t)(band - smem);
    const uint32_t *smem32 = reinterpret_cast<const uint32_t *>(smem);
    for (int k = 0;; k++) {
        const int s = k % kQsSlots;
        const int ci = stage_wait_full(s_stage, k);
        if (ci < 0) break;
        const QsMeta &me = s_meta[s];
        const int w = me.w, h = me.h, nw = me.nw, nh = me.nh, y0 = me.y0;
        const double m0 = me.m[0], m1 = me.m[1], m2 = me.m[2], m3 = me.m[3], m4 = me.m[4], m5 = me.m[5], m6 = me.m[6],
                     m7 = me.m[7], m8 = me.m[8];
        const uint32_t wpitch = (uint32_t)me.pitch, wbase = (uint32_t)me.base;
        const int wx0 = me.wx0, wy0 = me.wy0;
        const uint32_t umaxx = (uint32_t)me.umaxx, umaxy = (uint32_t)me.umaxy;
        const uint32_t ppitch = (uint32_t)w * 3u;  // patch rows in the band buffer
        const uint32_t *tab = tabs + (size_t)s * tab_n;
        T *dstf = kHasBatch<T> ? batch + (size_t)ci * 3 * plane : nullptr;
        uint8_t *dstu = kWriteU8 ? canvas_out + (size_t)ci * 3 * plane : nullptr;
        // this lane's two columns of a 64-column coordinate block
        const double ax0 = m0 * lane, ay0 = m3 * lane, aw0 = m6 * lane;
        const double ax1 = m0 * (lane + 32), ay1 = m3 * (lane + 32), aw1 = m6 * (lane + 32);
        bool bad = false;
        const int nbands = (nh + kQsG - 1) / kQsG;
        // strip height of the resampling pass: the one that keeps the 32 lanes busiest
        const int Gs = ((2 * nw + 31) / 32) * 5 < ((nw + 31) / 32) * 9 ? 2 : 4;
        for (int b = cw; b < nbands; b += kQsCW) {
            const int dyA = b * kQsG, dyB = min(nh, dyA + kQsG);
            const uint32_t recA = tab[area_tab_ybase(iw) + 8 * dyA], recB = tab[area_tab_ybase(iw) + 8 * (dyB - 1)];
            const int r0 = (int)(recA & 0xffffu);
            const int r1 = min(h - 1, (int)(recB & 0xffffu) + min((int)(recB >> 16), 4) - 1);
            if ((recA >> 16) > 4u || (recB >> 16) > 4u || r1 < r0 ||
                (uint32_t)(r1 - r0 + 1) * ppitch > (uint32_t)kQsBandBytes) {
                bad = true;  // more than four taps, or more patch rows than the buffer holds: the generic kernel
                continue;
            }
            // (i) the band's patch rows.  W >= 1e-3 on the whole patch and every term is finite (quad_plan_kernel): the
            // zero and NaN branches of warp_xy cannot be taken.  Every tap lies in the window by construction; the clamp
            // only keeps a violated assumption from reading outside the ring.
            // (Hoisting the row products m*r, or both columns of a lane in one basic block, were measured slower.)
            for (int r = r0; r <= r1; r++) {
                unsigned char *drow = band + (uint32_t)(r - r0) * ppitch;
                for (int bx = 0; bx < w; bx += 64) {
                    const double X0 = (m0 * bx + m1 * r) + m2, Y0 = (m3 * bx + m4 * r) + m5, W0 = (m6 * bx + m7 * r) + m8;
                    const int bwid = min(64, w - bx);
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        const int x1 = lane + 32 * j;
                        if (x1 < bwid) {
                            const double W = 32.0 / (W0 + (j ? aw1 : aw0));
                            const double fX = (X0 + (j ? ax1 : ax0)) * W, fY = (Y0 + (j ? ay1 : ay0)) * W;
                            const int X = __double2int_rn(fX), Y = __double2int_rn(fY);
                            const uint32_t fx = (uint32_t)X & 31u, fy = (uint32_t)Y & 31u;
                            const uint32_t ux = min((uint32_t)((X >> 5) - wx0), umaxx), uy = min((uint32_t)((Y >> 5) - wy0), umaxy);
                            const uint32_t addr = wbase + uy * wpitch + ux * 3u;
                            const uint32_t *pt = smem32 + (addr >> 2), *pb = pt + (wpitch >> 2);
                            const uint32_t sh = (addr & 3u) * 8u;
                            const uint32_t t0 = pt[0], t1 = pt[1], t2 = pt[2], c0 = pb[0], c1 = pb[1], c2 = pb[2];
                            // bytes R0 G0 B0 R1 | G1 B1 . .
                            const uint32_t ta = __funnelshift_r(t0, t1, sh), tb = __funnelshift_r(t1, t2, sh);
                            const uint32_t ca = __funnelshift_r(c0, c1, sh), cb = __funnelshift_r(c1, c2, sh);
                            const uint32_t gx = 32u - fx, gy = 32u - fy;
                            const uint32_t wr = gx | (fx << 24), wg = gx << 8, wb = gx << 16, wb1 = fx << 8;
                            const uint32_t rt = __dp4a(ta, wr, 0u), rb = __dp4a(ca, wr, 0u);
                            const uint32_t gt = __dp4a(tb, fx, __dp4a(ta, wg, 0u)), gb = __dp4a(cb, fx, __dp4a(ca, wg, 0u));
                            const uint32_t bt = __dp4a(tb, wb1, __dp4a(ta, wb, 0u)), bb = __dp4a(cb, wb1, __dp4a(ca, wb, 0u));
                            unsigned char *d = drow + (uint32_t)(bx + x1) * 3u;
                            d[0] = (unsigned char)((rt * gy + rb * fy + 512u) >> 10);
                            d[1] = (unsigned char)((gt * gy + gb * fy + 512u) >> 10);
                            d[2] = (unsigned char)((bt * gy + bb * fy + 512u) >> 10);
                        }
                    }
                }
            }
            __syncwarp();
            // (ii) the band's destination rows out of them (staged row r lives at band_off + (r - r0) * ppitch)
            const uint32_t soff = band_off - (uint32_t)r0 * ppitch;
            // (the strip height as a literal: the strip loop is unrolled for it)
            if (Gs == 2)
                bad = (me.x3 ? area4_strips<T, kWriteU8, 32, 3, true>(smem, soff, ppitch, 0u, 0u, tab, tab_n, ih, iw, nw, nh,
                                                                            y0, dstf, dstu, lane, 2, dyA, dyB)
                             : area4_strips<T, kWriteU8, 32, 4, true>(smem, soff, ppitch, 0u, 0u, tab, tab_n, ih, iw, nw, nh,
                                                                            y0, dstf, dstu, lane, 2, dyA, dyB)) || bad;
            else
                bad = (me.x3 ? area4_strips<T, kWriteU8, 32, 3, true>(smem, soff, ppitch, 0u, 0u, tab, tab_n, ih, iw, nw, nh,
                                                                            y0, dstf, dstu, lane, 4, dyA, dyB)
                             : area4_strips<T, kWriteU8, 32, 4, true>(smem, soff, ppitch, 0u, 0u, tab, tab_n, ih, iw, nw, nh,
                                                                            y0, dstf, dstu, lane, 4, dyA, dyB)) || bad;
            __syncwarp();  // the band buffer is rewritten by the next band
        }
        if (bad) redo[ci] = 1;  // the generic kernel redoes the quad (it rewrites the whole canvas)
        stage_release(s_stage, s);
    }
}

// quads for the generic kernel: not staged, or handed back
__global__ void __launch_bounds__(256) quad_fallback_list_kernel(const QuadPlan *__restrict__ qplans, int64_t n,
                                                                 const uint8_t *__restrict__ redo,
                                                                 int32_t *__restrict__ list, int32_t *__restrict__ list_n)
{
    ms_pdl_wait();
    for (int64_t ci = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ci < n; ci += (int64_t)gridDim.x * blockDim.x)
        if (!qplans[ci].staged || redo[ci]) list[atomicAdd(list_n, 1)] = (int32_t)ci;
}

// the patch alone (row-major h x w x 3), for one planned quad
__global__ void __launch_bounds__(256) quad_warp_kernel(const uint8_t *__restrict__ page, int img_h, int img_w,
                                                        const QuadPlan *__restrict__ qplan, int replicate, int bval,
                                                        uint8_t *__restrict__ patch)
{
    ms_pdl_wait();
    __shared__ QuadPlan s_qp;
    if (threadIdx.x == 0) s_qp = *qplan;
    __syncthreads();
    const QuadPlan &qp = s_qp;
    if (!qp.ok) return;
    const PageView pg{page, img_h, img_w, replicate, bval};
    const int64_t npx = (int64_t)qp.w * qp.h;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < npx; t += (int64_t)gridDim.x * blockDim.x) {
        const int y = (int)(t / qp.w), x = (int)(t - (int64_t)y * qp.w);
        int c0, c1, c2;
        warp_px(qp, pg, x, y, c0, c1, c2);
        patch[t * 3] = (unsigned char)c0;
        patch[t * 3 + 1] = (unsigned char)c1;
        patch[t * 3 + 2] = (unsigned char)c2;
    }
}

}  // namespace

size_t msk_quad_crop_scratch(int64_t n)
{
    const size_t k = (size_t)(n > 0 ? n : 0);
    return k * (sizeof(QuadPlan) + sizeof(Plan) + sizeof(StageDesc) + 1 + sizeof(int32_t)) + 8192;
}

static int quad_args_ok(int n_pages, int img_h, int img_w, int border_mode, int border_value, const char *who)
{
    if (n_pages <= 0 || img_h <= 0 || img_w <= 0 || img_h > 32767 || img_w > 32767) {
        ms_set_error("%s: pages must be 1..32767 pixels on a side (16-bit remap coordinates), got %dx%d", who, img_h, img_w);
        return MS_ERR_INVALID;
    }
    if (border_mode < 0 || border_mode > 1 || border_value < 0 || border_value > 255) {
        ms_set_error("%s: border_mode must be 0 (constant) or 1 (replicate), border_value 0..255", who);
        return MS_ERR_INVALID;
    }
    return MS_OK;
}

int msk_quad_crop(ms_ctx *ctx, const uint8_t *pages, int n_pages, int img_h, int img_w, const float *quads,
                  int quad_stride, const int32_t *page_of, int64_t n, int min_text_size, int border_mode,
                  int border_value, int out_h, int out_w, void *batch, int batch_dtype, uint8_t *canvas_u8,
                  int32_t *sizes_out, ms_bump bump, cudaStream_t st)
{
    if (n <= 0) return MS_OK;
    MS_TRY(quad_args_ok(n_pages, img_h, img_w, border_mode, border_value, "quad_crop"));
    if (out_h <= 0 || out_w <= 0 || quad_stride < 8 || (!batch && !canvas_u8) ||
        (int64_t)out_h * out_w > (1 << 20)) {
        ms_set_error("quad_crop: bad arguments");
        return MS_ERR_INVALID;
    }
    QuadPlan *qplans = bump.take<QuadPlan>((size_t)n);
    Plan *plans = bump.take<Plan>((size_t)n);
    StageDesc *work = bump.take<StageDesc>((size_t)n);
    uint8_t *redo = bump.take<uint8_t>((size_t)n);
    int32_t *list = bump.take<int32_t>((size_t)n);
    int32_t *cnt = bump.take<int32_t>(4);  // staged quads, ticket counter, fallback-list length
    if (!qplans || !plans || !work || !redo || !list || !cnt) {
        ms_set_error("quad_crop: scratch too small");
        return MS_ERR_CAPACITY;
    }
    // The staged kernel needs 16-byte aligned page rows (TMA bulk copies) and 32-bit quad indices; MS_B200_QUAD_NO_STAGE=1
    // sends every quad to the generic kernel (A/B runs and tests).
    const int tab_bytes = area_tab_words(out_h, out_w) * (int)sizeof(uint32_t);
    const int smem_s = kQsRing + 64 + kQsCW * kQsBandPitch + kQsSlots * tab_bytes;
    // (a 64 x 256 canvas' tables do not leave room for two CTAs per SM: generic kernel)
    const int stage_ok = (reinterpret_cast<uintptr_t>(pages) & 15) == 0 && ((size_t)img_w * 3) % 16 == 0 &&
                         n < ((int64_t)1 << 31) && !ctx->quad_no_stage && smem_s <= 112 * 1024;
    MS_CUDA(cudaMemsetAsync(cnt, 0, 4 * sizeof(int32_t), st));
    ctx->quad_cnt = cnt;
    ctx->quad_stream = st;
    MS_CUDA(cudaMemsetAsync(redo, 0, (size_t)n, st));
    int64_t pg = (n + 127) / 128;
    if (pg > (int64_t)ctx->num_sms * 16) pg = (int64_t)ctx->num_sms * 16;
    ms_launch(quad_plan_kernel, (int)pg, 128, 0, st, quads, quad_stride, page_of, n, n_pages, min_text_size, out_h, out_w,
                                             qplans, plans, sizes_out, pages, img_h, img_w, stage_ok, work, cnt);
    MS_LAUNCH_CHECK(ctx);
    const bool staged = stage_ok != 0;
    int64_t grid = (int64_t)ctx->num_sms * 4;  // 40 KB stage + 12 KB tables, 64 registers: four CTAs per SM
    if (grid > n) grid = n;
    const int smem = kQcPatchBytes + 16 + kQcMaxTab * (int)sizeof(AxisEnt);
    return launch_for_outputs(batch, batch_dtype, canvas_u8, [&](auto bt, auto u8) {
        using T = typename decltype(bt)::type;
        constexpr bool kU8 = decltype(u8)::value;
        T *out = static_cast<T *>(batch);
        const int vec_ok = batch_vec_ok<T>(batch, out_w);
        if (staged) {
            MS_TRY(ms_allow_smem(ctx, batch_slot<T, kU8>(MS_SMEM_QUAD_STAGED_U8), quad_crop_staged_kernel<T, kU8>, smem_s));
            ms_launch(quad_crop_staged_kernel<T, kU8>, ctx->num_sms * 2, kQsThreads, smem_s, st, qplans, plans, work, cnt,
                      cnt + 1, out_h, out_w, out, canvas_u8, vec_ok, redo);
            MS_LAUNCH_CHECK(ctx);
        }
        ms_launch(quad_fallback_list_kernel, (int)pg, 256, 0, st, qplans, n, redo, list, cnt + 2);
        MS_LAUNCH_CHECK(ctx);
        MS_TRY(ms_allow_smem(ctx, batch_slot<T, kU8>(MS_SMEM_QUAD_U8), quad_crop_kernel<T, kU8>, smem));
        ms_launch(quad_crop_kernel<T, kU8>, (int)grid, kQcThreads, smem, st, pages, img_h, img_w, qplans, plans, n,
                  border_mode, border_value, out_h, out_w, out, canvas_u8, vec_ok, list, cnt + 2);
        MS_LAUNCH_CHECK(ctx);
        return MS_OK;
    });
}

// One quad's patch.  *w / *h receive the patch size (0, 0: no patch); the pixels are produced only when they fit
// patch_cap bytes (device memory).  Synchronises `st` to read the size back.
int msk_quad_warp(ms_ctx *ctx, const uint8_t *page, int img_h, int img_w, const float *quad_dev, int border_mode,
                  int border_value, uint8_t *patch_dev, size_t patch_cap, int *w, int *h, ms_bump bump, cudaStream_t st)
{
    MS_TRY(quad_args_ok(1, img_h, img_w, border_mode, border_value, "quad_warp"));
    QuadPlan *qplan = bump.take<QuadPlan>(1);
    Plan *plan = bump.take<Plan>(1);
    int32_t *size = bump.take<int32_t>(2);
    if (!qplan || !plan || !size) {
        ms_set_error("quad_warp: scratch too small");
        return MS_ERR_CAPACITY;
    }
    ms_launch(quad_plan_kernel, 1, 128, 0, st, quad_dev, 8, nullptr, 1, 1, 0, 32, 128, qplan, plan, size, nullptr, img_h, img_w, 0,
                                        nullptr, nullptr);
    MS_LAUNCH_CHECK(ctx);
    int32_t hs[2] = {0, 0};
    MS_CUDA(cudaMemcpyAsync(hs, size, sizeof(hs), cudaMemcpyDeviceToHost, st));
    MS_CUDA(cudaStreamSynchronize(st));
    *w = hs[0];
    *h = hs[1];
    const size_t need = (size_t)hs[0] * hs[1] * 3;
    if (need == 0) return MS_OK;
    if (need > patch_cap) {
        ms_set_error("quad_warp: the %dx%d patch needs %zu bytes, capacity %zu", hs[0], hs[1], need, patch_cap);
        return MS_ERR_CAPACITY;
    }
    int64_t grid = ((int64_t)hs[0] * hs[1] + 255) / 256;
    if (grid > (int64_t)ctx->num_sms * 8) grid = (int64_t)ctx->num_sms * 8;
    ms_launch(quad_warp_kernel, (int)grid, 256, 0, st, page, img_h, img_w, qplan, border_mode, border_value, patch_dev);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}
