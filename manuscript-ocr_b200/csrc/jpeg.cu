// Baseline-JPEG decode on the device (DESIGN 4.5): ms_jpeg_inspect_host and ms_jpeg_decode_batch.
//
// Per batch: the host parses the markers (jpeg_core.cuh) and stages every device file's entropy-coded bytes and its
// descriptor (tables, geometry) in one pinned buffer, copied with one cudaMemcpyAsync.  Then, stream-ordered:
//   1. unstuff   jpg_end / jpg_count / jpg_scan / jpg_emit: the end of the entropy data (first marker that is not
//                RSTn), the bytes without stuffed zeros and RST markers, and the bit offset of every restart interval;
//   2. Huffman   jpg_guess / jpg_sync / jpg_fix: one thread per JPG_SUB_BITS of unstuffed data decodes the blocks
//                that start in its subsequence from a guessed state (bit offset, block within the MCU); threads of a
//                CTA then restart from their left neighbour's exit state until none changes (Klein & Wiseman's
//                self-synchronisation), JPG_SYNC_ROUNDS launches carry the states across CTAs, and one warp per file
//                walks the chain and re-decodes any subsequence whose entry still differs from its neighbour's exit,
//                so the result is exact whatever the data; jpg_base scans the block counts;
//   3. jpg_write decodes again from the final states and stores the coefficients (DC as differences);
//   4. jpg_dc    the DC prefix sums per component, reset at every restart interval;
//   5. jpg_idct  ISLOW IDCT of every block into per-component u8 planes (8 threads per block);
//   6. jpg_color upsampling and YCbCr -> RGB straight into the page.
// A page whose data does not decode exactly as the headers say gets MS_JPEG_BAD_ENTROPY and is left to the host.
#include <string.h>

#include <new>
#include <vector>

#include "jpeg_core.cuh"
#include "ms_internal.cuh"

#define JPG_CHUNK 4096       // entropy-coded bytes per unstuff CTA (256 threads x 16)
#define JPG_SYNC_ROUNDS 8    // cross-CTA synchronisation launches before the serial walk

struct jpg_fstate {
    unsigned long long end;  // first byte of the marker that ends the entropy-coded data (src_len when none)
    int32_t unst_len, nrst;
};

// ---- CTA scans ------------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T jpg_warp_incl(T v)
{
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T u = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (lane >= o) v += u;
    }
    return v;
}

// exclusive scan over the CTA (blockDim.x a multiple of 32, <= 1024); *total = the CTA's sum.  `sh` >= 33 entries.
template <typename T>
__device__ __forceinline__ T jpg_cta_excl(T v, T *sh, T *total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T inc = jpg_warp_incl(v);
    if (lane == 31) sh[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        T s = lane < nw ? sh[lane] : T(0);
        T si = jpg_warp_incl(s);
        if (lane < nw) sh[lane] = si - s;
        if (lane == 31) sh[32] = si;
    }
    __syncthreads();
    T r = inc - v + sh[wid];
    *total = sh[32];
    __syncthreads();
    return r;
}

__device__ __forceinline__ bool jpg_is_rst(uint8_t b) { return b >= 0xD0 && b <= 0xD7; }

// ---- 1. unstuff -----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) jpg_end_kernel(const jpg_file *files, const int32_t *chunk_file,
                                                      const uint8_t *src, jpg_fstate *fs, const int32_t *status)
{
    ms_pdl_wait();
    const int f = chunk_file[blockIdx.x];
    const jpg_file &F = files[f];
    const uint8_t *b = src + F.src_off;
    const int64_t i0 = (int64_t)(blockIdx.x - F.chunk_off) * JPG_CHUNK + threadIdx.x * 16;
    for (int j = 0; j < 16; j++) {
        const int64_t i = i0 + j;
        if (i >= F.src_len) break;
        if (b[i] != 0xFF) continue;
        if (i + 1 >= F.src_len || (b[i + 1] != 0 && !jpg_is_rst(b[i + 1]))) {
            atomicMin(&fs[f].end, (unsigned long long)i);
            break;
        }
    }
}

// kept byte / RST marker at i (< end)
__device__ __forceinline__ void jpg_classify(const uint8_t *b, int64_t i, bool &keep, bool &rst)
{
    const uint8_t c = b[i];
    const bool after_ff = i > 0 && b[i - 1] == 0xFF;
    rst = c == 0xFF && jpg_is_rst(b[i + 1]);
    keep = !rst && !(after_ff && (c == 0 || jpg_is_rst(c)));
}

__global__ void __launch_bounds__(256) jpg_count_kernel(const jpg_file *files, const int32_t *chunk_file,
                                                        const uint8_t *src, const jpg_fstate *fs, int32_t *chunk_kept,
                                                        int32_t *chunk_rst)
{
    ms_pdl_wait();
    __shared__ int32_t sh[33];
    const int f = chunk_file[blockIdx.x];
    const jpg_file &F = files[f];
    const uint8_t *b = src + F.src_off;
    const int64_t end = (int64_t)fs[f].end;
    const int64_t i0 = (int64_t)(blockIdx.x - F.chunk_off) * JPG_CHUNK + threadIdx.x * 16;
    int32_t nk = 0, nr = 0;
    for (int j = 0; j < 16; j++) {
        const int64_t i = i0 + j;
        if (i >= end) break;
        bool keep, rst;
        jpg_classify(b, i, keep, rst);
        nk += keep;
        nr += rst;
    }
    int32_t tk, tr;
    jpg_cta_excl(nk, sh, &tk);
    jpg_cta_excl(nr, sh, &tr);
    if (threadIdx.x == 0) {
        chunk_kept[blockIdx.x] = tk;
        chunk_rst[blockIdx.x] = tr;
    }
}

// per file: chunk prefixes, unstuffed length, restart-marker count and end-marker checks, segment table defaults
__global__ void __launch_bounds__(1024) jpg_scan_kernel(const jpg_file *files, const uint8_t *src, jpg_fstate *fs,
                                                        int32_t *chunk_kept, int32_t *chunk_rst, uint32_t *seg,
                                                        uint8_t *unst, int32_t *status)
{
    ms_pdl_wait();
    __shared__ int32_t sh[33];
    const jpg_file &F = files[blockIdx.x];
    int32_t ck = 0, cr = 0;
    for (int base = 0; base < F.nchunk; base += 1024) {
        const int c = base + threadIdx.x;
        int32_t k = c < F.nchunk ? chunk_kept[F.chunk_off + c] : 0, r = c < F.nchunk ? chunk_rst[F.chunk_off + c] : 0;
        int32_t tk, tr;
        int32_t ek = jpg_cta_excl(k, sh, &tk), er = jpg_cta_excl(r, sh, &tr);
        if (c < F.nchunk) {
            chunk_kept[F.chunk_off + c] = ck + ek;
            chunk_rst[F.chunk_off + c] = cr + er;
        }
        ck += tk;
        cr += tr;
    }
    uint32_t *sg = seg + F.seg_off;
    for (int s = threadIdx.x; s <= F.nseg; s += blockDim.x) sg[s] = s == 0 ? 0u : (uint32_t)ck * 8u;
    uint8_t *u = unst + F.unst_off;
    if (threadIdx.x < 16) u[ck + threadIdx.x] = 0xFF;
    if (threadIdx.x == 0) {
        fs[blockIdx.x].unst_len = ck;
        fs[blockIdx.x].nrst = cr;
        const int64_t end = (int64_t)fs[blockIdx.x].end;
        const uint8_t *b = src + F.src_off;
        bool bad = cr != F.nseg - 1;                                  // restart markers missing or extra
        if (end < F.src_len && (end + 1 >= F.src_len || b[end + 1] != 0xD9)) bad = true;  // not EOI: another scan, DNL
        if (bad) atomicOr(&status[F.index], JPG_ST_ENTROPY);
    }
}

__global__ void __launch_bounds__(256) jpg_emit_kernel(const jpg_file *files, const int32_t *chunk_file,
                                                       const uint8_t *src, const jpg_fstate *fs,
                                                       const int32_t *chunk_kept, const int32_t *chunk_rst,
                                                       uint32_t *seg, uint8_t *unst, int32_t *status)
{
    ms_pdl_wait();
    __shared__ int32_t sh[33];
    const int f = chunk_file[blockIdx.x];
    const jpg_file &F = files[f];
    const uint8_t *b = src + F.src_off;
    const int64_t end = (int64_t)fs[f].end;
    const int64_t i0 = (int64_t)(blockIdx.x - F.chunk_off) * JPG_CHUNK + threadIdx.x * 16;
    uint32_t km = 0, rm = 0;
    for (int j = 0; j < 16; j++) {
        const int64_t i = i0 + j;
        if (i >= end) break;
        bool keep, rst;
        jpg_classify(b, i, keep, rst);
        km |= (uint32_t)keep << j;
        rm |= (uint32_t)rst << j;
    }
    int32_t tk, tr;
    int32_t ok = jpg_cta_excl((int32_t)__popc(km), sh, &tk) + chunk_kept[blockIdx.x];
    int32_t orr = jpg_cta_excl((int32_t)__popc(rm), sh, &tr) + chunk_rst[blockIdx.x];
    uint8_t *u = unst + F.unst_off;
    uint32_t *sg = seg + F.seg_off;
    for (int j = 0; j < 16; j++) {
        const int64_t i = i0 + j;
        if ((km >> j) & 1) u[ok++] = b[i];
        if ((rm >> j) & 1) {
            if ((b[i + 1] & 7) != (orr & 7)) atomicOr(&status[F.index], JPG_ST_ENTROPY);  // RSTn out of sequence
            if (orr + 1 < F.nseg) sg[orr + 1] = (uint32_t)ok * 8u;
            orr++;
        }
    }
}

// ---- 2. Huffman decode and synchronisation ---------------------------------------------------------------------------
struct jpg_tables {
    jpg_huff dc[3], ac[3];
    int8_t comp_of[JPG_MAX_BPM];
};

__device__ __forceinline__ void jpg_load_tables(const jpg_file &F, jpg_tables &T)
{
    const int nc = F.ncomp;
    const uint4 *s0 = reinterpret_cast<const uint4 *>(F.dc), *s1 = reinterpret_cast<const uint4 *>(F.ac);
    uint4 *d0 = reinterpret_cast<uint4 *>(T.dc), *d1 = reinterpret_cast<uint4 *>(T.ac);
    const int n16 = nc * (int)(sizeof(jpg_huff) / 16);
    for (int i = threadIdx.x; i < n16; i += blockDim.x) {
        d0[i] = s0[i];
        d1[i] = s1[i];
    }
    if (threadIdx.x < JPG_MAX_BPM) T.comp_of[threadIdx.x] = F.comp_of[threadIdx.x];
    __syncthreads();
}

// Restart every thread whose entry differs from its left neighbour's exit until none changes.  Thread 0 keeps `entry`.
__device__ __forceinline__ void jpg_cta_converge(const jpg_file &F, const jpg_tables &T, const uint32_t *words,
                                                 const uint32_t *sg, uint64_t &entry, uint64_t &ex, int32_t &cnt,
                                                 uint32_t sub_end, uint64_t *xs)
{
    for (;;) {
        xs[threadIdx.x] = ex;
        __syncthreads();
        const uint64_t want = threadIdx.x ? xs[threadIdx.x - 1] : entry;
        const bool changed = want != entry;
        if (changed) {
            entry = want;
            ex = jpg_run<false>(F, T.dc, T.ac, T.comp_of, words, sg, entry, sub_end, cnt, nullptr, 0, nullptr);
        }
        if (!__syncthreads_or(changed)) break;
    }
}

__global__ void __launch_bounds__(JPG_SUB_CTA) jpg_guess_kernel(const jpg_file *files, const int32_t *sub_file,
                                                                const uint8_t *unst, const uint32_t *seg,
                                                                const int32_t *status, uint64_t *entry_out,
                                                                uint64_t *exit_out, int32_t *count_out)
{
    ms_pdl_wait();
    __shared__ jpg_tables T;
    __shared__ uint64_t xs[JPG_SUB_CTA];
    const jpg_file &F = files[sub_file[blockIdx.x]];
    if (status[F.index]) return;
    jpg_load_tables(F, T);
    const uint32_t *words = reinterpret_cast<const uint32_t *>(unst + F.unst_off);
    const uint32_t *sg = seg + F.seg_off;
    const uint32_t total = sg[F.nseg];
    const int tl = (blockIdx.x - F.sub_off / JPG_SUB_CTA) * JPG_SUB_CTA + threadIdx.x;
    const uint32_t st = (uint32_t)tl * JPG_SUB_BITS, sub_end = st + JPG_SUB_BITS;
    uint64_t entry = jpg_state(st < total ? st : total, 0);
    int32_t cnt;
    uint64_t ex = jpg_run<false>(F, T.dc, T.ac, T.comp_of, words, sg, entry, sub_end, cnt, nullptr, 0, nullptr);
    jpg_cta_converge(F, T, words, sg, entry, ex, cnt, sub_end, xs);
    const int64_t t = (int64_t)blockIdx.x * JPG_SUB_CTA + threadIdx.x;
    entry_out[t] = entry;
    exit_out[t] = ex;
    count_out[t] = cnt;
}

// One cross-CTA round: a CTA whose first subsequence's entry differs from the previous CTA's last exit restarts it
// and converges again.  (Reading a neighbour CTA's exit while that CTA updates it is benign: any exit read is a state
// some decode produced, and jpg_fix makes the chain consistent.)
__global__ void __launch_bounds__(JPG_SUB_CTA) jpg_sync_kernel(const jpg_file *files, const int32_t *sub_file,
                                                               const uint8_t *unst, const uint32_t *seg,
                                                               const int32_t *status, uint64_t *entry_io,
                                                               uint64_t *exit_io, int32_t *count_io)
{
    ms_pdl_wait();
    __shared__ jpg_tables T;
    __shared__ uint64_t xs[JPG_SUB_CTA];
    const jpg_file &F = files[sub_file[blockIdx.x]];
    if (status[F.index] || blockIdx.x * JPG_SUB_CTA == F.sub_off) return;
    const int64_t t0 = (int64_t)blockIdx.x * JPG_SUB_CTA;
    const uint64_t want = *(volatile const uint64_t *)&exit_io[t0 - 1];
    if (want == entry_io[t0]) return;  // uniform across the CTA
    jpg_load_tables(F, T);
    const uint32_t *words = reinterpret_cast<const uint32_t *>(unst + F.unst_off);
    const uint32_t *sg = seg + F.seg_off;
    const int64_t t = t0 + threadIdx.x;
    const int tl = (blockIdx.x - F.sub_off / JPG_SUB_CTA) * JPG_SUB_CTA + threadIdx.x;
    const uint32_t sub_end = (uint32_t)(tl + 1) * JPG_SUB_BITS;
    uint64_t entry = entry_io[t], ex = exit_io[t];
    int32_t cnt = count_io[t];
    if (threadIdx.x == 0) {
        entry = want;
        ex = jpg_run<false>(F, T.dc, T.ac, T.comp_of, words, sg, entry, sub_end, cnt, nullptr, 0, nullptr);
    }
    jpg_cta_converge(F, T, words, sg, entry, ex, cnt, sub_end, xs);
    entry_io[t] = entry;
    exit_io[t] = ex;
    count_io[t] = cnt;
}

// One warp per file: every subsequence whose entry is not its left neighbour's exit is decoded again, in order.
__global__ void __launch_bounds__(32) jpg_fix_kernel(const jpg_file *files, const uint8_t *unst, const uint32_t *seg,
                                                     const int32_t *status, uint64_t *entry_io, uint64_t *exit_io,
                                                     int32_t *count_io)
{
    ms_pdl_wait();
    __shared__ jpg_tables T;
    const jpg_file &F = files[blockIdx.x];
    if (status[F.index]) return;
    jpg_load_tables(F, T);
    const uint32_t *words = reinterpret_cast<const uint32_t *>(unst + F.unst_off);
    const uint32_t *sg = seg + F.seg_off;
    const int64_t first = F.sub_off, last = (int64_t)F.sub_off + F.nsub;
    int64_t t = first + 1;
    while (t < last) {
        const int64_t u = t + threadIdx.x;
        const bool mism = u < last && entry_io[u] != exit_io[u - 1];
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, mism);
        if (!m) {
            t += 32;
            continue;
        }
        t += __ffs(m) - 1;
        if (threadIdx.x == 0) {
            const uint64_t e = exit_io[t - 1];
            int32_t cnt;
            const uint32_t sub_end = (uint32_t)(t - first + 1) * JPG_SUB_BITS;
            exit_io[t] = jpg_run<false>(F, T.dc, T.ac, T.comp_of, words, sg, e, sub_end, cnt, nullptr, 0, nullptr);
            entry_io[t] = e;
            count_io[t] = cnt;
        }
        __syncwarp();
        t++;
    }
}

// block index of every subsequence's first block; the file's total must be its MCUs x blocks per MCU
__global__ void __launch_bounds__(1024) jpg_base_kernel(const jpg_file *files, const int32_t *count, int32_t *base,
                                                        int32_t *status)
{
    ms_pdl_wait();
    __shared__ int32_t sh[33];
    const jpg_file &F = files[blockIdx.x];
    if (status[F.index]) return;
    int32_t acc = 0;
    for (int b0 = 0; b0 < F.nsub; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        int32_t v = i < F.nsub ? count[F.sub_off + i] : 0, tot;
        int32_t e = jpg_cta_excl(v, sh, &tot);
        if (i < F.nsub) base[F.sub_off + i] = acc + e;
        acc += tot;
    }
    if (threadIdx.x == 0 && (int64_t)acc != (int64_t)F.mcux * F.mcuy * F.bpm) atomicOr(&status[F.index], JPG_ST_ENTROPY);
}

// ---- 3. coefficients ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(JPG_SUB_CTA) jpg_write_kernel(const jpg_file *files, const int32_t *sub_file,
                                                                const uint8_t *unst, const uint32_t *seg,
                                                                int32_t *status, const uint64_t *entry,
                                                                const int32_t *base, int16_t *coef)
{
    ms_pdl_wait();
    __shared__ jpg_tables T;
    const jpg_file &F = files[sub_file[blockIdx.x]];
    if (status[F.index]) return;
    jpg_load_tables(F, T);
    const uint32_t *words = reinterpret_cast<const uint32_t *>(unst + F.unst_off);
    const uint32_t *sg = seg + F.seg_off;
    const int64_t t = (int64_t)blockIdx.x * JPG_SUB_CTA + threadIdx.x;
    const int tl = (int)(t - F.sub_off);
    int32_t cnt, bad = 0;
    jpg_run<true>(F, T.dc, T.ac, T.comp_of, words, sg, entry[t], (uint32_t)(tl + 1) * JPG_SUB_BITS, cnt,
                  coef + F.coef_off * 64, base[t], &bad);
    if (bad) atomicOr(&status[F.index], JPG_ST_ENTROPY);
}

// ---- 4. DC prediction: per (file, component) segmented prefix sum over the component's blocks in scan order -----------
__global__ void __launch_bounds__(1024) jpg_dc_kernel(const jpg_file *files, const int32_t *status, int16_t *coef)
{
    ms_pdl_wait();
    __shared__ int32_t sv[32], sf[32];
    __shared__ int32_t carry;
    const jpg_file &F = files[blockIdx.x];
    const int comp = blockIdx.y;
    if (comp >= F.ncomp || status[F.index]) return;
    const int nc = F.comp_h_blocks[comp], first = F.first_of[comp];
    const int64_t mcus = (int64_t)F.mcux * F.mcuy, n = mcus * nc;
    int16_t *cf = coef + F.coef_off * 64;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t j0 = 0; j0 < n; j0 += 4 * 1024) {
        int32_t v[4];
        int flag = 0, sum = 0;
        for (int k = 0; k < 4; k++) {
            const int64_t j = j0 + (int64_t)threadIdx.x * 4 + k;
            v[k] = 0;
            if (j < n) {
                const int64_t m = j / nc;
                const int q = (int)(j - m * nc);
                v[k] = cf[(m * F.bpm + first + q) * 64];
                if (q == 0 && (m == 0 || (F.ri > 0 && m % F.ri == 0))) {
                    flag = 1;
                    sum = 0;
                }
            }
            sum += v[k];
        }
        // inclusive segmented scan of (flag, sum) over the CTA
        int f = flag, s = sum;
        for (int o = 1; o < 32; o <<= 1) {
            int fo = __shfl_up_sync(0xFFFFFFFFu, f, o), so = __shfl_up_sync(0xFFFFFFFFu, s, o);
            if (lane >= o && !f) s += so;
            if (lane >= o) f |= fo;
        }
        if (lane == 31) {
            sv[wid] = s;
            sf[wid] = f;
        }
        __syncthreads();
        if (wid == 0) {
            int wf = sf[lane], ws = sv[lane];
            for (int o = 1; o < 32; o <<= 1) {
                int fo = __shfl_up_sync(0xFFFFFFFFu, wf, o), so = __shfl_up_sync(0xFFFFFFFFu, ws, o);
                if (lane >= o && !wf) ws += so;
                if (lane >= o) wf |= fo;
            }
            sv[lane] = ws;
            sf[lane] = wf;
        }
        __syncthreads();
        // exclusive prefix for this thread: warp-exclusive part combined with the previous warps' and the carry
        int ef = __shfl_up_sync(0xFFFFFFFFu, f, 1), es = __shfl_up_sync(0xFFFFFFFFu, s, 1);
        if (lane == 0) {
            ef = 0;
            es = 0;
        }
        int pf = 0, ps = carry;
        if (wid > 0) {
            pf = sf[wid - 1];
            ps = pf ? sv[wid - 1] : carry + sv[wid - 1];
        }
        int run = ef ? es : ps + es;
        for (int k = 0; k < 4; k++) {
            const int64_t j = j0 + (int64_t)threadIdx.x * 4 + k;
            if (j < n) {
                const int64_t m = j / nc;
                const int q = (int)(j - m * nc);
                if (q == 0 && (m == 0 || (F.ri > 0 && m % F.ri == 0))) run = 0;
                run += v[k];
                cf[(m * F.bpm + first + q) * 64] = (int16_t)run;
            }
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry = run;
        __syncthreads();
    }
}

// ---- 5. IDCT: 8 threads per block, rows in, columns, rows out ---------------------------------------------------------
__global__ void __launch_bounds__(256) jpg_idct_kernel(const jpg_file *files, int nf, const int32_t *status,
                                                       const int16_t *coef, int64_t total_blocks, uint8_t *planes)
{
    ms_pdl_wait();
    __shared__ int32_t ws[32][8][9];
    const int g = threadIdx.x >> 3, r = threadIdx.x & 7;
    const int64_t blk = (int64_t)blockIdx.x * 32 + g;
    const bool live = blk < total_blocks;
    int f = 0;
    if (live) {
        int lo = 0, hi = nf - 1;
        while (lo < hi) {
            int mid = (lo + hi + 1) >> 1;
            if (files[mid].coef_off <= blk) lo = mid;
            else hi = mid - 1;
        }
        f = lo;
    }
    const jpg_file &F = files[f];
    const int64_t b = blk - F.coef_off;
    const int64_t m = b / (live ? F.bpm : 1);
    const int q = (int)(b - m * F.bpm), comp = live ? F.comp_of[q] : 0;
    const bool run = live && !status[F.index];
    if (run) {
        const int4 raw = reinterpret_cast<const int4 *>(coef + blk * 64)[r];
        const int16_t *c = reinterpret_cast<const int16_t *>(&raw);
        for (int x = 0; x < 8; x++) ws[g][r][x] = (int32_t)c[x] * (int32_t)F.q[comp][r * 8 + x];
    }
    __syncwarp();
    int32_t v[8], o[8];
    if (run) {
        for (int y = 0; y < 8; y++) v[y] = ws[g][y][r];
        jpg_idct_1d(v, o, 11);  // columns: CONST_BITS - PASS1_BITS
    }
    __syncwarp();
    if (run)
        for (int y = 0; y < 8; y++) ws[g][y][r] = o[y];
    __syncwarp();
    if (run) {
        for (int x = 0; x < 8; x++) v[x] = ws[g][r][x];
        jpg_idct_1d(v, o, 18);  // rows: CONST_BITS + PASS1_BITS + 3
        const int hc = comp == 0 ? F.hs : 1, vc = comp == 0 ? F.vs : 1;
        const int bx = (int)(m % F.mcux) * hc + F.blk_x[q], by = (int)(m / F.mcux) * vc + F.blk_y[q];
        uint32_t lo = 0, hi = 0;
        for (int x = 0; x < 4; x++) lo |= (uint32_t)jpg_idct_limit(o[x]) << (8 * x);
        for (int x = 0; x < 4; x++) hi |= (uint32_t)jpg_idct_limit(o[4 + x]) << (8 * x);
        uint8_t *dst = planes + F.plane_off[comp] + (int64_t)(by * 8 + r) * F.plane_w[comp] + bx * 8;
        *reinterpret_cast<uint2 *>(dst) = make_uint2(lo, hi);
    }
}

// ---- 6. upsampling and colour ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) jpg_color_kernel(const jpg_file *files, const int32_t *status,
                                                        const uint8_t *planes)
{
    ms_pdl_wait();
    const jpg_file &F = files[blockIdx.y];
    if (status[F.index] || !F.out) return;
    const int64_t npx = (int64_t)F.h * F.w;
    const uint8_t *p0 = planes + F.plane_off[0];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (int64_t)gridDim.x * blockDim.x) {
        const int y = (int)(i / F.w), x = (int)(i - (int64_t)y * F.w);
        uint8_t *px = F.out + i * 3;
        const int Y = p0[(int64_t)y * F.plane_w[0] + x];
        if (F.ncomp == 1) {
            px[0] = px[1] = px[2] = (uint8_t)Y;
            continue;
        }
        const int cb = jpg_chroma(planes + F.plane_off[1], F.plane_w[1], F.comp_w[1], F.comp_h[1], x, y, F.hs, F.vs,
                                  F.up);
        const int cr = jpg_chroma(planes + F.plane_off[2], F.plane_w[2], F.comp_w[2], F.comp_h[2], x, y, F.hs, F.vs,
                                  F.up);
        uint8_t rgb[3];
        jpg_ycc_rgb(Y, cb, cr, rgb);
        px[0] = rgb[0];
        px[1] = rgb[1];
        px[2] = rgb[2];
    }
}

// ---- entry points ---------------------------------------------------------------------------------------------------
extern "C" int ms_jpeg_inspect_host(const uint8_t *data, int64_t size, ms_jpeg_info *out)
{
    if (!data || !out || size < 0) {
        ms_set_error("ms_jpeg_inspect_host: NULL argument");
        return MS_ERR_INVALID;
    }
    static thread_local jpg_parsed p;
    jpg_parse(data, size, p);
    *out = p.info;
    return MS_OK;
}

static inline size_t jpg_al16(size_t b) { return (b + 15) & ~size_t(15); }

int ms_jpeg_decode_batch_impl(ms_ctx *ctx, const uint8_t *const *files, const int64_t *sizes, int n,
                              uint8_t *const *out_pages, int32_t *out_status, cudaStream_t st)
{
    // ---- parse, lay out ----
    std::vector<jpg_file> fv;
    std::vector<const uint8_t *> srcp;
    std::vector<int32_t> status(n);
    std::vector<int32_t> chunk_file, sub_file;
    int64_t src_bytes = 0, unst_bytes = 0, blocks = 0, plane_bytes = 0, max_px = 0;
    int32_t nseg_total = 0, nchunk = 0, nsub = 0;
    {
        jpg_parsed *p = new (std::nothrow) jpg_parsed;
        if (!p) {
            ms_set_error("ms_jpeg_decode_batch: out of host memory");
            return MS_ERR_INVALID;
        }
        for (int i = 0; i < n; i++) {
            jpg_parse(files[i], files[i] ? sizes[i] : 0, *p);
            status[i] = p->info.device ? MS_JPEG_OK : p->info.reason;
            if (!p->info.device) continue;
            if (!out_pages[i]) {
                status[i] = MS_JPEG_SCAN;
                continue;
            }
            jpg_file F = p->F;
            F.index = i;
            F.out = out_pages[i];
            F.src_off = src_bytes;
            src_bytes += jpg_al16(F.src_len + 1);
            F.unst_off = unst_bytes;
            unst_bytes += jpg_al16(F.src_len + 32);
            F.coef_off = blocks;
            blocks += (int64_t)F.mcux * F.mcuy * F.bpm;
            for (int k = 0; k < F.ncomp; k++) {
                F.plane_off[k] = plane_bytes;
                plane_bytes += jpg_al16((size_t)F.plane_w[k] * F.plane_h[k]);
            }
            F.seg_off = nseg_total;
            nseg_total += F.nseg + 1;
            F.chunk_off = nchunk;
            F.nchunk = (int32_t)((F.src_len + JPG_CHUNK - 1) / JPG_CHUNK);
            if (F.nchunk < 1) F.nchunk = 1;
            nchunk += F.nchunk;
            F.sub_off = nsub;
            int64_t ns = ((int64_t)F.src_len * 8 + JPG_SUB_BITS - 1) / JPG_SUB_BITS;
            F.nsub = (int32_t)((ns + JPG_SUB_CTA - 1) / JPG_SUB_CTA * JPG_SUB_CTA);
            if (F.nsub < JPG_SUB_CTA) F.nsub = JPG_SUB_CTA;
            nsub += F.nsub;
            const int fi = (int)fv.size();
            for (int c = 0; c < F.nchunk; c++) chunk_file.push_back(fi);
            for (int c = 0; c < F.nsub / JPG_SUB_CTA; c++) sub_file.push_back(fi);
            if ((int64_t)F.h * F.w > max_px) max_px = (int64_t)F.h * F.w;
            fv.push_back(F);
            srcp.push_back(files[i] + p->scan_off);
        }
        delete p;
    }
    const int nf = (int)fv.size();
    if (nf == 0) {
        memcpy(out_status, status.data(), sizeof(int32_t) * n);
        return MS_OK;
    }
    // ---- host staging: descriptors, maps, per-file state, statuses, entropy-coded bytes; one copy ----
    std::vector<jpg_fstate> fs0(nf);
    for (int i = 0; i < nf; i++) fs0[i] = jpg_fstate{(unsigned long long)fv[i].src_len, 0, 0};
    const size_t o_files = 0, o_cf = jpg_al16(o_files + sizeof(jpg_file) * nf);
    const size_t o_sf = jpg_al16(o_cf + sizeof(int32_t) * nchunk), o_fs = jpg_al16(o_sf + sizeof(int32_t) * sub_file.size());
    const size_t o_st = jpg_al16(o_fs + sizeof(jpg_fstate) * nf), o_src = jpg_al16(o_st + sizeof(int32_t) * n);
    const size_t stage_bytes = o_src + (size_t)src_bytes;
    if (ctx->jpeg_pending) {  // the previous call's copy out of the pinned buffer
        MS_CUDA(cudaEventSynchronize(ctx->jpeg_ev));
        ctx->jpeg_pending = 0;
    }
    if (stage_bytes > ctx->jpeg_pinned_bytes) {
        if (ctx->jpeg_pinned) MS_CUDA(cudaFreeHost(ctx->jpeg_pinned));
        ctx->jpeg_pinned = nullptr;
        ctx->jpeg_pinned_bytes = 0;
        const size_t want = stage_bytes + stage_bytes / 4 + (1 << 20);
        MS_CUDA(cudaMallocHost((void **)&ctx->jpeg_pinned, want));
        ctx->jpeg_pinned_bytes = want;
    }
    char *h = ctx->jpeg_pinned;
    memcpy(h + o_files, fv.data(), sizeof(jpg_file) * nf);
    memcpy(h + o_cf, chunk_file.data(), sizeof(int32_t) * nchunk);
    memcpy(h + o_sf, sub_file.data(), sizeof(int32_t) * sub_file.size());
    memcpy(h + o_fs, fs0.data(), sizeof(jpg_fstate) * nf);
    memcpy(h + o_st, status.data(), sizeof(int32_t) * n);
    for (int i = 0; i < nf; i++) memcpy(h + o_src + fv[i].src_off, srcp[i], (size_t)fv[i].src_len);

    // ---- device scratch from the arena ----
    char *stage_d = nullptr;
    int32_t *chunk_kept = nullptr, *chunk_rst = nullptr, *count = nullptr, *base = nullptr;
    uint32_t *seg = nullptr;
    uint8_t *unst = nullptr, *planes = nullptr;
    uint64_t *entry = nullptr, *exitv = nullptr;
    int16_t *coef = nullptr;
    auto carve = [&](ms_bump &bp) {
        stage_d = bp.take<char>(stage_bytes);
        chunk_kept = bp.take<int32_t>(nchunk);
        chunk_rst = bp.take<int32_t>(nchunk);
        seg = bp.take<uint32_t>(nseg_total);
        unst = bp.take<uint8_t>((size_t)unst_bytes);
        entry = bp.take<uint64_t>(nsub);
        exitv = bp.take<uint64_t>(nsub);
        count = bp.take<int32_t>(nsub);
        base = bp.take<int32_t>(nsub);
        coef = bp.take<int16_t>((size_t)blocks * 64);
        planes = bp.take<uint8_t>((size_t)plane_bytes + 16);
    };
    ms_bump probe{nullptr, 0, 0};
    carve(probe);
    MS_TRY(ms_arena_reserve(ctx, probe.off));
    ms_bump bp{ctx->arena, 0, ctx->arena_bytes};
    carve(bp);
    MS_CUDA(cudaMemcpyAsync(stage_d, h, stage_bytes, cudaMemcpyHostToDevice, st));
    MS_CUDA(cudaEventRecord(ctx->jpeg_ev, st));
    ctx->jpeg_pending = 1;
    const jpg_file *d_files = reinterpret_cast<const jpg_file *>(stage_d + o_files);
    const int32_t *d_cf = reinterpret_cast<const int32_t *>(stage_d + o_cf);
    const int32_t *d_sf = reinterpret_cast<const int32_t *>(stage_d + o_sf);
    jpg_fstate *d_fs = reinterpret_cast<jpg_fstate *>(stage_d + o_fs);
    int32_t *d_st = reinterpret_cast<int32_t *>(stage_d + o_st);
    const uint8_t *d_src = reinterpret_cast<const uint8_t *>(stage_d + o_src);
    const int nsub_cta = nsub / JPG_SUB_CTA;

    ms_launch(jpg_end_kernel, dim3(nchunk), dim3(256), 0, st, d_files, d_cf, d_src, d_fs, d_st);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_count_kernel, dim3(nchunk), dim3(256), 0, st, d_files, d_cf, d_src, d_fs, chunk_kept, chunk_rst);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_scan_kernel, dim3(nf), dim3(1024), 0, st, d_files, d_src, d_fs, chunk_kept, chunk_rst, seg, unst,
              d_st);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_emit_kernel, dim3(nchunk), dim3(256), 0, st, d_files, d_cf, d_src, d_fs, chunk_kept, chunk_rst, seg,
              unst, d_st);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_guess_kernel, dim3(nsub_cta), dim3(JPG_SUB_CTA), 0, st, d_files, d_sf, unst, seg, d_st, entry, exitv,
              count);
    MS_LAUNCH_CHECK(ctx);
    for (int r = 0; r < JPG_SYNC_ROUNDS; r++) {
        ms_launch(jpg_sync_kernel, dim3(nsub_cta), dim3(JPG_SUB_CTA), 0, st, d_files, d_sf, unst, seg, d_st, entry,
                  exitv, count);
        MS_LAUNCH_CHECK(ctx);
    }
    ms_launch(jpg_fix_kernel, dim3(nf), dim3(32), 0, st, d_files, unst, seg, d_st, entry, exitv, count);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_base_kernel, dim3(nf), dim3(1024), 0, st, d_files, count, base, d_st);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_write_kernel, dim3(nsub_cta), dim3(JPG_SUB_CTA), 0, st, d_files, d_sf, unst, seg, d_st, entry, base,
              coef);
    MS_LAUNCH_CHECK(ctx);
    ms_launch(jpg_dc_kernel, dim3(nf, 3), dim3(1024), 0, st, d_files, d_st, coef);
    MS_LAUNCH_CHECK(ctx);
    const int64_t idct_ctas = (blocks + 31) / 32;
    ms_launch(jpg_idct_kernel, dim3((unsigned)idct_ctas), dim3(256), 0, st, d_files, nf, d_st, coef, blocks, planes);
    MS_LAUNCH_CHECK(ctx);
    int gx = (int)((max_px + 255) / 256);
    const int cap = 4 * ctx->num_sms * 8 / nf + 1;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    ms_launch(jpg_color_kernel, dim3(gx, nf), dim3(256), 0, st, d_files, d_st, planes);
    MS_LAUNCH_CHECK(ctx);
    MS_CUDA(cudaMemcpyAsync(out_status, d_st, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    return MS_OK;
}
