// Baseline-JPEG decode: the marker parser (host) and the per-thread routines of the device decode (jpeg.cu), written
// once for both sides so that the entropy decode, the IDCT, the upsampling and the colour conversion are the code the
// kernels run.  The arithmetic restates libjpeg-turbo's (the library cv2.imread calls): jdhuff.c decode_mcu,
// jidctint.c jpeg_idct_islow, jdsample.c (fancy h2v1 / h1v2 / h2v2, plain replication) and jdcolor.c ycc_rgb_convert.
#pragma once
#include <stdint.h>
#include <string.h>

#include "../../include/manuscript_b200.h"

#if defined(__CUDACC__)
#define JPG_HD __host__ __device__ __forceinline__
#else
#define JPG_HD inline
#endif

#define JPG_SUB_BITS 1024     // bits of unstuffed entropy data per decode thread (one subsequence)
#define JPG_SUB_CTA 128       // subsequences per CTA; a CTA never spans two files
#define JPG_MAX_BPM 10        // blocks per MCU of the supported samplings (4:2:0 and 4:1:1: 6)
#define JPG_MAX_BYTES (256u << 20)  // larger entropy segments go to the host (bit offsets are 32-bit)

// status / reason codes (include/manuscript_b200.h)
#define JPG_ST_ENTROPY MS_JPEG_BAD_ENTROPY

// One Huffman table as decoded on the device: a 9-bit lookahead (len << 8 | symbol, 0 = code longer than 9 bits or
// none) and libjpeg's maxcode / valoffset for the longer codes.
struct alignas(16) jpg_huff {
    uint16_t lut[512];
    int32_t maxcode[18];
    int32_t valoff[18];
    uint8_t vals[256];
};

// One file of a device batch.  Block b of the scan is MCU b / bpm, block b % bpm of it.
struct jpg_file {
    int64_t src_off;            // staged entropy-coded bytes (from the end of the SOS header to the end of the file)
    int64_t src_len;
    int64_t unst_off;           // unstuffed bytes (words of 4, big-endian), capacity src_len + 16
    int64_t coef_off;           // first block in the coefficient buffer
    int64_t plane_off[3];       // component planes (u8, plane_w x plane_h)
    uint8_t *out;               // (h, w, 3) RGB on the device
    int32_t index;              // position in the caller's list
    int32_t h, w, ncomp, bpm, mcux, mcuy, ri, nseg;
    int32_t seg_off;            // nseg + 1 entries of the segment-start table (bit offsets)
    int32_t sub_off, nsub;      // subsequences (nsub a multiple of JPG_SUB_CTA)
    int32_t chunk_off, nchunk;  // 4 KB chunks of the entropy-coded bytes
    int32_t hs, vs;             // luma sampling (chroma is 1x1)
    int32_t plane_w[3], plane_h[3], comp_w[3], comp_h[3], comp_h_blocks[3];
    int32_t up;                 // chroma upsampling: 0 none, 1 fancy, 2 replication
    int8_t comp_of[JPG_MAX_BPM], blk_x[JPG_MAX_BPM], blk_y[JPG_MAX_BPM], first_of[3];
    uint16_t q[3][64];          // dequantisation, natural order
    jpg_huff dc[3], ac[3];
};

// natural order of the k-th zigzag coefficient (jutils.c jpeg_natural_order)
#define JPG_ZIGZAG                                                                                                   \
    {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,   \
     7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46,  \
     53, 60, 61, 54, 47, 55, 62, 63}
static const uint8_t jpg_zz_host[64] = JPG_ZIGZAG;
#if defined(__CUDACC__)
static __constant__ uint8_t jpg_zz_dev[64] = JPG_ZIGZAG;
#endif
JPG_HD int jpg_natural(int k)
{
#if defined(__CUDA_ARCH__)
    return jpg_zz_dev[k];
#else
    return jpg_zz_host[k];
#endif
}

// ---- bits ---------------------------------------------------------------------------------------------------------
JPG_HD uint32_t jpg_bswap(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, 0, 0x0123);
#else
    return (x >> 24) | ((x >> 8) & 0xFF00u) | ((x << 8) & 0xFF0000u) | (x << 24);
#endif
}

// the 32 bits of the stream from bit p on (words: the unstuffed bytes as little-endian u32 loads)
JPG_HD uint32_t jpg_peek32(const uint32_t *words, uint32_t p)
{
    uint32_t i = p >> 5, s = p & 31;
    uint32_t w0 = jpg_bswap(words[i]), w1 = jpg_bswap(words[i + 1]);
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(w1, w0, s);
#else
    return s ? (w0 << s) | (w1 >> (32 - s)) : w0;
#endif
}

// one code of table h from the top bits of w: length (0 = invalid) and symbol
JPG_HD int jpg_huff_decode(const jpg_huff *h, uint32_t w, int &sym)
{
    uint32_t e = h->lut[w >> 23];
    if (e) {
        sym = e & 0xFF;
        return (int)(e >> 8);
    }
    for (int l = 10; l <= 16; l++) {
        int32_t code = (int32_t)(w >> (32 - l));
        if (code <= h->maxcode[l]) {
            sym = h->vals[(code + h->valoff[l]) & 0xFF];
            return l;
        }
    }
    return 0;
}

// HUFF_EXTEND
JPG_HD int jpg_extend(uint32_t v, int s) { return (v < (1u << (s - 1))) ? (int)v + (int)((~0u << s) + 1u) : (int)v; }

// One block (jdhuff.c decode_mcu for one block, DC as the difference) from bit p; none of its bits may reach `end`.
// blk (64 int16, zeroed by the caller) receives the coefficients in natural order when not NULL.  Returns false on an
// invalid code, a code or value crossing `end`, or a coefficient index past 63 (the device leaves those to the host).
JPG_HD bool jpg_decode_block(const uint32_t *words, uint32_t p, uint32_t end, const jpg_huff *dc, const jpg_huff *ac,
                             uint32_t &p_out, int16_t *blk)
{
    int sym;
    uint32_t w = jpg_peek32(words, p);
    int len = jpg_huff_decode(dc, w, sym);
    if (!len || sym > 15) return false;
    uint32_t p2 = p + (uint32_t)(len + sym);
    if (p2 > end) return false;
    if (blk) blk[0] = sym ? (int16_t)jpg_extend((w << len) >> (32 - sym), sym) : (int16_t)0;
    p = p2;
    for (int k = 1; k < 64;) {
        w = jpg_peek32(words, p);
        len = jpg_huff_decode(ac, w, sym);
        if (!len) return false;
        int r = sym >> 4, s = sym & 15;
        if (s) {
            k += r;
            if (k > 63) return false;
            p2 = p + (uint32_t)(len + s);
            if (p2 > end) return false;
            if (blk) blk[jpg_natural(k)] = (int16_t)jpg_extend((w << len) >> (32 - s), s);
            k++;
        } else {
            p2 = p + (uint32_t)len;
            if (p2 > end) return false;
            if (r != 15) {
                p = p2;
                break;
            }
            k += 16;
        }
        p = p2;
    }
    p_out = p;
    return true;
}

// A decode state at a block boundary: bit position and block within the MCU.
JPG_HD uint64_t jpg_state(uint32_t p, int c) { return ((uint64_t)p << 8) | (uint32_t)c; }
JPG_HD uint32_t jpg_state_p(uint64_t s) { return (uint32_t)(s >> 8); }
JPG_HD int jpg_state_c(uint64_t s) { return (int)(s & 0xFF); }

// Decodes the blocks that start in [entry, sub_end) -- a block that starts before sub_end is finished even when it ends
// past it -- and returns the state after them.  seg (nseg + 1 bit offsets): restart intervals; an interval's first
// block starts in a known state (c = 0), and a block that fails to decode is retried one bit later, so a thread that
// started from a wrong guess still reaches some state deterministically.  Started from the true state, the blocks and
// the exit state are those of the file.  With `coef` (WRITE) the blocks are stored from block index blk0 on and every
// interval is checked: first block at index s * ri * bpm, no block past its end, no failure before its end (*bad).
template <bool WRITE>
JPG_HD uint64_t jpg_run(const jpg_file &F, const jpg_huff *dc, const jpg_huff *ac, const int8_t *comp_of,
                        const uint32_t *words, const uint32_t *seg, uint64_t entry, uint32_t sub_end, int32_t &count,
                        int16_t *coef, int64_t blk0, int32_t *bad)
{
    uint32_t p = jpg_state_p(entry);
    int c = jpg_state_c(entry);
    const int nseg = F.nseg;
    const uint32_t total = seg[nseg];
    int32_t n = 0;
    if (p >= total) {
        count = 0;
        return jpg_state(total, 0);
    }
    int lo = 0, hi = nseg - 1;  // last segment with seg[s] <= p
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (seg[mid] <= p) lo = mid;
        else hi = mid - 1;
    }
    int s = lo;
    uint32_t seg_end = seg[s + 1];
    const int64_t per_seg = F.ri > 0 ? (int64_t)F.ri * F.bpm : (int64_t)F.mcux * F.mcuy * F.bpm;
    const int64_t total_blocks = (int64_t)F.mcux * F.mcuy * F.bpm;
    bool checked = false;
    for (;;) {
        if (p >= seg_end) {
            if (s + 1 >= nseg) {
                p = total;
                c = 0;
                break;
            }
            s++;
            p = seg[s];
            seg_end = seg[s + 1];
            c = 0;
            checked = false;
            continue;
        }
        if (p >= sub_end) break;
        const int64_t b = blk0 + n;
        int64_t s_end = (int64_t)(s + 1) * per_seg;
        if (s_end > total_blocks) s_end = total_blocks;
        if (WRITE && !checked && p == seg[s]) {
            if (b != (int64_t)s * per_seg) *bad = 1;
            checked = true;
        }
        const int comp = comp_of[c];
        int16_t *blk = nullptr;
        if (WRITE && b < s_end && b >= (int64_t)s * per_seg) {
            blk = coef + b * 64;
            for (int i = 0; i < 64; i++) blk[i] = 0;
        }
        uint32_t p2;
        if (!jpg_decode_block(words, p, seg_end, dc + comp, ac + comp, p2, blk)) {
            if (WRITE && b < s_end) *bad = 1;
            p++;
            continue;
        }
        if (WRITE && b >= s_end) *bad = 1;
        p = p2;
        c = (c + 1 == F.bpm) ? 0 : c + 1;
        n++;
    }
    count = n;
    return jpg_state(p, c);
}

// ---- IDCT (jidctint.c jpeg_idct_islow) ---------------------------------------------------------------------------
#define JPG_FIX_0_298631336 2446
#define JPG_FIX_0_390180644 3196
#define JPG_FIX_0_541196100 4433
#define JPG_FIX_0_765366865 6270
#define JPG_FIX_0_899976223 7373
#define JPG_FIX_1_175875602 9633
#define JPG_FIX_1_501321110 12299
#define JPG_FIX_1_847759065 15137
#define JPG_FIX_1_961570560 16069
#define JPG_FIX_2_053119869 16819
#define JPG_FIX_2_562915447 20995
#define JPG_FIX_3_072711026 25172

// one 1-D pass on v[0..7] (dequantised), results DESCALEd by `shift` into o[0..7]
JPG_HD void jpg_idct_1d(const int32_t *v, int32_t *o, int shift)
{
    int32_t z2 = v[2], z3 = v[6];
    int32_t z1 = (z2 + z3) * JPG_FIX_0_541196100;
    int32_t tmp2 = z1 + z3 * (-JPG_FIX_1_847759065);
    int32_t tmp3 = z1 + z2 * JPG_FIX_0_765366865;
    int32_t tmp0 = (int32_t)((uint32_t)(v[0] + v[4]) << 13);
    int32_t tmp1 = (int32_t)((uint32_t)(v[0] - v[4]) << 13);
    int32_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = v[7];
    tmp1 = v[5];
    tmp2 = v[3];
    tmp3 = v[1];
    z1 = tmp0 + tmp3;
    z2 = tmp1 + tmp2;
    z3 = tmp0 + tmp2;
    int32_t z4 = tmp1 + tmp3;
    int32_t z5 = (z3 + z4) * JPG_FIX_1_175875602;
    tmp0 = tmp0 * JPG_FIX_0_298631336;
    tmp1 = tmp1 * JPG_FIX_2_053119869;
    tmp2 = tmp2 * JPG_FIX_3_072711026;
    tmp3 = tmp3 * JPG_FIX_1_501321110;
    z1 = z1 * (-JPG_FIX_0_899976223);
    z2 = z2 * (-JPG_FIX_2_562915447);
    z3 = z3 * (-JPG_FIX_1_961570560);
    z4 = z4 * (-JPG_FIX_0_390180644);
    z3 += z5;
    z4 += z5;
    tmp0 += z1 + z3;
    tmp1 += z2 + z4;
    tmp2 += z2 + z3;
    tmp3 += z1 + z4;
    const int32_t r = 1 << (shift - 1);
    o[0] = (tmp10 + tmp3 + r) >> shift;
    o[7] = (tmp10 - tmp3 + r) >> shift;
    o[1] = (tmp11 + tmp2 + r) >> shift;
    o[6] = (tmp11 - tmp2 + r) >> shift;
    o[2] = (tmp12 + tmp1 + r) >> shift;
    o[5] = (tmp12 - tmp1 + r) >> shift;
    o[3] = (tmp13 + tmp0 + r) >> shift;
    o[4] = (tmp13 - tmp0 + r) >> shift;
}

// range_limit[x & RANGE_MASK] of the IDCT output (jdmaster.c prepare_range_limit_table): wraps like the table
JPG_HD uint8_t jpg_idct_limit(int32_t x)
{
    int32_t u = ((x & 1023) + 128) & 1023;
    return u < 256 ? (uint8_t)u : u < 640 ? (uint8_t)255 : (uint8_t)0;
}

// ---- upsampling (jdsample.c) and YCbCr -> RGB (jdcolor.c) ---------------------------------------------------------
// chroma value at output pixel (x, y) from a plane of pitch pw whose component is cw x ch samples
JPG_HD int jpg_chroma(const uint8_t *pl, int pw, int cw, int ch, int x, int y, int hs, int vs, int up)
{
    if (up == 0) return pl[(size_t)y * pw + x];
    if (up == 2) return pl[(size_t)(y / vs) * pw + x / hs];
    if (vs == 1) {  // h2v1
        const uint8_t *row = pl + (size_t)y * pw;
        int j = x >> 1, v = row[j] * 3;
        return (x & 1) ? (v + row[j + 1 < cw ? j + 1 : cw - 1] + 2) >> 2 : (v + row[j > 0 ? j - 1 : 0] + 1) >> 2;
    }
    int r = y >> 1, o = (y & 1) ? (r + 1 < ch ? r + 1 : ch - 1) : (r > 0 ? r - 1 : 0);
    const uint8_t *r0 = pl + (size_t)r * pw, *r1 = pl + (size_t)o * pw;
    if (hs == 1) return (r0[x] * 3 + r1[x] + ((y & 1) ? 2 : 1)) >> 2;  // h1v2
    int j = x >> 1;                                                      // h2v2
    int cs = r0[j] * 3 + r1[j];
    if (x & 1) {
        int jn = j + 1 < cw ? j + 1 : cw - 1;
        return (cs * 3 + r0[jn] * 3 + r1[jn] + 7) >> 4;
    }
    int jp = j > 0 ? j - 1 : 0;
    return (cs * 3 + r0[jp] * 3 + r1[jp] + 8) >> 4;
}

JPG_HD uint8_t jpg_clamp255(int v) { return v < 0 ? 0 : v > 255 ? 255 : (uint8_t)v; }

JPG_HD void jpg_ycc_rgb(int y, int cb, int cr, uint8_t *rgb)
{
    const int32_t half = 1 << 15;
    int32_t xb = cb - 128, xr = cr - 128;
    int32_t r = (91881 * xr + half) >> 16;
    int32_t b = (116130 * xb + half) >> 16;
    int32_t g = ((-22554 * xb + half) + (-46802 * xr)) >> 16;
    rgb[0] = jpg_clamp255(y + r);
    rgb[1] = jpg_clamp255(y + g);
    rgb[2] = jpg_clamp255(y + b);
}

// ---- host: marker parser ------------------------------------------------------------------------------------------
// What the parser learns about one file; `F` is filled for files the device takes (info.device == 1).
struct jpg_parsed {
    ms_jpeg_info info;
    int64_t scan_off;  // first byte of the entropy-coded data
    jpg_file F;
};

static inline int jpg_u16(const uint8_t *p) { return (p[0] << 8) | p[1]; }

static bool jpg_build_huff(const uint8_t *bits, const uint8_t *vals, int nvals, bool is_dc, jpg_huff *h)
{
    memset(h, 0, sizeof(*h));
    int size[257], code[257], n = 0;
    for (int l = 1; l <= 16; l++)
        for (int i = 0; i < bits[l - 1]; i++) size[n++] = l;
    if (n != nvals || n > 256) return false;
    size[n] = 0;
    int c = 0, si = size[0], k = 0;
    while (size[k]) {
        while (size[k] == si) code[k++] = c++;
        if (c >= (1 << si)) return false;
        c <<= 1;
        si++;
    }
    k = 0;
    for (int l = 1; l <= 16; l++) {
        if (bits[l - 1]) {
            h->valoff[l] = k - code[k];
            k += bits[l - 1];
            h->maxcode[l] = code[k - 1];
        } else {
            h->maxcode[l] = -1;
        }
    }
    h->maxcode[17] = 0x7FFFFFFF;
    for (int i = 0; i < n; i++) {
        if (is_dc && vals[i] > 15) return false;
        h->vals[i] = vals[i];
        if (size[i] <= 9) {
            int sh = 9 - size[i];
            for (int j = 0; j < (1 << sh); j++) h->lut[(code[i] << sh) | j] = (uint16_t)((size[i] << 8) | vals[i]);
        }
    }
    return true;
}

// EXIF orientation of an APP1 payload: 1..8, 0 = no orientation tag, -1 = unreadable
static int jpg_exif_orientation(const uint8_t *p, int n)
{
    if (n < 14 || memcmp(p, "Exif\0\0", 6) != 0) return 0;
    const uint8_t *t = p + 6;
    int tn = n - 6;
    bool le;
    if (t[0] == 'I' && t[1] == 'I') le = true;
    else if (t[0] == 'M' && t[1] == 'M') le = false;
    else return -1;
    auto rd16 = [&](int o) -> int { return le ? t[o] | (t[o + 1] << 8) : (t[o] << 8) | t[o + 1]; };
    auto rd32 = [&](int o) -> uint32_t {
        return le ? (uint32_t)t[o] | ((uint32_t)t[o + 1] << 8) | ((uint32_t)t[o + 2] << 16) | ((uint32_t)t[o + 3] << 24)
                  : ((uint32_t)t[o] << 24) | ((uint32_t)t[o + 1] << 16) | ((uint32_t)t[o + 2] << 8) | t[o + 3];
    };
    if (rd16(2) != 42) return -1;
    uint32_t ifd = rd32(4);
    if (ifd + 2 > (uint32_t)tn) return -1;
    int cnt = rd16((int)ifd);
    if (ifd + 2 + 12u * cnt > (uint32_t)tn) return -1;
    for (int i = 0; i < cnt; i++) {
        int e = (int)ifd + 2 + 12 * i;
        if (rd16(e) == 0x0112) {
            int v = rd16(e + 8);
            return (rd16(e + 2) == 3 && v >= 1 && v <= 8) ? v : -1;
        }
    }
    return 0;
}

// Parses the markers up to the first scan.  Fills p.info (size as cv2.imread returns it, decision and reason) and, for a
// device file, p.F's geometry and tables (layout offsets are the caller's).
static void jpg_parse(const uint8_t *d, int64_t n, jpg_parsed &p)
{
    memset(&p, 0, sizeof(p));
    ms_jpeg_info &I = p.info;
    I.reason = MS_JPEG_NOT_JPEG;
    if (!d || n < 4 || d[0] != 0xFF || d[1] != 0xD8) return;
    struct comp {
        int id, h, v, tq, td, ta;
    } cp[4];
    uint8_t qdef[4] = {0, 0, 0, 0}, hdef[8] = {0};
    static thread_local uint16_t qt[4][64];
    static thread_local jpg_huff ht[8];  // dc 0..3, ac 4..7
    int nf = 0, ri = 0, sof = -1, prec = 0, orient = 0;
    bool jfif = false, adobe = false;
    int64_t i = 2;
    for (;;) {
        while (i < n && d[i] != 0xFF) i++;  // garbage between markers: libjpeg skips it with a warning
        while (i < n && d[i] == 0xFF) i++;
        if (i + 2 >= n) return;  // truncated header
        const int m = d[i++];
        if (m == 0xD8 || m == 0xD9 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) return;  // not where a header continues
        const int len = jpg_u16(d + i);
        if (len < 2 || i + len > n) return;
        const uint8_t *s = d + i + 2;
        const int sl = len - 2;
        if (m >= 0xC0 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {  // SOFn
            if (sof >= 0 || sl < 6) return;
            sof = m;
            prec = s[0];
            I.height = jpg_u16(s + 1);
            I.width = jpg_u16(s + 3);
            nf = s[5];
            I.components = nf;
            if (nf < 1 || nf > 4 || sl < 6 + 3 * nf) return;
            for (int k = 0; k < nf; k++) {
                cp[k].id = s[6 + 3 * k];
                cp[k].h = s[7 + 3 * k] >> 4;
                cp[k].v = s[7 + 3 * k] & 15;
                cp[k].tq = s[8 + 3 * k];
                if (cp[k].h < 1 || cp[k].h > 4 || cp[k].v < 1 || cp[k].v > 4 || cp[k].tq > 3) return;
            }
            if (m == 0xC2 || m == 0xC6 || m == 0xCA || m == 0xCE) {
                I.reason = MS_JPEG_PROGRESSIVE;
                break;
            }
        } else if (m == 0xC4) {  // DHT
            int o = 0;
            while (o < sl) {
                if (o + 17 > sl) return;
                int tc = s[o] >> 4, th = s[o] & 15, cnt = 0;
                for (int l = 0; l < 16; l++) cnt += s[o + 1 + l];
                if (tc > 1 || th > 3 || cnt > 256 || o + 17 + cnt > sl) return;
                if (!jpg_build_huff(s + o + 1, s + o + 17, cnt, tc == 0, &ht[tc * 4 + th])) {
                    hdef[tc * 4 + th] = 2;  // defined but unusable: a scan that uses it goes to the host
                } else {
                    hdef[tc * 4 + th] = 1;
                }
                o += 17 + cnt;
            }
        } else if (m == 0xDB) {  // DQT
            int o = 0;
            while (o < sl) {
                int pq = s[o] >> 4, tq = s[o] & 15, sz = pq ? 128 : 64;
                if (pq > 1 || tq > 3 || o + 1 + sz > sl) return;
                for (int k = 0; k < 64; k++)
                    qt[tq][jpg_natural(k)] = pq ? (uint16_t)jpg_u16(s + o + 1 + 2 * k) : s[o + 1 + k];
                qdef[tq] = 1;
                o += 1 + sz;
            }
        } else if (m == 0xDD) {  // DRI
            if (sl < 2) return;
            ri = jpg_u16(s);
        } else if (m == 0xE0) {
            if (sl >= 5 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xE1) {
            int o = jpg_exif_orientation(s, sl);
            if (o != 0 && orient == 0) orient = o;
        } else if (m == 0xEE) {
            if (sl >= 5 && memcmp(s, "Adobe", 5) == 0) adobe = true;
        } else if (m == 0xDA) {  // SOS
            if (sof < 0 || sl < 1) return;
            const int ns = s[0];
            if (ns < 1 || ns > 4 || sl < 1 + 2 * ns + 3) return;
            I.reason = MS_JPEG_OK;
            p.scan_off = i + len;
            if (sof != 0xC0 && sof != 0xC1) I.reason = MS_JPEG_UNSUPPORTED_CODING;
            else if (prec != 8) I.reason = MS_JPEG_UNSUPPORTED_CODING;
            else if (nf != 1 && nf != 3) I.reason = MS_JPEG_COLOR;
            else if (nf == 3 && (adobe || (!jfif && cp[0].id == 82 && cp[1].id == 71 && cp[2].id == 66)))
                I.reason = MS_JPEG_COLOR;
            else if (I.height == 0 || I.width == 0) I.reason = MS_JPEG_SCAN;  // DNL
            if (I.reason == MS_JPEG_OK) {
                if (ns != nf || s[1 + 2 * ns] != 0 || s[2 + 2 * ns] != 63 || s[3 + 2 * ns] != 0)
                    I.reason = MS_JPEG_SCAN;
                for (int k = 0; k < ns && I.reason == MS_JPEG_OK; k++) {
                    if (s[1 + 2 * k] != cp[k].id) I.reason = MS_JPEG_SCAN;
                    cp[k].td = s[2 + 2 * k] >> 4;
                    cp[k].ta = s[2 + 2 * k] & 15;
                    if (cp[k].td > 3 || cp[k].ta > 3 || hdef[cp[k].td] != 1 || hdef[4 + cp[k].ta] != 1 ||
                        !qdef[cp[k].tq])
                        I.reason = MS_JPEG_SCAN;
                }
            }
            if (I.reason == MS_JPEG_OK && nf == 3) {
                const bool chroma11 = cp[1].h == 1 && cp[1].v == 1 && cp[2].h == 1 && cp[2].v == 1;
                const int hs = cp[0].h, vs = cp[0].v;
                const bool luma_ok = (hs == 1 && vs == 1) || (hs == 2 && vs == 1) || (hs == 1 && vs == 2) ||
                                     (hs == 2 && vs == 2) || (hs == 4 && vs == 1);
                if (!chroma11 || !luma_ok) I.reason = MS_JPEG_SAMPLING;
            }
            if (I.reason == MS_JPEG_OK && (orient < 0 || orient > 1)) I.reason = MS_JPEG_ORIENTATION;
            if (I.reason == MS_JPEG_OK && n - p.scan_off > (int64_t)JPG_MAX_BYTES) I.reason = MS_JPEG_SCAN;
            break;
        }
        i += len;
    }
    if (orient >= 5 && orient <= 8) {  // cv2.imread applies the EXIF orientation: transposed size
        int t = I.height;
        I.height = I.width;
        I.width = t;
    }
    if (orient != 0 && orient != 1 && I.reason == MS_JPEG_OK) I.reason = MS_JPEG_ORIENTATION;
    I.luma_h = nf >= 1 ? cp[0].h : 0;
    I.luma_v = nf >= 1 ? cp[0].v : 0;
    I.restart_interval = ri;
    I.device = I.reason == MS_JPEG_OK;
    if (!I.device) return;

    jpg_file &F = p.F;
    F.h = I.height;
    F.w = I.width;
    F.ncomp = nf;
    F.ri = ri;
    if (nf == 1) {  // a one-component scan is non-interleaved: one block per MCU, raster order
        F.hs = F.vs = 1;
        F.bpm = 1;
        F.mcux = (F.w + 7) / 8;
        F.mcuy = (F.h + 7) / 8;
        F.comp_of[0] = 0;
        F.first_of[0] = 0;
        F.plane_w[0] = F.mcux * 8;
        F.plane_h[0] = F.mcuy * 8;
        F.comp_w[0] = F.w;
        F.comp_h[0] = F.h;
        F.comp_h_blocks[0] = 1;
        F.up = 0;
    } else {
        F.hs = cp[0].h;
        F.vs = cp[0].v;
        F.mcux = (F.w + 8 * F.hs - 1) / (8 * F.hs);
        F.mcuy = (F.h + 8 * F.vs - 1) / (8 * F.vs);
        int b = 0;
        for (int k = 0; k < 3; k++) {
            const int h = k == 0 ? F.hs : 1, v = k == 0 ? F.vs : 1;
            F.first_of[k] = (int8_t)b;
            for (int yy = 0; yy < v; yy++)
                for (int xx = 0; xx < h; xx++) {
                    F.comp_of[b] = (int8_t)k;
                    F.blk_x[b] = (int8_t)xx;
                    F.blk_y[b] = (int8_t)yy;
                    b++;
                }
            F.plane_w[k] = F.mcux * h * 8;
            F.plane_h[k] = F.mcuy * v * 8;
            F.comp_w[k] = (int)(((int64_t)F.w * h + F.hs - 1) / F.hs);
            F.comp_h[k] = (int)(((int64_t)F.h * v + F.vs - 1) / F.vs);
            F.comp_h_blocks[k] = h * v;
        }
        F.bpm = b;
        // jdsample.c jinit_upsampler: fancy h2v1 / h2v2 when the chroma is wider than 2 samples, h1v2 always,
        // replication otherwise (and for 4:1:1)
        if (F.hs == 1 && F.vs == 1) F.up = 0;
        else if (F.hs == 1 && F.vs == 2) F.up = 1;
        else if (F.hs == 2 && F.comp_w[1] > 2) F.up = 1;
        else F.up = 2;
    }
    const int64_t mcus = (int64_t)F.mcux * F.mcuy;
    F.nseg = ri > 0 ? (int)((mcus + ri - 1) / ri) : 1;
    for (int k = 0; k < nf; k++) {
        memcpy(F.q[k], qt[cp[k].tq], sizeof(F.q[k]));
        F.dc[k] = ht[cp[k].td];
        F.ac[k] = ht[4 + cp[k].ta];
    }
    F.src_len = n - p.scan_off;
}
