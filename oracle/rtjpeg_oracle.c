/*
 * rtjpeg_oracle.c -- TEST INFRASTRUCTURE ONLY (see rtjpeg_oracle.h).
 *
 * Plain-C restatement of the reference's RTjpeg YUV420 decode, written from
 * the behaviour of /root/reference/lib/RTjpeg.c (non-MMX C path).  Each
 * function cites the reference lines it follows.  The structure is not the
 * reference's: unpacking, the 1-D transform and the macroblock walk are
 * separate table-driven pieces so that tests can exercise them one by one.
 *
 * Pinned by tests/test_oracle.py against (a) the unmodified reference
 * compiled into oracle/_ref/ and (b) tests/golden/ fixtures produced by it.
 */
#include "rtjpeg_oracle.h"

#include <stdlib.h>
#include <string.h>

/* zig-zag position -> raster index.  Same map as RTjpeg_ZZ (RTjpeg.c:59-74),
 * generated here instead of tabulated: anti-diagonals d = r + c, walked
 * downwards (towards larger row) when d is odd... the reference's order is the
 * transpose of JPEG's, i.e. position 1 is raster 8 (row 1, col 0). */
static uint8_t zz_map[64];
static int     zz_ready;

static void zz_build(void)
{
    int k = 0;
    for (int d = 0; d < 15; d++) {
        int lo = d < 8 ? 0 : d - 7;
        int hi = d < 8 ? d : 7;
        /* even diagonals run from (row lo, col hi) to (row hi, col lo)?  The
         * reference sequence 0 | 8 1 | 2 9 16 | 24 17 10 3 | ... shows: odd d
         * starts at the largest row, even d starts at the largest column. */
        if (d & 1) {
            for (int r = hi; r >= lo; r--) zz_map[k++] = (uint8_t)(r * 8 + (d - r));
        } else {
            for (int c = hi; c >= lo; c--) zz_map[k++] = (uint8_t)((d - c) * 8 + c);
        }
    }
    zz_ready = 1;
}

static inline const uint8_t *zz(void)
{
    if (!zz_ready) zz_build();
    return zz_map;
}

/* JPEG Annex K base tables, raster order (RTjpeg.c:87-107). */
static const uint8_t base_luma[64] = {
    16, 11, 10, 16, 24, 40, 51, 61,   12, 12, 14, 19, 26, 58, 60, 55,
    14, 13, 16, 24, 40, 57, 69, 56,   14, 17, 22, 29, 51, 87, 80, 62,
    18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
    49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99
};
static const uint8_t base_chroma[64] = {
    17, 18, 24, 47, 99, 99, 99, 99,   18, 21, 26, 66, 99, 99, 99, 99,
    24, 26, 56, 99, 99, 99, 99, 99,   47, 66, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99,   99, 99, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99,   99, 99, 99, 99, 99, 99, 99, 99
};

/* AAN scale factors in Q32 (RTjpeg.c:76-85).  The table is separable:
 * entry (r,c) = round-to-table of s[r]*s[c]*2^32 with s[0]=1,
 * s[k]=sqrt(2)*cos(k*pi/16); the reference stores the rounded products, so
 * they are tabulated (8x8 symmetric) rather than recomputed in floating point. */
static const uint64_t aan_q32[64] = {
    4294967296ULL, 5957222912ULL, 5611718144ULL, 5050464768ULL, 4294967296ULL, 3374581504ULL, 2324432128ULL, 1184891264ULL,
    5957222912ULL, 8263040512ULL, 7783580160ULL, 7005009920ULL, 5957222912ULL, 4680582144ULL, 3224107520ULL, 1643641088ULL,
    5611718144ULL, 7783580160ULL, 7331904512ULL, 6598688768ULL, 5611718144ULL, 4408998912ULL, 3036936960ULL, 1548224000ULL,
    5050464768ULL, 7005009920ULL, 6598688768ULL, 5938608128ULL, 5050464768ULL, 3968072960ULL, 2733115392ULL, 1393296000ULL,
    4294967296ULL, 5957222912ULL, 5611718144ULL, 5050464768ULL, 4294967296ULL, 3374581504ULL, 2324432128ULL, 1184891264ULL,
    3374581504ULL, 4680582144ULL, 4408998912ULL, 3968072960ULL, 3374581504ULL, 2651326208ULL, 1826357504ULL, 931136000ULL,
    2324432128ULL, 3224107520ULL, 3036936960ULL, 2733115392ULL, 2324432128ULL, 1826357504ULL, 1258030336ULL, 641204288ULL,
    1184891264ULL, 1643641088ULL, 1548224000ULL, 1393296000ULL, 1184891264ULL, 931136000ULL, 641204288ULL, 326894240ULL
};

/* Number of leading zig-zag AC positions whose pre-AAN dequantiser is <= 8:
 * those coefficients travel as raw signed bytes (RTjpeg.c:2362-2367, and the
 * same loop in set_tables :2388-2393).  The reference loop has no upper bound;
 * it is capped at 63 here (a table that is <= 8 everywhere). */
static int raw_prefix_len(const int32_t *pre)
{
    const uint8_t *z = zz();
    int k = 0;
    while (k < 63 && pre[z[k + 1]] <= 8) k++;
    return k;
}

static void apply_aan(int32_t *t)
{
    /* RTjpeg_idct_init, RTjpeg.c:1208-1217 */
    for (int i = 0; i < 64; i++)
        t[i] = (int32_t)(((uint64_t)(uint32_t)t[i] * aan_q32[i]) >> 32);
}

void rtjo_tables_from_quality(int Q, rtjo_tables *out)
{
    /* RTjpeg_set_quality :2408-2412 clamps, RTjpeg_calc_tbls :2344-2361 derives */
    if (Q < 1) Q = 1;
    if (Q > 255) Q = 255;
    uint64_t qual = (uint64_t)Q << 25;
    for (int i = 0; i < 64; i++) {
        int32_t lq = (int32_t)((qual / ((uint64_t)base_luma[i] << 16)) >> 3);
        int32_t cq = (int32_t)((qual / ((uint64_t)base_chroma[i] << 16)) >> 3);
        if (lq == 0) lq = 1;
        if (cq == 0) cq = 1;
        out->liqt[i] = 65536 / (lq << 3);
        out->ciqt[i] = 65536 / (cq << 3);
    }
    out->lb8 = raw_prefix_len(out->liqt);
    out->cb8 = raw_prefix_len(out->ciqt);
    apply_aan(out->liqt);
    apply_aan(out->ciqt);
}

void rtjo_tables_from_raw(const uint32_t raw[128], rtjo_tables *out)
{
    /* RTjpeg_set_tables :2380-2395 */
    for (int i = 0; i < 64; i++) {
        out->liqt[i] = (int32_t)raw[i];
        out->ciqt[i] = (int32_t)raw[64 + i];
    }
    out->lb8 = raw_prefix_len(out->liqt);
    out->cb8 = raw_prefix_len(out->ciqt);
    apply_aan(out->liqt);
    apply_aan(out->ciqt);
}

void rtjo_decoder_reset(rtjo_decoder *d)
{
    /* RTjpeg_init :2495-2502: everything zero, so format 0 = YUV420 and no tables */
    memset(d, 0, sizeof(*d));
}

/* Byte length of the block that starts at s (1 for a skip marker), without
 * touching coefficients; *eob receives the count of zig-zag positions up to the
 * last explicitly coded one.  Grammar: RTjpeg_s2b, RTjpeg.c:157-186. */
static int block_extent(const uint8_t *s, size_t avail, int bt8, int *eob)
{
    if (avail < 1) return -1;
    if (s[0] == 0xFF) { *eob = 0; return 1; }
    size_t n = 1 + (size_t)bt8;          /* DC + raw bytes */
    int pos = 1 + bt8;                   /* next zig-zag position to fill */
    int last = pos;                      /* positions 0..bt8 are always explicit */
    if (n > avail) return -1;
    while (pos < 64) {
        if (n >= avail) return -1;
        int8_t b = (int8_t)s[n++];
        if (b > 63) pos += b - 63;       /* run of zeros */
        else { pos++; last = pos; }      /* one coefficient */
    }
    *eob = last;
    return (int)n;
}

int rtjo_unpack_block(const uint8_t *s, int bt8, const int32_t *iqt, int16_t blk[64])
{
    /* RTjpeg_s2b :157-186.  Products are formed in uint32 and truncated to
     * int16, exactly like `data[i] = strm[ci] * qtbl[i]` with qtbl uint32_t*. */
    const uint8_t *z = zz();
    memset(blk, 0, 64 * sizeof(int16_t));
    blk[0] = (int16_t)((uint32_t)s[0] * (uint32_t)iqt[0]);
    int n = 1, pos = 1;
    for (; pos <= bt8; pos++, n++)
        blk[z[pos]] = (int16_t)((uint32_t)(int32_t)(int8_t)s[n] * (uint32_t)iqt[z[pos]]);
    while (pos < 64) {
        int8_t b = (int8_t)s[n++];
        if (b > 63) {
            pos += b - 63;
        } else {
            blk[z[pos]] = (int16_t)((uint32_t)(int32_t)b * (uint32_t)iqt[z[pos]]);
            pos++;
        }
    }
    return n;
}

/* Fixed-point multiply of the reference (MULTIPLY, RTjpeg.c:1206): constants
 * carry 8 fractional bits, rounding is +128 then arithmetic shift. */
static inline int32_t fxmul(int32_t v, int32_t c) { return (int32_t)(v * c + 128) >> 8; }

/* One 8-point pass (RTjpeg.c:2240-2283 for columns, :2289-2326 for rows; both
 * passes run the same flow graph).  in[] natural order, out[] natural order. */
static void aan8(const int32_t in[8], int32_t out[8])
{
    enum { C1 = 277, C2 = 362, C3 = 473, C4 = 669 };
    int32_t s04 = in[0] + in[4], d04 = in[0] - in[4];
    int32_t s26 = in[2] + in[6];
    int32_t m26 = fxmul(in[2] - in[6], C2) - s26;
    int32_t e0 = s04 + s26, e3 = s04 - s26, e1 = d04 + m26, e2 = d04 - m26;

    int32_t z13 = in[5] + in[3], z10 = in[5] - in[3];
    int32_t z11 = in[1] + in[7], z12 = in[1] - in[7];
    int32_t o7 = z11 + z13;
    int32_t o11 = fxmul(z11 - z13, C2);
    int32_t z5 = fxmul(z10 + z12, C3);
    int32_t o10 = fxmul(z12, C1) - z5;
    int32_t o12 = fxmul(z10, -C4) + z5;
    int32_t o6 = o12 - o7;
    int32_t o5 = o11 - o6;
    int32_t o4 = o10 + o5;

    out[0] = e0 + o7; out[7] = e0 - o7;
    out[1] = e1 + o6; out[6] = e1 - o6;
    out[2] = e2 + o5; out[5] = e2 - o5;
    out[4] = e3 + o4; out[3] = e3 - o4;
}

void rtjo_idct_block(const int16_t blk[64], uint8_t *dst, int pitch)
{
    /* RTjpeg_idct C path, RTjpeg.c:2209-2332.  The reference's DC-only column
     * shortcut (:2223-2238) is value-identical to the general flow graph
     * because fxmul(0, c) == 0, so it is not special-cased here. */
    int32_t ws[64];
    for (int c = 0; c < 8; c++) {
        int32_t in[8], out[8];
        for (int r = 0; r < 8; r++) in[r] = blk[r * 8 + c];
        aan8(in, out);
        for (int r = 0; r < 8; r++) ws[r * 8 + c] = out[r];
    }
    for (int r = 0; r < 8; r++) {
        int32_t out[8];
        aan8(&ws[r * 8], out);
        for (int c = 0; c < 8; c++) {
            int16_t p = (int16_t)((out[c] + 4) >> 3);      /* DESCALE :1200 */
            dst[r * pitch + c] = (uint8_t)(p > 235 ? 235 : (p < 16 ? 16 : p)); /* RL :1204 */
        }
    }
}

long rtjo_walk_payload(const uint8_t *payload, size_t len, int nmb,
                       int lb8, int cb8, uint32_t *offsets, uint8_t *eob)
{
    size_t at = 0;
    for (int mb = 0; mb < nmb; mb++) {
        for (int k = 0; k < 6; k++) {
            int e;
            int n = block_extent(payload + at, len - at, k < 4 ? lb8 : cb8, &e);
            if (n < 0) return -1;
            if (offsets) offsets[mb * 6 + k] = e ? (uint32_t)at : 0xFFFFFFFFu;
            if (eob) eob[mb * 6 + k] = (uint8_t)e;
            at += (size_t)n;
        }
    }
    return (long)at;
}

long rtjo_decode_packet(rtjo_decoder *d, const uint8_t *pkt, size_t pkt_len,
                        uint8_t *y, uint8_t *u, uint8_t *v)
{
    if (pkt_len < 12) return -1;
    /* header fields, include/RTjpeg.h:100-109 (packed, little endian) */
    int w = pkt[6] | (pkt[7] << 8);
    int h = pkt[8] | (pkt[9] << 8);
    int q = pkt[10];
    /* lazy reconfiguration, RTjpeg_decompress :3568-3579 */
    if (w != d->width || h != d->height) { d->width = w; d->height = h; }
    if (q != d->Q) {
        int qc = q < 1 ? 1 : q;          /* set_quality stores the clamped value */
        d->Q = qc;
        rtjo_tables_from_quality(qc, &d->t);
    }
    const uint8_t *s = pkt + 12;
    size_t left = pkt_len - 12, at = 0;
    int cw = w >> 1;
    int16_t blk[64];
    /* macroblock walk, RTjpeg_decompressYUV420 :2688-2749: rows of 16 luma
     * lines, 16 luma columns per step, six blocks Y00 Y01 Y10 Y11 U V */
    for (int my = 0; my < (h >> 4); my++) {
        for (int mx = 0; mx < (w >> 4); mx++) {
            for (int k = 0; k < 6; k++) {
                int bt8 = k < 4 ? d->t.lb8 : d->t.cb8;
                const int32_t *iq = k < 4 ? d->t.liqt : d->t.ciqt;
                int e;
                int n = block_extent(s + at, left - at, bt8, &e);
                if (n < 0) return -1;
                if (e) {
                    uint8_t *dst;
                    int pitch;
                    if (k < 4) {
                        pitch = w;
                        dst = y + (size_t)(my * 16 + (k >> 1) * 8) * w + mx * 16 + (k & 1) * 8;
                    } else {
                        pitch = cw;
                        dst = (k == 4 ? u : v) + (size_t)(my * 8) * cw + mx * 8;
                    }
                    rtjo_unpack_block(s + at, bt8, iq, blk);
                    rtjo_idct_block(blk, dst, pitch);
                }
                at += (size_t)n;
            }
        }
    }
    return (long)at;
}

/* Plane bytes of one picture in the three formats RTjpeg_decompress dispatches on
 * (RTjpeg.c:3580-3585): 0 = YUV420, 1 = YUV422, 2 = 8-bit grey ("RGB8"). */
size_t rtjo_frame_bytes(int fmt, int w, int h)
{
    return fmt == 0 ? (size_t)w * h * 3 / 2 : fmt == 1 ? (size_t)w * h * 2 : (size_t)w * h;
}

long rtjo_decode_packet_fmt(rtjo_decoder *d, int fmt, const uint8_t *pkt, size_t pkt_len,
                            uint8_t *y, uint8_t *u, uint8_t *v)
{
    if (fmt == 0) return rtjo_decode_packet(d, pkt, pkt_len, y, u, v);
    if (pkt_len < 12) return -1;
    int w = pkt[6] | (pkt[7] << 8);
    int h = pkt[8] | (pkt[9] << 8);
    int q = pkt[10];
    if (w != d->width || h != d->height) { d->width = w; d->height = h; }
    if (q != d->Q) {
        int qc = q < 1 ? 1 : q;
        d->Q = qc;
        rtjo_tables_from_quality(qc, &d->t);
    }
    const uint8_t *s = pkt + 12;
    size_t left = pkt_len - 12, at = 0;
    int cw = w >> 1;
    int16_t blk[64];
    if (fmt == 1) {
        /* RTjpeg_decompressYUV422 :2639-2686: rows of 8 lines, 16 luma columns per step, four
         * blocks Y0 Y1 U V; chroma is half width, FULL height */
        for (int by = 0; by < (h >> 3); by++) {
            for (int mx = 0; mx < (w >> 4); mx++) {
                for (int k = 0; k < 4; k++) {
                    int bt8 = k < 2 ? d->t.lb8 : d->t.cb8;
                    const int32_t *iq = k < 2 ? d->t.liqt : d->t.ciqt;
                    int e;
                    int n = block_extent(s + at, left - at, bt8, &e);
                    if (n < 0) return -1;
                    if (e) {
                        uint8_t *dst = k < 2 ? y + (size_t)(by * 8) * w + mx * 16 + k * 8
                                             : (k == 2 ? u : v) + (size_t)(by * 8) * cw + mx * 8;
                        rtjo_unpack_block(s + at, bt8, iq, blk);
                        rtjo_idct_block(blk, dst, k < 2 ? w : cw);
                    }
                    at += (size_t)n;
                }
            }
        }
    } else {
        /* RTjpeg_decompress8 :2751-2772: luma blocks only, raster order */
        for (int by = 0; by < (h >> 3); by++) {
            for (int bx = 0; bx < (w >> 3); bx++) {
                int e;
                int n = block_extent(s + at, left - at, d->t.lb8, &e);
                if (n < 0) return -1;
                if (e) {
                    rtjo_unpack_block(s + at, d->t.lb8, d->t.liqt, blk);
                    rtjo_idct_block(blk, y + (size_t)(by * 8) * w + bx * 8, w);
                }
                at += (size_t)n;
            }
        }
    }
    return (long)at;
}

/* ------------------------------------------------------------------ */
/* colour converters (RTjpeg.c:3071-3486)                              */
/* ------------------------------------------------------------------ */

/* The fixed-point matrix of RTjpeg.c:3071-3075: 16 fractional bits, luma offset 16, chroma offset 128. */
enum { RTJO_KY = 76284, RTJO_KCRR = 76284, RTJO_KCRG = 53281, RTJO_KCBG = 25625, RTJO_KCBB = 132252 };

static inline uint8_t sat8(int32_t v) { return (uint8_t)(v > 255 ? 255 : (v < 0 ? 0 : v)); }

/* one pixel: y, and the chroma pair shared by its 2x1 (4:2:2) or 2x2 (4:2:0) neighbourhood; u = planes[1] is Cb,
 * v = planes[2] is Cr (:3084-3085, :3097-3100) */
static inline void px_rgb(int yv, int cb, int cr, uint8_t *r, uint8_t *g, uint8_t *b)
{
    int32_t y = (yv - 16) * RTJO_KY;
    *r = sat8((y + (cr - 128) * RTJO_KCRR) >> 16);
    *g = sat8((y - (cr - 128) * RTJO_KCRG - (cb - 128) * RTJO_KCBG) >> 16);
    *b = sat8((y + (cb - 128) * RTJO_KCBB) >> 16);
}

size_t rtjo_convert_bpp(int kind)
{
    static const size_t bpp[7] = {4, 4, 3, 3, 2, 1, 3};
    return kind >= 0 && kind < 7 ? bpp[kind] : 0;
}

/* kind: 0 yuv420rgb32 (:3123) 1 yuv420bgr32 (:3192) 2 yuv420rgb24 (:3261) 3 yuv420bgr24 (:3326)
 *       4 yuv420rgb16 (:3391) 5 yuv420rgb8 (:3477, the luma plane copied) 6 yuv422rgb24 (:3077).
 * Row r of the picture is written at out + r * pitch; the fourth byte of a 32-bit pixel is not written,
 * exactly as the reference steps over it (:3147, :3157, ...). */
void rtjo_convert(int kind, int w, int h, const uint8_t *y, const uint8_t *u, const uint8_t *v,
                  uint8_t *out, size_t pitch)
{
    const int cw = w >> 1;
    for (int r = 0; r < h; r++) {
        uint8_t *o = out + (size_t)r * pitch;
        const uint8_t *yr = y + (size_t)r * w;
        if (kind == 5) { memcpy(o, yr, (size_t)w); continue; }
        const size_t crow = (size_t)(kind == 6 ? r : r >> 1) * cw;        /* 4:2:2 chroma has the full height */
        for (int x = 0; x < w; x++) {
            uint8_t R, G, B;
            px_rgb(yr[x], u[crow + (x >> 1)], v[crow + (x >> 1)], &R, &G, &B);
            switch (kind) {
            case 0: o[4 * x] = R; o[4 * x + 1] = G; o[4 * x + 2] = B; break;
            case 1: o[4 * x] = B; o[4 * x + 1] = G; o[4 * x + 2] = R; break;
            case 2: case 6: o[3 * x] = R; o[3 * x + 1] = G; o[3 * x + 2] = B; break;
            case 3: o[3 * x] = B; o[3 * x + 1] = G; o[3 * x + 2] = R; break;
            case 4: {                                                       /* 5-6-5, low byte first (:3420-3425) */
                int t = (B >> 3) | ((G >> 2) << 5) | ((R >> 3) << 11);
                o[2 * x] = (uint8_t)(t & 0xff);
                o[2 * x + 1] = (uint8_t)(t >> 8);
                break;
            }
            default: break;
            }
        }
    }
}

/* ------------------------------------------------------------------ */
/* encoder (RTjpeg_compress, RTjpeg.c:3488-3524)                       */
/* ------------------------------------------------------------------ */

/* Quantiser tables of the encoder for quality Q: RTjpeg_calc_tbls (:2344-2361) makes lqt, liqt = 65536 / (lqt << 3)
 * and folds liqt back into lqt = (65536 / liqt) >> 3; RTjpeg_dct_init (:277-286) then divides by the AAN factors. */
void rtjo_encoder_tables(int Q, int32_t lqt[64], int32_t cqt[64], int *lb8, int *cb8)
{
    rtjo_tables t;
    if (Q < 1) Q = 1;
    if (Q > 255) Q = 255;
    uint64_t qual = (uint64_t)Q << 25;
    int32_t lpre[64], cpre[64];
    for (int i = 0; i < 64; i++) {
        int32_t lq = (int32_t)((qual / ((uint64_t)base_luma[i] << 16)) >> 3);
        int32_t cq = (int32_t)((qual / ((uint64_t)base_chroma[i] << 16)) >> 3);
        if (lq == 0) lq = 1;
        if (cq == 0) cq = 1;
        lpre[i] = 65536 / (lq << 3);
        cpre[i] = 65536 / (cq << 3);
        lq = (65536 / lpre[i]) >> 3;
        cq = (65536 / cpre[i]) >> 3;
        lqt[i] = (int32_t)(((uint64_t)lq << 32) / aan_q32[i]);
        cqt[i] = (int32_t)(((uint64_t)cq << 32) / aan_q32[i]);
    }
    (void)t;
    *lb8 = raw_prefix_len(lpre);
    *cb8 = raw_prefix_len(cpre);
}

/* One 8-point pass of the forward transform (RTjpeg_dctY :303-340 rows, :346-389 columns): the flow graph is the
 * same in both, only what is done with its eight results differs.  in: eight samples; e[0..7]: the results before
 * the pass's own scaling -- e0 = s0 + s1 terms ... as laid out below. */
static void fdct8(const int32_t x[8], int32_t *r0, int32_t *r4, int32_t *r2, int32_t *r6,
                  int32_t *r5, int32_t *r3, int32_t *r1, int32_t *r7)
{
    int32_t t0 = x[0] + x[7], t7 = x[0] - x[7], t1 = x[1] + x[6], t6 = x[1] - x[6];
    int32_t t2 = x[2] + x[5], t5 = x[2] - x[5], t3 = x[3] + x[4], t4 = x[3] - x[4];
    int32_t t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    *r0 = t10 + t11;                     /* scaled by << 8 (rows) or DESCALE10 (columns) by the caller */
    *r4 = t10 - t11;
    int32_t z1 = (t12 + t13) * 181;
    *r2 = (t13 << 8) + z1;
    *r6 = (t13 << 8) - z1;
    t10 = t4 + t5; t11 = t5 + t6; t12 = t6 + t7;
    int32_t z5 = (t10 - t12) * 98, z2 = t10 * 139 + z5, z4 = t12 * 334 + z5, z3 = t11 * 181;
    int32_t z11 = (t7 << 8) + z3, z13 = (t7 << 8) - z3;
    *r5 = z13 + z2; *r3 = z13 - z2; *r1 = z11 + z4; *r7 = z11 - z4;
}

/* RTjpeg_dctY (:288-390) followed by RTjpeg_quant (:245-252): 8x8 samples at src (row pitch `pitch`) -> 64 quantised
 * coefficients in raster order. */
void rtjo_fdct_quant(const uint8_t *src, int pitch, const int32_t qt[64], int16_t out[64])
{
    int32_t ws[64];
    for (int r = 0; r < 8; r++) {
        int32_t x[8], a0, a4;
        for (int c = 0; c < 8; c++) x[c] = src[(size_t)r * pitch + c];
        fdct8(x, &a0, &a4, &ws[r * 8 + 2], &ws[r * 8 + 6], &ws[r * 8 + 5], &ws[r * 8 + 3], &ws[r * 8 + 1], &ws[r * 8 + 7]);
        ws[r * 8 + 0] = a0 << 8;
        ws[r * 8 + 4] = a4 << 8;
    }
    for (int c = 0; c < 8; c++) {
        int32_t x[8], a0, a4, a2, a6, a5, a3, a1, a7;
        for (int r = 0; r < 8; r++) x[r] = ws[r * 8 + c];
        fdct8(x, &a0, &a4, &a2, &a6, &a5, &a3, &a1, &a7);
        int16_t col[8];
        col[0] = (int16_t)((a0 + 128) >> 8);            /* DESCALE10 */
        col[4] = (int16_t)((a4 + 128) >> 8);
        col[2] = (int16_t)((a2 + 32768) >> 16);         /* DESCALE20 */
        col[6] = (int16_t)((a6 + 32768) >> 16);
        col[5] = (int16_t)((a5 + 32768) >> 16);
        col[3] = (int16_t)((a3 + 32768) >> 16);
        col[1] = (int16_t)((a1 + 32768) >> 16);
        col[7] = (int16_t)((a7 + 32768) >> 16);
        for (int r = 0; r < 8; r++) out[r * 8 + c] = col[r];
    }
    for (int i = 0; i < 64; i++) out[i] = (int16_t)((out[i] * qt[i] + 32767) >> 16);
}

/* RTjpeg_b2s (:109-155): DC as an unsigned byte 0..254, bt8 raw signed bytes, then coefficients -64..63 and zero
 * runs 63 + n.  Returns the bytes written (2 + bt8 .. 64). */
int rtjo_pack_block(const int16_t blk[64], int bt8, uint8_t *out)
{
    const uint8_t *z = zz();
    int co = 1, ci;
    int v = blk[z[0]];
    out[0] = (uint8_t)(v > 254 ? 254 : (v < 0 ? 0 : v));
    for (ci = 1; ci <= bt8; ci++) {
        v = blk[z[ci]];
        out[co++] = (uint8_t)(int8_t)(v > 0 ? (v > 127 ? 127 : v) : (v < -128 ? -128 : v));
    }
    for (; ci < 64; ci++) {
        v = blk[z[ci]];
        if (v > 0) out[co++] = (uint8_t)(int8_t)(v > 63 ? 63 : v);
        else if (v < 0) out[co++] = (uint8_t)(int8_t)(v < -64 ? -64 : v);
        else {
            int start = ci;
            do ci++; while (ci < 64 && blk[z[ci]] == 0);
            out[co++] = (uint8_t)(63 + (ci - start));
            ci--;
        }
    }
    return co;
}

void rtjo_encoder_init(rtjo_encoder *e, int fmt, int w, int h, int Q, int key_rate, int lm, int cm)
{
    memset(e, 0, sizeof(*e));
    e->fmt = fmt; e->width = w; e->height = h;
    e->Q = Q < 1 ? 1 : (Q > 255 ? 255 : Q);
    rtjo_encoder_tables(e->Q, e->lqt, e->cqt, &e->lb8, &e->cb8);
    /* RTjpeg_set_intra (:2455-2490) clamps and clears the previous blocks */
    e->key_rate = key_rate < 0 ? 0 : (key_rate > 255 ? 255 : key_rate);
    e->lmask = lm < 0 ? 0 : (lm > 16 ? 16 : lm);
    e->cmask = cm < 0 ? 0 : (cm > 16 ? 16 : cm);
    e->nblk = fmt == 0 ? (w >> 4) * (h >> 4) * 6 : fmt == 1 ? (w >> 4) * (h >> 3) * 4 : (w >> 3) * (h >> 3);
    e->old = (int16_t *)calloc((size_t)e->nblk * 64, sizeof(int16_t));
}

void rtjo_encoder_free(rtjo_encoder *e) { free(e->old); e->old = NULL; }

/* One picture (tight planes) -> one packet at out (12-byte header + block stream); returns its size.
 * RTjpeg_compress (:3488-3524): key_rate == 0 codes every block (RTjpeg_compressYUV420 :2510-2563 and its siblings),
 * otherwise every block is first compared with the block last SENT at its place (RTjpeg_bcomp :2827-2838: a block
 * within +-mask of it in every coefficient becomes the byte 0xFF and leaves the stored block as it is) -- on "key"
 * pictures too, against blocks of zeros (RTjpeg_mcompressYUV420 :2841-2922). */
long rtjo_encode_frame(rtjo_encoder *e, const uint8_t *y, const uint8_t *u, const uint8_t *v, uint8_t *out)
{
    const int w = e->width, h = e->height, cw = w >> 1, fmt = e->fmt;
    /* The 8-bit branch is rtjo_encode_frame8: RTjpeg_compress8 / RTjpeg_mcompress8 hand RTjpeg_dctY the picture
     * width where it expects width / 8 (:2627, :3005; dctY steps rows by rskip << 3, :337), so every block is read
     * with a row stride of 8 * width -- up to 56 rows past the plane, which a tight picture does not have. */
    if (fmt != 0 && fmt != 1) return -1;
    const int inter = e->key_rate != 0;
    if (inter && e->key_count == 0) memset(e->old, 0, (size_t)e->nblk * 64 * sizeof(int16_t));
    uint8_t *sp = out + 12;
    const int unit = fmt == 0 ? 6 : fmt == 1 ? 4 : 1, unit_luma = fmt == 0 ? 4 : fmt == 1 ? 2 : 1;
    const int ux = fmt == 2 ? w >> 3 : w >> 4, uy = fmt == 0 ? h >> 4 : h >> 3;
    int16_t blk[64];
    int16_t *old = e->old;
    for (int gy = 0; gy < uy; gy++)
        for (int gx = 0; gx < ux; gx++)
            for (int k = 0; k < unit; k++) {
                const uint8_t *src;
                int pitch;
                if (k < unit_luma) {
                    pitch = w;
                    if (fmt == 0) src = y + (size_t)(gy * 16 + (k >> 1) * 8) * w + gx * 16 + (k & 1) * 8;
                    else if (fmt == 1) src = y + (size_t)(gy * 8) * w + gx * 16 + k * 8;
                    else src = y + (size_t)(gy * 8) * w + gx * 8;
                } else {
                    pitch = cw;
                    src = (k == unit_luma ? u : v) + (size_t)(gy * 8) * cw + gx * 8;
                }
                const int luma = k < unit_luma;
                rtjo_fdct_quant(src, pitch, luma ? e->lqt : e->cqt, blk);
                int skip = 0;
                if (inter) {
                    const int mask = luma ? e->lmask : e->cmask;
                    skip = 1;
                    for (int i = 0; i < 64; i++)
                        if (abs(old[i] - blk[i]) > mask) { skip = 0; break; }
                    if (!skip) memcpy(old, blk, sizeof(blk));
                    old += 64;
                }
                if (skip) *sp++ = 0xFF;
                else sp += rtjo_pack_block(blk, luma ? e->lb8 : e->cb8, sp);
            }
    const long ds = (long)(sp - out);
    out[0] = (uint8_t)ds; out[1] = (uint8_t)(ds >> 8); out[2] = (uint8_t)(ds >> 16); out[3] = (uint8_t)(ds >> 24);
    out[4] = 12; out[5] = 0;
    out[6] = (uint8_t)w; out[7] = (uint8_t)(w >> 8); out[8] = (uint8_t)h; out[9] = (uint8_t)(h >> 8);
    out[10] = (uint8_t)e->Q;
    out[11] = inter ? (uint8_t)e->key_count : 0;
    if (inter && ++e->key_count > e->key_rate) e->key_count = 0;
    return ds;
}

/* The 8-bit branch as the reference runs it (RTjpeg_compress8, RTjpeg_mcompress8), for a grey plane y that the caller
 * follows with at least 56 * width readable bytes.  Both hand RTjpeg_dctY the picture width where it expects
 * width / 8 (:2627, :3005), so every block is read with a row stride of 8 * width; RTjpeg_compress8 also steps one
 * pixel row (not eight) from a row of blocks to the next, RTjpeg_mcompress8 eight.  What lies behind the plane goes
 * into the packet: the same bytes there give the same packet.  Pinned by the grey fixtures of tests/golden/ on every
 * picture whose reads stay inside the pictures that follow it there. */
long rtjo_encode_frame8(rtjo_encoder *e, const uint8_t *y, uint8_t *out)
{
    const int w = e->width, h = e->height;
    if (e->fmt != 2) return -1;
    const int inter = e->key_rate != 0;
    if (inter && e->key_count == 0) memset(e->old, 0, (size_t)e->nblk * 64 * sizeof(int16_t));
    uint8_t *sp = out + 12;
    int16_t blk[64];
    int16_t *old = e->old;
    for (int by = 0; by < (h >> 3); by++)
        for (int bx = 0; bx < (w >> 3); bx++) {
            rtjo_fdct_quant(y + (size_t)by * (inter ? 8 : 1) * w + bx * 8, 8 * w, e->lqt, blk);
            int skip = 0;
            if (inter) {
                skip = 1;
                for (int i = 0; i < 64; i++)
                    if (abs(old[i] - blk[i]) > e->lmask) { skip = 0; break; }
                if (!skip) memcpy(old, blk, sizeof(blk));
                old += 64;
            }
            if (skip) *sp++ = 0xFF;
            else sp += rtjo_pack_block(blk, e->lb8, sp);
        }
    const long ds = (long)(sp - out);
    out[0] = (uint8_t)ds; out[1] = (uint8_t)(ds >> 8); out[2] = (uint8_t)(ds >> 16); out[3] = (uint8_t)(ds >> 24);
    out[4] = 12; out[5] = 0;
    out[6] = (uint8_t)w; out[7] = (uint8_t)(w >> 8); out[8] = (uint8_t)h; out[9] = (uint8_t)(h >> 8);
    out[10] = (uint8_t)e->Q;
    out[11] = inter ? (uint8_t)e->key_count : 0;
    if (inter && ++e->key_count > e->key_rate) e->key_count = 0;
    return ds;
}
