/*
 * rtjpeg_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of the RTjpeg paths of gmerlin-avdecoder this repository rebuilds -- decode (three formats),
 * colour converters, encoder (reference: lib/RTjpeg.c, include/RTjpeg.h).  It exists so that tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline leg can check the CUDA
 * path.  Nothing in the shipped library (gmerlin-avdecoder_b200/) may include,
 * link or call this file.
 *
 * Parity pin: the reference holds no golden vectors for this path (SURVEY.md
 * section 4), so the restatement is pinned against the reference itself,
 * compiled unmodified from /root/reference by oracle/Makefile into
 * oracle/_ref/, and against fixtures under tests/golden/ made by that build.
 */
#ifndef RTJPEG_ORACLE_H
#define RTJPEG_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Dequantisation tables for one quality value (reference: RTjpeg_calc_tbls
 * lib/RTjpeg.c:2344-2369 followed by RTjpeg_idct_init :1208-1217). */
typedef struct {
    int32_t liqt[64];   /* luma, raster order, AAN-scaled   */
    int32_t ciqt[64];   /* chroma, raster order, AAN-scaled */
    int     lb8;        /* #raw 8-bit coefficients after DC, luma   */
    int     cb8;        /* #raw 8-bit coefficients after DC, chroma */
} rtjo_tables;

/* Decoder instance state that survives between frames (reference: RTjpeg_t,
 * include/RTjpeg.h:54-92, decoder-relevant members only). */
typedef struct {
    int         width, height, Q;
    rtjo_tables t;
} rtjo_decoder;

/* Q is clamped to 1..255 exactly as RTjpeg_set_quality does (:2408-2412). */
void rtjo_tables_from_quality(int Q, rtjo_tables *out);

/* 128 raw (pre-AAN) u32 table entries, as RTjpeg_set_tables takes (:2380-2395). */
void rtjo_tables_from_raw(const uint32_t raw[128], rtjo_tables *out);

void rtjo_decoder_reset(rtjo_decoder *d);

/* One packet (12-byte header + payload) into persistent tight-pitch planes.
 * Mirrors RTjpeg_decompress (:3565-3586) with f == RTJ_YUV420.
 * Returns the number of payload bytes consumed, or -1 if the packet would be
 * read past pkt_len (the reference has no such check; the oracle refuses
 * instead of reading out of bounds). */
long rtjo_decode_packet(rtjo_decoder *d, const uint8_t *pkt, size_t pkt_len,
                        uint8_t *y, uint8_t *u, uint8_t *v);

/* Block walker: byte offset (relative to the payload start) of each of the
 * nblocks blocks, 0xFFFFFFFF for a skipped block, plus per-block end-of-block
 * count (number of zig-zag positions up to and including the last coded one;
 * 0 for a skipped block).  Returns payload bytes consumed or -1 on overrun. */
long rtjo_walk_payload(const uint8_t *payload, size_t len, int nblocks_mb6,
                       int lb8, int cb8, uint32_t *offsets, uint8_t *eob);

/* Single 8x8 block primitives, exposed for unit tests. */
int  rtjo_unpack_block(const uint8_t *s, int bt8, const int32_t *iqt, int16_t blk[64]);
void rtjo_idct_block(const int16_t blk[64], uint8_t *dst, int pitch);

/* The other two formats of RTjpeg_decompress (RTjpeg.c:3580-3585): fmt 1 = YUV422
 * (RTjpeg_decompressYUV422 :2639-2686; u, v are (w/2) x h), fmt 2 = 8-bit grey
 * (RTjpeg_decompress8 :2751-2772; u, v unused).  fmt 0 forwards to rtjo_decode_packet. */
size_t rtjo_frame_bytes(int fmt, int w, int h);
long rtjo_decode_packet_fmt(rtjo_decoder *d, int fmt, const uint8_t *pkt, size_t pkt_len,
                            uint8_t *y, uint8_t *u, uint8_t *v);

/* The encoder half (RTjpeg_compress, RTjpeg.c:3488-3524), see rtjpeg_oracle.c. */
typedef struct {
    int      fmt, width, height, Q;
    int32_t  lqt[64], cqt[64];       /* quantiser multipliers, raster order, AAN-divided */
    int      lb8, cb8;
    int      key_rate, key_count, lmask, cmask;
    int      nblk;
    int16_t *old;                    /* the block last sent at every place, stream order */
} rtjo_encoder;
void rtjo_encoder_tables(int Q, int32_t lqt[64], int32_t cqt[64], int *lb8, int *cb8);
void rtjo_fdct_quant(const uint8_t *src, int pitch, const int32_t qt[64], int16_t out[64]);
int  rtjo_pack_block(const int16_t blk[64], int bt8, uint8_t *out);
void rtjo_encoder_init(rtjo_encoder *e, int fmt, int w, int h, int Q, int key_rate, int lm, int cm);
void rtjo_encoder_free(rtjo_encoder *e);
long rtjo_encode_frame(rtjo_encoder *e, const uint8_t *y, const uint8_t *u, const uint8_t *v, uint8_t *out);
/* fmt 2 as the reference codes it, reading up to 56 rows behind the plane (see rtjpeg_oracle.c) */
long rtjo_encode_frame8(rtjo_encoder *e, const uint8_t *y, uint8_t *out);

/* Colour converters of RTjpeg.c:3071-3486 (RTjpeg_yuv420rgb32 ... RTjpeg_yuv422rgb24), see rtjpeg_oracle.c. */
size_t rtjo_convert_bpp(int kind);
void rtjo_convert(int kind, int w, int h, const uint8_t *y, const uint8_t *u, const uint8_t *v,
                  uint8_t *out, size_t pitch);

#ifdef __cplusplus
}
#endif
#endif
