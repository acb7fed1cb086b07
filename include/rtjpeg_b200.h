/*
 * rtjpeg_b200.h -- C ABI of the B200-native RTjpeg codec (decoder, colour converters, encoder).
 *
 * Two levels, both plain C (pointers and sizes only, no CUDA or torch types):
 *
 *   Level 1  the reference's own codec API, same names, same argument meaning,
 *            so that librtjpeg_b200.so can stand in for lib/RTjpeg.o when
 *            libgmerlin_avdec is linked.  Every prototype cites the reference
 *            declaration it replaces (paths relative to the gmerlin-avdecoder
 *            tree).
 *   Level 2  a batch interface (many packets -> many frames in one call), which
 *            is what keeps a B200 busy; Level 1 is its one-frame special case.
 *
 * Scope: lib/RTjpeg.c -- RTjpeg_decompress in its three formats (YUV420, the
 * one gmerlin-avdecoder's plugin uses, YUV422 and 8-bit grey), the colour
 * converters, and RTjpeg_compress for YUV420 and YUV422.
 */
#ifndef RTJPEG_B200_H
#define RTJPEG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------ */
/* Level 1: drop-in for include/RTjpeg.h                                     */
/* ------------------------------------------------------------------------ */

/* Opaque, as in include/RTjpeg.h:96 (`typedef void RTjpeg_t;`). */
typedef void RTjpeg_t;

/* Picture formats, include/RTjpeg.h:111-113. */
#define RTJ_YUV420 0
#define RTJ_YUV422 1
#define RTJ_RGB8   2

/* The colour converters of include/RTjpeg.h:128-136, as numbered by rtjgpu_convert_device. */
#define RTJ_CONV_RGB32        0   /* RTjpeg_yuv420rgb32, lib/RTjpeg.c:3123: R G B x */
#define RTJ_CONV_BGR32        1   /* RTjpeg_yuv420bgr32, :3192: B G R x */
#define RTJ_CONV_RGB24        2   /* RTjpeg_yuv420rgb24, :3261 */
#define RTJ_CONV_BGR24        3   /* RTjpeg_yuv420bgr24, :3326 */
#define RTJ_CONV_RGB16        4   /* RTjpeg_yuv420rgb16, :3391: 5-6-5, low byte first */
#define RTJ_CONV_RGB8         5   /* RTjpeg_yuv420rgb8, :3477: the luma plane */
#define RTJ_CONV_YUV422_RGB24 6   /* RTjpeg_yuv422rgb24, :3077 */

/* Element types of rtjgpu_decode_device_chw_window's planar output. */
#define RTJ_CHW_U8   0            /* the converter's byte */
#define RTJ_CHW_F16  1            /* IEEE binary16 */
#define RTJ_CHW_BF16 2            /* bfloat16 */
#define RTJ_CHW_F32  3            /* IEEE binary32 */

/* Fixed packet header length, include/RTjpeg.h:139 (RTJPEG_HEADER_SIZE). */
#define RTJPEG_B200_HEADER_BYTES 12

/* include/RTjpeg.h:115, lib/RTjpeg.c:2495.  New instance: no size, quality 0,
 * format YUV420.  Binds to the CUDA device named by $RTJPEG_B200_DEVICE
 * (default 0).  Returns NULL when no CUDA device can be used -- there is no
 * CPU fallback. */
RTjpeg_t *RTjpeg_init(void);

/* include/RTjpeg.h:116, lib/RTjpeg.c:2504. */
void RTjpeg_close(RTjpeg_t *rtj);

/* include/RTjpeg.h:117, lib/RTjpeg.c:2408.  Clamps *quality to 1..255 in
 * place, derives both dequantisation tables, returns 0. */
int RTjpeg_set_quality(RTjpeg_t *rtj, int *quality);

/* include/RTjpeg.h:118, lib/RTjpeg.c:2421.  Stores the format, returns 0.
 * RTjpeg_decompress refuses (error RTJGPU_E_FORMAT) a value outside 0..2. */
int RTjpeg_set_format(RTjpeg_t *rtj, int *format);

/* include/RTjpeg.h:119, lib/RTjpeg.c:2427.  Returns -1 when a dimension is
 * outside 0..65535, else 0. */
int RTjpeg_set_size(RTjpeg_t *rtj, int *w, int *h);

/* include/RTjpeg.h:120, lib/RTjpeg.c:2455.  Encoder-side knob; accepted and
 * clamped (key 0..255, masks 0..16) for source compatibility, no effect on
 * decoding. */
int RTjpeg_set_intra(RTjpeg_t *rtj, int *key, int *lm, int *cm);

/* include/RTjpeg.h:137, lib/RTjpeg.c:2371.  Writes the 128 AAN-scaled table
 * entries currently in force (luma 0..63, chroma 64..127). */
void RTjpeg_get_tables(RTjpeg_t *rtj, uint32_t *tables);

/* include/RTjpeg.h:138, lib/RTjpeg.c:2380.  Loads 128 raw (not AAN-scaled)
 * table entries; they stay in force until a packet whose quality byte differs
 * from the instance's current quality arrives (lib/RTjpeg.c:3575). */
void RTjpeg_set_tables(RTjpeg_t *rtj, uint32_t *tables);

/* include/RTjpeg.h:126, lib/RTjpeg.c:3565.  One packet (12-byte header +
 * payload) into planes[0..2] = Y, U, V, tight pitch (width, width/2, width/2;
 * YUV422: U and V have the full height; grey: planes[0] only).
 * Blocks the stream marks as skipped are left untouched in the caller's
 * planes, exactly like the reference.  Like the reference it returns nothing
 * and trusts the header's framesize; errors are reported out of band through
 * RTjpeg_b200_last_error(). */
void RTjpeg_decompress(RTjpeg_t *rtj, uint8_t *sp, uint8_t **planes);

/* include/RTjpeg.h:123, lib/RTjpeg.c:3488.  One picture (planes[0..2] = Y, U, V, tight pitch, in the instance's
 * format: YUV420 or YUV422) into one packet at sp -- 12-byte header + block stream, byte for byte the reference's,
 * inter-frame block skipping (RTjpeg_set_intra) included.  Returns the packet's size in bytes; the caller sizes sp
 * (worst case 12 + 64 bytes per block), as with the reference.  The reference's 8-bit format is not offered: its
 * encoder reads outside the plane (lib/RTjpeg.c:2627); 0 is returned and RTJGPU_E_FORMAT left for
 * RTjpeg_b200_last_error. */
int RTjpeg_compress(RTjpeg_t *rtj, uint8_t *sp, uint8_t **planes);

/* include/RTjpeg.h:128-136, lib/RTjpeg.c:3077-3486.  Colour conversion of one decoded picture: planes[0..2] = Y, Cb, Cr
 * (tight pitch, the instance's width and height), rows[r] = start of output row r.  Bit-exact integer arithmetic of
 * the reference (16 fractional bits).  The 32-bit converters step over the fourth byte of a pixel like the reference
 * does (:3147). */
void RTjpeg_yuv420rgb32(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);   /* include/RTjpeg.h:128, lib/RTjpeg.c:3123 */
void RTjpeg_yuv420bgr32(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);   /* :129, lib/RTjpeg.c:3192 */
void RTjpeg_yuv420rgb24(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);   /* :130, lib/RTjpeg.c:3261 */
void RTjpeg_yuv420bgr24(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);   /* :131, lib/RTjpeg.c:3326 */
void RTjpeg_yuv420rgb16(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);   /* :132, lib/RTjpeg.c:3391 */
void RTjpeg_yuv420rgb8(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);    /* :133, lib/RTjpeg.c:3477 */
void RTjpeg_yuv422rgb24(RTjpeg_t *rtj, uint8_t **planes, uint8_t **rows);   /* :135, lib/RTjpeg.c:3077 */
#define RTjpeg_yuv422rgb8(x, y, z) RTjpeg_yuv420rgb8(x, y, z)               /* :136 */

/* Same as RTjpeg_decompress but with the packet length known to the caller
 * (gavl_packet_t.buf.len in lib/video_rtjpeg.c:81), so a truncated packet is
 * refused instead of read past.  Returns 0 or a negative RTJGPU_E_* code. */
int RTjpeg_b200_decompress_n(RTjpeg_t *rtj, const uint8_t *sp, size_t len, uint8_t **planes);

/* Sticky error of the instance (0 = none); cleared by the call. */
int RTjpeg_b200_last_error(RTjpeg_t *rtj);

/* ------------------------------------------------------------------------ */
/* Level 2: batch decode                                                     */
/* ------------------------------------------------------------------------ */

enum {
    RTJGPU_OK          =  0,
    RTJGPU_E_CUDA      = -1,   /* a CUDA call failed; see rtjgpu_last_cuda_error */
    RTJGPU_E_ARG       = -2,   /* bad argument */
    RTJGPU_E_HEADER    = -3,   /* packet shorter than its header / framesize */
    RTJGPU_E_SIZE      = -4,   /* width/height zero, not a multiple of 16, or changing inside a batch */
    RTJGPU_E_FORMAT    = -5,   /* not YUV420 */
    RTJGPU_E_OVERRUN   = -6,   /* a frame's block stream runs past its packet */
    RTJGPU_E_TOOBIG    = -7,   /* batch exceeds the limits below */
    RTJGPU_E_NOMEM     = -8
};

#define RTJGPU_MAX_FRAMES_PER_BATCH 65534      /* source-frame indices are 16 bit */
#define RTJGPU_MAX_PAYLOAD_BYTES    (1u << 25) /* per frame; block offsets are 25 bit */
#define RTJGPU_STREAM_SLACK_BYTES   128        /* readable bytes required after the last packet of a device stream */

/* Which table set a frame uses: 0 = all-zero tables of a never-configured
 * instance (lib/RTjpeg.c:2495-2502), 1..255 = quality, 256 = the custom set
 * loaded with rtjgpu_set_custom_tables. */
#define RTJGPU_TABLE_ZERO   0
#define RTJGPU_TABLE_CUSTOM 256

/* One frame of a batch, as the kernels see it (16 bytes, device-resident). */
typedef struct rtjgpu_frame_desc {
    uint64_t offset;   /* of the packet header inside the stream buffer; multiple of 4 */
    uint32_t length;   /* packet bytes available (header + payload) */
    uint16_t table;    /* RTJGPU_TABLE_* / quality */
    uint16_t flags;    /* reserved, 0 */
} rtjgpu_frame_desc;

typedef struct rtjgpu_ctx rtjgpu_ctx;

/* Decoder state that crosses batch boundaries (lib/RTjpeg.c:3565-3579 keeps
 * the same three values in RTjpeg_t). */
typedef struct rtjgpu_state {
    int width, height;   /* 0,0 = unset */
    int table;           /* RTJGPU_TABLE_* currently in force */
    int quality;         /* rtj->Q: 0 on a fresh instance */
} rtjgpu_state;

/* Per-stage device time of the last rtjgpu_decode_device call, milliseconds
 * (CUDA events on the launch stream; filled only when timing is enabled).  In the pipelined arrangement
 * (rtjgpu_set_pipeline) the stages overlap: scan_ms is then the time until the last slice is scanned,
 * resolve_ms 0 and idct_ms the remainder. */
typedef struct rtjgpu_timing {
    float scan_ms;      /* K1 block-offset scan */
    float resolve_ms;   /* K3 last-writer resolution (0 when the batch has no skipped block) */
    float idct_ms;      /* K2 unpack + dequantise + IDCT + store */
    float total_ms;
} rtjgpu_timing;

/* Per-batch counters produced on the device, valid after rtjgpu_sync(). */
typedef struct rtjgpu_batch_info {
    uint64_t skipped_blocks;    /* 0xFF markers in the batch */
    uint64_t payload_bytes;     /* bytes the scan consumed, summed over frames */
    uint32_t bad_frames;        /* frames whose block stream overran the packet */
    int32_t  first_bad_frame;   /* -1 when none */
} rtjgpu_batch_info;

int  rtjgpu_create(int device, rtjgpu_ctx **out);
void rtjgpu_destroy(rtjgpu_ctx *ctx);
int  rtjgpu_device_count(void);
const char *rtjgpu_strerror(int code);
/* cudaError_t of the last failing CUDA call on this context, as int. */
int  rtjgpu_last_cuda_error(const rtjgpu_ctx *ctx);

/* Which flavour of the block-offset scan (K1) runs.  AUTO (the default) picks by batch size: many frames -- one CTA per
 * frame, SYNC (lanes walk the stream from guessed states and repair what was guessed wrong; frames whose streams do not
 * synchronise are handed to CHUNK's kernel, or, where the tables have a raw prefix, to the macroblock-level kernel --
 * which also takes every raw-prefix frame of a batch in which none was expected); few, large frames (and the one-frame RTjpeg_decompress) -- SEGMENT: the 8 KB segments of a frame go to separate
 * CTAs, with a frame-level chain between a summary pass and an emit pass.  CHUNK = one CTA per frame walks the frame's
 * segments in turn, every byte position examined in parallel inside a segment (round 1's kernel; its cost does not depend
 * on the content).  LANE / WARP / WALK force a serial walk instead: one thread per frame or one warp per frame.  Every
 * flavour is an independent implementation of the grammar and gives the same entries; the parity suite runs under each. */
#define RTJGPU_SCAN_AUTO    0
#define RTJGPU_SCAN_LANE    1
#define RTJGPU_SCAN_WARP    2
#define RTJGPU_SCAN_CHUNK   3
#define RTJGPU_SCAN_SEGMENT 4
#define RTJGPU_SCAN_WALK    5     /* one thread per frame, payload staged through shared memory with cp.async (not for raw-prefix frames) */
#define RTJGPU_SCAN_SYNC    6     /* one CTA per frame, every lane walks from its chunk's synchronisation point; no frame is handed over */
int  rtjgpu_set_scan_mode(rtjgpu_ctx *ctx, int mode);

/* How a large device batch is worked through.  SERIAL (what AUTO stands for at present): every stage on cuda_stream, one
 * after the other; per-stage times (rtjgpu_timing) are separable.  SLICED: in slices of frames, the scan of slice s + 1 on
 * a second CUDA stream beside resolve + IDCT of slice s; the call still orders everything after the work already on
 * cuda_stream and cuda_stream after its own work.  (Measured on a B200, DESIGN.md section 4: both stages are bound by
 * instruction issue, side by side they take each other's slots -- +1 .. 3 % on intra batches, -13 % on skip-heavy ones;
 * kept for hardware where that differs.)  slice_frames: frames per slice, 0 = keep the current value (default 1184);
 * rounded up to a multiple of 32.  K3's look-back for last writers never leaves a slice in either arrangement. */
#define RTJGPU_PIPELINE_AUTO   0
#define RTJGPU_PIPELINE_SERIAL 1
#define RTJGPU_PIPELINE_SLICED 2
int  rtjgpu_set_pipeline(rtjgpu_ctx *ctx, int mode, int slice_frames);

/* Picture format of the batches this context decodes (RTJ_YUV420, the default, RTJ_YUV422 or RTJ_RGB8 =
 * 8-bit grey): what RTjpeg_set_format is to an RTjpeg_t (lib/RTjpeg.c:2421, dispatch :3580-3585).  Frames
 * come out as tight planes: YUV420 w*h*3/2 bytes (Y, U, V), YUV422 w*h*2 bytes (Y, then U and V of
 * (w/2) x h), grey w*h bytes.  Width and height must be multiples of 16 in every format here. */
/* How K2 (IDCT + store) walks a device batch.  frames = 1: one CTA per (frame, row of macroblocks), every frame for itself.
 * frames = n > 1: a CTA works through n consecutive frames of its row, the row's pixels staying in shared memory from frame to
 * frame -- what a frame skips (lib/RTjpeg.c:2704: the block keeps what the persistent picture of lib/video_rtjpeg.c:81 held) is
 * then not touched at all, instead of being decoded again from its last writer's stream for every frame it persists in.
 * frames = 0 (the default): 8 when the batch before this one held skip markers, else 1 -- only the device knows about this
 * batch's markers at launch time, and streams do not change their nature from batch to batch.  The frames are the same either
 * way, bit for bit. */
int  rtjgpu_set_frame_runs(rtjgpu_ctx *ctx, int frames);
int  rtjgpu_set_format(rtjgpu_ctx *ctx, int format);

/* The converters above over a batch that is resident on the device -- typically the frames
 * rtjgpu_decode_device has just written.  d_frames: F tight pictures src_frame_bytes apart (Y, then Cb and Cr:
 * quarter size for the yuv420 kinds, half size for RTJ_CONV_YUV422_RGB24, unused by RTJ_CONV_RGB8).  Picture row r
 * of frame f goes to d_out + f * frame_pitch + r * row_pitch; row_pitch must be a multiple of 16.  Unlike the
 * reference, which steps over the fourth byte of a 32-bit pixel (lib/RTjpeg.c:3147), this call writes `alpha`
 * there.  Runs on cuda_stream. */
int  rtjgpu_convert_device(rtjgpu_ctx *ctx, int kind, const uint8_t *d_frames, size_t src_frame_bytes,
                           int F, int w, int h, uint8_t *d_out, size_t row_pitch, size_t frame_pitch,
                           int alpha, void *cuda_stream);
/* Bytes per pixel a converter writes (4, 3, 2 or 1); 0 for an unknown kind. */
int  rtjgpu_convert_bpp(int kind);

/* ---- encoder: RTjpeg_compress (lib/RTjpeg.c:3488-3524) over a batch that is resident on the device ---------
 * YUV420 and YUV422 (rtjgpu_set_format); the reference's 8-bit encoder reads outside its plane (:2627) and is not
 * offered.  A context carries one encoder: its tables (rtjgpu_encoder_set_quality = RTjpeg_set_quality :2408), the
 * inter-frame parameters (rtjgpu_encoder_set_intra = RTjpeg_set_intra :2455; key_rate 0 = every block coded), the
 * key counter and the blocks last sent, which carry over from call to call exactly as in an RTjpeg_t.
 * rtjgpu_encoder_reset puts counter and blocks back to those of a fresh instance. */
int  rtjgpu_encoder_set_quality(rtjgpu_ctx *ctx, int quality);
int  rtjgpu_encoder_set_intra(rtjgpu_ctx *ctx, int key_rate, int lm, int cm);
int  rtjgpu_encoder_reset(rtjgpu_ctx *ctx);
/* d_frames: F tight pictures of the context's format.  The packets (12-byte RTjpeg_frameheader + block stream, byte
 * for byte what RTjpeg_compress writes) go to d_stream back to back, each starting on a multiple of 4 bytes, and
 * d_offsets[0..F] (device memory) receives where each starts and where the last ends -- the layout rtjgpu_plan and
 * rtjgpu_decode_device take.  When the packets do not fit `capacity` nothing is written; rtjgpu_get_encode_info tells.
 * Asynchronous on cuda_stream. */
int  rtjgpu_encode_device(rtjgpu_ctx *ctx, const uint8_t *d_frames, int F, int w, int h,
                          uint8_t *d_stream, size_t capacity, uint64_t *d_offsets, void *cuda_stream);
/* Waits for the last rtjgpu_encode_device or rtjgpu_encode_device_seq: bytes its packets take, and whether they did not
 * fit. */
int  rtjgpu_get_encode_info(rtjgpu_ctx *ctx, uint64_t *bytes, int *overflow);

/* MANY INDEPENDENT STREAMS ENCODED IN ONE CALL, each with an encoder state of its own.  A handle is what an RTjpeg_t
 * carries for RTjpeg_compress -- tables, inter-frame parameters, key counter, the blocks last sent -- bound to one context
 * (so to its device).  rtjgpu_seqenc_create: a fresh instance's encoder (quality 0 = zero tables, key_rate 0).  The
 * setters are those of the context's encoder: set_quality clamps to 1..255 (it need not wait for the device: a handle's
 * tables are staged per call); set_intra clamps key_rate 0..255 and the masks 0..16 and clears the stored blocks but not
 * the key counter; reset puts counter and blocks back to a fresh instance's.  rtjgpu_seqenc_key_count: the key counter
 * the next picture gets.  A handle is freed by rtjgpu_seqenc_destroy, which waits for the work on
 * the device that may still use its stored blocks; it may outlive its context but is of no use then. */
typedef struct rtjgpu_seqenc rtjgpu_seqenc;
int  rtjgpu_seqenc_create(rtjgpu_ctx *ctx, rtjgpu_seqenc **out);
void rtjgpu_seqenc_destroy(rtjgpu_seqenc *e);
int  rtjgpu_seqenc_set_quality(rtjgpu_seqenc *e, int quality);
int  rtjgpu_seqenc_set_intra(rtjgpu_seqenc *e, int key_rate, int lm, int cm);
int  rtjgpu_seqenc_reset(rtjgpu_seqenc *e);
int  rtjgpu_seqenc_key_count(const rtjgpu_seqenc *e);
/* F output frames = S sequences laid end to end: sequence s is output frames [seq_first[s], seq_first[s + 1]), its
 * pictures are read from frames[s] (consecutive tight pictures of the context's format, 8-byte aligned, device memory)
 * and encoded with encs[s]'s state.  One pointer may serve several sequences (a rate ladder: the same pictures under
 * handles of different qualities); a handle may serve only one.  The packets of all sequences go to d_stream back to back,
 * each on a multiple of 4 bytes, and d_offsets[0..F] is laid out as by rtjgpu_encode_device: sequence s can be planned
 * with rtjgpu_plan over offsets[seq_first[s] .. seq_first[s + 1]] and its own rtjgpu_state, and decoded with
 * rtjgpu_decode_device_seq.  Sequence s's packets are byte for byte what RTjpeg_compress gives on that sequence alone
 * with the handle's history: key counter, stored blocks, quality and intra settings carried from earlier calls.  The
 * handles' counters advance at the call; their stored blocks are written by the device, so calls naming the same handle
 * must be ordered (one CUDA stream, as the workspace shared with rtjgpu_encode_device requires too).  When the packets do
 * not fit `capacity` nothing is written to d_stream, rtjgpu_get_encode_info tells, and every handle has advanced as if
 * they had been written: size d_stream with rtjgpu_encode_bound.  seq_first, frames and encs are host arrays (S + 1, S and
 * S entries), not read after the call returns.  Every argument is checked before anything is launched: RTJGPU_E_FORMAT for
 * the grey format; RTJGPU_E_ARG for seq_first as rtjgpu_decode_device_seq takes it (S >= 1, 0 .. F strictly increasing),
 * a NULL or misaligned picture pointer, a NULL handle, one of another context, or one named twice.  Asynchronous on
 * cuda_stream. */
int  rtjgpu_encode_device_seq(rtjgpu_ctx *ctx, int F, int w, int h, int S, const int *seq_first,
                              const uint8_t *const *frames, rtjgpu_seqenc *const *encs,
                              uint8_t *d_stream, size_t capacity, uint64_t *d_offsets, void *cuda_stream);
/* The most bytes F packets of format (RTJ_YUV420 or RTJ_YUV422) and size w x h can take, padding included: a capacity
 * that never overflows.  Host arithmetic; 0 for a format the encoder does not take or a bad size. */
size_t rtjgpu_encode_bound(int format, int w, int h, int F);

/* Raw (pre-AAN) tables for RTJGPU_TABLE_CUSTOM, the set_tables path. */
int  rtjgpu_set_custom_tables(rtjgpu_ctx *ctx, const uint32_t raw[128]);

/* Host-side planning: parse the headers of F packets laid out in one buffer
 * (packet f starts at offsets[f]; offsets[F] is the end of the buffer),
 * apply the lazy reconfiguration rules of RTjpeg_decompress
 * (lib/RTjpeg.c:3568-3579) starting from *state, and fill desc[F].  All frames
 * of a batch must share one size (split the batch where it changes).  *state
 * is advanced past the batch on success. */
int  rtjgpu_plan(const uint8_t *stream, const uint64_t *offsets, int F,
                 rtjgpu_state *state, rtjgpu_frame_desc *desc);
/* The same with the packets' TRUE lengths (lengths[f] bytes from offsets[f], at most the slot): what a caller that
 * knows them -- gavl_packet_t.buf.len in lib/video_rtjpeg.c:81 -- should use.  The header's framesize field is then
 * ignored altogether, as the reference ignores it (lib/RTjpeg.c:3565-3586).  rtjgpu_plan, which only sees slots that
 * may end in alignment padding, lets a framesize smaller than the slot bound the packet. */
int  rtjgpu_plan_n(const uint8_t *stream, const uint64_t *offsets, const uint32_t *lengths, int F,
                   rtjgpu_state *state, rtjgpu_frame_desc *desc);

/* Device-resident decode: stream, descriptors, output and carry all live in
 * device memory.  d_out receives F tight YUV420 frames (w*h*3/2 bytes each,
 * Y then U then V).  d_carry (w*h*3/2 bytes, may be NULL = zero-filled planes)
 * is the picture before the first frame: skipped blocks that no frame of the
 * batch has written yet are taken from it (lib/video_rtjpeg.c:81 decodes into
 * one persistent frame).  cuda_stream is a cudaStream_t passed as void*
 * (NULL = the legacy default stream).  Asynchronous: returns after the launches.
 * Alignment (RTJGPU_E_ARG otherwise): d_stream 4 bytes -- and every packet offset a multiple of 4, which rtjgpu_plan
 * checks --, d_desc 8, d_out 16 (frames are w*h*3/2 bytes, a multiple of 16, apart), d_carry 8.  Every
 * rtjgpu_decode_device* call, the _rgb ones included, and rtjgpu_scan_device (d_stream and d_desc) check the same. */
int  rtjgpu_decode_device(rtjgpu_ctx *ctx, const uint8_t *d_stream,
                          const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                          uint8_t *d_out, const uint8_t *d_carry, void *cuda_stream);

/* Device-resident decode STRAIGHT TO PACKED PIXELS: rtjgpu_decode_device with one of the reference's yuv420 converters
 * (RTJ_CONV_RGB32 / BGR32 / RGB24 / BGR24 / RGB16: RTjpeg_yuv420rgb32 ..., lib/RTjpeg.c:3123-3475) fused into the kernel
 * that makes the pixels -- a macroblock row (16 luma rows, 8 of Cb and Cr) is converted while it still sits in shared
 * memory, so the planes are never written to, nor read back from, device memory.  Bit for bit what RTjpeg_decompress
 * followed by the converter gives.  Picture row r of frame f goes to d_rgb + f * frame_pitch + r * row_pitch (both
 * multiples of 16, as d_rgb); the fourth byte of a 32-bit pixel receives `alpha`.  d_carry: the picture before the batch
 * as PLANES (w*h*3/2 bytes, or NULL = zeros), as for rtjgpu_decode_device; d_last_yuv (w*h*3/2 bytes, 16-byte aligned, or
 * NULL) receives the batch's last frame as planes -- the next batch's d_carry.  Contexts in RTJ_YUV420 format only.
 * Meant for streams of ordinary quality: blocks outside the sparse classes (more than seven coefficients) are decoded
 * by a slow path inside the kernel here, not by the separate general kernel. */
int  rtjgpu_decode_device_rgb(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F,
                              int w, int h, int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch, int alpha,
                              const uint8_t *d_carry, uint8_t *d_last_yuv, void *cuda_stream);

/* MANY INDEPENDENT STREAMS IN ONE CALL.  F frames = S independent sequences laid end to end in d_desc: sequence s is frames
 * [seq_first[s], seq_first[s + 1]).  A skipped block whose position no earlier frame OF THE SAME SEQUENCE coded is taken from
 * carries[s] (w*h*bytes-per-format picture, 8-byte aligned, device memory), or zeros where carries == NULL or carries[s] ==
 * NULL.  seq_first and carries are HOST arrays (S + 1 and S entries), read before the call returns.  Everything else as
 * rtjgpu_decode_device: d_out receives F frames, asynchronous on cuda_stream, every format.  Every sequence has the batch's
 * picture size and format; RTJGPU_TABLE_CUSTOM frames of any sequence use the context's one custom set.  Plan each sequence
 * with its own rtjgpu_state (rtjgpu_plan over its own offsets).  RTJGPU_E_ARG, before anything is launched, for S < 1 or
 * S > F, seq_first[0] != 0, seq_first[S] != F, seq_first not strictly increasing (no empty sequence), or a misaligned
 * carry.  S = 1 is rtjgpu_decode_device with carries[0]. */
int  rtjgpu_decode_device_seq(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                              int S, const int *seq_first, uint8_t *d_out, const uint8_t *const *carries, void *cuda_stream);
/* The same with rtjgpu_decode_device_rgb's fused converter; last_yuv (host array of S device pointers, or NULL; entries may
 * be NULL, 16-byte aligned) receives the LAST frame of each sequence as planes: that sequence's next carry.  YUV420 only. */
int  rtjgpu_decode_device_rgb_seq(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                  int S, const int *seq_first, int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch,
                                  int alpha, const uint8_t *const *carries, uint8_t *const *last_yuv, void *cuda_stream);

/* ONLY THE FRAMES A CALLER ASKS FOR.  The batch (F, S, seq_first, carries) is exactly that of rtjgpu_decode_device_seq; sel is
 * a HOST array of n batch frame indices, strictly increasing, each in [0, F), 0 <= n <= F, not read after the call returns.
 * Frame sel[k] goes to d_out + k * frame_bytes (tight planes of the context's format), byte for byte what
 * rtjgpu_decode_device_seq gives at row sel[k]; nothing else of d_out is written.  A frame needs only its own entries and
 * those of its skipped blocks' last writers, never the pixels of the frames before it: every frame is still scanned (K1)
 * and resolved (K3), only the selected ones are decoded and stored (K2).  Afterwards rtjgpu_get_batch_info and
 * rtjgpu_get_skip_counts describe all F frames.  To continue the streams in a later call, select each sequence's last frame:
 * its output is that sequence's next carry (selecting only the last frames is a seek).  Upload no trailing frames that no
 * selection needs: they are scanned all the same.  n = 0: the batch is scanned and resolved and nothing is written (d_out
 * may then be NULL).  n = F is rtjgpu_decode_device_seq; otherwise K2 decodes one frame per CTA whatever
 * rtjgpu_set_frame_runs says.  Every argument is checked before anything is launched: rtjgpu_decode_device_seq's rules
 * (alignment included), and RTJGPU_E_ARG for n < 0, n > F, sel == NULL with n > 0, or an index out of range, repeated or
 * out of order.  Asynchronous on cuda_stream. */
int  rtjgpu_decode_device_select(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                 int S, const int *seq_first, const uint8_t *const *carries,
                                 int n, const int *sel, uint8_t *d_out, void *cuda_stream);
/* The same with rtjgpu_decode_device_rgb_seq's fused converter: frame sel[k] goes to d_rgb + k * frame_pitch.  last_yuv has
 * its _rgb_seq meaning: each sequence's last frame leaves as planes (its next carry) whether or not it is selected; an
 * unselected last frame is decoded to planes only.  n = 0 (d_rgb may then be NULL) writes those planes and nothing else:
 * the streams advance by one batch and no picture is kept.  RTJGPU_E_FORMAT on a context that is not RTJ_YUV420. */
int  rtjgpu_decode_device_rgb_select(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                     int S, const int *seq_first, const uint8_t *const *carries,
                                     int n, const int *sel, int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch,
                                     int alpha, uint8_t *const *last_yuv, void *cuda_stream);

/* ONLY THE PART OF THE PICTURE A CALLER ASKS FOR.  The batch (F, S, seq_first, carries) and the selection (n, sel) are exactly
 * those of rtjgpu_decode_device_select.  origins is a HOST array of 2 S ints, (x, y) of sequence s's window, read before the
 * call returns; the window is cw x ch pixels for every sequence.  Selected frame sel[k] goes to d_out + k * window_bytes,
 * window_bytes = the tight planes of a cw x ch picture of the context's format (Y cw x ch, then U and V: (cw/2) x (ch/2) in
 * YUV420, (cw/2) x ch in YUV422; grey Y only), each plane byte for byte the crop of what rtjgpu_decode_device_select writes
 * for that frame.  A window is no carry: last_yuv (host array of S device pointers, or NULL; entries may be NULL, 16-byte
 * aligned) receives each sequence's last frame of the batch as FULL planes, selected or not -- that sequence's next carry.
 * n = 0 writes those planes only (d_out may then be NULL).  Nothing else is written; afterwards rtjgpu_get_batch_info and
 * rtjgpu_get_skip_counts describe all F frames, and K2 decodes one frame per CTA whatever rtjgpu_set_frame_runs says.  Only
 * the units that cover a window are decoded; a sequence's last frame that is selected is decoded twice (window and planes).
 * Every argument is checked before anything is launched: rtjgpu_decode_device_select's rules, and RTJGPU_E_ARG for cw or ch
 * <= 0, cw or any x not a multiple of 16, ch or any y odd, origins == NULL, a window that does not lie inside the picture, or
 * a misaligned last_yuv entry.  Asynchronous on cuda_stream. */
int  rtjgpu_decode_device_window(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                 int S, const int *seq_first, const uint8_t *const *carries,
                                 int n, const int *sel, int cw, int ch, const int *origins,
                                 uint8_t *d_out, uint8_t *const *last_yuv, void *cuda_stream);
/* The same with rtjgpu_decode_device_rgb_select's fused converter: window row r of frame sel[k] goes to d_rgb + k * frame_pitch
 * + r * row_pitch, cw * bytes-per-pixel bytes, byte for byte the crop of rtjgpu_decode_device_rgb_select's picture (alpha in
 * the fourth byte).  last_yuv as above.  RTJGPU_E_ARG also for a pitch that is not a multiple of 16, row_pitch < cw * bpp or
 * frame_pitch < ch * row_pitch; RTJGPU_E_FORMAT on a context that is not RTJ_YUV420. */
int  rtjgpu_decode_device_rgb_window(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                     int S, const int *seq_first, const uint8_t *const *carries,
                                     int n, const int *sel, int cw, int ch, const int *origins,
                                     int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch, int alpha,
                                     uint8_t *const *last_yuv, void *cuda_stream);
/* STRAIGHT TO A MODEL'S INPUT.  The batch, selection, window, origins, carries and last_yuv of rtjgpu_decode_device_rgb_window,
 * with its rules and error codes; what leaves is planar and typed.  Slot k is a tight [3][ch][cw] array of dtype (RTJ_CHW_U8,
 * F16, BF16 or F32: 1, 2, 2 or 4 bytes an element) at d_out + k * 3 * ch * cw * esize; d_out 16-byte aligned, NULL only when
 * n = 0.  kind is RTJ_CONV_RGB24 or RTJ_CONV_BGR24: channel c is byte c of that converter's pixel, v (0..255), bit for bit
 * what rtjgpu_decode_device_rgb_window writes.  RTJ_CHW_U8 stores v, and scale and bias must be NULL.  The float types store
 * t = fadd_rn(fmul_rn((float)v, scale[c]), bias[c]) -- two float32 roundings, no FMA -- as float32, or rounded to nearest even
 * to binary16 or bfloat16 (overflow to +-inf and subnormals as that rounding gives them).  scale and bias are HOST arrays of 3
 * floats indexed by output channel, read before the call returns; NULL means 1 and 0.  mirror is a HOST array of S ints, or
 * NULL: mirror[s] != 0 mirrors every window of sequence s left to right (output column j is window column cw - 1 - j; the
 * origin still says where the window lies).  RTJGPU_E_ARG also for a dtype or kind other than these, a scale or bias on
 * RTJ_CHW_U8, a scale or bias that is not finite, or a misaligned d_out; RTJGPU_E_FORMAT on a context that is not RTJ_YUV420.
 * Asynchronous on cuda_stream. */
int  rtjgpu_decode_device_chw_window(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                     int S, const int *seq_first, const uint8_t *const *carries,
                                     int n, const int *sel, int cw, int ch, const int *origins, const int *mirror,
                                     int kind, int dtype, const float *scale, const float *bias,
                                     void *d_out, uint8_t *const *last_yuv, void *cuda_stream);

/* Host-buffer decode: packets in host memory in, frames in host memory out.
 * The batch is cut into chunks that move through pinned staging buffers with
 * cudaMemcpyAsync on several streams so that copies overlap the kernels.
 * h_carry_inout (may be NULL) supplies the picture before the first frame and
 * receives the last decoded frame.  Synchronous.  flags: RTJGPU_HOST_* below. */
#define RTJGPU_HOST_IN_PINNED   1   /* h_stream is page-locked: DMA straight from it */
#define RTJGPU_HOST_OUT_PINNED  2   /* h_out is page-locked: DMA straight into it */
int  rtjgpu_decode_host(rtjgpu_ctx *ctx, const uint8_t *h_stream, const uint64_t *offsets, int F,
                        rtjgpu_state *state, uint8_t *h_out, uint8_t *h_carry_inout, int flags);
/* ... with the packets' true lengths (see rtjgpu_plan_n); lengths == NULL is rtjgpu_decode_host. */
int  rtjgpu_decode_host_n(rtjgpu_ctx *ctx, const uint8_t *h_stream, const uint64_t *offsets, const uint32_t *lengths, int F,
                          rtjgpu_state *state, uint8_t *h_out, uint8_t *h_carry_inout, int flags);

/* Per-frame skipped-block counts of the last successful rtjgpu_decode_host call (F entries, F at most that call's). */
int  rtjgpu_get_host_skip_counts(rtjgpu_ctx *ctx, uint32_t *counts, int F);

/* Wait for everything this context has launched. */
int  rtjgpu_sync(rtjgpu_ctx *ctx);

void rtjgpu_enable_timing(rtjgpu_ctx *ctx, int on);
int  rtjgpu_get_timing(rtjgpu_ctx *ctx, rtjgpu_timing *out);      /* last timed batch; waits for it */
/* Stage times of the timed device batch issued `calls_ago` calls before the last
 * one (0 = the last); the context keeps the most recent 256.  Reading after a
 * run of batches costs no synchronisation inside the run. */
int  rtjgpu_get_timing_at(rtjgpu_ctx *ctx, int calls_ago, rtjgpu_timing *out);
int  rtjgpu_get_batch_info(rtjgpu_ctx *ctx, rtjgpu_batch_info *out); /* syncs */

/* Per-frame skipped-block counts of the last device batch (F entries, host
 * array); a frame with count 0 is a "clean" frame, the only safe place to cut
 * an inter-coded stream into independent segments (SURVEY.md section 0-5). */
int  rtjgpu_get_skip_counts(rtjgpu_ctx *ctx, uint32_t *counts, int F);

/* Diagnostic: the first n block entries K1 made for the last device batch (frame-major, nblk per frame), 32 bits each --
 * 0xFFFFFFFF a skipped block; bit 31 set: a block of at most three coefficients carried in the entry itself (DC byte,
 * then the coefficients at zig-zag 1 and 2); else byte offset in the frame's payload (25 bits) and end-of-block
 * bound - 1 (6 bits above them).  After rtjgpu_scan_device these are K1's entries as made; after a decode, K3 has replaced
 * the marker of every skipped block whose last writer's entry is of the second kind (and was written under the same
 * tables) by a copy of that entry with bit 30 set -- the last writer in the same sequence (rtjgpu_decode_device_seq).  What RTjpeg_decompress uses to copy back only the blocks a frame coded, and what
 * the parity tests compare with the reference grammar's walk.  Synchronous. */
int  rtjgpu_get_entries(rtjgpu_ctx *ctx, uint32_t *entries, size_t n);

/* Number of kernels this library has launched on the context so far. */
uint64_t rtjgpu_launch_count(const rtjgpu_ctx *ctx);

/* K1 alone: the block-offset scan of a device-resident batch, without decoding it.  Afterwards rtjgpu_get_skip_counts
 * and rtjgpu_get_batch_info tell which frames are clean and whether every packet holds its picture -- what a host needs
 * to cut an inter-coded stream into shards before it decodes anything.  Same arguments as rtjgpu_decode_device. */
int  rtjgpu_scan_device(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                        void *cuda_stream);

/* Host-side multi-GPU split (pure host arithmetic, no CUDA).  Frames are coded against the picture before them
 * (lib/video_rtjpeg.c:81 decodes every packet into one persistent frame; a block marked 0xFF keeps what is there,
 * lib/RTjpeg.c:2704), so a stream can only be cut where the next frame rewrites everything: at a CLEAN frame
 * (clean[f] != 0: no skip marker in frame f, rtjgpu_get_skip_counts; the header's `key` byte is only a hint).
 *
 * rtjgpu_split_shards: n contiguous shards of roughly equal frame count, every cut on the clean frame nearest to the
 * ideal place (behind the previous cut).  first[n + 1] receives the shard starts (first[n] = F).  Returns the number
 * of shards that came out EMPTY because the clean frames ran out (0 = every shard has work), or a negative RTJGPU_E_*.
 *
 * rtjgpu_split_shards_lead: never an empty shard while F >= n.  A cut moves at most half a shard to reach a clean frame;
 * where there is none it stays at the ideal place and lead[i] tells how many frames BEFORE first[i] shard i has to
 * decode as well (back to the last clean frame, or to frame 0 and the caller's picture) and throw away: shard i
 * decodes frames [first[i] - lead[i], first[i + 1]) and keeps the last first[i + 1] - first[i] of them. */
int  rtjgpu_split_shards(const uint8_t *clean, int F, int n, int *first);
int  rtjgpu_split_shards_lead(const uint8_t *clean, int F, int n, int *first, int *lead);

/* Host-only table derivation, no CUDA involved (what the context uploads at
 * creation): the 128 AAN-scaled entries RTjpeg_get_tables would return after
 * RTjpeg_set_quality(Q) (lib/RTjpeg.c:2344-2369, :1208-1217), respectively after
 * RTjpeg_set_tables(raw) (:2380-2395), plus the raw-prefix lengths lb8 / cb8. */
void rtjgpu_tables_for_quality(int Q, uint32_t scaled[128], int *lb8, int *cb8);
void rtjgpu_tables_from_raw(const uint32_t raw[128], uint32_t scaled[128], int *lb8, int *cb8);

/* The 128 raw (not AAN-scaled) entries RTjpeg_set_tables takes for quality Q -- what a
 * NuppelVideo writer puts into the file's 'D'/'R' packet. */
void rtjgpu_raw_tables_for_quality(int Q, uint32_t raw[128]);

/* ------------------------------------------------------------------------ */
/* NuppelVideo / MythTV container in front of the decoder (host only)         */
/* ------------------------------------------------------------------------ */
/* lib/demux_nuv.c tags its video 'NUV ' and hands it to libavcodec; these helpers instead
 * rewrap the RTjpeg-coded frames of a .nuv file as 'RTJ0' packets for the decoder above. */
typedef struct rtjnuv_header {
    int      width, height;          /* lib/demux_nuv.c:78-80 */
    int      interlaced;             /* :84-89 */
    int      is_mythtv;              /* :69-72 */
    double   aspect, fps;            /* :93-94 */
    uint32_t video_packets, audio_packets;   /* :95-96 */
    int      has_tables;             /* a 'D' packet of subtype 'R' was found (:157-176) */
    uint32_t tables[128];            /* its contents: raw tables for RTjpeg_set_tables */
    uint64_t data_start;             /* offset of the first frame after the codec data (:241) */
} rtjnuv_header;

typedef struct rtjnuv_packet {
    uint8_t  type;                   /* 'V' video, 'A' audio, 'D' extradata, 'S' seek point, 'X' MythTV ext, ... */
    uint8_t  comptype;               /* video: '0' raw, '1' RTjpeg, '2' RTjpeg + LZO, '3' raw + LZO, 'N' black, 'L' repeat */
    uint8_t  keyframe, filters;
    uint32_t timecode;               /* milliseconds */
    uint32_t size;                   /* payload bytes (0 for seek points) */
    uint64_t payload_offset;
} rtjnuv_packet;

int rtjnuv_probe(const uint8_t *data, size_t len);                                 /* lib/demux_nuv.c:44 */
int rtjnuv_open(const uint8_t *data, size_t len, rtjnuv_header *out);              /* lib/demux_nuv.c:58 */
int rtjnuv_next(const uint8_t *data, size_t len, uint64_t *pos, rtjnuv_packet *out);   /* lib/demux_nuv.c:246; 1 = a packet, 0 = end */
/* Every RTjpeg-coded ('1') or repeated ('L', written as a frame of skip markers) video frame as an
 * 'RTJ0' packet: out receives the packets 16-byte aligned, offsets[0..*nframes] their starts (pass
 * out = NULL to size the buffer: offsets[*nframes] is the total).  Headers carry quality 0: decode
 * with rtjgpu_set_custom_tables(hdr->tables) and a state {width, height, RTJGPU_TABLE_CUSTOM, 0}.
 * *unsupported counts video frames of other compression types, which are left out. */
int rtjnuv_extract_rtj0(const uint8_t *data, size_t len, const rtjnuv_header *hdr, uint8_t *out, size_t out_cap,
                        uint64_t *offsets, uint32_t *timecodes, int max_frames, int *nframes, int *unsupported);

/* Pinned host memory helpers for callers that stage packets themselves. */
void *rtjgpu_host_alloc(size_t bytes);
void  rtjgpu_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* RTJPEG_B200_H */
