/*
 * rtj_common.h -- internal definitions shared by the host code and the kernels.
 */
#ifndef RTJ_COMMON_H
#define RTJ_COMMON_H

#include <stdint.h>
#include "../../include/rtjpeg_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- K1 output: one 32-bit entry per 8x8 block ------------------------------
 *   general   bit 31 = 0, bits 25..30 = E - 1, bits 0..24 = byte offset of the block
 *             inside its frame's payload.  E (1..64) is an end-of-block bound: every
 *             zig-zag position >= E is zero.
 *   inline    bit 31 = 1, bits 24..30 = 0: a block with E <= 3 carried in the entry
 *             itself -- bits 0..7 the DC byte (unsigned), bits 8..15 and 16..23 the
 *             signed coefficients at zig-zag 1 and 2 (0 where a run token covers
 *             them).  K2 never touches the payload for such a block.
 *   skipped   0xFFFFFFFF: the stream's 0xFF marker (lib/RTjpeg.c:2704).
 */
#define RTJ_ENT_OFF_BITS 25
#define RTJ_ENT_OFF_MASK ((1u << RTJ_ENT_OFF_BITS) - 1u)
#define RTJ_ENT(off, eob) ((uint32_t)(off) | ((uint32_t)((eob) - 1) << RTJ_ENT_OFF_BITS))
#define RTJ_ENT_SKIP 0xFFFFFFFFu
#define RTJ_ENT_INLINE_BIT 0x80000000u
#define RTJ_ENT_INLINE(dc, c1, c2) \
    (RTJ_ENT_INLINE_BIT | ((uint32_t)(dc) & 0xFFu) | (((uint32_t)(c1) & 0xFFu) << 8) | (((uint32_t)(c2) & 0xFFu) << 16))
/* K3 replaces the skip marker of a block whose last writer's entry is inline -- and was written under the same tables --
 * by a COPY of that entry (bit 30 tells): such a block needs no look-up of its last writer in K2 any more. */
#define RTJ_ENT_COPY_BIT 0x40000000u
#define RTJ_ENT_IS_SKIP(e) ((e) == RTJ_ENT_SKIP)
#define RTJ_ENT_IS_INLINE(e) (((e) & RTJ_ENT_INLINE_BIT) != 0u && (e) != RTJ_ENT_SKIP)
#define RTJ_ENT_EOB(e) ((int)(((e) >> RTJ_ENT_OFF_BITS) & 63u) + 1)

/* ---- picture formats (include/RTjpeg.h:111-113; RTjpeg_decompress dispatches on them, lib/RTjpeg.c:3580-3585) --
 * A picture is walked in UNITS: YUV420 a 16x16 macroblock of 4 luma + 2 chroma blocks (lib/RTjpeg.c:2701-2745),
 * YUV422 a 16x8 unit of 2 luma + 2 chroma blocks (:2654-2681, chroma half width, full height), 8-bit grey
 * a single 8x8 luma block (:2761-2770). */
#define RTJ_FMT_UNIT_BLOCKS(fmt) ((fmt) == 0 ? 6 : (fmt) == 1 ? 4 : 1)
#define RTJ_FMT_UNIT_LUMA(fmt)   ((fmt) == 0 ? 4 : (fmt) == 1 ? 2 : 1)
#define RTJ_FMT_UNITS_X(fmt, w)  ((fmt) == 2 ? (w) >> 3 : (w) >> 4)
#define RTJ_FMT_UNITS_Y(fmt, h)  ((fmt) == 0 ? (h) >> 4 : (h) >> 3)
#define RTJ_FMT_NBLK(fmt, w, h)  (RTJ_FMT_UNITS_X(fmt, w) * RTJ_FMT_UNITS_Y(fmt, h) * RTJ_FMT_UNIT_BLOCKS(fmt))
#define RTJ_FMT_FRAME_BYTES(fmt, w, h) \
    ((fmt) == 0 ? (size_t)(w) * (h) * 3 / 2 : (fmt) == 1 ? (size_t)(w) * (h) * 2 : (size_t)(w) * (h))

/* K3 output for skipped blocks: index of the last frame of the batch that
 * coded the block, or RTJ_SRC_CARRY when none has yet. */
#define RTJ_SRC_CARRY 0xFFFFu

/* Per-frame word of a batch of several sequences: the frame where f's sequence starts and that sequence's index
 * (both below 2^16: F <= RTJGPU_MAX_FRAMES_PER_BATCH).  A last writer before RTJ_SEQ_FIRST(...) belongs to another
 * sequence and does not count. */
#define RTJ_SEQ(first, index) ((uint32_t)(first) | (uint32_t)(index) << 16)
#define RTJ_SEQ_FIRST(v) ((v) & 0xFFFFu)
#define RTJ_SEQ_INDEX(v) ((v) >> 16)

/* One job of K2 in a call that decodes a selection of the batch's frames (rtjgpu_decode_device[_rgb]_select): the frame
 * and the output slot it goes to, both below 2^16 (n <= F <= RTJGPU_MAX_FRAMES_PER_BATCH).  RTJ_JOB_NO_SLOT (fused RGB
 * only): an unselected last frame of a sequence, decoded to planes for that sequence's last_yuv and nothing else. */
#define RTJ_JOB(frame, slot) ((uint32_t)(frame) | (uint32_t)(slot) << 16)
#define RTJ_JOB_FRAME(v) ((v) & 0xFFFFu)
#define RTJ_JOB_SLOT(v) ((v) >> 16)
#define RTJ_JOB_NO_SLOT 0xFFFFu

/* Per-sequence word of a call that decodes a window of its frames (rtjgpu_decode_device[_rgb]_window): the window's origin
 * in pixels, x a multiple of 16 and y even, both below 2^16 (they lie inside a picture of at most 65535 x 65535). */
#define RTJ_WIN(x, y) ((uint32_t)(x) | (uint32_t)(y) << 16)
#define RTJ_WIN_X(v) ((v) & 0xFFFFu)
#define RTJ_WIN_Y(v) ((v) >> 16)
/* rtjgpu_decode_device_chw_window: the sequence's windows leave mirrored left to right.  Bit 0 of x, free since x is a
 * multiple of 16: RTJ_WIN_X(v) / 16 is the window's first unit either way. */
#define RTJ_WIN_MIRROR 1u

#define RTJ_NUM_TABLES 257

/* Dequantisation tables as the kernels read them: zig-zag order (entry k is
 * the AAN-scaled multiplier of the k-th coefficient of the stream), luma then
 * chroma, plus the raw-prefix lengths lb8/cb8 (lib/RTjpeg.c:2362-2367). */
typedef struct rtj_dev_table {
    int32_t iq[2][64];
    int32_t bt8[2];
    int32_t pad[2];
} rtj_dev_table;

/* Host-side tables in the reference's own (raster) order. */
typedef struct rtj_host_table {
    int32_t liqt[64];
    int32_t ciqt[64];
    int     lb8, cb8;
} rtj_host_table;

extern const uint8_t rtj_zigzag[64];   /* position -> raster, lib/RTjpeg.c:59-74 */

void rtj_table_from_quality(int Q, rtj_host_table *out);           /* lib/RTjpeg.c:2344-2369 + 1208-1217 */
void rtj_table_from_raw(const uint32_t raw[128], rtj_host_table *out); /* lib/RTjpeg.c:2380-2395 */
void rtj_table_to_device_layout(const rtj_host_table *in, rtj_dev_table *out);
void rtj_encoder_table_from_quality(int Q, int32_t qt[128], int *lb8, int *cb8);   /* lib/RTjpeg.c:2344-2369 + 277-286 */

/* A batch is worked through in SLICES of frames (rtj_batch.cpp, run_kernels): K1 of slice s + 1 shares the SMs
 * with K3 / K2 of slice s.  Slices are whole chunks of RTJ_RESOLVE_T frames, at most RTJ_MAX_SLICES per batch. */
#define RTJ_RESOLVE_T  32
#define RTJ_K2_RUN_FRAMES 8      /* frames a CTA of K2 works through in turn on streams that skip blocks */
#define RTJ_MAX_SLICES 128

/* Device counters of one batch (lives in device memory, mirrored on request). */
typedef struct rtj_dev_info {
    unsigned long long skipped_blocks;
    unsigned long long payload_bytes;
    unsigned int       bad_frames;
    int                first_bad_frame;
    unsigned int       hard_blocks;      /* K2 -> K2b queue: mid-size blocks, filled from the front ... */
    unsigned int       hard_full;        /* ... and long blocks, filled from the back */
    unsigned int       raw_frames;       /* frames whose tables have a raw prefix (K1 counts them; AUTO's next choice of arrangement goes by it) */
    unsigned int       raw_walked;       /* ... of these, taken up by the self-synchronising walk (rtj_scan_sync_kernel<.., true>) */
    unsigned int       raw_given_up;     /* ... and left to rtj_scan_mb_kernel by it: streams that do not forget their past */
    unsigned int       slice_skips[RTJ_MAX_SLICES];   /* 0xFF markers per slice of frames (K1), what K3 decides on */
} rtj_dev_info;

/* ---- segment-parallel scan (few, large frames): a frame's 8 KB segments are parsed by separate
 * CTAs.  Where a segment is entered depends on everything before it, so the work is split in three:
 * every segment first reports, for EVERY possible entry offset, where a parse would leave it and how
 * many units (blocks or macroblocks) it would start; one thread per frame chains these summaries;
 * then every segment is parsed again from its now known entry and emits its entries. */
#define RTJ_SEG_BYTES    8192      /* segment of a frame without raw prefix (rtj_scan_chunk.cu) */
#define RTJ_SEG_BYTES_MB 4096      /* segment of a frame with raw prefix (rtj_scan_mb.cu) */
#define RTJ_SEG_NE    384          /* entry offsets a segment is summarised for (64 used without raw prefix) */
#define RTJ_SEG_UNUSED 0xFFFFFFFFu
#define RTJ_SEG_DEL_BYTES 9216     /* block lengths of one segment as level 0 leaves them (either kernel), for the second pass */
typedef struct rtj_seg_plan {
    uint32_t *sum;      /* [F][maxseg][RTJ_SEG_NE]  exit offset | units << 9 */
    uint32_t *entry;    /* [F][maxseg]  entry offset of the segment */
    uint32_t *base;     /* [F][maxseg]  first block index; RTJ_SEG_UNUSED = the frame is complete before it */
    int32_t  *nbf;      /* [F]  blocks the frame's stream holds, capped at nblk */
    uint8_t  *del;      /* [F][maxseg][RTJ_SEG_DEL_BYTES]  level 0 of the first pass, kept for the second; NULL: worked out again */
    int       maxseg;
    /* frames of many segments: the chain hops groups of RTJ_SEG_GROUP segments (gsum == NULL: it hops segments) */
    uint32_t *gsum;     /* [F][ngroups][RTJ_SEG_NE]  exit offset | units << 9 of a group */
    uint32_t *gentry;   /* [F][ngroups]  entry offset of the group's first segment */
    uint32_t *gbase;    /* [F][ngroups]  first block index; RTJ_SEG_UNUSED = behind the payload */
    int       ngroups;
} rtj_seg_plan;
#define RTJ_SEG_GROUP 16
#define RTJ_SEG_GROUP_MIN_SEGS 64      /* frames of fewer segments are chained segment by segment */

/* ---- kernel launchers (rtj_kernels.cu); stream is a cudaStream_t ----------- */
typedef struct rtj_launch_args {
    const uint8_t           *d_stream;
    const rtjgpu_frame_desc *d_desc;
    const rtj_dev_table     *d_tables;
    int                      F, w, h;
    int                      f0, f1;        /* the frames this launch covers (a slice); K1 segment-parallel and the serial flavours: 0, F */
    int                      slice;         /* index of the slice [f0, f1) */
    int                      row0, row1;    /* the rows of units K2 of this launch covers (all of them, as things are) */
    int                      k2_run;        /* frames a CTA of K2 works through in turn, the strip staying on chip (1: one frame per CTA) */
    unsigned long long      *h_skips_seen;  /* pinned host word K3 leaves the batch's skip count in (what the next batch's k2_run goes by), or NULL */
    void                    *d_walk;        /* [F] int2: rtj_scan_walk_kernel's state between slices of blocks */
    uint32_t                *d_redo;        /* [F] rtj_scan_sync_kernel: frames it leaves to rtj_scan_chunk_kernel / rtj_scan_mb_kernel (RTJ_REDO_*) */
    int                      raw_expected;  /* the batch before held frames with a raw prefix: launch the walk that takes them */
    int                      fmt;           /* RTJ_YUV420 / RTJ_YUV422 / RTJ_RGB8 */
    uint32_t                *d_ent;         /* [F][nblk] */
    uint16_t                *d_src;         /* [F][nblk] */
    uint32_t                *d_frame_skips; /* [F] */
    rtj_dev_info            *d_info;
    uint32_t                *d_hardq;       /* [F * nblk][2] K2 -> K2b queue: destination block, source block (frame * nblk + block) */
    uint16_t                *d_chunk_last;  /* [ceil(F / 32)][nblk] K3: last writer inside each chunk of frames */
    uint32_t                *d_chunk_mask;  /* [ceil(F / 32)][nblk] K3: which of the chunk's frames skipped the position */
    const uint16_t          *d_k3_in;       /* [nblk] K3: last writer before this slice (NULL: the first slice) */
    uint16_t                *d_k3_out;      /* [nblk] K3: last writer before the next slice */
    uint32_t                *d_k3_count;    /* [nblk / 128 + 1] K3: CTAs of rtj_resolve_last_kernel that are done with a group of positions */
    uint8_t                 *d_out;
    const uint8_t           *d_carry;
    const void              *d_lut;         /* K2: position table of this geometry (rtj_launch_build_lut) */
    /* K2 with the fused colour conversion (fused_rgb != 0): packed pixels instead of planes.  d_rgb may be NULL only when no
     * frame is converted (a selection of none whose sequences' last frames still leave as planes into last_yuv) */
    int                      fused_rgb;
    uint8_t                 *d_rgb;
    size_t                   rgb_row_pitch, rgb_frame_pitch;
    int                      rgb_kind;      /* RTJ_CONV_RGB32 / BGR32 / RGB24 / BGR24 / RGB16 */
    unsigned                 rgb_alpha;
    uint8_t                 *d_last_yuv;    /* the batch's last frame as planes too, or NULL */
    /* a batch of several independent sequences (rtjgpu_decode_device_seq); all NULL for one sequence, which takes
     * d_carry / d_last_yuv instead */
    const uint32_t          *d_seq;         /* [F] RTJ_SEQ(first frame of f's sequence, index of that sequence) */
    const uint8_t *const    *d_carries;     /* [S] picture before each sequence, entries NULL = zeros */
    uint8_t *const          *d_last_yuvs;   /* [S] RGB: where each sequence's last frame leaves as planes, entries may be NULL */
    int                      scan_mode;     /* RTJGPU_SCAN_* */
    rtj_seg_plan             seg;           /* workspace of the segment-parallel scan (sum == NULL: not available) */
    /* a selection of frames (rtjgpu_decode_device[_rgb]_select; d_jobs NULL: every frame, at its own index): K2 runs one
     * frame per CTA over jobs [j0, j1) of the batch's njobs RTJ_JOB words, sorted by frame */
    const uint32_t          *d_jobs;
    int                      j0, j1, njobs;
    /* a window of the selected frames (rtjgpu_decode_device[_rgb]_window; win_w == 0: none): win_w x win_h pixels at each
     * sequence's RTJ_WIN origin in d_win, over the most rows of units any sequence's window spans (win_rows).  win_last: the
     * launch of the sequences' last frames, a whole-picture window that leaves as planes to d_last_yuvs */
    const uint32_t          *d_win;
    int                      win_w, win_h, win_rows, win_last;
    /* the window leaves planar and typed (rtjgpu_decode_device_chw_window; chw == 0: packed, as rgb_kind says): slot k a
     * tight [3][win_h][win_w] array of chw_dtype (RTJ_CHW_*) at d_rgb + k * rgb_frame_pitch, rows rgb_row_pitch bytes apart.
     * Channel c = byte c of rgb_kind's pixel (RGB24 / BGR24), stored as fadd_rn(fmul_rn(v, chw_scale[c]), chw_bias[c]) */
    int                      chw, chw_dtype;
    float                    chw_scale[3], chw_bias[3];
} rtj_launch_args;

int rtj_launch_scan(const rtj_launch_args *a, void *stream);          /* returns the number of launches (>0) or -cudaError */
/* phase: 0 = one CTA per frame does everything, 1 = segment summaries, 2 = segment emit */
int rtj_launch_scan_chunk(const rtj_launch_args *a, int phase, void *stream);    /* rtj_scan_chunk.cu */
int rtj_scan_chunk_init(void);
int rtj_launch_scan_chunk_redo(const rtj_launch_args *a, const uint32_t *redo, void *stream);   /* one CTA per frame, flagged frames only */
/* rtj_scan_sync.cu.  redo[f]: 0 = the frame is done; else the kernel it is left to */
#define RTJ_REDO_CHUNK 1u
#define RTJ_REDO_MB    2u
int rtj_launch_scan_sync(const rtj_launch_args *a, uint32_t *redo, int handover, void *stream);
int rtj_launch_scan_sync_raw(const rtj_launch_args *a, uint32_t *redo, int handover, void *stream);   /* the frames marked RTJ_REDO_MB */
int rtj_scan_sync_init(void);
int rtj_launch_scan_mb(const rtj_launch_args *a, int phase, const uint32_t *redo, void *stream);       /* rtj_scan_mb.cu; redo (phase 0): only the frames marked RTJ_REDO_MB */
int rtj_launch_scan_walk(const rtj_launch_args *a, int b0, int b1, void *stream);   /* rtj_scan_walk.cu: blocks [b0, b1) of every frame */
int rtj_scan_walk_init(void);

int rtj_scan_mb_init(void);
int rtj_launch_resolve(const rtj_launch_args *a, void *stream);
int rtj_launch_idct(const rtj_launch_args *a, void *stream);           /* K2 over the slice */
int rtj_launch_idct_hard(const rtj_launch_args *a, void *stream);      /* K2b over the batch's queue, after the last slice */
/* d_lut: rtj_lut_bytes() bytes -- where each block of a row of units goes, for K2 */
size_t rtj_lut_bytes(int fmt, int w, int h);
int rtj_launch_build_lut(int fmt, int w, int h, void *d_lut, void *stream);
int rtj_idct_init(void);      /* rtj_idct.cu */
/* rtj_convert.cu: returns a cudaError */
int rtj_launch_convert(int kind, const uint8_t *d_src, size_t src_frame_bytes, int F, int w, int h,
                       uint8_t *d_out, size_t row_pitch, size_t frame_pitch, unsigned alpha, void *stream);
int rtj_convert_bpp(int kind);

/* rtj_encode.cu.  What one encode call needs on the device; all pointers device memory. */
typedef struct rtj_encode_args {
    const uint8_t *d_frames;       /* F tight pictures */
    int            F, w, h, fmt;   /* fmt: RTJ_YUV420 or RTJ_YUV422 */
    const int32_t *d_qt;           /* [128] quantiser multipliers, raster order, luma then chroma */
    int            lb8, cb8, quality;
    int            key_rate, key_count0, lmask, cmask;
    int16_t       *d_old;          /* [nblk][64] the block last sent at every place: state between calls */
    uint8_t       *d_slots;        /* [F][nblk][64] workspace: every block's bytes */
    uint8_t       *d_lens;         /* [F][nblk] workspace */
    uint32_t      *d_boff;         /* [F][nblk] workspace: byte offset of every block inside its packet's payload */
    uint32_t      *d_fsize;        /* [F] workspace: packet sizes */
    uint8_t       *d_stream;       /* out: packets back to back, each starting on a multiple of 4 */
    size_t         capacity;
    uint64_t      *d_offsets;      /* out: [F + 1] */
    uint64_t      *d_total;        /* out: [2] bytes needed, 1 if they did not fit */
} rtj_encode_args;
int rtj_launch_encode(const rtj_encode_args *a, void *stream);      /* returns launches (> 0) or -cudaError */

/* rtjgpu_encode_device_seq: S sequences, each with its own encoder state, laid end to end in the output frames.  E1 takes
 * a table of runs instead of one key period: a run is frames [f0, f1) of one sequence that chain their stored blocks, cut
 * where that sequence's key counter is 0 (intra sequences: one picture a run). */
typedef struct rtj_enc_run {
    int32_t  f0, f1;               /* output frames */
    uint32_t seq;                  /* sequence index | RTJ_ENC_RUN_* */
} rtj_enc_run;
#define RTJ_ENC_RUN_CONT  0x80000000u   /* starts from the handle's stored blocks (else from zeros) */
#define RTJ_ENC_RUN_LAST  0x40000000u   /* the sequence's last run: leaves its blocks in the handle */
#define RTJ_ENC_RUN_INDEX 0x0000FFFFu
typedef struct rtj_enc_seq {
    const uint8_t *d_frames;       /* the sequence's first picture; its pictures are consecutive */
    int16_t       *d_old;          /* [nblk][64] the handle's stored blocks (inter sequences) */
    int32_t        first;          /* output frame of the first picture */
    int32_t        quality;        /* row of the all-quality multiplier table */
    int32_t        lb8, cb8, lmask, cmask;
} rtj_enc_seq;
/* Per output frame: the header's quality and key bytes (RTJ_ENC_FRAME(quality, key)). */
#define RTJ_ENC_FRAME(q, key) ((uint32_t)(q) | (uint32_t)(key) << 8)
/* a->d_qt: [256][128] the multipliers of every quality (row 0 zeros); a->d_frames, quality, lb8 ... unused.  Runs
 * [0, n_intra) are intra, [n_intra, n_intra + n_inter) inter. */
int rtj_launch_encode_seq(const rtj_encode_args *a, const rtj_enc_run *d_runs, int n_intra, int n_inter,
                          const rtj_enc_seq *d_seqs, const uint32_t *d_frame_words, void *stream);
int rtj_kernels_init(void);   /* one-time function attributes (dynamic shared memory opt-in) */

#ifdef __cplusplus
}
#endif
#endif
