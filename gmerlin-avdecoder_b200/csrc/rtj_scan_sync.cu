/*
 * rtj_scan_sync.cu -- K1, self-synchronising flavour: the block-offset scan of one frame by a CTA whose
 * lanes each WALK a piece of the run-length stream, byte by byte, as a small state machine.
 *
 * What it replaces: the `sp += RTjpeg_s2b(...)` / `sp++` pointer chase of RTjpeg_decompressYUV420
 * (lib/RTjpeg.c:2701-2745), block lengths by the rules of RTjpeg_s2b (:157-186).  A parse of the stream is in
 * one of 64 states before every byte: "the next byte starts a block" (a DC byte, or the skip marker 0xFF,
 * :2704), or "r of the block's 63 places behind the DC are still to be filled" (r = 1..63; a byte 64..127 is a run
 * token that fills byte - 63 places, any other byte a coefficient that fills one, :171-183).  Where a block starts
 * depends on every byte before it -- but only through that one state.
 *
 * rtj_scan_chunk.cu makes the scan parallel by working out, for EVERY byte position, the length of the block
 * that would start there (~64 thread instructions per payload byte).  This kernel relies on a property of the
 * grammar instead: run-length streams FORGET.  Start a walk anywhere, in any state, and within a handful of blocks
 * it starts a block at a byte where the true parse starts one too -- from there on the two are the same walk
 * (measured on the bench stream: 6 bytes in the median, 49 at the 90th percentile).  One CTA per frame, 128 lanes
 * (256 in small batches, where a frame's latency is the batch's):
 *
 *   lead-in   the payload is cut into one chunk per lane.  Every lane walks the 64 bytes in front of its chunk from
 *             a GUESSED state ("a block starts here") ...
 *   walk      ... and then its chunk, ~8 instructions a byte, leaving one bit per byte: "a block starts here".
 *             Lane 0 starts from the frame's first byte (or from the state the previous segment ended in).
 *   check     a chunk must have been entered in the state its left neighbour ended in.  Where not (one chunk in ten
 *             with so short a lead-in), a repair walk starts from that state and runs until it falls in step with
 *             the walk made before; the rest of the chunk's bit map and its exit state then stand.  A repair that
 *             reaches the chunk's end changes the exit state, and the next chunk is checked again: after round k the
 *             first k chunks are final whatever the stream.  The guesses cost time when they are wrong, never
 *             exactness (tests/test_sync_model.py pins the argument on the CPU).
 *   emit      every lane lists the starts of its own chunk (a branch-free loop: one start per turn, the same
 *             instructions for every lane), and the 32-bit entries are made by all threads, four blocks each per
 *             turn, exactly as rtj_scan_chunk.cu makes them; stores coalesced.
 *
 * Streams that do not forget (every block 64 coefficient bytes long: noise at a high quality) would turn the check
 * into a serial walk, one chunk a round.  The CTA sees that after the first round -- too many repairs that never fell
 * in step -- and hands the frame over (redo[f] = 1) to rtj_scan_chunk_kernel, which is launched behind this kernel and
 * takes the flagged frames only; its cost does not depend on the content.
 *
 * The payload is read straight from the packet, 16 bytes a lane and read (a lane's reads lie in a row: every 32-byte
 * sector comes from L2 once), two reads under way; shared memory only holds the bit map and the list of starts
 * (26 KB, 80 registers: six CTAs, 24 warps per SM).  Frames of more than 40 KB are worked through in segments, the state
 * carried from one to the next.  (Earlier versions -- the set of all 64 states tracked as a bit mask until one is
 * left; the payload in shared memory by one bulk copy -- are in the history and in DESIGN.md section 4.)
 *
 * Frames whose tables have a raw 8-bit prefix (lb8 / cb8 != 0: a quality above 170) are walked by the kernel's second
 * instantiation (RAW), launched behind the first: the state then also holds the block's place in its unit, see SyTab below.
 * Same entries (rtj_common.h), counters and malformed-stream policy as the other flavours.
 */
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#include "rtj_common.h"

namespace {

constexpr unsigned FULL = 0xFFFFFFFFu;
/* Lanes a frame (the CTA's threads): 128, or 256 in small batches, where a frame's latency is what counts; 64 is kept for
 * comparison (rtj_launch_scan_sync picks). */
constexpr int SY_MAX_THREADS = 256;
constexpr int SY_LEAD = 4;                                 /* 16-byte pieces of the lead-in walk in front of a chunk (64 bytes) */
#ifndef SY_RAW_WARPS
#define SY_RAW_WARPS 28                                       /* resident warps per SM the raw-prefix instantiation is compiled for */
#endif
constexpr int SY_LEAD_RAW = 12;                            /* ... for frames with a raw prefix (192 bytes) */
constexpr int SY_SEG_MAX = 40960;                          /* bytes of a frame worked on at a time */
__host__ __device__ constexpr int sy_pmax(int threads) { return (SY_SEG_MAX / (16 * threads)) & ~1; }             /* pieces per chunk at most (even): a chunk's bit map is whole 32-bit words */
__host__ __device__ constexpr int sy_pmin(int threads) { return sy_pmax(threads) < 18 ? sy_pmax(threads) : 18; }   /* ... at least (even): short frames use fewer lanes, not shorter chunks */
constexpr int SY_LA = 80;                                  /* bytes walked behind a segment that is not the frame's last: the block that
                                                            * starts on its last byte (<= 64 bytes) and the start behind it, whole pieces */
constexpr int SY_WORDS = (SY_SEG_MAX + SY_LA + 31) / 32 + 1;   /* bit map words */
constexpr int SY_STAGE = 10240;                            /* block starts staged per emit round */
constexpr int SY_MAX_LOST = 8;                             /* more chunks than this whose repair walk never fell in step: not this kernel's stream */

static_assert(sy_pmin(SY_MAX_THREADS) >= SY_LEAD + 2, "a lead-in lies inside the chunk in front");
static_assert((sy_pmax(64) & 1) == 0 && (sy_pmax(128) & 1) == 0 && (sy_pmax(256) & 1) == 0 && (sy_pmin(64) & 1) == 0 && (sy_pmin(256) & 1) == 0,
              "a chunk's bit map is whole 32-bit words");
static_assert(SY_SEG_MAX + SY_LA + 16 < 65536, "positions inside a segment are 16 bit");

struct SyShared {
    uint32_t bits[SY_WORDS];             /* bit p: a block starts at byte p of the segment */
    uint16_t starts[SY_STAGE + 2];       /* one emit round's block starts */
    int16_t  exitst[SY_MAX_THREADS];     /* the state every lane's walk left its chunk in (raw-prefix frames: and the block's place in its unit) */
    int      wsum[SY_MAX_THREADS / 32];
    int      carry;                      /* state at the first byte of the next segment */
    int      nb;                         /* blocks started so far in this frame */
    int      skips;
    int      consumed;
    int      sentinel;                   /* first block start behind the segment's blocks */
};

/* One state over four bytes.  r > 0: places of the block still to fill; r <= 0: the next byte starts a block (a DC byte: 63
 * places behind it; the skip marker 0xFF: a block of its own).  A run token 01xxxxxx fills x + 1 places, any other byte one.
 * bm gets a bit for every byte that starts a block.
 *
 * The kernel is bound by the ALU pipe (LOP3 / SHF / PRMT / ISETP / SEL: one warp instruction every two clocks), while the
 * FMA pipe idles.  dp4a with a one-hot second operand picks a byte out of a word AND adds it to the state in one
 * instruction of the FMA pipe (measured, tools/pipe_rates2.cu: 0.5 / clock, pairs 1:1 with LOP3): the per-byte step is
 * two of them, one compare and one select. */
/* Frames whose tables have a RAW PREFIX (lib/RTjpeg.c:2362-2367, read by RTjpeg_s2b :165-169: the first bt8 bytes behind the
 * DC are coefficients whatever their value; bt8 differs between luma and chroma) need two more things in the state: which
 * block of its unit (macroblock: 4 luma + 2 chroma) the walk is in, and whether it is still inside the prefix.  The place in
 * the unit is kept as a PRMT selector, 0x7770 | place: one PRMT looks up the threshold above which r means "inside the
 * prefix" (63 - bt8 of the block's plane), another the selector of the next place.  Bytes 0 .. 5 of the two tables are the
 * places, byte 7 is what the selector's upper nibbles pick: 0 in the thresholds, 0x77 in the successors. */
struct SyTab {
    uint32_t thlo, thhi, nlo, nhi;
};
constexpr uint32_t SY_SEL = 0x77777770u;
__device__ __forceinline__ SyTab sy_make_tab(int unit, int unit_luma, int lb8, int cb8)
{
    unsigned long long th = 0, nx = 0x7700000000000000ull;
    for (int p = 0; p < unit; p++) {
        th |= (unsigned long long)(63 - min(p < unit_luma ? lb8 : cb8, 63)) << (8 * p);
        nx |= (unsigned long long)(0x70 | (p + 1 == unit ? 0 : p + 1)) << (8 * p);
    }
    SyTab t;
    t.thlo = (uint32_t)th; t.thhi = (uint32_t)(th >> 32); t.nlo = (uint32_t)nx; t.nhi = (uint32_t)(nx >> 32);
    return t;
}
/* a walk's state as one word: r in the low byte (signed), the place in the unit above it */
__device__ __forceinline__ int sy_pack(int r, uint32_t c) { return (r & 0xFF) | (int)((c & 7u) << 8); }
__device__ __forceinline__ int sy_r(int st) { return (int)(int8_t)st; }
__device__ __forceinline__ uint32_t sy_c(int st) { return SY_SEL | (uint32_t)(st >> 8); }

template <bool BITS, int bit0, bool RAW>
__device__ __forceinline__ void walk4(uint32_t W, int &r, uint32_t &c, const SyTab &tb, uint32_t &bm)
{
    const uint32_t runs = W & ~(W >> 1) & 0x40404040u;                   /* bit 6 of every run token */
    const uint32_t NX = ~(W & (runs - (runs >> 6)));                     /* per byte, as a signed byte: -(what it fills) */
    const uint32_t y = ~W;
    const uint32_t z = ~((y & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) & W & 0x80808080u;   /* bit 7 of every byte that is 0xFF */
    const uint32_t G = 0x3F3F3F3Fu & ~(z - (z >> 7));                    /* the state behind a block's first byte: 63, or 0 behind a skip marker */
    /* One byte: the new state is r - (what the byte fills); r - 1 inside a raw prefix; G's byte where a block starts.  All three
     * are dp4a (FMA pipe); the later two are PREDICATED and overwrite the first, so that no select is spent on the choice: the
     * ALU pipe -- the kernel's bound -- sees one compare (two with a prefix), the table look-ups and the bit for the map. */
#ifdef SY_SELECT_STEP                                       /* (A/B builds: the step with selects, as it was) */
#define SY_STEP(k)                                                                                   \
    {                                                                                                \
        int t, g;                                                                                    \
        asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(NX), "r"(1u << (8 * k)), "r"(r));         \
        asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(g) : "r"(G), "r"(1u << (8 * k)), "r"(0));          \
        const bool at = r <= 0;                                                                      \
        if (RAW) {                                                                                   \
            const int thr = (int)__byte_perm(tb.thlo, tb.thhi, c);                                   \
            const uint32_t cn = __byte_perm(tb.nlo, tb.nhi, c);                                      \
            int t1;                                                                                  \
            asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(t1) : "r"(0xFFFFFFFFu), "r"(1u), "r"(r));      \
            t = r > thr ? t1 : t;                                                                    \
            c = at ? cn : c;                                                                         \
        }                                                                                            \
        r = at ? g : t;                                                                              \
        if (BITS) asm("{ .reg .pred p; setp.ne.u32 p, %1, 0; @p add.u32 %0, %0, %2; }" : "+r"(bm) : "r"((unsigned)at), "n"(1u << (bit0 + k))); \
    }
#else
#define SY_STEP(k)                                                                                   \
    if (!RAW) {                                                                                      \
        if (BITS)                                                                                    \
            asm("{ .reg .pred pa; .reg .s32 rn;\n\t"                                                 \
                "setp.le.s32 pa, %0, 0;\n\t"                                                         \
                "dp4a.s32.u32 rn, %2, %4, %0;\n\t"                                                   \
                "@pa dp4a.u32.u32 rn, %3, %4, %5;\n\t"                                               \
                "@pa add.u32 %1, %1, %6;\n\t"                                                        \
                "mov.s32 %0, rn; }"                                                                  \
                : "+r"(r), "+r"(bm) : "r"(NX), "r"(G), "r"(1u << (8 * k)), "r"(0), "n"(1u << (bit0 + k)));   \
        else                                                                                         \
            asm("{ .reg .pred pa; .reg .s32 rn;\n\t"                                                 \
                "setp.le.s32 pa, %0, 0;\n\t"                                                         \
                "dp4a.s32.u32 rn, %1, %3, %0;\n\t"                                                   \
                "@pa dp4a.u32.u32 rn, %2, %3, %4;\n\t"                                               \
                "mov.s32 %0, rn; }"                                                                  \
                : "+r"(r) : "r"(NX), "r"(G), "r"(1u << (8 * k)), "r"(0));                            \
    } else {                                                                                         \
        /* inside the prefix (r above the plane's threshold) every byte is a coefficient: one place; the block that starts \
         * here is the unit's next */                                                                \
        if (BITS)                                                                                    \
            asm("{ .reg .pred pa, pr; .reg .s32 rn; .reg .b32 th;\n\t"                               \
                "setp.le.s32 pa, %0, 0;\n\t"                                                         \
                "prmt.b32 th, %7, %8, %1;\n\t"                                                       \
                "setp.gt.s32 pr, %0, th;\n\t"                                                        \
                "dp4a.s32.u32 rn, %3, %5, %0;\n\t"                                                   \
                "@pr dp4a.s32.u32 rn, %11, %12, %0;\n\t"                                             \
                "@pa dp4a.u32.u32 rn, %4, %5, %6;\n\t"                                               \
                "@pa prmt.b32 %1, %9, %10, %1;\n\t"                                                  \
                "@pa add.u32 %2, %2, %13;\n\t"                                                       \
                "mov.s32 %0, rn; }"                                                                  \
                : "+r"(r), "+r"(c), "+r"(bm)                                                         \
                : "r"(NX), "r"(G), "r"(1u << (8 * k)), "r"(0), "r"(tb.thlo), "r"(tb.thhi), "r"(tb.nlo), "r"(tb.nhi), \
                  "r"(0xFFFFFFFFu), "r"(1u), "n"(1u << (bit0 + k)));                                 \
        else                                                                                         \
            asm("{ .reg .pred pa, pr; .reg .s32 rn; .reg .b32 th;\n\t"                               \
                "setp.le.s32 pa, %0, 0;\n\t"                                                         \
                "prmt.b32 th, %6, %7, %1;\n\t"                                                       \
                "setp.gt.s32 pr, %0, th;\n\t"                                                        \
                "dp4a.s32.u32 rn, %2, %4, %0;\n\t"                                                   \
                "@pr dp4a.s32.u32 rn, %10, %11, %0;\n\t"                                             \
                "@pa dp4a.u32.u32 rn, %3, %4, %5;\n\t"                                               \
                "@pa prmt.b32 %1, %8, %9, %1;\n\t"                                                   \
                "mov.s32 %0, rn; }"                                                                  \
                : "+r"(r), "+r"(c)                                                                   \
                : "r"(NX), "r"(G), "r"(1u << (8 * k)), "r"(0), "r"(tb.thlo), "r"(tb.thhi), "r"(tb.nlo), "r"(tb.nhi), \
                  "r"(0xFFFFFFFFu), "r"(1u));                                                        \
    }
#endif
    SY_STEP(0) SY_STEP(1) SY_STEP(2) SY_STEP(3)
#undef SY_STEP
}

/* What the walks read: the segment's 16-byte pieces straight from the packet (a lane's pieces lie in a row, so each 128-byte
 * line is fetched once and then lives in L1 for the lane's next seven reads).  Bytes behind the payload read 0x7F, a run token
 * that ends any block; the bytes in front of it (the payload starts 0..12 bytes into its first piece) read 0xFF, "skip
 * markers" whose starts do not count.  The packet's own memory is never read past its last 16-byte line. */
struct SySeg {
    const uint4 *src;        /* piece 0 */
    int lim;                 /* the payload ends at byte lim of the segment */
    int first;               /* ... and starts at byte first (0 but for the frame's first segment) */
};
__device__ __forceinline__ uint32_t sy_fix_word(uint32_t w, int at, int lim, int first)      /* at: byte position of the word */
{
    if (at + 4 > lim) {
        const int nv = lim - at;
        const uint32_t m = nv <= 0 ? 0u : (1u << (8 * nv)) - 1u;
        w = (w & m) | (0x7F7F7F7Fu & ~m);
    }
    if (at < first) {
        const int nf = first - at;
        const uint32_t m = nf >= 4 ? 0xFFFFFFFFu : (1u << (8 * nf)) - 1u;
        w |= m;
    }
    return w;
}
__device__ __forceinline__ uint4 sy_piece(const SySeg &sg, int i)
{
    const int at = i * 16;
    uint4 w = make_uint4(0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x7F7F7F7Fu);
    if (at < sg.lim) {
        w = __ldg(sg.src + i);
        if (at + 16 > sg.lim || at < sg.first) {
            w.x = sy_fix_word(w.x, at, sg.lim, sg.first);
            w.y = sy_fix_word(w.y, at + 4, sg.lim, sg.first);
            w.z = sy_fix_word(w.z, at + 8, sg.lim, sg.first);
            w.w = sy_fix_word(w.w, at + 12, sg.lim, sg.first);
        }
    }
    return w;
}

/* pieces [p0, p1) from state r; BITS: leave the starts in the bit map.  Pieces that lie wholly inside the payload -- all but
 * the frame's first and last -- are read without a look at the payload's bounds, one piece ahead of their use. */
template <bool BITS, bool RAW>
__device__ __forceinline__ uint32_t walk16(const uint4 w, int &r, uint32_t &c, const SyTab &tb, uint16_t *bits16, int i)
{
    uint32_t bm = 0;
    walk4<BITS, 0, RAW>(w.x, r, c, tb, bm);
    walk4<BITS, 4, RAW>(w.y, r, c, tb, bm);
    walk4<BITS, 8, RAW>(w.z, r, c, tb, bm);
    walk4<BITS, 12, RAW>(w.w, r, c, tb, bm);
    if (BITS) bits16[i] = (uint16_t)bm;
    return bm;
}
/* st: the state -- r itself, or sy_pack(r, place) for frames with a raw prefix */
template <bool BITS, bool RAW>
__device__ __noinline__ int walk_pieces(const SySeg sg, uint16_t *bits16, int p0, int p1, int st, const SyTab tb)
{
    constexpr int D = 2;                                               /* pieces on their way at any time (measured at 128 lanes a frame: 1: 0.233 ms, 2: 0.231, 3: 0.237, 4: 0.247) */
    int r = RAW ? sy_r(st) : st;
    uint32_t c = RAW ? sy_c(st) : 0u;
    int i = p0;
    if (i < p1 && i == 0 && sg.first) { walk16<BITS, RAW>(sy_piece(sg, 0), r, c, tb, bits16, 0); i = 1; }
    const int pin = min(p1, sg.lim >> 4);
    if (i + D <= pin) {
        /* a new sector comes from L2, several hundred clocks, and the walk of one piece takes about as long */
        uint4 buf[D];
#pragma unroll
        for (int j = 0; j < D; j++) buf[j] = __ldg(sg.src + i + j);
        for (; i + D <= pin; i += D) {
#pragma unroll
            for (int j = 0; j < D; j++) {
                const uint4 cur = buf[j];
                buf[j] = __ldg(sg.src + min(i + D + j, pin - 1));
                walk16<BITS, RAW>(cur, r, c, tb, bits16, i + j);
            }
        }
    }
    for (; i < p1; i++) walk16<BITS, RAW>(sy_piece(sg, i), r, c, tb, bits16, i);     /* the last few, and what lies behind the payload */
    return RAW ? sy_pack(r, c) : r;
}

/* A repair walk: the chunk again, from the state it should have been entered in -- but only until it falls in step with the
 * walk made before: a byte at which both start a block.  From there on the two are the same walk (and wrongly entered walks
 * fall in step within a few blocks: that is what the lead-in relies on), so the rest of the chunk's bit map and its exit
 * state stand.  Returns false if that did not happen inside the chunk; st is then the chunk's new exit state.
 * With a raw prefix the two walks must also agree on WHICH block of its unit starts at that byte.  The bit map does not say;
 * the number of starts each walk has made since the chunk's first byte does: place = place at entry + starts so far.
 * was: the state the first walk entered the chunk in. */
template <bool RAW>
__device__ __noinline__ bool walk_repair(const SySeg sg, uint16_t *bits16, int p0, int p1, int &st, int was, int unit, const SyTab tb)
{
    int r = RAW ? sy_r(st) : st;
    uint32_t c = RAW ? sy_c(st) : 0u;
    /* places are taken BEHIND a start (the state's place is that of the block under way): the walks agree at a common
     * start if (place at entry + starts up to and including it) is the same for both, modulo the unit */
    int ahead = RAW ? (was >> 8) - (st >> 8) + unit : 0;               /* the first walk's place less this walk's, >= 0 */
    for (int i = p0; i < p1; i++) {
        const uint32_t before = bits16[i];
        const uint32_t now = walk16<true, RAW>(sy_piece(sg, i), r, c, tb, bits16, i);
        const uint32_t both = now & before;
        if (!RAW) {
            if (both) { st = r; return true; }
        } else {
            if (both) {
                /* at the piece's last common start: walks in step at an earlier one are in step there too */
                const uint32_t upto = (2u << (31 - __clz((int)both))) - 1u;
                if ((ahead + __popc(before & upto) - __popc(now & upto) + 16 * unit) % unit == 0) { st = sy_pack(r, c); return true; }
            }
            ahead += __popc(before) - __popc(now);
            ahead = (ahead % unit + unit) % unit;
        }
    }
    st = RAW ? sy_pack(r, c) : r;
    return false;
}

/* The 32-bit entry of a block (rtj_common.h): head = its first four bytes (DC, token 1, 2, 3), last = its last byte,
 * dl = its length, off = its offset in the payload.  The entry loop makes some 76 of them per lane and frame, so every
 * instruction here counts: the kernel is bound by the ALU pipe. */
__device__ __forceinline__ uint32_t sy_entry(uint32_t head, uint32_t last, int dl, int off, int bt8 = 0)
{
    /* positions >= eob are zero: a final run token (64..127) of n zeros ends at 64, so it starts at 64 - n = 127 - last;
     * any other last byte: 64 (bt8 = 63: no tokens at all).  Taken as unsigned, 127 - last is 0..63 for a run token, 64..127
     * for a byte below 64 and above 2^31 for one above 127, so one clamp does the choice (dl - 1 <= 63: a block is at most
     * 64 bytes) */
    uint32_t eob = min(max(127u - last, (uint32_t)(dl - 1)), 64u);
    if (bt8 >= 63) eob = 64u;
    /* inline (eob <= 3): the DC, and tokens 1 and 2 where they lie in front of eob and are not run tokens.  Byte-wise, bit 7
     * of x says "drop this byte": in bytes 1 and 2, ~head & (head << 1) marks a token 01xxxxxx, and 0x81 - eob / 0x82 - eob
     * (no borrow for eob <= 3) one at or behind eob; byte 0 reads 0x80.  PRMT spreads those bits over their bytes
     * (selector nibbles 9, A: sign of byte 1, 2; 8: byte 0's, dropping token 3; 4: zero, keeping the DC). */
    const uint32_t x = (~head & (head << 1)) | (0x00828180u - eob * 0x00010100u);
    uint32_t drop;
    asm("prmt.b32 %0, %1, 0, 0x8A94;" : "=r"(drop) : "r"(x));
    const uint32_t e_inl = RTJ_ENT_INLINE_BIT | (head & ~drop);
    const uint32_t e_gen = RTJ_ENT(off, eob);
    return (head & 0xFFu) == 0xFFu ? RTJ_ENT_SKIP : (bt8 == 0 && eob <= 3u ? e_inl : e_gen);      /* 0xFF: a skipped block */
}

} // namespace

/* redo[f]: 0 the frame is done, RTJ_REDO_CHUNK / RTJ_REDO_MB it is left to rtj_scan_chunk_kernel / rtj_scan_mb_kernel (rtj_common.h).
 * RAW = false takes the frames without a raw prefix and marks the others RTJ_REDO_MB; RAW = true, launched behind it where
 * such frames are expected, takes those.  handover = 0: never give a frame up (the parity suite's cross-check). */
template <int SY_THREADS, bool RAW>
__global__ void __launch_bounds__(SY_THREADS, (RAW ? SY_RAW_WARPS * 32 : 512) / SY_THREADS)
rtj_scan_sync_kernel(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                     const rtj_dev_table *__restrict__ tables, int F, int nblk,
                     uint32_t *__restrict__ ent, uint32_t *__restrict__ frame_skips,
                     rtj_dev_info *__restrict__ info, uint32_t *__restrict__ redo, int handover, int f0, int slice,
                     int unit, int unit_luma, int lead)
{
    extern __shared__ __align__(16) uint8_t sy_smem[];
    SyShared &sh = *reinterpret_cast<SyShared *>(sy_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    /* the kernels launched behind this one (the hand-over pass, the raw-prefix pass: both find nothing to do on most batches)
     * may take their places on the SMs while this grid's last CTAs are still at work */
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (RAW) asm volatile("griddepcontrol.wait;" ::: "memory");       /* the flags of the kernels in front are final */
    const int f = blockIdx.x + f0;
    if (f >= F) return;
    const rtjgpu_frame_desc d = desc[f];
    const rtj_dev_table &tab = tables[min((int)d.table, RTJ_NUM_TABLES - 1)];
    const int lb8 = tab.bt8[0], cb8 = tab.bt8[1];
    if (!RAW) {
        const bool raw = (lb8 | cb8) != 0;                             /* raw prefix: the other instantiation's frame, or rtj_scan_mb_kernel's */
        if (tid == 0) {
            redo[f] = raw ? RTJ_REDO_MB : 0u;
            if (raw) atomicAdd(&info->raw_frames, 1u);
        }
        if (raw) return;
    } else {
        if (redo[f] != RTJ_REDO_MB) return;
        if (tid == 0) atomicAdd(&info->raw_walked, 1u);
    }
    const SyTab tb = RAW ? sy_make_tab(unit, unit_luma, lb8, cb8) : SyTab{0u, 0u, 0u, 0u};
    const int MARG = RAW ? SY_LA : 8;                                  /* bytes behind the payload's end in which the start behind the last block lies */

    const uint8_t *pay = stream + d.offset + RTJPEG_B200_HEADER_BYTES;
    const int len = d.length > RTJPEG_B200_HEADER_BYTES ? (int)d.length - RTJPEG_B200_HEADER_BYTES : 0;
    const int mis = (int)(reinterpret_cast<uintptr_t>(pay) & 15);     /* 0, 4, 8 or 12: packets start 4-byte aligned */
    const uint8_t *gbase = pay - mis;                                   /* 16-byte aligned, never before the packet */
    uint32_t *out = ent + (size_t)f * nblk;
    uint16_t *bits16 = reinterpret_cast<uint16_t *>(sh.bits);

    /* positions: byte p of the frame is gbase[p]; the payload is [mis, end).  A frame that fits one segment leaves room for
     * the start behind its last block (end + 1 at most) inside the lanes' chunks. */
    const int end = len > 0 ? mis + len : 0;
    constexpr int SY_WARPS = SY_THREADS / 32, SY_PMAX = sy_pmax(SY_THREADS), SY_PMIN = sy_pmin(SY_THREADS);
    const int P = end + MARG > SY_SEG_MAX ? SY_PMAX : max(SY_PMIN, ((end + MARG + SY_THREADS * 32 - 1) / (SY_THREADS * 32)) * 2);
    const int SEG = SY_THREADS * P * 16;

    if (tid == 0) {
        sh.carry = 0;
        sh.nb = 0;
        sh.skips = 0;
        sh.consumed = 0;
    }
    __syncthreads();

    for (int seg0 = 0; seg0 < end; seg0 += SEG) {
        const int nb0 = sh.nb;
        if (nb0 >= nblk) break;                                        /* uniform: everybody reads the same word */
        SySeg sg;
        sg.src = reinterpret_cast<const uint4 *>(gbase + seg0);
        sg.lim = end - seg0;
        sg.first = seg0 == 0 ? mis : 0;
        const int lim = sg.lim, first = sg.first;
        const int climit = min(SEG, lim);                              /* starts before it are this segment's blocks */
        const bool more = lim + MARG > SEG;                            /* the frame goes on behind this segment */
        const int ptot = more ? (SEG + SY_LA) >> 4 : (lim + MARG + 15) >> 4;   /* pieces to walk: up to the start behind the last block */

        /* ---- lead-in: every lane walks the SY_LEAD pieces in front of its chunk from a guessed state ("a block starts
         *      here").  Run-length streams forget their past within a handful of blocks: at the chunk's first byte the
         *      walk is, more often than not, in the true state.  Whether it is, is checked below -- never assumed. ---- */
        const int p0 = tid * P, p1 = min(p0 + P, ptot);                /* this lane's chunk, in pieces */
        /* raw prefix: the guess is "the first block of a unit starts here" -- a walk that is wrong about the place falls out of
         * step with the stream at the next block of the other plane, and in again a few blocks on, with another place: it
         * takes some 80 bytes in the median (170 at the 99th percentile) until place and byte are both right, hence the longer
         * lead-in.  The frame's first byte is the one place known: behind the `first` bytes in front of the payload, which
         * read as skip markers and each count as a block, the unit's first block must start. */
        const int guess = RAW ? sy_pack(0, (uint32_t)(unit - 1)) : 0;
        int r_in = guess;                                              /* the state the chunk is entered in */
        if (tid == 0) r_in = seg0 != 0 ? sh.carry : RAW ? sy_pack(0, (uint32_t)(((unit - 1 - first) % unit + unit) % unit)) : 0;
        else if (p0 < ptot) r_in = walk_pieces<false, RAW>(sg, nullptr, p0 - (RAW ? lead : SY_LEAD), p0, guess, tb);

        /* ---- walk: the chunk, from that state; one bit per byte that starts a block ---- */
        int r_out = walk_pieces<true, RAW>(sg, bits16, p0, p1, r_in, tb);
        sh.exitst[tid] = (int16_t)r_out;
        __syncthreads();

        /* ---- check: a chunk must have been entered in the state its left neighbour ended in.  Where not (the lead-in is
         *      short: one lane in ten), a repair walk starts from that state and runs until it falls in step with the first
         *      walk, a few blocks on; the chunk's exit state stands then.  A repair that runs to the chunk's end without
         *      falling in step changes the exit state, and the next chunk is checked again: after round k the first k chunks
         *      are final whatever the stream, so the result never depends on the guesses -- they only cost time. ---- */
        for (int round = 0;; round++) {
            const int want = tid > 0 ? (int)sh.exitst[tid - 1] : r_in;
            /* states <= 0 all mean "a block starts here" */
            const bool dirty = tid > 0 && p0 < ptot &&
                               (RAW ? (max(sy_r(want), 0) != max(sy_r(r_in), 0) || (want >> 8) != (r_in >> 8)) : max(want, 0) != max(r_in, 0));
            if (__syncthreads_count(dirty) == 0) break;
            bool lost = false;
            if (dirty) {
                int r = want;
                if (!walk_repair<RAW>(sg, bits16, p0, p1, r, r_in, unit, tb)) {
                    lost = true;
                    r_out = r;
                    sh.exitst[tid] = (int16_t)r;
                }
                r_in = want;
            }
            const int nlost = __syncthreads_count(lost);
            if (handover && round == 0 && nlost > SY_MAX_LOST) {
                /* a stream that does not forget its past: leave the frame to the kernel whose cost does not depend on the content */
                if (tid == 0) {
                    redo[f] = RAW ? RTJ_REDO_MB : RTJ_REDO_CHUNK;
                    if (RAW) atomicAdd(&info->raw_given_up, 1u);
                }
                return;
            }
        }
        if (more && tid == SY_THREADS - 1) {
            /* the state the next segment starts in; the look-ahead behind this one */
            sh.carry = r_out;
            walk_pieces<true, RAW>(sg, bits16, SY_THREADS * P, ptot, r_out, tb);
        }
        __syncthreads();

        /* ---- the first start at or behind climit is where the segment's last block ends; the starts that do not count
         *      (in front of the payload, behind climit) leave the bit map ---- */
        if (tid == 0) {
            const int wend = (ptot * 16 + 31) >> 5;
            int s = climit;
            for (int w = climit >> 5; w < wend; w++) {
                uint32_t v = sh.bits[w];
                if (w == (climit >> 5)) v &= ~((1u << (climit & 31)) - 1u);
                if (w == wend - 1 && ((ptot * 16) & 31)) v &= 0xFFFFu;
                if (v) { s = w * 32 + __ffs((int)v) - 1; break; }
            }
            sh.sentinel = s;
            sh.bits[0] &= ~((1u << first) - 1u);                                     /* first <= 12 */
            for (int w = climit >> 5; w < wend; w++) sh.bits[w] = w == (climit >> 5) ? sh.bits[w] & ((1u << (climit & 31)) - 1u) : 0u;
        }
        __syncthreads();

        /* ---- count: every lane the starts of its own chunk; a scan over the lanes ---- */
        const int w0 = p0 >> 1, w1 = (min(p0 + P, ptot) + 1) >> 1;     /* the chunk's bit map words (P is even) */
        int cnt = 0;
        for (int w = w0; w < w1; w++) cnt += __popc(sh.bits[w]);
        int base, total;
        {
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += up;
            }
            if (lane == 31) sh.wsum[warp] = incl;
            __syncthreads();
            base = incl - cnt;
            total = 0;
#pragma unroll
            for (int k = 0; k < SY_WARPS; k++) {
                const int s = sh.wsum[k];
                if (k < warp) base += s;
                total += s;
            }
        }

        /* ---- emit: the list of starts (every lane its chunk's), then one block per thread ---- */
        const int nemit = min(total, nblk - nb0);
        int myskips = 0;
        const uint32_t *gw = reinterpret_cast<const uint32_t *>(gbase + seg0);
        const uint8_t *gb = gbase + seg0;
        const int offb = seg0 - mis;                                   /* a block's offset in the payload less its start */
#ifdef SY_AB_COUNT_ONLY
        /* (A/B builds only: the kernel stops after the count -- no list of starts, no entries but a harmless one per block,
         * stored as the entry loop stores them -- to time what the emit stage costs) */
        for (int b = tid; b < nemit; b += SY_THREADS) out[nb0 + b] = RTJ_ENT(0, 1);
        if (tid == 0) sh.consumed = len;
        for (int lo = 0; lo < 0; lo += SY_STAGE) {
#else
        for (int lo = 0; lo < nemit; lo += SY_STAGE) {
#endif
            const int n = min(SY_STAGE, nemit - lo);
            {
                /* One start per turn, the same instructions for every lane whatever its words hold (nothing to diverge on):
                 * a lane out of bits takes its next word in the same turn.  Turns: the busiest lane's starts + words. */
                const bool mine = base <= lo + n && base + cnt > lo;
                int turns = mine ? cnt + (w1 - w0) : 0;
#pragma unroll
                for (int o = 16; o; o >>= 1) turns = max(turns, __shfl_xor_sync(FULL, turns, o));
                /* (a lane whose starts all lie outside this round never stores: its indices are out of [0, n]) */
                int idx = base - lo, w = w0, pos0 = 0;
                uint32_t v = 0;
                const uint32_t starts_s = (uint32_t)__cvta_generic_to_shared(sh.starts);
                for (int t = 0; t < turns; t++) {
                    const uint32_t vn = sh.bits[min(w, SY_WORDS - 1)];
                    if (v == 0u) { v = w < w1 ? vn : 0u; pos0 = w * 32; w++; }
                    const int b = __ffs((int)v) - 1;
                    const bool ok = v != 0u && (unsigned)idx <= (unsigned)n;
                    asm volatile("{ .reg .pred p; setp.ne.u32 p, %0, 0; @p st.shared.u16 [%1], %2; }"
                                 :: "r"((unsigned)ok), "r"(starts_s + 2u * (unsigned)idx), "h"((uint16_t)(pos0 + b)) : "memory");
                    idx += v != 0u ? 1 : 0;
                    v &= v - 1u;
                }
            }
            if (tid == 0 && lo + n == total) sh.starts[n] = (uint16_t)sh.sentinel;
            __syncthreads();
            /* the payload read so far ends where the list's last block ends: starts[n] (the sentinel, or the start behind it) */
            if (tid == 0 && lo + n == nemit) sh.consumed = max(sh.consumed, offb + (int)sh.starts[n]);
            /* four blocks a thread and turn: the loads of all four are under way before any is used (the payload comes
             * from L2 by now: several hundred clocks) */
            uint32_t *op = out + nb0 + lo;
            constexpr int U = 4;
            /* whole: all four blocks lie in the list (every turn but a thread's last) -- no clamps, no tests */
            auto emit4 = [&](const int k, const bool whole) {
                int qq[U], nx[U];
                uint32_t h0[U], h1[U], lb[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int ku = whole || u == 0 ? k + u * SY_THREADS : min(k + u * SY_THREADS, n - 1);
                    qq[u] = sh.starts[ku];
                    nx[u] = sh.starts[ku + 1];
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const uint32_t *wp = gw + ((unsigned)qq[u] >> 2);
                    h0[u] = __ldg(wp);
                    h1[u] = __ldg(wp + 1);
                    lb[u] = __ldg(gb + (unsigned)nx[u] - 1);
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    /* raw prefix: the block's place in its unit tells its plane, and that the prefix's length */
                    const int bt8 = RAW ? ((nb0 + lo + k + u * SY_THREADS) % unit < unit_luma ? lb8 : cb8) : 0;
                    /* (the funnel shift takes its count modulo 32: qq * 8 is (qq & 3) * 8) */
                    const uint32_t head = __funnelshift_r(h0[u], h1[u], (unsigned)qq[u] * 8u);
                    const uint32_t e = sy_entry(head, lb[u], nx[u] - qq[u], qq[u] + offb, bt8);
                    if (whole || k + u * SY_THREADS < n) {
                        op[k + u * SY_THREADS] = e;
                        if ((head & 0xFFu) == 0xFFu) myskips++;                    /* e == RTJ_ENT_SKIP */
                    }
                }
            };
            int k = tid;
            for (; k + (U - 1) * SY_THREADS < n; k += U * SY_THREADS) emit4(k, true);
            if (k < n) emit4(k, false);
            /* the payload's last bytes: a block that starts on one of the last three, or that is cut short, must see 0x7F
             * behind the payload, not what follows the packet in memory -- at most the list's last four blocks */
            if (lo + n == total && lim < climit + SY_LA) {
                __syncthreads();
                const int k = n - 1 - tid;
                if (tid < 4 && k >= 0) {
                    const int qq = sh.starts[k], nx = sh.starts[k + 1];
                    if (qq + 4 > lim || nx > lim) {
                        const uint32_t *wp = gw + (qq >> 2);
                        uint32_t head = __funnelshift_r(__ldg(wp), __ldg(wp + 1), (unsigned)(qq & 3) * 8);
                        uint32_t last = __ldg(gb + min(nx, lim) - 1);
                        if (qq + 4 > lim) {
                            const uint32_t m = (1u << (8 * (lim - qq))) - 1u;           /* 1..3 bytes are the payload's */
                            head = (head & m) | (0x7F7F7F7Fu & ~m);
                        }
                        if (nx > lim) last = 0x7Fu;                                    /* the last block, cut short */
                        op[k] = sy_entry(head, last, nx - qq, qq + offb, RAW ? ((nb0 + lo + k) % unit < unit_luma ? lb8 : cb8) : 0);
                    }
                }
            }
            __syncthreads();
        }
        {
#pragma unroll
            for (int o = 16; o; o >>= 1) myskips += __shfl_xor_sync(FULL, myskips, o);
            if (lane == 0 && myskips) atomicAdd(&sh.skips, myskips);
            if (tid == 0) sh.nb = nb0 + total;
        }
        __syncthreads();
    }

    /* a frame whose stream ends early or mid-block: flag it, give the missing blocks a harmless entry */
    const int nbf = min(sh.nb, nblk);
    for (int b = nbf + tid; b < nblk; b += SY_THREADS) out[b] = RTJ_ENT(min(len, (int)RTJ_ENT_OFF_MASK), 1);
    if (tid == 0) {
        const int consumed = sh.consumed, skips = sh.skips;
        if (RAW) redo[f] = 0u;
        frame_skips[f] = (uint32_t)skips;
        if (skips) {
            atomicAdd(&info->skipped_blocks, (unsigned long long)skips);
            atomicAdd(&info->slice_skips[slice], (unsigned)skips);
        }
        atomicAdd(&info->payload_bytes, (unsigned long long)min(consumed, len));
        if (nbf < nblk || consumed > len || len > (int)RTJGPU_MAX_PAYLOAD_BYTES) {
            atomicAdd(&info->bad_frames, 1u);
            atomicMin((unsigned int *)&info->first_bad_frame, (unsigned int)f);
        }
    }
}

namespace {

template <int T, bool RAW>
cudaError_t sy_attr()
{
    return cudaFuncSetAttribute(rtj_scan_sync_kernel<T, RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SyShared));
}

template <int T, bool RAW>
cudaError_t sy_launch(const rtj_launch_args *a, uint32_t *redo, int handover, int lead, cudaStream_t st)
{
    const int nblk = RTJ_FMT_NBLK(a->fmt, a->w, a->h);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(a->f1 - a->f0));
    cfg.blockDim = dim3(T);
    cfg.dynamicSmemBytes = sizeof(SyShared);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = RAW ? 1 : 0;                         /* the raw-prefix pass sits behind the other and may take its place early */
    return cudaLaunchKernelEx(&cfg, rtj_scan_sync_kernel<T, RAW>, a->d_stream, a->d_desc, a->d_tables, a->f1, nblk, a->d_ent, a->d_frame_skips,
                              a->d_info, redo, handover, a->f0, a->slice, RTJ_FMT_UNIT_BLOCKS(a->fmt), RTJ_FMT_UNIT_LUMA(a->fmt), lead);
}

} // namespace

extern "C" int rtj_scan_sync_init(void)
{
    cudaError_t e = sy_attr<64, false>();
    if (e == cudaSuccess) e = sy_attr<128, false>();
    if (e == cudaSuccess) e = sy_attr<256, false>();
    if (e == cudaSuccess) e = sy_attr<64, true>();
    if (e == cudaSuccess) e = sy_attr<128, true>();
    return e == cudaSuccess ? 0 : (int)e;
}

/* redo: [F] flags; handover = 0: never give a frame up */
extern "C" int rtj_launch_scan_sync(const rtj_launch_args *a, uint32_t *redo, int handover, void *stream)
{
    const int nf = a->f1 - a->f0;
    /* Lanes a frame.  Few frames: 256 (a frame's latency is the batch's: 1920x1088, 120 frames: 0.20 ms with 64 lanes, 0.11 with
     * 128, 0.09 with 256).  Many: 128 -- 320-byte chunks at the bench point; 64 lanes with chunks twice as long spend less on
     * lead-ins but are 6 % slower there (0.255 against 0.239 ms per 4096 frames), 256 lose to their lead-ins (96: 0.254, 160: 0.276). */
    static const int forced = getenv("RTJPEG_B200_SYNC_THREADS") ? atoi(getenv("RTJPEG_B200_SYNC_THREADS")) : 0;
    const int threads = forced ? forced : nf <= 300 ? 256 : 128;
    cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t e = threads >= 256 ? sy_launch<256, false>(a, redo, handover, 0, st)
                          : threads >= 128 ? sy_launch<128, false>(a, redo, handover, 0, st)
                                           : sy_launch<64, false>(a, redo, handover, 0, st);
    return (int)e;
}

/* The frames with a raw prefix (rtj_launch_scan_sync has marked them): launched behind it where the batch is expected to
 * hold such frames; what it gives up (dense streams: noise at a high quality) stays marked for rtj_scan_mb_kernel. */
extern "C" int rtj_launch_scan_sync_raw(const rtj_launch_args *a, uint32_t *redo, int handover, void *stream)
{
    static const int forced = getenv("RTJPEG_B200_SYNC_RAW_THREADS") ? atoi(getenv("RTJPEG_B200_SYNC_RAW_THREADS")) : 0;
    static const int lead_env = getenv("RTJPEG_B200_SYNC_RAW_LEAD") ? atoi(getenv("RTJPEG_B200_SYNC_RAW_LEAD")) : 0;
    const int threads = forced ? forced : 128;
    /* lead-in, in 16-byte pieces: inside the chunk in front, whatever the frame's size */
    const int lead = min(max(lead_env ? lead_env : SY_LEAD_RAW, 1), sy_pmin(threads >= 128 ? 128 : 64) - 2);
    cudaStream_t st = (cudaStream_t)stream;
    return (int)(threads >= 128 ? sy_launch<128, true>(a, redo, handover, lead, st) : sy_launch<64, true>(a, redo, handover, lead, st));
}
