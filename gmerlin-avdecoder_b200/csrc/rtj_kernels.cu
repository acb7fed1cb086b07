/*
 * rtj_kernels.cu -- sm_100a kernels of the RTjpeg decoder: serial scans, last-writer resolve, scan plan.
 *
 *   K1  (serial flavours)   rtj_scan_lane_kernel / rtj_scan_warp_kernel: one thread or one warp walks one frame's
 *                           run-length stream and emits a 32-bit entry (payload offset + end-of-block bound, or
 *                           "skipped") for every 8x8 block.  Replaces the `sp += RTjpeg_s2b(...)` pointer chase of
 *                           RTjpeg_decompressYUV420 (lib/RTjpeg.c:2701-2745) and the length logic of RTjpeg_s2b
 *                           (:157-186).  Kept as cross-checks; what AUTO runs is in rtj_scan_sync.cu (the walk, one
 *                           instantiation for frames without a raw prefix, one for those with), rtj_scan_chunk.cu and
 *                           rtj_scan_mb.cu (what the walks hand over, without / with a raw prefix; the segment passes).
 *                           rtj_launch_scan below picks.
 *   K3  rtj_resolve_last_kernel + rtj_resolve_kernel
 *                           per block position, a last-writer scan over the frames of the batch: for every skipped
 *                           block, which earlier frame coded it last (and, where that frame's entry carries the block
 *                           inline, a copy of it).  Replaces the implicit "skipped blocks keep the previous picture"
 *                           state of the reference (lib/video_rtjpeg.c:81 decodes every packet into the same
 *                           persistent frame).
 *   K1  rtj_scan_plan_*     the frame-level chain between the two passes of the segment-parallel arrangement.
 *
 * K2 (unpack + dequantise + integer AAN IDCT + clamp + store, rtj_idct_kernel) and K2b are in rtj_idct.cu.
 *
 * All arithmetic is 32-bit integer and bit-exact with the reference: no tensor
 * cores, no floating point.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "rtj_common.h"

namespace {

constexpr unsigned FULL = 0xFFFFFFFFu;

/* ------------------------------------------------------------------------ */
/* K1: block-offset scan                                                      */
/* ------------------------------------------------------------------------ */

constexpr int SCAN_WARPS = 4;

} // namespace

extern "C" __global__ void __launch_bounds__(SCAN_WARPS * 32)
rtj_scan_warp_kernel(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                const rtj_dev_table *__restrict__ tables, int F, int nblk,
                uint32_t *__restrict__ ent, uint32_t *__restrict__ frame_skips,
                rtj_dev_info *__restrict__ info, int raw_only, int unit, int unit_luma)
{
    const int lane = threadIdx.x & 31;
    const int f = blockIdx.x * SCAN_WARPS + (threadIdx.x >> 5);
    if (f >= F) return;

    const rtjgpu_frame_desc d = desc[f];
    const uint8_t *pay = stream + d.offset + RTJPEG_B200_HEADER_BYTES;
    const int len = d.length > RTJPEG_B200_HEADER_BYTES ? (int)d.length - RTJPEG_B200_HEADER_BYTES : 0;
    const rtj_dev_table &tab = tables[min((int)d.table, RTJ_NUM_TABLES - 1)];     /* descriptors are the caller's memory */
    const int lb8 = tab.bt8[0];
    const int cb8 = tab.bt8[1];
    if (raw_only && (lb8 | cb8) == 0) return;        /* rtj_scan_chunk_kernel has done this frame */
    uint32_t *out = ent + (size_t)f * nblk;

    /* warp-uniform parser state */
    int pos = 0;        /* payload offset of lane 0's byte */
    int blk = 0;        /* blocks emitted so far */
    int k6 = 0;         /* index of the current block inside its macroblock, 0..5 */
    int rawleft = 0;    /* DC/raw bytes of the current block still to pass */
    int need = 0;       /* zig-zag positions still to fill by tokens (0: not inside a block) */
    int cur_off = 0;    /* payload offset of the current block */
    int skips = 0;
    int consumed = 0;
    uint32_t held = 0;  /* entry of block (blk & ~31) + lane, flushed every 32 blocks */

    while (blk < nblk) {
        /* one byte per lane; past the packet a 0x7F run token ends any block */
        const int at = pos + lane;
        const int b = at < len ? (int)pay[at] : 0x7F;
        const int sb = (int)(signed char)b;
        const bool isrun = sb > 63;
        const int a = isrun ? sb - 63 : 1;         /* positions this byte fills when read as a token */
        int S = a;                                   /* inclusive scan of a over the window */
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int up = __shfl_up_sync(FULL, S, o);
            if (lane >= o) S += up;
        }
        const int T = S - a;                         /* exclusive scan */
        const unsigned runmask = __ballot_sync(FULL, isrun);
        const int Slast = __shfl_sync(FULL, S, 31);

        int s = 0;                                   /* first unread lane of the window */
        while (s < 32 && blk < nblk) {
            bool done = false;
            uint32_t e_out = 0;
            if (rawleft == 0 && need == 0) {         /* at a block boundary */
                const int first = __shfl_sync(FULL, b, s);
                if (first == 0xFF) {                 /* skipped block: one byte, lib/RTjpeg.c:2704 */
                    s += 1;
                    skips++;
                    done = true;
                    e_out = RTJ_ENT_SKIP;
                } else {
                    const int bt8 = k6 < unit_luma ? lb8 : cb8;
                    cur_off = pos + s;
                    rawleft = 1 + bt8;               /* DC byte + raw 8-bit coefficients */
                    need = 63 - bt8;
                }
            }
            if (!done && rawleft > 0) {
                const int adv = min(rawleft, 32 - s);
                s += adv;
                rawleft -= adv;
                if (rawleft > 0) break;              /* raw prefix continues in the next window */
                if (need == 0) {                     /* 63 raw coefficients: no token tail */
                    done = true;
                    e_out = RTJ_ENT(min(cur_off, len), 64);
                } else if (s == 32) {
                    break;
                }
            }
            if (!done) {
                /* token tail: first lane e >= s where the filled positions reach `need` */
                const int base = __shfl_sync(FULL, T, s);
                const unsigned m = __ballot_sync(FULL, S - base >= need) & (FULL << s);
                if (m == 0) {                        /* block continues in the next window */
                    need -= Slast - base;
                    s = 32;
                    break;
                }
                const int e = __ffs(m) - 1;
                const int Te = __shfl_sync(FULL, T, e);
                /* positions >= eob are zero: a final run token starts at the bound */
                int eob = ((runmask >> e) & 1u) ? 64 - need + (Te - base) : 64;
                eob = max(1, min(eob, 64));
                e_out = RTJ_ENT(min(cur_off, len), eob);
                s = e + 1;
                need = 0;
                done = true;
            }
            if (done) {
                if (lane == (blk & 31)) held = e_out;
                blk++;
                k6 = k6 == unit - 1 ? 0 : k6 + 1;
                if ((blk & 31) == 0) out[blk - 32 + lane] = held;
            }
        }
        consumed = pos + s;
        pos += 32;
    }
    if (lane < (blk & 31)) out[(blk & ~31) + lane] = held;

    if (lane == 0) {
        frame_skips[f] = (uint32_t)skips;
        if (skips) {
            atomicAdd(&info->skipped_blocks, (unsigned long long)skips);
            atomicAdd(&info->slice_skips[0], (unsigned)skips);          /* the serial flavours scan the batch in one go */
        }
        atomicAdd(&info->payload_bytes, (unsigned long long)min(consumed, len));
        if (consumed > len || len > (int)RTJGPU_MAX_PAYLOAD_BYTES) {
            atomicAdd(&info->bad_frames, 1u);
            atomicMin((unsigned int *)&info->first_bad_frame, (unsigned int)f);
        }
    }
}


/* ------------------------------------------------------------------------ */
/* K1, lane-serial flavour: one THREAD walks one frame                        */
/* ------------------------------------------------------------------------ */
/*
 * The block grammar is a serial state machine (lib/RTjpeg.c:157-186): where a block
 * ends depends on every token before it.  One lane walks one frame, four tokens
 * per step with SIMD-within-a-register arithmetic:
 *
 *   t                     four token bytes
 *   r = t & ~(t>>1) & 0x40404040        bit 6 of every byte of the form 01xxxxxx (a run token, 64..127)
 *   x = t & ((r>>6) * 0x3F)             run length - 1 in run bytes, 0 in coefficient bytes
 *   P = x * 0x01010101 + 0x04030201     byte k = positions filled by tokens 0..k  (each token fills 1 + x_k)
 *   c = (P + (128-need) * 0x01010101) & 0x80808080
 *                                       bit 7 of byte k set  <=>  tokens 0..k fill >= need positions
 *
 * so the first set bit of c names the block's last token.  Byte overflows and carries
 * can only occur at or after that first crossing and never disturb it.  A lane costs
 * ~1 issue slot per block, so thousands of frames parse at a sliver of the machine;
 * the price is latency (one dependent chain per frame), which large batches hide.
 * The warp-cooperative flavour above serves batches with few, large frames.
 */
namespace {

__device__ __forceinline__ uint32_t ld_u32_unaligned(const uint32_t *__restrict__ base4, int byte_off)
{
    const uint32_t *wp = base4 + (byte_off >> 2);
    return __funnelshift_r(__ldg(wp), __ldg(wp + 1), (unsigned)(byte_off & 3) * 8);
}

struct LaneResult { int blk, skips, consumed; };

/* SWAR pieces: see the comment above.  swar_x: run length - 1 in run bytes, 0 elsewhere. */
__device__ __forceinline__ uint32_t swar_runs(uint32_t t) { return t & ~(t >> 1) & 0x40404040u; }
__device__ __forceinline__ uint32_t swar_x(uint32_t t, uint32_t r) { return t & ((r >> 6) * 0x3Fu); }

template <bool RAW>
__device__ __forceinline__ LaneResult lane_scan_frame(const uint8_t *__restrict__ pay, int len, int lb8, int cb8,
                                                     uint32_t *__restrict__ out, int nblk, int unit, int unit_luma)
{
    const uint32_t *base4 = reinterpret_cast<const uint32_t *>(pay);     /* packets start 4-byte aligned */
    int o = 0, blk = 0, skips = 0, k6 = 0;
    /* Lanes of a warp move in lockstep, so one lane missing L1 stalls all 32 (and with 128 sector
     * look-ups per step somebody always misses).  A real load touches the sector each lane will need
     * ~40 blocks from now; its value is consumed four steps later, by when even a DRAM miss is back. */
    uint32_t touch0 = 0, touch1 = 0, touch2 = 0, touch3 = 0, sink = 0;
    while (blk < nblk && o < len) {
        const int bt8 = RAW ? (k6 < unit_luma ? lb8 : cb8) : 0;
        if (RAW) k6 = k6 == unit - 1 ? 0 : k6 + 1;
        sink ^= touch3;
        touch3 = touch2; touch2 = touch1; touch1 = touch0;
        touch0 = __ldg(base4 + (min(o + 160, len + (int)RTJGPU_STREAM_SLACK_BYTES - 4) >> 2));   /* never behind the slack */

        /* the block's first byte and its first eight tokens */
        uint32_t first, t0, t1;
        {
            const uint32_t *wp = base4 + (o >> 2);
            const unsigned sh = (unsigned)(o & 3) * 8;
            const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2), w3 = __ldg(wp + 3);
            const uint32_t u0 = __funnelshift_r(w0, w1, sh), u1 = __funnelshift_r(w1, w2, sh),
                           u2 = __funnelshift_r(w2, w3, sh);
            first = u0 & 0xFFu;
            t0 = __funnelshift_r(u0, u1, 8);          /* bytes o+1 .. o+4 */
            t1 = __funnelshift_r(u1, u2, 8);          /* bytes o+5 .. o+8 */
        }
        int tok = o + 1 + bt8;
        if (RAW) {
            const uint32_t *wp = base4 + (tok >> 2);
            const unsigned sh = (unsigned)(tok & 3) * 8;
            const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
            t0 = __funnelshift_r(w0, w1, sh);
            t1 = __funnelshift_r(w1, w2, sh);
        }
        const bool isff = first == 0xFFu;             /* skipped block: one byte, lib/RTjpeg.c:2704 */
        int need = 63 - bt8;                          /* positions the token tail has to fill */

        /* eight tokens at once, no branches: the common block (<= 9 bytes) resolves here */
        const uint32_t K = (uint32_t)(128 - need) * 0x01010101u;
        const uint32_t r0 = swar_runs(t0), r1 = swar_runs(t1);
        const uint32_t P0 = swar_x(t0, r0) * 0x01010101u + 0x04030201u;
        const uint32_t P1 = swar_x(t1, r1) * 0x01010101u + 0x04030201u + (P0 >> 24) * 0x01010101u;
        const uint32_t c0 = (P0 + K) & 0x80808080u, c1 = (P1 + K) & 0x80808080u;
        uint32_t c = c0 ? c0 : c1, t = c0 ? t0 : t1, r = c0 ? r0 : r1;
        int ntok = c0 ? 0 : 4;
        if (!isff && c == 0 && need > 0) {            /* long block: keep going four tokens at a time */
            need -= (int)(P1 >> 24);
            ntok = 8;
            for (;;) {
                if (tok + ntok >= len + 64) { c = 0x80u; r = 0; break; }       /* runaway on a truncated frame */
                t = ld_u32_unaligned(base4, tok + ntok);
                r = swar_runs(t);
                const uint32_t P = swar_x(t, r) * 0x01010101u + 0x04030201u;
                c = (P + (uint32_t)(128 - need) * 0x01010101u) & 0x80808080u;
                if (c) break;
                need -= (int)(P >> 24);
                ntok += 4;
            }
        }
        const int bit = __ffs((int)c) - 1;            /* 7, 15, 23 or 31 */
        ntok += (bit >> 3) + 1;
        const uint32_t bk = (t >> (bit - 7)) & 0xFFu;
        /* positions >= eob are zero: a final run of n zeros ends at 64, so it starts at 64 - n */
        int eob = ((r >> (bit - 1)) & 1u) ? 63 - (int)(bk & 0x3Fu) : 64;
        if (need <= 0) { ntok = 0; eob = 64; }        /* 63 raw coefficients: no token tail */
        out[blk++] = isff ? RTJ_ENT_SKIP : RTJ_ENT(min(o, len), max(eob, 1));
        skips += isff;
        o = isff ? o + 1 : tok + ntok;
    }
    if (sink == 0x5eed5eedu && (touch0 ^ touch1 ^ touch2) == 0x0badf00du) skips = -1;     /* keeps the touch loads alive; never true in effect */
    LaneResult res = {blk, skips, o};
    return res;
}

} // namespace

extern "C" __global__ void __launch_bounds__(32)
rtj_scan_lane_kernel(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                     const rtj_dev_table *__restrict__ tables, int F, int nblk,
                     uint32_t *__restrict__ ent, uint32_t *__restrict__ frame_skips,
                     rtj_dev_info *__restrict__ info, int raw_only, int unit, int unit_luma)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const rtjgpu_frame_desc d = desc[f];
    const uint8_t *pay = stream + d.offset + RTJPEG_B200_HEADER_BYTES;
    const int len = d.length > RTJPEG_B200_HEADER_BYTES ? (int)d.length - RTJPEG_B200_HEADER_BYTES : 0;
    const rtj_dev_table &tab = tables[min((int)d.table, RTJ_NUM_TABLES - 1)];     /* descriptors are the caller's memory */
    const int lb8 = tab.bt8[0];
    const int cb8 = tab.bt8[1];
    if (raw_only && (lb8 | cb8) == 0) return;        /* rtj_scan_chunk_kernel has done this frame */
    uint32_t *out = ent + (size_t)f * nblk;

    const LaneResult res = (lb8 == 0 && cb8 == 0) ? lane_scan_frame<false>(pay, len, 0, 0, out, nblk, unit, unit_luma)
                                                  : lane_scan_frame<true>(pay, len, lb8, cb8, out, nblk, unit, unit_luma);

    /* a frame whose stream ends early or mid-block: flag it, give the missing blocks a harmless entry */
    const bool bad = res.blk < nblk || res.consumed > len;
    for (int b = res.blk; b < nblk; b++) out[b] = RTJ_ENT(len, 1);
    frame_skips[f] = (uint32_t)res.skips;
    if (res.skips) {
        atomicAdd(&info->skipped_blocks, (unsigned long long)res.skips);
        atomicAdd(&info->slice_skips[0], (unsigned)res.skips);
    }
    atomicAdd(&info->payload_bytes, (unsigned long long)min(res.consumed, len));
    if (bad || len > (int)RTJGPU_MAX_PAYLOAD_BYTES) {
        atomicAdd(&info->bad_frames, 1u);
        atomicMin((unsigned int *)&info->first_bad_frame, (unsigned int)f);
    }
}

/* ------------------------------------------------------------------------ */
/* K3: last-writer resolution of skipped blocks                               */
/* ------------------------------------------------------------------------ */

/*
 * Two kernels over (block position, chunk of RESOLVE_T frames), so that the scan over the batch's
 * frames -- serial in the reference, where it is simply "the picture persists" -- is spread over
 * F / RESOLVE_T times nblk threads:
 *   rtj_resolve_last_kernel   last frame of the chunk that coded the position (or none)
 *   rtj_resolve_kernel        carry-in = nearest earlier chunk with a writer, then the walk over the
 *                             chunk's own frames that gives every skipped block its last writer.
 * Both work on one SLICE of the batch, frames [f0, f1) = chunks [c_lo, c_hi): the look-back stays inside
 * the slice (a few chunks), and what lies before the slice comes as one value per position, `carry_in`,
 * which the previous slice's last chunk left in its `carry_out`.  A slice whose frames -- and all frames
 * before them -- hold no skip marker has nothing to resolve: every position was written by frame f1 - 1.
 * (slice_skips[0 .. slice] are final when K3 of that slice runs; the batch-wide count is not, K1 of later
 * slices may be running.)
 * A batch of several independent sequences (rtjgpu_decode_device_seq) changes nothing but rtj_resolve_kernel's walk:
 * a last writer in front of the frame's own sequence is taken as none.  rtj_resolve_last_kernel's running maximum and
 * the shortcut above stay exact -- the nearest writer before a frame is the only one that can lie in its sequence.
 */
constexpr int RESOLVE_T = RTJ_RESOLVE_T;

__device__ __forceinline__ bool k3_any_skips(const rtj_dev_info *__restrict__ info, int slice)
{
    unsigned any = 0;
    for (int s = 0; s <= slice; s++) any |= info->slice_skips[s];
    return any != 0;
}

extern "C" __global__ void __launch_bounds__(128)
rtj_resolve_last_kernel(const uint32_t *__restrict__ ent, uint16_t *__restrict__ chunk_last, uint32_t *__restrict__ chunk_mask,
                        int f0, int f1, int nblk, const rtj_dev_info *__restrict__ info, int slice, uint32_t *__restrict__ arrived)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");      /* rtj_resolve_kernel may take its places */
    if (!k3_any_skips(info, slice)) return;          /* nothing to resolve so far */
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < nblk)
        for (int c = f0 / RESOLVE_T + blockIdx.y; c * RESOLVE_T < f1; c += gridDim.y) {
            const int fa = c * RESOLVE_T, fb = min(f1, fa + RESOLVE_T);
            unsigned last = RTJ_SRC_CARRY;
            uint32_t skipped = 0;                            /* bit j: frame fa + j skipped the position -- rtj_resolve_kernel reads only the others */
            uint32_t e[16];
            int f = fa;
            for (; f + 16 <= fb; f += 16) {
#pragma unroll
                for (int j = 0; j < 16; j++) e[j] = ent[(size_t)(f + j) * nblk + b];
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    if (!RTJ_ENT_IS_SKIP(e[j])) last = (unsigned)(f + j);
                    else skipped |= 1u << (f + j - fa);
                }
            }
            for (; f < fb; f++) {
                if (!RTJ_ENT_IS_SKIP(ent[(size_t)f * nblk + b])) last = (unsigned)f;
                else skipped |= 1u << (f - fa);
            }
            chunk_last[(size_t)c * nblk + b] = (uint16_t)last;
            chunk_mask[(size_t)c * nblk + b] = skipped;
        }
    /* The CTA that arrives last for this group of positions turns chunk_last into a running maximum down the slice's chunks
     * -- chunk_last[c] := the last writer in chunks c_lo .. c -- so that rtj_resolve_kernel finds its carry-in with ONE read
     * however long nobody wrote a position (a static background: the look-back used to walk chunk by chunk, once per later
     * chunk). */
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned n = atomicAdd(&arrived[blockIdx.x], 1u);
        s_last = n == gridDim.y - 1;
        if (s_last) arrived[blockIdx.x] = 0u;                /* ready for the next launch */
    }
    __syncthreads();
    if (!s_last || b >= nblk) return;
    __threadfence();
    const int c_lo = f0 / RESOLVE_T, c_hi = (f1 + RESOLVE_T - 1) / RESOLVE_T;
    unsigned run = RTJ_SRC_CARRY;
    int c = c_lo;
    for (; c + 8 <= c_hi; c += 8) {
        unsigned v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = __ldcg(&chunk_last[(size_t)(c + j) * nblk + b]);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (v[j] != RTJ_SRC_CARRY) run = v[j];
            chunk_last[(size_t)(c + j) * nblk + b] = (uint16_t)run;
        }
    }
    for (; c < c_hi; c++) {
        const unsigned v = __ldcg(&chunk_last[(size_t)c * nblk + b]);
        if (v != RTJ_SRC_CARRY) run = v;
        chunk_last[(size_t)c * nblk + b] = (uint16_t)run;
    }
}

/* (seven CTAs an SM: 72 registers, what the kernel held before the sequence check -- registers are allocated in eights) */
extern "C" __global__ void __launch_bounds__(128, 7)
rtj_resolve_kernel(uint32_t *__restrict__ ent, const uint16_t *__restrict__ chunk_last, const uint32_t *__restrict__ chunk_mask,
                   uint16_t *__restrict__ src, int f0, int f1, int nblk, const rtj_dev_info *__restrict__ info, int slice,
                   const uint16_t *__restrict__ carry_in, uint16_t *__restrict__ carry_out,
                   const rtjgpu_frame_desc *__restrict__ desc, unsigned long long *__restrict__ skips_seen,
                   const uint32_t *__restrict__ seq)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    /* how many blocks the batch skipped, left where the host sees it without asking (pinned memory): the next batch's
     * arrangement of K2 goes by it */
    if (skips_seen && b == 0 && blockIdx.y == 0) {
        skips_seen[0] = info->skipped_blocks;
        skips_seen[1] = info->raw_frames;                           /* ... and AUTO's choice of K1's arrangement */
        if (info->raw_walked) skips_seen[2] = info->raw_given_up;   /* (a batch in which the walk was not tried says nothing about it) */
    }
    if (b >= nblk) return;
    if (!k3_any_skips(info, slice)) {                               /* (K1's counters: final before rtj_resolve_last_kernel started) */
        if (blockIdx.y == 0) carry_out[b] = (uint16_t)(f1 - 1);     /* every frame so far wrote every position */
        return;
    }
    /* launched with programmatic stream serialisation behind rtj_resolve_last_kernel: resident early, its notes final from here */
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int c_lo = f0 / RESOLVE_T;
    for (int c0 = c_lo + blockIdx.y; c0 * RESOLVE_T < f1; c0 += gridDim.y) {
        const int fa = c0 * RESOLVE_T, fb = min(f1, fa + RESOLVE_T);
        unsigned last = c0 > c_lo ? chunk_last[(size_t)(c0 - 1) * nblk + b] : RTJ_SRC_CARRY;   /* rtj_resolve_last_kernel's running maximum */
        if (last == RTJ_SRC_CARRY && carry_in) last = carry_in[b];
        /* Several sequences in the batch (seq != NULL): a last writer in front of the frame's own sequence is none -- the block
         * comes from that sequence's carry.  One comparison at the chunk's first frame covers the running maximum and carry_in
         * (RTJ_SRC_CARRY is above every frame index); behind it, a frame that starts a sequence starts from none. */
        uint32_t starts = 0;                                         /* bit j: frame fa + j starts a sequence */
        if (seq) {
            if (RTJ_SEQ_FIRST(seq[fa]) > last) last = RTJ_SRC_CARRY;
#pragma unroll 1
            for (int j = 1; j < fb - fa; j++) starts |= (RTJ_SEQ_FIRST(seq[fa + j]) == (unsigned)(fa + j) ? 1u : 0u) << j;
        }
        /* the last writer's entry, when it is an inline one (the block travels in it), and the tables it was written under:
         * a skipped block of a frame with the same tables gets a copy of it (RTJ_ENT_COPY_BIT) in the place of its marker */
        uint32_t last_e = 0;
        unsigned last_tab = 0;
        if (last != RTJ_SRC_CARRY) {
            const uint32_t e = ent[(size_t)last * nblk + b];
            if (RTJ_ENT_IS_INLINE(e)) { last_e = e | RTJ_ENT_COPY_BIT; last_tab = desc[last].table; }
        }
        /* skipped blocks are known from the first pass's mask: only the coded entries are read.  A skipped block gets a copy of
         * its last writer's inline entry, or -- where there is none to copy -- its last writer's frame in src[] (K2 looks there
         * only for entries that are still skip markers). */
        const uint32_t skipped = chunk_mask[(size_t)c0 * nblk + b];
        uint32_t e[8];
        unsigned tab[8];
        int f = fa;
        for (; f + 8 <= fb; f += 8) {
#pragma unroll
            for (int j = 0; j < 8; j++) {
                e[j] = (skipped >> (f + j - fa)) & 1u ? RTJ_ENT_SKIP : ent[(size_t)(f + j) * nblk + b];
                tab[j] = desc[f + j].table;
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                if ((starts >> (f + j - fa)) & 1u) { last = RTJ_SRC_CARRY; last_e = 0; }
                if (RTJ_ENT_IS_SKIP(e[j])) {
                    if (last_e && tab[j] == last_tab) ent[(size_t)(f + j) * nblk + b] = last_e;
                    else src[(size_t)(f + j) * nblk + b] = (uint16_t)last;
                } else {
                    last = (unsigned)(f + j);
                    last_e = RTJ_ENT_IS_INLINE(e[j]) ? (e[j] | RTJ_ENT_COPY_BIT) : 0u;
                    last_tab = tab[j];
                }
            }
        }
        for (; f < fb; f++) {
            const uint32_t ee = (skipped >> (f - fa)) & 1u ? RTJ_ENT_SKIP : ent[(size_t)f * nblk + b];
            const unsigned tb = desc[f].table;
            if ((starts >> (f - fa)) & 1u) { last = RTJ_SRC_CARRY; last_e = 0; }
            if (RTJ_ENT_IS_SKIP(ee)) {
                if (last_e && tb == last_tab) ent[(size_t)f * nblk + b] = last_e;
                else src[(size_t)f * nblk + b] = (uint16_t)last;
            } else {
                last = (unsigned)f;
                last_e = RTJ_ENT_IS_INLINE(ee) ? (ee | RTJ_ENT_COPY_BIT) : 0u;
                last_tab = tb;
            }
        }
        if (fb == f1) carry_out[b] = (uint16_t)last;                 /* the slice's last chunk: what the next slice starts from */
    }
}

/* ------------------------------------------------------------------------ */
/* K1, segment-parallel flavour: the frame-level chain between the two passes */
/* ------------------------------------------------------------------------ */

/* what the frame-level chain needs to know about a frame */
struct PlanFrame { int len, unit, segbytes, nseg; bool raw; };

__device__ __forceinline__ PlanFrame plan_frame(const rtjgpu_frame_desc *__restrict__ desc, const rtj_dev_table *__restrict__ tables,
                                                int f, int maxseg, int unit_blocks)
{
    const rtjgpu_frame_desc d = desc[f];
    PlanFrame p;
    p.len = d.length > RTJPEG_B200_HEADER_BYTES ? (int)d.length - RTJPEG_B200_HEADER_BYTES : 0;
    /* with a raw prefix the summaries count macroblocks (rtj_scan_mb.cu), without it blocks */
    const rtj_dev_table &tab = tables[min((int)d.table, RTJ_NUM_TABLES - 1)];
    const bool raw = (tab.bt8[0] | tab.bt8[1]) != 0;
    p.raw = raw;
    p.unit = raw ? unit_blocks : 1;
    p.segbytes = raw ? RTJ_SEG_BYTES_MB : RTJ_SEG_BYTES;
    p.nseg = (int)min((long long)maxseg, ((long long)p.len + p.segbytes - 1) / p.segbytes);   /* segments that hold payload */
    return p;
}

/* The frame's closing: blocks it holds, the missing ones' harmless entries, the flag of a frame without any block (every
 * other frame is closed by the segment that holds its last block). */
__device__ __forceinline__ void plan_close(int f, int nb, int nblk, int len, uint32_t *__restrict__ ent, uint32_t *__restrict__ frame_skips,
                                           rtj_dev_info *__restrict__ info, const rtj_seg_plan &sp)
{
    const int nbf = min(nb, nblk);
    sp.nbf[f] = nbf;
    frame_skips[f] = 0;
    for (int b = nbf; b < nblk; b++) ent[(size_t)f * nblk + b] = RTJ_ENT(min(len, (int)RTJ_ENT_OFF_MASK), 1);
    if (nbf == 0 && nblk > 0) {
        atomicAdd(&info->bad_frames, 1u);
        atomicMin((unsigned int *)&info->first_bad_frame, (unsigned int)f);
    }
}

/* segments [s0, s1) of frame f from (entry e, nb blocks before): their entry offsets and first block indices; segments behind
 * the payload or behind the frame's last block are marked unused.  Returns the blocks before segment s1. */
__device__ __forceinline__ int plan_walk(const PlanFrame &p, int f, int s0, int s1, int e, int nb, int nblk, const rtj_seg_plan &sp)
{
    for (int seg = s0; seg < s1; seg++) {
        const size_t idx = (size_t)f * sp.maxseg + seg;
        if (seg >= p.nseg || nb >= nblk) { sp.base[idx] = RTJ_SEG_UNUSED; continue; }
        sp.entry[idx] = (uint32_t)e;
        sp.base[idx] = (uint32_t)nb;
        const uint32_t v = sp.sum[idx * RTJ_SEG_NE + e];
        e = min((int)(v & 511u), RTJ_SEG_NE - 1);
        nb += p.unit * (int)(v >> 9);
    }
    return nb;
}

/* One thread per frame: the whole chain.  For frames of a few dozen segments. */
extern "C" __global__ void __launch_bounds__(64)
rtj_scan_plan_kernel(const rtjgpu_frame_desc *__restrict__ desc, const rtj_dev_table *__restrict__ tables, int F, int nblk,
                     uint32_t *__restrict__ ent, uint32_t *__restrict__ frame_skips, rtj_dev_info *__restrict__ info,
                     const rtj_seg_plan sp, int unit_blocks)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const PlanFrame p = plan_frame(desc, tables, f, sp.maxseg, unit_blocks);
    if (p.raw) atomicAdd(&info->raw_frames, 1u);
    const int nb = plan_walk(p, f, 0, sp.maxseg, 0, 0, nblk, sp);
    plan_close(f, nb, nblk, p.len, ent, frame_skips, info, sp);
}

/*
 * Frames of hundreds of segments (a dense 1920x1088 frame: 500): the chain above is as many dependent loads from a table
 * that does not fit the L2 -- 0.39 ms for a batch of 128 such frames, a tenth of the whole scan.  In three steps instead:
 *   groups   every group of RTJ_SEG_GROUP segments is summarised like a segment is: for every entry offset, where the parse
 *            leaves the group and how many units it starts (one thread per entry offset, 16 dependent loads, all groups
 *            of all frames at once)
 *   chain    one thread per frame hops group to group
 *   fill     one thread per group walks its segments from the group's now known entry
 */
extern "C" __global__ void __launch_bounds__(RTJ_SEG_NE)
rtj_scan_plan_group_kernel(const rtjgpu_frame_desc *__restrict__ desc, const rtj_dev_table *__restrict__ tables, const rtj_seg_plan sp,
                           int unit_blocks)
{
    const int f = blockIdx.y, g = blockIdx.x, e0 = threadIdx.x;
    const PlanFrame p = plan_frame(desc, tables, f, sp.maxseg, unit_blocks);
    const int s0 = g * RTJ_SEG_GROUP, s1 = min(s0 + RTJ_SEG_GROUP, sp.maxseg);
    if (s1 > p.nseg) return;                         /* a group that is not all payload is walked, not summarised */
    int e = e0, units = 0;
    for (int seg = s0; seg < s1; seg++) {
        const uint32_t v = sp.sum[((size_t)f * sp.maxseg + seg) * RTJ_SEG_NE + e];
        e = min((int)(v & 511u), RTJ_SEG_NE - 1);
        units += (int)(v >> 9);
    }
    sp.gsum[((size_t)f * sp.ngroups + g) * RTJ_SEG_NE + e0] = (uint32_t)e | ((uint32_t)units << 9);
}

extern "C" __global__ void __launch_bounds__(64)
rtj_scan_plan_chain_kernel(const rtjgpu_frame_desc *__restrict__ desc, const rtj_dev_table *__restrict__ tables, int F,
                           const rtj_seg_plan sp, int unit_blocks)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const PlanFrame p = plan_frame(desc, tables, f, sp.maxseg, unit_blocks);
    int e = 0, nb = 0;
    for (int g = 0; g < sp.ngroups; g++) {
        const size_t idx = (size_t)f * sp.ngroups + g;
        sp.gentry[idx] = (uint32_t)e;
        sp.gbase[idx] = (uint32_t)nb;
        if (min((g + 1) * RTJ_SEG_GROUP, sp.maxseg) > p.nseg) {          /* the payload ends in this group: nothing behind it matters */
            for (int g2 = g + 1; g2 < sp.ngroups; g2++) sp.gbase[(size_t)f * sp.ngroups + g2] = RTJ_SEG_UNUSED;
            break;
        }
        const uint32_t v = sp.gsum[idx * RTJ_SEG_NE + e];
        e = (int)(v & 511u);
        nb += p.unit * (int)(v >> 9);
    }
}

extern "C" __global__ void __launch_bounds__(64)
rtj_scan_plan_fill_kernel(const rtjgpu_frame_desc *__restrict__ desc, const rtj_dev_table *__restrict__ tables, int F, int nblk,
                          uint32_t *__restrict__ ent, uint32_t *__restrict__ frame_skips, rtj_dev_info *__restrict__ info,
                          const rtj_seg_plan sp, int unit_blocks)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= F * sp.ngroups) return;
    const int f = t / sp.ngroups, g = t - f * sp.ngroups;
    const PlanFrame p = plan_frame(desc, tables, f, sp.maxseg, unit_blocks);
    if (p.raw && g == 0) atomicAdd(&info->raw_frames, 1u);
    const int s0 = g * RTJ_SEG_GROUP, s1 = min(s0 + RTJ_SEG_GROUP, sp.maxseg);
    const uint32_t gb = sp.gbase[(size_t)f * sp.ngroups + g];
    int nb;
    if (gb == RTJ_SEG_UNUSED) {
        nb = nblk;                                                     /* behind the payload: every segment unused */
        for (int seg = s0; seg < s1; seg++) sp.base[(size_t)f * sp.maxseg + seg] = RTJ_SEG_UNUSED;
    } else
        nb = plan_walk(p, f, s0, s1, (int)sp.gentry[(size_t)f * sp.ngroups + g], (int)gb, nblk, sp);
    /* the group that holds the payload's last segment knows how many blocks the frame's stream holds */
    const int glast = p.nseg > 0 ? (p.nseg - 1) / RTJ_SEG_GROUP : 0;
    if (g == glast) plan_close(f, p.nseg > 0 ? nb : 0, nblk, p.len, ent, frame_skips, info, sp);
}

extern "C" int rtj_kernels_init(void)
{
    int e = rtj_idct_init();
    if (e) return e;
    if ((e = rtj_scan_mb_init())) return e;
    if ((e = rtj_scan_walk_init())) return e;
    if ((e = rtj_scan_sync_init())) return e;
    return rtj_scan_chunk_init();
}

extern "C" int rtj_launch_scan(const rtj_launch_args *a, void *stream)
{
    const int nblk = RTJ_FMT_NBLK(a->fmt, a->w, a->h);
    cudaStream_t st = (cudaStream_t)stream;
    /* AUTO: the chunk-parallel kernels -- rtj_scan_chunk_kernel takes every frame without a raw prefix,
     * rtj_scan_mb_kernel the others; each returns at once on the other's frames. */
    if (a->scan_mode == RTJGPU_SCAN_SYNC || (a->scan_mode == RTJGPU_SCAN_AUTO && !a->seg.sum)) {
        /* one CTA per frame.  Frames without a raw prefix: the self-synchronising walk; the frames it hands over (streams
         * that do not forget their past) are scanned by rtj_scan_chunk_kernel right behind it.  SYNC keeps every such
         * frame in the walk (the cross-check of the parity suite). */
        /* Frames with a raw prefix: the walk's other instantiation, launched where the batch before held such frames (or the
         * flavour is forced); what it gives up -- and, where it was not launched, every such frame -- is rtj_scan_mb_kernel's. */
        const int handover = a->scan_mode == RTJGPU_SCAN_AUTO;
        const bool raw_pass = a->scan_mode == RTJGPU_SCAN_SYNC || a->raw_expected;
        uint32_t *redo = a->d_redo;
        int e = rtj_launch_scan_sync(a, redo, handover, stream);
        if (!e && handover) e = rtj_launch_scan_chunk_redo(a, redo, stream);
        if (!e && raw_pass) e = rtj_launch_scan_sync_raw(a, redo, handover, stream);
        if (!e) e = rtj_launch_scan_mb(a, 0, redo, stream);
        return e ? -e : 2 + (handover ? 1 : 0) + (raw_pass ? 1 : 0);
    }
    if (a->scan_mode == RTJGPU_SCAN_AUTO || a->scan_mode == RTJGPU_SCAN_CHUNK || a->scan_mode == RTJGPU_SCAN_SEGMENT) {
        if (a->seg.sum) {
            /* few frames: their segments are parsed by separate CTAs -- summaries, frame-level chain, emit */
            int e = rtj_launch_scan_chunk(a, 1, stream);
            if (!e) e = rtj_launch_scan_mb(a, 1, nullptr, stream);
            if (e) return -e;
            int launches = 5;
            if (a->seg.gsum) {
                const int ub = RTJ_FMT_UNIT_BLOCKS(a->fmt);
                rtj_scan_plan_group_kernel<<<dim3((unsigned)a->seg.ngroups, (unsigned)a->F), RTJ_SEG_NE, 0, st>>>(a->d_desc, a->d_tables, a->seg, ub);
                rtj_scan_plan_chain_kernel<<<(a->F + 63) / 64, 64, 0, st>>>(a->d_desc, a->d_tables, a->F, a->seg, ub);
                rtj_scan_plan_fill_kernel<<<(a->F * a->seg.ngroups + 63) / 64, 64, 0, st>>>(a->d_desc, a->d_tables, a->F, nblk, a->d_ent,
                                                                                          a->d_frame_skips, a->d_info, a->seg, ub);
                launches = 7;
            } else
                rtj_scan_plan_kernel<<<(a->F + 63) / 64, 64, 0, st>>>(a->d_desc, a->d_tables, a->F, nblk, a->d_ent,
                                                                      a->d_frame_skips, a->d_info, a->seg,
                                                                      RTJ_FMT_UNIT_BLOCKS(a->fmt));
            if ((e = (int)cudaGetLastError())) return -e;
            e = rtj_launch_scan_chunk(a, 2, stream);
            if (!e) e = rtj_launch_scan_mb(a, 2, nullptr, stream);
            return e ? -e : launches;
        }
        int e = rtj_launch_scan_chunk(a, 0, stream);
        if (e) return -e;
        e = rtj_launch_scan_mb(a, 0, nullptr, stream);
        return e ? -e : 2;
    }
    /* rtjgpu_set_scan_mode() forces one serial flavour for every frame: one lane per frame (cheap in
     * issue slots, latency hidden only by very large batches) or one warp per frame. */
    if (a->scan_mode == RTJGPU_SCAN_WALK) {
        /* the walker takes the frames without raw prefix, rtj_scan_mb_kernel the others */
        int e = rtj_launch_scan_walk(a, 0, nblk, stream);
        if (!e) e = rtj_launch_scan_mb(a, 0, nullptr, stream);
        return e ? -e : 2;
    }
    if (a->scan_mode == RTJGPU_SCAN_LANE) {
        rtj_scan_lane_kernel<<<(a->F + 31) / 32, 32, 0, st>>>(
            a->d_stream, a->d_desc, a->d_tables, a->F, nblk, a->d_ent, a->d_frame_skips, a->d_info, 0,
            RTJ_FMT_UNIT_BLOCKS(a->fmt), RTJ_FMT_UNIT_LUMA(a->fmt));
    } else {
        const int grid = (a->F + SCAN_WARPS - 1) / SCAN_WARPS;
        rtj_scan_warp_kernel<<<grid, SCAN_WARPS * 32, 0, st>>>(
            a->d_stream, a->d_desc, a->d_tables, a->F, nblk, a->d_ent, a->d_frame_skips, a->d_info, 0,
            RTJ_FMT_UNIT_BLOCKS(a->fmt), RTJ_FMT_UNIT_LUMA(a->fmt));
    }
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -(int)e;
}

extern "C" int rtj_launch_resolve(const rtj_launch_args *a, void *stream)
{
    const int nblk = RTJ_FMT_NBLK(a->fmt, a->w, a->h);
    /* a batch without skip markers only pays for the launches: keep the grid modest and let a CTA
     * stride over the chunks of frames */
    const int nchunks = (a->f1 - a->f0 + RESOLVE_T - 1) / RESOLVE_T;    /* f0 is a multiple of RESOLVE_T */
    static const int ymax = getenv("RTJPEG_B200_K3Y") ? atoi(getenv("RTJPEG_B200_K3Y")) : 32;
    dim3 grid((unsigned)((nblk + 127) / 128), (unsigned)(nchunks < ymax ? nchunks : ymax));
    rtj_resolve_last_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(a->d_ent, a->d_chunk_last, a->d_chunk_mask, a->f0, a->f1, nblk, a->d_info, a->slice, a->d_k3_count);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(128);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, rtj_resolve_kernel, a->d_ent, (const uint16_t *)a->d_chunk_last, (const uint32_t *)a->d_chunk_mask,
                                             a->d_src, a->f0, a->f1, nblk, (const rtj_dev_info *)a->d_info, a->slice, a->d_k3_in, a->d_k3_out,
                                             a->d_desc, a->h_skips_seen, a->d_seq);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaGetLastError();
}
