/*
 * rtj_idct.cu -- K2 of the RTjpeg decoder: unpack + dequantise + integer AAN IDCT +
 * clamp + planar store, for sm_100a.
 *
 *   rtj_idct_kernel       one CTA per (frame, macroblock row [, strip]).  Replaces the value
 *                         path of RTjpeg_s2b (lib/RTjpeg.c:162-183), RTjpeg_idct (:2209-2332)
 *                         and the destination arithmetic of RTjpeg_decompressYUV420
 *                         (:2690-2744).  The strip's blocks are renumbered so that a warp
 *                         owns 32 horizontally adjacent 8x8 blocks (conflict-free shared
 *                         stores); the picture strip leaves the SM as TMA bulk stores.
 *                         Blocks are handled by sparsity class:
 *                           T2     E <= 3 (DC + zig-zag 1, 2): decoded right away, two pixels
 *                                  per instruction in packed 16-bit arithmetic
 *                           M7     E <= 7 (adds (0,2), (1,1), (2,0), (3,0)): deferred, decoded
 *                                  in class-homogeneous groups of 32
 *                           CARRY  skipped and never written in this batch: copied from the
 *                                  picture that precedes the batch
 *                           HARD   everything else (long blocks, blocks whose last writer
 *                                  used other tables): queued in device memory for ...
 *   rtj_idct_hard_kernel  ... the general decoder, one thread per queued block, which patches
 *                         its 8x8 pixels straight into the output frames afterwards.
 *
 * All arithmetic is integer and bit-exact with the reference.  The packed 16-bit epilogues
 * are used only where a bound on the block's coefficients proves that no pixel leaves
 * 16..235 and nothing overflows 16 bits; otherwise the same block takes the reference's
 * 32-bit DESCALE / clamp sequence.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "rtj_common.h"
#include "rtj_convert.cuh"

namespace {

constexpr unsigned FULL = 0xFFFFFFFFu;

/* MULTIPLY of the reference (lib/RTjpeg.c:1206): 8 fractional bits, +128, arithmetic shift. */
__device__ __forceinline__ int fxmul(int v, int c) { return (v * c + 128) >> 8; }

/* low 16 bits, sign-extended: the `int16_t` stores of RTjpeg_s2b and DESCALE */
__device__ __forceinline__ int wrap16(int v) { return (int)(short)v; }

/* 8-point AAN flow graph shared by both passes (lib/RTjpeg.c:2240-2283, :2289-2326).
 * Inputs that are literal zeros fold away at compile time: fxmul(0, c) == 0. */
__device__ __forceinline__ void aan8(int x0, int x1, int x2, int x3, int x4, int x5, int x6, int x7,
                                     int (&y)[8])
{
    const int s04 = x0 + x4, d04 = x0 - x4;
    const int s26 = x2 + x6;
    const int m26 = fxmul(x2 - x6, 362) - s26;
    const int e0 = s04 + s26, e3 = s04 - s26, e1 = d04 + m26, e2 = d04 - m26;

    const int z13 = x5 + x3, z10 = x5 - x3, z11 = x1 + x7, z12 = x1 - x7;
    const int o7 = z11 + z13;
    const int o11 = fxmul(z11 - z13, 362);
    const int z5 = fxmul(z10 + z12, 473);
    const int o10 = fxmul(z12, 277) - z5;
    const int o12 = fxmul(z10, -669) + z5;
    const int o6 = o12 - o7;
    const int o5 = o11 - o6;
    const int o4 = o10 + o5;

    y[0] = e0 + o7; y[7] = e0 - o7;
    y[1] = e1 + o6; y[6] = e1 - o6;
    y[2] = e2 + o5; y[5] = e2 - o5;
    y[4] = e3 + o4; y[3] = e3 - o4;
}

/* Four row outputs (already carrying the +4 rounding term) -> four clamped bytes.
 * DESCALE (lib/RTjpeg.c:1200) narrows to int16 before RL (:1204) clamps to 16..235;
 * packing the low halves reproduces that narrowing exactly. */
__device__ __forceinline__ uint32_t descale_pack4(int y0, int y1, int y2, int y3)
{
    uint32_t a = __byte_perm((uint32_t)(y0 >> 3), (uint32_t)(y1 >> 3), 0x5410);
    uint32_t b = __byte_perm((uint32_t)(y2 >> 3), (uint32_t)(y3 >> 3), 0x5410);
    a = __vmaxs2(__vmins2(a, 0x00EB00EBu), 0x00100010u);
    b = __vmaxs2(__vmins2(b, 0x00EB00EBu), 0x00100010u);
    return __byte_perm(a, b, 0x6420);
}

/* zig-zag position k sits at (row, col): lib/RTjpeg.c:59-74 */
#define RTJ_ZZ_LIST(X) \
    X(0,0,0) X(1,1,0) X(2,0,1) X(3,0,2) X(4,1,1) X(5,2,0) X(6,3,0) X(7,2,1) \
    X(8,1,2) X(9,0,3) X(10,0,4) X(11,1,3) X(12,2,2) X(13,3,1) X(14,4,0) X(15,5,0) \
    X(16,4,1) X(17,3,2) X(18,2,3) X(19,1,4) X(20,0,5) X(21,0,6) X(22,1,5) X(23,2,4) \
    X(24,3,3) X(25,4,2) X(26,5,1) X(27,6,0) X(28,7,0) X(29,6,1) X(30,5,2) X(31,4,3) \
    X(32,3,4) X(33,2,5) X(34,1,6) X(35,0,7) X(36,1,7) X(37,2,6) X(38,3,5) X(39,4,4) \
    X(40,5,3) X(41,6,2) X(42,7,1) X(43,7,2) X(44,6,3) X(45,5,4) X(46,4,5) X(47,3,6) \
    X(48,2,7) X(49,3,7) X(50,4,6) X(51,5,5) X(52,6,4) X(53,7,3) X(54,7,4) X(55,6,5) \
    X(56,5,6) X(57,4,7) X(58,5,7) X(59,6,6) X(60,7,5) X(61,7,6) X(62,6,7) X(63,7,7)

/*
 * Byte source of one block for the sparse classes: the first 4*NW bytes sit in
 * registers (aligned 32-bit loads, funnel-shifted to the block's byte offset) and
 * leave through the low byte, so the token walk issues no dependent loads.
 */
template <int NW>
struct RegBytes {
    uint32_t u[NW];
    __device__ __forceinline__ RegBytes() {}
    __device__ __forceinline__ explicit RegBytes(const uint8_t *__restrict__ src)
    {
        const uintptr_t a = reinterpret_cast<uintptr_t>(src);
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
        const unsigned sh = (unsigned)(a & 3) * 8;
        uint32_t w[NW + 1];
#pragma unroll
        for (int i = 0; i <= NW; i++) w[i] = __ldg(wp + i);      /* independent loads; slack bytes follow the stream */
#pragma unroll
        for (int i = 0; i < NW; i++) u[i] = __funnelshift_r(w[i], w[i + 1], sh);
    }
    __device__ __forceinline__ int peek_u8() const { return (int)(u[0] & 0xFFu); }
    __device__ __forceinline__ int peek_s8() const { return (int)(signed char)(u[0] & 0xFFu); }
    __device__ __forceinline__ void advance(bool take)
    {
        const unsigned sh = take ? 8u : 0u;
#pragma unroll
        for (int i = 0; i < NW - 1; i++) u[i] = __funnelshift_r(u[i], u[i + 1], sh);
        u[NW - 1] >>= sh;
    }
};

/* Byte source for dense blocks: straight from global memory, one byte at a time. */
struct MemBytes {
    const uint8_t *q;
    __device__ __forceinline__ explicit MemBytes(const uint8_t *__restrict__ src) : q(src) {}
    __device__ __forceinline__ int peek_u8() const { return (int)__ldg(q); }
    __device__ __forceinline__ int peek_s8() const { return (int)(signed char)__ldg(q); }
    __device__ __forceinline__ void advance(bool take) { q += take ? 1 : 0; }
};

/* Coefficients 0..K-1 of one block, dequantised (lib/RTjpeg.c:162-183): x[0] is the DC term
 * (unsigned byte) with DESCALE's +4 rounding term folded in -- it reaches every output
 * unchanged because the DC path has no multiply -- x[k] the k-th zig-zag coefficient.
 * iq holds the multipliers in zig-zag order, bt8 is the raw-prefix length. */
template <int K, typename Bytes, typename IQ>
__device__ __forceinline__ void unpack_block(Bytes &by, IQ iq, int bt8, int (&x)[K])
{
    x[0] = wrap16(by.peek_u8() * iq[0]) + 4;
    by.advance(true);
    int z = 0;          /* zero positions still owed by the last run token */
#pragma unroll
    for (int k = 1; k < K; k++) {
        const bool take = z == 0;
        const int bb = by.peek_s8();
        const bool run = take && k > bt8 && bb > 63;
        const int v = (take && !run) ? bb : 0;
        z = take ? (run ? bb - 64 : 0) : z - 1;
        by.advance(take);
        x[k] = wrap16(v * iq[k]);
    }
}

/* The same for a block of at most 16 coefficients under a raw prefix of BT8 bytes (lib/RTjpeg.c:165-169; 4, 8 or 9 with the
 * tables of a quality above 170): the DC byte and the prefix sit at fixed places of the 24 bytes held in registers, and
 * only the 15 - BT8 places behind them are walked as tokens, over a window of three words instead of six. */
template <int BT8, typename IQ>
__device__ __forceinline__ void unpack_block16_prefix(const RegBytes<6> &by, IQ iq, int (&x)[16])
{
    static_assert(BT8 >= 1 && BT8 <= 11, "the tokens behind the prefix fit twelve bytes that start inside the first three words");
    x[0] = wrap16((int)(by.u[0] & 0xFFu) * iq[0]) + 4;
#pragma unroll
    for (int k = 1; k <= BT8; k++) x[k] = wrap16((int)(signed char)((by.u[k >> 2] >> (8 * (k & 3))) & 0xFFu) * iq[k]);
    constexpr int b0 = BT8 + 1, w0 = b0 >> 2;
    constexpr unsigned sh = (unsigned)(b0 & 3) * 8u;
    RegBytes<3> t;
#pragma unroll
    for (int i = 0; i < 3; i++) t.u[i] = __funnelshift_r(by.u[w0 + i], w0 + i + 1 < 6 ? by.u[w0 + i + 1] : 0u, sh);
    int z = 0;
#pragma unroll
    for (int k = BT8 + 1; k < 16; k++) {
        const bool take = z == 0;
        const int bb = t.peek_s8();
        const bool run = take && bb > 63;
        const int v = (take && !run) ? bb : 0;
        z = take ? (run ? bb - 64 : 0) : z - 1;
        t.advance(take);
        x[k] = wrap16(v * iq[k]);
    }
}

/* General 8x8 inverse transform of a block whose zig-zag positions >= K are zero:
 * the reference's two passes with its DESCALE / clamp epilogue. */
template <int K>
__device__ __forceinline__ void idct_general(const int (&x)[K], uint32_t (&px)[16])
{
    int m[8][8];
#pragma unroll
    for (int r = 0; r < 8; r++)
#pragma unroll
        for (int c = 0; c < 8; c++) m[r][c] = 0;
#define RTJ_PUT(k, r, c) if ((k) < K) m[r][c] = x[(k) < K ? (k) : 0];
    RTJ_ZZ_LIST(RTJ_PUT)
#undef RTJ_PUT

    /* pass 1: columns (lib/RTjpeg.c:2221-2285) */
    int ws[8][8];
#pragma unroll
    for (int c = 0; c < 8; c++) {
        int y[8];
        aan8(m[0][c], m[1][c], m[2][c], m[3][c], m[4][c], m[5][c], m[6][c], m[7][c], y);
#pragma unroll
        for (int r = 0; r < 8; r++) ws[r][c] = y[r];
    }
    /* pass 2: rows, descale, clamp (lib/RTjpeg.c:2287-2330) */
#pragma unroll
    for (int r = 0; r < 8; r++) {
        int y[8];
        aan8(ws[r][0], ws[r][1], ws[r][2], ws[r][3], ws[r][4], ws[r][5], ws[r][6], ws[r][7], y);
        px[2 * r] = descale_pack4(y[0], y[1], y[2], y[3]);
        px[2 * r + 1] = descale_pack4(y[4], y[5], y[6], y[7]);
    }
}

/* odd half of the flow graph when x1 is its only input: (o7, o6, o5, o4) */
__device__ __forceinline__ void odd_from_x1(int x1, int &o7, int &o6, int &o5, int &o4)
{
    const int z5 = fxmul(x1, 473);
    o7 = x1;
    o6 = z5 - x1;                       /* o12 = fxmul(0, -669) + z5 = z5 */
    o5 = fxmul(x1, 362) - o6;
    o4 = fxmul(x1, 277) - z5 + o5;
}

/* (v << 5) of two values side by side in 16-bit halves, modulo 2^16 each */
__device__ __forceinline__ uint32_t pack_scaled(int lo, int hi)
{
    return __byte_perm((uint32_t)lo << 5, (uint32_t)hi << 5, 0x5410);
}

/* Packed epilogue arithmetic.  A pixel is (y >> 3) with y = a + d known to lie in 128..1887
 * (so neither clamp acts and DESCALE's int16 narrowing is the identity).  Halves hold
 * (value << 5) modulo 2^16: the pixel is then the upper BYTE of its half.  The non-negative
 * term carries a guard of 16 below the binary point, so the +-1 that a carry or borrow out of
 * the low half leaks into the high half never reaches bit 5.  One 32-bit add or subtract
 * makes two pixels, one PRMT gathers four. */
constexpr uint32_t PK_DUP = 0x00200020u;    /* v * PK_DUP = (v << 5) in both halves, 0 <= v < 2048 */
constexpr uint32_t PK_GUARD = 0x00100010u;

/*
 * T2: at most DC, zig-zag 1 (row 1, column 0) and zig-zag 2 (row 0, column 1).  Column 1 of
 * the first pass is constant down the rows, so the odd half of every ROW pass is the same
 * eight values D[j] and pixel (r, j) = A[r] + D[j], A = the column-0 pass.
 * x0 = dequantised DC + 4, x1 = zig-zag 1, q = zig-zag 2.
 */
__device__ __forceinline__ bool t2_safe(int x0, int x1, int q)
{
    /* |A[r] - x0| <= |x1| + 3 and |D[j]| <= |q| + 3: every odd term is below its input in magnitude */
    const int spread = abs(x1) + abs(q) + 6;
    return x0 - spread >= 128 && x0 + spread <= 1887;
}

__device__ __forceinline__ void t2_pixels(int x0, int x1, int q, bool packed, uint32_t (&px)[16])
{
    int a7, a6, a5, a4, d7, d6, d5, d4;
    odd_from_x1(x1, a7, a6, a5, a4);
    odd_from_x1(q, d7, d6, d5, d4);
    /* A[0]=x0+a7 A[7]=x0-a7 A[1]=x0+a6 A[6]=x0-a6 A[2]=x0+a5 A[5]=x0-a5 A[4]=x0+a4 A[3]=x0-a4;
     * D[0]=d7 D[7]=-d7 D[1]=d6 D[6]=-d6 D[2]=d5 D[5]=-d5 D[4]=d4 D[3]=-d4 */
    if (packed) {
        /* pixel (r, j) = x0 + a(r) + d(j): the four pairs x0 + d(j) are made once, a row adds or subtracts its a(r) */
        const uint32_t X = (uint32_t)x0 * PK_DUP + PK_GUARD;
        const uint32_t d01 = pack_scaled(d7, d6);         /* (D0, D1) */
        const uint32_t d23 = pack_scaled(d5, -d4);        /* (D2, D3) */
        const uint32_t X01 = X + d01, X23 = X + d23;
        const uint32_t X45 = X - __byte_perm(d23, 0u, 0x1032);   /* (D4, D5) = -(D3, D2) */
        const uint32_t X67 = X - __byte_perm(d01, 0u, 0x1032);   /* (D6, D7) = -(D1, D0) */
        const uint32_t k7 = (uint32_t)a7 * PK_DUP, k6 = (uint32_t)a6 * PK_DUP, k5 = (uint32_t)a5 * PK_DUP, k4 = (uint32_t)a4 * PK_DUP;
        /* modulo 2^32 these are the sums of the reference's rows, (x0 +- a) * PK_DUP + PK_GUARD +- d with x0 +- a >= 0 */
#define RTJ_T2_ROW(r, op, k) \
        px[2 * (r)] = __byte_perm(X01 op k, X23 op k, 0x7531); \
        px[2 * (r) + 1] = __byte_perm(X45 op k, X67 op k, 0x7531);
        RTJ_T2_ROW(0, +, k7) RTJ_T2_ROW(1, +, k6) RTJ_T2_ROW(2, +, k5) RTJ_T2_ROW(3, -, k4)
        RTJ_T2_ROW(4, +, k4) RTJ_T2_ROW(5, -, k5) RTJ_T2_ROW(6, -, k6) RTJ_T2_ROW(7, -, k7)
#undef RTJ_T2_ROW
    } else {
        const int A[8] = {x0 + a7, x0 + a6, x0 + a5, x0 - a4, x0 + a4, x0 - a5, x0 - a6, x0 - a7};
#pragma unroll
        for (int r = 0; r < 8; r++) {
            px[2 * r] = descale_pack4(A[r] + d7, A[r] + d6, A[r] + d5, A[r] - d4);
            px[2 * r + 1] = descale_pack4(A[r] + d4, A[r] - d5, A[r] - d6, A[r] - d7);
        }
    }
}

/*
 * M7: zig-zag positions 0..6 = (0,0) (1,0) (0,1) (0,2) (1,1) (2,0) (3,0).  Column 0 has four
 * inputs, column 1 two, column 2 is constant (x[3] in every row).  In the row pass the even
 * half is then w0[r] plus one of four constants and the odd half depends on w1[r] alone.
 */
__device__ __forceinline__ bool m7_safe(const int (&x)[7])
{
    /* every pixel stays within x[0] +- spread: |odd terms| <= |x1| + 1.18 |x3| + 3, even terms within
     * |x2| + 1 of x0 (the gains of the flow graph), applied to both passes */
    const int spread = abs(x[1]) + abs(x[5]) + abs(x[6]) + (abs(x[6]) >> 2) + abs(x[2]) + abs(x[4]) + abs(x[3]) + 16;
    return x[0] - spread >= 128 && x[0] + spread <= 1887;
}

__device__ __forceinline__ void m7_pixels(const int (&x)[7], bool packed, uint32_t (&px)[16])
{
    /* pass 1, column 0: inputs rows 0..3 = x0 x1 x5 x6 */
    int w0[8];
    {
        const int x0 = x[0], x1 = x[1], x2 = x[5], x3 = x[6];
        const int t12 = fxmul(x2, 362) - x2;
        const int e0 = x0 + x2, e3 = x0 - x2, e1 = x0 + t12, e2 = x0 - t12;
        const int o7 = x1 + x3;
        const int d13 = x1 - x3;
        const int o11 = fxmul(d13, 362);
        const int z5 = fxmul(d13, 473);
        const int o10 = fxmul(x1, 277) - z5;
        const int o12 = fxmul(-x3, -669) + z5;
        const int o6 = o12 - o7, o5 = o11 - o6, o4 = o10 + o5;
        w0[0] = e0 + o7; w0[7] = e0 - o7; w0[1] = e1 + o6; w0[6] = e1 - o6;
        w0[2] = e2 + o5; w0[5] = e2 - o5; w0[4] = e3 + o4; w0[3] = e3 - o4;
    }
    /* pass 1, column 1: inputs rows 0, 1 = x2 x4 */
    int w1[8];
    {
        int o7, o6, o5, o4;
        odd_from_x1(x[4], o7, o6, o5, o4);
        const int x0 = x[2];
        w1[0] = x0 + o7; w1[7] = x0 - o7; w1[1] = x0 + o6; w1[6] = x0 - o6;
        w1[2] = x0 + o5; w1[5] = x0 - o5; w1[4] = x0 + o4; w1[3] = x0 - o4;
    }
    /* pass 2: even half = w0[r] + {+c2, +t12, -t12, -c2}, odd half from w1[r] */
    const int c2 = x[3];
    const int t12 = fxmul(c2, 362) - c2;
    if (packed) {
        const uint32_t ce01 = pack_scaled(c2, t12);
        const uint32_t ce23 = pack_scaled(-t12, -c2);
#pragma unroll
        for (int r = 0; r < 8; r++) {
            int o7, o6, o5, o4;
            odd_from_x1(w1[r], o7, o6, o5, o4);
            const uint32_t a2 = (uint32_t)w0[r] * PK_DUP + PK_GUARD;
            const uint32_t e01 = a2 + ce01, e23 = a2 + ce23;          /* (e0, e1), (e2, e3): non-negative halves */
            const uint32_t o76 = pack_scaled(o7, o6), o5m4 = pack_scaled(o5, -o4);
            px[2 * r] = __byte_perm(e01 + o76, e23 + o5m4, 0x7531);      /* y0 y1 y2 y3 */
            px[2 * r + 1] = __byte_perm(e23 - o5m4, e01 - o76, 0x5713);  /* y4 y5 y6 y7 */
        }
    } else {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            int o7, o6, o5, o4;
            odd_from_x1(w1[r], o7, o6, o5, o4);
            const int e0 = w0[r] + c2, e1 = w0[r] + t12, e2 = w0[r] - t12, e3 = w0[r] - c2;
            px[2 * r] = descale_pack4(e0 + o7, e1 + o6, e2 + o5, e3 - o4);
            px[2 * r + 1] = descale_pack4(e3 + o4, e2 - o5, e1 - o6, e0 - o7);
        }
    }
}

constexpr int IDCT_MAX_MB = 128;     /* macroblocks per CTA strip */
constexpr int IDCT_THREADS = 128;

enum { Q_M7 = 0, Q_CARRY, Q_HARD, NQ, CLS_T2 = NQ, CLS_NONE = -1 };

__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, unsigned bytes)
{
    /* TMA 1-D bulk copy shared -> global (UBLKCP) */
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes) : "memory");
}

/*
 * Strip geometry, per picture format (rtj_common.h).  A strip of `mbs` units holds BLK*mbs blocks in
 * stream order i = BLK*unit + sub: YUV420 Y00 Y01 Y10 Y11 U V (lib/RTjpeg.c:2704-2739), YUV422
 * Y0 Y1 U V (:2654-2681), grey Y (:2761-2770).  The kernel works in "picture order" p -- luma block
 * rows left to right, then U, then V -- so consecutive p are horizontally adjacent 8-byte runs of the
 * shared picture strip and a warp's stores never conflict.  The strip holds the luma rows
 * (16 or 8 rows), then 8 U rows and 8 V rows of half the width.
 */
struct PicPos {
    int i;          /* stream-order index inside the strip */
    int off;        /* byte offset of the block's first row inside the shared strip (< 65536) */
};

template <int FMT> struct Geo;

template <> struct Geo<0> {                 /* YUV420: units of 16x16 */
    static constexpr int BLK = 6, UNIT_W = 16, LUMA_ROWS = 16, TILE = 384, CHROMA_AT = 256, PLANES = 3;
    __device__ static __forceinline__ PicPos pic_pos(int p, int mbs)        /* branch-free; luma positions come first */
    {
        const bool luma = p < 4 * mbs;
        const int half = luma ? 2 * mbs : mbs;
        const int t = luma ? p : p - 4 * mbs;
        const int hi = t >= half ? 1 : 0;
        const int c = t - (hi ? half : 0);
        PicPos r;
        r.i = luma ? 3 * c - 2 * (c & 1) + 2 * hi              /* 6 * (c >> 1) + 2 * hi + (c & 1) */
                   : 6 * c + 4 + hi;
        r.off = 8 * c + (luma ? hi * 128 * mbs : (256 + hi * 64) * mbs);     /* V follows the 8 rows of U */
        return r;
    }
    /* block bi (stream order inside the strip that starts at unit mx0 of unit row my) in a tight-pitch picture */
    __device__ static __forceinline__ const uint8_t *carry_src(const uint8_t *pic, int bi, int my, int mx0, int w, int h, int &pitch)
    {
        const int mb = bi / 6, sub = bi - mb * 6;
        if (sub < 4) {
            pitch = w;
            return pic + (size_t)(my * 16 + (sub >> 1) * 8) * w + (mx0 + mb) * 16 + (sub & 1) * 8;
        }
        pitch = w >> 1;
        return pic + (size_t)w * h + (sub == 5 ? (size_t)(w >> 1) * (h >> 1) : 0) + (size_t)(my * 8) * pitch + (mx0 + mb) * 8;
    }
};

template <> struct Geo<1> {                 /* YUV422: units of 16x8, chroma half width and full height */
    static constexpr int BLK = 4, UNIT_W = 16, LUMA_ROWS = 8, TILE = 256, CHROMA_AT = 128, PLANES = 3;
    __device__ static __forceinline__ PicPos pic_pos(int p, int mbs)
    {
        const bool luma = p < 2 * mbs;
        const int t = luma ? p : p - 2 * mbs;
        const int hi = (!luma && t >= mbs) ? 1 : 0;
        const int c = t - hi * mbs;
        PicPos r;
        r.i = luma ? 2 * c - (c & 1) : 4 * c + 2 + hi;         /* 4 * (c >> 1) + (c & 1) */
        r.off = 8 * c + (luma ? 0 : (128 + hi * 64) * mbs);
        return r;
    }
    __device__ static __forceinline__ const uint8_t *carry_src(const uint8_t *pic, int bi, int my, int mx0, int w, int h, int &pitch)
    {
        const int un = bi >> 2, sub = bi & 3;
        if (sub < 2) {
            pitch = w;
            return pic + (size_t)(my * 8) * w + (mx0 + un) * 16 + sub * 8;
        }
        pitch = w >> 1;
        return pic + (size_t)w * h + (sub == 3 ? (size_t)pitch * h : 0) + (size_t)(my * 8) * pitch + (mx0 + un) * 8;
    }
};

template <> struct Geo<2> {                 /* 8-bit grey: units of 8x8, luma only */
    static constexpr int BLK = 1, UNIT_W = 8, LUMA_ROWS = 8, TILE = 64, CHROMA_AT = 64, PLANES = 1;
    __device__ static __forceinline__ PicPos pic_pos(int p, int mbs)
    {
        PicPos r;
        r.i = p;
        r.off = 8 * p;
        return r;
    }
    __device__ static __forceinline__ const uint8_t *carry_src(const uint8_t *pic, int bi, int my, int mx0, int w, int h, int &pitch)
    {
        pitch = w;
        return pic + (size_t)(my * 8) * w + (mx0 + bi) * 8;
    }
};

template <int FMT>
__device__ __forceinline__ bool off_is_chroma(int off, int mbs) { return Geo<FMT>::PLANES == 3 && off >= Geo<FMT>::CHROMA_AT * mbs; }

/* tile_s: the strip's address in the shared window (32 bit: one add per row, no generic pointers) */
template <int FMT>
__device__ __forceinline__ void store_block(unsigned tile_s, int off, int mbs, const uint32_t (&px)[16])
{
    const unsigned luma_pitch = (unsigned)(Geo<FMT>::UNIT_W * mbs);
    const unsigned pitch = off_is_chroma<FMT>(off, mbs) ? luma_pitch >> 1 : luma_pitch;
    unsigned sa = tile_s + (unsigned)off;
#pragma unroll
    for (int r = 0; r < 8; r++, sa += pitch)
        asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(sa), "r"(px[2 * r]), "r"(px[2 * r + 1]) : "memory");
}

/* Where block i (stream order, whole frame) of frame f lives in the tight-pitch output planes. */
__device__ __forceinline__ uint8_t *block_dst(uint8_t *base, int fmt, int i, int w, int h, int &pitch)
{
    const int cw = w >> 1;
    if (fmt == 0) {
        const int mbw = w >> 4;
        const int mb = i / 6, sub = i - mb * 6;
        const int my = mb / mbw, mx = mb - my * mbw;
        if (sub < 4) { pitch = w; return base + (size_t)(my * 16 + (sub >> 1) * 8) * w + mx * 16 + (sub & 1) * 8; }
        pitch = cw;
        return base + (size_t)w * h + (sub == 5 ? (size_t)cw * (h >> 1) : 0) + (size_t)(my * 8) * cw + mx * 8;
    }
    if (fmt == 1) {
        const int uw = w >> 4;
        const int un = i >> 2, sub = i & 3;
        const int by = un / uw, ux = un - by * uw;
        if (sub < 2) { pitch = w; return base + (size_t)(by * 8) * w + ux * 16 + sub * 8; }
        pitch = cw;
        return base + (size_t)w * h + (sub == 3 ? (size_t)cw * h : 0) + (size_t)(by * 8) * cw + ux * 8;
    }
    const int bw = w >> 3;
    const int by = i / bw, bx = i - by * bw;
    pitch = w;
    return base + (size_t)(by * 8) * w + bx * 8;
}

/* what the kernel takes from the host */
struct K2Params {
    const uint8_t *stream;
    const rtjgpu_frame_desc *desc;
    const rtj_dev_table *tables;
    const uint32_t *ent;
    const uint16_t *srcf;
    int nblk, w, h, seg_mb, nstrips;
    int f0, F;                       /* first frame of this launch (blockIdx.y = 0); frames of the batch */
    int reserve;                     /* launch the RES instantiation */
    int f_end, run;                  /* one behind the launch's last frame; frames a CTA works through in turn (blockIdx.y counts runs) */
    int row0, rows;                  /* first row of units of this launch (blockIdx.x = 0); rows of units of a picture */
    uint8_t *out;
    const uint8_t *carry;
    int fmt;
    uint32_t *hardq;
    unsigned hardq_cap;              /* entries of hardq: F * nblk */
    rtj_dev_info *info;
    const uint32_t *pos;             /* SINGLE: pic_pos of every position of a row, i | off << 16 (rtj_build_lut_kernel) */
    /* RGB: the strip leaves as packed pixels (out / fmt unused) */
    uint8_t *rgb;                    /* picture row r of frame f at rgb + f * rgb_frame_pitch + r * rgb_row_pitch */
    size_t rgb_row_pitch, rgb_frame_pitch;
    int rgb_kind;                    /* RTJ_CONV_RGB32 / BGR32 / RGB24 / BGR24 / RGB16 */
    unsigned rgb_alpha;
    uint8_t *last_yuv;               /* RGB: the batch's last frame as planes as well (the next batch's carry), or NULL */
    /* several independent sequences in the batch (NULL: one, which takes carry / last_yuv): per frame RTJ_SEQ(first frame
     * of its sequence, sequence index); per sequence its carry and, RGB, where its last frame leaves as planes */
    const uint32_t *seq;
    const uint8_t *const *carries;
    uint8_t *const *last_yuvs;
    int ahead;                       /* frames between a CTA and the one that follows it on the same SM slot */
    int wq;                          /* slots of one warp's queue */
    /* SEL: blockIdx.y names job j0 + blockIdx.y of the batch's njobs RTJ_JOB words (frame, output slot), sorted by frame;
     * `ahead` then counts jobs */
    const uint32_t *jobs;
    int j0, njobs;
    /* WIN: a window of win_w x win_h pixels of every job's frame, at the origin of the frame's sequence (RTJ_WIN words,
     * per sequence; seq is never NULL).  win_last = 0: the window leaves to out + slot * frame_bytes(win_w, win_h) as tight
     * planes, or as packed pixels; 1: the window is the whole picture and leaves as planes to last_yuvs[sequence] */
    const uint32_t *win;
    int win_w, win_h, win_last;
    /* RGB_CHW: the window leaves planar and typed to rgb (rtj_launch_args::chw): channel c of rgb_kind's pixel, as chw_dtype,
     * scaled and offset by chw_scale[c], chw_bias[c] */
    int chw_dtype;
    float chw_scale[3], chw_bias[3];
};

/* The general decoder for one block that K2's sparse classes do not take (long blocks; blocks whose last writer used
 * other tables): gidx = frame * nblk + block.  `full`: more than 16 coefficients -- the reference's two full passes, fed
 * byte by byte; else the first 16 zig-zag positions (rows 0..5, columns 0..4) from 24 bytes held in registers. */
__device__ __forceinline__ void decode_general(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                                               const rtj_dev_table *__restrict__ tables, const uint32_t *__restrict__ ent,
                                               const uint16_t *__restrict__ srcf, int nblk, uint32_t gidx, int chroma, bool full,
                                               uint32_t (&px)[16])
{
    const unsigned f = gidx / (unsigned)nblk;
    const int i = (int)(gidx - f * (unsigned)nblk);
    uint32_t e = ent[gidx];
    unsigned sf = f;
    if (RTJ_ENT_IS_SKIP(e)) {                    /* queued skipped blocks always have a writer in the batch */
        sf = srcf[gidx];
        e = ent[(size_t)sf * nblk + i];
    }
    const rtj_dev_table *t = &tables[min((int)desc[sf].table, RTJ_NUM_TABLES - 1)];
    const uint8_t *src = stream + desc[sf].offset + RTJPEG_B200_HEADER_BYTES + (e & RTJ_ENT_OFF_MASK);
    if (RTJ_ENT_IS_INLINE(e)) {
        const int x0 = wrap16((int)(e & 0xFFu) * t->iq[chroma][0]) + 4;
        const int x1 = wrap16((int)(signed char)((e >> 8) & 0xFFu) * t->iq[chroma][1]);
        const int q = wrap16((int)(signed char)((e >> 16) & 0xFFu) * t->iq[chroma][2]);
        t2_pixels(x0, x1, q, false, px);
    } else if (full) {
        MemBytes by(src);
        int x[64];
        unpack_block<64>(by, t->iq[chroma], t->bt8[chroma], x);
        idct_general<64>(x, px);
    } else {
        RegBytes<6> by(src);
        int x[16];
        unpack_block<16>(by, t->iq[chroma], t->bt8[chroma], x);
        idct_general<16>(x, px);
    }
}

/* the same as a call (the fused-RGB kernel's rare path: kept out of line so that it does not set the kernel's registers) */
__device__ __noinline__ void decode_general_call(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                                                 const rtj_dev_table *__restrict__ tables, const uint32_t *__restrict__ ent,
                                                 const uint16_t *__restrict__ srcf, int nblk, uint32_t gidx, int chroma, int full,
                                                 uint32_t *__restrict__ px16)
{
    uint32_t px[16];
    decode_general(stream, desc, tables, ent, srcf, nblk, gidx, chroma, full != 0, px);
#pragma unroll
    for (int r = 0; r < 16; r++) px16[r] = px[r];
}

constexpr int K2_WARPS = IDCT_THREADS / 32;
constexpr int K2_PF_LINES = 12;                   /* 128-byte lines of payload asked into L2 for the CTA that follows */

} // namespace

/*
 * One CTA per (frame, macroblock row [, strip]).  A warp takes 32 picture positions per round,
 * decodes the T2 blocks among them at once and parks the others in its own queue (M7 from the
 * front, CARRY / HARD from the back), without atomics.  After one barrier the M7 blocks of all
 * warps are decoded pooled, 32 per pass; CARRY blocks are copied and HARD blocks handed to the
 * device queue by the warp that found them.  A second barrier, and the picture strip leaves.
 *
 * SINGLE: the strip is the whole macroblock row (frames up to IDCT_MAX_MB macroblocks wide): no
 * strip arithmetic, and the strip is contiguous in the tight-pitch output planes -> TMA bulk stores.
 */
/* RGBK: RGB_NONE = planes leave; RTJ_CONV_RGB32 .. RTJ_CONV_RGB16 = that converter fused into the store (one kernel per
 * kind: the conversion doubles the kernel's arithmetic and wants its registers); RGB_ANY = the kind is read at run time
 * (strips of very wide pictures: not worth five more kernels); RGB_CHW = a window that leaves planar and typed
 * (rtjgpu_decode_device_chw_window: WIN kernels only; the channel order and the element type are read at run time) */
constexpr int RGB_NONE = -1, RGB_ANY = 99, RGB_CHW = 100;

/* RUN: a CTA works through P.run frames in turn (below); false: one frame, and none of the run's bookkeeping is compiled in */
/* RES: a warp reserves its places in K2b's queue with one request per row (streams in which most blocks go that way: a quality
 * above 170; chosen by the batch before, like RUN) */
/* SEL: a selection of frames (rtjgpu_decode_device[_rgb]_select).  One frame per CTA, taken from job blockIdx.y of P.jobs: a
 * frame needs only its own entries and its last writers' (K3), never the pixels of the frames before it.  Its pixels go to
 * the job's output slot -- K2b's queue names the slot as the place they go to --; a fused-RGB job without a slot (an
 * unselected last frame of a sequence) leaves as planes for last_yuv only. */
/* WIN: a window of every selected frame (rtjgpu_decode_device[_rgb]_window), strips only.  blockIdx.x walks the strips and
 * rows of units of the window of the frame's sequence, from its origin; a CTA below its own window returns at once.  HARD
 * blocks are decoded here by the general path, as in the fused-RGB kernels: no K2b, so no block of K2b's would have to be
 * clipped.  The strip is complete in shared memory before it leaves, clipped to the window's rows. */
template <bool SINGLE, int FMT, int WARPS, int RGBK, bool RUN, bool RES = false, bool SEL = false, bool WIN = false>
__global__ void __launch_bounds__(WARPS * 32, WARPS == 4 ? 8 : 10)
rtj_idct_kernel(const K2Params P)
{
    constexpr bool RGB = RGBK != RGB_NONE;
    static_assert(!RGB || FMT == 0, "the fused converters are the reference's yuv420 ones");
    static_assert(!SEL || (!RUN && !RES), "a selection is decoded one frame per CTA, without K2b's reservations");
    static_assert(!WIN || (SEL && !SINGLE), "a window is a selection, decoded in strips");
    constexpr bool CHW = RGBK == RGB_CHW;
    static_assert(!CHW || WIN, "the planar typed form is a window's");
    constexpr bool GENERAL = RGB || WIN;                     /* HARD blocks decoded in this kernel, not queued for K2b */
    constexpr int THREADS = WARPS * 32;
    typedef Geo<FMT> G;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.wait;" ::: "memory");        /* resident before K3 is done (launch_pdl); K3's entries are final from here */
    const unsigned job_at = SEL ? (unsigned)P.j0 + blockIdx.y : 0u;
    const uint32_t job = SEL ? __ldg(P.jobs + job_at) : 0u;
    /* A CTA works through a RUN of frames of its row of units, the strip staying in shared memory from frame to frame: what a
     * frame skips (lib/RTjpeg.c:2704 -- the block keeps what the picture held) is then simply not touched, instead of being
     * decoded again from its last writer's stream for every frame it persists in.  P.run == 1: one frame per CTA. */
    const unsigned f_first = SEL ? RTJ_JOB_FRAME(job) : (unsigned)P.f0 + blockIdx.y * (RUN ? (unsigned)P.run : 1u);
    const unsigned f_last = RUN ? min(f_first + (unsigned)P.run, (unsigned)P.f_end) : f_first + 1u;       /* one behind */
    constexpr bool runs = RUN;
    const int w = P.w, h = P.h, mbw = w / G::UNIT_W;           /* units per picture row */
    /* WIN: the window's origin -- wx in units, wy in pixels -- and the unit it starts in */
    const uint32_t worg = WIN && !P.win_last ? __ldg(P.win + RTJ_SEQ_INDEX(P.seq[f_first])) : 0u;
    const int wx = WIN ? (int)RTJ_WIN_X(worg) / G::UNIT_W : 0, wy = WIN ? (int)RTJ_WIN_Y(worg) : 0;
    const int strip = SINGLE ? 0 : (int)(blockIdx.x % (unsigned)P.nstrips);
    const int my = (WIN ? wy / G::LUMA_ROWS : P.row0) + (SINGLE ? (int)blockIdx.x : (int)(blockIdx.x / (unsigned)P.nstrips));
    if (WIN && my > (wy + P.win_h - 1) / G::LUMA_ROWS) return;  /* below this sequence's window (before any barrier) */
    const int mx0 = (WIN ? wx : 0) + strip * P.seg_mb;
    const int mbs = SINGLE ? mbw : min(P.seg_mb, (WIN ? wx + P.win_w / G::UNIT_W : mbw) - mx0);
    const int nb = mbs * G::BLK;
    const unsigned strip_blk0 = (unsigned)(my * mbw + mx0) * (unsigned)G::BLK;

    uint8_t *tile = smem;                                            /* TILE * mbs bytes: Y, U, V */
    const unsigned tile_s = (unsigned)__cvta_generic_to_shared(tile);
    int *s_hard = reinterpret_cast<int *>(tile + G::TILE * mbs);     /* HARD blocks of the strip, per warp */
    static_assert(WARPS == 3 || WARPS == 4, "s_hard holds four counters per kind");
    if (WARPS == 3 && tid == 1) { s_hard[3] = 0; s_hard[7] = 0; }
    const int wq = P.wq;                                             /* queue slots of one warp: every block it looked at */
    uint32_t *wq_e = reinterpret_cast<uint32_t *>(s_hard + 8) + warp * wq;      /* this warp's queue: entries ... */
    uint32_t *wq_p = reinterpret_cast<uint32_t *>(s_hard + 8) + (K2_WARPS + warp) * wq;   /* ... strip offset | source << 16 */
    const int rounds = (nb + THREADS - 1) / THREADS;
    /* the positions of a whole row are the same for every row of every frame: a table, hot in L1 (padded to a
     * multiple of THREADS); strips of wider pictures work them out */
    auto pos_of = [&](int p) -> PicPos {
        if (SINGLE) {
            const uint32_t v = __ldg(P.pos + p);
            PicPos r;
            r.i = (int)(v & 0xFFFFu);
            r.off = (int)(v >> 16);
            return r;
        }
        return G::pic_pos(p, mbs);
    };
    unsigned valid = 0;              /* bit r: the strip holds the picture's pixels at this thread's position of round r */

    for (unsigned f = f_first; f < f_last; f++) {
    /* a frame that starts a sequence of its own holds nothing of the frame before: like the run's first frame, it keeps nothing */
    if (runs && P.seq && RTJ_SEQ_FIRST(P.seq[f]) == f) valid = 0u;
    const unsigned frame_blk0 = f * (unsigned)P.nblk + strip_blk0;   /* F * nblk < 2^32 (checked by the host) */
    const uint32_t *my_ent = P.ent + frame_blk0;
    /* A CTA lives a few microseconds, of which the first read of its entries from DRAM -- under the write traffic of
     * this kernel -- is a good part.  So it asks for the entries it will want next into L2 now: those of the CTA that will
     * take its place when it retires (same strip, P.ahead frames on), or, working through a run, those of its next frame. */
    unsigned pf = runs ? 1u : (unsigned)P.ahead;
    bool pf_ok = runs ? f + 1u < f_last : f + pf < (unsigned)P.F;
    if (SEL) {                                                       /* ... the frame of the job P.ahead jobs on */
        const unsigned ja = job_at + (unsigned)P.ahead;
        pf_ok = ja < (unsigned)P.njobs;
        pf = pf_ok ? RTJ_JOB_FRAME(__ldg(P.jobs + ja)) - f : 0u;     /* jobs are sorted by frame: pf > 0 */
    }
    if (pf_ok && tid * 32 < nb)
        asm volatile("prefetch.global.L2 [%0];" :: "l"(my_ent + (size_t)pf * (unsigned)P.nblk + tid * 32));

    /* everything that does not depend on anything else is fetched first: the first round's entry
     * and the frame descriptor; the table constants follow the descriptor */
    PicPos pp_next = pos_of(tid);
    uint32_t e_first = tid < nb ? my_ent[pp_next.i] : 0u;
    const rtjgpu_frame_desc fd = P.desc[f];
    const unsigned mytable = min((unsigned)fd.table, (unsigned)RTJ_NUM_TABLES - 1u);     /* descriptors are the caller's memory */
    const rtj_dev_table *tb = &P.tables[mytable];
    const uint8_t *frame_pay = P.stream + fd.offset + RTJPEG_B200_HEADER_BYTES;
    const int bt8_l = tb->bt8[0], bt8_c = tb->bt8[1];
    /* T2 needs three multipliers per plane type: registers */
    const int lq0 = tb->iq[0][0], lq1 = tb->iq[0][1], lq2 = tb->iq[0][2];
    const int cq0 = tb->iq[1][0], cq1 = tb->iq[1][1], cq2 = tb->iq[1][2];

    /* ---- pass 1, picture order: T2 blocks decode right away, the rest is queued ---- */
    int nfront = 0, nback = 0;                               /* warp-uniform queue fill: M7 | CARRY, HARD */
    bool saw_skip = false;
    for (int r = 0; r < rounds; r++) {
        const int p = r * THREADS + tid;
        const PicPos pp = pp_next;
        const bool chroma = off_is_chroma<FMT>(pp.off, mbs);
        uint32_t e = e_first;
        if (r + 1 < rounds) {                                /* next round's entry: in flight during this round */
            pp_next = pos_of(p + THREADS);
            e_first = p + THREADS < nb ? my_ent[pp_next.i] : 0u;
        }
        int cls = CLS_NONE;
        int x0 = 0, x1 = 0, q = 0;
        bool safe = true;
        unsigned sf = f;
        /* working through a run: a block this frame skips (its marker, or K3's copy of an inline last writer: both carry
         * bits 31 and 30) whose pixels the strip still holds from the frame before is left alone */
        const bool keep = runs && f != f_first && ((valid >> r) & 1u) && (e & 0xC0000000u) == 0xC0000000u;
        if (p < nb && !keep) {
            if (RTJ_ENT_IS_SKIP(e)) {                        /* skipped: take the entry of its last writer */
                saw_skip = true;
                const unsigned s = P.srcf[frame_blk0 + pp.i];
                if (s != RTJ_SRC_CARRY) {
                    sf = s;
                    e = P.ent[s * (unsigned)P.nblk + strip_blk0 + pp.i];
                }
            }
            if (RTJ_ENT_IS_SKIP(e)) cls = Q_CARRY;
            else if (sf != f && P.desc[sf].table != mytable) cls = Q_HARD;
            else if (RTJ_ENT_IS_INLINE(e)) {
                cls = CLS_T2;
                x0 = wrap16((int)(e & 0xFFu) * (chroma ? cq0 : lq0)) + 4;
                x1 = wrap16((int)(signed char)((e >> 8) & 0xFFu) * (chroma ? cq1 : lq1));
                q = wrap16((int)(signed char)((e >> 16) & 0xFFu) * (chroma ? cq2 : lq2));
            } else {
                const int eob = RTJ_ENT_EOB(e);
                if (eob <= 3) {
                    cls = CLS_T2;
                    const uint8_t *src = (sf == f ? frame_pay : P.stream + P.desc[sf].offset + RTJPEG_B200_HEADER_BYTES)
                                         + (e & RTJ_ENT_OFF_MASK);
                    RegBytes<1> by(src);
                    int x[3];
                    unpack_block<3>(by, tb->iq[chroma], chroma ? bt8_c : bt8_l, x);
                    x0 = x[0]; x1 = x[1]; q = x[2];
                } else if (eob <= 7) cls = Q_M7;
                else cls = Q_HARD;
            }
            if (cls == CLS_T2) safe = t2_safe(x0, x1, q);
        }
        /* what is decoded or copied into the strip leaves it valid; a HARD block's pixels only reach the frame in device memory */
        if (runs && !keep) valid = (valid & ~(1u << r)) | ((cls != CLS_NONE && (RGB || cls != Q_HARD)) ? 1u << r : 0u);
        const bool packed = __all_sync(FULL, safe);          /* one epilogue flavour per warp */
        if (cls == CLS_T2) {
            uint32_t px[16];
            t2_pixels(x0, x1, q, packed, px);
            store_block<FMT>(tile_s, pp.off, mbs, px);
        }
        const unsigned mM = __ballot_sync(FULL, cls == Q_M7);
        const unsigned mB = __ballot_sync(FULL, cls == Q_CARRY || cls == Q_HARD);
        const unsigned below = (1u << lane) - 1u;
        if (cls == Q_M7) {
            const int at = nfront + __popc(mM & below);
            wq_e[at] = e;
            wq_p[at] = (uint32_t)pp.off | (sf << 16);
        } else if (cls == Q_CARRY || cls == Q_HARD) {
            const int at = wq - 1 - (nback + __popc(mB & below));
            /* HARD blocks split once more for the general kernel: long ones (E > 16) apart from the rest */
            const bool full = cls == Q_HARD && !RTJ_ENT_IS_INLINE(e) && RTJ_ENT_EOB(e) > 16;
            wq_e[at] = (uint32_t)pp.i | (cls == Q_CARRY ? 0x80000000u : 0u) | (full ? 0x40000000u : 0u);
            wq_p[at] = (uint32_t)pp.off | (sf << 16);
        }
        nfront += __popc(mM);
        nback += __popc(mB);
    }
    /* ... where this row held skipped blocks, the last writers of that frame's row (two bytes a block) ... */
    if (pf_ok && __any_sync(FULL, saw_skip) && lane * 64 < nb && warp == 0)
        asm volatile("prefetch.global.L2 [%0];" :: "l"(P.srcf + frame_blk0 + (size_t)pf * (unsigned)P.nblk + lane * 64));
    /* ... and the part of that frame's payload where its blocks of this row should lie, if the payload is spread
     * evenly over the rows: the M7 blocks read it */
    if (pf_ok && warp == WARPS - 1 && lane < K2_PF_LINES) {
        const rtjgpu_frame_desc nd = P.desc[f + pf];
        const unsigned rows_total = (unsigned)P.rows;
        const unsigned plen = nd.length > RTJPEG_B200_HEADER_BYTES ? nd.length - RTJPEG_B200_HEADER_BYTES : 0u;
        const unsigned at = (unsigned)(((unsigned long long)plen * (unsigned)my) / rows_total);
        const unsigned o = (at & ~127u) + (unsigned)lane * 128u;
        if (o < plen) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.stream + nd.offset + RTJPEG_B200_HEADER_BYTES + o));
    }
    /* ---- pass 2: the M7 blocks of all four warps pooled, 32 at a time (a macroblock row of typical
     *      material holds ~55 of them: two full passes of the flow graph instead of four part-filled
     *      ones).  The queues stay where the warps wrote them; an index is mapped to (warp, slot)
     *      through the four counts. ---- */
    if (lane == 0) s_hard[4 + warp] = nfront;
    __syncthreads();
    const int n0 = s_hard[4], n1 = n0 + s_hard[5], n2 = n1 + s_hard[6], nM = n2 + s_hard[7];
    const uint32_t *q_e = reinterpret_cast<const uint32_t *>(s_hard + 8);
    const uint32_t *q_p = q_e + K2_WARPS * wq;
    /* the last warps start first: warp 0 is the one with a part-filled extra round behind it */
    for (int c0 = (WARPS - 1 - warp) * 32; c0 < nM; c0 += WARPS * 32) {
        const int idx = c0 + lane;
        int x[7] = {1008, 0, 0, 0, 0, 0, 0};
        const bool live = idx < nM;
        int off = 0;
        if (live) {
            const int qw = (idx >= n0) + (idx >= n1) + (idx >= n2);
            const int at = qw * wq + idx - (qw == 0 ? 0 : qw == 1 ? n0 : qw == 2 ? n1 : n2);
            const uint32_t e = q_e[at];
            const uint32_t ps = q_p[at];
            const unsigned sf = ps >> 16;
            off = (int)(ps & 0xFFFFu);
            const bool chroma = off_is_chroma<FMT>(off, mbs);
            const uint8_t *src = (sf == f ? frame_pay : P.stream + P.desc[sf].offset + RTJPEG_B200_HEADER_BYTES)
                                 + (e & RTJ_ENT_OFF_MASK);
            RegBytes<2> by(src);
            unpack_block<7>(by, tb->iq[chroma], chroma ? bt8_c : bt8_l, x);
        }
        const bool packed = __all_sync(FULL, m7_safe(x));
        if (live) {
            uint32_t px[16];
            m7_pixels(x, packed, px);
            store_block<FMT>(tile_s, off, mbs, px);
        }
    }
    /* ---- CARRY blocks are copied from the picture before the batch, HARD blocks leave for
     *      rtj_idct_hard_kernel through the device queue ---- */
    int nhard = 0;
    if (nback) {                                             /* warp-uniform */
        /* The warp's places in the device queue, both ends: ONE request per warp and row -- an atomic on a word every CTA of
         * the grid adds to, a trip to L2 and back -- instead of one per 32 blocks: above a quality of 170 every luma block
         * goes this way, eight requests one behind the other.  The counts come from the warp's own queue. */
        unsigned qbase16 = 0, qbaseF = 0;
        /* (a template parameter: as a run-time choice the code costs the kernel 0.65 % on streams that never use it) */
        const bool reserve = RES && !RGB && nback > 32;      /* (a single pass asks for itself, as ever) */
        if (reserve) {
            int nq16 = 0, nqF = 0;
            for (int c0 = 0; c0 < nback; c0 += 32) {
                const uint32_t ie = c0 + lane < nback ? wq_e[wq - 1 - (c0 + lane)] : 0x80000000u;
                const unsigned mH = __ballot_sync(FULL, !(ie >> 31)), mF = __ballot_sync(FULL, (ie >> 30) == 1u);
                nq16 += __popc(mH & ~mF);
                nqF += __popc(mF);
            }
            if (lane == 0) {
                if (nq16) qbase16 = atomicAdd(&P.info->hard_blocks, (unsigned)nq16);
                if (nqF) qbaseF = atomicAdd(&P.info->hard_full, (unsigned)nqF);
            }
            qbase16 = __shfl_sync(FULL, qbase16, 0);
            qbaseF = __shfl_sync(FULL, qbaseF, 0);
        }
        for (int c0 = 0; c0 < nback; c0 += 32) {
            const int idx = c0 + lane;
            const bool live = idx < nback;
            uint32_t ie = 0x80000000u;
            int off = 0;
            unsigned hsf = f;                                    /* the frame whose stream holds a HARD block: its last writer */
            if (live) { ie = wq_e[wq - 1 - idx]; const uint32_t ps = wq_p[wq - 1 - idx]; off = (int)(ps & 0xFFFFu); hsf = ps >> 16; }
            const bool hard = live && !(ie >> 31);
            const bool full = hard && ((ie >> 30) & 1u);
            const int bi = (int)(ie & 0x3FFFFFFFu);              /* stream-order index inside the strip */
            if (GENERAL) {
                /* no planes for rtj_idct_hard_kernel to patch (packed pixels, or a window's): the general decoder runs here,
                 * out of line */
                if (hard) {
                    uint32_t px[16];
                    decode_general_call(P.stream, P.desc, P.tables, P.ent, P.srcf, P.nblk, frame_blk0 + (unsigned)bi,
                                        off_is_chroma<FMT>(off, mbs) ? 1 : 0, full ? 1 : 0, px);
                    store_block<FMT>(tile_s, off, mbs, px);
                }
            }
            const unsigned mH = GENERAL ? 0u : __ballot_sync(FULL, hard && !full), mF = GENERAL ? 0u : __ballot_sync(FULL, full);
            if (mH | mF) {
                /* the device queue is filled from both ends: mid-size blocks from the front, long ones from the back */
                unsigned base = qbase16, baseF = qbaseF;
                if (reserve) {
                    qbase16 += (unsigned)__popc(mH);
                    qbaseF += (unsigned)__popc(mF);
                } else {
                    if (lane == 0) {
                        if (mH) base = atomicAdd(&P.info->hard_blocks, (unsigned)__popc(mH));
                        if (mF) baseF = atomicAdd(&P.info->hard_full, (unsigned)__popc(mF));
                    }
                    base = __shfl_sync(FULL, base, 0);
                    baseF = __shfl_sync(FULL, baseF, 0);
                }
                const unsigned below = (1u << lane) - 1u;
                /* a queue entry: the block's place in its frame (and whether it is a chroma block), the frame the pixels
                 * go to and the frame whose stream holds the block (its last writer) */
                const uint2 rec = make_uint2((strip_blk0 + (unsigned)bi) | (off_is_chroma<FMT>(off, mbs) ? 0x80000000u : 0u),
                                             (SEL ? RTJ_JOB_SLOT(job) : f) | (hsf << 16));
                if (hard && !full) reinterpret_cast<uint2 *>(P.hardq)[base + __popc(mH & below)] = rec;
                if (full) reinterpret_cast<uint2 *>(P.hardq)[P.hardq_cap - 1u - (baseF + __popc(mF & below))] = rec;
                /* (the luma blocks among them in the upper half: a strip whose luma blocks are all HARD keeps its luma rows) */
                const unsigned mC = __ballot_sync(FULL, off_is_chroma<FMT>(off, mbs));
                nhard += __popc(mH) + __popc(mF) + (__popc((mH | mF) & ~mC) << 16);
            }
            if (live && !hard) {
                uint32_t px[16];
                const uint8_t *carry = P.seq ? P.carries[RTJ_SEQ_INDEX(P.seq[f])] : P.carry;    /* the picture before f's sequence */
                if (carry) {
                    int pitch;
                    const uint8_t *cp = G::carry_src(carry, bi, my, mx0, w, h, pitch);
#pragma unroll
                    for (int r = 0; r < 8; r++) {
                        const uint2 v = *reinterpret_cast<const uint2 *>(cp + (size_t)r * pitch);
                        px[2 * r] = v.x;
                        px[2 * r + 1] = v.y;
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < 16; r++) px[r] = 0;
                }
                store_block<FMT>(tile_s, off, mbs, px);
            }
        }
    }
    if (lane == 0) s_hard[warp] = nhard;

    /* ---- the strip leaves the SM (a strip made of HARD blocks only has nothing to say) ---- */
    if (SINGLE) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    const int lw = G::UNIT_W * mbs;                              /* luma bytes per strip row */
    bool planes_leave = true, luma_leaves = true;
    uint8_t *last_planes = P.last_yuv;                          /* RGB: where the frame leaves as planes too, if it does */
    if (CHW) {
        /* The window's pixels as the RGB branch below makes them (RGB24 / BGR24), planar: a thread takes 8 pixels of two rows,
         * and stores each row's three channels, 8 elements each (8-, 16- or 2 x 16-byte stores, contiguous across the warp).
         * Mirrored, a chunk's bytes are reversed before they are converted and the chunk goes to the mirrored column. */
        using namespace rtjcv;
        const int chunks = lw >> 3;
        const uint8_t *tU = tile + G::CHROMA_AT * mbs, *tV = tU + 64 * mbs;
        const int top = my * 16 - wy;
        const int rp0 = max(0, -top) >> 1, rp1 = min(16, P.win_h - top) >> 1;
        const bool mirror = (worg & RTJ_WIN_MIRROR) != 0u;
        const int dtype = P.chw_dtype;
        const int es = dtype == RTJ_CHW_U8 ? 1 : dtype == RTJ_CHW_F32 ? 4 : 2;
        const size_t rowp = P.rgb_row_pitch, planep = rowp * (size_t)P.win_h;
        const int cr = P.rgb_kind == RTJ_CONV_BGR24 ? 2 : 0;        /* the channel red goes to; blue to the other end */
        uint8_t *const base = P.rgb + (size_t)RTJ_JOB_SLOT(job) * P.rgb_frame_pitch;
        uint8_t *const pr = base + cr * planep, *const pg = base + planep, *const pb = base + (2 - cr) * planep;
        const float sr = P.chw_scale[cr], sg = P.chw_scale[1], sb = P.chw_scale[2 - cr];
        const float br = P.chw_bias[cr], bg = P.chw_bias[1], bb = P.chw_bias[2 - cr];
        const int items = (rp1 - rp0) * chunks;
        for (int item = tid; item < items; item += THREADS) {
            const int rp = rp0 + item / chunks, c = item - (rp - rp0) * chunks;
            const uint2 y0 = *reinterpret_cast<const uint2 *>(tile + (2 * rp) * lw + c * 8);
            const uint2 y1 = *reinterpret_cast<const uint2 *>(tile + (2 * rp + 1) * lw + c * 8);
            const uint32_t ub = *reinterpret_cast<const uint32_t *>(tU + rp * (lw >> 1) + c * 4);
            const uint32_t vb = *reinterpret_cast<const uint32_t *>(tV + rp * (lw >> 1) + c * 4);
            Chroma ct[4];
#pragma unroll
            for (int k = 0; k < 4; k++) ct[k] = chroma_terms((ub >> (8 * k)) & 0xFFu, (vb >> (8 * k)) & 0xFFu);
            const int x = (mx0 - wx) * 16 + c * 8;                  /* the chunk's first column in the window */
            const size_t col = (size_t)(mirror ? P.win_w - 8 - x : x) * es;
#pragma unroll
            for (int k = 0; k < 2; k++) {
                Rgb8 v = rgb8(k ? y1 : y0, ct);
                if (mirror) { v.r = reverse8(v.r); v.g = reverse8(v.g); v.b = reverse8(v.b); }
                const size_t off = (size_t)(top + 2 * rp + k) * rowp + col;   /* strip row 2 rp + k is window row top + 2 rp + k */
                chw8(dtype, v.r, sr, br, pr + off);
                chw8(dtype, v.g, sg, bg, pg + off);
                chw8(dtype, v.b, sb, bb, pb + off);
            }
        }
        planes_leave = false;                                   /* the last frames have a launch of their own */
    } else if (RGB) {
        /* The strip -- 16 luma rows, 8 rows of Cb and of Cr: exactly what the reference's converters read for 16 output
         * rows (lib/RTjpeg.c:3123-3190) -- leaves as packed pixels.  A thread takes 8 pixels of two rows (one chroma row):
         * aligned 8- / 4-byte shared loads, 16- / 8-byte global stores, contiguous across the warp. */
        using namespace rtjcv;
        const int chunks = lw >> 3;
        const uint8_t *tU = tile + G::CHROMA_AT * mbs, *tV = tU + 64 * mbs;
        const int kind = RGBK == RGB_ANY ? P.rgb_kind : RGBK;
        const int bpp = (kind == RTJ_CONV_RGB32 || kind == RTJ_CONV_BGR32) ? 4 : kind == RTJ_CONV_RGB16 ? 2 : 3;
        /* WIN: strip row r is window row top + r; the row pairs inside the window are [rp0, rp1) (top, wy and win_h are even) */
        const int top = my * 16 - wy;
        const int rp0 = WIN ? max(0, -top) >> 1 : 0, rp1 = WIN ? min(16, P.win_h - top) >> 1 : 8;
        uint8_t *base = WIN ? P.rgb + (size_t)RTJ_JOB_SLOT(job) * P.rgb_frame_pitch + (size_t)((mx0 - wx) * 16) * bpp
                            : P.rgb + (size_t)(SEL ? RTJ_JOB_SLOT(job) : f) * P.rgb_frame_pitch + (size_t)(my * 16) * P.rgb_row_pitch
                              + (size_t)(mx0 * 16) * bpp;
        const int items = SEL && RTJ_JOB_SLOT(job) == RTJ_JOB_NO_SLOT ? 0 : (rp1 - rp0) * chunks;    /* SEL: planes for last_yuv only */
        for (int item = tid; item < items; item += THREADS) {
            const int rp = rp0 + item / chunks, c = item - (rp - rp0) * chunks;
            const uint2 y0 = *reinterpret_cast<const uint2 *>(tile + (2 * rp) * lw + c * 8);
            const uint2 y1 = *reinterpret_cast<const uint2 *>(tile + (2 * rp + 1) * lw + c * 8);
            const uint32_t ub = *reinterpret_cast<const uint32_t *>(tU + rp * (lw >> 1) + c * 4);
            const uint32_t vb = *reinterpret_cast<const uint32_t *>(tV + rp * (lw >> 1) + c * 4);
            Chroma ct[4];
#pragma unroll
            for (int k = 0; k < 4; k++) ct[k] = chroma_terms((ub >> (8 * k)) & 0xFFu, (vb >> (8 * k)) & 0xFFu);
            uint8_t *o = base + (size_t)((WIN ? top : 0) + 2 * rp) * P.rgb_row_pitch + (size_t)c * (8 * bpp);
            switch (kind) {
            case RTJ_CONV_RGB32: row8<RTJ_CONV_RGB32>(y0, ct, P.rgb_alpha, o); row8<RTJ_CONV_RGB32>(y1, ct, P.rgb_alpha, o + P.rgb_row_pitch); break;
            case RTJ_CONV_BGR32: row8<RTJ_CONV_BGR32>(y0, ct, P.rgb_alpha, o); row8<RTJ_CONV_BGR32>(y1, ct, P.rgb_alpha, o + P.rgb_row_pitch); break;
            case RTJ_CONV_RGB24: row8<RTJ_CONV_RGB24>(y0, ct, P.rgb_alpha, o); row8<RTJ_CONV_RGB24>(y1, ct, P.rgb_alpha, o + P.rgb_row_pitch); break;
            case RTJ_CONV_BGR24: row8<RTJ_CONV_BGR24>(y0, ct, P.rgb_alpha, o); row8<RTJ_CONV_BGR24>(y1, ct, P.rgb_alpha, o + P.rgb_row_pitch); break;
            default:             row8<RTJ_CONV_RGB16>(y0, ct, P.rgb_alpha, o); row8<RTJ_CONV_RGB16>(y1, ct, P.rgb_alpha, o + P.rgb_row_pitch); break;
            }
        }
        /* the last frame also leaves as planes: the next batch's carry -- with several sequences, the last frame of each
         * (WIN: the strips cover the window only; the last frames have a launch of their own) */
        if (WIN) last_planes = nullptr;
        else if (P.seq) {
            const unsigned nx = f + 1u;
            last_planes = nx == (unsigned)P.F || RTJ_SEQ_FIRST(P.seq[nx]) == nx ? P.last_yuvs[RTJ_SEQ_INDEX(P.seq[f])] : nullptr;
        } else if (f + 1u != (unsigned)P.F) last_planes = nullptr;
        if (!last_planes) planes_leave = false;
    } else if (WIN) {
        /* The window's planes, tight at the window's pitch: the strip's rows inside the window, in the strip path's vector
         * widths.  Strip luma row r is window row top + r, strip chroma row r window chroma row ctop + r. */
        const int ww = P.win_w, wh = P.win_h, wcw = ww >> 1;
        constexpr int VS = FMT == 0 ? 2 : 1;                     /* vertical chroma subsampling */
        uint8_t *const planes = P.win_last ? P.last_yuvs[RTJ_SEQ_INDEX(P.seq[f])]
                                           : P.out + (size_t)RTJ_JOB_SLOT(job) * RTJ_FMT_FRAME_BYTES(FMT, ww, wh);
        const int top = my * G::LUMA_ROWS - wy, ctop = my * 8 - wy / VS;
        const int r0 = max(0, -top), r1 = min(G::LUMA_ROWS, wh - top);
        const int c0 = max(0, -ctop), c1 = min(8, wh / VS - ctop);
        uint8_t *oy = planes + (mx0 - wx) * G::UNIT_W;
        uint8_t *ou = planes + (size_t)ww * wh + (mx0 - wx) * 8;
        uint8_t *ov = ou + (size_t)wcw * (wh / VS);
        const uint8_t *tileU = tile + G::CHROMA_AT * mbs, *tileV = tileU + 64 * mbs;
        for (int r = r0 + warp; r < r1; r += WARPS) {
            if (G::UNIT_W == 16) {
                for (int c = lane; c < mbs; c += 32)
                    *reinterpret_cast<uint4 *>(oy + (size_t)(top + r) * ww + c * 16) = *reinterpret_cast<const uint4 *>(tile + r * lw + c * 16);
            } else {
                for (int c = lane; c < mbs; c += 32)
                    *reinterpret_cast<uint2 *>(oy + (size_t)(top + r) * ww + c * 8) = *reinterpret_cast<const uint2 *>(tile + r * lw + c * 8);
            }
        }
        if (G::PLANES == 3) {
            const int segC = lw >> 1;
            for (int r = warp; r < 16; r += WARPS) {
                const int pl = r >> 3, rr = r & 7;
                if (rr < c0 || rr >= c1) continue;
                for (int c = lane; c < (segC >> 3); c += 32)
                    *reinterpret_cast<uint2 *>((pl ? ov : ou) + (size_t)(ctop + rr) * wcw + c * 8) =
                        *reinterpret_cast<const uint2 *>((pl ? tileV : tileU) + rr * segC + c * 8);
            }
        }
        planes_leave = false;
    } else {
        /* What rtj_idct_hard*_kernel patch need not be written here first.  All blocks HARD: nothing leaves; all luma blocks
         * (a quality above 170, where every luma block carries ten coefficients or more): the chroma rows only. */
        const int hs = s_hard[0] + s_hard[1] + s_hard[2] + s_hard[3];
        if ((hs & 0xFFFF) == nb) planes_leave = false;
        else if (G::PLANES == 3 && (hs >> 16) == nb - 2 * mbs) luma_leaves = false;
    }
    if (planes_leave) {
    const size_t fsz = RTJ_FMT_FRAME_BYTES(FMT, w, h);
    const int cw = w >> 1;
    uint8_t *const planes = RGB ? last_planes : P.out + (size_t)(SEL ? RTJ_JOB_SLOT(job) : f) * fsz;
    uint8_t *oy = planes + (size_t)(my * G::LUMA_ROWS) * w + mx0 * G::UNIT_W;
    uint8_t *ou = planes + (size_t)w * h + (size_t)(my * 8) * cw + mx0 * 8;
    uint8_t *ov = ou + (FMT == 0 ? (size_t)cw * (h >> 1) : (size_t)cw * h);
    const uint8_t *tileU = tile + G::CHROMA_AT * mbs, *tileV = tileU + 64 * mbs;
    if (SINGLE) {
        /* the luma rows and the 2 x 8 chroma rows are each one contiguous run in the tight-pitch planes:
         * TMA bulk stores issued by one thread */
        if (tid == 0) {
            if (luma_leaves) bulk_store(oy, tile, (unsigned)(G::LUMA_ROWS * lw));
            if (G::PLANES == 3) {
                bulk_store(ou, tileU, 64u * (unsigned)mbs);
                bulk_store(ov, tileV, 64u * (unsigned)mbs);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
    } else {
        if (!luma_leaves) {
        } else if (G::UNIT_W == 16) {
            for (int r = warp; r < G::LUMA_ROWS; r += WARPS)
                for (int c = lane; c < mbs; c += 32)                 /* 16-byte vectors per luma row */
                    *reinterpret_cast<uint4 *>(oy + (size_t)r * w + c * 16) =
                        *reinterpret_cast<const uint4 *>(tile + r * lw + c * 16);
        } else {
            for (int r = warp; r < G::LUMA_ROWS; r += WARPS)
                for (int c = lane; c < mbs; c += 32)                 /* 8-byte vectors: a grey strip may be an odd number of blocks */
                    *reinterpret_cast<uint2 *>(oy + (size_t)r * w + c * 8) =
                        *reinterpret_cast<const uint2 *>(tile + r * lw + c * 8);
        }
        if (G::PLANES == 3) {
            const int segC = lw >> 1;
            for (int r = warp; r < 16; r += WARPS) {
                const int pl = r >> 3, rr = r & 7;
                for (int c = lane; c < (segC >> 3); c += 32)     /* 8-byte vectors per chroma row */
                    *reinterpret_cast<uint2 *>((pl ? ov : ou) + (size_t)rr * cw + c * 8) =
                        *reinterpret_cast<const uint2 *>((pl ? tileV : tileU) + rr * segC + c * 8);
            }
        }
    }
    }
    /* the run's next frame writes into the strip: everybody is done reading it (thread 0 has waited for its bulk stores) */
    if (runs) __syncthreads();
    }
}

template <int FMT>
__global__ void rtj_build_lut_kernel(uint32_t *__restrict__ pos, int mbs, int npad)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npad) return;
    const PicPos r = Geo<FMT>::pic_pos(min(p, mbs * Geo<FMT>::BLK - 1), mbs);       /* the padding repeats the last position */
    pos[p] = (uint32_t)r.i | (uint32_t)r.off << 16;
}

/* ------------------------------------------------------------------------ */
/* K2b: the general decoder for queued blocks                                  */
/* ------------------------------------------------------------------------ */

/*
 * The queue holds blocks of at most 16 coefficients (and blocks carried inline whose last writer used other tables) at its
 * front, longer blocks at its back; an entry names the block's place in its frame, the frame its pixels go to and the
 * frame whose stream holds it.
 *
 * rtj_idct_hard16_kernel: the front.  One thread per block: the first 16 zig-zag positions touch rows 0..5 and columns 0..4
 * only and fit 24 bytes held in registers.
 */
extern "C" __global__ void __launch_bounds__(128)
rtj_idct_hard16_kernel(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                       const rtj_dev_table *__restrict__ tables, const uint32_t *__restrict__ ent,
                       int nblk, int w, int h, int fmt, uint8_t *__restrict__ out, const uint32_t *__restrict__ hardq,
                       const rtj_dev_info *__restrict__ info)
{
    /* resident before K2 is done (launch_pdl): its queue is final after the wait.  rtj_idct_hard_kernel, launched behind this
     * kernel, takes the other end of the queue: from here on it may start alongside. */
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const unsigned n16 = info->hard_blocks;
    const size_t fsz = RTJ_FMT_FRAME_BYTES(fmt, w, h);
    const unsigned stride = gridDim.x * blockDim.x;
    const unsigned k0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (k0 >= n16) return;
    /* A block is three reads deep -- the queue's record, the entry and descriptor it names, the bytes those point at -- and
     * a thread works through some forty blocks: with the reads of one block made only when the block before is stored, the
     * warps spent half their time waiting (long scoreboard on each of the three).  Three stages, three blocks under way:
     * while block j is unpacked and transformed, the bytes of j + 1, the entry of j + 2 and the record of j + 3 are on their
     * way.  (Records past the queue's end repeat its last one: read, never used.) */
    struct Src {
        uint32_t e;
        uint32_t table;
        const uint8_t *bytes;
    };
    const uint2 *Q = reinterpret_cast<const uint2 *>(hardq);
    auto ld_rec = [&](unsigned k) { return Q[min(k, n16 - 1u)]; };
    auto ld_src = [&](const uint2 rec) {
        const unsigned sf = rec.y >> 16;
        Src r;
        r.e = ent[(size_t)sf * nblk + (rec.x & 0x7FFFFFFFu)];
        const rtjgpu_frame_desc sd = desc[sf];
        r.table = sd.table;
        r.bytes = stream + sd.offset + RTJPEG_B200_HEADER_BYTES;
        return r;
    };
    /* (an inline entry holds no offset: its bytes are not used, any address inside the packet will do) */
    auto ld_bytes = [&](const Src &sr) { return RegBytes<6>(sr.bytes + (RTJ_ENT_IS_INLINE(sr.e) ? 0u : (sr.e & RTJ_ENT_OFF_MASK))); };
    uint2 rec0 = ld_rec(k0), rec1 = ld_rec(k0 + stride), rec2 = ld_rec(k0 + 2u * stride);
    Src sr0 = ld_src(rec0), sr1 = ld_src(rec1);
    RegBytes<6> by = ld_bytes(sr0);
    for (unsigned k = k0; k < n16; k += stride) {
        const RegBytes<6> by1 = ld_bytes(sr1);
        const Src sr2 = ld_src(rec2);
        const uint2 rec3 = ld_rec(k + 3u * stride);

        const int i = (int)(rec0.x & 0x7FFFFFFFu), chroma = (int)(rec0.x >> 31);
        const unsigned f = rec0.y & 0xFFFFu;
        const uint32_t e = sr0.e;
        const rtj_dev_table *t = &tables[min((int)sr0.table, RTJ_NUM_TABLES - 1)];
        uint32_t px[16];
        if (RTJ_ENT_IS_INLINE(e)) {
            const int x0 = wrap16((int)(e & 0xFFu) * t->iq[chroma][0]) + 4;
            const int x1 = wrap16((int)(signed char)((e >> 8) & 0xFFu) * t->iq[chroma][1]);
            const int q = wrap16((int)(signed char)((e >> 16) & 0xFFu) * t->iq[chroma][2]);
            t2_pixels(x0, x1, q, false, px);
        } else {
            int x[16];
            const int bt8 = t->bt8[chroma];
            if (bt8 == 9) unpack_block16_prefix<9>(by, t->iq[chroma], x);            /* the prefixes of the quality tables */
            else if (bt8 == 8) unpack_block16_prefix<8>(by, t->iq[chroma], x);
            else if (bt8 == 4) unpack_block16_prefix<4>(by, t->iq[chroma], x);
            else unpack_block<16>(by, t->iq[chroma], bt8, x);
            idct_general<16>(x, px);
        }
        int pitch;
        uint8_t *dst = block_dst(out + (size_t)f * fsz, fmt, i, w, h, pitch);
#pragma unroll
        for (int r = 0; r < 8; r++)
            *reinterpret_cast<uint2 *>(dst + (size_t)r * pitch) = make_uint2(px[2 * r], px[2 * r + 1]);
        rec0 = rec1; rec1 = rec2; rec2 = rec3;
        sr0 = sr1; sr1 = sr2;
        by = by1;
    }
}

/*
 * rtj_idct_hard_kernel: the back -- long blocks.  EIGHT LANES per block, four blocks per warp.  (One thread per block, 110
 * registers, the block's bytes fetched one by one in a dependent chain, kept 16 warps per SM waiting for memory: 43 % of
 * the issue slots used on a dense 1920x1088 stream.)  The block's up to 64 bytes arrive as one coalesced read, eight bytes
 * a lane.  Every byte's place in the zig-zag order is a prefix sum of what the bytes before it fill (lib/RTjpeg.c:162-183:
 * DC and the raw prefix one place each, a run token b - 63, any other token one), made within the lane and scanned over
 * the eight lanes; the dequantised coefficients are scattered into an 8x8 matrix in shared memory.  First pass
 * (:2221-2285): one COLUMN per lane; second pass (:2287-2330): one ROW per lane, after a transposition through shared
 * memory; every lane stores its row's eight pixels.
 */
__constant__ uint8_t c_zz_raster[64] = {
#define RTJ_RASTER(k, r, c) (r) * 8 + (c),
    RTJ_ZZ_LIST(RTJ_RASTER)
#undef RTJ_RASTER
};

constexpr int HB_THREADS = 128;

extern "C" __global__ void __launch_bounds__(HB_THREADS)
rtj_idct_hard_kernel(const uint8_t *__restrict__ stream, const rtjgpu_frame_desc *__restrict__ desc,
                     const rtj_dev_table *__restrict__ tables, const uint32_t *__restrict__ ent,
                     int nblk, int w, int h, int fmt,
                     uint8_t *__restrict__ out, const uint32_t *__restrict__ hardq, unsigned hardq_cap,
                     const rtj_dev_info *__restrict__ info)
{
    __shared__ __align__(16) int16_t s_m[HB_THREADS / 8][72];        /* coefficients, raster order; 36 words a block: the four blocks of a warp on different banks */
    __shared__ int32_t s_w[HB_THREADS / 8][8][9];                     /* first-pass results, rows padded to nine words */
    __shared__ uint8_t s_zz[64];                                      /* zig-zag place -> raster place (indexed per lane: not for the constant cache) */
    if (threadIdx.x < 64) s_zz[threadIdx.x] = c_zz_raster[threadIdx.x];
    __syncthreads();
    const unsigned total = info->hard_full;
    const size_t fsz = RTJ_FMT_FRAME_BYTES(fmt, w, h);
    const int lane = threadIdx.x & 31, l = lane & 7, grp = threadIdx.x >> 3;
    int16_t *M = s_m[grp];
    const int16_t *Mc = M + l;                                        /* this lane's column */
    int32_t *Wc = &s_w[grp][0][l];                                    /* ... of the first pass's results: row r at Wc[9 r] */
    const int32_t *Wr = &s_w[grp][l][0];                              /* this lane's row */
    const unsigned stride = gridDim.x * (HB_THREADS / 8);
    /* As in rtj_idct_hard16_kernel a block is three reads deep (queue record; entry and descriptor; bytes), and a warp works
     * through some twenty groups of four blocks: three groups under way, one stage apart, so that the reads of a group are
     * made while the two groups in front of it are transformed.  (Lanes past the queue's end read block 0 of frame 0.) */
    struct Src {
        uint32_t e, table;
        const uint32_t *wp;          /* the lane's three words */
        unsigned sh;
    };
    auto ld_rec = [&](unsigned kb) {
        const unsigned k = kb + (unsigned)(lane >> 3);
        return k < total ? reinterpret_cast<const uint2 *>(hardq)[hardq_cap - 1u - k] : make_uint2(0u, 0u);
    };
    auto ld_src = [&](unsigned kb, const uint2 rec) {
        const unsigned k = kb + (unsigned)(lane >> 3);
        const unsigned sf = rec.y >> 16;
        Src r;
        r.e = k < total ? ent[(size_t)sf * nblk + (rec.x & 0x7FFFFFFFu)] : 0u;
        const rtjgpu_frame_desc sd = desc[sf];
        r.table = sd.table;
        const uintptr_t a = reinterpret_cast<uintptr_t>(stream + sd.offset + RTJPEG_B200_HEADER_BYTES);
        r.wp = reinterpret_cast<const uint32_t *>(a);      /* packets start on a multiple of 4; the block's offset is added when the entry is there */
        r.sh = 0;
        return r;
    };
    struct Words {
        uint32_t w0, w1, w2;
        unsigned sh;
    };
    auto ld_words = [&](const Src &sr) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(sr.wp) + (sr.e & RTJ_ENT_OFF_MASK);
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3) + 2 * l;
        Words w;
        w.w0 = __ldg(wp); w.w1 = __ldg(wp + 1); w.w2 = __ldg(wp + 2);                    /* slack bytes follow the stream */
        w.sh = (unsigned)(a & 3) * 8;
        return w;
    };
    const unsigned kb0 = (blockIdx.x * (HB_THREADS / 32) + (threadIdx.x >> 5)) * 4;
    if (kb0 >= total) return;                                                           /* warp-uniform */
    uint2 rec0 = ld_rec(kb0), rec1 = ld_rec(kb0 + stride), rec2 = ld_rec(kb0 + 2u * stride);
    Src sr0 = ld_src(kb0, rec0), sr1 = ld_src(kb0 + stride, rec1);
    Words wd = ld_words(sr0);
    for (unsigned kb = kb0; kb < total; kb += stride) {       /* warp-uniform */
        const Words wd1 = ld_words(sr1);
        const Src sr2 = ld_src(kb + 2u * stride, rec2);
        const uint2 rec3 = ld_rec(kb + 3u * stride);

        const unsigned k = kb + (unsigned)(lane >> 3);
        const bool live = k < total;
        const uint2 rec = rec0;
        const int i = (int)(rec.x & 0x7FFFFFFFu), chroma = (int)(rec.x >> 31);
        const unsigned f = rec.y & 0xFFFFu;
        const rtj_dev_table *t = &tables[min((int)sr0.table, RTJ_NUM_TABLES - 1)];
        const int32_t *iq = t->iq[chroma];
        const int bt8 = t->bt8[chroma];

        /* the block's bytes 8l .. 8l + 7 */
        const uint32_t b0 = __funnelshift_r(wd.w0, wd.w1, wd.sh), b1 = __funnelshift_r(wd.w1, wd.w2, wd.sh);
        rec0 = rec1; rec1 = rec2; rec2 = rec3;
        sr0 = sr1; sr1 = sr2;
        wd = wd1;
        /* what every byte fills: DC and the raw prefix (bytes 0 .. bt8) one place each, a run token b - 63, else one */
        uint32_t x0, x1;
        {
            const uint32_t r0 = b0 & ~(b0 >> 1) & 0x40404040u, r1 = b1 & ~(b1 >> 1) & 0x40404040u;
            x0 = (b0 & ((r0 >> 6) * 0x3Fu)) + 0x01010101u;
            x1 = (b1 & ((r1 >> 6) * 0x3Fu)) + 0x01010101u;
            const int nraw = min(max(bt8 + 1 - 8 * l, 0), 8);
            const uint32_t m0 = nraw >= 4 ? 0xFFFFFFFFu : (1u << (8 * nraw)) - 1u;
            const uint32_t m1 = nraw >= 8 ? 0xFFFFFFFFu : nraw <= 4 ? 0u : (1u << (8 * (nraw - 4))) - 1u;
            x0 = (x0 & ~m0) | (0x01010101u & m0);
            x1 = (x1 & ~m1) | (0x01010101u & m1);
        }
        /* zig-zag place of each of the lane's bytes: places filled before it -- within the lane, then over the eight lanes */
        int pos[8];
        {
            int acc = 0;
#pragma unroll
            for (int m = 0; m < 8; m++) { pos[m] = acc; acc += (int)(((m < 4 ? x0 : x1) >> (8 * (m & 3))) & 0xFFu); }
            int incl = acc;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const int up = __shfl_up_sync(FULL, incl, o, 8);
                if (l >= o) incl += up;
            }
            const int before = incl - acc;
#pragma unroll
            for (int m = 0; m < 8; m++) pos[m] += before;
        }
        *reinterpret_cast<uint4 *>(M + 8 * l) = make_uint4(0u, 0u, 0u, 0u);
        __syncwarp();
        if (pos[0] < 64) {
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const uint32_t bv = ((m < 4 ? b0 : b1) >> (8 * (m & 3))) & 0xFFu;
                const bool lit = 8 * l + m <= bt8 || (bv - 64u) >= 64u;           /* not a run token */
                if (lit && pos[m] < 64) {
                    const int c = (l | m) == 0 ? (int)bv : (int)(signed char)bv;  /* the DC byte is unsigned (lib/RTjpeg.c:164) */
                    M[s_zz[pos[m]]] = (int16_t)(c * __ldg(iq + pos[m]));
                }
            }
        }
        __syncwarp();
        /* first pass: column l */
        {
            int y[8];
            aan8((int)Mc[0] + (l == 0 ? 4 : 0),                         /* DESCALE's rounding term rides on the DC path */
                 Mc[8], Mc[16], Mc[24], Mc[32], Mc[40], Mc[48], Mc[56], y);
#pragma unroll
            for (int r = 0; r < 8; r++) Wc[9 * r] = y[r];
        }
        __syncwarp();
        /* second pass: row l, descale, clamp */
        {
            int y[8];
            aan8(Wr[0], Wr[1], Wr[2], Wr[3], Wr[4], Wr[5], Wr[6], Wr[7], y);
            if (live) {
                int pitch;
                uint8_t *dst = block_dst(out + (size_t)f * fsz, fmt, i, w, h, pitch);
                *reinterpret_cast<uint2 *>(dst + (size_t)l * pitch) =
                    make_uint2(descale_pack4(y[0], y[1], y[2], y[3]), descale_pack4(y[4], y[5], y[6], y[7]));
            }
        }
        __syncwarp();
    }
}

namespace {

inline int idct_seg_mb(int mbw, int *nstrips)
{
    const int n = (mbw + IDCT_MAX_MB - 1) / IDCT_MAX_MB;
    *nstrips = n;
    return (mbw + n - 1) / n;
}

/* warps per CTA: three when that spreads the strip's passes of 32 blocks evenly and four does not (a 720-wide row is 9
 * passes: three rounds of three warps, where four warps would leave three of twelve slots empty and wait for the fourth) */
inline int idct_warps(int nb)
{
    const int passes = (nb + 31) / 32;
    const int waste4 = (passes + 3) / 4 * 4 - passes, waste3 = (passes + 2) / 3 * 3 - passes;
    return waste3 < waste4 ? 3 : 4;
}

inline int idct_wq(int nb, int warps) { return (nb + warps * 32 - 1) / (warps * 32) * 32; }

inline size_t idct_smem_bytes(int seg_mb, int fmt, int warps)
{
    const int blk = fmt == 0 ? 6 : fmt == 1 ? 4 : 1;
    size_t s = (size_t)seg_mb * (fmt == 0 ? 384 : fmt == 1 ? 256 : 64);    /* the picture strip */
    s += 32;                                         /* counters */
    s += (size_t)2 * K2_WARPS * idct_wq(seg_mb * blk, warps) * 4;          /* warp queues (laid out for four) */
    return (s + 15) & ~(size_t)15;
}

int g_sm_count = 0;

template <bool SINGLE, int FMT, int WARPS, int RGBK>
cudaError_t k2_attr()
{
    cudaError_t e = cudaFuncSetAttribute(rtj_idct_kernel<SINGLE, FMT, WARPS, RGBK, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)idct_smem_bytes(IDCT_MAX_MB, FMT, 3));
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(rtj_idct_kernel<SINGLE, FMT, WARPS, RGBK, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)idct_smem_bytes(IDCT_MAX_MB, FMT, 3));
    if (RGBK == RGB_NONE && e == cudaSuccess)
        e = cudaFuncSetAttribute(rtj_idct_kernel<SINGLE, FMT, WARPS, RGB_NONE, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)idct_smem_bytes(IDCT_MAX_MB, FMT, 3));
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(rtj_idct_kernel<SINGLE, FMT, WARPS, RGBK, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)idct_smem_bytes(IDCT_MAX_MB, FMT, 3));
    if constexpr (!SINGLE) {
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(rtj_idct_kernel<false, FMT, WARPS, RGBK, false, false, true, true>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)idct_smem_bytes(IDCT_MAX_MB, FMT, 3));
    }
    return e;
}

/* a launch with programmatic stream serialisation: the grid may become resident while the kernel in front of it in the stream
 * is still at work; it calls griddepcontrol.wait before it touches what that kernel makes */
template <typename K, typename... A>
cudaError_t launch_pdl(K kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, A... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

template <int FMT, int RGBK>
cudaError_t k2_launch(K2Params &P, int grid_x, int F, cudaStream_t st)
{
    constexpr int RGBS = RGBK == RGB_NONE ? RGB_NONE : RGB_ANY;          /* what the strip kernels are instantiated with */
    const int blk = FMT == 0 ? 6 : FMT == 1 ? 4 : 1;
    const int warps = idct_warps(P.seg_mb * blk);
    P.wq = idct_wq(P.seg_mb * blk, warps);
    const int resident = (g_sm_count > 0 ? g_sm_count : 148) * (warps == 4 ? 8 : 10);
    P.ahead = (resident + grid_x - 1) / grid_x;
    const size_t smem = idct_smem_bytes(P.seg_mb, FMT, warps);
    P.run = P.run < 1 ? 1 : P.run;
    const dim3 grid((unsigned)grid_x, (unsigned)((F + P.run - 1) / P.run));
    cudaError_t e;
    if (P.jobs) {
        /* a selection: one frame per CTA whatever P.run says (the caller sets it to 1), no reservations in K2b's queue */
        if (P.nstrips == 1) {
            if (warps == 4) e = launch_pdl(rtj_idct_kernel<true, FMT, 4, RGBK, false, false, true>, grid, dim3(128), smem, st, P);
            else e = launch_pdl(rtj_idct_kernel<true, FMT, 3, RGBK, false, false, true>, grid, dim3(96), smem, st, P);
        } else {
            if (warps == 4) e = launch_pdl(rtj_idct_kernel<false, FMT, 4, RGBS, false, false, true>, grid, dim3(128), smem, st, P);
            else e = launch_pdl(rtj_idct_kernel<false, FMT, 3, RGBS, false, false, true>, grid, dim3(96), smem, st, P);
        }
    } else if (P.run > 1) {
        if (P.nstrips == 1) {
            if (warps == 4) e = launch_pdl(rtj_idct_kernel<true, FMT, 4, RGBK, true>, grid, dim3(128), smem, st, P);
            else e = launch_pdl(rtj_idct_kernel<true, FMT, 3, RGBK, true>, grid, dim3(96), smem, st, P);
        } else {
            if (warps == 4) e = launch_pdl(rtj_idct_kernel<false, FMT, 4, RGBS, true>, grid, dim3(128), smem, st, P);
            else e = launch_pdl(rtj_idct_kernel<false, FMT, 3, RGBS, true>, grid, dim3(96), smem, st, P);
        }
    } else if (RGBK == RGB_NONE && P.reserve) {
        if (P.nstrips == 1) {
            if (warps == 4) e = launch_pdl(rtj_idct_kernel<true, FMT, 4, RGB_NONE, false, true>, grid, dim3(128), smem, st, P);
            else e = launch_pdl(rtj_idct_kernel<true, FMT, 3, RGB_NONE, false, true>, grid, dim3(96), smem, st, P);
        } else {
            if (warps == 4) e = launch_pdl(rtj_idct_kernel<false, FMT, 4, RGB_NONE, false, true>, grid, dim3(128), smem, st, P);
            else e = launch_pdl(rtj_idct_kernel<false, FMT, 3, RGB_NONE, false, true>, grid, dim3(96), smem, st, P);
        }
    } else if (P.nstrips == 1) {
        if (warps == 4) e = launch_pdl(rtj_idct_kernel<true, FMT, 4, RGBK, false>, grid, dim3(128), smem, st, P);
        else e = launch_pdl(rtj_idct_kernel<true, FMT, 3, RGBK, false>, grid, dim3(96), smem, st, P);
    } else {
        if (warps == 4) e = launch_pdl(rtj_idct_kernel<false, FMT, 4, RGBS, false>, grid, dim3(128), smem, st, P);
        else e = launch_pdl(rtj_idct_kernel<false, FMT, 3, RGBS, false>, grid, dim3(96), smem, st, P);
    }
    return e != cudaSuccess ? e : cudaGetLastError();
}

/* a window of a selection (P.win_w != 0): the strip kernels, one frame per CTA; RGBK is RGB_NONE, RGB_ANY or RGB_CHW */
template <int FMT, int RGBK>
cudaError_t k2_launch_win(K2Params &P, int grid_x, int njobs, cudaStream_t st)
{
    const int blk = FMT == 0 ? 6 : FMT == 1 ? 4 : 1;
    const int warps = idct_warps(P.seg_mb * blk);
    P.wq = idct_wq(P.seg_mb * blk, warps);
    const int resident = (g_sm_count > 0 ? g_sm_count : 148) * (warps == 4 ? 8 : 10);
    P.ahead = (resident + grid_x - 1) / grid_x;
    P.run = 1;
    const size_t smem = idct_smem_bytes(P.seg_mb, FMT, warps);
    const dim3 grid((unsigned)grid_x, (unsigned)njobs);
    const cudaError_t e = warps == 4 ? launch_pdl(rtj_idct_kernel<false, FMT, 4, RGBK, false, false, true, true>, grid, dim3(128), smem, st, P)
                                     : launch_pdl(rtj_idct_kernel<false, FMT, 3, RGBK, false, false, true, true>, grid, dim3(96), smem, st, P);
    return e != cudaSuccess ? e : cudaGetLastError();
}

template <int FMT, int RGBK>
cudaError_t k2_attrs()
{
    constexpr int RGBS = RGBK == RGB_NONE ? RGB_NONE : RGB_ANY;
    cudaError_t e = k2_attr<true, FMT, 4, RGBK>();
    if (e == cudaSuccess) e = k2_attr<false, FMT, 4, RGBS>();
    if (e == cudaSuccess) e = k2_attr<true, FMT, 3, RGBK>();
    if (e == cudaSuccess) e = k2_attr<false, FMT, 3, RGBS>();
    return e;
}

} // namespace

extern "C" int rtj_idct_init(void)
{
    cudaError_t e = k2_attrs<0, RGB_NONE>();
    if (e == cudaSuccess) e = k2_attrs<0, RTJ_CONV_RGB32>();
    if (e == cudaSuccess) e = k2_attrs<0, RTJ_CONV_BGR32>();
    if (e == cudaSuccess) e = k2_attrs<0, RTJ_CONV_RGB24>();
    if (e == cudaSuccess) e = k2_attrs<0, RTJ_CONV_BGR24>();
    if (e == cudaSuccess) e = k2_attrs<0, RTJ_CONV_RGB16>();
    if (e == cudaSuccess) e = k2_attrs<1, RGB_NONE>();
    if (e == cudaSuccess) e = k2_attrs<2, RGB_NONE>();
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(rtj_idct_kernel<false, 0, 4, RGB_CHW, false, false, true, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)idct_smem_bytes(IDCT_MAX_MB, 0, 3));
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(rtj_idct_kernel<false, 0, 3, RGB_CHW, false, false, true, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)idct_smem_bytes(IDCT_MAX_MB, 0, 3));
    if (e != cudaSuccess) return (int)e;
    int dev = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    return 0;
}

/* The position table of rtj_idct_kernel<SINGLE = true> for this geometry: 4 bytes per position of one row of units. */
extern "C" size_t rtj_lut_bytes(int fmt, int w, int h)
{
    const int nb = RTJ_FMT_UNITS_X(fmt, w) * RTJ_FMT_UNIT_BLOCKS(fmt);
    return (size_t)((nb + 383) / 384 * 384) * sizeof(uint32_t);      /* whole rounds of 96 and of 128 threads */
}

extern "C" int rtj_launch_build_lut(int fmt, int w, int h, void *d_lut, void *stream)
{
    const int mbs = RTJ_FMT_UNITS_X(fmt, w);
    const int npad = (int)(rtj_lut_bytes(fmt, w, h) / sizeof(uint32_t));
    uint32_t *pos = reinterpret_cast<uint32_t *>(d_lut);
    cudaStream_t st = (cudaStream_t)stream;
    if (mbs > IDCT_MAX_MB) return 0;                 /* strips: no table */
    if (fmt == 0) rtj_build_lut_kernel<0><<<(npad + 127) / 128, 128, 0, st>>>(pos, mbs, npad);
    else if (fmt == 1) rtj_build_lut_kernel<1><<<(npad + 127) / 128, 128, 0, st>>>(pos, mbs, npad);
    else rtj_build_lut_kernel<2><<<(npad + 127) / 128, 128, 0, st>>>(pos, mbs, npad);
    return (int)cudaGetLastError();
}

extern "C" int rtj_launch_idct(const rtj_launch_args *a, void *stream)
{
    const int fmt = a->fmt;
    const int ux = RTJ_FMT_UNITS_X(fmt, a->w), uy = RTJ_FMT_UNITS_Y(fmt, a->h);
    cudaStream_t st = (cudaStream_t)stream;
    K2Params P;
    P.stream = a->d_stream; P.desc = a->d_desc; P.tables = a->d_tables; P.ent = a->d_ent; P.srcf = a->d_src;
    P.nblk = RTJ_FMT_NBLK(fmt, a->w, a->h); P.w = a->w; P.h = a->h;
    P.seg_mb = idct_seg_mb(ux, &P.nstrips);
    P.out = a->d_out; P.carry = a->d_carry; P.hardq = a->d_hardq; P.info = a->d_info;
    P.hardq_cap = (unsigned)((size_t)a->F * (size_t)P.nblk);
    P.fmt = fmt;
    P.pos = reinterpret_cast<const uint32_t *>(a->d_lut);
    P.f0 = a->f0; P.F = a->F; P.f_end = a->f1; P.run = a->k2_run; P.reserve = a->raw_expected;
    P.row0 = a->row0; P.rows = uy;
    const int grid_x = P.nstrips * (a->row1 - a->row0);
    int nf = a->f1 - a->f0;
    P.jobs = a->d_jobs; P.j0 = a->j0; P.njobs = a->njobs;
    if (a->d_jobs) {                                 /* a selection: the launch's jobs, one frame per CTA */
        nf = a->j1 - a->j0;
        P.run = 1;
        if (nf <= 0) return (int)cudaErrorInvalidValue;
    }
    P.rgb = a->d_rgb; P.rgb_row_pitch = a->rgb_row_pitch; P.rgb_frame_pitch = a->rgb_frame_pitch;
    P.rgb_kind = a->rgb_kind; P.rgb_alpha = a->rgb_alpha & 0xFFu; P.last_yuv = a->d_last_yuv;
    P.seq = a->d_seq; P.carries = a->d_carries; P.last_yuvs = a->d_last_yuvs;
    P.win = a->d_win; P.win_w = a->win_w; P.win_h = a->win_h; P.win_last = a->win_last;
    P.chw_dtype = a->chw_dtype;
    for (int c = 0; c < 3; c++) { P.chw_scale[c] = a->chw_scale[c]; P.chw_bias[c] = a->chw_bias[c]; }
    if (a->win_w) {
        /* a window: strips cut from the window's width, over the most rows of units any sequence's window spans */
        if (!a->d_jobs || !a->d_seq || a->win_rows <= 0) return (int)cudaErrorInvalidValue;
        P.seg_mb = idct_seg_mb(RTJ_FMT_UNITS_X(fmt, a->win_w), &P.nstrips);
        const int gx = P.nstrips * a->win_rows;
        if (a->chw && !a->win_last) return fmt == 0 ? (int)k2_launch_win<0, RGB_CHW>(P, gx, nf, st) : (int)cudaErrorInvalidValue;
        if (a->fused_rgb && !a->win_last) return fmt == 0 ? (int)k2_launch_win<0, RGB_ANY>(P, gx, nf, st) : (int)cudaErrorInvalidValue;
        return (int)(fmt == 0 ? k2_launch_win<0, RGB_NONE>(P, gx, nf, st) : fmt == 1 ? k2_launch_win<1, RGB_NONE>(P, gx, nf, st)
                                                                       : k2_launch_win<2, RGB_NONE>(P, gx, nf, st));
    }
    if (a->fused_rgb) {
        if (fmt != 0) return (int)cudaErrorInvalidValue;
        switch (a->rgb_kind) {
        case RTJ_CONV_RGB32: return (int)k2_launch<0, RTJ_CONV_RGB32>(P, grid_x, nf, st);
        case RTJ_CONV_BGR32: return (int)k2_launch<0, RTJ_CONV_BGR32>(P, grid_x, nf, st);
        case RTJ_CONV_RGB24: return (int)k2_launch<0, RTJ_CONV_RGB24>(P, grid_x, nf, st);
        case RTJ_CONV_BGR24: return (int)k2_launch<0, RTJ_CONV_BGR24>(P, grid_x, nf, st);
        case RTJ_CONV_RGB16: return (int)k2_launch<0, RTJ_CONV_RGB16>(P, grid_x, nf, st);
        default: return (int)cudaErrorInvalidValue;
        }
    }
    cudaError_t e = fmt == 0 ? k2_launch<0, RGB_NONE>(P, grid_x, nf, st) : fmt == 1 ? k2_launch<1, RGB_NONE>(P, grid_x, nf, st)
                                                                        : k2_launch<2, RGB_NONE>(P, grid_x, nf, st);
    return (int)e;
}

extern "C" int rtj_launch_idct_hard(const rtj_launch_args *a, void *stream)
{
    /* the queue's length is only known on the device: a fixed grid strides over it */
    const int sms = g_sm_count > 0 ? g_sm_count : 148;
    const int nblk = RTJ_FMT_NBLK(a->fmt, a->w, a->h);
    cudaError_t e16 = launch_pdl(rtj_idct_hard16_kernel, dim3((unsigned)(sms * 7)), dim3(128), 0, (cudaStream_t)stream,      /* 70 registers: seven CTAs a SM */
                                 a->d_stream, a->d_desc, a->d_tables, (const uint32_t *)a->d_ent, nblk, a->w, a->h, a->fmt, a->d_out,
                                 (const uint32_t *)a->d_hardq, (const rtj_dev_info *)a->d_info);
    if (e16 != cudaSuccess) return (int)e16;
    /* (programmatic stream serialisation, no wait: the two kernels patch different blocks; what both depend on -- K2's queue --
     * was complete before the first of them started) */
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(sms * 16));
    cfg.blockDim = dim3(HB_THREADS);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, rtj_idct_hard_kernel, a->d_stream, a->d_desc, a->d_tables, (const uint32_t *)a->d_ent, nblk,
                                             a->w, a->h, a->fmt, a->d_out, (const uint32_t *)a->d_hardq,
                                             (unsigned)((size_t)a->F * (size_t)nblk), (const rtj_dev_info *)a->d_info);
    return e != cudaSuccess ? (int)e : (int)cudaGetLastError();
}
