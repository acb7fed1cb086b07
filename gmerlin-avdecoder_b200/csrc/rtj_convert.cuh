/*
 * rtj_convert.cuh -- the arithmetic of the reference's colour converters (lib/RTjpeg.c:3071-3486), shared by the
 * stand-alone converter kernels (rtj_convert.cu) and K2's fused RGB epilogue (rtj_idct.cu).  Bit for bit the
 * reference's: 16 fractional bits, (Y - 16) * 76284, Cr/Cb - 128 times 76284 / 53281 / 25625 / 132252 (:3071-3075),
 * arithmetic shift, clamp to 0..255.
 */
#ifndef RTJ_CONVERT_CUH
#define RTJ_CONVERT_CUH

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "rtj_common.h"

namespace rtjcv {

constexpr int KY = 76284, KCRR = 76284, KCRG = 53281, KCBG = 25625, KCBB = 132252;

/* sat(a) << 8 | sat(b) in the low half, c's low half above it: two clamps to 0..255 and the packing in one I2IP */
__device__ __forceinline__ uint32_t pack_sat(int a, int b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

struct Chroma { int r, g, b; };          /* the three chroma terms of a 2x1 / 2x2 neighbourhood */

__device__ __forceinline__ Chroma chroma_terms(uint32_t cb, uint32_t cr)
{
    Chroma c;
    c.r = ((int)cr - 128) * KCRR;
    c.g = ((int)cr - 128) * KCRG + ((int)cb - 128) * KCBG;
    c.b = ((int)cb - 128) * KCBB;
    return c;
}

/* 8 pixels of one row: luma bytes in yw (little endian, pixel 0 lowest), chroma terms per pixel pair.
 * KIND as in include/rtjpeg_b200.h (RTJ_CONV_*). */
template <int KIND>
__device__ __forceinline__ void row8(const uint2 yw, const Chroma (&c)[4], uint32_t alpha, uint8_t *__restrict__ o)
{
    int R[8], G[8], B[8];                /* before the clamp */
#pragma unroll
    for (int x = 0; x < 8; x++) {
        const uint32_t yb = ((x < 4 ? yw.x : yw.y) >> (8 * (x & 3))) & 0xFFu;
        const int y = ((int)yb - 16) * KY;
        R[x] = (y + c[x >> 1].r) >> 16;
        G[x] = (y - c[x >> 1].g) >> 16;
        B[x] = (y + c[x >> 1].b) >> 16;
    }
    if (KIND == RTJ_CONV_RGB32 || KIND == RTJ_CONV_BGR32) {
        uint32_t p[8];
#pragma unroll
        for (int x = 0; x < 8; x++) {
            const bool rgb = KIND == RTJ_CONV_RGB32;
            p[x] = pack_sat(G[x], rgb ? R[x] : B[x], pack_sat((int)alpha, rgb ? B[x] : R[x], 0u));
        }
        reinterpret_cast<uint4 *>(o)[0] = make_uint4(p[0], p[1], p[2], p[3]);
        reinterpret_cast<uint4 *>(o)[1] = make_uint4(p[4], p[5], p[6], p[7]);
    } else if (KIND == RTJ_CONV_RGB16) {
        uint32_t p[4];
#pragma unroll
        for (int x = 0; x < 8; x += 2) {
            const uint32_t gr0 = pack_sat(G[x], R[x], 0u), b0 = pack_sat(0, B[x], 0u);          /* G << 8 | R, B */
            const uint32_t gr1 = pack_sat(G[x + 1], R[x + 1], 0u), b1 = pack_sat(0, B[x + 1], 0u);
            const uint32_t lo = (b0 >> 3) | ((gr0 >> 10) << 5) | (((gr0 & 0xFFu) >> 3) << 11);
            const uint32_t hi = (b1 >> 3) | ((gr1 >> 10) << 5) | (((gr1 & 0xFFu) >> 3) << 11);
            p[x >> 1] = lo | hi << 16;
        }
        *reinterpret_cast<uint4 *>(o) = make_uint4(p[0], p[1], p[2], p[3]);
    } else {                             /* 24 bits: four pixels are twelve bytes, three words */
        const bool rgb = KIND != RTJ_CONV_BGR24;
        const int *F0 = rgb ? R : B, *F2 = rgb ? B : R;        /* first and third byte of a pixel */
        uint32_t wd[6];
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int x = 4 * q;
            wd[3 * q] = pack_sat(G[x], F0[x], pack_sat(F0[x + 1], F2[x], 0u));
            wd[3 * q + 1] = pack_sat(F2[x + 1], G[x + 1], pack_sat(G[x + 2], F0[x + 2], 0u));
            wd[3 * q + 2] = pack_sat(F0[x + 3], F2[x + 2], pack_sat(F2[x + 3], G[x + 3], 0u));
        }
        reinterpret_cast<uint2 *>(o)[0] = make_uint2(wd[0], wd[1]);
        reinterpret_cast<uint2 *>(o)[1] = make_uint2(wd[2], wd[3]);
        reinterpret_cast<uint2 *>(o)[2] = make_uint2(wd[4], wd[5]);
    }
}

/* The same 8 pixels as row8 computes them, clamped, one channel at a time: 8 bytes each, pixel 0 lowest */
struct Rgb8 { uint2 r, g, b; };

__device__ __forceinline__ Rgb8 rgb8(const uint2 yw, const Chroma (&c)[4])
{
    int R[8], G[8], B[8];
#pragma unroll
    for (int x = 0; x < 8; x++) {
        const uint32_t yb = ((x < 4 ? yw.x : yw.y) >> (8 * (x & 3))) & 0xFFu;
        const int y = ((int)yb - 16) * KY;
        R[x] = (y + c[x >> 1].r) >> 16;
        G[x] = (y - c[x >> 1].g) >> 16;
        B[x] = (y + c[x >> 1].b) >> 16;
    }
    auto bytes8 = [](const int (&v)[8]) {
        return make_uint2(pack_sat(v[1], v[0], pack_sat(v[3], v[2], 0u)), pack_sat(v[5], v[4], pack_sat(v[7], v[6], 0u)));
    };
    return Rgb8{bytes8(R), bytes8(G), bytes8(B)};
}

/* 8 bytes in reverse order: a chunk of a mirrored window */
__device__ __forceinline__ uint2 reverse8(uint2 v)
{
    return make_uint2(__byte_perm(v.y, 0u, 0x0123), __byte_perm(v.x, 0u, 0x0123));
}

/* 8 elements of one channel of a planar window (rtjgpu_decode_device_chw_window) to o: the bytes v themselves (RTJ_CHW_U8,
 * 8 bytes), or fadd_rn(fmul_rn(v, s), b) -- two roundings, never contracted -- as binary16 / bfloat16 (16 bytes) or float32
 * (32 bytes) */
__device__ __forceinline__ void chw8(int dtype, uint2 v, float s, float b, uint8_t *__restrict__ o)
{
    if (dtype == RTJ_CHW_U8) {
        *reinterpret_cast<uint2 *>(o) = v;
        return;
    }
    float t[8];
#pragma unroll
    for (int x = 0; x < 8; x++)
        t[x] = __fadd_rn(__fmul_rn((float)(((x < 4 ? v.x : v.y) >> (8 * (x & 3))) & 0xFFu), s), b);
    if (dtype == RTJ_CHW_F32) {
        reinterpret_cast<float4 *>(o)[0] = make_float4(t[0], t[1], t[2], t[3]);
        reinterpret_cast<float4 *>(o)[1] = make_float4(t[4], t[5], t[6], t[7]);
        return;
    }
    uint32_t p[4];
#pragma unroll
    for (int x = 0; x < 8; x += 2) {
        if (dtype == RTJ_CHW_F16) {
            const __half2 hv = __floats2half2_rn(t[x], t[x + 1]);
            p[x >> 1] = *reinterpret_cast<const uint32_t *>(&hv);
        } else {
            const __nv_bfloat162 bv = __floats2bfloat162_rn(t[x], t[x + 1]);
            p[x >> 1] = *reinterpret_cast<const uint32_t *>(&bv);
        }
    }
    *reinterpret_cast<uint4 *>(o) = make_uint4(p[0], p[1], p[2], p[3]);
}

} // namespace rtjcv

#endif
