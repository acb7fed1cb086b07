/*
 * rtj_encode.cu -- the encoder half of lib/RTjpeg.c for sm_100a: RTjpeg_compress (:3488-3524) over a batch of
 * pictures that are resident in HBM, YUV420 and YUV422.
 *
 *   E1  rtj_encode_blocks_kernel   one thread per (run of pictures, block place): forward AAN transform
 *                                  (RTjpeg_dctY :288-390), quantisation (RTjpeg_quant :245-252), the comparison
 *                                  with the block last sent at that place (RTjpeg_bcomp :2827-2838) and the
 *                                  run-length coding (RTjpeg_b2s :109-155) into a 64-byte slot.  The comparison
 *                                  chains a block place from picture to picture, but only up to the next picture
 *                                  whose key counter is 0 -- there the reference clears the stored blocks
 *                                  (:3505) -- so runs of key_rate + 1 pictures are independent of each other.
 *   E2  rtj_encode_layout_kernel   per picture: exclusive scan of the block lengths, packet size
 *   E3  rtj_encode_offsets_kernel  exclusive scan of the packet sizes (each rounded up to 4 bytes)
 *   E4  rtj_encode_gather_kernel   blocks and headers (RTjpeg_frameheader, include/RTjpeg.h:100-109) into place
 *
 * All arithmetic is the reference's, bit for bit.  The 8-bit format is not offered: RTjpeg_compress8 reads its
 * blocks with a row stride of 8 * width (:2627), outside the plane -- there is nothing defined to reproduce.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "rtj_common.h"

namespace {

constexpr int EN_THREADS = 128;

/* zig-zag position k sits at raster index ZZ(k): lib/RTjpeg.c:59-74 */
__device__ constexpr int EN_ZZ[64] = {
    0, 8, 1, 2, 9, 16, 24, 17, 10, 3, 4, 11, 18, 25, 32, 40, 33, 26, 19, 12, 5, 6, 13, 20, 27, 34, 41, 48, 56, 49, 42, 35,
    28, 21, 14, 7, 15, 22, 29, 36, 43, 50, 57, 58, 51, 44, 37, 30, 23, 31, 38, 45, 52, 59, 60, 53, 46, 39, 47, 54, 61, 62, 55, 63};

/* ... and raster index i is zig-zag position EN_RANK[i] */
__device__ constexpr int EN_RANK[64] = {
    0, 2, 3, 9, 10, 20, 21, 35, 1, 4, 8, 11, 19, 22, 34, 36, 5, 7, 12, 18, 23, 33, 37, 48, 6, 13, 17, 24, 32, 38, 47, 49, 14, 16, 25, 31, 39, 46, 50, 57, 15, 26, 30, 40, 45, 51, 56, 58, 27, 29, 41, 44, 52, 55, 59, 62, 28, 42, 43, 53, 54, 60, 61, 63};

/* the 8-point flow graph shared by both passes (:303-340, :346-389); r0 and r4 come out unscaled */
__device__ __forceinline__ void fdct8(const int (&x)[8], int &r0, int &r1, int &r2, int &r3, int &r4, int &r5, int &r6, int &r7)
{
    const int t0 = x[0] + x[7], t7 = x[0] - x[7], t1 = x[1] + x[6], t6 = x[1] - x[6];
    const int t2 = x[2] + x[5], t5 = x[2] - x[5], t3 = x[3] + x[4], t4 = x[3] - x[4];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    r0 = t10 + t11;
    r4 = t10 - t11;
    const int z1 = (t12 + t13) * 181;
    r2 = (t13 << 8) + z1;
    r6 = (t13 << 8) - z1;
    const int u10 = t4 + t5, u11 = t5 + t6, u12 = t6 + t7;
    const int z5 = (u10 - u12) * 98, z2 = u10 * 139 + z5, z4 = u12 * 334 + z5, z3 = u11 * 181;
    const int z11 = (t7 << 8) + z3, z13 = (t7 << 8) - z3;
    r5 = z13 + z2; r3 = z13 - z2; r1 = z11 + z4; r7 = z11 - z4;
}

/* where block i (stream order) of a picture lives: byte offset of its first row and the row pitch */
__device__ __forceinline__ size_t block_at(int fmt, int i, int w, int h, int &pitch)
{
    const int cw = w >> 1, uw = w >> 4;
    if (fmt == RTJ_YUV420) {
        const int mb = i / 6, sub = i - mb * 6, my = mb / uw, mx = mb - my * uw;
        if (sub < 4) { pitch = w; return (size_t)(my * 16 + (sub >> 1) * 8) * w + mx * 16 + (sub & 1) * 8; }
        pitch = cw;
        return (size_t)w * h + (sub == 5 ? (size_t)cw * (h >> 1) : 0) + (size_t)(my * 8) * cw + mx * 8;
    }
    const int un = i >> 2, sub = i & 3, by = un / uw, ux = un - by * uw;
    if (sub < 2) { pitch = w; return (size_t)(by * 8) * w + ux * 16 + sub * 8; }
    pitch = cw;
    return (size_t)w * h + (sub == 3 ? (size_t)cw * h : 0) + (size_t)(by * 8) * cw + ux * 8;
}

} // namespace

/* INTER: pictures are compared with the blocks last sent (key_rate != 0); false: none of that is compiled in.
 * SEQ: rtjgpu_encode_device_seq -- run blockIdx.y is runs[blockIdx.y], and its sequence's record gives pictures, stored
 * blocks, tables and masks; false: one sequence, runs cut by period / first_boundary, runs and seqs unused. */
template <bool INTER, bool SEQ = false>
__global__ void __launch_bounds__(EN_THREADS, INTER ? 3 : 4)
rtj_encode_blocks_kernel(const rtj_encode_args A, int nblk, int nruns, int period, int first_boundary,
                         const rtj_enc_run *__restrict__ runs, const rtj_enc_seq *__restrict__ seqs)
{
    __shared__ int32_t s_qt[128];                           /* the quantiser's multipliers: read 64 times a block */
    /* a row a thread: the block's token values in zig-zag order, then -- in place -- its bytes (RTjpeg_b2s never writes more
     * bytes than it has read places); 17 words: the rows of a warp on different banks */
    __shared__ uint32_t s_zz[EN_THREADS][17];
    /* INTER: the quantised block itself, two values a word as the stored blocks hold them, for the comparison (kept out of
     * the registers: the transform's 64 intermediate values live there) */
    __shared__ uint32_t s_q[INTER ? EN_THREADS : 1][33];
    const int run = blockIdx.y;
    const rtj_enc_run R = SEQ ? runs[run] : rtj_enc_run{};
    const rtj_enc_seq *const Q = SEQ ? seqs + (R.seq & RTJ_ENC_RUN_INDEX) : nullptr;
    s_qt[threadIdx.x] = SEQ ? A.d_qt[Q->quality * 128 + threadIdx.x] : A.d_qt[threadIdx.x];
    static_assert(EN_THREADS == 128, "one multiplier a thread");
    __syncthreads();
    const int b = blockIdx.x * EN_THREADS + threadIdx.x;
    if (b >= nblk) return;
    /* the pictures of this run: [f0, f1).  Run 0 may continue a run of the call before (key_count0 != 0). */
    constexpr bool inter = INTER;
    int f0, f1;
    if (SEQ) { f0 = R.f0; f1 = R.f1; }
    else if (!inter) { f0 = run; f1 = run + 1; }
    else if (first_boundary == 0) { f0 = run * period; f1 = min(f0 + period, A.F); }
    else if (run == 0) { f0 = 0; f1 = min(first_boundary, A.F); }
    else { f0 = first_boundary + (run - 1) * period; f1 = min(f0 + period, A.F); }
    const size_t fsz = RTJ_FMT_FRAME_BYTES(A.fmt, A.w, A.h);
    int pitch;
    const size_t at = block_at(A.fmt, b, A.w, A.h, pitch);
    const bool luma = A.fmt == RTJ_YUV420 ? (b % 6) < 4 : (b & 3) < 2;
    const int32_t *qt = s_qt + (luma ? 0 : 64);
    const int bt8 = SEQ ? (luma ? Q->lb8 : Q->cb8) : (luma ? A.lb8 : A.cb8);
    const int mask = SEQ ? (luma ? Q->lmask : Q->cmask) : (luma ? A.lmask : A.cmask);
    /* SEQ: output frame f is picture f - Q->first of the sequence's pictures */
    const uint8_t *const pics = SEQ ? Q->d_frames : nullptr;
    const int fbase = SEQ ? Q->first : 0;

    /* the block last sent here, two coefficients per register */
    uint32_t old[INTER ? 32 : 1];
    const bool continues = inter && (SEQ ? (R.seq & RTJ_ENC_RUN_CONT) != 0 : run == 0 && A.key_count0 != 0);
    if (INTER) {
#pragma unroll
        for (int k = 0; k < 32; k++) old[k] = continues ? reinterpret_cast<const uint32_t *>((SEQ ? Q->d_old : A.d_old) + (size_t)b * 64)[k] : 0u;
    }

    for (int f = f0; f < f1; f++) {
        const uint8_t *src = SEQ ? pics + (size_t)(f - fbase) * fsz + at : A.d_frames + (size_t)f * fsz + at;
        int ws[64];
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint2 p = *reinterpret_cast<const uint2 *>(src + (size_t)r * pitch);
            int x[8];
#pragma unroll
            for (int c = 0; c < 8; c++) x[c] = (int)(((c < 4 ? p.x : p.y) >> (8 * (c & 3))) & 0xFFu);
            int r0, r4;
            fdct8(x, r0, ws[r * 8 + 1], ws[r * 8 + 2], ws[r * 8 + 3], r4, ws[r * 8 + 5], ws[r * 8 + 6], ws[r * 8 + 7]);
            ws[r * 8 + 0] = r0 << 8;
            ws[r * 8 + 4] = r4 << 8;
        }
        uint8_t *row = reinterpret_cast<uint8_t *>(s_zz[threadIdx.x]);
        int16_t *qrow = reinterpret_cast<int16_t *>(s_q[INTER ? threadIdx.x : 0]);
        int dc = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) {
            int x[8], y[8];
#pragma unroll
            for (int r = 0; r < 8; r++) x[r] = ws[r * 8 + c];
            fdct8(x, y[0], y[1], y[2], y[3], y[4], y[5], y[6], y[7]);
#pragma unroll
            for (int r = 0; r < 8; r++) {
                /* DESCALE10 for rows 0 and 4, DESCALE20 for the others (:272-273), each narrowed to int16; then RTjpeg_quant */
                const int v = (int)(short)((r == 0 || r == 4) ? (y[r] + 128) >> 8 : (y[r] + 32768) >> 16);
                const int q = (int)(short)((v * qt[r * 8 + c] + 32767) >> 16);
                if (INTER) qrow[r * 8 + c] = (int16_t)q;
                /* what RTjpeg_b2s (:109-155) makes of the value at its zig-zag place: clamped to a byte inside the raw prefix,
                 * to -64 .. 63 behind it */
                const int place = EN_RANK[r * 8 + c];
                if (place == 0) dc = q;
                else {
                    const int lim = place <= bt8 ? 127 : 63;
                    row[place] = (uint8_t)(q > 0 ? min(q, lim) : max(q, -lim - 1));
                }
            }
        }
        bool skip = false;
        if (INTER) {
            bool same = true;
#pragma unroll
            for (int k = 0; k < (INTER ? 32 : 0); k++) {
                const uint32_t nw = s_q[INTER ? threadIdx.x : 0][k];
                const int o0 = (int)(short)(old[k] & 0xFFFFu), o1 = (int)(short)(old[k] >> 16);
                const int n0 = (int)(short)(nw & 0xFFFFu), n1 = (int)(short)(nw >> 16);
                same = same && abs(o0 - n0) <= mask && abs(o1 - n1) <= mask;
            }
            skip = same;
            if (!same) {
#pragma unroll
                for (int k = 0; k < (INTER ? 32 : 0); k++) old[k] = s_q[INTER ? threadIdx.x : 0][k];
            }
        }
        uint8_t *slot = A.d_slots + ((size_t)f * nblk + b) * 64;
        int co = 1;
        if (skip) row[0] = 0xFF;
        else {
            row[0] = (uint8_t)(dc > 254 ? 254 : (dc < 0 ? 0 : dc));
            /* the last place that gets a byte of its own: the last value that is not zero, or the raw prefix's end;
             * everything behind it is one run token (most blocks of ordinary material end within the first ten places) */
            int last = 0;
            for (int wv = 15; wv >= 0; wv--) {
                uint32_t x4 = s_zz[threadIdx.x][wv];
                if (wv == 0) x4 &= 0xFFFFFF00u;
                if (x4) { last = 4 * wv + 3 - (__clz((int)x4) >> 3); break; }
            }
            last = max(last, min(bt8, 63));
            int zeros = 0;
            for (int ci = 1; ci <= last; ci++) {
                const int v = (int)(signed char)row[ci];
                if (ci <= bt8) row[co++] = (uint8_t)v;
                else if (v != 0) {
                    if (zeros) { row[co++] = (uint8_t)(63 + zeros); zeros = 0; }
                    row[co++] = (uint8_t)v;
                } else zeros++;
            }
            zeros += 63 - last;                                        /* the places behind `last` are zero */
            if (zeros) row[co++] = (uint8_t)(63 + zeros);
        }
        /* the bytes leave as words (what lies behind the block's last byte in its slot is never read) */
        for (int k = 0; k < (co + 3) >> 2; k++) reinterpret_cast<uint32_t *>(slot)[k] = s_zz[threadIdx.x][k];
        A.d_lens[(size_t)f * nblk + b] = (uint8_t)co;
    }
    /* the run that ends the batch (SEQ: its sequence) leaves its blocks for the next call */
    if (INTER && (SEQ ? (R.seq & RTJ_ENC_RUN_LAST) != 0 : f1 == A.F)) {
#pragma unroll
        for (int k = 0; k < (INTER ? 32 : 0); k++) reinterpret_cast<uint32_t *>((SEQ ? Q->d_old : A.d_old) + (size_t)b * 64)[k] = old[k];
    }
}

/* per picture: where every block's bytes go inside the payload, and the packet size */
extern "C" __global__ void __launch_bounds__(256)
rtj_encode_layout_kernel(const uint8_t *__restrict__ lens, uint32_t *__restrict__ boff, uint32_t *__restrict__ fsize, int nblk)
{
    __shared__ uint32_t warp_tot[8];
    __shared__ uint32_t carry;
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nblk; b0 += 256) {
        const int b = b0 + tid;
        const uint32_t len = b < nblk ? lens[(size_t)f * nblk + b] : 0u;
        uint32_t incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        uint32_t base = carry;
        for (int k = 0; k < warp; k++) base += warp_tot[k];
        if (b < nblk) boff[(size_t)f * nblk + b] = base + incl - len;
        __syncthreads();
        if (tid == 255) carry = base + incl;
        __syncthreads();
    }
    if (tid == 0) fsize[f] = carry + RTJPEG_B200_HEADER_BYTES;
}

/* packet offsets: every packet starts on a multiple of 4 (what rtjgpu_decode_device asks of its input) */
extern "C" __global__ void __launch_bounds__(1024)
rtj_encode_offsets_kernel(const uint32_t *__restrict__ fsize, int F, uint64_t *__restrict__ offsets, uint64_t *__restrict__ total,
                          size_t capacity)
{
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int f0 = 0; f0 < F; f0 += 1024) {
        const int f = f0 + tid;
        const unsigned long long sz = f < F ? (unsigned long long)((fsize[f] + 3u) & ~3u) : 0ull;
        unsigned long long incl = sz;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        unsigned long long base = carry;
        for (int k = 0; k < warp; k++) base += warp_tot[k];
        if (f < F) offsets[f] = base + incl - sz;
        __syncthreads();
        if (tid == 1023) carry = base + incl;
        __syncthreads();
    }
    if (tid == 0) {
        offsets[F] = carry;
        total[0] = carry;
        total[1] = carry > (unsigned long long)capacity ? 1ull : 0ull;
    }
}

/* SEQ: the header's quality and key bytes come from frame_words[f] (RTJ_ENC_FRAME) */
template <bool SEQ = false>
__global__ void __launch_bounds__(EN_THREADS)
rtj_encode_gather_kernel(const rtj_encode_args A, int nblk, int period, const uint32_t *__restrict__ frame_words)
{
    if (A.d_total[1]) return;                               /* the stream buffer is too small: nothing is written */
    const int f = blockIdx.y;
    uint8_t *pkt = A.d_stream + A.d_offsets[f];
    const int b = blockIdx.x * EN_THREADS + threadIdx.x;
    if (b == 0) {
        /* RTjpeg_frameheader (include/RTjpeg.h:100-109), filled as RTjpeg_compress does (:3515-3522) */
        const uint32_t ds = A.d_fsize[f];
        const uint32_t fw = SEQ ? frame_words[f] : 0u;
        const int key = SEQ ? (int)(fw >> 8) & 0xFF : A.key_rate == 0 ? 0 : (A.key_count0 + f) % period;
        const int quality = SEQ ? (int)fw & 0xFF : A.quality;
        pkt[0] = (uint8_t)ds; pkt[1] = (uint8_t)(ds >> 8); pkt[2] = (uint8_t)(ds >> 16); pkt[3] = (uint8_t)(ds >> 24);
        pkt[4] = RTJPEG_B200_HEADER_BYTES; pkt[5] = 0;
        pkt[6] = (uint8_t)A.w; pkt[7] = (uint8_t)(A.w >> 8); pkt[8] = (uint8_t)A.h; pkt[9] = (uint8_t)(A.h >> 8);
        pkt[10] = (uint8_t)quality; pkt[11] = (uint8_t)key;
        for (uint32_t k = ds; k < ((ds + 3u) & ~3u); k++) pkt[k] = 0;       /* the padding up to the next packet */
    }
    if (b >= nblk) return;
    const size_t i = (size_t)f * nblk + b;
    const uint8_t *slot = A.d_slots + i * 64;
    uint8_t *dst = pkt + RTJPEG_B200_HEADER_BYTES + A.d_boff[i];
    const int n = A.d_lens[i];
    for (int k = 0; k < n; k++) dst[k] = slot[k];
}

namespace {

/* E2, E3 and E4 behind E1: the same for both entry points but for where E4 takes its header bytes */
template <bool SEQ>
int launch_layout_and_gather(const rtj_encode_args *a, int nblk, int period, const uint32_t *frame_words, cudaStream_t st)
{
    const unsigned gx = (unsigned)((nblk + EN_THREADS - 1) / EN_THREADS);
    cudaError_t e;
    rtj_encode_layout_kernel<<<(unsigned)a->F, 256, 0, st>>>(a->d_lens, a->d_boff, a->d_fsize, nblk);
    if ((e = cudaGetLastError()) != cudaSuccess) return -(int)e;
    rtj_encode_offsets_kernel<<<1, 1024, 0, st>>>(a->d_fsize, a->F, a->d_offsets, a->d_total, a->capacity);
    if ((e = cudaGetLastError()) != cudaSuccess) return -(int)e;
    rtj_encode_gather_kernel<SEQ><<<dim3(gx, (unsigned)a->F), EN_THREADS, 0, st>>>(*a, nblk, period, frame_words);
    if ((e = cudaGetLastError()) != cudaSuccess) return -(int)e;
    return 3;
}

} // namespace

extern "C" int rtj_launch_encode(const rtj_encode_args *a, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const int nblk = RTJ_FMT_NBLK(a->fmt, a->w, a->h);
    const int period = a->key_rate + 1;
    const bool inter = a->key_rate != 0;
    const int first_boundary = inter ? (period - a->key_count0 % period) % period : 0;
    int nruns;
    if (!inter) nruns = a->F;
    else if (first_boundary == 0) nruns = (a->F + period - 1) / period;
    else nruns = 1 + (a->F > first_boundary ? (a->F - first_boundary + period - 1) / period : 0);
    const unsigned gx = (unsigned)((nblk + EN_THREADS - 1) / EN_THREADS);
    if (inter) rtj_encode_blocks_kernel<true><<<dim3(gx, (unsigned)nruns), EN_THREADS, 0, st>>>(*a, nblk, nruns, period, first_boundary, nullptr, nullptr);
    else rtj_encode_blocks_kernel<false><<<dim3(gx, (unsigned)nruns), EN_THREADS, 0, st>>>(*a, nblk, nruns, period, first_boundary, nullptr, nullptr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return -(int)e;
    const int n = launch_layout_and_gather<false>(a, nblk, period, nullptr, st);
    return n < 0 ? n : 1 + n;
}

extern "C" int rtj_launch_encode_seq(const rtj_encode_args *a, const rtj_enc_run *d_runs, int n_intra, int n_inter,
                                     const rtj_enc_seq *d_seqs, const uint32_t *d_frame_words, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const int nblk = RTJ_FMT_NBLK(a->fmt, a->w, a->h);
    const unsigned gx = (unsigned)((nblk + EN_THREADS - 1) / EN_THREADS);
    int launches = 0;
    cudaError_t e;
    if (n_intra) {
        rtj_encode_blocks_kernel<false, true><<<dim3(gx, (unsigned)n_intra), EN_THREADS, 0, st>>>(*a, nblk, n_intra, 0, 0, d_runs, d_seqs);
        if ((e = cudaGetLastError()) != cudaSuccess) return -(int)e;
        launches++;
    }
    if (n_inter) {
        rtj_encode_blocks_kernel<true, true><<<dim3(gx, (unsigned)n_inter), EN_THREADS, 0, st>>>(*a, nblk, n_inter, 0, 0,
                                                                                               d_runs + n_intra, d_seqs);
        if ((e = cudaGetLastError()) != cudaSuccess) return -(int)e;
        launches++;
    }
    const int n = launch_layout_and_gather<true>(a, nblk, 0, d_frame_words, st);
    return n < 0 ? n : launches + n;
}
