/*
 * ref_driver.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Thin driver around the UNMODIFIED reference object (lib/RTjpeg.c compiled
 * where it lies under /root/reference by oracle/Makefile, its RTjpeg_* symbols
 * renamed to ref_RTjpeg_* with objcopy so that the object can sit in the same
 * process as the drop-in library that exports the original names).
 *
 * It provides what the reference has no tool for (SURVEY.md section 4):
 *   - packets of caller-supplied pictures from the reference's own RTjpeg_compress (:3488),
 *   - sequential and threaded decode with the reference's RTjpeg_decompress
 *     (:3565) for parity checks and for the CPU baseline timing.
 * No reference source text is reproduced here; only its public API
 * (include/RTjpeg.h:115-139) is called.
 */
#define _GNU_SOURCE
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

typedef void RTjpeg_t;
extern RTjpeg_t *ref_RTjpeg_init(void);
extern void ref_RTjpeg_close(RTjpeg_t *);
extern int ref_RTjpeg_set_quality(RTjpeg_t *, int *);
extern int ref_RTjpeg_set_format(RTjpeg_t *, int *);
extern int ref_RTjpeg_set_size(RTjpeg_t *, int *, int *);
extern int ref_RTjpeg_set_intra(RTjpeg_t *, int *, int *, int *);
extern int ref_RTjpeg_compress(RTjpeg_t *, uint8_t *, uint8_t **);
extern void ref_RTjpeg_decompress(RTjpeg_t *, uint8_t *, uint8_t **);
extern void ref_RTjpeg_get_tables(RTjpeg_t *, uint32_t *);
extern void ref_RTjpeg_set_tables(RTjpeg_t *, uint32_t *);

/* ------------------------------------------------------------------ */
/* encode                                                              */
/* ------------------------------------------------------------------ */

typedef struct {
    int w, h, Q, key_rate, lm, cm;      /* key_rate < 0: no set_intra call (pure intra) */
    int noise_y, noise_c, dark;
    uint32_t seed;
} refdrv_clip;

static RTjpeg_t *make_encoder(const refdrv_clip *c)
{
    RTjpeg_t *e = ref_RTjpeg_init();
    int fmt = 0, w = c->w, h = c->h, q = c->Q;
    ref_RTjpeg_set_format(e, &fmt);
    ref_RTjpeg_set_size(e, &w, &h);
    ref_RTjpeg_set_quality(e, &q);
    if (c->key_rate >= 0) {
        int k = c->key_rate, lm = c->lm, cm = c->cm;
        ref_RTjpeg_set_intra(e, &k, &lm, &cm);
    }
    return e;
}

/* worst-case packet: header + 64 bytes per block */
size_t refdrv_packet_bound(int w, int h) { return 12 + (size_t)(w / 16) * (h / 16) * 6 * 64 + 64; }

/*
 * Encode caller-supplied frames (F tight YUV420 frames back to back) with ONE
 * encoder instance, sequentially.  Packets are written back to back into out
 * (each start rounded up to `align` bytes), offsets[F+1] receives their starts
 * (offsets[F] = end of the last one, unaligned).  Returns bytes used or 0 if
 * cap is too small.
 */
size_t refdrv_encode_frames(const refdrv_clip *c, const uint8_t *frames, int F,
                            uint8_t *out, size_t cap, uint64_t *offsets, int align)
{
    RTjpeg_t *e = make_encoder(c);
    size_t fsz = (size_t)c->w * c->h * 3 / 2, at = 0, bound = refdrv_packet_bound(c->w, c->h);
    uint8_t *tmp = (uint8_t *)malloc(bound);
    for (int f = 0; f < F; f++) {
        const uint8_t *base = frames + fsz * f;
        uint8_t *pl[3] = { (uint8_t *)base, (uint8_t *)base + (size_t)c->w * c->h,
                           (uint8_t *)base + (size_t)c->w * c->h * 5 / 4 };
        int n = ref_RTjpeg_compress(e, tmp, pl);
        at = (at + (size_t)align - 1) / (size_t)align * (size_t)align;
        if (at + (size_t)n > cap) { free(tmp); ref_RTjpeg_close(e); return 0; }
        memcpy(out + at, tmp, (size_t)n);
        offsets[f] = at;
        at += (size_t)n;
    }
    offsets[F] = at;
    free(tmp);
    ref_RTjpeg_close(e);
    return at;
}

/* ------------------------------------------------------------------ */
/* decode                                                              */
/* ------------------------------------------------------------------ */

/*
 * Sequential decode of F packets with ONE reference decoder instance into one
 * persistent plane set (initialised from `init`, w*h*3/2 bytes, or zero if
 * NULL), exactly the shape of decode_rtjpeg (video_rtjpeg.c:62-90) minus gavl.
 * After each frame the planes are copied to frames_out + f*w*h*3/2 when
 * frames_out != NULL.  last_out (w*h*3/2) receives the final planes.
 */
void refdrv_decode_seq(const uint8_t *stream, const uint64_t *offsets, int F, int w, int h,
                       const uint8_t *init, uint8_t *frames_out, uint8_t *last_out)
{
    size_t ysz = (size_t)w * h, fsz = ysz * 3 / 2;
    uint8_t *pl_mem = (uint8_t *)malloc(fsz);
    if (init) memcpy(pl_mem, init, fsz); else memset(pl_mem, 0, fsz);
    uint8_t *pl[3] = { pl_mem, pl_mem + ysz, pl_mem + ysz * 5 / 4 };
    RTjpeg_t *d = ref_RTjpeg_init();
    for (int f = 0; f < F; f++) {
        ref_RTjpeg_decompress(d, (uint8_t *)stream + offsets[f], pl);
        if (frames_out) memcpy(frames_out + fsz * f, pl_mem, fsz);
    }
    if (last_out) memcpy(last_out, pl_mem, fsz);
    ref_RTjpeg_close(d);
    free(pl_mem);
}

typedef struct {
    const uint8_t *stream;
    const uint64_t *offsets;
    const int *seg;             /* segment start frame indices, nseg+1 entries */
    int s0, s1;                 /* segment range owned by this worker */
    int w, h;
    uint8_t *frames_out;        /* may be NULL */
    int zero_init;              /* clear the planes at every segment start */
    uint64_t checksum;
    const uint32_t *raw;        /* NULL, or 128 raw tables loaded with RTjpeg_set_tables before the first packet */
} dec_job;


static void *dec_worker(void *arg)
{
    dec_job *j = (dec_job *)arg;
    size_t ysz = (size_t)j->w * j->h, fsz = ysz * 3 / 2;
    uint8_t *pl_mem = (uint8_t *)malloc(fsz);
    uint8_t *pl[3] = { pl_mem, pl_mem + ysz, pl_mem + ysz * 5 / 4 };
    RTjpeg_t *d = ref_RTjpeg_init();
    if (j->raw) {
        /* the set_tables path: they stay in force while the packets' quality byte equals the decoder's Q (0 on a
         * fresh instance, lib/RTjpeg.c:3575-3579) */
        uint32_t tmp[128];
        int ww = j->w, hh = j->h;
        memcpy(tmp, j->raw, sizeof(tmp));
        ref_RTjpeg_set_size(d, &ww, &hh);
        ref_RTjpeg_set_tables(d, tmp);
    }
    uint64_t acc = 0;
    for (int s = j->s0; s < j->s1; s++) {
        if (j->zero_init || s == j->s0) memset(pl_mem, 0, fsz);
        for (int f = j->seg[s]; f < j->seg[s + 1]; f++) {
            ref_RTjpeg_decompress(d, (uint8_t *)j->stream + j->offsets[f], pl);
            if (j->frames_out) memcpy(j->frames_out + fsz * f, pl_mem, fsz);
            else acc += pl_mem[(size_t)f % fsz];     /* keep the decode observable */
        }
    }
    j->checksum = acc;
    ref_RTjpeg_close(d);
    free(pl_mem);
    return NULL;
}

/*
 * Threaded decode, the CPU-baseline shape of BASELINE.md section 3: `threads`
 * workers, each with a private reference decoder and a private plane set,
 * whole segments per worker (segments = independent frame ranges: single
 * frames for intra-only streams, clean-frame-delimited runs for inter
 * streams; with zero_init each segment starts from zeroed planes, which is what
 * parity needs; the timing leg passes 0 for intra-only streams so the baseline
 * is not charged a memset the reference would not do).  Returns wall seconds
 * for the decode only (CLOCK_MONOTONIC).
 */
double refdrv_decode_threaded_tables(const uint8_t *stream, const uint64_t *offsets,
                                     const int *seg, int nseg, int w, int h, int threads,
                                     int zero_init, uint8_t *frames_out, const uint32_t *raw);

double refdrv_decode_threaded(const uint8_t *stream, const uint64_t *offsets,
                              const int *seg, int nseg, int w, int h, int threads,
                              int zero_init, uint8_t *frames_out)
{
    return refdrv_decode_threaded_tables(stream, offsets, seg, nseg, w, h, threads, zero_init, frames_out, NULL);
}

/* the same with every worker's decoder given raw tables through RTjpeg_set_tables first (packets carry quality 0) */
double refdrv_decode_threaded_tables(const uint8_t *stream, const uint64_t *offsets,
                                     const int *seg, int nseg, int w, int h, int threads,
                                     int zero_init, uint8_t *frames_out, const uint32_t *raw)
{
    if (threads < 1) threads = 1;
    if (threads > nseg) threads = nseg;
    dec_job *jobs = (dec_job *)calloc((size_t)threads, sizeof(dec_job));
    pthread_t *th = (pthread_t *)calloc((size_t)threads, sizeof(pthread_t));
    /* balance by frame count */
    int F = seg[nseg];
    int s = 0;
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int i = 0; i < threads; i++) {
        long want = (long)F * (i + 1) / threads;
        int e = s;
        while (e < nseg && seg[e + 1] <= want) e++;
        if (i == threads - 1) e = nseg;
        jobs[i] = (dec_job){ stream, offsets, seg, s, e, w, h, frames_out, zero_init, 0, raw };
        s = e;
        pthread_create(&th[i], NULL, dec_worker, &jobs[i]);
    }
    for (int i = 0; i < threads; i++) pthread_join(th[i], NULL);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    free(jobs); free(th);
    return (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
}

/* Tables as the reference derives them, for pinning the host table builder. */
void refdrv_tables_for_quality(int Q, uint32_t out[128])
{
    RTjpeg_t *d = ref_RTjpeg_init();
    int q = Q;
    ref_RTjpeg_set_quality(d, &q);
    ref_RTjpeg_get_tables(d, out);
    ref_RTjpeg_close(d);
}

/* Decode one packet on a decoder that was given raw tables via set_tables
 * first (the NUV 'D'/'R' extradata path, SURVEY.md section 8a7). */
void refdrv_decode_with_tables(const uint32_t raw[128], const uint8_t *pkt, int w, int h,
                               uint8_t *planes_inout)
{
    size_t ysz = (size_t)w * h;
    uint8_t *pl[3] = { planes_inout, planes_inout + ysz, planes_inout + ysz * 5 / 4 };
    RTjpeg_t *d = ref_RTjpeg_init();
    uint32_t tmp[128];
    memcpy(tmp, raw, sizeof(tmp));
    int ww = w, hh = h;
    ref_RTjpeg_set_size(d, &ww, &hh);
    ref_RTjpeg_set_tables(d, tmp);
    /* quality byte of the packet must equal the decoder's Q (0 on a fresh
     * instance) or decompress re-derives tables from it (:3575-3579) */
    ref_RTjpeg_decompress(d, (uint8_t *)pkt, pl);
    ref_RTjpeg_close(d);
}

/* ------------------------------------------------------------------ */
/* the other two formats (YUV422, 8-bit grey)                          */
/* ------------------------------------------------------------------ */

static size_t fmt_frame_bytes(int fmt, int w, int h)
{
    return fmt == 0 ? (size_t)w * h * 3 / 2 : fmt == 1 ? (size_t)w * h * 2 : (size_t)w * h;
}

static void fmt_planes(int fmt, int w, int h, uint8_t *base, uint8_t *pl[3])
{
    size_t ysz = (size_t)w * h, csz = fmt == 0 ? ysz / 4 : fmt == 1 ? ysz / 2 : 0;
    pl[0] = base;
    pl[1] = base + ysz;
    pl[2] = base + ysz + csz;
}

/* Encode caller-supplied frames (tight planes of format fmt) with one reference encoder. */
size_t refdrv_encode_frames_fmt(const refdrv_clip *c, int fmt, const uint8_t *frames, int F,
                                uint8_t *out, size_t cap, uint64_t *offsets, int align)
{
    RTjpeg_t *e = ref_RTjpeg_init();
    int f0 = fmt, w = c->w, h = c->h, q = c->Q;
    ref_RTjpeg_set_format(e, &f0);
    ref_RTjpeg_set_size(e, &w, &h);
    ref_RTjpeg_set_quality(e, &q);
    if (c->key_rate >= 0) {
        int k = c->key_rate, lm = c->lm, cm = c->cm;
        ref_RTjpeg_set_intra(e, &k, &lm, &cm);
    }
    size_t fsz = fmt_frame_bytes(fmt, c->w, c->h), at = 0;
    size_t bound = 12 + (size_t)(c->w / 8) * (c->h / 8) * 2 * 64 + 64;
    uint8_t *tmp = (uint8_t *)malloc(bound);
    for (int f = 0; f < F; f++) {
        uint8_t *pl[3];
        fmt_planes(fmt, c->w, c->h, (uint8_t *)frames + fsz * f, pl);
        int n = ref_RTjpeg_compress(e, tmp, pl);
        at = (at + (size_t)align - 1) / (size_t)align * (size_t)align;
        if (at + (size_t)n > cap) { free(tmp); ref_RTjpeg_close(e); return 0; }
        memcpy(out + at, tmp, (size_t)n);
        offsets[f] = at;
        at += (size_t)n;
    }
    offsets[F] = at;
    free(tmp);
    ref_RTjpeg_close(e);
    return at;
}

/* Sequential reference decode in format fmt into one persistent plane set. */
void refdrv_decode_seq_fmt(const uint8_t *stream, const uint64_t *offsets, int F, int w, int h, int fmt,
                           const uint8_t *init, uint8_t *frames_out, uint8_t *last_out)
{
    size_t fsz = fmt_frame_bytes(fmt, w, h);
    uint8_t *pl_mem = (uint8_t *)malloc(fsz);
    if (init) memcpy(pl_mem, init, fsz); else memset(pl_mem, 0, fsz);
    uint8_t *pl[3];
    fmt_planes(fmt, w, h, pl_mem, pl);
    RTjpeg_t *d = ref_RTjpeg_init();
    int f0 = fmt;
    ref_RTjpeg_set_format(d, &f0);
    for (int f = 0; f < F; f++) {
        ref_RTjpeg_decompress(d, (uint8_t *)stream + offsets[f], pl);
        if (frames_out) memcpy(frames_out + fsz * f, pl_mem, fsz);
    }
    if (last_out) memcpy(last_out, pl_mem, fsz);
    ref_RTjpeg_close(d);
    free(pl_mem);
}

/* ------------------------------------------------------------------ */
/* colour converters                                                   */
/* ------------------------------------------------------------------ */

extern void ref_RTjpeg_yuv420rgb32(RTjpeg_t *, uint8_t **, uint8_t **);
extern void ref_RTjpeg_yuv420bgr32(RTjpeg_t *, uint8_t **, uint8_t **);
extern void ref_RTjpeg_yuv420rgb24(RTjpeg_t *, uint8_t **, uint8_t **);
extern void ref_RTjpeg_yuv420bgr24(RTjpeg_t *, uint8_t **, uint8_t **);
extern void ref_RTjpeg_yuv420rgb16(RTjpeg_t *, uint8_t **, uint8_t **);
extern void ref_RTjpeg_yuv420rgb8(RTjpeg_t *, uint8_t **, uint8_t **);
extern void ref_RTjpeg_yuv422rgb24(RTjpeg_t *, uint8_t **, uint8_t **);

/* The reference's converter `kind` (numbered as in rtjpeg_oracle.c) over one picture given as tight planes
 * y, u, v; picture row r goes to out + r * pitch. */
void refdrv_convert(int kind, int w, int h, const uint8_t *y, const uint8_t *u, const uint8_t *v,
                    uint8_t *out, size_t pitch)
{
    RTjpeg_t *d = ref_RTjpeg_init();
    int ww = w, hh = h;
    ref_RTjpeg_set_size(d, &ww, &hh);
    uint8_t *pl[3] = {(uint8_t *)y, (uint8_t *)u, (uint8_t *)v};
    uint8_t **rows = (uint8_t **)malloc(sizeof(uint8_t *) * (size_t)h);
    for (int r = 0; r < h; r++) rows[r] = out + (size_t)r * pitch;
    switch (kind) {
    case 0: ref_RTjpeg_yuv420rgb32(d, pl, rows); break;
    case 1: ref_RTjpeg_yuv420bgr32(d, pl, rows); break;
    case 2: ref_RTjpeg_yuv420rgb24(d, pl, rows); break;
    case 3: ref_RTjpeg_yuv420bgr24(d, pl, rows); break;
    case 4: ref_RTjpeg_yuv420rgb16(d, pl, rows); break;
    case 5: ref_RTjpeg_yuv420rgb8(d, pl, rows); break;
    case 6: ref_RTjpeg_yuv422rgb24(d, pl, rows); break;
    default: break;
    }
    free(rows);
    ref_RTjpeg_close(d);
}
