/*
 * rtjo_driver.c -- TEST INFRASTRUCTURE ONLY.
 *
 * What tests/, smoke() and bench.py need around the restatement (rtjpeg_oracle.c) to stand on their own,
 * without the reference's sources:
 *   - the seeded synthetic YUV420 source (SURVEY.md section 8d, configs 2-4),
 *   - stream production with the restated RTjpeg_compress, several encoders at once,
 *   - threaded decode with the restated RTjpeg_decompress for the large parity checks.
 * The restatement is pinned to the reference's own packets and pictures by tests/golden/ (test_encode.py,
 * test_oracle.py), so the streams made here are the ones the reference's encoder makes from the same source.
 */
#define _GNU_SOURCE
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "rtjpeg_oracle.h"

/* ------------------------------------------------------------------ */
/* synthetic source                                                    */
/* ------------------------------------------------------------------ */

static inline uint32_t xs32(uint32_t *s)
{
    uint32_t x = *s;
    x ^= x << 13; x ^= x >> 17; x ^= x << 5;
    return *s = x;
}

static inline uint8_t clip_video(int v) { return (uint8_t)(v < 16 ? 16 : (v > 235 ? 235 : v)); }

/*
 * Frame t of the synthetic clip into tight planes (Y w*h, U and V (w/2)*(h/2)).
 *   Y = 128 + 60 sin((x+3t) 0.05) cos(y 0.07) + checker(40 px, +-25, phase flips
 *       every 8 frames) + uniform noise in [-noise_y, +noise_y]
 *   U,V = smooth sinusoids around 128 (+ uniform noise in [-noise_c, +noise_c])
 * dark != 0 additionally paints the left third flat Y=16 (adversarial case:
 * "key" frames that still contain skip markers, SURVEY.md section 0-5).
 */
void rtjo_synth_frame(int w, int h, int t, uint32_t seed, int noise_y, int noise_c,
                      int dark, uint8_t *y, uint8_t *u, uint8_t *v)
{
    uint32_t rng = seed * 2654435761u + (uint32_t)t * 40503u + 1u;
    if (!rng) rng = 1;
    float *sx = (float *)malloc(sizeof(float) * (size_t)w);
    for (int x = 0; x < w; x++) sx[x] = sinf((float)(x + 3 * t) * 0.05f);
    int flip = (t >> 3) & 1;
    for (int yy = 0; yy < h; yy++) {
        float cy = 60.0f * cosf((float)yy * 0.07f);
        for (int x = 0; x < w; x++) {
            int chk = (((x / 40) + (yy / 40) + flip) & 1) ? 25 : -25;
            int n = noise_y ? (int)(xs32(&rng) % (uint32_t)(2 * noise_y + 1)) - noise_y : 0;
            int val = 128 + (int)lrintf(sx[x] * cy) + chk + n;
            if (dark && x < w / 3) val = 16;
            y[(size_t)yy * w + x] = clip_video(val);
        }
    }
    int cw = w / 2, ch = h / 2;
    for (int yy = 0; yy < ch; yy++) {
        for (int x = 0; x < cw; x++) {
            int nu = noise_c ? (int)(xs32(&rng) % (uint32_t)(2 * noise_c + 1)) - noise_c : 0;
            int nv = noise_c ? (int)(xs32(&rng) % (uint32_t)(2 * noise_c + 1)) - noise_c : 0;
            int uu = 128 + (int)lrintf(40.0f * sinf((float)(x + t) * 0.03f) * cosf((float)yy * 0.02f)) + nu;
            int vv = 128 + (int)lrintf(40.0f * cosf((float)(x - 2 * t) * 0.025f) * sinf((float)yy * 0.035f)) + nv;
            u[(size_t)yy * cw + x] = clip_video(uu);
            v[(size_t)yy * cw + x] = clip_video(vv);
        }
    }
    free(sx);
}

/* ------------------------------------------------------------------ */
/* encode                                                              */
/* ------------------------------------------------------------------ */

/* A synthetic clip and the settings of the encoder that codes it (mirrored by oracle.py's Clip). */
typedef struct {
    int w, h, Q, key_rate, lm, cm;      /* key_rate <= 0: every block coded (RTjpeg_set_intra never called) */
    int noise_y, noise_c, dark;
    uint32_t seed;
} rtjo_clip;

/* worst-case packet: header + 64 bytes per block */
size_t rtjo_packet_bound(int w, int h) { return 12 + (size_t)(w / 16) * (h / 16) * 6 * 64 + 64; }

typedef struct {
    const rtjo_clip *c;
    int f0, f1;                 /* synthetic frame index range */
    uint8_t **pkts;             /* per-frame malloc'd packets */
    uint32_t *sizes;
} enc_job;

static void *enc_worker(void *arg)
{
    enc_job *j = (enc_job *)arg;
    const rtjo_clip *c = j->c;
    rtjo_encoder e;
    rtjo_encoder_init(&e, 0, c->w, c->h, c->Q, c->key_rate, c->lm, c->cm);
    size_t ysz = (size_t)c->w * c->h;
    uint8_t *frame = (uint8_t *)malloc(ysz * 3 / 2);
    uint8_t *tmp = (uint8_t *)malloc(rtjo_packet_bound(c->w, c->h));
    uint8_t *pl[3] = { frame, frame + ysz, frame + ysz * 5 / 4 };
    for (int f = j->f0; f < j->f1; f++) {
        rtjo_synth_frame(c->w, c->h, f, c->seed, c->noise_y, c->noise_c, c->dark, pl[0], pl[1], pl[2]);
        long n = rtjo_encode_frame(&e, pl[0], pl[1], pl[2], tmp);
        j->pkts[f] = (uint8_t *)malloc((size_t)n);
        memcpy(j->pkts[f], tmp, (size_t)n);
        j->sizes[f] = (uint32_t)n;
    }
    free(tmp); free(frame);
    rtjo_encoder_free(&e);
    return NULL;
}

/*
 * Synthesize + encode F frames of the clip with `threads` workers.  Each worker owns a private encoder and a
 * contiguous frame range that starts on a GOP boundary (multiple of key_rate+1), so the result is byte-identical
 * to a single sequential encoder (the encoder zeroes its blocks at every key frame and holds no other inter-frame
 * state).  Packets are written back to back into out (each start rounded up to `align` bytes), offsets[F+1]
 * receives their starts (offsets[F] = end of the last one, unaligned).  Returns bytes used, or 0 if cap is too small.
 */
size_t rtjo_encode_clip(const rtjo_clip *c, int F, int threads, uint8_t *out, size_t cap, uint64_t *offsets, int align)
{
    if (threads < 1) threads = 1;
    int gop = c->key_rate > 0 ? c->key_rate + 1 : 1;
    int ngop = (F + gop - 1) / gop;
    if (threads > ngop) threads = ngop;
    uint8_t **pkts = (uint8_t **)calloc((size_t)F, sizeof(uint8_t *));
    uint32_t *sizes = (uint32_t *)calloc((size_t)F, sizeof(uint32_t));
    enc_job *jobs = (enc_job *)calloc((size_t)threads, sizeof(enc_job));
    pthread_t *th = (pthread_t *)calloc((size_t)threads, sizeof(pthread_t));
    for (int i = 0; i < threads; i++) {
        int g0 = (int)((long)ngop * i / threads), g1 = (int)((long)ngop * (i + 1) / threads);
        jobs[i].c = c; jobs[i].f0 = g0 * gop; jobs[i].f1 = g1 * gop > F ? F : g1 * gop;
        jobs[i].pkts = pkts; jobs[i].sizes = sizes;
        pthread_create(&th[i], NULL, enc_worker, &jobs[i]);
    }
    for (int i = 0; i < threads; i++) pthread_join(th[i], NULL);
    size_t at = 0;
    int ok = 1;
    for (int f = 0; f < F; f++) {
        at = (at + (size_t)align - 1) / (size_t)align * (size_t)align;
        if (ok && at + sizes[f] <= cap) memcpy(out + at, pkts[f], sizes[f]); else ok = 0;
        offsets[f] = at;
        at += sizes[f];
        free(pkts[f]);
    }
    offsets[F] = at;
    free(pkts); free(sizes); free(jobs); free(th);
    return ok ? at : 0;
}

/* ------------------------------------------------------------------ */
/* decode                                                              */
/* ------------------------------------------------------------------ */

typedef struct {
    const uint8_t *stream;
    const uint64_t *offsets;
    const int *seg;             /* segment start frame indices, nseg+1 entries */
    int s0, s1;                 /* segment range owned by this worker */
    int w, h;
    uint8_t *frames_out;
    int zero_init;              /* clear the planes at every segment start */
    const uint32_t *raw;        /* NULL, or 128 raw tables in force before the first packet (RTjpeg_set_tables) */
    int err;
} dec_job;

static void *dec_worker(void *arg)
{
    dec_job *j = (dec_job *)arg;
    size_t ysz = (size_t)j->w * j->h, fsz = ysz * 3 / 2;
    uint8_t *pl = (uint8_t *)malloc(fsz);
    rtjo_decoder d;
    rtjo_decoder_reset(&d);
    if (j->raw) {
        /* they stay in force while the packets' quality byte equals the decoder's Q, 0 on a fresh instance */
        d.width = j->w; d.height = j->h; d.Q = 0;
        rtjo_tables_from_raw(j->raw, &d.t);
    }
    for (int s = j->s0; s < j->s1; s++) {
        if (j->zero_init || s == j->s0) memset(pl, 0, fsz);
        for (int f = j->seg[s]; f < j->seg[s + 1]; f++) {
            const uint8_t *pkt = j->stream + j->offsets[f];
            if (rtjo_decode_packet(&d, pkt, (size_t)(j->offsets[f + 1] - j->offsets[f]), pl, pl + ysz, pl + ysz * 5 / 4) < 0)
                j->err = 1;
            memcpy(j->frames_out + fsz * f, pl, fsz);
        }
    }
    free(pl);
    return NULL;
}

/*
 * Restated decode of independent frame ranges (segments: seg[0..nseg], frame seg[s] starts segment s) on `threads`
 * workers, each with a private decoder and plane set; every segment starts from zeroed planes when zero_init, else
 * only a worker's first one does.  frames_out receives w*h*3/2 bytes per frame.  Returns -1 if a packet was
 * truncated, else 0.
 */
int rtjo_decode_threaded(const uint8_t *stream, const uint64_t *offsets, const int *seg, int nseg, int w, int h,
                         int threads, int zero_init, uint8_t *frames_out, const uint32_t *raw)
{
    if (threads < 1) threads = 1;
    if (threads > nseg) threads = nseg;
    if (threads < 1) return 0;
    dec_job *jobs = (dec_job *)calloc((size_t)threads, sizeof(dec_job));
    pthread_t *th = (pthread_t *)calloc((size_t)threads, sizeof(pthread_t));
    int F = seg[nseg], s = 0, err = 0;
    for (int i = 0; i < threads; i++) {           /* balance by frame count */
        long want = (long)F * (i + 1) / threads;
        int e = s;
        while (e < nseg && seg[e + 1] <= want) e++;
        if (i == threads - 1) e = nseg;
        jobs[i] = (dec_job){ stream, offsets, seg, s, e, w, h, frames_out, zero_init, raw, 0 };
        s = e;
        pthread_create(&th[i], NULL, dec_worker, &jobs[i]);
    }
    for (int i = 0; i < threads; i++) {
        pthread_join(th[i], NULL);
        err |= jobs[i].err;
    }
    free(jobs); free(th);
    return err ? -1 : 0;
}
