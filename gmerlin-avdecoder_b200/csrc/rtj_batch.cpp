/*
 * rtj_batch.cpp -- batch context of the B200 RTjpeg decoder (Level 2 of
 * include/rtjpeg_b200.h): device tables, workspaces, the device-resident
 * decode and the pinned-memory host pipeline.
 *
 * Host-side counterpart of what RTjpeg_decompress (lib/RTjpeg.c:3565-3586)
 * does before it starts walking blocks: header parse and lazy size / quality
 * reconfiguration -- done here once per batch on the CPU (rtjgpu_plan), the
 * block work itself runs in rtj_kernels.cu.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "rtj_common.h"

namespace {

/* An owning, grow-only buffer of T in device memory (cudaMalloc) or pinned host memory (cudaMallocHost).  reserve(n)
 * keeps what it holds when that has room for n elements; otherwise it frees it BEFORE it allocates -- a workspace can be
 * gigabytes, and holding the old and the new one at once would double the peak while it grows -- and keeps nothing of
 * the old contents.  The frees are the synchronous ones: they wait for work still in flight on the memory
 * (rtjgpu_seqenc_destroy relies on that). */
template <typename T, bool PINNED = false>
class Buf {
public:
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    ~Buf() { release(); }

    T *get() const { return p_; }
    size_t cap() const { return cap_; }          /* elements */

    [[nodiscard]] cudaError_t reserve(size_t n)
    {
        if (n <= cap_) return cudaSuccess;
        release();
        void *p = nullptr;
        const cudaError_t e = PINNED ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
        if (e != cudaSuccess) return e;
        p_ = static_cast<T *>(p);
        cap_ = n;
        return cudaSuccess;
    }
    /* reserve() of memory the caller can do without: a failed allocation is no error and leaves the buffer empty */
    [[nodiscard]] bool try_reserve(size_t n)
    {
        if (reserve(n) == cudaSuccess) return true;
        cudaGetLastError();
        return false;
    }
    void release()
    {
        if (p_) {
            if (PINNED) cudaFreeHost(p_);
            else cudaFree(p_);
        }
        p_ = nullptr;
        cap_ = 0;
    }

private:
    T     *p_ = nullptr;
    size_t cap_ = 0;
};

template <typename T> using PinnedBuf = Buf<T, true>;

struct Workspace {
    Buf<uint32_t>     d_ent;                 /* [F][nblk] */
    Buf<uint16_t>     d_src;                 /* [F][nblk] */
    Buf<uint32_t>     d_hardq;               /* [F][nblk][2] */
    Buf<uint16_t>     d_chunk;               /* K3's notes: chunk_mask(), chunk_last() */
    Buf<uint8_t>      d_k3;                  /* K3's hand-over: k3_carry(), k3_count(), laid out for k3_nblk positions */
    int               k3_nblk = 0;
    Buf<int2>         d_walk;                /* [F]: where every frame's walker stands between slices */
    Buf<uint32_t>     d_skips;               /* frame_skips(), redo() */
    Buf<rtj_dev_info> d_info;
    /* segment-parallel scan */
    Buf<uint32_t>     d_seg_sum, d_seg_entry, d_seg_base;
    Buf<int32_t>      d_seg_nbf;
    Buf<uint8_t>      d_seg_del;
    Buf<uint32_t>     d_seg_gsum, d_seg_gentry, d_seg_gbase;
    /* K2's position table, rebuilt when the geometry changes */
    Buf<uint8_t>      d_lut;
    int               lut_fmt = -1, lut_w = 0, lut_h = 0;
    /* the sequence layout of a batch of several sequences (seq_upload) */
    Buf<uint8_t>      d_seq;

    /* K3's per-chunk notes: a 32-bit skip mask and a 16-bit last writer per (chunk of frames, position), the masks first */
    static size_t chunk_words(size_t nchunk) { return 3 * nchunk; }
    uint32_t *chunk_mask() const { return reinterpret_cast<uint32_t *>(d_chunk.get()); }
    uint16_t *chunk_last() const { return d_chunk.get() + d_chunk.cap() / 3 * 2; }
    /* [2][nblk] last writers handed from slice to slice, and behind them K3's arrival counters, one per 128 positions
     * (zero between launches: the last arrival resets its own) */
    static size_t k3_carry_bytes(size_t nblk) { return (2 * nblk * sizeof(uint16_t) + 15) & ~(size_t)15; }
    static size_t k3_count_bytes(size_t nblk) { return (nblk / 128 + 1) * sizeof(uint32_t); }
    uint16_t *k3_carry() const { return reinterpret_cast<uint16_t *>(d_k3.get()); }
    uint32_t *k3_count() const { return reinterpret_cast<uint32_t *>(d_k3.get() + k3_carry_bytes(k3_nblk)); }
    /* [F] skipped blocks of every frame, and behind them [F] K1's hand-over flags */
    uint32_t *frame_skips() const { return d_skips.get(); }
    uint32_t *redo() const { return d_skips.get() + d_skips.cap() / 2; }
};

constexpr int HOST_SLOTS = 3;
constexpr int TIMING_RING = 256;

/* The two streams a large device batch is worked through on (run_kernels): K1 slice by slice on `scan`,
 * K3 / K2 of every slice behind it on `idct`, forked from and joined to the caller's stream with events. */
struct Pipeline {
    cudaStream_t scan = nullptr, idct = nullptr;
    cudaEvent_t  fork = nullptr, join = nullptr;
    cudaEvent_t  scanned[RTJ_MAX_SLICES] = {};
    bool         ready = false;
};

struct HostSlot {
    cudaStream_t       stream = nullptr;
    cudaEvent_t        decoded = nullptr;     /* kernels of the chunk in this slot have finished */
    Workspace          ws;
    Buf<uint8_t>       d_in, d_out;
    Buf<rtjgpu_frame_desc> d_desc;
    PinnedBuf<uint8_t> h_in, h_out;
    PinnedBuf<rtjgpu_frame_desc> h_desc;
    PinnedBuf<rtj_dev_info> h_info;           /* read-back of the chunk's counters */
    /* pending drain of h_out into the caller's memory */
    uint8_t           *pending_dst = nullptr;
    size_t             pending_bytes = 0;
    bool               busy = false;
};

} // namespace

struct rtjgpu_ctx {
    int            device = 0;
    int            last_cuda = 0;
    Buf<rtj_dev_table> d_tables;
    rtj_host_table h_tables[RTJ_NUM_TABLES];
    Workspace      ws;                        /* rtjgpu_decode_device */
    PinnedBuf<rtj_dev_info> h_info_reset;     /* template {0,0,0,-1} */
    PinnedBuf<rtj_dev_info> h_info;           /* read-back */
    int            last_F = 0;
    void          *last_stream = nullptr;
    bool           timing = false;
    cudaEvent_t    ev[TIMING_RING][4] = {};   /* stage brackets of the last TIMING_RING device batches */
    uint64_t       timed_calls = 0;
    uint64_t       launches = 0;
    HostSlot       slot[HOST_SLOTS];
    bool           slots_ready = false;
    Buf<uint8_t>   d_host_carry;              /* carry plane of the host pipeline */
    int            scan_mode = RTJGPU_SCAN_AUTO;
    int            format = RTJ_YUV420;
    Pipeline       pipe;
    int            pipeline_mode = RTJGPU_PIPELINE_AUTO;
    int            slice_frames = 1184, slice0_frames = 1184;   /* multiples of RTJ_RESOLVE_T */
    bool           scan_priority = false;
    int            frame_run = 0;             /* rtjgpu_set_frame_runs: 0 = by the batch before, 1 = off, n = forced */
    PinnedBuf<unsigned long long> h_skips_seen;    /* [3] skipped blocks, raw-prefix frames of the last batch whose K3 has run; raw-prefix frames
                                                    * the self-synchronising walk gave up when it was last tried */
    bool           slices_forced = false;     /* rtjgpu_set_pipeline / the environment gave a slice size: it holds in either arrangement */
    /* encoder: configuration, state between calls, workspace */
    int            enc_quality = 0, enc_lb8 = 0, enc_cb8 = 0;
    int            enc_key_rate = 0, enc_key_count = 0, enc_lm = 0, enc_cm = 0;
    bool           enc_clear_old = true;
    int            enc_w = 0, enc_h = 0, enc_fmt = -1;
    Buf<int32_t>   d_enc_qt;                  /* [128] */
    Buf<int16_t>   d_enc_old;                 /* [nblk][64] */
    Buf<uint8_t>   d_enc_slots, d_enc_lens;   /* [F][nblk][64], [F][nblk] */
    Buf<uint32_t>  d_enc_boff, d_enc_fsize;   /* [F][nblk], [F] */
    Buf<uint64_t>  d_enc_total;               /* [2] */
    PinnedBuf<uint64_t> h_enc_total;          /* [2] */
    void          *enc_stream = nullptr;
    /* rtjgpu_encode_device_seq: the multipliers of every quality (row 0: the zero tables of a fresh instance), made at the
     * first rtjgpu_seqenc_create; the run table, sequence records and frame words of a call (device copy) */
    Buf<int32_t>   d_enc_qt_all;
    int            enc_lb8_all[256] = {}, enc_cb8_all[256] = {};
    Buf<uint8_t>   d_enc_seq;
    uint64_t       enc_seq_calls = 0;         /* stamps the handles of a call: one seen twice is a duplicate */
    std::vector<rtj_enc_run> enc_runs;        /* host scratch of a call */
    uint64_t       host_bad = 0;              /* overrun frames seen by the current rtjgpu_decode_host call */
    PinnedBuf<uint32_t> h_host_skips;         /* per-frame skip counts of that call */
    int            host_F = 0;
    /* pinned staging of the sequence layouts of rtjgpu_decode_device[_rgb]_seq: two buffers taken in turn, each reused only
     * when its last copy to the device is done */
    PinnedBuf<uint8_t> h_seq[2];
    cudaEvent_t    seq_copied[2] = {};
    bool           seq_pending[2] = {};
    int            seq_turn = 0;
    std::vector<uint32_t> sel_jobs;           /* host scratch of rtjgpu_decode_device[_rgb]_select: K2's job list (RTJ_JOB) */
    std::vector<uint32_t> win_words;          /* host scratch of rtjgpu_decode_device[_rgb]_window: [S] RTJ_WIN origins, then
                                               * the jobs of the sequences' last frames (RTJ_JOB(frame, sequence)) */
};

namespace {

#define CK(ctx, call)                                             \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) {                                 \
            (ctx)->last_cuda = (int)e__;                          \
            return RTJGPU_E_CUDA;                                 \
        }                                                         \
    } while (0)

int ws_reserve(rtjgpu_ctx *ctx, Workspace *ws, int F, int nblk)
{
    const size_t need = (size_t)F * (size_t)nblk;
    CK(ctx, ws->d_ent.reserve(need));
    CK(ctx, ws->d_src.reserve(need));
    CK(ctx, ws->d_hardq.reserve(2 * need));          /* two words an entry: destination and source block */
    /* (sized on their own: few frames of a large picture need more of these than many frames of a small one) */
    CK(ctx, ws->d_chunk.reserve(Workspace::chunk_words(((size_t)F / RTJ_RESOLVE_T + 1) * (size_t)nblk)));
    if (nblk > ws->k3_nblk) {                       /* a new layout: allocated afresh, its counters zeroed */
        ws->d_k3.release();
        ws->k3_nblk = 0;
        const size_t carry = Workspace::k3_carry_bytes(nblk), count = Workspace::k3_count_bytes(nblk);
        CK(ctx, ws->d_k3.reserve(carry + count));
        CK(ctx, cudaMemset(ws->d_k3.get() + carry, 0, count));
        ws->k3_nblk = nblk;
    }
    CK(ctx, ws->d_skips.reserve(2 * (size_t)F));
    CK(ctx, ws->d_walk.reserve((size_t)F));
    CK(ctx, ws->d_info.reserve(1));
    return RTJGPU_OK;
}

/* Workspace of the segment-parallel scan, when the batch qualifies: forced by the scan mode, or AUTO
 * with a batch too small to fill the device with one CTA per frame.  Fills *sp (sum == NULL: not used). */
/* AUTO's choice between one CTA per frame and the segment-parallel arrangement.  The host knows the batch's geometry, not
 * its payload (packets and descriptors are device memory): a block of ordinary material is ~4 bytes.  Measured on a B200
 * (DESIGN.md section 3): one CTA per frame takes ~40 us per 40 KB segment of a frame whatever the batch, until the batch
 * fills the device; the segment-parallel passes take ~55 us + 11 ns per KB of batch.  Frames of one segment (up to about
 * 720x576) are never worth cutting up; large frames are, in small batches (a single 1920x1088 frame: 0.06 against 0.18 ms). */
bool auto_wants_segments(const rtjgpu_ctx *ctx, int F, int nblk)
{
    /* Frames with a raw prefix (quality above 170) are another matter: their kernel walks 4 KB segments at ~25 us each, and
     * a frame is many of them.  Whether a batch holds such frames only the device knows; the batch before is the guide (its
     * count arrives in pinned memory, like the skip count that K2's arrangement goes by). */
    /* (The self-synchronising walk takes such frames at a few us per 40 KB when their streams forget their past -- ordinary
     * material does; noise at a high quality does not, and is what the segment-parallel passes remain for.) */
    const volatile unsigned long long *seen = ctx->h_skips_seen.get();
    if (seen[1]) {
        if (seen[2]) return F <= 256;
        /* measured at a quality of 255 (~9 bytes a block): the walk ~21 us per 40 KB segment of a frame whatever the batch
         * (720x576: 0.067 ms for 1 .. 96 frames; 1920x1088: 0.22 - 0.25 ms for 4 .. 32), the segment-parallel passes
         * ~90 us + 20 ns per KB of batch (720x576: 0.097 / 0.133 / 0.239 ms for 1 / 32 / 96 frames; 1920x1088: 0.123 / 0.370 ms
         * for 4 / 32): segments for a handful of large frames only */
        const double raw_kb = (double)nblk * 9.0 / 1024.0;
        const int raw_nseg = (int)((raw_kb + 39.99) / 40.0);
        return 0.090 + 2.0e-5 * (double)F * raw_kb < 0.021 * (double)raw_nseg;
    }
    const double frame_kb = (double)nblk * 4.0 / 1024.0;
    const int nseg = (int)((frame_kb + 39.99) / 40.0);
    return nseg > 1 && 0.055 + 1.1e-5 * (double)F * frame_kb < 0.040 * (double)nseg;
}
constexpr size_t SEG_MAX_SUM_BYTES = (size_t)1 << 30;
constexpr size_t SEG_MAX_DEL_BYTES = (size_t)2 << 30;

int seg_reserve(rtjgpu_ctx *ctx, Workspace *ws, int F, int nblk, int scan_mode, rtj_seg_plan *sp)
{
    memset(sp, 0, sizeof(*sp));
    if (scan_mode != RTJGPU_SCAN_SEGMENT && !(scan_mode == RTJGPU_SCAN_AUTO && auto_wants_segments(ctx, F, nblk))) return RTJGPU_OK;
    /* a frame needs at most 64 bytes per block */
    const size_t maxseg = ((size_t)nblk * 64 + RTJ_SEG_BYTES_MB - 1) / RTJ_SEG_BYTES_MB + 1;   /* the smaller segment size rules */
    const size_t nseg = (size_t)F * maxseg, nsum = nseg * RTJ_SEG_NE;
    if (nsum * sizeof(uint32_t) > SEG_MAX_SUM_BYTES) return RTJGPU_OK;          /* too big: one CTA per frame instead */
    CK(ctx, ws->d_seg_sum.reserve(nsum));
    CK(ctx, ws->d_seg_entry.reserve(nseg));
    CK(ctx, ws->d_seg_base.reserve(nseg));
    CK(ctx, ws->d_seg_nbf.reserve((size_t)F));
    /* the block lengths of the first pass are kept for the second when that fits (it saves the larger half of the second);
     * no room: the second pass works them out again */
    if (nseg * RTJ_SEG_DEL_BYTES <= SEG_MAX_DEL_BYTES)
        sp->del = ws->d_seg_del.try_reserve(nseg * RTJ_SEG_DEL_BYTES) ? ws->d_seg_del.get() : nullptr;
    if (maxseg >= RTJ_SEG_GROUP_MIN_SEGS) {
        const size_t ngroups = (maxseg + RTJ_SEG_GROUP - 1) / RTJ_SEG_GROUP, ng = (size_t)F * ngroups;
        CK(ctx, ws->d_seg_gsum.reserve(ng * RTJ_SEG_NE));
        CK(ctx, ws->d_seg_gentry.reserve(ng));
        CK(ctx, ws->d_seg_gbase.reserve(ng));
        sp->gsum = ws->d_seg_gsum.get(); sp->gentry = ws->d_seg_gentry.get(); sp->gbase = ws->d_seg_gbase.get();
        sp->ngroups = (int)ngroups;
    }
    sp->sum = ws->d_seg_sum.get(); sp->entry = ws->d_seg_entry.get(); sp->base = ws->d_seg_base.get(); sp->nbf = ws->d_seg_nbf.get();
    sp->maxseg = (int)maxseg;
    return RTJGPU_OK;
}

int pipeline_init(rtjgpu_ctx *ctx)
{
    Pipeline &p = ctx->pipe;
    if (p.ready) return RTJGPU_OK;
    int least = 0, greatest = 0;
    CK(ctx, cudaDeviceGetStreamPriorityRange(&least, &greatest));
    CK(ctx, cudaStreamCreateWithPriority(&p.scan, cudaStreamNonBlocking, ctx->scan_priority ? greatest : least));
    CK(ctx, cudaStreamCreateWithPriority(&p.idct, cudaStreamNonBlocking, least));
    CK(ctx, cudaEventCreateWithFlags(&p.fork, cudaEventDisableTiming));
    CK(ctx, cudaEventCreateWithFlags(&p.join, cudaEventDisableTiming));
    for (int i = 0; i < RTJ_MAX_SLICES; i++) CK(ctx, cudaEventCreateWithFlags(&p.scanned[i], cudaEventDisableTiming));
    p.ready = true;
    return RTJGPU_OK;
}

void pipeline_release(Pipeline *p)
{
    if (p->scan) cudaStreamDestroy(p->scan);
    if (p->idct) cudaStreamDestroy(p->idct);
    if (p->fork) cudaEventDestroy(p->fork);
    if (p->join) cudaEventDestroy(p->join);
    for (int i = 0; i < RTJ_MAX_SLICES; i++) if (p->scanned[i]) cudaEventDestroy(p->scanned[i]);
    *p = Pipeline();
}

/* The slices of a batch: [first[i], first[i + 1]), whole chunks of RTJ_RESOLVE_T frames, at most RTJ_MAX_SLICES. */
int plan_slices(const rtjgpu_ctx *ctx, int F, int *first)
{
    auto up = [](int v) { return (v + RTJ_RESOLVE_T - 1) / RTJ_RESOLVE_T * RTJ_RESOLVE_T; };
    int s0 = up(std::max(ctx->slice0_frames, 1)), sl = up(std::max(ctx->slice_frames, 1));
    /* stage after stage, slices only serve to bound K3's look-back: few and large (two launches each) */
    if (ctx->pipeline_mode != RTJGPU_PIPELINE_SLICED && !ctx->slices_forced) s0 = sl = std::max(sl, 4096);
    if (F > s0 && (F - s0 + sl - 1) / sl + 1 > RTJ_MAX_SLICES) sl = up((F - s0 + RTJ_MAX_SLICES - 2) / (RTJ_MAX_SLICES - 1));
    int n = 0;
    first[0] = 0;
    for (int at = 0; at < F; n++) {
        at = std::min(F, at + (n == 0 ? s0 : sl));
        first[n + 1] = at;
    }
    return n;
}

/* The sequences of a device batch as the caller gave them: host arrays.  first == NULL: rtjgpu_decode_device[_rgb], one
 * sequence whose carry and last_yuv are carries[0] / last_yuv[0]. */
struct SeqIn {
    int                   S = 1;
    const int            *first = nullptr;       /* [S + 1] */
    const uint8_t *const *carries = nullptr;     /* [S], or NULL: zeros */
    uint8_t *const       *last_yuv = nullptr;    /* [S], or NULL */
    const uint8_t *carry(int s) const { return carries ? carries[s] : nullptr; }
    uint8_t *last(int s) const { return last_yuv ? last_yuv[s] : nullptr; }
};

/* A selection of the batch's frames as the caller gave it: n batch frame indices, strictly increasing (host array). */
struct SelIn {
    int        n;
    const int *idx;
};

/* where K2's pixels go when they leave as packed RGB (rtjgpu_decode_device_rgb); the last frames as planes go to the
 * sequences' last_yuv */
struct RgbOut {
    uint8_t *d_rgb;
    size_t   row_pitch, frame_pitch;
    int      kind;
    int      alpha;              /* its low byte */
};

/* A window of the selected frames as the caller gave it: cw x ch pixels at origins[2 s], origins[2 s + 1] of sequence s
 * (host array).  The sequences' last frames leave whole, as planes, to their last_yuv. */
struct WinIn {
    int        cw, ch;
    const int *origins;
};

/* What a device decode is given: the batch, its sequences, which frames it wants and where they go -- planes to d_out, or
 * packed pixels (rgb != NULL), of the whole picture or of a window (win != NULL, with a selection).  rtjgpu_scan_device
 * gives the batch alone. */
struct DecodeCall {
    const uint8_t           *d_stream;
    const rtjgpu_frame_desc *d_desc;
    int                      F, w, h;
    cudaStream_t             stream;
    SeqIn                    q;
    const SelIn             *sel = nullptr;      /* NULL: every frame, at its own index */
    const WinIn             *win = nullptr;
    uint8_t                 *d_out = nullptr;
    const RgbOut            *rgb = nullptr;

    DecodeCall(const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h, void *stream)
        : d_stream(d_stream), d_desc(d_desc), F(F), w(w), h(h), stream((cudaStream_t)stream) {}
};

/* The device copies of a call's tables (seq_upload): the sequence layout (S > 1; all NULL for one sequence: the kernels
 * take the one-stream path), and a selection's K2 jobs, sorted by frame, on the device and on the host (where the slices'
 * ranges of jobs are looked up) */
struct CallDev {
    const uint32_t       *seq = nullptr;         /* [F] RTJ_SEQ(first, index) */
    const uint8_t *const *carries = nullptr;     /* [S] */
    uint8_t *const       *last_yuvs = nullptr;   /* [S] */
    const uint32_t       *d_jobs = nullptr, *h_jobs = nullptr;
    int                   njobs = 0;
    /* a window (the layout goes up for S = 1 too): [S] RTJ_WIN origins, and the jobs of the last-frame launch */
    const uint32_t       *win = nullptr, *d_last_jobs = nullptr;
    int                   nlast = 0;
};

/* What K1 reads of rtj_launch_args, for all frames of c on ws; every other field zero */
rtj_launch_args k1_args(const rtjgpu_ctx *ctx, const Workspace &ws, const DecodeCall &c)
{
    rtj_launch_args a;
    memset(&a, 0, sizeof(a));
    a.d_stream = c.d_stream; a.d_desc = c.d_desc; a.d_tables = ctx->d_tables.get();
    a.F = c.F; a.w = c.w; a.h = c.h;
    a.f0 = 0; a.f1 = c.F;
    a.fmt = ctx->format;
    a.row1 = RTJ_FMT_UNITS_Y(ctx->format, c.h);
    a.raw_expected = ((volatile unsigned long long *)ctx->h_skips_seen.get())[1] != 0;
    a.d_walk = ws.d_walk.get(); a.d_redo = ws.redo();
    a.d_ent = ws.d_ent.get(); a.d_frame_skips = ws.frame_skips(); a.d_info = ws.d_info.get();
    a.scan_mode = ctx->scan_mode;
    return a;
}

/*
 * K1 -> K3 -> K2 -> K2b of call c on workspace ws, with c's tables on the device in dev.  ev != NULL brackets the stages
 * with events.
 *
 * The batch is worked through in slices of frames.  Serial arrangement (small batches, the segment-parallel and the
 * serial scans, RTJGPU_PIPELINE_SERIAL): everything on the caller's stream -- K1 over the batch, K3 slice by slice
 * (its look-back never leaves a slice), K2 over the batch.  Pipelined arrangement (allow_pipe, two slices or more):
 * K1 of slice s + 1 runs on a second stream next to K3 / K2 of slice s.  K1 is bound by the ALU pipe and by its
 * barriers, K2 by the FMA pipe: side by side on an SM they fill each other's idle issue slots.  K1's stream has the
 * higher priority, so the CTAs of its next slice (one wave, sized by the slice) take their share of every SM as
 * K2's short-lived CTAs retire.  The last writer of a skipped block lies in an earlier frame, i.e. in a slice
 * that is already scanned, so nothing else has to be ordered.
 */
int run_kernels(rtjgpu_ctx *ctx, Workspace *ws, const DecodeCall &c, const CallDev &dev, cudaEvent_t *ev, bool allow_pipe)
{
    const int F = c.F, nblk = RTJ_FMT_NBLK(ctx->format, c.w, c.h);
    const cudaStream_t st = c.stream;
    const RgbOut *rgb = c.rgb;
    const bool sel = c.sel != nullptr;
    rtj_launch_args a = k1_args(ctx, *ws, c);
    a.d_jobs = dev.d_jobs; a.njobs = dev.njobs;
    /* a selection: jobs [j0, j1) are those of frames [f0, f1) (K2 skips a slice that has none) */
    auto job_range = [&](int f0, int f1) {
        auto at = [&](int f) {
            return (int)(std::partition_point(dev.h_jobs, dev.h_jobs + dev.njobs,
                                              [f](uint32_t j) { return (int)RTJ_JOB_FRAME(j) < f; }) - dev.h_jobs);
        };
        a.j0 = at(f0); a.j1 = at(f1);
    };
    /* K2 works through runs of frames with the strip staying on chip when the stream skips blocks -- which only the device
     * knows for this batch.  The batch before is the guide (its count arrives in pinned memory; a count that is not there yet
     * is the one before it): streams do not change their nature from batch to batch, and either arrangement is exact. */
    a.k2_run = ctx->frame_run ? ctx->frame_run : (*(volatile unsigned long long *)ctx->h_skips_seen.get() ? RTJ_K2_RUN_FRAMES : 1);
    a.h_skips_seen = ctx->h_skips_seen.get();
    a.d_src = ws->d_src.get(); a.d_hardq = ws->d_hardq.get(); a.d_chunk_last = ws->chunk_last(); a.d_chunk_mask = ws->chunk_mask();
    a.d_k3_out = ws->k3_carry(); a.d_k3_count = ws->k3_count();
    a.d_out = c.d_out; a.d_carry = c.q.S > 1 ? nullptr : c.q.carry(0);
    if (rgb) {
        a.fused_rgb = 1;
        a.d_rgb = rgb->d_rgb; a.rgb_row_pitch = rgb->row_pitch; a.rgb_frame_pitch = rgb->frame_pitch;
        a.rgb_kind = rgb->kind; a.rgb_alpha = (unsigned)rgb->alpha & 0xFFu; a.d_last_yuv = c.q.S > 1 ? nullptr : c.q.last(0);
    }
    a.d_seq = dev.seq; a.d_carries = dev.carries; a.d_last_yuvs = dev.last_yuvs;
    /* a window: K2 of the selected frames over the rows of units the windows span; then one launch over the sequences' last
     * frames, whole, to their last_yuv (a window is no carry).  No K2b: the window kernels decode HARD blocks themselves. */
    const WinIn *win = c.win;
    if (win) {
        const int lr = ctx->format == RTJ_YUV420 ? 16 : 8;
        a.d_win = dev.win; a.win_w = win->cw; a.win_h = win->ch; a.win_rows = 0;
        for (int s = 0; s < c.q.S; s++) {
            const int y = win->origins[2 * s + 1];
            a.win_rows = std::max(a.win_rows, (y + win->ch - 1) / lr - y / lr + 1);
        }
    }
    auto last_frames_launch = [&](cudaStream_t s) {
        rtj_launch_args l = a;
        l.d_jobs = dev.d_last_jobs; l.j0 = 0; l.j1 = l.njobs = dev.nlast;
        l.win_w = c.w; l.win_h = c.h; l.win_rows = RTJ_FMT_UNITS_Y(ctx->format, c.h); l.win_last = 1;
        return rtj_launch_idct(&l, s);
    };
    {
        const int rc = seg_reserve(ctx, ws, F, nblk, ctx->scan_mode, &a.seg);
        if (rc) return rc;
    }

    if (ws->lut_fmt != ctx->format || ws->lut_w != c.w || ws->lut_h != c.h) {
        ws->lut_fmt = -1;                           /* until the table of this geometry is built */
        CK(ctx, ws->d_lut.reserve(rtj_lut_bytes(ctx->format, c.w, c.h)));
        const int e0 = rtj_launch_build_lut(ctx->format, c.w, c.h, ws->d_lut.get(), st);
        if (e0) { ctx->last_cuda = e0; return RTJGPU_E_CUDA; }
        ws->lut_fmt = ctx->format; ws->lut_w = c.w; ws->lut_h = c.h;
        ctx->launches += 1;
    }
    a.d_lut = ws->d_lut.get();

    int first[RTJ_MAX_SLICES + 1];
    const int nslices = plan_slices(ctx, F, first);
    const bool chunk_scan = !a.seg.sum && (ctx->scan_mode == RTJGPU_SCAN_AUTO || ctx->scan_mode == RTJGPU_SCAN_CHUNK);
    const bool piped = allow_pipe && chunk_scan && nslices >= 2 && ctx->pipeline_mode == RTJGPU_PIPELINE_SLICED;
    auto slice_args = [&](int i) {
        a.f0 = first[i]; a.f1 = first[i + 1]; a.slice = i;
        a.d_k3_in = i == 0 ? nullptr : ws->k3_carry() + (size_t)(i & 1) * nblk;
        a.d_k3_out = ws->k3_carry() + (size_t)((i + 1) & 1) * nblk;
    };
#define LAUNCHED(call, count)                                                  \
    do {                                                                       \
        const int e__ = (call);                                                \
        if (e__ < 0 || ((count) && e__ > 0)) { ctx->last_cuda = e__ < 0 ? -e__ : e__; return RTJGPU_E_CUDA; } \
        ctx->launches += (count) ? (uint64_t)(count) : (uint64_t)e__;          \
    } while (0)

    CK(ctx, cudaMemcpyAsync(ws->d_info.get(), ctx->h_info_reset.get(), sizeof(rtj_dev_info), cudaMemcpyHostToDevice, st));
    if (ev) CK(ctx, cudaEventRecord(ev[0], st));
    if (!piped) {
        LAUNCHED(rtj_launch_scan(&a, st), 0);                  /* returns its launches */
        if (ev) CK(ctx, cudaEventRecord(ev[1], st));
        for (int i = 0; i < nslices; i++) {
            slice_args(i);                                      /* (the one scan over the batch counted its skips as slice 0) */
            LAUNCHED(rtj_launch_resolve(&a, st), 2);
        }
        a.f0 = 0; a.f1 = F;
        if (ev) CK(ctx, cudaEventRecord(ev[2], st));
        if (sel) job_range(0, F);
        if (!sel || a.j1 > a.j0) {                              /* (an empty selection: K1 and K3 only) */
            LAUNCHED(rtj_launch_idct(&a, st), 1);
            if (!rgb && !win) LAUNCHED(rtj_launch_idct_hard(&a, st), 2);
        }
        if (win && dev.nlast) LAUNCHED(last_frames_launch(st), 1);
        if (ev) CK(ctx, cudaEventRecord(ev[3], st));
        return RTJGPU_OK;
    }

    {
        const int rc = pipeline_init(ctx);
        if (rc) return rc;
    }
    Pipeline &p = ctx->pipe;
    CK(ctx, cudaEventRecord(p.fork, st));
    CK(ctx, cudaStreamWaitEvent(p.scan, p.fork, 0));
    CK(ctx, cudaStreamWaitEvent(p.idct, p.fork, 0));
    for (int i = 0; i < nslices; i++) {
        slice_args(i);
        LAUNCHED(rtj_launch_scan(&a, p.scan), 0);
        CK(ctx, cudaEventRecord(p.scanned[i], p.scan));
        CK(ctx, cudaStreamWaitEvent(p.idct, p.scanned[i], 0));
        LAUNCHED(rtj_launch_resolve(&a, p.idct), 2);
        if (sel) job_range(first[i], first[i + 1]);
        if (!sel || a.j1 > a.j0) LAUNCHED(rtj_launch_idct(&a, p.idct), 1);     /* (a slice without a selected frame: no K2) */
    }
    if (ev) {                                                   /* stages overlap: scan = until the last slice is scanned, idct = the rest */
        CK(ctx, cudaEventRecord(ev[1], p.scan));
        CK(ctx, cudaEventRecord(ev[2], p.scan));
    }
    a.f0 = 0; a.f1 = F;
    if (!rgb && !win && (!sel || dev.njobs > 0)) LAUNCHED(rtj_launch_idct_hard(&a, p.idct), 2);
    if (win && dev.nlast) LAUNCHED(last_frames_launch(p.idct), 1);
    CK(ctx, cudaEventRecord(p.join, p.idct));
    CK(ctx, cudaStreamWaitEvent(st, p.join, 0));
    if (ev) CK(ctx, cudaEventRecord(ev[3], st));
#undef LAUNCHED
    return RTJGPU_OK;
}

inline uint32_t rd_u32le(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
inline uint16_t rd_u16le(const uint8_t *p) { return (uint16_t)(p[0] | p[1] << 8); }

/* The picture sizes the library takes: both sides positive multiples of 16 that fit the header's 16-bit fields */
inline bool valid_size(int w, int h) { return w > 0 && h > 0 && !(w & 15) && !(h & 15) && w <= 65535 && h <= 65535; }

/* The checks of the _seq calls that the one-stream calls do not have. */
int seq_check(int F, const SeqIn &q)
{
    if (q.S < 1 || q.S > F || !q.first || q.first[0] != 0 || q.first[q.S] != F) return RTJGPU_E_ARG;
    for (int s = 0; s < q.S; s++) {
        if (q.first[s + 1] <= q.first[s]) return RTJGPU_E_ARG;              /* no empty sequence */
        if (((uintptr_t)q.carry(s) & 7) || ((uintptr_t)q.last(s) & 15)) return RTJGPU_E_ARG;
    }
    return RTJGPU_OK;
}

/* Small per-call tables go up with cudaMemcpyAsync on the launch stream, staged in one of two pinned buffers taken in
 * turn; a buffer is written again only once its previous copy is done, and the caller's arrays are not read after the
 * call returns.  stage_begin hands out the buffer to fill (bytes of it), stage_end copies it to d_dst. */
int stage_begin(rtjgpu_ctx *ctx, size_t bytes, uint8_t **h)
{
    const int t = ctx->seq_turn;
    if (!ctx->seq_copied[t]) CK(ctx, cudaEventCreateWithFlags(&ctx->seq_copied[t], cudaEventDisableTiming));
    if (ctx->seq_pending[t]) {
        CK(ctx, cudaEventSynchronize(ctx->seq_copied[t]));
        ctx->seq_pending[t] = false;
    }
    CK(ctx, ctx->h_seq[t].reserve(bytes));
    *h = ctx->h_seq[t].get();
    return RTJGPU_OK;
}

int stage_end(rtjgpu_ctx *ctx, void *d_dst, size_t bytes, cudaStream_t st)
{
    const int t = ctx->seq_turn;
    CK(ctx, cudaMemcpyAsync(d_dst, ctx->h_seq[t].get(), bytes, cudaMemcpyHostToDevice, st));
    CK(ctx, cudaEventRecord(ctx->seq_copied[t], st));
    ctx->seq_pending[t] = true;
    ctx->seq_turn = t ^ 1;
    return RTJGPU_OK;
}

/* The device copy of c's layout of S > 1 sequences, in the workspace: [F] RTJ_SEQ words, then [S] carry pointers, then
 * [S] last_yuv pointers -- and behind them, for a selection, its ctx->sel_jobs, and for a window its ctx->win_words: one
 * copy either way.  S = 1 uploads the jobs alone, unless there is a window: the window kernels take every sequence's
 * origin, carry and last_yuv from the layout. */
int seq_upload(rtjgpu_ctx *ctx, Workspace *ws, const DecodeCall &c, CallDev *out)
{
    const SeqIn &q = c.q;
    const bool layout = q.S > 1 || c.win;
    const size_t words = layout ? ((size_t)c.F * sizeof(uint32_t) + 7) & ~(size_t)7 : 0, ptrs = layout ? (size_t)q.S * sizeof(void *) : 0;
    const size_t jbytes = c.sel ? ctx->sel_jobs.size() * sizeof(uint32_t) : 0;
    const size_t wbytes = c.win ? ctx->win_words.size() * sizeof(uint32_t) : 0;
    const size_t bytes = words + 2 * ptrs + jbytes + wbytes;
    uint8_t *h;
    int rc = stage_begin(ctx, bytes, &h);
    if (rc) return rc;
    CK(ctx, ws->d_seq.reserve(bytes));
    if (layout) {
        uint32_t *hw = reinterpret_cast<uint32_t *>(h);
        for (int s = 0; s < q.S; s++)
            for (int f = q.first[s]; f < q.first[s + 1]; f++) hw[f] = RTJ_SEQ(q.first[s], s);
        const uint8_t **hc = reinterpret_cast<const uint8_t **>(h + words);
        uint8_t **hl = reinterpret_cast<uint8_t **>(h + words + ptrs);
        for (int s = 0; s < q.S; s++) { hc[s] = q.carry(s); hl[s] = q.last(s); }
    }
    if (jbytes) memcpy(h + words + 2 * ptrs, ctx->sel_jobs.data(), jbytes);
    if (wbytes) memcpy(h + words + 2 * ptrs + jbytes, ctx->win_words.data(), wbytes);
    const uint8_t *d = ws->d_seq.get();
    if ((rc = stage_end(ctx, ws->d_seq.get(), bytes, c.stream))) return rc;
    if (layout) {
        out->seq = reinterpret_cast<const uint32_t *>(d);
        out->carries = reinterpret_cast<const uint8_t *const *>(d + words);
        out->last_yuvs = reinterpret_cast<uint8_t *const *>(d + words + ptrs);
    }
    if (c.sel) {
        out->d_jobs = reinterpret_cast<const uint32_t *>(d + words + 2 * ptrs);
        out->h_jobs = ctx->sel_jobs.data();
        out->njobs = (int)ctx->sel_jobs.size();
    }
    if (c.win) {
        const uint32_t *wd = reinterpret_cast<const uint32_t *>(d + words + 2 * ptrs + jbytes);
        out->win = wd;
        out->d_last_jobs = wd + q.S;
        out->nlast = (int)ctx->win_words.size() - q.S;
    }
    return RTJGPU_OK;
}

int sel_check(int F, const SelIn &s)
{
    if (s.n < 0 || s.n > F || (s.n > 0 && !s.idx)) return RTJGPU_E_ARG;
    for (int k = 0; k < s.n; k++)
        if (s.idx[k] < 0 || s.idx[k] >= F || (k > 0 && s.idx[k] <= s.idx[k - 1])) return RTJGPU_E_ARG;
    return RTJGPU_OK;
}

/* K2's jobs of a selection (into ctx->sel_jobs), sorted by frame: selected frame sel[k] to slot k; with rgb_last, also every
 * sequence's last frame that is not selected but has a last_yuv, to planes only. */
void sel_jobs(rtjgpu_ctx *ctx, const SeqIn &q, const SelIn &s, bool rgb_last)
{
    std::vector<uint32_t> &jobs = ctx->sel_jobs;
    jobs.clear();
    int k = 0;
    for (int i = 0; i < q.S; i++) {
        const int last = q.first[i + 1] - 1;
        bool last_selected = false;
        for (; k < s.n && s.idx[k] <= last; k++) {
            jobs.push_back(RTJ_JOB(s.idx[k], k));
            last_selected = s.idx[k] == last;
        }
        if (rgb_last && q.last(i) && !last_selected) jobs.push_back(RTJ_JOB(last, RTJ_JOB_NO_SLOT));
    }
}

/* The checks every device call makes once its sequences and selection are known to be consistent (decode()): pointers,
 * alignment, geometry, batch size -- in this order, and before anything is reserved or launched.  Without `output`
 * (rtjgpu_scan_device) the output, carry and last_yuv pointers are not looked at.  Sets the device and *nblk. */
int check_batch(rtjgpu_ctx *ctx, const DecodeCall &c, bool output, int *nblk)
{
    uint8_t *const dst = c.rgb ? c.rgb->d_rgb : c.d_out;
    if (!c.d_stream || !c.d_desc || (output && !dst && !(c.sel && c.sel->n == 0))) return RTJGPU_E_ARG;
    /* K1 reads the stream as 32-bit words, K2 leaves its strips as 16-byte bulk stores and reads the carry as 8-byte rows */
    if (((uintptr_t)c.d_stream & 3) || ((uintptr_t)c.d_desc & 7)) return RTJGPU_E_ARG;
    if (output && (((uintptr_t)dst & 15) || ((uintptr_t)c.q.carry(0) & 7) || ((uintptr_t)c.q.last(0) & 15))) return RTJGPU_E_ARG;
    /* a window: x and cw multiples of 16, y and ch even, inside the picture -- every output row starts 8- or 16-byte aligned
     * and the two luma rows of a chroma row stay together */
    if (output && c.win) {
        const WinIn &v = *c.win;
        if (v.cw <= 0 || v.ch <= 0 || (v.cw & 15) || (v.ch & 1) || !v.origins) return RTJGPU_E_ARG;
        for (int s = 0; s < c.q.S; s++) {
            const int x = v.origins[2 * s], y = v.origins[2 * s + 1];
            if (x < 0 || y < 0 || (x & 15) || (y & 1) || x > c.w - v.cw || y > c.h - v.ch) return RTJGPU_E_ARG;
        }
    }
    if (output && c.rgb) {
        const RgbOut &o = *c.rgb;
        const int ow = c.win ? c.win->cw : c.w, oh = c.win ? c.win->ch : c.h;     /* the picture that leaves */
        if ((o.row_pitch & 15) || (o.frame_pitch & 15) || o.row_pitch < (size_t)ow * rtj_convert_bpp(o.kind)
            || o.frame_pitch < o.row_pitch * (size_t)oh)
            return RTJGPU_E_ARG;
    }
    if (!valid_size(c.w, c.h)) return RTJGPU_E_SIZE;
    if (c.F > RTJGPU_MAX_FRAMES_PER_BATCH) return RTJGPU_E_TOOBIG;
    CK(ctx, cudaSetDevice(ctx->device));
    *nblk = RTJ_FMT_NBLK(ctx->format, c.w, c.h);
    if ((uint64_t)c.F * (uint64_t)*nblk >= (1ull << 32)) return RTJGPU_E_TOOBIG;   /* block indices are 32 bit */
    if ((uint64_t)RTJ_FMT_FRAME_BYTES(ctx->format, c.w, c.h) >= (1ull << 32)) return RTJGPU_E_TOOBIG;   /* and so are offsets inside a frame */
    return RTJGPU_OK;
}

/* Every rtjgpu_decode_device* call: rtjgpu_decode_device is the one-sequence case of rtjgpu_decode_device_seq, which is
 * rtjgpu_decode_device_select selecting every frame; the same three with packed pixels out (c.rgb) */
int decode(rtjgpu_ctx *ctx, DecodeCall c)
{
    if (!ctx || c.F < 0) return RTJGPU_E_ARG;
    if (c.rgb) {
        if (ctx->format != RTJ_YUV420) return RTJGPU_E_FORMAT;                 /* the reference's converters are yuv420 ones */
        const int k = c.rgb->kind;
        if (k != RTJ_CONV_RGB32 && k != RTJ_CONV_BGR32 && k != RTJ_CONV_RGB24 && k != RTJ_CONV_BGR24 && k != RTJ_CONV_RGB16)
            return RTJGPU_E_FORMAT;
    }
    int rc;
    if (c.q.first && (rc = seq_check(c.F, c.q))) return rc;
    if (c.sel) {
        if ((rc = sel_check(c.F, *c.sel))) return rc;
        /* every frame: the full call, runs of frames and last frames as planes included (a window stays a selection) */
        if (c.sel->n == c.F && !c.win) c.sel = nullptr;
    }
    if (c.F == 0) { ctx->last_F = 0; return RTJGPU_OK; }
    int nblk;
    if ((rc = check_batch(ctx, c, true, &nblk))) return rc;
    if ((rc = ws_reserve(ctx, &ctx->ws, c.F, nblk))) return rc;
    CallDev dev;
    if (c.sel) sel_jobs(ctx, c.q, *c.sel, c.rgb != nullptr && !c.win);
    if (c.win) {
        /* the sequences' origins, then the jobs of the last-frame launch: each sequence's last frame that has a last_yuv */
        std::vector<uint32_t> &ww = ctx->win_words;
        ww.clear();
        for (int s = 0; s < c.q.S; s++) ww.push_back(RTJ_WIN(c.win->origins[2 * s], c.win->origins[2 * s + 1]));
        for (int s = 0; s < c.q.S; s++)
            if (c.q.last(s)) ww.push_back(RTJ_JOB(c.q.first[s + 1] - 1, s));
    }
    if ((c.q.S > 1 || c.win || (c.sel && !ctx->sel_jobs.empty())) && (rc = seq_upload(ctx, &ctx->ws, c, &dev))) return rc;
    cudaEvent_t *ev = ctx->timing ? ctx->ev[ctx->timed_calls % TIMING_RING] : nullptr;
    rc = run_kernels(ctx, &ctx->ws, c, dev, ev, true);
    if (ev && rc == RTJGPU_OK) ctx->timed_calls++;
    ctx->last_F = c.F;
    ctx->last_stream = c.stream;
    return rc;
}

/* The encoder's workspace for F pictures of nblk blocks, shared by rtjgpu_encode_device and rtjgpu_encode_device_seq
 * (both on the stream of the call that uses it), and the totals rtjgpu_get_encode_info reads back */
int enc_reserve(rtjgpu_ctx *ctx, size_t nblk, int F)
{
    const size_t nb = nblk * (size_t)F;
    CK(ctx, ctx->d_enc_total.reserve(2));
    CK(ctx, ctx->h_enc_total.reserve(2));
    CK(ctx, ctx->d_enc_slots.reserve(nb * 64));
    CK(ctx, ctx->d_enc_lens.reserve(nb));
    CK(ctx, ctx->d_enc_boff.reserve(nb));
    CK(ctx, ctx->d_enc_fsize.reserve((size_t)F));
    return RTJGPU_OK;
}

} // namespace

extern "C" {

const char *rtjgpu_strerror(int code)
{
    switch (code) {
    case RTJGPU_OK:        return "ok";
    case RTJGPU_E_CUDA:    return "CUDA call failed";
    case RTJGPU_E_ARG:     return "bad argument";
    case RTJGPU_E_HEADER:  return "packet shorter than its header or framesize";
    case RTJGPU_E_SIZE:    return "width/height zero, not a multiple of 16, or changing inside a batch";
    case RTJGPU_E_FORMAT:  return "unknown picture format or converter";
    case RTJGPU_E_OVERRUN: return "block stream runs past the end of its packet";
    case RTJGPU_E_TOOBIG:  return "batch exceeds RTJGPU_MAX_FRAMES_PER_BATCH / RTJGPU_MAX_PAYLOAD_BYTES";
    case RTJGPU_E_NOMEM:   return "out of memory";
    default:               return "unknown error";
    }
}

int rtjgpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int rtjgpu_create(int device, rtjgpu_ctx **out)
{
    if (!out) return RTJGPU_E_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || device < 0 || device >= n) return RTJGPU_E_CUDA;   /* no CPU fallback */
    rtjgpu_ctx *ctx = new (std::nothrow) rtjgpu_ctx();
    if (!ctx) return RTJGPU_E_NOMEM;
    ctx->device = device;
    /* development knobs (tools/): slice sizes of the pipelined arrangement, K1's stream priority */
    if (const char *v = getenv("RTJPEG_B200_SLICE")) { ctx->slice_frames = ctx->slice0_frames = std::max(32, atoi(v)); ctx->slices_forced = true; }
    if (const char *v = getenv("RTJPEG_B200_SLICE0")) ctx->slice0_frames = std::max(32, atoi(v));
    if (const char *v = getenv("RTJPEG_B200_SCAN_PRIO")) ctx->scan_priority = atoi(v) != 0;
    if (const char *v = getenv("RTJPEG_B200_SCAN")) ctx->scan_mode = std::min(std::max(atoi(v), 0), (int)RTJGPU_SCAN_SYNC);
    if (const char *v = getenv("RTJPEG_B200_K2_RUN")) ctx->frame_run = std::min(std::max(atoi(v), 0), 64);
    if (const char *v = getenv("RTJPEG_B200_PIPELINE")) ctx->pipeline_mode = std::min(std::max(atoi(v), 0), (int)RTJGPU_PIPELINE_SLICED);
    int rc = RTJGPU_OK;
    do {
        if ((e = cudaSetDevice(device)) != cudaSuccess) { rc = RTJGPU_E_CUDA; break; }
        if (int k = rtj_kernels_init()) { e = (cudaError_t)k; rc = RTJGPU_E_CUDA; break; }
        /* table 0: never-configured instance (all zero, lb8 = cb8 = 0); 1..255: quality; 256: custom */
        memset(ctx->h_tables, 0, sizeof(ctx->h_tables));
        std::vector<rtj_dev_table> dev(RTJ_NUM_TABLES);
        for (int q = 1; q <= 255; q++) rtj_table_from_quality(q, &ctx->h_tables[q]);
        for (int t = 0; t < RTJ_NUM_TABLES; t++) rtj_table_to_device_layout(&ctx->h_tables[t], &dev[t]);
        if ((e = ctx->d_tables.reserve(RTJ_NUM_TABLES)) != cudaSuccess) { rc = RTJGPU_E_CUDA; break; }
        if ((e = cudaMemcpy(ctx->d_tables.get(), dev.data(), sizeof(rtj_dev_table) * RTJ_NUM_TABLES, cudaMemcpyHostToDevice)) != cudaSuccess) { rc = RTJGPU_E_CUDA; break; }
        if ((e = ctx->h_info_reset.reserve(1)) != cudaSuccess) { rc = RTJGPU_E_CUDA; break; }
        if ((e = ctx->h_info.reserve(1)) != cudaSuccess) { rc = RTJGPU_E_CUDA; break; }
        if ((e = ctx->h_skips_seen.reserve(3)) != cudaSuccess) { rc = RTJGPU_E_CUDA; break; }
        unsigned long long *seen = ctx->h_skips_seen.get();
        seen[0] = seen[1] = seen[2] = 0;
        rtj_dev_info *reset = ctx->h_info_reset.get();
        memset(reset, 0, sizeof(rtj_dev_info));
        reset->first_bad_frame = -1;
        *ctx->h_info.get() = *reset;
        for (int i = 0; i < TIMING_RING * 4 && rc == RTJGPU_OK; i++)
            if ((e = cudaEventCreate(&ctx->ev[i / 4][i % 4])) != cudaSuccess) rc = RTJGPU_E_CUDA;
    } while (0);
    if (rc != RTJGPU_OK) {
        ctx->last_cuda = (int)e;
        rtjgpu_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return RTJGPU_OK;
}

void rtjgpu_destroy(rtjgpu_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    pipeline_release(&ctx->pipe);
    for (HostSlot &s : ctx->slot) {
        if (s.decoded) cudaEventDestroy(s.decoded);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    for (cudaEvent_t e : ctx->seq_copied) if (e) cudaEventDestroy(e);
    for (int i = 0; i < TIMING_RING * 4; i++) if (ctx->ev[i / 4][i % 4]) cudaEventDestroy(ctx->ev[i / 4][i % 4]);
    delete ctx;                                 /* (and with it every buffer it holds) */
}

int rtjgpu_last_cuda_error(const rtjgpu_ctx *ctx) { return ctx ? ctx->last_cuda : 0; }
uint64_t rtjgpu_launch_count(const rtjgpu_ctx *ctx) { return ctx ? ctx->launches : 0; }
void rtjgpu_enable_timing(rtjgpu_ctx *ctx, int on) { if (ctx) ctx->timing = on != 0; }

int rtjgpu_set_scan_mode(rtjgpu_ctx *ctx, int mode)
{
    if (!ctx || mode < RTJGPU_SCAN_AUTO || mode > RTJGPU_SCAN_SYNC) return RTJGPU_E_ARG;
    ctx->scan_mode = mode;
    return RTJGPU_OK;
}

int rtjgpu_set_pipeline(rtjgpu_ctx *ctx, int mode, int slice_frames)
{
    if (!ctx || mode < RTJGPU_PIPELINE_AUTO || mode > RTJGPU_PIPELINE_SLICED || slice_frames < 0) return RTJGPU_E_ARG;
    ctx->pipeline_mode = mode;
    if (slice_frames) {
        ctx->slice_frames = ctx->slice0_frames = (slice_frames + RTJ_RESOLVE_T - 1) / RTJ_RESOLVE_T * RTJ_RESOLVE_T;
        ctx->slices_forced = true;
    }
    return RTJGPU_OK;
}

int rtjgpu_set_frame_runs(rtjgpu_ctx *ctx, int frames)
{
    if (!ctx || frames < 0 || frames > 64) return RTJGPU_E_ARG;
    ctx->frame_run = frames;
    return RTJGPU_OK;
}

int rtjgpu_set_format(rtjgpu_ctx *ctx, int format)
{
    if (!ctx || format < RTJ_YUV420 || format > RTJ_RGB8) return RTJGPU_E_ARG;
    ctx->format = format;
    return RTJGPU_OK;
}

/* ---- encoder ---------------------------------------------------------------------------------------- */

int rtjgpu_encoder_set_quality(rtjgpu_ctx *ctx, int quality)
{
    if (!ctx) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    if (quality < 1) quality = 1;
    if (quality > 255) quality = 255;
    int32_t qt[128];
    rtj_encoder_table_from_quality(quality, qt, &ctx->enc_lb8, &ctx->enc_cb8);
    CK(ctx, ctx->d_enc_qt.reserve(128));
    if (ctx->enc_stream) CK(ctx, cudaStreamSynchronize((cudaStream_t)ctx->enc_stream));   /* a batch may still read the old tables */
    CK(ctx, cudaMemcpy(ctx->d_enc_qt.get(), qt, sizeof(qt), cudaMemcpyHostToDevice));
    ctx->enc_quality = quality;
    return RTJGPU_OK;
}

int rtjgpu_encoder_set_intra(rtjgpu_ctx *ctx, int key_rate, int lm, int cm)
{
    if (!ctx) return RTJGPU_E_ARG;
    ctx->enc_key_rate = key_rate < 0 ? 0 : key_rate > 255 ? 255 : key_rate;
    ctx->enc_lm = lm < 0 ? 0 : lm > 16 ? 16 : lm;
    ctx->enc_cm = cm < 0 ? 0 : cm > 16 ? 16 : cm;
    ctx->enc_clear_old = true;           /* lib/RTjpeg.c:2488: the stored blocks are cleared; the key counter is not touched */
    return RTJGPU_OK;
}

int rtjgpu_encoder_reset(rtjgpu_ctx *ctx)
{
    if (!ctx) return RTJGPU_E_ARG;
    ctx->enc_key_count = 0;
    ctx->enc_clear_old = true;
    return RTJGPU_OK;
}

int rtjgpu_encode_device(rtjgpu_ctx *ctx, const uint8_t *d_frames, int F, int w, int h,
                         uint8_t *d_stream, size_t capacity, uint64_t *d_offsets, void *cuda_stream)
{
    if (!ctx || F < 0) return RTJGPU_E_ARG;
    if (ctx->format != RTJ_YUV420 && ctx->format != RTJ_YUV422) return RTJGPU_E_FORMAT;
    if (!valid_size(w, h)) return RTJGPU_E_SIZE;
    if (F > RTJGPU_MAX_FRAMES_PER_BATCH) return RTJGPU_E_TOOBIG;
    if (!d_offsets || (F && (!d_frames || !d_stream)) || ((uintptr_t)d_frames & 7) || ((uintptr_t)d_stream & 3)) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t nblk = (size_t)RTJ_FMT_NBLK(ctx->format, w, h);
    if (!ctx->d_enc_qt.get()) {          /* never configured: the all-zero tables of a fresh RTjpeg_t (lib/RTjpeg.c:2499) */
        CK(ctx, ctx->d_enc_qt.reserve(128));
        CK(ctx, cudaMemset(ctx->d_enc_qt.get(), 0, 128 * sizeof(int32_t)));
    }
    int rc = enc_reserve(ctx, nblk, F);             /* (F = 0: the totals alone) */
    if (rc) return rc;
    if (ctx->enc_w != w || ctx->enc_h != h || ctx->enc_fmt != ctx->format) {
        ctx->enc_w = w; ctx->enc_h = h; ctx->enc_fmt = ctx->format;
        ctx->enc_clear_old = true;
    }
    CK(ctx, ctx->d_enc_old.reserve(nblk * 64));
    if (ctx->enc_clear_old) {
        CK(ctx, cudaMemsetAsync(ctx->d_enc_old.get(), 0, nblk * 64 * sizeof(int16_t), st));
        ctx->enc_clear_old = false;
    }
    ctx->enc_stream = cuda_stream;
    if (F == 0) {
        CK(ctx, cudaMemsetAsync(d_offsets, 0, sizeof(uint64_t), st));
        CK(ctx, cudaMemsetAsync(ctx->d_enc_total.get(), 0, 2 * sizeof(uint64_t), st));
        return RTJGPU_OK;
    }
    rtj_encode_args a;
    a.d_frames = d_frames; a.F = F; a.w = w; a.h = h; a.fmt = ctx->format;
    a.d_qt = ctx->d_enc_qt.get(); a.lb8 = ctx->enc_lb8; a.cb8 = ctx->enc_cb8; a.quality = ctx->enc_quality;
    a.key_rate = ctx->enc_key_rate; a.key_count0 = ctx->enc_key_count; a.lmask = ctx->enc_lm; a.cmask = ctx->enc_cm;
    a.d_old = ctx->d_enc_old.get(); a.d_slots = ctx->d_enc_slots.get(); a.d_lens = ctx->d_enc_lens.get(); a.d_boff = ctx->d_enc_boff.get();
    a.d_fsize = ctx->d_enc_fsize.get(); a.d_stream = d_stream; a.capacity = capacity; a.d_offsets = d_offsets;
    a.d_total = ctx->d_enc_total.get();
    const int e = rtj_launch_encode(&a, cuda_stream);
    if (e < 0) { ctx->last_cuda = -e; return RTJGPU_E_CUDA; }
    ctx->launches += (uint64_t)e;
    if (ctx->enc_key_rate) ctx->enc_key_count = (ctx->enc_key_count + F) % (ctx->enc_key_rate + 1);
    return RTJGPU_OK;
}

int rtjgpu_get_encode_info(rtjgpu_ctx *ctx, uint64_t *bytes, int *overflow)
{
    if (!ctx || !ctx->d_enc_total.get()) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)ctx->enc_stream;
    const uint64_t *total = ctx->h_enc_total.get();
    CK(ctx, cudaMemcpyAsync(ctx->h_enc_total.get(), ctx->d_enc_total.get(), 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    if (bytes) *bytes = total[0];
    if (overflow) *overflow = total[1] != 0;
    return RTJGPU_OK;
}

/* ---- encoder states of their own: rtjgpu_encode_device_seq ---------------------------------------------- */

struct rtjgpu_seqenc {
    rtjgpu_ctx *ctx = nullptr;
    int         device = 0;                 /* ctx's, kept for rtjgpu_seqenc_destroy */
    int         quality = 0, key_rate = 0, key_count = 0, lm = 0, cm = 0;
    bool        cleared = true;             /* the stored blocks are zeros: a run that starts here does not read them */
    int         w = 0, h = 0, fmt = -1;     /* geometry of the stored blocks */
    Buf<int16_t> d_old;                     /* [nblk][64], allocated at the first inter call */
    uint64_t    call = 0;                   /* rtjgpu_ctx::enc_seq_calls of the last call that named it */
};

int rtjgpu_seqenc_create(rtjgpu_ctx *ctx, rtjgpu_seqenc **out)
{
    if (!ctx || !out) return RTJGPU_E_ARG;
    *out = nullptr;
    if (!ctx->d_enc_qt_all.get()) {
        CK(ctx, cudaSetDevice(ctx->device));
        std::vector<int32_t> qt(256 * 128, 0);
        for (int q = 1; q <= 255; q++) rtj_encoder_table_from_quality(q, &qt[(size_t)q * 128], &ctx->enc_lb8_all[q], &ctx->enc_cb8_all[q]);
        CK(ctx, ctx->d_enc_qt_all.reserve(qt.size()));
        const cudaError_t e = cudaMemcpy(ctx->d_enc_qt_all.get(), qt.data(), qt.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { ctx->d_enc_qt_all.release(); ctx->last_cuda = (int)e; return RTJGPU_E_CUDA; }
    }
    rtjgpu_seqenc *e = new (std::nothrow) rtjgpu_seqenc();
    if (!e) return RTJGPU_E_NOMEM;
    e->ctx = ctx;
    e->device = ctx->device;
    *out = e;
    return RTJGPU_OK;
}

void rtjgpu_seqenc_destroy(rtjgpu_seqenc *e)
{
    if (!e) return;
    if (e->d_old.get()) cudaSetDevice(e->device);  /* freeing d_old waits for the work that may still read or write it */
    delete e;
}

int rtjgpu_seqenc_set_quality(rtjgpu_seqenc *e, int quality)
{
    if (!e) return RTJGPU_E_ARG;
    e->quality = quality < 1 ? 1 : quality > 255 ? 255 : quality;
    return RTJGPU_OK;
}

int rtjgpu_seqenc_set_intra(rtjgpu_seqenc *e, int key_rate, int lm, int cm)
{
    if (!e) return RTJGPU_E_ARG;
    e->key_rate = key_rate < 0 ? 0 : key_rate > 255 ? 255 : key_rate;
    e->lm = lm < 0 ? 0 : lm > 16 ? 16 : lm;
    e->cm = cm < 0 ? 0 : cm > 16 ? 16 : cm;
    e->cleared = true;                      /* lib/RTjpeg.c:2488, as rtjgpu_encoder_set_intra */
    return RTJGPU_OK;
}

int rtjgpu_seqenc_reset(rtjgpu_seqenc *e)
{
    if (!e) return RTJGPU_E_ARG;
    e->key_count = 0;
    e->cleared = true;
    return RTJGPU_OK;
}

int rtjgpu_seqenc_key_count(const rtjgpu_seqenc *e) { return e ? e->key_count : RTJGPU_E_ARG; }

size_t rtjgpu_encode_bound(int format, int w, int h, int F)
{
    if ((format != RTJ_YUV420 && format != RTJ_YUV422) || !valid_size(w, h) || F < 0) return 0;
    /* a block takes at most 64 bytes (DC byte and one byte per place, RTjpeg_b2s :109-155); header and block bytes are a
     * multiple of 4 already, so no packet needs padding */
    return (size_t)F * (RTJPEG_B200_HEADER_BYTES + 64 * (size_t)RTJ_FMT_NBLK(format, w, h));
}

int rtjgpu_encode_device_seq(rtjgpu_ctx *ctx, int F, int w, int h, int S, const int *seq_first,
                             const uint8_t *const *frames, rtjgpu_seqenc *const *encs,
                             uint8_t *d_stream, size_t capacity, uint64_t *d_offsets, void *cuda_stream)
{
    if (!ctx) return RTJGPU_E_ARG;
    if (ctx->format != RTJ_YUV420 && ctx->format != RTJ_YUV422) return RTJGPU_E_FORMAT;
    if (!valid_size(w, h)) return RTJGPU_E_SIZE;
    if (F > RTJGPU_MAX_FRAMES_PER_BATCH) return RTJGPU_E_TOOBIG;
    SeqIn q;
    q.S = S; q.first = seq_first;
    if (F < 1 || !seq_first || seq_check(F, q) || !frames || !encs || !d_stream || !d_offsets || ((uintptr_t)d_stream & 3))
        return RTJGPU_E_ARG;
    const uint64_t call = ++ctx->enc_seq_calls;
    for (int s = 0; s < S; s++) {
        rtjgpu_seqenc *e = encs[s];
        if (!frames[s] || ((uintptr_t)frames[s] & 7) || !e || e->ctx != ctx || e->call == call) return RTJGPU_E_ARG;
        e->call = call;
    }
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t nblk = (size_t)RTJ_FMT_NBLK(ctx->format, w, h);
    int rc = enc_reserve(ctx, nblk, F);
    if (rc) return rc;
    for (int s = 0; s < S; s++) {
        rtjgpu_seqenc *e = encs[s];
        if (e->w != w || e->h != h || e->fmt != ctx->format) { e->w = w; e->h = h; e->fmt = ctx->format; e->cleared = true; }
        if (e->key_rate && e->d_old.cap() < nblk * 64) {
            CK(ctx, e->d_old.reserve(nblk * 64));
            e->cleared = true;
        }
    }

    /* Runs: every sequence cut where its key counter is 0 -- there RTjpeg_compress clears the stored blocks (:3505) --,
     * intra sequences one picture a run; the counter and the header bytes follow RTjpeg_compress picture by picture. */
    const size_t seqs_bytes = (size_t)S * sizeof(rtj_enc_seq);
    const size_t words_bytes = ((size_t)F * sizeof(uint32_t) + 7) & ~(size_t)7;
    std::vector<rtj_enc_run> &runs = ctx->enc_runs;
    runs.clear();
    int n_intra = 0;
    for (int s = 0; s < S; s++)
        if (!encs[s]->key_rate) n_intra += seq_first[s + 1] - seq_first[s];
    runs.resize((size_t)n_intra);
    const size_t bytes_bound = seqs_bytes + words_bytes + ((size_t)F + S) * sizeof(rtj_enc_run);
    uint8_t *hb;
    if ((rc = stage_begin(ctx, bytes_bound, &hb))) return rc;
    rtj_enc_seq *hs = reinterpret_cast<rtj_enc_seq *>(hb);
    uint32_t *hw = reinterpret_cast<uint32_t *>(hb + seqs_bytes);
    int at_intra = 0;
    for (int s = 0; s < S; s++) {
        const rtjgpu_seqenc *e = encs[s];
        const int a = seq_first[s], b = seq_first[s + 1];
        rtj_enc_seq &r = hs[s];
        r.d_frames = frames[s]; r.d_old = e->d_old.get(); r.first = a; r.quality = e->quality;
        r.lb8 = ctx->enc_lb8_all[e->quality]; r.cb8 = ctx->enc_cb8_all[e->quality]; r.lmask = e->lm; r.cmask = e->cm;
        if (!e->key_rate) {
            for (int f = a; f < b; f++) {
                runs[at_intra++] = rtj_enc_run{f, f + 1, (uint32_t)s};
                hw[f] = RTJ_ENC_FRAME(e->quality, 0);
            }
            continue;
        }
        int c = e->key_count, f0 = a;
        uint32_t flags = c != 0 && !e->cleared ? RTJ_ENC_RUN_CONT : 0u;
        for (int f = a; f < b; f++) {
            if (c == 0 && f > f0) {
                runs.push_back(rtj_enc_run{f0, f, (uint32_t)s | flags});
                f0 = f; flags = 0;
            }
            hw[f] = RTJ_ENC_FRAME(e->quality, c);
            c = c + 1 > e->key_rate ? 0 : c + 1;
        }
        runs.push_back(rtj_enc_run{f0, b, (uint32_t)s | flags | RTJ_ENC_RUN_LAST});
    }
    const size_t runs_bytes = runs.size() * sizeof(rtj_enc_run);
    const size_t bytes = seqs_bytes + words_bytes + runs_bytes;
    memcpy(hb + seqs_bytes + words_bytes, runs.data(), runs_bytes);
    CK(ctx, ctx->d_enc_seq.reserve(bytes));
    const uint8_t *d = ctx->d_enc_seq.get();
    if ((rc = stage_end(ctx, ctx->d_enc_seq.get(), bytes, st))) return rc;

    rtj_encode_args a;
    memset(&a, 0, sizeof(a));
    a.F = F; a.w = w; a.h = h; a.fmt = ctx->format; a.d_qt = ctx->d_enc_qt_all.get();
    a.d_slots = ctx->d_enc_slots.get(); a.d_lens = ctx->d_enc_lens.get(); a.d_boff = ctx->d_enc_boff.get();
    a.d_fsize = ctx->d_enc_fsize.get(); a.d_stream = d_stream; a.capacity = capacity; a.d_offsets = d_offsets;
    a.d_total = ctx->d_enc_total.get();
    ctx->enc_stream = cuda_stream;
    const int n = rtj_launch_encode_seq(&a, reinterpret_cast<const rtj_enc_run *>(d + seqs_bytes + words_bytes),
                                        n_intra, (int)runs.size() - n_intra, reinterpret_cast<const rtj_enc_seq *>(d),
                                        reinterpret_cast<const uint32_t *>(d + seqs_bytes), cuda_stream);
    if (n < 0) { ctx->last_cuda = -n; return RTJGPU_E_CUDA; }
    ctx->launches += (uint64_t)n;
    /* the handles move on as RTjpeg_compress would have, whether the packets fit or not */
    for (int s = 0; s < S; s++) {
        rtjgpu_seqenc *e = encs[s];
        if (!e->key_rate) continue;
        int c = e->key_count;
        for (int f = seq_first[s]; f < seq_first[s + 1]; f++) c = c + 1 > e->key_rate ? 0 : c + 1;
        e->key_count = c;
        e->cleared = false;
    }
    return RTJGPU_OK;
}

int rtjgpu_convert_bpp(int kind) { return rtj_convert_bpp(kind); }

int rtjgpu_convert_device(rtjgpu_ctx *ctx, int kind, const uint8_t *d_frames, size_t src_frame_bytes,
                          int F, int w, int h, uint8_t *d_out, size_t row_pitch, size_t frame_pitch,
                          int alpha, void *cuda_stream)
{
    if (!ctx || F < 0) return RTJGPU_E_ARG;
    const int bpp = rtj_convert_bpp(kind);
    if (!bpp) return RTJGPU_E_FORMAT;
    if (F == 0) return RTJGPU_OK;
    if (!d_frames || !d_out) return RTJGPU_E_ARG;
    if (!valid_size(w, h)) return RTJGPU_E_SIZE;
    if (F > 65535) return RTJGPU_E_TOOBIG;                                   /* frames are the grid's second dimension */
    if ((row_pitch & 15) || row_pitch < (size_t)w * bpp || frame_pitch < row_pitch * (size_t)h
        || ((uintptr_t)d_out & 15) || ((uintptr_t)d_frames & 7) || (src_frame_bytes & 7) || (frame_pitch & 15))
        return RTJGPU_E_ARG;
    const size_t ysz = (size_t)w * h;
    const size_t need = kind == RTJ_CONV_RGB8 ? ysz : kind == RTJ_CONV_YUV422_RGB24 ? 2 * ysz : ysz + ysz / 2;
    if (src_frame_bytes < need) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    const int e = rtj_launch_convert(kind, d_frames, src_frame_bytes, F, w, h, d_out, row_pitch, frame_pitch,
                                     (unsigned)alpha, cuda_stream);
    if (e) { ctx->last_cuda = e; return RTJGPU_E_CUDA; }
    ctx->launches += 1;
    return RTJGPU_OK;
}

int rtjgpu_set_custom_tables(rtjgpu_ctx *ctx, const uint32_t raw[128])
{
    if (!ctx || !raw) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    rtj_table_from_raw(raw, &ctx->h_tables[RTJGPU_TABLE_CUSTOM]);
    rtj_dev_table dev;
    rtj_table_to_device_layout(&ctx->h_tables[RTJGPU_TABLE_CUSTOM], &dev);
    /* ordered after the batches this context has queued (its own streams and the caller's last one); other contexts'
     * work on the device is none of its business */
    if (cudaStreamSynchronize((cudaStream_t)ctx->last_stream) != cudaSuccess) {    /* the caller's stream may be gone by now */
        cudaGetLastError();
        CK(ctx, cudaDeviceSynchronize());
    }
    if (ctx->pipe.ready) { CK(ctx, cudaStreamSynchronize(ctx->pipe.scan)); CK(ctx, cudaStreamSynchronize(ctx->pipe.idct)); }
    if (ctx->slots_ready) for (int i = 0; i < HOST_SLOTS; i++) CK(ctx, cudaStreamSynchronize(ctx->slot[i].stream));
    CK(ctx, cudaMemcpy(ctx->d_tables.get() + RTJGPU_TABLE_CUSTOM, &dev, sizeof(dev), cudaMemcpyHostToDevice));
    return RTJGPU_OK;
}

/* internal: host tables in the reference's raster order (for RTjpeg_get_tables) */
const rtj_host_table *rtj_ctx_host_table(const rtjgpu_ctx *ctx, int table)
{
    if (!ctx || table < 0 || table >= RTJ_NUM_TABLES) return nullptr;
    return &ctx->h_tables[table];
}

int rtjgpu_plan(const uint8_t *stream, const uint64_t *offsets, int F, rtjgpu_state *state, rtjgpu_frame_desc *desc)
{
    return rtjgpu_plan_n(stream, offsets, nullptr, F, state, desc);
}

int rtjgpu_plan_n(const uint8_t *stream, const uint64_t *offsets, const uint32_t *lengths, int F, rtjgpu_state *state,
                  rtjgpu_frame_desc *desc)
{
    if (!stream || !offsets || !state || (F > 0 && !desc) || F < 0) return RTJGPU_E_ARG;
    if (F > RTJGPU_MAX_FRAMES_PER_BATCH) return RTJGPU_E_TOOBIG;
    rtjgpu_state st = *state;
    int bw = 0, bh = 0;
    for (int f = 0; f < F; f++) {
        if (offsets[f + 1] < offsets[f]) return RTJGPU_E_ARG;
        uint64_t avail = offsets[f + 1] - offsets[f];
        if (lengths) {
            if (lengths[f] > avail) return RTJGPU_E_ARG;
            avail = lengths[f];
        }
        if (avail < RTJPEG_B200_HEADER_BYTES) return RTJGPU_E_HEADER;
        if (offsets[f] & 3u) return RTJGPU_E_ARG;
        const uint8_t *p = stream + offsets[f];
        /* packed little-endian header, include/RTjpeg.h:100-109 */
        const uint32_t framesize = rd_u32le(p);
        const int w = rd_u16le(p + 6), h = rd_u16le(p + 8), q = p[10];
        /* the reference never reads framesize/headersize (lib/RTjpeg.c:3565-3586).  With the packets' true lengths
         * given, neither does this; without them the slot [offsets[f], offsets[f + 1]) may end in alignment padding,
         * and the smaller of framesize and the slot bounds every read */
        uint64_t len = avail;
        if (!lengths && framesize >= RTJPEG_B200_HEADER_BYTES && framesize < len) len = framesize;
        if (len - RTJPEG_B200_HEADER_BYTES > RTJGPU_MAX_PAYLOAD_BYTES) return RTJGPU_E_TOOBIG;
        if (w != st.width || h != st.height) { st.width = w; st.height = h; }   /* :3568-3574 */
        if (!valid_size(w, h)) return RTJGPU_E_SIZE;                             /* the row loop of :2701 needs /16 */
        if (f == 0) { bw = w; bh = h; }
        else if (w != bw || h != bh) return RTJGPU_E_SIZE;
        if (q != st.quality) {                                                   /* :3575-3579 */
            const int qc = q < 1 ? 1 : q;                                        /* set_quality clamps, :2410-2412 */
            st.quality = qc;
            st.table = qc;
        }
        desc[f].offset = offsets[f];
        desc[f].length = (uint32_t)len;
        desc[f].table = (uint16_t)st.table;
        desc[f].flags = 0;
    }
    *state = st;
    return RTJGPU_OK;
}

int rtjgpu_decode_device(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F,
                         int w, int h, uint8_t *d_out, const uint8_t *d_carry, void *cuda_stream)
{
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.carries = &d_carry;
    c.d_out = d_out;
    return decode(ctx, c);
}

int rtjgpu_decode_device_seq(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                             int S, const int *seq_first, uint8_t *d_out, const uint8_t *const *carries, void *cuda_stream)
{
    if (!seq_first) return RTJGPU_E_ARG;
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.S = S; c.q.first = seq_first; c.q.carries = carries;
    c.d_out = d_out;
    return decode(ctx, c);
}

int rtjgpu_decode_device_rgb(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F,
                             int w, int h, int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch, int alpha,
                             const uint8_t *d_carry, uint8_t *d_last_yuv, void *cuda_stream)
{
    const RgbOut o{d_rgb, row_pitch, frame_pitch, kind, alpha};
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.carries = &d_carry; c.q.last_yuv = &d_last_yuv;
    c.rgb = &o;
    return decode(ctx, c);
}

int rtjgpu_decode_device_rgb_seq(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                 int S, const int *seq_first, int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch,
                                 int alpha, const uint8_t *const *carries, uint8_t *const *last_yuv, void *cuda_stream)
{
    if (!seq_first) return RTJGPU_E_ARG;
    const RgbOut o{d_rgb, row_pitch, frame_pitch, kind, alpha};
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.S = S; c.q.first = seq_first; c.q.carries = carries; c.q.last_yuv = last_yuv;
    c.rgb = &o;
    return decode(ctx, c);
}

int rtjgpu_decode_device_select(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                int S, const int *seq_first, const uint8_t *const *carries,
                                int n, const int *sel, uint8_t *d_out, void *cuda_stream)
{
    if (!seq_first) return RTJGPU_E_ARG;
    const SelIn s{n, sel};
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.S = S; c.q.first = seq_first; c.q.carries = carries;
    c.sel = &s;
    c.d_out = d_out;
    return decode(ctx, c);
}

int rtjgpu_decode_device_rgb_select(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                    int S, const int *seq_first, const uint8_t *const *carries,
                                    int n, const int *sel, int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch,
                                    int alpha, uint8_t *const *last_yuv, void *cuda_stream)
{
    if (!seq_first) return RTJGPU_E_ARG;
    const SelIn s{n, sel};
    const RgbOut o{d_rgb, row_pitch, frame_pitch, kind, alpha};
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.S = S; c.q.first = seq_first; c.q.carries = carries; c.q.last_yuv = last_yuv;
    c.sel = &s;
    c.rgb = &o;
    return decode(ctx, c);
}

int rtjgpu_decode_device_window(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                int S, const int *seq_first, const uint8_t *const *carries,
                                int n, const int *sel, int cw, int ch, const int *origins,
                                uint8_t *d_out, uint8_t *const *last_yuv, void *cuda_stream)
{
    if (!seq_first) return RTJGPU_E_ARG;
    const SelIn s{n, sel};
    const WinIn v{cw, ch, origins};
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.S = S; c.q.first = seq_first; c.q.carries = carries; c.q.last_yuv = last_yuv;
    c.sel = &s;
    c.win = &v;
    c.d_out = d_out;
    return decode(ctx, c);
}

int rtjgpu_decode_device_rgb_window(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                                    int S, const int *seq_first, const uint8_t *const *carries,
                                    int n, const int *sel, int cw, int ch, const int *origins,
                                    int kind, uint8_t *d_rgb, size_t row_pitch, size_t frame_pitch, int alpha,
                                    uint8_t *const *last_yuv, void *cuda_stream)
{
    if (!seq_first) return RTJGPU_E_ARG;
    const SelIn s{n, sel};
    const WinIn v{cw, ch, origins};
    const RgbOut o{d_rgb, row_pitch, frame_pitch, kind, alpha};
    DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    c.q.S = S; c.q.first = seq_first; c.q.carries = carries; c.q.last_yuv = last_yuv;
    c.sel = &s;
    c.win = &v;
    c.rgb = &o;
    return decode(ctx, c);
}

int rtjgpu_sync(rtjgpu_ctx *ctx)
{
    if (!ctx) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaDeviceSynchronize());
    return RTJGPU_OK;
}

int rtjgpu_get_timing_at(rtjgpu_ctx *ctx, int calls_ago, rtjgpu_timing *out)
{
    if (!ctx || !out || calls_ago < 0 || calls_ago >= TIMING_RING) return RTJGPU_E_ARG;
    memset(out, 0, sizeof(*out));
    if ((uint64_t)calls_ago >= ctx->timed_calls) return RTJGPU_E_ARG;
    cudaEvent_t *ev = ctx->ev[(ctx->timed_calls - 1 - (uint64_t)calls_ago) % TIMING_RING];
    CK(ctx, cudaEventSynchronize(ev[3]));
    CK(ctx, cudaEventElapsedTime(&out->scan_ms, ev[0], ev[1]));
    CK(ctx, cudaEventElapsedTime(&out->resolve_ms, ev[1], ev[2]));
    CK(ctx, cudaEventElapsedTime(&out->idct_ms, ev[2], ev[3]));
    CK(ctx, cudaEventElapsedTime(&out->total_ms, ev[0], ev[3]));
    return RTJGPU_OK;
}

int rtjgpu_get_timing(rtjgpu_ctx *ctx, rtjgpu_timing *out)
{
    if (!ctx || !out) return RTJGPU_E_ARG;
    memset(out, 0, sizeof(*out));
    if (!ctx->timed_calls) return RTJGPU_OK;
    return rtjgpu_get_timing_at(ctx, 0, out);
}

int rtjgpu_get_batch_info(rtjgpu_ctx *ctx, rtjgpu_batch_info *out)
{
    if (!ctx || !out) return RTJGPU_E_ARG;
    memset(out, 0, sizeof(*out));
    out->first_bad_frame = -1;
    if (ctx->last_F == 0 || !ctx->ws.d_info.get()) return RTJGPU_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaDeviceSynchronize());
    const rtj_dev_info *info = ctx->h_info.get();
    CK(ctx, cudaMemcpy(ctx->h_info.get(), ctx->ws.d_info.get(), sizeof(rtj_dev_info), cudaMemcpyDeviceToHost));
    out->skipped_blocks = info->skipped_blocks;
    out->payload_bytes = info->payload_bytes;
    out->bad_frames = info->bad_frames;
    out->first_bad_frame = info->first_bad_frame;
    return RTJGPU_OK;
}

int rtjgpu_get_skip_counts(rtjgpu_ctx *ctx, uint32_t *counts, int F)
{
    if (!ctx || !counts || F < 0 || F > ctx->last_F) return RTJGPU_E_ARG;
    if (F == 0) return RTJGPU_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaDeviceSynchronize());
    CK(ctx, cudaMemcpy(counts, ctx->ws.frame_skips(), (size_t)F * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return RTJGPU_OK;
}

int rtjgpu_get_entries(rtjgpu_ctx *ctx, uint32_t *entries, size_t n)
{
    if (!ctx || !entries || n > ctx->ws.d_ent.cap()) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaDeviceSynchronize());
    CK(ctx, cudaMemcpy(entries, ctx->ws.d_ent.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return RTJGPU_OK;
}

/* nearest clean frame to `ideal` inside [lo, hi], the later one on a tie; -1: none */
static int nearest_clean(const uint8_t *clean, int ideal, int lo, int hi)
{
    for (int d = 0; ideal - d >= lo || ideal + d <= hi; d++) {
        if (ideal + d >= lo && ideal + d <= hi && clean[ideal + d]) return ideal + d;
        if (ideal - d >= lo && ideal - d <= hi && clean[ideal - d]) return ideal - d;
    }
    return -1;
}

int rtjgpu_split_shards(const uint8_t *clean, int F, int n, int *first)
{
    if (!clean || !first || n < 1 || F < 0) return RTJGPU_E_ARG;
    first[0] = 0;
    int empty = 0;
    for (int i = 1; i < n; i++) {
        /* the clean frame nearest to the ideal cut, behind the previous cut and leaving a frame for every later shard
         * where the clean frames allow it; without any, the shard comes out empty -- and is counted */
        const int ideal = (int)((long long)F * i / n);
        const int lo = first[i - 1] + 1, hi = F - 1;
        int cut = lo <= hi ? nearest_clean(clean, std::min(std::max(ideal, lo), hi), lo, hi) : -1;
        if (cut < 0) cut = F;
        first[i] = cut;
    }
    first[n] = F;
    for (int i = 0; i < n; i++) empty += first[i + 1] == first[i];
    return F == 0 ? 0 : empty;
}

int rtjgpu_split_shards_lead(const uint8_t *clean, int F, int n, int *first, int *lead)
{
    if (!clean || !first || !lead || n < 1 || F < 0) return RTJGPU_E_ARG;
    first[0] = 0;
    lead[0] = 0;                                            /* frame 0 starts from the caller's picture */
    const int win = std::max(1, F / (2 * n));              /* how far a cut may move to find a clean frame: half a shard */
    for (int i = 1; i < n; i++) {
        const int ideal = (int)((long long)F * i / n);
        const int lo = std::min(first[i - 1] + 1, F);
        const int hi = std::max(lo, F - (n - i));                          /* a frame for every shard, while F >= n */
        const int at = std::min(std::max(ideal, lo), hi);
        if (at >= F) { first[i] = F; lead[i] = 0; continue; }              /* fewer frames than shards: an empty one */
        const int c = nearest_clean(clean, at, std::max(lo, at - win), std::min(hi, at + win));
        if (c >= 0) { first[i] = c; lead[i] = 0; continue; }
        /* no clean frame near: cut at the ideal place and decode again from the last clean frame before it --
         * or from frame 0 and the caller's picture when there is none */
        int back = at;
        while (back > 0 && !clean[back]) back--;
        first[i] = at;
        lead[i] = at - back;
    }
    first[n] = F;
    return RTJGPU_OK;
}

int rtjgpu_scan_device(rtjgpu_ctx *ctx, const uint8_t *d_stream, const rtjgpu_frame_desc *d_desc, int F, int w, int h,
                       void *cuda_stream)
{
    if (!ctx || F < 0) return RTJGPU_E_ARG;
    if (F == 0) { ctx->last_F = 0; return RTJGPU_OK; }
    const DecodeCall c(d_stream, d_desc, F, w, h, cuda_stream);
    int nblk, rc;
    if ((rc = check_batch(ctx, c, false, &nblk))) return rc;
    if ((rc = ws_reserve(ctx, &ctx->ws, F, nblk))) return rc;
    rtj_launch_args a = k1_args(ctx, ctx->ws, c);
    if ((rc = seg_reserve(ctx, &ctx->ws, F, nblk, ctx->scan_mode, &a.seg))) return rc;
    CK(ctx, cudaMemcpyAsync(ctx->ws.d_info.get(), ctx->h_info_reset.get(), sizeof(rtj_dev_info), cudaMemcpyHostToDevice, c.stream));
    const int e = rtj_launch_scan(&a, c.stream);
    if (e < 0) { ctx->last_cuda = -e; return RTJGPU_E_CUDA; }
    ctx->launches += (uint64_t)e;
    ctx->last_F = F;
    ctx->last_stream = cuda_stream;
    return RTJGPU_OK;
}

static void export_table(const rtj_host_table &t, uint32_t scaled[128], int *lb8, int *cb8)
{
    for (int i = 0; i < 64; i++) {
        scaled[i] = (uint32_t)t.liqt[i];
        scaled[64 + i] = (uint32_t)t.ciqt[i];
    }
    if (lb8) *lb8 = t.lb8;
    if (cb8) *cb8 = t.cb8;
}

void rtjgpu_tables_for_quality(int Q, uint32_t scaled[128], int *lb8, int *cb8)
{
    rtj_host_table t;
    rtj_table_from_quality(Q, &t);
    export_table(t, scaled, lb8, cb8);
}

void rtjgpu_tables_from_raw(const uint32_t raw[128], uint32_t scaled[128], int *lb8, int *cb8)
{
    rtj_host_table t;
    rtj_table_from_raw(raw, &t);
    export_table(t, scaled, lb8, cb8);
}

void *rtjgpu_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}

void rtjgpu_host_free(void *p) { if (p) cudaFreeHost(p); }

/* ------------------------------------------------------------------------ */
/* host pipeline                                                              */
/* ------------------------------------------------------------------------ */

static int slots_init(rtjgpu_ctx *ctx)
{
    if (ctx->slots_ready) return RTJGPU_OK;
    for (int i = 0; i < HOST_SLOTS; i++) {
        CK(ctx, cudaStreamCreateWithFlags(&ctx->slot[i].stream, cudaStreamNonBlocking));
        CK(ctx, cudaEventCreateWithFlags(&ctx->slot[i].decoded, cudaEventDisableTiming));
        CK(ctx, ctx->slot[i].h_info.reserve(1));
    }
    ctx->slots_ready = true;
    return RTJGPU_OK;
}

static int slot_drain(rtjgpu_ctx *ctx, HostSlot &s)
{
    if (!s.busy) return RTJGPU_OK;
    const cudaError_t e = cudaStreamSynchronize(s.stream);
    if (e == cudaSuccess) {
        ctx->host_bad += s.h_info.get()->bad_frames;
        if (s.pending_dst) memcpy(s.pending_dst, s.h_out.get(), s.pending_bytes);
    }
    s.pending_dst = nullptr;              /* whatever happened: never again touch the memory of the call that queued this */
    s.pending_bytes = 0;
    s.busy = false;
    if (e != cudaSuccess) { ctx->last_cuda = (int)e; return RTJGPU_E_CUDA; }
    return RTJGPU_OK;
}

int rtjgpu_decode_host(rtjgpu_ctx *ctx, const uint8_t *h_stream, const uint64_t *offsets, int F,
                       rtjgpu_state *state, uint8_t *h_out, uint8_t *h_carry_inout, int flags)
{
    return rtjgpu_decode_host_n(ctx, h_stream, offsets, nullptr, F, state, h_out, h_carry_inout, flags);
}

int rtjgpu_decode_host_n(rtjgpu_ctx *ctx, const uint8_t *h_stream, const uint64_t *offsets, const uint32_t *lengths, int F,
                         rtjgpu_state *state, uint8_t *h_out, uint8_t *h_carry_inout, int flags)
{
    if (!ctx || !state || F < 0) return RTJGPU_E_ARG;
    if (F == 0) return RTJGPU_OK;
    if (!h_stream || !offsets || !h_out) return RTJGPU_E_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = slots_init(ctx);
    if (rc) return rc;

    /* geometry from the first header; rtjgpu_plan re-checks every frame */
    if ((lengths ? (uint64_t)lengths[0] : offsets[1] - offsets[0]) < RTJPEG_B200_HEADER_BYTES) return RTJGPU_E_HEADER;
    const int w = rd_u16le(h_stream + offsets[0] + 6), h = rd_u16le(h_stream + offsets[0] + 8);
    if (!valid_size(w, h)) return RTJGPU_E_SIZE;
    const size_t fsz = RTJ_FMT_FRAME_BYTES(ctx->format, w, h);
    const int nblk = RTJ_FMT_NBLK(ctx->format, w, h);

    /* chunk size: ~64 MB of output per chunk keeps three slots in flight without
     * hoarding memory; at least 1, at most the batch limit */
    int chunk = (int)std::max<size_t>(1, (64u << 20) / fsz);
    chunk = std::min(chunk, RTJGPU_MAX_FRAMES_PER_BATCH);
    chunk = std::min(chunk, F);

    CK(ctx, ctx->d_host_carry.reserve(fsz));
    CK(ctx, ctx->h_host_skips.reserve((size_t)F));
    ctx->host_F = 0;
    const bool have_carry = h_carry_inout != nullptr;
    if (have_carry)
        CK(ctx, cudaMemcpy(ctx->d_host_carry.get(), h_carry_inout, fsz, cudaMemcpyHostToDevice));

    const uint8_t *d_prev = have_carry ? ctx->d_host_carry.get() : nullptr;
    cudaEvent_t prev_decoded = nullptr;
    rtjgpu_state st = *state;
    int result = RTJGPU_OK;
    ctx->host_bad = 0;
    std::vector<uint64_t> rel;

    /* inside the loop a failing CUDA call must not return: the slots already in flight hold pointers into this call's
     * h_out and have to be drained first */
#define CKB(call)                                                                          \
    { const cudaError_t e__ = (call); if (e__ != cudaSuccess) { ctx->last_cuda = (int)e__; result = RTJGPU_E_CUDA; break; } }
    for (int c0 = 0, ci = 0; c0 < F; c0 += chunk, ci++) {
        const int n = std::min(chunk, F - c0);
        HostSlot &s = ctx->slot[ci % HOST_SLOTS];
        if ((rc = slot_drain(ctx, s))) { result = rc; break; }

        const uint64_t b0 = offsets[c0], b1 = offsets[c0 + n];
        const size_t in_bytes = (size_t)(b1 - b0);
        CKB(s.d_in.reserve(in_bytes + RTJGPU_STREAM_SLACK_BYTES));
        CKB(s.d_out.reserve(fsz * (size_t)n));
        CKB(s.d_desc.reserve((size_t)n));
        CKB(s.h_desc.reserve((size_t)n));
        if ((rc = ws_reserve(ctx, &s.ws, n, nblk))) { result = rc; break; }

        /* descriptors relative to the chunk's own device buffer */
        rel.resize((size_t)n + 1);
        for (int i = 0; i <= n; i++) rel[(size_t)i] = offsets[c0 + i] - b0;
        if ((rc = rtjgpu_plan_n(h_stream + b0, rel.data(), lengths ? lengths + c0 : nullptr, n, &st, s.h_desc.get()))) { result = rc; break; }
        if (st.width != w || st.height != h) { result = RTJGPU_E_SIZE; break; }

        const uint8_t *src = h_stream + b0;
        if (!(flags & RTJGPU_HOST_IN_PINNED)) {
            CKB(s.h_in.reserve(in_bytes));
            memcpy(s.h_in.get(), src, in_bytes);
            src = s.h_in.get();
        }
        CKB(cudaMemcpyAsync(s.d_in.get(), src, in_bytes, cudaMemcpyHostToDevice, s.stream));
        CKB(cudaMemsetAsync(s.d_in.get() + in_bytes, 0x7F, RTJGPU_STREAM_SLACK_BYTES, s.stream));
        CKB(cudaMemcpyAsync(s.d_desc.get(), s.h_desc.get(), sizeof(rtjgpu_frame_desc) * (size_t)n, cudaMemcpyHostToDevice, s.stream));
        if (prev_decoded) CKB(cudaStreamWaitEvent(s.stream, prev_decoded, 0));   /* carry comes from the previous chunk */
        DecodeCall c(s.d_in.get(), s.d_desc.get(), n, w, h, s.stream);
        c.q.carries = &d_prev;
        c.d_out = s.d_out.get();
        if ((rc = run_kernels(ctx, &s.ws, c, CallDev(), nullptr, false))) { result = rc; break; }
        CKB(cudaEventRecord(s.decoded, s.stream));
        CKB(cudaMemcpyAsync(s.h_info.get(), s.ws.d_info.get(), sizeof(rtj_dev_info), cudaMemcpyDeviceToHost, s.stream));
        CKB(cudaMemcpyAsync(ctx->h_host_skips.get() + c0, s.ws.frame_skips(), sizeof(uint32_t) * (size_t)n, cudaMemcpyDeviceToHost, s.stream));
        prev_decoded = s.decoded;
        d_prev = s.d_out.get() + fsz * (size_t)(n - 1);

        uint8_t *dst = h_out + fsz * (size_t)c0;
        if (flags & RTJGPU_HOST_OUT_PINNED) {
            CKB(cudaMemcpyAsync(dst, s.d_out.get(), fsz * (size_t)n, cudaMemcpyDeviceToHost, s.stream));
            s.pending_dst = nullptr;
        } else {
            CKB(s.h_out.reserve(fsz * (size_t)n));
            CKB(cudaMemcpyAsync(s.h_out.get(), s.d_out.get(), fsz * (size_t)n, cudaMemcpyDeviceToHost, s.stream));
            s.pending_dst = dst;
            s.pending_bytes = fsz * (size_t)n;
        }
        s.busy = true;
    }
#undef CKB
    /* drain in issue order so that later chunks' carries are complete */
    for (int i = 0; i < HOST_SLOTS; i++) {
        int rc2 = slot_drain(ctx, ctx->slot[i]);
        if (rc2 && !result) result = rc2;
    }
    if (result == RTJGPU_OK && ctx->host_bad) result = RTJGPU_E_OVERRUN;
    if (result == RTJGPU_OK || result == RTJGPU_E_OVERRUN) {
        if (have_carry) memcpy(h_carry_inout, h_out + fsz * (size_t)(F - 1), fsz);
        *state = st;
        ctx->host_F = F;
    }
    return result;
}

int rtjgpu_get_host_skip_counts(rtjgpu_ctx *ctx, uint32_t *counts, int F)
{
    if (!ctx || !counts || F < 0 || F > ctx->host_F) return RTJGPU_E_ARG;
    if (F) memcpy(counts, ctx->h_host_skips.get(), sizeof(uint32_t) * (size_t)F);
    return RTJGPU_OK;
}

} // extern "C"
