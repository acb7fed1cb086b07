"""K1, self-synchronising flavour (csrc/rtj_scan_sync.cu): the paths the general parity suite does not reach by itself --
frames of several segments, streams whose parse does NOT synchronise (repair rounds when the flavour is forced, the
hand-over to the chunk-parallel kernel under AUTO), and entry tables / counters identical to the chunk-parallel kernel's on
damaged streams.  Pixels are checked against the reference (lib/RTjpeg.c compiled by oracle/Makefile)."""
import ctypes as C

import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from gpu_util import first_diff, gpu_decode
from streams import clip, reference_frames

pytestmark = pytest.mark.gpu


def _ctx(mode):
    c = g.BatchContext(0)
    c.set_scan_mode(mode)
    return c


def _entries(ctx, s, o, w, h):
    """rtjgpu_scan_device alone: the entry table as K1 leaves it, and the batch counters."""
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, w, h)
    ctx.set_format(0)
    ctx.scan_device(b.stream.data_ptr(), b.desc.data_ptr(), b.F, w, h, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    nblk = (w // 16) * (h // 16) * 6
    ent = np.zeros(b.F * nblk, dtype=np.uint32)
    L = g.load_library()
    L.rtjgpu_get_entries.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    assert L.rtjgpu_get_entries(ctx._h, C.c_void_p(ent.ctypes.data), ent.size) == 0
    bi = ctx.batch_info()
    return ent.reshape(b.F, nblk), (bi.skipped_blocks, bi.payload_bytes, bi.bad_frames, bi.first_bad_frame)


@pytest.mark.parametrize("kw", [dict(Q=128), dict(Q=128, key_rate=3, lm=2, cm=2), dict(Q=170, noise_y=12, noise_c=4)])
def test_frames_of_several_segments(kw):
    """1920x1088: 150 .. 400 KB of payload a frame, four to ten segments, the state carried from one to the next."""
    kw = dict(kw)
    Q = kw.pop("Q")
    w, h, F = 1920, 1088, 3
    s, o = clip(w, h, Q, F, **kw)
    assert int(O.packet_sizes(s, o).min()) > 2 * 40960                   # three segments or more
    want = reference_frames(s, o, w, h)
    with _ctx(capi.SCAN_SYNC) as c:
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        assert c.batch_info().bad_frames == 0


def _dense_packets(w, h, n, seed):
    rng = np.random.default_rng(seed)
    return [O.random_wellformed_packet(rng, w, h, 128, skip_prob=0.02, dense_prob=0.97, extreme=False) for _ in range(n)]


def test_stream_that_does_not_synchronise_forced():
    """Nearly every block is 64 coefficient bytes long: a walk entered in the wrong state stays wrong for whole chunks.  With
    the flavour forced, the repair rounds must still arrive at the one true parse."""
    w, h = 320, 240
    pk = _dense_packets(w, h, 3, 5)
    s, o = O.pack_packets(pk)
    want = reference_frames(s, o, w, h)
    with _ctx(capi.SCAN_SYNC) as c, _ctx(capi.SCAN_CHUNK) as k:
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        e1, i1 = _entries(c, s, o, w, h)
        e2, i2 = _entries(k, s, o, w, h)
        assert np.array_equal(e1, e2) and i1 == i2


def test_stream_that_does_not_synchronise_is_handed_over_under_auto():
    """AUTO with a batch large enough for one CTA per frame: frames whose chunks are entered in the wrong state too often go
    to the chunk-parallel kernel, the others stay; pixels and counters as ever."""
    w, h = 320, 240
    dense = _dense_packets(w, h, 2, 9)
    s0, o0 = clip(w, h, 128, 2, noise_y=6)
    sizes = O.packet_sizes(s0, o0)
    calm = [s0[int(o0[i]):int(o0[i]) + int(sizes[i])] for i in range(2)]
    order = [dense[0], calm[0], dense[1], calm[1]] * 75                 # 300 frames: above AUTO's segment-parallel limit
    s, o = O.pack_packets(order)
    want4 = reference_frames(*O.pack_packets(order[:4]), w, h)
    with _ctx(capi.SCAN_AUTO) as c:
        got, _ = gpu_decode(c, s, o, w, h)
        bi = c.batch_info()
        assert bi.bad_frames == 0
        assert bi.payload_bytes == sum(p.size - 12 for p in order)
    # intra frames, no skip markers in the calm ones; the dense ones hold a few: compare frame by frame with its sequence's reference
    seq = reference_frames(s, o, w, h)
    assert np.array_equal(got, seq), first_diff(got, seq, w, h)
    assert np.array_equal(seq[:4], want4)


@pytest.mark.parametrize("cut", [1, 2, 3, 7, 64, 1000, -1, -2, -5, -63])
def test_damaged_streams_same_entries_as_the_chunk_kernel(cut):
    """A packet cut short (from the front: keep `cut` payload bytes; from the back: drop -cut bytes), followed by garbage
    in the stream's slack: both kernels see the same blocks, flag the same frame and count the same bytes."""
    w, h = 208, 112
    s, o = clip(w, h, 128, 3, key_rate=2, lm=2, cm=2, noise_y=10)
    sizes = O.packet_sizes(s, o)
    n1 = int(sizes[1])
    keep = 12 + cut if cut > 0 else n1 + cut
    pk = [s[int(o[0]):int(o[0]) + int(sizes[0])], s[int(o[1]):int(o[1]) + keep].copy(), s[int(o[2]):int(o[2]) + int(sizes[2])]]
    pk[1][0:4] = np.frombuffer(np.uint32(pk[1].size).tobytes(), dtype=np.uint8)
    s2, o2 = O.pack_packets(pk, align=4)                                 # packets 4-byte aligned: every misalignment of the payload
    with _ctx(capi.SCAN_SYNC) as c, _ctx(capi.SCAN_CHUNK) as k:
        e1, i1 = _entries(c, s2, o2, w, h)
        e2, i2 = _entries(k, s2, o2, w, h)
    assert i1 == i2 and i1[2] == 1 and i1[3] == 1
    assert np.array_equal(e1, e2)


@pytest.mark.parametrize("align", [4, 16])
def test_every_payload_misalignment_and_frame_size(align):
    """Frames of very different sizes back to back (a one-macroblock frame next to a large one is not possible in one
    batch: sizes vary through the content instead), packets at every 4-byte alignment: entries as the chunk kernel's."""
    w, h = 352, 288
    s, o = clip(w, h, 100, 9, key_rate=4, lm=1, cm=1, noise_y=14, noise_c=3)
    sizes = O.packet_sizes(s, o)
    pk = [s[int(o[i]):int(o[i]) + int(sizes[i])] for i in range(9)]
    s2, o2 = O.pack_packets(pk, align=align)
    with _ctx(capi.SCAN_SYNC) as c, _ctx(capi.SCAN_CHUNK) as k:
        e1, i1 = _entries(c, s2, o2, w, h)
        e2, i2 = _entries(k, s2, o2, w, h)
        assert np.array_equal(e1, e2) and i1 == i2 and i1[2] == 0
        got, _ = gpu_decode(c, s2, o2, w, h)
    want = reference_frames(s2, o2, w, h)
    assert np.array_equal(got, want), first_diff(got, want, w, h)


def test_workspace_few_large_frames_after_many_small_ones():
    """One context, first many frames of a small picture, then few frames of a large one with skipped blocks: the second
    batch needs fewer entries than the first but more of K3's per-chunk notes (one row per 32 frames AND position)."""
    with _ctx(capi.SCAN_AUTO) as c:
        s, o = clip(64, 48, 128, 600, key_rate=8, lm=1, cm=1, noise_y=4)
        got, _ = gpu_decode(c, s, o, 64, 48)
        want = reference_frames(s, o, 64, 48)
        assert np.array_equal(got, want), first_diff(got, want, 64, 48)
        w, h = 1280, 720
        s, o = clip(w, h, 128, 3, key_rate=2, lm=2, cm=2, noise_y=4)
        got, _ = gpu_decode(c, s, o, w, h)
        want = reference_frames(s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)


@pytest.mark.parametrize("F", [40, 400, 700])
def test_every_lane_count(F):
    """The kernel runs 256, 128 or 64 lanes a frame by the size of the batch (few frames: more lanes, shorter chunks)."""
    w, h = 176, 144
    s, o = clip(w, h, 110, F, key_rate=11, lm=1, cm=2, noise_y=9, noise_c=2)
    want = reference_frames(s, o, w, h)
    with _ctx(capi.SCAN_SYNC) as c, _ctx(capi.SCAN_CHUNK) as k:
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        e1, i1 = _entries(c, s, o, w, h)
        e2, i2 = _entries(k, s, o, w, h)
        assert np.array_equal(e1, e2) and i1 == i2


# ---- frames with a raw prefix (quality above 170): the walk's other instantiation ------------------------------------------

@pytest.mark.parametrize("Q,w,h", [(171, 208, 112), (200, 208, 112), (255, 208, 112), (255, 720, 576), (228, 1280, 720)])
def test_raw_prefix_frames_walked(Q, w, h):
    """SYNC forces the walk for every frame: pixels as the reference's, entries and counters as rtj_scan_mb_kernel's (CHUNK).
    720x576 at Q=255 is three segments a frame, 1280x720 six."""
    s, o = clip(w, h, Q, 3, noise_y=5, noise_c=2)
    assert O.tables_from_quality(Q).lb8 > 0
    want = reference_frames(s, o, w, h)
    with _ctx(capi.SCAN_SYNC) as c, _ctx(capi.SCAN_CHUNK) as k:
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        e1, i1 = _entries(c, s, o, w, h)
        e2, i2 = _entries(k, s, o, w, h)
        assert i1 == i2 and i1[2] == 0
        assert np.array_equal(e1, e2)


def test_raw_prefix_inter_stream_and_quality_changes():
    """Skip markers between blocks with a prefix, and frames with and without prefix in one batch (each kernel takes its own)."""
    w, h = 176, 144
    a = clip(w, h, 255, 6, key_rate=3, lm=2, cm=2, noise_y=6)
    b = clip(w, h, 120, 6, noise_y=6)
    c_ = clip(w, h, 190, 6, key_rate=2, lm=1, cm=1, noise_y=3, noise_c=3)
    from streams import interleave
    s, o = interleave([a, b, c_])
    want = reference_frames(s, o, w, h)
    for mode in (capi.SCAN_SYNC, capi.SCAN_AUTO):
        with _ctx(mode) as c, _ctx(capi.SCAN_CHUNK) as k:
            for _ in range(2):                                           # AUTO: the second batch expects raw-prefix frames
                got, _ = gpu_decode(c, s, o, w, h)
                assert np.array_equal(got, want), first_diff(got, want, w, h)
            e1, i1 = _entries(c, s, o, w, h)
            e2, i2 = _entries(k, s, o, w, h)
            assert i1 == i2 and np.array_equal(e1, e2)


def test_raw_prefix_dense_stream_is_given_up_under_auto():
    """Noise at a high quality: blocks of 64 bytes, a parse that never forgets.  Forced, the repair rounds get there; under
    AUTO the walk gives such frames up and rtj_scan_mb_kernel takes them -- from the third batch on in the segment-parallel
    arrangement (the host has seen that the walk does not pay)."""
    w, h = 320, 240
    s, o = clip(w, h, 255, 3, noise_y=100, noise_c=60)
    assert int(O.packet_sizes(s, o).min()) > 50 * (w // 16) * (h // 16) * 6 // 2
    want = reference_frames(s, o, w, h)
    with _ctx(capi.SCAN_SYNC) as c:
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
    with _ctx(capi.SCAN_AUTO) as c:
        for _ in range(4):
            got, _ = gpu_decode(c, s, o, w, h)
            assert np.array_equal(got, want), first_diff(got, want, w, h)
            assert c.batch_info().bad_frames == 0


@pytest.mark.parametrize("cut", [1, 5, 11, 12, 64, 1000, -1, -2, -9, -12, -63])
def test_raw_prefix_damaged_streams_same_entries_as_the_mb_kernel(cut):
    w, h = 208, 112
    s, o = clip(w, h, 255, 3, key_rate=2, lm=2, cm=2, noise_y=10)
    sizes = O.packet_sizes(s, o)
    n1 = int(sizes[1])
    keep = 12 + cut if cut > 0 else n1 + cut
    pk = [s[int(o[0]):int(o[0]) + int(sizes[0])], s[int(o[1]):int(o[1]) + keep].copy(), s[int(o[2]):int(o[2]) + int(sizes[2])]]
    pk[1][0:4] = np.frombuffer(np.uint32(pk[1].size).tobytes(), dtype=np.uint8)
    s2, o2 = O.pack_packets(pk, align=4)
    with _ctx(capi.SCAN_SYNC) as c, _ctx(capi.SCAN_CHUNK) as k:
        e1, i1 = _entries(c, s2, o2, w, h)
        e2, i2 = _entries(k, s2, o2, w, h)
    assert i1 == i2 and i1[2] == 1 and i1[3] == 1
    assert np.array_equal(e1, e2)


@pytest.mark.parametrize("fmt", [1, 2])
@pytest.mark.parametrize("Q", [190, 255])
def test_raw_prefix_other_unit_sizes(fmt, Q):
    """YUV422 (units of 2 luma + 2 chroma blocks) and 8-bit grey (every block luma): the place tables follow the format."""
    from streams import reference_frames_fmt
    w, h = 176, 144
    s, o = O.encode_clip_fmt(w, h, Q, 4, fmt, 2, 1, 1, noise_y=5, noise_c=2)
    init = np.full(O.frame_bytes(fmt, w, h), 0x3C, dtype=np.uint8)
    want = reference_frames_fmt(s, o, w, h, fmt, init)
    with _ctx(capi.SCAN_SYNC) as c:
        c.set_format(fmt)
        got, _ = gpu_decode(c, s, o, w, h, carry=init, fmt=fmt)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        assert c.batch_info().bad_frames == 0


def test_raw_prefix_few_large_frames_under_auto():
    """AUTO, batch after batch of two 1920x1088 frames at a quality of 255: the first batch knows nothing (rtj_scan_mb_kernel
    takes the frames), the second expects raw-prefix frames and -- a handful of large frames -- goes segment-parallel, and a
    batch of 40 frames of the same stream is walked.  Pixels as the reference's every time."""
    w, h = 1920, 1088
    s, o = clip(w, h, 255, 2, noise_y=4, noise_c=1)
    want = reference_frames(s, o, w, h)
    sizes = O.packet_sizes(s, o)
    pk = [s[int(o[i]):int(o[i]) + int(sizes[i])] for i in range(2)]
    s40, o40 = O.pack_packets(pk * 20)
    with _ctx(capi.SCAN_AUTO) as c:
        for _ in range(3):
            got, _ = gpu_decode(c, s, o, w, h)
            assert np.array_equal(got, want), first_diff(got, want, w, h)
            assert c.batch_info().bad_frames == 0
        got, _ = gpu_decode(c, s40, o40, w, h)
        for k in range(20):
            assert np.array_equal(got[2 * k:2 * k + 2], want), first_diff(got[2 * k:2 * k + 2], want, w, h)
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)


def test_batches_with_and_without_raw_prefix_in_turn():
    """What a batch is arranged by -- raw-prefix frames, skipped blocks in the batch before -- is a guess about THIS batch:
    one context, batches of different nature in turn, every guess wrong once.  Pixels as the reference's each time."""
    w, h = 352, 288
    clips = [clip(w, h, 255, 5, noise_y=5, noise_c=2),                       # raw prefix, intra
             clip(w, h, 128, 5, key_rate=3, lm=2, cm=2, noise_y=5),          # no prefix, skipped blocks
             clip(w, h, 200, 5, key_rate=2, lm=1, cm=1, noise_y=5),          # raw prefix, skipped blocks
             clip(w, h, 100, 5, noise_y=5)]                                  # no prefix, intra
    want = [reference_frames(s, o, w, h) for s, o in clips]
    with _ctx(capi.SCAN_AUTO) as c:
        for turn in (0, 1, 2, 3, 0, 2, 1, 3, 3, 0):
            s, o = clips[turn]
            got, _ = gpu_decode(c, s, o, w, h)
            assert np.array_equal(got, want[turn]), (turn, first_diff(got, want[turn], w, h))
            assert c.batch_info().bad_frames == 0
