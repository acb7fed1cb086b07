"""The sliced / pipelined arrangement of a device batch (rtjgpu_set_pipeline): K1 of slice s + 1 beside K3 / K2 of
slice s on two streams, and K3's slice-to-slice hand-over of last writers.  Bit-exact against the reference in every
arrangement, with slices small enough that these short clips cross many of them."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from oracle import oracle as O
from gpu_util import first_diff, gpu_decode
from streams import clip, reference_frames

pytestmark = pytest.mark.gpu


def _ctx(pipeline, slice_frames, scan=capi.SCAN_CHUNK):
    c = g.BatchContext(0)
    c.set_scan_mode(scan)                  # one CTA per frame even for these small batches: the arrangement that is sliced
    c.set_pipeline(pipeline, slice_frames)
    return c


ARRANGEMENTS = [(capi.PIPELINE_SLICED, 32), (capi.PIPELINE_SLICED, 64), (capi.PIPELINE_SLICED, 96), (capi.PIPELINE_SERIAL, 32),
                (capi.PIPELINE_SERIAL, 576)]


def splice(w, h, base_pkt, keep):
    """A packet made of base_pkt's blocks where keep[b], of skip markers elsewhere (built from the grammar only:
    the oracle's walker says where the blocks of base_pkt start)."""
    nmb = (w // 16) * (h // 16)
    pay = base_pkt[12:]
    n, offs, _ = O.walk_payload(pay, nmb, 0, 0)
    ends = list(offs[1:]) + [n]
    out = bytearray(base_pkt[:12].tobytes())
    for b in range(nmb * 6):
        out += pay[int(offs[b]):int(ends[b])].tobytes() if keep[b] else b"\xff"
    pkt = np.frombuffer(bytes(out), dtype=np.uint8).copy()
    pkt[0:4] = np.frombuffer(np.uint32(len(pkt)).tobytes(), dtype=np.uint8)
    return pkt


@pytest.mark.parametrize("pipeline,slice_frames", ARRANGEMENTS)
def test_inter_clip_across_slices(pipeline, slice_frames):
    w, h, F = 320, 240, 200
    s, o = clip(w, h, 128, F, key_rate=29, lm=3, cm=3)
    init = np.full(w * h * 3 // 2, 0x41, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    with _ctx(pipeline, slice_frames) as c:
        got, _ = gpu_decode(c, s, o, w, h, carry=init)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        bi = c.batch_info()
        assert bi.bad_frames == 0 and bi.skipped_blocks > 0
        # the per-frame skip counts are the clean-frame detector of the multi-GPU split
        counts = c.skip_counts(F)
        assert int(counts.sum()) == bi.skipped_blocks and counts[0] == 0 and counts[30] == 0


@pytest.mark.parametrize("pipeline,slice_frames", ARRANGEMENTS)
def test_last_writer_many_chunks_back(pipeline, slice_frames):
    """Frame 0 coded; 130 frames of skip markers only; then partial updates: the last writer of most blocks lies four
    resolve chunks (and, with small slices, several slices) back; positions updated once keep that writer afterwards."""
    w, h = 160, 96
    nblk = (w // 16) * (h // 16) * 6
    s, o = clip(w, h, 128, 12)                                   # intra frames to take blocks from
    sizes = O.packet_sizes(s, o)
    base = [s[int(o[f]):int(o[f]) + int(sizes[f])] for f in range(12)]
    rng = np.random.default_rng(7)
    pkts = [base[0]]
    pkts += [splice(w, h, base[1], np.zeros(nblk, bool)) for _ in range(130)]
    for t in range(40):                                          # sparse updates, a different tenth of the picture each
        pkts.append(splice(w, h, base[2 + t % 10], rng.random(nblk) < 0.1))
    pkts += [splice(w, h, base[1], np.zeros(nblk, bool)) for _ in range(70)]
    pkts.append(splice(w, h, base[11], rng.random(nblk) < 0.5))
    st, of = O.pack_packets(pkts)
    init = np.full(w * h * 3 // 2, 0x99, dtype=np.uint8)
    want = reference_frames(st, of, w, h, init)
    with _ctx(pipeline, slice_frames) as c:
        got, _ = gpu_decode(c, st, of, w, h, carry=init)
        assert np.array_equal(got, want), first_diff(got, want, w, h)


@pytest.mark.parametrize("pipeline,slice_frames", [(capi.PIPELINE_SLICED, 32), (capi.PIPELINE_SERIAL, 64)])
def test_never_written_positions_take_the_carry(pipeline, slice_frames):
    """No frame of the batch writes the left half of the picture: those blocks come from the picture before the
    batch in every slice."""
    w, h = 160, 96
    nblk = (w // 16) * (h // 16) * 6
    s, o = clip(w, h, 128, 4)
    sizes = O.packet_sizes(s, o)
    base = [s[int(o[f]):int(o[f]) + int(sizes[f])] for f in range(4)]
    mbx = (np.arange(nblk) // 6) % (w // 16)
    right = mbx >= (w // 32)
    rng = np.random.default_rng(11)
    pkts = [splice(w, h, base[t % 4], right & (rng.random(nblk) < 0.3)) for t in range(150)]
    st, of = O.pack_packets(pkts)
    init = rng.integers(16, 236, w * h * 3 // 2).astype(np.uint8)
    want = reference_frames(st, of, w, h, init)
    with _ctx(pipeline, slice_frames) as c:
        got, _ = gpu_decode(c, st, of, w, h, carry=init)
        assert np.array_equal(got, want), first_diff(got, want, w, h)


def test_pipelined_equals_serial_on_the_bench_shape():
    """720x576 Q128 intra, 1300 frames: two and a quarter slices of the default size, pipelined, against the
    serial arrangement of the same library and against the reference on a sample of frames."""
    w, h, F = 720, 576, 1300
    s, o = clip(w, h, 128, F)
    with _ctx(capi.PIPELINE_SERIAL, 0, scan=capi.SCAN_AUTO) as c:
        serial, _ = gpu_decode(c, s, o, w, h)
    with _ctx(capi.PIPELINE_SLICED, 0, scan=capi.SCAN_AUTO) as c:
        piped, _ = gpu_decode(c, s, o, w, h)
        assert c.batch_info().bad_frames == 0
    assert np.array_equal(serial, piped)
    for f in (0, 575, 576, 1151, 1152, 1299):
        want = reference_frames(s[int(o[f]):int(o[f + 1])], np.array([0, int(o[f + 1]) - int(o[f])], dtype=np.uint64), w, h)
        assert np.array_equal(piped[f], want[0]), f


# ---- the walker flavour of K1 (rtj_scan_walk.cu): one lane per frame, payload staged through shared memory ----------

@pytest.fixture
def walker():
    c = g.BatchContext(0)
    c.set_scan_mode(capi.SCAN_WALK)
    yield c
    c.close()


def test_walker_inter_clip(walker):
    w, h, F = 320, 240, 200
    s, o = clip(w, h, 128, F, key_rate=29, lm=3, cm=3)
    init = np.full(w * h * 3 // 2, 0x41, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    got, _ = gpu_decode(walker, s, o, w, h, carry=init)
    assert np.array_equal(got, want), first_diff(got, want, w, h)
    bi = walker.batch_info()
    assert bi.bad_frames == 0 and bi.skipped_blocks > 0
    assert bi.payload_bytes == int(O.packet_sizes(s, o).astype(np.int64).sum()) - 12 * F
    counts = walker.skip_counts(F)
    assert int(counts.sum()) == bi.skipped_blocks and counts[0] == 0 and counts[30] == 0


def test_walker_intra_bench_shape(walker):
    w, h, F = 720, 576, 40
    s, o = clip(w, h, 128, F)
    want = reference_frames(s, o, w, h)
    got, _ = gpu_decode(walker, s, o, w, h)
    assert np.array_equal(got, want), first_diff(got, want, w, h)
    assert walker.batch_info().skipped_blocks == 0


def test_walker_long_static_stretch(walker):
    """Frame 0 coded, 130 frames of skip markers only, then sparse updates: K3's running maximum over the chunks."""
    w, h = 160, 96
    nblk = (w // 16) * (h // 16) * 6
    s, o = clip(w, h, 128, 12)
    sizes = O.packet_sizes(s, o)
    base = [s[int(o[f]):int(o[f]) + int(sizes[f])] for f in range(12)]
    rng = np.random.default_rng(7)
    pkts = [splice(w, h, base[1], rng.random(nblk) < 0.5)]          # not even frame 0 writes everything: the carry shows through
    pkts += [splice(w, h, base[1], np.zeros(nblk, bool)) for _ in range(130)]
    pkts += [splice(w, h, base[2 + t % 10], rng.random(nblk) < 0.1) for t in range(40)]
    st, of = O.pack_packets(pkts)
    init = rng.integers(16, 236, w * h * 3 // 2).astype(np.uint8)
    want = reference_frames(st, of, w, h, init)
    got, _ = gpu_decode(walker, st, of, w, h, carry=init)
    assert np.array_equal(got, want), first_diff(got, want, w, h)


def test_walker_leaves_raw_prefix_frames_to_the_other_scan(walker):
    """Q=255 frames (raw prefix 9: another grammar) between Q=128 frames, inter-coded: both scans feed the same slices."""
    from streams import interleave
    w, h, F = 160, 96, 24
    a = clip(w, h, 128, F, key_rate=5, lm=2, cm=2)
    b = clip(w, h, 255, F, key_rate=5, lm=2, cm=2, seed=3)
    st, of = interleave([a, b])
    init = np.full(w * h * 3 // 2, 0x70, dtype=np.uint8)
    want = reference_frames(st, of, w, h, init)
    got, _ = gpu_decode(walker, st, of, w, h, carry=init)
    assert np.array_equal(got, want), first_diff(got, want, w, h)
    assert walker.batch_info().bad_frames == 0


def test_walker_flags_truncated_frames(walker):
    w, h, F = 160, 96, 9
    s, o = clip(w, h, 128, F)
    sizes = O.packet_sizes(s, o).astype(np.int64)
    pk = [s[int(o[f]):int(o[f]) + int(sizes[f])].copy() for f in range(F)]
    for f, cut in ((2, 0.5), (5, 0.1), (7, 0.97)):
        n = 12 + int((len(pk[f]) - 12) * cut)
        pk[f] = pk[f][:n].copy()
        pk[f][0:4] = np.frombuffer(np.uint32(n).tobytes(), dtype=np.uint8)
    st, of = O.pack_packets(pk)
    got, _ = gpu_decode(walker, st, of, w, h)
    bi = walker.batch_info()
    assert bi.bad_frames == 3 and bi.first_bad_frame == 2
    want = reference_frames(s, o, w, h)
    for f in (0, 1, 3, 4, 6, 8):
        assert np.array_equal(got[f], want[f]), f


@pytest.mark.parametrize("fmt", [1, 2])
def test_walker_other_formats(walker, fmt):
    from streams import reference_frames_fmt
    w, h, F = 96, 64, 20
    s, o = O.encode_clip_fmt(w, h, 128, F, fmt, key_rate=4, lm=2, cm=2)
    init = np.full(O.frame_bytes(fmt, w, h), 0x50, dtype=np.uint8)
    want = reference_frames_fmt(s, o, w, h, fmt, init=init)
    got, _ = gpu_decode(walker, s, o, w, h, carry=init, fmt=fmt)
    assert np.array_equal(got, want)
