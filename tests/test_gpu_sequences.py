"""rtjgpu_decode_device_seq / rtjgpu_decode_device_rgb_seq: many independent inter-coded streams in one device batch, each
with its own carry picture.  Expected frames: every sequence decoded on its own by the reference (or the restatement) from
its own picture before the first frame -- a skipped block never takes pixels from another sequence."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from gpu_util import first_diff
from streams import clip, reference_frames, reference_frames_fmt

pytestmark = pytest.mark.gpu

W, H = 160, 96
FSZ = W * H * 3 // 2

# (Q, F, keyword arguments of clip): inter clips of different seeds, qualities (255: raw prefix) and GOPs; sequences of
# length 1 and lengths that are not multiples of 32
SPECS = [
    (128, 45, dict(key_rate=14, lm=2, cm=2, dark=1, seed=1)),
    (32, 1, dict(key_rate=14, lm=4, cm=4, dark=1, seed=2)),        # one frame, skipping against the encoder's zero blocks
    (32, 33, dict(key_rate=9, lm=4, cm=4, dark=1, seed=5)),
    (255, 20, dict(key_rate=6, lm=2, cm=2, seed=7)),
    (200, 1, dict(key_rate=3, lm=2, cm=2, seed=8)),
    (128, 70, dict(key_rate=29, lm=3, cm=3, dark=1, seed=9)),
]


def _carry(seed):
    return np.random.default_rng(seed).integers(0, 256, FSZ).astype(np.uint8)


@pytest.fixture(scope="module")
def case1():
    seqs = [clip(W, H, Q, F, **kw) for Q, F, kw in SPECS]
    carries = [_carry(11), _carry(12), None, _carry(14), None, _carry(16)]      # distinct pictures and NULL
    want = np.concatenate([reference_frames(s, o, W, H, c) for (s, o), c in zip(seqs, carries)])
    return seqs, carries, want


def decode_seq(ctx, seqs, carries, w=W, h=H, fmt=0, states=None):
    b, sf = D.upload_sequences(seqs, w, h, fmt=fmt, states=states)
    b.out.fill_(0xCD)
    cts = None if carries is None else [None if c is None else torch.from_numpy(c).cuda() for c in carries]
    D.decode_sequences(ctx, b, sf, cts)
    torch.cuda.synchronize()
    assert ctx.batch_info().bad_frames == 0
    return b.out.cpu().numpy(), b, sf


def test_inter_sequences_one_call(case1):
    seqs, carries, want = case1
    with g.BatchContext(0) as ctx:
        got, _, sf = decode_seq(ctx, seqs, carries)
        assert ctx.batch_info().skipped_blocks > 0
    assert list(sf) == [0, 45, 46, 79, 99, 100, 170]
    assert np.array_equal(got, want), first_diff(got, want, W, H)


def test_no_leak_between_sequences():
    """B is dark Q=32 material whose 'key' frames still skip blocks: without the sequence boundary, its skipped blocks
    would be filled from A's frames."""
    w, h = 720, 576
    a = clip(w, h, 128, 20, key_rate=7, lm=2, cm=2, seed=3)
    bseq = clip(w, h, 32, 45, key_rate=14, lm=4, cm=4, dark=1)
    ca = np.full(w * h * 3 // 2, 0x50, dtype=np.uint8)
    cb = np.full(w * h * 3 // 2, 0x37, dtype=np.uint8)
    want_b = reference_frames(*bseq, w, h, cb)
    with g.BatchContext(0) as ctx:
        got, b, sf = decode_seq(ctx, [a, bseq], [ca, cb], w, h)
        assert np.array_equal(got[20:], want_b), first_diff(got[20:], want_b, w, h)
        # the same packets as ONE stream: B's skipped blocks come from A's last frames -- different pixels
        b.out.fill_(0xCD)
        D.decode(ctx, b, torch.from_numpy(ca).cuda())
        torch.cuda.synchronize()
        one = b.out.cpu().numpy()
    assert not np.array_equal(one[20:], want_b)


@pytest.mark.parametrize("mode", [capi.SCAN_AUTO, capi.SCAN_LANE, capi.SCAN_WARP, capi.SCAN_CHUNK, capi.SCAN_SEGMENT,
                                  capi.SCAN_WALK, capi.SCAN_SYNC])
def test_every_scan_mode(case1, mode):
    seqs, carries, want = case1
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(mode)
        got, _, _ = decode_seq(ctx, seqs, carries)
    assert np.array_equal(got, want), first_diff(got, want, W, H)


@pytest.mark.parametrize("run", [1, 2, 8, 64])
def test_frame_runs(case1, run):
    """K2 working through runs of frames: a frame that starts a sequence keeps nothing of the strip."""
    seqs, carries, want = case1
    with g.BatchContext(0) as ctx:
        ctx.set_frame_runs(run)
        got, _, _ = decode_seq(ctx, seqs, carries)
    assert np.array_equal(got, want), first_diff(got, want, W, H)


@pytest.mark.parametrize("mode", [capi.SCAN_AUTO, capi.SCAN_CHUNK])
def test_sliced_pipeline(case1, mode):
    """Slices of 32 frames: sequences start inside slices, and sequences span several of them (K3's carry_in)."""
    seqs, carries, want = case1
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(mode)
        ctx.set_pipeline(capi.PIPELINE_SLICED, 32)
        got, _, _ = decode_seq(ctx, seqs, carries)
    assert np.array_equal(got, want), first_diff(got, want, W, H)


@pytest.mark.parametrize("fmt", [1, 2])
def test_other_formats(fmt):
    fsz = O.frame_bytes(fmt, W, H)
    seqs = [O.encode_clip_fmt(W, H, 128, 40, fmt, 9, 2, 2, noise_y=4, seed=1),
            O.encode_clip_fmt(W, H, 32, 1, fmt, 3, 4, 4, dark=1, seed=2),
            O.encode_clip_fmt(W, H, 200, 35, fmt, 6, 2, 2, seed=3)]
    rng = np.random.default_rng(fmt)
    carries = [rng.integers(0, 256, fsz).astype(np.uint8), None, rng.integers(0, 256, fsz).astype(np.uint8)]
    want = np.concatenate([reference_frames_fmt(s, o, W, H, fmt, c) for (s, o), c in zip(seqs, carries)])
    with g.BatchContext(0) as ctx:
        got, _, _ = decode_seq(ctx, seqs, carries, fmt=fmt)
        assert ctx.batch_info().skipped_blocks > 0
        ctx.set_format(0)
    assert np.array_equal(got, want), first_diff(got, want, W, H)


def _expect_rgb(frames, kind, pitch, alpha):
    bpp = capi.CONV_BPP[kind]
    out = np.full((len(frames), H, pitch), 0xCD, dtype=np.uint8)
    for f, fr in enumerate(frames):
        out[f, :, :W * bpp] = (O.ref_convert if O.have_ref() else O.convert)(kind, fr, W, H, pitch=W * bpp, fill=alpha)
    return out


@pytest.mark.parametrize("kind", [capi.CONV_RGB32, capi.CONV_BGR24, capi.CONV_RGB16])
def test_fused_rgb(case1, kind):
    seqs, carries, want = case1
    bpp = capi.CONV_BPP[kind]
    pitch = (W * bpp + 15) // 16 * 16
    b, sf = D.upload_sequences(seqs, W, H)
    out = torch.full((b.F, H, pitch), 0xCD, dtype=torch.uint8, device="cuda")
    lasts = [None if s in (1, 4) else torch.full((FSZ,), 0xEE, dtype=torch.uint8, device="cuda") for s in range(len(seqs))]
    cts = [None if c is None else torch.from_numpy(c).cuda() for c in carries]
    with g.BatchContext(0) as ctx:
        ctx.set_format(0)
        ctx.decode_device_rgb_seq(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), kind, out.data_ptr(), pitch,
                                  H * pitch, 0x5A, [None if c is None else c.data_ptr() for c in cts],
                                  [None if t is None else t.data_ptr() for t in lasts], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
    assert np.array_equal(out.cpu().numpy(), _expect_rgb(want, kind, pitch, 0x5A))
    for s, t in enumerate(lasts):
        if t is not None:
            assert np.array_equal(t.cpu().numpy(), want[sf[s + 1] - 1]), s


def test_streaming_two_calls():
    """The second call's carries are each sequence's last frame in the first call's output; plan states carry over."""
    specs = [sp for sp in SPECS if sp[1] > 2]
    clips = [clip(W, H, Q, F, **kw) for Q, F, kw in specs]
    inits = [_carry(21), None, _carry(23), _carry(24)]
    want = [reference_frames(s, o, W, H, c) for (s, o), c in zip(clips, inits)]
    cut = [F // 2 for _, F, _ in specs]
    first = [(s, o[:k + 1]) for (s, o), k in zip(clips, cut)]
    second = [(s, o[k:]) for (s, o), k in zip(clips, cut)]
    states = [capi.State(0, 0, capi.TABLE_ZERO, 0) for _ in clips]
    with g.BatchContext(0) as ctx:
        got1, b1, sf1 = decode_seq(ctx, first, inits, states=states)
        b2, sf2 = D.upload_sequences(second, W, H, states=states)
        b2.out.fill_(0xCD)
        ctx.decode_device_seq(b2.stream.data_ptr(), b2.desc.data_ptr(), b2.F, W, H, list(sf2), b2.out.data_ptr(),
                              [b1.out[int(sf1[s + 1]) - 1].data_ptr() for s in range(len(clips))],
                              torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got2 = b2.out.cpu().numpy()
    for s in range(len(clips)):
        got = np.concatenate([got1[sf1[s]:sf1[s + 1]], got2[sf2[s]:sf2[s + 1]]])
        assert np.array_equal(got, want[s]), (s, first_diff(got, want[s], W, H))


def test_shards_in_one_call():
    """A config5-style stream cut by rtjgpu_split_shards_lead; every shard, lead-in frames included, is one sequence of a
    single call: garbage before every shard but the one that starts at frame 0."""
    w, h, F, n = 720, 576, 120, 8
    s, o = clip(w, h, 128, F, key_rate=29, lm=4, cm=4)
    init = np.full(w * h * 3 // 2, 0x62, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    garbage = np.random.default_rng(5).integers(0, 256, w * h * 3 // 2).astype(np.uint8)
    with g.BatchContext(0) as ctx:
        desc, _ = g.plan(s, o)
        bt = D.upload(s, desc, w, h)
        ctx.scan_device(bt.stream.data_ptr(), bt.desc.data_ptr(), F, w, h, torch.cuda.current_stream().cuda_stream)
        clean = (ctx.skip_counts(F) == 0).astype(np.uint8)
        first, lead = g.split_shards_lead(clean, n)
        assert (lead > 0).any()
        starts = [int(first[i] - lead[i]) for i in range(n)]
        seqs = [(s, o[a:int(first[i + 1]) + 1]) for i, a in enumerate(starts)]
        got, _, sf = decode_seq(ctx, seqs, [init if a == 0 else garbage for a in starts], w, h)
    for i in range(n):
        kept = got[int(sf[i]) + int(lead[i]):int(sf[i + 1])]
        assert np.array_equal(kept, want[int(first[i]):int(first[i + 1])]), (i, first_diff(kept, want[int(first[i]):int(first[i + 1])], w, h))


def test_one_sequence_is_decode_device(case1):
    seqs, carries, _ = case1
    s, o = seqs[0]
    ct = torch.from_numpy(carries[0]).cuda()
    with g.BatchContext(0) as ctx:
        b, sf = D.upload_sequences([seqs[0]], W, H)
        D.decode(ctx, b, ct)                                   # warm-up: position table, skip statistics of the stream
        torch.cuda.synchronize()
        n0 = ctx.launch_count()
        b.out.fill_(0xCD)
        D.decode(ctx, b, ct)
        torch.cuda.synchronize()
        n1 = ctx.launch_count()
        one = b.out.cpu().numpy()
        b.out.fill_(0xCD)
        D.decode_sequences(ctx, b, sf, [ct])
        torch.cuda.synchronize()
        n2 = ctx.launch_count()
        seq = b.out.cpu().numpy()
    assert list(sf) == [0, len(o) - 1]
    assert np.array_equal(seq, one)
    assert n2 - n1 == n1 - n0


def test_invalid_arguments():
    a, b2 = clip(64, 48, 128, 3, key_rate=2, lm=2, cm=2), clip(64, 48, 128, 2, key_rate=2, lm=2, cm=2, seed=2)
    b, sf = D.upload_sequences([a, b2], 64, 48)
    carry = torch.zeros(64 * 48 * 3 // 2 + 16, dtype=torch.uint8, device="cuda")
    rgb = torch.empty((5, 48, 64 * 4), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf)
        torch.cuda.synchronize()
        n0 = ctx.launch_count()

        def call(first, carries=None, F=5):
            ctx.decode_device_seq(b.stream.data_ptr(), b.desc.data_ptr(), F, 64, 48, first, b.out.data_ptr(), carries, st)

        def call_rgb(first, carries=None, last=None):
            ctx.decode_device_rgb_seq(b.stream.data_ptr(), b.desc.data_ptr(), 5, 64, 48, first, capi.CONV_RGB32, rgb.data_ptr(),
                                      64 * 4, 48 * 64 * 4, 0, carries, last, st)

        bad = [lambda: call([0]),                                     # S = 0
               lambda: call([0, 1, 2, 3], F=2),                       # S > F
               lambda: call([1, 3, 5]),                               # seq_first[0] != 0
               lambda: call([0, 3, 4]),                               # seq_first[S] != F
               lambda: call([0, 3, 3, 5]),                            # an empty sequence
               lambda: call([0, 4, 3, 5]),                            # not increasing
               lambda: call([0, 3, 5], [carry.data_ptr(), carry.data_ptr() + 4]),      # misaligned carry
               lambda: call_rgb([0, 3, 5], None, [carry.data_ptr(), carry.data_ptr() + 8]),   # misaligned last_yuv
               lambda: call_rgb([0, 2, 6])]
        for i, fn in enumerate(bad):
            with pytest.raises(g.RTjpegError) as e:
                fn()
            assert e.value.code == capi.E_ARG, i
        torch.cuda.synchronize()
        assert ctx.launch_count() == n0
        ctx.set_format(1)
        with pytest.raises(g.RTjpegError) as e:
            call_rgb([0, 3, 5])
        assert e.value.code == capi.E_FORMAT
        assert ctx.launch_count() == n0
