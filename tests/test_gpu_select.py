"""rtjgpu_decode_device_select / rtjgpu_decode_device_rgb_select: only the frames a caller asks for, out of a device batch of
many independent sequences.  Expected frames: every sequence decoded on its own by the reference (or the restatement) from
its own picture before the first frame, at the selected rows.  Output buffers are poisoned with 0xCD and carry one guard
frame behind the last slot, which must stay poisoned: nothing but the selected frames is written."""
import ctypes as C

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
POISON = 0xCD

# (Q, F, keyword arguments of clip): inter clips of different seeds, qualities (255: raw prefix, every luma block through
# K2b's queue) and GOPs; sequences of length 1 and lengths that are not multiples of 32
SPECS = [
    (128, 45, dict(key_rate=14, lm=2, cm=2, dark=1, seed=1)),
    (32, 1, dict(key_rate=14, lm=4, cm=4, dark=1, seed=2)),
    (32, 33, dict(key_rate=9, lm=4, cm=4, dark=1, seed=5)),
    (255, 20, dict(key_rate=6, lm=2, cm=2, seed=7)),
    (200, 1, dict(key_rate=3, lm=2, cm=2, seed=8)),
    (128, 70, dict(key_rate=29, lm=3, cm=3, dark=1, seed=9)),
]


def _carry(seed, fsz=FSZ):
    return np.random.default_rng(seed).integers(0, 256, fsz).astype(np.uint8)


@pytest.fixture(scope="module")
def case1():
    seqs = [clip(W, H, Q, F, **kw) for Q, F, kw in SPECS]
    carries = [_carry(11), _carry(12), None, _carry(14), None, _carry(16)]      # distinct pictures and NULL
    want = np.concatenate([reference_frames(s, o, W, H, c) for (s, o), c in zip(seqs, carries)])
    return seqs, carries, want


def _dev(carries):
    return None if carries is None else [None if c is None else torch.from_numpy(c).cuda() for c in carries]


def _lengths(sf):
    return [int(sf[s + 1] - sf[s]) for s in range(len(sf) - 1)]


def run_select(ctx, b, sf, sel, cts):
    """One select call into a poisoned buffer of n + 1 frames; returns the n frames, checks the guard frame."""
    sel = np.asarray(sel, dtype=np.int64)
    out = torch.full((len(sel) + 1, b.frame_bytes), POISON, dtype=torch.uint8, device="cuda")
    D.decode_select(ctx, b, sf, sel, cts, out=out)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert (got[len(sel)] == POISON).all(), "the call wrote behind its last slot"
    return got[:len(sel)]


def check(got, want, sel, w=W, h=H):
    exp = want[np.asarray(sel, dtype=np.int64)]
    assert np.array_equal(got, exp), first_diff(got, exp, w, h)


PICKS = {
    "every2": lambda n, rng: np.arange(0, n, 2),
    "every3_from1": lambda n, rng: np.arange(1, n, 3),
    "every7": lambda n, rng: np.arange(0, n, 7),
    "random_a": lambda n, rng: np.flatnonzero(rng.random(n) < 0.3),
    "random_b": lambda n, rng: rng.permutation(n)[:max(1, n // 5)],
    "first": lambda n, rng: np.array([0]),
    "last": lambda n, rng: np.array([n - 1]),
}


@pytest.mark.parametrize("pick", list(PICKS))
def test_selection_matches_reference(case1, pick):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    rng = np.random.default_rng(sum(map(ord, pick)))
    sel = g.select_frames(sf, [PICKS[pick](n, rng) for n in _lengths(sf)])
    with g.BatchContext(0) as ctx:
        got = run_select(ctx, b, sf, sel, _dev(carries))
        bi = ctx.batch_info()
        assert bi.bad_frames == 0 and bi.skipped_blocks > 0
    check(got, want, sel)


def test_all_frames_is_the_seq_call(case1):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    cts = _dev(carries)
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf, cts)                      # warm-up: position table, skip statistics of the stream
        torch.cuda.synchronize()
        n0 = ctx.launch_count()
        b.out.fill_(POISON)
        D.decode_sequences(ctx, b, sf, cts)
        torch.cuda.synchronize()
        n1 = ctx.launch_count()
        full = b.out.cpu().numpy()
        got = run_select(ctx, b, sf, np.arange(b.F), cts)
        n2 = ctx.launch_count()
    assert np.array_equal(got, full)
    assert np.array_equal(got, want), first_diff(got, want, W, H)
    assert n2 - n1 == n1 - n0                                    # the full call's launches, runs of frames included


def test_streaming_three_calls():
    """Each call selects every third frame of each sequence and its last frame; the next call's carries are the previous
    call's outputs of those last frames.  Plan states carry over."""
    specs = [sp for sp in SPECS if sp[1] > 3]
    clips = [clip(W, H, Q, F, **kw) for Q, F, kw in specs]
    inits = [_carry(21), None, _carry(23), _carry(24)]
    want = [reference_frames(s, o, W, H, c) for (s, o), c in zip(clips, inits)]
    cuts = [[0, F // 3, 2 * F // 3, F] for _, F, _ in specs]
    states = [capi.State(0, 0, capi.TABLE_ZERO, 0) for _ in clips]
    cts = _dev(inits)
    with g.BatchContext(0) as ctx:
        for call in range(3):
            batch = [(s, o[c[call]:c[call + 1] + 1]) for (s, o), c in zip(clips, cuts)]
            b, sf = D.upload_sequences(batch, W, H, states=states)
            picks = [np.union1d(np.arange(call, n, 3), [n - 1]) for n in _lengths(sf)]
            sel = g.select_frames(sf, picks)
            out = torch.full((len(sel) + 1, FSZ), POISON, dtype=torch.uint8, device="cuda")
            D.decode_select(ctx, b, sf, sel, cts, out=out)
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            assert (got[len(sel)] == POISON).all()
            k = 0
            for s in range(len(clips)):
                for i in picks[s]:
                    f = cuts[s][call] + int(i)
                    assert np.array_equal(got[k], want[s][f]), (call, s, f, first_diff(got[k:k + 1], want[s][f:f + 1], W, H))
                    k += 1
            # each sequence's last frame is the next call's carry
            last_slot = np.searchsorted(sel, np.asarray(sf[1:]) - 1)
            cts = [out[int(j)] for j in last_slot]


def splice(w, h, base_pkt, keep):
    """A packet made of base_pkt's blocks where keep[b], of skip markers elsewhere (built from the grammar only: the
    oracle's walker says where the blocks of base_pkt start)."""
    nmb = (w // 16) * (h // 16)
    pay = base_pkt[12:]
    n, offs, _ = O.walk_payload(pay, nmb, 0, 0)
    ends = list(offs[1:]) + [n]
    out = bytearray(base_pkt[:12].tobytes())
    for bl in range(nmb * 6):
        out += pay[int(offs[bl]):int(ends[bl])].tobytes() if keep[bl] else b"\xff"
    pkt = np.frombuffer(bytes(out), dtype=np.uint8).copy()
    pkt[0:4] = np.frombuffer(np.uint32(len(pkt)).tobytes(), dtype=np.uint8)
    return pkt


@pytest.mark.parametrize("pipeline,slice_frames", [(capi.PIPELINE_SERIAL, 0), (capi.PIPELINE_SLICED, 32)])
def test_far_last_writer_and_carry(pipeline, slice_frames):
    """Frame 0 codes half the blocks, 130 frames of skip markers follow, then sparse updates: a selected frame 120 takes
    half its blocks from frame 0 (four K3 chunks back) and the other half from the carry, which no frame before it wrote."""
    nblk = (W // 16) * (H // 16) * 6
    s, o = clip(W, H, 128, 12)
    sizes = O.packet_sizes(s, o)
    base = [s[int(o[f]):int(o[f]) + int(sizes[f])] for f in range(12)]
    rng = np.random.default_rng(7)
    pkts = [splice(W, H, base[1], rng.random(nblk) < 0.5)]
    pkts += [splice(W, H, base[1], np.zeros(nblk, bool)) for _ in range(130)]
    pkts += [splice(W, H, base[2 + t % 10], rng.random(nblk) < 0.1) for t in range(40)]
    st, of = O.pack_packets(pkts)
    other = clip(W, H, 128, 30, key_rate=14, lm=2, cm=2, seed=4)
    inits = [_carry(31), _carry(32)]
    want = np.concatenate([reference_frames(st, of, W, H, inits[0]), reference_frames(*other, W, H, inits[1])])
    b, sf = D.upload_sequences([(st, of), other], W, H)
    sel = g.select_frames(sf, [[120, 130, 131, 150, 170], [0, 29]])
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(capi.SCAN_CHUNK)
        ctx.set_pipeline(pipeline, slice_frames)
        got = run_select(ctx, b, sf, sel, _dev(inits))
    check(got, want, sel)


@pytest.mark.parametrize("mode", [capi.SCAN_AUTO, capi.SCAN_LANE, capi.SCAN_WARP, capi.SCAN_CHUNK, capi.SCAN_SEGMENT,
                                  capi.SCAN_WALK, capi.SCAN_SYNC])
def test_every_scan_mode(case1, mode):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    sel = g.select_frames(sf, [np.arange(n - 1, -1, -3) for n in _lengths(sf)])
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(mode)
        got = run_select(ctx, b, sf, sel, _dev(carries))
    check(got, want, sel)


@pytest.mark.parametrize("mode", [capi.SCAN_AUTO, capi.SCAN_CHUNK])
def test_sliced_pipeline_with_empty_slices(case1, mode):
    """Slices of 32 frames; [32, 64) and [64, 96) hold no selected frame (their K2 launch is left out)."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    sel = np.array([3, 10, 31, 99, 100, 101, 140, 169])
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(mode)
        ctx.set_pipeline(capi.PIPELINE_SLICED, 32)
        got = run_select(ctx, b, sf, sel, _dev(carries))
    check(got, want, sel)


def test_frame_runs_setting_does_not_matter(case1):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    sel = g.select_frames(sf, [np.arange(0, n, 4) for n in _lengths(sf)])
    outs = []
    with g.BatchContext(0) as ctx:
        for run in (1, 8, 64):
            ctx.set_frame_runs(run)
            outs.append(run_select(ctx, b, sf, sel, _dev(carries)))
    for got in outs:
        assert np.array_equal(got, outs[0])
    check(outs[0], want, sel)


@pytest.mark.parametrize("fmt", [1, 2])
def test_other_formats(fmt):
    fsz = O.frame_bytes(fmt, W, H)
    seqs = [O.encode_clip_fmt(W, H, 128, 40, fmt, 9, 2, 2, noise_y=4, seed=1),
            O.encode_clip_fmt(W, H, 32, 1, fmt, 3, 4, 4, dark=1, seed=2),
            O.encode_clip_fmt(W, H, 200, 35, fmt, 6, 2, 2, seed=3)]
    rng = np.random.default_rng(fmt)
    carries = [rng.integers(0, 256, fsz).astype(np.uint8), None, rng.integers(0, 256, fsz).astype(np.uint8)]
    want = np.concatenate([reference_frames_fmt(s, o, W, H, fmt, c) for (s, o), c in zip(seqs, carries)])
    b, sf = D.upload_sequences(seqs, W, H, fmt=fmt)
    sel = g.select_frames(sf, [np.arange(1, n, 3) if n > 1 else [0] for n in _lengths(sf)])
    with g.BatchContext(0) as ctx:
        got = run_select(ctx, b, sf, sel, _dev(carries))
        ctx.set_format(0)
    check(got, want, sel)


def test_high_quality_hard_queue():
    """Q = 255: every luma block goes through K2b's queue, whose records name the output slot, not the frame."""
    seqs = [clip(W, H, 255, 40, key_rate=9, lm=2, cm=2, seed=3), clip(W, H, 255, 25, key_rate=4, lm=2, cm=2, seed=6)]
    carries = [_carry(41), _carry(42)]
    want = np.concatenate([reference_frames(s, o, W, H, c) for (s, o), c in zip(seqs, carries)])
    b, sf = D.upload_sequences(seqs, W, H)
    sel = g.select_frames(sf, [[5, 17, 30, 39], [0, 12, 24]])
    with g.BatchContext(0) as ctx:
        got = run_select(ctx, b, sf, sel, _dev(carries))
    check(got, want, sel)


def test_wide_picture_strips():
    """2080 px: wider than one CTA's strip of 128 macroblocks, so the strip instantiations run (planes and fused RGB)."""
    w, h = 2080, 32
    fsz = w * h * 3 // 2
    seqs = [clip(w, h, 128, 12, key_rate=5, lm=2, cm=2, seed=1), clip(w, h, 200, 9, key_rate=3, lm=2, cm=2, seed=2)]
    carries = [_carry(51, fsz), _carry(52, fsz)]
    want = np.concatenate([reference_frames(s, o, w, h, c) for (s, o), c in zip(seqs, carries)])
    b, sf = D.upload_sequences(seqs, w, h)
    sel = g.select_frames(sf, [[1, 4, 11], [0, 7]])
    with g.BatchContext(0) as ctx:
        got = run_select(ctx, b, sf, sel, _dev(carries))
        check(got, want, sel, w, h)
        kind, pitch = capi.CONV_RGB32, w * 4 + 16
        out = torch.full((len(sel) + 1, h, pitch), POISON, dtype=torch.uint8, device="cuda")
        lasts = [torch.full((fsz,), 0xEE, dtype=torch.uint8, device="cuda") for _ in seqs]
        cts = _dev(carries)
        ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, w, h, list(sf), list(sel), kind, out.data_ptr(),
                                     pitch, h * pitch, 0x5A, [c.data_ptr() for c in cts], [t.data_ptr() for t in lasts],
                                     torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert np.array_equal(got[:len(sel)], _expect_rgb(want[sel], kind, pitch, 0x5A, w, h))
    assert (got[len(sel)] == POISON).all()
    for s, t in enumerate(lasts):
        assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s


def _expect_rgb(frames, kind, pitch, alpha, w=W, h=H):
    bpp = capi.CONV_BPP[kind]
    out = np.full((len(frames), h, pitch), POISON, dtype=np.uint8)
    for f, fr in enumerate(frames):
        out[f, :, :w * bpp] = (O.ref_convert if O.have_ref() else O.convert)(kind, fr, w, h, pitch=w * bpp, fill=alpha)
    return out


@pytest.mark.parametrize("kind", [capi.CONV_RGB32, capi.CONV_BGR32, capi.CONV_RGB24, capi.CONV_BGR24, capi.CONV_RGB16])
def test_fused_rgb(case1, kind):
    """Padded pitches; last_yuv for every sequence but one, the last frames of sequences 0 and 3 selected, those of 2 and 5
    not (decoded to planes only), sequences 1 and 4 of one frame each."""
    seqs, carries, want = case1
    bpp = capi.CONV_BPP[kind]
    pitch = (W * bpp + 15) // 16 * 16 + 32
    b, sf = D.upload_sequences(seqs, W, H)
    n = _lengths(sf)
    picks = [[0, 10, n[0] - 1], [0], [2, 20], [n[3] - 1], [], [5, 33, 34]]
    sel = g.select_frames(sf, picks)
    out = torch.full((len(sel) + 1, H, pitch), POISON, dtype=torch.uint8, device="cuda")
    lasts = [None if s == 4 else torch.full((FSZ,), 0xEE, dtype=torch.uint8, device="cuda") for s in range(len(seqs))]
    cts = _dev(carries)
    with g.BatchContext(0) as ctx:
        ctx.set_format(0)
        ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), list(sel), kind, out.data_ptr(),
                                     pitch, H * pitch, 0x5A, [None if c is None else c.data_ptr() for c in cts],
                                     [None if t is None else t.data_ptr() for t in lasts], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
    got = out.cpu().numpy()
    assert np.array_equal(got[:len(sel)], _expect_rgb(want[sel], kind, pitch, 0x5A))
    assert (got[len(sel)] == POISON).all()
    for s, t in enumerate(lasts):
        if t is not None:
            assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s


def test_fused_rgb_nothing_selected_advances_the_streams(case1):
    """n = 0 with no RGB buffer at all (d_rgb NULL): every sequence's last frame still leaves as planes into its last_yuv --
    the streams advance by one batch and no picture is kept."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    lasts = [None if s == 4 else torch.full((FSZ + 16,), POISON, dtype=torch.uint8, device="cuda") for s in range(len(seqs))]
    cts = _dev(carries)
    with g.BatchContext(0) as ctx:
        ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), [], capi.CONV_RGB32, None,
                                     W * 4, H * W * 4, 0, [None if c is None else c.data_ptr() for c in cts],
                                     [None if t is None else t.data_ptr() for t in lasts], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
    for s, t in enumerate(lasts):
        if t is not None:
            got = t.cpu().numpy()
            assert np.array_equal(got[:FSZ], want[int(sf[s + 1]) - 1]), s
            assert (got[FSZ:] == POISON).all(), s


def test_one_sequence():
    """S = 1 (seq_first = {0, F}): the job list goes up alone and K2 takes the one carry and the batch's last frame as the
    sequence's.  Planes at a sparse selection; fused RGB with last_yuv where the last frame is not selected; and n = 0 with
    only last_yuv."""
    s, o = clip(W, H, 128, 50, key_rate=14, lm=2, cm=2, dark=1, seed=3)
    init = _carry(71)
    want = reference_frames(s, o, W, H, init)
    b, sf = D.upload_sequences([(s, o)], W, H)
    assert list(sf) == [0, 50]
    ct = torch.from_numpy(init).cuda()
    sel = np.array([0, 7, 31, 32, 48])
    kind, pitch = capi.CONV_BGR24, W * 3 + 16
    st = torch.cuda.current_stream().cuda_stream
    with g.BatchContext(0) as ctx:
        got = run_select(ctx, b, sf, sel, [ct])
        check(got, want, sel)
        out = torch.full((len(sel) + 1, H, pitch), POISON, dtype=torch.uint8, device="cuda")
        last = torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda")
        ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), list(sel), kind, out.data_ptr(),
                                     pitch, H * pitch, 0x33, [ct.data_ptr()], [last.data_ptr()], st)
        torch.cuda.synchronize()
        rgb = out.cpu().numpy()
        assert np.array_equal(rgb[:len(sel)], _expect_rgb(want[sel], kind, pitch, 0x33))
        assert (rgb[len(sel)] == POISON).all()
        assert np.array_equal(last.cpu().numpy(), want[49])
        last.fill_(POISON)
        ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), [], kind, None,
                                     pitch, H * pitch, 0, [ct.data_ptr()], [last.data_ptr()], st)
        torch.cuda.synchronize()
        assert np.array_equal(last.cpu().numpy(), want[49])


def test_many_sequences_at_720x576():
    """64 sequences of 8 frames, each starting anywhere in a GOP of one of two clips, every fourth frame selected."""
    w, h, k = 720, 576, 8
    fsz = w * h * 3 // 2
    clips = [clip(w, h, 128, 40, key_rate=29, lm=2, cm=2, seed=seed) for seed in (1, 2)]
    seqs = []
    for s in range(64):
        cs, co = clips[s % 2]
        a = (s * 7) % (40 - k + 1)
        seqs.append((cs, co[a:a + k + 1]))
    init = _carry(61, fsz)
    b, sf = D.upload_sequences(seqs, w, h)
    sel = g.select_frames(sf, [np.arange(s % 4, k, 4) for s in range(64)])
    with g.BatchContext(0) as ctx:
        got = run_select(ctx, b, sf, sel, [torch.from_numpy(init).cuda()] * 64)
    k_at = 0
    for s, (cs, co) in enumerate(seqs):
        want = reference_frames(cs, co, w, h, init)
        for i in range(s % 4, k, 4):
            assert np.array_equal(got[k_at], want[i]), (s, i, first_diff(got[k_at:k_at + 1], want[i:i + 1], w, h))
            k_at += 1
    assert k_at == len(sel)


def test_nothing_selected_and_batch_info(case1):
    """n = 0: the batch is scanned and resolved, nothing is written.  After any select call, batch info and skip counts
    describe all F frames, as after the full call."""
    seqs, carries, _ = case1
    b, sf = D.upload_sequences(seqs, W, H)
    cts = _dev(carries)
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf, cts)
        torch.cuda.synchronize()
        bi = ctx.batch_info()
        full = (bi.skipped_blocks, bi.payload_bytes, bi.bad_frames, bi.first_bad_frame)
        counts = ctx.skip_counts(b.F)
        assert full[0] > 0
        for sel in (np.zeros(0, dtype=np.int64), g.select_frames(sf, [np.arange(0, n, 4) for n in _lengths(sf)])):
            got = run_select(ctx, b, sf, sel, cts)
            assert got.shape[0] == len(sel)
            bi = ctx.batch_info()
            assert (bi.skipped_blocks, bi.payload_bytes, bi.bad_frames, bi.first_bad_frame) == full
            assert np.array_equal(ctx.skip_counts(b.F), counts)


def test_invalid_arguments():
    a, b2 = clip(64, 48, 128, 3, key_rate=2, lm=2, cm=2), clip(64, 48, 128, 2, key_rate=2, lm=2, cm=2, seed=2)
    b, sf = D.upload_sequences([a, b2], 64, 48)
    fsz = 64 * 48 * 3 // 2
    carry = torch.zeros(fsz + 16, dtype=torch.uint8, device="cuda")
    out = torch.empty((6, fsz), dtype=torch.uint8, device="cuda")
    rgb = torch.empty((5, 48, 64 * 4), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    L = g.load_library()
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf)
        torch.cuda.synchronize()
        n0 = ctx.launch_count()

        def call(sel, first=(0, 3, 5), carries=None, d_out=None, F=5):
            ctx.decode_device_select(b.stream.data_ptr(), b.desc.data_ptr(), F, 64, 48, list(first), list(sel),
                                     d_out if d_out is not None else out.data_ptr(), carries, st)

        def call_rgb(sel, first=(0, 3, 5), last=None):
            ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), 5, 64, 48, list(first), list(sel), capi.CONV_RGB32,
                                         rgb.data_ptr(), 64 * 4, 48 * 64 * 4, 0, None, last, st)

        def raw(n, sel_ptr):
            first = (C.c_int * 3)(0, 3, 5)
            return L.rtjgpu_decode_device_select(ctx._h, C.c_void_p(b.stream.data_ptr()), C.c_void_p(b.desc.data_ptr()), 5, 64,
                                                 48, 2, first, None, n, sel_ptr, C.c_void_p(out.data_ptr()), C.c_void_p(st))

        bad = [lambda: call([5]),                                     # out of range
               lambda: call([-1, 2]),                                 # negative
               lambda: call([1, 1]),                                  # repeated
               lambda: call([3, 1]),                                  # out of order
               lambda: call([0, 1, 2, 3, 4, 4]),                      # n > F
               lambda: call([0], first=(0, 3, 3, 5)),                 # seq_first: an empty sequence
               lambda: call([0], first=(0, 3, 4)),                    # seq_first[S] != F
               lambda: call([0], carries=[carry.data_ptr(), carry.data_ptr() + 4]),     # misaligned carry
               lambda: call([0], d_out=out.data_ptr() + 8),           # misaligned output
               lambda: call_rgb([0], last=[carry.data_ptr(), carry.data_ptr() + 8]),    # misaligned last_yuv
               lambda: call_rgb([0, 5])]
        for i, fn in enumerate(bad):
            with pytest.raises(g.RTjpegError) as e:
                fn()
            assert e.value.code == capi.E_ARG, i
        assert raw(-1, None) == capi.E_ARG                            # n < 0
        assert raw(2, None) == capi.E_ARG                             # sel NULL with n > 0
        torch.cuda.synchronize()
        assert ctx.launch_count() == n0
        ctx.set_format(1)
        with pytest.raises(g.RTjpegError) as e:
            call_rgb([0, 3])
        assert e.value.code == capi.E_FORMAT
        assert ctx.launch_count() == n0
