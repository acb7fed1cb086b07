"""rtjgpu_decode_device_window / rtjgpu_decode_device_rgb_window: only a window of each selected frame, at an origin per
sequence, out of a device batch of many independent sequences.  Expected windows: every sequence decoded on its own by the
reference (or the restatement) from its own picture before the first frame, the selected frames cropped in numpy -- and for
packed pixels converted first by the oracle's converter, then cropped.  Output buffers are poisoned with 0xCD and carry one
guard slot behind the last one, which must stay poisoned."""
import ctypes as C

import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from streams import clip, reference_frames, reference_frames_fmt

pytestmark = pytest.mark.gpu

W, H = 160, 96
FSZ = W * H * 3 // 2
POISON = 0xCD

# inter clips of different seeds, qualities (255: raw prefix, every luma block HARD; 200: many blocks HARD) and GOPs;
# sequences of one frame and lengths that are not multiples of 32
SPECS = [
    (128, 45, dict(key_rate=14, lm=2, cm=2, dark=1, seed=1)),
    (32, 1, dict(key_rate=14, lm=4, cm=4, dark=1, seed=2)),
    (200, 33, dict(key_rate=9, lm=2, cm=2, seed=5)),
    (255, 20, dict(key_rate=6, lm=2, cm=2, seed=7)),
    (128, 70, dict(key_rate=29, lm=3, cm=3, dark=1, seed=9)),
]


def _carry(seed, fsz=FSZ):
    return np.random.default_rng(seed).integers(0, 256, fsz).astype(np.uint8)


@pytest.fixture(scope="module")
def case1():
    seqs = [clip(W, H, Q, F, **kw) for Q, F, kw in SPECS]
    carries = [_carry(11), None, _carry(13), _carry(14), None]      # distinct pictures and NULL
    want = np.concatenate([reference_frames(s, o, W, H, c) for (s, o), c in zip(seqs, carries)])
    return seqs, carries, want


def _dev(carries):
    return None if carries is None else [None if c is None else torch.from_numpy(c).cuda() for c in carries]


def _lengths(sf):
    return [int(sf[s + 1] - sf[s]) for s in range(len(sf) - 1)]


def _seq_of(sf, f):
    return int(np.searchsorted(np.asarray(sf), f, side="right") - 1)


def crop_planes(frame, fmt, w, h, x, y, cw, ch):
    """The window (x, y, cw, ch) of one frame's tight planes, as the tight planes of a cw x ch picture."""
    fr = np.asarray(frame).reshape(-1)
    Y = fr[:w * h].reshape(h, w)[y:y + ch, x:x + cw]
    if fmt == 2:
        return Y.reshape(-1).copy()
    vs = 2 if fmt == 0 else 1
    cwp, chp = w // 2, h // vs
    U = fr[w * h:w * h + cwp * chp].reshape(chp, cwp)[y // vs:(y + ch) // vs, x // 2:(x + cw) // 2]
    V = fr[w * h + cwp * chp:w * h + 2 * cwp * chp].reshape(chp, cwp)[y // vs:(y + ch) // vs, x // 2:(x + cw) // 2]
    return np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)])


def expect_planes(want, sf, sel, origins, size, fmt=0, w=W, h=H):
    cw, ch = size
    return np.stack([crop_planes(want[f], fmt, w, h, *origins[_seq_of(sf, f)], cw, ch) for f in sel]) if len(sel) else \
        np.zeros((0, O.frame_bytes(fmt, cw, ch)), np.uint8)


def expect_rgb(want, sf, sel, origins, size, kind, alpha, w=W, h=H):
    cw, ch = size
    bpp = capi.CONV_BPP[kind]
    out = []
    for f in sel:
        x, y = origins[_seq_of(sf, f)]
        pic = (O.ref_convert if O.have_ref() else O.convert)(kind, want[f], w, h, pitch=w * bpp, fill=alpha)
        out.append(np.asarray(pic).reshape(h, w * bpp)[y:y + ch, x * bpp:(x + cw) * bpp])
    return np.stack(out)


def _origins(S, xy):
    return [tuple(xy)] * S if np.ndim(xy) == 1 else [tuple(o) for o in xy]


def run_window(ctx, b, sf, sel, size, origins, cts, last=None):
    """One window call into a poisoned buffer of n + 1 slots; returns the n windows, checks the guard slot."""
    sel = np.asarray(sel, dtype=np.int64)
    wb = capi.frame_bytes(b.fmt, *size)
    out = torch.full((len(sel) + 1, wb), POISON, dtype=torch.uint8, device="cuda")
    D.decode_window(ctx, b, sf, sel, size, origins, cts, last=last, out=out)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert (got[len(sel)] == POISON).all(), "the call wrote behind its last slot"
    return got[:len(sel)]


def run_rgb_window(ctx, b, sf, sel, size, origins, kind, alpha, cts, last=None, pad=32):
    """The fused form into poisoned rows padded by `pad` bytes, one guard slot behind the last; returns [n, ch, cw * bpp]."""
    cw, ch = size
    bpp = capi.CONV_BPP[kind]
    pitch = cw * bpp + pad
    out = torch.full((len(sel) + 1, ch, pitch), POISON, dtype=torch.uint8, device="cuda")
    ctx.decode_device_rgb_window(b.stream.data_ptr(), b.desc.data_ptr(), b.F, b.w, b.h, list(sf), [int(v) for v in sel],
                                 size, _origins(len(sf) - 1, origins), kind, out.data_ptr(), pitch, ch * pitch, alpha,
                                 None if cts is None else [None if c is None else c.data_ptr() for c in cts],
                                 None if last is None else [None if t is None else t.data_ptr() for t in last],
                                 torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert (got[len(sel)] == POISON).all(), "the call wrote behind its last slot"
    assert (got[:len(sel), :, cw * bpp:] == POISON).all(), "the call wrote behind a window row"
    return got[:len(sel), :, :cw * bpp]


# (size, origins): one origin for all sequences, or one per sequence (five sequences)
WINDOWS = {
    "top_left": ((48, 32), (0, 0)),
    "bottom_right": ((64, 30), (W - 64, H - 30)),
    "top_right": ((32, 16), (W - 32, 0)),
    "bottom_left": ((80, 40), (0, H - 40)),
    "full": ((W, H), (0, 0)),
    "one_unit": ((16, 16), (64, 32)),
    "two_rows": ((W, 2), (0, 50)),
    "mid_unit": ((96, 20), (32, 6)),
    "per_sequence": ((48, 24), [(0, 0), (112, 72), (16, 6), (96, 38), (64, 70)]),
}


@pytest.mark.parametrize("name", list(WINDOWS))
def test_planes_window_matches_reference(case1, name):
    seqs, carries, want = case1
    size, org = WINDOWS[name]
    b, sf = D.upload_sequences(seqs, W, H)
    origins = _origins(len(seqs), org)
    sel = g.select_frames(sf, [np.arange(n % 3, n, 3) for n in _lengths(sf)])
    with g.BatchContext(0) as ctx:
        got = run_window(ctx, b, sf, sel, size, origins, _dev(carries))
        assert ctx.batch_info().bad_frames == 0
    exp = expect_planes(want, sf, sel, origins, size)
    for k in range(len(sel)):
        assert np.array_equal(got[k], exp[k]), (name, k, int(sel[k]))


def test_full_window_is_the_select_call(case1):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    cts = _dev(carries)
    sel = g.select_frames(sf, [np.arange(0, n, 2) for n in _lengths(sf)])
    with g.BatchContext(0) as ctx:
        ref = D.decode_select(ctx, b, sf, sel, cts)
        torch.cuda.synchronize()
        got = run_window(ctx, b, sf, sel, (W, H), (0, 0), cts)
        all_frames = run_window(ctx, b, sf, np.arange(b.F), (W, H), (0, 0), cts)
    assert np.array_equal(got, ref.cpu().numpy())
    assert np.array_equal(all_frames, want)


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
    lasts = [torch.full((fsz,), POISON, dtype=torch.uint8, device="cuda"), None,
             torch.full((fsz,), POISON, dtype=torch.uint8, device="cuda")]
    with g.BatchContext(0) as ctx:
        for size, org in (((48, 26), [(16, 6), (0, 0), (112, 70)]), ((W, H), [(0, 0)] * 3), ((16, 2), [(144, 94)] * 3)):
            got = run_window(ctx, b, sf, sel, size, org, _dev(carries), last=lasts)
            exp = expect_planes(want, sf, sel, org, size, fmt)
            assert np.array_equal(got, exp), (fmt, size)
            for s in (0, 2):
                assert np.array_equal(lasts[s].cpu().numpy(), want[int(sf[s + 1]) - 1]), (fmt, s)
        ctx.set_format(0)


@pytest.mark.parametrize("kind", [capi.CONV_RGB32, capi.CONV_BGR32, capi.CONV_RGB24, capi.CONV_BGR24, capi.CONV_RGB16])
def test_fused_rgb(case1, kind):
    """Padded pitches, distinct origins (one mid-unit), last_yuv for every sequence but one; the last frames of sequences 0
    and 3 selected, those of 2 and 4 not."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    n = _lengths(sf)
    sel = g.select_frames(sf, [[0, 10, n[0] - 1], [0], [2, 20], [n[3] - 1], [5, 33, 34]])
    size, org = (64, 36), [(0, 0), (96, 60), (16, 6), (80, 34), (32, 12)]
    lasts = [None if s == 1 else torch.full((FSZ,), 0xEE, dtype=torch.uint8, device="cuda") for s in range(len(seqs))]
    with g.BatchContext(0) as ctx:
        got = run_rgb_window(ctx, b, sf, sel, size, org, kind, 0x5A, _dev(carries), last=lasts)
        assert ctx.batch_info().bad_frames == 0
    assert np.array_equal(got, expect_rgb(want, sf, sel, org, size, kind, 0x5A))
    for s, t in enumerate(lasts):
        if t is not None:
            assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s


def test_fused_rgb_full_window_is_the_select_call(case1):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    cts = _dev(carries)
    sel = g.select_frames(sf, [np.arange(0, n, 4) for n in _lengths(sf)])
    kind = capi.CONV_RGB24
    with g.BatchContext(0) as ctx:
        ref = torch.full((len(sel), H, W * 3), POISON, dtype=torch.uint8, device="cuda")
        ctx.decode_device_rgb_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), list(sel), kind, ref.data_ptr(),
                                     W * 3, H * W * 3, 0, [None if c is None else c.data_ptr() for c in cts], None,
                                     torch.cuda.current_stream().cuda_stream)
        got = D.decode_rgb_window(ctx, b, sf, sel, (W, H), (0, 0), kind, carries=cts)
        torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy().reshape(len(sel), H, W * 3), ref.cpu().numpy())


def test_wide_picture_strips():
    """2080 px: a window of 2064 px is cut into two strips; a window of 96 px crosses the boundary between the strips of
    the whole picture (x = 1040).  Planes and fused RGB."""
    w, h = 2080, 32
    fsz = w * h * 3 // 2
    seqs = [clip(w, h, 128, 12, key_rate=5, lm=2, cm=2, seed=1), clip(w, h, 200, 9, key_rate=3, lm=2, cm=2, seed=2)]
    carries = [_carry(51, fsz), _carry(52, fsz)]
    want = np.concatenate([reference_frames(s, o, w, h, c) for (s, o), c in zip(seqs, carries)])
    b, sf = D.upload_sequences(seqs, w, h)
    sel = g.select_frames(sf, [[1, 4, 11], [0, 7]])
    lasts = [torch.full((fsz,), POISON, dtype=torch.uint8, device="cuda") for _ in seqs]
    with g.BatchContext(0) as ctx:
        for size, org in (((2064, 30), [(16, 2), (0, 0)]), ((96, 16), [(1008, 8), (992, 16)])):
            got = run_window(ctx, b, sf, sel, size, org, _dev(carries), last=lasts)
            assert np.array_equal(got, expect_planes(want, sf, sel, org, size, 0, w, h)), size
            for s, t in enumerate(lasts):
                assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s
            rgb = run_rgb_window(ctx, b, sf, sel, size, org, capi.CONV_RGB32, 0x11, _dev(carries))
            assert np.array_equal(rgb, expect_rgb(want, sf, sel, org, size, capi.CONV_RGB32, 0x11, w, h)), size


def test_last_yuv_null_entries_and_unselected_last_frames(case1):
    """last_yuv for sequences 0, 2 and 3 (1 and 4 NULL); the last frame of 0 selected, those of 2 and 3 not; a 16-byte
    guard behind every last picture."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    n = _lengths(sf)
    sel = g.select_frames(sf, [[3, n[0] - 1], [0], [1], [0, 5], [9]])
    lasts = [torch.full((FSZ + 16,), POISON, dtype=torch.uint8, device="cuda") if s in (0, 2, 3) else None
             for s in range(len(seqs))]
    org = [(32, 16)] * len(seqs)
    with g.BatchContext(0) as ctx:
        got = run_window(ctx, b, sf, sel, (32, 32), org, _dev(carries), last=lasts)
    assert np.array_equal(got, expect_planes(want, sf, sel, org, (32, 32)))
    for s, t in enumerate(lasts):
        if t is not None:
            v = t.cpu().numpy()
            assert np.array_equal(v[:FSZ], want[int(sf[s + 1]) - 1]), s
            assert (v[FSZ:] == POISON).all(), s


def test_streaming_three_calls():
    """Each call takes a window of every third frame of each sequence; the next call's carries are the previous call's
    last_yuv.  Plan states carry over."""
    specs = [sp for sp in SPECS if sp[1] > 3]
    clips = [clip(W, H, Q, F, **kw) for Q, F, kw in specs]
    inits = [_carry(21), None, _carry(23), _carry(24)]
    want = [reference_frames(s, o, W, H, c) for (s, o), c in zip(clips, inits)]
    cuts = [[0, F // 3, 2 * F // 3, F] for _, F, _ in specs]
    states = [capi.State(0, 0, capi.TABLE_ZERO, 0) for _ in clips]
    org = [(0, 0), (16, 8), (128, 64), (48, 30)]
    size = (32, 32)
    cts = _dev(inits)
    with g.BatchContext(0) as ctx:
        for call in range(3):
            batch = [(s, o[c[call]:c[call + 1] + 1]) for (s, o), c in zip(clips, cuts)]
            b, sf = D.upload_sequences(batch, W, H, states=states)
            picks = [np.arange(call, n, 3) for n in _lengths(sf)]
            sel = g.select_frames(sf, picks)
            lasts = [torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda") for _ in clips]
            got = run_window(ctx, b, sf, sel, size, org, cts, last=lasts)
            k = 0
            for s in range(len(clips)):
                for i in picks[s]:
                    f = cuts[s][call] + int(i)
                    assert np.array_equal(got[k], crop_planes(want[s][f], 0, W, H, *org[s], *size)), (call, s, f)
                    k += 1
                assert np.array_equal(lasts[s].cpu().numpy(), want[s][cuts[s][call + 1] - 1]), (call, s)
            cts = lasts


def test_nothing_selected_null_output(case1):
    """n = 0, d_out NULL: only the last frames leave, as planes; batch info and skip counts describe all F frames."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    cts = _dev(carries)
    lasts = [torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda") for _ in seqs]
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf, cts)
        torch.cuda.synchronize()
        bi = ctx.batch_info()
        full = (bi.skipped_blocks, bi.payload_bytes, bi.bad_frames, bi.first_bad_frame)
        counts = ctx.skip_counts(b.F)
        out = D.decode_window(ctx, b, sf, [], (32, 32), (0, 0), cts, last=lasts)
        torch.cuda.synchronize()
        assert out.shape[0] == 0
        bi = ctx.batch_info()
        assert (bi.skipped_blocks, bi.payload_bytes, bi.bad_frames, bi.first_bad_frame) == full
        assert np.array_equal(ctx.skip_counts(b.F), counts)
        for t in lasts:
            t.fill_(POISON)
        ctx.decode_device_rgb_window(b.stream.data_ptr(), b.desc.data_ptr(), b.F, W, H, list(sf), [], (32, 32),
                                     [(0, 0)] * len(seqs), capi.CONV_RGB32, None, 128, 128 * 32, 0,
                                     [None if c is None else c.data_ptr() for c in cts], [t.data_ptr() for t in lasts],
                                     torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    for s, t in enumerate(lasts):
        assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s


@pytest.mark.parametrize("mode", [capi.SCAN_AUTO, capi.SCAN_CHUNK])
def test_sliced_pipeline_with_empty_slices(case1, mode):
    """Slices of 32 frames; [32, 64) and [64, 96) hold no selected frame (their K2 launch is left out)."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    sel = np.array([3, 10, 31, 99, 100, 101, 140, 168])
    org = [(16, 6), (0, 0), (144, 70), (64, 40), (32, 70)]
    lasts = [torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda") for _ in seqs]
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(mode)
        ctx.set_pipeline(capi.PIPELINE_SLICED, 32)
        got = run_window(ctx, b, sf, sel, (16, 26), org, _dev(carries), last=lasts)
    assert np.array_equal(got, expect_planes(want, sf, sel, org, (16, 26)))
    for s, t in enumerate(lasts):
        assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s


def test_one_sequence():
    """S = 1: the origin goes up in the same table as for many sequences."""
    s, o = clip(W, H, 128, 50, key_rate=14, lm=2, cm=2, dark=1, seed=3)
    init = _carry(71)
    want = reference_frames(s, o, W, H, init)
    b, sf = D.upload_sequences([(s, o)], W, H)
    sel = np.array([0, 7, 31, 32, 48])
    last = torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda")
    with g.BatchContext(0) as ctx:
        got = run_window(ctx, b, sf, sel, (64, 48), (48, 24), [torch.from_numpy(init).cuda()], last=[last])
    assert np.array_equal(got, expect_planes(want, sf, sel, [(48, 24)], (64, 48)))
    assert np.array_equal(last.cpu().numpy(), want[49])


def test_many_sequences_at_720x576():
    """64 sequences of 8 frames at 720x576, a 224x224 window per sequence at its own origin, every fourth frame; the fused
    RGB24 form of the same."""
    w, h, k = 720, 576, 8
    fsz = w * h * 3 // 2
    clips = [clip(w, h, 128, 40, key_rate=29, lm=2, cm=2, seed=seed) for seed in (1, 2)]
    seqs = []
    for s in range(64):
        cs, co = clips[s % 2]
        a = (s * 7) % (40 - k + 1)
        seqs.append((cs, co[a:a + k + 1]))
    init = _carry(61, fsz)
    rng = np.random.default_rng(5)
    org = [(int(rng.integers(0, (w - 224) // 16 + 1)) * 16, int(rng.integers(0, (h - 224) // 2 + 1)) * 2) for _ in range(64)]
    b, sf = D.upload_sequences(seqs, w, h)
    sel = g.select_frames(sf, [np.arange(s % 4, k, 4) for s in range(64)])
    cts = [torch.from_numpy(init).cuda()] * 64
    with g.BatchContext(0) as ctx:
        got = run_window(ctx, b, sf, sel, (224, 224), org, cts)
        rgb = D.decode_rgb_window(ctx, b, sf, sel, (224, 224), org, capi.CONV_RGB24, carries=cts).cpu().numpy()
    k_at = 0
    for s, (cs, co) in enumerate(seqs):
        want = reference_frames(cs, co, w, h, init)
        for i in range(s % 4, k, 4):
            assert np.array_equal(got[k_at], crop_planes(want[i], 0, w, h, *org[s], 224, 224)), (s, i)
            pic = (O.ref_convert if O.have_ref() else O.convert)(capi.CONV_RGB24, want[i], w, h, pitch=w * 3, fill=255)
            exp = np.asarray(pic).reshape(h, w * 3)[org[s][1]:org[s][1] + 224, org[s][0] * 3:(org[s][0] + 224) * 3]
            assert np.array_equal(rgb[k_at].reshape(224, 224 * 3), exp), (s, i)
            k_at += 1
    assert k_at == len(sel)


def test_invalid_arguments():
    a, b2 = clip(64, 48, 128, 3, key_rate=2, lm=2, cm=2), clip(64, 48, 128, 2, key_rate=2, lm=2, cm=2, seed=2)
    b, sf = D.upload_sequences([a, b2], 64, 48)
    fsz = 64 * 48 * 3 // 2
    last = torch.zeros(fsz + 16, dtype=torch.uint8, device="cuda")
    out = torch.empty((6, fsz), dtype=torch.uint8, device="cuda")
    rgb = torch.empty((5, 48, 64 * 4), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    L = g.load_library()
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf)
        torch.cuda.synchronize()
        n0 = ctx.launch_count()

        def call(sel=(0, 3), size=(32, 32), org=((0, 0), (16, 16)), lasts=None, first=(0, 3, 5)):
            ctx.decode_device_window(b.stream.data_ptr(), b.desc.data_ptr(), 5, 64, 48, list(first), list(sel), size, org,
                                     out.data_ptr(), None, lasts, st)

        def call_rgb(size=(32, 32), org=((0, 0), (16, 16)), row_pitch=64 * 4, frame_pitch=48 * 64 * 4):
            ctx.decode_device_rgb_window(b.stream.data_ptr(), b.desc.data_ptr(), 5, 64, 48, [0, 3, 5], [0, 3], size, org,
                                         capi.CONV_RGB32, rgb.data_ptr(), row_pitch, frame_pitch, 0, None, None, st)

        def raw_null_origins():
            first, sel = (C.c_int * 3)(0, 3, 5), (C.c_int * 1)(0)
            return L.rtjgpu_decode_device_window(ctx._h, C.c_void_p(b.stream.data_ptr()), C.c_void_p(b.desc.data_ptr()), 5,
                                                 64, 48, 2, first, None, 1, sel, 32, 32, None, C.c_void_p(out.data_ptr()),
                                                 None, C.c_void_p(st))

        bad = [lambda: call(size=(0, 32)),                            # cw <= 0
               lambda: call(size=(32, 0)),                            # ch <= 0
               lambda: call(size=(-16, 32)),
               lambda: call(size=(24, 32)),                           # cw not a multiple of 16
               lambda: call(size=(32, 31)),                           # ch odd
               lambda: call(org=((8, 0), (0, 0))),                    # x not a multiple of 16
               lambda: call(org=((0, 0), (0, 3))),                    # y odd
               lambda: call(org=((-16, 0), (0, 0))),                  # outside the picture
               lambda: call(org=((0, 0), (48, 0))),                   # ... on the right
               lambda: call(org=((0, 18), (0, 0))),                   # ... at the bottom
               lambda: call(size=(80, 16)),                           # wider than the picture
               lambda: call(lasts=[last.data_ptr(), last.data_ptr() + 8]),     # misaligned last_yuv
               lambda: call(sel=(3, 1)),                              # the selection's rules
               lambda: call(first=(0, 3, 4)),                         # ... and the batch's
               lambda: call_rgb(row_pitch=32 * 4 - 16),               # row_pitch < cw * bpp
               lambda: call_rgb(row_pitch=32 * 4 + 8),                # pitch not a multiple of 16
               lambda: call_rgb(frame_pitch=32 * 32 * 4 + 8),
               lambda: call_rgb(org=((0, 0), (40, 0)))]
        for i, fn in enumerate(bad):
            with pytest.raises(g.RTjpegError) as e:
                fn()
            assert e.value.code == capi.E_ARG, i
        assert raw_null_origins() == capi.E_ARG                       # origins NULL
        torch.cuda.synchronize()
        assert ctx.launch_count() == n0
        call_rgb(row_pitch=32 * 4, frame_pitch=32 * 32 * 4)          # a tight window is fine
        torch.cuda.synchronize()
        n1 = ctx.launch_count()
        ctx.set_format(1)
        with pytest.raises(g.RTjpegError) as e:
            call_rgb()
        assert e.value.code == capi.E_FORMAT
        assert ctx.launch_count() == n1
