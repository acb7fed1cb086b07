"""rtjgpu_decode_device_chw_window: a window of each selected frame straight to a model's input -- planar channels of the
RGB24 / BGR24 converter, as uint8, float16, bfloat16 or float32, scaled and offset per channel, mirrored per sequence.
Expected values: the per-sequence reference decodes of test_gpu_window, converted by the oracle's converter, cropped, split
into channels and mirrored in numpy, then v * scale + bias in numpy float32 (two roundings) and rounded to the element type
on the CPU.  Results are compared as bit patterns.  Output buffers are poisoned with 0xCD and carry one guard slot behind
the last one, which must stay poisoned."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from streams import clip, reference_frames
from test_gpu_window import FSZ, H, POISON, SPECS, W, _carry, _dev, _lengths, _origins, _seq_of, case1, crop_planes  # noqa: F401

pytestmark = pytest.mark.gpu

DTYPES = [torch.uint8, torch.float16, torch.bfloat16, torch.float32]
BITS = {torch.uint8: (torch.uint8, np.uint8), torch.float16: (torch.int16, np.uint16),
        torch.bfloat16: (torch.int16, np.uint16), torch.float32: (torch.int32, np.uint32)}
KINDS = {"rgb": capi.CONV_RGB24, "bgr": capi.CONV_BGR24}
IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))

_pics = {}


def rgb_pictures(want, kind, w=W, h=H):
    """Every frame of `want` through the oracle's converter: [F, h, w, 3] (cached per array and converter)."""
    key = (id(want), kind)
    if key not in _pics:
        conv = O.ref_convert if O.have_ref() else O.convert
        _pics[key] = (want, np.stack([np.asarray(conv(kind, f, w, h, pitch=w * 3)).reshape(h, w, 3) for f in want]))
    return _pics[key][1]


def expect_u8(pics, sf, sel, origins, size, mirror):
    """[n, 3, ch, cw] uint8: the window of each selected frame, channel c = byte c of the converter's pixel."""
    cw, ch = size
    out = np.zeros((len(sel), 3, ch, cw), np.uint8)
    for k, f in enumerate(sel):
        s = _seq_of(sf, f)
        x, y = origins[s]
        v = pics[f][y:y + ch, x:x + cw].transpose(2, 0, 1)
        out[k] = v[..., ::-1] if mirror is not None and mirror[s] else v
    return out


def expect_bits(v, dtype, scale=None, bias=None):
    """The stored bit patterns of byte values v [n, 3, ch, cw] as dtype: float32 v * scale + bias (two roundings)."""
    if dtype == torch.uint8:
        return v
    s = np.ones(3, np.float32) if scale is None else np.asarray(scale, np.float32)
    b = np.zeros(3, np.float32) if bias is None else np.asarray(bias, np.float32)
    t = v.astype(np.float32) * s[None, :, None, None]
    t = t + b[None, :, None, None]
    assert t.dtype == np.float32
    if dtype == torch.float32:
        return t.view(np.uint32)
    if dtype == torch.float16:
        return t.astype(np.float16).view(np.uint16)
    return torch.from_numpy(t).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def bits(t):
    tv, nv = BITS[t.dtype]
    return t.view(tv).cpu().numpy().view(nv)


def run_chw(ctx, b, sf, sel, size, origins, dtype, order="rgb", mirror=None, scale=None, bias=None, cts=None, last=None,
            mean=None, std=None):
    """One call into a poisoned [n + 1, 3, ch, cw] buffer; returns the bit patterns of the n windows, checks the guard."""
    cw, ch = size
    n = len(sel)
    buf = torch.full((n + 1, 3 * ch * cw * capi.CHW_ESIZE[D.CHW_DTYPES[dtype]]), POISON, dtype=torch.uint8, device="cuda")
    out = buf.view(dtype).view(n + 1, 3, ch, cw)[:n]
    D.decode_chw_window(ctx, b, sf, sel, size, origins, dtype=dtype, mean=mean, std=std, scale=scale, bias=bias, order=order,
                        mirror=mirror, carries=cts, last=last, out=out)
    torch.cuda.synchronize()
    assert (buf[n] == POISON).all().item(), "the call wrote behind its last slot"
    return bits(out)


MIRRORS = {"none": lambda S: None, "all": lambda S: [1] * S, "alternate": lambda S: [s % 2 for s in range(S)]}
# corners, a full-picture window, and an origin per sequence
WINDOWS = [((48, 32), (0, 0)), ((64, 30), (W - 64, H - 30)), ((W, H), (0, 0)),
           ((48, 24), [(0, 0), (112, 72), (16, 6), (96, 38), (64, 70)])]


@pytest.mark.parametrize("mirror", list(MIRRORS))
@pytest.mark.parametrize("order", list(KINDS))
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_dtype_order_mirror(case1, dtype, order, mirror):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    S = len(seqs)
    mir = MIRRORS[mirror](S)
    pics = rgb_pictures(want, KINDS[order])
    sel = g.select_frames(sf, [np.arange(n % 3, n, 3) for n in _lengths(sf)])
    scale, bias = (None, None) if dtype == torch.uint8 else ((0.5, -1.25, 3.0), (-7.0, 0.125, 100.0))
    with g.BatchContext(0) as ctx:
        for size, org in WINDOWS:
            origins = _origins(S, org)
            got = run_chw(ctx, b, sf, sel, size, origins, dtype, order, mir, scale, bias, _dev(carries))
            exp = expect_bits(expect_u8(pics, sf, sel, origins, size, mir), dtype, scale, bias)
            assert np.array_equal(got, exp), (size, org)
        assert ctx.batch_info().bad_frames == 0


# hand-picked per-channel coefficients: f16 overflow to +-inf, f16 subnormals, a negative scale, ties of bf16 and of f16
COEFFS = {
    "imagenet": capi.normalize_coefficients(*IMAGENET),
    "null": (None, None),
    "f16_inf": ((300.0, -300.0, 1.0), (0.0, 0.0, 65000.0)),
    "subnormal": ((1e-7, -3e-8, 2.0 ** -24), (0.0, 0.0, 0.0)),
    "negative": ((-1.0, -0.0078125, -2.5), (255.0, 1.0, -0.5)),
    "ties": ((1.0, 1.0, 1.0), (0.5, 256.0, 1024.5)),
}


@pytest.mark.parametrize("coeffs", list(COEFFS))
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32], ids=str)
def test_normalisation(case1, dtype, coeffs):
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    S = len(seqs)
    scale, bias = COEFFS[coeffs]
    pics = rgb_pictures(want, capi.CONV_RGB24)
    sel = g.select_frames(sf, [np.arange(0, n, 2) for n in _lengths(sf)])
    size, org = (64, 48), [(16, 2), (0, 0), (96, 48), (32, 20), (80, 10)]
    mir = [1, 0, 0, 1, 1]
    with g.BatchContext(0) as ctx:
        got = run_chw(ctx, b, sf, sel, size, org, dtype, "rgb", mir, scale, bias, _dev(carries))
        if coeffs == "imagenet":             # mean / std through the wrapper are the same coefficients
            again = run_chw(ctx, b, sf, sel, size, org, dtype, "rgb", mir, cts=_dev(carries), mean=IMAGENET[0],
                            std=IMAGENET[1])
            assert np.array_equal(again, got)
    exp = expect_bits(expect_u8(pics, sf, sel, org, size, mir), dtype, scale, bias)
    assert np.array_equal(got, exp)
    if coeffs == "f16_inf" and dtype == torch.float16:
        assert (got == 0x7C00).any() and (got == 0xFC00).any()
    if coeffs == "subnormal" and dtype == torch.float16:
        assert ((got & 0x7C00) == 0).any() and ((got & 0x3FF) != 0).any()


def test_u8_is_the_rgb_window_permuted(case1):
    """The same batch through rtjgpu_decode_device_rgb_window (RGB24), permuted to CHW on the device."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    sel = g.select_frames(sf, [np.arange(1, n, 2) if n > 1 else [0] for n in _lengths(sf)])
    org = [(16, 2), (0, 0), (96, 48), (32, 20), (80, 10)]
    with g.BatchContext(0) as ctx:
        for order, kind in KINDS.items():
            rgb = D.decode_rgb_window(ctx, b, sf, sel, (64, 48), org, kind, carries=_dev(carries))
            chw = D.decode_chw_window(ctx, b, sf, sel, (64, 48), org, dtype=torch.uint8, order=order, carries=_dev(carries))
            torch.cuda.synchronize()
            assert torch.equal(chw, rgb.permute(0, 3, 1, 2).contiguous()), order


def test_wide_picture_mirrored_across_strips():
    """2304 px: a window of 2288 px is cut into two strips; mirrored, each strip's chunks land in the other half of the
    window.  A 96 px window across the picture's middle too."""
    w, h = 2304, 64
    fsz = w * h * 3 // 2
    seqs = [clip(w, h, 128, 10, key_rate=4, lm=2, cm=2, seed=1), clip(w, h, 200, 7, key_rate=3, lm=2, cm=2, seed=2)]
    carries = [_carry(51, fsz), _carry(52, fsz)]
    want = np.concatenate([reference_frames(s, o, w, h, c) for (s, o), c in zip(seqs, carries)])
    pics = rgb_pictures(want, capi.CONV_RGB24, w, h)
    b, sf = D.upload_sequences(seqs, w, h)
    sel = g.select_frames(sf, [[1, 4, 9], [0, 6]])
    with g.BatchContext(0) as ctx:
        for size, org in (((2288, 30), [(16, 2), (0, 34)]), ((96, 16), [(1104, 8), (1136, 48)]), ((w, h), [(0, 0)] * 2)):
            for dtype in (torch.uint8, torch.float16, torch.float32):
                got = run_chw(ctx, b, sf, sel, size, org, dtype, "rgb", [1, 1], cts=_dev(carries))
                exp = expect_bits(expect_u8(pics, sf, sel, org, size, [1, 1]), dtype)
                assert np.array_equal(got, exp), (size, dtype)


def test_last_yuv_and_streaming_two_calls():
    """last_yuv byte for byte what decode_window writes for the same call, and the next call's carries."""
    specs = [sp for sp in SPECS if sp[1] > 3]
    clips = [clip(W, H, Q, F, **kw) for Q, F, kw in specs]
    inits = [_carry(21), None, _carry(23), _carry(24)]
    want = [reference_frames(s, o, W, H, c) for (s, o), c in zip(clips, inits)]
    cuts = [[0, F // 2, F] for _, F, _ in specs]
    states = [capi.State(0, 0, capi.TABLE_ZERO, 0) for _ in clips]
    org, size, mir = [(0, 0), (16, 8), (128, 64), (48, 30)], (32, 32), [0, 1, 1, 0]
    cts = _dev(inits)
    with g.BatchContext(0) as ctx:
        for call in range(2):
            batch = [(s, o[c[call]:c[call + 1] + 1]) for (s, o), c in zip(clips, cuts)]
            b, sf = D.upload_sequences(batch, W, H, states=states)
            picks = [np.arange(call, n, 2) for n in _lengths(sf)]
            sel = g.select_frames(sf, picks)
            lasts = [torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda") for _ in clips]
            ref = [torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda") for _ in clips]
            D.decode_window(ctx, b, sf, sel, size, org, cts, last=ref)
            got = run_chw(ctx, b, sf, sel, size, org, torch.bfloat16, "bgr", mir, *capi.normalize_coefficients(*IMAGENET),
                          cts=cts, last=lasts)
            k = 0
            for s in range(len(clips)):
                assert torch.equal(lasts[s], ref[s]), (call, s)
                assert np.array_equal(lasts[s].cpu().numpy(), want[s][cuts[s][call + 1] - 1]), (call, s)
                for i in picks[s]:
                    f = cuts[s][call] + int(i)
                    pic = (O.ref_convert if O.have_ref() else O.convert)(capi.CONV_BGR24, want[s][f], W, H, pitch=W * 3)
                    v = np.asarray(pic).reshape(H, W, 3)[org[s][1]:org[s][1] + 32, org[s][0]:org[s][0] + 32].transpose(2, 0, 1)
                    v = v[..., ::-1] if mir[s] else v
                    exp = expect_bits(v[None], torch.bfloat16, *capi.normalize_coefficients(*IMAGENET))[0]
                    assert np.array_equal(got[k], exp), (call, s, f)
                    k += 1
            cts = lasts


def test_subsets_and_nothing_selected(case1):
    """1 in 8, the last frame only, and n = 0 with a NULL output: only the last frames leave, as planes."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    S = len(seqs)
    pics = rgb_pictures(want, capi.CONV_RGB24)
    n = _lengths(sf)
    org = [(16, 2), (0, 0), (96, 48), (32, 20), (80, 10)]
    mir = [0, 1, 0, 1, 0]
    with g.BatchContext(0) as ctx:
        for picks in ([np.arange(s, m, 8) if m > s else [0] for s, m in enumerate(n)], [[m - 1] for m in n]):
            sel = g.select_frames(sf, picks)
            got = run_chw(ctx, b, sf, sel, (64, 48), org, torch.float16, "rgb", mir, cts=_dev(carries))
            assert np.array_equal(got, expect_bits(expect_u8(pics, sf, sel, org, (64, 48), mir), torch.float16))
        lasts = [torch.full((FSZ,), POISON, dtype=torch.uint8, device="cuda") for _ in seqs]
        out = D.decode_chw_window(ctx, b, sf, [], (32, 32), (0, 0), dtype=torch.float16, mirror=True, carries=_dev(carries),
                                  last=lasts)
        torch.cuda.synchronize()
        assert tuple(out.shape) == (0, 3, 32, 32)
        for t in lasts:
            t.fill_(POISON)
        L = g.load_library()
        first = (C.c_int * (S + 1))(*[int(v) for v in sf])
        org_c = (C.c_int * (2 * S))(*([0] * 2 * S))
        cts = _dev(carries)
        rc = L.rtjgpu_decode_device_chw_window(ctx._h, C.c_void_p(b.stream.data_ptr()), C.c_void_p(b.desc.data_ptr()), b.F,
                                               W, H, S, first, capi._ptr_array([None if c is None else c.data_ptr() for c in cts]),
                                               0, None, 32, 32, org_c, None, capi.CONV_RGB24, capi.CHW_F32, None, None, None,
                                               capi._ptr_array([t.data_ptr() for t in lasts]),
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == capi.OK
        torch.cuda.synchronize()
    for s, t in enumerate(lasts):
        assert np.array_equal(t.cpu().numpy(), want[int(sf[s + 1]) - 1]), s


@pytest.mark.parametrize("mode", [capi.SCAN_AUTO, capi.SCAN_CHUNK, capi.SCAN_SYNC])
def test_sliced_pipeline_and_scan_modes(case1, mode):
    """The sliced pipeline (slices of 32 frames, some without a selected frame) and several scan modes: the same bytes as
    the serial call."""
    seqs, carries, want = case1
    b, sf = D.upload_sequences(seqs, W, H)
    sel = np.array([3, 10, 31, 99, 100, 101, 140, 168])
    org = [(16, 6), (0, 0), (144, 70), (64, 40), (32, 70)]
    mir = [1, 0, 1, 0, 1]
    coeffs = capi.normalize_coefficients(*IMAGENET)
    with g.BatchContext(0) as ctx:
        ctx.set_pipeline(capi.PIPELINE_SERIAL, 0)
        serial = run_chw(ctx, b, sf, sel, (16, 26), org, torch.float16, "rgb", mir, *coeffs, cts=_dev(carries))
        ctx.set_scan_mode(mode)
        ctx.set_pipeline(capi.PIPELINE_SLICED, 32)
        got = run_chw(ctx, b, sf, sel, (16, 26), org, torch.float16, "rgb", mir, *coeffs, cts=_dev(carries))
    assert np.array_equal(got, serial)
    exp = expect_bits(expect_u8(rgb_pictures(want, capi.CONV_RGB24), sf, sel, org, (16, 26), mir), torch.float16, *coeffs)
    assert np.array_equal(got, exp)


def test_invalid_arguments():
    a, b2 = clip(64, 48, 128, 3, key_rate=2, lm=2, cm=2), clip(64, 48, 128, 2, key_rate=2, lm=2, cm=2, seed=2)
    b, sf = D.upload_sequences([a, b2], 64, 48)
    fsz = 64 * 48 * 3 // 2
    last = torch.zeros(fsz + 16, dtype=torch.uint8, device="cuda")
    out = torch.full((3 * 3 * 48 * 64 * 4 + 64,), POISON, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    L = g.load_library()
    with g.BatchContext(0) as ctx:
        D.decode_sequences(ctx, b, sf)
        torch.cuda.synchronize()
        n0 = ctx.launch_count()

        def call(sel=(0, 3), size=(32, 32), org=((0, 0), (16, 16)), kind=capi.CONV_RGB24, dtype=capi.CHW_F16, scale=None,
                 bias=None, at=0, lasts=None, first=(0, 3, 5), mirror=(1, 0)):
            ctx.decode_device_chw_window(b.stream.data_ptr(), b.desc.data_ptr(), 5, 64, 48, list(first), list(sel), size, org,
                                         kind, dtype, out.data_ptr() + at, mirror, scale, bias, None, lasts, st)

        def raw(scale, bias, dtype=capi.CHW_F32):
            first, sel, org = (C.c_int * 3)(0, 3, 5), (C.c_int * 1)(0), (C.c_int * 4)(0, 0, 0, 0)
            f3 = lambda v: None if v is None else (C.c_float * 3)(*v)        # noqa: E731 (NaN and inf as they are)
            return L.rtjgpu_decode_device_chw_window(ctx._h, C.c_void_p(b.stream.data_ptr()), C.c_void_p(b.desc.data_ptr()),
                                                     5, 64, 48, 2, first, None, 1, sel, 32, 32, org, None, capi.CONV_RGB24,
                                                     dtype, f3(scale), f3(bias), C.c_void_p(out.data_ptr()), None,
                                                     C.c_void_p(st))

        bad = [lambda: call(dtype=4), lambda: call(dtype=-1),                                  # dtype
               lambda: call(kind=capi.CONV_RGB32), lambda: call(kind=capi.CONV_RGB16),          # kind
               lambda: call(kind=capi.CONV_RGB8), lambda: call(kind=7),
               lambda: call(dtype=capi.CHW_U8, scale=(1, 1, 1)),                               # u8 is not scaled
               lambda: call(dtype=capi.CHW_U8, bias=(0, 0, 0)),
               lambda: call(at=8), lambda: call(at=4),                                          # d_out misaligned
               lambda: call(size=(24, 32)), lambda: call(size=(32, 31)),                        # the window's rules
               lambda: call(org=((8, 0), (0, 0))), lambda: call(org=((0, 0), (48, 0))),
               lambda: call(org=((0, 18), (0, 0))), lambda: call(size=(0, 32)),
               lambda: call(lasts=[last.data_ptr(), last.data_ptr() + 8]),
               lambda: call(sel=(3, 1)), lambda: call(sel=(0, 5)),                              # the selection's
               lambda: call(first=(0, 3, 4))]                                                   # ... and the batch's
        for i, fn in enumerate(bad):
            with pytest.raises(g.RTjpegError) as e:
                fn()
            assert e.value.code == capi.E_ARG, i
        for s, bb in (((math.nan, 1, 1), None), ((1, math.inf, 1), None), (None, (0, 0, -math.inf)), (None, (math.nan, 0, 0))):
            assert raw(s, bb) == capi.E_ARG, (s, bb)
        torch.cuda.synchronize()
        assert ctx.launch_count() == n0
        assert (out == POISON).all().item(), "a refused call wrote"
        call(dtype=capi.CHW_F32, scale=(1, 2, 3), bias=(0, -1, 1))             # and the same call, right, is fine
        torch.cuda.synchronize()
        n1 = ctx.launch_count()
        assert n1 > n0
        ctx.set_format(1)
        with pytest.raises(g.RTjpegError) as e:
            call()
        assert e.value.code == capi.E_FORMAT
        ctx.set_format(0)
        assert ctx.launch_count() == n1
