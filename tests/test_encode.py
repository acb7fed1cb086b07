"""The encoder half, RTjpeg_compress (lib/RTjpeg.c:3488-3524): the oracle's restatement against the unmodified reference
(CPU; packets must be byte-identical), the CUDA encoder against both through the C ABI (GPU), and the round trip through
this library's own decoder."""
import numpy as np
import pytest

from oracle import oracle as O
from streams import golden, reference_frames

CASES = [  # fmt, w, h, Q, key_rate, lm
    (0, 64, 48, 128, -1, 0), (0, 96, 64, 200, 5, 2), (0, 48, 32, 255, 3, 1), (0, 160, 32, 32, 2, 6), (0, 32, 32, 171, 255, 16),
    (1, 64, 48, 128, -1, 0), (1, 96, 64, 228, 4, 2), (1, 160, 32, 32, 2, 6),
]


def _pictures(fmt, w, h, n=10, seed=5):
    """A moving synthetic clip, one full-range random picture and a repeated picture (every block skipped)."""
    rng = np.random.default_rng(seed)
    s, o = O.encode_clip(O.make_clip(w, h, 255, noise_y=20, noise_c=6, dark=1), n, threads=1)
    fr = O.frames_in_format(reference_frames(s, o, w, h), w, h, fmt)
    return np.concatenate([fr, rng.integers(0, 256, (1, fr.shape[1])).astype(np.uint8), fr[-1:], fr[-1:]])


@pytest.mark.skipif(not O.have_ref(), reason="reference build absent (oracle/_ref)")
@pytest.mark.parametrize("fmt,w,h,Q,kr,lm", CASES)
def test_restatement_matches_live_reference_encoder(fmt, w, h, Q, kr, lm):
    fr = _pictures(fmt, w, h)
    a_s, a_o = O.encode_frames_fmt(O.make_clip(w, h, Q, kr, lm, lm), fmt, fr)
    b_s, b_o = O.encode_frames_oracle(fr, w, h, fmt, Q, kr, lm, lm)
    assert np.array_equal(a_o, b_o) and np.array_equal(a_s, b_s)


def test_restatement_matches_golden_encoder():
    g = golden("encode_64x48")
    for fmt, key in ((0, "420"), (1, "422")):
        s, o = O.encode_frames_oracle(g["pics" + key], 64, 48, fmt, int(g["Q"]), int(g["key_rate"]), int(g["lm"]), int(g["cm"]))
        assert np.array_equal(s, g["stream" + key]) and np.array_equal(o, g["offsets" + key])


# The streams of tests/golden/ and the settings make_golden.py made them with: the reference's own encoder over the
# seeded source.  A grey picture is read up to 56 rows past its end (rtjo_encode_frame8); where that reached past the
# last picture the fixture holds what lay behind it then, so only the first `exact` packets are compared.
CLIPS = [  # name, fmt, w, h, Q, frames, clip settings, exact
    ("intra_64x48_q128", 0, 64, 48, 128, 4, dict(noise_y=6, noise_c=3), 4),
    ("intra_320x240_q128", 0, 320, 240, 128, 2, {}, 2),
    ("inter_64x48_q200_gop6", 0, 64, 48, 200, 14, dict(key_rate=5, lm=2, cm=2, noise_y=30, noise_c=8), 14),
    ("inter_dark_96x64_q32_gop4", 0, 96, 64, 32, 10, dict(key_rate=3, lm=4, cm=4, dark=1), 10),
    ("dense_48x32_q255", 0, 48, 32, 255, 3, dict(noise_y=110, noise_c=90), 3),
    ("yuv422_inter_64x48_q200_gop4", 1, 64, 48, 200, 9, dict(key_rate=3, lm=2, cm=2, noise_y=30, noise_c=8), 9),
    ("yuv422_intra_96x32_q128", 1, 96, 32, 128, 3, dict(noise_y=6, noise_c=3), 3),
    ("grey_inter_64x48_q255_gop4", 2, 64, 48, 255, 9, dict(key_rate=3, lm=2, cm=2, noise_y=40), 7),
    ("grey_intra_96x32_q64", 2, 96, 32, 64, 3, dict(noise_y=6), 2),
]


@pytest.mark.parametrize("name,fmt,w,h,Q,F,kw,exact", CLIPS)
def test_clip_streams_match_golden(name, fmt, w, h, Q, F, kw, exact):
    """The synthetic clips tests and bench.py decode come from the restated encoder: the reference's packets, byte for byte."""
    g = golden(name)
    if fmt == 0:
        s, o = O.encode_clip(O.make_clip(w, h, Q, **kw), F, threads=3)
    else:
        kw = dict(kw)
        kr, lm, cm = kw.pop("key_rate", -1), kw.pop("lm", 0), kw.pop("cm", 0)
        s, o = O.encode_clip_fmt(w, h, Q, F, fmt, kr, lm, cm, **kw)
    if exact == F:
        assert np.array_equal(s, g["stream"]) and np.array_equal(o, g["offsets"])
    got, want = O.packet_sizes(s, o), O.packet_sizes(g["stream"], g["offsets"])
    for f in range(exact):
        assert np.array_equal(s[int(o[f]):int(o[f]) + int(got[f])],
                              g["stream"][int(g["offsets"][f]):int(g["offsets"][f]) + int(want[f])]), f


def test_grey_encoder_is_refused():
    with pytest.raises(ValueError):
        O.encode_frames_oracle(np.zeros((1, 64 * 48), dtype=np.uint8), 64, 48, 2, 128)


def _want(fr, w, h, fmt, Q, kr, lm, align=4):
    if O.have_ref():
        return O.encode_frames_fmt(O.make_clip(w, h, Q, kr, lm, lm), fmt, fr, align=align)
    return O.encode_frames_oracle(fr, w, h, fmt, Q, kr, lm, lm, align=align)


def _gpu_encode(ctx, fr, w, h, fmt):
    import torch
    F = fr.shape[0]
    cap = F * (12 + (w // 8) * (h // 8) * 2 * 64 + 16)
    d_fr = torch.from_numpy(fr).cuda()
    d_stream = torch.full((cap,), 0xEE, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(F + 1, dtype=torch.int64, device="cuda")
    ctx.set_format(fmt)
    try:
        ctx.encode_device(d_fr.data_ptr(), F, w, h, d_stream.data_ptr(), cap, d_off.data_ptr(), torch.cuda.current_stream().cuda_stream)
        nbytes, overflow = ctx.encode_info()
    finally:
        ctx.set_format(0)
    assert not overflow
    return d_stream[:nbytes].cpu().numpy(), d_off.cpu().numpy().astype(np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,w,h,Q,kr,lm", CASES + [(0, 720, 576, 128, 29, 2), (1, 320, 240, 64, 0, 0), (0, 1920, 1088, 255, 3, 1)])
def test_encode_device_matches_reference(fmt, w, h, Q, kr, lm):
    import gmerlin_avdecoder_b200 as g
    fr = _pictures(fmt, w, h, n=6 if w > 1000 else 10)
    want_s, want_o = _want(fr, w, h, fmt, Q, kr, lm)
    with g.BatchContext(0) as ctx:
        ctx.encoder_config(Q, max(kr, 0), lm, lm)
        got_s, got_o = _gpu_encode(ctx, fr, w, h, fmt)
        # the reference driver ends its offsets at the last packet's last byte, the device at the next multiple of 4
        end = int(want_o[-1])
        assert np.array_equal(got_o[:-1], want_o[:-1]) and int(got_o[-1]) == (end + 3) // 4 * 4 == got_s.size
        assert np.array_equal(got_s[:end], want_s[:end]) and not got_s[end:].any()
        # the encoder's state carries over: the same clip in two calls gives the same packets
        ctx.encoder_config(Q, max(kr, 0), lm, lm)
        a_s, a_o = _gpu_encode(ctx, fr[:5], w, h, fmt)
        b_s, b_o = _gpu_encode(ctx, fr[5:], w, h, fmt)
        assert np.array_equal(np.concatenate([a_s, b_s])[:end], want_s[:end])


@pytest.mark.gpu
def test_encode_decode_round_trip_on_device():
    """Encode on the device, decode what came out with this library's own decoder, compare with the reference decoding the
    reference's packets: the whole loop without the host touching a pixel."""
    import torch
    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import device as D
    w, h, Q, kr, lm = 320, 240, 128, 9, 2
    fr = _pictures(0, w, h, n=24)
    with g.BatchContext(0) as ctx:
        ctx.encoder_config(Q, kr, lm, lm)
        s, o = _gpu_encode(ctx, fr, w, h, 0)
        desc, _ = g.plan(s, o)
        b = D.upload(s, desc, w, h)
        D.decode(ctx, b)
        torch.cuda.synchronize()
        got = b.out.cpu().numpy()
    want_s, want_o = _want(fr, w, h, 0, Q, kr, lm)
    want = O.ref_decode_seq(want_s, want_o, w, h) if O.have_ref() else O.decode_stream(want_s, want_o, w, h)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_encode_overflow_is_reported():
    import torch
    import gmerlin_avdecoder_b200 as g
    fr = _pictures(0, 64, 48)
    with g.BatchContext(0) as ctx:
        ctx.encoder_config(200)
        d_fr = torch.from_numpy(fr).cuda()
        d_stream = torch.full((256,), 0xEE, dtype=torch.uint8, device="cuda")
        d_off = torch.zeros(fr.shape[0] + 1, dtype=torch.int64, device="cuda")
        ctx.encode_device(d_fr.data_ptr(), fr.shape[0], 64, 48, d_stream.data_ptr(), 256, d_off.data_ptr(), torch.cuda.current_stream().cuda_stream)
        nbytes, overflow = ctx.encode_info()
        assert overflow and nbytes > 256
        assert (d_stream.cpu().numpy() == 0xEE).all()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [0, 1])
def test_rtjpeg_compress_drop_in(fmt):
    import gmerlin_avdecoder_b200 as g
    w, h, Q, kr, lm = 96, 64, 171, 3, 1
    fr = _pictures(fmt, w, h)
    want_s, want_o = _want(fr, w, h, fmt, Q, kr, lm)
    sizes = O.packet_sizes(want_s, want_o)
    r = g.RTjpeg()
    r.set_format(fmt)
    assert r.set_size(w, h) == 0 and r.set_quality(Q) == Q
    r.set_intra(kr, lm, lm)
    for f in range(fr.shape[0]):
        pkt = r.compress(fr[f], w, h)
        assert np.array_equal(pkt, want_s[int(want_o[f]):int(want_o[f]) + int(sizes[f])]), f
    assert r.last_error() == 0
    r.set_format(2)
    assert r.compress(fr[0][:w * h], w, h).size == 0 and r.last_error() == g.capi.E_FORMAT
    r.close()
