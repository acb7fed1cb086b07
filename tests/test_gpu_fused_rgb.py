"""rtjgpu_decode_device_rgb: decode with one of the reference's yuv420 colour converters fused into K2 (SURVEY.md section
8f-4: "fused colour conversion").  Expected pixels: the compiled reference's RTjpeg_decompress followed by its
RTjpeg_yuv420rgb32 / bgr32 / rgb24 / bgr24 / rgb16 (lib/RTjpeg.c:3123-3475) -- byte for byte."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from streams import clip, interleave, reference_frames

pytestmark = pytest.mark.gpu

KINDS = [capi.CONV_RGB32, capi.CONV_BGR32, capi.CONV_RGB24, capi.CONV_BGR24, capi.CONV_RGB16]


def decode_rgb(ctx, s, o, w, h, kind, pad=0, alpha=0x5A, carry=None, want_last=False):
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, w, h)
    bpp = capi.CONV_BPP[kind]
    pitch = (w * bpp + pad + 15) // 16 * 16
    out = torch.full((b.F, h, pitch), 0xCD, dtype=torch.uint8, device="cuda")
    last = torch.full((w * h * 3 // 2,), 0xEE, dtype=torch.uint8, device="cuda") if want_last else None
    ct = None if carry is None else torch.from_numpy(np.ascontiguousarray(carry)).cuda()
    ctx.set_format(0)
    ctx.decode_device_rgb(b.stream.data_ptr(), b.desc.data_ptr(), b.F, w, h, kind, out.data_ptr(), pitch, h * pitch, alpha,
                          None if ct is None else ct.data_ptr(), None if last is None else last.data_ptr(),
                          torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert ctx.batch_info().bad_frames == 0
    return out.cpu().numpy(), pitch, None if last is None else last.cpu().numpy()


def expect(frames, w, h, kind, pitch, alpha):
    """The reference's converter over the reference's frames; bytes it does not write -- the fourth byte of a 32-bit pixel,
    which the batch call fills with alpha, and the row padding, which it leaves alone -- are set accordingly."""
    bpp = capi.CONV_BPP[kind]
    out = np.empty((len(frames), h, pitch), dtype=np.uint8)
    for f, fr in enumerate(frames):
        px = (O.ref_convert if O.have_ref() else O.convert)(kind, fr, w, h, pitch=w * bpp, fill=alpha)
        out[f, :, :w * bpp] = px
        out[f, :, w * bpp:] = 0xCD
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_intra_720x576(kind):
    w, h, F = 720, 576, 5
    s, o = clip(w, h, 128, F)
    frames = reference_frames(s, o, w, h)
    with g.BatchContext(0) as ctx:
        got, pitch, last = decode_rgb(ctx, s, o, w, h, kind, pad=48, want_last=True)
    assert np.array_equal(got, expect(frames, w, h, kind, pitch, 0x5A))
    assert np.array_equal(last, frames[-1])


@pytest.mark.parametrize("kind", [capi.CONV_RGB32, capi.CONV_BGR24, capi.CONV_RGB16])
@pytest.mark.parametrize("scan,pipeline,slice_frames", [(capi.SCAN_AUTO, capi.PIPELINE_SLICED, 0), (capi.SCAN_CHUNK, capi.PIPELINE_SLICED, 32),
                                                        (capi.SCAN_CHUNK, capi.PIPELINE_SERIAL, 64)])
def test_inter_with_carry(kind, scan, pipeline, slice_frames):
    """Skipped blocks come from their last writer or from the picture before the batch -- planes, whatever leaves."""
    w, h, F = 320, 240, 90
    s, o = clip(w, h, 128, F, key_rate=29, lm=3, cm=3, dark=1)
    init = np.random.default_rng(2).integers(16, 236, w * h * 3 // 2).astype(np.uint8)
    frames = reference_frames(s, o, w, h, init)
    with g.BatchContext(0) as ctx:
        ctx.set_scan_mode(scan)
        ctx.set_pipeline(pipeline, slice_frames)
        got, pitch, last = decode_rgb(ctx, s, o, w, h, kind, carry=init, want_last=True)
        assert ctx.batch_info().skipped_blocks > 0
    assert np.array_equal(got, expect(frames, w, h, kind, pitch, 0x5A))
    assert np.array_equal(last, frames[-1])


@pytest.mark.parametrize("kind", [capi.CONV_BGR32, capi.CONV_RGB24])
def test_blocks_outside_the_sparse_classes(kind):
    """Q=255 (raw prefix: every luma block takes the general decoder) interleaved with Q=128 and Q=32 frames, inter-coded:
    long blocks and blocks whose last writer used other tables are decoded inside the fused kernel."""
    w, h, F = 160, 96, 18
    st, of = interleave([clip(w, h, 128, F, key_rate=5, lm=2, cm=2), clip(w, h, 255, F, key_rate=5, lm=2, cm=2, seed=3),
                         clip(w, h, 32, F, key_rate=5, lm=2, cm=2, seed=5, noise_y=40)])
    init = np.full(w * h * 3 // 2, 0x70, dtype=np.uint8)
    frames = reference_frames(st, of, w, h, init)
    with g.BatchContext(0) as ctx:
        got, pitch, _ = decode_rgb(ctx, st, of, w, h, kind, carry=init)
    assert np.array_equal(got, expect(frames, w, h, kind, pitch, 0x5A))


def test_wide_picture_in_strips():
    """More than 128 macroblocks wide: K2 works on strips of a macroblock row, the fused epilogue on strips of pixels."""
    w, h, F = 2080, 32, 3
    s, o = clip(w, h, 128, F, key_rate=2, lm=2, cm=2)
    frames = reference_frames(s, o, w, h)
    with g.BatchContext(0) as ctx:
        got, pitch, last = decode_rgb(ctx, s, o, w, h, capi.CONV_RGB32, want_last=True)
    assert np.array_equal(got, expect(frames, w, h, capi.CONV_RGB32, pitch, 0x5A))
    assert np.array_equal(last, frames[-1])


def test_arguments():
    w, h = 64, 48
    s, o = clip(w, h, 128, 2)
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, w, h)
    out = torch.empty((2, h, w * 4), dtype=torch.uint8, device="cuda")
    with g.BatchContext(0) as ctx:
        def call(kind=capi.CONV_RGB32, ptr=None, pitch=w * 4):
            ctx.decode_device_rgb(b.stream.data_ptr(), b.desc.data_ptr(), 2, w, h, kind, out.data_ptr() if ptr is None else ptr,
                                  pitch, h * pitch)
        call()
        for bad in (dict(kind=capi.CONV_RGB8), dict(kind=capi.CONV_YUV422_RGB24), dict(kind=99)):
            with pytest.raises(g.RTjpegError) as e:
                call(**bad)
            assert e.value.code == capi.E_FORMAT
        for bad in (dict(ptr=out.data_ptr() + 4), dict(pitch=w * 4 - 16), dict(pitch=w * 4 + 8)):
            with pytest.raises(g.RTjpegError) as e:
                call(**bad)
            assert e.value.code == capi.E_ARG
        ctx.set_format(1)
        with pytest.raises(g.RTjpegError) as e:
            call()
        assert e.value.code == capi.E_FORMAT
