"""K2 working through RUNS of frames (rtjgpu_set_frame_runs): a CTA keeps its row's pixels in shared memory from frame to frame
and leaves what a frame skips untouched -- the reference's persistent picture (lib/video_rtjpeg.c:81, lib/RTjpeg.c:2704) at the
scale of a macroblock row.  The frames must not depend on the run length; expected pixels come from the compiled reference."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from gpu_util import first_diff, gpu_decode
from streams import clip, interleave, reference_frames
from test_gpu_fused_rgb import decode_rgb, expect

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("run", [1, 2, 8, 64])
def test_inter_batch_any_run_length(run):
    """300 inter frames (above AUTO's segment-parallel limit: K1 one CTA a frame, K3 over ten chunks of frames): skipped blocks
    whose last writers are inline, mid-size and long blocks, blocks nobody has written yet (carried in from the picture before
    the batch), key frames in the middle of runs."""
    w, h, F = 352, 288, 300
    s, o = clip(w, h, 150, F, key_rate=13, lm=2, cm=1, noise_y=14, noise_c=4)
    init = np.full(w * h * 3 // 2, 0x47, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    with g.BatchContext(0) as c:
        c.set_frame_runs(run)
        got, _ = gpu_decode(c, s, o, w, h, carry=init)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        assert c.batch_info().bad_frames == 0 and c.batch_info().skipped_blocks > 0


def test_frames_that_start_with_skips_and_no_carry():
    """The batch's first frames skip blocks that no frame of the batch has written and no picture is carried in: zeros, and
    they persist through the runs until somebody writes."""
    w, h = 208, 112
    s, o = clip(w, h, 128, 9, key_rate=20, lm=4, cm=4, noise_y=3)
    sizes = O.packet_sizes(s, o)
    pk = [s[int(o[i]):int(o[i]) + int(sizes[i])] for i in range(1, 9)]          # drop the key frame
    s2, o2 = O.pack_packets(pk)
    want = reference_frames(s2, o2, w, h)
    with g.BatchContext(0) as c:
        c.set_frame_runs(5)
        got, _ = gpu_decode(c, s2, o2, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)


def test_quality_changes_inside_runs():
    """Two clips of different quality interleaved: a skipped block's last writer used other tables (the general decoder's
    business when every frame stands for itself).  Inside a run the pixels simply stay."""
    w, h = 160, 96
    a = clip(w, h, 60, 6, key_rate=5, lm=2, cm=2, noise_y=8)
    b = clip(w, h, 200, 6, key_rate=5, lm=2, cm=2, noise_y=8, seed=3)
    s, o = interleave([a, b])
    want = reference_frames(s, o, w, h)
    for run in (1, 4):
        with g.BatchContext(0) as c:
            c.set_frame_runs(run)
            got, _ = gpu_decode(c, s, o, w, h)
            assert np.array_equal(got, want), (run, first_diff(got, want, w, h))


def test_default_follows_the_batch_before():
    """frames = 0: the arrangement of a batch goes by the skip count of the batch before it.  Whatever it picks, the frames
    are the reference's: an inter batch twice (every frame for itself, then runs), an intra batch behind it (runs once more,
    on a stream without a single skipped block), the intra batch again."""
    w, h = 352, 288
    si, oi = clip(w, h, 128, 300, key_rate=9, lm=1, cm=1, noise_y=5)
    sa, oa = clip(w, h, 128, 300, noise_y=5)
    want_i, want_a = reference_frames(si, oi, w, h), reference_frames(sa, oa, w, h)
    with g.BatchContext(0) as c:
        for _ in range(2):
            got, _ = gpu_decode(c, si, oi, w, h)
            assert np.array_equal(got, want_i), first_diff(got, want_i, w, h)
        for _ in range(2):
            got, _ = gpu_decode(c, sa, oa, w, h)
            assert np.array_equal(got, want_a), first_diff(got, want_a, w, h)


@pytest.mark.parametrize("kind", [capi.CONV_RGB32, capi.CONV_BGR24])
def test_fused_rgb_in_runs(kind):
    w, h, F = 352, 288, 40
    s, o = clip(w, h, 128, F, key_rate=7, lm=2, cm=2, noise_y=10)
    init = np.full(w * h * 3 // 2, 0x60, dtype=np.uint8)
    frames = reference_frames(s, o, w, h, init)
    with g.BatchContext(0) as ctx:
        ctx.set_frame_runs(6)
        got, pitch, last = decode_rgb(ctx, s, o, w, h, kind, carry=init, want_last=True)
    assert np.array_equal(got, expect(frames, w, h, kind, pitch, 0x5A))
    assert np.array_equal(last, frames[-1])


def test_wide_picture_in_strips_and_runs():
    """2064 wide: two strips per row of macroblocks (the kernel without the position table and bulk stores)."""
    w, h = 2064, 48
    s, o = clip(w, h, 128, 12, key_rate=5, lm=2, cm=2, noise_y=10)
    want = reference_frames(s, o, w, h)
    with g.BatchContext(0) as c:
        c.set_frame_runs(4)
        got, _ = gpu_decode(c, s, o, w, h)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
