"""BASELINE.json configs[4]: ONE inter-coded stream cut at clean frames (rtjgpu_split_shards_lead) and every shard
decoded by the CUDA path from nothing, on as many devices as are visible (shard i on device i mod #devices; on a
one-GPU box the shards run one after the other, which still proves that independently started shards reproduce the
sequential picture sequence).  Expected frames: the unmodified reference decoding the whole stream sequentially into
one persistent picture (lib/video_rtjpeg.c:81; skipped blocks keep what is there, lib/RTjpeg.c:2704)."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from gpu_util import first_diff
from streams import clip, reference_frames

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def contexts():
    cs = [g.BatchContext(d) for d in range(torch.cuda.device_count())]
    yield cs
    for c in cs:
        c.close()


def clean_frames(ctx, s, o, w, h):
    """K1 alone over the whole stream: a frame without a skip marker is clean (the header's key byte is only a hint)."""
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, w, h, device=ctx.device)
    with torch.cuda.device(ctx.device):
        ctx.scan_device(b.stream.data_ptr(), b.desc.data_ptr(), b.F, w, h, torch.cuda.current_stream().cuda_stream)
        counts = ctx.skip_counts(b.F)
    assert ctx.batch_info().bad_frames == 0
    return (counts == 0).astype(np.uint8)


def decode_shard(ctx, s, o, a, b, w, h, carry):
    """Frames [a, b) of the stream as a batch of their own on ctx's device."""
    sub = s[int(o[a]):int(o[b])]
    rel = (o[a:b + 1] - o[a]).astype(np.uint64)
    desc, _ = g.plan(sub, rel)
    with torch.cuda.device(ctx.device):
        bt = D.upload(sub, desc, w, h, device=ctx.device)
        bt.out.fill_(0xCD)
        D.decode(ctx, bt, torch.from_numpy(carry).to(bt.out.device))
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
        return bt.out.cpu().numpy()


def sharded(contexts, s, o, w, h, n, init):
    F = len(o) - 1
    clean = clean_frames(contexts[0], s, o, w, h)
    first, lead = g.split_shards_lead(clean, n)
    assert first[0] == 0 and first[-1] == F and (np.diff(first) > 0).all()
    garbage = np.random.default_rng(5).integers(0, 256, w * h * 3 // 2).astype(np.uint8)
    out = np.empty((F, w * h * 3 // 2), dtype=np.uint8)
    for i in range(n):
        a = int(first[i] - lead[i])
        # only a shard that starts at frame 0 sees the caller's picture; every other one starts from garbage, which a
        # clean first frame must overwrite completely
        fr = decode_shard(contexts[i % len(contexts)], s, o, a, int(first[i + 1]), w, h, init if a == 0 else garbage)
        out[int(first[i]):int(first[i + 1])] = fr[int(lead[i]):]
    return out, clean, first, lead


@pytest.mark.parametrize("n", [2, 4, 8])
def test_config5_1920x1088_inter_sharded(contexts, n):
    w, h, F = 1920, 1088, 64
    s, o = clip(w, h, 128, F, key_rate=7, lm=2, cm=2)
    init = np.full(w * h * 3 // 2, 0x30, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    got, clean, first, lead = sharded(contexts, s, o, w, h, n, init)
    assert clean[::8].all() and clean.sum() == 8 and (lead == 0).all()       # cuts on the GOP boundaries, nothing decoded twice
    assert np.array_equal(got, want), first_diff(got, want, w, h)


@pytest.mark.parametrize("n", [2, 4, 8])
def test_config5_720x576_gop30_sharded(contexts, n):
    w, h, F = 720, 576, 120
    s, o = clip(w, h, 128, F, key_rate=29, lm=4, cm=4)
    init = np.full(w * h * 3 // 2, 0x62, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    got, clean, first, lead = sharded(contexts, s, o, w, h, n, init)
    if n == 8:
        assert (lead > 0).any()             # eight shards over four GOPs: half of them decode back to their GOP's key frame
    assert np.array_equal(got, want), first_diff(got, want, w, h)


@pytest.mark.parametrize("n", [2, 4])
def test_key_frames_with_skips_shard_correctly(contexts, n):
    """Dark flat material at Q=32: the encoder's 'key' frames still carry skip markers (SURVEY.md section 0-5), so
    cutting at fh->key == 0 would be wrong.  No frame is clean: every shard leads back to frame 0 and the caller's
    picture -- redundant, but right."""
    w, h, F = 720, 576, 45
    s, o = clip(w, h, 32, F, key_rate=14, lm=4, cm=4, dark=1)
    keys = np.array([s[int(o[f]) + 11] for f in range(F)])
    assert (keys == 0).sum() == 3                                          # what the header claims
    init = np.full(w * h * 3 // 2, 0x37, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    got, clean, first, lead = sharded(contexts, s, o, w, h, n, init)
    assert clean.sum() == 0 and list(lead) == list(first[:-1])
    assert np.array_equal(got, want), first_diff(got, want, w, h)
    # and the cut the header suggests does go wrong (so the test above means something)
    wrong = decode_shard(contexts[0], s, o, 15, 30, w, h, np.zeros(w * h * 3 // 2, np.uint8))
    assert not np.array_equal(wrong, want[15:30])
