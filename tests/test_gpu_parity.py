"""Parity of the CUDA path (through the C ABI) with the reference: bit-exact Y/U/V."""
import ctypes as C

import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from gpu_util import first_diff, gpu_decode
from streams import clip, golden, interleave, reference_frames, reference_frames_threaded

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["auto", "chunk", "lane", "warp", "walk", "sync", "runs", "segment"])
def ctx(request):
    """Every parity case runs under all flavours of the block-offset scan (K1): the default (which
    picks the segment-parallel arrangement for the small batches of this suite and one CTA per frame
    for the full-size one), one CTA per frame forced, and each serial kernel alone."""
    c = g.BatchContext(0)
    c.set_scan_mode({"auto": capi.SCAN_AUTO, "chunk": capi.SCAN_CHUNK, "lane": capi.SCAN_LANE,
                     "warp": capi.SCAN_WARP, "walk": capi.SCAN_WALK, "sync": capi.SCAN_SYNC, "runs": capi.SCAN_AUTO, "segment": capi.SCAN_SEGMENT}[request.param])
    if request.param == "runs":
        c.set_frame_runs(3)              # K2 works through runs of three frames, the strip staying on chip
    c.flavour = request.param
    yield c
    c.close()


GOLDEN = ["intra_64x48_q128", "intra_320x240_q128", "inter_64x48_q200_gop6",
          "inter_dark_96x64_q32_gop4", "dense_48x32_q255", "random_48x32"]


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_fixtures(ctx, name):
    gd = golden(name)
    w, h = int(gd["w"]), int(gd["h"])
    init = np.full(w * h * 3 // 2, int(gd["init_fill"]), dtype=np.uint8)
    got, _ = gpu_decode(ctx, gd["stream"], gd["offsets"], w, h, carry=init)
    want = gd["frames"] if "frames" in gd else reference_frames(gd["stream"], gd["offsets"], w, h, init)
    assert np.array_equal(got, want), first_diff(got, want, w, h)
    assert ctx.batch_info().bad_frames == 0


def _check_clip(ctx, w, h, Q, F, init_fill=0, **kw):
    s, o = clip(w, h, Q, F, **kw)
    init = np.full(w * h * 3 // 2, init_fill, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    got, _ = gpu_decode(ctx, s, o, w, h, carry=init if init_fill else None)
    assert np.array_equal(got, want), first_diff(got, want, w, h)
    bi = ctx.batch_info()
    assert bi.bad_frames == 0
    assert bi.payload_bytes == int(O.packet_sizes(s, o).astype(np.int64).sum()) - 12 * F
    return s, o, bi


def test_config1_320x240_intra(ctx):
    _check_clip(ctx, 320, 240, 128, 16)


@pytest.mark.parametrize("Q", [32, 128, 255])
def test_config2_720x576_intra(ctx, Q):
    _, _, bi = _check_clip(ctx, 720, 576, Q, 24)
    assert bi.skipped_blocks == 0


@pytest.mark.parametrize("lm,cm", [(1, 1), (4, 4)])
def test_config3_720x576_inter_gop30(ctx, lm, cm):
    _, _, bi = _check_clip(ctx, 720, 576, 128, 64, key_rate=29, lm=lm, cm=cm, init_fill=0x55)
    assert bi.skipped_blocks > 0
    counts = ctx.skip_counts(64)
    assert counts.sum() == bi.skipped_blocks
    assert counts[0] == 0 and counts[30] == 0 and counts[60] == 0


def test_config3_key_frames_with_skips(ctx):
    # dark flat third at Q=32: "key" frames still carry 0xFF markers (SURVEY.md section 0-5)
    s, o, bi = _check_clip(ctx, 720, 576, 32, 45, key_rate=14, lm=4, cm=4, dark=1, init_fill=0x37)
    counts = ctx.skip_counts(45)
    assert counts[0] > 0 and counts[15] > 0


def test_config4_1920x1088_dense(ctx):
    _check_clip(ctx, 1920, 1088, 255, 4, noise_y=60, noise_c=20)
    _check_clip(ctx, 1920, 1088, 255, 2, noise_y=110, noise_c=0)


@pytest.mark.parametrize("Q", [1, 2, 32, 170, 171, 199, 200, 227, 228, 255])
def test_random_wellformed_streams(ctx, Q):
    rng = np.random.default_rng(100 + Q)
    pk = [O.random_wellformed_packet(rng, 160, 96, Q, skip_prob=p, dense_prob=dp)
          for p, dp in ((0.0, 0.3), (0.2, 0.3), (0.5, 1.0), (0.1, 0.0))]
    s, o = O.pack_packets(pk)
    init = rng.integers(0, 256, 160 * 96 * 3 // 2).astype(np.uint8)
    want = reference_frames(s, o, 160, 96, init)
    got, _ = gpu_decode(ctx, s, o, 160, 96, carry=init)
    assert np.array_equal(got, want), first_diff(got, want, 160, 96)


def test_quality_changes_and_foreign_table_sources(ctx):
    # two inter-coded clips of different quality, interleaved frame by frame: skipped blocks
    # of a Q=90 frame are last written by a Q=210 frame and the other way round
    a = clip(208, 112, 90, 24, key_rate=7, lm=3, cm=3, noise_y=3, seed=4)
    b = clip(208, 112, 210, 24, key_rate=5, lm=2, cm=2, noise_y=3, seed=4)
    s, o = interleave([a, b])
    init = np.full(208 * 112 * 3 // 2, 0x42, dtype=np.uint8)
    want = reference_frames(s, o, 208, 112, init)
    got, st = gpu_decode(ctx, s, o, 208, 112, carry=init)
    assert np.array_equal(got, want), first_diff(got, want, 208, 112)
    assert st.quality == 210


def test_quality_zero_on_fresh_and_configured_decoder(ctx):
    rng = np.random.default_rng(9)
    pkt = O.random_wellformed_packet(rng, 64, 64, 1, skip_prob=0.3)
    pkt[10] = 0
    s, o = O.pack_packets([pkt, pkt])
    init = np.full(64 * 64 * 3 // 2, 0x55, dtype=np.uint8)
    want = reference_frames(s, o, 64, 64, init)
    got, _ = gpu_decode(ctx, s, o, 64, 64, carry=init)              # fresh: zero tables
    assert np.array_equal(got, want)
    good = O.random_wellformed_packet(rng, 64, 64, 77, skip_prob=0.0)
    s, o = O.pack_packets([good, pkt])
    want = reference_frames(s, o, 64, 64, init)
    got, _ = gpu_decode(ctx, s, o, 64, 64, carry=init)              # configured: falls to Q=1
    assert np.array_equal(got, want)


def test_carry_across_batches(ctx):
    s, o = clip(160, 96, 128, 40, key_rate=29, lm=2, cm=2, noise_y=3)
    want = reference_frames(s, o, 160, 96)
    first, st = gpu_decode(ctx, s, o[:18], 160, 96)
    second, _ = gpu_decode(ctx, s[int(o[17]):], o[17:] - o[17], 160, 96, carry=first[-1], state=st)
    assert np.array_equal(np.concatenate([first, second]), want)


def _scan_only(ctx, s, o, w, h):
    """K1 alone (rtjgpu_scan_device): the entries as the scan makes them, before K3 touches the skipped ones."""
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, w, h)
    ctx.set_format(0)
    ctx.scan_device(b.stream.data_ptr(), b.desc.data_ptr(), b.F, w, h, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert ctx.batch_info().bad_frames == 0
    return b


def test_scan_entries_match_oracle_walker(ctx):
    s, o = clip(208, 112, 200, 6, key_rate=2, lm=3, cm=3, noise_y=25, noise_c=5)
    w, h = 208, 112
    nblk = (w // 16) * (h // 16) * 6
    _scan_only(ctx, s, o, w, h)
    L = g.load_library()
    ent = np.zeros(6 * nblk, dtype=np.uint32)
    L.rtjgpu_get_entries.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    assert L.rtjgpu_get_entries(ctx._h, C.c_void_p(ent.ctypes.data), ent.size) == 0
    ent = ent.reshape(6, nblk)
    t = O.tables_from_quality(200)
    sizes = O.packet_sizes(s, o)
    for f in range(6):
        n, offs, eob = O.walk_payload(s[int(o[f]) + 12:int(o[f]) + int(sizes[f])], nblk // 6, t.lb8, t.cb8)
        coded = eob > 0
        assert ((ent[f] == 0xFFFFFFFF) == ~coded).all()
        # Q=200: luma blocks carry a raw prefix (never inline); chroma blocks (cb8 = 0) may go inline
        inline = coded & (ent[f] >> 31 == 1)
        chroma = (np.arange(nblk) % 6) >= 4
        assert not (inline & ~chroma).any()
        assert (eob[inline] <= 3).all()
        if ctx.flavour in ("lane", "warp"):
            assert not inline.any()                      # these serial kernels never emit inline entries
        gen = coded & ~inline
        assert ((ent[f] & 0x1FFFFFF)[gen] == offs[gen]).all()
        # the kernel's bound may exceed the exact end-of-block, never undercut it
        keob = ((ent[f] >> 25) & 63) + 1
        assert (keob[gen] >= eob[gen]).all()
        assert (keob[gen] == eob[gen]).mean() > 0.99


def test_scan_entries_inline_format(ctx):
    """Frames without a raw prefix: the chunk-parallel scan carries blocks with an end-of-block
    bound <= 3 inside the entry (DC and two coefficients), the rest by offset.  The lane and warp
    kernels carry every block by offset."""
    s, o = clip(208, 112, 128, 4, key_rate=1, lm=2, cm=2, noise_y=12, noise_c=3)
    w, h = 208, 112
    nblk = (w // 16) * (h // 16) * 6
    _scan_only(ctx, s, o, w, h)
    L = g.load_library()
    ent = np.zeros(4 * nblk, dtype=np.uint32)
    L.rtjgpu_get_entries.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    assert L.rtjgpu_get_entries(ctx._h, C.c_void_p(ent.ctypes.data), ent.size) == 0
    ent = ent.reshape(4, nblk)
    sizes = O.packet_sizes(s, o)
    inline_scan = ctx.flavour not in ("lane", "warp")
    seen_inline = seen_general = 0
    for f in range(4):
        pay = s[int(o[f]) + 12:int(o[f]) + int(sizes[f])]
        n, offs, eob = O.walk_payload(pay, nblk // 6, 0, 0)
        for b in range(nblk):
            e = int(ent[f, b])
            if eob[b] == 0:
                assert e == 0xFFFFFFFF
            elif e >> 31:
                assert eob[b] <= 3 and (e >> 24) == 0x80
                p = int(offs[b])
                assert (e & 0xFF) == pay[p]
                want = [0, 0]
                if eob[b] >= 2:
                    want[0] = int(pay[p + 1]) if not 64 <= pay[p + 1] < 128 else 0
                if eob[b] >= 3:
                    want[1] = int(pay[p + 2]) if not 64 <= pay[p + 2] < 128 else 0
                assert ((e >> 8) & 0xFF, (e >> 16) & 0xFF) == tuple(want)
                seen_inline += 1
            else:
                # a scan that makes inline entries gives every general one a bound of at least 4
                assert (e & 0x1FFFFFF) == offs[b] and ((e >> 25) & 63) + 1 >= max(int(eob[b]), 4 if inline_scan else 0)
                seen_general += 1
    assert seen_general and bool(seen_inline) == inline_scan


def test_k3_gives_skipped_blocks_a_copy_of_an_inline_last_writer(ctx):
    """After a decode, the marker of a skipped block whose last writer's entry is an inline one (same tables) has been
    replaced by that entry with bit 30 set; every other skipped block keeps its marker (all of them after the lane and
    warp kernels, which make no inline entries)."""
    w, h, F = 208, 112, 12
    s, o = clip(w, h, 128, F, key_rate=5, lm=3, cm=3, noise_y=6)
    nblk = (w // 16) * (h // 16) * 6
    L = g.load_library()
    L.rtjgpu_get_entries.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    _scan_only(ctx, s, o, w, h)
    k1 = np.zeros(F * nblk, dtype=np.uint32)
    assert L.rtjgpu_get_entries(ctx._h, C.c_void_p(k1.ctypes.data), k1.size) == 0
    k1 = k1.reshape(F, nblk)
    gpu_decode(ctx, s, o, w, h)
    k3 = np.zeros(F * nblk, dtype=np.uint32)
    assert L.rtjgpu_get_entries(ctx._h, C.c_void_p(k3.ctypes.data), k3.size) == 0
    k3 = k3.reshape(F, nblk)
    copies = 0
    last = np.full(nblk, -1)
    for f in range(F):
        skip = k1[f] == 0xFFFFFFFF
        assert np.array_equal(k3[f][~skip], k1[f][~skip])                  # coded blocks are left alone
        for b in np.flatnonzero(skip):
            lw = last[b]
            inl = lw >= 0 and (k1[lw, b] >> 31) == 1
            if inl:
                assert k3[f, b] == (k1[lw, b] | 0x40000000), (f, b)
                copies += 1
            else:
                assert k3[f, b] == 0xFFFFFFFF, (f, b)
        last[~skip] = f
    if ctx.flavour in ("lane", "warp"):
        assert copies == 0
    else:
        assert copies > 100


def test_edge_geometries(ctx):
    _check_clip(ctx, 16, 16, 128, 3, noise_y=20)                      # one macroblock
    _check_clip(ctx, 2064, 16, 128, 2, noise_y=10)                    # 129 macroblocks: two strips per row
    _check_clip(ctx, 16, 272, 255, 2, noise_y=40, key_rate=1, lm=1, cm=1)
    _check_clip(ctx, 4112, 32, 60, 1, noise_y=4)                      # three strips


def test_empty_batch(ctx):
    ctx.decode_device(0, 0, 0, 64, 48, 0)
    out = np.zeros((0, 10), dtype=np.uint8)
    ctx.decode_host(np.zeros(16, dtype=np.uint8), np.zeros(1, dtype=np.uint64), out)


def test_truncated_frame_is_flagged_not_overread(ctx):
    s, o = clip(160, 96, 128, 3, noise_y=8)
    sizes = O.packet_sizes(s, o)
    # cut the second packet short: keep the header's framesize honest about what is there
    cut = int(o[1]) + int(sizes[1]) // 2
    pk = [s[int(o[0]):int(o[0]) + int(sizes[0])], s[int(o[1]):cut].copy(), s[int(o[2]):int(o[2]) + int(sizes[2])]]
    pk[1][0:4] = np.frombuffer(np.uint32(pk[1].size).tobytes(), dtype=np.uint8)
    s2, o2 = O.pack_packets(pk)
    got, _ = gpu_decode(ctx, s2, o2, 160, 96)
    bi = ctx.batch_info()
    assert bi.bad_frames == 1 and bi.first_bad_frame == 1
    want = reference_frames(s, o, 160, 96)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])   # neighbours unaffected


def test_decode_host_pipeline(ctx):
    ctx.set_scan_mode(capi.SCAN_AUTO)
    # 250 frames of 720x576 = three chunks through the pinned staging slots
    s, o = clip(720, 576, 128, 250, key_rate=29, lm=2, cm=2, noise_y=2)
    w, h = 720, 576
    fsz = w * h * 3 // 2
    init = np.full(fsz, 0x21, dtype=np.uint8)
    want = reference_frames(s, o, w, h, init)
    out = np.empty((250, fsz), dtype=np.uint8)
    carry = init.copy()
    st = ctx.decode_host(s, o, out, carry=carry)
    assert np.array_equal(out, want), first_diff(out, want, w, h)
    assert np.array_equal(carry, want[-1])
    assert (st.width, st.height, st.quality) == (720, 576, 128)
    # pinned in/out: same result through the direct-DMA path
    ps = torch.from_numpy(s).pin_memory()
    po = torch.empty((250, fsz), dtype=torch.uint8).pin_memory()
    ctx.decode_host(ps.numpy(), o, po.numpy(), carry=init.copy(),
                    flags=g.HOST_IN_PINNED | g.HOST_OUT_PINNED)
    assert np.array_equal(po.numpy(), want)
    # a truncated frame surfaces as an error code
    bad = s.copy()
    bad[int(o[5]):int(o[5]) + 4] = np.frombuffer(np.uint32(40).tobytes(), dtype=np.uint8)
    with pytest.raises(g.RTjpegError) as e:
        ctx.decode_host(bad, o, out)
    assert e.value.code == capi.E_OVERRUN


@pytest.fixture(scope="module")
def full_size_clip():
    return clip(720, 576, 128, 4096)


def test_full_size_config2_4096_frames(ctx, full_size_clip):
    """BASELINE.json configs[1] at full size under every flavour, checked frame by frame against the
    reference (threaded across the host's cores), plus the determinism property: decoding the same
    batch twice gives identical bytes."""
    import os
    w, h, F = 720, 576, 4096
    s, o = full_size_clip
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, w, h)
    D.decode(ctx, b)
    torch.cuda.synchronize()
    assert ctx.batch_info().bad_frames == 0
    first = b.out.clone()
    D.decode(ctx, b)
    torch.cuda.synchronize()
    assert torch.equal(first, b.out)
    threads = os.cpu_count() or 1
    for c0 in range(0, F, 512):
        # decode this chunk with the reference (each intra frame is its own segment)
        sub_o = o[c0:c0 + 513] if c0 + 512 < F else o[c0:]
        n = len(sub_o) - 1
        want = reference_frames_threaded(s, sub_o, np.arange(n + 1, dtype=np.int32), w, h, threads, zero_init=False)
        got = b.out[c0:c0 + n].cpu().numpy()
        assert np.array_equal(got, want), first_diff(got, want, w, h)


@pytest.mark.parametrize("w,h", [(720, 576), (1920, 1088)])
def test_frames_of_skip_markers_only(ctx, w, h):
    """A frame that is nothing but 0xFF bytes -- one block per byte, 8192 blocks in a scan segment, more than one
    emit round holds -- after a coded frame, at a quality without and one with a raw prefix."""
    nblk = (w // 16) * (h // 16) * 6
    for Q in (128, 255):
        s, o = clip(w, h, Q, 2, noise_y=6)
        sizes = O.packet_sizes(s, o)
        first = s[int(o[0]):int(o[0]) + int(sizes[0])]
        allskip = np.full(12 + nblk, 0xFF, dtype=np.uint8)
        allskip[:12] = first[:12]
        allskip[0:4] = np.frombuffer(np.uint32(12 + nblk).tobytes(), dtype=np.uint8)
        second = s[int(o[1]):int(o[1]) + int(sizes[1])]
        s2, o2 = O.pack_packets([first, allskip, allskip, second, allskip])
        init = np.full(w * h * 3 // 2, 0x30, dtype=np.uint8)
        want = reference_frames(s2, o2, w, h, init)
        got, _ = gpu_decode(ctx, s2, o2, w, h, carry=init)
        assert np.array_equal(got, want), first_diff(got, want, w, h)
        assert np.array_equal(want[1], want[0]) and ctx.batch_info().skipped_blocks == 3 * nblk
