"""NuppelVideo container in front of the decoder (SURVEY.md section 8f-1): the reader follows
lib/demux_nuv.c, the decode of the rewrapped frames is pinned against lib/RTjpeg.c through the
reference's own RTjpeg_set_tables + RTjpeg_decompress."""
import numpy as np
import pytest

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from oracle import oracle as O
from nuv_writer import frame, write_nuv
from streams import clip, reference_frames


def _payloads(s, o):
    sizes = O.packet_sizes(s, o)
    return [s[int(o[f]) + 12:int(o[f]) + int(sizes[f])] for f in range(len(o) - 1)]


def _reference_frames_with_tables(raw, stream, offsets, w, h):
    """lib/RTjpeg.c decode of 'RTJ0' packets on an instance configured with RTjpeg_set_tables(raw)."""
    planes = np.zeros(w * h * 3 // 2, dtype=np.uint8)
    out = []
    for f in range(len(offsets) - 1):
        pkt = stream[int(offsets[f]):int(offsets[f + 1])]
        planes = (O.ref_decode_with_tables if O.have_ref() else O.decode_with_tables)(raw, pkt, w, h, planes)
        out.append(planes.copy())
    return np.stack(out)


def test_raw_tables_reproduce_the_quality_tables():
    for Q in (1, 32, 128, 171, 255):
        raw = g.raw_tables_for_quality(Q)
        scaled, lb8, cb8 = g.tables_from_raw(raw)
        want, wl, wc = g.tables_for_quality(Q)
        assert np.array_equal(scaled, want) and (lb8, cb8) == (wl, wc)


def test_reader_follows_demux_nuv():
    w, h, Q = 64, 48, 128
    s, o = clip(w, h, Q, 6, key_rate=2, lm=2, cm=2, noise_y=6)
    pay = _payloads(s, o)
    raw = g.raw_tables_for_quality(Q)
    vids = [pay[0], pay[1], ("L",), pay[2], ("N",), pay[3], ("0", bytes(w * h * 3 // 2)), pay[4], pay[5]]
    data = write_nuv(w, h, 25.0, raw, vids, keyframes=[1, 0, 0, 0, 1, 0, 1, 0, 0], audio_every=2, seek_every=4)
    assert g.nuv_probe(data) and not g.nuv_probe(data[4:])
    hd = g.nuv_open(data)
    assert (hd.width, hd.height, hd.interlaced, hd.is_mythtv) == (w, h, 0, 0)
    assert hd.fps == 25.0 and hd.video_packets == len(vids) and hd.audio_packets == 4
    assert hd.has_tables and np.array_equal(np.array(hd.tables[:]), raw)
    assert hd.data_start == 72 + 12 + 512
    pk = g.nuv_packets(data, hd)
    assert [p[0] for p in pk].count("V") == len(vids) and [p[0] for p in pk].count("A") == 4
    assert [p[0] for p in pk].count("S") == 3 and all(p[4] == 0 for p in pk if p[0] == "S")
    assert [p[1] for p in pk if p[0] == "V"] == ["1", "1", "L", "1", "N", "1", "0", "1", "1"]
    stream, offsets, tc, unsupported = g.nuv_extract_rtj0(data, hd)
    assert unsupported == 2 and len(offsets) - 1 == 7           # 'N' and '0' are left to libavcodec
    assert list(tc) == [0, 40, 80, 120, 200, 280, 320]
    # packets: RTjpeg_frameheader + the block stream; the repeated frame is a frame of skip markers
    nblk = (w // 16) * (h // 16) * 6
    for i, want in enumerate([pay[0], pay[1], np.full(nblk, 0xFF, np.uint8), pay[2], pay[3], pay[4], pay[5]]):
        p = stream[int(offsets[i]):int(offsets[i + 1])]
        assert int.from_bytes(p[0:4].tobytes(), "little") == 12 + len(want) and p[4] == 12 and p[5] == 0
        assert int.from_bytes(p[6:8].tobytes(), "little") == w and int.from_bytes(p[8:10].tobytes(), "little") == h
        assert p[10] == 0 and np.array_equal(p[12:12 + len(want)], want)
    # what lib/RTjpeg.c makes of them (set_tables path) is what it makes of the original stream
    direct = reference_frames(s, o, w, h)
    got = _reference_frames_with_tables(raw, stream, offsets, w, h)
    assert np.array_equal(got[[0, 1, 3, 4, 5, 6]], direct)
    assert np.array_equal(got[2], got[1])                      # 'L': the picture repeats
    # the restatement agrees
    st = capi.State(w, h, capi.TABLE_CUSTOM, 0)
    desc, st2 = g.plan(stream, offsets, st)
    assert (desc["table"] == capi.TABLE_CUSTOM).all() and st2.quality == 0


def test_reader_rejects_damage():
    w, h = 32, 32
    raw = g.raw_tables_for_quality(90)
    data = write_nuv(w, h, 30.0, raw, [bytes([0x80, 126] * 24)])
    with pytest.raises(g.RTjpegError):
        g.nuv_open(data[:60])                                  # file header cut short
    with pytest.raises(g.RTjpegError):
        g.nuv_open(data[:72 + 12 + 100])                       # tables cut short
    hd = g.nuv_open(data)
    cut = data[:len(data) - 10]                                # last frame cut short: it is not reported
    assert [p[0] for p in g.nuv_packets(cut, hd)] == []
    odd = write_nuv(40, 32, 30.0, raw, [bytes(4)])
    with pytest.raises(g.RTjpegError) as e:
        g.nuv_extract_rtj0(odd, g.nuv_open(odd))               # width not a multiple of 16
    assert e.value.code == capi.E_SIZE
    # MythTV files: codec data ends with the 'X' packet
    myth = bytearray(data)
    myth[0:12] = b"MythTVVideo\0"
    ext = frame("X", "\0", 0, 0, bytes(512))
    myth = np.frombuffer(bytes(myth[:72 + 12 + 512]) + ext + bytes(myth[72 + 12 + 512:]), dtype=np.uint8)
    hm = g.nuv_open(myth)
    assert hm.is_mythtv and hm.data_start == 72 + 12 + 512 + 12 + 512


@pytest.mark.gpu
def test_config0_nuv_320x240_keyframe_only_on_gpu():
    """BASELINE.json configs[0], literally: a .nuv RTjpeg 320x240 YUV420 keyframe-only clip."""
    import torch
    from gmerlin_avdecoder_b200 import device as D
    w, h, Q, F = 320, 240, 128, 64
    s, o = clip(w, h, Q, F)
    raw = g.raw_tables_for_quality(Q)
    data = write_nuv(w, h, 25.0, raw, _payloads(s, o), audio_every=5, seek_every=16)
    hd = g.nuv_open(data)
    stream, offsets, tc, unsupported = g.nuv_extract_rtj0(data, hd)
    assert unsupported == 0 and len(offsets) - 1 == F
    want = reference_frames(s, o, w, h)                        # the reference on the original 'RTJ0' stream
    with g.BatchContext(0) as ctx:
        ctx.set_custom_tables(np.array(hd.tables[:], dtype=np.uint32))
        desc, _ = g.plan(stream, offsets, capi.State(w, h, capi.TABLE_CUSTOM, 0))
        b = D.upload(stream, desc, w, h, device=0)
        D.decode(ctx, b)
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
        assert np.array_equal(b.out.cpu().numpy(), want)
        # the host entry point with the same state
        out = np.empty((F, w * h * 3 // 2), dtype=np.uint8)
        ctx.decode_host(stream, offsets, out, state=capi.State(w, h, capi.TABLE_CUSTOM, 0))
        assert np.array_equal(out, want)
