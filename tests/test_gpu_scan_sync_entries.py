"""K1's entry loop (csrc/rtj_scan_sync.cu, sy_entry and the emit stage): the entry table the self-synchronising walk
makes (SYNC, both instantiations), byte for byte against the chunk-parallel kernels' (CHUNK: an independent
implementation of the same entries), at the bench point's geometry and quality, with a raw prefix (Q = 255), and on
frames cut short so that their last blocks start in the payload's last bytes or run past its end.  320 frames: the
batch size from which the walk runs 128 lanes a frame, as at the bench point."""
import numpy as np
import pytest

from gmerlin_avdecoder_b200 import capi
from oracle import oracle as O
from streams import clip
from test_gpu_scan_sync import _ctx, _entries

pytestmark = pytest.mark.gpu

W, H, F = 720, 576, 320


def _same_entries(s, o, w, h):
    with _ctx(capi.SCAN_SYNC) as a, _ctx(capi.SCAN_CHUNK) as k:
        e1, i1 = _entries(a, s, o, w, h)
        e2, i2 = _entries(k, s, o, w, h)
    assert i1 == i2
    bad = np.argwhere(e1 != e2)
    assert bad.size == 0, "frame %d block %d: %#010x, chunk kernel %#010x" % (
        bad[0][0], bad[0][1], e1[tuple(bad[0])], e2[tuple(bad[0])])
    return e1, i1


@pytest.mark.parametrize("Q", [128, 255])
def test_bench_point_entries(Q):
    """720x576 intra at the bench quality, and at Q = 255 (raw prefix 9: the walk's second instantiation)."""
    s, o = clip(W, H, Q, F)
    e, info = _same_entries(s, o, W, H)
    assert info[2] == 0                                                   # no bad frames
    inline = (e & 0x80000000) != 0
    assert inline.any() and (~inline).any()                               # both kinds of entry are made


@pytest.mark.parametrize("Q", [128, 255])
def test_frames_cut_in_their_last_bytes(Q):
    """Every frame cut by 1 .. 40 bytes at its end: last blocks that start in the final three bytes (the tail path of the
    emit stage), blocks cut short mid-way, and frames cut exactly behind a block."""
    s, o = clip(W, H, Q, F)
    sizes = O.packet_sizes(s, o)
    pk = []
    for f in range(F):
        keep = int(sizes[f]) - 1 - f % 40
        p = s[int(o[f]):int(o[f]) + keep].copy()
        p[0:4] = np.frombuffer(np.uint32(p.size).tobytes(), dtype=np.uint8)
        pk.append(p)
    s2, o2 = O.pack_packets(pk, align=4)                                  # every misalignment of the payload
    _, info = _same_entries(s2, o2, W, H)
    assert info[2] >= 1
