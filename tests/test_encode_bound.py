"""rtjgpu_encode_bound (host arithmetic): a capacity for rtjgpu_encode_device[_seq] that the packets never exceed."""
import numpy as np
import pytest

import gmerlin_avdecoder_b200 as g
from oracle import oracle as O


@pytest.mark.parametrize("fmt,w,h", [(0, 64, 48), (1, 64, 48), (0, 720, 576), (1, 160, 32)])
def test_bound_holds_the_worst_packets(fmt, w, h):
    """Full-range random pictures at quality 255 (every block coded, raw prefix): the largest packets the encoder makes,
    laid out 4-byte aligned as the device lays them out -- within the bound, and the bound within the capacity the
    encoder tests give (12 + 2 * 64 bytes per 8x8 luma block + 16 per picture)."""
    F = 3
    rng = np.random.default_rng(fmt * 7 + w)
    fr = rng.integers(0, 256, (F, O.frame_bytes(fmt, w, h))).astype(np.uint8)
    s, o = O.encode_frames_oracle(fr, w, h, fmt, 255, 0, 0, 0, align=4)
    used = (int(o[-1]) + 3) // 4 * 4
    bound = g.encode_bound(fmt, w, h, F)
    assert used <= bound <= F * (12 + (w // 8) * (h // 8) * 2 * 64 + 16)
    nblk = (w // 16) * (h // 16) * 6 if fmt == 0 else (w // 16) * (h // 8) * 4
    assert bound == F * (12 + 64 * nblk)
    assert used > bound * 3 // 4                 # random pictures come close to it


def test_bound_refuses_what_the_encoder_refuses():
    assert g.encode_bound(2, 64, 48, 1) == 0      # grey: no encoder
    assert g.encode_bound(0, 60, 48, 1) == 0      # not a multiple of 16
    assert g.encode_bound(0, 64, 48, -1) == 0
    assert g.encode_bound(0, 64, 48, 0) == 0
