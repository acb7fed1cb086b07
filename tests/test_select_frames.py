"""capi.select_frames (host only): per-sequence frame indices into the sorted batch indices that
rtjgpu_decode_device_select takes, and what it refuses."""
import numpy as np
import pytest

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi


def test_local_indices_become_sorted_batch_indices():
    seq_first = [0, 5, 6, 13, 17]
    sel = g.select_frames(seq_first, [[4, 0, 2], [0], np.array([6, 1]), []])
    assert sel.dtype == np.int64
    assert list(sel) == [0, 2, 4, 5, 7, 12]
    # output slot k of the call holds batch frame sel[k]: map each back to (sequence, local index)
    seq = np.searchsorted(seq_first, sel, side="right") - 1
    assert list(zip(seq.tolist(), (sel - np.asarray(seq_first)[seq]).tolist())) == [(0, 0), (0, 2), (0, 4), (1, 0), (2, 1), (2, 6)]


def test_every_kth_and_last_frames():
    seq_first = np.array([0, 30, 60, 75])
    every4 = capi.select_frames(seq_first, [np.arange(0, n, 4) for n in np.diff(seq_first)])
    assert list(every4[:8]) == [0, 4, 8, 12, 16, 20, 24, 28]
    assert (np.diff(every4) > 0).all()
    last = capi.select_frames(seq_first, [[n - 1] for n in np.diff(seq_first)])
    assert list(last) == [29, 59, 74]
    every = capi.select_frames(seq_first, [np.arange(n) for n in np.diff(seq_first)])
    assert list(every) == list(range(75))


def test_nothing_selected():
    sel = capi.select_frames([0, 3, 5], [[], []])
    assert sel.size == 0 and sel.dtype == np.int64


@pytest.mark.parametrize("picks", [
    [[3], [0]],          # past the end of sequence 0 (3 frames)
    [[0], [2]],          # past the end of sequence 1 (2 frames)
    [[-1], []],          # negative
    [[1, 1], []],        # named twice
    [[2, 0, 2], [1]],    # named twice, out of order
    [[0]],               # one index array for two sequences
])
def test_rejects(picks):
    with pytest.raises(ValueError):
        capi.select_frames([0, 3, 5], picks)
