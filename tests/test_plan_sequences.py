"""capi.plan_sequences (host only): several independent packet sequences packed into one batch for
rtjgpu_decode_device_seq, each planned with its own state."""
import numpy as np

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from streams import clip


def test_plan_sequences_matches_plan_per_sequence():
    seqs = [clip(64, 48, 128, 5, key_rate=2, lm=2, cm=2),
            clip(64, 48, 255, 1, seed=3),
            clip(64, 48, 32, 7, key_rate=3, lm=4, cm=4, dark=1, seed=5)]
    # a sequence that starts inside its buffer, off the 16-byte grid of the others
    s3, o3 = clip(64, 48, 200, 6, key_rate=2, lm=2, cm=2, seed=7)
    seqs.append((s3, o3[2:]))
    stream, offsets, desc, seq_first, states = g.plan_sequences(seqs)
    assert list(seq_first) == [0, 5, 6, 13, 17]
    assert len(offsets) == 18 and len(desc) == 17 and offsets[-1] == stream.size
    for i, (s, o) in enumerate(seqs):
        a, b = int(seq_first[i]), int(seq_first[i + 1])
        want, st = g.plan(s, o)
        shift = offsets[a] - o[0]
        assert np.array_equal(offsets[a:b], o[:-1] + shift)
        assert (offsets[a:b] % 16 == o[:-1] % 16).all()
        assert np.array_equal(desc[a:b]["offset"], want["offset"] + shift)
        for k in ("length", "table", "flags"):
            assert np.array_equal(desc[a:b][k], want[k]), k
        assert (states[i].width, states[i].height, states[i].table, states[i].quality) == (st.width, st.height, st.table, st.quality)
        for f in range(b - a):         # the packets themselves
            n = int(want["length"][f])
            assert np.array_equal(stream[int(desc[a + f]["offset"]):][:n], s[int(o[f]):][:n])


def test_plan_sequences_advances_given_states():
    s, o = clip(64, 48, 128, 8, key_rate=3, lm=2, cm=2)
    st = capi.State(0, 0, capi.TABLE_ZERO, 0)
    g.plan_sequences([(s, o[:4])], [st])
    _, _, desc, _, states = g.plan_sequences([(s, o[3:])], [st])
    assert states[0] is st
    want, _ = g.plan(s, o)
    assert np.array_equal(desc["table"], want["table"][3:])
    assert (st.width, st.height, st.quality) == (64, 48, 128)
