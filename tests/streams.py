"""Stream fixtures shared by the test modules (test infrastructure)."""
import hashlib
import os

import numpy as np

from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def reference_frames(stream, offsets, w, h, init=None):
    """Expected output: the unmodified reference when its build is present, else the restatement
    (which test_oracle.py pins to the reference through the golden fixtures)."""
    if O.have_ref():
        return O.ref_decode_seq(stream, offsets, w, h, init=init)
    return O.decode_stream(stream, offsets, w, h, init=init)


def reference_frames_threaded(stream, offsets, segments, w, h, threads, zero_init=True, raw_tables=None):
    """reference_frames for independent frame ranges (see oracle.decode_threaded), on `threads` host cores."""
    if O.have_ref():
        return O.ref_decode_threaded(stream, offsets, segments, w, h, threads, zero_init=zero_init, keep=True,
                                     raw_tables=raw_tables)[1]
    return O.decode_threaded(stream, offsets, segments, w, h, threads, zero_init=zero_init, raw_tables=raw_tables)


def clip(w, h, Q, F, **kw):
    c = O.make_clip(w, h, Q, **kw)
    return O.encode_clip(c, F)


def interleave(streams):
    """Round-robin interleave of several (stream, offsets) packet sequences of equal length."""
    pk = []
    n = len(streams[0][1]) - 1
    for f in range(n):
        for s, o in streams:
            size = int(O.packet_sizes(s, o)[f])
            pk.append(s[int(o[f]):int(o[f]) + size])
    return O.pack_packets(pk)


def reference_frames_fmt(stream, offsets, w, h, fmt, init=None):
    if O.have_ref():
        return O.ref_decode_seq_fmt(stream, offsets, w, h, fmt, init=init)
    return O.decode_stream_fmt(stream, offsets, w, h, fmt, init=init)
