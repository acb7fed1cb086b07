"""ctypes front-end to the oracle -- TEST INFRASTRUCTURE ONLY.

Two libraries live behind this module:

* ``oracle/liboracle.so``      -- the plain-C restatement (oracle/rtjpeg_oracle.c) and what drives it:
  the seeded synthetic clips, their streams and threaded decode (oracle/rtjo_driver.c);
* ``oracle/_ref/librtjref.so`` -- the UNMODIFIED reference (``lib/RTjpeg.c`` compiled
  from /root/reference by ``oracle/Makefile``) plus ``oracle/ref_driver.c``.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import this module.  The shipped
package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "librtjref.so")
REFERENCE_ROOT = "/root/reference"

_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_i32p = C.POINTER(C.c_int32)


def build(want_ref: bool = True) -> None:
    """Compile the restatement, and the reference when its sources are present."""
    subprocess.check_call(["make", "-s", "-C", HERE, "all"])
    if want_ref and os.path.isdir(REFERENCE_ROOT):
        subprocess.check_call(["make", "-s", "-C", HERE, "ref"])


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def _np_u8(a) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a


def _ptr(a: np.ndarray, typ=_u8p):
    return a.ctypes.data_as(typ)


# --------------------------------------------------------------------------
# restatement
# --------------------------------------------------------------------------

class _Tables(C.Structure):
    _fields_ = [("liqt", C.c_int32 * 64), ("ciqt", C.c_int32 * 64), ("lb8", C.c_int), ("cb8", C.c_int)]


class _Decoder(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("Q", C.c_int), ("t", _Tables)]


_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            build(want_ref=False)
        L = C.CDLL(ORACLE_SO)
        L.rtjo_tables_from_quality.argtypes = [C.c_int, C.POINTER(_Tables)]
        L.rtjo_tables_from_raw.argtypes = [_u32p, C.POINTER(_Tables)]
        L.rtjo_decoder_reset.argtypes = [C.POINTER(_Decoder)]
        L.rtjo_decode_packet.argtypes = [C.POINTER(_Decoder), _u8p, C.c_size_t, _u8p, _u8p, _u8p]
        L.rtjo_decode_packet.restype = C.c_long
        L.rtjo_decode_packet_fmt.argtypes = [C.POINTER(_Decoder), C.c_int, _u8p, C.c_size_t, _u8p, _u8p, _u8p]
        L.rtjo_decode_packet_fmt.restype = C.c_long
        L.rtjo_walk_payload.argtypes = [_u8p, C.c_size_t, C.c_int, C.c_int, C.c_int, _u32p, _u8p]
        L.rtjo_walk_payload.restype = C.c_long
        L.rtjo_unpack_block.argtypes = [_u8p, C.c_int, _i32p, C.POINTER(C.c_int16)]
        L.rtjo_unpack_block.restype = C.c_int
        L.rtjo_idct_block.argtypes = [C.POINTER(C.c_int16), _u8p, C.c_int]
        L.rtjo_synth_frame.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_int,
                                       _u8p, _u8p, _u8p]
        L.rtjo_packet_bound.argtypes = [C.c_int, C.c_int]
        L.rtjo_packet_bound.restype = C.c_size_t
        L.rtjo_encode_clip.argtypes = [C.POINTER(Clip), C.c_int, C.c_int, _u8p, C.c_size_t, _u64p, C.c_int]
        L.rtjo_encode_clip.restype = C.c_size_t
        L.rtjo_decode_threaded.argtypes = [_u8p, _u64p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int,
                                           C.c_int, _u8p, _u32p]
        L.rtjo_decode_threaded.restype = C.c_int
        _oracle = L
    return _oracle


@dataclass
class Tables:
    liqt: np.ndarray
    ciqt: np.ndarray
    lb8: int
    cb8: int


def tables_from_quality(Q: int) -> Tables:
    t = _Tables()
    oracle_lib().rtjo_tables_from_quality(Q, C.byref(t))
    return Tables(np.array(t.liqt, dtype=np.int32), np.array(t.ciqt, dtype=np.int32), t.lb8, t.cb8)


def tables_from_raw(raw) -> Tables:
    raw = np.ascontiguousarray(raw, dtype=np.uint32)
    assert raw.size == 128
    t = _Tables()
    oracle_lib().rtjo_tables_from_raw(_ptr(raw, _u32p), C.byref(t))
    return Tables(np.array(t.liqt, dtype=np.int32), np.array(t.ciqt, dtype=np.int32), t.lb8, t.cb8)


class OracleDecoder:
    """Sequential decoder with persistent planes, the shape of decode_rtjpeg
    (reference lib/video_rtjpeg.c:62-90) without gavl."""

    def __init__(self):
        self._d = _Decoder()
        oracle_lib().rtjo_decoder_reset(C.byref(self._d))
        self.planes = None

    def decode(self, pkt, planes: np.ndarray | None = None) -> np.ndarray:
        pkt = _np_u8(pkt)
        w = int(pkt[6]) | int(pkt[7]) << 8
        h = int(pkt[8]) | int(pkt[9]) << 8
        fsz = w * h * 3 // 2
        if planes is not None:
            self.planes = planes
        if self.planes is None or self.planes.size != fsz:
            self.planes = np.zeros(fsz, dtype=np.uint8)
        p = self.planes
        n = oracle_lib().rtjo_decode_packet(
            C.byref(self._d), _ptr(pkt), pkt.size,
            _ptr(p), C.cast(p.ctypes.data + w * h, _u8p), C.cast(p.ctypes.data + w * h * 5 // 4, _u8p))
        if n < 0:
            raise ValueError("packet overrun")
        self.consumed = int(n)
        return p


def decode_stream(stream, offsets, w: int, h: int, init: np.ndarray | None = None,
                  keep_all: bool = True) -> np.ndarray:
    """Restatement decode of a whole stream; returns [F, w*h*3/2] (or the last frame)."""
    stream = _np_u8(stream)
    F = len(offsets) - 1
    fsz = w * h * 3 // 2
    dec = OracleDecoder()
    dec.planes = np.zeros(fsz, dtype=np.uint8) if init is None else np.array(init, dtype=np.uint8).copy()
    out = np.empty((F, fsz), dtype=np.uint8) if keep_all else None
    for f in range(F):
        dec.decode(stream[int(offsets[f]):int(offsets[f + 1])])
        if keep_all:
            out[f] = dec.planes
    return out if keep_all else dec.planes.copy()


def walk_payload(payload, nmb: int, lb8: int, cb8: int):
    payload = _np_u8(payload)
    offs = np.empty(nmb * 6, dtype=np.uint32)
    eob = np.empty(nmb * 6, dtype=np.uint8)
    n = oracle_lib().rtjo_walk_payload(_ptr(payload), payload.size, nmb, lb8, cb8, _ptr(offs, _u32p), _ptr(eob))
    return int(n), offs, eob


def idct_block(blk: np.ndarray) -> np.ndarray:
    blk = np.ascontiguousarray(blk, dtype=np.int16).reshape(64)
    out = np.zeros(64, dtype=np.uint8)
    oracle_lib().rtjo_idct_block(blk.ctypes.data_as(C.POINTER(C.c_int16)), _ptr(out), 8)
    return out.reshape(8, 8)


# --------------------------------------------------------------------------
# unmodified reference + driver
# --------------------------------------------------------------------------

class Clip(C.Structure):
    """Mirror of rtjo_clip (oracle/rtjo_driver.c) and refdrv_clip (oracle/ref_driver.c)."""
    _fields_ = [("w", C.c_int), ("h", C.c_int), ("Q", C.c_int), ("key_rate", C.c_int),
                ("lm", C.c_int), ("cm", C.c_int), ("noise_y", C.c_int), ("noise_c", C.c_int),
                ("dark", C.c_int), ("seed", C.c_uint32)]


def make_clip(w, h, Q, key_rate=-1, lm=0, cm=0, noise_y=2, noise_c=0, dark=0, seed=1) -> Clip:
    return Clip(w, h, Q, key_rate, lm, cm, noise_y, noise_c, dark, seed)


_ref = None


def ref_lib():
    global _ref
    if _ref is None:
        if not have_ref():
            if os.path.isdir(REFERENCE_ROOT):
                build(want_ref=True)
            else:
                raise FileNotFoundError(
                    f"{REF_SO} missing and {REFERENCE_ROOT} absent: build it where the reference is mounted")
        L = C.CDLL(REF_SO)
        L.refdrv_packet_bound.argtypes = [C.c_int, C.c_int]
        L.refdrv_packet_bound.restype = C.c_size_t
        L.refdrv_encode_frames.argtypes = [C.POINTER(Clip), _u8p, C.c_int, _u8p, C.c_size_t, _u64p, C.c_int]
        L.refdrv_encode_frames.restype = C.c_size_t
        L.refdrv_decode_seq.argtypes = [_u8p, _u64p, C.c_int, C.c_int, C.c_int, _u8p, _u8p, _u8p]
        L.refdrv_encode_frames_fmt.argtypes = [C.POINTER(Clip), C.c_int, _u8p, C.c_int, _u8p, C.c_size_t, _u64p, C.c_int]
        L.refdrv_encode_frames_fmt.restype = C.c_size_t
        L.refdrv_decode_seq_fmt.argtypes = [_u8p, _u64p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, _u8p, _u8p]
        L.refdrv_decode_threaded.argtypes = [_u8p, _u64p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, _u8p]
        L.refdrv_decode_threaded.restype = C.c_double
        L.refdrv_decode_threaded_tables.argtypes = [_u8p, _u64p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int,
                                                    C.c_int, C.c_int, _u8p, _u32p]
        L.refdrv_decode_threaded_tables.restype = C.c_double
        L.refdrv_tables_for_quality.argtypes = [C.c_int, _u32p]
        L.refdrv_decode_with_tables.argtypes = [_u32p, _u8p, C.c_int, C.c_int, _u8p]
        _ref = L
    return _ref


def synth_frame(w, h, t, seed=1, noise_y=2, noise_c=0, dark=0) -> np.ndarray:
    out = np.empty(w * h * 3 // 2, dtype=np.uint8)
    oracle_lib().rtjo_synth_frame(w, h, t, seed, noise_y, noise_c, dark, _ptr(out),
                                  C.cast(out.ctypes.data + w * h, _u8p),
                                  C.cast(out.ctypes.data + w * h * 5 // 4, _u8p))
    return out


def encode_clip(clip: Clip, F: int, threads: int = 0, align: int = 16):
    """Synthesize and encode F frames with the restated encoder (oracle/rtjo_driver.c), which
    tests/golden/ pins to the reference's own packets.

    Returns (stream uint8[...], offsets uint64[F+1]); packet f is
    stream[offsets[f]:offsets[f]+framesize]; every start is `align`-aligned."""
    L = oracle_lib()
    threads = threads or (os.cpu_count() or 1)
    cap = int(L.rtjo_packet_bound(clip.w, clip.h) + align) * F + 64
    # worst-case capacity can be large (64 B/block); fall back to a generous typical bound first
    typical = max(1 << 20, (clip.w * clip.h * 3 // 2 + 4096) * F)
    for c in (min(cap, typical), cap):
        buf = np.zeros(c, dtype=np.uint8)
        offs = np.empty(F + 1, dtype=np.uint64)
        used = L.rtjo_encode_clip(C.byref(clip), F, threads, _ptr(buf), c, _ptr(offs, _u64p), align)
        if used or F == 0:
            return buf[:int(used)].copy(), offs
    raise RuntimeError("encode buffer too small")


def encode_frames(clip: Clip, frames: np.ndarray, align: int = 16):
    """Encode caller-supplied YUV420 frames [F, w*h*3/2] sequentially with one encoder."""
    L = ref_lib()
    frames = _np_u8(frames)
    F = frames.shape[0]
    cap = int(L.refdrv_packet_bound(clip.w, clip.h) + align) * max(F, 1) + 64
    buf = np.zeros(cap, dtype=np.uint8)
    offs = np.empty(F + 1, dtype=np.uint64)
    used = L.refdrv_encode_frames(C.byref(clip), _ptr(frames), F, _ptr(buf), cap, _ptr(offs, _u64p), align)
    if not used and F:
        raise RuntimeError("encode buffer too small")
    return buf[:int(used)].copy(), offs


def ref_encode_clip(clip: Clip, F: int, align: int = 16):
    """The clip of encode_clip coded by the reference's own RTjpeg_compress, one encoder in sequence: what the streams of
    tests/golden/ are made with, so that they pin the restated encoder to the reference."""
    frames = np.stack([synth_frame(clip.w, clip.h, t, clip.seed, clip.noise_y, clip.noise_c, clip.dark) for t in range(F)])
    return encode_frames(clip, frames, align)


def ref_encode_clip_fmt(w: int, h: int, Q: int, F: int, fmt: int, key_rate: int = -1, lm: int = 0, cm: int = 0, **kw):
    """encode_clip_fmt with the reference doing both the round trip of the source and the coding in format fmt."""
    s, o = ref_encode_clip(make_clip(w, h, 255, **kw), F)
    frames = frames_in_format(ref_decode_seq(s, o, w, h), w, h, fmt)
    return encode_frames_fmt(make_clip(w, h, Q, key_rate, lm, cm), fmt, frames)


def ref_decode_seq(stream, offsets, w, h, init=None, keep_all=True):
    """Reference decode, one decoder instance, persistent planes."""
    stream = _np_u8(stream)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    F = len(offsets) - 1
    fsz = w * h * 3 // 2
    frames = np.empty((F, fsz), dtype=np.uint8) if keep_all else None
    last = np.empty(fsz, dtype=np.uint8)
    initp = None if init is None else _ptr(_np_u8(init))
    # the reference reads without bounds checks: give it slack past the end
    padded = np.concatenate([stream, np.full(256, 0x7F, dtype=np.uint8)])
    ref_lib().refdrv_decode_seq(_ptr(padded), _ptr(offsets, _u64p), F, w, h, initp,
                                None if frames is None else _ptr(frames), _ptr(last))
    return frames if keep_all else last


def ref_decode_threaded(stream, offsets, segments, w, h, threads, zero_init=True, keep=False, raw_tables=None):
    """Threaded reference decode; returns (seconds, frames or None).  raw_tables: 128 raw entries every worker loads
    with RTjpeg_set_tables first (the packets then carry quality 0)."""
    stream = _np_u8(stream)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    seg = np.ascontiguousarray(segments, dtype=np.int32)
    F = int(seg[-1])
    fsz = w * h * 3 // 2
    frames = np.empty((F, fsz), dtype=np.uint8) if keep else None
    raw = None if raw_tables is None else np.ascontiguousarray(raw_tables, dtype=np.uint32)
    secs = ref_lib().refdrv_decode_threaded_tables(_ptr(stream), _ptr(offsets, _u64p),
                                                   seg.ctypes.data_as(C.POINTER(C.c_int)), len(seg) - 1,
                                                   w, h, threads, 1 if zero_init else 0,
                                                   None if frames is None else _ptr(frames),
                                                   None if raw is None else _ptr(raw, _u32p))
    return float(secs), frames


def ref_tables_for_quality(Q: int) -> np.ndarray:
    out = np.empty(128, dtype=np.uint32)
    ref_lib().refdrv_tables_for_quality(Q, _ptr(out, _u32p))
    return out


def ref_decode_with_tables(raw, pkt, w, h, planes: np.ndarray) -> np.ndarray:
    raw = np.ascontiguousarray(raw, dtype=np.uint32)
    pkt = np.concatenate([_np_u8(pkt), np.full(256, 0x7F, dtype=np.uint8)])
    planes = np.array(planes, dtype=np.uint8).copy()
    ref_lib().refdrv_decode_with_tables(_ptr(raw, _u32p), _ptr(pkt), w, h, _ptr(planes))
    return planes


# --------------------------------------------------------------------------
# stream helpers shared by tests and bench (pure numpy, no codec arithmetic)
# --------------------------------------------------------------------------

def packet_sizes(stream: np.ndarray, offsets: np.ndarray) -> np.ndarray:
    """framesize field (u32 LE at +0) of every packet."""
    o = np.asarray(offsets[:-1], dtype=np.int64)
    b = stream
    return (b[o].astype(np.uint32) | b[o + 1].astype(np.uint32) << 8 |
            b[o + 2].astype(np.uint32) << 16 | b[o + 3].astype(np.uint32) << 24)


def random_wellformed_packet(rng: np.random.Generator, w: int, h: int, Q: int, skip_prob=0.2,
                             dense_prob=0.3, extreme=True) -> np.ndarray:
    """A syntactically valid packet with arbitrary token values (SURVEY.md appendix A.5):
    exercises the int16 wrap of the dequantiser, every raw-prefix class and long blocks.
    Built from the grammar only -- no codec arithmetic involved."""
    t = tables_from_quality(Q)
    nmb = (w // 16) * (h // 16)
    out = bytearray()
    out += bytes(12)
    for mb in range(nmb):
        for k in range(6):
            bt8 = t.lb8 if k < 4 else t.cb8
            if rng.random() < skip_prob:
                out.append(0xFF)
                continue
            out.append(int(rng.integers(0, 255)))          # DC 0..254
            for _ in range(bt8):
                out.append(int(rng.integers(-128, 128)) & 0xFF)
            pos = 1 + bt8
            dense = rng.random() < dense_prob
            while pos < 64:
                if not dense and rng.random() < 0.5:
                    run = int(rng.integers(1, 64 - pos + 1))   # never overshoots 64
                    out.append(63 + run)
                    pos += run
                else:
                    lo, hi = (-128, 64) if extreme else (-8, 9)
                    out.append(int(rng.integers(lo, hi)) & 0xFF)
                    pos += 1
    n = len(out)
    hdr = np.zeros(12, dtype=np.uint8)
    hdr[0:4] = np.frombuffer(np.uint32(n).tobytes(), dtype=np.uint8)
    hdr[4] = 12
    hdr[6:8] = np.frombuffer(np.uint16(w).tobytes(), dtype=np.uint8)
    hdr[8:10] = np.frombuffer(np.uint16(h).tobytes(), dtype=np.uint8)
    hdr[10] = Q
    pkt = np.frombuffer(bytes(out), dtype=np.uint8).copy()
    pkt[:12] = hdr
    return pkt


def pack_packets(pkts, align: int = 16):
    """Concatenate packets with aligned starts -> (stream, offsets[F+1])."""
    offs = np.zeros(len(pkts) + 1, dtype=np.uint64)
    at = 0
    for i, p in enumerate(pkts):
        at = (at + align - 1) // align * align
        offs[i] = at
        at += len(p)
    offs[len(pkts)] = at
    buf = np.zeros(at, dtype=np.uint8)
    for i, p in enumerate(pkts):
        buf[int(offs[i]):int(offs[i]) + len(p)] = p
    return buf, offs


# ---- the other two formats of RTjpeg_decompress: 1 = YUV422, 2 = 8-bit grey ------------------

def frame_bytes(fmt: int, w: int, h: int) -> int:
    return w * h * 3 // 2 if fmt == 0 else w * h * 2 if fmt == 1 else w * h


def frames_in_format(frames420: np.ndarray, w: int, h: int, fmt: int) -> np.ndarray:
    """Synthetic YUV420 frames [F, w*h*3/2] -> tight planes of format fmt (422: chroma rows doubled
    and roughened a little so that the two rows of a pair differ; grey: luma only)."""
    frames420 = _np_u8(frames420)
    F = frames420.shape[0]
    ysz = w * h
    if fmt == 0:
        return frames420.copy()
    if fmt == 2:
        return np.ascontiguousarray(frames420[:, :ysz])
    out = np.empty((F, 2 * ysz), dtype=np.uint8)
    out[:, :ysz] = frames420[:, :ysz]
    for k, lo in ((0, ysz), (1, ysz + ysz // 4)):
        c = frames420[:, lo:lo + ysz // 4].reshape(F, h // 2, w // 2).astype(np.int16)
        up = np.repeat(c, 2, axis=1)
        up[:, 1::2, :] += ((np.arange(w // 2) % 5) - 2)[None, None, :]
        out[:, ysz + k * (ysz // 2):ysz + (k + 1) * (ysz // 2)] = np.clip(up, 16, 235).astype(np.uint8).reshape(F, -1)
    return out


def encode_frames_fmt(clip: Clip, fmt: int, frames: np.ndarray, align: int = 16):
    """Reference RTjpeg_compress in format fmt over caller-supplied tight planes [F, frame_bytes]."""
    L = ref_lib()
    frames = _np_u8(frames)
    F = frames.shape[0]
    if fmt == 2:
        # RTjpeg_compress8 / RTjpeg_mcompress8 read every block with a row stride of 8 * width (they hand RTjpeg_dctY the
        # width where it expects width / 8, RTjpeg.c:2627, :3005): up to 56 rows behind the plane.  Give them zeros to read.
        padded = np.zeros(frames.size + 64 * clip.w, dtype=np.uint8)
        padded[:frames.size] = frames.reshape(-1)
        frames = padded[:F * frames.shape[1]].reshape(F, -1)
    cap = (12 + (clip.w // 8) * (clip.h // 8) * 2 * 64 + 64 + align) * max(F, 1) + 64
    buf = np.zeros(cap, dtype=np.uint8)
    offs = np.empty(F + 1, dtype=np.uint64)
    used = L.refdrv_encode_frames_fmt(C.byref(clip), fmt, _ptr(frames), F, _ptr(buf), cap, _ptr(offs, _u64p), align)
    if not used and F:
        raise RuntimeError("encode buffer too small")
    return buf[:int(used)].copy(), offs


def ref_decode_seq_fmt(stream, offsets, w, h, fmt, init=None):
    stream = _np_u8(stream)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    F = len(offsets) - 1
    fsz = frame_bytes(fmt, w, h)
    frames = np.empty((F, fsz), dtype=np.uint8)
    last = np.empty(fsz, dtype=np.uint8)
    initp = None if init is None else _ptr(_np_u8(init))
    padded = np.concatenate([stream, np.full(256, 0x7F, dtype=np.uint8)])
    ref_lib().refdrv_decode_seq_fmt(_ptr(padded), _ptr(offsets, _u64p), F, w, h, fmt, initp, _ptr(frames), _ptr(last))
    return frames


def decode_stream_fmt(stream, offsets, w: int, h: int, fmt: int, init: np.ndarray | None = None) -> np.ndarray:
    """Restatement decode of a whole stream in format fmt; returns [F, frame_bytes]."""
    stream = _np_u8(stream)
    L = oracle_lib()
    F = len(offsets) - 1
    fsz = frame_bytes(fmt, w, h)
    ysz = w * h
    csz = ysz // 4 if fmt == 0 else ysz // 2 if fmt == 1 else 0
    planes = np.zeros(fsz, dtype=np.uint8) if init is None else np.array(init, dtype=np.uint8).copy()
    d = _Decoder()
    L.rtjo_decoder_reset(C.byref(d))
    out = np.empty((F, fsz), dtype=np.uint8)
    for f in range(F):
        pkt = np.ascontiguousarray(stream[int(offsets[f]):int(offsets[f + 1])])
        base = planes.ctypes.data
        y = C.cast(base, _u8p)
        u = C.cast(base + ysz, _u8p)
        v = C.cast(base + ysz + csz, _u8p)
        n = L.rtjo_decode_packet_fmt(C.byref(d), fmt, _ptr(pkt), pkt.size, y, u, v)
        if n < 0:
            raise ValueError("truncated packet")
        out[f] = planes
    return out


def encode_clip_fmt(w: int, h: int, Q: int, F: int, fmt: int, key_rate: int = -1, lm: int = 0, cm: int = 0, **kw):
    """A synthetic clip in format fmt: the seeded YUV420 source of rtjo_driver.c (taken through one
    high-quality round trip), reshaped by frames_in_format and coded in that format by the restated
    RTjpeg_compress.  Returns (stream, offsets)."""
    src = make_clip(w, h, 255, **kw)
    s, o = encode_clip(src, F, threads=1)
    frames = frames_in_format(decode_stream(s, o, w, h), w, h, fmt)
    if fmt == 2:
        return encode_frames_grey(frames, w, h, Q, key_rate, lm)
    return encode_frames_oracle(frames, w, h, fmt, Q, key_rate, lm, cm)


# ---- colour converters (RTjpeg.c:3071-3486) ---------------------------------------------------

CONV_RGB32, CONV_BGR32, CONV_RGB24, CONV_BGR24, CONV_RGB16, CONV_RGB8, CONV_YUV422_RGB24 = range(7)
CONV_BPP = (4, 4, 3, 3, 2, 1, 3)


def _convert(fn, kind: int, frame: np.ndarray, w: int, h: int, pitch: int | None, fill: int) -> np.ndarray:
    frame = _np_u8(frame)
    pitch = w * CONV_BPP[kind] if pitch is None else pitch
    ysz = w * h
    csz = ysz // 2 if kind == CONV_YUV422_RGB24 else ysz // 4
    if kind == CONV_RGB8:
        assert frame.size >= ysz
    else:
        assert frame.size >= ysz + 2 * csz
    out = np.full(h * pitch, fill, dtype=np.uint8)
    base = frame.ctypes.data
    fn(kind, w, h, C.cast(base, _u8p), C.cast(base + ysz, _u8p), C.cast(base + ysz + csz, _u8p), _ptr(out), pitch)
    return out.reshape(h, pitch)


def convert(kind: int, frame: np.ndarray, w: int, h: int, pitch: int | None = None, fill: int = 0) -> np.ndarray:
    """Restatement of the reference's converter `kind` over one tight picture; bytes the converter does not
    write (the fourth byte of a 32-bit pixel, row padding) keep the value `fill`."""
    L = oracle_lib()
    L.rtjo_convert.argtypes = [C.c_int, C.c_int, C.c_int, _u8p, _u8p, _u8p, _u8p, C.c_size_t]
    L.rtjo_convert.restype = None
    return _convert(L.rtjo_convert, kind, frame, w, h, pitch, fill)


def ref_convert(kind: int, frame: np.ndarray, w: int, h: int, pitch: int | None = None, fill: int = 0) -> np.ndarray:
    """The unmodified reference's converter (RTjpeg_yuv420rgb32 ...)."""
    L = ref_lib()
    L.refdrv_convert.argtypes = [C.c_int, C.c_int, C.c_int, _u8p, _u8p, _u8p, _u8p, C.c_size_t]
    L.refdrv_convert.restype = None
    return _convert(L.refdrv_convert, kind, frame, w, h, pitch, fill)


# ---- encoder (RTjpeg_compress, RTjpeg.c:3488-3524) --------------------------------------------

class _Encoder(C.Structure):
    _fields_ = [("fmt", C.c_int), ("width", C.c_int), ("height", C.c_int), ("Q", C.c_int),
                ("lqt", C.c_int32 * 64), ("cqt", C.c_int32 * 64), ("lb8", C.c_int), ("cb8", C.c_int),
                ("key_rate", C.c_int), ("key_count", C.c_int), ("lmask", C.c_int), ("cmask", C.c_int),
                ("nblk", C.c_int), ("old", C.c_void_p)]


def encode_frames_oracle(frames: np.ndarray, w: int, h: int, fmt: int, Q: int, key_rate: int = 0, lm: int = 0, cm: int = 0,
                         align: int = 16):
    """Restatement of RTjpeg_compress over tight pictures [F, frame_bytes(fmt)]; returns (stream, offsets) laid out like
    encode_frames_fmt (packets `align`-aligned).  key_rate <= 0 is intra-only, as when RTjpeg_set_intra is never called."""
    L = oracle_lib()
    L.rtjo_encoder_init.argtypes = [C.POINTER(_Encoder), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.rtjo_encoder_free.argtypes = [C.POINTER(_Encoder)]
    L.rtjo_encode_frame.argtypes = [C.POINTER(_Encoder), _u8p, _u8p, _u8p, _u8p]
    L.rtjo_encode_frame.restype = C.c_long
    frames = _np_u8(frames)
    F = frames.shape[0]
    ysz = w * h
    csz = ysz // 4 if fmt == 0 else ysz // 2 if fmt == 1 else 0
    e = _Encoder()
    L.rtjo_encoder_init(C.byref(e), fmt, w, h, Q, max(key_rate, 0), lm, cm)
    bound = 12 + (w // 8) * (h // 8) * 2 * 64 + 64
    tmp = np.zeros(bound, dtype=np.uint8)
    pkts = []
    for f in range(F):
        base = frames[f].ctypes.data
        n = L.rtjo_encode_frame(C.byref(e), C.cast(base, _u8p), C.cast(base + ysz, _u8p), C.cast(base + ysz + csz, _u8p), _ptr(tmp))
        if n < 0:
            L.rtjo_encoder_free(C.byref(e))
            raise ValueError("the 8-bit encoder of the reference reads outside its plane; not restated")
        pkts.append(tmp[:n].copy())
    L.rtjo_encoder_free(C.byref(e))
    return pack_packets(pkts, align)


def encode_frames_grey(frames: np.ndarray, w: int, h: int, Q: int, key_rate: int = 0, lm: int = 0, align: int = 16):
    """The reference's RTjpeg_compress in the 8-bit format over grey pictures [F, w*h] (rtjo_encode_frame8): it reads
    every picture up to 56 rows past its end, which is the next picture or, behind the last one, zeros."""
    L = oracle_lib()
    L.rtjo_encoder_init.argtypes = [C.POINTER(_Encoder), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.rtjo_encoder_free.argtypes = [C.POINTER(_Encoder)]
    L.rtjo_encode_frame8.argtypes = [C.POINTER(_Encoder), C.c_void_p, _u8p]
    L.rtjo_encode_frame8.restype = C.c_long
    frames = _np_u8(frames)
    F = frames.shape[0]
    padded = np.zeros(frames.size + 64 * w, dtype=np.uint8)
    padded[:frames.size] = frames.reshape(-1)
    e = _Encoder()
    L.rtjo_encoder_init(C.byref(e), 2, w, h, Q, max(key_rate, 0), lm, lm)
    tmp = np.zeros(12 + (w // 8) * (h // 8) * 64 + 64, dtype=np.uint8)
    pkts = []
    for f in range(F):
        n = L.rtjo_encode_frame8(C.byref(e), padded.ctypes.data + f * w * h, _ptr(tmp))
        pkts.append(tmp[:n].copy())
    L.rtjo_encoder_free(C.byref(e))
    return pack_packets(pkts, align)


def decode_threaded(stream, offsets, segments, w: int, h: int, threads: int = 0, zero_init: bool = True,
                    raw_tables=None) -> np.ndarray:
    """Restatement decode of independent frame ranges on `threads` workers (segments: first frame of each range, then
    the frame count); returns [F, w*h*3/2].  raw_tables: 128 raw entries every worker's decoder starts with, as
    RTjpeg_set_tables leaves them (the packets then carry quality 0)."""
    stream = _np_u8(stream)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    seg = np.ascontiguousarray(segments, dtype=np.int32)
    F = int(seg[-1])
    frames = np.empty((F, w * h * 3 // 2), dtype=np.uint8)
    raw = None if raw_tables is None else np.ascontiguousarray(raw_tables, dtype=np.uint32)
    rc = oracle_lib().rtjo_decode_threaded(_ptr(stream), _ptr(offsets, _u64p), seg.ctypes.data_as(C.POINTER(C.c_int)),
                                           len(seg) - 1, w, h, threads or (os.cpu_count() or 1), 1 if zero_init else 0,
                                           _ptr(frames), None if raw is None else _ptr(raw, _u32p))
    if rc < 0:
        raise ValueError("truncated packet")
    return frames


def decode_with_tables(raw, pkt, w: int, h: int, planes: np.ndarray) -> np.ndarray:
    """Restatement decode of one packet on a fresh decoder given raw tables first (RTjpeg_set_tables: they stay in force
    while the packet's quality byte is 0)."""
    d = _Decoder()
    oracle_lib().rtjo_decoder_reset(C.byref(d))
    raw = np.ascontiguousarray(raw, dtype=np.uint32)
    oracle_lib().rtjo_tables_from_raw(_ptr(raw, _u32p), C.byref(d.t))
    d.width, d.height, d.Q = w, h, 0
    pkt = _np_u8(pkt)
    p = np.array(planes, dtype=np.uint8).copy()
    n = oracle_lib().rtjo_decode_packet(C.byref(d), _ptr(pkt), pkt.size, _ptr(p), C.cast(p.ctypes.data + w * h, _u8p),
                                        C.cast(p.ctypes.data + w * h * 5 // 4, _u8p))
    if n < 0:
        raise ValueError("truncated packet")
    return p
