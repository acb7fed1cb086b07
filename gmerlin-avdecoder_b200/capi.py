"""ctypes binding of the C ABI declared in include/rtjpeg_b200.h.

The library is built in-tree by ``make -C gmerlin-avdecoder_b200`` (see
``build_library``).  Loading fails loudly when the shared object is missing and
every context constructor fails loudly when no CUDA device is usable: there is
no CPU path in this package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import weakref

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# RTJPEG_B200_LIBFILE: development switch, another build of the same library (kernel variants side by side)
LIB_PATH = os.environ.get("RTJPEG_B200_LIBFILE") or os.path.join(PKG_DIR, "lib", "librtjpeg_b200.so")
PLUGIN_PATH = os.path.join(PKG_DIR, "lib", "librtjpeg_b200_bgav.so")

# mirrors of the C structs ---------------------------------------------------

FRAME_DESC_DTYPE = np.dtype([("offset", "<u8"), ("length", "<u4"), ("table", "<u2"), ("flags", "<u2")])
assert FRAME_DESC_DTYPE.itemsize == 16


class State(C.Structure):
    """rtjgpu_state: decoder state that crosses batch boundaries."""
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("table", C.c_int), ("quality", C.c_int)]


class Timing(C.Structure):
    _fields_ = [("scan_ms", C.c_float), ("resolve_ms", C.c_float), ("idct_ms", C.c_float), ("total_ms", C.c_float)]


class BatchInfo(C.Structure):
    _fields_ = [("skipped_blocks", C.c_uint64), ("payload_bytes", C.c_uint64),
                ("bad_frames", C.c_uint32), ("first_bad_frame", C.c_int32)]


class NuvHeader(C.Structure):
    """rtjnuv_header: what lib/demux_nuv.c:58-243 reads before the first frame."""
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("interlaced", C.c_int), ("is_mythtv", C.c_int),
                ("aspect", C.c_double), ("fps", C.c_double), ("video_packets", C.c_uint32), ("audio_packets", C.c_uint32),
                ("has_tables", C.c_int), ("tables", C.c_uint32 * 128), ("data_start", C.c_uint64)]


class NuvPacket(C.Structure):
    _fields_ = [("type", C.c_uint8), ("comptype", C.c_uint8), ("keyframe", C.c_uint8), ("filters", C.c_uint8),
                ("timecode", C.c_uint32), ("size", C.c_uint32), ("payload_offset", C.c_uint64)]


OK = 0
E_CUDA, E_ARG, E_HEADER, E_SIZE, E_FORMAT, E_OVERRUN, E_TOOBIG, E_NOMEM = -1, -2, -3, -4, -5, -6, -7, -8
HOST_IN_PINNED, HOST_OUT_PINNED = 1, 2
STREAM_SLACK_BYTES = 128
TABLE_ZERO, TABLE_CUSTOM = 0, 256
SCAN_AUTO, SCAN_LANE, SCAN_WARP, SCAN_CHUNK, SCAN_SEGMENT, SCAN_WALK, SCAN_SYNC = 0, 1, 2, 3, 4, 5, 6
PIPELINE_AUTO, PIPELINE_SERIAL, PIPELINE_SLICED = 0, 1, 2

_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


class RTjpegError(RuntimeError):
    def __init__(self, code: int, what: str = ""):
        self.code = code
        msg = load_library().rtjgpu_strerror(code).decode() if _lib is not None else str(code)
        super().__init__(f"{what}: {msg} ({code})" if what else f"{msg} ({code})")


def build_library(verbose: bool = False) -> None:
    """Compile every CUDA/C++ source for sm_100a into gmerlin-avdecoder_b200/lib/."""
    cmd = ["make", "-C", PKG_DIR, "all"]
    if not verbose:
        cmd.insert(1, "-s")
    subprocess.check_call(cmd)


_lib = None


def load_library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} is missing: run `make -C {PKG_DIR}` (or __graft_entry__.build()); "
            "there is no fallback implementation")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    # Level 1
    L.RTjpeg_init.restype = vp
    L.RTjpeg_close.argtypes = [vp]
    L.RTjpeg_close.restype = None
    for name in ("RTjpeg_set_quality", "RTjpeg_set_format"):
        getattr(L, name).argtypes = [vp, C.POINTER(C.c_int)]
    L.RTjpeg_set_size.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.RTjpeg_set_intra.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.RTjpeg_get_tables.argtypes = [vp, _u32p]
    L.RTjpeg_get_tables.restype = None
    L.RTjpeg_set_tables.argtypes = [vp, _u32p]
    L.RTjpeg_set_tables.restype = None
    L.RTjpeg_decompress.argtypes = [vp, _u8p, C.POINTER(_u8p)]
    L.RTjpeg_decompress.restype = None
    L.RTjpeg_b200_decompress_n.argtypes = [vp, _u8p, C.c_size_t, C.POINTER(_u8p)]
    L.RTjpeg_b200_last_error.argtypes = [vp]
    # Level 2
    L.rtjgpu_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.rtjgpu_destroy.argtypes = [vp]
    L.rtjgpu_destroy.restype = None
    L.rtjgpu_strerror.argtypes = [C.c_int]
    L.rtjgpu_strerror.restype = C.c_char_p
    L.rtjgpu_last_cuda_error.argtypes = [vp]
    L.rtjgpu_set_custom_tables.argtypes = [vp, _u32p]
    L.rtjgpu_set_scan_mode.argtypes = [vp, C.c_int]
    L.rtjgpu_set_format.argtypes = [vp, C.c_int]
    L.rtjgpu_set_pipeline.argtypes = [vp, C.c_int, C.c_int]
    L.rtjgpu_set_frame_runs.argtypes = [vp, C.c_int]
    L.rtjgpu_convert_device.argtypes = [vp, C.c_int, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, C.c_size_t,
                                        C.c_int, vp]
    L.rtjgpu_convert_bpp.argtypes = [C.c_int]
    L.rtjgpu_encoder_set_quality.argtypes = [vp, C.c_int]
    L.rtjgpu_encoder_set_intra.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.rtjgpu_encoder_reset.argtypes = [vp]
    L.rtjgpu_encode_device.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, vp, vp]
    L.rtjgpu_get_encode_info.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
    L.rtjgpu_seqenc_create.argtypes = [vp, C.POINTER(vp)]
    L.rtjgpu_seqenc_destroy.argtypes = [vp]
    L.rtjgpu_seqenc_destroy.restype = None
    L.rtjgpu_seqenc_set_quality.argtypes = [vp, C.c_int]
    L.rtjgpu_seqenc_set_intra.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.rtjgpu_seqenc_reset.argtypes = [vp]
    L.rtjgpu_seqenc_key_count.argtypes = [vp]
    L.rtjgpu_encode_device_seq.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(vp),
                                           C.POINTER(vp), vp, C.c_size_t, vp, vp]
    L.rtjgpu_encode_bound.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    L.rtjgpu_encode_bound.restype = C.c_size_t
    L.RTjpeg_compress.argtypes = [vp, _u8p, C.POINTER(_u8p)]
    for name in CONVERTERS:
        getattr(L, name).argtypes = [vp, C.POINTER(_u8p), C.POINTER(_u8p)]
        getattr(L, name).restype = None
    L.rtjgpu_plan.argtypes = [_u8p, _u64p, C.c_int, C.POINTER(State), vp]
    L.rtjgpu_decode_device.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.rtjgpu_decode_device_rgb.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, C.c_size_t, C.c_int,
                                           vp, vp, vp]
    L.rtjgpu_decode_device_seq.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), vp,
                                           C.POINTER(vp), vp]
    L.rtjgpu_decode_device_rgb_seq.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int, vp,
                                               C.c_size_t, C.c_size_t, C.c_int, C.POINTER(vp), C.POINTER(vp), vp]
    L.rtjgpu_decode_device_select.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(vp),
                                              C.c_int, C.POINTER(C.c_int), vp, vp]
    L.rtjgpu_decode_device_rgb_select.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int),
                                                  C.POINTER(vp), C.c_int, C.POINTER(C.c_int), C.c_int, vp, C.c_size_t,
                                                  C.c_size_t, C.c_int, C.POINTER(vp), vp]
    L.rtjgpu_decode_device_window.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(vp),
                                              C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_int), vp,
                                              C.POINTER(vp), vp]
    L.rtjgpu_decode_device_rgb_window.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int),
                                                  C.POINTER(vp), C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int,
                                                  C.POINTER(C.c_int), C.c_int, vp, C.c_size_t, C.c_size_t, C.c_int,
                                                  C.POINTER(vp), vp]
    L.rtjgpu_decode_device_chw_window.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int),
                                                  C.POINTER(vp), C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int,
                                                  C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.c_int,
                                                  C.POINTER(C.c_float), C.POINTER(C.c_float), vp, C.POINTER(vp), vp]
    L.rtjgpu_decode_host.argtypes = [vp, _u8p, _u64p, C.c_int, C.POINTER(State), _u8p, _u8p, C.c_int]
    L.rtjgpu_sync.argtypes = [vp]
    L.rtjgpu_enable_timing.argtypes = [vp, C.c_int]
    L.rtjgpu_enable_timing.restype = None
    L.rtjgpu_get_timing.argtypes = [vp, C.POINTER(Timing)]
    L.rtjgpu_get_timing_at.argtypes = [vp, C.c_int, C.POINTER(Timing)]
    L.rtjgpu_get_batch_info.argtypes = [vp, C.POINTER(BatchInfo)]
    L.rtjgpu_get_skip_counts.argtypes = [vp, _u32p, C.c_int]
    L.rtjgpu_launch_count.argtypes = [vp]
    L.rtjgpu_launch_count.restype = C.c_uint64
    L.rtjgpu_split_shards.argtypes = [_u8p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    L.rtjgpu_split_shards_lead.argtypes = [_u8p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.rtjgpu_scan_device.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
    L.rtjgpu_tables_for_quality.argtypes = [C.c_int, _u32p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.rtjgpu_tables_for_quality.restype = None
    L.rtjgpu_tables_from_raw.argtypes = [_u32p, _u32p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.rtjgpu_tables_from_raw.restype = None
    L.rtjgpu_raw_tables_for_quality.argtypes = [C.c_int, _u32p]
    L.rtjgpu_raw_tables_for_quality.restype = None
    L.rtjnuv_probe.argtypes = [_u8p, C.c_size_t]
    L.rtjnuv_open.argtypes = [_u8p, C.c_size_t, C.POINTER(NuvHeader)]
    L.rtjnuv_next.argtypes = [_u8p, C.c_size_t, _u64p, C.POINTER(NuvPacket)]
    L.rtjnuv_extract_rtj0.argtypes = [_u8p, C.c_size_t, C.POINTER(NuvHeader), _u8p, C.c_size_t, _u64p, _u32p,
                                      C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.rtjgpu_host_alloc.argtypes = [C.c_size_t]
    L.rtjgpu_host_alloc.restype = vp
    L.rtjgpu_host_free.argtypes = [vp]
    L.rtjgpu_host_free.restype = None
    _lib = L
    return L


# the converters of include/RTjpeg.h:128-136, indexed by RTJ_CONV_*
CONV_RGB32, CONV_BGR32, CONV_RGB24, CONV_BGR24, CONV_RGB16, CONV_RGB8, CONV_YUV422_RGB24 = range(7)
CONVERTERS = ("RTjpeg_yuv420rgb32", "RTjpeg_yuv420bgr32", "RTjpeg_yuv420rgb24", "RTjpeg_yuv420bgr24",
              "RTjpeg_yuv420rgb16", "RTjpeg_yuv420rgb8", "RTjpeg_yuv422rgb24")
CONV_BPP = (4, 4, 3, 3, 2, 1, 3)

# element types of rtjgpu_decode_device_chw_window, indexed by RTJ_CHW_*, and their sizes in bytes
CHW_U8, CHW_F16, CHW_BF16, CHW_F32 = range(4)
CHW_ESIZE = (1, 2, 2, 4)


def normalize_coefficients(mean, std):
    """The per-channel scale and bias of rtjgpu_decode_device_chw_window that mean torchvision's normalisation of a byte v,
    (v / 255 - mean) / std: scale = 1 / (255 std), bias = -mean / std.  Computed in float64, rounded once to float32.
    Returns (scale, bias), two float32 arrays of 3."""
    mean = np.asarray(mean, dtype=np.float64).reshape(-1)
    std = np.asarray(std, dtype=np.float64).reshape(-1)
    if mean.shape != (3,) or std.shape != (3,):
        raise ValueError("normalize_coefficients: mean and std take 3 values, one per channel")
    if not (np.isfinite(mean).all() and np.isfinite(std).all()) or (std == 0).any():
        raise ValueError("normalize_coefficients: mean and std must be finite, std nonzero")
    return (1.0 / (255.0 * std)).astype(np.float32), (-mean / std).astype(np.float32)


def frame_bytes(fmt: int, w: int, h: int) -> int:
    """Tight planes of one picture: YUV420 w*h*3/2, YUV422 w*h*2, 8-bit grey w*h."""
    return w * h * 3 // 2 if fmt == 0 else w * h * 2 if fmt == 1 else w * h


def _u8(a: np.ndarray):
    return a.ctypes.data_as(_u8p)


def _int_array(v):
    return (C.c_int * max(len(v), 1))(*[int(x) for x in v])


def _ptr_array(v):
    """A host array of device addresses (None entries: NULL), or NULL for v = None."""
    if v is None:
        return None
    return (C.c_void_p * max(len(v), 1))(*[int(x) if x else None for x in v])


def _origins_array(origins):
    """[(x, y), ...] -> the host array of 2 S ints the window calls take, or NULL for None."""
    if origins is None:
        return None
    return _int_array([int(v) for xy in origins for v in xy])


def _float3(v):
    """3 floats -> a host float array, or NULL for None."""
    if v is None:
        return None
    v = np.asarray(v, dtype=np.float32).reshape(-1)
    if v.shape != (3,):
        raise ValueError("3 values, one per channel, expected")
    return (C.c_float * 3)(*[float(x) for x in v])


def _check(rc: int, what: str) -> None:
    if rc != OK:
        raise RTjpegError(rc, what)


# Level 2 ----------------------------------------------------------------------

def plan(stream: np.ndarray, offsets: np.ndarray, state: State | None = None):
    """rtjgpu_plan: header parse + lazy reconfiguration -> (descriptors, state)."""
    L = load_library()
    stream = np.ascontiguousarray(stream, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    F = len(offsets) - 1
    st = State(0, 0, TABLE_ZERO, 0) if state is None else state
    desc = np.zeros(max(F, 1), dtype=FRAME_DESC_DTYPE)
    _check(L.rtjgpu_plan(_u8(stream), offsets.ctypes.data_as(_u64p), F, C.byref(st),
                         C.c_void_p(desc.ctypes.data)), "rtjgpu_plan")
    return desc[:F], st


def plan_sequences(seqs, states=None):
    """Several independent packet sequences into one batch for rtjgpu_decode_device_seq.  seqs: list of (stream, offsets) as
    for plan().  Every sequence's packets keep their slots and their alignment modulo 16 in one buffer; each sequence is
    planned on its own with its own state (states: list of State advanced in place, or None = fresh ones).
    Returns (stream, offsets[F + 1], desc[F], seq_first[S + 1], states)."""
    if states is None:
        states = [State(0, 0, TABLE_ZERO, 0) for _ in seqs]
    assert len(states) == len(seqs)
    bases, at = [], 0
    for _, offsets in seqs:
        lo, hi = int(offsets[0]), int(offsets[-1])
        base = (at + 15) // 16 * 16 + lo % 16           # the packets' starts keep their place modulo 16
        bases.append(base)
        at = base + hi - lo
    out = np.zeros(at, dtype=np.uint8)
    offs, descs, seq_first = [], [], [0]
    for (stream, offsets), base, st in zip(seqs, bases, states):
        offsets = np.asarray(offsets, dtype=np.uint64)
        lo, hi = int(offsets[0]), int(offsets[-1])
        out[base:base + hi - lo] = np.asarray(stream, dtype=np.uint8)[lo:hi]
        o = offsets - np.uint64(lo) + np.uint64(base)
        desc, _ = plan(out, o, st)
        offs.append(o[:-1])
        descs.append(desc)
        seq_first.append(seq_first[-1] + len(desc))
    offsets = np.concatenate(offs + [np.array([at], dtype=np.uint64)])
    return out, offsets, np.concatenate(descs), np.array(seq_first, dtype=np.int64), states


def select_frames(seq_first, picks) -> np.ndarray:
    """Per-sequence frame indices -> the batch frame indices rtjgpu_decode_device_select takes.  picks: a list of S index
    arrays, picks[s] local to sequence s (0 .. its length - 1, any order).  Returns the sorted global indices (int64); output
    slot k of the select call is then the k-th of them.  Raises ValueError for an index outside its sequence or one named
    twice."""
    seq_first = np.asarray(seq_first, dtype=np.int64)
    S = len(seq_first) - 1
    if len(picks) != S:
        raise ValueError(f"select_frames: {len(picks)} index arrays for {S} sequences")
    out = []
    for s, p in enumerate(picks):
        p = np.asarray(p, dtype=np.int64).reshape(-1)
        n = int(seq_first[s + 1] - seq_first[s])
        if p.size and (p.min() < 0 or p.max() >= n):
            raise ValueError(f"select_frames: sequence {s} has {n} frames, index out of range")
        p = np.sort(p)
        if p.size > 1 and (np.diff(p) == 0).any():
            raise ValueError(f"select_frames: sequence {s}: an index named twice")
        out.append(p + seq_first[s])
    return np.concatenate(out) if out else np.zeros(0, dtype=np.int64)


def encode_bound(fmt: int, w: int, h: int, F: int) -> int:
    """rtjgpu_encode_bound: the most bytes F packets of format fmt and size w x h can take (0: not encodable)."""
    return int(load_library().rtjgpu_encode_bound(fmt, w, h, F))


def tables_for_quality(Q: int):
    """Host-only: (scaled[128], lb8, cb8) as RTjpeg_set_quality would leave them."""
    out = np.zeros(128, dtype=np.uint32)
    a, b = C.c_int(), C.c_int()
    load_library().rtjgpu_tables_for_quality(Q, out.ctypes.data_as(_u32p), C.byref(a), C.byref(b))
    return out, a.value, b.value


def tables_from_raw(raw: np.ndarray):
    raw = np.ascontiguousarray(raw, dtype=np.uint32)
    out = np.zeros(128, dtype=np.uint32)
    a, b = C.c_int(), C.c_int()
    load_library().rtjgpu_tables_from_raw(raw.ctypes.data_as(_u32p), out.ctypes.data_as(_u32p), C.byref(a), C.byref(b))
    return out, a.value, b.value


def raw_tables_for_quality(Q: int) -> np.ndarray:
    """The 128 raw (not AAN-scaled) entries RTjpeg_set_tables takes for quality Q."""
    out = np.zeros(128, dtype=np.uint32)
    load_library().rtjgpu_raw_tables_for_quality(Q, out.ctypes.data_as(_u32p))
    return out


# NuppelVideo container (host only) --------------------------------------------

def nuv_probe(data: np.ndarray) -> bool:
    data = np.ascontiguousarray(data, dtype=np.uint8)
    return bool(load_library().rtjnuv_probe(_u8(data), data.size))


def nuv_open(data: np.ndarray) -> NuvHeader:
    data = np.ascontiguousarray(data, dtype=np.uint8)
    h = NuvHeader()
    _check(load_library().rtjnuv_open(_u8(data), data.size, C.byref(h)), "rtjnuv_open")
    return h


def nuv_packets(data: np.ndarray, hdr: NuvHeader):
    """Every frame header behind the codec data: list of (type, comptype, keyframe, timecode, size, payload_offset)."""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    L = load_library()
    pos = C.c_uint64(hdr.data_start)
    p = NuvPacket()
    out = []
    while L.rtjnuv_next(_u8(data), data.size, C.byref(pos), C.byref(p)):
        out.append((chr(p.type), chr(p.comptype), int(p.keyframe), int(p.timecode), int(p.size), int(p.payload_offset)))
    return out


def nuv_extract_rtj0(data: np.ndarray, hdr: NuvHeader):
    """The file's RTjpeg video frames as 'RTJ0' packets -> (stream, offsets, timecodes, unsupported)."""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    L = load_library()
    cap = max(int(hdr.video_packets), sum(1 for p in nuv_packets(data, hdr) if p[0] == "V"))
    offsets = np.zeros(cap + 1, dtype=np.uint64)
    n, bad = C.c_int(), C.c_int()
    _check(L.rtjnuv_extract_rtj0(_u8(data), data.size, C.byref(hdr), None, 0, offsets.ctypes.data_as(_u64p), None,
                                 cap, C.byref(n), C.byref(bad)), "rtjnuv_extract_rtj0 (sizing)")
    total = int(offsets[n.value])
    stream = np.full(total + STREAM_SLACK_BYTES, 0x7F, dtype=np.uint8)
    tc = np.zeros(cap, dtype=np.uint32)
    _check(L.rtjnuv_extract_rtj0(_u8(data), data.size, C.byref(hdr), _u8(stream), total, offsets.ctypes.data_as(_u64p),
                                 tc.ctypes.data_as(_u32p), cap, C.byref(n), C.byref(bad)), "rtjnuv_extract_rtj0")
    return stream, offsets[:n.value + 1].copy(), tc[:n.value].copy(), int(bad.value)


def split_shards(clean: np.ndarray, n: int, allow_empty: bool = True) -> np.ndarray:
    """rtjgpu_split_shards: cuts on clean frames only -> first[n + 1].  A shard comes out empty when the clean frames
    run out; allow_empty=False raises instead."""
    L = load_library()
    clean = np.ascontiguousarray(clean, dtype=np.uint8)
    first = (C.c_int * (n + 1))()
    rc = L.rtjgpu_split_shards(_u8(clean), len(clean), n, first)
    if rc < 0:
        raise RTjpegError(rc, "rtjgpu_split_shards")
    if rc > 0 and not allow_empty:
        raise ValueError(f"rtjgpu_split_shards: {rc} of {n} shards are empty (not enough clean frames); use split_shards_lead")
    return np.array(first[:], dtype=np.int64)


def split_shards_lead(clean: np.ndarray, n: int):
    """rtjgpu_split_shards_lead -> (first[n + 1], lead[n]): shard i decodes frames [first[i] - lead[i], first[i + 1])
    and keeps the last first[i + 1] - first[i]."""
    L = load_library()
    clean = np.ascontiguousarray(clean, dtype=np.uint8)
    first = (C.c_int * (n + 1))()
    lead = (C.c_int * n)()
    _check(L.rtjgpu_split_shards_lead(_u8(clean), len(clean), n, first, lead), "rtjgpu_split_shards_lead")
    return np.array(first[:], dtype=np.int64), np.array(lead[:], dtype=np.int64)


class BatchContext:
    """rtjgpu_ctx: one per device and per decoding thread."""

    def __init__(self, device: int = 0):
        self._L = load_library()
        h = C.c_void_p()
        rc = self._L.rtjgpu_create(device, C.byref(h))
        if rc != OK or not h.value:
            raise RTjpegError(rc or E_CUDA, f"rtjgpu_create(device={device}): no usable CUDA device, and no CPU fallback")
        self._h = h
        self.device = device
        self._encoders = weakref.WeakSet()      # SeqEncoder handles of this context, freed with it

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            for e in list(getattr(self, "_encoders", ())):
                e.close()
            self._L.rtjgpu_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_scan_mode(self, mode: int) -> None:
        """0 = auto, 1 = one thread per frame, 2 = one warp per frame."""
        _check(self._L.rtjgpu_set_scan_mode(self._h, mode), "rtjgpu_set_scan_mode")

    def set_frame_runs(self, frames: int = 0) -> None:
        """rtjgpu_set_frame_runs: 0 = by the batch before, 1 = every frame for itself, n = runs of n frames per CTA of K2."""
        _check(self._L.rtjgpu_set_frame_runs(self._h, frames), "rtjgpu_set_frame_runs")

    def set_pipeline(self, mode: int = PIPELINE_AUTO, slice_frames: int = 0) -> None:
        """PIPELINE_SERIAL (= AUTO at present): stage after stage; PIPELINE_SLICED: scan of slice s + 1 beside resolve + IDCT of slice s."""
        _check(self._L.rtjgpu_set_pipeline(self._h, mode, slice_frames), "rtjgpu_set_pipeline")

    def set_format(self, fmt: int) -> None:
        """RTJ_YUV420 (default), RTJ_YUV422 or RTJ_RGB8 (8-bit grey) for the batches that follow."""
        _check(self._L.rtjgpu_set_format(self._h, fmt), "rtjgpu_set_format")

    def convert_device(self, kind: int, d_frames: int, src_frame_bytes: int, F: int, w: int, h: int, d_out: int,
                       row_pitch: int, frame_pitch: int, alpha: int = 0, cuda_stream: int | None = None) -> None:
        """The reference's colour converter `kind` (CONV_*) over F device-resident pictures."""
        _check(self._L.rtjgpu_convert_device(self._h, kind, C.c_void_p(d_frames), src_frame_bytes, F, w, h,
                                             C.c_void_p(d_out), row_pitch, frame_pitch, alpha,
                                             C.c_void_p(cuda_stream or 0)), "rtjgpu_convert_device")

    def encoder_config(self, quality: int, key_rate: int = 0, lm: int = 0, cm: int = 0) -> None:
        """RTjpeg_set_quality + RTjpeg_set_intra on a fresh encoder (key counter 0, no block sent yet)."""
        _check(self._L.rtjgpu_encoder_set_quality(self._h, quality), "rtjgpu_encoder_set_quality")
        _check(self._L.rtjgpu_encoder_set_intra(self._h, key_rate, lm, cm), "rtjgpu_encoder_set_intra")
        _check(self._L.rtjgpu_encoder_reset(self._h), "rtjgpu_encoder_reset")

    def encode_device(self, d_frames: int, F: int, w: int, h: int, d_stream: int, capacity: int, d_offsets: int,
                      cuda_stream: int | None = None) -> None:
        _check(self._L.rtjgpu_encode_device(self._h, C.c_void_p(d_frames), F, w, h, C.c_void_p(d_stream), capacity,
                                            C.c_void_p(d_offsets), C.c_void_p(cuda_stream or 0)), "rtjgpu_encode_device")

    def seq_encoder(self, quality: int | None = None, key_rate: int = 0, lm: int = 0, cm: int = 0) -> "SeqEncoder":
        """rtjgpu_seqenc_create: an encoder state of its own for encode_device_seq; quality None leaves a fresh instance's
        (0, zero tables)."""
        e = SeqEncoder(self)
        self._encoders.add(e)
        if quality is not None:
            e.set_quality(quality)
        if key_rate or lm or cm:
            e.set_intra(key_rate, lm, cm)
        return e

    def encode_device_seq(self, F: int, w: int, h: int, seq_first, frames, encoders, d_stream: int, capacity: int,
                          d_offsets: int, cuda_stream: int | None = None) -> None:
        """rtjgpu_encode_device_seq: frames a list of S device addresses (each sequence's first picture), encoders a list
        of S SeqEncoder (None: NULL, which the library refuses)."""
        S = len(seq_first) - 1
        _check(self._L.rtjgpu_encode_device_seq(self._h, F, w, h, S, _int_array(seq_first), _ptr_array(frames),
                                                _ptr_array([None if e is None else e._h.value for e in encoders]), C.c_void_p(d_stream), capacity,
                                                C.c_void_p(d_offsets), C.c_void_p(cuda_stream or 0)), "rtjgpu_encode_device_seq")

    def encode_info(self):
        b, o = C.c_uint64(), C.c_int()
        _check(self._L.rtjgpu_get_encode_info(self._h, C.byref(b), C.byref(o)), "rtjgpu_get_encode_info")
        return int(b.value), bool(o.value)

    def set_custom_tables(self, raw: np.ndarray) -> None:
        raw = np.ascontiguousarray(raw, dtype=np.uint32)
        assert raw.size == 128
        _check(self._L.rtjgpu_set_custom_tables(self._h, raw.ctypes.data_as(_u32p)), "rtjgpu_set_custom_tables")

    def decode_device(self, d_stream: int, d_desc: int, F: int, w: int, h: int, d_out: int,
                      d_carry: int | None = None, cuda_stream: int | None = None) -> None:
        """All pointers are raw device addresses (e.g. torch.Tensor.data_ptr())."""
        _check(self._L.rtjgpu_decode_device(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h,
                                            C.c_void_p(d_out), C.c_void_p(d_carry or 0),
                                            C.c_void_p(cuda_stream or 0)), "rtjgpu_decode_device")

    def decode_device_rgb(self, d_stream: int, d_desc: int, F: int, w: int, h: int, kind: int, d_rgb: int, row_pitch: int,
                          frame_pitch: int, alpha: int = 0, d_carry: int | None = None, d_last_yuv: int | None = None,
                          cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device with the converter `kind` (CONV_*) fused into the decode: packed pixels out."""
        _check(self._L.rtjgpu_decode_device_rgb(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, kind,
                                                C.c_void_p(d_rgb), row_pitch, frame_pitch, alpha, C.c_void_p(d_carry or 0),
                                                C.c_void_p(d_last_yuv or 0), C.c_void_p(cuda_stream or 0)),
               "rtjgpu_decode_device_rgb")

    def decode_device_seq(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, d_out: int,
                          carries=None, cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_seq: seq_first[S + 1] frame indices, carries a list of S device addresses (None = zeros)
        or None."""
        S = len(seq_first) - 1
        _check(self._L.rtjgpu_decode_device_seq(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                _int_array(seq_first), C.c_void_p(d_out), _ptr_array(carries),
                                                C.c_void_p(cuda_stream or 0)), "rtjgpu_decode_device_seq")

    def decode_device_rgb_seq(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, kind: int, d_rgb: int,
                              row_pitch: int, frame_pitch: int, alpha: int = 0, carries=None, last_yuv=None,
                              cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_rgb_seq: last_yuv a list of S device addresses (None = not wanted) or None."""
        S = len(seq_first) - 1
        _check(self._L.rtjgpu_decode_device_rgb_seq(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                    _int_array(seq_first), kind, C.c_void_p(d_rgb), row_pitch, frame_pitch,
                                                    alpha, _ptr_array(carries), _ptr_array(last_yuv),
                                                    C.c_void_p(cuda_stream or 0)), "rtjgpu_decode_device_rgb_seq")

    def decode_device_select(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, sel, d_out: int,
                             carries=None, cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_select: the batch of decode_device_seq, only frames sel (batch indices, strictly increasing;
        see select_frames) decoded, frame sel[k] to d_out + k * frame_bytes."""
        S = len(seq_first) - 1
        _check(self._L.rtjgpu_decode_device_select(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                   _int_array(seq_first), _ptr_array(carries), len(sel), _int_array(sel),
                                                   C.c_void_p(d_out or 0), C.c_void_p(cuda_stream or 0)),
               "rtjgpu_decode_device_select")

    def decode_device_rgb_select(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, sel, kind: int,
                                 d_rgb: int, row_pitch: int, frame_pitch: int, alpha: int = 0, carries=None, last_yuv=None,
                                 cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_rgb_select: frame sel[k] to d_rgb + k * frame_pitch; last_yuv as for decode_device_rgb_seq
        (each sequence's last frame as planes, selected or not)."""
        S = len(seq_first) - 1
        _check(self._L.rtjgpu_decode_device_rgb_select(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                       _int_array(seq_first), _ptr_array(carries), len(sel), _int_array(sel),
                                                       kind, C.c_void_p(d_rgb or 0), row_pitch, frame_pitch, alpha,
                                                       _ptr_array(last_yuv), C.c_void_p(cuda_stream or 0)),
               "rtjgpu_decode_device_rgb_select")

    def decode_device_window(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, sel, size, origins,
                             d_out: int, carries=None, last_yuv=None, cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_window: the selection of decode_device_select, only a window of size (cw, ch) of each frame,
        at origins[s] = (x, y) of its sequence, frame sel[k] to d_out + k * window_bytes as tight planes.  last_yuv: a list
        of S device addresses (None = not wanted) or None, receiving each sequence's last frame whole."""
        S = len(seq_first) - 1
        cw, ch = size
        _check(self._L.rtjgpu_decode_device_window(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                   _int_array(seq_first), _ptr_array(carries), len(sel), _int_array(sel),
                                                   cw, ch, _origins_array(origins), C.c_void_p(d_out or 0),
                                                   _ptr_array(last_yuv), C.c_void_p(cuda_stream or 0)),
               "rtjgpu_decode_device_window")

    def decode_device_rgb_window(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, sel, size, origins,
                                 kind: int, d_rgb: int, row_pitch: int, frame_pitch: int, alpha: int = 0, carries=None,
                                 last_yuv=None, cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_rgb_window: window row r of frame sel[k] to d_rgb + k * frame_pitch + r * row_pitch;
        last_yuv as for decode_device_window."""
        S = len(seq_first) - 1
        cw, ch = size
        _check(self._L.rtjgpu_decode_device_rgb_window(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                       _int_array(seq_first), _ptr_array(carries), len(sel), _int_array(sel),
                                                       cw, ch, _origins_array(origins), kind, C.c_void_p(d_rgb or 0),
                                                       row_pitch, frame_pitch, alpha, _ptr_array(last_yuv),
                                                       C.c_void_p(cuda_stream or 0)),
               "rtjgpu_decode_device_rgb_window")

    def decode_device_chw_window(self, d_stream: int, d_desc: int, F: int, w: int, h: int, seq_first, sel, size, origins,
                                 kind: int, dtype: int, d_out: int, mirror=None, scale=None, bias=None, carries=None,
                                 last_yuv=None, cuda_stream: int | None = None) -> None:
        """rtjgpu_decode_device_chw_window: the window of frame sel[k] to d_out + k * 3 * ch * cw * CHW_ESIZE[dtype] as a
        tight [3][ch][cw] array of dtype (CHW_*), channel c byte c of kind's pixel (CONV_RGB24 / CONV_BGR24).  mirror: S flags
        or None; scale, bias: 3 floats each or None (1 and 0); last_yuv as for decode_device_window."""
        S = len(seq_first) - 1
        cw, ch = size
        mir = None if mirror is None else _int_array([1 if m else 0 for m in mirror])
        _check(self._L.rtjgpu_decode_device_chw_window(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h, S,
                                                       _int_array(seq_first), _ptr_array(carries), len(sel), _int_array(sel),
                                                       cw, ch, _origins_array(origins), mir, kind, dtype, _float3(scale),
                                                       _float3(bias), C.c_void_p(d_out or 0), _ptr_array(last_yuv),
                                                       C.c_void_p(cuda_stream or 0)),
               "rtjgpu_decode_device_chw_window")

    def decode_host(self, stream: np.ndarray, offsets: np.ndarray, out: np.ndarray, state: State | None = None,
                    carry: np.ndarray | None = None, flags: int = 0) -> State:
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        F = len(offsets) - 1
        st = State(0, 0, TABLE_ZERO, 0) if state is None else state
        assert stream.dtype == np.uint8 and out.dtype == np.uint8 and out.flags.c_contiguous
        _check(self._L.rtjgpu_decode_host(self._h, _u8(stream), offsets.ctypes.data_as(_u64p), F, C.byref(st),
                                          _u8(out), None if carry is None else _u8(carry), flags),
               "rtjgpu_decode_host")
        return st

    def scan_device(self, d_stream: int, d_desc: int, F: int, w: int, h: int, cuda_stream: int | None = None) -> None:
        """K1 only: afterwards skip_counts() / batch_info() describe the batch without it having been decoded."""
        _check(self._L.rtjgpu_scan_device(self._h, C.c_void_p(d_stream), C.c_void_p(d_desc), F, w, h,
                                          C.c_void_p(cuda_stream or 0)), "rtjgpu_scan_device")

    def sync(self) -> None:
        _check(self._L.rtjgpu_sync(self._h), "rtjgpu_sync")

    def enable_timing(self, on: bool = True) -> None:
        self._L.rtjgpu_enable_timing(self._h, 1 if on else 0)

    def timing(self) -> Timing:
        t = Timing()
        _check(self._L.rtjgpu_get_timing(self._h, C.byref(t)), "rtjgpu_get_timing")
        return t

    def timing_at(self, calls_ago: int) -> Timing:
        t = Timing()
        _check(self._L.rtjgpu_get_timing_at(self._h, calls_ago, C.byref(t)), "rtjgpu_get_timing_at")
        return t

    def batch_info(self) -> BatchInfo:
        b = BatchInfo()
        _check(self._L.rtjgpu_get_batch_info(self._h, C.byref(b)), "rtjgpu_get_batch_info")
        return b

    def skip_counts(self, F: int) -> np.ndarray:
        out = np.zeros(F, dtype=np.uint32)
        _check(self._L.rtjgpu_get_skip_counts(self._h, out.ctypes.data_as(_u32p), F), "rtjgpu_get_skip_counts")
        return out

    def launch_count(self) -> int:
        return int(self._L.rtjgpu_launch_count(self._h))


class SeqEncoder:
    """rtjgpu_seqenc: one stream's encoder state (tables, key counter, blocks last sent), bound to a BatchContext."""

    def __init__(self, ctx: BatchContext):
        self._L = ctx._L
        h = C.c_void_p()
        _check(self._L.rtjgpu_seqenc_create(ctx._h, C.byref(h)), "rtjgpu_seqenc_create")
        self._h = h

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.rtjgpu_seqenc_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def set_quality(self, quality: int) -> None:
        _check(self._L.rtjgpu_seqenc_set_quality(self._h, quality), "rtjgpu_seqenc_set_quality")

    def set_intra(self, key_rate: int, lm: int = 0, cm: int = 0) -> None:
        _check(self._L.rtjgpu_seqenc_set_intra(self._h, key_rate, lm, cm), "rtjgpu_seqenc_set_intra")

    def reset(self) -> None:
        _check(self._L.rtjgpu_seqenc_reset(self._h), "rtjgpu_seqenc_reset")

    @property
    def key_count(self) -> int:
        return int(self._L.rtjgpu_seqenc_key_count(self._h))


# Level 1 ----------------------------------------------------------------------

class RTjpeg:
    """The reference's codec object (include/RTjpeg.h:115-139) -- decode side."""

    def __init__(self):
        self._L = load_library()
        h = self._L.RTjpeg_init()
        if not h:
            raise RTjpegError(E_CUDA, "RTjpeg_init: no usable CUDA device, and no CPU fallback")
        self._h = C.c_void_p(h)

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.RTjpeg_close(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def set_quality(self, q: int) -> int:
        v = C.c_int(q)
        self._L.RTjpeg_set_quality(self._h, C.byref(v))
        return v.value

    def set_format(self, fmt: int) -> None:
        v = C.c_int(fmt)
        self._L.RTjpeg_set_format(self._h, C.byref(v))
        self._fmt = fmt

    def set_size(self, w: int, h: int) -> int:
        a, b = C.c_int(w), C.c_int(h)
        return self._L.RTjpeg_set_size(self._h, C.byref(a), C.byref(b))

    def set_intra(self, key: int, lm: int, cm: int):
        a, b, c = C.c_int(key), C.c_int(lm), C.c_int(cm)
        self._L.RTjpeg_set_intra(self._h, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def get_tables(self) -> np.ndarray:
        out = np.zeros(128, dtype=np.uint32)
        self._L.RTjpeg_get_tables(self._h, out.ctypes.data_as(_u32p))
        return out

    def set_tables(self, raw: np.ndarray) -> None:
        raw = np.ascontiguousarray(raw, dtype=np.uint32).copy()
        self._L.RTjpeg_set_tables(self._h, raw.ctypes.data_as(_u32p))

    def _planes(self, planes: np.ndarray, w: int, h: int):
        assert planes.dtype == np.uint8 and planes.flags.c_contiguous
        fmt = getattr(self, "_fmt", 0)
        if planes.size < frame_bytes(fmt, w, h):      # header lies about the geometry: the library refuses it before any plane access
            w = h = 0
        base = planes.ctypes.data
        csz = w * h // 4 if fmt == 0 else w * h // 2 if fmt == 1 else 0
        arr = (_u8p * 3)(C.cast(base, _u8p), C.cast(base + w * h, _u8p), C.cast(base + w * h + csz, _u8p))
        return arr

    def decompress(self, pkt: np.ndarray, planes: np.ndarray) -> None:
        """RTjpeg_decompress: planes is one tight buffer (Y|U|V in the current format) updated in place."""
        pkt = np.ascontiguousarray(pkt, dtype=np.uint8)
        w = int(pkt[6]) | int(pkt[7]) << 8
        h = int(pkt[8]) | int(pkt[9]) << 8
        self._L.RTjpeg_decompress(self._h, _u8(pkt), self._planes(planes, w, h))

    def decompress_n(self, pkt: np.ndarray, planes: np.ndarray) -> int:
        pkt = np.ascontiguousarray(pkt, dtype=np.uint8)
        if pkt.size < 12:
            return self._L.RTjpeg_b200_decompress_n(self._h, _u8(pkt), pkt.size, self._planes(planes, 0, 0))
        w = int(pkt[6]) | int(pkt[7]) << 8
        h = int(pkt[8]) | int(pkt[9]) << 8
        return self._L.RTjpeg_b200_decompress_n(self._h, _u8(pkt), pkt.size, self._planes(planes, w, h))

    def compress(self, planes: np.ndarray, w: int, h: int) -> np.ndarray:
        """RTjpeg_compress: one tight picture in the current format -> one packet."""
        fmt = getattr(self, "_fmt", 0)
        ysz = w * h
        csz = ysz // 4 if fmt == 0 else ysz // 2 if fmt == 1 else 0
        assert planes.dtype == np.uint8 and planes.flags.c_contiguous
        base = planes.ctypes.data
        pl = (_u8p * 3)(C.cast(base, _u8p), C.cast(base + ysz, _u8p), C.cast(base + ysz + csz, _u8p))
        out = np.zeros(12 + (w // 8) * (h // 8) * 2 * 64 + 64, dtype=np.uint8)
        n = self._L.RTjpeg_compress(self._h, _u8(out), pl)
        return out[:n].copy()

    def convert(self, kind: int, planes: np.ndarray, w: int, h: int, out: np.ndarray) -> None:
        """RTjpeg_yuv420rgb32 & co.: planes is one tight picture (Y|Cb|Cr), out a [h, pitch] byte array whose rows
        are handed over as the reference's `rows`."""
        assert planes.dtype == np.uint8 and planes.flags.c_contiguous and out.dtype == np.uint8 and out.ndim == 2
        ysz = w * h
        csz = 0 if kind == CONV_RGB8 else ysz // 2 if kind == CONV_YUV422_RGB24 else ysz // 4
        base = planes.ctypes.data
        pl = (_u8p * 3)(C.cast(base, _u8p), C.cast(base + ysz, _u8p), C.cast(base + ysz + csz, _u8p))
        rows = (_u8p * h)(*[C.cast(out[r].ctypes.data, _u8p) for r in range(h)])
        getattr(self._L, CONVERTERS[kind])(self._h, pl, rows)

    def last_error(self) -> int:
        return int(self._L.RTjpeg_b200_last_error(self._h))
