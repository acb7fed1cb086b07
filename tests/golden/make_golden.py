#!/usr/bin/env python3
"""Generate tests/golden/*.npz from the UNMODIFIED reference.

Run in the authoring container, where /root/reference is mounted:

    python tests/golden/make_golden.py

Every expected output in the fixtures comes from the reference's own
RTjpeg_decompress (lib/RTjpeg.c:3565) / RTjpeg_set_quality+get_tables
(:2408, :2371), compiled by oracle/Makefile into oracle/_ref/.  Streams come
from the reference's own RTjpeg_compress (:3488, through oracle.ref_encode_clip
and ref_encode_clip_fmt) fed by the seeded synthetic source in
oracle/rtjo_driver.c, or -- for the `random_*` cases -- from the grammar-only
packet generator in oracle/oracle.py (no codec arithmetic).  Never from the
restated encoder: these streams are what pins it.
The reference ships no fixtures of its own (SURVEY.md section 4); these files
are the pin.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def clip_case(name, w, h, Q, F, key_rate=-1, lm=0, cm=0, noise_y=2, noise_c=0, dark=0, seed=1,
              init_fill=0, keep_planes=True):
    clip = O.make_clip(w, h, Q, key_rate, lm, cm, noise_y=noise_y, noise_c=noise_c, dark=dark, seed=seed)
    stream, offs = O.ref_encode_clip(clip, F)
    init = np.full(w * h * 3 // 2, init_fill, dtype=np.uint8)
    frames = O.ref_decode_seq(stream, offs, w, h, init=init)
    d = dict(stream=stream, offsets=offs, w=w, h=h, Q=Q, init_fill=init_fill,
             sha=np.array([sha(f) for f in frames]))
    if keep_planes:
        d["frames"] = frames
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print(f"{name}: {F} frames, {stream.size} stream bytes")


def random_case(name, w, h, qualities, per_q=2, seed=5):
    rng = np.random.default_rng(seed)
    pkts = []
    for q in qualities:
        for i in range(per_q):
            pkts.append(O.random_wellformed_packet(rng, w, h, q, skip_prob=0.2 if i else 0.0))
    stream, offs = O.pack_packets(pkts)
    init = np.full(w * h * 3 // 2, 0x55, dtype=np.uint8)
    frames = O.ref_decode_seq(stream, offs, w, h, init=init)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), stream=stream, offsets=offs, w=w, h=h,
                        init_fill=0x55, frames=frames, sha=np.array([sha(f) for f in frames]),
                        qualities=np.repeat(np.array(qualities), per_q))
    print(f"{name}: {len(pkts)} packets, {stream.size} stream bytes")


def tables_case():
    tabs = np.stack([O.ref_tables_for_quality(q) for q in range(1, 256)])   # [255, 128] AAN-scaled
    # lb8/cb8 are private to the reference; they are observable through the stream grammar,
    # so the fixture records what the restatement derives and test_oracle re-checks it by
    # decoding (random_* cases cover every raw-prefix class)
    np.savez_compressed(os.path.join(OUT, "tables.npz"), tables=tabs)
    print("tables: 255 x 128")


def set_tables_case(seed=11):
    """The set_tables path (NUV 'D'/'R' extradata): raw tables, quality byte 0."""
    rng = np.random.default_rng(seed)
    w, h = 48, 32
    cases = []
    for variant in range(3):
        raw = rng.integers(1, 40, size=128).astype(np.uint32)
        if variant == 1:
            # every multiplier <= 8 except the last zig-zag position: raw prefix of 62 bytes.
            # (A table that is <= 8 EVERYWHERE makes the reference's unbounded scan,
            # lib/RTjpeg.c:2388-2393, read past RTjpeg_ZZ[63]: undefined there, not pinned.)
            raw[:] = rng.integers(1, 9, size=128)
            raw[63] = 20
            raw[127] = 20
        if variant == 2:
            raw[:64] = rng.integers(9, 200, size=64)     # lb8 = 0
        t = O.tables_from_raw(raw)
        # build a packet with that grammar (quality byte 0 keeps the custom tables in force)
        nmb = (w // 16) * (h // 16)
        body = bytearray(12)
        for mb in range(nmb):
            for k in range(6):
                bt8 = t.lb8 if k < 4 else t.cb8
                body.append(int(rng.integers(0, 255)))
                for _ in range(bt8):
                    body.append(int(rng.integers(-128, 128)) & 0xFF)
                pos = 1 + bt8
                while pos < 64:
                    if rng.random() < 0.5:
                        run = int(rng.integers(1, 64 - pos + 1))
                        body.append(63 + run)
                        pos += run
                    else:
                        body.append(int(rng.integers(-20, 21)) & 0xFF)
                        pos += 1
        pkt = np.frombuffer(bytes(body), dtype=np.uint8).copy()
        pkt[0:4] = np.frombuffer(np.uint32(pkt.size).tobytes(), dtype=np.uint8)
        pkt[4] = 12
        pkt[6:8] = np.frombuffer(np.uint16(w).tobytes(), dtype=np.uint8)
        pkt[8:10] = np.frombuffer(np.uint16(h).tobytes(), dtype=np.uint8)
        pkt[10] = 0
        planes = O.ref_decode_with_tables(raw, pkt, w, h, np.full(w * h * 3 // 2, 0x33, dtype=np.uint8))
        cases.append((raw, pkt, planes))
    np.savez_compressed(os.path.join(OUT, "set_tables.npz"), w=w, h=h, init_fill=0x33,
                        **{f"raw{i}": c[0] for i, c in enumerate(cases)},
                        **{f"pkt{i}": c[1] for i, c in enumerate(cases)},
                        **{f"planes{i}": c[2] for i, c in enumerate(cases)})
    print("set_tables: 3 cases")


def fmt_case(name, fmt, w, h, Q, F, key_rate=-1, lm=0, cm=0, init_fill=0, **kw):
    """YUV422 (fmt 1) and 8-bit grey (fmt 2): the other two branches of RTjpeg_decompress (:3580-3585)."""
    stream, offs = O.ref_encode_clip_fmt(w, h, Q, F, fmt, key_rate, lm, cm, **kw)
    init = np.full(O.frame_bytes(fmt, w, h), init_fill, dtype=np.uint8)
    frames = O.ref_decode_seq_fmt(stream, offs, w, h, fmt, init=init)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), stream=stream, offsets=offs, w=w, h=h, Q=Q, fmt=fmt,
                        init_fill=init_fill, frames=frames, sha=np.array([sha(f) for f in frames]))
    print(f"{name}: {F} frames, {stream.size} stream bytes")


def convert_case(seed=21):
    """The colour converters (lib/RTjpeg.c:3077-3486) over one full-range random picture per chroma layout."""
    rng = np.random.default_rng(seed)
    w, h = 48, 32
    pic420 = rng.integers(0, 256, w * h * 3 // 2).astype(np.uint8)
    pic422 = rng.integers(0, 256, w * h * 2).astype(np.uint8)
    names = ["rgb32", "bgr32", "rgb24", "bgr24", "rgb16", "rgb8", "yuv422rgb24"]
    d = {n: O.ref_convert(k, pic422 if k == O.CONV_YUV422_RGB24 else pic420, w, h, fill=0x5A) for k, n in enumerate(names)}
    np.savez_compressed(os.path.join(OUT, "convert_48x32.npz"), pic420=pic420, pic422=pic422,
                        sha420=hashlib.sha256(pic420.tobytes()).hexdigest()[:16], **d)
    print("convert_48x32: 7 converters")


def encode_case():
    """RTjpeg_compress (lib/RTjpeg.c:3488) over a short clip in both chroma layouts: the reference's packets, byte for byte."""
    w, h, Q, kr, lm = 64, 48, 171, 3, 2
    s, o = O.ref_encode_clip(O.make_clip(w, h, 255, noise_y=20, noise_c=6, dark=1), 7)
    yuv = O.ref_decode_seq(s, o, w, h)
    d = dict(Q=Q, key_rate=kr, lm=lm, cm=lm)
    for fmt, key in ((0, "420"), (1, "422")):
        pics = O.frames_in_format(yuv, w, h, fmt)
        pics = np.concatenate([pics, pics[-1:]])
        st, of = O.encode_frames_fmt(O.make_clip(w, h, Q, kr, lm, lm), fmt, pics)
        d["pics" + key], d["stream" + key], d["offsets" + key] = pics, st, of
    np.savez_compressed(os.path.join(OUT, "encode_64x48.npz"), **d)
    print("encode_64x48: 8 pictures x 2 formats")


if __name__ == "__main__":
    O.build()
    assert O.have_ref(), "needs /root/reference"
    clip_case("intra_64x48_q128", 64, 48, 128, 4, noise_y=6, noise_c=3)
    clip_case("intra_320x240_q128", 320, 240, 128, 2, keep_planes=False)          # configs[0] geometry
    clip_case("inter_64x48_q200_gop6", 64, 48, 200, 14, key_rate=5, lm=2, cm=2, noise_y=30, noise_c=8,
              init_fill=0x55)
    clip_case("inter_dark_96x64_q32_gop4", 96, 64, 32, 10, key_rate=3, lm=4, cm=4, dark=1, init_fill=0x55)
    clip_case("dense_48x32_q255", 48, 32, 255, 3, noise_y=110, noise_c=90)
    random_case("random_48x32", 48, 32, [1, 32, 170, 171, 200, 228, 255])
    tables_case()
    set_tables_case()
    convert_case()
    encode_case()
    fmt_case("yuv422_inter_64x48_q200_gop4", 1, 64, 48, 200, 9, key_rate=3, lm=2, cm=2, noise_y=30, noise_c=8, init_fill=0x55)
    fmt_case("yuv422_intra_96x32_q128", 1, 96, 32, 128, 3, noise_y=6, noise_c=3)
    fmt_case("grey_inter_64x48_q255_gop4", 2, 64, 48, 255, 9, key_rate=3, lm=2, cm=2, noise_y=40, init_fill=0x55)
    fmt_case("grey_intra_96x32_q64", 2, 96, 32, 64, 3, noise_y=6)
