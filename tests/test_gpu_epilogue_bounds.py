"""The packed 16-bit epilogues of K2 (rtj_idct.cu: t2_pixels / m7_pixels behind t2_safe / m7_safe) are used where a
bound on the block's coefficients says that no pixel leaves 16..235 and nothing overflows its 16-bit half.  A bound is
not proved by samples: here the T2 class is swept EXHAUSTIVELY -- every DC byte 0..254 with every pair of coefficient
bytes -128..63 at zig-zag 1 and 2, under luma and under chroma tables, for several qualities and for custom tables
with large multipliers -- and the M7 class on more than 10^7 blocks whose DC runs over all 255 values for every
coefficient pattern (so both edges of the bound are crossed for each), all against the compiled reference
(lib/RTjpeg.c:157-186, :1196-1206, :2209-2332).

Layout trick: pictures are ONE macroblock wide (16 x 65520), so a macroblock row -- the unit K2's CTA works on, and
the unit within which a warp takes ONE epilogue flavour -- holds four luma and two chroma blocks.  All blocks under
test in a row carry the same DC and the same coefficient magnitudes (signs vary), so the warp's choice is exactly
the bound's verdict for that input: every input the bound accepts is computed by the packed arithmetic."""
import os

import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from streams import reference_frames_threaded

pytestmark = pytest.mark.gpu

W, ROWS = 16, 4095
H = ROWS * 16
FSZ = W * H * 3 // 2


def benign(iq0: int) -> np.ndarray:
    """A DC-only block (DC byte, then one run token for the other 63 positions) for the blocks that are not under test.
    They share the warp with the blocks that are, so they must not be what forces the warp off the packed path: a DC
    that dequantises to mid-range (x0 = DC * iq0 + 4 near 1000) wherever the table allows one."""
    return np.array([int(np.clip(round(1000 / iq0), 1, 254)), 0x7E], dtype=np.uint8)


def dc_multipliers(quality, raw_tables=None):
    t = O.tables_from_quality(quality) if raw_tables is None else O.tables_from_raw(raw_tables)
    assert t.lb8 == 0 and t.cb8 == 0
    return int(t.liqt[0]), int(t.ciqt[0])

COEF = np.arange(-128, 64, dtype=np.int16)               # a literal coefficient byte: -128..63 (64..127 are run tokens)


def build_stream(rows: np.ndarray, benign_row: np.ndarray, quality: int):
    R, L = rows.shape
    F = (R + ROWS - 1) // ROWS
    allrows = np.concatenate([rows, np.tile(benign_row, (F * ROWS - R, 1))]) if F * ROWS > R else rows
    size = 12 + ROWS * L
    slot = (size + 15) // 16 * 16
    stream = np.zeros(F * slot, dtype=np.uint8)
    view = stream.reshape(F, slot)
    hdr = np.zeros(12, dtype=np.uint8)
    hdr[0:4] = np.frombuffer(np.uint32(size).tobytes(), np.uint8)
    hdr[4] = 12
    hdr[6:8] = np.frombuffer(np.uint16(W).tobytes(), np.uint8)
    hdr[8:10] = np.frombuffer(np.uint16(H).tobytes(), np.uint8)
    hdr[10] = quality
    view[:, :12] = hdr
    view[:, 12:size] = allrows.reshape(F, ROWS * L)
    offsets = (np.arange(F + 1, dtype=np.uint64) * np.uint64(slot))
    return stream, offsets


def check_against_reference(stream, offsets, quality, raw_tables=None, chunk=96):
    """GPU decode of the whole batch, reference decode chunk by chunk; returns the number of rows compared."""
    F = len(offsets) - 1
    threads = min(len(os.sched_getaffinity(0)), 64)
    with g.BatchContext(0) as ctx:
        state = None
        if raw_tables is not None:
            ctx.set_custom_tables(raw_tables)
            state = capi.State(W, H, capi.TABLE_CUSTOM, 0)
        desc, _ = g.plan(stream, offsets, state)
        b = D.upload(stream, desc, W, H)
        b.out.fill_(0xCD)
        D.decode(ctx, b)
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
        for a in range(0, F, chunk):
            e = min(F, a + chunk)
            want = reference_frames_threaded(stream, np.ascontiguousarray(offsets[a:e + 1]),
                                             np.arange(e - a + 1, dtype=np.int32), W, H, threads, raw_tables=raw_tables)
            got = b.out[a:e].cpu().numpy()
            if not np.array_equal(got, want):
                f, o = np.argwhere(got != want)[0]
                plane = "Y" if o < W * H else "C"
                row = (o // (16 * 16)) if plane == "Y" else ((o - W * H) % (W * H // 4)) // (8 * 8)
                raise AssertionError(f"frame {a + f} offset {o} ({plane}, macroblock row {row}): got {got[f, o]} want {want[f, o]}")
    return F * ROWS


def t2_rows(luma: bool, iq0):
    """Every (DC, c1, c2): 255 x 192 x 192 rows.  The blocks under test: DC, c1, c2, run of 61.  iq0: the DC multipliers
    (luma, chroma) of the tables in force, for the blocks that are not under test."""
    BL, BC = benign(iq0[0]), benign(iq0[1])
    dc = np.arange(255, dtype=np.uint8)
    c = COEF.astype(np.int8).view(np.uint8)
    DC, C1, C2 = np.meshgrid(dc, c, c, indexing="ij")
    n = DC.size
    blk = np.empty((n, 4), dtype=np.uint8)
    blk[:, 0] = DC.ravel(); blk[:, 1] = C1.ravel(); blk[:, 2] = C2.ravel(); blk[:, 3] = 63 + 61
    if luma:
        ben = np.tile(BC, (n, 1))
        # the four luma blocks of a row: (c1, c2), (c1, -c2), (-c1, c2), (-c1, -c2) where the negation is a literal too
        def neg(x):
            v = x.view(np.int8).astype(np.int16)
            m = np.where((-v >= -128) & (-v <= 63), -v, v)
            return m.astype(np.int8).view(np.uint8)
        b1 = blk.copy(); b1[:, 2] = neg(blk[:, 2])
        b2 = blk.copy(); b2[:, 1] = neg(blk[:, 1])
        b3 = b2.copy(); b3[:, 2] = neg(blk[:, 2])
        rows = np.concatenate([blk, b1, b2, b3, ben, ben], axis=1)
        benign_row = np.concatenate([[BL[0], 0, 0, 63 + 61]] * 4 + [BC] * 2).astype(np.uint8)
    else:
        ben = np.tile(BL, (n, 1))
        b1 = blk.copy()
        rows = np.concatenate([ben, ben, ben, ben, blk, b1], axis=1)
        benign_row = np.concatenate([BL] * 4 + [[BC[0], 0, 0, 63 + 61]] * 2).astype(np.uint8)
    return rows, benign_row


CUSTOM = {
    # raw (pre-AAN) tables, lib/RTjpeg.c:2380-2395; entry 8 is zig-zag 1 and must exceed 8 or a raw prefix appears
    "wide_dc": dict(dc=7, c=30),        # x0 = 7 DC + 4 spans almost exactly the legal range; large coefficient steps
    "coarse": dict(dc=40, c=200),       # products that wrap the int16 of the dequantiser (lib/RTjpeg.c:170-180)
}


def custom_raw(dc, c):
    raw = np.full(128, c, dtype=np.uint32)
    raw[0] = raw[64] = dc
    return raw


@pytest.mark.parametrize("luma", [True, False], ids=["luma", "chroma"])
@pytest.mark.parametrize("quality", [1, 32, 128, 170])
def test_t2_exhaustive(quality, luma):
    rows, pad = t2_rows(luma, dc_multipliers(quality))
    stream, offsets = build_stream(rows, pad, quality)
    assert check_against_reference(stream, offsets, quality) >= 255 * 192 * 192


@pytest.mark.parametrize("luma", [True, False], ids=["luma", "chroma"])
@pytest.mark.parametrize("name", sorted(CUSTOM))
def test_t2_exhaustive_custom_tables(name, luma):
    raw = custom_raw(**CUSTOM[name])
    rows, pad = t2_rows(luma, dc_multipliers(0, raw))
    stream, offsets = build_stream(rows, pad, 0)
    assert check_against_reference(stream, offsets, 0, raw_tables=raw) >= 255 * 192 * 192


def m7_rows(rng, nsets, luma, iq0):
    """nsets coefficient patterns (six magnitudes for zig-zag 1..6, mostly small, some large, a few extreme) times all 255
    DC bytes; the blocks of a row share DC and magnitudes and differ in signs.  Block: DC, c1..c6, run of 57."""
    kind = rng.random(nsets)
    mag = np.where(kind[:, None] < 0.6, rng.integers(0, 6, (nsets, 6)),
                   np.where(kind[:, None] < 0.9, rng.integers(0, 40, (nsets, 6)), rng.integers(0, 129, (nsets, 6))))
    mag[:, 3:] = np.maximum(mag[:, 3:], 1 * (rng.random((nsets, 3)) < 0.7))          # keep E > 3 for most rows: the M7 class
    nb = 4 if luma else 2
    dc = np.arange(255, dtype=np.uint8)
    n = nsets * 255
    blocks = []
    for _ in range(nb):
        sign = rng.integers(0, 2, (nsets, 6)) * 2 - 1
        v = mag * sign
        v = np.where(v > 63, -v, v)                                                   # +64..+128 is not a literal: take the negative
        v = np.clip(v, -128, 63).astype(np.int8).view(np.uint8)
        blk = np.empty((nsets, 255, 8), dtype=np.uint8)
        blk[:, :, 0] = dc[None, :]
        blk[:, :, 1:7] = v[:, None, :]
        blk[:, :, 7] = 63 + 57
        blocks.append(blk.reshape(n, 8))
    BL, BC = benign(iq0[0]), benign(iq0[1])
    if luma:
        ben = np.tile(BC, (n, 1))
        rows = np.concatenate(blocks + [ben, ben], axis=1)
        benign_row = np.concatenate([[BL[0], 0, 0, 0, 0, 0, 1, 63 + 57]] * 4 + [BC] * 2).astype(np.uint8)
    else:
        ben = np.tile(BL, (n, 1))
        rows = np.concatenate([ben] * 4 + blocks, axis=1)
        benign_row = np.concatenate([BL] * 4 + [[BC[0], 0, 0, 0, 0, 0, 1, 63 + 57]] * 2).astype(np.uint8)
    return rows, benign_row


@pytest.mark.parametrize("quality,luma,nsets", [(128, True, 10400), (32, True, 2000), (170, True, 2000), (1, True, 1000),
                                                (128, False, 6000), (32, False, 2000)])
def test_m7_dc_sweeps(quality, luma, nsets):
    rng = np.random.default_rng(1000 * quality + luma)
    rows, pad = m7_rows(rng, nsets, luma, dc_multipliers(quality))
    stream, offsets = build_stream(rows, pad, quality)
    check_against_reference(stream, offsets, quality)


def test_m7_custom_tables():
    rng = np.random.default_rng(77)
    raw = custom_raw(**CUSTOM["wide_dc"])
    rows, pad = m7_rows(rng, 3000, True, dc_multipliers(0, raw))
    stream, offsets = build_stream(rows, pad, 0)
    check_against_reference(stream, offsets, 0, raw_tables=raw)
