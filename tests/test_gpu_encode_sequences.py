"""rtjgpu_encode_device_seq: many independent streams encoded in one device batch, each with an encoder state (rtjgpu_seqenc)
of its own.  Expected packets: every sequence encoded on its own by the reference's RTjpeg_compress where it is built, else
by the restatement, with that sequence's history -- byte for byte, sequence by sequence."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from oracle import oracle as O
from gpu_util import first_diff
from streams import clip, reference_frames

pytestmark = pytest.mark.gpu

W, H = 96, 64


def _pictures(fmt, w, h, n=12, seed=5):
    """A moving synthetic clip, then one full-range random picture and a repeated picture (every block skipped)."""
    rng = np.random.default_rng(seed)
    s, o = O.encode_clip(O.make_clip(w, h, 255, noise_y=20, noise_c=6, dark=1, seed=seed), n, threads=1)
    fr = O.frames_in_format(reference_frames(s, o, w, h), w, h, fmt)
    return np.concatenate([fr, rng.integers(0, 256, (1, fr.shape[1])).astype(np.uint8), fr[-1:], fr[-1:]])


def _packets(stream, offsets):
    """Every packet's bytes, framesize long (what RTjpeg_compress returned for it)."""
    sizes = O.packet_sizes(stream, offsets)
    return [np.asarray(stream[int(offsets[f]):int(offsets[f]) + int(sizes[f])]) for f in range(len(offsets) - 1)]


def _want(fr, w, h, fmt, Q, kr, lm):
    """One sequence encoded from a fresh instance: RTjpeg_set_quality(Q), RTjpeg_set_intra(kr, lm, lm) -> packets."""
    if O.have_ref():
        s, o = O.encode_frames_fmt(O.make_clip(w, h, Q, kr if kr else -1, lm, lm), fmt, fr, align=4)
    else:
        s, o = O.encode_frames_oracle(fr, w, h, fmt, Q, kr, lm, lm, align=4)
    return _packets(s, o)


def _encode(ctx, pics, encs, w=W, h=H, fmt=0):
    """encode_sequences -> list of S packet lists, checking the layout: packets back to back on multiples of 4, padding 0."""
    d_stream, d_off, sf, nbytes = D.encode_sequences(ctx, [torch.from_numpy(np.ascontiguousarray(p)).cuda() if isinstance(p, np.ndarray)
                                                           else p for p in pics], encs, w, h, fmt)
    s = d_stream.cpu().numpy()
    o = d_off.cpu().numpy().astype(np.uint64)
    assert o[0] == 0 and int(o[-1]) == nbytes and (o % 4 == 0).all()
    sizes = O.packet_sizes(s, o).astype(np.int64)
    assert np.array_equal(np.diff(o.astype(np.int64)), (sizes + 3) // 4 * 4)
    for f in range(len(o) - 1):
        assert not s[int(o[f]) + int(sizes[f]):int(o[f + 1])].any()
    pk = _packets(s, o)
    return [pk[int(sf[i]):int(sf[i + 1])] for i in range(len(sf) - 1)]


def _same(got, want, what=""):
    assert len(got) == len(want), (what, len(got), len(want))
    for f, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), f"{what}: packet {f} differs ({a.size} vs {b.size} bytes)"


def _next_count(c, kr, n):
    for _ in range(n if kr else 0):
        c = 0 if c + 1 > kr else c + 1
    return c


# (Q, key_rate, lm, first picture, pictures): intra; GOP 6 over 14 pictures; raw prefix (Q255) over the random and the
# repeated pictures; masks 16 with key_rate 255; one picture; 13 pictures at GOP 5
SPECS = [(128, 0, 0, 0, 9), (200, 5, 2, 0, 14), (255, 3, 1, 3, 12), (171, 255, 16, 0, 10), (64, 2, 6, 7, 1), (32, 4, 2, 2, 13)]


@pytest.mark.parametrize("fmt", [0, 1])
def test_sequences_one_call(fmt):
    pics = _pictures(fmt, W, H)
    with g.BatchContext(0) as ctx:
        encs = [ctx.seq_encoder(Q, kr, lm, lm) for Q, kr, lm, _, _ in SPECS]
        got = _encode(ctx, [pics[a:a + n] for _, _, _, a, n in SPECS], encs, fmt=fmt)
        for i, (Q, kr, lm, a, n) in enumerate(SPECS):
            _same(got[i], _want(pics[a:a + n], W, H, fmt, Q, kr, lm), f"sequence {i}")
            assert encs[i].key_count == _next_count(0, kr, n)


def test_state_carries_across_calls():
    """Every handle's sequence split at its own places over several calls; handles absent from some calls, the order of
    the handles changing from call to call.  The packets put together are those of one pass."""
    pics = _pictures(0, W, H)
    N = pics.shape[0]
    settings = [(200, 5, 2), (128, 0, 0), (255, 3, 1), (64, 29, 3)]
    cuts = {0: [0, 5, 9, N], 1: [0, 7, N], 2: [0, 1, N], 3: [0, N]}
    calls = [[2, 0, 1], [0, 3], [1, 0, 2]]
    with g.BatchContext(0) as ctx:
        encs = [ctx.seq_encoder(*s, s[2]) for s in settings]
        done = {i: 0 for i in cuts}
        got = {i: [] for i in cuts}
        for order in calls:
            pieces = []
            for i in order:
                a, b = cuts[i][done[i]], cuts[i][done[i] + 1]
                pieces.append(pics[a:b])
            out = _encode(ctx, pieces, [encs[i] for i in order])
            for i, pk in zip(order, out):
                got[i] += pk
                done[i] += 1
                n = cuts[i][done[i]]
                assert encs[i].key_count == _next_count(0, settings[i][1], n), (i, n)
        for i, (Q, kr, lm) in enumerate(settings):
            assert done[i] == len(cuts[i]) - 1
            _same(got[i], _want(pics, W, H, 0, Q, kr, lm), f"handle {i}")


def _ctx_encode(ctx, fr, w=W, h=H):
    F = fr.shape[0]
    cap = g.encode_bound(0, w, h, F)
    d_fr = torch.from_numpy(np.ascontiguousarray(fr)).cuda()
    d_stream = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(F + 1, dtype=torch.int64, device="cuda")
    ctx.encode_device(d_fr.data_ptr(), F, w, h, d_stream.data_ptr(), cap, d_off.data_ptr(), torch.cuda.current_stream().cuda_stream)
    nbytes, overflow = ctx.encode_info()
    assert not overflow
    return _packets(d_stream[:nbytes].cpu().numpy(), d_off.cpu().numpy().astype(np.uint64))


def test_settings_between_calls_match_context_encoder():
    """set_quality / set_intra / reset between calls on one handle (a second handle goes along untouched): the packets
    of the context's own encoder doing the same."""
    pics = _pictures(0, W, H, n=20)
    steps = [(6, None), (3, ("quality", 64)), (4, ("intra", 3, 1, 1)), (3, ("reset",)), (2, ("quality", 255)),
             (2, ("intra", 0, 0, 0)), (3, ("intra", 7, 2, 2))]
    L = capi.load_library()
    with g.BatchContext(0) as ref, g.BatchContext(0) as ctx:
        ref.encoder_config(200, 5, 2, 2)
        e = ctx.seq_encoder(200, 5, 2, 2)
        other = ctx.seq_encoder(128, 9, 1, 1)
        at, want_other, got_other = 0, [], []
        for n, op in steps:
            if op and op[0] == "quality":
                L.rtjgpu_encoder_set_quality(ref._h, op[1])
                e.set_quality(op[1])
            elif op and op[0] == "intra":
                L.rtjgpu_encoder_set_intra(ref._h, *op[1:])
                e.set_intra(*op[1:])
            elif op and op[0] == "reset":
                L.rtjgpu_encoder_reset(ref._h)
                e.reset()
            fr = pics[at:at + n]
            want = _ctx_encode(ref, fr)
            got, go = _encode(ctx, [fr, pics[at:at + n][::-1].copy()], [e, other])
            _same(got, want, f"after {op}")
            got_other += go
            want_other.append(pics[at:at + n][::-1])
            at += n
        _same(got_other, _want(np.concatenate(want_other), W, H, 0, 128, 9, 1), "untouched handle")


def test_no_leak_between_handles():
    """Two inter sequences at different qualities, each picture the other's last: where a handle would compare with the
    other's stored blocks, blocks would be skipped that must be coded (and the other way round)."""
    pics = _pictures(0, W, H)
    x, y = pics[2].copy(), pics[2].copy()
    y[:W * H // 2] = pics[9][:W * H // 2]               # the upper half of the luma differs
    with g.BatchContext(0) as ctx:
        a, b = ctx.seq_encoder(200, 30, 2, 2), ctx.seq_encoder(64, 30, 2, 2)
        g1 = _encode(ctx, [x[None], y[None]], [a, b])
        g2 = _encode(ctx, [y[None], x[None]], [b, a])        # order swapped: b now encodes y again, a x
        g3 = _encode(ctx, [y[None], x[None]], [a, b])
    _same(g1[0] + g2[1] + g3[0], _want(np.stack([x, x, y]), W, H, 0, 200, 30, 2), "a")
    _same(g1[1] + g2[0] + g3[1], _want(np.stack([y, y, x]), W, H, 0, 64, 30, 2), "b")
    # the last picture of each sequence differs from its own stored blocks: no block of the changed half is skipped
    assert g3[0][0].size > g2[1][0].size and g3[1][0].size > g2[0][0].size


@pytest.mark.parametrize("fmt,Q,kr,lm", [(0, 200, 5, 2), (1, 128, 4, 2), (0, 255, 0, 0), (1, 32, 255, 16)])
def test_one_sequence_equals_encode_device(fmt, Q, kr, lm):
    pics = _pictures(fmt, W, H)
    with g.BatchContext(0) as ref, g.BatchContext(0) as ctx:
        ref.encoder_config(Q, kr, lm, lm)
        ref.set_format(fmt)
        e = ctx.seq_encoder(Q, kr, lm, lm)
        for a, b in ((0, 4), (4, pics.shape[0])):
            cap = g.encode_bound(fmt, W, H, b - a)
            d_fr = torch.from_numpy(pics[a:b].copy()).cuda()
            d_s = torch.zeros(cap, dtype=torch.uint8, device="cuda")
            d_o = torch.zeros(b - a + 1, dtype=torch.int64, device="cuda")
            ref.encode_device(d_fr.data_ptr(), b - a, W, H, d_s.data_ptr(), cap, d_o.data_ptr(), torch.cuda.current_stream().cuda_stream)
            nb, _ = ref.encode_info()
            d_stream, d_off, _, nbytes = D.encode_sequences(ctx, [d_fr], [e], W, H, fmt)
            assert nbytes == nb
            assert torch.equal(d_off, d_o) and torch.equal(d_stream[:nb], d_s[:nb])


def test_rate_ladder_one_picture_pointer():
    pics = _pictures(0, W, H)
    d = torch.from_numpy(pics).cuda()
    ladder = [(32, 5, 2), (128, 5, 2), (255, 5, 2)]
    with g.BatchContext(0) as ctx:
        encs = [ctx.seq_encoder(Q, kr, lm, lm) for Q, kr, lm in ladder]
        got = _encode(ctx, [d, d, d], encs)
    for (Q, kr, lm), pk in zip(ladder, got):
        _same(pk, _want(pics, W, H, 0, Q, kr, lm), f"Q{Q}")


def test_transcode_round_trip_on_device():
    """decode_sequences -> encode_sequences at another quality -> per-sequence plan -> decode_sequences.  Only packets and
    offsets visit the host; the result equals the reference decoding the reference's re-encode of its own decode."""
    w, h = 160, 96
    srcs = [clip(w, h, 128, 17, key_rate=14, lm=2, cm=2, dark=1, seed=1), clip(w, h, 200, 9, key_rate=4, lm=2, cm=2, seed=3),
            clip(w, h, 64, 1, seed=4)]
    Q, kr, lm = 64, 9, 2
    with g.BatchContext(0) as ctx:
        b, sf = D.upload_sequences(srcs, w, h)
        D.decode_sequences(ctx, b, sf)
        encs = [ctx.seq_encoder(Q, kr, lm, lm) for _ in srcs]
        d_stream, d_off, sf2, nbytes = D.encode_sequences(ctx, [b.out[int(sf[i]):int(sf[i + 1])] for i in range(len(srcs))], encs, w, h)
        assert list(sf2) == list(sf)
        host = d_stream[:nbytes].cpu().numpy()
        offs = d_off.cpu().numpy().astype(np.uint64)
        desc = np.concatenate([g.plan(host, offs[sf[i]:sf[i + 1] + 1])[0] for i in range(len(srcs))])
        F = int(sf[-1])
        out = torch.full((F, w * h * 3 // 2), 0xCD, dtype=torch.uint8, device="cuda")
        b2 = D.DeviceBatch(d_stream, torch.from_numpy(desc.view(np.uint8).copy()).cuda(), out, F, w, h, 0)
        D.decode_sequences(ctx, b2, sf2)
        torch.cuda.synchronize()
        got = out.cpu().numpy()
    want = []
    for s, o in srcs:
        fr = reference_frames(s, o, w, h)
        ws, wo = (O.encode_frames_fmt(O.make_clip(w, h, Q, kr, lm, lm), 0, fr) if O.have_ref()
                  else O.encode_frames_oracle(fr, w, h, 0, Q, kr, lm, lm))
        want.append(reference_frames(ws, wo, w, h))
    want = np.concatenate(want)
    assert np.array_equal(got, want), first_diff(got, want, w, h)


def test_many_sequences_at_scale():
    """720x576, 64 sequences of 8 pictures at GOP 30, every handle warmed to a different key phase first."""
    w, h, S, k, kr, lm, Q = 720, 576, 64, 8, 29, 2, 128
    pool = _pictures(0, w, h, n=20, seed=3)
    warm = [(7 * s) % 30 for s in range(S)]
    first = [s % (pool.shape[0] - k) for s in range(S)]
    seqs = [np.concatenate([pool[::-1]] * 3)[:warm[s]] for s in range(S)]
    with g.BatchContext(0) as ctx:
        encs = [ctx.seq_encoder(Q, kr, lm, lm) for _ in range(S)]
        warmed = [s for s in range(S) if warm[s]]
        _encode(ctx, [seqs[s] for s in warmed], [encs[s] for s in warmed], w, h)
        got = _encode(ctx, [pool[first[s]:first[s] + k] for s in range(S)], encs, w, h)
        for s in range(S):
            assert encs[s].key_count == (warm[s] + k) % 30
    for s in range(0, S, 3):                 # every third sequence against its one-pass expectation
        want = _want(np.concatenate([seqs[s], pool[first[s]:first[s] + k]]), w, h, 0, Q, kr, lm)
        _same(got[s], want[warm[s]:], f"sequence {s}")


def test_overflow_writes_nothing_and_state_advances():
    pics = _pictures(0, W, H)
    with g.BatchContext(0) as ctx:
        e1, e2 = ctx.seq_encoder(200, 5, 2, 2), ctx.seq_encoder(128, 0, 0, 0)
        d = torch.from_numpy(pics).cuda()
        d_stream = torch.full((256,), 0xEE, dtype=torch.uint8, device="cuda")
        d_off = torch.zeros(2 * 4 + 1, dtype=torch.int64, device="cuda")
        ctx.encode_device_seq(8, W, H, [0, 4, 8], [d.data_ptr(), d.data_ptr()], [e1, e2], d_stream.data_ptr(), 256,
                              d_off.data_ptr(), torch.cuda.current_stream().cuda_stream)
        nbytes, overflow = ctx.encode_info()
        assert overflow and nbytes > 256
        assert (d_stream.cpu().numpy() == 0xEE).all()
        assert e1.key_count == 4 and e2.key_count == 0
        got = _encode(ctx, [pics[4:], pics[4:]], [e1, e2])
    _same(got[0], _want(pics, W, H, 0, 200, 5, 2)[4:], "inter")
    _same(got[1], _want(pics, W, H, 0, 128, 0, 0)[4:], "intra")


def test_argument_errors_launch_nothing():
    pics = _pictures(0, W, H, n=4)
    d = torch.from_numpy(pics).cuda()
    p = d.data_ptr()
    cap = g.encode_bound(0, W, H, 6)
    d_stream = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(7, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    with g.BatchContext(0) as ctx, g.BatchContext(0) as other:
        a, b = ctx.seq_encoder(128, 5, 2, 2), ctx.seq_encoder(64)
        foreign = other.seq_encoder(128)

        def call(first, frames, encs, fmt=0):
            ctx.set_format(fmt)
            try:
                ctx.encode_device_seq(6, W, H, first, frames, encs, d_stream.data_ptr(), cap, d_off.data_ptr(), st)
            except g.RTjpegError as e:
                return e.code
            finally:
                ctx.set_format(0)
            return 0

        n0 = ctx.launch_count()
        assert call([0, 3, 6], [p, p], [a, a]) == capi.E_ARG                   # one handle twice
        assert call([0, 3, 6], [p, p], [a, foreign]) == capi.E_ARG             # a handle of another context
        assert call([0, 3, 6], [p, p], [a, None]) == capi.E_ARG                # no handle
        assert call([1, 3, 6], [p, p], [a, b]) == capi.E_ARG                   # seq_first[0] != 0
        assert call([0, 3, 5], [p, p], [a, b]) == capi.E_ARG                   # seq_first[S] != F
        assert call([0, 3, 3, 6], [p, p, p], [a, b, foreign]) == capi.E_ARG    # an empty sequence
        assert call([0, 6, 3], [p, p], [a, b]) == capi.E_ARG                   # not increasing
        assert call([0, 3, 6], [p, None], [a, b]) == capi.E_ARG                # no pictures
        assert call([0, 3, 6], [p, p + 4], [a, b]) == capi.E_ARG               # pictures not 8-byte aligned
        assert call([0, 3, 6], [p, p], [a, b], fmt=2) == capi.E_FORMAT         # the grey format
        assert ctx.launch_count() == n0
        assert a.key_count == 0 and b.key_count == 0
        assert call([0, 3, 6], [p, p], [a, b]) == 0
        assert ctx.launch_count() > n0 and a.key_count == 3
        foreign.close()
