"""Device-side plumbing for the device-resident entry point (torch owns the memory).

PyTorch is used for exactly three things here: allocating HBM, host<->device
copies, and handing the current CUDA stream to the library.  No torch op touches
the pixel data.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import capi


@dataclass
class DeviceBatch:
    """One batch resident in HBM: packets, descriptors and the output frames."""
    stream: torch.Tensor      # uint8, packets back to back + STREAM_SLACK_BYTES of 0x7F
    desc: torch.Tensor        # uint8 view of rtjgpu_frame_desc[F]
    out: torch.Tensor         # uint8 [F, w*h*3/2]
    F: int
    w: int
    h: int
    payload_bytes: int        # sum over frames of (packet length - 12)
    fmt: int = 0              # RTJ_YUV420 / RTJ_YUV422 / RTJ_RGB8 (grey)

    @property
    def frame_bytes(self) -> int:
        return capi.frame_bytes(self.fmt, self.w, self.h)


def upload(stream: np.ndarray, desc: np.ndarray, w: int, h: int, device: int | str = 0,
           out: torch.Tensor | None = None, fmt: int = 0) -> DeviceBatch:
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    F = len(desc)
    host = np.full(stream.size + capi.STREAM_SLACK_BYTES, 0x7F, dtype=np.uint8)
    host[:stream.size] = stream
    d_stream = torch.from_numpy(host).to(dev)
    d_desc = torch.from_numpy(np.ascontiguousarray(desc).view(np.uint8).copy()).to(dev)
    if out is None:
        out = torch.empty((F, capi.frame_bytes(fmt, w, h)), dtype=torch.uint8, device=dev)
    payload = int(desc["length"].astype(np.int64).sum()) - 12 * F
    return DeviceBatch(d_stream, d_desc, out, F, w, h, payload, fmt)


def decode(ctx: capi.BatchContext, b: DeviceBatch, carry: torch.Tensor | None = None,
           stream: torch.cuda.Stream | None = None) -> None:
    """Launch K1/K3/K2 for the batch on `stream` (default: torch's current stream)."""
    st = stream if stream is not None else torch.cuda.current_stream(b.out.device)
    ctx.set_format(b.fmt)
    ctx.decode_device(b.stream.data_ptr(), b.desc.data_ptr(), b.F, b.w, b.h, b.out.data_ptr(),
                      None if carry is None else carry.data_ptr(), st.cuda_stream)


def upload_sequences(seqs, w: int, h: int, device: int | str = 0, fmt: int = 0, states=None, out: torch.Tensor | None = None):
    """Several independent packet sequences [(stream, offsets), ...] as one batch (capi.plan_sequences): each is planned
    with its own state (states: list of capi.State, advanced in place, or None).  out: as for upload() (a caller that only
    decodes selections, decode_select, may pass an empty tensor).  Returns (DeviceBatch, seq_first[S + 1])."""
    stream, _, desc, seq_first, _ = capi.plan_sequences(seqs, states)
    return upload(stream, desc, w, h, device=device, out=out, fmt=fmt), seq_first


def decode_sequences(ctx: capi.BatchContext, b: DeviceBatch, seq_first, carries=None,
                     stream: torch.cuda.Stream | None = None) -> None:
    """rtjgpu_decode_device_seq over a batch of upload_sequences: carries is a list of S tensors (the picture before each
    sequence) or None entries (zeros), or None."""
    st = stream if stream is not None else torch.cuda.current_stream(b.out.device)
    ctx.set_format(b.fmt)
    ptrs = None if carries is None else [None if c is None else c.data_ptr() for c in carries]
    ctx.decode_device_seq(b.stream.data_ptr(), b.desc.data_ptr(), b.F, b.w, b.h, list(seq_first), b.out.data_ptr(), ptrs,
                          st.cuda_stream)


def decode_select(ctx: capi.BatchContext, b: DeviceBatch, seq_first, sel, carries=None, out: torch.Tensor | None = None,
                  stream: torch.cuda.Stream | None = None) -> torch.Tensor:
    """rtjgpu_decode_device_select over a batch of upload_sequences: only the batch frames sel (strictly increasing; see
    capi.select_frames) are decoded, frame sel[k] to row k of the result.  carries as for decode_sequences.  out: a
    [n, frame_bytes] uint8 tensor to fill (default: a new one; b.out is not used).  Returns out."""
    st = stream if stream is not None else torch.cuda.current_stream(b.stream.device)
    sel = [int(x) for x in np.asarray(sel, dtype=np.int64).reshape(-1)]
    if out is None:
        out = torch.empty((len(sel), b.frame_bytes), dtype=torch.uint8, device=b.stream.device)
    assert out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= len(sel) * b.frame_bytes
    ctx.set_format(b.fmt)
    ptrs = None if carries is None else [None if c is None else c.data_ptr() for c in carries]
    ctx.decode_device_select(b.stream.data_ptr(), b.desc.data_ptr(), b.F, b.w, b.h, list(seq_first), sel,
                             out.data_ptr() if len(sel) else None, ptrs, st.cuda_stream)
    return out


def _window_args(seq_first, sel, size, origins, last):
    S = len(seq_first) - 1
    sel = [int(x) for x in np.asarray(sel, dtype=np.int64).reshape(-1)]
    cw, ch = int(size[0]), int(size[1])
    origins = [tuple(origins)] * S if np.ndim(origins) == 1 else [tuple(o) for o in origins]
    last_ptrs = None if last is None else [None if t is None else t.data_ptr() for t in last]
    return sel, cw, ch, origins, last_ptrs


def decode_window(ctx: capi.BatchContext, b: DeviceBatch, seq_first, sel, size, origins, carries=None, last=None,
                  out: torch.Tensor | None = None, stream: torch.cuda.Stream | None = None) -> torch.Tensor:
    """rtjgpu_decode_device_window over a batch of upload_sequences: the batch frames sel (as for decode_select), only a
    window of size = (cw, ch) pixels of each, at origins -- one (x, y) for every sequence, or S pairs.  Frame sel[k] goes
    to row k of the result as the tight planes of a cw x ch picture.  last: a list of S tensors (or None entries) that
    receive each sequence's last frame whole, as planes (the next call's carries), or None.  out: a [n, window_bytes]
    uint8 tensor to fill (default: a new one).  Returns out."""
    st = stream if stream is not None else torch.cuda.current_stream(b.stream.device)
    sel, cw, ch, origins, last_ptrs = _window_args(seq_first, sel, size, origins, last)
    if out is None:
        out = torch.empty((len(sel), capi.frame_bytes(b.fmt, cw, ch)), dtype=torch.uint8, device=b.stream.device)
    assert out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= len(sel) * capi.frame_bytes(b.fmt, cw, ch)
    ctx.set_format(b.fmt)
    ptrs = None if carries is None else [None if c is None else c.data_ptr() for c in carries]
    ctx.decode_device_window(b.stream.data_ptr(), b.desc.data_ptr(), b.F, b.w, b.h, list(seq_first), sel, (cw, ch), origins,
                             out.data_ptr() if len(sel) else None, ptrs, last_ptrs, st.cuda_stream)
    return out


def decode_rgb_window(ctx: capi.BatchContext, b: DeviceBatch, seq_first, sel, size, origins, kind: int, alpha: int = 255,
                      carries=None, last=None, out: torch.Tensor | None = None,
                      stream: torch.cuda.Stream | None = None) -> torch.Tensor:
    """rtjgpu_decode_device_rgb_window: decode_window with one of the reference's yuv420 converters (capi.CONV_RGB32 ...
    RGB16) fused in.  Returns a tight [n, ch, cw, bpp] uint8 tensor (out, if given, must be one), alpha in the fourth byte
    of 32-bit pixels.  YUV420 batches only."""
    st = stream if stream is not None else torch.cuda.current_stream(b.stream.device)
    sel, cw, ch, origins, last_ptrs = _window_args(seq_first, sel, size, origins, last)
    bpp = capi.CONV_BPP[kind]
    if out is None:
        out = torch.empty((len(sel), ch, cw, bpp), dtype=torch.uint8, device=b.stream.device)
    assert out.dtype == torch.uint8 and out.is_contiguous() and tuple(out.shape) == (len(sel), ch, cw, bpp)
    ctx.set_format(b.fmt)
    ptrs = None if carries is None else [None if c is None else c.data_ptr() for c in carries]
    ctx.decode_device_rgb_window(b.stream.data_ptr(), b.desc.data_ptr(), b.F, b.w, b.h, list(seq_first), sel, (cw, ch),
                                 origins, kind, out.data_ptr() if len(sel) else None, cw * bpp, ch * cw * bpp, alpha, ptrs,
                                 last_ptrs, st.cuda_stream)
    return out


def encode_sequences(ctx: capi.BatchContext, pictures, encoders, w: int, h: int, fmt: int = 0,
                     stream: torch.cuda.Stream | None = None):
    """rtjgpu_encode_device_seq: pictures a list of S uint8 device tensors (or views), each one sequence's consecutive
    tight w x h pictures of format fmt; encoders a list of S capi.SeqEncoder.  Returns (d_stream, d_offsets, seq_first,
    nbytes): the packets in a buffer sized by capi.encode_bound (plus STREAM_SLACK_BYTES, so that it can be decoded as
    it is), offsets[F + 1] on the device, seq_first[S + 1] and the bytes the packets take.  Waits for the encode."""
    assert len(pictures) == len(encoders) and len(pictures) > 0
    fsz = capi.frame_bytes(fmt, w, h)
    counts = []
    for p in pictures:
        assert p.dtype == torch.uint8 and p.is_contiguous() and p.numel() % fsz == 0, "tight pictures of the format"
        counts.append(p.numel() // fsz)
    seq_first = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    F = int(seq_first[-1])
    dev = pictures[0].device
    st = stream if stream is not None else torch.cuda.current_stream(dev)
    cap = capi.encode_bound(fmt, w, h, F)
    d_stream = torch.full((cap + capi.STREAM_SLACK_BYTES,), 0x7F, dtype=torch.uint8, device=dev)
    d_offsets = torch.empty(F + 1, dtype=torch.int64, device=dev)
    ctx.set_format(fmt)
    ctx.encode_device_seq(F, w, h, list(seq_first), [p.data_ptr() for p in pictures], encoders, d_stream.data_ptr(), cap,
                          d_offsets.data_ptr(), st.cuda_stream)
    nbytes, overflow = ctx.encode_info()
    assert not overflow, "rtjgpu_encode_bound was exceeded"
    return d_stream, d_offsets, seq_first, nbytes
