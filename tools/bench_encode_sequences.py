#!/usr/bin/env python3
"""Many independent streams encoded per device batch: rtjgpu_encode_device_seq against one call per stream.

Pictures: two 720x576 YUV420 clips coded at Q=128 (GOP 30), decoded on the device.  Sequence s takes k consecutive
pictures of one of them, starting anywhere, and is encoded again at Q=128, GOP 30, lm = cm = 2 (the intra line: key_rate
0) by a handle of its own, every handle first warmed by (7 s) % 30 pictures so that the key phases differ.  For each
layout S x k it reports pictures/s of
  seq      one rtjgpu_encode_device_seq call
  calls    S rtjgpu_encode_device_seq calls of one sequence each, on the same stream, with the same handles
  ceiling  the same S * k pictures as ONE stream (one buffer) in one rtjgpu_encode_device call: about the same work,
           what one call could at best reach
and a transcode line: rtjgpu_decode_device_seq of the S source sequences, then rtjgpu_encode_device_seq of what it wrote.
Pictures, packets and offsets stay in HBM.  Times: CUDA events around `steps` passes after `warmup` passes.  Prints one
JSON line with the card's name and power limit.

    python tools/bench_encode_sequences.py [--layouts 512x8,128x30,16x240,intra:512x8] [--steps 20] [--warmup 3]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_sequences import card  # noqa: E402

W, H, Q, GOP, CLIP_FRAMES = 720, 576, 128, 30, 240


def timed(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", default="512x8,128x30,16x240,intra:512x8")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import device as D
    from oracle import oracle as O

    assert torch.cuda.is_available(), "bench_encode_sequences measures the B200 path: no CUDA device"
    fsz = W * H * 3 // 2
    clips = [O.encode_clip(O.make_clip(W, H, Q, key_rate=GOP - 1, lm=2, cm=2, seed=seed), CLIP_FRAMES) for seed in (1, 2)]
    ctx = g.BatchContext(0)
    pools = []
    for s, o in clips:                          # the clips' pictures, decoded on the device
        desc, _ = g.plan(s, o)
        b = D.upload(s, desc, W, H)
        D.decode(ctx, b)
        pools.append(b.out)
    torch.cuda.synchronize()
    st = torch.cuda.current_stream()
    results = []
    for lay in args.layouts.split(","):
        intra = lay.startswith("intra:")
        S, k = (int(x) for x in lay.split(":")[-1].split("x"))
        kr, lm = (0, 0) if intra else (GOP - 1, 2)
        starts = [(s * 37) % (CLIP_FRAMES - k + 1) for s in range(S)]
        pics = [pools[s % 2][a:a + k] for s, a in enumerate(starts)]
        F = S * k
        sf = [s * k for s in range(S + 1)]
        cap = g.encode_bound(0, W, H, F)
        d_stream = torch.empty(cap, dtype=torch.uint8, device="cuda")
        d_off = torch.empty(F + 1, dtype=torch.int64, device="cuda")
        encs = [ctx.seq_encoder(Q, kr, lm, lm) for _ in range(S)]
        for s, e in enumerate(encs):            # key phases of their own
            n = (7 * s) % GOP
            if n:
                ctx.encode_device_seq(n, W, H, [0, n], [pools[0].data_ptr()], [e], d_stream.data_ptr(), cap, d_off.data_ptr(),
                                      st.cuda_stream)
        ptrs = [p.data_ptr() for p in pics]
        one = torch.cat(pics)                   # the ceiling's one buffer
        ctx.encoder_config(Q, kr, lm, lm)
        ctx.set_format(0)

        def run_seq():
            ctx.encode_device_seq(F, W, H, sf, ptrs, encs, d_stream.data_ptr(), cap, d_off.data_ptr(), st.cuda_stream)

        def run_calls():
            for s in range(S):
                ctx.encode_device_seq(k, W, H, [0, k], [ptrs[s]], [encs[s]], d_stream.data_ptr(), cap, d_off.data_ptr(),
                                      st.cuda_stream)

        def run_one():
            ctx.encode_device(one.data_ptr(), F, W, H, d_stream.data_ptr(), cap, d_off.data_ptr(), st.cuda_stream)

        row = {"layout": lay, "S": S, "k": k, "pictures": F, "key_rate": kr, "lm": lm}
        for name, fn in (("seq", run_seq), ("calls", run_calls), ("ceiling", run_one), ("seq_again", run_seq)):
            ms = timed(fn, args.steps, args.warmup)
            row[name] = {"ms_per_pass": ms, "pictures_per_s": F / (ms * 1e-3)}
        nbytes, overflow = ctx.encode_info()
        assert not overflow
        row["bytes_per_picture"] = nbytes / F
        row["seq_over_calls"] = row["seq"]["pictures_per_s"] / row["calls"]["pictures_per_s"]
        row["seq_over_ceiling"] = row["seq"]["pictures_per_s"] / row["ceiling"]["pictures_per_s"]
        if not intra:
            # transcode: the S source sequences decoded in one call, then encoded again in one call
            seqs = [(clips[s % 2][0], clips[s % 2][1][a:a + k + 1]) for s, a in enumerate(starts)]
            b, bsf = D.upload_sequences(seqs, W, H)
            views = [b.out[int(bsf[s]):int(bsf[s + 1])].data_ptr() for s in range(S)]

            def run_transcode():
                ctx.decode_device_seq(b.stream.data_ptr(), b.desc.data_ptr(), F, W, H, list(bsf), b.out.data_ptr(), None,
                                      st.cuda_stream)
                ctx.encode_device_seq(F, W, H, sf, views, encs, d_stream.data_ptr(), cap, d_off.data_ptr(), st.cuda_stream)

            ms = timed(run_transcode, args.steps, args.warmup)
            row["transcode"] = {"ms_per_pass": ms, "pictures_per_s": F / (ms * 1e-3)}
            del b
        for e in encs:
            e.close()
        results.append(row)
        del d_stream, one
        torch.cuda.empty_cache()
        print(json.dumps(row), file=sys.stderr, flush=True)
    ctx.close()
    print(json.dumps({"metric": "720x576 Q128 re-encode, GOP 30 lm=cm=2 (intra: key_rate 0), pictures/s per layout",
                      "card": card(), "steps": args.steps, "warmup": args.warmup, "layouts": results}))


if __name__ == "__main__":
    main()
