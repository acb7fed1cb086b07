#!/usr/bin/env python3
"""Many independent streams per device batch: rtjgpu_decode_device_seq against one call per stream.

For each layout S x k (S sequences of k frames, 720x576 YUV420, Q=128, GOP 30, lm = cm = 2) it reports frames/s of
  seq      one rtjgpu_decode_device_seq call, every sequence with its own carry picture
  calls    S rtjgpu_decode_device calls on the same stream, each over its sequence's frames with its own carry
  ceiling  the same S * k frames as ONE stream in one rtjgpu_decode_device call (wrong pixels across the sequence
           boundaries, about the same work: what one call could at best reach)
Packets, descriptors and carries are resident in HBM; the frames stay there.  Times: CUDA events around `steps` passes
after `warmup` passes.  Prints one JSON line with the card's name and power limit.

    python tools/bench_sequences.py [--layouts 512x8,128x30,16x240] [--steps 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, Q, GOP, CLIP_FRAMES = 720, 576, 128, 30, 240


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", default="512x8,128x30,16x240")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import device as D
    from oracle import oracle as O

    assert torch.cuda.is_available(), "bench_sequences measures the B200 path: no CUDA device"
    clips = [O.encode_clip(O.make_clip(W, H, Q, key_rate=GOP - 1, lm=2, cm=2, seed=seed), CLIP_FRAMES) for seed in (1, 2)]
    fsz = W * H * 3 // 2
    carry = torch.from_numpy(np.random.default_rng(0).integers(0, 256, fsz).astype(np.uint8)).cuda()
    st = torch.cuda.current_stream()
    results = []
    for lay in args.layouts.split(","):
        S, k = (int(x) for x in lay.split("x"))
        assert k <= CLIP_FRAMES
        seqs = []
        for s in range(S):                      # sequence s: k frames of one of the clips, starting anywhere in a GOP
            cs, co = clips[s % 2]
            a = (s * 37) % (CLIP_FRAMES - k + 1)
            seqs.append((cs, co[a:a + k + 1]))
        b, sf = D.upload_sequences(seqs, W, H)
        F = b.F
        carries = [carry.data_ptr()] * S
        ctx = g.BatchContext(0)

        def run_seq():
            ctx.decode_device_seq(b.stream.data_ptr(), b.desc.data_ptr(), F, W, H, list(sf), b.out.data_ptr(), carries, st.cuda_stream)

        def run_calls():
            for s in range(S):
                a = int(sf[s])
                ctx.decode_device(b.stream.data_ptr(), b.desc.data_ptr() + 16 * a, int(sf[s + 1]) - a, W, H,
                                  b.out.data_ptr() + fsz * a, carry.data_ptr(), st.cuda_stream)

        def run_one():
            ctx.decode_device(b.stream.data_ptr(), b.desc.data_ptr(), F, W, H, b.out.data_ptr(), carry.data_ptr(), st.cuda_stream)

        row = {"layout": lay, "S": S, "k": k, "frames": F}
        for name, fn in (("seq", run_seq), ("calls", run_calls), ("ceiling", run_one), ("seq_again", run_seq)):
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            row[name] = {"ms_per_pass": ms, "frames_per_s": F / (ms * 1e-3)}
        row["seq_over_calls"] = row["seq"]["frames_per_s"] / row["calls"]["frames_per_s"]
        row["seq_over_ceiling"] = row["seq"]["frames_per_s"] / row["ceiling"]["frames_per_s"]
        results.append(row)
        ctx.close()
        del b
        torch.cuda.empty_cache()
        print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps({"metric": "720x576 GOP-30 lm=cm=2 sequences, frames/s per layout", "card": card(), "steps": args.steps,
                      "warmup": args.warmup, "layouts": results}))


if __name__ == "__main__":
    main()
