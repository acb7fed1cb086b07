#!/usr/bin/env python3
"""Decoding straight to a model's input: rtjgpu_decode_device_chw_window against what callers write today.

Layouts S x k (S sequences of k frames, 720x576 YUV420, Q=128): 128x30 and 16x240 inter (GOP 30, lm = cm = 2, every
sequence starting anywhere in a GOP of one of two clips), and 1x4096 of bench.py's intra stream -- the setup of
tools/bench_window.py.  Window: 224x224 (--size) at a random origin per sequence; selections: every frame and every 8th frame of each
sequence; every other sequence mirrored.  On the same batch:
  (a) the fused call: float16 with ImageNet's mean and std, and uint8;
  (b) rtjgpu_decode_device_rgb_window, RGB24 alone (the floor);
  (c) (b) followed by the plain eager torch post-process callers write today: for float16
      permute(0, 3, 1, 2) -> float32 -> mul_(scale) -> add_(bias) -> float16, for uint8 permute(0, 3, 1, 2).contiguous().
Packets, descriptors and carries are resident in HBM; the outputs stay there.  Times: CUDA events around `steps` passes
after `warmup` passes, (b) timed before and after the others (their mean is the floor).

Writes one JSON line, with the card's name, power limit and clocks read in the same run, to --out and to stdout.

    python tools/bench_chw_window.py [--layouts 128x30,16x240,1x4096] [--size 224x224] [--steps 20] [--warmup 3]
                                     [--out profiles/chw_window_bench_line.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_window import CLIP_FRAMES, GOP, H, Q, SELECTIONS, W, card  # noqa: E402

IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layouts", default="128x30,16x240,1x4096")
    ap.add_argument("--size", default="224x224", help="the window, cw x ch (720x576: the whole picture)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "chw_window_bench_line.json"))
    args = ap.parse_args()
    CW, CH = (int(v) for v in args.size.split("x"))

    import torch
    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import capi
    from gmerlin_avdecoder_b200 import device as D
    from oracle import oracle as O

    assert torch.cuda.is_available(), "bench_chw_window measures the B200 path: no CUDA device"
    threads = min(os.cpu_count() or 1, 64)
    clips = [O.encode_clip(O.make_clip(W, H, Q, key_rate=GOP - 1, lm=2, cm=2, seed=seed), CLIP_FRAMES, threads=threads)
             for seed in (1, 2)]
    fsz = W * H * 3 // 2
    carry = torch.from_numpy(np.random.default_rng(0).integers(0, 256, fsz).astype(np.uint8)).cuda()
    st = torch.cuda.current_stream()
    vp = C.c_void_p
    scale, bias = capi.normalize_coefficients(*IMAGENET)
    scale_c, bias_c = (C.c_float * 3)(*[float(v) for v in scale]), (C.c_float * 3)(*[float(v) for v in bias])
    scale_t = torch.from_numpy(scale).cuda().view(1, 3, 1, 1)
    bias_t = torch.from_numpy(bias).cuda().view(1, 3, 1, 1)

    def ok(rc):
        assert rc == 0, rc

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    results = []
    for lay in args.layouts.split(","):
        S, k = (int(x) for x in lay.split("x"))
        if S == 1 and k > CLIP_FRAMES:          # bench.py's intra stream (BASELINE.json configs[1])
            seqs = [O.encode_clip(O.make_clip(W, H, Q, key_rate=-1, seed=1), k, threads=threads)]
            kind = "intra"
        else:
            assert k <= CLIP_FRAMES
            seqs = []
            for s in range(S):
                cs, co = clips[s % 2]
                a = (s * 37) % (CLIP_FRAMES - k + 1)
                seqs.append((cs, co[a:a + k + 1]))
            kind = "inter"
        b, sf = D.upload_sequences(seqs, W, H)
        F = b.F
        ctx = g.BatchContext(0)
        L = ctx._L
        first = (C.c_int * (S + 1))(*[int(x) for x in sf])
        carries = (vp * S)(*([carry.data_ptr()] * S))
        lens = [int(sf[s + 1] - sf[s]) for s in range(S)]
        rng = np.random.default_rng(S * 1000 + k)
        org = [(int(rng.integers(0, (W - CW) // 16 + 1)) * 16, int(rng.integers(0, (H - CH) // 2 + 1)) * 2) for _ in range(S)]
        org_c = (C.c_int * (2 * S))(*[v for xy in org for v in xy])
        mirror_c = (C.c_int * S)(*[s % 2 for s in range(S)])
        row = {"layout": lay, "stream": kind, "S": S, "k": k, "frames": F, "size": [CW, CH]}
        for sname, step in SELECTIONS:
            sel = capi.select_frames(sf, [np.arange(0, n, step) for n in lens])
            n = len(sel)
            sel_c = (C.c_int * max(n, 1))(*[int(x) for x in sel])
            rgb = torch.empty((n, CH, CW, 3), dtype=torch.uint8, device="cuda")
            f16 = torch.empty((n, 3, CH, CW), dtype=torch.float16, device="cuda")
            u8 = torch.empty((n, 3, CH, CW), dtype=torch.uint8, device="cuda")

            def batch():
                return (ctx._h, vp(b.stream.data_ptr()), vp(b.desc.data_ptr()), F, W, H, S, first, carries, n, sel_c)

            def run_rgb():
                ok(L.rtjgpu_decode_device_rgb_window(*batch(), CW, CH, org_c, capi.CONV_RGB24, vp(rgb.data_ptr()), CW * 3,
                                                     CH * CW * 3, 0, None, vp(st.cuda_stream)))

            def run_f16():
                ok(L.rtjgpu_decode_device_chw_window(*batch(), CW, CH, org_c, mirror_c, capi.CONV_RGB24, capi.CHW_F16, scale_c,
                                                     bias_c, vp(f16.data_ptr()), None, vp(st.cuda_stream)))

            def run_u8():
                ok(L.rtjgpu_decode_device_chw_window(*batch(), CW, CH, org_c, mirror_c, capi.CONV_RGB24, capi.CHW_U8, None,
                                                     None, vp(u8.data_ptr()), None, vp(st.cuda_stream)))

            def run_rgb_torch_f16():
                run_rgb()
                rgb.permute(0, 3, 1, 2).float().mul_(scale_t).add_(bias_t).half()

            def run_rgb_torch_u8():
                run_rgb()
                rgb.permute(0, 3, 1, 2).contiguous()

            b0 = timed(run_rgb)
            t = {"fused_f16_imagenet_ms": timed(run_f16), "fused_u8_ms": timed(run_u8),
                 "rgb_window_torch_f16_ms": timed(run_rgb_torch_f16), "rgb_window_torch_u8_ms": timed(run_rgb_torch_u8)}
            b1 = timed(run_rgb)
            floor = (b0 + b1) / 2
            t["rgb_window_ms"] = floor
            t["rgb_window_ms_before_after"] = [b0, b1]
            t["f16_over_rgb_window"] = t["fused_f16_imagenet_ms"] / floor
            t["f16_over_torch_f16"] = t["fused_f16_imagenet_ms"] / t["rgb_window_torch_f16_ms"]
            t["u8_over_rgb_window"] = t["fused_u8_ms"] / floor
            t["u8_over_torch_u8"] = t["fused_u8_ms"] / t["rgb_window_torch_u8_ms"]
            # bytes that leave: RGB24 packed, f16 planar (the fused call), and what the torch post-process reads and writes
            px = n * CW * CH * 3
            t["selected"] = n
            t["bytes_out"] = {"rgb24": px, "f16": 2 * px, "u8": px, "torch_f16_read_write": 27 * px}
            row[sname] = t
            print(json.dumps({"layout": lay, "selection": sname, **t}), file=sys.stderr, flush=True)
            del rgb, f16, u8
        results.append(row)
        ctx.close()
        del b
        torch.cuda.empty_cache()
    line = json.dumps({"metric": f"720x576 Q128, {CW}x{CH} windows at a random origin per sequence: rtjgpu_decode_device_chw_window "
                                 "(f16 ImageNet-normalised, u8) against rtjgpu_decode_device_rgb_window RGB24 alone and "
                                 "followed by the eager torch post-process", "card": card(), "steps": args.steps,
                       "warmup": args.warmup, "layouts": results})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
