#!/usr/bin/env python3
"""Decoding a window of the selected frames: rtjgpu_decode_device_window against rtjgpu_decode_device_select of the same
frames, and the fused rtjgpu_decode_device_rgb_window (RGB24) against rtjgpu_decode_device_rgb_select.

Layouts S x k (S sequences of k frames, 720x576 YUV420, Q=128): 128x30 and 16x240 inter (GOP 30, lm = cm = 2, every
sequence starting anywhere in a GOP of one of two clips), and 1x4096 of bench.py's intra stream.  Windows: the full picture,
the letterbox 720x432 at y = 72, a centred 352x288 (x = 176: the nearest multiple of 16 to 184), and 224x224 at a random
origin per sequence.  Selections: every frame and every 8th frame of each sequence.  No last_yuv: the calls launch K2 over
the selected frames only; the 224x224 window is also timed with a last_yuv for every sequence (the launch of the last
frames, whole).  Packets, descriptors and carries are resident in HBM; the outputs stay there.  Times: CUDA
events around `steps` passes after `warmup` passes, the reference call timed before and after the window call (their mean
is the reference).  Then, on a context with the library's stage timing (rtjgpu_timing), the median idct stage of the same
passes over the macroblocks each call decodes: K2's device time per decoded macroblock (ps, all SMs at once) for the
window kernel (the strip family) and for the select call (the SINGLE kernel of 720-wide pictures, plus K2b where blocks go
that way).

Writes one JSON line, with the card's name and power limit read in the same run, to --out and to stdout.

    python tools/bench_window.py [--layouts 128x30,16x240,1x4096] [--steps 20] [--warmup 3] [--out profiles/window_bench_line.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, Q, GOP, CLIP_FRAMES = 720, 576, 128, 30, 240
SELECTIONS = [("every_1", 1), ("every_8", 8)]


def windows(S, rng):
    """name -> ((cw, ch), [(x, y)] * S)"""
    rand = [(int(rng.integers(0, (W - 224) // 16 + 1)) * 16, int(rng.integers(0, (H - 224) // 2 + 1)) * 2) for _ in range(S)]
    return {"full": ((W, H), [(0, 0)] * S), "letterbox_720x432": ((720, 432), [(0, 72)] * S),
            "centre_352x288": ((352, 288), [(176, 144)] * S), "random_224x224": ((224, 224), rand)}


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
    ap.add_argument("--layouts", default="128x30,16x240,1x4096")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "window_bench_line.json"))
    args = ap.parse_args()

    import torch
    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import capi
    from gmerlin_avdecoder_b200 import device as D
    from oracle import oracle as O

    assert torch.cuda.is_available(), "bench_window measures the B200 path: no CUDA device"
    threads = min(os.cpu_count() or 1, 64)
    clips = [O.encode_clip(O.make_clip(W, H, Q, key_rate=GOP - 1, lm=2, cm=2, seed=seed), CLIP_FRAMES, threads=threads)
             for seed in (1, 2)]
    fsz = W * H * 3 // 2
    carry = torch.from_numpy(np.random.default_rng(0).integers(0, 256, fsz).astype(np.uint8)).cuda()
    st = torch.cuda.current_stream()
    vp = C.c_void_p

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

    def idct_median(ctx, fn):
        for _ in range(args.warmup):
            fn()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return float(np.median([ctx.timing_at(i).idct_ms for i in range(args.steps)]))

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
        ctx, tctx = g.BatchContext(0), g.BatchContext(0)
        tctx.enable_timing(True)
        L = ctx._L
        first = (C.c_int * (S + 1))(*[int(x) for x in sf])
        carries = (vp * S)(*([carry.data_ptr()] * S))
        lens = [int(sf[s + 1] - sf[s]) for s in range(S)]
        seq_of = np.repeat(np.arange(S), lens)
        row = {"layout": lay, "stream": kind, "S": S, "k": k, "frames": F, "windows": {}}
        for wname, ((cw, ch), org) in windows(S, np.random.default_rng(S * 1000 + k)).items():
            org_c = (C.c_int * (2 * S))(*[v for xy in org for v in xy])
            wrow = {"size": [cw, ch]}
            for sname, step in SELECTIONS:
                sel = capi.select_frames(sf, [np.arange(0, n, step) for n in lens])
                n = len(sel)
                sel_c = (C.c_int * max(n, 1))(*[int(x) for x in sel])
                # macroblocks K2 decodes: the full picture for select, the units that cover each frame's window
                mb_sel = n * (W // 16) * (H // 16)
                rows = np.array([(y + ch - 1) // 16 - y // 16 + 1 for _, y in org])
                mb_win = int(rows[seq_of[sel]].sum()) * (cw // 16)
                out_sel = torch.empty((n, fsz), dtype=torch.uint8, device="cuda")
                out_win = torch.empty((n, cw * ch * 3 // 2), dtype=torch.uint8, device="cuda")
                rgb_sel = torch.empty((n, H, W * 3), dtype=torch.uint8, device="cuda")
                rgb_win = torch.empty((n, ch, cw * 3), dtype=torch.uint8, device="cuda")

                def batch(c):
                    return (c._h, vp(b.stream.data_ptr()), vp(b.desc.data_ptr()), F, W, H, S, first, carries, n, sel_c)

                def run_sel(c=ctx):
                    ok(L.rtjgpu_decode_device_select(*batch(c), vp(out_sel.data_ptr()), vp(st.cuda_stream)))

                def run_win(c=ctx):
                    ok(L.rtjgpu_decode_device_window(*batch(c), cw, ch, org_c, vp(out_win.data_ptr()), None, vp(st.cuda_stream)))

                def run_rgb_sel(c=ctx):
                    ok(L.rtjgpu_decode_device_rgb_select(*batch(c), capi.CONV_RGB24, vp(rgb_sel.data_ptr()), W * 3, H * W * 3,
                                                         0, None, vp(st.cuda_stream)))

                def run_rgb_win(c=ctx):
                    ok(L.rtjgpu_decode_device_rgb_window(*batch(c), cw, ch, org_c, capi.CONV_RGB24, vp(rgb_win.data_ptr()),
                                                         cw * 3, ch * cw * 3, 0, None, vp(st.cuda_stream)))

                res = {"selected": n}
                for form, ref_fn, win_fn in (("planes", run_sel, run_win), ("rgb24", run_rgb_sel, run_rgb_win)):
                    r0 = timed(ref_fn)
                    wms = timed(win_fn)
                    r1 = timed(ref_fn)
                    ref = (r0 + r1) / 2
                    res[form] = {"window_ms": wms, "select_ms": ref, "select_ms_before_after": [r0, r1], "over_select": wms / ref}
                if wname == "random_224x224":
                    # the same window call with every sequence's last frame also leaving whole to a last_yuv: the second
                    # launch, which runs behind the window launch on the same stream
                    lasts = torch.empty((S, fsz), dtype=torch.uint8, device="cuda")
                    lasts_c = (vp * S)(*[lasts[s].data_ptr() for s in range(S)])

                    def run_win_last(c=ctx):
                        ok(L.rtjgpu_decode_device_window(*batch(c), cw, ch, org_c, vp(out_win.data_ptr()), lasts_c,
                                                         vp(st.cuda_stream)))

                    wl = timed(run_win_last)
                    res["planes"]["window_with_last_yuv_ms"] = wl
                    res["planes"]["last_yuv_launch_ms"] = wl - res["planes"]["window_ms"]
                    del lasts
                k2_sel = idct_median(tctx, lambda: run_sel(tctx))
                k2_win = idct_median(tctx, lambda: run_win(tctx))
                res["k2"] = {"select_idct_ms": k2_sel, "window_idct_ms": k2_win, "select_mb": mb_sel, "window_mb": mb_win,
                             "select_ps_per_mb": 1e9 * k2_sel / mb_sel, "window_ps_per_mb": 1e9 * k2_win / max(mb_win, 1)}
                wrow[sname] = res
                del out_sel, out_win, rgb_sel, rgb_win
            row["windows"][wname] = wrow
            print(json.dumps({"layout": lay, "window": wname, **wrow}), file=sys.stderr, flush=True)
        results.append(row)
        ctx.close()
        tctx.close()
        del b
        torch.cuda.empty_cache()
    line = json.dumps({"metric": "720x576 Q128 windows of selected frames: rtjgpu_decode_device[_rgb]_window against "
                                 "the _select call of the same frames", "card": card(), "steps": args.steps,
                       "warmup": args.warmup, "layouts": results})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
