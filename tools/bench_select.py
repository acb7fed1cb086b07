#!/usr/bin/env python3
"""Decoding a selection of a batch's frames: rtjgpu_decode_device_select against the full rtjgpu_decode_device_seq call.

Layouts S x k (S sequences of k frames, 720x576 YUV420, Q=128): 128x30 and 16x240 inter (GOP 30, lm = cm = 2, every
sequence starting anywhere in a GOP of one of two clips), and 1x4096 of bench.py's intra stream.  Selections: every k-th
frame of each sequence (k = 1, 2, 4, 8, 30) and each sequence's last frame only.  For each it reports the select call's ms
per pass, the full call's ms on the same batch (timed before and after the selections; their mean is the reference), the
ratio, batch frames consumed per second and the output bytes.  Also the fused RGB32 select at 1 in 8 against the full
rtjgpu_decode_device_rgb_seq call.  Packets, descriptors and carries are resident in HBM; the frames stay there.  Times:
CUDA events around `steps` passes after `warmup` passes.  Prints one JSON line with the card's name and power limit.

--wide WxHxF: the strip kernels of pictures wider than 2048 px (one CTA takes part of a macroblock row), whose selection
instantiations spill where the full call's do not: an intra stream (so the full call, too, decodes one frame per CTA), the full
call against a selection of all frames but the last, with the library's per-stage times (rtjgpu_timing) -- K2's time per
decoded frame in either.  "" leaves it out.

    python tools/bench_select.py [--layouts 128x30,16x240,1x4096] [--wide 2560x1440x256] [--steps 20] [--warmup 3]
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
SELECTIONS = [("every_1", 1), ("every_2", 2), ("every_4", 4), ("every_8", 8), ("every_30", 30), ("last_only", None)]


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
    ap.add_argument("--wide", default="2560x1440x256")
    args = ap.parse_args()

    import torch
    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import capi
    from gmerlin_avdecoder_b200 import device as D
    from oracle import oracle as O

    assert torch.cuda.is_available(), "bench_select measures the B200 path: no CUDA device"
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

    results = []
    for lay in args.layouts.split(","):
        S, k = (int(x) for x in lay.split("x"))
        if S == 1 and k > CLIP_FRAMES:          # bench.py's intra stream (BASELINE.json configs[1])
            seqs = [O.encode_clip(O.make_clip(W, H, Q, key_rate=-1, seed=1), k, threads=threads)]
            kind = "intra"
        else:
            assert k <= CLIP_FRAMES
            seqs = []
            for s in range(S):                  # sequence s: k frames of one of the clips, starting anywhere in a GOP
                cs, co = clips[s % 2]
                a = (s * 37) % (CLIP_FRAMES - k + 1)
                seqs.append((cs, co[a:a + k + 1]))
            kind = "inter"
        b, sf = D.upload_sequences(seqs, W, H)
        F = b.F
        ctx = g.BatchContext(0)
        L = ctx._L
        # the host arrays of every call are made once: the timed loops enqueue the calls and nothing else
        first = (C.c_int * (S + 1))(*[int(x) for x in sf])
        carries = (vp * S)(*([carry.data_ptr()] * S))
        args_batch = (ctx._h, vp(b.stream.data_ptr()), vp(b.desc.data_ptr()), F, W, H, S, first)

        def run_full():
            ok(L.rtjgpu_decode_device_seq(*args_batch, vp(b.out.data_ptr()), carries, vp(st.cuda_stream)))

        row = {"layout": lay, "stream": kind, "S": S, "k": k, "frames": F, "full_output_bytes": F * fsz}
        full_ms = [timed(run_full)]
        sels = {}
        for name, step in SELECTIONS:
            lens = [int(sf[s + 1] - sf[s]) for s in range(S)]
            picks = [np.arange(0, n, step) if step else np.array([n - 1]) for n in lens]
            sel = capi.select_frames(sf, picks)
            n = len(sel)
            sel_c = (C.c_int * max(n, 1))(*[int(x) for x in sel])
            out = torch.empty((n, fsz), dtype=torch.uint8, device="cuda")

            def run_sel():
                ok(L.rtjgpu_decode_device_select(*args_batch, carries, n, sel_c, vp(out.data_ptr()), vp(st.cuda_stream)))

            ms = timed(run_sel)
            sels[name] = {"selected": n, "ms_per_pass": ms, "frames_consumed_per_s": F / (ms * 1e-3), "output_bytes": n * fsz}
            del out
        full_ms.append(timed(run_full))
        full = sum(full_ms) / 2
        row["full"] = {"ms_per_pass": full, "ms_before_after": full_ms, "frames_consumed_per_s": F / (full * 1e-3)}
        for v in sels.values():
            v["over_full"] = v["ms_per_pass"] / full
        row["select"] = sels

        # the fused RGB32 converter, 1 in 8, against the full fused call
        pitch = W * 4
        sel = capi.select_frames(sf, [np.arange(0, int(sf[s + 1] - sf[s]), 8) for s in range(S)])
        n = len(sel)
        sel_c = (C.c_int * max(n, 1))(*[int(x) for x in sel])
        rgb_full = torch.empty((F, H, pitch), dtype=torch.uint8, device="cuda")
        rgb_sel = torch.empty((n, H, pitch), dtype=torch.uint8, device="cuda")

        def run_rgb_full():
            ok(L.rtjgpu_decode_device_rgb_seq(*args_batch, capi.CONV_RGB32, vp(rgb_full.data_ptr()), pitch, H * pitch, 0,
                                              carries, None, vp(st.cuda_stream)))

        def run_rgb_sel():
            ok(L.rtjgpu_decode_device_rgb_select(*args_batch, carries, n, sel_c, capi.CONV_RGB32, vp(rgb_sel.data_ptr()), pitch,
                                                 H * pitch, 0, None, vp(st.cuda_stream)))

        rf = timed(run_rgb_full)
        rs = timed(run_rgb_sel)
        rf2 = timed(run_rgb_full)
        row["rgb32_every_8"] = {"selected": n, "select_ms": rs, "full_ms": (rf + rf2) / 2, "full_ms_before_after": [rf, rf2],
                                "over_full": rs / ((rf + rf2) / 2), "output_bytes": n * H * pitch}
        results.append(row)
        ctx.close()
        del b, rgb_full, rgb_sel
        torch.cuda.empty_cache()
        print(json.dumps(row), file=sys.stderr, flush=True)
    wide = None
    if args.wide:
        ww, wh, wf = (int(x) for x in args.wide.split("x"))
        b, sf = D.upload_sequences([O.encode_clip(O.make_clip(ww, wh, Q, key_rate=-1, seed=3), wf, threads=threads)], ww, wh)
        ctx = g.BatchContext(0)
        ctx.enable_timing(True)
        L = ctx._L
        first = (C.c_int * 2)(0, wf)
        args_batch = (ctx._h, vp(b.stream.data_ptr()), vp(b.desc.data_ptr()), wf, ww, wh, 1, first)
        sel_c = (C.c_int * (wf - 1))(*range(wf - 1))
        out = torch.empty((wf - 1, b.frame_bytes), dtype=torch.uint8, device="cuda")

        def run_wide_full():
            ok(L.rtjgpu_decode_device_seq(*args_batch, vp(b.out.data_ptr()), None, vp(st.cuda_stream)))

        def run_wide_sel():
            ok(L.rtjgpu_decode_device_select(*args_batch, None, wf - 1, sel_c, vp(out.data_ptr()), vp(st.cuda_stream)))

        def stages():
            t = [ctx.timing_at(i) for i in range(args.steps)]
            return {f: float(np.median([getattr(x, f) for x in t])) for f in ("scan_ms", "resolve_ms", "idct_ms", "total_ms")}

        wide = {"picture": f"{ww}x{wh}", "frames": wf, "stream": "intra"}
        for name, fn, nf in (("full", run_wide_full, wf), ("select_all_but_last", run_wide_sel, wf - 1),
                             ("full_again", run_wide_full, wf)):
            ms = timed(fn)
            sg = stages()
            wide[name] = {"ms_per_pass": ms, "stages_median": sg, "k2_us_per_frame": 1e3 * sg["idct_ms"] / nf}
        full_k2 = (wide["full"]["k2_us_per_frame"] + wide["full_again"]["k2_us_per_frame"]) / 2
        wide["k2_per_frame_select_over_full"] = wide["select_all_but_last"]["k2_us_per_frame"] / full_k2
        ctx.close()
        del b, out
        torch.cuda.empty_cache()
        print(json.dumps(wide), file=sys.stderr, flush=True)
    print(json.dumps({"metric": "720x576 Q128 selected frames: rtjgpu_decode_device_select against the full _seq call",
                      "card": card(), "steps": args.steps, "warmup": args.warmup, "layouts": results, "wide": wide}))


if __name__ == "__main__":
    main()
