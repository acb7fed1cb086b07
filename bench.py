#!/usr/bin/env python3
"""bench.py -- RTjpeg 720x576 YUV420 decoded frames/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]              # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...       # the reference's CPU decoder (oracle/_ref)
    python bench.py --dump-outputs DIR ...                            # + what the last timed step decoded, as .npy
    torchrun --nproc-per-node N ... bench.py --gpus N ...             # one rank per GPU

A "step" is one pass of the hot path (K1 scan -> K3 resolve -> K2 idct -> K2b hard blocks) over one batch of
4096 synthetic 720x576 frames (BASELINE.json configs[1]: intra-only, Q=128).  The batch is produced once, outside
every timed region, by RTjpeg_compress as oracle/ restates it (tests/golden/ pins it to the reference's own packets,
byte for byte) from the seeded source in oracle/rtjo_driver.c: the same arguments give the same batch.  The headline
is weak scaling: every rank decodes its own 4096-frame batch (its own seed); batches are independent, there is no
data-path collective.

value     whole-job frames/s, packets and descriptors already resident in HBM, frames left in HBM; the library's
          default arrangement (rtjgpu_set_pipeline AUTO: the scan of one slice of frames beside resolve + IDCT of the
          slice before it, on two streams forked from and joined to the caller's).
e2e       same metric through the C ABI's host entry point (rtjgpu_decode_host): packets in pinned host memory,
          frames returned to pinned host memory, both copies inside the timed region.
roofline  dominant kernel (K2), timed ALONE: separate steps in the serial arrangement (every stage on the caller's
          stream, CUDA events recorded by the library between the stages); algorithmic bytes = payload read + planes
          written.  whole_path_frac is the same bytes over the headline step time.
on_device_consumers   end to end with the frames consumed on the device (fused RGB32 out; transcode through the GPU encoder)
other_configs   the parity configs of BASELINE.json (inter GOP 30 at two masks, Q32 / Q255, 1920x1088 dense), measured in
          the same process after the headline (rank 0, N = 1).
config5   BASELINE.json configs[4]: ONE inter-coded 1920x1088 stream, cut at clean frames on the host
          (rtjgpu_split_shards_lead over the headers' key hints, verified with K1's skip counts), every shard decoded
          by its rank's GPU, frames left there.  Strong scaling: the stream is the same at every N.
cpu_baseline  the unmodified reference decoder (oracle/_ref) on this box's host cores; left out where it is not built
          (oracle/Makefile `ref` compiles it from the reference's sources, which the repository does not hold).
--dump-outputs DIR  after the timed steps, what the last of them left in HBM: frames.npy, a fixed seeded sample of 16
          decoded frames (float32, frame_index.npy says which), and frame_sums.npy, the byte sum of every frame (float64).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H, QUALITY, FRAMES = 720, 576, 128, 4096
METRIC = "RTjpeg 720x576 YUV420 decoded frames/sec"
WORKLOAD = "configs[1]: RTjpeg 720x576 YUV420 intra-only Q=128, 4096-frame synthetic batch per GPU"
SM_SUBPARTITIONS = 148 * 4

C5_W, C5_H, C5_Q, C5_GOP, C5_FRAMES = 1920, 1088, 128, 30, 960


def make_workload(frames: int, seed: int, w=W, h=H, q=QUALITY, **kw):
    """Synthetic clip -> packets by the restated compressor (not timed)."""
    from oracle import oracle as O
    kw.setdefault("noise_y", 2)
    kw.setdefault("noise_c", 0)
    clip = O.make_clip(w, h, q, key_rate=kw.pop("key_rate", -1), seed=seed, **kw)
    t0 = time.time()
    stream, offsets = O.encode_clip(clip, frames, threads=min(os.cpu_count() or 1, 64))
    return stream, offsets, time.time() - t0


def config_dict(payload_per_frame: float, frames: int) -> dict:
    """The workload as both arms state it (the driver compares the arms' `config`)."""
    fsz = W * H * 3 // 2
    return {
        "workload": WORKLOAD, "frames_per_gpu_per_step": frames, "quality": QUALITY,
        "payload_bytes_per_frame": payload_per_frame, "planar_bytes_per_frame": fsz,
        "l2": "inputs larger than L2: every step reads %.0f MB and writes %.0f MB"
              % (payload_per_frame * frames / 1e6, frames * fsz / 1e6),
        "stream_source": "RTjpeg_compress (restated, the reference's packets byte for byte) on a seeded synthetic clip (untimed)",
    }


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def reference_decode_fps(stream, offsets, frames: int, threads: int, reps: int, w=W, h=H, segments=None):
    """Reference RTjpeg_decompress over `frames` frames, `threads` private decoders; intra: frames striped (every frame
    its own segment); inter: whole clean-frame-delimited segments per thread.  Returns the list of frames/s."""
    from oracle import oracle as O
    sub = offsets[:frames + 1]
    seg = np.arange(frames + 1, dtype=np.int32) if segments is None else np.asarray(segments, dtype=np.int32)
    fps = []
    for _ in range(reps):
        secs, _ = O.ref_decode_threaded(stream, sub, seg, w, h, threads, zero_init=segments is not None, keep=False)
        fps.append(frames / secs)
    return fps


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML from before the warm-up to the end of the timed steps."""

    def __init__(self, index: int, period: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.util = []
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            getattr(nv, "nvmlClocksEventReasonApplicationsClocksSetting", 0x2): "applications_clocks_setting",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_min_mhz": min(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
            "window": "from before the warm-up steps to the end of the timed steps",
        }


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_facts():
    """What one committed ncu capture says about the kernels at configs[1] (profiles/traffic.json): DRAM bytes and warp
    instructions per launch.  Not measured by this run; times and clocks are."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:  # noqa: BLE001
        return {}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return                                           # rank 0 alone runs and prints the CPU arm
    stream, offsets, _ = make_workload(args.frames, seed=1)
    threads = host_threads()
    frames = args.frames
    from oracle import oracle as O
    payload = float(O.packet_sizes(stream, offsets).astype(np.int64).sum() - 12 * frames) / frames
    for _ in range(max(args.warmup, 1)):
        reference_decode_fps(stream, offsets, min(frames, 512), threads, 1)
    t0 = time.time()
    fps = reference_decode_fps(stream, offsets, frames, threads, args.steps)
    wall = time.time() - t0
    value = frames * args.steps / sum(frames / f for f in fps)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": config_dict(payload, frames),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "reference",
                         "sample": f"{args.steps} steps over all {frames} frames of the batch, unmodified lib/RTjpeg.c "
                                   f"RTjpeg_decompress, {threads} threads each with a private decoder and plane set",
                         "median": statistics.median(fps), "all": fps},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


# ---------------------------------------------------------------------------------------------------------------
# the CUDA arm
# ---------------------------------------------------------------------------------------------------------------

def time_steps(torch, D, ctx, batch, steps, sync):
    """`steps` device-resident decodes between two events on the current stream -> (ms total, launches)."""
    l0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    ev0.record()
    for _ in range(steps):
        D.decode(ctx, batch)
    ev1.record()
    sync()
    return ev0.elapsed_time(ev1), ctx.launch_count() - l0


def stage_times(torch, g, D, ctx, batch, steps):
    """Per-stage times in the SERIAL arrangement (each kernel alone on the device), mean over `steps`."""
    ctx.set_pipeline(g.PIPELINE_SERIAL)
    ctx.enable_timing(True)
    for _ in range(2):
        D.decode(ctx, batch)
    torch.cuda.synchronize()
    for _ in range(steps):
        D.decode(ctx, batch)
    torch.cuda.synchronize()
    ts = [ctx.timing_at(i) for i in range(steps)]
    ctx.enable_timing(False)
    ctx.set_pipeline(g.PIPELINE_AUTO)
    return {"scan": sum(t.scan_ms for t in ts) / steps, "resolve": sum(t.resolve_ms for t in ts) / steps,
            "idct": sum(t.idct_ms for t in ts) / steps, "total": sum(t.total_ms for t in ts) / steps}


def other_config(torch, g, D, name, w, h, q, frames, peak, sm_hz, steps=10, **kw):
    stream, offsets, _ = make_workload(frames, seed=1, w=w, h=h, q=q, **kw)
    desc, _ = g.plan(stream, offsets)
    ctx = g.BatchContext(0)
    b = D.upload(stream, desc, w, h, device=0)
    for _ in range(3):
        D.decode(ctx, b)
        torch.cuda.synchronize()      # the library arranges a batch by what the batch before held (skipped blocks, raw prefixes)
    info = ctx.batch_info()
    assert info.bad_frames == 0
    ms, _ = time_steps(torch, D, ctx, b, steps, torch.cuda.synchronize)
    ms /= steps
    st = stage_times(torch, g, D, ctx, b, min(steps, 10))
    algo = b.payload_bytes + frames * w * h * 3 // 2
    nblk = (w // 16) * (h // 16) * 6
    out = {
        "case": name, "w": w, "h": h, "quality": q, "frames": frames,
        "payload_bytes_per_frame": b.payload_bytes / frames,
        "skipped_blocks_frac": info.skipped_blocks / (frames * nblk),
        "ms_per_step": ms, "frames_per_s": frames / (ms * 1e-3),
        "hbm_frac": algo / (ms * 1e-3) / 1e9 / peak,
        "stage_ms_serial": st,
    }
    ctx.close()
    del b
    torch.cuda.empty_cache()
    return out


def on_device_consumers(torch, g, D, peak, F=1024, steps=5):
    """End to end through host buffers with the frames CONSUMED ON THE DEVICE, so that 622 KB a frame need not cross PCIe
    (`e2e` above is bound by exactly that): packets in, decode, then (a) the reference's yuv420 -> RGB32 conversion fused into
    the decode and the packed pixels out, (b) the GPU encoder (a transcode at another quality) and packets out.  configs[1]
    geometry and stream, F frames a step; pinned host buffers; copies inside the timed region, wall clock."""
    from gmerlin_avdecoder_b200 import capi
    w, h = 720, 576
    stream, offsets, _ = make_workload(F, seed=1)
    desc, _ = g.plan(stream, offsets)
    h_in = torch.from_numpy(stream).pin_memory()
    h_desc = torch.from_numpy(desc.view(np.uint8)).pin_memory()
    d_in = torch.empty(stream.size + g.STREAM_SLACK_BYTES, dtype=torch.uint8, device="cuda")
    d_desc = torch.empty(h_desc.numel(), dtype=torch.uint8, device="cuda")
    out = {}
    st = torch.cuda.current_stream().cuda_stream
    with g.BatchContext(torch.cuda.current_device()) as ctx:
        # (a) decode -> RGB32 on the device -> host
        pitch = w * 4
        d_rgb = torch.empty((F, h, pitch), dtype=torch.uint8, device="cuda")
        h_rgb = torch.empty((F, h, pitch), dtype=torch.uint8).pin_memory()

        def rgb_step():
            d_in[:stream.size].copy_(h_in, non_blocking=True)
            d_desc.copy_(h_desc, non_blocking=True)
            ctx.decode_device_rgb(d_in.data_ptr(), d_desc.data_ptr(), F, w, h, capi.CONV_RGB32, d_rgb.data_ptr(), pitch, h * pitch,
                                  0xFF, None, None, st)
            h_rgb.copy_(d_rgb, non_blocking=True)
            torch.cuda.synchronize()

        # (b) decode -> encode at Q = 64 on the device -> host
        d_yuv = torch.empty((F, w * h * 3 // 2), dtype=torch.uint8, device="cuda")
        cap = stream.size * 2 + (1 << 20)
        d_pk = torch.empty(cap, dtype=torch.uint8, device="cuda")
        d_off = torch.zeros(F + 1, dtype=torch.int64, device="cuda")
        h_pk = torch.empty(cap, dtype=torch.uint8).pin_memory()
        sizes = {}

        def transcode_step():
            d_in[:stream.size].copy_(h_in, non_blocking=True)
            d_desc.copy_(h_desc, non_blocking=True)
            ctx.decode_device(d_in.data_ptr(), d_desc.data_ptr(), F, w, h, d_yuv.data_ptr(), None, st)
            ctx.encoder_config(64, 0, 0, 0)
            ctx.encode_device(d_yuv.data_ptr(), F, w, h, d_pk.data_ptr(), cap, d_off.data_ptr(), st)
            nbytes, overflow = ctx.encode_info()                       # (syncs: the size of what goes back)
            assert not overflow
            h_pk[:nbytes].copy_(d_pk[:nbytes], non_blocking=True)
            torch.cuda.synchronize()
            sizes["out"] = nbytes

        for name, fn in (("decode_rgb32_d2h", rgb_step), ("decode_encode_d2h", transcode_step)):
            fn()
            fn()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            dt = time.perf_counter() - t0
            d2h = int(F * h * pitch) if name == "decode_rgb32_d2h" else int(sizes["out"])
            out[name] = {"value": F * steps / dt, "unit": "frames/s", "frames_per_step": F, "steps": steps,
                         "h2d_bytes_per_step": int(stream.size + h_desc.numel()), "d2h_bytes_per_step": d2h}
    return out


def run_config5(torch, dist, g, D, rank, world, local, steps, peak):
    """configs[4]: one inter-coded 1920x1088 stream, GOP 30, cut at clean frames, one shard per rank."""
    from oracle import oracle as O
    w, h, F = C5_W, C5_H, C5_FRAMES
    fsz = w * h * 3 // 2
    stream, offsets, _ = make_workload(F, seed=7, w=w, h=h, q=C5_Q, key_rate=C5_GOP - 1, lm=2, cm=2)   # the same stream on every rank
    sizes = O.packet_sizes(stream, offsets).astype(np.int64)
    # the cut: the headers' key byte is the hint (0 on the encoder's key frames, include/RTjpeg.h:100-109) ...
    hint = np.array([stream[int(offsets[f]) + 11] == 0 for f in range(F)], dtype=np.uint8)
    first, lead = g.split_shards_lead(hint, world)
    a, b_end = int(first[rank] - lead[rank]), int(first[rank + 1])
    ctx = g.BatchContext(local)
    verified = False
    while True:
        sub = stream[int(offsets[a]):int(offsets[b_end])]
        rel = (offsets[a:b_end + 1] - offsets[a]).astype(np.uint64)
        desc, _ = g.plan(sub, rel)
        bt = D.upload(sub, desc, w, h, device=local)
        D.decode(ctx, bt)
        torch.cuda.synchronize()
        assert ctx.batch_info().bad_frames == 0
        # ... K1's skip count of the shard's first frame is the proof: a frame without skip markers rewrites everything
        if a == 0 or ctx.skip_counts(1)[0] == 0:
            verified = True
            break
        a2 = a - 1                                       # the hint lied (key frames with skips): lead back to the hint before
        while a2 > 0 and not hint[a2]:
            a2 -= 1
        a = a2
    keep0 = int(first[rank]) - a                          # frames decoded only to rebuild the shard's first picture
    for _ in range(3):
        D.decode(ctx, bt)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ms, launches = time_steps(torch, D, ctx, bt, steps, sync)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / steps
    # bit-exactness of this rank's shard on its last GOP, against the oracle decoding that GOP on the host
    g0 = max(k for k in range(int(first[rank]), b_end) if hint[k]) if b_end > int(first[rank]) else b_end
    ok = True
    if b_end > g0:
        want = O.decode_stream(stream, offsets[g0:b_end + 1], w, h, keep_all=False)
        ok = bool(np.array_equal(bt.out[b_end - a - 1].cpu().numpy(), want))
    okt = torch.tensor([1 if ok and verified else 0], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    payload = int(sizes.sum()) - 12 * F
    algo = payload + F * fsz
    out = {
        "workload": "configs[4]: ONE RTjpeg 1920x1088 YUV420 inter-coded stream (GOP %d, lm=cm=2, Q=%d), %d frames, cut at clean "
                    "frames into %d shards, one per GPU; frames stay on the owning device" % (C5_GOP, C5_Q, F, world),
        "scaling": "strong", "frames": F, "n_gpus": world, "value": F / (ms_step * 1e-3), "unit": "frames/s",
        "ms_per_step": ms_step, "steps": steps,
        "shard_starts": [int(x) for x in first], "lead_frames": [int(x) for x in lead],
        "redundant_frames_this_rank": keep0,
        "payload_bytes_per_frame": payload / F, "planar_bytes_per_frame": fsz,
        "algorithmic_GBps_total": algo / (ms_step * 1e-3) / 1e9,
        "per_gpu_hbm_frac": algo / world / (ms_step * 1e-3) / 1e9 / peak,
        "cut": "header key hints, verified on the device: skip count of every shard's first frame is 0",
        "bit_exact_last_frame_of_every_shard_vs_reference": bool(okt.item()),
        "gpu_launches_this_rank": launches,
        "collectives_in_data_path": 0,
    }
    if rank == 0 and O.have_ref():
        threads = host_threads()
        gops = list(range(0, F, C5_GOP)) + [F]
        sample = min(F, 240)
        segs = [x for x in gops if x <= sample]
        reference_decode_fps(stream, offsets, sample, threads, 1, w, h, segments=segs)
        fps = reference_decode_fps(stream, offsets, sample, threads, 3, w, h, segments=segs)
        out["cpu_reference"] = {"value": statistics.median(fps), "unit": "frames/s", "cores": threads, "kind": "reference",
                                "sample": f"median of 3 passes over the first {sample} frames, whole GOPs per thread, "
                                          f"unmodified lib/RTjpeg.c, {threads} threads", "all": fps}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES, help="frames per GPU per step (default: the metric's 4096)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="host-path steps (default: min(steps, 10))")
    ap.add_argument("--cpu-sample", type=int, default=2048, help="frames per CPU-baseline pass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step decoded to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import gmerlin_avdecoder_b200 as g
    from gmerlin_avdecoder_b200 import device as D
    from oracle import oracle as O

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the decoder has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    F = args.frames
    fsz = W * H * 3 // 2
    stream, offsets, gen_s = make_workload(F, seed=1 + rank)
    desc, _ = g.plan(stream, offsets)
    ctx = g.BatchContext(local)
    batch = D.upload(stream, desc, W, H, device=local)
    algo_bytes = batch.payload_bytes + F * fsz            # SURVEY.md section 8d: payload read + planes written

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident steps: the library's default arrangement ---------------------------------
    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(warmup):
        D.decode(ctx, batch)
    barrier()
    info = ctx.batch_info()
    assert info.bad_frames == 0
    ms, launches = time_steps(torch, D, ctx, batch, args.steps, barrier)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batch.out)

    t_ms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = world * F * args.steps / (ms_max * 1e-3)

    # ---- the stages alone (serial arrangement), for the roofline of the dominant kernel ------------
    stage_ms = stage_times(torch, g, D, ctx, batch, min(args.steps, 20))

    # ---- end to end through the host entry point -----------------------------------------------
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    h_in = torch.from_numpy(stream).pin_memory()
    h_out = torch.empty((F, fsz), dtype=torch.uint8).pin_memory()
    flags = g.HOST_IN_PINNED | g.HOST_OUT_PINNED
    ctx.decode_host(h_in.numpy(), offsets, h_out.numpy(), flags=flags)          # warm-up (allocations)
    ctx.decode_host(h_in.numpy(), offsets, h_out.numpy(), flags=flags)
    barrier()
    l0 = ctx.launch_count()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.decode_host(h_in.numpy(), offsets, h_out.numpy(), flags=flags)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_launches = ctx.launch_count() - l0
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * F * e2e_steps / float(t_e.item())
    # the host path's last chunk must equal the device path's frames (same bytes, two routes)
    assert torch.equal(h_out[-1].cuda(), batch.out[-1]), "host path and device path disagree"
    del h_out, h_in

    peak, peak_src = measured_hbm_peak()
    line = None
    if rank == 0:
        facts = ncu_facts()
        sm_hz = (clocks.get("sm_mhz") or 1965) * 1e6
        k2_ms = stage_ms["idct"]
        achieved = algo_bytes / (k2_ms * 1e-3) / 1e9

        def issue_frac(kernel, ms_):
            inst = facts.get(kernel, {}).get("warp_instructions_per_launch_configs1")
            return None if not inst or F != FRAMES else inst / (SM_SUBPARTITIONS * sm_hz * ms_ * 1e-3)

        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": config_dict(batch.payload_bytes / F, F),
            "arrangement": "rtjgpu_set_pipeline AUTO = serial: K1 (rtj_scan_sync_kernel, + the chunk kernel for frames it hands over), K3, K2, K2b one after the other on the caller's stream",
            "clocks": clocks,
            "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "frames/s", "steps": e2e_steps,
                    "h2d_bytes_per_step": int(stream.size + desc.nbytes), "d2h_bytes_per_step": int(F * fsz),
                    "gpu_launches": e2e_launches,
                    "api": "rtjgpu_decode_host, pinned host buffers in and out"},
            "roofline": {
                "bound": "hbm", "kernel": "K2 rtj_idct_kernel + K2b rtj_idct_hard_kernel (one event bracket; K2b is ~4 % of it)",
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": facts.get("rtj_idct_kernel", {}).get("dram_bytes_per_launch_configs1"),
                "traffic_source": facts.get("source"),
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes,
                "kernel_ms": k2_ms,
                "timed": "alone: %d separate steps in the serial arrangement, CUDA events between the stages on the launch stream"
                         % min(args.steps, 20),
                "stage_ms_serial": stage_ms,
                "whole_path_frac": algo_bytes / (ms_max / args.steps * 1e-3) / 1e9 / peak,
                "whole_path_frac_serial": algo_bytes / (stage_ms["total"] * 1e-3) / 1e9 / peak,
                "int_issue_frac": {
                    "what": "warp instructions per launch (one committed ncu capture) / (592 SM sub-partitions x SM clock "
                            "x this run's kernel time): share of the issue slots used",
                    "K1": issue_frac("rtj_scan_sync_kernel", stage_ms["scan"]),
                    "K2": issue_frac("rtj_idct_kernel", k2_ms),
                    "whole_path": (None if F != FRAMES or not facts.get("rtj_idct_kernel", {}).get("warp_instructions_per_launch_configs1")
                                   or not facts.get("rtj_scan_sync_kernel", {}).get("warp_instructions_per_launch_configs1")
                                   else (facts["rtj_idct_kernel"]["warp_instructions_per_launch_configs1"]
                                         + facts["rtj_scan_sync_kernel"]["warp_instructions_per_launch_configs1"])
                                   / (SM_SUBPARTITIONS * sm_hz * ms_max / args.steps * 1e-3)),
                },
            },
        }
        if world == 1 and not args.no_cpu_baseline and O.have_ref():
            threads = host_threads()
            sample = min(F, args.cpu_sample)
            reference_decode_fps(stream, offsets, sample, threads, 2)             # warm the threads and the caches
            fps = reference_decode_fps(stream, offsets, sample, threads, 5)
            line["cpu_baseline"] = {
                "value": statistics.median(fps), "unit": "frames/s", "cores": threads, "kind": "reference",
                "sample": f"median of 5 passes (after 2 warm-up passes) over the first {sample} frames of the same batch, "
                          f"unmodified lib/RTjpeg.c RTjpeg_decompress, {threads} threads each with a private decoder",
                "all": fps,
            }
    ctx.close()
    del batch
    torch.cuda.empty_cache()

    if rank == 0 and world == 1 and not args.no_other_configs:
        sm_hz = (clocks.get("sm_mhz") or 1965) * 1e6
        line["other_configs"] = [
            other_config(torch, g, D, "configs[2]: 720x576 inter GOP 30, lm=cm=1", 720, 576, 128, 2048, peak, sm_hz, key_rate=29, lm=1, cm=1),
            other_config(torch, g, D, "configs[2]: 720x576 inter GOP 30, lm=cm=4", 720, 576, 128, 2048, peak, sm_hz, key_rate=29, lm=4, cm=4),
            other_config(torch, g, D, "configs[1] at Q=32", 720, 576, 32, 2048, peak, sm_hz),
            other_config(torch, g, D, "configs[1] at Q=255 (raw prefix 9)", 720, 576, 255, 1024, peak, sm_hz),
            other_config(torch, g, D, "configs[3]: 1920x1088 Q=255 dense", 1920, 1088, 255, 128, peak, sm_hz, steps=5,
                         noise_y=60, noise_c=20),
        ]

    if rank == 0 and world == 1 and not args.no_other_configs:
        try:
            line["on_device_consumers"] = on_device_consumers(torch, g, D, peak)
        except Exception as exc:  # noqa: BLE001 -- informational: the line stands without it
            line["on_device_consumers"] = {"error": repr(exc)}

    if not args.no_config5:
        c5 = run_config5(torch, dist, g, D, rank, world, local, max(3, min(args.steps, 20)), peak)
        if rank == 0:
            line["config5"] = c5

    if rank == 0:
        _emit(line)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir: str, frames) -> None:
    """What a caller of the device path receives, the decoded frames [F, w*h*3/2] in HBM, sampled to 16 frames chosen by a
    fixed seed (40 MB as float32) plus the byte sum of every frame, so that two builds can be compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    F = frames.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(F, size=min(F, 16), replace=False))
    np.save(os.path.join(out_dir, "frame_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "frames.npy"), frames[torch.from_numpy(idx).to(frames.device)].cpu().numpy().astype(np.float32))
    # a few frames at a time: the int64 sum of the whole batch at once would need a temporary of 8 bytes per pixel
    sums = torch.cat([frames[i:i + 64].sum(dim=1, dtype=torch.int64) for i in range(0, F, 64)])
    np.save(os.path.join(out_dir, "frame_sums.npy"), sums.cpu().numpy().astype(np.float64))


def _emit(line: dict) -> None:
    """The one JSON line, on the process's real stdout."""
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


_REAL_STDOUT = sys.stdout

if __name__ == "__main__":
    # Libraries write banners to file descriptor 1 (NCCL prints "NCCL version ..." there when its communicator comes up):
    # everything that is not the JSON line goes to stderr instead.
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    main()
