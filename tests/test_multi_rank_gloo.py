"""The N>1 path on CPU: two ranks over gloo, each owning one shard of an inter-coded stream.

The data path has no collective (SURVEY.md section 8e): a batch is cut on the host at clean
frames (rtjgpu_split_shards_lead) and every rank decodes its shard from nothing.  What can be
checked without a GPU is the host-side logic: that every rank derives the same cut from the
same per-frame skip counts, that the shards tile the batch, that a shard which cannot start on
a clean frame leads back to one, and that decoding the shards independently reproduces the
sequential picture sequence.  The ORACLE stands in for the decoder here -- as the checker, the
only role it is allowed.  The CUDA decode of independently started shards is what
tests/test_gpu_shards.py checks on the GPU box, and bench.py's `config5` leg times it with one
rank per GPU."""
import hashlib
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import gmerlin_avdecoder_b200 as g
from oracle import oracle as O
from streams import golden


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _clean_frames(s, o, w, h, Q):
    t = O.tables_from_quality(Q)
    sizes = O.packet_sizes(s, o)
    nmb = (w // 16) * (h // 16)
    return np.array([(O.walk_payload(s[int(o[f]) + 12:int(o[f]) + int(sizes[f])], nmb, t.lb8, t.cb8)[2] != 0).all()
                     for f in range(len(o) - 1)], dtype=np.uint8)


def _rank_main(rank, world, port, name, w, h, Q, out_dir, mask_clean):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        gd = golden(name)
        s, o = gd["stream"], gd["offsets"]
        F = len(o) - 1
        clean = _clean_frames(s, o, w, h, Q)
        if mask_clean:                                          # pretend the clean frames near the cut are not: the shard must lead back
            clean = clean.copy()
            clean[F // 2 - 2:F // 2 + 3] = 0
        first, lead = g.split_shards_lead(clean, world)         # every rank computes the same cut
        cuts = [torch.zeros(2 * world + 1, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(cuts, torch.from_numpy(np.concatenate([first, lead])))
        assert all(torch.equal(c, cuts[0]) for c in cuts)
        a, b = int(first[rank]), int(first[rank + 1])
        assert b > a and (not mask_clean or rank == 0 or lead[rank] > 0)
        lo = a - int(lead[rank])
        garbage = np.full(w * h * 3 // 2, 0xA5, dtype=np.uint8)   # a shard that does not start at frame 0 starts from anything
        frames = O.decode_stream(s, o[lo:b + 1], w, h, init=None if lo == 0 else garbage)[a - lo:]
        # per-frame digests travel, the frames stay where they were decoded
        dig = torch.zeros(F, 16, dtype=torch.uint8)
        for i in range(b - a):
            dig[a + i] = torch.frombuffer(bytearray(hashlib.md5(frames[i].tobytes()).digest()), dtype=torch.uint8)
        dist.all_reduce(dig, op=dist.ReduceOp.SUM)                # shards are disjoint: a sum is a gather
        done = torch.tensor([b - a], dtype=torch.int64)
        dist.all_reduce(done, op=dist.ReduceOp.SUM)
        if rank == 0:
            assert int(done.item()) == F                          # the shards tile the batch
            whole = O.decode_stream(s, o, w, h)
            for f in range(F):
                want = np.frombuffer(hashlib.md5(whole[f].tobytes()).digest(), dtype=np.uint8)
                assert np.array_equal(dig[f].numpy(), want), f"frame {f} differs between sharded and sequential decode"
            open(os.path.join(out_dir, "ok"), "w").write("%d %d" % (a, b))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mask_clean", [False, True])
@pytest.mark.parametrize("name,w,h,Q", [("inter_64x48_q200_gop6", 64, 48, 200)])
def test_two_ranks_decode_disjoint_shards(tmp_path, name, w, h, Q, mask_clean):
    world = 2
    mp.spawn(_rank_main, args=(world, _free_port(), name, w, h, Q, str(tmp_path), mask_clean), nprocs=world, join=True)
    assert (tmp_path / "ok").exists()


@pytest.mark.skipif(not O.have_ref(), reason="reference build absent (oracle/_ref): the arm times the reference's own decoder")
def test_reference_arm_runs_on_rank_zero_only(tmp_path):
    """bench.py --impl reference under a multi-rank launch: rank 0 prints the line, the others exit 0."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0", "--frames", "16", "--cpu-sample", "16"],
                       env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ""
    env["RANK"] = "0"; env["LOCAL_RANK"] = "0"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0", "--frames", "16", "--cpu-sample", "16"],
                       env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "reference"
