#!/usr/bin/env python
"""Own-alignment STC-007 stitching (STC007DataStitcher.doFrameReassembleAuto) sharded over N GPUs by sharding.stitch_shard.

  torchrun --nproc_per_node N tools/bench_stitch_shards.py [--frames F] [--steps K] [--warmup W] [--cwd] [--stitch-warmup K]

Workload: the config-5 clean tape (bench.py's periodic PAL 720x576 segment repeated to --frames frames), field order and video
standard preset (PAL / TFF, 14 bit, P+Q), CWD as --cwd says.  Each rank decodes its own frames to line records once, outside
the timed region; a step is stitch_shard over the rank's records: record exchange, warm-up, the shard, the verify gather and any
redo.  Prints one JSON line: stitched lines/s per step (CUDA events, the slowest rank), the warm-up share of the step, redo
rounds and redone ranks, the card's name and power limit (read in the same run), and a blake2b digest of the gathered sample
stream + flags, which must be the same at every N.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card_info(index):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")[:2]]
        return {"name": name, "power_limit": limit}
    except Exception as e:      # noqa: BLE001 -- reported, not fatal
        return {"name": None, "power_limit": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--period", type=int, default=30)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--cwd", action="store_true")
    ap.add_argument("--stitch-warmup", type=int, default=None, help="frames of the state warm-up (default sharding.STITCH_WARMUP_FRAMES)")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    from sdvpcmdecoder_b200 import operators as ops, sharding, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    tr = sharding.DistTransport(rank, world)
    seg = synth.make_stc007(args.period, seed=1234, periodic=True)["luma"]
    n, H = args.frames, seg.shape[1]
    a, b = sharding.frame_range(n, rank, world)
    luma = np.ascontiguousarray(np.concatenate([seg[f % args.period][None] for f in range(a, b)]))
    h = ops.capi.Handle(local)
    recs = ops.VideoToDigital(h).doBinarize(torch.from_numpy(luma).cuda())
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(1); st.setResolutionPreset(False); st.setCWDCorrection(args.cwd)
    kw = {} if args.stitch_warmup is None else {"warmup": args.stitch_warmup}
    torch.cuda.synchronize()

    def step():
        return sharding.stitch_shard(st, recs, n, H, tr, video_std=1, **kw)
    for _ in range(args.warmup):
        step()
    ms, warm, rounds, redone = [], [], [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        out, stats = step()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1), stats["warmup_s"] * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms.append(float(t[0])); warm.append(float(t[1]))
        rounds.append(stats["rounds"])
        r = torch.tensor([stats["redone"]], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(r)
        redone.append(int(r))
    # digest of the gathered stream (the last step's output)
    _, s, f, _ = out
    mine = torch.cat([s.reshape(-1).view(torch.uint8), f.reshape(-1)]).contiguous()
    digest = None
    if world > 1:
        sizes = [torch.zeros(2, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([s.numel() * 2, f.numel()], dtype=torch.int64, device="cuda"))
        if rank == 0:
            parts = [mine]
            for g in range(1, world):
                buf = torch.empty(int(sizes[g].sum()), dtype=torch.uint8, device="cuda")
                dist.recv(buf, g)
                parts.append(buf)
        else:
            dist.send(mine, 0)
    else:
        parts, sizes = [mine], [torch.tensor([s.numel() * 2, f.numel()])]
    if rank == 0:
        hs, hf = hashlib.blake2b(digest_size=16), hashlib.blake2b(digest_size=16)
        for p, sz in zip(parts, sizes):
            host = p.cpu().numpy()
            k = int(sz[0])
            hs.update(host[:k].tobytes()); hf.update(host[k:].tobytes())
        digest = {"samples": hs.hexdigest(), "flags": hf.hexdigest()}
        med = float(np.median(ms))
        line = {"tool": "bench_stitch_shards", "gpus": world, "frames": n, "lines": n * H, "cwd": args.cwd,
                "stitch_warmup_frames": args.stitch_warmup or sharding.STITCH_WARMUP_FRAMES,
                "step_ms": ms, "median_ms": med, "lines_per_s": n * H / (med * 1e-3),
                "warmup_share": float(np.median(np.array(warm) / np.array(ms))),
                "redo_rounds": [len(r) for r in rounds], "redone_ranks": redone, "digest": digest, "card": card_info(local)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
