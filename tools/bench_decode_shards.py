#!/usr/bin/env python
"""Line decode (VideoToDigital.doBinarize) sharded over N GPUs: the plain sharded decode (every shard starts its chain empty, what
bench.py measures) against sharding.decode_shard (the chain state handed from shard to shard, exact).

  torchrun --nproc_per_node N tools/bench_decode_shards.py [--frames F] [--steps K] [--warmup W] [--decode-warmup K]
  python tools/bench_decode_shards.py --local-ranks N ...    (N handles on one GPU as ranks, threads: protocol counts, not speed)

Workload: the config-5 clean tape (bench.py's periodic PAL 720x576 segment repeated to --frames frames), MODE_NORMAL, duplicate
check on.  Each rank holds its own frames in device memory.  A step of the plain decode is one doBinarize over them; a step of
decode_shard is the luma hand-over, the warm-up decode, the shard, the state saves, the verify gather and any redo.  Prints one
JSON line: per-step times of both (CUDA events, the slowest rank), the warm-up, save and verify parts of decode_shard, redo
rounds and redone ranks, whether decode_shard's records equal the plain shards' (they may differ at the shard heads), and the card's name and power limit (read in the
same run).
"""
from __future__ import annotations

import argparse
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


def rank_body(args, tr, device, reduce_max):
    """The measurement on one rank; reduce_max(list of floats) -> the maximum over the ranks."""
    import torch
    from sdvpcmdecoder_b200 import operators as ops, sharding, synth
    rank, world = tr.rank, tr.world
    seg = synth.make_stc007(args.period, seed=1234, periodic=True)["luma"]
    n = args.frames
    a, b = sharding.frame_range(n, rank, world)
    luma = torch.from_numpy(np.ascontiguousarray(np.concatenate([seg[f % args.period][None] for f in range(a, b)]))).to(device)
    v2d = ops.VideoToDigital(ops.capi.Handle(device.index))
    kw = {} if args.decode_warmup is None else {"warmup": args.decode_warmup}
    edges = [sharding.frame_range(n, g, world)[0] for g in range(world)] + [n]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        torch.cuda.synchronize(device)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize(device)
        return out, e0.elapsed_time(e1)
    res = {"plain_ms": [], "shard_ms": [], "warmup_ms": [], "save_ms": [], "verify_ms": [], "rounds": [], "redone": []}
    plain = shard = None
    for i in range(args.warmup + args.steps):
        plain, t_plain = timed(lambda: v2d.doBinarize(luma))
        (shard, stats), t_shard = timed(lambda: sharding.decode_shard(v2d, luma, tr, edges=edges, **kw))
        m = reduce_max([t_plain, t_shard, stats["warmup_s"] * 1e3, stats["save_s"] * 1e3, stats["verify_s"] * 1e3, float(stats["redone"])])
        if i >= args.warmup:
            for k, v in zip(("plain_ms", "shard_ms", "warmup_ms", "save_ms", "verify_ms"), m[:5]):
                res[k].append(v)
            res["rounds"].append(len(stats["rounds"]))
            res["redone"].append(int(m[5]))
    res["equal_to_plain"] = bool(torch.equal(plain, shard))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--period", type=int, default=30)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--decode-warmup", type=int, default=None, help="frames of the chain warm-up (default sharding.DECODE_WARMUP_FRAMES)")
    ap.add_argument("--local-ranks", type=int, default=0, help="N > 0: N handles on GPU 0 as ranks (threads), no torch.distributed")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    from sdvpcmdecoder_b200 import sharding

    if args.local_ranks > 0:
        world, local = args.local_ranks, 0
        hub = sharding.LocalTransport(world)
        slots = [None] * world

        def fn(tr):
            def reduce_max(v):
                g = tr.all_gather(torch.tensor(v, dtype=torch.float64))
                return g.max(dim=0).values.tolist()
            slots[tr.rank] = rank_body(args, tr, torch.device("cuda", 0), reduce_max)
        hub.run(fn)
        res, rank = slots[0], 0
        res["equal_to_plain"] = all(s["equal_to_plain"] for s in slots)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        rank = int(os.environ.get("RANK", "0"))
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        if world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        tr = sharding.DistTransport(rank, world)

        def reduce_max(v):
            t = torch.tensor(v, dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.tolist()
        res = rank_body(args, tr, torch.device("cuda", local), reduce_max)
        if world > 1:
            ok = torch.tensor([int(res["equal_to_plain"])], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            res["equal_to_plain"] = bool(ok.item())
    if rank == 0:
        med = {k: float(np.median(res[k])) for k in ("plain_ms", "shard_ms", "warmup_ms", "save_ms", "verify_ms")}
        line = {"tool": "bench_decode_shards", "gpus": world, "local_ranks": args.local_ranks, "frames": args.frames,
                "decode_warmup_frames": sharding.DECODE_WARMUP_FRAMES if args.decode_warmup is None else args.decode_warmup,
                "median": med, "steps": {k: res[k] for k in ("plain_ms", "shard_ms", "warmup_ms", "save_ms", "verify_ms")},
                "redo_rounds": res["rounds"], "redone_ranks": res["redone"],
                "shard_records_equal_plain": res["equal_to_plain"], "card": card_info(local)}
        print(json.dumps(line), flush=True)
    if args.local_ranks == 0 and world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
