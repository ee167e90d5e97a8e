"""The own-alignment stitcher's shard protocol (sharding.stitch_shard) with 2-4 CPU processes (gloo) and a stub stitcher whose
carried state is a small tensor: which ranks redo in each round, that the hand-off settles within [world] rounds, that a
guess equal to the truth causes no redo, and that the shards' outputs concatenate to the unsharded run."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_FRAMES = 12


class StubStitcher:
    """The three methods stitch_shard uses.  One record per frame; the state after a frame is a hash of every frame of the file
    since its start (memory=None: a wrong guess never heals) or just the last frame's record (memory=1: any warm-up is exact).
    The output of a call is the state after each frame it consumes (file_end = 0 leaves the last frame, as the real stitcher)."""

    def __init__(self, memory):
        self.memory = memory
        self.state = torch.zeros(2, dtype=torch.int64)

    def doFrameReassembleAuto(self, recs, n_frames, height, file_start=True, file_end=True):
        assert height == 1 and recs.shape[0] == n_frames
        if file_start:
            self.state = torch.zeros(2, dtype=torch.int64)
        out = []
        for f in range(n_frames if file_end else n_frames - 1):
            v = int(recs[f, 0])
            s0 = v if self.memory == 1 else (int(self.state[0]) * 31 + v) % 1000003
            self.state = torch.tensor([s0, 1], dtype=torch.int64)
            out.append(self.state.clone())
        return torch.stack(out) if out else torch.zeros((0, 2), dtype=torch.int64)

    def saveState(self):
        return self.state.clone()

    def loadState(self, t):
        self.state = t.clone()


def _tape():
    return (torch.arange(N_FRAMES, dtype=torch.int64) * 7919 % 1009 + 1).reshape(-1, 1)


def _worker(rank, world, port, out_dir, memory, warmup):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sdvpcmdecoder_b200 import sharding
    a, b = sharding.frame_range(N_FRAMES, rank, world)
    out, stats = sharding.stitch_shard(StubStitcher(memory), _tape()[a:b].clone(), N_FRAMES, 1, sharding.DistTransport(), warmup=warmup)
    torch.save({"out": out, "rounds": stats["rounds"], "redone": stats["redone"], "warmup_frames": stats["warmup_frames"]},
               os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def _run(tmp_path, world, memory, warmup, port_ofs):
    sys.path.insert(0, ROOT)
    port = 28600 + (os.getpid() % 300) * 8 + port_ofs
    mp.spawn(_worker, args=(world, port, str(tmp_path), memory, warmup), nprocs=world, join=True)
    res = [torch.load(os.path.join(str(tmp_path), f"rank{r}.pt")) for r in range(world)]
    whole = StubStitcher(memory).doFrameReassembleAuto(_tape(), N_FRAMES, 1)
    assert torch.equal(torch.cat([r["out"] for r in res]), whole)
    assert all(r["rounds"] == res[0]["rounds"] for r in res), "every rank must see the same rounds"
    return res


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3, 4])
def test_wrong_guesses_settle_rank_by_rank(tmp_path, world):
    """A state that never heals and a warm-up too short to reach the file start: every rank but 0 guesses wrong, and in round r
    the ranks from r+1 on redo (each one's predecessor changed its end state in round r-1); done within [world] rounds."""
    res = _run(tmp_path, world, None, 2, world)
    rounds = res[0]["rounds"]
    assert rounds == [list(range(r + 1, world)) for r in range(world - 1)]
    assert len(rounds) <= world
    assert [r["redone"] for r in res] == [min(g, world - 1) if g else 0 for g in range(world)]


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 4])
def test_guess_equal_to_truth_causes_no_redo(tmp_path, world):
    """The state heals after one frame, so a 2-frame warm-up guesses right: one gather, no redo."""
    res = _run(tmp_path, world, 1, 2, 10 + world)
    assert res[0]["rounds"] == [] and all(r["redone"] == 0 for r in res)


@pytest.mark.timeout(300)
def test_warmup_from_the_file_start_is_exact(tmp_path):
    """A warm-up that reaches frame 0 (records passed along the ranks when shards are shorter than it) starts where the file
    starts: exact by construction, even for a state that never heals."""
    res = _run(tmp_path, 4, None, 70, 20)
    assert res[0]["rounds"] == []
    assert [r["warmup_frames"] for r in res] == [0, 3, 6, 9]
