"""Frame-range sharding of a tape over the ranks of one node (one process per GPU, torch.distributed).

The decode path shards by contiguous frame ranges.  The plain sharded line decode needs nothing from the neighbours (each
shard starts its VideoToDigital chain empty, exactly like the reference at file start); decode_shard instead hands the chain
state from shard to shard, so that the shards equal one call over the whole tape.  The STC-007 deinterleaver reads 112 lines
ahead (7 x 16 lines, stc007datablock.h:44-58), so shard g needs the first 112 line records of shard g+1: one small
point-to-point message per boundary (NCCL send/recv over NVLink on GPUs, gloo in the CPU tests).  The one thing that
flows the other way is the stitcher's broken-block countdown: a BROKEN block near the end of shard g masks the first blocks
of shard g+1 (carry_countdowns: one 8-byte all_gather per decode, a second round only for the shards it affects).
Samples stay sharded.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

HALO_LINES = 112            # STC007DataBlock::MIN_DEINT_DATA
LEAD_IN_LINES = 80          # lines queued ahead of the first frame of a file (stc007datastitcher.cpp:4733-4737)


def frame_range(n_frames: int, rank: int, world: int):
    """Frames [a, b) of the tape decoded by this rank."""
    return rank * n_frames // world, (rank + 1) * n_frames // world


def shard_lead_in(rank: int) -> int:
    """Only the first shard carries the file's lead-in lines."""
    return LEAD_IN_LINES if rank == 0 else 0


def first_block(n_frames: int, rank: int, world: int, lines_per_field: int) -> int:
    """Index, in the unsharded block stream, of this rank's first data block."""
    a, _ = frame_range(n_frames, rank, world)
    return 0 if rank == 0 else LEAD_IN_LINES + a * 2 * lines_per_field


def block_count(n_frames: int, rank: int, world: int, lines_per_field: int) -> int:
    a, b = frame_range(n_frames, rank, world)
    return shard_lead_in(rank) + (b - a) * 2 * lines_per_field


def exchange_halo(recs: torch.Tensor, halo: torch.Tensor | None, rank: int, world: int):
    """Send this shard's first 112 line records to the previous rank, receive the next rank's into [halo].

    recs: [n_lines, 32] uint8 record buffer of this shard; halo: [112, 32] uint8 (None on the last rank).
    Returns [halo] (None on the last rank)."""
    return exchange_halo_finish(exchange_halo_start(recs, halo, rank, world), halo, rank, world)


def exchange_halo_start(recs: torch.Tensor, halo: torch.Tensor | None, rank: int, world: int):
    """First half of exchange_halo(): post the send / receive and return the requests.  Only the shard's first 112 line
    records need to be final -- VideoToDigital.doBinarize(on_first_frame=...) calls back at that point, while the rest of
    the shard is still being decoded."""
    if world == 1:
        return []
    ops = []
    if rank > 0:
        ops.append(dist.P2POp(dist.isend, recs[:HALO_LINES], rank - 1))
    if rank < world - 1:
        ops.append(dist.P2POp(dist.irecv, halo, rank + 1))
    return dist.batch_isend_irecv(ops) if ops else []


def exchange_halo_finish(reqs, halo: torch.Tensor | None, rank: int, world: int):
    for r in reqs:
        r.wait()
    return halo if (world > 1 and rank < world - 1) else None


def carry_countdowns(state: dict, redo, rank: int, world: int, device=None) -> dict:
    """Hand the broken-block countdown from shard to shard.

    STC007DataStitcher::broken_countdown is a member (stc007datastitcher.cpp:79, 6785-6863): a BROKEN block within the last
    broken_mask_dur blocks of shard g masks the first blocks of shard g+1.  Every rank runs its deinterleave pass first with
    countdown_in = 0 (all ranks at once); [state] is what the library reports for that pass (STC007DataStitcher.countdown():
    countdown_in / countdown_out / depends_on_in).  Then, the same on every rank: gather all countdown_out; the true input
    of rank g is the output of rank g-1; ranks whose input was something else call redo(countdown_in) -> new state (the
    library only redoes the blocks inside the windows) and the gather repeats.  Rank 0's output is final from the start,
    rank 1's after one round, ...: at most [world] rounds, one round (a single 8-byte all_gather) on a tape without
    BROKEN blocks near the shard boundaries.  Returns the final state of this rank."""
    if world == 1:
        return state
    used = [0] * world
    for _ in range(world + 1):
        mine = torch.tensor([int(state["countdown_out"]), int(bool(state["depends_on_in"]))], dtype=torch.int32, device=device)
        allv = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        outs = [int(v[0]) for v in allv]
        want = [0] + outs[:-1]
        changed = [g for g in range(world) if want[g] != used[g]]
        if not changed:
            return state
        if rank in changed:
            state = redo(want[rank])
        used = want
    raise RuntimeError("countdown hand-off did not settle")


def carry_countdowns_device(state_dev: torch.Tensor, gathered: torch.Tensor, redo, rank: int, world: int) -> int:
    """carry_countdowns() for the GPU path: [state_dev] is the int32[4] device tensor STC007DataStitcher.countdown_to() filled
    (countdown_in, countdown_out, windows, depends), [gathered] an int32 [world, 4] device tensor.  One all_gather over NCCL
    straight from device memory and one read-back per round; redo(countdown_in) runs the deinterleave call again and refills
    [state_dev].  Returns the number of rounds in which this rank had to redo its windows (0 on a tape without BROKEN blocks at
    the shard boundaries)."""
    if world == 1:
        return 0
    used = [0] * world
    redone = 0
    for _ in range(world + 1):
        dist.all_gather_into_tensor(gathered.view(-1), state_dev.view(-1)[:4].contiguous())
        outs = [int(v) for v in gathered.view(world, 4)[:, 1].cpu()]
        want = [0] + outs[:-1]
        changed = [g for g in range(world) if want[g] != used[g]]
        if not changed:
            return redone
        if rank in changed:
            redo(want[rank])
            redone += 1
        used = want
    raise RuntimeError("countdown hand-off did not settle")


class CountdownHandoff:
    """carry_countdowns_device() without a host round trip in the step: post() gathers the countdown states over NCCL and starts
    their copy into pinned host memory (nothing blocks); settle() -- called when the host synchronises with the device anyway,
    e.g. at the start of the next step, and before the results are used -- looks at the copy and runs the redo rounds if a
    shard's predecessor left a window open (never on a tape without BROKEN blocks at the shard boundaries)."""

    def __init__(self, rank: int, world: int, device):
        self.rank, self.world = rank, world
        self.gathered = torch.zeros((world, 4), dtype=torch.int32, device=device)
        self.host = torch.zeros((world, 4), dtype=torch.int32).pin_memory()
        self.event = torch.cuda.Event()
        self.pending = None
        self.redone = 0

    def post(self, state_dev: torch.Tensor, redo):
        if self.world == 1:
            return
        dist.all_gather_into_tensor(self.gathered.view(-1), state_dev.view(-1)[:4].contiguous())
        self.host.copy_(self.gathered, non_blocking=True)
        self.event.record()
        self.pending = (state_dev, redo)

    def settle(self):
        if self.pending is None:
            return
        state_dev, redo = self.pending
        self.pending = None
        self.event.synchronize()
        outs = [int(v) for v in self.host[:, 1]]
        used = [0] * self.world
        for _ in range(self.world + 1):
            want = [0] + outs[:-1]
            changed = [g for g in range(self.world) if want[g] != used[g]]
            if not changed:
                return
            if self.rank in changed:
                redo(want[self.rank])
                self.redone += 1
            used = want
            dist.all_gather_into_tensor(self.gathered.view(-1), state_dev.view(-1)[:4].contiguous())
            outs = [int(v) for v in self.gathered[:, 1].cpu()]
        raise RuntimeError("countdown hand-off did not settle")


# ---- the own-alignment stitcher (STC007DataStitcher.doFrameReassembleAuto) over frame shards
#
# Its carried state (previous frame, 65-entry order / resolution histories, countdown, the last 112 queued lines) depends on
# the whole tape before a shard, so each shard guesses it and the guesses are verified: rank g stitches the K frames in front of
# its first frame from a file start (a warm-up whose output is thrown away), continues over its own frames from the state that
# leaves, then compares that state with the end state of rank g-1.  The states are canonical blobs (saveState), so equality is
# byte equality.  A rank whose guess was wrong loads the true state and runs again; rank 0 is exact, so after round r the
# first r+1 shards are final: at most [world] rounds.

STITCH_WARMUP_FRAMES = 70       # the 65-entry histories refill, plus a margin


class DistTransport:
    """Records and state blobs between the ranks of a torch.distributed process group (NCCL from device memory, gloo on CPUs)."""

    def __init__(self, rank: int | None = None, world: int | None = None):
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world

    def send(self, t: torch.Tensor, dst: int):
        dist.send(t.contiguous(), dst)

    def recv(self, t: torch.Tensor, src: int):
        dist.recv(t, src)

    def all_gather(self, t: torch.Tensor) -> torch.Tensor:
        out = [torch.empty_like(t) for _ in range(self.world)]
        dist.all_gather(out, t.contiguous())
        return torch.stack(out)


class LocalTransport:
    """Ranks as threads of one process (several handles on one GPU): what DistTransport does, through in-process mailboxes.
    LocalTransport(world).run(fn) calls fn(transport of rank r) for every rank at once and returns the results in rank order."""

    def __init__(self, world: int, timeout: float = 600.0):
        import queue
        import threading
        self.world, self.timeout = world, timeout
        self._boxes = {(s, d): queue.Queue() for s in range(world) for d in range(world)}
        self._barrier = threading.Barrier(world, timeout=timeout)
        self._slots = [None] * world

    class _Rank:
        def __init__(self, hub, rank):
            self.hub, self.rank, self.world = hub, rank, hub.world

        def send(self, t, dst):
            self.hub._boxes[(self.rank, dst)].put(t.clone())

        def recv(self, t, src):
            import queue
            import time
            end = time.monotonic() + self.hub.timeout
            while True:     # (in slices, so that a rank that failed ends the others' waits)
                if self.hub._barrier.broken:
                    raise RuntimeError("another rank failed")
                try:
                    t.copy_(self.hub._boxes[(src, self.rank)].get(timeout=0.5))
                    return
                except queue.Empty:
                    if time.monotonic() > end:
                        raise

        def all_gather(self, t):
            self.hub._slots[self.rank] = t.clone()
            self.hub._barrier.wait()
            out = torch.stack(self.hub._slots)
            self.hub._barrier.wait()
            return out

    def run(self, fn):
        import threading
        results, errors = [None] * self.world, []

        def body(r):
            try:
                results[r] = fn(LocalTransport._Rank(self, r))
            except BaseException as e:      # noqa: BLE001 -- re-raised below; the others must not wait for this rank
                errors.append(e)
                self._barrier.abort()
        threads = [threading.Thread(target=body, args=(r,)) for r in range(self.world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return results


def stitch_shard(stitcher, recs: torch.Tensor, n_frames: int, lines_per_frame: int, transport,
                 warmup: int = STITCH_WARMUP_FRAMES, edges=None, **stitch_kw):
    """Own-alignment stitching of this rank's frames [a, b) = frame_range(n_frames, rank, world) so that the shards' outputs
    concatenate to one doFrameReassembleAuto call over the whole tape.

    stitcher: an STC007DataStitcher on this rank's handle (doFrameReassembleAuto, saveState, loadState); recs: the line records of
    frames [a, b) ([(b-a)*lines_per_frame, 32]); transport: DistTransport or LocalTransport rank; edges: world+1 frame indices
    [0, a_1, .., n_frames] for shards other than frame_range's; stitch_kw goes to doFrameReassembleAuto.
    Steps: (1) receive the records of the [warmup] frames before a from rank-1 (passed along when shards are shorter) and of
    frame b from rank+1, the frame the stitcher looks ahead to; (2) warm-up: frames [a-warmup, a] from a file start,
    output discarded, its end state is the guess at a (exact when a-warmup <= 0); (3) continue over [a, b] (the last rank over [a, n)
    with file_end), save the end state; (4) all-gather (state started from, end state) of every rank, redo the ranks whose start
    differs from their predecessor's end, repeat until none does.
    Returns (the doFrameReassembleAuto output of the final run, stats): the shard's blocks start at the first of the 112 lines
    carried in from rank-1 (rank 0: at the lead-in); stats = warmup_frames, warmup_s, total_s, rounds (the ranks redone in each
    round), redone (runs of this rank after the first)."""
    import time
    rank, world, H = transport.rank, transport.world, lines_per_frame
    if edges is None:
        edges = [frame_range(n_frames, g, world)[0] for g in range(world)] + [n_frames]
    if len(edges) != world + 1 or edges[0] != 0 or edges[-1] != n_frames or any(edges[g + 1] <= edges[g] for g in range(world)):
        raise ValueError("every shard needs at least one frame, and the shards must cover the tape")
    a, b = edges[rank], edges[rank + 1]
    if recs.shape[0] != (b - a) * H:
        raise ValueError("recs must hold the line records of this rank's frames")
    t0 = time.perf_counter()
    # (1) records
    k = min(warmup, a)
    head = recs.new_empty((k * H,) + tuple(recs.shape[1:]))
    if rank > 0:
        transport.recv(head, rank - 1)
    if rank < world - 1:
        k_next = min(warmup, b)
        transport.send(torch.cat([head, recs])[(k + b - a - k_next) * H:], rank + 1)
    if rank > 0:
        transport.send(recs[:H], rank - 1)
    last = rank == world - 1
    run_recs = recs
    if not last:
        ahead = recs.new_empty((H,) + tuple(recs.shape[1:]))
        transport.recv(ahead, rank + 1)
        run_recs = torch.cat([recs, ahead])
    # (2) warm-up
    if rank > 0:
        stitcher.doFrameReassembleAuto(torch.cat([head, recs[:H]]), k + 1, H, file_start=True, file_end=False, **stitch_kw)
        start = stitcher.saveState()
    t_warm = time.perf_counter() - t0

    # (3) the shard
    def run():
        out = stitcher.doFrameReassembleAuto(run_recs, run_recs.shape[0] // H, H, file_start=(rank == 0), file_end=last, **stitch_kw)
        return out, (None if last else stitcher.saveState())
    out, end = run()
    if world == 1:
        return out, {"warmup_frames": 0, "warmup_s": t_warm, "total_s": time.perf_counter() - t0, "rounds": [], "redone": 0}
    # (4) verify / redo (nobody compares with rank 0's start or the last rank's end: placeholders of the blob's shape)
    if rank == 0:
        start = end
    if last:
        end = start

    def redo(state):
        nonlocal out
        stitcher.loadState(state)
        out, end = run()
        return state if last else end
    rounds, redone = settle_states(transport, start, end, redo, "stitcher state")
    return out, {"warmup_frames": k, "warmup_s": t_warm, "total_s": time.perf_counter() - t0, "rounds": rounds, "redone": redone}


def settle_states(transport, start: torch.Tensor, end: torch.Tensor, redo, what: str = "state"):
    """The verify / redo rounds of a shard hand-off.  [start]: the state this rank's run started from, [end]: the state it ended
    with (canonical blobs: equality is byte equality; placeholders of the same shape where nobody compares them).  Every round
    all-gathers the (start, end) pairs; every rank g > 0 whose start differs from rank g-1's end calls redo(that end) -> its new
    end state.  Rank 0 is exact, so after round r the first r+1 shards are final: at most [world] rounds.
    Returns (rounds: the ranks redone in each round, the same list on every rank; redone: the redo calls of this rank)."""
    rank, world = transport.rank, transport.world
    rounds, redone = [], 0
    if world == 1:
        return rounds, redone
    for _ in range(world + 1):
        both = transport.all_gather(torch.stack([start, end]))
        bad = [g for g in range(1, world) if not torch.equal(both[g, 0], both[g - 1, 1])]
        if not bad:
            return rounds, redone
        rounds.append(bad)
        if rank in bad:
            start = both[rank - 1, 1].clone()
            end = redo(start)
            redone += 1
    raise RuntimeError(f"{what} hand-off did not settle")


# ---- line decode (VideoToDigital.doBinarize) over frame shards, exact
#
# The plain sharded decode starts every shard with an empty chain, as the reference does at a file start; on a damaged tape the
# records at a shard's head can then differ from one call over the whole tape (Tier-B fields, the words of lines that fail their
# CRC, with ignore_crc the samples).  decode_shard makes the shards exact with the protocol of stitch_shard: rank g decodes the
# [warmup] frames in front of its first frame as a new file (records thrown away), continues over its own frames from the chain
# state that leaves, and the (start, end) chain states (VideoToDigital.saveState, canonical) are verified by settle_states.
#
# The chain forgets: its presets follow the last good line, the damper the last 9 lines, the frame average the last 16 frames.
# DECODE_WARMUP_FRAMES is that 16-frame reach plus a margin -- a guess until measured on damaged tapes.

DECODE_WARMUP_FRAMES = 20


def decode_shard(v2d, luma: torch.Tensor, transport, warmup: int = DECODE_WARMUP_FRAMES, edges=None, want_aux: bool = False):
    """Line decode of this rank's frames [a, b) = frame_range(n_frames, rank, world) so that the shards' records (and aux)
    concatenate to one doBinarize call over the whole tape, in every format.

    v2d: a VideoToDigital on this rank's handle (PCM type, mode, duplicate check and fine settings as for the whole tape; one
    chain segment); luma: CUDA uint8 [b-a, H, W], this rank's frames; transport: DistTransport or LocalTransport rank; edges:
    world+1 frame indices [0, a_1, .., n_frames] for shards other than frame_range's (n_frames is then edges[-1]; without edges
    it is the sum of the shards' frame counts, gathered).
    Steps: (1) receive the luma of the [warmup] frames before a from rank-1 (passed along when shards are shorter); (2) decode
    them as a new file, records discarded: the chain state this leaves is the guess at a (exact when the warm-up reaches frame
    0); (3) continue over [a, b), save the end state; (4) settle_states: ranks whose start differs from their predecessor's end
    load that end and decode again.  Rank 0 decodes from a file start.  warmup must be >= 1 on ranks > 0: a file start is no
    state to continue (frame 0 carries the NEW_FILE line).
    The STC-007 halo (the first 112 records of rank g+1) is final only when this returns: exchange it afterwards, not from
    doBinarize's on_first_frame hook.
    Returns (records, stats) or ((records, aux), stats); stats as stitch_shard's (warmup_frames, warmup_s, total_s, rounds,
    redone) plus save_s and verify_s (time spent saving states and in the verify / redo rounds)."""
    import time
    rank, world = transport.rank, transport.world
    n_own = luma.shape[0]
    if edges is None:
        counts = transport.all_gather(torch.tensor([n_own], dtype=torch.int64, device=luma.device)).view(-1).tolist()
        edges = [0]
        for c in counts:
            edges.append(edges[-1] + int(c))
    n_frames = edges[-1]
    if len(edges) != world + 1 or edges[0] != 0 or any(edges[g + 1] <= edges[g] for g in range(world)):
        raise ValueError("every shard needs at least one frame, and the shards must cover the tape")
    a, b = edges[rank], edges[rank + 1]
    if n_own != b - a:
        raise ValueError("luma must hold this rank's frames")
    if rank > 0 and warmup < 1:
        raise ValueError("decode_shard needs warmup >= 1 on ranks > 0: a file start is no chain state to continue")
    if getattr(v2d, "chain_segments", 1) > 1:
        raise ValueError("decode_shard decodes one file: chain_segments must be 1")
    t0 = time.perf_counter()
    # (1) luma of the frames in front
    k = min(warmup, a)
    head = luma.new_empty((k,) + tuple(luma.shape[1:]))
    if rank > 0:
        transport.recv(head, rank - 1)
    if rank < world - 1:
        k_next = min(warmup, b)
        transport.send(torch.cat([head, luma])[k + (b - a) - k_next:], rank + 1)
    # (2) warm-up
    t_save = 0.0
    if rank > 0:
        v2d.doBinarize(head)
        ts = time.perf_counter()
        start = v2d.saveState()
        t_save += time.perf_counter() - ts
    t_warm = time.perf_counter() - t0

    # (3) the shard
    def run():
        nonlocal t_save
        out = v2d.doBinarize(luma, want_aux=want_aux, continue_file=(rank > 0))
        ts = time.perf_counter()
        end = v2d.saveState()
        t_save += time.perf_counter() - ts
        return out, end
    out, end = run()
    if rank == 0:
        start = end

    # (4) verify / redo
    def redo(state):
        nonlocal out
        v2d.loadState(state)
        out, e = run()
        return e
    tv = time.perf_counter()
    rounds, redone = settle_states(transport, start, end, redo, "line-decode chain state")
    t_verify = time.perf_counter() - tv
    return out, {"warmup_frames": k, "warmup_s": t_warm, "total_s": time.perf_counter() - t0, "rounds": rounds, "redone": redone,
                 "save_s": t_save, "verify_s": t_verify}


def bind_to_gpu_numa_node(device_index: int):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so that host buffers allocated afterwards (the
    pinned luma / sample buffers of the host entry points) are local to the GPU's PCIe root: with one process per GPU
    every H2D stream then reads its own socket's memory.  Returns the node, or None when the platform does not say
    (no sysfs entry, a single node, or a VM that hides the topology) -- nothing is changed in that case."""
    import os
    try:
        p = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except (OSError, ValueError, AttributeError, RuntimeError):
        return None
