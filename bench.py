#!/usr/bin/env python
"""bench.py -- decoded video lines/s of the STC-007 decode path (binarize + CRCC + deinterleave/P/Q) on 1..8 B200.

Workload (BASELINE.json config 5 = config 1 at tape length): an STC-007 PAL tape of --frames frames (default 90 000 =
1 hour, 720x576 8-bit luma, 51.84 M lines, 37.3 GB), frame-sharded contiguously over the ranks ("strong" scaling: the
tape is fixed, each rank decodes frames [rank*F/N, (rank+1)*F/N) and receives the 112-line halo of the next shard over
NCCL).  The tape is synthetic: a periodic encoder output (sdvpcmdecoder_b200/synth.py, period --period frames) repeated
end to end, which is one continuous valid tape; it is resident in HBM before the timed region.  A step = one pass of the
whole path over the rank's shard.  Inputs are far larger than L2 (126 MB), so nothing is served from cache between steps.

  python bench.py [--gpus N] [--steps K] [--warmup W]            product arm (one process per GPU under torchrun)
  python bench.py --impl reference ...                           the reference's own CPU path (oracle/_ref) on the host cores
  python bench.py ... --dump-outputs DIR                         also write what the last timed step computed (see dump_outputs)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W = 576, 720
LPF = 294
BYTES_BULK = W + 32          # bulk kernel: luma row read + 32-byte line record written
BYTES_DEINT = 32 + 18        # deinterleave kernel: line record read + 6 int16 samples + 6 flag bytes written
BYTES_PATH = W + 64          # SURVEY.md section 8(d): W + 24 + 24 + 16 rounded to the record sizes used there


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_traffic(frames):
    """dram__bytes_read.sum + dram__bytes_write.sum of one stc007_bulk_kernel launch from the committed ncu --set full
    capture (profiles/r2_bulk_deint_ncu_full.txt, taken at the 90 000-frame workload), in bytes; None for other sizes."""
    if frames != 90000:
        return None
    try:
        got = {}
        for line in open(os.path.join(ROOT, "profiles", "r2_bulk_deint_ncu_full.txt")):
            p = line.split()
            if p and p[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and p[0] not in got:      # first capture in the file = current kernel
                got[p[0]] = float(p[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[p[2]]
        return sum(got.values()) or None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.05] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], None, set()
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(p[0])); mx = float(p[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_segment(period):
    from sdvpcmdecoder_b200 import synth
    return synth.make_stc007(period, seed=1234, periodic=True)


DUMP_BYTES = 60_000_000      # all files of one --dump-outputs run together (headers aside), under 64 MB


def dump_outputs(out_dir, samples, flags, first_block, rank, world):
    """Write what a caller of the decode path receives -- the samples [nb, 6] (int16) and the sample flags [nb, 6] -- as float32
    .npy files, with the global index of every block as float64.  A tape too large for DUMP_BYTES is represented by a fixed
    sample of its blocks (seeded, so two runs with the same arguments write the same blocks).  Under torchrun every rank writes
    its own shard's files, named *.rank<r>.npy."""
    import torch
    nb = samples.shape[0]
    k = min(nb, DUMP_BYTES // world // (6 * 4 * 2 + 8))
    rows = np.arange(nb) if k == nb else np.sort(np.random.default_rng(1234 + rank).choice(nb, k, replace=False))
    idx = torch.from_numpy(rows).to(samples.device)
    suffix = "" if world == 1 else f".rank{rank}"
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"samples{suffix}.npy"), samples[idx].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, f"flags{suffix}.npy"), flags[idx].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, f"block_index{suffix}.npy"), (rows + first_block).astype(np.float64))


# ------------------------------------------------------------------------------------------------ reference arm / CPU baseline
_TAPE_CACHE = {}


def _cpu_tape(frames, period=30):
    if (frames, period) not in _TAPE_CACHE:
        seg = make_segment(period)["luma"]
        reps = (frames + period - 1) // period
        _TAPE_CACHE[(frames, period)] = np.ascontiguousarray(np.concatenate([seg] * reps)[:frames])
    return _TAPE_CACHE[(frames, period)]


def cpu_reference_rate(frames_per_pipe, pipes, period=30):
    """Frame-sharded reference pipelines (VideoToDigital + STC007DataStitcher, 2 worker threads each) on the host cores.
    Returns (lines/s, seconds, threads).  The tape is generated outside the timed part."""
    from oracle import refbind as R
    if not R.available():
        return None
    luma = _cpu_tape(frames_per_pipe, period)
    cfg = R.StitchCfg(video_std=1, field_order=1, resolution=1, p_corr=1, q_corr=1, cwd=0)
    out = [None] * pipes

    def work(i):
        pairs, _, _ = R.pipeline_run(R.TYPE_STC007, R.MODE_NORMAL, luma, cfg, taps=False)
        out[i] = len(pairs)

    ths = [threading.Thread(target=work, args=(i,)) for i in range(pipes)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    assert all(o and o > frames_per_pipe * 1500 for o in out), out
    return pipes * frames_per_pipe * H / dt, dt, 2 * pipes


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 2
    pipes = max(1, ncpu // 2)
    frames = args.ref_frames
    from oracle import refbind as R
    if not R.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libsdvref.so missing (reference tree was not present at build time)"}))
        return
    for _ in range(args.warmup):
        cpu_reference_rate(max(10, frames // 4), pipes)
    _cpu_tape(frames)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        rate, dt, thr = cpu_reference_rate(frames, pipes)
        total += pipes * frames * H
    dt = time.perf_counter() - t0
    value = total / dt
    sample = f"{pipes} concurrent reference pipelines x {frames} PAL frames per step (same synthetic tape), shim msleep 200 us"
    line = {"metric": "decoded video lines/sec (bin+CRC+deint)", "value": value, "unit": "lines/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "STC-007 PAL 720x576 tape, MODE_NORMAL, dup-check on, PAL/TFF/14-bit preset, P+Q on, CWD off (bounded sample)",
                       "frames_per_step": pipes * frames},
            "cpu_baseline": {"value": value, "unit": "lines/s", "cores": ncpu, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "lines/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))



# ------------------------------------------------------------------------------------------------ BASELINE configs 1-4 (N = 1)
def _median_ms(fn, reps, torch):
    """Median device time of fn() over [reps] runs (CUDA events on the current stream, synchronised on both sides)."""
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), [float(t) for t in ts]


def _ref_rate(pcm_type, luma, cfg_kw):
    """Reference pipeline (VideoToDigital + stitcher threads, oracle/_ref) on a bounded sample; (lines/s, seconds) or None."""
    from oracle import refbind as R
    if not R.available():
        return None
    cfg = R.StitchCfg(**cfg_kw)
    t0 = time.perf_counter()
    R.pipeline_run(pcm_type, R.MODE_NORMAL, luma, cfg, taps=False)
    dt = time.perf_counter() - t0
    return luma.shape[0] * luma.shape[1] / dt, dt


def bench_configs(h, dev, peak, frames=1000, reps=20, c4_frames=1000, c4_reps=3, cpu=True):
    """BASELINE.json configs 1-4 on one GPU, device-resident input, whole path to samples: lines/s (median of [reps] device
    timings), fraction of the HBM roofline at SURVEY section 8(d)'s bytes per line, and the reference pipeline on a bounded
    sample of the same tape.  Parity of every one of them is what tests/ -m gpu checks; these are their speeds."""
    import torch
    from sdvpcmdecoder_b200 import capi, operators, synth
    from oracle import refbind as R
    out = []

    def entry(cid, workload, lines, ms, all_ms, bytes_per_line, extra=None, ref=None, ref_sample=None):
        v = lines / (ms * 1e-3)
        e = {"id": cid, "workload": workload, "lines": lines, "lines_per_s": v, "ms": ms, "reps": len(all_ms), "ms_min": min(all_ms), "ms_max": max(all_ms),
             "roofline": {"bound": "hbm", "bytes_per_line": bytes_per_line, "achieved": v * bytes_per_line / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": v * bytes_per_line / 1e9 / peak}}
        if extra:
            e.update(extra)
        if ref is not None:
            e["cpu_baseline"] = {"value": ref[0], "unit": "lines/s", "cores": 2, "kind": "reference", "sample": ref_sample + f", {ref[1]:.1f} s"}
        out.append(e)

    # ---- config 1: STC-007 PAL clean
    t = synth.make_stc007(50, seed=1234, periodic=True)
    luma = torch.from_numpy(np.ascontiguousarray(np.tile(t["luma"], (frames // 50, 1, 1)))).to(dev)
    v2d = operators.VideoToDigital(h)
    st = operators.STC007DataStitcher(h)
    recs = torch.empty((frames * H, 32), dtype=torch.uint8, device=dev)
    nb = st.block_count(frames)
    smp = torch.empty((nb, 6), dtype=torch.int16, device=dev)
    fl = torch.empty((nb, 6), dtype=torch.uint8, device=dev)

    def c1():
        v2d.doBinarize(luma, out=recs)
        st.doFrameReassemble(recs, frames, H, samples=smp, flags=fl)
    c1(); c1()
    ms, all_ms = _median_ms(c1, reps, torch)
    v2d.warm_start = False
    ms_cold, all_cold = _median_ms(c1, reps, torch)
    v2d.warm_start = True

    def c1_auto():
        v2d.doBinarize(luma, out=recs)
        st.doFrameReassembleAuto(recs, frames, H, video_std=1)
    c1_auto()
    ms_auto, _ = _median_ms(c1_auto, max(3, reps // 4), torch)
    st.setCWDCorrection(True)           # the reference's default: on a clean tape no frame holds a line CWD may patch, the scan is the cost
    c1_auto()
    ms_auto_cwd, _ = _median_ms(c1_auto, max(3, reps // 4), torch)
    st.setCWDCorrection(False)
    ref = _ref_rate(R.TYPE_STC007, np.ascontiguousarray(np.tile(t["luma"], (2, 1, 1))),
                    dict(video_std=1, field_order=1, resolution=1, p_corr=1, q_corr=1, cwd=0)) if cpu else None
    entry(1, f"config 1: STC-007 PAL 720x576 clean, {frames} frames, MODE_NORMAL + CRCC + dup-check, PAL/TFF/14-bit preset geometry, P+Q", frames * H, ms, all_ms, BYTES_PATH,
          {"cold_start": {"ms": ms_cold, "lines_per_s": frames * H / (ms_cold * 1e-3), "note": "no warm start (sdv_bin_config.reserved[2] bit 0): first-frame chain not hidden"},
           "own_alignment": {"ms": ms_auto, "lines_per_s": frames * H / (ms_auto * 1e-3), "ms_with_cwd": ms_auto_cwd,
                             "note": "sdv_stc007_stitch_frames: trim + field-stitching decisions + assembly as the reference makes them, instead of preset geometry; "
                                     "ms_with_cwd: the same with Cross-Word Decoding enabled (setCWDCorrection(true))"}},
          ref, "one reference pipeline (2 threads) on 100 frames of the same tape")
    del luma, recs, smp, fl

    # ---- config 2 / 3: PCM-1, PCM-16x0 (SI)
    for cid, fmt in ((2, "pcm1"), (3, "pcm16x0")):
        if fmt == "pcm1":
            t = synth.make_pcm1(50)
            ptype, rtype, stitch, bpl = capi.TYPE_PCM1, R.TYPE_PCM1, operators.PCM1DataStitcher(h), W + 64
            name = "config 2: PCM-1 NTSC 720x480 clean"
        else:
            t = synth.make_pcm16x0(50)
            ptype, rtype, stitch, bpl = capi.TYPE_PCM16X0, R.TYPE_PCM16X0, operators.PCM16X0DataStitcher(h), W + 96
            name = "config 3: PCM-16x0 (SI) NTSC 44.1 kHz 720x480 clean"
        luma = torch.from_numpy(np.ascontiguousarray(np.tile(t["luma"], (frames // 50, 1, 1)))).to(dev)
        vf = operators.VideoToDigital(h)
        vf.setPCMType(ptype)

        def cf():
            r = vf.doBinarize(luma)
            stitch.doFrameReassemble(r, frames, 480)
        cf(); cf()
        ms, all_ms = _median_ms(cf, reps, torch)
        ref = _ref_rate(rtype, np.ascontiguousarray(t["luma"][:30]), dict(field_order=1, auto_line_offset=1, pcm16x0_format=1, p_corr=1)) if cpu else None
        entry(cid, f"{name}, {frames} frames, MODE_NORMAL (4 coordinate prescans per frame) + CRCC + stitcher + deinterleave", frames * 480, ms, all_ms, bpl,
              {"stats": vf.stats()}, ref, "one reference pipeline (2 threads) on 30 frames of the same tape")
        del luma

    # ---- config 4: damaged STC-007 (every frame through the sequential chain + reference-level sweeps)
    base = synth.make_stc007(c4_frames, seed=4)
    dmg = synth.damage_stc007(base["luma"], seed=4567)
    luma = torch.from_numpy(dmg).to(dev)
    v4 = operators.VideoToDigital(h)
    s4 = operators.STC007DataStitcher(h)

    def c4():
        r = v4.doBinarize(luma)
        s4.doFrameReassembleAuto(r, c4_frames, H, video_std=1)
    c4()
    ms, all_ms = _median_ms(c4, c4_reps, torch)
    st4 = v4.stats()
    seg = max(2, min(c4_frames // 2, 4 * 148))
    v4.chain_segments = seg
    c4()
    ms_seg, all_seg = _median_ms(c4, c4_reps, torch)
    v4.chain_segments = 1
    s4.setCWDCorrection(True)
    c4()
    ms_cwd, _ = _median_ms(c4, c4_reps, torch)
    cwd_chains = s4.handle.last_stats()["reserved"]
    s4.setCWDCorrection(False)
    ref = _ref_rate(R.TYPE_STC007, np.ascontiguousarray(dmg[:10]), dict(video_std=1, field_order=1, resolution=1, p_corr=1, q_corr=1, cwd=0)) if cpu else None
    entry(4, f"config 4: STC-007 PAL with gain/offset jitter, noise sigma 12, blur, dropouts, killed markers (synth.damage_stc007 seed 4567), {c4_frames} frames, "
             "one file (chain_segments = 1: the reference's semantics), own alignment, P+Q", c4_frames * H, ms, all_ms, BYTES_PATH,
          {"bound_note": "latency / integer-issue bound (sequential chain + reference-level sweeps), not HBM: profiles/r2_config4_relay.md, profiles/r2_config4_ncu.txt",
           "relay": {"pieces": st4["reserved"] >> 16, "pieces_decoded_again": st4["reserved"] & 0xFFFF,
                     "note": "relay mode: many chains at once, every piece verified to start from the true chain state (exact single-file semantics)"},
           "lines_chain": st4["lines_chain"],
           "with_cwd": {"ms": ms_cwd, "lines_per_s": c4_frames * H / (ms_cwd * 1e-3),
                        "chains": cwd_chains,
                        "note": "the same with Cross-Word Decoding (setCWDCorrection(true), the reference's default): chains of damaged frames walked on the device"},
           "segments": {"chain_segments": seg, "ms": ms_seg, "lines_per_s": c4_frames * H / (ms_seg * 1e-3),
                        "note": "NOT the reference's semantics: the tape decoded as that many independent files"}},
          ref, "one reference pipeline (2 threads) on 10 frames of the same tape")
    return out

# ------------------------------------------------------------------------------------------------ product arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=90000, help="tape length in frames (whole job)")
    ap.add_argument("--period", type=int, default=60, help="period of the synthetic tape in frames")
    ap.add_argument("--e2e-frames", type=int, default=9000, help="frames per rank of the host-buffer (end-to-end) measurement")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--ref-frames", type=int, default=150, help="frames per reference pipeline and step (--impl reference)")
    ap.add_argument("--cpu-frames", type=int, default=400, help="frames of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE config 1-4 entries (N = 1 only)")
    ap.add_argument("--config-frames", type=int, default=1000)
    ap.add_argument("--config-reps", type=int, default=20)
    ap.add_argument("--config4-frames", type=int, default=1000)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--late-halo", action="store_true", help="exchange the halo after the whole shard is decoded")
    ap.add_argument("--no-countdown-exchange", action="store_true",
                    help="skip the hand-off of the broken-block countdown between shards (not exact on tapes with BROKEN blocks at shard boundaries)")
    ap.add_argument("--fuse", action="store_true", help="finish the in-frame data blocks inside the bulk pass (sdv_stc007_fuse_next_decode; slower, see DESIGN 3.3)")
    ap.add_argument("--no-lazy", action="store_true", help="wait for the bulk pass inside every decode call (no lazy verification)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the samples and flags of the last one to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from sdvpcmdecoder_b200 import capi, operators, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU: the product has no CPU path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    numa_node = None if args.no_numa_bind else sharding.bind_to_gpu_numa_node(local)      # before any pinned allocation
    sampler = ClockSampler(local) if rank == 0 else None

    F = args.frames
    a, b = sharding.frame_range(F, rank, world)
    n = b - a
    seg = make_segment(args.period)
    seg_dev = torch.from_numpy(seg["luma"]).to(dev)
    luma = seg_dev[(torch.arange(a, b, device=dev) % args.period)]            # [n, H, W] resident in HBM
    assert luma.is_contiguous() and luma.shape == (n, H, W)

    h = capi.Handle(local)
    v2d = operators.VideoToDigital(h)
    st = operators.STC007DataStitcher(h)
    st.lead_in = sharding.shard_lead_in(rank)
    nb = st.block_count(n)
    recs = torch.empty((n * H, 32), dtype=torch.uint8, device=dev)
    samples = torch.empty((nb, 6), dtype=torch.int16, device=dev)
    flags = torch.empty((nb, 6), dtype=torch.uint8, device=dev)
    halo = torch.zeros((112, 32), dtype=torch.uint8, device=dev) if rank < world - 1 else None
    cd_state = torch.zeros(4, dtype=torch.int32, device=dev)
    handoff = sharding.CountdownHandoff(rank, world, dev)
    lazy = not args.no_lazy
    last_halo = [None]
    lazy_redone = [0]

    def finish_previous():
        """The previous step's lazy decode: if a frame was not clean after all (never on this tape) the library has decoded the tape
        again; what was computed from the records is computed again."""
        if lazy and v2d.verify():
            lazy_redone[0] += 1
            handoff.settle()
            st.doFrameReassemble(recs, n, H, samples=samples, flags=flags, halo=last_halo[0])

    def step():
        # The previous step's countdown hand-off is settled AFTER this step's decode is under way (the decode call waits for its
        # first frame anyway; by then the gathered countdowns have long arrived), so the device never idles on it.  A redo it asked
        # for would run on this step's records: the same tape here; a pipeline with other data per batch keeps a batch's records
        # until its hand-off is settled.
        # Lazy verification (sdv_bin_config.reserved[2] bit 1): the decode call returns once the first frame has confirmed the
        # warm-start presets; that the bulk pass took every frame is looked at when the NEXT step starts -- the deinterleave pass
        # and the hand-off are enqueued behind the bulk pass meanwhile, and the host is never behind the device.
        finish_previous()
        if args.fuse:
            # the bulk pass also finishes the data blocks that lie inside a frame (sdv_stc007_fuse_next_decode); the deinterleave
            # call below then only does the blocks that reach into the next frame.  Measured slower (DESIGN 3.3): off by default.
            st.fuseWithNextDecode(samples, flags)
        if world == 1 or args.late_halo:
            v2d.doBinarize(luma, out=recs, lazy=lazy)
            handoff.settle()
            h_in = sharding.exchange_halo(recs, halo, rank, world)
        else:
            # the halo (first 112 line records) leaves as soon as the first frame is final, beside the bulk pass
            reqs = []
            v2d.doBinarize(luma, out=recs, lazy=lazy, on_first_frame=lambda: reqs.extend(sharding.exchange_halo_start(recs, halo, rank, world)))
            handoff.settle()
            h_in = sharding.exchange_halo_finish(reqs, halo, rank, world)
        last_halo[0] = h_in
        st.doFrameReassemble(recs, n, H, samples=samples, flags=flags, halo=h_in)
        if world > 1 and not args.no_countdown_exchange:
            # the stitcher's broken-block countdown crosses shard boundaries: gather every shard's countdown_out (posted here,
            # looked at when the host next waits for the device anyway), redo the windows of a shard whose predecessor leaves one
            # open (never on this clean tape; the exchange itself is the cost)
            st.countdown_to(cd_state)

            def redo(c_in):
                st.doFrameReassemble(recs, n, H, samples=samples, flags=flags, halo=h_in, countdown_in=c_in)
                st.countdown_to(cd_state)
            handoff.post(cd_state, redo)

    def barrier():
        finish_previous()
        handoff.settle()            # (inside the timed region: a step is not done before its hand-off is)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    h.timings(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step()
    finish_previous()
    handoff.settle()
    e1.record()
    barrier()
    t_wall1 = time.perf_counter()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    tm = h.timings(reset=True)
    launches_timed = int(tm["kernel_launches"])
    stats = v2d.stats()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, samples, flags, sharding.first_block(F, rank, world, LPF), rank, world)

    # ---- the same K steps without the warm start (a one-shot decode of a tape is a cold call on every GPU)
    v2d.warm_start = False
    step()
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(args.steps):
        step()
    finish_previous()
    handoff.settle()
    c1.record()
    barrier()
    cms = torch.tensor([c0.elapsed_time(c1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(cms, op=dist.ReduceOp.MAX)
    cold_ms = float(cms.item()) / args.steps
    v2d.warm_start = True
    h.timings(reset=True)

    # ---- the work was real: every block flagged valid equals the source audio, and the tape interior is all valid
    check = None
    if not args.no_check:
        audio = torch.from_numpy(seg["audio"].astype(np.int32)).to(dev)           # periodic source blocks
        nper = audio.shape[0]
        g0 = sharding.first_block(F, rank, world, LPF)                             # global index of local block 0
        src = torch.arange(nb, device=dev, dtype=torch.int64) + (g0 - (operators.LEAD_IN_LINES - seg["j0"]))
        exp = (audio[src % nper] << 2).to(torch.int16)
        ok = (flags & 1).bool().all(dim=1)
        good = ((samples == exp).all(dim=1) | ~ok)[src >= 0]
        interior = torch.ones(nb, dtype=torch.bool, device=dev)
        if rank == 0:
            interior[:400] = False
        if rank == world - 1:
            interior[-400:] = False
        res = torch.tensor([int((~good).sum()), int((~ok & interior).sum()), int(ok.sum())], device=dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(res)
        check = {"blocks_wrong": int(res[0]), "interior_blocks_invalid": int(res[1]), "blocks_valid": int(res[2])}
        del audio, src, exp, ok, good, interior

    # ---- end to end through the host-buffer entry point (H2D + decode + D2H inside the timed region)
    ne = min(args.e2e_frames, n)
    e2e = None
    if ne > 0 and args.e2e_steps > 0:
        host = torch.empty((ne, H, W), dtype=torch.uint8, pin_memory=True)
        hn = host.numpy()
        for i in range(0, ne, args.period):
            m = min(args.period, ne - i)
            hn[i:i + m] = seg["luma"][:m]
        nbe = operators.LEAD_IN_LINES + ne * 2 * LPF
        s_host = torch.empty((nbe, 6), dtype=torch.int16, pin_memory=True)
        f_host = torch.empty((nbe, 6), dtype=torch.uint8, pin_memory=True)
        operators.decode_tape_host(h, hn, samples_out=s_host.numpy(), flags_out=f_host.numpy())       # warm-up (allocations)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            operators.decode_tape_host(h, hn, samples_out=s_host.numpy(), flags_out=f_host.numpy())
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * ne * H * args.e2e_steps / float(dt.item()), "unit": "lines/s",
               "h2d_bytes_per_step": world * ne * H * W, "d2h_bytes_per_step": world * nbe * 18,
               "frames_per_rank": ne, "steps": args.e2e_steps, "numa_node_rank0": numa_node,
               "scaling": "weak (every rank decodes its own e2e-frames tape from pinned host memory; value = sum over ranks)",
               "bound": "PCIe H2D of the luma (720 B per line against 18 B of samples back); ranks share the host's memory controllers",
               "valid_blocks": int((f_host.numpy()[:, 0] & 1).sum())}

    if rank == 0:
        peak, peak_src = _peaks()
        lines_total = F * H
        value = lines_total * args.steps / (ms_total * 1e-3)
        bulk_gbs = tm["bulk_lines"] * BYTES_BULK / (tm["bulk_ms"] * 1e-3) / 1e9 if tm["bulk_ms"] > 0 else 0.0
        deint_gbs = tm["deint_blocks"] * BYTES_DEINT / (tm["deint_ms"] * 1e-3) / 1e9 if tm["deint_ms"] > 0 else 0.0
        path_gbs = (n * H * args.steps) * BYTES_PATH / (ms_total * 1e-3) / 1e9          # rank 0's shard over its step time
        line = {
            "metric": "decoded video lines/sec (bin+CRC+deint)", "value": value, "unit": "lines/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "STC-007 PAL 720x576 8-bit luma tape, MODE_NORMAL binarization + CRCC + dup-check, PAL/TFF/14-bit assembly, P+Q correction, CWD off",
                       "frames": F, "lines": lines_total, "frames_per_gpu": n, "period_frames": args.period,
                       "sharding": f"contiguous frame ranges over {world} GPU(s), 112-line halo from the next shard (NCCL send/recv)"
                                   + ("" if (world == 1 or args.no_countdown_exchange) else ", broken-block countdown handed to the next shard (one 16-byte all_gather per step, its copy to the host read when the next step starts)"),
                       "l2": "inputs (37.3 GB tape) exceed L2; no flush needed"},
            "roofline": {"bound": "hbm", "kernel": "stc007_bulk_kernel", "achieved": bulk_gbs, "peak": peak, "unit": "GB/s",
                         "frac": bulk_gbs / peak, "traffic": _ncu_traffic(F),
                         "traffic_source": "profiles/r2_bulk_deint_ncu_full.txt (ncu --set full capture of this kernel at this workload, not re-measured in this run)",
                         "peak_source": peak_src,
                         "peak_note": "peak is a copy figure (half reads, half writes); this kernel is 96 % reads and can pass it: "
                                      "ncu puts it at 85 % of the DRAM pin rate (profiles/r2_bulk_deint_ncu_full.txt)",
                         "bytes_per_line": BYTES_BULK, "avg_launch_ms": tm["bulk_ms"] / max(tm["bulk_launches"], 1),
                         "launches": tm["bulk_launches"],
                         "deint_kernel": {"achieved": deint_gbs, "frac": deint_gbs / peak, "bytes_per_block": BYTES_DEINT,
                                          "avg_launch_ms": tm["deint_ms"] / max(tm["deint_launches"], 1)},
                         "path": {"achieved": path_gbs, "frac": path_gbs / peak, "bytes_per_line": BYTES_PATH}},
            "cold": {"ms_per_step": cold_ms, "value": lines_total / (cold_ms * 1e-3), "unit": "lines/s",
                     "note": "warm start off (sdv_bin_config.reserved[2] bit 0): the first-frame chain runs ahead of the bulk pass instead of beside it"},
            "e2e": e2e, "gpu_launches": launches_timed, "clocks": clocks,
            "stats": {"lines_bulk": stats["lines_fast"], "lines_chain": stats["lines_chain"], "kernel_launches_per_decode": stats["kernel_launches"],
                      "lazy_verification": lazy, "lazy_redone": lazy_redone[0], "fused_deinterleave": bool(args.fuse)},
            "check": check,
        }
        if world == 1 and not args.no_configs:
            del luma, recs, samples, flags
            torch.cuda.empty_cache()
            line["configs"] = bench_configs(h, dev, peak, frames=args.config_frames, reps=args.config_reps, c4_frames=args.config4_frames,
                                            cpu=not args.no_cpu_baseline)
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_rate(args.cpu_frames, 1)
            if r is not None:
                line["cpu_baseline"] = {"value": r[0], "unit": "lines/s", "cores": 2, "kind": "reference",
                                        "sample": f"one reference pipeline (VideoToDigital thread + STC007DataStitcher thread) on {args.cpu_frames} frames of the same tape, {r[1]:.1f} s, shim msleep 200 us"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
