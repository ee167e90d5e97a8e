"""GPU fuzz of the STC-007 kernels over seed ranges, with the case builders of tests/test_gpu_stc007_fuzz.py: random line decode
(STC-007 against the C oracle, M2 against the host build), long tapes past one bulk wave, relay / batches / segments on damaged
tapes, the frame assembly fed the GPU's records, the preset-geometry path fused and separate.  Needs a GPU; not part of the suite.
The oracle runs on the CPU, so the seeds are spread over --jobs processes, each with its own decoder handles.
    PYTHONPATH=. python tools/gpu_fuzz_stc007.py [--lines A B] [--m2 A B] [--long A B] [--relay A B] [--stitch A B]
                                                 [--preset A B] [--jobs N]"""
import argparse
import multiprocessing as mp
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

LONG_WIDTHS = (720, 1000, 1920, 2048)


def run(task):
    """(kind, seed) -> (kind, seed, mismatches, what the case covered); an exception is a mismatch."""
    import traceback
    try:
        return case(*task)
    except Exception:
        return task[0], task[1], [f"{task[0]} seed {task[1]} raised: {traceback.format_exc()}"], {}


def case(kind, seed):
    import torch
    from tests import test_gpu_stc007_fuzz as T
    if kind == "lines":
        c = T.line_case(seed)
        bad, frac = T.check_line_case(c)
        n, H, W = c["luma"].shape
        return kind, seed, bad, dict(frac=frac, short=bool(H % 32 and n > 1), compact=bool(W % 16))
    if kind == "m2":
        return kind, seed, T.check_line_case(T.m2_case(seed))[0], {}
    if kind == "long":
        W = LONG_WIDTHS[seed % len(LONG_WIDTHS)]
        wave = T.bulk_wave(W, torch.cuda.get_device_properties(0).multi_processor_count)
        return kind, seed, T.check_long_case(T.long_case(seed, W, wave)), {}
    if kind == "relay":
        return kind, seed, T.check_relay_case(T.relay_case(seed)), {}
    if kind == "stitch":
        bad, used = T.stitch_case(seed)
        return kind, seed, bad, dict(used=used)
    return kind, seed, T.check_preset_case(T.preset_case(seed)), {}


def main():
    ap = argparse.ArgumentParser()
    for k in ("lines", "m2", "long", "relay", "stitch", "preset"):
        ap.add_argument("--" + k, nargs=2, type=int, default=(0, 0), metavar=("FIRST", "END"))
    ap.add_argument("--jobs", type=int, default=1)
    a = ap.parse_args()
    tasks = [(k, s) for k in ("relay", "long", "stitch", "preset", "m2", "lines") for s in range(*getattr(a, k))]
    runs = {k: 0 for k in ("lines", "m2", "long", "relay", "stitch", "preset")}
    bad, fracs, short, compact, used = [], [], 0, 0, []
    t0 = time.time()
    with mp.get_context("spawn").Pool(max(1, a.jobs)) as pool:
        for i, (kind, seed, msgs, cov) in enumerate(pool.imap_unordered(run, tasks)):
            runs[kind] += 1
            bad += msgs
            if kind == "lines" and cov:
                fracs.append(cov["frac"])
                short += cov["short"]
                compact += cov["compact"]
            used += cov.get("used", [])
            if msgs or (i + 1) % 10 == 0:
                print(f"{i + 1}/{len(tasks)} {kind} {seed}: mismatches so far {len(bad)}  {time.time() - t0:.0f}s", flush=True)
    from tests.test_gpu_stc007_fuzz import stitch_coverage
    from tests.test_stc007_fuzz import sweep_coverage
    for m in bad:
        print("MISMATCH", m)
    print("cases", runs, f"{time.time() - t0:.0f}s")
    print("line sweep: (mostly valid, mixed)", sweep_coverage(fracs), "multi-frame crops ending on a short bulk step", short,
          "compact-slot widths", compact)
    print("stitcher settings (detect in / preset in):", stitch_coverage(used))
    print("ALL OK" if not bad else f"{len(bad)} MISMATCHES")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
