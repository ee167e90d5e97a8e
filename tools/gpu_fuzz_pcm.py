"""GPU fuzz of the PCM-1 / PCM-16x0 kernels against the host build of the device code, over a seed range, with the case builders
of tests/test_gpu_pcm_fuzz.py: random line decode (both formats), MODE_INSANE slices, bulk/chain hand-off on longer tapes, the
three frame assemblies fed the GPU's records.  Needs a GPU; not part of the suite.
    PYTHONPATH=. python tools/gpu_fuzz_pcm.py <first seed> <last seed + 1>"""
import sys
import time

from sdvpcmdecoder_b200 import capi
from tests import test_gpu_pcm_fuzz as T


def main():
    import torch
    from sdvpcmdecoder_b200 import operators
    a, b = int(sys.argv[1]), int(sys.argv[2])
    ctx = (capi.Handle(0), operators, torch)
    runs = {"lines": 0, "insane": 0, "handoff": 0, "pcm1_stitch": 0, "x0_preset": 0, "x0_auto": 0}
    bad = []
    fracs = []
    t0 = time.time()
    for seed in range(a, b):
        for fmt in (T.P1, T.X0):
            msg, frac, _ = T.check_line_case(ctx, T.line_case(fmt, seed))
            fracs.append(frac)
            runs["lines"] += 1
            bad += [msg] if msg else []
            if seed % 10 == 0:
                msg = T.check_line_case(ctx, T.insane_case(fmt, seed))[0]
                runs["insane"] += 1
                bad += [msg] if msg else []
            if seed % 25 == 0:
                W = [720, 1000, 1920][(seed // 25) % 3]
                n = 200 if W == 1920 else 40
                case = T.handoff_case(fmt, seed, W, n)
                msg, _, st = T.check_line_case(ctx, case)
                runs["handoff"] += 1
                bad += [msg] if msg else []
                if not 0 < st["frames_skipped"] < n:
                    bad.append(f"{case['desc']}: frames_skipped {st['frames_skipped']}")
        for key, fn in (("pcm1_stitch", T.p1_stitch_case), ("x0_preset", T.x0_preset_case), ("x0_auto", T.x0_auto_case)):
            bad += fn(ctx, seed)
            runs[key] += 1
        print(seed, "mismatches so far", len(bad), "%.0fs" % (time.time() - t0), flush=True)
    for m in bad:
        print("MISMATCH", m)
    print("cases", runs, "line sweep (mostly valid, mixed)", T.sweep_coverage(fracs))
    print("ALL OK" if not bad else f"{len(bad)} MISMATCHES")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
