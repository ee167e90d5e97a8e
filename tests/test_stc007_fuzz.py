"""Random STC-007 / M2 tapes through the host build of the device code (tests/hostemu: the host loop of sdv_bin_decode_frames
with scalar stand-ins for the bulk kernel) against the C oracle: widths from 160 to 2048 px, crops down to 2 rows, levels,
PAL / NTSC, Control Block, 16-bit F1, modes 0-3, the duplicate check on and off.  This pins the logic the kernels share with
the host build at these shapes on machines without a GPU; tests/test_gpu_stc007_fuzz.py runs the same builders through the
kernels, so a mismatch there that this module does not show points at what only the GPU runs.

The case builders are plain functions of a seed, shared with tests/test_gpu_stc007_fuzz.py and tools/gpu_fuzz_stc007.py."""
import numpy as np

from oracle import oraclebind as O
from sdvpcmdecoder_b200 import synth
from tests import util

FIELDS = ["words", "flags"] + util.REC_FIELDS[1:] + ["mark_stages"] + ["aux." + n for n in util.AUX_FIELDS]
# 160 px: too few pixels per bit cell, no line decodes; 200 / 280 px: most lines still decode
LINE_WIDTHS = (160, 200, 280, 352, 500, 640, 720, 722, 728, 1000, 1024, 1448, 1920, 2048)
# crops: the bulk kernel steps through a frame 32 rows at a time (BULK_ROWS), so 330, 170, 62, 24 and 2 end on a short step;
# 330, 170, 62 and 2 also have an odd number of rows per field
CROPS = (320, 330, 170, 96, 62, 24, 2)


def oracle_arrays(o):
    """The oracle's line records as the arrays util.line_arrays gives of the product's (records, aux)."""
    return util.line_arrays(util.lines_from_oracle(o), o)


def record_row(k, H):
    """Record k of a frame -> its row: a frame's records are its odd-field rows (0, 2, ...) then its even-field rows."""
    hf = H // 2
    return 2 * (k % hf) + k // hf


def lines_diff(H, got, want):
    """'' when two lists of line arrays (util.line_arrays / oracle_arrays) are equal; else every field that differs, with the
    number of records and the first differing (frame, row) and both values."""
    out = []
    for name, u, v in zip(FIELDS, got, want):
        if len(u) != len(v):
            return f"{len(u)} records, reference {len(v)}"
        d = u != v
        if d.ndim > 1:
            d = d.reshape(len(u), -1).any(axis=1)
        if d.any():
            i = np.nonzero(d)[0][:4]
            at = [(int(k) // H, record_row(int(k) % H, H)) for k in i]
            out.append(f"{name}: {int(d.sum())} records, first (frame, row) {at} got {u[i].tolist()} reference {v[i].tolist()}")
    return "; ".join(out)


def valid_fraction(flags):
    return float((flags & 1).mean()) if len(flags) else 0.0


def sweep_coverage(fracs):
    """(cases with at least 90 % valid lines, cases that mix valid and invalid lines)."""
    f = np.asarray(fracs)
    return int((f >= 0.9).sum()), int(((f > 0.02) & (f < 0.98)).sum())


def _crop(rng, luma):
    """In about 35 % of cases a crop of CROPS rows at an even top row."""
    H = luma.shape[1]
    if rng.rand() < 0.35:
        H = min(int(rng.choice(CROPS)), H)
        top = 2 * int(rng.randint(0, (luma.shape[1] - H) // 2 + 1))
        luma = luma[:, top:top + H]
    return np.ascontiguousarray(luma), H


def _damage(rng, luma, seed, black, white):
    return synth.damage_stc007(luma, seed=seed + 1, sigma=float(rng.choice([0., 4., 10., 20.])), jitter=bool(rng.rand() < 0.4),
                               blur=bool(rng.rand() < 0.4), dropout_frac=float(rng.choice([0., 0.02, 0.1])),
                               marker_kill_frac=float(rng.choice([0., 0.02])), src_black=black, src_white=white)


def line_case(seed):
    """A random STC-007 tape: width, data coordinates scaled with it, levels, PAL / NTSC, Control Block, 16-bit F1, mode 0-3,
    duplicate check, 1-4 frames, damage in 80 % of cases, crops in about 35 %."""
    rng = np.random.RandomState(seed)
    W = int(rng.choice(LINE_WIDTHS))
    m = W / 720.0
    x0 = int(round(rng.randint(2, 40) * m))
    x1 = int(W - round(rng.randint(2, 40) * m))
    black, white = int(rng.randint(5, 60)), int(rng.randint(120, 250))
    n = int(rng.randint(1, 5))
    pal, cb, f16 = bool(rng.rand() < 0.6), bool(rng.rand() < 0.2), bool(rng.rand() < 0.2)
    mode, dup = int(rng.randint(0, 4)), bool(rng.rand() < 0.7)
    luma = synth.make_stc007(n, seed=seed, pal=pal, width=W, x0=x0, x1=x1, black=black, white=white, control_block=cb, f1_16bit=f16)["luma"]
    damage = bool(rng.rand() < 0.8)
    if damage:
        luma = _damage(rng, luma, seed, black, white)
    luma, H = _crop(rng, luma)
    desc = (f"seed {seed} {n}x{H}x{W} {'PAL' if pal else 'NTSC'} mode {mode} dup {dup} x {x0} {x1} bw {black} {white} "
            f"control_block {cb} f1_16bit {f16} damage {damage}")
    return dict(seed=seed, luma=luma, mode=mode, dup=dup, m2=False, desc=desc)


def m2_case(seed):
    """A random M2 tape (STC-007 lines, quiet passages that trip the almost-silent rule of the duplicate check): width, levels,
    PAL / NTSC, mode, 1-3 frames, damage in half the cases, crops in about 35 %."""
    rng = np.random.RandomState(90000 + seed)
    W = int(rng.choice((720, 722, 1000, 1448, 1920)))
    m = W / 720.0
    x0, x1 = int(round(rng.randint(2, 30) * m)), int(W - round(rng.randint(2, 30) * m))
    black, white = int(rng.randint(5, 50)), int(rng.randint(140, 240))
    n, pal = int(rng.randint(1, 4)), bool(rng.rand() < 0.6)
    quiet = float(rng.choice([0.1, 0.3, 0.6]))
    mode, dup = int(rng.randint(0, 4)), bool(rng.rand() < 0.8)
    luma = synth.make_stc007(n, seed=seed, pal=pal, width=W, x0=x0, x1=x1, black=black, white=white, quiet_frac=quiet)["luma"]
    damage = bool(rng.rand() < 0.5)
    if damage:
        luma = _damage(rng, luma, seed, black, white)
    luma, H = _crop(rng, luma)
    desc = f"seed {seed} M2 {n}x{H}x{W} {'PAL' if pal else 'NTSC'} quiet {quiet} mode {mode} dup {dup} x {x0} {x1} bw {black} {white} damage {damage}"
    return dict(seed=seed, luma=luma, mode=mode, dup=dup, m2=True, desc=desc)


def reference_lines(case):
    """The reference of a case as line arrays: the C oracle; for M2, which the oracle has no mode for, the host build."""
    if case["m2"]:
        rec, aux, _ = util.emu_v2d(case["luma"], case["mode"], case["dup"], hybrid=True, m2=True)
        return util.line_arrays(rec, aux)
    return oracle_arrays(O.v2d_stc007(case["mode"], case["luma"], case["dup"]))


def coverage_line_sweep(cases, fracs):
    """(mostly valid, mixed, crops with H % 32 != 0 and more than one frame, widths that are not a multiple of 16)."""
    mostly, mixed = sweep_coverage(fracs)
    short = sum(1 for c in cases if c["luma"].shape[1] % 32 and c["luma"].shape[0] > 1)
    compact = sum(1 for c in cases if c["luma"].shape[2] % 16)
    return mostly, mixed, short, compact


LINE_SEEDS = range(40)


def test_random_line_decode_host_build_equals_oracle():
    bad, fracs, cases = [], [], []
    for seed in LINE_SEEDS:
        case = line_case(seed)
        want = reference_lines(case)
        rec, aux, _ = util.emu_v2d(case["luma"], case["mode"], case["dup"], hybrid=True)
        d = lines_diff(case["luma"].shape[1], util.line_arrays(rec, aux), want)
        if d:
            bad.append(f"{case['desc']}: {d}")
        fracs.append(valid_fraction(want[1]))
        cases.append(case)
    assert not bad, "\n".join(bad)
    cov = coverage_line_sweep(cases, fracs)
    assert cov[0] >= 6 and cov[1] >= 6 and cov[2] >= 3 and cov[3] >= 6, (cov, np.round(fracs, 2).tolist())


def test_m2_host_build_equals_its_chain():
    """M2: the host loop of sdv_bin_decode_frames (bulk stand-in + chain) against every line through the chain alone."""
    bad = []
    for seed in range(4):
        case = m2_case(seed)
        luma = case["luma"]
        rec, aux, _ = util.emu_v2d(luma, case["mode"], case["dup"], hybrid=True, m2=True)
        crec, caux, _ = util.emu_v2d(luma, case["mode"], case["dup"], hybrid=False, m2=True)
        d = lines_diff(luma.shape[1], util.line_arrays(rec, aux), util.line_arrays(crec, caux))
        if d:
            bad.append(f"{case['desc']}: {d}")
    assert not bad, "\n".join(bad)
