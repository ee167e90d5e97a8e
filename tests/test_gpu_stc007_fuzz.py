"""Randomised differential tests of the STC-007 kernels against the C oracle (and, for M2 and the frame assembly, which the oracle
has no mode for, against the host build of the same device code).  tests/test_stc007_fuzz.py runs the line-decode builders
through the host build on the CPU, so a difference here points at what only the GPU runs: the persistent bulk kernel (its grid
loop, compact slots, the short last 32-row step of a frame), the bulk/chain hand-off after the first wave, the warm start,
relay mode and its verification, continuation across calls, segment mode, the fused deinterleave and the stitch kernels.

The case builders are plain functions of a seed, so that tools/gpu_fuzz_stc007.py can run them over long seed ranges."""
import numpy as np
import pytest

from oracle import oraclebind as O
from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX, BLOCK_REC
from tests import util
from tests.test_gpu_pcm_fuzz import decode_pitched
from tests.test_pcm16x0_stitch import edge_damage
from tests.test_stc007_fuzz import (line_case, m2_case, reference_lines, lines_diff, oracle_arrays, valid_fraction,
                                    coverage_line_sweep)
from tests.test_stc007_stitch import shift_rows

pytestmark = pytest.mark.gpu

STC = "stc007"


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators
    assert torch.cuda.is_available()
    return capi.Handle(0), operators, torch


# ------------------------------------------------------------------------------------------------ decode and compare
def decode(h, luma, mode=2, dup=True, m2=False, continue_file=False, **attrs):
    """VideoToDigital on the GPU (luma: host array or CUDA tensor) -> (records, aux, stats, device records).  attrs: VideoToDigital
    attributes (warm_start, relay, chain_segments)."""
    import torch
    from sdvpcmdecoder_b200 import operators as ops
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(capi.TYPE_M2 if m2 else capi.TYPE_STC007)
    v2d.setBinarizationMode(mode)
    v2d.setCheckLineDup(dup)
    for k, v in attrs.items():
        setattr(v2d, k, v)
    dev = luma if isinstance(luma, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(luma)).cuda()
    recs, aux = v2d.doBinarize(dev, want_aux=True, continue_file=continue_file)
    torch.cuda.synchronize()
    return ops.records_to_numpy(recs, LINE_REC), ops.records_to_numpy(aux, LINE_AUX), v2d.stats(), recs


def arrays(rec, aux):
    """Every field of the records and every field of aux but its padding (the product's output), in util.line_arrays order."""
    return util.line_arrays(rec, aux) + [rec["reserved"]]


def same_records(a, b):
    return all(np.array_equal(u, v) for u, v in zip(arrays(*a), arrays(*b)))


# ------------------------------------------------------------------------------------------------ A1 / A2: random line decode
def check_line_case(case):
    """Cold and then warm decode on a fresh handle against the reference; every 4th seed also through a pitched, unaligned
    buffer (stride W+3, offset 1), byte-identical to the contiguous call.  -> (mismatches, valid fraction of the reference)."""
    import torch
    luma = case["luma"]
    n, H, W = luma.shape
    want = reference_lines(case)
    bad = []
    h = capi.Handle(0)
    try:
        dev = torch.from_numpy(luma).cuda()
        for call in ("cold", "warm"):
            rec, aux, st, _ = decode(h, dev, case["mode"], case["dup"], case["m2"])
            d = lines_diff(H, util.line_arrays(rec, aux), want)
            if d:
                bad.append(f"{case['desc']} {call}: {d}")
        if case["seed"] % 4 == 0 and not case["m2"]:
            base = decode_pitched(h, STC, luma, W, 0, case["mode"], case["dup"])
            rec, aux, _ = decode_pitched(h, STC, luma, W + 3, 1, case["mode"], case["dup"], seed=case["seed"])
            if not (np.array_equal(rec.view(np.uint8), base[0].view(np.uint8)) and np.array_equal(aux.view(np.uint8), base[1].view(np.uint8))):
                bad.append(f"{case['desc']} stride {W + 3} offset 1: not byte-identical to the contiguous call")
            d = lines_diff(H, util.line_arrays(rec, aux), want)
            if d:
                bad.append(f"{case['desc']} stride {W + 3} offset 1: {d}")
    finally:
        h.close()
    return bad, valid_fraction(want[1])


LINE_SEEDS = range(60)


def test_random_line_decode_equals_oracle(ctx):
    bad, fracs, cases = [], [], []
    for seed in LINE_SEEDS:
        case = line_case(seed)
        msg, frac = check_line_case(case)
        bad += msg
        fracs.append(frac)
        cases.append(case)
    assert not bad, "\n".join(bad)
    # a sweep that decodes nothing proves nothing: enough tapes mostly valid, enough mixed, enough multi-frame crops that end
    # on a short bulk step (decoded cold and warm), enough widths that put the bulk kernel on compact slots
    cov = coverage_line_sweep(cases, fracs)
    assert cov[0] >= 10 and cov[1] >= 10 and cov[2] >= 4 and cov[3] >= 8, (cov, np.round(fracs, 2).tolist())


def test_random_m2_decode_equals_host_build(ctx):
    bad = [m for s in range(8) for m in check_line_case(m2_case(s))[0]]
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ A3: past one bulk wave
BULK_SMEM_HEADER = 128 + 3 * 512        # csrc/stc007_bulk.cuh


def bulk_wave(W, num_sms):
    """Frames one wave of the persistent bulk kernel covers on a contiguous tape of width W: the grid of decode_frames_impl
    (88 % of the SMs) times the warps per block of bulk_plan (2 stages x 32 rows of slot bytes each in 227 KiB, at most 4)."""
    copy = (W + 15) & ~15
    slot = W if W % 16 == 0 else (copy if (copy // 16) & 1 else copy + 16)
    warps = min(4, (227 * 1024 - BULK_SMEM_HEADER) // (2 * 32 * slot))
    grid = num_sms * 88 // 100 if num_sms > 8 else num_sms
    return grid * warps


def long_case(seed, W, wave):
    """A clean tape of 1.2-1.5 bulk waves (6 synthesised frames repeated) with 4-6 frames damaged sparsely, at least one inside
    the first wave and one behind it: a dropout band, a blank first line, one line with another gain, a line with a valid CRC
    but the words of another frame."""
    rng = np.random.RandomState(seed)
    m = W / 720.0
    n_frames = int(wave * rng.uniform(1.2, 1.5))
    src = synth.make_stc007(6, seed=seed, width=W, x0=int(round(14 * m)), x1=W - int(round(14 * m)))["luma"]
    luma = np.ascontiguousarray(np.tile(src, (-(-n_frames // 6), 1, 1))[:n_frames])
    H = luma.shape[1]
    frames = {int(rng.randint(2, wave - 1)), int(rng.randint(wave + 2, n_frames))}
    want = int(rng.randint(4, 7))
    while len(frames) < want:
        frames.add(int(rng.randint(1, n_frames)))
    hits = []
    for f in sorted(frames):
        kind, r = int(rng.randint(4)), int(rng.randint(0, H))
        if kind == 0:
            ln = int(rng.randint(100, 400) * m)
            x = int(rng.randint(0, W - ln))
            luma[f, r:r + int(rng.randint(2, 9)), x:x + ln] = 255 if rng.randint(2) else 0
        elif kind == 1:
            r = int(rng.randint(2))
            luma[f, r] = 16
        elif kind == 2:
            g = float(rng.choice([0.55, 0.75, 1.25]))
            luma[f, r] = np.clip((luma[f, r].astype(np.float32) - 16) * g + 16, 0, 255).astype(np.uint8)
        else:
            luma[f, r] = src[(f % 6 + 1 + int(rng.randint(5))) % 6, int(rng.randint(0, H))]
        hits.append((f, kind, r))
    return dict(luma=luma, desc=f"seed {seed} {n_frames}x{H}x{W} wave {wave} damage (frame, kind, row) {hits}")


def check_long_case(case):
    """Cold, warm and warm_start = False against the oracle, the three records identical, every call served by the bulk kernel
    and the chain.  -> list of mismatches."""
    import torch
    luma = case["luma"]
    n, H, W = luma.shape
    want = oracle_arrays(O.v2d_stc007(2, luma, True))
    dev = torch.from_numpy(luma).cuda()
    bad, runs = [], []
    h = capi.Handle(0)
    try:
        for call, kw in (("cold", {}), ("warm", {}), ("warm_start off", {"warm_start": False})):
            rec, aux, st, _ = decode(h, dev, **kw)
            d = lines_diff(H, util.line_arrays(rec, aux), want)
            if d:
                bad.append(f"{case['desc']} {call}: {d}")
            if not 0 < st["frames_skipped"] < n:
                bad.append(f"{case['desc']} {call}: frames_skipped {st['frames_skipped']} of {n}")
            runs.append((rec, aux))
    finally:
        h.close()
        del dev
    if not all(same_records(runs[0], r) for r in runs[1:]):
        bad.append(f"{case['desc']}: the records of the three calls differ")
    return bad


@pytest.mark.parametrize("width", [720, 1000, 1920, 2048])
def test_long_tapes_past_one_bulk_wave(ctx, width):
    import torch
    wave = bulk_wave(width, torch.cuda.get_device_properties(0).multi_processor_count)
    bad = check_long_case(long_case(8000 + width, width, wave))
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ A4: relay, batches, segments
def relay_case(seed):
    """40-64 frames of BASELINE config-4 damage (the chain never settles: relay mode after the first frames), PAL or NTSC; every
    third seed with a stretch of frames of a second capture with other coordinates spliced in.  Random batch cuts: a 1-frame
    batch, a cut inside the first 2 frames, cuts inside the relay span (every frame of such a tape is damaged, so every cut is
    right behind a damaged frame); and a segment count of 2-7."""
    rng = np.random.RandomState(70000 + seed)
    n, pal = int(rng.randint(40, 65)), bool(seed % 2 == 0)
    luma = synth.damage_stc007(synth.make_stc007(n, seed=7100 + seed, pal=pal)["luma"], seed=7200 + seed)
    splice = None
    if seed % 3 == 1:
        a = int(rng.randint(n // 3, n // 2))
        splice = (a, a + int(rng.randint(4, 13)))
        t2 = synth.make_stc007(n, seed=7300 + seed, pal=pal, x0=22, x1=698)["luma"]
        luma[splice[0]:splice[1]] = synth.damage_stc007(t2, seed=7400 + seed)[splice[0]:splice[1]]
    r1 = int(rng.randint(3, n // 2))
    r2 = int(rng.randint(n // 2, n - 1))
    cuts = sorted({0, 1, 2, r1, r1 + 1, r2, n})
    segments = int(rng.randint(2, 8))
    return dict(luma=np.ascontiguousarray(luma), cuts=cuts, segments=segments,
                desc=f"seed {seed} {n}x{luma.shape[1]}x720 splice {splice} cuts {cuts} segments {segments}")


def check_relay_case(case):
    """One call against the oracle (relay mode ran), relay off, batches with continue_file, segment mode.  -> mismatches."""
    import torch
    luma, cuts, S = case["luma"], case["cuts"], case["segments"]
    n, H, _ = luma.shape
    want = oracle_arrays(O.v2d_stc007(2, luma, True))
    dev = torch.from_numpy(luma).cuda()
    bad = []
    h = capi.Handle(0)
    try:
        one = decode(h, dev)
        d = lines_diff(H, util.line_arrays(*one[:2]), want)
        if d:
            bad.append(f"{case['desc']} one call: {d}")
        if not one[2]["reserved"] >> 16:
            bad.append(f"{case['desc']}: relay mode did not run {one[2]}")
        if not same_records(decode(capi.Handle(0), dev, relay=False)[:2], one[:2]):
            bad.append(f"{case['desc']}: relay off differs from relay on")
        parts = [decode(h, dev[a:b], continue_file=(a > 0))[:2] for a, b in zip(cuts[:-1], cuts[1:])]
        got = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]))
        if not same_records(got, one[:2]):
            bad.append(f"{case['desc']} batches: {lines_diff(H, util.line_arrays(*got), util.line_arrays(*one[:2]))}")
        rec, aux, _, _ = decode(h, dev, chain_segments=S)
        for s in range(S):
            a, b = s * n // S, (s + 1) * n // S
            d = lines_diff(H, util.line_arrays(rec[a * H:b * H], aux[a * H:b * H]), oracle_arrays(O.v2d_stc007(2, luma[a:b], True)))
            if d:
                bad.append(f"{case['desc']} segment {s} frames [{a}, {b}): {d}")
    finally:
        h.close()
    return bad


RELAY_SEEDS = range(3)


def test_continuing_batch_after_a_wrong_warm_guess(ctx):
    """A continuing call on a handle with warm presets whose first frame does not confirm them (here: damaged) once failed with
    "nothing to continue": the start-over without the guess had lost the file.  Found by the batch cuts of the relay tapes."""
    luma = synth.make_stc007(8, seed=7500)["luma"]
    luma[4:6] = synth.damage_stc007(luma[4:6], seed=7501)
    h = capi.Handle(0)
    try:
        one = decode(h, luma)[:2]
        assert not lines_diff(576, util.line_arrays(*one), oracle_arrays(O.v2d_stc007(2, luma, True)))
        parts = [decode(h, luma[a:b], continue_file=(a > 0))[:2] for a, b in ((0, 4), (4, 8))]
    finally:
        h.close()
    assert same_records((np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])), one)


def test_relay_batches_and_segments_on_damaged_tapes(ctx):
    bad = [m for s in RELAY_SEEDS for m in check_relay_case(relay_case(s))]
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ A5: frame assembly
def stitch_tape(seed):
    """3-5 frames, the recipe of tools/parity_fuzz_stitch.py: PAL / NTSC, 16-bit F1, vertical shifts, config-4 / heavy / dropout
    damage, one damaged frame, edge damage, a blank frame."""
    rng = np.random.RandomState(seed)
    pal, f16, frames = bool(rng.rand() < 0.7), bool(rng.rand() < 0.4), int(rng.randint(3, 6))
    luma = synth.make_stc007(frames, seed=seed, pal=pal, f1_16bit=f16)["luma"]
    if rng.rand() < 0.3:
        luma = shift_rows(luma, int(rng.randint(-3, 4)))
    kind = int(rng.randint(0, 6))
    if kind == 0:
        luma = synth.damage_stc007(luma, seed=seed + 1)
    elif kind == 1:
        luma = synth.damage_stc007(luma, seed=seed + 1, sigma=float(rng.uniform(10, 24)), dropout_frac=float(rng.uniform(0.02, 0.15)),
                                   marker_kill_frac=float(rng.uniform(0, 0.06)))
    elif kind == 2:
        luma = synth.damage_stc007(luma, seed=seed + 1, sigma=float(rng.uniform(2, 6)), dropout_frac=float(rng.uniform(0.1, 0.35)), marker_kill_frac=0.0)
    elif kind == 3:
        luma = luma.copy()
        f = int(rng.randint(0, frames))
        luma[f] = synth.damage_stc007(luma[f:f + 1], seed=seed + 1, sigma=4.0, dropout_frac=0.3)[0]
    elif kind == 4:
        luma = edge_damage(luma, seed=seed + 1, per_field=int(rng.randint(3, 90)))
    else:
        luma = shift_rows(luma, int(rng.choice([-40, -12, -6, 5, 9, 20, 60])))
    blank = None
    if rng.rand() < 0.15:
        luma = luma.copy()
        blank = int(rng.randint(0, frames))
        luma[blank] = 16
    return np.ascontiguousarray(luma), pal, f16, f"seed {seed} {frames}x{luma.shape[1]} {'PAL' if pal else 'NTSC'} f16 {f16} kind {kind} blank {blank}"


def stitch_settings(rng, pal, f16):
    """Random STC007DataStitcher settings, each drawn once and given to both sides."""
    p, q = [(True, True), (True, False), (False, False)][int(rng.choice(3, p=[0.6, 0.25, 0.15]))]
    return dict(video_std=int(rng.choice([0, 1 if pal else 2])), field_order=int(rng.choice([0, 1, 2], p=[0.45, 0.45, 0.1])),
                res16=[None, f16, not f16][int(rng.choice(3, p=[0.45, 0.45, 0.1]))], p_corr=p, q_corr=q,
                ignore_crc=bool(rng.rand() < 0.2), cwd=bool(rng.rand() < 0.5), broken_mask_dur=int(rng.choice([0, 64, 128, 255])),
                mask_seams=bool(rng.rand() < 0.8), fix_cut_above=bool(rng.rand() < 0.3),
                max_unch14=int(rng.choice([0x40, 0x10, 0x80])), max_unch16=int(rng.choice([0x20, 0x08, 0x40])))


def gpu_stitcher(h, s):
    from sdvpcmdecoder_b200 import operators as ops
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(s["field_order"]); st.setResolutionPreset(s["res16"])
    st.setPCorrection(s["p_corr"]); st.setQCorrection(s["q_corr"])
    st.setIgnoreCRC(s["ignore_crc"]); st.setForcedErrorCheck(not s["ignore_crc"])
    st.setCWDCorrection(s["cwd"]); st.setBrokenMaskDuration(s["broken_mask_dur"])
    st.setFineMaskSeams(s["mask_seams"]); st.setFineTopLineFix(s["fix_cut_above"])
    st.setFineMaxUnch14(s["max_unch14"]); st.setFineMaxUnch16(s["max_unch16"])
    return st


def stitch_case(seed):
    """The GPU's line records of a stitch tape (checked against the oracle), then doFrameReassembleAuto under 2-3 random settings
    against the host build under the same settings (blocks, samples, flags, frame info), and the same tape in 2-3 batches
    (file_start / file_end, the last frame of a batch again at the head of the next) against the single call.
    -> (mismatches, the settings used)."""
    import torch
    from sdvpcmdecoder_b200 import operators as ops
    rng = np.random.RandomState(50000 + seed)
    luma, pal, f16, desc = stitch_tape(seed)
    n, H, _ = luma.shape
    h = capi.Handle(0)
    used = []
    try:
        rec, aux, _, dev = decode(h, luma)
        d = lines_diff(H, util.line_arrays(rec, aux), oracle_arrays(O.v2d_stc007(2, luma, True)))
        if d:
            return [f"{desc}: line records: {d}"], used
        bad = []
        for _ in range(int(rng.randint(2, 4))):
            s = stitch_settings(rng, pal, f16)
            used.append(s)
            st = gpu_stitcher(h, s)
            blocks, samples, flags, info = st.doFrameReassembleAuto(dev, n, H, want_blocks=True, video_std=s["video_std"])
            torch.cuda.synchronize()
            got = (ops.records_to_numpy(blocks, BLOCK_REC), samples.cpu().numpy(), flags.cpu().numpy(), info)
            want = util.emu_stc007_stitch(rec, n, H, **s)
            wrong = [k for k, a, b in zip(("blocks", "samples", "flags", "info"), got, want) if not np.array_equal(a, b)]
            if wrong:
                bad.append(f"{desc} {s}: {wrong} differ from the host build ({len(got[0])} / {len(want[0])} blocks)")
                continue
            k = int(rng.randint(2, 4))
            cuts = [0] + sorted(int(c) for c in rng.choice(np.arange(1, n), size=min(k - 1, n - 1), replace=False)) + [n]
            parts = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                last = b == n
                hi = b if last else b + 1
                pb, ps, pf, pi = st.doFrameReassembleAuto(dev[a * H:hi * H], hi - a, H, want_blocks=True, video_std=s["video_std"],
                                                          file_start=(a == 0), file_end=last)
                torch.cuda.synchronize()
                parts.append((ops.records_to_numpy(pb, BLOCK_REC), ps.cpu().numpy(), pf.cpu().numpy(), pi))
            # info.start is the stream line of the frame in the call's own output: behind the blocks of the batches before
            for i in range(1, len(parts)):
                parts[i][3]["start"] += sum(len(p[1]) for p in parts[:i])
            cat = [np.concatenate([p[i] for p in parts]) for i in range(4)]
            wrong = [k for k, a, b in zip(("blocks", "samples", "flags"), cat, got) if not np.array_equal(a, b)]
            wrong += ["info." + k for k in capi.STC007_FRAME_INFO.names if not np.array_equal(cat[3][k], got[3][k])]
            if wrong:
                bad.append(f"{desc} {s} batches {cuts}: {wrong} differ from the single call")
    finally:
        h.close()
    return bad, used


def stitch_coverage(used):
    """Which of detect / preset each of video standard, field order and resolution took, and CWD off / on."""
    return {"std": {s["video_std"] == 0 for s in used}, "order": {s["field_order"] == 0 for s in used},
            "res": {s["res16"] is None for s in used}, "cwd": {s["cwd"] for s in used}}


STITCH_SEEDS = range(8)


def test_frame_assembly_on_gpu_records_equals_host_build(ctx):
    bad, used = [], []
    for seed in STITCH_SEEDS:
        b, u = stitch_case(seed)
        bad += b
        used += u
    assert not bad, "\n".join(bad)
    cov = stitch_coverage(used)
    assert all(v == {False, True} for v in cov.values()), cov


# ------------------------------------------------------------------------------------------------ A6: preset geometry, fused
def preset_case(seed):
    """A full-height tape at a random width: clean, with lines that carry a valid CRC and the words of another frame (BROKEN
    blocks, countdown windows), or with light damage; preset-geometry settings: lead-in 0 / 80, a halo or none, countdown_in,
    broken-mask duration, resolution mode, P / Q."""
    rng = np.random.RandomState(60000 + seed)
    W = int(rng.choice((720, 722, 1000, 1024, 1448, 1920)))
    m = W / 720.0
    n, pal = int(rng.randint(3, 8)), bool(rng.rand() < 0.6)
    x0, x1 = int(round(rng.randint(4, 30) * m)), int(W - round(rng.randint(4, 30) * m))
    luma = synth.make_stc007(n + 2, seed=seed, pal=pal, width=W, x0=x0, x1=x1)["luma"]
    luma, next_shard = np.ascontiguousarray(luma[:n]), np.ascontiguousarray(luma[n:])
    H = luma.shape[1]
    kind = int(rng.randint(3))
    if kind == 1:
        for _ in range(int(rng.randint(1, 5))):
            f, r = int(rng.randint(1, n)), int(rng.randint(0, H))
            luma[f, r] = luma[int(rng.randint(0, n)), int(rng.randint(0, H))]
    elif kind == 2:
        f = int(rng.randint(0, n))
        luma[f] = synth.damage_stc007(luma[f:f + 1], seed=seed + 1, sigma=6.0, dropout_frac=0.02)[0]
    p, q = [(True, True), (True, False), (False, False)][int(rng.randint(3))]
    cfg = dict(lead_in=int(rng.choice([0, 80])), halo=bool(rng.rand() < 0.5), countdown_in=int(rng.choice([0, 0, 5, 100, 255])),
               broken_mask_dur=int(rng.choice([0, 64, 128, 255])), res_mode=int(rng.choice(4, p=[0.55, 0.15, 0.15, 0.15])), p_corr=p, q_corr=q)
    return dict(luma=luma, next_shard=next_shard, pal=pal, cfg=cfg, desc=f"seed {seed} {n}x{H}x{W} {'PAL' if pal else 'NTSC'} kind {kind} {cfg}")


def host_preset(rec, n, H, pal, lead_in, halo, c):
    """Frame assembly with preset geometry (tests/test_sharding_gloo._assemble for PAL and NTSC) + the host build of the
    deinterleaver with the countdown carried in."""
    lpf = 294 if pal else 245
    hf, nb = H // 2, lead_in + n * 2 * lpf
    asm = np.zeros(nb + 112, LINE_REC)
    for fld in range(2 * n):
        src = (fld // 2) * H + (fld & 1) * hf
        asm[lead_in + fld * lpf:lead_in + fld * lpf + hf] = rec[src:src + hf]
    if halo is not None:
        asm[nb:nb + 112] = halo
    _, s, f, _ = util.emu_deint_carry(asm, c["countdown_in"], c["res_mode"], False, True, c["p_corr"], c["q_corr"], c["broken_mask_dur"])
    return s, f


def check_preset_case(case):
    """doFrameReassemble against the host build, then fused with the next decode (cold and warm handle) against the separate
    pass, byte for byte.  -> mismatches."""
    import torch
    from sdvpcmdecoder_b200 import operators as ops
    luma, c, pal = case["luma"], case["cfg"], case["pal"]
    n, H, _ = luma.shape
    bad = []
    h = capi.Handle(0)
    try:
        rec, aux, _, recs = decode(h, luma)
        d = lines_diff(H, util.line_arrays(rec, aux), oracle_arrays(O.v2d_stc007(2, luma, True)))
        if d:
            return [f"{case['desc']}: line records: {d}"]
        halo = None
        if c["halo"]:
            hh = capi.Handle(0)
            halo = decode(hh, case["next_shard"])[3][:112].clone()
            hh.close()

        def stitcher(hh):
            st = ops.STC007DataStitcher(hh)
            st.setVideoStandard(ops.VID_PAL if pal else ops.VID_NTSC)
            st.lead_in = c["lead_in"]
            st.setResMode(c["res_mode"]); st.setPCorrection(c["p_corr"]); st.setQCorrection(c["q_corr"])
            st.setBrokenMaskDuration(c["broken_mask_dur"])
            return st
        st = stitcher(h)
        _, s0, f0 = st.doFrameReassemble(recs, n, H, halo=halo, countdown_in=c["countdown_in"])
        torch.cuda.synchronize()
        s0, f0 = s0.cpu().numpy(), f0.cpu().numpy()
        es, ef = host_preset(rec, n, H, pal, c["lead_in"], None if halo is None else halo.cpu().numpy().reshape(-1).view(LINE_REC), c)
        if not (np.array_equal(s0, es) and np.array_equal(f0, ef)):
            bad.append(f"{case['desc']}: separate pass differs from the host build")
        dev = torch.from_numpy(luma).cuda()
        nb = st.block_count(n)
        smp = torch.empty((nb, 6), dtype=torch.int16, device="cuda")
        fl = torch.empty((nb, 6), dtype=torch.uint8, device="cuda")
        for call in ("cold", "warm"):
            hf = capi.Handle(0) if call == "cold" else h
            st = stitcher(hf)
            smp.fill_(12345); fl.fill_(99)
            st.fuseWithNextDecode(smp, fl, countdown_in=c["countdown_in"])
            v2d = ops.VideoToDigital(hf)
            r = v2d.doBinarize(dev)
            st.doFrameReassemble(r, n, H, samples=smp, flags=fl, halo=halo, countdown_in=c["countdown_in"])
            torch.cuda.synchronize()
            if not (np.array_equal(smp.cpu().numpy(), s0) and np.array_equal(fl.cpu().numpy(), f0)):
                bad.append(f"{case['desc']} fused {call}: differs from the separate pass")
            if hf is not h:
                hf.close()
    finally:
        h.close()
    return bad


PRESET_SEEDS = range(6)


def test_preset_geometry_fused_and_separate(ctx):
    bad = [m for s in PRESET_SEEDS for m in check_preset_case(preset_case(s))]
    assert not bad, "\n".join(bad)
