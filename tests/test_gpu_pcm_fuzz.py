"""Randomised differential tests of the PCM-1 / PCM-16x0 kernels against the host build of the same device code
(tests/hostemu: one-thread blocks, no bulk kernel), and of pitched / unaligned luma buffers through the C ABI for all three
formats.  The host build is pinned to the reference by the stored digests and the CPU suite, so a difference here points at
what only the GPU runs: the warp-per-frame bulk kernels (bulk copy or plain loads into compact slots, the grid loop over
frames), the block-wide prescan and chain kernels and their bulk/chain hand-off, the stitch kernels.

The case builders are plain functions of a seed, so that tools/gpu_fuzz_pcm.py can run them over long seed ranges."""
import ctypes as C

import numpy as np
import pytest

from oracle import oraclebind as O
from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX
from tests import util
from tests.test_pcm16x0_stitch import variant_b, shift_rows, edge_damage

pytestmark = pytest.mark.gpu

P1, X0, STC = "pcm1", "pcm16x0", "stc007"
PCM_TYPE = {P1: capi.TYPE_PCM1, X0: capi.TYPE_PCM16X0, STC: capi.TYPE_STC007}
FIELDS = ["words", "flags"] + util.REC_FIELDS[1:] + ["mark_stages"] + ["aux." + n for n in util.AUX_FIELDS]


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators
    assert torch.cuda.is_available()
    return capi.Handle(0), operators, torch


# ------------------------------------------------------------------------------------------------ decode and compare
def gpu_lines(ctx, fmt, luma, mode=2, dup=True):
    """VideoToDigital on the GPU -> (records, aux, stats)."""
    h, ops, torch = ctx
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(PCM_TYPE[fmt])
    v2d.setBinarizationMode(mode)
    v2d.setCheckLineDup(dup)
    recs, aux = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda(), want_aux=True)
    torch.cuda.synchronize()
    return ops.records_to_numpy(recs, LINE_REC), ops.records_to_numpy(aux, LINE_AUX), v2d.stats(), recs


def host_lines(fmt, luma, mode=2, dup=True):
    """The host build of the same line decode + chain -> (records, aux)."""
    rec, aux, _ = (util.emu_p1_v2d if fmt == P1 else util.emu_x0_v2d)(luma, mode, dup)
    return rec, aux


def lines_diff(fmt, height, got, want):
    """'' when the compared fields (util.line_arrays) of two (records, aux) pairs are equal; else every field that differs, with
    its first differing records as (frame, record of the frame) and both values."""
    x0 = fmt == X0
    a, b = util.line_arrays(*got, with_part=x0), util.line_arrays(*want, with_part=x0)
    per = height * (3 if x0 else 1)
    out = []
    for name, u, v in zip(FIELDS + (["part"] if x0 else []), a, b):
        if len(u) != len(v):
            return f"{len(u)} records, host build {len(v)}"
        d = u != v
        if d.ndim > 1:
            d = d.reshape(len(u), -1).any(axis=1)
        if d.any():
            i = np.nonzero(d)[0][:4]
            out.append(f"{name}: {int(d.sum())} records, first {[(int(k) // per, int(k) % per) for k in i]} gpu {u[i].tolist()} host {v[i].tolist()}")
    return "; ".join(out)


def valid_fraction(rec):
    return float((rec["flags"] & 1).mean()) if len(rec) else 0.0


# ------------------------------------------------------------------------------------------------ A1: random line decode
LINE_WIDTHS = (360, 500, 720, 722, 728, 1000, 1448, 1920, 2048)
CROPS = (240, 96, 62, 24)


def line_case(fmt, seed):
    """A random PCM-1 / PCM-16x0 tape: width, data coordinates scaled with it (off-screen at either edge too), levels, damage,
    mode, duplicate check, PCM-1 header lines, 1-4 frames, mostly 480 rows but also crops."""
    rng = np.random.RandomState(2 * seed + (fmt == X0))
    W = int(rng.choice(LINE_WIDTHS))
    m = W / 720.0
    x0 = int(round(rng.randint(-14, 40) * m))
    x1 = int(W - round(rng.randint(-14, 40) * m))
    black, white = int(rng.randint(5, 60)), int(rng.randint(120, 250))
    n = int(rng.randint(1, 5))
    mode, dup = int(rng.randint(0, 3)), bool(rng.rand() < 0.7)
    header = fmt == P1 and bool(rng.rand() < 0.3)
    if fmt == P1:
        luma = synth.make_pcm1(n, seed=seed, width=W, x0=x0, x1=x1, black=black, white=white, header=header)["luma"]
    else:
        luma = synth.make_pcm16x0(n, seed=seed, width=W, x0=x0, x1=x1, black=black, white=white)["luma"]
    damage = bool(rng.rand() < 0.8)
    if damage:
        luma = synth.damage_stc007(luma, seed=seed + 1, sigma=float(rng.choice([0., 4., 10., 20.])), jitter=bool(rng.rand() < 0.4),
                                   blur=bool(rng.rand() < 0.4), dropout_frac=float(rng.choice([0., 0.02, 0.1])),
                                   marker_kill_frac=float(rng.choice([0., 0.02])), src_black=black, src_white=white)
    H = 480
    if rng.rand() < 0.35:
        H = int(rng.choice(CROPS))
        top = 2 * int(rng.randint(0, (480 - H) // 2 + 1))
        luma = luma[:, top:top + H]
    desc = f"seed {seed} {fmt} {n}x{H}x{W} mode {mode} dup {dup} x {x0} {x1} bw {black} {white} header {header} damage {damage}"
    return dict(fmt=fmt, luma=np.ascontiguousarray(luma), mode=mode, dup=dup, desc=desc)


def check_line_case(ctx, case):
    """-> (mismatch or '', valid fraction of the host build's records, stats of the GPU call)."""
    luma = case["luma"]
    got = gpu_lines(ctx, case["fmt"], luma, case["mode"], case["dup"])
    want = host_lines(case["fmt"], luma, case["mode"], case["dup"])
    bad = lines_diff(case["fmt"], luma.shape[1], got[:2], want)
    return (case["desc"] + ": " + bad if bad else ""), valid_fraction(want[0]), got[2]


def sweep_coverage(fracs):
    """(cases with at least 90 % valid lines, cases that mix valid and invalid lines)."""
    f = np.asarray(fracs)
    return int((f >= 0.9).sum()), int(((f > 0.02) & (f < 0.98)).sum())


LINE_SEEDS = range(40)


@pytest.mark.parametrize("fmt", [P1, X0])
def test_random_line_decode_equals_host_build(ctx, fmt):
    bad, fracs = [], []
    for seed in LINE_SEEDS:
        msg, frac, _ = check_line_case(ctx, line_case(fmt, seed))
        fracs.append(frac)
        if msg:
            bad.append(msg)
    assert not bad, "\n".join(bad)
    # a sweep of tapes that decode nothing would prove nothing: enough of them must be mostly valid, enough must mix
    mostly, mixed = sweep_coverage(fracs)
    assert mostly >= 8 and mixed >= 8, (mostly, mixed, np.round(fracs, 2).tolist())


# ------------------------------------------------------------------------------------------------ A2: bulk/chain hand-off
def handoff_case(fmt, seed, W, n_frames, dup=True, n_src=6):
    """A clean tape (n_src frames repeated) with a few random frames damaged: a dropout band, a blank first line, one line with
    another gain, a line with a valid CRC but the words of another frame."""
    rng = np.random.RandomState(2 * seed + (fmt == X0))
    m = W / 720.0
    if fmt == P1:
        src = synth.make_pcm1(n_src, seed=seed, width=W, x0=int(round(8 * m)), x1=W - int(round(8 * m)))["luma"]
    else:
        src = synth.make_pcm16x0(n_src, seed=seed, width=W)["luma"]
    luma = np.ascontiguousarray(np.tile(src, (-(-n_frames // n_src), 1, 1))[:n_frames])
    H = luma.shape[1]
    hits = []
    for f in sorted(rng.choice(np.arange(1, n_frames), size=min(6, n_frames - 1), replace=False).tolist()):
        kind = int(rng.randint(4))
        r = int(rng.randint(0, H))
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
            other = (f % n_src + 1 + int(rng.randint(n_src - 1))) % n_src
            luma[f, r] = src[other, int(rng.randint(0, H))]
        hits.append((f, kind, r))
    return dict(fmt=fmt, luma=luma, mode=2, dup=dup, desc=f"seed {seed} {fmt} {n_frames}x{H}x{W} dup {dup} damage (frame, kind, row) {hits}")


HANDOFF_CASES = [(P1, 720, 40, True), (X0, 720, 40, False), (P1, 1000, 24, True), (X0, 1000, 24, True),
                 (P1, 1920, 200, True), (X0, 1920, 200, True)]


@pytest.mark.parametrize("fmt,width,n_frames,dup", HANDOFF_CASES)
def test_bulk_chain_handoff_on_long_tapes(ctx, fmt, width, n_frames, dup):
    """At 1920 px the bulk kernel runs one warp per block, so 200 frames loop inside a grid capped at the SM count."""
    case = handoff_case(fmt, 7000 + width + n_frames, width, n_frames, dup)
    msg, frac, st = check_line_case(ctx, case)
    assert not msg, msg
    assert 0 < st["frames_skipped"] < n_frames, (case["desc"], st)       # the bulk kernel served frames, the chain the others
    assert frac > 0.98


# ------------------------------------------------------------------------------------------------ A3: MODE_INSANE
def insane_case(fmt, seed):
    rng = np.random.RandomState(seed)
    W = int(rng.choice([640, 720, 960]))
    m = W / 720.0
    x0, x1 = int(round(rng.randint(2, 24) * m)), int(W - round(rng.randint(2, 24) * m))
    black, white = int(rng.randint(5, 60)), int(rng.randint(120, 250))
    H = int(rng.choice([32, 48, 64]))
    if fmt == P1:
        luma = synth.make_pcm1(1, seed=seed, width=W, x0=x0, x1=x1, black=black, white=white)["luma"]
    else:
        luma = synth.make_pcm16x0(1, seed=seed, width=W, x0=x0, x1=x1, black=black, white=white)["luma"]
    luma = synth.damage_stc007(luma, seed=seed + 1, sigma=float(rng.choice([4., 10.])), jitter=True, blur=bool(rng.rand() < 0.5),
                               dropout_frac=0.05, marker_kill_frac=0.02, src_black=black, src_white=white)
    dup = bool(rng.rand() < 0.7)
    return dict(fmt=fmt, luma=np.ascontiguousarray(luma[:, :H]), mode=3, dup=dup, desc=f"seed {seed} {fmt} 1x{H}x{W} MODE_INSANE dup {dup}")


@pytest.mark.parametrize("fmt", [P1, X0])
def test_mode_insane_equals_host_build(ctx, fmt):
    bad = [m for m in (check_line_case(ctx, insane_case(fmt, s))[0] for s in (1, 2, 3)) if m]
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ A4: frame assembly
def stitch_tape(fmt, rng, ei=False):
    """A 4-frame tape for the stitchers (parity_fuzz_p1_stitch / parity_fuzz_x0_stitch recipe): header line or control-bit
    layout, variant B spans, heavy noise, damage, blanked spans and frames, edge damage, vertical shift."""
    if fmt == P1:
        header = bool(rng.randint(2))
        base = synth.make_pcm1(4, seed=rng.randint(1 << 20), header=header)["luma"]
        tag = ["plain", "header"][header]
    else:
        ctrl = [(1, 2), (2,), (), (0, 1, 2, 3), (1,)][rng.randint(5)]
        base = synth.make_pcm16x0(4, seed=rng.randint(1 << 20), ei=ei, ctrl_lines=ctrl)["luma"]
        tag = f"ctrl {ctrl} {'EI' if ei else 'SI'}"
    kind = int(rng.randint(7))
    luma = base
    if kind == 1:
        luma = variant_b(base, seed=rng.randint(1000), frac=rng.choice([0.05, 0.2, 0.5]))
    if kind == 2:
        luma = synth.damage_stc007(base, seed=rng.randint(1000), jitter=False, blur=False, sigma=float(rng.choice([15, 25, 40])),
                                   dropout_frac=float(rng.choice([0.02, 0.1, 0.3])))
    if kind == 3:
        luma = synth.damage_stc007(base, seed=rng.randint(1000))
    if kind == 4:
        luma = base.copy()
        a = rng.randint(0, 400)
        luma[rng.randint(4), a:a + rng.randint(20, 300)] = 16
    if kind == 5:
        luma = base.copy()
        luma[rng.randint(4)] = 16
    if kind == 6:
        luma = edge_damage(base, seed=rng.randint(1000), per_field=int(rng.randint(25, 50)))
    sh = int(rng.choice([0, 0, 0, 1, 3, -2, -7, 12, -20, 50, -60]))
    return np.ascontiguousarray(shift_rows(luma, sh)), f"{tag} kind {kind} shift {sh}"


def gpu_recs_checked(ctx, fmt, luma, desc):
    """The GPU's line records of a stitch tape, after checking that they equal the host build's -> (device records, host copy)."""
    rec, aux, _, dev = gpu_lines(ctx, fmt, luma)
    bad = lines_diff(fmt, luma.shape[1], (rec, aux), host_lines(fmt, luma))
    return dev, rec, (desc + ": line records: " + bad if bad else "")


def info_diff(got, want, names):
    return [n for n in names if not np.array_equal(got[n], want[n])]


def p1_stitch_case(ctx, seed):
    """PCM1DataStitcher on the GPU's records against the host build's assembly + the C oracle's deinterleaver: TFF / BFF,
    ignore-CRC, automatic or random manual line offsets, frame info.  -> list of mismatches."""
    h, ops, torch = ctx
    rng = np.random.RandomState(seed)
    luma, desc = stitch_tape(P1, rng)
    desc = f"seed {seed} {P1} {desc}"
    n, H = luma.shape[:2]
    dev, rec, bad = gpu_recs_checked(ctx, P1, luma, desc)
    if bad:
        return [bad]
    out = []
    for _ in range(3):
        bff, ign = bool(rng.randint(2)), bool(rng.rand() < 0.3)
        ofs = None if rng.rand() < 0.5 else (int(rng.randint(-10, 11)), int(rng.randint(-10, 11)))
        st = ops.PCM1DataStitcher(h)
        st.setFieldOrder(st.ORDER_BFF if bff else st.ORDER_TFF)
        st.setIgnoreCRC(ign)
        if ofs is not None:
            st.setAutoLineOffset(False); st.setOddLineOffset(ofs[0]); st.setEvenLineOffset(ofs[1])
        smp, fl, info = st.doFrameReassemble(dev, n, H, want_info=True)
        torch.cuda.synchronize()
        info = ops.records_to_numpy(info, capi.PCM1_FRAME_INFO)
        sub, einfo = util.emu_p1_assemble(rec, n, H, bff, True, ofs)
        es, ef = O.deint_pcm1(np.stack([sub["left"], sub["right"]], axis=1), sub["flags"], ignore_crc=ign)
        wrong = [k for k, (a, b) in (("samples", (smp.cpu().numpy(), es)), ("flags", (fl.cpu().numpy(), ef & 3))) if not np.array_equal(a, b)]
        wrong += info_diff(info, einfo, [k for k in capi.PCM1_FRAME_INFO.names if k != "reserved"])
        if wrong:
            out.append(f"{desc} bff {bff} ignore_crc {ign} offsets {ofs}: {wrong}")
    return out


def x0_preset_case(ctx, seed):
    """PCM16X0DataStitcher.doFrameReassemble (preset alignment) on the GPU's records against the host build: random top paddings,
    seam masks, P correction, ignore-CRC, broken-block mask 0 / 81 / 255, frame info.  -> list of mismatches."""
    h, ops, torch = ctx
    rng = np.random.RandomState(seed)
    luma, desc = stitch_tape(X0, rng)
    desc = f"seed {seed} {X0} preset {desc}"
    n, H = luma.shape[:2]
    dev, rec, bad = gpu_recs_checked(ctx, X0, luma, desc)
    if bad:
        return [bad]
    out = []
    for _ in range(3):
        bff, ign, p_corr = bool(rng.randint(2)), bool(rng.rand() < 0.3), bool(rng.rand() < 0.7)
        top = (int(rng.randint(0, 13)), int(rng.randint(0, 13)))
        dur = int(rng.choice([0, 81, 255]))
        seams = rng.randint(0, 2, n).astype(np.uint8)
        st = ops.PCM16X0DataStitcher(h)
        st.setFieldOrder(st.ORDER_BFF if bff else st.ORDER_TFF)
        st.setIgnoreCRC(ign); st.setPCorrection(p_corr); st.setTopPadding(*top); st.setFineBrokeMask(dur)
        smp, fl, info = st.doFrameReassemble(dev, n, H, mask_seams=torch.from_numpy(seams).cuda(), want_info=True)
        torch.cuda.synchronize()
        es, ef, einfo = util.emu_x0_stitch_info(rec, n, H, bff, top, ign, p_corr, dur, seams)
        wrong = [k for k, (a, b) in (("samples", (smp.cpu().numpy(), es)), ("flags", (fl.cpu().numpy(), ef))) if not np.array_equal(a, b)]
        wrong += info_diff(info, einfo, capi.PCM16X0_FRAME_INFO.names)
        if wrong:
            out.append(f"{desc} bff {bff} ignore_crc {ign} p_corr {p_corr} top {top} broken_mask {dur} seams {seams.tolist()}: {wrong}")
    return out


def x0_auto_case(ctx, seed):
    """doFrameReassembleAuto (the alignment searched on the device and decided in the library), SI or EI, on the GPU's records
    against the host build of the same search.  -> list of mismatches."""
    h, ops, torch = ctx
    rng = np.random.RandomState(seed)
    ei = bool(rng.randint(2))
    luma, desc = stitch_tape(X0, rng, ei=ei)
    desc = f"seed {seed} {X0} auto {desc}"
    n, H = luma.shape[:2]
    dev, rec, bad = gpu_recs_checked(ctx, X0, luma, desc)
    if bad:
        return [bad]
    out = []
    for bff, p_corr in ((False, True), (True, True), (False, False)):
        ign = bool(rng.rand() < 0.25)
        st = ops.PCM16X0DataStitcher(h)
        st.setFormat(st.FORMAT_EI if ei else st.FORMAT_SI)
        st.setFieldOrder(st.ORDER_BFF if bff else st.ORDER_TFF)
        st.setIgnoreCRC(ign); st.setPCorrection(p_corr)
        smp, fl, al = st.doFrameReassembleAuto(dev, n, H)
        torch.cuda.synchronize()
        es, ef, eal = util.emu_x0_stitch_auto(rec, n, H, bff, ignore_crc=ign, p_corr=p_corr, ei=ei)
        wrong = [k for k, (a, b) in (("samples", (smp.cpu().numpy(), es)), ("flags", (fl.cpu().numpy(), ef)), ("alignment", (al, eal)))
                 if not np.array_equal(a, b)]
        if wrong:
            out.append(f"{desc} bff {bff} ignore_crc {ign} p_corr {p_corr}: {wrong} gpu {al.tolist()} host {eal.tolist()}")
    return out


STITCH_SEEDS = range(8)


@pytest.mark.parametrize("part", ["pcm1", "pcm16x0_preset", "pcm16x0_auto"])
def test_frame_assembly_on_gpu_records_equals_host_build(ctx, part):
    fn = {"pcm1": p1_stitch_case, "pcm16x0_preset": x0_preset_case, "pcm16x0_auto": x0_auto_case}[part]
    bad = [m for s in STITCH_SEEDS for m in fn(ctx, 100 + s)]
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ B: pitched / unaligned luma
def decode_pitched(h, fmt, luma, stride, off, mode=2, dup=True, seed=0):
    """sdv_bin_decode_frames on a device buffer of n*H*stride + off bytes with the frames written at [stride] from byte [off].
    Whatever is not a pixel -- the off bytes in front, the stride - W bytes behind every row -- is hostile: noise, and in every
    other row the pixels of another PCM line.  Output buffers are pre-filled with one byte pattern, so that two calls can be
    compared byte for byte.  -> (records, aux, stats)."""
    import torch
    n, H, W = luma.shape
    rng = np.random.RandomState(seed)
    host = rng.randint(0, 256, off + n * H * stride).astype(np.uint8)
    rows = host[off:].reshape(n * H, stride)
    flat = luma.reshape(n * H, W)
    rows[:, :W] = flat
    k = min(stride - W, W)
    if k > 0:
        rows[::2, W:W + k] = np.roll(flat, 7, axis=0)[::2, :k]
    buf = torch.from_numpy(host).cuda()
    assert buf.data_ptr() % 16 == 0
    nrec = n * H * (3 if fmt == X0 else 1)
    recs = torch.full((nrec, LINE_REC.itemsize), 0xA5, dtype=torch.uint8, device="cuda")
    aux = torch.full((nrec, LINE_AUX.itemsize), 0x5A, dtype=torch.uint8, device="cuda")
    cfg = capi.BinConfig(pcm_type=PCM_TYPE[fmt], mode=mode, check_line_dup=int(dup))
    h.check(capi.lib().sdv_bin_decode_frames(h.ptr, C.byref(cfg), C.c_void_p(buf.data_ptr() + off), n, H, W, stride,
                                             C.c_void_p(recs.data_ptr()), C.c_void_p(aux.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return recs.cpu().numpy().reshape(-1).view(LINE_REC), aux.cpu().numpy().reshape(-1).view(LINE_AUX), h.last_stats()


def pitch_tapes(fmt, W):
    """(name, luma, clean) of one format at one width: a clean tape and a sparsely damaged one."""
    m = W / 720.0
    if fmt == STC:
        clean = synth.make_stc007(4, seed=W, width=W, x0=int(14 * m), x1=W - int(14 * m))["luma"]
    elif fmt == P1:
        clean = synth.make_pcm1(4, seed=W, width=W, x0=int(8 * m), x1=W - int(8 * m))["luma"]
    else:
        clean = synth.make_pcm16x0(4, seed=W, width=W)["luma"]
    sparse = clean.copy()
    sparse[1, 100:104, int(200 * m):int(500 * m)] = 255
    sparse[2, 0, :] = 16
    x = sparse[3, 301].astype(np.float32)
    sparse[3, 301] = np.clip((x - 16) * 0.7 + 30, 0, 255).astype(np.uint8)
    return [("clean", clean, True), ("sparse", sparse, False)]


PITCHES = [(720, s, o) for s in (720, 736, 723, 4096) for o in (0, 1, 16) if (s, o) != (720, 0)] + [(2048, 4096, 0), (2048, 4096, 1)]


def pitch_case(fmt, W):
    """Every pitched / offset geometry of PITCHES at width W against the contiguous call and the host build (STC-007: the C
    oracle); STC-007 decodes cold and then warm on the same handle.  -> list of mismatches."""
    bad = []
    for name, luma, clean in pitch_tapes(fmt, W):
        n, H, _ = luma.shape
        if fmt == STC:
            want = O.v2d_stc007(2, luma, True)
        else:
            want = host_lines(fmt, luma)
        base = decode_pitched(capi.Handle(0), fmt, luma, W, 0)
        for s, o in [(s, o) for w, s, o in PITCHES if w == W]:
            h = capi.Handle(0)
            for call in (("cold", "warm") if fmt == STC else ("cold",)):
                rec, aux, st = decode_pitched(h, fmt, luma, s, o, seed=s + o)
                tag = f"{fmt} {name} {n}x{H}x{W} stride {s} offset {o} {call}"
                if not (np.array_equal(rec.view(np.uint8), base[0].view(np.uint8)) and np.array_equal(aux.view(np.uint8), base[1].view(np.uint8))):
                    bad.append(f"{tag}: not byte-identical to the contiguous call")
                if fmt == STC:
                    d = util.compare_line_records(want, rec, aux)
                else:
                    d = lines_diff(fmt, H, (rec, aux), want)
                if d:
                    bad.append(f"{tag}: {d}")
                if clean and st["frames_skipped"] == 0:
                    bad.append(f"{tag}: no frame taken from the bulk kernel {st}")
            h.close()
    return bad


@pytest.mark.parametrize("fmt", [STC, P1, X0])
@pytest.mark.parametrize("width", [720, 2048])
def test_pitched_and_unaligned_luma_through_c_abi(ctx, fmt, width):
    bad = pitch_case(fmt, width)
    assert not bad, "\n".join(bad)
