"""PCM-16x0 line decode on the GPU (through the C ABI) against the reference's sub-line records and sample streams (stored in
tests/golden/reference_streams.json) and the golden fixture."""
import os

import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX
from tests import util

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators
    assert torch.cuda.is_available()
    return capi.Handle(0), operators, torch


def _decode(ctx, luma, mode=2, dup=True):
    h, ops, torch = ctx
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(capi.TYPE_PCM16X0)
    v2d.setBinarizationMode(mode)
    v2d.setCheckLineDup(dup)
    recs, aux = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda(), want_aux=True)
    torch.cuda.synchronize()
    return ops.records_to_numpy(recs, LINE_REC), ops.records_to_numpy(aux, LINE_AUX), v2d.stats()


def _check(ctx, luma, mode=2, dup=True):
    """The product's three sub-line records of every line equal the reference's (VideoToDigital, the part of the line
    included); -> (records, stats)."""
    rec, aux, st = _decode(ctx, luma, mode, dup)
    bad = util.lines_mismatch("pcm16x0_lines", luma, (mode, dup), rec, aux, with_part=True)
    assert not bad, bad
    return rec, st


# the tapes of the line tests: (luma, mode, dup) lists, shared with tests/golden/make_golden.py
def clean_tape():
    return synth.make_pcm16x0(10)["luma"]


def drift_tape():
    a = synth.make_pcm16x0(3, seed=1)["luma"]
    b = synth.make_pcm16x0(3, seed=2, x0=9, x1=713)["luma"]
    return np.concatenate([a, b, a[:2]])


def damaged_runs(mode):
    base = synth.make_pcm16x0(2)["luma"]
    return [(t, mode, True) for t in (
        base,
        synth.damage_stc007(base, seed=100 + mode),
        synth.damage_stc007(base, seed=200 + mode, jitter=False, blur=False, sigma=25., dropout_frac=0.05),
        synth.make_pcm16x0(2, seed=11, x0=-5, x1=710)["luma"],
        synth.make_pcm16x0(2, seed=12, x0=6, x1=723)["luma"],
        synth.damage_stc007(synth.make_pcm16x0(2, seed=13, x0=-7, x1=725)["luma"], seed=5, jitter=False, blur=False, sigma=6., dropout_frac=0.02),
        synth.make_pcm16x0(1, seed=15, width=1440)["luma"])]


def sparse_tape():
    luma = synth.make_pcm16x0(8, seed=5)["luma"].copy()
    luma[3, 100:104, 200:500] = 255
    luma[6, 0, :] = 16
    return luma


def insane_runs():
    base = synth.make_pcm16x0(1)["luma"]
    return [(base[:, :64], 3, True), (synth.damage_stc007(base, seed=102)[:, :64], 3, True)]


WIDTHS = [640, 1024, 1920]


def width_runs(width):
    luma = synth.make_pcm16x0(3, seed=width, width=width)["luma"]
    return [(luma, 2, True), (synth.damage_stc007(luma[:2], seed=width + 1, sigma=6.0, dropout_frac=0.03, jitter=False, blur=False), 2, True)]


def line_runs():
    runs = [(clean_tape(), 2, dup) for dup in (True, False)] + [(drift_tape(), 2, dup) for dup in (True, False)]
    runs += [(sparse_tape(), 2, True)] + insane_runs()
    for mode in (0, 1, 2):
        runs += damaged_runs(mode)
    for w in WIDTHS:
        runs += width_runs(w)
    return runs


def test_clean_tape_all_fields_and_bulk_path(ctx):
    luma = clean_tape()
    for dup in (True, False):
        ref, st = _check(ctx, luma, dup=dup)
        assert st["frames_skipped"] == 10 and st["lines_chain"] == 0, (dup, st)
    assert (ref["flags"] & 1).mean() > 0.99


def test_coordinates_drift_between_frames(ctx):
    """Frames whose prescan coordinates differ: with the duplicate-line check on the reference keeps decoding with the
    history median, without it every frame follows its own prescan."""
    luma = drift_tape()
    for dup in (True, False):
        _check(ctx, luma, dup=dup)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_damaged_and_cut_tapes(ctx, mode):
    for luma, m, dup in damaged_runs(mode):
        _check(ctx, luma, m, dup)


def test_sparse_damage_mixes_bulk_and_chain(ctx):
    ref, st = _check(ctx, sparse_tape())
    assert 0 < st["frames_skipped"] < 8 and st["lines_chain"] > 0


def test_golden_sublines(ctx):
    from tests.test_pcm16x0_line import pcm16x0_cases
    g = np.load(os.path.join(GOLD, "pcm16x0_lines.npz"))
    cases = pcm16x0_cases()
    for name in ("clean", "damaged", "cutboth", "drift"):
        rec, aux, st = _decode(ctx, cases[name])
        assert np.array_equal(g[name + "_recs"].view(LINE_REC).reshape(-1), rec), name


def test_pipeline_samples_against_reference(ctx):
    from tests.test_pcm16x0_stitch import stitch_cases, ref_pairs, frames_match
    h, ops, torch = ctx
    for name, luma in stitch_cases().items():
        v2d = ops.VideoToDigital(h)
        v2d.setPCMType(capi.TYPE_PCM16X0)
        recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
        n = luma.shape[0]
        for bff, p_corr in ((False, True), (True, True), (False, False)):
            st = ops.PCM16X0DataStitcher(h)
            st.setFieldOrder(st.ORDER_BFF if bff else st.ORDER_TFF)
            st.setPCorrection(p_corr)
            s0, f0 = st.doFrameReassemble(recs, n, luma.shape[1])
            s1, f1 = st.doFrameReassemble(recs, n, luma.shape[1], mask_seams=torch.ones(n, dtype=torch.uint8, device="cuda"))
            torch.cuda.synchronize()
            m = frames_match(ref_pairs(luma, bff, p_corr), (s0.cpu().numpy(), f0.cpu().numpy()), (s1.cpu().numpy(), f1.cpu().numpy()), n)
            assert -1 not in m, (name, bff, p_corr, m)
            if name == "clean":
                assert m == [0] * n


def test_config3_round_trip(ctx):
    """BASELINE config 3 at full size (1000 frames, tiled from 40): every source sample pair comes back, bit-exact."""
    h, ops, torch = ctx
    t = synth.make_pcm16x0(40)
    luma = np.tile(t["luma"], (25, 1, 1))
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(capi.TYPE_PCM16X0)
    recs = v2d.doBinarize(torch.from_numpy(luma).cuda())
    smp, fl = ops.PCM16X0DataStitcher(h).doFrameReassemble(recs, 1000, 480)
    torch.cuda.synchronize()
    st = v2d.stats()
    src = np.tile(t["pairs"].view(np.int16).reshape(40, 1470, 2), (25, 1, 1))
    assert np.array_equal(smp.cpu().numpy().reshape(1000, 1470, 2), src)
    assert ((fl.cpu().numpy() & 3) == 3).all()
    assert st["frames_skipped"] == 1000 and st["lines_chain"] == 0


def test_mode_insane_reference_level_sweep(ctx):
    (a, ma, da), (b, mb, db) = insane_runs()
    _check(ctx, a, ma, da)
    ref, st = _check(ctx, b, mb, db)
    assert ((ref["flags"] >> 5) & 1).sum() > 0


def test_host_buffer_entry_points(ctx):
    """sdv_pcm1_decode_tape_host / sdv_pcm16x0_decode_tape_host: host luma in, host samples out, same as the device-buffer path."""
    h, ops, torch = ctx
    t = synth.make_pcm16x0(6)
    smp, fl, rec = ops.decode_tape_host_pcm16x0(h, t["luma"], want_recs=True)
    assert np.array_equal(smp.reshape(-1, 2), t["pairs"].view(np.int16)[:6 * 1470]) and ((fl & 3) == 3).all()
    assert len(rec) == 6 * 480 * 3 and (rec["flags"] & 1).mean() > 0.99
    t1 = synth.make_pcm1(6)
    smp, fl, rec = ops.decode_tape_host_pcm1(h, t1["luma"], want_recs=True)
    src = synth.pcm1_expand(t1["pairs"]).reshape(-1)[:6 * 2940]
    valid = (fl & 2) != 0
    assert valid.mean() > 0.97 and np.array_equal(smp[valid], src[valid])


@pytest.mark.parametrize("width", WIDTHS)
def test_frame_widths(ctx, width):
    for luma, m, dup in width_runs(width):
        _check(ctx, luma, m, dup)


def test_frame_info_control_bits(ctx):
    # sdv_pcm16x0_frames_to_samples_info against the golden decisions of the reference pipeline (sample rate, emphasis)
    from tests.test_pcm16x0_stitch import info_cases, GOLD_INFO
    h, ops, torch = ctx
    g = np.load(GOLD_INFO)
    for name, luma in info_cases().items():
        v2d = ops.VideoToDigital(h)
        v2d.setPCMType(capi.TYPE_PCM16X0)
        recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
        st = ops.PCM16X0DataStitcher(h)
        s0, f0 = st.doFrameReassemble(recs, luma.shape[0], luma.shape[1])
        s1, f1, info = st.doFrameReassemble(recs, luma.shape[0], luma.shape[1], want_info=True)
        torch.cuda.synchronize()
        assert torch.equal(s0, s1) and torch.equal(f0, f1)
        got = np.stack([info["sample_rate"], info["emphasis"].astype(np.uint16)], axis=1)
        assert np.array_equal(got, g[name]), name


def test_own_alignment_equals_reference_pipeline(ctx):
    """sdv_pcm16x0_frames_to_samples_auto through the C ABI: the library finds the vertical alignment of every field itself
    (padding sweep on the device, findSIPadding's decisions on the host) -- the reference's PCMSamplePair stream frame by frame,
    on configs 3 / 3B, damaged tapes and vertically shifted captures; and the host build of the same code gives the same
    alignment records."""
    from tests.test_pcm16x0_stitch import alignment_cases, ref_pairs, pairs_mismatch
    h, ops, torch = ctx
    for name, luma in alignment_cases().items():
        v2d = ops.VideoToDigital(h)
        v2d.setPCMType(capi.TYPE_PCM16X0)
        recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
        n = luma.shape[0]
        for bff, p_corr in ((False, True), (True, True), (False, False)):
            st = ops.PCM16X0DataStitcher(h)
            st.setFieldOrder(2 if bff else 1); st.setPCorrection(p_corr)
            smp, fl, al = st.doFrameReassembleAuto(recs, n, luma.shape[1])
            torch.cuda.synchronize()
            ref = ref_pairs(luma, bff, p_corr)
            assert not pairs_mismatch(ref, smp.cpu().numpy(), fl.cpu().numpy()), (name, bff, p_corr, pairs_mismatch(ref, smp.cpu().numpy(), fl.cpu().numpy()), al)
            es, ef, eal = util.emu_x0_stitch_auto(ops.records_to_numpy(recs, LINE_REC), n, luma.shape[1], bff, p_corr=p_corr)
            assert np.array_equal(al, eal), (name, bff, p_corr)


def test_ei_stitching_equals_reference_pipeline(ctx):
    """The EI format through the C ABI (sdv_pcm16x0_frames_to_samples_auto with ei_format = 1): tryEIPadding x 81 paddings per
    frame on the device, findEIFrameStitching's decisions in the library -- the reference's PCMSamplePair stream with
    setFormat(FORMAT_EI) frame by frame, on every tape of ei_cases(); the host build gives the same alignment records; the
    padding history carries over calls (file_start = 0) and is dropped by a change of format."""
    from tests.test_pcm16x0_stitch import ei_cases, ref_pairs, pairs_mismatch
    h, ops, torch = ctx
    for name, luma in ei_cases().items():
        v2d = ops.VideoToDigital(h)
        v2d.setPCMType(capi.TYPE_PCM16X0)
        recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
        n = luma.shape[0]
        for bff, p_corr in ((False, True), (True, True), (False, False)):
            st = ops.PCM16X0DataStitcher(h)
            st.setFormat(st.FORMAT_EI); st.setFieldOrder(2 if bff else 1); st.setPCorrection(p_corr)
            smp, fl, al = st.doFrameReassembleAuto(recs, n, luma.shape[1])
            torch.cuda.synchronize()
            ref = ref_pairs(luma, bff, p_corr, ei=True)
            assert not pairs_mismatch(ref, smp.cpu().numpy(), fl.cpu().numpy()), (name, bff, p_corr, pairs_mismatch(ref, smp.cpu().numpy(), fl.cpu().numpy()), al)
            es, ef, eal = util.emu_x0_stitch_auto(ops.records_to_numpy(recs, LINE_REC), n, luma.shape[1], bff, p_corr=p_corr, ei=True)
            assert np.array_equal(al, eal), (name, bff, p_corr)
            if name in ("clean", "shift3") and p_corr:
                # the preset-alignment entry in the EI format, given the paddings the search found (no field is cut on these tapes)
                assert (al["cut_lines"] == 0).all() and (al["mask_seams"] == 0).all()
                st.setTopPadding(int(al["top_padding"][0][0]), int(al["top_padding"][0][1]))
                ps, pf = st.doFrameReassemble(recs, n, luma.shape[1])
                assert not pairs_mismatch(ref, ps.cpu().numpy(), pf.cpu().numpy()), (name, bff, "preset EI")
            if name in ("shift50", "blanked_shift-20") and not bff and p_corr:
                # two calls of two frames = one call of four (the history of accepted paddings stays on the handle) ...
                rl = ops.records_to_numpy(recs, LINE_REC).reshape(n, -1)
                halves = []
                for k, fs in ((0, True), (2, False)):
                    part = torch.from_numpy(np.ascontiguousarray(rl[k:k + 2]).view(np.uint8)).cuda()
                    halves.append(st.doFrameReassembleAuto(part, 2, luma.shape[1], file_start=fs))
                assert np.array_equal(np.concatenate([x[0].cpu().numpy() for x in halves]), smp.cpu().numpy()), name      # = the reference's
                assert np.array_equal(np.concatenate([x[2] for x in halves]), al), name
                # ... and an SI call in between drops it
                st.setFormat(st.FORMAT_SI)
                st.doFrameReassembleAuto(recs, 1, luma.shape[1], file_start=False)
                st.setFormat(st.FORMAT_EI)
                part = torch.from_numpy(np.ascontiguousarray(rl[2:]).view(np.uint8)).cuda()
                fresh = st.doFrameReassembleAuto(part, 2, luma.shape[1], file_start=True)
                again = st.doFrameReassembleAuto(part, 2, luma.shape[1], file_start=False)      # history of "fresh"
                st.setFormat(st.FORMAT_SI)
                st.doFrameReassembleAuto(recs, 1, luma.shape[1], file_start=False)
                st.setFormat(st.FORMAT_EI)
                dropped = st.doFrameReassembleAuto(part, 2, luma.shape[1], file_start=False)
                assert np.array_equal(dropped[2], fresh[2]), name
                assert again[2].shape == fresh[2].shape


def test_ei_tape_round_trip_at_length(ctx):
    """500 EI frames: every source sample pair comes back through line decode + the EI stitcher, all flagged valid."""
    h, ops, torch = ctx
    t = synth.make_pcm16x0(50, seed=77, ei=True, ctrl_lines=(1, 2))
    luma = torch.from_numpy(np.ascontiguousarray(np.tile(t["luma"], (10, 1, 1)))).cuda()
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(capi.TYPE_PCM16X0)
    recs = v2d.doBinarize(luma)
    st = ops.PCM16X0DataStitcher(h)
    st.setFormat(st.FORMAT_EI)
    smp, fl, al = st.doFrameReassembleAuto(recs, 500, 480)
    src = np.tile(t["pairs"].view(np.int16)[:50 * 1470], (10, 1))
    assert np.array_equal(smp.cpu().numpy().reshape(-1, 2), src)
    assert ((fl.cpu().numpy() & 3) == 3).all()
    assert (al["result"][:, 0] == 4).all() and (al["result"][:, 1] == 5).all() and not al["mask_seams"].any()
