"""PCM-1 line decode on the GPU (through the C ABI) against the reference's line records and sample streams (stored in
tests/golden/reference_streams.json) and the golden fixtures."""
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
    v2d.setPCMType(capi.TYPE_PCM1)
    v2d.setBinarizationMode(mode)
    v2d.setCheckLineDup(dup)
    recs, aux = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda(), want_aux=True)
    torch.cuda.synchronize()
    return ops.records_to_numpy(recs, LINE_REC), ops.records_to_numpy(aux, LINE_AUX), v2d.stats()


def _check(ctx, luma, mode=2, dup=True):
    """The product's records of every line equal the reference's (VideoToDigital, flag bit 11 aside); -> (records, stats)."""
    rec, aux, st = _decode(ctx, luma, mode, dup)
    bad = util.lines_mismatch("pcm1_lines", luma, (mode, dup), rec, aux)
    assert not bad, bad
    return rec, st


# the tapes of the line tests: (luma, mode, dup) lists, shared with tests/golden/make_golden.py
def clean_tape():
    return synth.make_pcm1(12)["luma"]


def modes_runs(mode):
    base = synth.make_pcm1(3, seed=21 + mode)["luma"]
    return [(base, mode, True), (base, mode, False), (synth.make_pcm1(3, seed=7, header=True)["luma"], mode, True)]


def damaged_runs(mode):
    base = synth.make_pcm1(2)["luma"]
    return [(t, mode, True) for t in (
        synth.damage_stc007(base, seed=100 + mode),
        synth.damage_stc007(base, seed=200 + mode, jitter=False, blur=False, sigma=25., dropout_frac=0.05),
        synth.make_pcm1(2, seed=11, x0=-9, x1=705)["luma"],
        synth.make_pcm1(2, seed=12, x0=10, x1=726)["luma"],
        synth.damage_stc007(synth.make_pcm1(2, seed=13, x0=-12, x1=728)["luma"], seed=5, jitter=False, blur=False, sigma=6., dropout_frac=0.02),
        synth.make_pcm1(2, seed=14, x0=30, x1=690)["luma"])]


def sparse_tape():
    luma = synth.make_pcm1(10, seed=5)["luma"].copy()
    luma[3, 100:104, 200:500] = 255          # a dropout in frame 3
    luma[7, 0, :] = 16                       # first line of frame 7 blank
    return luma


def unaligned_tape():
    return synth.make_pcm1(3, seed=9, width=722, x0=9, x1=713)["luma"]


def insane_runs():
    base = synth.make_pcm1(1)["luma"]
    return [(base[:, :64], 3, True), (synth.damage_stc007(base, seed=102)[:, :120], 3, True)]


WIDTHS = [352, 1024, 1920]


def width_runs(width):
    m = width / 720.0
    luma = synth.make_pcm1(3, seed=width, width=width, x0=int(8 * m), x1=width - int(8 * m))["luma"]
    return [(luma, 2, True), (synth.damage_stc007(luma[:2], seed=width + 1, sigma=6.0, dropout_frac=0.03, jitter=False, blur=False), 2, True)]


def line_runs():
    runs = [(clean_tape(), 2, True), (sparse_tape(), 2, True), (unaligned_tape(), 2, True)] + insane_runs()
    for mode in (0, 1, 2):
        runs += modes_runs(mode) + damaged_runs(mode)
    for w in WIDTHS:
        runs += width_runs(w)
    return runs


MANUAL_OFFSETS = ((3, 2), (-8, 1), (-10, -10))


def test_clean_tape_all_fields_and_bulk_path(ctx):
    luma = clean_tape()
    ref, st = _check(ctx, luma)
    assert st["frames_skipped"] == 12 and st["lines_chain"] == 0      # every frame taken from the bulk kernel
    assert (ref["flags"] & 1).mean() > 0.99


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_modes_dup_and_header(ctx, mode):
    for luma, m, dup in modes_runs(mode):
        _check(ctx, luma, m, dup)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_damaged_and_cut_tapes(ctx, mode):
    for luma, m, dup in damaged_runs(mode):
        _check(ctx, luma, m, dup)


def test_sparse_damage_mixes_bulk_and_chain(ctx):
    ref, st = _check(ctx, sparse_tape())
    assert 0 < st["frames_skipped"] < 10 and st["lines_chain"] > 0


def test_unaligned_width(ctx):
    _check(ctx, unaligned_tape())


def test_mode_insane_reference_level_sweep(ctx):
    """MODE_INSANE: a full coordinate search at every reference level for every line that fails the presets (and for the
    four prescan lines of every frame).  Small frames: the reference needs seconds per swept line."""
    (a, ma, da), (b, mb, db) = insane_runs()
    _check(ctx, a, ma, da)
    ref, st = _check(ctx, b, mb, db)
    assert ((ref["flags"] >> 5) & 1).sum() > 0          # lines decoded by the sweep


def _samples(ctx, luma, mode=2, bff=False, ignore_crc=False):
    h, ops, torch = ctx
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(capi.TYPE_PCM1)
    v2d.setBinarizationMode(mode)
    recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    st = ops.PCM1DataStitcher(h)
    st.setFieldOrder(st.ORDER_BFF if bff else st.ORDER_TFF)
    st.setIgnoreCRC(ignore_crc)
    smp, fl, info = st.doFrameReassemble(recs, luma.shape[0], luma.shape[1], want_info=True)
    torch.cuda.synchronize()
    return smp.cpu().numpy(), fl.cpu().numpy() & 3, ops.records_to_numpy(info, capi.PCM1_FRAME_INFO), ops.records_to_numpy(recs, LINE_REC)


def test_pipeline_samples_against_reference(ctx):
    from tests.test_pcm1_line import pcm1_cases
    for name, luma in pcm1_cases().items():
        for bff in (False, True):
            smp, fl, info, _ = _samples(ctx, luma, 2, bff)
            bad = util.stream_mismatch_digests(util.golden_stream("pcm1", luma, (bff,)), [smp.reshape(-1), fl.reshape(-1)])
            assert not bad, (name, bff, bad)


def test_golden_lines_and_samples(ctx):
    from tests.test_pcm1_line import pcm1_cases
    g = np.load(os.path.join(GOLD, "pcm1_lines.npz"))
    cases = pcm1_cases()
    for name in ("clean", "header", "damaged", "cutboth"):
        smp, fl, info, rec = _samples(ctx, cases[name])
        assert np.array_equal(g[name + "_recs"].view(LINE_REC).reshape(-1), rec), name
        assert np.array_equal(g[name + "_samples"], smp) and np.array_equal(g[name + "_sflags"], fl), name


def test_config2_round_trip(ctx):
    """BASELINE config 2 at full size (1000 frames, tiled from 50): every source sample pair comes back, bit-exact."""
    t = synth.make_pcm1(50)
    luma = np.tile(t["luma"], (20, 1, 1))
    smp, fl, info, rec = _samples(ctx, luma)
    src = synth.pcm1_expand(t["pairs"]).reshape(50, 2, 735, 2)
    got = smp.reshape(1000, 2, 735, 2)
    valid = (fl.reshape(1000, 2, 735, 2) & 2) != 0
    want = np.tile(src, (20, 1, 1, 1))
    assert valid.mean() > 0.97                      # 5 uncaptured lines per field + the first line of every field
    assert np.array_equal(got[valid], want[valid])
    assert (rec["flags"] & 1).mean() > 0.99


def test_manual_line_offsets(ctx):
    from tests.test_pcm1_line import pcm1_cases
    h, ops, torch = ctx
    luma = pcm1_cases()["clean"]
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(capi.TYPE_PCM1)
    recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    for ofs in MANUAL_OFFSETS:
        st = ops.PCM1DataStitcher(h)
        st.setAutoLineOffset(False); st.setOddLineOffset(ofs[0]); st.setEvenLineOffset(ofs[1])
        smp, fl = st.doFrameReassemble(recs, luma.shape[0], luma.shape[1])
        torch.cuda.synchronize()
        ref = util.golden_stream("pcm1_offsets", luma, ofs)
        bad = util.stream_mismatch_digests(ref, [smp.cpu().numpy().reshape(-1), fl.cpu().numpy().reshape(-1) & 3])
        assert not bad, (ofs, bad)


@pytest.mark.parametrize("width", WIDTHS)
def test_frame_widths(ctx, width):
    for luma, m, dup in width_runs(width):
        _check(ctx, luma, m, dup)
