"""PCM-16x0 frame assembly + deinterleave with preset alignment (device code built for the host) against the reference
pipeline (VideoToDigital + PCM16X0DataStitcher, SI format).  The reference searches the vertical alignment itself; on
frames where its search is unsure it additionally masks the first data blocks (seam masking): the product takes that
per-frame decision as an input, so every reference frame must equal the product's frame with the mask off or on."""
import os

import numpy as np
import pytest

from oracle import refbind as R
from sdvpcmdecoder_b200 import synth
from tests import util

have_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref not built")


def variant_b(luma, seed=99, frac=0.08, span=72):
    """Config 3 variant B: a 72-pixel span blanked in 8 % of the lines."""
    rng = np.random.RandomState(seed)
    out = luma.copy().reshape(-1, luma.shape[2])
    for r in np.nonzero(rng.rand(out.shape[0]) < frac)[0]:
        st = rng.randint(0, luma.shape[2] - span)
        out[r, st:st + span] = 16
    return out.reshape(luma.shape)


def ref_pairs(luma, bff=False, p_corr=True, ei=False):
    """The stored PCMSamplePair stream of VideoToDigital + PCM16X0DataStitcher (FORMAT_SI or FORMAT_EI) on this tape: samples
    [n*490, 6] and flags & 7 per frame (tests/golden/reference_streams.json; provenance in make_golden.streams_golden)."""
    return util.golden_stream("pcm16x0", luma, (bff, p_corr, ei))


def pairs_mismatch(ref, smp, fl):
    """'' when samples [n*490, 6] i16 and flags [n*490, 6] u8 equal the reference stream ref_pairs() gave."""
    return util.stream_mismatch_digests(ref, [np.asarray(smp, np.int16), np.asarray(fl, np.uint8)])


def frames_match(ref, got0, got1, n_frames):
    """-> list of 0/1/-1 per frame: which product variant (mask off / on) the reference frame equals."""
    assert ref["rows"] == n_frames * 490 and ref["chunk"] == 490
    d0 = util.chunk_digests([np.asarray(got0[0], np.int16), np.asarray(got0[1], np.uint8)], 490)
    d1 = util.chunk_digests([np.asarray(got1[0], np.int16), np.asarray(got1[1], np.uint8)], 490)
    return [0 if r == a else 1 if r == b else -1 for r, a, b in zip(ref["digests"], d0, d1)]


def stitch_cases():
    base = synth.make_pcm16x0(3)["luma"]
    return {"clean": base, "variantB": variant_b(base),
            "noise": synth.damage_stc007(base, seed=202, jitter=False, blur=False, sigma=25., dropout_frac=0.05),
            "damaged": synth.damage_stc007(base, seed=102)}


def test_samples_against_reference_pipeline():
    for name, luma in stitch_cases().items():
        if name == "damaged":
            continue                # (the strict own-alignment test below covers it; this one accepts either masking variant)
        rec, _, _ = util.emu_x0_v2d(luma, 2, True)
        n = luma.shape[0]
        for bff, p_corr in ((False, True), (True, True), (False, False)):
            ref = ref_pairs(luma, bff, p_corr)
            got0 = util.emu_x0_stitch(rec, n, luma.shape[1], bff, p_corr=p_corr)
            got1 = util.emu_x0_stitch(rec, n, luma.shape[1], bff, p_corr=p_corr, mask_seams=np.ones(n, np.uint8))
            m = frames_match(ref, got0, got1, n)
            assert -1 not in m, (name, bff, p_corr, m)
            if name == "clean":
                assert m == [0] * n


def shift_rows(luma, k):
    o = np.full_like(luma, 16)
    if k > 0:
        o[:, k:] = luma[:, :-k]
    elif k < 0:
        o[:, :k] = luma[:, -k:]
    else:
        o[:] = luma
    return o


def edge_damage(luma, seed=31, per_field=35):
    """All three CRCs broken (levels still found) in the first and the last captured line of every field and in random lines, so
    that each field keeps 205 good lines: above 4/5 of the field, below MIN_GOOD_LINES_PF = 210 (pcm16x0datastitcher.h:135) --
    the trim must still go by the levels, not by the CRCs."""
    rng = np.random.RandomState(seed)
    o = luma.copy()
    h = luma.shape[1]
    for f in range(luma.shape[0]):
        for fld in range(2):
            rows = np.arange(fld, h, 2)
            pick = np.concatenate([rows[[0, -1]], rng.choice(rows[1:-1], per_field - 2, replace=False)])
            for r in pick:
                for x in (100, 340, 580):
                    o[f, r, x:x + 10] = 255 - o[f, r, x:x + 10]
    return o


def alignment_cases():
    """Tapes for the padding search: configs 3 / 3B, noise, damage, and captures shifted vertically (top padding 5 -> 7, fields
    cut at the head when the picture starts inside the second interleave block)."""
    c = dict(stitch_cases())
    base = synth.make_pcm16x0(3, seed=8)["luma"]
    for k in (2, 6, -4, 40, -30):
        c[f"shift{k}"] = shift_rows(base, k)
    c["shift6_variantB"] = variant_b(shift_rows(base, 6))
    c["edges_205good"] = edge_damage(base)
    return c


@pytest.mark.parametrize("name", sorted(alignment_cases()))
def test_own_alignment_equals_reference_pipeline(name):
    """sdv_pcm16x0_frames_to_samples_auto's logic (trySIPadding x 35 paddings per field, findSIPadding with its padding history,
    findSIDataAlignment, seam masking decided by the search itself) on the host build: every frame of the reference's
    PCMSamplePair stream, no tolerance for 'either variant'."""
    luma = alignment_cases()[name]
    rec, _, _ = util.emu_x0_v2d(luma, 2, True)
    n = luma.shape[0]
    for bff, p_corr in ((False, True), (True, True), (False, False)):
        ref = ref_pairs(luma, bff, p_corr)
        smp, fl, al = util.emu_x0_stitch_auto(rec, n, luma.shape[1], bff, p_corr=p_corr)
        assert not pairs_mismatch(ref, smp, fl), (name, bff, p_corr, pairs_mismatch(ref, smp, fl), al)
    if name == "shift-30":
        assert (al["cut_lines"] > 0).all() and (al["top_padding"] == 0).all()
    if name == "shift-4":
        assert (al["top_padding"] == 7).all()


def ei_cases():
    """EI-format tapes (one interleave unit per frame): clean, variant B, noise, heavy damage, vertically shifted captures (the
    padding between the fields grows or shrinks, fields lose their head), control bits absent or all active, a blanked frame
    and a blanked band (BROKE / NO_PAD results, the fall-back by control bits alone, the padding history re-used)."""
    base = synth.make_pcm16x0(4, ei=True, ctrl_lines=(1, 2))["luma"]
    c = {"clean": base, "variantB": variant_b(base),
         "noise": synth.damage_stc007(base, seed=202, jitter=False, blur=False, sigma=25., dropout_frac=0.05),
         "damaged": synth.damage_stc007(base, seed=102)}
    for k in (3, -7, 50, -60, 100):
        c[f"shift{k}"] = shift_rows(base, k)
    c["no_ctrl_shift12"] = shift_rows(synth.make_pcm16x0(4, seed=21, ei=True, ctrl_lines=())["luma"], 12)
    c["all_ctrl"] = synth.make_pcm16x0(4, seed=22, ei=True, ctrl_lines=(0, 1, 2, 3))["luma"]
    gap = synth.make_pcm16x0(4, seed=23, ei=True, ctrl_lines=(2,))["luma"].copy()
    gap[1] = 16
    gap[2, 100:330] = 16
    c["blanked_shift-20"] = shift_rows(gap, -20)
    c["variantB_heavy_shift100"] = shift_rows(variant_b(base, seed=5, frac=0.5), 100)
    c["edges_205good"] = edge_damage(base)
    # long stretches of digital silence: DS_RET_SILENCE (no padding, seams not masked), silent frames in the history
    c["half_silent"] = synth.make_pcm16x0(4, seed=5, ei=True, ctrl_lines=(1, 2), silent_frames=((1, 0, 900), (2, 600, 1470)))["luma"]
    c["silent_variantB_shift12"] = shift_rows(variant_b(synth.make_pcm16x0(
        4, seed=5, ei=True, ctrl_lines=(1, 2), silent_frames=((0, 100, 1000), (1, 0, 1200), (3, 300, 1300)))["luma"], seed=3, frac=0.2), 12)
    c["silent_frame"] = synth.make_pcm16x0(4, seed=6, ei=True, ctrl_lines=(1, 2), silent_frames=(1, 2))["luma"]
    return c


CPU_EI_CASES = ("clean", "variantB", "shift-60", "shift100", "no_ctrl_shift12", "blanked_shift-20", "edges_205good", "half_silent")


def _ei_check(name, luma, rec, stitch):
    n = luma.shape[0]
    decisions = set()
    for bff, p_corr in ((False, True), (True, True), (False, False)):
        ref = ref_pairs(luma, bff, p_corr, ei=True)
        smp, fl, al = stitch(rec, n, luma.shape[1], bff, p_corr)
        assert ref["rows"] == len(smp), (name, bff, p_corr, ref["rows"])
        assert not pairs_mismatch(ref, smp, fl), (name, bff, p_corr, pairs_mismatch(ref, smp, fl), al)
        decisions |= {(int(a["result"][0]), int(a["mask_seams"])) for a in al}
    return decisions


@pytest.mark.parametrize("name", CPU_EI_CASES)
def test_ei_stitching_equals_reference_pipeline(name):
    """The EI stitcher (tryEIPadding x 81 paddings per frame, findEIFrameStitching's decisions with the padding history,
    conditionEIFramePadding / findEIDataAlignment, data blocks from sub-lines b, b+490, b+980) on the host build: every
    frame of the reference's PCMSamplePair stream with setFormat(FORMAT_EI)."""
    luma = ei_cases()[name]
    rec, _, _ = util.emu_x0_v2d(luma, 2, True)
    d = _ei_check(name, luma, rec, lambda r, n, h, bff, p: util.emu_x0_stitch_auto(r, n, h, bff, p_corr=p, ei=True))
    if name == "clean":
        assert d == {(4, 0), (3, 1)}            # DS_RET_OK with P correction; no padding search (masked seams) without it
    if name == "blanked_shift-20":
        assert (3, 1) in d and (4, 0) in d
    if name == "half_silent":
        assert (1, 0) in d                      # DS_RET_SILENCE: the seams stay unmasked


def test_ei_stitching_against_golden():
    """The same against the committed fixture (line records of the reference + its sample stream): runs without oracle/_ref."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "pcm16x0_ei_stitch.npz"))
    for name in ("variantB", "shift-60"):
        rec = g[name + "_rec"].view(util.LINE_REC).reshape(-1)
        n = int(g[name + "_frames"])
        for i, (bff, p_corr) in enumerate(((False, True), (True, True), (False, False))):
            smp, fl, _ = util.emu_x0_stitch_auto(rec, n, 480, bff, p_corr=p_corr, ei=True)
            assert np.array_equal(g[f"{name}_smp{i}"], smp) and np.array_equal(g[f"{name}_fl{i}"], fl), (name, bff, p_corr)


def test_ei_round_trip_on_host():
    """Every source sample pair of the synthetic EI tape comes back (the 2 x 15 uncaptured sub-lines per frame through P)."""
    t = synth.make_pcm16x0(2, ei=True, ctrl_lines=(1, 2))
    rec, _, _ = util.emu_x0_v2d(t["luma"], 2, True)
    smp, fl, al = util.emu_x0_stitch_auto(rec, 2, 480, ei=True)
    src = t["pairs"].view(np.int16)[:2 * 2 * 735]
    assert np.array_equal(smp.reshape(-1, 2), src)
    assert ((fl & 3) == 3).all()
    assert (al["result"][:, 0] == 4).all() and (al["result"][:, 1] == 5).all() and (al["mask_seams"] == 0).all()


def test_config3_round_trip_on_host():
    """Every source sample pair of the synthetic SI tape comes back (the 15 uncaptured sub-lines per field through P)."""
    t = synth.make_pcm16x0(2)
    rec, _, _ = util.emu_x0_v2d(t["luma"], 2, True)
    smp, fl = util.emu_x0_stitch(rec, 2, 480)
    src = t["pairs"].view(np.int16)[:2 * 2 * 735]
    assert np.array_equal(smp.reshape(-1, 2), src)
    assert ((fl & 3) == 3).all()


# ---- control-bit decisions per frame (collectCtrlBitStats / getProbable*): sample rate and emphasis of the reference's pairs
def ref_frame_info(luma, bff=False):
    cfg = R.StitchCfg()
    cfg.field_order = 2 if bff else 1
    cfg.pcm16x0_format = 1
    cfg.p_corr = 1
    pairs, _, _ = R.pipeline_run(R.TYPE_PCM16X0, 2, luma, cfg, taps=False)
    a = pairs[pairs["service_type"] == 0].reshape(luma.shape[0], 1470)
    assert (a["sample_rate"] == a["sample_rate"][:, :1]).all() and (a["emphasis"] == a["emphasis"][:, :1]).all()
    return np.stack([a["sample_rate"][:, 0], a["emphasis"][:, 0].astype(np.uint16)], axis=1)


def info_cases():
    out = {"44k1": synth.make_pcm16x0(3, seed=1)["luma"],
           "44k056": synth.make_pcm16x0(3, seed=2, ctrl_lines=())["luma"],
           "emph_code": synth.make_pcm16x0(3, seed=3, ctrl_lines=(0, 1, 3))["luma"]}
    l = synth.make_pcm16x0(8, seed=5, ctrl_lines=(0, 1))["luma"].copy()
    l[3:6] = 16                              # nothing to vote with: the history decides (with the reference's inverted sense)
    out["blank_mid"] = l
    l = synth.make_pcm16x0(5, seed=6, ctrl_lines=(0, 1))["luma"].copy()
    l[:2] = 16                               # empty history
    out["blank_start"] = l
    out["noisy"] = synth.damage_stc007(synth.make_pcm16x0(4, seed=7, ctrl_lines=(1, 3))["luma"], seed=9, sigma=30., dropout_frac=0.3,
                                       jitter=False, blur=False)
    return out


GOLD_INFO = os.path.join(os.path.dirname(__file__), "golden", "pcm16x0_frame_info.npz")


def test_frame_info_against_golden():
    g = np.load(GOLD_INFO)
    for name, luma in info_cases().items():
        rec, _, _ = util.emu_x0_v2d(luma, 2, True)
        _, _, info = util.emu_x0_stitch_info(rec, luma.shape[0], luma.shape[1])
        got = np.stack([info["sample_rate"], info["emphasis"].astype(np.uint16)], axis=1)
        assert np.array_equal(got, g[name]), name
    assert (g["blank_mid"][:, 1] == [1, 1, 1, 0, 0, 0, 1, 1]).all()        # the fall-back's sense of "emphasis" is the voted one inverted


def test_frame_info_against_reference_live():
    """The reference's decisions on these tapes: its live run where the reference build is present, else the ones it wrote to
    tests/golden/pcm16x0_frame_info.npz."""
    g = np.load(GOLD_INFO)
    for name in ("emph_code", "blank_start"):
        luma = info_cases()[name]
        rec, _, _ = util.emu_x0_v2d(luma, 2, True)
        _, _, info = util.emu_x0_stitch_info(rec, luma.shape[0], luma.shape[1])
        got = np.stack([info["sample_rate"], info["emphasis"].astype(np.uint16)], axis=1)
        assert np.array_equal(got, ref_frame_info(luma) if R.available() else g[name]), name
