"""STC007DataStitcher with its own vertical alignment (sdv_stc007_stitch_frames): frame trim, the field-stitching decision
chain, frame assembly, seam masking and the broken-block countdown.

CPU part: the library's host decision chain (csrc/stc007_stitch_host.h) and the SDV_HD device code (csrc/stc007_stitch.cuh),
built as host code by tests/hostemu and fed with the oracle's line records, against the PCMSamplePair streams and data blocks
stored for these tapes in tests/golden/reference_streams.json -- damaged far beyond BASELINE config 4, shifted vertically, with
blank and partial frames, with field order / video standard preset or detected.  The stored streams stand for the reference
pipeline's (VideoToDigital + STC007DataStitcher) output; tests/golden/make_golden.py streams_golden() says where they come from
and what ties them to the reference.  GPU part (tests/test_gpu_stc007_stitch.py): the CUDA path through the C ABI against the
same streams.
"""
import os

import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from tests import util

HEAVY = dict(sigma=20.0, dropout_frac=0.1, marker_kill_frac=0.05)
GOLD = os.path.join(os.path.dirname(__file__), "golden", "stc007_stitch.npz")


def shift_rows(luma, k):
    """Move the picture k rows down (k < 0: up); rows that come into view are black."""
    o = np.full_like(luma, 16)
    if k > 0:
        o[:, k:] = luma[:, :-k]
    elif k < 0:
        o[:, :k] = luma[:, -k:]
    else:
        o[:] = luma
    return o


def stitch_cases():
    """name -> (luma, video_std, field_order, resolution preset (1 = 14 bit, 2 = 16 bit), p, q)."""
    c = {}
    t = synth.make_stc007(6, seed=401)
    c["config4"] = (synth.damage_stc007(t["luma"], seed=4567), 1, 1, 1, 1, 1)
    c["heavy"] = (synth.damage_stc007(t["luma"], seed=402, **HEAVY), 1, 1, 1, 1, 1)
    c["heavy_auto"] = (synth.damage_stc007(t["luma"], seed=403, **HEAVY), 0, 0, 1, 1, 1)
    c["noise25"] = (synth.damage_stc007(t["luma"], seed=404, sigma=25.0), 1, 1, 1, 1, 1)
    n = synth.make_stc007(6, seed=405, pal=False)
    c["ntsc_heavy_auto"] = (synth.damage_stc007(n["luma"], seed=406, **HEAVY), 0, 0, 1, 1, 1)
    jit = t["luma"].copy()
    for f, k in enumerate([0, 2, 2, 0, -2, 4]):
        jit[f] = shift_rows(t["luma"][f:f + 1], k)[0]
    c["vertical_jitter"] = (jit, 1, 1, 1, 1, 1)
    c["vertical_jitter_heavy"] = (synth.damage_stc007(jit, seed=407, **HEAVY), 1, 1, 1, 1, 1)
    c["shift3_heavy_auto"] = (synth.damage_stc007(shift_rows(t["luma"], 3), seed=408, **HEAVY), 0, 0, 1, 1, 1)
    sw = t["luma"].copy()
    sw[:, 0::2], sw[:, 1::2] = t["luma"][:, 1::2], t["luma"][:, 0::2]
    c["swapped_fields_auto"] = (sw, 1, 0, 1, 1, 1)
    c["wrong_order_preset"] = (synth.damage_stc007(t["luma"], seed=409, **HEAVY), 1, 2, 1, 1, 1)
    bl = synth.damage_stc007(t["luma"], seed=410, **HEAVY)
    bl[2] = 16
    bl[3, :200] = 16
    bl[4, 1::2] = 16
    c["blank_and_partial_frames"] = (bl, 0, 0, 1, 1, 1)
    c["p_only"] = (synth.damage_stc007(t["luma"], seed=411, **HEAVY), 1, 1, 1, 1, 0)
    c["res16"] = (synth.damage_stc007(t["luma"], seed=412, **HEAVY), 1, 1, 2, 1, 1)
    return c


BLOCKS_PER_FRAME = 588          # 2 x 294 assembled lines (PAL), one data block each: the unit of the stored digests


def reference_stream(luma, std, order, res, p, q, cwd=0):
    """The stored PCMSamplePair stream (l, r, flags & 7) and data blocks of VideoToDigital + STC007DataStitcher on this tape with
    these settings (tests/golden/reference_streams.json; provenance in make_golden.streams_golden)."""
    g = util.golden_stream("stc007", luma, (std, order, res, p, q, cwd))
    return g["pairs"], g["blocks"]


def pair_arrays(samples, flags):
    return samples.reshape(-1, 2), flags.reshape(-1, 2)


def block_arrays(blocks):
    return [blocks[n] for n in ("words", "line_crc", "word_valid", "audio_state", "resolution")] + [blocks["flags"] & 0x1F]


def stream_mismatch(pairs, samples, flags):
    return util.stream_mismatch_digests(pairs, pair_arrays(samples, flags))


def block_mismatch(ref_blocks, blocks):
    return util.stream_mismatch_digests(ref_blocks, block_arrays(blocks))


def oracle_lines(luma):
    """Line records of the oracle's VideoToDigital (equal to the reference's: tests/test_oracle.py) for the host-built stitcher."""
    from oracle import oraclebind as O
    return util.lines_from_oracle(O.v2d_stc007(capi.MODE_NORMAL, luma, True))


@pytest.mark.parametrize("name", sorted(stitch_cases()))
def test_host_chain_and_device_logic_against_reference_pipeline(name):
    luma, std, order, res, p, q = stitch_cases()[name]
    pairs, ref_blocks = reference_stream(luma, std, order, res, p, q)
    recs = oracle_lines(luma)
    blocks, samples, flags, info = util.emu_stc007_stitch(recs, luma.shape[0], luma.shape[1], video_std=std, field_order=order, res16=(res == 2),
                                                          p_corr=bool(p), q_corr=bool(q))
    assert not stream_mismatch(pairs, samples, flags)
    assert not block_mismatch(ref_blocks, blocks)
    if name in ("heavy", "vertical_jitter_heavy", "blank_and_partial_frames"):
        # the cases are there to leave the standard layout: make sure they do
        assert (info["flags"] & (capi.FA_MASK_INNER | capi.FA_MASK_PREV_OUTER)).any() or (info["inner"] != info["inner"][0]).any()


def test_golden_stream():
    """tests/golden/stc007_stitch.npz (the reference's PCMSamplePair stream, written by tests/golden/make_golden.py) against the
    host build of the stitcher fed with the golden line records -- runs where oracle/_ref does not exist."""
    g = np.load(GOLD)
    for name in ("heavy", "vertical_jitter_heavy"):
        recs = g[name + "_recs"].view(capi.LINE_REC).reshape(-1)
        n_frames, height = int(g[name + "_shape"][0]), int(g[name + "_shape"][1])
        _, samples, flags, _ = util.emu_stc007_stitch(recs, n_frames, height)
        got, gf = samples.reshape(-1, 2), flags.reshape(-1, 2)
        assert np.array_equal(got[:, 0], g[name + "_l"]) and np.array_equal(got[:, 1], g[name + "_r"])
        assert np.array_equal(gf[:, 0], g[name + "_fl"] & 7) and np.array_equal(gf[:, 1], g[name + "_fr"] & 7)


def test_padding_decision_table():
    """pad_decide (findPadding's ranking and acceptance rules) is reached through emu_stc007_stitch; here its edge: a clean
    tape keeps the previous frame's paddings without a new sweep, a blank tape reports silence and the standard layout."""
    t = synth.make_stc007(4, seed=420)
    from oracle import oraclebind as O
    recs = util.lines_from_oracle(O.v2d_stc007(2, t["luma"], True))
    _, _, _, info = util.emu_stc007_stitch(recs, 4, 576)
    assert (info["inner"] == 6).all() and (info["outer"] == 6).all() and (info["n1"] == 288).all()
    assert (info["flags"][:-1] & 3 == 3).all()          # the last frame has no frame behind it to stitch to
    blank = np.zeros(4 * 576, capi.LINE_REC)
    _, s, f, info = util.emu_stc007_stitch(blank, 4, 576)
    assert (info["n1"] == 0).all() and (info["inner"] == 294).all() and not s.any() and not (f & 1).any()


def resolution_cases():
    """Tapes for the audio-resolution detection (setResolutionPreset(SAMPLE_RES_UNKNOWN)): name -> luma."""
    c = {}
    t14 = synth.make_stc007(4, seed=431)
    t16 = synth.make_stc007(4, seed=432, f1_16bit=True)
    c["clean14"] = t14["luma"]
    c["clean16"] = t16["luma"]
    c["heavy16"] = synth.damage_stc007(t16["luma"], seed=433, **HEAVY)
    c["config4_16"] = synth.damage_stc007(t16["luma"], seed=4567)
    mix = t14["luma"].copy()
    mix[2:] = t16["luma"][2:]                       # a tape that switches from 14 to 16 bit
    c["switch_14_to_16"] = synth.damage_stc007(mix, seed=434)
    bl = synth.damage_stc007(t16["luma"], seed=435, **HEAVY)
    bl[1] = 16                                      # a blank frame: its fields are "unknown" and take the history's word
    bl[2, 1::2] = 16
    c["blank_frames_16"] = bl
    return c


# (the CPU suite runs a subset of the tapes to stay within minutes; the GPU tests run all of them against the same reference)
CPU_RESOLUTION_CASES = ["clean16", "heavy16", "switch_14_to_16", "blank_frames_16"]
CPU_CWD_CASES = ["config4", "heavy", "dropouts16", "heavy16_auto_res", "p_only", "sparse"]


@pytest.mark.parametrize("name", CPU_RESOLUTION_CASES)
def test_detected_audio_resolution_against_reference_pipeline(name):
    """getFieldResolution + detectAudioResolution + getDataBlockResolution: the resolution is not preset, every block and every
    seam takes the mode of the fields it touches."""
    luma = resolution_cases()[name]
    pairs, ref_blocks = reference_stream(luma, 1, 1, 0, 1, 1)
    recs = oracle_lines(luma)
    blocks, samples, flags, info = util.emu_stc007_stitch(recs, luma.shape[0], luma.shape[1], video_std=1, field_order=1, res16=None)
    assert not stream_mismatch(pairs, samples, flags)
    assert not block_mismatch(ref_blocks, blocks)
    if name == "clean16":
        assert (info["odd_res_mode"] == 3).all() and (blocks["resolution"][200:-200] == 1).all()
    if name == "clean14":
        assert (info["odd_res_mode"] == 0).all()


def cwd_cases():
    """Tapes for Cross-Word Decoding (setCWDCorrection(true), the reference's default): name -> (luma, std, order, res, p, q)."""
    c = {}
    t = synth.make_stc007(4, seed=451)
    c["config4"] = (synth.damage_stc007(t["luma"], seed=4567), 1, 1, 1, 1, 1)
    c["heavy"] = (synth.damage_stc007(t["luma"], seed=452, **HEAVY), 1, 1, 1, 1, 1)
    c["dropouts"] = (synth.damage_stc007(t["luma"], seed=453, sigma=4.0, dropout_frac=0.25, marker_kill_frac=0.0), 1, 1, 1, 1, 1)
    c["heavy_auto"] = (synth.damage_stc007(t["luma"], seed=454, **HEAVY), 0, 0, 1, 1, 1)
    c["p_only"] = (synth.damage_stc007(t["luma"], seed=455, sigma=4.0, dropout_frac=0.2), 1, 1, 1, 1, 0)
    t16 = synth.make_stc007(4, seed=456, f1_16bit=True)
    c["dropouts16"] = (synth.damage_stc007(t16["luma"], seed=457, sigma=4.0, dropout_frac=0.2), 1, 1, 2, 1, 1)
    c["heavy16_auto_res"] = (synth.damage_stc007(t16["luma"], seed=458, **HEAVY), 1, 1, 0, 1, 1)
    sparse = t["luma"].copy()                       # clean frames between damaged ones: separate chains
    sparse[1] = synth.damage_stc007(t["luma"][1:2], seed=459, sigma=4.0, dropout_frac=0.3)[0]
    sparse[3] = synth.damage_stc007(t["luma"][3:4], seed=460, sigma=4.0, dropout_frac=0.3)[0]
    c["sparse"] = (sparse, 1, 1, 1, 1, 1)
    c["clean"] = (t["luma"], 1, 1, 1, 1, 1)
    return c


@pytest.mark.parametrize("name", CPU_CWD_CASES)
def test_cwd_against_reference_pipeline(name):
    """performCWD + the deinterleaver's CWD stage: the PCMSamplePair stream and the data blocks of the reference pipeline with
    setCWDCorrection(true)."""
    luma, std, order, res, p, q = cwd_cases()[name]
    pairs, ref_blocks = reference_stream(luma, std, order, res, p, q, cwd=1)
    recs = oracle_lines(luma)
    blocks, samples, flags, info = util.emu_stc007_stitch(recs, luma.shape[0], luma.shape[1], video_std=std, field_order=order,
                                                          res16={0: None, 1: False, 2: True}[res], p_corr=bool(p), q_corr=bool(q), cwd=True)
    assert not stream_mismatch(pairs, samples, flags)
    assert not block_mismatch(ref_blocks, blocks)
    if name in ("dropouts", "heavy", "dropouts16"):
        # the cases are there for CWD to repair something: the stream must differ from the one without it
        pairs0, _ = reference_stream(luma, std, order, res, p, q, cwd=0)
        assert stream_mismatch(pairs0, samples, flags)
