"""GPU parity of sdv_stc007_stitch_frames (through the C ABI) with the UNMODIFIED reference pipeline: the product's
PCMSamplePair stream (l, r, three flags per sample) and its data blocks against those stored for VideoToDigital +
STC007DataStitcher on the same tapes (tests/golden/reference_streams.json; provenance in make_golden.streams_golden).  Needs a GPU."""
import os

import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC, BLOCK_REC
from tests import util
from tests.test_stc007_stitch import stitch_cases, reference_stream, stream_mismatch, block_mismatch, GOLD, HEAVY

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators
    assert torch.cuda.is_available()
    return capi.Handle(0), operators, torch


def _product(ctx, luma, std, order, res=1, p=1, q=1, **kw):
    h, ops, torch = ctx
    v2d = ops.VideoToDigital(h)
    recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(order); st.setResolutionPreset(res == 2); st.setPCorrection(bool(p)); st.setQCorrection(bool(q))
    blocks, samples, flags, info = st.doFrameReassembleAuto(recs, luma.shape[0], luma.shape[1], want_blocks=True, video_std=std, **kw)
    torch.cuda.synchronize()
    return ops.records_to_numpy(blocks, BLOCK_REC), samples.cpu().numpy(), flags.cpu().numpy(), info, recs, st


@pytest.mark.parametrize("name", sorted(stitch_cases()))
def test_sample_stream_equals_reference_pipeline(ctx, name):
    luma, std, order, res, p, q = stitch_cases()[name]
    pairs, ref_blocks = reference_stream(luma, std, order, res, p, q)
    blocks, samples, flags, info, _, _ = _product(ctx, luma, std, order, res, p, q)
    assert not stream_mismatch(pairs, samples, flags)
    assert not block_mismatch(ref_blocks, blocks)
    if name == "heavy":
        # the reference's 128-block countdown after a BROKEN block (stc007datastitcher.cpp:6778-6862) is pinned HERE, by the reference's
        # own stream: this tape has BROKEN blocks and no masked seam, so every block marked unsafe lies in such a window
        assert (blocks["flags"] & capi.BF_UNSAFE).any() and (blocks["flags"] & 2).any() and not (info["flags"] & (capi.FA_MASK_INNER | capi.FA_MASK_PREV_OUTER)).any()


CONFIG4_SEEDS = [4567, 4568, 4569, 4570, 4571]


def config4_tape(seed):
    return synth.damage_stc007(synth.make_stc007(24, seed=seed - 4000)["luma"], seed=seed)


def two_shard_tape():
    luma = synth.damage_stc007(synth.make_stc007(12, seed=441)["luma"], seed=442)        # BASELINE config 4 damage
    # BROKEN blocks just ahead of the boundary: lines with a valid CRC and foreign words (a splice) at the end of frame 5,
    # shard 0's last; the 128-block window they open reaches two blocks into shard 1
    luma[5, 561:576:2] = luma[4, 101:116:2]
    return luma


def ntsc16_tape():
    return synth.damage_stc007(synth.make_stc007(6, seed=441, pal=False, f1_16bit=True)["luma"], seed=442, **HEAVY)


def cwd_config4_tape():
    return synth.damage_stc007(synth.make_stc007(24, seed=567)["luma"], seed=4567)


@pytest.mark.parametrize("seed", CONFIG4_SEEDS)
def test_config4_sample_stream(ctx, seed):
    """BASELINE config 4 (damage_stc007 with its default mix) on 24 PAL frames, plain STC-007, PAL / TFF / 14-bit preset."""
    luma = config4_tape(seed)
    pairs, ref_blocks = reference_stream(luma, 1, 1, 1, 1, 1)
    blocks, samples, flags, info, _, _ = _product(ctx, luma, 1, 1)
    assert not stream_mismatch(pairs, samples, flags)
    assert not block_mismatch(ref_blocks, blocks)


def test_golden_stream(ctx):
    g = np.load(GOLD)
    for name in ("heavy", "vertical_jitter_heavy"):
        luma, std, order, res, p, q = stitch_cases()[name]
        blocks, samples, flags, info, recs, _ = _product(ctx, luma, std, order, res, p, q)
        h, ops, torch = ctx
        assert np.array_equal(ops.records_to_numpy(recs, LINE_REC), g[name + "_recs"].view(LINE_REC).reshape(-1))
        got, gf = samples.reshape(-1, 2), flags.reshape(-1, 2)
        assert np.array_equal(got[:, 0], g[name + "_l"]) and np.array_equal(got[:, 1], g[name + "_r"])
        assert np.array_equal(gf[:, 0], g[name + "_fl"] & 7) and np.array_equal(gf[:, 1], g[name + "_fr"] & 7)


def test_equals_host_emulation_incl_frame_info(ctx):
    """Same decisions as the host build of the same code: the per-frame summaries, every block record (unsafe marks incl.)."""
    for name in ("heavy", "blank_and_partial_frames", "swapped_fields_auto"):
        luma, std, order, res, p, q = stitch_cases()[name]
        blocks, samples, flags, info, recs, _ = _product(ctx, luma, std, order, res, p, q)
        h, ops, torch = ctx
        eb, es, ef, einfo = util.emu_stc007_stitch(ops.records_to_numpy(recs, LINE_REC), luma.shape[0], luma.shape[1], video_std=std, field_order=order)
        assert np.array_equal(info, einfo)
        assert np.array_equal(blocks, eb) and np.array_equal(samples, es) and np.array_equal(flags, ef)


def test_batches_continue_the_file(ctx):
    """file_start / file_end: a tape fed in batches (the last frame of a batch passed again at the head of the next, as the
    reference needs the frame behind the one it assembles) gives the stream of the single call."""
    h, ops, torch = ctx
    luma = synth.damage_stc007(synth.make_stc007(9, seed=431)["luma"], seed=432, **HEAVY)
    blocks, samples, flags, info, recs, st = _product(ctx, luma, 1, 1)
    H = luma.shape[1]
    out_s, out_f, out_b, n_info = [], [], [], 0
    cuts = [0, 3, 4, 7, 9]
    for i in range(len(cuts) - 1):
        a, b = cuts[i], cuts[i + 1]
        last = (b == 9)
        hi = b if last else b + 1
        bb, ss, ff, ii = st.doFrameReassembleAuto(recs[a * H:hi * H], hi - a, H, want_blocks=True, video_std=1, file_start=(a == 0), file_end=last)
        torch.cuda.synchronize()
        out_s.append(ss.cpu().numpy()); out_f.append(ff.cpu().numpy()); out_b.append(ops.records_to_numpy(bb, BLOCK_REC))
        assert len(ii) == b - a
        n_info += len(ii)
    assert n_info == 9
    assert np.array_equal(np.concatenate(out_s), samples) and np.array_equal(np.concatenate(out_f), flags)
    assert np.array_equal(np.concatenate(out_b), blocks)


def test_long_clean_tape_and_empty_input(ctx):
    h, ops, torch = ctx
    tape = synth.make_stc007(60, seed=433)
    blocks, samples, flags, info, recs, st = _product(ctx, tape["luma"], 1, 1)
    # the standard layout everywhere: the stream equals the preset-geometry path
    _, s2, f2 = st.doFrameReassemble(recs, 60, 576)
    torch.cuda.synchronize()
    assert np.array_equal(samples, s2.cpu().numpy()) and np.array_equal(flags, f2.cpu().numpy())
    assert (info["inner"] == 6).all() and (info["outer"] == 6).all()
    bb, ss, ff, ii = st.doFrameReassembleAuto(recs[:0], 0, 576, video_std=1)
    assert ss.shape[0] == 80 and len(ii) == 0            # lead-in and tail only: 80 + 112 lines, all empty
    with pytest.raises(capi.SdvError):
        st.doFrameReassembleAuto(recs[:576], 1, 576, video_std=1, file_start=False)     # nothing to continue after a file end


def test_countdown_carries_across_deinterleave_calls(ctx):
    """STC007DataStitcher::broken_countdown is a member: a BROKEN block shortly before the end of one call masks the first
    blocks of the next (sdv_deint_config.countdown_in / sdv_stc007_countdown).  Two calls over the halves of a line array
    equal one call over the whole, for every cut."""
    from tests.test_hostemu import _random_lines
    h, ops, torch = ctx
    lines = _random_lines(4000, seed=91, p_bad=0.03)
    d = ops.STC007Deinterleaver(h)
    d.broken_mask_dur = 128
    dev = torch.from_numpy(lines.view(np.uint8).reshape(-1, 32)).cuda()
    blocks, samples, flags = d.processBlocks(dev)
    torch.cuda.synchronize()
    full_b = ops.records_to_numpy(blocks, BLOCK_REC)
    assert (full_b["flags"] & capi.BF_UNSAFE).any()
    eb, es, ef = util.emu_deint(lines, 0, False, True, True, True, broken_mask_dur=128)
    assert np.array_equal(full_b, eb)
    st = ops.STC007DataStitcher(h)
    tested = 0
    broken = np.nonzero((full_b["flags"] & capi.BF_BROKEN) != 0)[0]
    for cut in [int(broken[len(broken) // 3]) + 40, int(broken[len(broken) // 2]) + 100, int(broken[-1]) + 5, 2000]:
        b1, s1, f1 = d.processBlocks(dev[:cut + 112])
        c = st.countdown()
        b2, s2, f2 = d.processBlocks(dev[cut:], countdown_in=c["countdown_out"])
        torch.cuda.synchronize()
        got = np.concatenate([ops.records_to_numpy(b1, BLOCK_REC), ops.records_to_numpy(b2, BLOCK_REC)])
        assert np.array_equal(got, full_b), cut
        tested += int(c["countdown_out"] > 0)
    assert tested >= 2


def test_two_shards_on_a_damaged_tape_equal_the_reference(ctx):
    """Frame-sharded decode as bench.py does it at N = 2 -- two handles, each shard's chain starting empty, the 112-line halo
    from the next shard, the broken-block countdown handed on (sharding.carry_countdowns' rule, here without the process
    group) -- against the reference pipeline's PCMSamplePair stream of the UNSHARDED damaged tape."""
    import torch
    from sdvpcmdecoder_b200 import operators as ops, sharding
    luma = two_shard_tape()
    pairs, ref_blocks = reference_stream(luma, 1, 1, 1, 1, 1)
    H, world = luma.shape[1], 2
    out_s, out_f, states, handles, stitchers, recs_all, halos = [], [], [], [], [], [], []
    for rank in range(world):
        a, b = sharding.frame_range(luma.shape[0], rank, world)
        h = capi.Handle(0)
        recs = ops.VideoToDigital(h).doBinarize(torch.from_numpy(np.ascontiguousarray(luma[a:b])).cuda())
        handles.append(h); recs_all.append(recs)
    for rank in range(world):
        a, b = sharding.frame_range(luma.shape[0], rank, world)
        st = ops.STC007DataStitcher(handles[rank])
        st.lead_in = sharding.shard_lead_in(rank)
        halo = recs_all[rank + 1][:sharding.HALO_LINES].clone() if rank < world - 1 else None
        _, s, f = st.doFrameReassemble(recs_all[rank], b - a, H, halo=halo)
        stitchers.append((st, b - a, halo)); states.append(st.countdown()); out_s.append(s); out_f.append(f)
    # the hand-off: shard g's true countdown_in is shard g-1's countdown_out
    used = [0] * world
    for _ in range(world + 1):
        want = [0] + [states[g]["countdown_out"] for g in range(world - 1)]
        changed = [g for g in range(world) if want[g] != used[g]]
        if not changed:
            break
        for g in changed:
            st, n, halo = stitchers[g]
            _, out_s[g], out_f[g] = st.doFrameReassemble(recs_all[g], n, H, halo=halo, countdown_in=want[g])
            states[g] = st.countdown()
        used = want
    torch.cuda.synchronize()
    samples = np.concatenate([s.cpu().numpy() for s in out_s])
    flags = np.concatenate([f.cpu().numpy() for f in out_f])
    assert not stream_mismatch(pairs, samples, flags)
    assert states[1]["countdown_in"] > 0, "the tape was meant to carry a countdown into the second shard"


def _product_auto_res(ctx, luma, std=1, order=1, **kw):
    h, ops, torch = ctx
    recs = ops.VideoToDigital(h).doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(order); st.setResolutionPreset(None)
    blocks, samples, flags, info = st.doFrameReassembleAuto(recs, luma.shape[0], luma.shape[1], want_blocks=True, video_std=std, **kw)
    torch.cuda.synchronize()
    return ops.records_to_numpy(blocks, BLOCK_REC), samples.cpu().numpy(), flags.cpu().numpy(), info, recs, st


def test_detected_audio_resolution(ctx):
    """setResolutionPreset(SAMPLE_RES_UNKNOWN): getFieldResolution on the device, detectAudioResolution in the library, the mode of
    every seam and every block from the fields it touches -- against the reference pipeline with the same preset."""
    from tests.test_stc007_stitch import resolution_cases
    for name, luma in sorted(resolution_cases().items()):
        pairs, ref_blocks = reference_stream(luma, 1, 1, 0, 1, 1)
        blocks, samples, flags, info, _, _ = _product_auto_res(ctx, luma)
        assert not stream_mismatch(pairs, samples, flags), name
        assert not block_mismatch(ref_blocks, blocks), name
    # everything detected at once (video standard, field order, resolution) on an NTSC 16-bit tape
    n16 = ntsc16_tape()
    pairs, ref_blocks = reference_stream(n16, 0, 0, 0, 1, 1)
    blocks, samples, flags, info, _, _ = _product_auto_res(ctx, n16, std=0, order=0)
    assert not stream_mismatch(pairs, samples, flags) and not block_mismatch(ref_blocks, blocks)


def test_detected_audio_resolution_in_batches(ctx):
    """The resolution history carries across calls (file_start = 0) like the rest of the stitcher state."""
    from tests.test_stc007_stitch import resolution_cases
    luma = resolution_cases()["blank_frames_16"]
    h, ops, torch = ctx
    recs = ops.VideoToDigital(h).doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(1); st.setResolutionPreset(None)
    H = luma.shape[1]
    _, s_all, f_all, _ = st.doFrameReassembleAuto(recs, luma.shape[0], H)
    s_all, f_all = s_all.cpu().numpy(), f_all.cpu().numpy()
    parts_s, parts_f = [], []
    for a, hi, fs, fe in [(0, 3, True, False), (2, 4, False, True)]:       # frames [0,3) then [2,4): the last frame of a batch comes again
        _, s, f, ii = st.doFrameReassembleAuto(recs[a * H:hi * H], hi - a, H, file_start=fs, file_end=fe)
        parts_s.append(s.cpu().numpy()); parts_f.append(f.cpu().numpy())
    assert np.array_equal(np.concatenate(parts_s), s_all) and np.array_equal(np.concatenate(parts_f), f_all)


def _product_cwd(ctx, luma, std, order, res, p, q, **kw):
    h, ops, torch = ctx
    recs = ops.VideoToDigital(h).doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(order); st.setResolutionPreset({0: None, 1: False, 2: True}[res]); st.setPCorrection(bool(p)); st.setQCorrection(bool(q))
    st.setCWDCorrection(True)
    blocks, samples, flags, info = st.doFrameReassembleAuto(recs, luma.shape[0], luma.shape[1], want_blocks=True, video_std=std, **kw)
    torch.cuda.synchronize()
    return ops.records_to_numpy(blocks, BLOCK_REC), samples.cpu().numpy(), flags.cpu().numpy(), info, recs, st


def test_cwd_sample_stream_equals_reference_pipeline(ctx):
    """Cross-Word Decoding (the reference's default): performCWD over chains of frames on the device + the deinterleaver's CWD
    stage, against the reference pipeline with setCWDCorrection(true)."""
    from tests.test_stc007_stitch import cwd_cases
    for name, (luma, std, order, res, p, q) in sorted(cwd_cases().items()):
        pairs, ref_blocks = reference_stream(luma, std, order, res, p, q, cwd=1)
        blocks, samples, flags, info, recs, st = _product_cwd(ctx, luma, std, order, res, p, q)
        assert not stream_mismatch(pairs, samples, flags), name
        assert not block_mismatch(ref_blocks, blocks), name
        if name in ("dropouts", "heavy"):
            assert (blocks["flags"] & capi.BF_CWD).any(), name
        if name == "clean":
            assert not (blocks["flags"] & capi.BF_CWD).any()


def test_cwd_config4_24_frames(ctx):
    luma = cwd_config4_tape()
    pairs, ref_blocks = reference_stream(luma, 1, 1, 1, 1, 1, cwd=1)
    blocks, samples, flags, info, _, _ = _product_cwd(ctx, luma, 1, 1, 1, 1, 1)
    assert not stream_mismatch(pairs, samples, flags)
    assert not block_mismatch(ref_blocks, blocks)


def test_cwd_in_batches_and_without_block_buffer(ctx):
    """The patched lines a call leaves in the queue carry over to the next call; the caller need not ask for block records."""
    from tests.test_stc007_stitch import cwd_cases
    h, ops, torch = ctx
    luma, std, order, res, p, q = cwd_cases()["heavy"]
    blocks, s_all, f_all, info, recs, st = _product_cwd(ctx, luma, std, order, res, p, q)
    H = luma.shape[1]
    _, s2, f2, _ = st.doFrameReassembleAuto(recs, luma.shape[0], H, want_blocks=False, video_std=std)
    assert np.array_equal(s2.cpu().numpy(), s_all) and np.array_equal(f2.cpu().numpy(), f_all)
    parts_s, parts_f = [], []
    for a, hi, fs, fe in [(0, 2, True, False), (1, 3, False, False), (2, 4, False, True)]:
        _, s, f, ii = st.doFrameReassembleAuto(recs[a * H:hi * H], hi - a, H, video_std=std, file_start=fs, file_end=fe)
        parts_s.append(s.cpu().numpy()); parts_f.append(f.cpu().numpy())
    assert np.array_equal(np.concatenate(parts_s), s_all) and np.array_equal(np.concatenate(parts_f), f_all)
