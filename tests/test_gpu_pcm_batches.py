"""PCM-1 / PCM-16x0 tapes fed in batches on the GPU: line decode with sdv_bin_config.reserved[3] (continue the file), the PCM-1
stitcher with file_start on the first batch only, the PCM-16x0 stitchers with continue_file, the host-buffer whole paths -- each
equal to one call over the whole tape -- and the calls a continuation refuses."""
import ctypes as C

import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX
from tests import util
from tests import test_gpu_pcm1_line as p1_tapes
from tests import test_gpu_pcm16x0_line as x0_tapes
from tests.test_gpu_pcm_fuzz import lines_diff
from tests.test_pcm_batches import cut_sets, same_bytes, P1, X0

pytestmark = pytest.mark.gpu
PCM_TYPE = {P1: capi.TYPE_PCM1, X0: capi.TYPE_PCM16X0}
TAPES = {P1: p1_tapes, X0: x0_tapes}
GOLDEN_KIND = {P1: "pcm1_lines", X0: "pcm16x0_lines"}


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators
    assert torch.cuda.is_available()
    return capi.Handle(0), operators, torch


def batches(n, cuts):
    b = [0] + list(cuts) + [n]
    return list(zip(b[:-1], b[1:]))


def decode_batches(ctx, fmt, luma, mode=2, dup=True, cuts=(), cont=True):
    """VideoToDigital.doBinarize over the batches of luma (cuts: batch boundaries); every batch after the first continues the
    file when cont.  -> (records, aux, per-call stats)."""
    h, ops, torch = ctx
    v2d = ops.VideoToDigital(h)
    v2d.setPCMType(PCM_TYPE[fmt])
    v2d.setBinarizationMode(mode)
    v2d.setCheckLineDup(dup)
    recs, auxs, stats = [], [], []
    for i, (a, b) in enumerate(batches(luma.shape[0], cuts)):
        r, x = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma[a:b])).cuda(), want_aux=True, continue_file=cont and i > 0)
        torch.cuda.synchronize()
        recs.append(ops.records_to_numpy(r, LINE_REC))
        auxs.append(ops.records_to_numpy(x, LINE_AUX))
        stats.append(v2d.stats())
    return np.concatenate(recs), np.concatenate(auxs), stats


def decode_pitched_batches(h, fmt, luma, cuts, stride, off, mode=2, dup=True):
    """sdv_bin_decode_frames per batch on a device buffer with rows [stride] apart from byte [off], the padding filled with noise."""
    import torch
    n, H, W = luma.shape
    per = 3 if fmt == X0 else 1
    recs, auxs = [], []
    for i, (a, b) in enumerate(batches(n, cuts)):
        host = np.random.RandomState(i).randint(0, 256, off + (b - a) * H * stride).astype(np.uint8)
        host[off:].reshape((b - a) * H, stride)[:, :W] = luma[a:b].reshape(-1, W)
        buf = torch.from_numpy(host).cuda()
        rec = torch.full(((b - a) * H * per, LINE_REC.itemsize), 0xA5, dtype=torch.uint8, device="cuda")
        aux = torch.full(((b - a) * H * per, LINE_AUX.itemsize), 0x5A, dtype=torch.uint8, device="cuda")
        cfg = capi.BinConfig(pcm_type=PCM_TYPE[fmt], mode=mode, check_line_dup=int(dup))
        cfg.reserved[3] = int(i > 0)
        h.check(capi.lib().sdv_bin_decode_frames(h.ptr, C.byref(cfg), C.c_void_p(buf.data_ptr() + off), b - a, H, W, stride,
                                                 C.c_void_p(rec.data_ptr()), C.c_void_p(aux.data_ptr()),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        recs.append(rec.cpu().numpy().reshape(-1).view(LINE_REC))
        auxs.append(aux.cpu().numpy().reshape(-1).view(LINE_AUX))
    return np.concatenate(recs), np.concatenate(auxs)


def extra_cuts(fmt, n):
    """Cuts right behind the damaged frames of the sparse tapes (PCM-1: 3 and 7, PCM-16x0: 3 and 6) and inside clean runs."""
    return ([4], [8], [4, 8]) if fmt == P1 else ([4], [7], [4, 7], [3], [5, 6])


# ------------------------------------------------------------------------------------------------ line records
@pytest.mark.parametrize("fmt", [P1, X0])
def test_line_records_in_batches_equal_one_call(ctx, fmt):
    """Every tape of the line tests, in 1-frame batches, cut in the middle and behind damaged frames: the concatenated records and
    aux equal one call byte for byte, the reference's stored records and the host build run in one pass."""
    x0 = fmt == X0
    for luma, mode, dup in TAPES[fmt].line_runs():
        n, H = luma.shape[:2]
        one = decode_batches(ctx, fmt, luma, mode, dup)
        bad = util.lines_mismatch(GOLDEN_KIND[fmt], luma, (mode, dup), one[0], one[1], with_part=x0)
        assert not bad, (fmt, luma.shape, mode, dup, bad)
        host = (util.emu_x0_v2d if x0 else util.emu_p1_v2d)(luma, mode, dup)
        assert not lines_diff(fmt, H, one[:2], host[:2]), (fmt, luma.shape, mode, dup, lines_diff(fmt, H, one[:2], host[:2]))
        for cuts in cut_sets(n, extra_cuts(fmt, n) if n in (8, 10) else ()):
            rec, aux, _ = decode_batches(ctx, fmt, luma, mode, dup, cuts)
            assert same_bytes(rec, one[0]) and same_bytes(aux, one[1]), (fmt, luma.shape, mode, dup, cuts, lines_diff(fmt, H, (rec, aux), one[:2]))


@pytest.mark.parametrize("fmt", [P1, X0])
def test_line_records_in_batches_draft_mode(ctx, fmt):
    """DRAFT mode (no prescan: the reference level and coordinates of every frame come from the carried chain)."""
    for luma in (TAPES[fmt].sparse_tape(), TAPES[fmt].clean_tape()):
        for dup in (True, False):
            one = decode_batches(ctx, fmt, luma, 0, dup)
            for cuts in cut_sets(luma.shape[0]):
                rec, aux, _ = decode_batches(ctx, fmt, luma, 0, dup, cuts)
                assert same_bytes(rec, one[0]) and same_bytes(aux, one[1]), (fmt, dup, cuts)


@pytest.mark.parametrize("fmt", [P1, X0])
def test_pitched_luma_in_batches(ctx, fmt):
    """Continuation through sdv_bin_decode_frames with pitched luma (stride W+16, base offset 1) equals the contiguous call."""
    h = ctx[0]
    for luma in (TAPES[fmt].sparse_tape(), TAPES[fmt].clean_tape()):
        one = decode_batches(ctx, fmt, luma)
        for cuts in ([3], [1, 2, 5]):
            rec, aux = decode_pitched_batches(h, fmt, luma, cuts, luma.shape[2] + 16, 1)
            assert same_bytes(rec, one[0]) and same_bytes(aux, one[1]), (fmt, cuts)


@pytest.mark.parametrize("fmt", [P1, X0])
def test_clean_tape_in_batches_stays_on_the_bulk_path(ctx, fmt):
    """On the clean tape every continuing call is served by the bulk pass (every frame skipped, no line through the chain),
    duplicate check on and off; the sparse tape in batches mixes both as one call does."""
    luma = TAPES[fmt].clean_tape()
    n = luma.shape[0]
    for dup in (True, False):
        _, _, one = decode_batches(ctx, fmt, luma, 2, dup)
        assert (one[0]["frames_skipped"] == n and one[0]["lines_chain"] == 0) or (fmt == P1 and not dup), (fmt, dup, one)
        all_bulk = one[0]["frames_skipped"] == n
        for cuts in ([1, 2, 3], [5], list(range(1, n))):
            _, _, stats = decode_batches(ctx, fmt, luma, 2, dup, cuts)
            for (a, b), st in zip(batches(n, cuts), stats):
                assert (not all_bulk) or (st["frames_skipped"] == b - a and st["lines_chain"] == 0), (fmt, dup, cuts, st)
            assert sum(s["frames_skipped"] for s in stats) == one[0]["frames_skipped"], (fmt, dup, cuts, stats, one)
    luma = TAPES[fmt].sparse_tape()
    _, _, one = decode_batches(ctx, fmt, luma)
    _, _, stats = decode_batches(ctx, fmt, luma, cuts=[4])
    print(fmt, "sparse tape, one call:", one[0], "| cut at 4:", stats)
    assert sum(s["frames_skipped"] for s in stats) == one[0]["frames_skipped"]
    assert sum(s["lines_chain"] for s in stats) == one[0]["lines_chain"]


# ------------------------------------------------------------------------------------------------ samples
def test_pcm1_samples_in_batches(ctx):
    """Batched line decode + PCM1DataStitcher with file_start on the first batch only = the single-call pipeline."""
    h, ops, torch = ctx
    for luma in (p1_tapes.clean_tape(), p1_tapes.sparse_tape(), synth.make_pcm1(5, seed=7, header=True)["luma"]):
        n, H = luma.shape[:2]
        rec, _, _ = decode_batches(ctx, P1, luma)
        st = ops.PCM1DataStitcher(h)
        s1, f1 = st.doFrameReassemble(torch.from_numpy(rec.view(np.uint8).reshape(-1, 32).copy()).cuda(), n, H)
        for cuts in cut_sets(n):
            rec_b, _, _ = decode_batches(ctx, P1, luma, cuts=cuts)
            assert same_bytes(rec_b, rec)
            parts = []
            for i, (a, b) in enumerate(batches(n, cuts)):
                r = torch.from_numpy(rec_b[a * H:b * H].view(np.uint8).reshape(-1, 32).copy()).cuda()
                parts.append(st.doFrameReassemble(r, b - a, H, file_start=i == 0))
            torch.cuda.synchronize()
            assert np.array_equal(np.concatenate([p[0].cpu().numpy() for p in parts]), s1.cpu().numpy()), cuts
            assert np.array_equal(np.concatenate([p[1].cpu().numpy() for p in parts]), f1.cpu().numpy()), cuts


def x0_stitch_batches(ctx, rec, n, H, cuts, auto, cont=True, ei=False):
    """The PCM-16x0 stitcher over the batches of the records: _auto (file_start on the first batch, continue_file on the others)
    or the preset geometry with _info.  -> (samples, flags, info, alignment or None)."""
    h, ops, torch = ctx
    st = ops.PCM16X0DataStitcher(h)
    if ei:
        st.setFormat(st.FORMAT_EI)
    out = []
    for i, (a, b) in enumerate(batches(n, cuts)):
        r = torch.from_numpy(rec[a * H * 3:b * H * 3].view(np.uint8).reshape(-1, 32).copy()).cuda()
        if auto:
            s, f, al, info = st.doFrameReassembleAuto(r, b - a, H, want_info=True, file_start=i == 0, continue_file=cont and i > 0)
            info = info.cpu().numpy().reshape(-1).view(capi.PCM16X0_FRAME_INFO)
        else:
            s, f, info = st.doFrameReassemble(r, b - a, H, want_info=True, continue_file=cont and i > 0)
            al = None
        out.append((s.cpu().numpy(), f.cpu().numpy(), info, al))
    cat = [np.concatenate([o[k] for o in out]) for k in range(3)]
    return cat[0], cat[1], cat[2], (np.concatenate([o[3] for o in out]) if auto else None)


def same_stitch(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b) if x is not None)


def test_pcm16x0_samples_in_batches(ctx):
    """Batched decode + _auto(file_start=0, continue_file=1) and the preset-geometry _info with continue_file=1 = one call, in
    samples, flags, info and alignment; the info cases split into batches still give the golden decisions."""
    from tests.test_pcm16x0_stitch import info_cases, GOLD_INFO
    g = np.load(GOLD_INFO)
    tapes = dict(info_cases())
    tapes["clean"] = x0_tapes.clean_tape()
    tapes["sparse"] = x0_tapes.sparse_tape()
    for name, luma in tapes.items():
        n, H = luma.shape[:2]
        rec, _, _ = decode_batches(ctx, X0, luma)
        for auto in (True, False):
            one = x0_stitch_batches(ctx, rec, n, H, [], auto)
            for cuts in cut_sets(n):
                rec_b, _, _ = decode_batches(ctx, X0, luma, cuts=cuts)
                assert same_bytes(rec_b, rec), (name, cuts)
                got = x0_stitch_batches(ctx, rec_b, n, H, cuts, auto)
                assert same_stitch(got, one), (name, auto, cuts)
                if name in g.files and not auto:
                    dec = np.stack([got[2]["sample_rate"], got[2]["emphasis"].astype(np.uint16)], axis=1)
                    assert np.array_equal(dec, g[name]), (name, cuts)


def history_tape():
    """80 frames: 40 voting 44.1 kHz with emphasis, 30 voting 44.056 kHz without, then 10 blank frames that have no vote of
    their own and take the majority of the 64 frames before -- which flips from the first kind to the second at frame 74."""
    a = synth.make_pcm16x0(8, seed=31, ctrl_lines=(0, 1))["luma"]
    b = synth.make_pcm16x0(6, seed=32, ctrl_lines=())["luma"]
    luma = np.concatenate([np.tile(a, (5, 1, 1)), np.tile(b, (5, 1, 1)), np.full((10,) + a.shape[1:], 16, np.uint8)])
    return luma


def test_pcm16x0_control_bit_history_across_calls(ctx):
    """A tape whose later frames have no valid votes: batched without continue_file, their info differs from one call's (empty
    history); with continue_file it equals it, also when the 64-frame window reaches back over several short calls."""
    luma = history_tape()
    n, H = luma.shape[:2]
    rec, _, _ = decode_batches(ctx, X0, luma, cuts=[40, 70])
    for auto in (True, False):
        one = x0_stitch_batches(ctx, rec, n, H, [], auto)
        rates = one[2]["sample_rate"]
        assert (rates[:40] == 44100).all() and (rates[40:70] == 44056).all(), rates
        assert (one[2]["frame_votes"][70:] & 1 == 0).all() and len(set(rates[70:].tolist())) == 2, rates[70:]
        for cuts in ([70], [72], list(range(5, 80, 5)), [69, 70, 71, 74, 75]):
            got = x0_stitch_batches(ctx, rec, n, H, cuts, auto)
            assert same_stitch(got, one), (auto, cuts)
        bad = x0_stitch_batches(ctx, rec, n, H, [70], auto, cont=False)
        assert not np.array_equal(bad[2], one[2]), auto


# ------------------------------------------------------------------------------------------------ host-buffer whole paths
def test_host_whole_paths_in_batches(ctx):
    h, ops, torch = ctx
    luma = p1_tapes.sparse_tape()
    one = ops.decode_tape_host_pcm1(h, luma, want_recs=True)
    parts = [ops.decode_tape_host_pcm1(h, np.ascontiguousarray(luma[a:b]), want_recs=True, continue_file=a > 0)
             for a, b in batches(luma.shape[0], [4, 7])]
    for k in range(3):
        assert same_bytes(np.concatenate([p[k] for p in parts]), one[k]), k
    luma = x0_tapes.sparse_tape()
    one = ops.decode_tape_host_pcm16x0(h, luma, want_recs=True)
    parts = [ops.decode_tape_host_pcm16x0(h, np.ascontiguousarray(luma[a:b]), want_recs=True, continue_file=a > 0)
             for a, b in batches(luma.shape[0], [4, 7])]
    for k in range(3):
        assert same_bytes(np.concatenate([p[k] for p in parts]), one[k]), k


# ------------------------------------------------------------------------------------------------ refused calls
def test_refused_continuations(ctx):
    _, ops, torch = ctx
    h = capi.Handle(0)
    p1 = torch.from_numpy(synth.make_pcm1(2)["luma"]).cuda()
    x0 = torch.from_numpy(synth.make_pcm16x0(2)["luma"]).cuda()
    stc = torch.from_numpy(synth.make_stc007(2)["luma"]).cuda()

    def v2d(t, mode=2, dup=True):
        v = ops.VideoToDigital(h)
        v.setPCMType(t); v.setBinarizationMode(mode); v.setCheckLineDup(dup)
        return v

    def refused(fn):
        with pytest.raises(capi.SdvError) as e:
            fn()
        assert e.value.code == capi.SDV_ERR_ARG, e.value

    refused(lambda: v2d(capi.TYPE_PCM1).doBinarize(p1, continue_file=True))             # fresh handle
    v2d(capi.TYPE_PCM1).doBinarize(p1)
    v2d(capi.TYPE_PCM1).doBinarize(p1[:0], continue_file=True)                          # no frames: nothing changes
    v2d(capi.TYPE_PCM1).doBinarize(p1, continue_file=True)
    refused(lambda: v2d(capi.TYPE_PCM16X0).doBinarize(p1, continue_file=True))          # other PCM type
    refused(lambda: v2d(capi.TYPE_PCM1).doBinarize(p1[:, :400].contiguous(), continue_file=True))    # other H
    refused(lambda: v2d(capi.TYPE_PCM1).doBinarize(p1[:, :, :700].contiguous(), continue_file=True))    # other W
    refused(lambda: v2d(capi.TYPE_PCM1, mode=1).doBinarize(p1, continue_file=True))     # other mode
    refused(lambda: v2d(capi.TYPE_PCM1, dup=False).doBinarize(p1, continue_file=True))  # other duplicate check
    seg = v2d(capi.TYPE_PCM1)
    seg.chain_segments = 2
    refused(lambda: seg.doBinarize(p1, continue_file=True))                             # not with chain segments
    v2d(capi.TYPE_PCM1).doBinarize(p1, continue_file=True)                              # the refusals left the file open
    # an STC-007 call in between does not break the PCM file, a PCM call does not break the STC-007 one
    v2d(capi.TYPE_STC007).doBinarize(stc)
    v2d(capi.TYPE_PCM1).doBinarize(p1, continue_file=True)
    v2d(capi.TYPE_STC007).doBinarize(stc, continue_file=True)
    # fine settings
    v = v2d(capi.TYPE_PCM1)
    v.setFineSettings(min_valid_crcs=4)
    refused(lambda: v.doBinarize(p1, continue_file=True))
    v.setDefaultFineSettings()
    v.doBinarize(p1)
    v.doBinarize(p1, continue_file=True)
    # the stitcher's control-bit history
    recs = v2d(capi.TYPE_PCM16X0).doBinarize(x0)
    st = ops.PCM16X0DataStitcher(capi.Handle(0))
    refused(lambda: st.doFrameReassemble(recs, 2, 480, continue_file=True))             # no earlier stitch call
    refused(lambda: st.doFrameReassembleAuto(recs, 2, 480, file_start=False, continue_file=True))
    st.doFrameReassemble(recs, 2, 480)
    st.doFrameReassemble(recs, 2, 480, continue_file=True)
    st.doFrameReassembleAuto(recs, 2, 480, file_start=False, continue_file=True)
    refused(lambda: st.doFrameReassembleAuto(recs, 2, 480, file_start=True, continue_file=True))    # file_start with continue_file
    st.doFrameReassembleAuto(recs, 2, 480)
    st.setFormat(st.FORMAT_EI)                                                           # across an SI / EI change
    refused(lambda: st.doFrameReassembleAuto(recs, 2, 480, file_start=False, continue_file=True))
    refused(lambda: st.doFrameReassemble(recs, 2, 480, continue_file=True))
    st.doFrameReassemble(recs, 2, 480)
    st.doFrameReassemble(recs, 2, 480, continue_file=True)
