"""The deinterleave pass of the standard setting (14-bit, forced check, P+Q) with samples and flags only -- where
stc007_deint_kernel finishes two adjacent blocks per lane (deint_pair_std14) -- against the host build of the one-block path
(deint_block_std14 through tests/hostemu, emu_deint_carry) on the same line records: samples, flags and the countdown left
over, byte for byte.  Damaged config-4 tapes (BROKEN blocks, countdown windows across tiles), odd block counts, the assembled
stream of a tape with and without a halo, PAL and NTSC, CRC ignored.  Run on the B200 box."""
import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC
from tests import util
from tests.test_hostemu import _random_lines, _lines_with_data_flags

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators
    assert torch.cuda.is_available()
    return capi.Handle(0), operators, torch


def _records(ctx, luma):
    h, ops, torch = ctx
    v2d = ops.VideoToDigital(h)
    recs = v2d.doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())
    torch.cuda.synchronize()
    return recs


def _config4_records(ctx, frames, seed, pal=True):
    luma = synth.damage_stc007(synth.make_stc007(frames, seed=seed - 4000, pal=pal)["luma"], seed=seed)
    return _records(ctx, luma), luma.shape[1]


def _plain(ctx, lines, countdown_in=0, ignore_crc=False):
    """The pass over a plain line array (sdv_deint_stc007), no block records: samples, flags, countdown out."""
    h, ops, torch = ctx
    d = ops.STC007Deinterleaver(h)
    d.broken_mask_dur = 128
    if ignore_crc:
        d.setIgnoreCRC(True)
    _, s, f = d.processBlocks(torch.from_numpy(lines.view(np.uint8).reshape(-1, 32)).cuda(), want_blocks=False, countdown_in=countdown_in)
    c = ops.STC007DataStitcher(h).countdown()
    return s.cpu().numpy(), f.cpu().numpy(), c["countdown_out"]


def _host(lines, countdown_in=0, ignore_crc=False):
    _, s, f, c = util.emu_deint_carry(lines, countdown_in=countdown_in, ignore_crc=ignore_crc, broken_mask_dur=128)
    return s, f, c


def _assert_same(got, want, what):
    (gs, gf, gc), (es, ef, ec) = got, want
    assert gs.shape == es.shape, what
    bad = np.nonzero((gs != es).any(axis=1) | (gf != ef).any(axis=1))[0]
    assert len(bad) == 0, (what, len(bad), bad[:8])
    assert gc == ec, (what, gc, ec)


@pytest.mark.parametrize("seed", [4101, 4102])
def test_damaged_records_plain_array(ctx, seed):
    """Config-4 damage (BROKEN blocks that open windows across tiles), whole records and an odd number of blocks, with and
    without a countdown carried in."""
    recs, _ = _config4_records(ctx, 6, seed)
    lines = ctx[1].records_to_numpy(recs, LINE_REC)
    e = _host(lines)
    assert (e[1][:, 0] & capi.SF_BLOCK_OK).mean() < 0.999, "the tape was meant to carry damage"
    _assert_same(_plain(ctx, lines), e, "whole")
    odd = lines[:len(lines) - 113]                     # n_blocks odd: the last lane holds one block
    assert (len(odd) - 112) % 2 == 1
    _assert_same(_plain(ctx, odd, countdown_in=77), _host(odd, countdown_in=77), "odd, countdown in")


def test_random_lines_with_broken_blocks(ctx):
    """Random damage with lying lines (BROKEN, not silent): the candidate bits and windows, several block counts."""
    lines = _random_lines(9001, seed=5, p_bad=0.03)
    e = _host(lines)
    assert (e[1][:, 0] == 0).any()
    _assert_same(_plain(ctx, lines), e, "9001")
    for n in (113, 114, 241, 1129, 4096 + 112 + 1):
        sub = np.ascontiguousarray(lines[:n])
        _assert_same(_plain(ctx, sub, countdown_in=n % 129), _host(sub, countdown_in=n % 129), n)


def test_ignore_crc(ctx):
    lines, _ = _lines_with_data_flags(3001, 23)
    _assert_same(_plain(ctx, lines, ignore_crc=True), _host(lines, ignore_crc=True), "ignore_crc")


def _assembled(lines_rec, n_frames, H, lpf, halo=None, lead_in=80):
    """The stream sdv_stc007_shard_to_samples deinterleaves, written out: lead-in, per field H/2 decoded lines and lpf - H/2
    empty ones, then the halo (at most 112 lines) or nothing."""
    hf = H // 2
    nb = lead_in + n_frames * 2 * lpf
    out = np.zeros(nb + 112, LINE_REC)
    for fld in range(2 * n_frames):
        a = lead_in + fld * lpf
        out[a:a + hf] = lines_rec[(fld >> 1) * H + (fld & 1) * hf:(fld >> 1) * H + (fld & 1) * hf + hf]
    if halo is not None:
        m = min(112, hf)
        out[nb:nb + m] = halo[:m]
    return out


@pytest.mark.parametrize("pal", [True, False])
@pytest.mark.parametrize("with_halo", [False, True])
def test_assembled_tape(ctx, pal, with_halo):
    """The geometry path (the bench's): a damaged tape's records as fields with the lead-in and the uncaptured lines, with the
    next shard's first 112 records as a halo or without; also equal to the pass with block records (one block per lane)."""
    h, ops, torch = ctx
    recs, H = _config4_records(ctx, 5, 4200 + 2 * int(pal) + int(with_halo), pal=pal)
    n_frames = recs.shape[0] // H
    halo_recs, _ = _config4_records(ctx, 1, 4300, pal=pal) if with_halo else (None, None)
    st = ops.STC007DataStitcher(h)
    st.setVideoStandard(ops.VID_PAL if pal else ops.VID_NTSC)
    lpf = ops.LINES_PER_FIELD[st.video_std]
    halo = halo_recs[:112].contiguous() if with_halo else None
    _, s, f = st.doFrameReassemble(recs, n_frames, H, halo=halo, countdown_in=5)
    c = st.countdown()["countdown_out"]
    got = (s.cpu().numpy(), f.cpu().numpy(), c)
    lines = _assembled(ops.records_to_numpy(recs, LINE_REC), n_frames, H, lpf,
                       ops.records_to_numpy(halo, LINE_REC) if with_halo else None)
    _assert_same(got, _host(lines, countdown_in=5), "assembled")
    _, s2, f2 = st.doFrameReassemble(recs, n_frames, H, halo=halo, countdown_in=5, want_blocks=True)
    assert np.array_equal(s2.cpu().numpy(), got[0]) and np.array_equal(f2.cpu().numpy(), got[1])


def test_clean_tape_takes_the_pair_path_everywhere(ctx):
    """The clean tape (one untrusted word in a sixth of the blocks): every interior block valid and equal to the host build."""
    h, ops, torch = ctx
    tape = synth.make_stc007(8)
    recs = _records(ctx, tape["luma"])
    st = ops.STC007DataStitcher(h)
    _, s, f = st.doFrameReassemble(recs, 8, 576)
    got = (s.cpu().numpy(), f.cpu().numpy(), st.countdown()["countdown_out"])
    lines = _assembled(ops.records_to_numpy(recs, LINE_REC), 8, 576, 294)
    _assert_same(got, _host(lines), "clean")
    ok = (got[1] & capi.SF_BLOCK_OK).all(axis=1)
    assert ok[300:-300].all()
