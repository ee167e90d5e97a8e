"""PCM-1 / PCM-16x0 line decode of a tape fed in batches, on the host build of the device code (tests/hostemu/pcm_chain_cont.cpp):
the chain run batch by batch, each batch continuing from the chain context the one before left (what a decode call with
sdv_bin_config.reserved[3] bit 0 does with the handle's context), gives the records and aux of one pass over the whole tape, byte
for byte."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX
from tests import util
from tests import test_gpu_pcm1_line as p1_tapes
from tests import test_gpu_pcm16x0_line as x0_tapes

P1, X0 = "pcm1", "pcm16x0"
CONT_SRC = os.path.join(util.HERE, "hostemu", "pcm_chain_cont.cpp")
CONT_LIB = os.path.join(os.path.dirname(util.EMU_LIB), "libpcm_chain_cont.so")
_cont = None


def cont_lib():
    """The host build of the PCM chains with a caller-owned context, compiled on first use (as util.build_hostemu does)."""
    global _cont
    if _cont is None:
        csrc = os.path.join(util.ROOT, "sdvpcmdecoder_b200", "csrc")
        deps = [CONT_SRC] + [os.path.join(csrc, f) for f in os.listdir(csrc)]
        if not (os.path.exists(CONT_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(CONT_LIB) for d in deps)):
            os.makedirs(os.path.dirname(CONT_LIB), exist_ok=True)
            subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w", "-o", CONT_LIB, CONT_SRC], check=True)
        _cont = C.CDLL(CONT_LIB)
    return _cont


def ctx_sizes():
    out = (C.c_int * 2)()
    cont_lib().emu_pcm_ctx_sizes(out)
    return {P1: out[0], X0: out[1]}


def host_batches(fmt, luma, mode, dup, cuts):
    """The host chain over luma[0:cuts[0]], luma[cuts[0]:cuts[1]], ...: the first batch opens the file, every later one continues
    from the chain context of the batch before.  -> (records, aux) of all batches, concatenated."""
    luma = np.ascontiguousarray(luma, dtype=np.uint8)
    n, H, W = luma.shape
    per = 3 if fmt == X0 else 1
    fn = cont_lib().emu_x0_v2d_chain_cont if fmt == X0 else cont_lib().emu_p1_v2d_chain_cont
    ctx = np.zeros(ctx_sizes()[fmt], np.uint8)
    recs, auxs = [], []
    for i, (a, b) in enumerate(zip([0] + list(cuts), list(cuts) + [n])):
        part = np.ascontiguousarray(luma[a:b])
        rec = np.zeros((b - a) * H * per, LINE_REC)
        aux = np.zeros((b - a) * H * per, LINE_AUX)
        ps = np.zeros(b - a, util.P1_PRESET)
        fn(mode, int(dup), util._p(part), b - a, H, W, util._p(rec), util._p(aux), util._p(ps), util._p(ctx), int(i > 0))
        recs.append(rec)
        auxs.append(aux)
    return np.concatenate(recs), np.concatenate(auxs)


def host_one_pass(fmt, luma, mode, dup):
    """The same chain over the whole tape in one call (equal to tests/hostemu's emu_p1_v2d_chain / emu_x0_v2d_chain: see
    test_one_pass_equals_hostemu)."""
    return host_batches(fmt, luma, mode, dup, [])


def cut_sets(n, extra=()):
    """Batch boundaries to try on a tape of n frames: 1-frame batches, one cut in the middle, and the given ones."""
    sets = [list(range(1, n)), [n // 2]] + [list(c) for c in extra]
    out = []
    for s in sets:
        s = sorted(set(c for c in s if 0 < c < n))
        if s and s not in out:
            out.append(s)
    return out


def same_bytes(a, b):
    return np.array_equal(a.view(np.uint8), b.view(np.uint8))


def check_batches(fmt, luma, mode, dup, cuts_list):
    one = host_one_pass(fmt, luma, mode, dup)
    for cuts in cuts_list:
        rec, aux = host_batches(fmt, luma, mode, dup, cuts)
        assert same_bytes(rec, one[0]) and same_bytes(aux, one[1]), (fmt, luma.shape, mode, dup, cuts)
    return one


# ---- PCM-1: every tape of the line tests (more than one frame) with every cut set, MODE_INSANE slices
def p1_runs():
    base = synth.make_pcm1(3)["luma"]
    insane = [(base[:, :64], 3, True), (synth.damage_stc007(base, seed=102)[:, :120], 3, True)]       # MODE_INSANE slices
    return [r for r in p1_tapes.line_runs() if r[0].shape[0] > 1] + insane


@pytest.mark.parametrize("i", range(len(p1_runs())))
def test_pcm1_batches_equal_one_pass(i):
    luma, mode, dup = p1_runs()[i]
    check_batches(P1, luma, mode, dup, cut_sets(luma.shape[0]))


def test_pcm1_cuts_after_damage_and_inside_clean_runs():
    """The sparse tape cut right behind each damaged frame (3 and 7), the clean tape inside its run of clean frames; duplicate
    check on and off."""
    for dup in (True, False):
        check_batches(P1, p1_tapes.sparse_tape(), 2, dup, [[4], [8], [4, 8], [3, 4, 7, 8]])
        check_batches(P1, p1_tapes.clean_tape(), 2, dup, [[5], [2, 9]])


def test_pcm1_draft_mode_carries_prescan_ref():
    """DRAFT mode: no prescan, every frame starts from the reference level and the coordinate history the chain carries."""
    for luma, _, _ in p1_tapes.damaged_runs(0)[:3] + [(p1_tapes.sparse_tape(), 0, True)]:
        for dup in (True, False):
            check_batches(P1, luma, 0, dup, cut_sets(luma.shape[0]))


def test_pcm1_continuing_differs_from_reopening():
    """Continuing matters: a batch that opens a new file instead (chain reset, frame 0 with NEW_FILE) gives other records -- so
    the equalities above are not the trivial ones."""
    for luma, mode, cut in ((p1_tapes.sparse_tape(), 2, 4), (p1_tapes.clean_tape(), 0, 6)):
        one = host_one_pass(P1, luma, mode, True)
        reopened, _ = host_one_pass(P1, luma[cut:], mode, True)
        assert not same_bytes(reopened, one[0][cut * luma.shape[1]:]), mode
        rec, aux = host_batches(P1, luma, mode, True, [cut])
        assert same_bytes(rec, one[0]) and same_bytes(aux, one[1]), mode


# ---- PCM-16x0: the same tapes, plus cuts after the damaged frames of the sparse tape (3 and 6) and inside the drift tape's runs
def x0_runs():
    base = synth.make_pcm16x0(2)["luma"]
    insane = [(base[:, :64], 3, True), (synth.damage_stc007(base, seed=102)[:, :64], 3, True)]       # MODE_INSANE slices
    draft = [(x0_tapes.sparse_tape(), 0, dup) for dup in (True, False)]
    return [r for r in x0_tapes.line_runs() if r[0].shape[0] > 1] + insane + draft


@pytest.mark.parametrize("i", range(len(x0_runs())))
def test_pcm16x0_batches_equal_one_pass(i):
    luma, mode, dup = x0_runs()[i]
    check_batches(X0, luma, mode, dup, cut_sets(luma.shape[0], extra=([4], [4, 7], [3], [5, 6]) if luma.shape[0] == 8 else ()))


def test_one_pass_equals_hostemu():
    """The one-pass run of this build is the host build of tests/hostemu, record for record."""
    for fmt, luma in ((P1, p1_tapes.sparse_tape()), (X0, x0_tapes.sparse_tape())):
        rec, aux = host_one_pass(fmt, luma, 2, True)
        ref = (util.emu_x0_v2d if fmt == X0 else util.emu_p1_v2d)(luma, 2, True)
        assert same_bytes(rec, ref[0]) and same_bytes(aux, ref[1]), fmt
