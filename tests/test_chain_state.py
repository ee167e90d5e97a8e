"""The line-decode chain state as a blob (chain_state.cuh, what sdv_bin_chain_state_save / _load run on the device), on the host
build of the device code (tests/hostemu/chain_state_cont.cpp): every format's chain run in pieces with pack -> unpack into a fresh
context between them gives the records and aux of one pass, byte for byte, and the packed bytes after a prefix do not depend on
how the prefix was cut.  Also sharding.decode_shard's protocol with a stub line decoder: the luma passed along when shards are
shorter than the warm-up, the verify / redo rounds, and the warmup >= 1 rule."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from sdvpcmdecoder_b200 import synth, sharding
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX
from tests import util
from tests import test_gpu_pcm1_line as p1_tapes
from tests import test_gpu_pcm16x0_line as x0_tapes
from tests.test_m2 import m2_tapes

SRC = os.path.join(util.HERE, "hostemu", "chain_state_cont.cpp")
LIB = os.path.join(os.path.dirname(util.EMU_LIB), "libchain_state_cont.so")
STC, M2, P1, X0 = "stc007", "m2", "pcm1", "pcm16x0"
KIND = {STC: 0, M2: 0, P1: 1, X0: 2}
_lib = None


def lib():
    """The host build, compiled on first use (as util.build_hostemu does)."""
    global _lib
    if _lib is None:
        csrc = os.path.join(util.ROOT, "sdvpcmdecoder_b200", "csrc")
        deps = [SRC, os.path.join(util.HERE, "hostemu", "pcm_chain_cont.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc)]
        if not (os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps)):
            os.makedirs(os.path.dirname(LIB), exist_ok=True)
            subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w", "-o", LIB, SRC], check=True)
        _lib = C.CDLL(LIB)
    return _lib


def pack(fmt, ctx):
    blob = np.zeros(lib().emu_chain_blob_bytes(), np.uint8)
    lib().emu_chain_pack(KIND[fmt], util._p(ctx), util._p(blob))
    return blob


def fresh_ctx(fmt, fill=0xA5):
    """A context that has never decoded anything, filled with garbage: what unpacking does not set would show."""
    return np.full(lib().emu_chain_ctx_size(KIND[fmt]), fill, np.uint8)


def unpack(fmt, blob):
    ctx = fresh_ctx(fmt)
    lib().emu_chain_unpack(KIND[fmt], util._p(blob), util._p(ctx))
    return ctx


def run(fmt, luma, mode, dup, cuts, handoff=True):
    """The chain over luma[0:cuts[0]], luma[cuts[0]:cuts[1]], ...: the first piece opens the file, every later one continues --
    from pack -> unpack of the state the piece before left (handoff) or from that context itself.
    -> (records, aux, blob after the last piece)."""
    luma = np.ascontiguousarray(luma, dtype=np.uint8)
    n, H, W = luma.shape
    per = 3 if fmt == X0 else 1
    ctx = fresh_ctx(fmt, 0)
    recs, auxs = [], []
    for i, (a, b) in enumerate(zip([0] + list(cuts), list(cuts) + [n])):
        if i > 0 and handoff:
            ctx = unpack(fmt, pack(fmt, ctx))
        part = np.ascontiguousarray(luma[a:b])
        rec = np.zeros((b - a) * H * per, LINE_REC)
        aux = np.zeros((b - a) * H * per, LINE_AUX)
        if fmt in (STC, M2):
            flags = int(dup) | (2 if fmt == M2 else 0)
            lib().emu_stc_v2d_chain_cont(mode, flags, util._p(part), b - a, H, W, util._p(rec), util._p(aux), util._p(ctx), int(i > 0))
        else:
            fn = lib().emu_x0_v2d_chain_cont if fmt == X0 else lib().emu_p1_v2d_chain_cont
            fn(mode, int(dup), util._p(part), b - a, H, W, util._p(rec), util._p(aux), None, util._p(ctx), int(i > 0))
        recs.append(rec)
        auxs.append(aux)
    return np.concatenate(recs), np.concatenate(auxs), pack(fmt, ctx)


def same(a, b):
    return np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _sparse_stc(n=8):
    luma = synth.make_stc007(n, seed=61)["luma"].copy()
    for f in (2, 5):
        luma[f, 200:203] = synth.damage_stc007(luma[f:f + 1, 200:203].copy(), seed=f, jitter=True)[0]
    return luma


def runs():
    """(format, luma, mode, duplicate check): the line-test tapes, damaged tapes, DRAFT mode and the duplicate check off."""
    dmg = synth.damage_stc007(synth.make_stc007(5, seed=62)["luma"], seed=63)
    out = [(STC, synth.make_stc007(4, seed=60)["luma"], 2, True), (STC, _sparse_stc(), 2, True), (STC, dmg, 2, True),
           (STC, dmg, 0, True), (STC, dmg, 2, False), (STC, synth.make_stc007(4, control_block=True)["luma"], 2, True)]
    out += [(M2, luma, 2, True) for _, luma in sorted(m2_tapes().items())]
    out += [(P1, p1_tapes.clean_tape()[:6], 2, True), (P1, p1_tapes.sparse_tape(), 2, True), (P1, p1_tapes.sparse_tape(), 2, False),
            (P1, p1_tapes.sparse_tape(), 0, True)]
    out += [(P1, luma, mode, dup) for luma, mode, dup in p1_tapes.damaged_runs(2)[:2] if luma.shape[0] > 1]
    out += [(X0, x0_tapes.clean_tape()[:5], 2, True), (X0, x0_tapes.drift_tape(), 2, True), (X0, x0_tapes.sparse_tape(), 2, True),
            (X0, x0_tapes.sparse_tape(), 2, False), (X0, x0_tapes.sparse_tape(), 0, True)]
    out += [(X0, luma, mode, dup) for luma, mode, dup in x0_tapes.damaged_runs(2)[:2] if luma.shape[0] > 1]
    return out


def _cut_sets(n, seed):
    rng = np.random.default_rng(seed)
    sets = [list(range(1, n)), [n // 2], sorted(rng.choice(np.arange(1, n), size=min(2, n - 1), replace=False).tolist())]
    return [s for i, s in enumerate(sets) if s and s not in sets[:i]]


@pytest.mark.parametrize("i", range(len(runs())))
def test_handoff_in_pieces_equals_one_pass(i):
    """Pack -> unpack into a fresh context at every cut: the records and aux of one pass, and the same end state."""
    fmt, luma, mode, dup = runs()[i]
    one = run(fmt, luma, mode, dup, [])
    for cuts in _cut_sets(luma.shape[0], i):
        got = run(fmt, luma, mode, dup, cuts)
        assert same(got[0], one[0]) and same(got[1], one[1]), (fmt, mode, dup, cuts)
        assert np.array_equal(got[2], one[2]), (fmt, mode, dup, cuts)


@pytest.mark.parametrize("i", range(len(runs())))
def test_blob_after_a_prefix_does_not_depend_on_the_cuts(i):
    """The bytes after frames [0, k) are the same for one pass, for pieces continued in place and for pieces handed over; and
    unpack -> pack gives them back."""
    fmt, luma, mode, dup = runs()[i]
    n = luma.shape[0]
    for k in sorted({1, n // 2, n - 1, n} - {0}):
        want = run(fmt, luma[:k], mode, dup, [])[2]
        assert np.array_equal(pack(fmt, unpack(fmt, want)), want)
        for cuts in _cut_sets(k, 100 + i) if k > 1 else []:
            for handoff in (False, True):
                assert np.array_equal(run(fmt, luma[:k], mode, dup, cuts, handoff)[2], want), (fmt, k, cuts, handoff)


def test_blob_holds_the_state_and_no_counters():
    """Two states that differ only in counters pack alike; a damaged tape and a clean one do not; entries past the history counts
    and the bytes behind the state are zero."""
    fmt, luma = STC, synth.make_stc007(3, seed=60)["luma"]
    a = run(fmt, luma, 2, True, [])[2]
    assert not np.array_equal(a, run(fmt, synth.damage_stc007(luma, seed=64), 2, True, [])[2])
    assert not a[:64].any() and not a[292:].any()
    n_last, n_long = int(a[80:84].view(np.int32)[0]), int(a[84:88].view(np.int32)[0])
    assert 0 < n_last <= 9 and 0 < n_long <= 16
    assert not a[120 + 4 * n_last:228].any() and not a[228 + 4 * n_long:292].any()


# ---- sharding.decode_shard with a stub line decoder
N_FRAMES = 12


class StubV2D:
    """What decode_shard uses of VideoToDigital.  One record per frame: the chain state after it, a hash of every frame since the
    file start (memory=None: a wrong guess never heals) or of the last frame only (memory=1).  [seen] logs every call's frames."""

    def __init__(self, memory=None):
        self.memory, self.state, self.seen = memory, None, []

    def doBinarize(self, luma, want_aux=False, continue_file=False):
        if continue_file and self.state is None:
            raise RuntimeError("nothing to continue")
        if not continue_file:
            self.state = torch.zeros(2, dtype=torch.int64)
        self.seen.append((bool(continue_file), [int(v) for v in luma[:, 0, 0]]))
        out = []
        for f in range(luma.shape[0]):
            v = int(luma[f, 0, 0])
            s0 = v if self.memory == 1 else (int(self.state[0]) * 31 + v) % 1000003
            self.state = torch.tensor([s0, 1], dtype=torch.int64)
            out.append(self.state.clone())
        recs = torch.stack(out)
        return (recs, -recs) if want_aux else recs

    def saveState(self):
        return self.state.clone()

    def loadState(self, t):
        self.state = t.clone()


def _luma():
    return (torch.arange(N_FRAMES, dtype=torch.int64) * 7919 % 251 + 1).to(torch.uint8).reshape(-1, 1, 1).repeat(1, 2, 3)


def _shards(edges, warmup, memory=None, want_aux=False):
    world = len(edges) - 1
    luma = _luma()
    stubs = [StubV2D(memory) for _ in range(world)]

    def fn(tr):
        a, b = edges[tr.rank], edges[tr.rank + 1]
        return sharding.decode_shard(stubs[tr.rank], luma[a:b].clone(), tr, warmup=warmup, edges=edges, want_aux=want_aux)
    res = sharding.LocalTransport(world).run(fn)
    whole = StubV2D(memory).doBinarize(luma)
    got = torch.cat([r[0][0] if want_aux else r[0] for r in res])
    assert torch.equal(got, whole)
    if want_aux:
        assert torch.equal(torch.cat([r[0][1] for r in res]), -whole)
    assert all(r[1]["rounds"] == res[0][1]["rounds"] for r in res)
    return [r[1] for r in res], stubs


def test_warmup_luma_is_passed_along_short_shards():
    """Shards of 3 frames: rank g decodes the frames [a-k, a) from a file start, k = min(warmup, a), taken from several ranks back.
    A 9-frame warm-up reaches frame 0 on every rank, so every guess is exact even for a state that never heals; a 7-frame one
    does not on the last rank, which redoes once."""
    edges = [0, 3, 6, 9, 12]
    tape = [int(v) for v in _luma()[:, 0, 0]]
    for warmup, redone in ((9, [0, 0, 0, 0]), (7, [0, 0, 0, 1])):
        stats, stubs = _shards(edges, warmup)
        assert [s["warmup_frames"] for s in stats] == [min(warmup, a) for a in edges[:-1]]
        assert [s["redone"] for s in stats] == redone
        for g in range(1, 4):
            a = edges[g]
            assert stubs[g].seen[0] == (False, tape[max(0, a - warmup):a])
            assert stubs[g].seen[1] == (True, tape[a:edges[g + 1]])


@pytest.mark.parametrize("world", [2, 3, 5])
def test_wrong_guesses_are_redone_rank_by_rank(world):
    """A state that never heals and a 1-frame warm-up: in round r the ranks from r+1 on redo; exact within [world] rounds."""
    edges = [N_FRAMES * g // world for g in range(world)] + [N_FRAMES]
    stats, _ = _shards(edges, 1, want_aux=True)
    assert stats[0]["rounds"] == [list(range(r + 1, world)) for r in range(world - 1)]
    assert [s["redone"] for s in stats] == [min(g, world - 1) if g else 0 for g in range(world)]


def test_right_guesses_cause_no_redo_and_one_frame_shards():
    """A state that heals after one frame: a 2-frame warm-up guesses right everywhere, 1-frame shards included."""
    stats, _ = _shards([0, 1, 2, 5, 6, 12], 2, memory=1)
    assert stats[0]["rounds"] == [] and all(s["redone"] == 0 for s in stats)


def test_edges_from_the_shard_sizes():
    """Without edges, the shards' frame counts are gathered."""
    luma = _luma()
    edges = [0, 5, 12]

    def fn(tr):
        return sharding.decode_shard(StubV2D(), luma[edges[tr.rank]:edges[tr.rank + 1]].clone(), tr, warmup=20)
    res = sharding.LocalTransport(2).run(fn)
    assert torch.equal(torch.cat([r[0] for r in res]), StubV2D().doBinarize(luma))
    assert [r[1]["warmup_frames"] for r in res] == [0, 5]


def test_warmup_must_be_positive_on_later_ranks():
    luma = _luma()
    with pytest.raises(ValueError, match="warmup"):
        sharding.LocalTransport(2).run(lambda tr: sharding.decode_shard(StubV2D(), luma[tr.rank * 6:(tr.rank + 1) * 6].clone(), tr,
                                                                        warmup=0, edges=[0, 6, 12]))
    # one rank: nothing to warm up, warmup = 0 is fine
    recs, stats = sharding.decode_shard(StubV2D(), luma.clone(), sharding.LocalTransport(1)._Rank(sharding.LocalTransport(1), 0),
                                        warmup=0, edges=[0, N_FRAMES])
    assert torch.equal(recs, StubV2D().doBinarize(luma)) and stats["rounds"] == []
