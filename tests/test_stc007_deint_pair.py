"""The two-blocks-at-once deinterleave of the standard setting (stc007_deint.cuh: deint_pair_std14 and its output packing, what
stc007_deint_kernel runs on pairs of adjacent blocks) against the one-block path deint_block_std14 + blk_output, both built as
host code (tests/hostemu/deint_pair.cpp): every field of both Blocks, the samples, the flag bytes and the BROKEN candidate
decision; and the pair path takes exactly the pairs in which each block has at most one untrusted word."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth
from tests import util

SRC = os.path.join(util.HERE, "hostemu", "deint_pair.cpp")
LIB = os.path.join(os.path.dirname(util.EMU_LIB), "libdeint_pair.so")
EMU_BLOCK = np.dtype([("words", "<u2", 8), ("line_crc", "u1"), ("word_valid", "u1"), ("resolution", "u1"), ("audio_state", "u1"),
                      ("samples", "<i2", 6), ("flags", "u1", 6), ("broken_ns", "u1"), ("pad", "u1")])
_lib = None


def lib():
    """The host build, compiled on first use (as util.build_hostemu does)."""
    global _lib
    if _lib is None:
        csrc = os.path.join(util.ROOT, "sdvpcmdecoder_b200", "csrc")
        deps = [SRC] + [os.path.join(csrc, f) for f in os.listdir(csrc)]
        if not (os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps)):
            os.makedirs(os.path.dirname(LIB), exist_ok=True)
            subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w", "-o", LIB, SRC], check=True)
        _lib = C.CDLL(LIB)
    return _lib


def run_both(words, ok):
    """words u16 [n, 2, 8], ok u8 [n, 2] -> (one-block path [n, 2], pair path [n, 2], covered bool [n])."""
    words = np.ascontiguousarray(words, np.uint16)
    ok = np.ascontiguousarray(ok, np.uint8)
    n = words.shape[0]
    assert EMU_BLOCK.itemsize == 40
    ref = np.zeros((n, 2), EMU_BLOCK)
    got = np.zeros((n, 2), EMU_BLOCK)
    cov = np.zeros(n, np.uint8)
    lib().emu_pair_scalar(n, util._p(words), util._p(ok), util._p(ref))
    lib().emu_pair_packed(n, util._p(words), util._p(ok), util._p(got), util._p(cov))
    return ref, got, cov.astype(bool)


def check(words, ok):
    ref, got, cov = run_both(words, ok)
    n_bad = np.array([[bin(0xFF & ~int(v)).count("1") for v in row] for row in ok])
    np.testing.assert_array_equal(cov, (n_bad <= 1).all(axis=1), "the pair path must take exactly the pairs with <= 1 untrusted word per block")
    for f in EMU_BLOCK.names:
        if f == "pad":
            continue
        a, b = ref[cov][f], got[cov][f]
        bad = np.nonzero((a != b).reshape(len(a), -1).any(axis=1))[0]
        assert len(bad) == 0, (f, len(bad), words[cov][bad[0] // 2] if len(bad) else None, ok[cov][bad[0] // 2] if len(bad) else None,
                               a[bad[0]], b[bad[0]])
    return ref, got, cov


def codewords(rng, n):
    """n valid blocks: six random 14-bit audio words with their P and Q."""
    a = rng.randint(0, 1 << 14, size=(n, 6)).astype(np.uint16)
    p, q = synth.stc007_pq(a)
    return np.concatenate([a, p[:, None], q[:, None]], axis=1)


def damage(rng, w, kind):
    """kind 0: syndromes zero; 1: only P's syndrome non-zero; 2: only Q's; 3: both (an audio word changed)."""
    w = w.copy()
    n = w.shape[0]
    e = rng.randint(1, 1 << 14, size=n).astype(np.uint16)
    if kind == 1:
        w[:, 6] ^= e
    elif kind == 2:
        w[:, 7] ^= e
    elif kind == 3:
        w[np.arange(n), rng.randint(0, 6, size=n)] ^= e
    return w


def all_ok_pairs():
    a, b = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    return np.stack([a.ravel(), b.ravel()], axis=1).astype(np.uint8)


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_every_pair_of_ok_masks(kind):
    """All 256 x 256 pairs of trusted-line masks, on codewords with zero syndromes, only Sp, only Sq or both non-zero; the untrusted
    words keep their value or are overwritten with garbage (what a line without a valid CRC brings)."""
    rng = np.random.RandomState(100 + kind)
    ok = all_ok_pairs()
    n = len(ok)
    w = np.stack([damage(rng, codewords(rng, n), kind), damage(rng, codewords(rng, n), kind)], axis=1)
    garbage = rng.rand(n, 2, 8) < 0.5
    bad_line = ((ok[:, :, None] >> np.arange(8)) & 1) == 0
    junk = rng.randint(0, 1 << 14, size=w.shape).astype(np.uint16)
    w = np.where(garbage & bad_line, junk, w)
    ref, got, cov = check(w, ok)
    assert cov.sum() == 9 * 9          # none or one of the 8 words untrusted, in each block
    st = ref[cov]["audio_state"]
    assert (st == 3).any() == (kind != 0)           # BROKEN blocks exactly when damaged
    assert (st == 1).any() or kind != 0             # corrections by P


def test_random_words_and_high_bits():
    """Random 16-bit words (bits 14 and 15 too: the checks see them, the samples drop them), mostly-trusted masks."""
    rng = np.random.RandomState(7)
    n = 200000
    w = rng.randint(0, 1 << 16, size=(n, 2, 8)).astype(np.uint16)
    near = np.stack([codewords(rng, n), codewords(rng, n)], axis=1)
    pick = rng.rand(n, 2, 1) < 0.5
    w = np.where(pick, near ^ (rng.rand(n, 2, 8) < 0.05) * np.uint16(0xC000), w)
    ok = np.full((n, 2), 0xFF, np.uint8)
    drop = rng.randint(0, 9, size=(n, 2))              # 8 = none
    ok = np.where(drop < 8, ok & ~(1 << np.minimum(drop, 7)).astype(np.uint8), ok).astype(np.uint8)
    check(w, ok)


def test_control_block_and_silent_patterns():
    """Silent blocks (all audio zero: BROKEN but never a window candidate) and a control-block line's word in a block."""
    rng = np.random.RandomState(11)
    ok = all_ok_pairs()
    n = len(ok)
    silent = np.zeros((n, 2, 8), np.uint16)
    kind = rng.randint(0, 4, size=(n, 2))
    e = rng.randint(1, 1 << 14, size=(n, 2)).astype(np.uint16)
    silent[:, :, 6] = np.where(kind == 1, e, 0)
    silent[:, :, 7] = np.where(kind == 2, e, 0)
    silent[:, :, 0] = np.where(kind == 3, e, 0)
    ref, got, cov = check(silent, ok)
    assert (ref[cov]["audio_state"] == 3).any()
    cb = np.array(synth.STC007_CTRL_BLOCK, np.uint16)
    w = np.stack([codewords(rng, n), codewords(rng, n)], axis=1)
    k = rng.randint(0, 8, size=(n, 2))
    w[np.arange(n)[:, None], np.arange(2)[None, :], k] = cb[k]
    check(w, ok)
