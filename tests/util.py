"""Shared helpers of the test-suite (TEST INFRASTRUCTURE)."""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX, BLOCK_REC

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EMU_SRC = os.path.join(HERE, "hostemu", "hostemu.cpp")
EMU_LIB = os.path.join(HERE, "hostemu", "_build", "libhostemu.so")
REF_STREAMS = os.path.join(HERE, "golden", "reference_streams.json")
_emu = None
_ref_streams = None


# ---- the reference pipeline's output streams, stored as digests (tests/golden/reference_streams.json, make_golden.py streams)
def tape_key(kind, luma, params):
    """Key of one reference run: the tape's bytes, its shape and the pipeline settings."""
    h = hashlib.blake2b(np.ascontiguousarray(luma).tobytes(), digest_size=16)
    h.update(repr((kind, tuple(luma.shape), tuple(int(p) for p in params))).encode())
    return h.hexdigest()


def chunk_digests(arrays, rows):
    """blake2b digest of every [rows] rows of the arrays (all of one length), in order: one digest per frame."""
    n = len(arrays[0])
    assert all(len(a) == n for a in arrays)
    out = []
    for a in range(0, n, rows):
        h = hashlib.blake2b(digest_size=16)
        for x in arrays:
            h.update(np.ascontiguousarray(x[a:a + rows]).tobytes())
        out.append(h.hexdigest())
    return out


def stream_entry(arrays, rows):
    """Stored form of a stream: a digest per frame (chunk of rows) over all arrays, and a digest per array over all frames."""
    return {"rows": int(len(arrays[0])), "chunk": rows, "digests": chunk_digests(arrays, rows),
            "fields": [chunk_digests([a], len(a))[0] for a in arrays]}


def stream_mismatch_digests(ref, arrays):
    """'' when the arrays equal the stored stream; else which frames (chunks) and which arrays (by position) differ."""
    if len(arrays[0]) != ref["rows"]:
        return f"{len(arrays[0])} rows, reference {ref['rows']}"
    got = chunk_digests(arrays, ref["chunk"])
    bad = [i for i, (a, b) in enumerate(zip(got, ref["digests"])) if a != b]
    fields = [i for i, (a, d) in enumerate(zip(arrays, ref["fields"])) if chunk_digests([a], len(a))[0] != d]
    return f"{len(bad)} of {len(got)} frames differ, first {bad[:6]}; arrays {fields} differ" if bad else ""


def golden_stream(kind, luma, params):
    """The stored reference stream(s) of this tape and these settings; a tape without one is an error, not a skip."""
    global _ref_streams
    if _ref_streams is None:
        with open(REF_STREAMS) as f:
            _ref_streams = json.load(f)
    key = tape_key(kind, luma, params)
    assert key in _ref_streams, f"no reference stream stored for this {kind} tape {tuple(luma.shape)} / {params} (make_golden.py streams)"
    return _ref_streams[key]


def build_hostemu():
    deps = [EMU_SRC] + [os.path.join(ROOT, "sdvpcmdecoder_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "sdvpcmdecoder_b200", "csrc"))]
    if os.path.exists(EMU_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(EMU_LIB) for d in deps):
        return
    os.makedirs(os.path.dirname(EMU_LIB), exist_ok=True)
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w", "-o", EMU_LIB, EMU_SRC], check=True)


def emu():
    global _emu
    if _emu is None:
        build_hostemu()
        _emu = C.CDLL(EMU_LIB)
    return _emu


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def emu_v2d(luma, mode=2, dup=True, hybrid=False, m2=False):
    luma = np.ascontiguousarray(luma, dtype=np.uint8)
    f, h, w = luma.shape
    rec = np.zeros(f * h, LINE_REC)
    aux = np.zeros(f * h, LINE_AUX)
    if hybrid:
        st = (C.c_longlong * 4)()
        emu().emu_v2d_hybrid(mode, int(dup) | (2 if m2 else 0), _p(luma), f, h, w, _p(rec), _p(aux), st)
        return rec, aux, list(st)
    emu().emu_v2d_chain(mode, int(dup) | (2 if m2 else 0), _p(luma), f, h, w, _p(rec), _p(aux))
    return rec, aux, None


def emu_deint(lines, res_mode=0, ignore_crc=False, force_check=True, p_corr=True, q_corr=True, broken_mask_dur=0, m2=False):
    lines = np.ascontiguousarray(lines)
    n = lines.shape[0]
    nb = max(n - 112, 0)
    blocks = np.zeros(nb, BLOCK_REC)
    samples = np.zeros((nb, 6), np.int16)
    flags = np.zeros((nb, 6), np.uint8)
    emu().emu_deint(_p(lines), n, res_mode | (0x100 if m2 else 0), int(ignore_crc), int(force_check), int(p_corr), int(q_corr), broken_mask_dur,
                    _p(blocks), _p(samples), _p(flags))
    return blocks, samples, flags


def emu_deint_carry(lines, countdown_in=0, res_mode=0, ignore_crc=False, force_check=True, p_corr=True, q_corr=True, broken_mask_dur=128):
    """emu_deint with the broken-block countdown carried in and out (what sdv_deint_config.countdown_in / sdv_stc007_countdown do)."""
    lines = np.ascontiguousarray(lines)
    n = lines.shape[0]
    nb = max(n - 112, 0)
    blocks = np.zeros(nb, BLOCK_REC)
    samples = np.zeros((nb, 6), np.int16)
    flags = np.zeros((nb, 6), np.uint8)
    out = C.c_int(0)
    emu().emu_deint_carry(_p(lines), n, res_mode, int(ignore_crc), int(force_check), int(p_corr), int(q_corr), broken_mask_dur,
                          _p(blocks), _p(samples), _p(flags), int(countdown_in), C.byref(out))
    return blocks, samples, flags, out.value


REC_FIELDS = ["words", "ref", "black", "white", "hyst", "data_start", "data_stop", "shift", "service_type"]
AUX_FIELDS = ["ref_low", "ref_high", "marker_start_bg", "marker_start_ed", "marker_stop_ed", "word_crc_mask", "word_valid_mask"]
ORACLE_ONLY_FLAGS = np.uint16((1 << 7) | (1 << 11))      # coordinate sweep / control bit: not STC-007


def compare_line_records(oracle_recs, rec, aux=None, tier_a_only=False, oracle_only_flags=None):
    """Field-by-field comparison of oracle/reference line records with product records.  Returns a list of mismatch strings."""
    bad = []
    o = oracle_recs
    assert len(o) == len(rec), (len(o), len(rec))
    if not np.array_equal(o["words"], rec["words"]):
        d = (o["words"] != rec["words"]).any(axis=1)
        bad.append(f"words: {int(d.sum())} lines, first {np.nonzero(d)[0][:5]}")
    fo = o["flags"] & ~(ORACLE_ONLY_FLAGS if oracle_only_flags is None else np.uint16(oracle_only_flags))
    fr = rec["flags"]
    if tier_a_only:
        fo, fr = fo & 7, fr & 7
    if not np.array_equal(fo, fr):
        d = fo != fr
        bad.append(f"flags: {int(d.sum())} lines, first {np.nonzero(d)[0][:5]} oracle {fo[d][:5]} got {fr[d][:5]}")
    if tier_a_only:
        return bad
    for n in REC_FIELDS[1:]:
        if not np.array_equal(o[n], rec[n]):
            d = o[n] != rec[n]
            bad.append(f"{n}: {int(d.sum())} lines, first {np.nonzero(d)[0][:5]} oracle {o[n][d][:5]} got {rec[n][d][:5]}")
    ms = (o["mark_st_stage"] | (o["mark_ed_stage"] << 4)).astype(np.uint8)
    if not np.array_equal(ms, rec["mark_stages"]):
        d = ms != rec["mark_stages"]
        bad.append(f"mark_stages: {int(d.sum())} lines, first {np.nonzero(d)[0][:5]}")
    if aux is not None:
        for n in AUX_FIELDS:
            if not np.array_equal(o[n], aux[n]):
                d = o[n] != aux[n]
                bad.append(f"aux.{n}: {int(d.sum())} lines, first {np.nonzero(d)[0][:5]}")
    return bad


def line_arrays(rec, aux, with_part=False):
    """The fields compare_line_records looks at, of product records + aux (with_part: the PCM-16x0 sub-line part in reserved),
    in the order the stored digests of reference line records use (tests/golden/reference_streams.json): words, flags,
    REC_FIELDS[1:], mark_stages, AUX_FIELDS[, reserved]."""
    a = [rec["words"], rec["flags"]] + [rec[n] for n in REC_FIELDS[1:]] + [rec["mark_stages"]] + [aux[n] for n in AUX_FIELDS]
    return a + [rec["reserved"]] if with_part else a


def lines_mismatch(kind, luma, params, rec, aux, with_part=False):
    """'' when the product's line records equal the reference's stored for this tape (one digest per frame)."""
    return stream_mismatch_digests(golden_stream(kind, luma, params), line_arrays(rec, aux, with_part))


def lines_from_oracle(o):
    """Oracle/reference line records -> product LINE_REC array (for feeding the deinterleaver)."""
    r = np.zeros(len(o), LINE_REC)
    r["words"] = o["words"]
    r["flags"] = o["flags"] & ~ORACLE_ONLY_FLAGS
    for n in REC_FIELDS[1:]:
        r[n] = o[n]
    r["mark_stages"] = (o["mark_st_stage"] | (o["mark_ed_stage"] << 4)).astype(np.uint8)
    return r


def compare_blocks(oracle_blocks, blocks, samples, flags):
    """Oracle block records (BLOCK_REC of refbind) vs product blocks / samples."""
    bad = []
    ob = oracle_blocks
    assert len(ob) == len(blocks), (len(ob), len(blocks))
    for n in ["words", "line_crc", "word_valid", "audio_state", "resolution"]:
        if not np.array_equal(ob[n], blocks[n]):
            d = ob[n] != blocks[n]
            d = d.any(axis=1) if d.ndim > 1 else d
            bad.append(f"block.{n}: {int(d.sum())} blocks, first {np.nonzero(d)[0][:5]}")
    of = ob["flags"] & 0x1F
    if not np.array_equal(of, blocks["flags"] & 0x1F):
        d = of != (blocks["flags"] & 0x1F)
        bad.append(f"block.flags: {int(d.sum())} blocks, first {np.nonzero(d)[0][:5]} oracle {of[d][:5]} got {blocks['flags'][d][:5]}")
    if not np.array_equal(ob["samples"], samples):
        d = (ob["samples"] != samples).any(axis=1)
        bad.append(f"samples: {int(d.sum())} blocks, first {np.nonzero(d)[0][:5]}")
    # outputSamplePair flags from the oracle's block state
    broken = (ob["flags"] & 2) != 0
    bvalid = ((ob["flags"] & 1) != 0) & ~broken
    exp = np.zeros((len(ob), 6), np.uint8)
    for i in range(6):
        wv = ((ob["word_valid"] >> i) & 1).astype(bool) & ~broken
        lc = ((ob["line_crc"] >> i) & 1).astype(bool) & bvalid
        exp[:, i] = bvalid * 1 + wv * 2 + lc * 4
    if not np.array_equal(exp, flags):
        d = (exp != flags).any(axis=1)
        bad.append(f"sample flags: {int(d.sum())} blocks, first {np.nonzero(d)[0][:5]}")
    return bad


P1_PRESET = np.dtype([("start", "<i2"), ("stop", "<i2"), ("valid", "u1"), ("ref", "u1"), ("pad", "u1", (2,))])


def emu_p1_v2d(luma, mode=2, dup=True):
    """PCM-1 line decode + chain through the host build of the device code (one-thread block)."""
    luma = np.ascontiguousarray(luma, dtype=np.uint8)
    f, h, w = luma.shape
    rec = np.zeros(f * h, LINE_REC)
    aux = np.zeros(f * h, LINE_AUX)
    ps = np.zeros(f, P1_PRESET)
    emu().emu_p1_v2d_chain(mode, int(dup), _p(luma), f, h, w, _p(rec), _p(aux), _p(ps))
    return rec, aux, ps


def ref_lines_in_frame_order(ref, keep=(0, 6, 7)):
    """Reference V2D record stream -> the product's record order (service lines other than header/control block dropped)."""
    m = np.isin(ref["service_type"], keep)
    return ref[m]


def emu_p1_assemble(recs, n_frames, height, bff=False, file_start=True, offsets=None):
    from sdvpcmdecoder_b200.capi import PCM1_SUBLINE, PCM1_FRAME_INFO
    recs = np.ascontiguousarray(recs)
    sub = np.zeros(n_frames * 2 * 735, PCM1_SUBLINE)
    info = np.zeros(n_frames, PCM1_FRAME_INFO)
    emu().emu_p1_assemble(_p(recs), n_frames, height, int(bff), int(file_start), int(offsets is not None), *(offsets or (0, 0)),
                          _p(sub), _p(info))
    return sub, info


def emu_x0_v2d(luma, mode=2, dup=True):
    """PCM-16x0 line decode + chain through the host build of the device code: three sub-line records per video line."""
    luma = np.ascontiguousarray(luma, dtype=np.uint8)
    f, h, w = luma.shape
    rec = np.zeros(f * h * 3, LINE_REC)
    aux = np.zeros(f * h * 3, LINE_AUX)
    ps = np.zeros(f, P1_PRESET)
    emu().emu_x0_v2d_chain(mode, int(dup), _p(luma), f, h, w, _p(rec), _p(aux), _p(ps))
    return rec, aux, ps


def x0_ref_to_product(ref):
    """Reference PCM-16x0 sub-line records -> the product's field layout (queue_order in words[4], part in reserved)."""
    r = ref.copy()
    r["words"][:, 4] = ref["queue_order"]
    return r


def emu_x0_stitch_info(recs, n_frames, height, bff=False, top=(5, 5), ignore_crc=False, p_corr=True, broken_mask_dur=81, mask_seams=None):
    from sdvpcmdecoder_b200 import capi
    recs = np.ascontiguousarray(recs)
    smp = np.zeros((n_frames * 490, 6), np.int16)
    fl = np.zeros((n_frames * 490, 6), np.uint8)
    info = np.zeros(n_frames, capi.PCM16X0_FRAME_INFO)
    ms = None if mask_seams is None else np.ascontiguousarray(mask_seams, dtype=np.uint8)
    emu().emu_x0_stitch_info(_p(recs), n_frames, height, int(bff), top[0], top[1], int(ignore_crc), int(p_corr), broken_mask_dur,
                             _p(ms) if ms is not None else None, _p(smp), _p(fl), _p(info))
    return smp, fl, info


def emu_x0_stitch(recs, n_frames, height, bff=False, top=(5, 5), ignore_crc=False, p_corr=True, broken_mask_dur=81, mask_seams=None):
    recs = np.ascontiguousarray(recs)
    smp = np.zeros((n_frames * 490, 6), np.int16)
    fl = np.zeros((n_frames * 490, 6), np.uint8)
    ms = None if mask_seams is None else np.ascontiguousarray(mask_seams, dtype=np.uint8)
    emu().emu_x0_stitch(_p(recs), n_frames, height, int(bff), top[0], top[1], int(ignore_crc), int(p_corr), broken_mask_dur,
                        _p(ms) if ms is not None else None, _p(smp), _p(fl))
    return smp, fl


def emu_stc007_stitch(recs, n_frames, height, video_std=1, field_order=1, res16=False, mask_seams=True, fix_cut_above=False,
                      max_unch14=0x40, max_unch16=0x20, file_end=True, ignore_crc=False, p_corr=True, q_corr=True, broken_mask_dur=128, m2=False, cwd=False):
    """STC007DataStitcher through the host build of the device code + the library's own decision chain (one-thread blocks)."""
    from sdvpcmdecoder_b200 import capi
    recs = np.ascontiguousarray(recs)
    cap = 80 + 112 + n_frames * 588
    blocks = np.zeros(cap, BLOCK_REC)
    samples = np.zeros((cap, 6), np.int16)
    flags = np.zeros((cap, 6), np.uint8)
    info = np.zeros(max(n_frames, 1), capi.STC007_FRAME_INFO)
    # res16: False / True = preset, None = detected per field
    st = (C.c_int * 10)(video_std, field_order, 2 if res16 is None else int(res16), int(mask_seams), int(fix_cut_above), max_unch14, max_unch16, 1, int(file_end), int(cwd))
    res_mode = 3 if res16 else 0
    nb = emu().emu_stc007_stitch(_p(recs), n_frames, height, st, res_mode, int(ignore_crc), int(p_corr), int(q_corr), broken_mask_dur, int(m2),
                                 _p(blocks), _p(samples), _p(flags), _p(info))
    assert nb >= 0
    return blocks[:nb], samples[:nb], flags[:nb], info[:n_frames if file_end else max(n_frames - 1, 0)]


def emu_x0_stitch_auto(recs, n_frames, height, bff=False, ignore_crc=False, p_corr=True, broken_mask_dur=81, mask_seams=True, ei=False):
    """PCM-16x0 (SI, or EI with ei=True) frames -> samples with the reference's own padding search (host build of the scan +
    the library's chain)."""
    from sdvpcmdecoder_b200 import capi
    recs = np.ascontiguousarray(recs)
    smp = np.zeros((n_frames * 490, 6), np.int16)
    fl = np.zeros((n_frames * 490, 6), np.uint8)
    al = np.zeros(n_frames, capi.PCM16X0_ALIGNMENT)
    fn = emu().emu_x0_stitch_auto_ei if ei else emu().emu_x0_stitch_auto
    fn(_p(recs), n_frames, height, int(bff), int(ignore_crc), int(p_corr), broken_mask_dur, int(mask_seams), _p(smp), _p(fl), _p(al))
    return smp, fl, al


def emu_set_fine(**fields):
    """Fine binarization settings (numeric fields of bin_preset_t) of the host build; no arguments = the defaults."""
    from oracle.refbind import FINE_FIELDS, FINE_DEFAULTS
    if not fields:
        emu().emu_set_fine(None)
        return
    v = dict(FINE_DEFAULTS)
    v.update(fields)
    emu().emu_set_fine((C.c_int * len(FINE_FIELDS))(*[int(v[k]) for k in FINE_FIELDS]))
