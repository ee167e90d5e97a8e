"""Generates the golden fixtures from the UNMODIFIED reference (oracle/_ref/libsdvref.so, built from /root/reference by
oracle/Makefile).  Run in the build container only:  python tests/golden/make_golden.py

  stc007_pipeline_pal.npz : PCMSamplePair stream of VideoToDigital + STC007DataStitcher (PAL/TFF/14-bit preset, P+Q on,
                            CWD off) on synth.make_stc007(8, seed=1234)
  stc007_lines_clean.npz / stc007_lines_damaged.npz : every STC007Line the reference VideoToDigital emits for a clean
                            and a damaged (synth.damage_stc007) tape, MODE_NORMAL
  stc007_deint.npz        : STC007Deinterleaver::processBlock results on random erased lines, all resolution modes
  stc007_try_padding.npz  : STC007DataStitcher::tryPadding (private member) for paddings 0..31 on eight field seams
  stc007_find_padding.npz : STC007DataStitcher::findPadding (private member) on 60 random seams x 18 settings
  pcm16x0_frame_info.npz  : sample rate / emphasis per frame of the reference's PCM-16x0 PCMSamplePair stream (control-bit votes + history)
  pcm16x0_deint.npz       : PCM16X0Deinterleaver::processBlock (SI) over 24 interleave blocks, six settings
  pcm1_deint.npz          : PCM1Deinterleaver::processBlock over 6 fields of random sub-lines, CRC checked / ignored
  pcm16x0_lines.npz       : every PCM16X0SubLine of VideoToDigital (MODE_NORMAL) for four tapes of
                            tests.test_pcm16x0_line.pcm16x0_cases()
  pcm16x0_ei_stitch.npz   : PCM-16x0 EI format: sub-line records of VideoToDigital and the PCMSamplePair stream of PCM16X0DataStitcher
                            (setFormat(FORMAT_EI); TFF / BFF / no P correction) for two tapes of tests.test_pcm16x0_stitch.ei_cases()
  stc007_stitch.npz       : line records of VideoToDigital and the PCMSamplePair stream of STC007DataStitcher (PAL/TFF/14-bit preset,
                            trim, paddings and masking its own) for two heavily damaged tapes of tests.test_stc007_stitch.stitch_cases()
                            (only this file: python tests/golden/make_golden.py stitch)
  pcm1_lines.npz          : every PCM1Line of VideoToDigital (MODE_NORMAL) and the PCMSamplePair stream of PCM1DataStitcher
                            (TFF, automatic line offset) for four tapes of tests.test_pcm1_line.pcm1_cases()
  reference_streams.json  : per-frame digests of the reference's line records (PCM-1, PCM-16x0, M2) and pipeline streams (STC-007,
                            PCM-1, PCM-16x0, M2) on the tapes of the parity tests (streams_golden(); needs no reference build:
                            python tests/golden/make_golden.py streams)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oraclebind as O, refbind as R  # noqa: E402
from sdvpcmdecoder_b200 import synth  # noqa: E402
from tests.test_hostemu import _random_lines  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def stitch_golden():
    from tests import util
    from tests.test_stc007_stitch import stitch_cases
    out = {}
    for name in ("heavy", "vertical_jitter_heavy"):
        luma, std, order, res, p, q = stitch_cases()[name]
        pairs, _, _ = R.pipeline_run(R.TYPE_STC007, R.MODE_NORMAL, luma, R.StitchCfg(video_std=std, field_order=order, resolution=res, p_corr=p, q_corr=q))
        pairs = pairs[pairs["service_type"] == 0]
        recs = util.lines_from_oracle(util.ref_lines_in_frame_order(R.v2d_run(R.TYPE_STC007, R.MODE_NORMAL, luma), keep=(0, 7)))
        out[name + "_recs"] = recs.view(np.uint8).reshape(len(recs), -1)
        out[name + "_shape"] = np.array(luma.shape)
        out[name + "_l"], out[name + "_r"], out[name + "_fl"], out[name + "_fr"] = pairs["l"], pairs["r"], pairs["flags_l"], pairs["flags_r"]
    np.savez_compressed(os.path.join(HERE, "stc007_stitch.npz"), **out)


def ei_stitch_golden():
    """PCM-16x0 EI format: the reference's sub-line records of two tapes + its PCMSamplePair stream for three settings."""
    from tests import util
    from tests.test_pcm16x0_line import ref_sublines
    from tests.test_pcm16x0_stitch import ei_cases
    out = {}
    for name in ("variantB", "shift-60"):
        luma = ei_cases()[name]
        ref = ref_sublines(luma)
        rec = util.lines_from_oracle(util.x0_ref_to_product(ref))
        rec["flags"], rec["reserved"] = ref["flags"], ref["line_part"]       # the control bit travels in the flags (bit 11)
        out[name + "_rec"] = rec.view(np.uint8).reshape(len(rec), -1)
        out[name + "_frames"] = np.array(luma.shape[0])
        for i, (bff, p_corr) in enumerate(((False, True), (True, True), (False, False))):
            smp, fl = _live_reference(("pcm16x0", luma, (bff, p_corr, True)), 490)["arrays"]
            got = util.emu_x0_stitch_auto(rec, luma.shape[0], luma.shape[1], bff, p_corr=p_corr, ei=True)
            assert np.array_equal(smp, got[0]) and np.array_equal(fl, got[1]), (name, bff, p_corr)
            out[f"{name}_smp{i}"], out[f"{name}_fl{i}"] = smp, fl
    np.savez_compressed(os.path.join(HERE, "pcm16x0_ei_stitch.npz"), **out)


def _stream_runs():
    """(kind, luma, params) of every reference pipeline run the parity tests compare with."""
    from tests import test_gpu_stc007_stitch as G
    from tests.test_stc007_stitch import stitch_cases, resolution_cases, cwd_cases
    from tests.test_pcm16x0_stitch import alignment_cases, ei_cases
    runs = [("stc007", luma, (std, order, res, p, q, 0)) for luma, std, order, res, p, q in stitch_cases().values()]
    runs += [("stc007", G.config4_tape(s), (1, 1, 1, 1, 1, 0)) for s in G.CONFIG4_SEEDS]
    runs += [("stc007", G.two_shard_tape(), (1, 1, 1, 1, 1, 0)), ("stc007", G.ntsc16_tape(), (0, 0, 0, 1, 1, 0)),
             ("stc007", G.cwd_config4_tape(), (1, 1, 1, 1, 1, 1))]
    runs += [("stc007", luma, (1, 1, 0, 1, 1, 0)) for luma in resolution_cases().values()]
    for name, (luma, std, order, res, p, q) in cwd_cases().items():
        runs.append(("stc007", luma, (std, order, res, p, q, 1)))
        if name in ("dropouts", "heavy", "dropouts16"):
            runs.append(("stc007", luma, (std, order, res, p, q, 0)))
    for ei, cases in ((False, alignment_cases()), (True, ei_cases())):
        runs += [("pcm16x0", luma, (bff, p_corr, ei)) for luma in cases.values() for bff, p_corr in ((False, True), (True, True), (False, False))]
    # line records of the GPU line tests, PCM-1 sample streams, M2
    from tests import test_gpu_pcm1_line as P1, test_gpu_pcm16x0_line as X0
    from tests.test_pcm1_line import pcm1_cases
    from tests.test_m2 import m2_tapes
    runs += [("pcm1_lines", luma, (mode, dup)) for luma, mode, dup in P1.line_runs()]
    runs += [("pcm16x0_lines", luma, (mode, dup)) for luma, mode, dup in X0.line_runs()]
    runs += [("pcm1", luma, (bff,)) for luma in pcm1_cases().values() for bff in (False, True)]
    runs += [("pcm1_offsets", pcm1_cases()["clean"], ofs) for ofs in P1.MANUAL_OFFSETS]
    runs += [(kind, luma, ()) for luma in m2_tapes().values() for kind in ("m2_lines", "m2")]
    return runs


def _stream(run):
    from tests import util
    from tests.test_stc007_stitch import oracle_lines, pair_arrays, block_arrays, BLOCKS_PER_FRAME
    kind, luma, params = run
    if kind == "stc007":
        std, order, res, p, q, cwd = params
        blocks, samples, flags, _ = util.emu_stc007_stitch(oracle_lines(luma), luma.shape[0], luma.shape[1], video_std=std, field_order=order,
                                                           res16={0: None, 1: False, 2: True}[res], p_corr=bool(p), q_corr=bool(q), cwd=bool(cwd))
        out = {"pairs": util.stream_entry(pair_arrays(samples, flags), 3 * BLOCKS_PER_FRAME),
               "blocks": util.stream_entry(block_arrays(blocks), BLOCKS_PER_FRAME)}
    elif kind == "pcm16x0":
        bff, p_corr, ei = params
        rec, _, _ = util.emu_x0_v2d(luma, 2, True)
        smp, fl, _ = util.emu_x0_stitch_auto(rec, luma.shape[0], luma.shape[1], bff, p_corr=p_corr, ei=ei)
        out = util.stream_entry([smp, fl], 490)
    elif kind in ("pcm1_lines", "pcm16x0_lines"):
        rec, aux, _ = (util.emu_p1_v2d if kind == "pcm1_lines" else util.emu_x0_v2d)(luma, *params)
        out = util.stream_entry(util.line_arrays(rec, aux, with_part=(kind == "pcm16x0_lines")), len(rec) // luma.shape[0])
    elif kind in ("pcm1", "pcm1_offsets"):
        from tests.test_pcm1_line import emu_samples
        rec, _, _ = util.emu_p1_v2d(luma, 2, True)
        if kind == "pcm1":
            smp, fl, _ = emu_samples(rec, luma.shape[0], luma.shape[1], params[0])
        else:
            sub, _ = util.emu_p1_assemble(rec, luma.shape[0], luma.shape[1], False, True, offsets=params)
            smp, fl = O.deint_pcm1(np.stack([sub["left"], sub["right"]], axis=1), sub["flags"])
        out = util.stream_entry([smp.reshape(-1), fl.reshape(-1) & 3], 2 * 2 * 735)
    else:
        from tests.test_m2 import assemble
        rec, aux, _ = util.emu_v2d(luma, 2, True, hybrid=True, m2=True)
        if kind == "m2_lines":
            out = util.stream_entry(util.line_arrays(rec, aux), luma.shape[1])
        else:
            _, s, f = util.emu_deint(assemble(rec, luma.shape[0]), 0, False, True, True, True, 128, m2=True)
            out = util.stream_entry([s.reshape(-1, 2), f.reshape(-1, 2)], 3 * BLOCKS_PER_FRAME)
    return util.tape_key(kind, luma, params), out


def _live_reference(run, chunk):
    """The same stream computed by the reference build (oracle/_ref), with the field selection and masking of the comparisons
    the parity tests made against it when they ran it live."""
    from tests import util
    from tests.test_stc007_stitch import block_arrays
    kind, luma, params = run
    n_lines = luma.shape[0] * luma.shape[1]

    def pairs_of(pcm_type, cfg, mask=7, shape=(-1, 2)):
        pairs, _, blocks = R.pipeline_run(pcm_type, R.MODE_NORMAL, luma, cfg)
        a = pairs[pairs["service_type"] == 0]
        return [np.stack([a["l"], a["r"]], 1).reshape(shape), (np.stack([a["flags_l"], a["flags_r"]], 1) & mask).astype(np.uint8).reshape(shape)], blocks

    def lines_of(ref, mask, with_part=False):
        a = [ref["words"], ref["flags"] & ~np.uint16(mask)] + [ref[n] for n in util.REC_FIELDS[1:]]
        a += [(ref["mark_st_stage"] | (ref["mark_ed_stage"] << 4)).astype(np.uint8)] + [ref[n] for n in util.AUX_FIELDS]
        return a + [ref["line_part"]] if with_part else a

    if kind == "stc007":
        std, order, res, p, q, cwd = params
        arrays, blocks = pairs_of(R.TYPE_STC007, R.StitchCfg(video_std=std, field_order=order, resolution=res, p_corr=p, q_corr=q, cwd=cwd))
        return {"pairs": dict(util.stream_entry(arrays, chunk["pairs"]), arrays=arrays),
                "blocks": dict(util.stream_entry(block_arrays(blocks), chunk["blocks"]), arrays=block_arrays(blocks))}
    if kind == "pcm16x0":
        bff, p_corr, ei = params
        arrays, _ = pairs_of(R.TYPE_PCM16X0, R.StitchCfg(field_order=2 if bff else 1, pcm16x0_format=2 if ei else 1, p_corr=int(p_corr)), shape=(-1, 6))
    elif kind == "pcm1":
        arrays, _ = pairs_of(R.TYPE_PCM1, R.StitchCfg(field_order=2 if params[0] else 1, auto_line_offset=1), mask=3, shape=-1)
    elif kind == "pcm1_offsets":
        cfg = R.StitchCfg(field_order=1, auto_line_offset=0)
        cfg.reserved[0], cfg.reserved[1] = params
        arrays, _ = pairs_of(R.TYPE_PCM1, cfg, mask=3, shape=-1)
    elif kind == "m2":
        arrays, _ = pairs_of(R.TYPE_M2, R.StitchCfg(video_std=1, field_order=1, resolution=1, p_corr=1, q_corr=1, cwd=0))
    elif kind == "pcm1_lines":
        mode, dup = params
        arrays = lines_of(util.ref_lines_in_frame_order(R.v2d_run(R.TYPE_PCM1, mode, luma, line_dup=dup))[:n_lines], 1 << 11)
    elif kind == "pcm16x0_lines":
        mode, dup = params
        ref = R.v2d_run(R.TYPE_PCM16X0, mode, luma, line_dup=dup)
        arrays = lines_of(util.x0_ref_to_product(ref[ref["service_type"] == 0][:3 * n_lines]), 0, with_part=True)
    else:
        ref = R.v2d_run(R.TYPE_M2, R.MODE_NORMAL, luma)
        arrays = lines_of(ref[(ref["service_type"] == 0) | (ref["service_type"] == 7)][:n_lines], util.ORACLE_ONLY_FLAGS)
    return dict(util.stream_entry(arrays, chunk), arrays=arrays)


def streams_golden():
    """reference_streams.json: the line records and PCMSamplePair streams (and STC-007 data blocks) the parity tests compare
    with, on every tape they use, as blake2b digests per frame and per compared field, keyed by tape and settings.

    They are computed with the oracle's line decode (STC-007) or the host build of the line decode (PCM-1, PCM-16x0, M2), the
    host build of the stitchers and the oracle's PCM-1 deinterleaver -- not by the reference itself, whose build (oracle/_ref)
    needs the reference sources, which this repository does not hold.  What ties them to the reference: where a fixture above
    holds the reference's own output for a tape, the file is checked against it here; the CUDA path, checked against the live
    reference on all of these tapes by the GPU parity tests (profiles/r2_gputest_full.log, 127 passed), must reproduce every
    entry; and where oracle/_ref is present, every entry is checked against a live run of the reference before it is written."""
    import json
    from concurrent.futures import ProcessPoolExecutor
    from tests import util
    from tests.test_stc007_stitch import stitch_cases, pair_arrays
    from tests.test_pcm16x0_stitch import ei_cases
    util.build_hostemu()
    runs = _stream_runs()
    with ProcessPoolExecutor() as ex:
        out = dict(ex.map(_stream, runs))
    if R.available():
        # every entry against a live run of the reference build
        for run in runs:
            key = util.tape_key(*run)
            chunk = {k: v["chunk"] for k, v in out[key].items()} if run[0] == "stc007" else out[key]["chunk"]
            live = _live_reference(run, chunk)
            strip = lambda e: {k: v for k, v in e.items() if k != "arrays"}      # noqa: E731
            live = {k: strip(v) for k, v in live.items()} if run[0] == "stc007" else strip(live)
            assert live == out[key], (run[0], run[2])
        print("every stream equals the live reference run")
    g = np.load(os.path.join(HERE, "stc007_stitch.npz"))
    for name in ("heavy", "vertical_jitter_heavy"):
        luma, std, order, res, p, q = stitch_cases()[name]
        ref = np.stack([g[name + "_l"], g[name + "_r"]], axis=1), np.stack([g[name + "_fl"] & 7, g[name + "_fr"] & 7], axis=1)
        assert out[util.tape_key("stc007", luma, (std, order, res, p, q, 0))]["pairs"]["digests"] == util.chunk_digests(ref, 3 * 588), name
    g = np.load(os.path.join(HERE, "pcm16x0_ei_stitch.npz"))
    for name in ("variantB", "shift-60"):
        for i, (bff, p_corr) in enumerate(((False, True), (True, True), (False, False))):
            ref = [g[f"{name}_smp{i}"], g[f"{name}_fl{i}"]]
            assert out[util.tape_key("pcm16x0", ei_cases()[name], (bff, p_corr, True))]["digests"] == util.chunk_digests(ref, 490), name
    with open(util.REF_STREAMS, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")


def main():
    if sys.argv[1:] == ["streams"]:
        return streams_golden()
    assert R.available(), "build oracle/_ref first (make -C oracle ref)"
    if sys.argv[1:] == ["stitch"]:
        return stitch_golden()
    if sys.argv[1:] == ["ei"]:
        return ei_stitch_golden()
    stitch_golden()
    ei_stitch_golden()
    # ---- pipeline
    n_frames, seed = 8, 1234
    tape = synth.make_stc007(n_frames, seed=seed)
    cfg = R.StitchCfg(video_std=1, field_order=1, resolution=1, p_corr=1, q_corr=1, cwd=0)
    pairs, _, _ = R.pipeline_run(R.TYPE_STC007, R.MODE_NORMAL, tape["luma"], cfg, taps=False)
    p = pairs[pairs["service_type"] == 0]
    np.savez_compressed(os.path.join(HERE, "stc007_pipeline_pal.npz"), n_frames=n_frames, seed=seed, first_pair=0,
                        l=p["l"], r=p["r"], flags_l=p["flags_l"], flags_r=p["flags_r"])
    # ---- line records
    for name, luma, mode in (("clean", synth.make_stc007(3, seed=11)["luma"], R.MODE_NORMAL),
                             ("damaged", synth.damage_stc007(synth.make_stc007(2, seed=12)["luma"], seed=4567), R.MODE_NORMAL)):
        r = R.v2d_run(R.TYPE_STC007, mode, luma)
        r = r[(r["service_type"] == 0) | (r["service_type"] == 7)]
        np.savez_compressed(os.path.join(HERE, f"stc007_lines_{name}.npz"), recs=r.view(np.uint8).reshape(len(r), -1), mode=mode)
    # ---- deinterleaver
    out = {}
    lines = _random_lines(2500, seed=321, p_bad=0.06, burst=True)
    out["words"] = lines["words"][:, :8]
    out["crc_ok"] = (lines["flags"] & 3).astype(np.uint8)
    for res_mode in range(4):
        b = R.deint_stc007(out["words"], out["crc_ok"], res_mode, False, True, True, True)
        out[f"blocks_{res_mode}"] = b.view(np.uint8).reshape(len(b), -1)
    np.savez_compressed(os.path.join(HERE, "stc007_deint.npz"), **out)
    # ---- PCM-1 deinterleaver
    from tests.test_pcm1 import make_sublines
    lr, flags = make_sublines(6, seed=123, p_bad=0.004)
    out = {"lr": lr, "flags": flags}
    for ign in (0, 1):
        smp, sfl = R.deint_pcm1(lr, flags, ign)
        out[f"samples_{ign}"], out[f"sflags_{ign}"] = smp, sfl
    np.savez_compressed(os.path.join(HERE, "pcm1_deint.npz"), **out)
    # ---- PCM-16x0 deinterleaver (SI)
    from tests.test_pcm16x0 import make_sublines as make16, SETTINGS
    w, fl, pl = make16(24, seed=456, p_bad=0.06, p_pick=0.08)
    out = {"words": w, "flags": fl, "picked_left": pl}
    for k, (ign, force, pc) in enumerate(SETTINGS):
        smp, sfl, st = R.deint_pcm16x0(w, fl, pl, ign, force, pc)
        out[f"samples_{k}"], out[f"sflags_{k}"], out[f"states_{k}"] = smp, sfl, st
    np.savez_compressed(os.path.join(HERE, "pcm16x0_deint.npz"), **out)
    # ---- PCM-16x0 deinterleaver, EI format
    from tests.test_pcm16x0 import make_sublines_ei, SETTINGS as X0_SETTINGS
    w, fl, pl = make_sublines_ei(2, 60, p_bad=0.08, p_pick=0.08)
    out = dict(words=w, flags=fl, picked_left=pl)
    for k, (ign, force, p) in enumerate(X0_SETTINGS):
        out[f"samples_{k}"], out[f"sflags_{k}"], out[f"states_{k}"] = R.deint_pcm16x0(w, fl, pl, ign, force, p, ei=True)
    np.savez_compressed(os.path.join(HERE, "pcm16x0_deint_ei.npz"), **out)
    # ---- STC-007 seam padding sweep (tryPadding)
    from tests.test_seam_sweep import fields, CASES
    out = {}
    for i, (lost, p_bad, nl, sil) in enumerate(CASES):
        f1, ok1, f2, ok2 = fields(i, lost, p_bad, nl, sil)
        for j, pq in enumerate(((1, 1), (1, 0), (0, 0))):
            out[f"stats_{i}_{j}"] = R.try_padding(f1, ok1, f2, ok2, 32, *pq)
    np.savez_compressed(os.path.join(HERE, "stc007_try_padding.npz"), **out)
    # ---- STC-007 seam padding decision (findPadding)
    from tests.test_seam_sweep import find_cases, FIND_SETTINGS
    res = np.zeros((len(find_cases()), len(FIND_SETTINGS), 3), dtype=np.uint16)
    for i, c in enumerate(find_cases()):
        for j, (std, r16, pq) in enumerate(FIND_SETTINGS):
            res[i, j] = R.find_padding(*c, std, r16, *pq)
    np.savez_compressed(os.path.join(HERE, "stc007_find_padding.npz"), res=res)
    # ---- PCM-16x0 control-bit decisions per frame
    from tests.test_pcm16x0_stitch import info_cases, ref_frame_info
    np.savez_compressed(os.path.join(HERE, "pcm16x0_frame_info.npz"), **{k: ref_frame_info(v) for k, v in info_cases().items()})
    # ---- PCM-1 line decode + stitcher
    from tests.test_pcm1_line import pcm1_cases, ref_lines, ref_samples
    from tests.util import lines_from_oracle
    import tests.util as U
    cases = pcm1_cases()
    out = {}
    for name in ("clean", "header", "damaged", "cutboth"):
        luma = cases[name]
        ref = ref_lines(luma, 2, True)
        r = lines_from_oracle(ref)
        r["flags"] = ref["flags"] & ~np.uint16(1 << 11)
        out[name + "_recs"] = r.view(np.uint8).reshape(len(r), -1)
        out[name + "_samples"], out[name + "_sflags"] = ref_samples(luma, 2, False)
    np.savez_compressed(os.path.join(HERE, "pcm1_lines.npz"), **out)
    # ---- PCM-16x0 line decode (three sub-line records per video line)
    from tests.test_pcm16x0_line import pcm16x0_cases, ref_sublines
    cases = pcm16x0_cases()
    out = {}
    for name in ("clean", "damaged", "cutboth", "drift"):
        ref = ref_sublines(cases[name], 2, True)
        r = lines_from_oracle(U.x0_ref_to_product(ref))
        r["flags"] = ref["flags"]
        r["reserved"] = ref["line_part"]
        out[name + "_recs"] = r.view(np.uint8).reshape(len(r), -1)
    np.savez_compressed(os.path.join(HERE, "pcm16x0_lines.npz"), **out)
    print("golden fixtures written")


if __name__ == "__main__":
    main()
