"""M2 sample format (VideoToDigital::TYPE_M2 = STC-007 lines whose samples use a range/sign expansion): the "almost silent"
rule of the duplicate-line check and the sample output change.  Device code built for the host and the GPU path against
the compiled reference (oracle/_ref)."""
import numpy as np
import pytest

from oracle import refbind as R
from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import LINE_REC, LINE_AUX
from tests import util

have_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref not built")
H, LPF = 576, 294


def m2_tapes():
    return {"quiet": synth.make_stc007(3, seed=5, quiet_frac=0.3)["luma"],
            "quiet_damaged": synth.damage_stc007(synth.make_stc007(3, seed=6, quiet_frac=0.3)["luma"], seed=9)}


def ref_lines(luma, pcm_type):
    ref = R.v2d_run(pcm_type, 2, luma)
    return ref[(ref["service_type"] == 0) | (ref["service_type"] == 7)][:luma.shape[0] * luma.shape[1]]


def ref_pairs(luma):
    cfg = R.StitchCfg(video_std=1, field_order=1, resolution=1, p_corr=1, q_corr=1, cwd=0)
    pairs, _, _ = R.pipeline_run(R.TYPE_M2, 2, luma, cfg, taps=False)
    return pairs[pairs["service_type"] == 0]


def assemble(recs, n_frames):
    hf = H // 2
    nb = 80 + n_frames * 2 * LPF
    asm = np.zeros(nb + 112, LINE_REC)
    for fld in range(2 * n_frames):
        src = (fld // 2) * H + (fld & 1) * hf
        asm[80 + fld * LPF:80 + fld * LPF + hf] = recs[src:src + hf]
    return asm


@have_ref
def test_m2_on_host_against_reference_live():
    for name, luma in m2_tapes().items():
        ref = ref_lines(luma, R.TYPE_M2)
        rec, aux, _ = util.emu_v2d(luma, 2, True, hybrid=True, m2=True)
        bad = util.compare_line_records(ref, rec, aux)
        assert not bad, (name, bad)
        assert (ref["flags"] != ref_lines(luma, R.TYPE_STC007)["flags"]).sum() > 100       # the format does change the outcome
        p = ref_pairs(luma)
        _, s, f = util.emu_deint(assemble(rec, luma.shape[0]), 0, False, True, True, True, 128, m2=True)
        s, f = s.reshape(-1, 2), f.reshape(-1, 2)
        assert len(p) == len(s)
        assert np.array_equal(p["l"], s[:, 0]) and np.array_equal(p["r"], s[:, 1]), name
        assert np.array_equal(p["flags_l"] & 7, f[:, 0]) and np.array_equal(p["flags_r"] & 7, f[:, 1]), name


@pytest.mark.gpu
def test_m2_gpu_against_reference():
    """The GPU path against the reference's line records and PCMSamplePair stream (tests/golden/reference_streams.json)."""
    import torch
    from sdvpcmdecoder_b200 import operators as ops
    h = capi.Handle(0)
    for name, luma in m2_tapes().items():
        v2d = ops.VideoToDigital(h)
        v2d.setPCMType(capi.TYPE_M2)
        recs, aux = v2d.doBinarize(torch.from_numpy(luma).cuda(), want_aux=True)
        st = ops.STC007DataStitcher(h)
        st.setM2SampleFormat(True)
        _, samples, flags = st.doFrameReassemble(recs, luma.shape[0], luma.shape[1])
        torch.cuda.synchronize()
        bad = util.lines_mismatch("m2_lines", luma, (), ops.records_to_numpy(recs, LINE_REC), ops.records_to_numpy(aux, LINE_AUX))
        assert not bad, (name, bad)
        bad = util.stream_mismatch_digests(util.golden_stream("m2", luma, ()), [samples.cpu().numpy().reshape(-1, 2), flags.cpu().numpy().reshape(-1, 2)])
        assert not bad, (name, bad)
