"""The own-alignment stitcher (sdv_stc007_stitch_frames) split over frame shards by sharding.stitch_shard, with several handles on
one GPU as ranks (LocalTransport): every sharded run must equal one call over the same records byte for byte -- samples, flags,
block records, and the per-frame summaries with `start` moved by the shard's offset -- and the state blob must round-trip
between handles and be canonical.  Needs a GPU."""
import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from sdvpcmdecoder_b200.capi import BLOCK_REC
from tests.test_stc007_stitch import stitch_cases, resolution_cases, HEAVY
from tests.test_gpu_stc007_stitch import config4_tape, two_shard_tape, cwd_config4_tape, ntsc16_tape, CONFIG4_SEEDS

pytestmark = pytest.mark.gpu
MAX_WORLD = 5


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators, sharding
    assert torch.cuda.is_available()
    return [capi.Handle(0) for _ in range(MAX_WORLD + 1)], operators, sharding, torch


def _stitcher(ops, h, order, res, p=1, q=1, cwd=False):
    st = ops.STC007DataStitcher(h)
    st.setFieldOrder(order); st.setResolutionPreset({0: None, 1: False, 2: True}[res]); st.setPCorrection(bool(p)); st.setQCorrection(bool(q))
    st.setCWDCorrection(cwd)
    return st


def _host(ops, out):
    b, s, f, i = out
    return ops.records_to_numpy(b, BLOCK_REC), s.cpu().numpy(), f.cpu().numpy(), i.copy()


def _records(ctx, luma):
    handles, ops, _, torch = ctx
    return ops.VideoToDigital(handles[0]).doBinarize(torch.from_numpy(np.ascontiguousarray(luma)).cuda())


def _whole(ctx, recs, n, H, std, settings):
    handles, ops, _, torch = ctx
    out = _stitcher(ops, handles[MAX_WORLD], **settings).doFrameReassembleAuto(recs, n, H, want_blocks=True, video_std=std)
    torch.cuda.synchronize()
    return _host(ops, out)


def _sharded(ctx, recs, n, H, std, settings, edges, warmup=None):
    """stitch_shard on len(edges)-1 ranks; returns the concatenated output and every rank's stats."""
    handles, ops, sharding, torch = ctx
    world = len(edges) - 1
    kw = {} if warmup is None else {"warmup": warmup}

    def rank_fn(tr):
        a, b = edges[tr.rank], edges[tr.rank + 1]
        st = _stitcher(ops, handles[tr.rank], **settings)
        out, stats = sharding.stitch_shard(st, recs[a * H:b * H], n, H, tr, edges=edges, want_blocks=True, video_std=std, **kw)
        torch.cuda.synchronize()
        return _host(ops, out), stats
    res = sharding.LocalTransport(world).run(rank_fn)
    parts, stats = [r[0] for r in res], [r[1] for r in res]
    off = 0
    for _, s, _, i in parts:
        i["start"] += off
        off += s.shape[0]
    cat = tuple(np.concatenate([p[k] for p in parts]) for k in range(4))
    return cat, stats


def _assert_equal(got, want, what=""):
    for k, name in enumerate(("blocks", "samples", "flags", "info")):
        assert got[k].shape == want[k].shape and np.array_equal(got[k], want[k]), f"{what}: {name} differ"


def _edges(n, world):
    return [n * g // world for g in range(world)] + [n]


def _check(ctx, luma, std, settings, layouts, what=""):
    """layouts: (edges, warmup) pairs; returns the stats of every run."""
    recs = _records(ctx, luma)
    n, H = luma.shape[0], luma.shape[1]
    want = _whole(ctx, recs, n, H, std, settings)
    out = []
    for edges, warmup in layouts:
        got, stats = _sharded(ctx, recs, n, H, std, settings, edges, warmup)
        _assert_equal(got, want, f"{what} edges={edges} warmup={warmup}")
        assert len(stats[0]["rounds"]) <= len(edges) - 1
        out.append(stats)
    return out


@pytest.mark.parametrize("name", sorted(stitch_cases()))
def test_stitch_cases_in_shards(ctx, name):
    """Every stitcher test tape with its settings (order and standard detection included): 2, 3 and 5 shards (1-frame shards at 5)
    at the default warm-up, and 3 shards with a 1-frame warm-up, which guesses and has to verify."""
    luma, std, order, res, p, q = stitch_cases()[name]
    n = luma.shape[0]
    _check(ctx, luma, std, dict(order=order, res=res, p=p, q=q),
           [(_edges(n, 2), None), (_edges(n, 3), None), (_edges(n, 5), None), (_edges(n, 3), 1)], name)


def test_detected_resolution_in_shards(ctx):
    for name, luma in sorted(resolution_cases().items()):
        n = luma.shape[0]
        _check(ctx, luma, 1, dict(order=1, res=0), [(_edges(n, 2), None), (_edges(n, 3), 1)], name)
    n16 = ntsc16_tape()
    _check(ctx, n16, 0, dict(order=0, res=0), [(_edges(6, 2), 1), (_edges(6, 4), 2)], "ntsc16 detect all")


@pytest.mark.parametrize("seed", CONFIG4_SEEDS)
@pytest.mark.parametrize("cwd", [False, True])
def test_config4_in_random_shards(ctx, seed, cwd):
    """24 damaged frames, CWD off and on: 2-5 shards at random cuts, shards shorter than the warm-up, warm-ups of 3 frames."""
    rng = np.random.default_rng(seed + 17 * cwd)
    layouts = []
    for world in (2, 3, 4, 5):
        cuts = sorted(rng.choice(np.arange(1, 24), size=world - 1, replace=False).tolist())
        layouts.append(([0] + cuts + [24], None))
        layouts.append(([0] + cuts + [24], 3))
    _check(ctx, config4_tape(seed), 1, dict(order=1, res=1, cwd=cwd), layouts, f"seed {seed} cwd {cwd}")


def test_cwd_cut_inside_dirty_chains(ctx):
    """Every cut of the CWD config-4 tape into two shards, so that some fall inside a chain of frames CWD patched: the patched lines
    in the queue travel in the state blob."""
    luma = cwd_config4_tape()
    recs = _records(ctx, luma)
    settings = dict(order=1, res=1, cwd=True)
    want = _whole(ctx, recs, 24, 576, 1, settings)
    assert (want[0]["flags"] & capi.BF_CWD).any()
    for cut in range(1, 24):
        for warmup in (None, 2):
            got, _ = _sharded(ctx, recs, 24, 576, 1, settings, [0, cut, 24], warmup)
            _assert_equal(got, want, f"cut {cut} warmup {warmup}")


def test_countdown_window_across_the_cut(ctx):
    """The BROKEN blocks at the end of shard 0 open a window that reaches into shard 1: the countdown is part of the state."""
    luma = two_shard_tape()
    settings = dict(order=1, res=1)
    _check(ctx, luma, 1, settings, [(_edges(12, 2), None), (_edges(12, 2), 2), (_edges(12, 3), 2)], "two_shard_tape")


def test_short_warmup_redoes_and_stays_exact(ctx):
    """Order detection and vertical shifts with a 2-frame warm-up: the guessed histories are short of entries, so a rank redoes
    at least once, and the output is still exact."""
    t = synth.make_stc007(16, seed=451)["luma"]
    from tests.test_stc007_stitch import shift_rows
    jit = t.copy()
    for f in range(16):
        jit[f] = shift_rows(t[f:f + 1], (0, 2, -2, 4)[f % 4])[0]
    luma = synth.damage_stc007(jit, seed=452, **HEAVY)
    stats = _check(ctx, luma, 0, dict(order=0, res=1), [(_edges(16, 4), 2), (_edges(16, 3), 2)], "shifted, order detected")
    for run in stats:
        assert run[0]["rounds"], "a wrong guess was expected"
        assert sum(s["redone"] for s in run) >= 1


def test_clean_tape_verifies_on_the_first_round(ctx):
    """A clean tape at the default warm-up: no redo -- on 60 frames in 4 shards, and where the warm-up really guesses (shard 1
    starting at frame 80 of 100, field order detected, so the 65-entry order history must match after rotation)."""
    luma = synth.make_stc007(60, seed=433)["luma"]
    for stats in _check(ctx, luma, 1, dict(order=1, res=1), [(_edges(60, 4), None)], "clean 60"):
        assert stats[0]["rounds"] == [] and all(s["redone"] == 0 for s in stats)
    luma = synth.make_stc007(100, seed=434)["luma"]
    for stats in _check(ctx, luma, 1, dict(order=0, res=1), [([0, 80, 100], None)], "clean 100"):
        assert stats[1]["warmup_frames"] == 70
        assert stats[0]["rounds"] == [] and all(s["redone"] == 0 for s in stats)


def test_save_load_continues_on_another_handle(ctx):
    """The batches of test_batches_continue_the_file: after every batch, the state saved on handle A and loaded into a fresh
    handle B lets B continue exactly as A does."""
    handles, ops, _, torch = ctx
    luma = synth.damage_stc007(synth.make_stc007(9, seed=431)["luma"], seed=432, **HEAVY)
    recs = _records(ctx, luma)
    H = luma.shape[1]
    cuts = [0, 3, 4, 7, 9]
    for cwd in (False, True):
        want = _whole(ctx, recs, 9, H, 1, dict(order=1, res=1, cwd=cwd))
        for switch in range(1, len(cuts) - 1):        # batches [0, switch) on A, the rest on B
            parts = []
            for i in range(len(cuts) - 1):
                a, b = cuts[i], cuts[i + 1]
                last = b == 9
                hi = b if last else b + 1
                st = _stitcher(ops, handles[0 if i < switch else 1], order=1, res=1, cwd=cwd)
                if i == switch:
                    blob = _stitcher(ops, handles[0], order=1, res=1, cwd=cwd).saveState()
                    handles[1].close(); handles[1] = capi.Handle(0)
                    st = _stitcher(ops, handles[1], order=1, res=1, cwd=cwd)
                    st.loadState(blob)
                parts.append(_host(ops, st.doFrameReassembleAuto(recs[a * H:hi * H], hi - a, H, want_blocks=True, video_std=1,
                                                                 file_start=(a == 0), file_end=last)))
            off = 0
            for p in parts:
                p[3]["start"] += off
                off += p[1].shape[0]
            _assert_equal(tuple(np.concatenate([p[k] for p in parts]) for k in range(4)), want, f"switch {switch} cwd {cwd}")


def test_equal_states_save_to_equal_bytes(ctx):
    """Frames [0, 80) and frames [5, 80) of a clean tape, field order detected, from a file start each: the same state at frame 80
    (the 65-entry order history full of the same order, its ring at different positions), so the same bytes."""
    handles, ops, _, torch = ctx
    luma = synth.make_stc007(81, seed=435)["luma"]
    recs = _records(ctx, luma)
    H = luma.shape[1]
    blobs = []
    for first in (0, 5):
        st = _stitcher(ops, handles[0], order=0, res=1)
        st.doFrameReassembleAuto(recs[first * H:81 * H], 81 - first, H, video_std=1, file_end=False)
        blobs.append(st.saveState().clone())
    torch.cuda.synchronize()
    assert blobs[0].numel() == int(capi.lib().sdv_stc007_stitch_state_bytes())
    assert torch.equal(blobs[0], blobs[1])


def test_bad_blobs_and_settings_are_refused(ctx):
    handles, ops, _, torch = ctx
    luma = cwd_config4_tape()[:6]
    recs = _records(ctx, luma)
    H = luma.shape[1]
    st = _stitcher(ops, handles[0], order=1, res=1, cwd=True)
    st.doFrameReassembleAuto(recs[:4 * H], 4, H, video_std=1, file_end=False)
    blob = st.saveState().clone()
    bad = blob.clone()
    bad[0] ^= 0xFF
    b = _stitcher(ops, handles[1], order=1, res=1, cwd=True)
    with pytest.raises(capi.SdvError):
        b.loadState(bad)
    # saved with CWD on, continued with CWD off
    b.loadState(blob)
    off = _stitcher(ops, handles[1], order=1, res=1, cwd=False)
    with pytest.raises(capi.SdvError):
        off.doFrameReassembleAuto(recs[3 * H:6 * H], 3, H, video_std=1, file_start=False)
    # ... and with resolution detection on
    b.loadState(blob)
    det = _stitcher(ops, handles[1], order=1, res=0, cwd=True)
    with pytest.raises(capi.SdvError):
        det.doFrameReassembleAuto(recs[3 * H:6 * H], 3, H, video_std=1, file_start=False)
    # the matching settings continue; after a file end there is nothing to save
    b.loadState(blob)
    b.doFrameReassembleAuto(recs[3 * H:6 * H], 3, H, video_std=1, file_start=False)
    with pytest.raises(capi.SdvError):
        b.saveState()


def test_sharded_decode_and_stitch_end_to_end(ctx):
    """A clean tape: every rank decodes its own frames (its line-decode chain starting empty) and the shards stitch with the
    protocol; the result equals the unsharded decode + one stitch call."""
    handles, ops, sharding, torch = ctx
    luma = synth.make_stc007(24, seed=436)["luma"]
    n, H = luma.shape[0], luma.shape[1]
    settings = dict(order=0, res=1, cwd=True)
    want = _whole(ctx, _records(ctx, luma), n, H, 0, settings)
    for world, warmup in ((3, None), (4, 2)):
        edges = _edges(n, world)

        def rank_fn(tr):
            a, b = edges[tr.rank], edges[tr.rank + 1]
            h = handles[tr.rank]
            recs = ops.VideoToDigital(h).doBinarize(torch.from_numpy(np.ascontiguousarray(luma[a:b])).cuda())
            kw = {} if warmup is None else {"warmup": warmup}
            out, stats = sharding.stitch_shard(_stitcher(ops, h, **settings), recs, n, H, tr, edges=edges, want_blocks=True, video_std=0, **kw)
            torch.cuda.synchronize()
            return _host(ops, out)
        parts = sharding.LocalTransport(world).run(rank_fn)
        off = 0
        for p in parts:
            p[3]["start"] += off
            off += p[1].shape[0]
        _assert_equal(tuple(np.concatenate([p[k] for p in parts]) for k in range(4)), want, f"world {world}")
