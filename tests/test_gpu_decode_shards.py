"""The line-decode chain state as a blob (sdv_bin_chain_state_save / _load, VideoToDigital.saveState / loadState) and the exact
sharded line decode built on it (sharding.decode_shard), in all four formats: a decode handed from one handle to another mid-tape,
and a tape decoded in 2-5 shards (several handles on one GPU as ranks, LocalTransport), must give the records and aux of one call
byte for byte -- the Tier-B fields at the shard heads included; the blob must be canonical; bad blobs and mismatched calls are
refused.  Needs a GPU."""
import numpy as np
import pytest

from sdvpcmdecoder_b200 import synth, capi
from tests import test_gpu_pcm1_line as p1_tapes
from tests import test_gpu_pcm16x0_line as x0_tapes
from tests.test_m2 import m2_tapes
from tests.test_gpu_stc007_stitch import config4_tape

pytestmark = pytest.mark.gpu
STC, M2, P1, X0 = "stc007", "m2", "pcm1", "pcm16x0"
TYPE = {STC: capi.TYPE_STC007, M2: capi.TYPE_M2, P1: capi.TYPE_PCM1, X0: capi.TYPE_PCM16X0}
FORMATS = (STC, M2, P1, X0)
MAX_WORLD = 5


@pytest.fixture(scope="module")
def ctx():
    import torch
    from sdvpcmdecoder_b200 import operators, sharding
    assert torch.cuda.is_available()
    return [capi.Handle(0) for _ in range(MAX_WORLD + 1)], operators, sharding, torch


def _v2d(ops, h, fmt, mode=2, dup=True, warm=True, relay=True):
    v = ops.VideoToDigital(h)
    v.setPCMType(TYPE[fmt]); v.setBinarizationMode(mode); v.setCheckLineDup(dup)
    v.warm_start, v.relay = warm, relay
    return v


def _dev(torch, luma):
    return torch.from_numpy(np.ascontiguousarray(luma)).cuda()


def _sparse_stc(n=12):
    luma = synth.make_stc007(n, seed=71)["luma"].copy()
    for f in (3, 7):
        luma[f, 200:203] = synth.damage_stc007(luma[f:f + 1, 200:203].copy(), seed=f, jitter=True)[0]
    return luma


def relay_tape():
    """Config-4 damage over 48 frames: one call goes into relay mode after two frames (32 frames or more left)."""
    return synth.damage_stc007(synth.make_stc007(48, seed=571)["luma"], seed=4567)


def tapes(fmt):
    if fmt == STC:
        return {"clean": synth.make_stc007(12, seed=70)["luma"], "sparse": _sparse_stc(), "config4": config4_tape(4567)}
    if fmt == M2:
        quiet = synth.make_stc007(10, seed=5, quiet_frac=0.3)["luma"]
        return {"clean": quiet, "sparse": _sparse_stc(10), "damaged": m2_tapes()["quiet_damaged"]}
    mod = p1_tapes if fmt == P1 else x0_tapes
    return {"clean": mod.clean_tape(), "sparse": mod.sparse_tape(), "damaged": synth.damage_stc007(mod.clean_tape(), seed=4567)}


def _host(torch, out):
    recs, aux = out
    torch.cuda.synchronize()
    return recs.cpu().numpy().copy(), aux.cpu().numpy().copy()


def one_call(ctx, fmt, luma, **kw):
    handles, ops, _, torch = ctx
    return _host(torch, _v2d(ops, handles[MAX_WORLD], fmt, **kw).doBinarize(_dev(torch, luma), want_aux=True))


def _equal(got, want, what):
    assert got[0].shape == want[0].shape and np.array_equal(got[0], want[0]), f"{what}: records differ"
    assert np.array_equal(got[1], want[1]), f"{what}: aux differ"


def _fresh(ctx, i):
    handles = ctx[0]
    handles[i].close()
    handles[i] = capi.Handle(0)
    return handles[i]


# ---- hand-over between handles
@pytest.mark.parametrize("fmt", FORMATS)
def test_handover_between_handles(ctx, fmt):
    """[0, k) on handle A, save, load on a fresh handle B (and on a second device when there is one), [k, n) on B: one call."""
    handles, ops, _, torch = ctx
    devices = [0] + ([1] if torch.cuda.device_count() > 1 else [])
    for name, luma in tapes(fmt).items():
        n = luma.shape[0]
        want = one_call(ctx, fmt, luma)
        for k in sorted({1, n // 2, n - 1}):
            for dev in devices:
                a = _v2d(ops, _fresh(ctx, 0), fmt)
                ra = a.doBinarize(_dev(torch, luma[:k]), want_aux=True)
                blob = a.saveState()
                hb = capi.Handle(dev) if dev else _fresh(ctx, 1)
                b = _v2d(ops, hb, fmt)
                with torch.cuda.device(dev):
                    b.loadState(blob.to(f"cuda:{dev}"))
                    rb = b.doBinarize(_dev(torch, luma[k:]).to(f"cuda:{dev}"), want_aux=True, continue_file=True)
                    torch.cuda.synchronize()
                if name == "clean" and fmt in (P1, X0):      # the running pair G derived on load: still all on the bulk pass
                    assert b.stats()["frames_skipped"] == n - k, (fmt, k, b.stats())
                ha, hb_ = _host(torch, ra), _host(torch, rb)
                _equal((np.concatenate([ha[0], hb_[0]]), np.concatenate([ha[1], hb_[1]])), want, f"{fmt} {name} k={k} dev={dev}")
                if dev:
                    hb.close()


def test_handover_inside_the_relay_span(ctx):
    """A config-4 tape long enough for relay mode: the cuts fall inside the span one call decodes in relay mode, and A's own call
    relays too (cut at 36); relay on and off on either side."""
    handles, ops, _, torch = ctx
    luma = relay_tape()
    want = one_call(ctx, STC, luma)
    assert np.array_equal(want[0], one_call(ctx, STC, luma, relay=False)[0])
    for k in (20, 36):
        for relay in (True, False):
            a = _v2d(ops, _fresh(ctx, 0), STC, relay=relay)
            ra = _host(torch, a.doBinarize(_dev(torch, luma[:k]), want_aux=True))
            b = _v2d(ops, _fresh(ctx, 1), STC, relay=not relay)
            b.loadState(a.saveState())
            rb = _host(torch, b.doBinarize(_dev(torch, luma[k:]), want_aux=True, continue_file=True))
            _equal((np.concatenate([ra[0], rb[0]]), np.concatenate([ra[1], rb[1]])), want, f"k={k} relay={relay}")


# ---- canonical bytes
def _blob_after(ctx, fmt, luma, cuts=(), warm=True, relay=True, warm_first=False, round_trip=False):
    handles, ops, _, torch = ctx
    v = _v2d(ops, _fresh(ctx, 0), fmt, warm=warm, relay=relay)
    if warm_first:
        v.doBinarize(_dev(torch, luma))                # the handle now holds warm-start presets for the next fresh call
    edges = [0] + list(cuts) + [luma.shape[0]]
    for i in range(len(edges) - 1):
        v.doBinarize(_dev(torch, luma[edges[i]:edges[i + 1]]), continue_file=i > 0)
    blob = v.saveState().clone()
    if round_trip:
        w = _v2d(ops, _fresh(ctx, 1), fmt)
        w.loadState(blob)
        blob = w.saveState().clone()
    torch.cuda.synchronize()
    return blob.cpu().numpy()


@pytest.mark.parametrize("fmt", FORMATS)
def test_equal_states_save_to_equal_bytes(ctx, fmt):
    """The blob after [0, k): one call, random batches, warm start on / off, relay on / off, save -> load -> save."""
    rng = np.random.default_rng(len(fmt))
    for name, luma in tapes(fmt).items():
        n = luma.shape[0]
        for k in sorted({n // 2, n}):
            want = _blob_after(ctx, fmt, luma[:k])
            assert want.size == int(capi.lib().sdv_bin_chain_state_bytes())
            variants = {"warm": dict(warm_first=True), "cold": dict(warm=False), "no relay": dict(relay=False),
                        "round trip": dict(round_trip=True)}
            if k > 1:
                variants["batches"] = dict(cuts=sorted(rng.choice(np.arange(1, k), size=min(3, k - 1), replace=False).tolist()))
                variants["1-frame batches"] = dict(cuts=list(range(1, k)))
            for what, kw in variants.items():
                assert np.array_equal(_blob_after(ctx, fmt, luma[:k], **kw), want), f"{fmt} {name} k={k}: {what}"
    if fmt == STC:
        luma = relay_tape()
        want = _blob_after(ctx, fmt, luma)
        assert np.array_equal(_blob_after(ctx, fmt, luma, relay=False), want)
        assert np.array_equal(_blob_after(ctx, fmt, luma, cuts=[20, 36]), want)


# ---- refusals
def test_refused_calls(ctx):
    handles, ops, _, torch = ctx
    luma = synth.make_stc007(4, seed=72)["luma"]
    dev = _dev(torch, luma)
    # nothing open of that kind
    v = _v2d(ops, _fresh(ctx, 0), STC)
    with pytest.raises(capi.SdvError):
        v.saveState()
    v.doBinarize(dev)
    for t in (capi.TYPE_PCM1, capi.TYPE_PCM16X0, capi.TYPE_M2):
        with pytest.raises(capi.SdvError):
            v.saveState(pcm_type=t)
    blob = v.saveState().clone()
    # a lazy call awaiting verification
    v.doBinarize(dev, lazy=True)
    with pytest.raises(capi.SdvError):
        v.saveState()
    with pytest.raises(capi.SdvError):
        v.loadState(blob)
    assert v.verify() is False
    v.saveState()
    # bad blobs: magic, version, size, type, mode, duplicate check, field state, history count, per-frame count, Binarizer mode,
    # unused bytes in the state, behind it and in the header, a history entry past its count
    b = _v2d(ops, _fresh(ctx, 1), STC)
    for at, val in ((0, 0x00), (4, 0x7F), (8, 0x01), (6, 0x09), (16, 0x09), (17, 0x02), (76, 0x09), (80, 0x63), (88, 0x01),
                    (67, 0x01), (400, 0x01), (114, 0x01), (20, 0x01)):
        bad = blob.clone()
        bad[at] = val if int(bad[at]) != val else (val ^ 0x10)
        with pytest.raises(capi.SdvError):
            b.loadState(bad)
    n_last = int(blob[80:84].cpu().numpy().view(np.int32)[0])
    if n_last < 9:
        bad = blob.clone()
        bad[120 + 4 * n_last] = 1
        with pytest.raises(capi.SdvError):
            b.loadState(bad)
    # other fine settings on the loading handle
    b.setFineSettings(min_valid_crcs=3)
    with pytest.raises(capi.SdvError):
        b.loadState(blob)
    b.setDefaultFineSettings()
    # a continuing call with another H, W, mode, duplicate check or type after a load
    for what, lum, kw in (("H", luma[:, :-2], {}), ("W", luma[:, :, :-2], {}), ("mode", luma, dict(mode=1)),
                          ("dup", luma, dict(dup=False)), ("type", luma, dict(fmt=M2))):
        b.loadState(blob)
        c = _v2d(ops, b.handle, kw.pop("fmt", STC), **kw)
        with pytest.raises(capi.SdvError):
            c.doBinarize(_dev(torch, lum), continue_file=True)
    b.loadState(blob)
    b.doBinarize(dev, continue_file=True)
    # the PCM kinds are refused in the same way
    p = _v2d(ops, _fresh(ctx, 2), P1)
    with pytest.raises(capi.SdvError):
        p.saveState()
    pl = p1_tapes.clean_tape()[:3]
    p.doBinarize(_dev(torch, pl))
    pblob = p.saveState().clone()
    with pytest.raises(capi.SdvError):
        p.saveState(pcm_type=capi.TYPE_PCM16X0)
    q = _v2d(ops, _fresh(ctx, 3), X0)
    q.loadState(pblob)
    with pytest.raises(capi.SdvError):
        q.doBinarize(_dev(torch, pl), continue_file=True)      # the open PCM file is a PCM-1 one


# ---- sharded
def sharded(ctx, fmt, luma, edges, warmup=None, **kw):
    handles, ops, sharding, torch = ctx
    world = len(edges) - 1
    wk = {} if warmup is None else {"warmup": warmup}

    def fn(tr):
        a, b = edges[tr.rank], edges[tr.rank + 1]
        v = _v2d(ops, handles[tr.rank], fmt, **kw)
        out, stats = sharding.decode_shard(v, _dev(torch, luma[a:b]), tr, edges=edges, want_aux=True, **wk)
        stats["last_call"] = v.stats()
        return _host(torch, out), stats
    res = sharding.LocalTransport(world).run(fn)
    got = (np.concatenate([r[0][0] for r in res]), np.concatenate([r[0][1] for r in res]))
    return got, [r[1] for r in res]


def _layouts(n, rng):
    out = []
    for world in (2, 3, 4, 5):
        if world > n:
            continue
        cuts = sorted(rng.choice(np.arange(1, n), size=world - 1, replace=False).tolist())
        out.append(([0] + cuts + [n], None))
        out.append(([0] + cuts + [n], 1))
    if n >= 5:
        out.append(([0, 1, 2, 3, 4, n], 2))            # 1-frame shards, shorter than the warm-up
    return out


@pytest.mark.parametrize("fmt", FORMATS)
def test_sharded_decode_equals_one_call(ctx, fmt):
    """2-5 shards at random cuts, 1-frame shards, shards shorter than the warm-up, and 1-frame warm-ups (forced guesses)."""
    rng = np.random.default_rng(17 + len(fmt))
    for name, luma in tapes(fmt).items():
        want = one_call(ctx, fmt, luma)
        for edges, warmup in _layouts(luma.shape[0], rng):
            got, stats = sharded(ctx, fmt, luma, edges, warmup)
            _equal(got, want, f"{fmt} {name} edges={edges} warmup={warmup}")
            assert len(stats[0]["rounds"]) <= len(edges) - 1


@pytest.mark.parametrize("fmt", FORMATS)
def test_clean_tape_settles_at_once_on_the_bulk_pass(ctx, fmt):
    """A clean tape at the default warm-up: one gather, no redo, and every shard's continuing call served by the bulk pass
    (STC-007 / M2: all but the frames the chain decodes before it hands over)."""
    luma = tapes(fmt)["clean"]
    n = luma.shape[0]
    edges = [0, n // 3, 2 * n // 3, n]
    got, stats = sharded(ctx, fmt, luma, edges)
    _equal(got, one_call(ctx, fmt, luma), f"{fmt} clean")
    assert stats[0]["rounds"] == [] and all(s["redone"] == 0 for s in stats)
    for g in range(1, 3):
        frames = edges[g + 1] - edges[g]
        skipped = stats[g]["last_call"]["frames_skipped"]
        assert skipped >= (frames if fmt in (P1, X0) else frames - 2), (fmt, g, skipped, frames)


def test_independent_shards_differ_at_the_heads(ctx):
    """Why the hand-off exists: on a damaged tape, shards that each start an empty chain (the plain sharded decode) give other
    records at the shard heads than one call -- decode_shard gives the same."""
    handles, ops, _, torch = ctx
    fmt = STC
    luma = tapes(fmt)["config4"]
    n = luma.shape[0]
    edges = [0, n // 2, n]
    want = one_call(ctx, fmt, luma)
    plain = [_host(torch, _v2d(ops, handles[g], fmt).doBinarize(_dev(torch, luma[edges[g]:edges[g + 1]]), want_aux=True)) for g in range(2)]
    assert not np.array_equal(np.concatenate([p[0] for p in plain]), want[0])
    _equal(sharded(ctx, fmt, luma, edges)[0], want, fmt)


def test_relay_tape_in_shards(ctx):
    luma = relay_tape()
    want = one_call(ctx, STC, luma)
    for edges, warmup in (([0, 20, 48], None), ([0, 10, 30, 48], 1), ([0, 5, 25, 40, 48], 3)):
        got, _ = sharded(ctx, STC, luma, edges, warmup)
        _equal(got, want, f"edges={edges} warmup={warmup}")


# ---- end to end, STC-007
def test_end_to_end_with_deinterleave_and_stitch(ctx):
    """A damaged tape: decode_shard, then the halo (the next shard's first 112 records, final only now), then the preset-geometry
    deinterleave with ignore_crc on and the broken-block countdown handed from shard to shard (the value carry_countdowns settles
    on: each shard's input is its predecessor's output); and decode_shard -> stitch_shard with CWD on.  Both equal the unsharded
    call byte for byte."""
    handles, ops, sharding, torch = ctx
    luma = config4_tape(4568)
    n, H = luma.shape[0], luma.shape[1]
    edges = [0, 7, 15, n]
    world = len(edges) - 1
    recs_all = _v2d(ops, handles[MAX_WORLD], STC).doBinarize(_dev(torch, luma))

    def deint(h, recs, nf, halo, cd, lead_in):
        st = ops.STC007DataStitcher(h)
        st.setIgnoreCRC(True); st.setBrokenMaskDuration(128)
        st.lead_in = lead_in
        _, s, f = st.doFrameReassemble(recs, nf, H, halo=halo, countdown_in=cd)
        torch.cuda.synchronize()
        return s.cpu().numpy(), f.cpu().numpy(), st.countdown()["countdown_out"]
    want_s, want_f, _ = deint(handles[MAX_WORLD], recs_all, n, None, 0, 80)
    cw = ops.STC007DataStitcher(handles[MAX_WORLD])
    cw.setFieldOrder(1); cw.setResolutionPreset(False); cw.setCWDCorrection(True)
    want_st = [x.cpu().numpy() if hasattr(x, "cpu") else x for x in cw.doFrameReassembleAuto(recs_all, n, H, want_blocks=True, video_std=1)]

    def fn(tr):
        a, b = edges[tr.rank], edges[tr.rank + 1]
        v = _v2d(ops, handles[tr.rank], STC)
        recs, _ = sharding.decode_shard(v, _dev(torch, luma[a:b]), tr, edges=edges)
        halo = None
        if tr.rank > 0:
            tr.send(recs[:sharding.HALO_LINES], tr.rank - 1)
        if tr.rank < world - 1:
            halo = recs.new_empty((sharding.HALO_LINES, recs.shape[1]))
            tr.recv(halo, tr.rank + 1)
        st = ops.STC007DataStitcher(handles[tr.rank])
        st.setFieldOrder(1); st.setResolutionPreset(False); st.setCWDCorrection(True)
        out, _ = sharding.stitch_shard(st, recs, n, H, tr, edges=edges, want_blocks=True, video_std=1)
        torch.cuda.synchronize()
        return recs, halo, [x.cpu().numpy() if hasattr(x, "cpu") else x for x in out]
    res = sharding.LocalTransport(world).run(fn)
    parts, cd = [], 0
    for g, (recs, halo, _) in enumerate(res):
        s, f, cd = deint(handles[g], recs, edges[g + 1] - edges[g], halo, cd, sharding.shard_lead_in(g))
        parts.append((s, f))
    assert np.array_equal(np.concatenate([p[0] for p in parts]), want_s)
    assert np.array_equal(np.concatenate([p[1] for p in parts]), want_f)
    off = 0
    outs = [r[2] for r in res]
    for o in outs:
        o[3]["start"] += off
        off += o[1].shape[0]
    for k in range(4):
        assert np.array_equal(np.concatenate([o[k] for o in outs]), want_st[k]), k
