"""Indexed streaming pushes (wwb_stream_push_indexed, wwb_context_step_indexed): each push names a subset of the
allocated slots, in any order, each with a chunk of its own length.

The arithmetic is the dense push's, only the addressing of streams and chunks differs, so every result is checked
against paths that are already trusted: the oracle's TriggerOracle / PipelineOracle per slot, the batch path bit for
bit, the dense push bit for bit on the dense shape, and a fresh context that only ever saw one slot's pushes.

Tolerances as in test_gpu_streaming.py: 1e-3 for f32 / tc, 2e-2 for tc_fast; triggers exact outside the band around
the threshold.
"""
import os

import numpy as np
import pytest

from conftest import WEIGHTS, load_weights
from oracle import restated as R
from streaming_helpers import (MAX_CHUNK, MAX_FRAMES, MODELS, PRECISIONS, SCRIPTS, SIZES, TOL, IndexedSchedule, IPush,
                               assert_same_rows, engine, host, indexed_script, pipeline_script, run_indexed, schedule,
                               script)
from wakeword_detection_b200 import synth

_ORACLE_CACHE = {}


# ------------------------------------------------------------------------------------ the oracle's run of a script
def oracle_run(model, name):
    """per push and entry: (posteriors, trigger, post_max as the device reports it: before the reset on a fall)"""
    key = (model, name)
    if key in _ORACLE_CACHE:
        return _ORACLE_CACHE[key]
    w = load_weights(model)
    sch = script(name)
    orc = [R.TriggerOracle(w, 0.5, sch.a) for _ in range(sch.cap)]
    out = []
    for p, chunks in zip(sch.pushes, sch.chunks):
        if p.reset is not None:
            for s in np.nonzero(p.reset)[0]:
                orc[s].reset()
        res = []
        for s, chunk, sp, ac in zip(p.ids, chunks, p.speech, p.active):
            o = orc[s]
            o.active = bool(ac)
            before, pm0 = len(o.posteriors), o.post_max
            o(chunk, bool(sp))
            new = np.array(o.posteriors[before:], np.float32)
            res.append((new, bool(not ac and (new > p.threshold).any()), max([pm0] + list(new))))
        out.append(res)
    _ORACLE_CACHE[key] = out
    return out


# ------------------------------------------------------------------------------------ the scripts (no GPU)
def test_indexed_scripts_cover_the_edges():
    """every chunk size, unsorted ids, a slot absent for >= 10 pushes, a push of only the highest slot, a push of every
    slot, and one push with an entry completing max_frames frames next to one completing none"""
    for name in SCRIPTS:
        sch = script(name)
        cap = sch.cap
        assert set(SIZES) <= {int(n) for p in sch.pushes for n in p.lens}
        assert any((np.diff(p.ids) < 0).any() for p in sch.pushes)
        assert all(len(set(p.ids.tolist())) == p.ids.size for p in sch.pushes)
        named = np.array([[s in p.ids for s in range(cap)] for p in sch.pushes])
        runs = [max(len(r) for r in "".join("1" if v else "0" for v in named[:, s]).split("1")) for s in range(cap)]
        assert max(runs) >= 10
        assert any(p.ids.tolist() == [cap - 1] for p in sch.pushes)
        assert any(sorted(p.ids.tolist()) == list(range(cap)) and (np.diff(p.ids) < 0).any() for p in sch.pushes)
        both = [i for i, fr in enumerate(sch.frames) if MAX_FRAMES in fr and 0 in fr]
        assert both
        i = both[0]
        for j in (sch.frames[i].index(MAX_FRAMES), sch.frames[i].index(0)):
            assert sch.pushes[i].speech[j] and not sch.pushes[i].active[j]
        assert {0.5, 0.9} == {p.threshold for p in sch.pushes}
        assert sum(p.reset is not None for p in sch.pushes) >= 3
        assert any(not p.speech.all() for p in sch.pushes) and any(p.active.any() for p in sch.pushes)


# ------------------------------------------------------------------------------------ 1: replay against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCRIPTS))
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", MODELS)
def test_indexed_replay_vs_oracle(model, precision, name):
    """n_post exact per entry, posteriors within tolerance, NaN tail, trigger exact outside the band, post_max"""
    sch = script(name)
    exp = oracle_run(model, name)
    eng = engine(model, precision, sch.cap)
    try:
        outs = run_indexed(eng, sch)
    finally:
        eng.close()
    tol = TOL[precision]
    n_win, fired = 0, 0
    for i, (o, e) in enumerate(zip(outs, exp)):
        post, npost, trig, pmax = o
        p = sch.pushes[i]
        assert post.shape == (p.ids.size, MAX_FRAMES)
        for j, (new, want_trig, want_pm) in enumerate(e):
            where = (name, i, j, int(p.ids[j]))
            assert npost[j] == new.size, where
            assert np.isnan(post[j, new.size:]).all(), where
            if new.size:
                assert np.abs(post[j, :new.size] - new).max() <= tol, where
                n_win += new.size
            if not (new.size and np.abs(new - p.threshold).min() <= tol):
                assert trig[j] == want_trig, where
            assert abs(float(pmax[j]) - want_pm) <= tol, (where, float(pmax[j]), want_pm)
            fired += want_trig
    print("%s %s %s: %d windows checked, %d oracle triggers" % (model, precision, name, n_win, fired))
    assert n_win > 500


# ------------------------------------------------------------------------------------ 2: bit-exact vs the batch path
@pytest.mark.gpu
@pytest.mark.parametrize("a", [0.0, 0.97])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", MODELS)
def test_indexed_equals_batch_path_bitwise(model, precision, a):
    """1024 slots, each push names a random ~30 % of them in random order with ragged lengths; speech throughout, never
    active.  Slot s consumes a prefix of its row of `pcm`, so its k-th posterior must equal, bit for bit,

        posteriors(cat(zeros(L-1, 40), filter(pcm_s, a)), hop=1)[s, k]

    (a frame of the batch filter reads only samples the slot has consumed).  Every slot is checked."""
    import torch
    from wakeword_detection_b200 import _cabi
    S, n_push = 1024, 24
    r = np.random.default_rng(int(a * 100) + 41)
    pushes = []
    for _ in range(n_push):
        ids = r.permutation(S)[:int(S * 0.3)].astype(np.int32)
        pushes.append((ids, r.choice(SIZES, size=ids.size).astype(np.int32)))
    used = np.zeros(S, np.int64)
    for ids, lens in pushes:
        used[ids] += lens
    N = int(used.max())
    eng = _cabi.Engine(load_weights(model), 0, precision)
    try:
        eng.stream_alloc(S, MAX_CHUNK)
        L = eng.L
        pcm = synth.device_pcm(S, N, seed=91, device=eng.device)
        mel = eng.filter(pcm, a)
        ref = eng.posteriors(torch.cat([torch.zeros((S, L - 1, 40), device=eng.device), mel], 1), hop=1)
        ref = ref.cpu().numpy().view(np.uint32)
        flat = pcm.reshape(-1)
        cur = np.zeros(S, np.int64)
        checked = 0
        for ids, lens in pushes:
            idx = np.concatenate([s * N + np.arange(cur[s], cur[s] + n) for s, n in zip(ids, lens)])
            post, npost, _, _ = eng.stream_push_indexed(ids, flat[torch.from_numpy(idx).to(eng.device)], lens,
                                                        pre_emphasis=a)
            post, npost = post.cpu().numpy(), npost.cpu().numpy()
            for j, (s, n) in enumerate(zip(ids, lens)):
                k0, k1 = R.num_frames(cur[s]), R.num_frames(cur[s] + n)
                assert npost[j] == k1 - k0, (s, j)
                assert np.array_equal(post[j, :k1 - k0].view(np.uint32), ref[s, k0:k1]), (s, j, k0)
                assert np.isnan(post[j, k1 - k0:]).all()
                checked += k1 - k0
            cur[ids] += lens
        assert (cur > 0).all() and checked > 0
    finally:
        eng.close()


# ------------------------------------------------------------------------------------ 3: the dense shape, bit for bit
@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_indexed_identity_equals_dense_push(model, precision):
    """Context A runs the ragged pre-emphasis script of test_gpu_streaming.py with wwb_stream_push (prefix pushes,
    masked resets, falls, active stretches); context B runs it with stream_push_indexed(ids=arange(S), lengths=[n]*S).
    All four outputs of every push are identical."""
    import torch
    sch = schedule("ragged_pe")
    ea, eb = engine(model, precision, sch.cap, sch.max_chunk), engine(model, precision, sch.cap, sch.max_chunk)
    try:
        for i, (p, chunk) in enumerate(zip(sch.pushes, sch.chunks)):
            if p.reset is not None:
                ea.stream_reset(p.reset)
                eb.stream_reset(p.reset)
            S = p.n_streams
            sp, ac = p.speech[:S].astype(np.uint8), p.active[:S].astype(np.uint8)
            x = torch.from_numpy(chunk).to(ea.device)
            a = host(ea.stream_push(x, sp, ac, sch.a, p.threshold))
            b = host(eb.stream_push_indexed(np.arange(S), x.reshape(-1), [p.n] * S, sp, ac, sch.a, p.threshold))
            assert_same_rows([a], [b])
    finally:
        ea.close()
        eb.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_indexed_identity_equals_dense_context_step(model):
    """wwb_context_step against wwb_context_step_indexed(arange(S), [320]*S) on two contexts: all seven outputs of
    every step are identical.  (The script is the CRNN one of the golden pipeline run: WaveNet analyses the same
    windows but does not activate on it.)"""
    import torch
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    cfg, pcm0, raw0 = pipeline_script()
    S, nf = 5, len(raw0)
    rng = np.random.default_rng(12)
    pcm = np.stack([np.roll(pcm0, 320 * 7 * s) for s in range(S)])
    raw = np.stack([raw0] + [np.roll(raw0, 7 * s) ^ (rng.random(nf) < 0.03) for s in range(1, S)])
    pa = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, S, pre_emphasis=0.97, **cfg)
    pb = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, S, pre_emphasis=0.97, **cfg)
    acts, n_win = 0, 0
    try:
        for i in range(nf):
            x = torch.from_numpy(np.ascontiguousarray(pcm[:, i * 320:(i + 1) * 320])).to(pa.engine.device)
            a = pa.step(x, raw[:, i])
            b = pb.engine.context_step_indexed(np.arange(S), x.reshape(-1), [320] * S, raw[:, i], 0.97, pb.threshold)
            assert a.keys() == b.keys()
            for k in a:
                assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), (i, k)
            acts += int(a["is_active"].sum())
            n_win += int(a["n_post"].sum())
    finally:
        pa.close()
        pb.close()
    assert n_win > 800 and (acts > 0 or model != "CRNN")


# ------------------------------------------------------------------------------------ 4: isolation
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_indexed_slots_are_isolated(model):
    """A 64-slot context gets interleaved pushes to many slots.  For each target slot, its rows equal bit for bit those
    of a fresh context that only ever saw that slot's pushes.  Slot 2, the neighbour in memory of target 1, has a VAD
    fall (its ring is cleared) in a push that lists it as entry 1 and target 1 as entry 2."""
    cap, n_push = 64, 30
    targets = (1, 3, 40, 63)
    r = np.random.default_rng(31)
    pushes = []
    for i in range(n_push):
        others = r.choice([s for s in range(cap) if s not in targets], size=int(r.integers(1, 20)), replace=False)
        tgt = [t for t in targets if r.random() < 0.7]
        ids = np.array(list(others) + tgt, np.int32)
        r.shuffle(ids)
        lens = r.choice(SIZES, size=ids.size)
        if i == 11:                       # slot 2 fills its ring ...
            ids, lens = np.array([2, 1], np.int32), [MAX_CHUNK, 513]
        if i == 12:                       # ... and falls as entry 1, next to target 1 as entry 2
            ids, lens = np.array([7, 2, 1, 3], np.int32), r.choice(SIZES, size=4)
        speech = np.ones(ids.size, bool)
        if i in (12, 13):
            speech[ids == 2] = False
        pushes.append(IPush(ids, lens, speech, np.zeros(ids.size), 0.5))
    sch = IndexedSchedule("iso", cap, 0.97, pushes, 32)
    eng = engine(model, "tc", cap)
    try:
        outs = run_indexed(eng, sch)
    finally:
        eng.close()
    for t in targets:
        fresh = engine(model, "tc", cap)
        try:
            n_win = 0
            for i, p in enumerate(sch.pushes):
                if t not in p.ids:
                    continue
                j = int(np.nonzero(p.ids == t)[0][0])
                got = host(fresh.stream_push_indexed([t], sch.chunks[i][j], [p.lens[j]], [p.speech[j]], [p.active[j]],
                                                      sch.a, p.threshold))
                assert_same_rows([tuple(x[j:j + 1] for x in outs[i])], [got])
                n_win += int(got[1][0])
            assert n_win > 20, t
        finally:
            fresh.close()


# ------------------------------------------------------------------------------------ 5: rejected calls
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_indexed_rejections_change_nothing(model):
    """Every malformed call raises (IndexError for the state / range checks, ValueError for NULL tables or PCM), and
    the next valid push still equals a reference context's bit for bit."""
    import ctypes as C
    import torch
    from wakeword_detection_b200 import _cabi
    w = load_weights(model)
    cap = 16
    sch = indexed_script("rej", cap, 16, 0.97, 23, (0.5,))

    unalloc = _cabi.Engine(w, 0, "tc")
    filt = _cabi.Engine({k: w[k] for k in ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")}, 0, "tc")
    try:
        with pytest.raises(IndexError):
            unalloc.stream_push_indexed([0], np.zeros(160, np.int16), [160])
        filt.stream_alloc(cap, MAX_CHUNK)
        with pytest.raises(IndexError):
            filt.stream_push_indexed([0], np.zeros(160, np.int16), [160])
    finally:
        unalloc.close()
        filt.close()

    def bad_calls(eng, i):
        z = lambda n: np.zeros(n, np.int16)
        bad = [
            ([], z(0), []),                                     # n_ids = 0
            (np.arange(cap + 1) % cap, z(cap + 1), [1] * (cap + 1)),   # n_ids > max_streams
            ([0, cap], z(2), [1, 1]),                           # id out of range
            ([3, -1], z(2), [1, 1]),
            ([5, 2, 5], z(3), [1, 1, 1]),                       # duplicate id
            ([1, 2], z(160), [160, 0]),                         # empty chunk
            ([1, 2], z(MAX_CHUNK + 2), [1, MAX_CHUNK + 1]),     # chunk too long
        ]
        for ids, pcm, lens in bad:
            with pytest.raises(IndexError):
                eng.stream_push_indexed(ids, pcm, lens, pre_emphasis=sch.a)
        with pytest.raises(IndexError):                          # no wwb_context_alloc on this ctx
            eng.context_step_indexed([0], z(160), [160])
        ids, lens = np.array([0, 1], np.int32), np.array([160, 160], np.int32)
        x = torch.zeros(320, dtype=torch.int16, device=eng.device)
        out = [torch.empty(2 * MAX_FRAMES, device=eng.device), torch.empty(2, dtype=torch.int32, device=eng.device),
               torch.empty(2, dtype=torch.uint8, device=eng.device), torch.empty(2, device=eng.device)]
        for args in ((None, lens.ctypes.data, x.data_ptr()), (ids.ctypes.data, None, x.data_ptr()),
                     (ids.ctypes.data, lens.ctypes.data, None)):
            rc = eng.lib.wwb_stream_push_indexed(eng.ctx, args[0], 2, args[1], args[2], None, None, C.c_float(0),
                                                 C.c_float(0.5), *[o.data_ptr() for o in out], eng._stream())
            assert rc == -1
            with pytest.raises(ValueError):
                eng._check(rc)

    ea, eb = engine(model, "tc", cap), engine(model, "tc", cap)
    try:
        a = run_indexed(ea, sch)
        b = run_indexed(eb, sch, before=lambda i: bad_calls(eb, i))
    finally:
        ea.close()
        eb.close()
    assert_same_rows(a, b)
    assert sum(int(o[1].sum()) for o in a) > 50


# ------------------------------------------------------------------------------------ 6: the device pipeline
@pytest.mark.gpu
def test_step_streams_vs_pipeline_oracle():
    """MultiStreamPipeline.step_streams: slots dispatched at different times (each slot skips its own pushes) and with
    different frame lengths, pre-emphasis 0.97, rise / fall / min / max-active delays of 40 / 60 / 200 / 1000 ms,
    against one PipelineOracle per slot fed the same frames in the same order."""
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    model, a = "CRNN", 0.97
    w = load_weights(model)
    cfg, pcm0, raw0 = pipeline_script()
    assert all(cfg[k] > 0 for k in ("vad_rise_delay", "vad_fall_delay", "min_active", "max_active"))
    cap, n_step = 8, 300
    rng = np.random.default_rng(13)
    lens_of = [320, 160, 319, 1, 320, 240, 7, 320]   # per slot: the frame length it sends
    rows = [np.roll(pcm0, 977 * s) for s in range(cap)]
    raws = [np.roll(raw0, 5 * s) ^ (rng.random(raw0.size) < 0.03) for s in range(cap)]
    pipe = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, cap, pre_emphasis=a, **cfg)
    oracles = [R.PipelineOracle(w, a=a, **cfg) for _ in range(cap)]
    cur, k = np.zeros(cap, np.int64), np.zeros(cap, np.int64)
    n_win, acts = 0, 0
    try:
        for i in range(n_step):
            ids = rng.permutation(cap)[:int(rng.integers(1, cap + 1))]
            frames, raw = [], []
            for s in ids:
                n = lens_of[s]
                frames.append(rows[s][cur[s]:cur[s] + n])
                raw.append(raws[s][k[s] % raws[s].size])
                cur[s] += n
                k[s] += 1
            out = pipe.step_streams(ids, frames, np.array(raw, np.uint8))
            sp, ac = out["is_speech"].cpu().numpy().astype(bool), out["is_active"].cpu().numpy().astype(bool)
            post, npost = out["post"].cpu().numpy(), out["n_post"].cpu().numpy()
            acts += int(ac.sum())
            for j, s in enumerate(ids):
                o = oracles[s]
                before = len(o.trig.posteriors)
                want_sp, want_ac = o(frames[j], raw[j])
                new = np.array(o.trig.posteriors[before:], np.float32)
                assert sp[j] == want_sp, (i, s)
                assert npost[j] == new.size, (i, s)
                if new.size:
                    assert np.abs(post[j, :new.size] - new).max() < 1e-3, (i, s)
                    n_win += new.size
                if not (new.size and np.abs(new - 0.5).min() <= 1e-3):
                    assert ac[j] == want_ac, (i, s)
    finally:
        pipe.close()
    print("step_streams: %d windows checked, %d active slot-steps" % (n_win, acts))
    assert n_win > 300 and acts > 0
