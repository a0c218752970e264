"""Per-slot trigger options (wwb_stream_set_options, Engine.stream_set_options, set_stream_options of the streaming
classes): a threshold that replaces the call's threshold for one slot, and a listening switch that pauses a slot on one
ctx.

A slot threshold is the scalar threshold of a push of that slot alone, and a paused slot is a slot the trigger sees as
active, so every result is checked bit for bit against a context without options fed the equivalent inputs, and against
the oracle: TriggerOracle per slot, and for trigger chains the reference's composition with paused stages skipped.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import WEIGHTS, load_weights
from oracle import restated as R
from streaming_helpers import MAX_CHUNK, TOL, assert_same_rows, engine, host, pipeline_script, run_indexed, script
from test_gpu_wakeword_chain import FRAME, N_FRAMES, STAGES, STREAMS, _cfg, _models, scenario
from wakeword_detection_b200 import _cabi

GAP = 2e-3   # every oracle posterior compared for a trigger is at least this far from its slot's threshold


# ------------------------------------------------------------------------------------ the binding (no GPU)
def test_symbol_and_argtypes():
    lib = _cabi.load_library()
    res, args = _cabi.PROTOTYPES["wwb_stream_set_options"]
    assert res is C.c_int
    assert args == [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    assert lib.wwb_stream_set_options.argtypes == args and lib.wwb_stream_set_options.restype is C.c_int
    assert lib.wwb_stream_set_options(None, None, 1, None, None, None) == -1


def test_python_argument_shapes():
    thr, lst = _cabi._stream_options(3, 0.5, [1, 0, True])
    assert thr.dtype == np.float32 and thr.tolist() == [0.5] * 3 and lst.dtype == np.uint8 and lst.tolist() == [1, 0, 1]
    assert _cabi._stream_options(2, None, None) == (None, None)
    assert np.isnan(_cabi._stream_options(2, [np.nan, np.inf])[0]).tolist() == [True, False]
    for bad in (dict(threshold=[0.1, 0.2]), dict(listening=np.ones((3, 1))), dict(listening=[0.5, 1, 1]),
                dict(listening=[-1, 0, 1]), dict(listening=[256, 0, 1])):
        with pytest.raises(ValueError):
            _cabi._stream_options(3, **bad)


# ------------------------------------------------------------------------------------ oracle runs of the indexed script
_ORACLE = {}


def oracle_pushes(model, name, paused=frozenset()):
    """per push and entry of the indexed script: (new posteriors, post_max as the device reports it); entry (i, slot) in
    `paused` is fed is_active = 1.  The threshold only decides the trigger, which the callers work out."""
    key = (model, name, paused)
    if key not in _ORACLE:
        w, sch = load_weights(model), script(name)
        orc = [R.TriggerOracle(w, 0.5, sch.a) for _ in range(sch.cap)]
        out = []
        for i, (p, chunks) in enumerate(zip(sch.pushes, sch.chunks)):
            if p.reset is not None:
                for s in np.nonzero(p.reset)[0]:
                    orc[s].reset()
            res = []
            for s, chunk, sp, ac in zip(p.ids, chunks, p.speech, p.active):
                o = orc[s]
                o.active = bool(ac) or (i, int(s)) in paused
                before, pm0 = len(o.posteriors), o.post_max
                o(chunk, bool(sp))
                new = np.array(o.posteriors[before:], np.float32)
                res.append((new, max([pm0] + list(new))))
            out.append(res)
        _ORACLE[key] = out
    return _ORACLE[key]


def _eff(t, call):
    return call if np.isnan(t) else t


def _far(new, t):
    return new.size == 0 or np.isinf(t) or np.abs(new.astype(np.float64) - t).min() >= GAP


def _check_vs_oracle(sch, outs, exp, thr_of, precision, paused=frozenset(), strict=True):
    """outs against the oracle: n_post exact, posteriors within TOL, post_max within TOL, the trigger exact.  strict:
    the threshold of every entry is asserted to be at least GAP from its posteriors; else the trigger is not compared
    where a posterior lies within TOL of the threshold (reported as in test_gpu_stream_indexed.py).  Returns the
    windows checked."""
    tol, n_win, n_band = TOL[precision], 0, 0
    for i, (o, e) in enumerate(zip(outs, exp)):
        post, npost, trig, pmax = o
        p = sch.pushes[i]
        for j, (new, want_pm) in enumerate(e):
            s = int(p.ids[j])
            t = thr_of(i, s)
            where = (i, j, s, t)
            if strict:
                assert _far(new, t), where
            assert npost[j] == new.size, where
            assert np.isnan(post[j, new.size:]).all(), where
            if new.size:
                assert np.abs(post[j, :new.size] - new).max() <= tol, where
            active = bool(p.active[j]) or (i, s) in paused
            if strict or not (new.size and np.abs(new - t).min() <= tol):
                assert trig[j] == (not active and bool((new > t).any())), where
            else:
                n_band += 1
            assert abs(float(pmax[j]) - want_pm) <= tol, where
            n_win += new.size
    print("%d windows checked against the oracle, %d entries in the band around the threshold" % (n_win, n_band))
    return n_win


# ------------------------------------------------------------------------------------ 1: explicit defaults
def _set_defaults(eng, cap):
    ids = np.random.default_rng(cap).permutation(cap)
    n = eng.launch_count()
    eng.stream_set_options(ids, np.full(cap, np.nan, np.float32), np.ones(cap, np.uint8))
    assert eng.launch_count() == n + 1            # one scatter kernel


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tc", "f32"])
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_explicit_defaults_indexed(model, precision):
    """NaN / 1 set on every slot: the ragged indexed script gives the untouched context's outputs bit for bit, with the
    same launches"""
    sch = script("idx")
    ea, eb = engine(model, precision, sch.cap), engine(model, precision, sch.cap)
    try:
        _set_defaults(eb, sch.cap)
        n0 = [ea.launch_count(), eb.launch_count()]
        a, b = run_indexed(ea, sch), run_indexed(eb, sch)
        assert ea.launch_count() - n0[0] == eb.launch_count() - n0[1]
    finally:
        ea.close()
        eb.close()
    assert_same_rows(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_explicit_defaults_dense_pipeline(model):
    """the dense MultiStreamPipeline script of the golden pipeline run, 5 streams, pre-emphasis 0.97"""
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    cfg, pcm0, raw0 = pipeline_script()
    S, nf = 5, len(raw0)
    pcm = np.stack([np.roll(pcm0, 320 * 7 * s) for s in range(S)])
    raw = np.stack([np.roll(raw0, 7 * s) for s in range(S)])
    pa = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, S, pre_emphasis=0.97, **cfg)
    pb = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, S, pre_emphasis=0.97, **cfg)
    try:
        _set_defaults(pb.engine, S)
        n0 = [pa.engine.launch_count(), pb.engine.launch_count()]
        for i in range(nf):
            x = pcm[:, i * 320:(i + 1) * 320]
            a, b = pa.step(x, raw[:, i]), pb.step(x, raw[:, i])
            for k in a:
                assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), (i, k)
        assert pa.engine.launch_count() - n0[0] == pb.engine.launch_count() - n0[1]
    finally:
        pa.close()
        pb.close()


@pytest.mark.gpu
def test_explicit_defaults_chain():
    """a K = 3 MultiWakewordPipeline over the chain scenario, defaults set as scalars on every stage"""
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    pcm, raw = scenario()
    S = len(STREAMS)
    pa, pb = MultiWakewordPipeline(_models(3), S, **_cfg()), MultiWakewordPipeline(_models(3), S, **_cfg())
    count = lambda p: [e.launch_count() for e in p.engines]
    try:
        n = count(pb)
        pb.set_stream_options(np.arange(S), threshold=np.nan, listening=1)
        assert count(pb) == [x + 1 for x in n]
        n0 = [count(pa), count(pb)]
        for i in range(N_FRAMES):
            x = pcm[:, i * FRAME:(i + 1) * FRAME]
            a, b = pa.step(x, raw[:, i]), pb.step(x, raw[:, i])
            for k in a:
                assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), (i, k)
        assert [x - y for x, y in zip(count(pa), n0[0])] == [x - y for x, y in zip(count(pb), n0[1])]
    finally:
        pa.close()
        pb.close()


# ------------------------------------------------------------------------------------ 2: per-slot thresholds
CANDIDATES = (np.nan, 0.05, -np.inf, 0.1, 0.2, 0.3, np.inf, 0.4, 0.6, 0.8)
PHASES = (0, 20, 40)   # the slot thresholds change before these pushes


def slot_thresholds(model, name):
    """[phase][slot] -> threshold: slot s takes the first candidate, in an order rotated by slot and phase, that is at
    least GAP from every oracle posterior of its entries in that phase (NaN: from the call's threshold of each push)"""
    sch, exp = script(name), oracle_pushes(model, name)
    bounds = list(PHASES) + [len(sch.pushes)]
    table = []
    for k in range(len(PHASES)):
        row = []
        for s in range(sch.cap):
            for c in range(len(CANDIDATES)):
                t = CANDIDATES[(c + s + 3 * k) % len(CANDIDATES)]
                ok = all(_far(exp[i][j][0], _eff(t, sch.pushes[i].threshold))
                         for i in range(bounds[k], bounds[k + 1]) for j in np.nonzero(sch.pushes[i].ids == s)[0])
                if ok:
                    row.append(t)
                    break
            else:
                raise AssertionError("no threshold candidate for slot %d in phase %d" % (s, k))
        table.append(np.array(row, np.float32))
    return table


def _phase(i):
    return int(np.searchsorted(PHASES, i, side="right")) - 1


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tc", "f32"])
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_slot_thresholds(model, precision):
    """The indexed script "idx" with per-slot thresholds (NaN, +-inf and values between 0.05 and 0.8) that change
    before pushes 20 and 40, set between pushes without a sync and read back only after the last push.  Each entry's
    post, n_post, trigger and post_max equal bit for bit those of the same slot pushed on a context without options
    with the slot's threshold as the call's scalar, and match TriggerOracle at that threshold."""
    sch = script("idx")
    table = slot_thresholds(model, "idx")
    thr_of = lambda i, s: _eff(float(table[_phase(i)][s]), sch.pushes[i].threshold)
    eb, ref = engine(model, precision, sch.cap), engine(model, precision, sch.cap)
    try:
        dev = []
        for i, p in enumerate(sch.pushes):
            if i in PHASES:
                order = np.random.default_rng(i).permutation(sch.cap)
                eb.stream_set_options(order, table[PHASES.index(i)][order])
            if p.reset is not None:
                eb.stream_reset(p.reset)
            dev.append(eb.stream_push_indexed(p.ids, sch.packed(i), p.lens, p.speech.astype(np.uint8),
                                              p.active.astype(np.uint8), sch.a, p.threshold))
        outs = [host(o) for o in dev]
        # the reference: each push split by effective threshold, every part pushed with it as the call's threshold
        want = []
        for i, p in enumerate(sch.pushes):
            if p.reset is not None:
                ref.stream_reset(p.reset)
            eff = np.array([thr_of(i, int(s)) for s in p.ids])
            rows = [None] * p.ids.size
            for t in np.unique(eff):
                js = np.nonzero(eff == t)[0]
                part = host(ref.stream_push_indexed(p.ids[js], np.concatenate([sch.chunks[i][j] for j in js]),
                                                    p.lens[js], p.speech[js].astype(np.uint8),
                                                    p.active[js].astype(np.uint8), sch.a, float(t)))
                for r, j in enumerate(js):
                    rows[j] = tuple(x[r] for x in part)
            want.append(tuple(np.stack([r[k] for r in rows]) for k in range(4)))
    finally:
        eb.close()
        ref.close()
    for i, (o, w) in enumerate(zip(outs, want)):
        for a, b in zip(o, w):
            assert np.array_equal(a, b, equal_nan=True), i
    exp = oracle_pushes(model, "idx")
    n_win = _check_vs_oracle(sch, outs, exp, thr_of, precision)
    # the slot thresholds decide differently from the call's: in both directions where the call's threshold triggers
    # at all (the WaveNet posteriors of this script stay below 0.5)
    up = down = calls = 0
    for i, (o, e) in enumerate(zip(outs, exp)):
        p = sch.pushes[i]
        for j, (new, _) in enumerate(e):
            call = (not p.active[j]) and bool((new > p.threshold).any())
            up += bool(o[2][j]) and not call
            down += call and not o[2][j]
            calls += call
    print("%s %s: %d windows, %d triggers gained and %d of %d lost through slot thresholds"
          % (model, precision, n_win, up, down, calls))
    assert n_win > 500 and up > 0 and (down > 0 or calls == 0)


# ------------------------------------------------------------------------------------ 3: pausing a slot
PAUSES = {0: range(12, 22), 2: range(12, 22), 3: range(12, 22), 5: range(28, 34)}   # slot -> pushes paused


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tc", "f32"])
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_pause_is_active(model, precision):
    """Slots paused over stretches of the indexed script (the listening switch set between pushes without a sync;
    slots 2 and 3 have VAD falls while paused, slot 0 the wake clip) give, on every row of every push, the outputs of a
    context without options fed is_active = 1 for those entries: after resuming a slot continues from its retained
    window, and the slots not paused are unaffected.  The same rows match TriggerOracle fed is_active = 1."""
    sch = script("idx")
    paused = frozenset((i, int(s)) for i, p in enumerate(sch.pushes) for s in p.ids if i in PAUSES.get(int(s), ()))
    edges = {}
    for s, r in PAUSES.items():
        edges.setdefault(r.start, ([], []))[0].append(s)
        edges.setdefault(r.stop, ([], []))[1].append(s)
    eb, ref = engine(model, precision, sch.cap), engine(model, precision, sch.cap)
    try:
        dev = []
        for i, p in enumerate(sch.pushes):
            if i in edges:
                off, on = edges[i]
                eb.stream_set_options(off + on, listening=[0] * len(off) + [1] * len(on))
            if p.reset is not None:
                eb.stream_reset(p.reset)
            dev.append(eb.stream_push_indexed(p.ids, sch.packed(i), p.lens, p.speech.astype(np.uint8),
                                              p.active.astype(np.uint8), sch.a, p.threshold))
        outs = [host(o) for o in dev]
        want = []
        for i, p in enumerate(sch.pushes):
            if p.reset is not None:
                ref.stream_reset(p.reset)
            act = np.array([a or (i, int(s)) in paused for s, a in zip(p.ids, p.active)], np.uint8)
            want.append(host(ref.stream_push_indexed(p.ids, sch.packed(i), p.lens, p.speech.astype(np.uint8), act,
                                                     sch.a, p.threshold)))
    finally:
        eb.close()
        ref.close()
    assert_same_rows(outs, want)
    # paused entries: nothing analysed, no trigger, the running maximum; some would have analysed frames, and some fall
    unpaused = oracle_pushes(model, "idx")
    would, falls = 0, 0
    was = np.ones(sch.cap, bool)
    for i, p in enumerate(sch.pushes):
        for j, s in enumerate(p.ids):
            if (i, int(s)) in paused:
                assert outs[i][1][j] == 0 and outs[i][2][j] == 0 and np.isnan(outs[i][0][j]).all(), (i, s)
                would += unpaused[i][j][0].size > 0
                falls += bool(was[s] and not p.speech[j])
            was[s] = p.speech[j]
    assert would > 10 and falls > 0
    exp = oracle_pushes(model, "idx", paused)
    assert _check_vs_oracle(sch, outs, exp, lambda i, s: sch.pushes[i].threshold, precision, paused, strict=False) > 500


# ------------------------------------------------------------------------------------ 4: selecting stages of a chain
LISTEN_ONLY = {0: 1, 1: 2, 3: 0, 4: 1, 5: 2, 6: 0}          # stream -> the one stage it listens to
STAGE_THR = (0.4, 0.7, 0.6)                                  # the single listeners' threshold in each stage
ALL_THR = {2: (0.3, np.nan, 0.95), 7: (np.nan, 0.5, np.nan), 8: (0.7, 0.8, 0.4)}   # streams listening to every stage


def _options():
    S, K = len(STREAMS), 3
    listen = np.ones((S, K), np.uint8)
    thr = np.full((S, K), np.nan, np.float32)
    for s, k in LISTEN_ONLY.items():
        listen[s] = 0
        listen[s, k] = 1
        thr[s, k] = STAGE_THR[k]
    for s, t in ALL_THR.items():
        thr[s] = t
    return listen, thr


class SelectOracle:
    """one stream through vad -> the stages it listens to -> activation timeout: a paused stage is fed is_active = 1
    and leaves the is_active of the later stages alone"""

    def __init__(self, ws, listen, thr, cfg):
        self.vad = R.VadDebounceOracle(cfg["frame_width"], cfg["vad_rise_delay"], cfg["vad_fall_delay"])
        self.trigs = [R.TriggerOracle(w, _eff(t, t0), a) for w, (_, t0, a), t in zip(ws, STAGES, thr)]
        self.listen = listen
        self.tmo = R.ActivationTimeoutOracle(cfg["frame_width"], cfg["min_active"], cfg["max_active"])
        self.is_speech, self.is_active = False, False

    def __call__(self, frame, raw):
        self.is_speech = self.vad(self.is_speech, raw)
        act, by, new = self.is_active, -1, []
        for k, t in enumerate(self.trigs):
            before = len(t.posteriors)
            t.active = act or not self.listen[k]
            t(frame, self.is_speech)
            new.append(np.array(t.posteriors[before:], np.float32))
            if self.listen[k]:
                if t.active and not act:
                    by = k
                act = t.active
        self.is_active = self.tmo(self.is_speech, act)
        return dict(is_speech=self.is_speech, is_active=self.is_active, activated=by >= 0,
                    deactivated=act and not self.is_active, activated_by=by, post=new)


_SELECT = {}


def select_oracle_run():
    if not _SELECT:
        pcm, raw = scenario()
        listen, thr = _options()
        ws = [load_weights(m) for m, _, _ in STAGES]
        orc = [SelectOracle(ws, listen[s], thr[s], _cfg()) for s in range(len(STREAMS))]
        _SELECT["steps"] = [[o(pcm[s, i * FRAME:(i + 1) * FRAME], raw[s, i]) for s, o in enumerate(orc)]
                            for i in range(N_FRAMES)]
    return _SELECT["steps"]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tc", "f32"])
def test_chain_stage_selection(precision):
    """K = 3 MultiWakewordPipeline over the chain scenario with per-slot, per-stage options ([n_ids, K] arrays): a stream
    that listens to stage k only equals, bit for bit, the same stream in a MultiStreamPipeline of stage k's model and
    pre-emphasis at the stream's stage-k threshold (stage k's post, n_post, post_max; is_speech, is_active, activated,
    deactivated), its other stages analyse nothing and activated_by is k or -1.  Every stream matches the chain oracle
    with paused stages and per-stage thresholds."""
    from wakeword_detection_b200.wakeword import MultiStreamPipeline, MultiWakewordPipeline
    pcm, raw = scenario()
    S, K = len(STREAMS), 3
    listen, thr = _options()
    steps = select_oracle_run()
    cfg = _cfg()
    pipe = MultiWakewordPipeline(_models(K), S, precision=precision, **cfg)
    solo = [MultiStreamPipeline(os.path.join(WEIGHTS, m), "Wavenet" if m == "Wavenet" else "CRNN", S, pre_emphasis=a,
                                posterior_threshold=STAGE_THR[k], precision=precision, **cfg)
            for k, (m, _, a) in enumerate(STAGES)]
    order = np.random.default_rng(3).permutation(S)
    n_win, near_frames, acts = 0, 0, {k: 0 for k in range(K)}
    try:
        pipe.set_stream_options(order, threshold=thr[order], listening=listen[order])
        for i in range(N_FRAMES):
            chunk = pcm[:, i * FRAME:(i + 1) * FRAME]
            got = host_dict(pipe.step(chunk, raw[:, i]))
            refs = [host_dict(p.step(chunk, raw[:, i])) for p in solo]
            for s, k in LISTEN_ONLY.items():
                ref = refs[k]
                for key in ("post", "n_post", "post_max"):
                    assert np.array_equal(got[key][k, s], ref[key][s], equal_nan=True), (i, s, key)
                for key in ("is_speech", "is_active", "activated", "deactivated"):
                    assert got[key][s] == ref[key][s], (i, s, key)
                assert got["activated_by"][s] == (k if got["activated"][s] else -1), (i, s)
                assert all(got["n_post"][j, s] == 0 for j in range(K) if j != k), (i, s)
                acts[k] += int(got["activated"][s])
            for s in range(S):
                want = steps[i][s]
                assert got["is_speech"][s] == want["is_speech"], (i, s)
                near = False
                for k in range(K):
                    p = want["post"][k]
                    assert got["n_post"][k, s] == p.size, (i, s, k)
                    if p.size:
                        assert np.abs(got["post"][k, s, :p.size] - p).max() < 1e-3, (i, s, k)
                        n_win += p.size
                        near |= np.abs(p - _eff(thr[s, k], STAGES[k][1])).min() <= 1e-3
                if near:
                    near_frames += 1
                    continue
                for key in ("is_active", "activated", "deactivated", "activated_by"):
                    assert int(got[key][s]) == int(want[key]), (i, s, key)
    finally:
        pipe.close()
        for p in solo:
            p.close()
    print("selection %s: %d windows, %d stream-frames in the band, activations of single listeners by stage %s"
          % (precision, n_win, near_frames, acts))
    assert acts[0] > 0 and acts[1] > 0


def host_dict(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


# ------------------------------------------------------------------------------------ 5: records and resets
@pytest.mark.gpu
def test_options_outside_records_and_kept_by_resets():
    """MultiStreamPipeline (CRNN, tc, 6 streams): export_streams bytes do not depend on the options; after
    import_streams (permuted ids), context_reset and a masked stream_reset the options are still in force: the
    pipeline that had them before equals one that got them after the same operation, and differs from one without."""
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    cfg, pcm0, raw0 = pipeline_script()
    S, cut, seg = 6, 60, 60
    pcm = np.stack([np.roll(pcm0, 320 * 11 * s) for s in range(S)])
    raw = np.stack([np.roll(raw0, 11 * s) for s in range(S)])
    ids = np.arange(S, dtype=np.int32)
    opts = dict(threshold=[0.2, np.inf, np.nan, -np.inf, 0.6, np.nan], listening=[1, 1, 0, 1, 1, 0])
    mk = lambda: MultiStreamPipeline(os.path.join(WEIGHTS, "CRNN"), "CRNN", S, pre_emphasis=0.97, **cfg)
    a, b, c, d = mk(), mk(), mk(), mk()
    step = lambda p, i: host_dict(p.step(pcm[:, i * 320:(i + 1) * 320], raw[:, i]))

    def b_equals_c_not_d(i0):
        differs = False
        for i in range(i0, i0 + seg):
            ob, oc, od = step(b, i), step(c, i), step(d, i)
            for k in ob:
                assert np.array_equal(ob[k], oc[k], equal_nan=True), (i, k)
            differs |= any(not np.array_equal(ob[k], od[k], equal_nan=True) for k in ob)
        assert differs

    try:
        for i in range(cut):
            step(a, i)
            step(b, i)
        b.set_stream_options(ids, **opts)
        rec = a.export_streams(ids).cpu().numpy()
        assert np.array_equal(b.export_streams(ids).cpu().numpy(), rec)
        b.import_streams(ids[::-1], rec[::-1])
        for p in (c, d):
            p.import_streams(ids, rec)
        c.set_stream_options(ids, **opts)
        b_equals_c_not_d(cut)
        for p in (b, c, d):
            p.reset()
        b_equals_c_not_d(cut + seg)
        for p in (b, c, d):
            p.engine.stream_reset([1, 0, 1, 1, 0, 1])
        b_equals_c_not_d(cut + 2 * seg)
    finally:
        for p in (a, b, c, d):
            p.close()


# ------------------------------------------------------------------------------------ 6: rejected calls
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_rejections_change_nothing(model):
    """Each malformed call raises with its message before any device work (the launch count stays), and the pushes
    after it equal those of a context that never saw it"""
    w = load_weights(model)
    sch = script("idx")

    unalloc = _cabi.Engine(w, 0, "tc")
    filt = _cabi.Engine({k: w[k] for k in ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")}, 0, "tc")
    try:
        with pytest.raises(IndexError, match="wwb_stream_alloc has not been called"):
            unalloc.stream_set_options([0], threshold=0.5)
        filt.stream_alloc(sch.cap, MAX_CHUNK)
        n = filt.launch_count()
        with pytest.raises(IndexError, match="filter only"):
            filt.stream_set_options([0], listening=0)
        assert filt.launch_count() == n
    finally:
        unalloc.close()
        filt.close()

    def bad_calls(eng, i):
        if i % 6:
            return
        n = eng.launch_count()
        so = eng.stream_set_options
        cases = [
            (IndexError, r"n_ids 0 outside \[1, 12\]", lambda: so([], threshold=[])),
            (IndexError, r"n_ids 13 outside \[1, 12\]", lambda: so(np.arange(13) % 12, threshold=0.1)),
            (IndexError, r"id 12 of entry 1 outside \[0, 12\)", lambda: so([0, 12], listening=0)),
            (IndexError, r"id -1 of entry 1 outside", lambda: so([3, -1], threshold=-np.inf, listening=0)),
            (IndexError, r"id 5 named twice \(entry 2\)", lambda: so([5, 2, 5], listening=[0, 0, 0])),
            (ValueError, "threshold and listening arrays both NULL", lambda: so([0])),
            (ValueError, r"listening value 2 \(entry 1\) is not 0 or 1", lambda: so([0, 4], np.inf, [0, 2])),
        ]
        for exc, msg, fn in cases:
            with pytest.raises(exc, match=msg):
                fn()
        thr = np.full(2, np.inf, np.float32)
        rc = eng.lib.wwb_stream_set_options(eng.ctx, None, 2, thr.ctypes.data, None, eng._stream())
        assert rc == -1 and b"NULL id table" in eng.lib.wwb_last_error(eng.ctx)
        assert eng.launch_count() == n, i

    ea, eb = engine(model, "tc", sch.cap), engine(model, "tc", sch.cap)
    try:
        a = run_indexed(ea, sch)
        b = run_indexed(eb, sch, before=lambda i: bad_calls(eb, i))
    finally:
        ea.close()
        eb.close()
    assert_same_rows(a, b)


@pytest.mark.gpu
def test_chain_arguments_checked_before_any_stage():
    """MultiWakewordPipeline.set_stream_options: a wrong shape or a bad listening value in any stage raises ValueError
    before the first stage's call (no stage launches anything); a valid call launches one scatter per stage"""
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    pipe = MultiWakewordPipeline(_models(2), 4, **_cfg())
    count = lambda: [e.launch_count() for e in pipe.engines]
    try:
        n = count()
        for kw, msg in ((dict(threshold=np.zeros((2, 3))), r"threshold must be a scalar, \[2\] or \[2, 2\]"),
                        (dict(threshold=np.zeros(3)), "threshold must be"),
                        (dict(listening=np.ones((2, 2, 1))), "listening must be"),
                        (dict(threshold=0.5, listening=[[1, 1], [1, 2]]), "listening values must be 0 or 1"),
                        (dict(listening=[[1, 1], [1, -1]]), "listening values must be 0 or 1")):
            with pytest.raises(ValueError, match=msg):
                pipe.set_stream_options([0, 1], **kw)
            assert count() == n, kw
        with pytest.raises(IndexError, match="named twice"):
            pipe.set_stream_options([1, 1], listening=[[1, 0], [0, 1]])
        assert count() == n
        pipe.set_stream_options([0, 1], threshold=[0.3, 0.4], listening=[[1, 0], [0, 1]])
        assert count() == [x + 1 for x in n]
    finally:
        pipe.close()
