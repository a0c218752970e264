"""Several wake words on the same streams: the device speech pipeline with one trigger stage per model
(wwb_context_step_chain / _indexed, wwb_stream_import_chain, MultiWakewordPipeline).

The oracle is the reference's composition restated: VadDebounceOracle, then one TriggerOracle per stage, each fed the
pipeline's is_active at the start of the frame OR'd with the triggers of the stages before it, then
ActivationTimeoutOracle, exactly as PipelineOracle chains them for one stage.  Posteriors within 1e-3; n_post, is_speech,
is_active, activated, deactivated and activated_by exact unless a posterior of the frame lies inside the 1e-3 band around
a stage's threshold (reported, as in test_gpu_streaming.py).  Everything else is checked bit for bit against paths that
are already trusted: wwb_context_step for one stage, a standalone MultiStreamTrigger per model, an uninterrupted run.
"""
import copy
import os

import numpy as np
import pytest

from conftest import WEIGHTS, load_weights
from oracle import restated as R
from streaming_helpers import pipeline_script, wake_clip
from wakeword_detection_b200 import _cabi, synth

FRAME = 320
# (model, posterior_threshold, pre_emphasis) of each stage: thresholds and pre-emphasis differ between the stages
STAGES = [("Wavenet", 0.5, 0.0), ("CRNN", 0.9, 0.97), ("CRNN_arik_original", 0.8, 0.5)]
N_FRAMES = 170


def _cfg():
    return pipeline_script()[0]   # rise / fall delays of 40 / 60 ms, min / max active 200 / 1000 ms


def _models(K):
    return [dict(model_dir=os.path.join(WEIGHTS, m), model_type="Wavenet" if m == "Wavenet" else "CRNN",
                 posterior_threshold=t, pre_emphasis=a) for m, t, a in STAGES[:K]]


# (wake clip or None, its scale, its first sample, noise stream) per stream; the comments name what each stream is for
# (first-trigger frames of the stages measured with the oracle on the CPU)
STREAMS = [
    ("crnn", 1.0, 3287, 7),      # stage 1 triggers first
    ("crnn", 0.25, 3164, 4),     # K = 2: stages 0 and 1 would trigger in the same frame; K = 3: stage 2 first
    ("wavenet", 0.25, 3082, 2),  # K = 3: stages 0 and 2 would trigger in the same frame
    ("wavenet", 1.0, 3000, 0),   # stage 0; the VAD never falls: max_active ends the activation
    (None, 1.0, 0, 0),           # no trigger
    (None, 1.0, 0, 1),           # no trigger, a flickering VAD
    ("crnn", 0.25, 3123, 3),     # stage 0; the VAD falls while active
    (None, 1.0, 0, 2),           # no trigger
    ("crnn", 0.25, 3205, 5),     # K = 2: stage 1 first; K = 3: stage 2 first
]


def scenario():
    """pcm [S, N_FRAMES * 320] int16 and raw VAD [S, N_FRAMES] bool"""
    n = N_FRAMES * FRAME
    pcm, raw = [], []
    rng = np.random.default_rng(17)
    for s, (clip, scale, off, j) in enumerate(STREAMS):
        x = synth.stream_int16(n, 2, 7, j)
        if clip:
            c = np.clip(wake_clip(clip).astype(np.float64) * scale, -32768, 32767).astype(np.int16)
            x[off:off + c.size] = c[:n - off]
        pcm.append(x)
        r = np.ones(N_FRAMES, bool)
        if s == 5:
            r = rng.random(N_FRAMES) < 0.8
        elif s == 6:
            r[95:100] = False          # a fall some 35 frames after its trigger (min_active is 10 frames)
        elif s != 3:
            r[140:146] = False         # a fall late in the run
        raw.append(r)
    return np.stack(pcm), np.stack(raw)


class ChainOracle:
    """one stream through vad -> trigger 0 -> ... -> trigger K-1 -> activation timeout (SpeechPipeline._dispatch with one
    WakewordTrigger stage per model, one shared SpeechContext)"""

    def __init__(self, ws, stages, cfg):
        self.vad = R.VadDebounceOracle(cfg["frame_width"], cfg["vad_rise_delay"], cfg["vad_fall_delay"])
        self.trigs = [R.TriggerOracle(w, t, a) for w, (_, t, a) in zip(ws, stages)]
        self.tmo = R.ActivationTimeoutOracle(cfg["frame_width"], cfg["min_active"], cfg["max_active"])
        self.is_speech, self.is_active = False, False
        self.shadowed = 0     # frames in which a later stage skipped a chunk on which it would have triggered

    def __call__(self, frame, raw):
        self.is_speech = self.vad(self.is_speech, raw)
        act, by = self.is_active, -1
        new = []
        for k, t in enumerate(self.trigs):
            if act and not self.is_active:      # an earlier stage triggered in this frame: would this one have too?
                probe = copy.copy(t)
                probe.frames, probe.posteriors, probe.active = t.frames.copy(), [], False
                probe(frame, self.is_speech)
                self.shadowed += probe.active
            before = len(t.posteriors)
            t.active = act
            t(frame, self.is_speech)
            new.append(np.array(t.posteriors[before:], np.float32))
            if t.active and not act:
                by = k
            act = t.active
        self.is_active = self.tmo(self.is_speech, act)
        return dict(is_speech=self.is_speech, is_active=self.is_active, activated=by >= 0,
                    deactivated=act and not self.is_active, activated_by=by, post=new)


_ORACLE_RUNS = {}


def oracle_run(K):
    """the oracle's outputs for every frame and stream of the scenario with the first K stages (cached: they do not
    depend on the precision)"""
    if K not in _ORACLE_RUNS:
        pcm, raw = scenario()
        ws = [load_weights(m) for m, _, _ in STAGES[:K]]
        oracles = [ChainOracle(ws, STAGES[:K], _cfg()) for _ in STREAMS]
        steps = [[o(pcm[s, i * FRAME:(i + 1) * FRAME], raw[s, i]) for s, o in enumerate(oracles)] for i in range(N_FRAMES)]
        _ORACLE_RUNS[K] = (steps, [o.shadowed for o in oracles])
    return _ORACLE_RUNS[K]


def host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


# ------------------------------------------------------------------------------------ 1: one stage is wwb_context_step
def _k1_inputs(cap, n_step, seed):
    cfg, pcm0, raw0 = pipeline_script()
    rng = np.random.default_rng(seed)
    rows = [np.roll(pcm0, 977 * s) for s in range(cap)]
    raws = [np.roll(raw0, 5 * s) ^ (rng.random(raw0.size) < 0.03) for s in range(cap)]
    return cfg, rows, raws


@pytest.mark.gpu
def test_one_stage_equals_context_step():
    """K = 1, CRNN tc, pre-emphasis 0.97, the golden pipeline script with rise and fall delays on 6 streams: every output
    of the dense chain step equals wwb_context_step's and every output of the indexed chain step (random subsets, ragged
    frames, permuted ids) equals wwb_context_step_indexed's, bit for bit; activated_by is 0 exactly where a trigger fired.
    Launches per call: a step launches two kernels (vad, timeout) more than a push of the same shape on a ctx of the same
    model, dense and indexed, and a one-stage chain step, which asks for activated_by, one more than the step."""
    model, a, thr, cap = "CRNN", 0.97, 0.5, 6
    cfg, rows, raws = _k1_inputs(cap, 0, 5)
    nf = min(len(r) for r in raws)
    engines = []
    try:
        for j in range(5):
            e = _cabi.Engine(load_weights(model), 0, "tc")
            e.stream_alloc(cap, FRAME)
            if j < 4:
                e.context_alloc(**cfg)
            engines.append(e)
        ref, chain, iref, ichain, push = engines
        rng = np.random.default_rng(9)
        cur, k = np.zeros(cap, np.int64), np.zeros(cap, np.int64)
        trig = 0
        for i in range(nf):
            pcm = np.stack([r[i * FRAME:(i + 1) * FRAME] for r in rows])
            vad = np.array([r[i] for r in raws], np.uint8)
            n0 = [e.launch_count() for e in (push, ref, chain)]
            push.stream_push(pcm, pre_emphasis=a, threshold=thr)
            want = host(ref.context_step(pcm, vad, a, thr))
            got = host(chain.context_step_chain([], pcm, vad, a, thr))
            d = [e.launch_count() - n for e, n in zip((push, ref, chain), n0)]
            assert d[1:] == [d[0] + 2, d[0] + 3], (i, d)
            for key in want:
                w, g = want[key], got[key]
                if key in ("post", "n_post", "post_max"):
                    g = g[0]
                assert np.array_equal(w, g, equal_nan=True), (i, key)
            trig += int(got["activated"].sum())
            assert np.array_equal(got["activated_by"], np.where(got["activated"] != 0, 0, -1)), i
            # the indexed form: a random subset of the slots in random order, each with its own frame length
            ids = rng.permutation(cap)[:int(rng.integers(1, cap + 1))].astype(np.int32)
            lens = rng.choice([FRAME, 160, 1, 319, 7], size=ids.size).astype(np.int32)
            frames = [rows[s][cur[s]:cur[s] + n] for s, n in zip(ids, lens)]
            packed = np.concatenate(frames)
            ivad = np.array([raws[s][k[s] % nf] for s in ids], np.uint8)
            cur[ids] += lens
            k[ids] += 1
            n0 = [e.launch_count() for e in (push, iref, ichain)]
            push.stream_push_indexed(ids, packed, lens, pre_emphasis=a, threshold=thr)
            want = host(iref.context_step_indexed(ids, packed, lens, ivad, a, thr))
            got = host(ichain.context_step_chain_indexed([], ids, packed, lens, ivad, a, thr))
            d = [e.launch_count() - n for e, n in zip((push, iref, ichain), n0)]
            assert d[1:] == [d[0] + 2, d[0] + 3], (i, d)
            for key in want:
                g = got[key][0] if key in ("post", "n_post", "post_max") else got[key]
                assert np.array_equal(want[key], g, equal_nan=True), (i, key)
        assert trig > 0
    finally:
        for e in engines:
            e.close()


# ------------------------------------------------------------------------------------ 2, 3: oracle replay, isolation
def _near(post, thr, tol=1e-3):
    return post.size > 0 and np.abs(post - thr).min() <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tc", "f32"])
@pytest.mark.parametrize("K", [2, 3])
def test_chain_vs_oracle(K, precision):
    """MultiWakewordPipeline.step over the scenario (WaveNet + CRNN, + CRNN_arik_original for K = 3; thresholds and
    pre-emphasis per stage) against ChainOracle: each stage activates some stream, on some stream stage 0 triggers in a
    frame in which a later stage would also have triggered (that stage skips the chunk and continues on its own grid),
    activations end through VAD falls and through max_active."""
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    steps, shadowed = oracle_run(K)
    pcm, raw = scenario()
    S = len(STREAMS)
    thr = [t for _, t, _ in STAGES[:K]]
    pipe = MultiWakewordPipeline(_models(K), S, precision=precision, **_cfg())
    n_win, worst, near_frames = 0, 0.0, 0
    by_seen, ends = set(), {"vad_fall": 0, "max_active": 0}
    try:
        for i in range(N_FRAMES):
            got = host(pipe.step(pcm[:, i * FRAME:(i + 1) * FRAME], raw[:, i]))
            for s in range(S):
                want = steps[i][s]
                assert got["is_speech"][s] == want["is_speech"], (i, s)
                near = False
                for k in range(K):
                    p = want["post"][k]
                    assert got["n_post"][k, s] == p.size, (i, s, k)
                    if p.size:
                        err = float(np.abs(got["post"][k, s, :p.size] - p).max())
                        assert err < 1e-3, (i, s, k, err)
                        worst, n_win = max(worst, err), n_win + p.size
                    assert np.isnan(got["post"][k, s, p.size:]).all()
                    near |= _near(p, thr[k])
                if near:
                    near_frames += 1
                    continue
                for key in ("is_active", "activated", "deactivated", "activated_by"):
                    assert int(got[key][s]) == int(want[key]), (i, s, key)
                if want["activated"]:
                    by_seen.add(want["activated_by"])
                if want["deactivated"]:
                    ends["max_active" if want["is_speech"] else "vad_fall"] += 1
    finally:
        pipe.close()
    print("chain K=%d %s: %d windows, max |err| %.3e, %d stream-frames in the band, activations by stage %s, "
          "ends %s, shadowed %s" % (K, precision, n_win, worst, near_frames, sorted(by_seen), ends, shadowed))
    assert by_seen == set(range(K))
    assert sum(shadowed) > 0
    assert ends["vad_fall"] > 0 and ends["max_active"] > 0


@pytest.mark.gpu
def test_stages_are_isolated():
    """On the streams where no stage triggers, stage k's posteriors equal those of a standalone MultiStreamTrigger of
    the same model, threshold and pre-emphasis fed the same audio and the chain's is_speech, bit for bit (K = 3, tc)."""
    from wakeword_detection_b200.wakeword import MultiStreamTrigger, MultiWakewordPipeline
    K = 3
    steps, _ = oracle_run(K)
    quiet = [s for s in range(len(STREAMS)) if not any(steps[i][s]["is_active"] for i in range(N_FRAMES))]
    assert len(quiet) >= 3
    pcm, raw = scenario()
    S = len(STREAMS)
    pipe = MultiWakewordPipeline(_models(K), S, **_cfg())
    solo = [MultiStreamTrigger(os.path.join(WEIGHTS, m), "Wavenet" if m == "Wavenet" else "CRNN", S, FRAME, a, t)
            for m, t, a in STAGES[:K]]
    n_win = 0
    try:
        for i in range(N_FRAMES):
            chunk = pcm[:, i * FRAME:(i + 1) * FRAME]
            got = host(pipe.step(chunk, raw[:, i]))
            for k in range(K):
                # the solo triggers see the chain's is_speech and is_active = 0: identical inputs on the quiet streams
                ref = solo[k].push(chunk, got["is_speech"], np.zeros(S, np.uint8))
                post, n_post = ref["post"].cpu().numpy(), ref["n_post"].cpu().numpy()
                assert np.array_equal(got["post"][k, quiet], post[quiet], equal_nan=True), (i, k)
                assert np.array_equal(got["n_post"][k, quiet], n_post[quiet]), (i, k)
                n_win += int(n_post[quiet].sum())
    finally:
        pipe.close()
        for t in solo:
            t.close()
    assert n_win > 1000


# ------------------------------------------------------------------------------------ 4: indexed subsets
def _records(pipe, cap):
    return [r.cpu().numpy() for r in pipe.export_streams(np.arange(cap, dtype=np.int32))]


@pytest.mark.gpu
def test_indexed_subsets_leave_other_slots_alone():
    """MultiWakewordPipeline.step_streams (K = 3, tc) over ragged subsets of 12 slots in permuted order: the records of
    every slot not named in a step are byte-identical before and after it in every stage; the named slots advance.
    A step naming every slot in permuted order gives the dense step's outputs, row for row."""
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    K, cap, n_step = 3, 12, 60
    cfg = _cfg()
    pcm, raw = scenario()
    rows = [pcm[s % len(STREAMS)] for s in range(cap)]
    raws = [np.roll(raw[s % len(STREAMS)], 3 * s) for s in range(cap)]
    rng = np.random.default_rng(23)
    pipe = MultiWakewordPipeline(_models(K), cap, **cfg)
    dense = MultiWakewordPipeline(_models(K), cap, **cfg)
    perm = MultiWakewordPipeline(_models(K), cap, **cfg)
    cur, k = np.zeros(cap, np.int64), np.zeros(cap, np.int64)
    moved = 0
    try:
        for i in range(n_step):
            ids = rng.permutation(cap)[:int(rng.integers(1, cap))].astype(np.int32)
            lens = rng.choice([FRAME, 160, 1, 319, 200], size=ids.size)
            frames = [rows[s][cur[s]:cur[s] + n] for s, n in zip(ids, lens)]
            vad = np.array([raws[s][k[s]] for s in ids], np.uint8)
            cur[ids] += lens
            k[ids] += 1
            before = _records(pipe, cap)
            out = host(pipe.step_streams(ids, frames, vad))
            after = _records(pipe, cap)
            others = np.setdiff1d(np.arange(cap), ids)
            for st in range(K):
                assert np.array_equal(before[st][others], after[st][others]), (i, st)
                moved += int((before[st][ids] != after[st][ids]).any(axis=1).sum())
            assert out["post"].shape[:2] == (K, ids.size) and out["activated_by"].shape == (ids.size,)

            # every slot, permuted, against the dense step (rows of the permuted step in ids order)
            chunk = pcm[:, i * FRAME:(i + 1) * FRAME][np.arange(cap) % len(STREAMS)]
            v = raw[np.arange(cap) % len(STREAMS), i].astype(np.uint8)
            p = rng.permutation(cap).astype(np.int32)
            want = host(dense.step(chunk, v))
            got = host(perm.step_streams(p, [chunk[s] for s in p], v[p]))
            for key in want:
                w = want[key][:, p] if key in ("post", "n_post", "post_max") else want[key][p]
                assert np.array_equal(w, got[key], equal_nan=True), (i, key)
    finally:
        for x in (pipe, dense, perm):
            x.close()
    assert moved > n_step


# ------------------------------------------------------------------------------------ 5: session records
@pytest.mark.gpu
def test_chain_records_move_and_reject_atomically():
    """K = 2 (WaveNet + CRNN, tc): after 80 steps every stage's records go into a fresh chain of 16 slots under permuted
    ids; continuing there gives the uninterrupted run's outputs bit for bit.  A batch whose stage-1 record 3 is corrupt
    raises ValueError naming stage 1 and record 3, and no slot of either stage changes."""
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    K, cut = 2, 80
    cfg = _cfg()
    pcm, raw = scenario()
    S = len(STREAMS)
    ids = np.arange(S, dtype=np.int32)
    a = MultiWakewordPipeline(_models(K), S, **cfg)
    b = MultiWakewordPipeline(_models(K), 16, **cfg)
    m = np.random.default_rng(4).permutation(16)[:S].astype(np.int32)
    try:
        outs = [host(a.step(pcm[:, i * FRAME:(i + 1) * FRAME], raw[:, i])) for i in range(cut)]
        recs = a.export_streams(ids)
        assert len(recs) == K
        d0 = _cabi.decode_stream_state(recs[0], 182)
        d1 = _cabi.decode_stream_state(recs[1], 151)
        assert (d0["flags"] == _cabi.STREAM_STATE_PIPELINE).all() and (d1["flags"] == 0).all()
        b.import_streams(m, recs)
        for st in range(K):
            assert np.array_equal(b.export_streams(m)[st].cpu().numpy(), recs[st].cpu().numpy()), st
        acts = 0
        for i in range(cut, N_FRAMES):
            chunk = pcm[:, i * FRAME:(i + 1) * FRAME]
            want = host(a.step(chunk, raw[:, i]))
            got = host(b.step_streams(m, list(chunk), raw[:, i]))
            for key in want:
                assert np.array_equal(want[key], got[key], equal_nan=True), (i, key)
            acts += int(want["activated"].sum())
        assert acts > 0 or any(o["activated"].any() for o in outs)

        before = [r.cpu().numpy() for r in b.export_streams(np.arange(16, dtype=np.int32))]
        bad = [r.clone() for r in a.export_streams(ids)]
        bad[1][3, :4] = 0                     # stage 1, record 3: bad magic
        with pytest.raises(ValueError, match=r"stage 1 record 3: bad magic"):
            b.import_streams(m, bad)
        after = [r.cpu().numpy() for r in b.export_streams(np.arange(16, dtype=np.int32))]
        for st in range(K):
            assert np.array_equal(before[st], after[st]), st
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------------------------ 6: rejections change nothing
def _raw_step(eng, engines, K, a=True, thr=True):
    """wwb_context_step_chain through ctypes with K stages from `engines` (not necessarily distinct) and optionally
    NULL pre-emphasis / threshold arrays; returns the status"""
    import ctypes as C
    import torch
    S = 4
    pcm = torch.zeros((S, FRAME), dtype=torch.int16, device=eng.device)
    ctxs = (C.c_void_p * max(K, 1))(*[e.ctx for e in engines[:max(K, 1)]])
    av = np.zeros(max(K, 1), np.float32)
    tv = np.full(max(K, 1), 0.5, np.float32)
    return eng.lib.wwb_context_step_chain(ctxs, K, pcm.data_ptr(), S, FRAME, None, av.ctypes.data if a else None,
                                          tv.ctypes.data if thr else None, None, None, None, None, None, None, None,
                                          None, None)


@pytest.mark.gpu
def test_chain_rejections_change_nothing():
    """Each check of the stage list returns its code before any device work, and afterwards the records of every slot
    of every stage are byte-identical to those taken before: a capacity mismatch, another device (with two GPUs), a
    filter-only ctx, stage 0 without wwb_context_alloc, a repeated ctx, K = 0 and K = 9, NULL pre-emphasis / threshold
    arrays, a chunk longer than a later stage's max_chunk, a repeated id, a bad record array."""
    import torch
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    cap = 4
    cfg = _cfg()
    pcm, raw = scenario()
    pipe = MultiWakewordPipeline(_models(2), cap, **cfg)
    w = load_weights("CRNN")
    extra = []

    def mk(cap_, chunk, filt=False, ctx_alloc=False, device=0):
        ww = {k: w[k] for k in ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")} if filt else w
        e = _cabi.Engine(ww, device, "tc")
        e.stream_alloc(cap_, chunk)
        if ctx_alloc:
            e.context_alloc(**cfg)
        extra.append(e)
        return e

    try:
        for i in range(30):
            pipe.step(pcm[:cap, i * FRAME:(i + 1) * FRAME], raw[:cap, i])
        ids = np.arange(cap, dtype=np.int32)
        e0, e1 = pipe.engines
        ref = _records(pipe, cap)
        chunk = pcm[:cap, :FRAME]
        vad = np.ones(cap, np.uint8)

        def unchanged():
            now = _records(pipe, cap)
            for st in range(2):
                assert np.array_equal(ref[st], now[st]), st

        cases = [
            (IndexError, "stage 1: stream state for 5 streams", lambda: e0.context_step_chain([mk(5, FRAME)], chunk, vad)),
            (IndexError, "filter only", lambda: e0.context_step_chain([mk(cap, FRAME, filt=True)], chunk, vad)),
            (IndexError, "wwb_context_alloc", lambda: e1.context_step_chain([e0], chunk, vad)),
            (ValueError, "the ctx of stage 0 again", lambda: e0.context_step_chain([e1, e0], chunk, vad)),
            (ValueError, "9 stages", lambda: e0.context_step_chain([e1] + [mk(cap, FRAME) for _ in range(7)], chunk, vad)),
            (IndexError, "stage 1: chunk of 320 samples", lambda: e0.context_step_chain([mk(cap, 200)], chunk, vad)),
            (IndexError, "stage 1: chunk of 320 samples",
             lambda: e0.context_step_chain_indexed([mk(cap, 200)], ids, chunk.reshape(-1), np.full(cap, FRAME), vad)),
            (IndexError, "named twice", lambda: e0.context_step_chain_indexed([e1], [0, 1, 1], chunk[:3].reshape(-1),
                                                                              np.full(3, FRAME), vad[:3])),
            (IndexError, "named twice", lambda: e0.stream_import_chain([e1], [2, 2], [x[:2] for x in ref])),
            (ValueError, "stage 1: records hold", lambda: e0.stream_import_chain([e1], ids, [ref[0], ref[1][:2]])),
        ]
        if torch.cuda.device_count() > 1:
            cases.append((ValueError, "on device 1", lambda: e0.context_step_chain([mk(cap, FRAME, device=1)], chunk, vad)))
        for exc, msg, fn in cases:
            with pytest.raises(exc, match=msg):
                fn()
            unchanged()
        # through the C ABI: K outside [1, 8] and NULL per-stage arrays
        assert _raw_step(e0, [e0, e1], 0) == -1 and b"0 stages" in e0.lib.wwb_last_error(e0.ctx)
        assert _raw_step(e0, [e0, e1], 2, a=False) == -1
        assert _raw_step(e0, [e0, e1], 2, thr=False) == -1
        assert b"NULL pre-emphasis or threshold" in e0.lib.wwb_last_error(e0.ctx)
        unchanged()
    finally:
        pipe.close()
        for e in extra:
            e.close()
