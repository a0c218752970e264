"""The many-stream streaming trigger (wwb_stream_push, csrc/filter.cu stream_*_kernel) against the oracle's
`TriggerOracle` (wakeword/tflite.py:123-246) and against the batch path.

A run is a script of pushes.  Each push gives the chunk length, how many of the allocated streams it covers (a
prefix), per-stream is_speech / is_active, the threshold and an optional masked reset applied before it.  The
script never depends on what the device returns, so one oracle run per (model, script) serves every precision.

Tolerances as in test_gpu_parity.py: posteriors 1e-3 absolute for f32 / tc, 2e-2 for tc_fast (single fp16
operands); trigger decisions exact unless a posterior of the push lies inside the band around the threshold.
"""
import numpy as np
import pytest

from conftest import GOLDEN, WEIGHTS, load_weights
from oracle import restated as R
from streaming_helpers import (CHUNKS, MODELS, PRECISIONS, SCHEDULES, TOL, Push, Schedule, assert_same_rows,
                               engine, host, schedule, wake_clip)
from wakeword_detection_b200 import synth

STATS = {}
_ORACLE_CACHE = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for (model, prec), (n, err) in sorted(STATS.items()):
        print("\n[stream replay] %s %s: %d windows checked against the oracle, max |err| %.3e" % (model, prec, n, err))


# ------------------------------------------------------------------------------------ the oracle's run of a schedule
def oracle_run(model, sname):
    """Per push and covered stream: (posteriors, trigger, post_max as the device reports it).  On a VAD fall the
    device reports the maximum before its reset (stream_finish_kernel writes it, then clears the state)."""
    key = (model, sname)
    if key in _ORACLE_CACHE:
        return _ORACLE_CACHE[key]
    w = load_weights(model)
    sch = schedule(sname)
    orc = [R.TriggerOracle(w, 0.5, sch.a) for _ in range(sch.cap)]
    out = []
    for p, chunk in zip(sch.pushes, sch.chunks):
        if p.reset is not None:
            for s in np.nonzero(p.reset)[0]:
                orc[s].reset()
        res = []
        for s in range(p.n_streams):
            o = orc[s]
            o.active = bool(p.active[s])
            before, pm0 = len(o.posteriors), o.post_max
            o(chunk[s], bool(p.speech[s]))
            new = np.array(o.posteriors[before:], np.float32)
            trig = bool(not p.active[s] and (new > p.threshold).any())
            res.append((new, trig, max([pm0] + list(new))))
        out.append(res)
    _ORACLE_CACHE[key] = out
    return out


def _push(eng, sch, i):
    import torch
    p = sch.pushes[i]
    S = p.n_streams
    c = torch.from_numpy(sch.chunks[i]).to(eng.device)
    return host(eng.stream_push(c, p.speech[:S].astype(np.uint8), p.active[:S].astype(np.uint8), sch.a, p.threshold))


def run_device(eng, sch, between=None):
    """every push of `sch` on `eng` (masked resets included); `between(i)` runs before push i"""
    outs = []
    for i, p in enumerate(sch.pushes):
        if between is not None:
            between(i)
        if p.reset is not None:
            eng.stream_reset(p.reset)
        outs.append(_push(eng, sch, i))
    return outs


def check_against_oracle(outs, exp, sch, tol, streams=None):
    """n_post exact, posteriors within tol, NaN tail, trigger exact outside the band, post_max within tol.
    Returns (windows checked, max |err|)."""
    mf = sch.max_frames
    n_win, worst = 0, 0.0
    for i, (o, e) in enumerate(zip(outs, exp)):
        post, npost, trig, pmax = o
        p = sch.pushes[i]
        for s in range(p.n_streams) if streams is None else [s for s in streams if s < p.n_streams]:
            new, want_trig, want_pm = e[s]
            where = (sch.name, i, s)
            assert npost[s] == new.size, where
            assert np.isnan(post[s, new.size:mf]).all(), where
            if new.size:
                err = float(np.abs(post[s, :new.size] - new).max())
                assert err <= tol, (where, err)
                worst = max(worst, err)
                n_win += new.size
            if not (new.size and np.abs(new - p.threshold).min() <= tol):
                assert trig[s] == want_trig, where
            assert abs(float(pmax[s]) - want_pm) <= tol, (where, float(pmax[s]), want_pm)
    return n_win, worst


# ------------------------------------------------------------------------------------ 0/1: the oracle side (no GPU)
def test_schedules_cover_the_edges():
    """the scripts reach what they claim to: every chunk size, a push completing max_frames, pushes completing none
    with and without frames before, fewer than 512 samples seen, falls, resets and prefixes (counted on the host)"""
    for name in SCHEDULES:
        sch = schedule(name)
        seen = np.zeros(sch.cap, np.int64)
        frames_per_push, small = [], False
        for p in sch.pushes:
            before = R.num_frames(seen[0])
            seen[:p.n_streams] += p.n
            frames_per_push.append(R.num_frames(seen[0]) - before)
            small |= seen[0] < R.FFT
        if name.startswith("ragged"):
            assert set(CHUNKS) <= {p.n for p in sch.pushes}
            assert small and sch.max_frames in frames_per_push
            assert 0 in frames_per_push[frames_per_push.index(sch.max_frames):]
            assert {sch.cap, sch.cap - 1, 1, sch.cap // 2} <= {p.n_streams for p in sch.pushes}
            assert any(p.reset is not None and p.reset.size < sch.cap for p in sch.pushes)
        else:
            assert frames_per_push[1:] == [sch.max_frames] * (len(sch.pushes) - 1)
    sch = schedule("ragged_pe")
    assert {0.5, 0.9} == {p.threshold for p in sch.pushes}
    pcm3 = np.concatenate([c[3] for c in sch.chunks if c.shape[0] > 3])
    assert (pcm3 == -32768).any() and (pcm3 == 32767).any()


@pytest.mark.parametrize("a", [0.0, 0.97])
def test_trigger_oracle_is_the_padded_window_formula(a):
    """TriggerOracle fed ragged chunks (speech throughout, never active) emits, for its k-th analysed frame, the
    posterior of rows [k+1, k+1+L) of [L zero rows ; mel_stream(pcm, a)]: the formula the GPU tests compare the
    stream path with.  (1e-6, not bits: numpy's BLAS may sum a batch of windows in another order than one window.)
    reset() keeps prev_sample: the first sample after a reset is pre-emphasised against the one before it.  That sample
    only ever sits at position 0 of the first frame after the reset, where the Hann window is 0, so no posterior
    depends on it: the device's reset may or may not clear prev_sample without any test here seeing it."""
    w = load_weights("CRNN_arik_original")
    L = int(w["mel_length"])
    r = np.random.default_rng(int(a * 100) + 3)
    pcm = synth.stream_int16(160 * 40 + 700, 2, 9, 1)
    o = R.TriggerOracle(w, 0.5, a)
    at = 0
    while at < pcm.size:
        n = int(r.choice(CHUNKS))
        o(pcm[at:at + n], True)
        at += n
    mel = R.mel_stream(R.int16_to_float(pcm), w, a)
    padded = np.concatenate([np.zeros((L, 40), np.float32), mel])
    k = np.arange(mel.shape[0])
    ref = R.posterior(padded[(k + 1)[:, None] + np.arange(L)[None, :]], w)
    assert len(o.posteriors) == mel.shape[0] > 30
    np.testing.assert_allclose(np.array(o.posteriors, np.float32), ref, rtol=0, atol=1e-6)
    prev = o.prev_sample
    assert prev == float(R.int16_to_float(pcm[-1:])[0])
    o.reset()
    assert o.prev_sample == prev and o.pending.size == 0 and o.post_max == 0.0 and not o.frames.any()


# ------------------------------------------------------------------------------------ 2: replay against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("sname", list(SCHEDULES))
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", MODELS)
def test_stream_replay_vs_oracle(model, precision, sname):
    sch = schedule(sname)
    exp = oracle_run(model, sname)
    eng = engine(model, precision, sch.cap, sch.max_chunk)
    try:
        assert eng.stream_max_frames() == sch.max_frames
        outs = run_device(eng, sch)
    finally:
        eng.close()
    tol = TOL[precision]
    n_win, worst = check_against_oracle(outs, exp, sch, tol)
    fired = sum(t for e in exp for (_, t, _) in e)
    n, err = STATS.get((model, precision), (0, 0.0))
    STATS[(model, precision)] = (n + n_win, max(err, worst))
    print("%s %s %s: %d windows checked, %d oracle triggers, max |err| %.3e" % (model, precision, sname, n_win, fired, worst))
    assert n_win > 0 and (fired > 0 or not sname.startswith("long"))     # the wake clips fire at 0.9 on every model


# ------------------------------------------------------------------------------------ 3: bit-exact vs the batch path
@pytest.mark.gpu
@pytest.mark.parametrize("a", [0.0, 0.97])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", MODELS)
def test_stream_equals_batch_path_bitwise(model, precision, a):
    """1024 streams, ragged chunks, speech throughout, no reset, never active: push i, frame q of stream s is the
    window that ends at that stream's k-th frame, so it must equal

        posteriors(cat(zeros(S, L-1, 40), filter(pcm, a)), hop=1)[s, k]

    bit for bit.  Both filters run frame_spectrum64 / mel_pair on the same fp32 pre-emphasised samples, and the
    explicit-list windows of a push take the per-window encoder schedule, which is bit-identical to the shared batch
    schedule (test_crnn_shared_columns_*, test_wavenet_shared_activations_*).  Every stream is checked."""
    import torch
    from wakeword_detection_b200 import _cabi
    S, max_chunk = 1024, 1601
    r = np.random.default_rng(int(a * 100) + 17)
    ns = [int(v) for v in r.choice(CHUNKS, size=16)]
    eng = _cabi.Engine(load_weights(model), 0, precision)
    try:
        eng.stream_alloc(S, max_chunk)
        mf = eng.stream_max_frames()
        L = eng.L
        pcm = synth.device_pcm(S, sum(ns), seed=77, device=eng.device)
        mel = eng.filter(pcm, a)
        F = mel.shape[1]
        ref = eng.posteriors(torch.cat([torch.zeros((S, L - 1, 40), device=eng.device), mel], 1), hop=1)
        assert ref.shape == (S, F)
        at, k = 0, 0
        for n in ns:
            post, npost, trig, pmax = eng.stream_push(pcm[:, at:at + n].contiguous(), pre_emphasis=a)
            at += n
            q = R.num_frames(at) - k
            assert bool((npost == q).all())
            assert torch.equal(post[:, :q], ref[:, k:k + q]), (k, q, float((post[:, :q] - ref[:, k:k + q]).abs().max()))
            assert bool(post[:, q:mf].isnan().all())
            k += q
        assert k == F
    finally:
        eng.close()


# ------------------------------------------------------------------------------------ 4: state isolation
def _small_schedule(cap, n_push, a, seed, n_streams=None, resets=None, speech=True):
    r = np.random.default_rng(seed)
    ns = [int(v) for v in r.choice(CHUNKS, size=n_push)]
    n_streams = n_streams or {}
    resets = resets or {}
    pushes = [Push(ns[i], n_streams.get(i, cap), np.full(cap, speech), np.zeros(cap), 0.5, resets.get(i))
              for i in range(n_push)]
    pcm = np.stack([synth.stream_int16(sum(ns) + 1, 2 + (s % 2) * 3, seed, s) for s in range(cap)])
    pcm[0, 600:600 + 35200] = wake_clip("crnn")[:sum(ns) + 1 - 600]
    return Schedule("small", cap, 1601, a, pcm, pushes)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_skipped_stream_keeps_its_state(model):
    """Stream cap-1 sits out pushes 4..8 (n_streams = cap-1): its later posteriors equal those of the same stream on a
    fresh context that never saw those pushes (bits), and the oracle's."""
    cap, skip = 4, range(4, 9)
    sch = _small_schedule(cap, 16, 0.97, 5, n_streams={i: cap - 1 for i in skip})
    w = load_weights(model)
    eng = engine(model, "tc", cap, 1601)
    fresh = engine(model, "tc", cap, 1601)
    try:
        a = run_device(eng, sch)
        keep = [i for i in range(len(sch.pushes)) if i not in skip]
        b = [_push(fresh, sch, i) for i in keep]
    finally:
        eng.close()
        fresh.close()
    s = cap - 1
    assert_same_rows([a[i] for i in keep], b, rows=s)
    o = R.TriggerOracle(w, 0.5, sch.a)
    n_win = 0
    for j, i in enumerate(keep):
        before = len(o.posteriors)
        o(sch.chunks[i][s], True)
        new = np.array(o.posteriors[before:], np.float32)
        assert b[j][1][s] == new.size
        if new.size:
            assert np.abs(b[j][0][s, :new.size] - new).max() <= TOL["tc"]
        n_win += new.size
    assert n_win > 20


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_masked_reset(model):
    """A reset with the 5-byte mask [1,0,1,0,0] before push 8 on 8 streams: streams 1, 3, 4 and 5..7 (past the mask)
    continue bit for bit as without the reset; streams 0 and 2 follow the oracle after its reset()."""
    cap, at = 8, 8
    mask = np.array([1, 0, 1, 0, 0], np.uint8)
    with_reset = _small_schedule(cap, 14, 0.97, 6, resets={at: mask})
    without = _small_schedule(cap, 14, 0.97, 6)
    w = load_weights(model)
    e1, e2 = engine(model, "tc", cap, 1601), engine(model, "tc", cap, 1601)
    try:
        a = run_device(e1, with_reset)
        b = run_device(e2, without)
    finally:
        e1.close()
        e2.close()
    untouched = np.array([1, 3, 4, 5, 6, 7])
    assert_same_rows(a, b, rows=untouched)
    assert_same_rows(a[:at], b[:at])
    for s in (0, 2):
        o = R.TriggerOracle(w, 0.5, with_reset.a)
        for i, chunk in enumerate(with_reset.chunks):
            if i == at:
                o.reset()
            before, pm0 = len(o.posteriors), o.post_max
            o(chunk[s], True)
            new = np.array(o.posteriors[before:], np.float32)
            post, npost, _, pmax = a[i]
            assert npost[s] == new.size, (i, s)
            if new.size:
                assert np.abs(post[s, :new.size] - new).max() <= TOL["tc"], (i, s)
            assert abs(float(pmax[s]) - max([pm0] + list(new))) <= TOL["tc"], (i, s)
    # the reset changed what streams 0 / 2 see (their windows after it start from zero rows again)
    assert any(not np.array_equal(x[0][[0, 2]], y[0][[0, 2]], equal_nan=True) for x, y in zip(a[at:], b[at:]))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_rejected_pushes_and_batch_calls_leave_the_state_alone(model, precision):
    """Baseline run on a fresh context, then the same script on three more fresh contexts: (a) unchanged, (b) with
    rejected pushes (n > max_chunk, n_streams > cap, n = 0 raise IndexError) before some pushes, (c) with filter /
    posteriors / pipeline calls on a batch that regrows the context's workspaces between pushes.  Window slots come
    from an atomicAdd, so (a) is also the determinism check: post, n_post, trigger and post_max agree bit for bit."""
    import torch
    cap = 64
    sch = _small_schedule(cap, 12, 0.97, 8, n_streams={5: cap // 2})
    runs = {}
    big = synth.device_pcm(48, 160 * 600 + 512, seed=3, device=torch.device("cuda", 0))

    def rejected(eng, i):
        if i % 4 == 2:
            with pytest.raises(IndexError):
                eng.stream_push(np.zeros((cap, sch.max_chunk + 1), np.int16), pre_emphasis=sch.a)
            with pytest.raises(IndexError):
                eng.stream_push(np.zeros((cap + 1, 160), np.int16), pre_emphasis=sch.a)
            with pytest.raises(IndexError):
                eng.stream_push(np.zeros((cap, 0), np.int16), pre_emphasis=sch.a)

    def batch_calls(eng, i):
        if i % 3 == 1:
            mel = eng.filter(big, 0.5)
            eng.posteriors(mel, hop=1)
            eng.pipeline(big, hop=2, pre_emphasis=0.97)

    for name, between in (("base", None), ("again", None), ("rejected", rejected), ("batch", batch_calls)):
        eng = engine(model, precision, cap, 1601)
        try:
            runs[name] = run_device(eng, sch, None if between is None else (lambda i, e=eng, f=between: f(e, i)))
        finally:
            eng.close()
    for name in ("again", "rejected", "batch"):
        assert_same_rows(runs["base"], runs[name])
    assert sum(int(o[1].sum()) for o in runs["base"]) > 100


# ------------------------------------------------------------------------------------ 5: the device pipeline, a = 0.97
@pytest.mark.gpu
def test_device_pipeline_with_pre_emphasis_vs_oracle():
    """wwb_context_step (vad debounce -> trigger -> activation timeout) with pre_emphasis = 0.97 against PipelineOracle
    on the raw-VAD scripts of test_device_pipeline_state_machine_replays_reference_run (that one runs a = 0)."""
    import os
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    wname, name, a = "CRNN", "crnn", 0.97
    w = load_weights(wname)
    g = np.load(os.path.join(GOLDEN, "reference_pipeline.npz"))
    cfg = dict(zip(("frame_width", "vad_rise_delay", "vad_fall_delay", "min_active", "max_active"), [int(v) for v in g["cfg"]]))
    pcm0, raw0 = g["pipe_%s_pcm" % name], g["pipe_%s_raw" % name]
    nf = len(raw0)
    S = 5
    rng = np.random.default_rng(11)
    pcm = np.stack([np.roll(pcm0, 320 * 7 * s) for s in range(S)])
    raw = np.stack([raw0] + [np.roll(raw0, 7 * s) ^ (rng.random(nf) < 0.03) for s in range(1, S)])
    raw[4] = True
    pipe = MultiStreamPipeline(os.path.join(WEIGHTS, wname), wname, S, pre_emphasis=a, **cfg)
    oracles = [R.PipelineOracle(w, a=a, **cfg) for _ in range(S)]
    n_win, worst, acts = 0, 0.0, 0
    try:
        for i in range(nf):
            out = pipe.step(pcm[:, i * 320:(i + 1) * 320], raw[:, i])
            sp, ac = out["is_speech"].cpu().numpy().astype(bool), out["is_active"].cpu().numpy().astype(bool)
            post, npost = out["post"].cpu().numpy(), out["n_post"].cpu().numpy()
            acts += int(ac.sum())
            for s in range(S):
                o = oracles[s]
                before = len(o.trig.posteriors)
                want_sp, want_ac = o(pcm[s, i * 320:(i + 1) * 320], raw[s, i])
                new = np.array(o.trig.posteriors[before:], np.float32)
                near = new.size and np.abs(new - 0.5).min() <= 1e-3
                assert sp[s] == want_sp, (i, s)
                assert npost[s] == new.size, (i, s)
                if new.size:
                    err = float(np.abs(post[s, :new.size] - new).max())
                    assert err < 1e-3, (i, s, err)
                    worst, n_win = max(worst, err), n_win + new.size
                if not near:
                    assert ac[s] == want_ac, (i, s)
    finally:
        pipe.close()
    print("context_step a=%.2f: %d windows checked, max |err| %.3e, %d active stream-frames" % (a, n_win, worst, acts))
    assert n_win > 800 and acts > 0          # the script analyses 865 windows (the oracle's count, every one compared)
