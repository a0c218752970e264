"""What the streaming tests share (test_gpu_streaming, test_gpu_stream_indexed, test_gpu_stream_state): the models and
tolerances, the push scripts (dense schedules and indexed scripts, built on the host, never from device results), the
engine constructor, the push and run helpers and the mel check.

Tolerances as in test_gpu_parity.py: posteriors 1e-3 absolute for f32 / tc, 2e-2 for tc_fast (single fp16 operands).
"""
import os

import numpy as np

from conftest import GOLDEN, load_weights
from oracle import restated as R
from wakeword_detection_b200 import synth

MODELS = ("CRNN", "CRNN_arik_original", "Wavenet")
PRECISIONS = ("f32", "tc", "tc_fast")
TOL = {"f32": 1e-3, "tc": 1e-3, "tc_fast": 2e-2}
CHUNKS = (1, 7, 159, 160, 161, 319, 320, 511, 512, 513, 1599, 1600, 1601)
MAX_CHUNK = 1601
SIZES = (1, 7, 159, 160, 161, 319, 320, 511, 512, 513, MAX_CHUNK - 1, MAX_CHUNK)
MAX_FRAMES = (MAX_CHUNK - 1) // R.HOP + 1

MEL_RTOL = 1e-4
MEL_STATS = {"bins": 0, "at_floor": 0, "max_err": 0.0, "max_err_over_tol": 0.0}


def check_mel(got, ref):
    """BASELINE.md 4: |d| <= 1e-4 * max(|ref|, 1) on EVERY bin, no exemptions (the FFT is fp64 like the
    reference's, csrc/fft64.cuh).  Bins whose reference value is exactly 0.0 (energy at or below the 1e-5 floor) are
    counted, not exempted: they obey the same bound.  Running statistics are printed at the end of the session."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape
    tol = MEL_RTOL * np.maximum(np.abs(ref), 1.0)
    err = np.abs(got - ref)
    MEL_STATS["bins"] += int(ref.size)
    MEL_STATS["at_floor"] += int((ref == 0.0).sum())
    if ref.size:
        MEL_STATS["max_err"] = max(MEL_STATS["max_err"], float(err.max()))
        MEL_STATS["max_err_over_tol"] = max(MEL_STATS["max_err_over_tol"], float((err / tol).max()))
        i = np.unravel_index(np.argmax(err / tol), err.shape)
        assert np.all(err <= tol), "mel error %.3e over tolerance %.3e (ref=%.5f)" % (err[i], tol[i], ref[i])
    return float(err.max()) if ref.size else 0.0


def wake_clip(name):
    """the int16 PCM of the golden wake-word clip of `name` ("crnn" / "wavenet")"""
    return np.load(os.path.join(GOLDEN, "wake_%s_pcm.npy" % name))


# ------------------------------------------------------------------------------------ dense push schedules
class Push:
    def __init__(self, n, n_streams, speech, active, threshold, reset=None):
        self.n, self.n_streams, self.threshold = int(n), int(n_streams), float(threshold)
        self.speech = np.asarray(speech, bool)
        self.active = np.asarray(active, bool)
        self.reset = None if reset is None else np.asarray(reset, np.uint8)


class Schedule:
    """pushes + per-stream PCM; stream s consumes its own PCM only in the pushes that cover it."""

    def __init__(self, name, cap, max_chunk, a, pcm, pushes):
        self.name, self.cap, self.max_chunk, self.a = name, cap, max_chunk, float(a)
        self.pushes = pushes
        cur = np.zeros(cap, np.int64)
        self.chunks = []
        for p in pushes:
            S = p.n_streams
            assert 1 <= S <= cap and 1 <= p.n <= max_chunk
            c = np.stack([pcm[s, cur[s]:cur[s] + p.n] for s in range(S)])
            assert c.shape == (S, p.n), "stream PCM too short for the script"
            self.chunks.append(c)
            cur[:S] += p.n
        self.max_frames = (max_chunk - 1) // R.HOP + 1


def _clip_runs(n, seed):
    """noise with runs at both int16 rails: -32768 / 32767 become -1.0000305 / 1.0 before the clip to [-1, 1]"""
    x = synth.stream_int16(n, 0, seed, 3)
    r = np.random.default_rng(seed)
    for at in r.integers(0, n - 400, size=max(1, n // 3000)):
        x[at:at + r.integers(40, 400)] = -32768 if r.random() < 0.5 else 32767
    return x


def stream_pcm(cap, n, seed):
    pcm = np.stack([synth.stream_int16(n, (s % 5) + (s % 5 > 2), seed, s) for s in range(cap)])
    pcm[0, 3000:3000 + 35200] = wake_clip("crnn")[:n - 3000]
    if cap > 4:
        pcm[4, 6000:6000 + 35200] = wake_clip("wavenet")[:n - 6000]
    if cap > 3:
        pcm[3] = _clip_runs(n, seed)
    return pcm


def _ragged(name, cap, n_push, a, seed, thresholds):
    """max_chunk = 1601 on one allocation: every chunk size of CHUNKS, a push that completes exactly max_frames frames,
    pushes that complete none, pushes over prefixes of the streams, masked resets (one mask shorter than cap) and the
    speech / activation scripts below."""
    r = np.random.default_rng(seed)
    ns = list(CHUNKS)                                   # 1 + 7 + 159 + 160 + 161 = 488 < 512 samples after five pushes
    total = sum(ns)
    fix = (R.FFT + 159 - total) % R.HOP or R.HOP        # leaves 511 samples pending: the next 1601 completes 11 frames
    ns += [fix, 1601]
    ns += [int(v) for v in r.choice(CHUNKS, size=n_push - len(ns))]
    speech = np.ones((n_push, cap), bool)
    active = np.zeros((n_push, cap), bool)
    speech[:10, 1] = False                              # stream 1: silence, then speech (no fall)
    speech[25:30, 2] = False                            # stream 2: speech, a fall at push 25 (reset), speech again
    if cap > 5:
        speech[45:47, 5] = False
    active[40:48, 0] = True                             # streams 0 / 4: active for a stretch, then sampling again
    if cap > 4:
        active[50:56, 4] = True
    n_streams = np.full(n_push, cap)
    n_streams[12:17] = cap - 1                          # the last stream sits out five pushes
    n_streams[20:22] = 1
    n_streams[33:36] = cap // 2
    resets = {28: [0, 1, 0, 1, 0, 1][:cap - 1]}         # shorter than cap: the streams past its end keep their state
    if n_push > 52:
        m = np.zeros(cap, np.uint8)
        m[[0, cap - 1]] = 1
        resets[52] = m
    pushes = [Push(ns[i], n_streams[i], speech[i], active[i], thresholds[(i // 8) % len(thresholds)], resets.get(i))
              for i in range(n_push)]
    pcm = stream_pcm(cap, sum(ns) + 1, seed)
    return Schedule(name, cap, 1601, a, pcm, pushes)


def _long(name, a):
    """max_chunk = 16000: 97 then 100 (= max_frames) frames per push"""
    cap, n_push = 2, 4
    pcm = np.stack([synth.stream_int16(16000 * n_push, 2, 5, s) for s in range(cap)])
    pcm[0, 8000:8000 + 35200] = wake_clip("crnn")
    pcm[1, 20000:20000 + 35200] = wake_clip("wavenet")
    pushes = [Push(16000, cap, np.ones(cap), np.zeros(cap), 0.9) for _ in range(n_push)]
    return Schedule(name, cap, 16000, a, pcm, pushes)


SCHEDULES = {
    "ragged_pe": lambda: _ragged("ragged_pe", 10, 64, 0.97, 1, (0.5, 0.9)),
    "ragged": lambda: _ragged("ragged", 7, 40, 0.0, 2, (0.5,)),
    "long_pe": lambda: _long("long_pe", 0.97),
}
_SCHED_CACHE = {}


def schedule(name):
    if name not in _SCHED_CACHE:
        _SCHED_CACHE[name] = SCHEDULES[name]()
    return _SCHED_CACHE[name]


# ------------------------------------------------------------------------------------ indexed push scripts
class IPush:
    def __init__(self, ids, lens, speech, active, threshold, reset=None):
        self.ids = np.asarray(ids, np.int32)
        self.lens = np.asarray(lens, np.int32)
        self.speech = np.asarray(speech, bool)      # per entry
        self.active = np.asarray(active, bool)      # per entry
        self.threshold = float(threshold)
        self.reset = None if reset is None else np.asarray(reset, np.uint8)   # [cap] mask applied before the push


def _frames_done(pending, n, active, fall):
    """the samples a stream keeps pending and the frames its chunk completes (TriggerOracle's sample loop)"""
    if active:
        return pending, 0
    pending += n
    k = 0
    while pending >= R.FFT:
        pending -= R.HOP
        k += 1
    return (0 if fall else pending), k


class IndexedSchedule:
    """pushes + per-slot PCM; slot s consumes its own PCM in the order of the pushes that name it.  `frames[i][j]` is
    the number of frames entry j of push i completes (counted on the host)."""

    def __init__(self, name, cap, a, pushes, seed):
        self.name, self.cap, self.a, self.pushes = name, cap, float(a), pushes
        need = np.zeros(cap, np.int64)
        for p in pushes:
            need[p.ids] += p.lens
        pcm = stream_pcm(cap, max(int(need.max()) + 1, 40000), seed)
        pcm[0], pcm[4] = np.roll(pcm[0], -2500), np.roll(pcm[4], -5500)   # the wake clips start at sample 500
        cur = np.zeros(cap, np.int64)
        pend = np.zeros(cap, np.int64)
        speech = np.ones(cap, bool)
        self.chunks, self.frames = [], []
        for p in pushes:
            if p.reset is not None:
                pend[p.reset[:cap] != 0] = 0
            self.chunks.append([pcm[s, cur[s]:cur[s] + n] for s, n in zip(p.ids, p.lens)])
            fr = []
            for s, n, sp, ac in zip(p.ids, p.lens, p.speech, p.active):
                pend[s], k = _frames_done(pend[s], n, ac, speech[s] and not sp)
                speech[s] = sp
                fr.append(k)
            self.frames.append(fr)
            cur[p.ids] += p.lens

    def packed(self, i):
        return np.concatenate(self.chunks[i])


def indexed_script(name, cap, n_push, a, seed, thresholds):
    """Random subsets of the slots in random order, each slot with its own chunk length from SIZES, plus:
    slot `absent` sits out pushes 10..21, push 3 names only the highest slot, push 7 every slot (shuffled), push 31
    has entries that complete max_frames frames and 0 frames, speech falls, active stretches and masked resets.
    Slots 0 and 4 (the wake clips) are named in most pushes."""
    r = np.random.default_rng(seed)
    absent = cap // 2
    speech = np.ones((n_push, cap), bool)
    active = np.zeros((n_push, cap), bool)
    speech[5:9, 1] = False                      # silence then speech
    speech[14:17, 2] = False                    # a fall on slot 2 (clears its ring) ...
    speech[14:16, 3] = False                    # ... and on its neighbour 3
    speech[40:44, cap - 1] = False
    active[20:27, 0] = True                     # slots 0 / 4: active for a stretch, then sampling again
    active[36:41, 4] = True
    resets = {12: np.arange(cap) % 3 == 0, 26: np.arange(cap) == cap - 1, 45: np.arange(cap) % 2 == 1}
    pend = np.zeros(cap, np.int64)
    was = np.ones(cap, bool)
    pushes = []
    for i in range(n_push):
        if i == 3:
            ids = [cap - 1]
        elif i == 7:
            ids = list(r.permutation(cap))
        else:
            pool = [s for s in range(cap) if not (10 <= i <= 21 and s == absent)]
            ids = list(r.choice(pool, size=int(r.integers(1, len(pool) + 1)), replace=False))
            ids += [s for s in (0, 4) if s not in ids and r.random() < 0.8]
            r.shuffle(ids)
        lens = [int(v) for v in r.choice(SIZES, size=len(ids))]
        reset = resets.get(i)
        if reset is not None:
            pend[reset] = 0
        if i in (30, 31):
            rest = [s for s in ids if s not in (5, 6)]
            ids, lens = [5, 6] + rest, [0, 0] + lens[-len(rest):] if rest else [0, 0]
            if i == 30:       # slot 5 to exactly 511 pending samples, slot 6 to at most 510
                lens[0] = 511 - int(pend[5]) if pend[5] < 511 else R.HOP
                lens[1] = 1 if pend[6] <= 509 else 200
            else:             # slot 5: 1601 samples complete max_frames frames; slot 6: 1 sample completes none
                ids[0], ids[1] = 6, 5
                lens[0], lens[1] = 1, MAX_CHUNK
        ids = np.array(ids, np.int32)
        sp, ac = speech[i, ids], active[i, ids]
        for s, n, spk, act in zip(ids, lens, sp, ac):
            pend[s], _ = _frames_done(pend[s], n, act, was[s] and not spk)
            was[s] = spk
        pushes.append(IPush(ids, lens, sp, ac, thresholds[(i // 8) % len(thresholds)],
                            None if reset is None else reset.astype(np.uint8)))
    return IndexedSchedule(name, cap, a, pushes, seed)


SCRIPTS = {
    "idx": lambda: indexed_script("idx", 12, 56, 0.0, 21, (0.5, 0.9)),
    "idx_pe": lambda: indexed_script("idx_pe", 12, 56, 0.97, 22, (0.9, 0.5)),
}
_SCRIPT_CACHE = {}


def script(name):
    if name not in _SCRIPT_CACHE:
        _SCRIPT_CACHE[name] = SCRIPTS[name]()
    return _SCRIPT_CACHE[name]


def pipeline_script():
    """the pipeline config and the CRNN PCM / raw VAD script of the golden pipeline run"""
    g = np.load(os.path.join(GOLDEN, "reference_pipeline.npz"))
    cfg = dict(zip(("frame_width", "vad_rise_delay", "vad_fall_delay", "min_active", "max_active"), [int(v) for v in g["cfg"]]))
    pcm0, raw0 = g["pipe_crnn_pcm"], g["pipe_crnn_raw"]
    return cfg, pcm0, raw0


# ------------------------------------------------------------------------------------ engines, pushes and runs
def engine(model, precision, cap, max_chunk=MAX_CHUNK, device=0):
    """an Engine on `device` with stream state for cap streams of up to max_chunk samples per push"""
    from wakeword_detection_b200 import _cabi
    eng = _cabi.Engine(load_weights(model), device, precision)
    eng.stream_alloc(cap, max_chunk)
    return eng


def host(res):
    """a push's device outputs (post, n_post, trigger, post_max) as numpy arrays"""
    return tuple(x.cpu().numpy() for x in res)


def push_indexed(eng, sch, i, m=None):
    """push i of the indexed script `sch`, slot s as slot m[s]"""
    p = sch.pushes[i]
    ids = p.ids if m is None else m[p.ids]
    return host(eng.stream_push_indexed(ids, sch.packed(i), p.lens, p.speech.astype(np.uint8), p.active.astype(np.uint8),
                                        sch.a, p.threshold))


def _reset(eng, sch, i, m=None, cap=None):
    p = sch.pushes[i]
    if p.reset is None:
        return
    if m is None:
        eng.stream_reset(p.reset)
        return
    mask = np.zeros(cap, np.uint8)
    mask[m[np.nonzero(p.reset)[0]]] = 1
    eng.stream_reset(mask)


def run_indexed(eng, sch, start=0, stop=None, m=None, cap=None, before=None):
    """pushes start..stop-1 of the indexed script `sch` with their resets, slot s as slot m[s] of a context with cap
    slots; before(i) runs before push i's reset"""
    outs = []
    for i in range(start, len(sch.pushes) if stop is None else stop):
        if before is not None:
            before(i)
        _reset(eng, sch, i, m, cap)
        outs.append(push_indexed(eng, sch, i, m))
    return outs


def assert_same_rows(o1, o2, rows=slice(None)):
    """the outputs of two runs equal on `rows` of every push (NaN equal to NaN)"""
    for i, (x, y) in enumerate(zip(o1, o2)):
        for a, b in zip(x, y):
            assert np.array_equal(a[rows], b[rows], equal_nan=True), i
