"""Stream state records (wwb_stream_export / wwb_stream_import, csrc/stream_state.cu): a stream's state out of its slot
and back, into the same slot, another slot, another context (other capacity, max_chunk, precision) or another GPU.

The record is the reference's WakewordTrigger state (oracle: TriggerOracle), plus the VAD debounce and ActivationTimeout
state on a pipeline context (PipelineOracle).  Every check below is against the oracle or against an uninterrupted run of
the same script, bit for bit: after an import the slot's window holds the same rows as the exporting slot's, so every
later posterior is computed from the same inputs.

The scripts are the indexed ones of test_gpu_stream_indexed.py (streaming_helpers.py builds them).
"""
import ctypes as C
import os
import re
import struct

import numpy as np
import pytest

from conftest import ROOT, WEIGHTS, load_weights
from oracle import restated as R
from streaming_helpers import (MODELS, PRECISIONS, SCRIPTS, TOL, check_mel, engine, host, pipeline_script, run_indexed,
                               script)
from wakeword_detection_b200 import _cabi

# after these pushes of the indexed scripts the tests export every slot.  30: slot 5 holds exactly 511 pending samples;
# 14 / 16: slot 2's ring was just cleared by a VAD fall; 23: slot 0 inside its active stretch (20..26); 12: after a masked
# reset; 12 .. 21: slot 6 (cap // 2) is absent from the pushes
CUTS = (3, 11, 12, 14, 15, 16, 21, 23, 30, 31, 55)
B_CAP, B_CHUNK = 40, 4000      # the importing context: other capacity, other ring size

OFFSETS = {"magic": 0, "version": 4, "flags": 6, "kind": 8, "mel_length": 12, "n_pending": 16, "prev_sample": 20,
           "post_max": 24, "was_speech": 28, "is_speech": 29, "is_active": 30, "t_is_speech": 31, "run_value": 32,
           "run_length": 36, "active_length": 40, "reserved": 44}
PIPE_FIELDS = ("is_speech", "is_active", "t_is_speech", "run_value", "run_length", "active_length")


class HeaderC(C.Structure):
    """a C caller's view of wwb_stream_state_header"""
    _fields_ = [("magic", C.c_uint32), ("version", C.c_uint16), ("flags", C.c_uint16), ("kind", C.c_int32),
                ("mel_length", C.c_int32), ("n_pending", C.c_int32), ("prev_sample", C.c_float), ("post_max", C.c_float),
                ("was_speech", C.c_uint8), ("is_speech", C.c_uint8), ("is_active", C.c_uint8), ("t_is_speech", C.c_uint8),
                ("run_value", C.c_int32), ("run_length", C.c_int32), ("active_length", C.c_int32),
                ("reserved", C.c_uint32)]


# ------------------------------------------------------------------------------------ 1: the layout (no GPU)
def test_record_header_layout():
    """the numpy dtype, a ctypes mirror and the header's own declaration agree: 48 bytes, the documented offsets"""
    dt = _cabi.STREAM_STATE_HEADER
    assert dt.itemsize == 48 and C.sizeof(HeaderC) == 48
    assert list(dt.names) == list(OFFSETS) == [f[0] for f in HeaderC._fields_]
    for k, off in OFFSETS.items():
        assert dt.fields[k][1] == off, k
        assert getattr(HeaderC, k).offset == off, k
    text = open(os.path.join(ROOT, "include", "wwb200.h")).read()
    body = re.search(r"typedef struct \{([^{}]*)\} wwb_stream_state_header;", text).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    declared = [n for decl in body.split(";") for n in re.findall(r"(\w+)\s*$", decl.strip())]
    assert declared == list(OFFSETS)
    assert re.search(r"#define WWB_STREAM_STATE_MAGIC 0x53425757u", text)
    assert re.search(r"#define WWB_STREAM_STATE_VERSION 1\b", text)
    assert re.search(r"#define WWB_VERSION 100\b", text)
    assert _cabi.stream_state_dtype(151).itemsize == 26256
    assert _cabi.stream_state_dtype(182).itemsize == 31216
    assert struct.pack("<I", _cabi.STREAM_STATE_MAGIC) == b"WWBS"


def test_decode_round_trips_a_hand_built_record():
    import torch
    L, n = 182, 3
    r = np.random.default_rng(0)
    rec = np.zeros(n, _cabi.stream_state_dtype(L))
    h = rec["header"]
    vals = {"magic": [_cabi.STREAM_STATE_MAGIC] * n, "version": [1] * n, "flags": [0, 1, 1], "kind": [1] * n,
            "mel_length": [L] * n, "n_pending": [0, 511, 37], "prev_sample": r.standard_normal(n),
            "post_max": r.random(n), "was_speech": [1, 0, 1], "is_speech": [0, 1, 1], "is_active": [0, 1, 0],
            "t_is_speech": [0, 0, 1], "run_value": [0, 1, 0], "run_length": [0, 7, 123], "active_length": [0, 31, 2],
            "reserved": [0] * n}
    for k, v in vals.items():
        h[k] = v
    rec["pending"][1, :511] = r.standard_normal(511)
    rec["pending"][2, :37] = r.standard_normal(37)
    rec["mel"] = r.standard_normal((n, L, 40))
    raw = rec.view(np.uint8).reshape(n, -1)
    assert raw.shape == (n, 48 + 4 * 512 + 160 * L)
    # an independent packing of entry 1's header and of its body offsets
    f = lambda k: h[k][1].item()
    packed = struct.pack("<IHHiiiffBBBBiiiI", *[f(k) for k in OFFSETS])
    assert raw[1, :48].tobytes() == packed
    assert raw[1, 48:48 + 2048].tobytes() == rec["pending"][1].astype("<f4").tobytes()
    assert raw[1, 2096:].tobytes() == rec["mel"][1].astype("<f4").tobytes()
    for src in (raw, torch.from_numpy(raw.copy()), raw.reshape(-1)):
        d = _cabi.decode_stream_state(src, L)
        for k in OFFSETS:
            assert np.array_equal(d[k], h[k]), k
        assert np.array_equal(d["pending"], rec["pending"]) and np.array_equal(d["mel"], rec["mel"])
    with pytest.raises(ValueError):
        _cabi.decode_stream_state(raw[:, :-4], L)


# ------------------------------------------------------------------------------------ helpers
def _same_bits(xs, ys):
    """outputs of two runs bit for bit; the second context's post rows may be longer (a larger max_chunk): NaN there"""
    assert len(xs) == len(ys)
    for i, (x, y) in enumerate(zip(xs, ys)):
        mf = x[0].shape[1]
        assert np.array_equal(x[0].view(np.uint32), y[0][:, :mf].view(np.uint32)), i
        assert np.isnan(y[0][:, mf:]).all(), i
        for a, b in zip(x[1:], y[1:]):
            assert np.array_equal(a, b), i


def _slots(sch):
    return np.arange(sch.cap, dtype=np.int32)


_SNAP_CACHE = {}


def oracle_states(model, name):
    """per cut: the TriggerOracle of every slot after that push (copies of the state a record carries)"""
    key = (model, name)
    if key in _SNAP_CACHE:
        return _SNAP_CACHE[key]
    w = load_weights(model)
    sch = script(name)
    orc = [R.TriggerOracle(w, 0.5, sch.a) for _ in range(sch.cap)]
    snaps = {}
    for i, (p, chunks) in enumerate(zip(sch.pushes, sch.chunks)):
        if p.reset is not None:
            for s in np.nonzero(p.reset)[0]:
                orc[s].reset()
        for s, chunk, sp, ac in zip(p.ids, chunks, p.speech, p.active):
            orc[s].active = bool(ac)
            orc[s](chunk, bool(sp))
        if i in CUTS:
            snaps[i] = [dict(pending=o.pending.copy(), prev_sample=o.prev_sample, was_speech=o.was_speech,
                             frames=o.frames.copy(), post_max=o.post_max) for o in orc]
    _SNAP_CACHE[key] = snaps
    return snaps


def check_trigger_state(d, j, o, L, tol):
    """entry j of decoded records against a TriggerOracle snapshot"""
    n = o["pending"].size
    assert d["magic"][j] == _cabi.STREAM_STATE_MAGIC and d["version"][j] == 1 and d["mel_length"][j] == L
    assert d["n_pending"][j] == n
    assert np.array_equal(d["pending"][j, :n], o["pending"])
    assert not d["pending"][j, n:].any() and d["reserved"][j] == 0
    assert d["prev_sample"][j] == np.float32(o["prev_sample"])
    assert bool(d["was_speech"][j]) == o["was_speech"]
    check_mel(d["mel"][j], o["frames"])
    assert abs(float(d["post_max"][j]) - o["post_max"]) <= tol


# ------------------------------------------------------------------------------------ 2: the record is the reference's state
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCRIPTS))
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_export_is_the_oracle_state(model, precision, name):
    """After each cut every slot's record equals its TriggerOracle's state: n_pending, the pending samples, prev_sample
    and was_speech exactly (the device's int16 division is the correctly rounded one and pre-emphasis the same two f32
    operations), a zero pending tail, the window within the mel bound, post_max within the posterior tolerance."""
    sch = script(name)
    snaps = oracle_states(model, name)
    eng = engine(model, precision, sch.cap)
    L = eng.L
    seen = {"511": False, "fall": False, "active": False}
    try:
        assert eng.stream_state_bytes() == 48 + 2048 + 160 * L
        for i in range(len(sch.pushes)):
            run_indexed(eng, sch, i, i + 1)
            if i not in CUTS:
                continue
            rec = eng.stream_export(_slots(sch))
            assert rec.shape == (sch.cap, eng.stream_state_bytes()) and rec.device == eng.device
            d = _cabi.decode_stream_state(rec, L)
            assert (d["kind"] == eng.kind).all() and not d["flags"].any()
            assert not any(d[k].any() for k in PIPE_FIELDS)
            for s in range(sch.cap):
                check_trigger_state(d, s, snaps[i][s], L, TOL[precision])
            p = sch.pushes[i]
            seen["511"] |= bool((d["n_pending"] == 511).any())
            seen["fall"] |= bool(2 in p.ids and not d["was_speech"][2] and not d["mel"][2].any())
            seen["active"] |= bool(any(s == 0 and ac for s, ac in zip(p.ids, p.active)) and d["mel"][0].any())
    finally:
        eng.close()
    assert all(seen.values()), seen


# ------------------------------------------------------------------------------------ 3: moved, the stream continues bit for bit
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCRIPTS))
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("model", MODELS)
def test_moved_streams_continue_bit_exact(model, precision, name):
    """Context A (12 slots, max_chunk 1601) runs the script.  At cuts 23 and 30 every slot is exported and imported into a
    context B (40 slots, max_chunk 4000: another capacity and ring size) at permuted slot ids, after B's slots were
    filled with other audio.  B continues the script with the ids and reset masks mapped: every output row of every later
    push equals A's bit for bit."""
    import torch
    sch = script(name)
    recs = {}
    a = engine(model, precision, sch.cap)

    def export_at_cuts(i):
        if i - 1 in (23, 30):
            recs[i - 1] = a.stream_export(_slots(sch))

    try:
        outs_a = run_indexed(a, sch, before=export_at_cuts)
    finally:
        a.close()
    r = np.random.default_rng(7)
    for cut in (23, 30):
        m = r.permutation(B_CAP)[:sch.cap].astype(np.int32)
        b = engine(model, precision, B_CAP, B_CHUNK)
        try:
            noise = torch.randint(-3000, 3000, (B_CAP, B_CHUNK), dtype=torch.int16, device=b.device)
            for _ in range(2):
                b.stream_push(noise, pre_emphasis=0.5)
            b.stream_import(m, recs[cut])
            outs_b = run_indexed(b, sch, cut + 1, m=m, cap=B_CAP)
        finally:
            b.close()
        _same_bits(outs_a[cut + 1:], outs_b)
    assert sum(int(o[1].sum()) for o in outs_a[24:]) > 100


# ------------------------------------------------------------------------------------ 4: across precisions
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCRIPTS))
@pytest.mark.parametrize("model", MODELS)
def test_tc_export_continues_on_f32(model, name):
    """Records exported from a tc context at cut 23 and imported into an f32 context: the window rows do not depend on
    the precision, so posteriors, n_post and triggers equal those of an f32 context that ran the whole script.  post_max
    carries the tc maximum: it equals max(imported post_max, new posteriors) until the slot's next VAD fall or reset,
    and the f32 run's after it."""
    sch = script(name)
    cut = 23
    src, ref, dst = engine(model, "tc", sch.cap), engine(model, "f32", sch.cap), engine(model, "f32", sch.cap)
    try:
        run_indexed(src, sch, 0, cut + 1)
        rec = src.stream_export(_slots(sch))
        outs_ref = run_indexed(ref, sch)
        dst.stream_import(_slots(sch), rec)
        outs = run_indexed(dst, sch, cut + 1)
    finally:
        src.close()
        ref.close()
        dst.close()
    d = _cabi.decode_stream_state(rec, int(load_weights(model)["mel_length"]))
    pm = {s: np.float32(d["post_max"][s]) for s in range(sch.cap)}      # None: follows the f32 run
    was = {s: bool(d["was_speech"][s]) for s in range(sch.cap)}
    carried = 0
    for k, (o, e) in enumerate(zip(outs, outs_ref[cut + 1:])):
        i = cut + 1 + k
        p = sch.pushes[i]
        assert np.array_equal(o[0], e[0], equal_nan=True) and np.array_equal(o[1], e[1]) and np.array_equal(o[2], e[2]), i
        if p.reset is not None:
            for s in np.nonzero(p.reset)[0]:
                pm[s] = None
        for j, s in enumerate(p.ids):
            if pm[s] is None:
                assert o[3][j] == e[3][j], (i, s)
            else:
                n = int(o[1][j])
                pm[s] = max([pm[s]] + list(o[0][j, :n]))
                assert o[3][j] == pm[s], (i, s)
                carried += 1
            if was[s] and not p.speech[j]:
                pm[s] = None
            was[s] = bool(p.speech[j])
    assert carried > 20


# ------------------------------------------------------------------------------------ 5: rewind and reset
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_rewind_and_fresh_import(model):
    """(a) Slots 0 and 4 are exported at cut 23; their pushes of the rest of the script are replayed on their own, the
    records are imported back and the same pushes replayed again: the outputs repeat bit for bit.
    (b) A fresh context's record imported into the used slot 4 makes it a fresh stream: its outputs over slot 4's first
    pushes of the script equal those of a fresh context."""
    sch = script("idx_pe")
    cut = 23
    eng = engine(model, "tc", sch.cap)
    try:
        run_indexed(eng, sch, 0, cut + 1)
        slots = np.array([0, 4], np.int32)
        rec = eng.stream_export(slots)
        solo = [(i, j) for i in range(cut + 1, len(sch.pushes)) for j, s in enumerate(sch.pushes[i].ids) if s in slots]

        def replay(e, items, slot_of=lambda s: s):
            outs = []
            for i, j in items:
                p = sch.pushes[i]
                outs.append(host(e.stream_push_indexed([slot_of(p.ids[j])], sch.chunks[i][j], [p.lens[j]], [p.speech[j]],
                                                       [p.active[j]], sch.a, p.threshold)))
            return outs

        first = replay(eng, solo)
        eng.stream_import(slots, rec)
        again = replay(eng, solo)
        _same_bits(first, again)
        assert sum(int(o[1][0]) for o in first) > 30

        # (b) slot 4 (used, mid-stream) gets slot 1 of a fresh context of another capacity and max_chunk
        fresh_src = engine(model, "tc", 3, 320)
        blank = fresh_src.stream_export([1])
        fresh_src.close()
        early = [(i, j) for i in range(len(sch.pushes)) for j, s in enumerate(sch.pushes[i].ids) if s == 4][:20]
        eng.stream_import([4], blank)
        got = replay(eng, early)
        fresh = engine(model, "tc", sch.cap)
        try:
            want = replay(fresh, early, lambda s: 9)
        finally:
            fresh.close()
        _same_bits(want, got)
        assert sum(int(o[1][0]) for o in got) > 20
    finally:
        eng.close()


# ------------------------------------------------------------------------------------ 6: isolation and purity
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_export_is_pure_and_import_is_isolated(model):
    """An export of every slot before every push (and a second one right after it, byte-identical) leaves the outputs of
    the whole script bit-identical to a run without exports.  Importing other slots' records into slots 2, 7 and 9: those
    slots then export exactly the imported records, and every other slot exports the bytes it exported before."""
    import torch
    sch = script("idx_pe")
    plain, probed = engine(model, "tc", sch.cap), engine(model, "tc", sch.cap)
    ids = _slots(sch)
    try:
        outs_plain = run_indexed(plain, sch)

        def probe(i):
            e1 = probed.stream_export(ids)
            e2 = probed.stream_export(ids)
            assert torch.equal(e1, e2), i

        outs_probed = run_indexed(probed, sch, before=probe)
        _same_bits(outs_plain, outs_probed)

        before = probed.stream_export(ids)
        named, src = np.array([2, 7, 9], np.int32), np.array([5, 0, 11])
        probed.stream_import(named, before[torch.from_numpy(src).to(probed.device)])
        after = probed.stream_export(ids)
        rows = lambda x: torch.from_numpy(np.asarray(x, np.int64)).to(probed.device)
        others = np.setdiff1d(ids, named)
        assert torch.equal(after[rows(others)], before[rows(others)])
        assert torch.equal(after[rows(named)], before[rows(src)])
    finally:
        plain.close()
        probed.close()


# ------------------------------------------------------------------------------------ 7: the device pipeline
def _pipeline_run_inputs(cap, n_step, seed):
    cfg, pcm0, raw0 = pipeline_script()
    rng = np.random.default_rng(seed)
    lens_of = [320, 160, 319, 1, 320, 240, 7, 320]
    rows = [np.roll(pcm0, 977 * s) for s in range(cap)]
    raws = [np.roll(raw0, 5 * s) ^ (rng.random(raw0.size) < 0.03) for s in range(cap)]
    cur, k = np.zeros(cap, np.int64), np.zeros(cap, np.int64)
    steps = []
    for _ in range(n_step):
        ids = rng.permutation(cap)[:int(rng.integers(1, cap + 1))].astype(np.int32)
        frames, raw = [], []
        for s in ids:
            n = lens_of[s % len(lens_of)]
            frames.append(rows[s][cur[s]:cur[s] + n])
            raw.append(raws[s][k[s] % raws[s].size])
            cur[s] += n
            k[s] += 1
        steps.append((ids, frames, np.array(raw, np.uint8)))
    return cfg, steps


def _pipe_host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
def test_pipeline_records_and_continuation():
    """MultiStreamPipeline.step_streams, CRNN, pre-emphasis 0.97, rise / fall / min / max-active delays of the golden
    pipeline config, 8 slots, 300 steps; every slot is exported after every step.
    - Each record's pipeline fields equal the PipelineOracle's (vad.run_value / run_length, is_speech, tmo.is_speech,
      tmo.active_length, trig.active), flags bit 0 set, and its trigger fields equal the oracle's trigger state.
    - At a step where slots are active and others mid-debounce, the records go into a second pipeline context
      (16 slots, permuted ids), which continues the run: all seven outputs equal the uninterrupted run's bit for bit.
    - A trigger-only record imported into a pipeline slot with live pipeline state gives that slot the initial
      pipeline state and the record's trigger state."""
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    model, a, cap = "CRNN", 0.97, 8
    w = load_weights(model)
    L = int(w["mel_length"])
    cfg, steps = _pipeline_run_inputs(cap, 300, 13)
    assert all(cfg[k] > 0 for k in ("vad_rise_delay", "vad_fall_delay", "min_active", "max_active"))
    ids_all = np.arange(cap, dtype=np.int32)
    oracles = [R.PipelineOracle(w, a=a, **cfg) for _ in range(cap)]
    pipe = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, cap, pre_emphasis=a, **cfg)
    outs, recs, cut = [], [], None
    try:
        for i, (ids, frames, raw) in enumerate(steps):
            outs.append(_pipe_host(pipe.step_streams(ids, frames, raw)))
            near = set()
            for j, s in enumerate(ids):
                before = len(oracles[s].trig.posteriors)
                oracles[s](frames[j], raw[j])
                new = np.array(oracles[s].trig.posteriors[before:])
                if new.size and np.abs(new - 0.5).min() <= 1e-3:
                    near.add(s)      # the trigger decision may differ within the posterior tolerance
            rec = pipe.export_streams(ids_all)
            recs.append(rec)
            d = _cabi.decode_stream_state(rec, L)
            assert (d["flags"] == _cabi.STREAM_STATE_PIPELINE).all(), i
            for s, o in enumerate(oracles):
                want = {"run_value": int(o.vad.run_value), "run_length": o.vad.run_length, "is_speech": int(o.is_speech),
                        "t_is_speech": int(o.tmo.is_speech), "active_length": o.tmo.active_length,
                        "is_active": int(o.trig.active)}
                got = {k: int(d[k][s]) for k in want}
                if s not in near:
                    assert got == want, (i, s, got, want)
                t = o.trig
                check_trigger_state(d, s, dict(pending=t.pending, prev_sample=t.prev_sample, was_speech=t.was_speech,
                                               frames=t.frames, post_max=t.post_max), L, 1e-3)
            mid = [s for s, o in enumerate(oracles) if int(o.vad.run_value) != int(o.is_speech)]
            if cut is None and i >= 60 and any(o.trig.active for o in oracles) and mid:
                cut = i
    finally:
        pipe.close()
    assert cut is not None

    m = np.random.default_rng(3).permutation(16)[:cap].astype(np.int32)
    pipe_b = MultiStreamPipeline(os.path.join(WEIGHTS, model), model, 16, pre_emphasis=a, **cfg)
    try:
        pipe_b.import_streams(m, recs[cut])
        assert torch_equal(pipe_b.export_streams(m), recs[cut])
        n_win = 0
        for i in range(cut + 1, len(steps)):
            ids, frames, raw = steps[i]
            got = _pipe_host(pipe_b.step_streams(m[ids], frames, raw))
            assert got.keys() == outs[i].keys()
            for k in got:
                assert np.array_equal(got[k], outs[i][k], equal_nan=True), (i, k)
            n_win += int(got["n_post"].sum())
        assert n_win > 100

        # a trigger-only record (no pipeline state) into slot m[s] of the pipeline context
        trig = engine(model, "tc", 2, 1601)
        try:
            pcm = np.concatenate([c for c in steps[0][1]] + [np.zeros(600, np.int16)])[:600]
            trig.stream_push_indexed([1], pcm, [600], pre_emphasis=a)
            solo = trig.stream_export([1])
        finally:
            trig.close()
        ds = _cabi.decode_stream_state(solo, L)
        assert ds["flags"][0] == 0 and ds["n_pending"][0] > 0
        live = pipe_b.export_streams(m)
        dl = _cabi.decode_stream_state(live, L)
        s = int(np.argmax([sum(int(dl[k][j]) for k in PIPE_FIELDS) for j in range(cap)]))
        assert any(dl[k][s] for k in PIPE_FIELDS)
        pipe_b.import_streams(m[s:s + 1], solo)
        dn = _cabi.decode_stream_state(pipe_b.export_streams(m[s:s + 1]), L)
        assert dn["flags"][0] == _cabi.STREAM_STATE_PIPELINE
        for k in PIPE_FIELDS:
            assert dn[k][0] == 0, k
        for k in ("n_pending", "prev_sample", "post_max", "was_speech", "pending", "mel"):
            assert np.array_equal(dn[k], ds[k]), k
    finally:
        pipe_b.close()


def torch_equal(x, y):
    import torch
    return torch.equal(x.to(y.device), y)


# ------------------------------------------------------------------------------------ 8: rejected calls change nothing
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_rejections_change_nothing(model):
    """Table errors raise IndexError before any device work; bad records raise ValueError naming the entry and the
    reason, and no record of the batch is applied (also when only the last one is bad).  After each, an export of every
    slot is byte-identical to the one taken before.  A dense context_step rejected for its chunk length, a NULL pcm or a
    filter-only ctx launches no kernel: the VAD debounce and trigger state of every slot export unchanged."""
    import torch
    w = load_weights(model)
    other = "Wavenet" if model == "CRNN" else "CRNN"
    unalloc = _cabi.Engine(w, 0, "tc")
    filt = _cabi.Engine({k: w[k] for k in ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")}, 0, "tc")
    try:
        filt.stream_alloc(4, 320)
        for e in (unalloc, filt):
            assert e.stream_state_bytes() == 0
            with pytest.raises(IndexError):
                e.stream_export([0])
            with pytest.raises(IndexError):
                e.stream_import([0], np.zeros((1, 48), np.uint8))
        filt.context_alloc()
        n0 = filt.launch_count()
        with pytest.raises(IndexError):
            filt.context_step(np.zeros((4, 160), np.int16))
        assert filt.launch_count() == n0
    finally:
        unalloc.close()
        filt.close()
    pipe = engine(model, "tc", 4, 320)
    try:
        pipe.context_alloc()
        noise = torch.randint(-3000, 3000, (4, 320), dtype=torch.int16, device=pipe.device)
        for raw in ([1, 0, 1, 0], [1, 1, 0, 0]):
            pipe.context_step(noise, raw)
        four = np.arange(4, dtype=np.int32)
        p0, n0 = pipe.stream_export(four), pipe.launch_count()
        with pytest.raises(IndexError):
            pipe.context_step(np.zeros((4, 321), np.int16))
        assert pipe.lib.wwb_context_step(pipe.ctx, None, 4, 320, None, C.c_float(0), C.c_float(0.5), *([None] * 7),
                                         pipe._stream()) == -1
        assert pipe.launch_count() == n0
        assert torch.equal(pipe.stream_export(four), p0)
    finally:
        pipe.close()
    src = engine(other, "tc", 2, 320)
    try:
        foreign = src.stream_export([0, 1])
    finally:
        src.close()

    sch = script("idx_pe")
    cap = sch.cap
    eng = engine(model, "tc", sch.cap)
    nb = eng.stream_state_bytes()
    try:
        run_indexed(eng, sch, 0, 31)
        ids = _slots(sch)
        e0 = eng.stream_export(ids)

        def unchanged():
            assert torch.equal(eng.stream_export(ids), e0)

        for bad in ([], np.arange(cap + 1) % cap, [0, cap], [3, -1], [5, 2, 5]):
            bad = np.asarray(bad, np.int32)
            with pytest.raises(IndexError):
                eng.stream_export(bad)
            recs = e0[torch.from_numpy(np.arange(bad.size) % cap).to(eng.device)]
            with pytest.raises(IndexError):
                eng.stream_import(bad, recs)
            unchanged()
        out = torch.empty((2, nb), dtype=torch.uint8, device=eng.device)
        status = torch.zeros(2, dtype=torch.int32, device=eng.device)
        two = np.array([0, 1], np.int32)
        assert eng.lib.wwb_stream_export(eng.ctx, None, 2, out.data_ptr(), eng._stream()) == -1
        assert eng.lib.wwb_stream_export(eng.ctx, two.ctypes.data, 2, None, eng._stream()) == -1
        assert eng.lib.wwb_stream_export(eng.ctx, two.ctypes.data, 2, out.data_ptr() + 4, eng._stream()) == -1
        assert eng.lib.wwb_stream_import(eng.ctx, two.ctypes.data, 2, out.data_ptr(), None, eng._stream()) == -1
        unchanged()

        # six good records of other slots (applying them would change slots 0..5), then one field of one made bad
        n = 6
        good = e0[torch.from_numpy(np.array([7, 9, 11, 8, 10, 6])).to(eng.device)].cpu().numpy()
        hdr = lambda r: r[:, :48].view(_cabi.STREAM_STATE_HEADER)[:, 0]

        def corrupt(j, field=None, value=None, record=None):
            r = good.copy()
            if record is not None:
                k = min(nb, record.size)
                r[j] = 0
                r[j, :k] = record[:k]
            else:
                hdr(r)[field][j] = value
            return r

        L = eng.L
        cases = [(corrupt(3, "magic", 0x53425758), 3, "magic"),
                 (corrupt(3, "version", 2), 3, "version"),
                 (corrupt(3, record=foreign[0].cpu().numpy()), 3, "model kind"),
                 (corrupt(3, "mel_length", L - 1), 3, "mel_length"),
                 (corrupt(3, "n_pending", 512), 3, "n_pending"),
                 (corrupt(3, "n_pending", -1), 3, "n_pending"),
                 (corrupt(3, "flags", 2), 3, "flag"),
                 (corrupt(3, "flags", 0x8001), 3, "flag"),
                 (corrupt(n - 1, "magic", 0), n - 1, "magic")]
        r2 = corrupt(4, "version", 0)
        hdr(r2)["n_pending"][2] = 600
        cases.append((r2, 2, "n_pending"))                        # two bad records: the lower entry is reported
        for recs, j, why in cases:
            with pytest.raises(ValueError, match=r"^record %d: .*%s" % (j, why)):
                eng.stream_import(np.arange(n), recs)
            unchanged()
        # the status the C ABI reports for the last-only case: 1 + entry, reason code
        dev = torch.from_numpy(cases[-2][0]).to(eng.device)
        assert eng.lib.wwb_stream_import(eng.ctx, np.arange(n, dtype=np.int32).ctypes.data, n, dev.data_ptr(),
                                         status.data_ptr(), eng._stream()) == 0
        assert status.cpu().tolist() == [n, 1]
        unchanged()
        # and the same batch without the bad record is applied
        eng.stream_import(np.arange(n), good)
        assert torch.equal(eng.stream_export(np.arange(n)).cpu(), torch.from_numpy(good))
    finally:
        eng.close()


# ------------------------------------------------------------------------------------ 9: across GPUs
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["CRNN", "Wavenet"])
def test_move_to_another_gpu(model):
    """Records exported on cuda:0 at cut 23, moved with .to("cuda:1") and imported into a context on device 1 (40 slots,
    max_chunk 4000, permuted ids): the rest of the script gives A's outputs bit for bit."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    sch = script("idx_pe")
    cut = 23
    a = engine(model, "tc", sch.cap)
    try:
        run_indexed(a, sch, 0, cut + 1)
        rec = a.stream_export(_slots(sch))
        outs_a = run_indexed(a, sch, cut + 1)
    finally:
        a.close()
    m = np.random.default_rng(9).permutation(B_CAP)[:sch.cap].astype(np.int32)
    b = engine(model, "tc", B_CAP, B_CHUNK, device=1)
    try:
        moved = rec.to("cuda:1")
        b.stream_import(m, moved)
        with torch.cuda.device(1):
            outs_b = run_indexed(b, sch, cut + 1, m=m, cap=B_CAP)
    finally:
        b.close()
    _same_bits(outs_a, outs_b)
