"""CRNN models of any window length L = 17..256 frames: the conv geometry, the kernels at every precision, sliding
windows on both column paths, streaming pushes, state records, the trigger chain and the Python drop-ins, on synthetic
models drawn at the shipped models' weight stds.

The lengths cover every residue mod 8 and both ends of the range.  L = 1, 2, 3 mod 8 (17, 50, 97, 99, 201) give three or
four padded conv columns, the others two; L = 17 has no interior column at all.  The truth is the oracle in float64
(oracle.restated, dtype=np.float64).  Tolerances as in test_gpu_synthetic_models.py: 1e-3 (2e-2 for tc_fast)."""
import os

import numpy as np
import pytest

from conftest import WEIGHTS, load_weights
from crnn_models import calibrate, geometry, mel_windows, shared_launches, synth_crnn
from oracle import restated as R
from streaming_helpers import CHUNKS, MAX_CHUNK, assert_same_rows, stream_pcm, wake_clip
from wakeword_detection_b200 import synth

F64 = np.float64
POST_ATOL = 1e-3
FAST_ATOL = 2e-2
LENGTHS = [17, 24, 50, 97, 99, 101, 124, 150, 151, 201, 256]
STATS = []


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for line in STATS:
        print("\n[crnn L] " + line)


_MODELS = {}


def model(L, n_out=2, seed=0):
    """(weights, windows, float64 encoder / detect / posteriors), cached"""
    key = (L, n_out, seed)
    if key not in _MODELS:
        X = mel_windows(L)
        w = calibrate(synth_crnn(seed, L, n_out), X)
        enc = R.encode(X, w, F64)
        det = R.detect(enc, w, F64)
        assert np.mean((det[:, -1] >= 0.05) & (det[:, -1] <= 0.95)) >= 0.5, "posteriors saturated"
        _MODELS[key] = (w, X, enc, det, det[:, -1])
    return _MODELS[key]


def _err(a, b):
    return float(np.abs(np.asarray(a, F64) - np.asarray(b, F64)).max())


def _engine(w, precision):
    from wakeword_detection_b200 import _cabi
    return _cabi.Engine(w, 0, precision)


# ------------------------------------------------------------------------------------ CPU
def test_geometry_table():
    """the padded columns per residue mod 8, as the kernels derive them"""
    assert geometry(151) == (19, 6, [0, 18])
    assert geometry(97) == (13, 9, [0, 1, 11, 12]) and geometry(99) == (13, 8, [0, 11, 12])
    assert geometry(17) == (3, 9, [0, 1, 2]) and geometry(256) == (32, 6, [0, 31])
    for L in range(17, 257):
        T, pad_lo, padded = geometry(L)
        assert 12 <= 8 * T + 12 - L <= 19
        assert len(padded) == min(T, 2 + (L % 8 in (1, 2)) + (L % 8 in (1, 2, 3))), L


@pytest.mark.parametrize("L", LENGTHS)
def test_oracle_conv_is_tf_same(L):
    """oracle.crnn_conv equals a direct float64 loop convolution with the TF SAME rule (out = ceil(in / stride), the
    padding total split with the smaller half first) at every length"""
    r = np.random.default_rng(L)
    w = {"conv_w": r.standard_normal((32, 5, 20)), "conv_b": r.standard_normal(32)}
    x = r.random((2, L, 40)) * 4
    T = -(-L // 8)
    pt = max((T - 1) * 8 + 20 - L, 0)
    pf = max((20 - 1) * 2 + 5 - 40, 0)
    want = np.zeros((2, T, 20, 32))
    for t in range(T):
        for f in range(20):
            acc = np.tile(w["conv_b"], (2, 1))
            for kt in range(20):
                i = 8 * t + kt - pt // 2
                if not 0 <= i < L:
                    continue
                for kf in range(5):
                    j = 2 * f + kf - pf // 2
                    if 0 <= j < 40:
                        acc = acc + x[:, i, j, None] * w["conv_w"][None, :, kf, kt]
            want[:, t, f] = np.maximum(acc, 0)
    got = R.crnn_conv(x, w, F64)
    assert got.shape == (2, T, 640)
    assert np.abs(got - want.reshape(2, T, 640)).max() < 1e-10


# ------------------------------------------------------------------------------------ GPU: independent windows
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "tc", "tc_fast"])
@pytest.mark.parametrize("n_out", [1, 2])
@pytest.mark.parametrize("L", LENGTHS)
def test_windows_vs_float64(L, n_out, precision):
    """encoder output, detect output and posteriors of independent windows against float64; decisions exact outside
    the band around 0.5"""
    w, X, enc64, det64, ref = model(L, n_out)
    tol = FAST_ATOL if precision == "tc_fast" else POST_ATOL
    eng = _engine(w, precision)
    try:
        assert eng.L == L
        enc_t = eng.encode(X)
        enc = enc_t.cpu().numpy()
        det = eng.detect(enc_t).cpu().numpy()
        post = eng.posteriors(X, hop=1).cpu().numpy()[:, 0]
    finally:
        eng.close()
    e = (_err(enc, enc64), _err(det, det64), _err(post, ref))
    STATS.append("L=%d n_out=%d %s: enc %.2e det %.2e post %.2e" % ((L, n_out, precision) + e))
    assert det.shape == det64.shape and np.isfinite(post).all()
    assert max(e) < tol, e
    if precision != "tc_fast":
        band = np.abs(ref - 0.5) <= POST_ATOL
        assert np.array_equal((post > 0.5)[~band], (ref > 0.5)[~band])


# ------------------------------------------------------------------------------------ GPU: sliding windows
def _posteriors(eng, X, hop, no_share):
    os.environ["WWB_CRNN_NO_SHARE"] = "1" if no_share else "0"
    try:
        n0 = eng.launch_count()
        out = eng.posteriors(X, hop=hop).clone()
        return out, eng.launch_count() - n0
    finally:
        os.environ["WWB_CRNN_NO_SHARE"] = "0"


@pytest.mark.gpu
@pytest.mark.parametrize("L", LENGTHS)
def test_sliding_shared_columns_bit_identical(L):
    """Hops 1, 2, 4 and 8 over streams of 2700 frames (several strips per stream and phase, several 128-window
    recurrence tiles; at hop 2 the 120-window position ring where the padded columns are only the first and the last):
    the shared-column path is taken, equals the per-window tiles (WWB_CRNN_NO_SHARE=1) bit for bit and equals f32 within
    1e-3, at n_out 1 and 2"""
    import torch
    for n_out in (1, 2):
        w = model(L, n_out)[0]
        tc, f32 = _engine(w, "tc"), _engine(w, "f32")
        try:
            torch.manual_seed(L + n_out)
            X = torch.rand((2, 2700, 40), device=tc.device) * 5
            for hop in (1, 2, 4, 8):
                a, na = _posteriors(tc, X, hop, True)
                b, nb = _posteriors(tc, X, hop, False)
                assert a.shape == (2, (2700 - L) // hop + 1)
                assert (na, nb) == (4, shared_launches(L)), (hop, na, nb)
                assert bool((a == b).all()), hop
                err = float((b - f32.posteriors(X, hop=hop)).abs().max())
                assert err < POST_ATOL, (hop, err)
        finally:
            tc.close()
            f32.close()


# ------------------------------------------------------------------------------------ GPU: streaming and records
def _stream_run(eng, chunks, thr, ids=None):
    """dense pushes (ids None) or indexed pushes of every stream in the order `ids`; returns the host outputs"""
    outs = []
    for c in chunks:
        if ids is None:
            res = eng.stream_push(c, np.ones(len(c), np.uint8), np.zeros(len(c), np.uint8), 0.0, thr)
        else:
            lens = np.array([c.shape[1]] * len(ids), np.int32)
            res = eng.stream_push_indexed(ids.astype(np.int32), np.concatenate([c[s] for s in ids]), lens,
                                          np.ones(len(ids), np.uint8), np.zeros(len(ids), np.uint8), 0.0, thr)
        outs.append(tuple(x.cpu().numpy() for x in res))
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "tc"])
@pytest.mark.parametrize("L", [97, 124])
def test_streaming_and_records(L, precision):
    """Ragged dense pushes (every chunk size of CHUNKS) and indexed pushes (slots in permuted order) against
    TriggerOracle, the threshold crossed in both directions.  The state record is 48 + 2048 + 160 L bytes; an export /
    import round trip into a second context continues bit-exact; an import into a context of another L is refused with
    `record 0: ...` and leaves every slot as it was.  The threshold is the median of the oracle's posteriors."""
    from wakeword_detection_b200 import _cabi
    w = model(L)[0]
    cap = 4
    ns = list(CHUNKS) * 2
    pcm = stream_pcm(cap, sum(ns) + 1, 5)
    chunks, cur = [], 0
    for n in ns:
        chunks.append(pcm[:, cur:cur + n])
        cur += n
    orc = [R.TriggerOracle(w, 0.5, 0.0) for _ in range(cap)]
    want = []   # [push][stream] the oracle's new posteriors (they do not depend on the threshold)
    for c in chunks:
        want.append([])
        for s in range(cap):
            o = orc[s]
            o.active = False
            before = len(o.posteriors)
            o(c[s], True)
            want[-1].append(np.array(o.posteriors[before:], np.float32))
    thr = float(np.median(np.concatenate([p for row in want for p in row])))
    perm = np.array([2, 0, 3, 1])
    mk = []

    def engine(wt=w):
        e = _cabi.Engine(wt, 0, precision)
        e.stream_alloc(cap, MAX_CHUNK)
        mk.append(e)
        return e

    try:
        dense, indexed = engine(), engine()
        assert dense.stream_state_bytes() == 48 + 2048 + 160 * L
        outs = _stream_run(dense, chunks, thr)
        iouts = _stream_run(indexed, chunks, thr, perm)
        worst, n_win, fired, quiet = 0.0, 0, 0, 0
        for i, (post, npost, trig, _) in enumerate(outs):
            ipost, inpost = iouts[i][0], iouts[i][1]
            for s in range(cap):
                new = want[i][s]
                j = int(np.nonzero(perm == s)[0][0])
                assert npost[s] == new.size and inpost[j] == new.size, (i, s)
                if new.size:
                    err = max(_err(post[s, :new.size], new), _err(ipost[j, :new.size], new))
                    assert err <= POST_ATOL, (i, s, err)
                    worst, n_win = max(worst, err), n_win + new.size
                    if np.abs(new - thr).min() > POST_ATOL:
                        assert bool(trig[s]) == bool((new > thr).any()), (i, s)
                        fired += bool(trig[s])
                        quiet += not bool(trig[s])
        assert n_win > 100 and fired > 0 and quiet > 0, (n_win, fired, quiet)
        STATS.append("stream L=%d %s: %d windows, max |err| vs TriggerOracle %.2e, %d pushes fired, %d quiet"
                     % (L, precision, n_win, worst, fired, quiet))
        # export after push `half`, import into a fresh context, continue both
        half = 13
        a, b = engine(), engine()
        _stream_run(a, chunks[:half], thr)
        rec = a.stream_export(np.arange(cap))
        b.stream_import(np.arange(cap), rec)
        assert_same_rows(_stream_run(b, chunks[half:], thr), outs[half:])
        # records written at another length (their mel_length field; a record's size follows from it): refused, nothing
        # changes
        c, d = engine(), engine()
        _stream_run(c, chunks[:half], thr)
        _stream_run(d, chunks[:half], thr)
        bad = rec.cpu().numpy().copy()
        bad[:, 12:16] = np.frombuffer(np.int32(L + 8).tobytes(), np.uint8)
        with pytest.raises(ValueError, match="record 0: mel_length"):
            c.stream_import(np.arange(cap), bad)
        assert_same_rows(_stream_run(c, chunks[half:], thr), _stream_run(d, chunks[half:], thr))
    finally:
        for e in mk:
            e.close()


# ------------------------------------------------------------------------------------ GPU: the chain and the drop-ins
FRAME = 320


@pytest.mark.gpu
def test_chain_with_three_lengths(tmp_path):
    """MultiWakewordPipeline with the shipped WaveNet (182), a synthetic CRNN at L = 97 and the shipped CRNN (151)
    against VadDebounceOracle -> one TriggerOracle per stage -> ActivationTimeoutOracle: posteriors within 1e-3,
    is_speech exact, is_active / activated / deactivated / activated_by exact outside the threshold band"""
    from wakeword_detection_b200 import weights as W
    from wakeword_detection_b200.wakeword import MultiWakewordPipeline
    w97 = model(97)[0]
    d97 = tmp_path / "crnn97"
    d97.mkdir()
    W.save_npz(w97, str(d97 / "weights.npz"))
    stages = [(os.path.join(WEIGHTS, "Wavenet"), "Wavenet", load_weights("Wavenet"), 0.5),
              (str(d97), "CRNN", w97, 0.6),
              (os.path.join(WEIGHTS, "CRNN"), "CRNN", load_weights("CRNN"), 0.9)]
    cfg = dict(frame_width=20, vad_rise_delay=40, vad_fall_delay=60, min_active=200, max_active=1000)
    n_frames, S = 150, 5
    pcm = np.stack([synth.stream_int16(n_frames * FRAME, 2, 7, j) for j in range(S)])
    for s, (clip, off) in enumerate((("crnn", 3287), ("wavenet", 3000), (None, 0), ("crnn", 9000), (None, 0))):
        if clip:
            c = wake_clip(clip)
            pcm[s, off:off + c.size] = c[:pcm.shape[1] - off]
    raw = np.ones((S, n_frames), bool)
    raw[2, 60:64] = False
    raw[3, 120:126] = False
    vad = [R.VadDebounceOracle(cfg["frame_width"], cfg["vad_rise_delay"], cfg["vad_fall_delay"]) for _ in range(S)]
    trig = [[R.TriggerOracle(w, t, 0.0) for _, _, w, t in stages] for _ in range(S)]
    tmo = [R.ActivationTimeoutOracle(cfg["frame_width"], cfg["min_active"], cfg["max_active"]) for _ in range(S)]
    speech, active = [False] * S, [False] * S
    pipe = MultiWakewordPipeline([dict(model_dir=d, model_type=t, posterior_threshold=th) for d, t, _, th in stages],
                                 S, precision="tc", **cfg)
    by_seen, near_frames, worst = set(), 0, 0.0
    try:
        for i in range(n_frames):
            got = {k: v.cpu().numpy() for k, v in pipe.step(pcm[:, i * FRAME:(i + 1) * FRAME], raw[:, i]).items()}
            for s in range(S):
                frame = pcm[s, i * FRAME:(i + 1) * FRAME]
                speech[s] = vad[s](speech[s], raw[s, i])
                act, by, near = active[s], -1, False
                for k, t in enumerate(trig[s]):
                    before = len(t.posteriors)
                    t.active = act
                    t(frame, speech[s])
                    p = np.array(t.posteriors[before:], np.float32)
                    assert got["n_post"][k, s] == p.size, (i, s, k)
                    if p.size:
                        err = _err(got["post"][k, s, :p.size], p)
                        assert err < POST_ATOL, (i, s, k, err)
                        worst = max(worst, err)
                        near |= bool(np.abs(p - stages[k][3]).min() <= POST_ATOL)
                    if t.active and not act:
                        by = k
                    act = t.active
                active[s] = tmo[s](speech[s], act)
                assert bool(got["is_speech"][s]) == speech[s], (i, s)
                if near:
                    near_frames += 1
                    continue
                want = dict(is_active=active[s], activated=by >= 0, deactivated=act and not active[s], activated_by=by)
                for key, v in want.items():
                    assert int(got[key][s]) == int(v), (i, s, key)
                if by >= 0:
                    by_seen.add(by)
    finally:
        pipe.close()
    STATS.append("chain WaveNet + CRNN L=97 + CRNN: max |err| %.2e, activations by stage %s, %d stream-frames in the band"
                 % (worst, sorted(by_seen), near_frames))
    assert by_seen, "no stage activated"


@pytest.mark.gpu
def test_drop_ins_at_another_length(tmp_path):
    """TFLiteModel reports the window in its input shape, WakewordTrigger sizes its frame window from it, and
    evaluate_tf_lite_opts runs with --timesteps 97: posteriors of the clips within 1e-3 of float64"""
    from wakeword_detection_b200 import evaluate_tf_lite_opts as ETO
    from wakeword_detection_b200 import weights as W
    from wakeword_detection_b200.models import TFLiteModel
    from wakeword_detection_b200.wakeword import WakewordTrigger
    w, X, _, _, ref = model(97)
    d = tmp_path / "m"
    d.mkdir()
    W.save_npz(w, str(d / "weights.npz"))
    enc = TFLiteModel(model_path=str(d / "encode.tflite"))
    assert list(enc.input_details[0]["shape"]) == [1, 40, 97, 1]
    trig = WakewordTrigger(model_dir=str(d), model_type="CRNN")
    assert trig.mel_length == 97 and trig.frame_window._store.shape == (98, 40)
    trig.close()
    clips = {"c%02d" % i: X[i] for i in range(len(X))}
    ETO.save_npz(str(tmp_path / "test.npz"), clips, {k: i % 2 for i, k in enumerate(clips)})
    args = ETO.parse_args(["--tf_models_dir", str(d), "--dataset_dir", str(tmp_path), "--testset", "test.npz",
                           "--timesteps", "97"])
    Xl, _ = ETO.load_data(str(tmp_path / "test.npz"), 97, 40)
    e, dt = ETO.load_tf_models(str(d))
    assert _err(ETO.posteriors(e, dt, Xl, "CRNN"), ref) < POST_ATOL
    assert ETO.main(args) == 0 and (d / "tf_lite_results.npy").is_file()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [16, 257])
def test_lengths_outside_the_range_are_refused(L):
    w = dict(model(17)[0], mel_length=np.int32(L))
    for precision in ("f32", "tc"):
        with pytest.raises(ValueError, match=r"CRNN window of %d frames unsupported \(expected 17\.\.256\)" % L):
            _engine(w, precision)
