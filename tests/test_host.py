"""CPU tests of the host-side logic: ring buffer semantics, sharding, the counter
all-reduce on gloo with world_size 2, window/clip bookkeeping."""
import os
import sys

import numpy as np
import pytest

from conftest import REFERENCE, ROOT
from wakeword_detection_b200 import dist as wdist
from wakeword_detection_b200.ring_buffer import RingBuffer
from wakeword_detection_b200 import evaluate_models as EM


def _drive(rb, ops, log):
    for op, arg in ops:
        try:
            if op == "write":
                rb.write(arg)
            elif op == "read":
                log.append(("read", rb.read().copy()))
            elif op == "read_all":
                log.append(("all", rb.read_all().copy()))
            elif op == "seek":
                rb.seek(arg)
            elif op == "rewind":
                rb.rewind()
            elif op == "reset":
                rb.reset()
            elif op == "fill":
                rb.fill(arg)
            log.append((op, rb.is_empty, rb.is_full))
        except IndexError as e:
            log.append(("IndexError", str(e)))


def _check_log(mine, theirs):
    assert len(mine) == len(theirs)
    for a, b in zip(mine, theirs):
        assert a[0] == b[0]
        if isinstance(a[1], np.ndarray):      # the data a read / read_all returned
            assert isinstance(b[1], (list, np.ndarray))
            np.testing.assert_array_equal(a[1].reshape(-1), np.asarray(b[1], np.float32).reshape(-1))
        else:                                 # (is_empty, is_full) after the operation, or the IndexError message
            assert tuple(a[1:]) == tuple(b[1:])


def test_ring_buffer_matches_reference_semantics():
    """The RingBuffer replays the stored operation log of tests/golden/ring_buffer_log.json
    (make_golden_ring_buffer.py); with WWB_REFERENCE pointing at a checkout of the reference, its own
    spokestack/ring_buffer.py is driven through the same operations as well."""
    import json
    from conftest import GOLDEN
    g = json.load(open(os.path.join(GOLDEN, "ring_buffer_log.json")))
    ops = [tuple(o) for o in g["ops"]]
    mine = []
    _drive(RingBuffer(shape=[g["capacity"]]), ops, mine)
    assert len(ops) == 401 and sum(e[0] == "IndexError" for e in mine) > 0   # the log does exercise misuse
    _check_log(mine, g["log"])
    # invariants that hold without the reference
    rb = RingBuffer(shape=[3])
    assert rb.capacity == 3 and rb.is_empty and not rb.is_full
    for v in (1, 2, 3):
        rb.write(v)
    assert rb.is_full
    with pytest.raises(IndexError):
        rb.write(4)
    rb.rewind().seek(1)
    rb.write(4)
    np.testing.assert_array_equal(rb.read_all(), [2, 3, 4])
    assert rb.is_empty
    with pytest.raises(IndexError):
        rb.read()
    if not REFERENCE:
        return
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_ring_buffer", os.path.join(REFERENCE, "spokestack", "ring_buffer.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    theirs = []
    _drive(mod.RingBuffer(shape=[g["capacity"]]), ops, theirs)
    _check_log(mine, theirs)


def test_shard_range_partitions():
    for n in (0, 1, 7, 100, 4096):
        for world in (1, 2, 3, 8):
            spans = [wdist.shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1
    chunks = wdist.time_chunks(1000, 4)
    assert chunks[0][2] == 0 and chunks[-1][3] == 0 and chunks[1][2] == 16 and chunks[1][3] == 14


def test_chunked_far_count_equals_whole(golden):
    """Sharding one trajectory into time chunks with halos gives the same edge count
    (checked here with the numpy oracle on logical ranks; the device version is in the gpu tests)."""
    from oracle import restated as R
    p = golden["pm_traj"]
    thr = R.thresholds_eval()
    sm = R.smooth_same(p)
    whole = np.array([R.rising_edges(sm, t) for t in thr])
    total = np.zeros_like(whole)
    for b, e, lo, hi in wdist.time_chunks(len(p), 4):
        seg = p[b - lo:e + hi]
        sms = np.array([np.sum(seg[max(0, i - 15):i + 15] / 30.0) for i in range(len(seg))])
        for ti, t in enumerate(thr):
            above = sms > t
            for i in range(lo, lo + (e - b)):
                prev = above[i - 1] if i > 0 else False
                total[ti] += int(above[i] and not prev)
    np.testing.assert_array_equal(total, whole)


def _gloo_worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from wakeword_detection_b200 import dist as wd
    assert wd.rank_world() == (rank, world)
    a = torch.arange(5, dtype=torch.int64) * (rank + 1)
    b = torch.full((3,), rank + 10, dtype=torch.int64)
    ra, rb = wd.all_reduce_counters(a, b)
    if rank == 0:
        out.put((ra.tolist(), rb.tolist()))
    dist.destroy_process_group()


def test_counter_all_reduce_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 1000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ra, rb = q.get(timeout=120)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ra == [0, 3, 6, 9, 12] and rb == [21, 21, 21]


def test_eval_clip_padding_matches_oracle():
    from oracle import restated as R
    rng = np.random.default_rng(1)
    for n in (1, 319, 320, 4321, 16000):
        x = rng.standard_normal(n).astype(np.float32)
        np.testing.assert_array_equal(EM._padded_stream(x, 16000, 320), R.eval_clip_samples(x))


def test_wav_roundtrip(tmp_path):
    pcm = (np.random.default_rng(2).standard_normal(4000) * 3000).astype(np.int16)
    EM.concatenate_FA([pcm, pcm], 2, tmp_path / "x.wav")
    x = EM.load_wav(tmp_path / "x.wav", 16000)
    assert x.shape[0] == 8000 + 1600 and x.dtype == np.float32
    np.testing.assert_array_equal(x[:4000], pcm.astype(np.float32) / 32768.0)
    assert abs(EM.duration_test(tmp_path / "x.wav", 16000) - 0.6) < 1e-9
    with pytest.raises(ValueError):
        EM.load_wav(tmp_path / "x.wav", 8000)


def test_parse_args_flags():
    a = EM.parse_args(["--model_type", "Wavenet", "--models_dir", os.path.join(ROOT, "weights", "Wavenet")])
    assert a.model_type == "Wavenet" and a.sample_rate == 16000 and a.frame_width == 20
    assert a.neg_samples == "not_hey_snips_long.wav" and a.examine_audio is False


def test_tf_lite_opts_load_data_npz_and_metrics(tmp_path, capsys):
    """evaluate_tf_lite_opts.py:35-47 (truncate / zero-pad to `timesteps`, file order, uint8 labels) and :69-87
    (metric definitions, including the reference's swapped recall / precision names)."""
    from wakeword_detection_b200 import evaluate_tf_lite_opts as ETO
    rng = np.random.default_rng(0)
    clips = {"b_long": rng.random((200, 40), dtype=np.float32), "a_short": rng.random((37, 40), dtype=np.float32),
             "c_exact": rng.random((151, 40), dtype=np.float32)}
    labels = {"b_long": 1, "a_short": 0, "c_exact": 1}
    path = str(tmp_path / "test.npz")
    ETO.save_npz(path, clips, labels)
    X, y = ETO.load_data(path, 151, 40)
    assert X.shape == (3, 151, 40) and X.dtype == np.float32 and y.dtype == np.uint8
    assert list(y) == [1, 0, 1]                                   # keys in file order, not sorted
    assert np.array_equal(X[0], clips["b_long"][:151])
    assert np.array_equal(X[1, :37], clips["a_short"]) and not X[1, 37:].any()
    assert np.array_equal(X[2], clips["c_exact"])
    r = ETO.metrics([1, 0, 1, 1, 0, 0], [1, 0, 0, 1, 1, 0])
    assert (r["true_positive"], r["false_positive"], r["false_negative"], r["true_negative"]) == (2, 1, 1, 2)
    assert r["recall"] == 2 / 3 and r["precision"] == 2 / 3 and abs(r["accuracy"] - 2 / 3) < 1e-12
    a = ETO.parse_args([])
    assert (a.tf_models_dir, a.testset, a.timesteps, a.num_features, a.model_type) == ("CRNN_tf_model", "test.h5", 151, 40, "CRNN")


def test_fft64_header_matches_numpy(tmp_path):
    """csrc/fft64.cuh (the fp64 FFT the K1 kernel runs) compiled for the CPU with its 16 lanes emulated in lock step
    (tests/fft64_host.cpp) against np.fft.rfft: index algebra and accuracy of the exact device code, no GPU needed."""
    import subprocess
    exe = str(tmp_path / "fft64_host")
    subprocess.check_call(["g++", "-O2", "-std=c++14", "-o", exe, os.path.join(ROOT, "tests", "fft64_host.cpp")])
    rng = np.random.default_rng(0)
    t = np.arange(512)
    fr = (rng.standard_normal((6, 512)) * 0.1).astype(np.float32)
    fr[1] = np.clip(np.round(32767 * 1.4 * np.sin(2 * np.pi * 440 / 16000 * t)) / 32767, -1, 1)
    fr[2] = 0
    fr[3] = (0.9 * np.sin(2 * np.pi * 300 / 16000 * t) + 2e-4 * np.sin(2 * np.pi * 5200 / 16000 * t)).astype(np.float32)
    out = subprocess.run([exe], input=fr.tobytes(), capture_output=True, check=True).stdout
    mag = np.frombuffer(out, np.float32).reshape(6, 257)
    ref = np.abs(np.fft.rfft(fr * np.hanning(512), n=512)).astype(np.float32)
    assert np.all(mag[2] == 0)
    assert np.all(np.abs(mag - ref) <= 2e-7 * ref + 1e-30)


def test_pcm_scaling_without_division_is_exact():
    """filter.cu:pcm_to_float replaces s / 32767 by q0 = s*r, q = fma(fma(-q0, 32767, s), r, q0): equal to the IEEE
    quotient numpy computes (wakeword/tflite.py:150) for all 65536 int16 values (fma emulated exactly in fp64: the
    products have <= 48 significant bits and the sums cancel to few bits)."""
    s = np.arange(-32768, 32768).astype(np.float32)
    r = np.float32(3.0518509447574615e-05)
    assert r == np.float32(1.0) / np.float32(32767.0)
    q0 = (s * r).astype(np.float32)
    rem = (s.astype(np.float64) - q0.astype(np.float64) * 32767.0).astype(np.float32)
    assert np.all(rem.astype(np.float64) == s.astype(np.float64) - q0.astype(np.float64) * 32767.0)   # exact
    q = (rem.astype(np.float64) * np.float64(r) + q0.astype(np.float64)).astype(np.float32)
    assert np.array_equal(q, s / np.float32(32767.0))


def test_fp16_weight_variant_loader_and_dequantize_folding():
    """SURVEY 8(f) row 3: `*-quant.tflite` = trained constants stored as float16 behind DEQUANTIZE ops, float32 math
    (wwdetect/CRNN/convert_CRNN_tflite.py:23-37).  The reader folds the op; without the files the variant is derived by the
    converter's rounding; a missing `-quant` file raises like the interpreter unless derivation is asked for."""
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200 import tflite_reader as tr, weights as W
    from wakeword_detection_b200.models import TFLiteModel
    # DEQUANTIZE folding on a hand-built graph: fp16 constant -> DEQUANTIZE -> FULLY_CONNECTED
    w16 = np.array([[0.1, -2.5], [3.0, 1e-3]], np.float16)
    tensors = [tr.Tensor(0, "in", [1, 2], np.float32, 0, None), tr.Tensor(1, "w16", [2, 2], np.float16, 1, w16),
               tr.Tensor(2, "w32", [2, 2], np.float32, 0, None), tr.Tensor(3, "out", [1, 2], np.float32, 0, None)]
    ops = [tr.Op(6, "DEQUANTIZE", [1], [2]), tr.Op(9, "FULLY_CONNECTED", [0, 2, -1], [3], {"act": 0})]
    m = tr.fold_dequantize(tr.Model(3, "t", [tr.SubGraph("main", tensors, [0], [3], ops)]))
    assert [o.name for o in m.main.ops] == ["FULLY_CONNECTED"]
    assert m.main.tensors[2].data.dtype == np.float32 and np.array_equal(m.main.tensors[2].data, w16.astype(np.float32))
    for name in ("CRNN", "Wavenet"):
        d = os.path.join(WEIGHTS, name)
        w = W.load_model_dir(d, name)
        q = W.load_model_dir(d, name, quant=True)
        assert str(q["quant_source"]) == "derived"
        changed = 0
        for k, v in w.items():
            if k in ("mel_w", "mel_b", "mel_length", "dilation") or not isinstance(v, np.ndarray) or v.dtype != np.float32 or v.ndim == 0:
                assert np.array_equal(q[k], v)                  # the filter and the geometry are untouched
                continue
            assert np.array_equal(q[k], q[k].astype(np.float16).astype(np.float32))   # exactly representable in fp16
            assert np.abs(q[k] - v).max() <= 2.0 ** -11 * max(np.abs(v).max(), 6.2e-5) + 6e-8
            changed += int((q[k] != v).any())
        assert changed >= 8
        q2 = W.quantize_fp16(q)
        assert all(np.array_equal(q2[k], q[k]) for k in q if k != "quant_source")
        with pytest.raises(ValueError):
            TFLiteModel(os.path.join(d, "encode-quant.tflite"))   # not shipped: opening it fails like the interpreter
    with pytest.raises(ValueError):
        TFLiteModel(os.path.join(WEIGHTS, "CRNN", "filter-quant.tflite"), derive_quant=True)


def load_weights_host(name):
    from conftest import load_weights
    return load_weights(name)


def test_vad_debounce_and_activation_timeout_dropins_replay_reference_run():
    """tests/golden/reference_pipeline.npz = the reference's own VoiceActivityDetector / WakewordTrigger /
    ActivationTimeout dispatched frame by frame (make_golden_pipeline.py).  The host drop-ins reproduce the VAD debounce
    from the scripted raw decisions and, given the trigger's activations, the timeout's deactivations; so does the
    oracle's PipelineOracle end to end (CRNN run, CPU)."""
    import os
    from conftest import GOLDEN
    from oracle import restated as R
    from wakeword_detection_b200.activation_timeout import ActivationTimeout
    from wakeword_detection_b200.context import SpeechContext
    from wakeword_detection_b200.vad import VoiceActivityDetector, VoiceActivityTrigger
    g = np.load(os.path.join(GOLDEN, "reference_pipeline.npz"))
    cfg = dict(zip(("frame_width", "vad_rise_delay", "vad_fall_delay", "min_active", "max_active"), [int(v) for v in g["cfg"]]))
    for name in ("crnn", "wavenet"):
        raw, speech, active = g["pipe_%s_raw" % name], g["pipe_%s_speech" % name], g["pipe_%s_active" % name]
        it = iter(raw)
        vad = VoiceActivityDetector(detector=lambda b, sr: bool(next(it)), **cfg)
        tmo = ActivationTimeout(**cfg)
        ctx = SpeechContext()
        prev = False
        for i in range(len(raw)):
            vad(ctx, np.zeros(320, np.int16))
            assert ctx.is_speech == bool(speech[i]), (name, i)
            # the trigger's part: an activation shows up as a rising edge that the timeout did not cause
            if active[i] and not prev:
                ctx.is_active = True
            tmo(ctx)
            assert ctx.is_active == bool(active[i]), (name, i)
            prev = bool(active[i])
    vt, ctx = VoiceActivityTrigger(), SpeechContext()
    ctx.is_speech = True
    vt(ctx)
    assert ctx.is_active
    with pytest.raises(ImportError):
        VoiceActivityDetector()            # webrtcvad is not installed here: the decision function must be injected
    w = load_weights_host("CRNN")
    o = R.PipelineOracle(w, **cfg)
    pcm, raw = g["pipe_crnn_pcm"], g["pipe_crnn_raw"]
    got = [o(pcm[i * 320:(i + 1) * 320], raw[i]) for i in range(len(raw))]
    assert [s for s, _ in got] == list(g["pipe_crnn_speech"]) and [a for _, a in got] == list(g["pipe_crnn_active"])


class _OracleEngine:
    """CPU stand-in for `_cabi.Engine` in the host-logic tests of the sharded evaluation: same methods, answers from the
    oracle (tests may use oracle/; the product path never does)."""

    def __init__(self, w):
        import torch
        from oracle import restated as R
        self.w, self.R, self.torch = w, R, torch
        self.device = torch.device("cpu")
        self.L = int(w["mel_length"])

    def num_frames(self, n):
        return 0 if n < 512 else (n - 512) // 160 + 1

    def num_windows(self, f, hop):
        return 0 if f < self.L else (f - self.L) // hop + 1

    def pipeline(self, pcm, hop=2, pre_emphasis=0.0):
        R = self.R
        x = pcm.numpy()
        nw = self.num_windows(self.num_frames(x.shape[1]), hop)
        out = np.zeros((x.shape[0], nw), np.float32)
        for i in range(x.shape[0]):
            mel = R.mel_stream(x[i], self.w)
            if nw:
                j = np.arange(nw)
                out[i] = R.posterior(mel[(hop * j)[:, None] + np.arange(self.L)[None, :]], self.w)
        return self.torch.from_numpy(out)

    def eval_counts(self, post, seg_off, thresholds, mode, smooth=30, halo_lo=None, halo_hi=None):
        R = self.R
        p = np.asarray(post, np.float32).reshape(-1)
        seg = np.asarray(seg_off)
        counts = np.zeros(len(thresholds), np.int64)
        for k in range(len(seg) - 1):
            part = p[seg[k]:seg[k + 1]]
            if mode == "frr_max":
                counts += np.array([int(part.max() > t) for t in thresholds])
            else:
                lo = halo_lo[k] if halo_lo is not None else 0
                hi = halo_hi[k] if halo_hi is not None else 0
                sm = R.smooth_same(part)
                for ti, t in enumerate(thresholds):
                    above = sm > t
                    idx = np.arange(lo, part.size - hi)
                    prev = np.where(idx > 0, above[np.maximum(idx - 1, 0)], False)
                    counts[ti] += int((above[idx] & ~prev).sum())
        return self.torch.from_numpy(counts)


def _sharded_eval_inputs():
    from conftest import GOLDEN
    from wakeword_detection_b200 import synth
    wake = np.load(os.path.join(GOLDEN, "wake_crnn_pcm.npy")).astype(np.float32) / 32768.0
    pos = [wake, np.clip(synth.stream_float(20321, 2, 9, 1), -1, 1).astype(np.float32), wake[3000:30000],
           np.clip(synth.stream_float(16777, 0, 9, 2), -1, 1).astype(np.float32), wake[:33001]]
    far = np.concatenate([np.clip(synth.stream_float(40000, 5, 9, 3), -1, 1).astype(np.float32), wake,
                          np.clip(synth.stream_float(52345, 2, 9, 4), -1, 1).astype(np.float32), wake[:30000]])
    return pos, far


def _sharded_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    pos, far = _sharded_eval_inputs()
    eng = _OracleEngine(load_weights_host("CRNN"))
    thr = np.arange(0.5, 0.99999, 0.05)
    acc, edg = EM.evaluate_sharded("", "CRNN", pos, far, 20, 16000, thr, engine=eng)
    out.put((rank, acc.tolist(), edg.tolist()))
    dist.destroy_process_group()


def test_sharded_evaluation_gloo_world2_equals_single_process():
    """utils/evaluate_models.py:280-327 over two ranks (gloo on CPU, posteriors from the oracle): wake-word clips in
    contiguous runs with the carried window, the long false-accept clip in two time chunks with PCM + counter halos,
    ONE all-reduce - the counters equal the single-process sweep on every rank.  Also the pure partition rules."""
    import torch.multiprocessing as mp
    pos, far = _sharded_eval_inputs()
    eng = _OracleEngine(load_weights_host("CRNN"))
    thr = np.arange(0.5, 0.99999, 0.05)
    kp = EM.get_posterior("", "CRNN", "false_negatives", pos, 20, 16000, engine=eng)
    nk = EM.get_posterior("", "CRNN", "false_accepts", [far], 20, 16000, engine=eng)
    acc1, edg1 = EM.sweep_counts(kp, nk, thr, eng)
    assert acc1[0] >= 3 and edg1[0] >= 2                  # the wake clips fire in both sets
    # a rank's run of clips, started with the carried window, gives the same maxima as the whole list
    carries = EM.carry_before_clips([len(c) for c in pos], 16000, 320)
    assert carries[0] == 0 and carries[1] == 480
    tail = EM.get_posterior("", "CRNN", "false_negatives", pos[2:], 20, 16000, engine=eng, carry_len=carries[2])
    np.testing.assert_array_equal(np.array(tail, np.float32), np.array(kp[2:], np.float32))
    # time chunks of the FAR clip: the chunk's posteriors are the global trajectory's, for any world size
    for world in (2, 3):
        got = []
        for r in range(world):
            part, lo, hi, n_win = EM.far_chunk_posteriors(far, 20, 16000, r, world, eng)
            assert n_win == len(nk)
            got.append(part[lo:part.size - hi])
            b, e, _, _ = wdist.time_chunks(n_win, world)[r]
            np.testing.assert_allclose(part, np.array(nk[b - lo:e + hi], np.float32), atol=2e-6)
        assert sum(g.size for g in got) == len(nk)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 7) % 1000
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(2)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, acc, edg in res:
        assert acc == acc1.tolist() and edg == edg1.tolist()


def test_load_wav_range(tmp_path):
    pcm = (np.random.default_rng(3).standard_normal(5000) * 3000).astype(np.int16)
    EM.concatenate_FA([pcm], 1, tmp_path / "y.wav")
    whole = EM.load_wav(tmp_path / "y.wav", 16000)
    assert EM.clip_num_samples(tmp_path / "y.wav", 16000) == 5000 and EM.clip_num_samples(whole, 16000) == 5000
    for a, b in ((0, 5000), (-100, 300), (4900, 5200), (1234, 2345), (6000, 6100)):
        want = np.zeros(b - a, np.float32)
        lo, hi = max(a, 0), min(b, 5000)
        if hi > lo:
            want[lo - a:hi - a] = whole[lo:hi]
        np.testing.assert_array_equal(EM.load_wav_range(tmp_path / "y.wav", a, b, 16000), want)
        np.testing.assert_array_equal(EM.load_wav_range(whole, a, b, 16000), want)


def test_wfst_smoothing_is_the_lattice_shortest_path():
    """wwdetect/wfst.py:17-71 on the reference's own two test posteriors (:75-97): the Viterbi recursion equals the
    brute-force minimum over all 2^10 label paths of the lattice the reference builds (pynini cannot run here)."""
    import itertools
    from wakeword_detection_b200 import wfst
    t1 = [[0.8, 0.2], [0.9, 0.1], [0.5, 0.5], [0.4, 0.6], [0.2, 0.8], [0.6, 0.4], [0.3, 0.7], [0.4, 0.6], [0.5, 0.5], [0.9, 0.1]]
    t2 = [[0.8, 0.2], [0.9, 0.1], [0.5, 0.5], [0.55, 0.45], [0.2, 0.8], [0.6, 0.4], [0.7, 0.3], [0.8, 0.2], [0.3, 0.7], [0.9, 0.1]]
    for probs in (t1, t2):
        obs = -np.log(np.array(probs))
        best, best_cost = None, np.inf
        for path in itertools.product((0, 1), repeat=len(probs)):
            c = -np.log(0.5) + obs[0, path[0]]
            for t in range(1, len(probs)):
                c += obs[t, path[t]] - (1.0 if path[t] == path[t - 1] else 0.0)
            if c < best_cost - 1e-12:
                best, best_cost = list(path), c
        got, cost = wfst.best_path(probs)
        assert got == best and abs(cost - best_cost) < 1e-9
    # the stay bonus keeps the path in the wake-word state through the single contrary frame of test 1 and out of it in test 2
    assert wfst.smooth(t1) == "other other other wakeword wakeword wakeword wakeword wakeword other other"
    assert wfst.smooth(t2) == " ".join(["other"] * 10)        # the errant single wake-word frame is smoothed away


def test_keyword_oracle_replays_reference_run():
    """tests/golden/reference_keyword.npz = the reference's own KeywordRecognizer over 5 s of audio with scripted
    activations (make_golden_keyword.py): the oracle's restatement produces the same events at the same frames and the
    same encode windows."""
    import os
    from conftest import GOLDEN
    sys.path.insert(0, GOLDEN)
    import keyword_stub as KS
    from oracle import restated as R
    g = np.load(os.path.join(GOLDEN, "reference_keyword.npz"))
    o = R.KeywordOracle(load_weights_host("CRNN"), KS.Encode(), KS.Detect(), threshold=float(g["kw_threshold"]))
    pcm, active = g["kw_pcm"], g["kw_active"]
    events, frames = [], []
    for i in range(len(active)):
        ev = o(pcm[i * 320:(i + 1) * 320], bool(active[i]))
        events += ev
        frames += [i] * len(ev)
        assert np.abs(o.encoded - g["kw_enc_window"][i]).max() < 1e-4, i
    assert frames == list(g["kw_event_frame"])
    assert [e[0] for e in events] == list(g["kw_event_kind"])
    classes = ["up", "down", "stop"]
    assert [classes[e[1]] if e[1] >= 0 else "" for e in events] == list(g["kw_event_class"])
    assert np.abs(np.array([e[2] for e in events]) - g["kw_event_conf"]).max() < 1e-4
