"""GPU parity tests: the CUDA path, called through the C ABI (ctypes `Engine`), against
the CPU oracle on the same seeded inputs, against the committed golden vectors from the
reference's own glue, and — at benchmark sizes — through size-independent properties.

Tolerances (BASELINE.md §4): mel |d| <= 1e-4*max(|ref|,1) on every bin (no exemptions); encoder outputs and
posteriors 1e-3 absolute; trigger decisions and FAR/FRR counts exact.
"""
import numpy as np
import pytest

from conftest import get_engine, load_weights
from oracle import restated as R
from streaming_helpers import MEL_STATS, check_mel
from wakeword_detection_b200 import synth

pytestmark = pytest.mark.gpu

POST_ATOL = 1e-3

@pytest.fixture(scope="module", autouse=True)
def _mel_report():
    yield
    print("\n[mel parity] %d bins checked (%d at the 1e-5 floor, same bound), max |err| %.3e = %.4f of the tolerance"
          % (MEL_STATS["bins"], MEL_STATS["at_floor"], MEL_STATS["max_err"], MEL_STATS["max_err_over_tol"]))


# ------------------------------------------------------------------------------------ filter
@pytest.mark.parametrize("cls", range(synth.N_CLASSES))
def test_filter_int16_classes(cls, w_crnn):
    eng = get_engine("CRNN")
    n = 16000 + 37 * cls
    pcm = synth.stream_int16(n, cls, seed=1, stream=cls)
    mel = eng.filter(pcm[None]).cpu().numpy()[0]
    ref = R.mel_stream(R.int16_to_float(pcm), w_crnn)
    check_mel(mel, ref)


def test_filter_silence_is_exact_zero():
    eng = get_engine("CRNN")
    mel = eng.filter(np.zeros((3, 4000), np.int16)).cpu().numpy()
    assert mel.shape == (3, 22, 40) and np.all(mel == 0.0)


@pytest.mark.parametrize("a", [0.0, 0.97])
def test_filter_float_batch_preemphasis(a, w_crnn):
    eng = get_engine("CRNN")
    x = np.stack([np.clip(synth.stream_float(9000, c, 2, c), -1, 1) for c in (0, 2, 5)]).astype(np.float32)
    mel = eng.filter(x, a).cpu().numpy()
    for i in range(3):
        check_mel(mel[i], R.mel_stream(x[i], w_crnn, a))


def test_filter_golden_vectors(golden, w_crnn):
    eng = get_engine("CRNN")
    n = int(golden["filter_consumed_pe0"])
    mel = eng.filter(golden["filter_in"][None, :n]).cpu().numpy()[0]
    check_mel(mel, golden["filter_mel_pe0"])
    mel = eng.filter(golden["filter_in"][None, :n], 0.97).cpu().numpy()[0]
    check_mel(mel, golden["filter_mel_pe97"])


def test_filter_edge_sizes(w_crnn):
    eng = get_engine("CRNN")
    assert eng.filter(np.zeros((2, 511), np.int16)).shape == (2, 0, 40)
    assert eng.filter(np.zeros((0, 4000), np.int16)).shape == (0, 22, 40)
    pcm = synth.stream_int16(512 + 160 * 16, 2, 3, 0)          # 17 frames: one full tile + 1
    for n in (512, 671, 672, 512 + 160 * 15, 512 + 160 * 16):
        mel = eng.filter(pcm[None, :n]).cpu().numpy()[0]
        check_mel(mel, R.mel_stream(R.int16_to_float(pcm[:n]), w_crnn))
    # unaligned rows (odd pitch) take the scalar load path
    big = synth.batch_int16(3, 3001, seed=4)
    mel = eng.filter(big).cpu().numpy()
    for i in range(3):
        check_mel(mel[i], R.mel_stream(R.int16_to_float(big[i]), w_crnn))


def _hdr_signals(n=8000):
    """High-dynamic-range PCM: bands 60-120 dB below the frame's loudest bin but above the 1e-5 mel floor - the
    cases an fp32 FFT gets wrong (round 1: 4.6e-4) and the reference's fp64 FFT does not."""
    t = np.arange(n) / 16000.0
    rng = np.random.default_rng(7)
    sigs = [
        1.4 * np.sin(2 * np.pi * 440.0 * t),                                               # clipping sine
        0.999 * np.sin(2 * np.pi * 1000.0 * t),                                            # full-scale clean tone
        0.9 * np.sin(2 * np.pi * 300.0 * t) + 2e-4 * np.sin(2 * np.pi * 5200.0 * t),       # tone + tone 73 dB down
        0.95 * np.sin(2 * np.pi * 7000.0 * t) + 1e-3 * rng.standard_normal(n),             # HF tone over a -60 dB noise bed
        0.5 * np.sign(np.sin(2 * np.pi * 125.0 * t)),                                      # square wave (1/k harmonics)
        0.8 * np.sin(2 * np.pi * (200.0 + 3000.0 * t) * t),                                # chirp
        0.6 + 0.0 * t,                                                                     # DC
        np.where(np.arange(n) % 700 == 0, 0.99, 0.0) + 3e-4 * rng.standard_normal(n),      # clicks over a quiet bed
    ]
    return np.stack([np.round(np.clip(x, -1, 1) * 32767).astype(np.int16) for x in sigs])


def test_filter_high_dynamic_range(w_crnn):
    eng = get_engine("CRNN")
    pcm = _hdr_signals()
    mel = eng.filter(pcm).cpu().numpy()
    worst = 0.0
    for i in range(pcm.shape[0]):
        worst = max(worst, check_mel(mel[i], R.mel_stream(R.int16_to_float(pcm[i]), w_crnn)))
    print("high-dynamic-range set: max |err| %.3e" % worst)


def test_filter_bench_shape_vs_oracle(w_crnn):
    """The headline shape (512 streams x 10 s, 64-frame work items): first / middle / last streams against the oracle."""
    eng = get_engine("CRNN")
    pcm = synth.device_pcm(512, 160000, seed=1234, device=eng.device)
    mel = eng.filter(pcm)
    for sidx in (0, 1, 255, 510, 511):
        ref = R.mel_stream(R.int16_to_float(pcm[sidx].cpu().numpy()), w_crnn)
        check_mel(mel[sidx].cpu().numpy(), ref)


def test_filter_mel_model_callable(w_crnn):
    eng = get_engine("CRNN")
    rng = np.random.default_rng(0)
    mag = (rng.random((33, 257)) * 4).astype(np.float32)
    mag[0] = 0
    got = eng.mel_from_magnitude(mag).cpu().numpy()
    check_mel(got, R.mel_from_magnitude(mag, w_crnn))


def test_filter_full_size_properties():
    """config 2 shape (many 2 s clips): doubling the PCM adds exactly 0.5*ln 2 to every mel
    value above the floor; results do not depend on the batch a stream is in."""
    import torch
    eng = get_engine("CRNN")
    S, N = 4096, 32000
    pcm = synth.device_pcm(S, N, seed=7, device=eng.device)
    pcm = torch.clamp(pcm, -16000, 16000)
    mel1 = eng.filter(pcm)
    mel2 = eng.filter(pcm * 2)
    assert mel1.shape == (S, 197, 40)
    mask = mel1 > 1.0
    d = (mel2 - mel1)[mask]
    assert float((d - 0.5 * np.log(2.0)).abs().max()) < 2e-4
    sub = eng.filter(pcm[1000:1003].clone())
    assert torch.equal(sub, mel1[1000:1003])
    assert bool(torch.isfinite(mel1).all())


# ------------------------------------------------------------------------------------ encoders
def _windows(name, w, n_extra=24):
    import os
    from conftest import GOLDEN
    adv = np.load(os.path.join(GOLDEN, "wake_%s_mel.npy" % name))
    L = int(w["mel_length"])
    mels = [R.mel_stream(np.clip(synth.stream_float(16000 * 3, c, 5, c), -1, 1).astype(np.float32), w)
            for c in range(synth.N_CLASSES)]
    rnd = [m[j:j + L] for m in mels for j in range(0, m.shape[0] - L, 41)][:n_extra]
    zero = np.zeros((1, L, 40), np.float32)
    return np.concatenate([adv, np.stack(rnd), zero]).astype(np.float32)


@pytest.mark.parametrize("precision", ["f32", "tc"])
@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("CRNN_arik_original", "crnn"), ("CRNN_arik_nosilence", "crnn"),
                                        ("CRNN_arik_nosilence_enhanced", "crnn"), ("Wavenet", "wavenet")])
def test_encode_detect_vs_oracle(wname, name, precision):
    w = load_weights(wname)
    eng = get_engine(wname, precision)
    X = _windows(name, w)
    if name == "wavenet":
        X = X[::2]
    enc = eng.encode(X)
    ref_enc = R.encode(X, w)
    assert np.abs(enc.cpu().numpy() - ref_enc).max() < POST_ATOL
    det = eng.detect(enc).cpu().numpy()
    ref_det = R.detect(ref_enc, w)
    assert det.shape == ref_det.shape
    assert np.abs(det - ref_det).max() < POST_ATOL
    # detect on the oracle's encoder output as well (the two models are separate callables)
    det2 = eng.detect(ref_enc).cpu().numpy()
    assert np.abs(det2 - ref_det).max() < POST_ATOL
    post = eng.posteriors(X.reshape(X.shape[0], X.shape[1], 40), hop=1).cpu().numpy()[:, 0]
    ref = ref_det[:, -1]
    assert np.abs(post - ref).max() < POST_ATOL
    assert ref.max() > {"CRNN_arik_original": 0.6, "CRNN_arik_nosilence_enhanced": 0.8}.get(wname, 0.9) and ref.min() < 0.1   # spans the range
    # decisions: exact outside the tolerance band around the threshold
    band = np.abs(ref - 0.5) <= POST_ATOL
    assert np.array_equal((post > 0.5)[~band], (ref > 0.5)[~band])


@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_tc_fast_mode_is_close_but_outside_parity(wname, name):
    """single-fp16 operands: documented as outside the 1e-3 bound; must still be sane"""
    w = load_weights(wname)
    X = _windows(name, w)
    ref = R.posterior(X, w)
    fast = get_engine(wname, "tc_fast").posteriors(X, hop=1).cpu().numpy()[:, 0]
    exact = get_engine(wname, "tc").posteriors(X, hop=1).cpu().numpy()[:, 0]
    assert np.abs(fast - ref).max() < 2e-2
    assert np.abs(exact - ref).max() < 2e-4 < POST_ATOL     # the split path is ~fp32
    assert np.abs(exact - ref).max() <= np.abs(fast - ref).max()


def test_crnn_tc_many_tiles_matches_f32_path():
    """8191 independent windows (ragged last tile of every kernel) through both paths."""
    import torch
    e32, etc = get_engine("CRNN", "f32"), get_engine("CRNN", "tc")
    pcm = synth.device_pcm(64, 160 * 300 + 512, seed=3, device=e32.device)
    mel = e32.filter(pcm)
    wins = mel.unfold(1, 151, 1).permute(0, 1, 3, 2)[:, :128].reshape(-1, 151, 40)[:8191].contiguous()
    a = e32.posteriors(wins, hop=1)[:, 0]
    b = etc.posteriors(wins, hop=1)[:, 0]
    assert float((a - b).abs().max()) < 2e-4
    enc_a, enc_b = e32.encode(wins[:300]), etc.encode(wins[:300])
    assert float((enc_a - enc_b).abs().max()) < 2e-4


def test_wavenet_tc_many_groups_matches_f32_path():
    """4097 windows (1025 groups of 4, ragged last group, > 6 groups per SM) through both paths,
    sliding hop-1 windows of real filter output; also the encoder output tensor."""
    e32, etc = get_engine("Wavenet", "f32"), get_engine("Wavenet", "tc")
    pcm = synth.device_pcm(17, 160 * 421 + 512, seed=5, device=e32.device)
    mel = e32.filter(pcm)                      # [17, 422, 40] -> 241 windows per stream
    a = e32.posteriors(mel, hop=1)
    b = etc.posteriors(mel, hop=1)
    assert a.shape == (17, 241)
    assert float((a - b).abs().max()) < 2e-4
    wins = mel.unfold(1, 182, 1).permute(0, 1, 3, 2)[:, :5].reshape(-1, 182, 40).contiguous()
    ea, eb = e32.encode(wins), etc.encode(wins)
    assert float((ea - eb).abs().max()) < 5e-4 * max(1.0, float(ea.abs().max()))
    da, db = e32.detect(ea), etc.detect(eb)
    assert float((da - db).abs().max()) < 2e-4


@pytest.mark.parametrize("n", [1, 2, 3, 5, 6, 7, 9])
def test_wavenet_ragged_groups_vs_oracle(n):
    """Fewer windows than a group of 4 holds, and every remainder of the last group: the rows of the missing windows are
    masked, the posteriors of the present ones equal the oracle's and do not depend on what else is in the batch."""
    w = load_weights("Wavenet")
    eng = get_engine("Wavenet", "tc")
    X = _windows("wavenet", w)[:9]
    post = eng.posteriors(X[:n], hop=1).cpu().numpy()[:, 0]
    assert post.shape == (n,)
    assert np.abs(post - R.posterior(X[:n], w)).max() < POST_ATOL
    full = eng.posteriors(X, hop=1).cpu().numpy()[:, 0]
    assert np.array_equal(post, full[:n])


def test_known_answers_on_device():
    for wname, L, want in (("CRNN", 151, 0.00343328), ("CRNN_arik_original", 151, 0.13182628),
                           ("Wavenet", 182, 0.12610082)):
        eng = get_engine(wname)
        p = eng.posteriors(np.zeros((2, L, 40), np.float32), hop=1).cpu().numpy()
        assert p.shape == (2, 1) and np.abs(p - want).max() < 1e-5


@pytest.mark.parametrize("wname", ["CRNN", "Wavenet"])
def test_posteriors_sliding_windows(wname):
    w = load_weights(wname)
    eng = get_engine(wname)
    L = int(w["mel_length"])
    x = np.stack([np.clip(synth.stream_float(16000 * 2 + 777, c, 6, c), -1, 1) for c in (2, 0)]).astype(np.float32)
    mel = eng.filter(x)
    F = mel.shape[1]
    p2 = eng.posteriors(mel, hop=2).cpu().numpy()
    p1 = eng.posteriors(mel, hop=1).cpu().numpy()
    assert p2.shape == (2, (F - L) // 2 + 1) and p1.shape == (2, F - L + 1)
    np.testing.assert_array_equal(p1[:, ::2][:, :p2.shape[1]], p2)      # same windows, same bits
    melh = mel.cpu().numpy()
    j = np.arange(0, p2.shape[1], 7)
    for s in range(2):
        win = melh[s][(2 * j)[:, None] + np.arange(L)[None, :]]
        assert np.abs(p2[s, j] - R.posterior(win, w)).max() < POST_ATOL
    # too few frames -> no windows
    assert eng.posteriors(mel[:, :L - 1], hop=2).shape == (2, 0)


@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_pipeline_device_and_host(wname, name, wake_pcm):
    w = load_weights(wname)
    eng = get_engine(wname)
    pcm = np.stack([wake_pcm[name][:32000], synth.stream_int16(32000, 2, 8, 1)])
    post = eng.pipeline(pcm, hop=2).cpu().numpy()
    host = eng.pipeline_host(pcm, hop=2)
    np.testing.assert_array_equal(post, host)
    for s in range(2):
        mel = R.mel_stream(R.int16_to_float(pcm[s]), w)
        nw = R.eval_windows(mel.shape[0], int(w["mel_length"]))
        j = np.arange(0, nw, 3)
        ref = R.posterior(mel[(2 * j)[:, None] + np.arange(int(w["mel_length"]))[None, :]], w)
        assert np.abs(post[s, j] - ref).max() < POST_ATOL
    assert post[0].max() > 0.9 and post[1].max() < 0.5


def test_sweep_host_pipeline_two_jobs_in_flight(wake_pcm):
    """wwb_sweep_submit / wwb_sweep_wait: host PCM -> ONE copy + ONE filter pass -> CRNN and WaveNet posteriors and the
    FAR / FRR counters in host memory; two jobs in flight.  Results equal the device-buffer path bit for bit, and the
    synchronous wwb_pipeline_host accepts pageable numpy buffers."""
    from wakeword_detection_b200 import _cabi
    crnn, wn = get_engine("CRNN"), get_engine("Wavenet")
    S, N = 70, 64000
    thr = R.thresholds_eval()
    jobs = []
    for j in range(3):
        pcm = _cabi.pinned_empty((S, N), np.int16)
        pcm[:] = synth.batch_int16(S, N, seed=40 + j)
        pcm[j, 1000:1000 + 35200] = wake_pcm["crnn"]
        pcm[j + 5, 20000:20000 + 35200] = wake_pcm["wavenet"]
        jobs.append(pcm)
    recs = [crnn.sweep_submit(jobs[0], 2, thr, others=[wn]), crnn.sweep_submit(jobs[1], 2, thr, others=[wn])]
    with pytest.raises(IndexError):
        crnn.sweep_submit(jobs[2], 2, thr, others=[wn])              # two jobs are in flight already
    crnn.sweep_wait()
    recs.append(crnn.sweep_submit(jobs[2], 2, thr, others=[wn]))
    crnn.sweep_wait()
    crnn.sweep_wait()
    with pytest.raises(IndexError):
        crnn.sweep_wait()
    for pcm, rec in zip(jobs, recs):
        for m, eng in enumerate((crnn, wn)):
            post = eng.pipeline(pcm.copy(), hop=2)
            np.testing.assert_array_equal(rec["post"][m], post.cpu().numpy())
            seg = np.arange(S + 1) * post.shape[1]
            np.testing.assert_array_equal(rec["far"][m], eng.eval_counts(post, seg, thr, "far_edges").cpu().numpy())
            np.testing.assert_array_equal(rec["frr"][m], eng.eval_counts(post, seg, thr, "frr_max").cpu().numpy())
            assert rec["frr"][m][0] >= 1                              # the spliced clip fires its model
    # synchronous single-model call, pageable input and output
    pageable = np.array(jobs[0])
    out = wn.pipeline_host(pageable, hop=2)
    np.testing.assert_array_equal(out, recs[0]["post"][1])
    small = crnn.pipeline_host(pageable[:3, :16000], hop=2)
    np.testing.assert_array_equal(small, crnn.pipeline(pageable[:3, :16000].copy(), hop=2).cpu().numpy())
    assert crnn.pipeline_host(np.zeros((2, 400), np.int16), hop=2).shape == (2, 0)


def test_crnn_batch_config3_properties():
    """config 3 shape: 8192 windows in one launch; the batch a window sits in must not
    change its result, and window order is preserved."""
    import torch
    eng = get_engine("CRNN")
    pcm = synth.device_pcm(64, 160 * 300 + 512, seed=3, device=eng.device)
    mel = eng.filter(pcm)                                    # [64, 301, 40]
    wins = mel.unfold(1, 151, 1).permute(0, 1, 3, 2)[:, :128].reshape(-1, 151, 40).contiguous()   # 8192
    assert wins.shape[0] == 8192
    p = eng.posteriors(wins, hop=1)[:, 0]
    perm = torch.randperm(8192, device=eng.device)
    pp = eng.posteriors(wins[perm].contiguous(), hop=1)[:, 0]
    assert torch.equal(pp, p[perm])
    assert torch.equal(eng.posteriors(wins[77:78].contiguous(), hop=1)[:, 0], p[77:78])
    assert bool(((p >= 0) & (p <= 1)).all())


def test_wavenet_config4_streaming_shape():
    """config 4 shape: 4096 streams, one new mel frame per push (hop 1)."""
    import torch
    eng = get_engine("Wavenet")
    S = 4096
    if eng._stream_cap is None:
        eng.stream_alloc(S, 320)
    else:
        eng.stream_reset()
    pcm = synth.device_pcm(S, 160 * 6 + 512, seed=9, device=eng.device)
    eng2 = get_engine("Wavenet")
    mel = eng2.filter(pcm)                                   # 7 frames per stream
    posts = []
    o = 0
    for n in (320, 192, 160, 160, 160, 160, 160, 160):
        post, npost, trig, pmax = eng.stream_push(pcm[:, o:o + n].contiguous())
        o += n
        want = 0 if o < 512 else 1
        assert int(npost.min()) == want and int(npost.max()) == want
        if want:
            posts.append(post[:, 0].clone())
    assert len(posts) == 7
    # window k = 182-k zeros + the first k mel frames: check two streams against the batch path
    for k in (1, 7):
        win = torch.zeros((2, 182, 40), device=eng.device)
        win[:, 182 - k:] = mel[:2, :k]
        ref = eng2.posteriors(win, hop=1)[:, 0]
        assert float((posts[k - 1][:2] - ref).abs().max()) < 1e-6


# ------------------------------------------------------------------------------------ BASELINE configs vs the oracle
def _bench_pcm(eng, name, wake_pcm, S=512, N=160000):
    """The headline shape: 512 streams x 10 s of device-generated PCM with the wake clip spliced into three streams
    (start, middle, end of the batch; at the start, in the middle and at the end of the stream)."""
    import torch
    pcm = synth.device_pcm(S, N, seed=1234, device=eng.device)
    wk = torch.from_numpy(wake_pcm[name]).to(eng.device)
    for sidx, at in ((0, 0), (S // 2 - 1, 60000), (S - 1, N - wk.numel())):
        pcm[sidx, at:at + wk.numel()] = wk
    return pcm


@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_bench_shape_posteriors_vs_oracle(wname, name, wake_pcm):
    """BASELINE config 5 step shape (512 x 10 s, hop 2) through wwb_pipeline against the oracle on >= 2000 windows:
    every window of the first / last stream, of the three streams that carry a wake clip and of two noise streams.  Decisions are exact outside the tolerance band (wakeword/tflite.py:233-239, evaluate_models.py:70-86)."""
    w = load_weights(wname)
    eng = get_engine(wname)
    L = int(w["mel_length"])
    pcm = _bench_pcm(eng, name, wake_pcm)
    post = eng.pipeline(pcm, hop=2).cpu().numpy()
    nw = post.shape[1]
    assert nw == R.eval_windows(997, L)
    checked, worst, flips = 0, 0.0, 0
    fired = []
    for sidx in (0, 1, 255, 300, 511):
        mel = R.mel_stream(R.int16_to_float(pcm[sidx].cpu().numpy()), w)
        j = np.arange(nw)
        ref = R.posterior(mel[(2 * j)[:, None] + np.arange(L)[None, :]], w)
        err = np.abs(post[sidx, j] - ref)
        worst = max(worst, float(err.max()))
        checked += j.size
        band = np.abs(ref - 0.5) <= POST_ATOL
        flips += int(((post[sidx, j] > 0.5) != (ref > 0.5))[~band].sum())
        fired.append(bool((ref > 0.5).any()))
    print("%s bench shape: %d windows checked, max |err| %.3e, %d decision flips outside the band" % (wname, checked, worst, flips))
    assert checked >= 2000 and worst < POST_ATOL and flips == 0
    assert fired == [True, False, True, False, True]            # the spliced clips fire, the noise streams do not


def test_crnn_config3_vs_oracle():
    """BASELINE config 3: 8192 independent [151, 40] windows in one wwb_posteriors call (per-window tiles, no column
    sharing) against the oracle on 2049 of them (every 4th, and the last)."""
    w = load_weights("CRNN")
    eng = get_engine("CRNN")
    pcm = synth.device_pcm(64, 160 * 300 + 512, seed=3, device=eng.device)
    mel = eng.filter(pcm)                                    # [64, 301, 40]
    wins = mel.unfold(1, 151, 1).permute(0, 1, 3, 2)[:, :128].reshape(-1, 151, 40).contiguous()
    adv = np.load(__import__("os").path.join(__import__("conftest").GOLDEN, "wake_crnn_mel.npy"))
    wins[4:4 * adv.shape[0] + 4:4] = __import__("torch").from_numpy(adv).to(eng.device)   # windows across the posterior range
    assert wins.shape[0] == 8192
    post = eng.posteriors(wins, hop=1)[:, 0].cpu().numpy()
    j = np.unique(np.concatenate([np.arange(0, 8192, 4), [8191]]))
    ref = R.posterior(wins[j].cpu().numpy(), w)
    err = np.abs(post[j] - ref)
    band = np.abs(ref - 0.5) <= POST_ATOL
    print("config 3: %d windows checked, max |err| %.3e" % (j.size, err.max()))
    assert err.max() < POST_ATOL and ref.max() > 0.9
    assert np.array_equal((post[j] > 0.5)[~band], (ref > 0.5)[~band])


def test_wavenet_config4_stream_push_vs_oracle(wake_pcm, w_wavenet):
    """BASELINE config 4: 4096 streams, one new mel frame per wwb_stream_push (hop 1, 160-sample chunks), 220 pushes.
    64 streams are checked against the oracle: 4 of them (two carry the wake clip) on every push incl. trigger latch and
    posterior max, the others on every 8th push.  Window k = the last 182 rows of [182 zero rows ; first k+1 mel frames]
    (wakeword/tflite.py:102, :193-215)."""
    import torch
    from wakeword_detection_b200 import _cabi
    w = w_wavenet
    S, n_push, L = 4096, 220, 182
    eng = _cabi.Engine(w, 0, "tc")
    eng.stream_alloc(S, 160)
    pcm = synth.device_pcm(S, 160 * n_push, seed=21, device=eng.device)
    wk = torch.from_numpy(wake_pcm["wavenet"]).to(eng.device)
    full = [0, 7, 2048, 4095]
    pcm[0, :wk.numel()] = wk[:160 * n_push]
    pcm[2048, 1600:1600 + wk.numel()] = wk[:160 * n_push - 1600]
    part = [int(s) for s in np.linspace(1, 4094, 60).astype(int)]
    posts, trigs, pmax = [], [], None
    active = torch.zeros(S, dtype=torch.uint8, device=eng.device)
    for i in range(n_push):
        post, npost, trig, pmax = eng.stream_push(pcm[:, i * 160:(i + 1) * 160].contiguous(), is_active=active)
        want = 0 if (i + 1) * 160 < 512 else 1
        act = active.bool()
        assert bool((npost[~act] == want).all()) and bool((npost[act] == 0).all())
        active |= trig
        posts.append(post[:, 0].clone())
        trigs.append(trig.clone())
    posts = torch.stack(posts).cpu().numpy()            # [push, stream]
    trigs = torch.stack(trigs).cpu().numpy().astype(bool)
    first_frame_push = 3                                # 512 samples are complete during push 3 (0-based)
    checked, worst = 0, 0.0
    for sidx in full + part:
        mel = R.mel_stream(R.int16_to_float(pcm[sidx].cpu().numpy()), w)
        padded = np.concatenate([np.zeros((L, 40), np.float32), mel])
        ks = np.arange(mel.shape[0]) if sidx in full else np.arange(0, mel.shape[0], 8)
        ref = R.posterior(padded[(ks + 1)[:, None] + np.arange(L)[None, :]], w)
        got = posts[ks + first_frame_push, sidx]
        live = ~np.isnan(got)                           # after the trigger latched the stream stops sampling (:139-140)
        err = np.abs(got[live] - ref[live])
        worst = max(worst, float(err.max()))
        checked += int(live.sum())
        if sidx in full:
            over = np.nonzero(ref > 0.5)[0]
            band = np.abs(ref - 0.5) <= POST_ATOL
            if over.size and not band.any():
                k0 = int(over[0])
                assert trigs[k0 + first_frame_push, sidx] and trigs[:, sidx].sum() == 1
                assert np.isnan(posts[k0 + first_frame_push + 1:, sidx]).all()
                assert abs(float(pmax[sidx]) - ref[:k0 + 1].max()) < POST_ATOL
            elif not over.size:
                assert not trigs[:, sidx].any() and live.all()
                assert abs(float(pmax[sidx]) - ref.max()) < POST_ATOL
    print("config 4: %d pushes checked on 64 streams, max |err| %.3e" % (checked, worst))
    assert worst < POST_ATOL and checked >= 2000
    assert trigs[:, 0].any() and trigs[:, 2048].any()
    eng.close()



def test_crnn_streaming_many_windows_per_push(w_crnn):
    """4096 streams x 1600-sample chunks = up to 40960 windows per wwb_stream_push (beyond one 37888-window chunk of the
    CRNN path): the push scores them all; two streams are checked against the oracle's trigger state machine, and a
    capacity the library cannot serve is refused at wwb_stream_alloc, before any state exists."""
    import torch
    from wakeword_detection_b200 import _cabi
    eng = _cabi.Engine(w_crnn, 0, "tc")
    S = 4096
    eng.stream_alloc(S, 1600)
    assert eng.stream_max_frames() == 10
    pcm = synth.device_pcm(S, 1600 * 4, seed=33, device=eng.device)
    oracles = {sidx: R.TriggerOracle(w_crnn) for sidx in (0, 4095)}
    for i in range(4):
        post, npost, trig, pmax = eng.stream_push(pcm[:, i * 1600:(i + 1) * 1600].contiguous())
        want = 7 if i == 0 else 10                     # (1600 - 512) // 160 + 1 = 7 frames complete in the first chunk
        assert int(npost.min()) == want and int(npost.max()) == want
        for sidx, o in oracles.items():
            before = len(o.posteriors)
            o(pcm[sidx, i * 1600:(i + 1) * 1600].cpu().numpy(), True)
            ref = np.array(o.posteriors[before:], np.float32)
            assert np.abs(post[sidx, :want].cpu().numpy() - ref).max() < POST_ATOL
    eng.close()
    big = _cabi.Engine(w_crnn, 0, "tc")
    with pytest.raises(ValueError):
        big.stream_alloc(200000, 1600)                 # 2 M windows per push: refused up front
    big.close()


# ------------------------------------------------------------------------------------ counters
def test_eval_counts_vs_oracle(golden):
    eng = get_engine("CRNN")
    rng = np.random.default_rng(4)
    traj = golden["pm_traj"].astype(np.float32)
    for thr in (R.thresholds_eval(), R.thresholds_plot()):
        sm = R.smooth_same(traj)
        want = np.array([R.rising_edges(sm, t) for t in thr])
        got = eng.eval_counts(traj, [0, traj.size], thr, "far_edges").cpu().numpy()
        np.testing.assert_array_equal(got, want)
        # several segments: counts add, nothing leaks across segment boundaries
        cuts = [0, 900, 2500, 5000]
        want2 = sum(np.array([R.rising_edges(R.smooth_same(traj[a:b]), t) for t in thr])
                    for a, b in zip(cuts[:-1], cuts[1:]))
        got2 = eng.eval_counts(traj, cuts, thr, "far_edges").cpu().numpy()
        np.testing.assert_array_equal(got2, want2)
        pos = rng.random(777).astype(np.float32)
        seg = np.concatenate([[0], np.cumsum(rng.integers(1, 9, size=150))])
        seg = seg[seg <= 777]
        mx = np.array([pos[a:b].max() for a, b in zip(seg[:-1], seg[1:])])
        want3 = np.array([(mx > t).sum() for t in thr])
        got3 = eng.eval_counts(pos, seg, thr, "frr_max").cpu().numpy()
        np.testing.assert_array_equal(got3, want3)


def test_eval_counts_time_chunks_sum_to_whole(golden):
    from wakeword_detection_b200 import dist as wd
    eng = get_engine("CRNN")
    traj = golden["pm_traj"].astype(np.float32)
    thr = R.thresholds_eval()
    whole = eng.eval_counts(traj, [0, traj.size], thr, "far_edges").cpu().numpy()
    for world in (2, 4, 8):
        total = np.zeros_like(whole)
        for b, e, lo, hi in wd.time_chunks(traj.size, world):
            part = traj[b - lo:e + hi]
            total += eng.eval_counts(part, [0, part.size], thr, "far_edges", halo_lo=[lo], halo_hi=[hi]).cpu().numpy()
        np.testing.assert_array_equal(total, whole)


def test_plot_eval_models_process_results_dropin(golden):
    """utils/plot_eval_models.py:84-129: the 491-threshold sweep of `process_results` from one pass of the counter kernels
    equals the reference's own `threshold_accepts` loop on the golden trajectory (pm_accepts) and the FRR definition."""
    from wakeword_detection_b200 import plot_eval_models as PM
    eng = get_engine("CRNN")
    traj = golden["pm_traj"]                                   # an (already smooth) trajectory in [0, 1]
    rng = np.random.default_rng(8)
    wake = rng.random(333).astype(np.float32)
    res = PM.process_results({"CRNN": {"wakeword": wake, "smooth_not_wakeword": traj}}, 333, 2.5, engine=eng)["CRNN"]
    thr = golden["pm_thr"]
    np.testing.assert_array_equal(res["thresholds"], thr)
    traj32 = traj.astype(np.float32).astype(np.float64)        # the kernel reads float32 posteriors
    acc = np.array([PM.threshold_accepts(traj32, t) for t in thr])
    assert res["FAR"] == sorted((acc / 2.5).tolist())
    assert res["FRR"] == sorted(((333 - np.array([(wake > t).sum() for t in thr])) / 333).tolist())[::-1]
    assert res["smooth_FAR"].shape == (462,) and res["smooth_FRR"].shape == (462,)
    for t in (0.5, 0.7, 0.9):
        assert PM.threshold_accepts(traj32, t, engine=eng) == PM.threshold_accepts(traj32, t)
    same = np.array([PM.threshold_accepts(traj, t) for t in thr])
    assert (same == golden["pm_accepts"]).all()                # the host form is the reference's loop


def test_eval_counts_errors():
    eng = get_engine("CRNN")
    with pytest.raises(ValueError):
        eng.eval_counts(np.zeros(10, np.float32), [0, 5, 5, 10], [0.5, 0.6], "frr_max")     # empty clip
    with pytest.raises(ValueError):
        eng.eval_counts(np.zeros(10, np.float32), [0, 10], [0.6, 0.5], "far_edges")         # unsorted
    # a trajectory shorter than the smoothing window: np.convolve(..., 'same') swaps its operands and returns 30 values
    short = np.array([0.9, 0.95, 0.2, 0.99, 0.97, 0.1, 0.1, 0.98, 0.9, 0.96], np.float32)
    thr = np.array([0.1, 0.2, 0.25, 0.3, 0.5])
    sm = np.convolve(short, np.ones(30) / 30, mode="same")
    assert sm.size == 30
    want = np.array([R.rising_edges(sm, t) for t in thr])
    np.testing.assert_array_equal(eng.eval_counts(short, [0, 10], thr, "far_edges").cpu().numpy(), want)
    both = np.concatenate([short, np.linspace(0, 1, 50).astype(np.float32)])
    want2 = want + np.array([R.rising_edges(R.smooth_same(both[10:]), t) for t in thr])
    np.testing.assert_array_equal(eng.eval_counts(both, [0, 10, 60], thr, "far_edges").cpu().numpy(), want2)


# ------------------------------------------------------------------------------------ drop-ins
@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_wakeword_trigger_replays_golden(wname, name, golden):
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200.wakeword import WakewordTrigger
    from wakeword_detection_b200.context import SpeechContext
    trig = WakewordTrigger(model_dir=os.path.join(WEIGHTS, wname), model_type=wname)
    assert trig.mel_length == (151 if name == "crnn" else 182) and trig.mel_width == 40
    assert trig.hop_length == 160 and trig.encode_width == (64 if name == "crnn" else 32)
    ctx = SpeechContext()
    pcm, sp = golden["trig_%s_pcm" % name], golden["trig_%s_speech" % name]
    posts, at = [], -1
    for i in range(len(sp)):
        ctx.is_speech = bool(sp[i])
        trig(ctx, pcm[i * 320:(i + 1) * 320])
        posts += list(trig.last_posteriors)
        if ctx.is_active:
            at = i
            break
    ref = golden["trig_%s_post" % name]
    assert len(posts) == len(ref)
    assert np.abs(np.array(posts) - ref).max() < POST_ATOL
    assert at == int(golden["trig_%s_active_at" % name])
    assert abs(trig._posterior_max - float(golden["trig_%s_post_max" % name])) < POST_ATOL
    # once active the stage stops sampling (wakeword/tflite.py:139-140)
    trig(ctx, pcm[:320])
    assert len(trig.last_posteriors) == 0
    # VAD fall resets the windows (:143-146)
    ctx.is_active = False
    ctx.is_speech = False
    trig(ctx, pcm[:320])
    assert trig._posterior_max == 0.0
    with pytest.raises(ValueError):
        WakewordTrigger(model_dir=os.path.join(WEIGHTS, wname), model_type=wname, fft_window_type="hamming")
    trig.close()


def test_multistream_trigger_vs_oracle(wake_pcm, w_crnn):
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200.wakeword import MultiStreamTrigger
    S = 5
    ms = MultiStreamTrigger(os.path.join(WEIGHTS, "CRNN"), "CRNN", S, 320)
    pcm = np.stack([np.concatenate([synth.stream_int16(1600 * s, 0, 2, s), wake_pcm["crnn"]])[:32000] for s in range(S)])
    speech = np.ones((100, S), bool)
    speech[:, 1] = False                       # stream 1: VAD never opens -> no posteriors
    speech[40:44, 2] = False                   # stream 2: a VAD fall resets it mid-way
    oracles = [R.TriggerOracle(w_crnn) for _ in range(S)]
    active = np.zeros(S, bool)
    for i in range(100):
        out = ms.push(pcm[:, i * 320:(i + 1) * 320], speech[i], active)
        npost = out["n_post"].cpu().numpy()
        post = out["post"].cpu().numpy()
        trig = out["trigger"].cpu().numpy().astype(bool)
        for s in range(S):
            o = oracles[s]
            before = len(o.posteriors)
            o.active = bool(active[s])
            o(pcm[s, i * 320:(i + 1) * 320], bool(speech[i, s]))
            new = np.array(o.posteriors[before:], np.float32)
            assert npost[s] == len(new), (i, s)
            if len(new):
                assert np.abs(post[s, :len(new)] - new).max() < POST_ATOL
                band = np.abs(new - 0.5) <= POST_ATOL
                if not band.any():
                    assert trig[s] == bool((new > 0.5).any() and not active[s])
        active |= trig
    assert active[0] and not active[1]
    ms.close()


@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_device_pipeline_state_machine_replays_reference_run(wname, name):
    """SURVEY 8f row 2: vad debounce -> trigger -> activation timeout for many streams on the device
    (wwb_context_step) against (a) the golden run of the reference's own three stages (stream 0) and (b) the oracle's
    PipelineOracle on streams with other raw-VAD scripts / audio (time-shifted copies)."""
    import os
    from conftest import GOLDEN, WEIGHTS
    from wakeword_detection_b200.wakeword import MultiStreamPipeline
    w = load_weights(wname)
    g = np.load(os.path.join(GOLDEN, "reference_pipeline.npz"))
    cfg = dict(zip(("frame_width", "vad_rise_delay", "vad_fall_delay", "min_active", "max_active"), [int(v) for v in g["cfg"]]))
    pcm0, raw0 = g["pipe_%s_pcm" % name], g["pipe_%s_raw" % name]
    nf = len(raw0)
    S = 5
    rng = np.random.default_rng(11)
    pcm = np.stack([np.roll(pcm0, 320 * 7 * s) for s in range(S)])
    raw = np.stack([raw0] + [np.roll(raw0, 7 * s) ^ (rng.random(nf) < 0.03) for s in range(1, S)])
    raw[4] = True                                        # a stream whose VAD never falls: only max_active ends activations
    pipe = MultiStreamPipeline(os.path.join(WEIGHTS, wname), wname, S, **cfg)
    oracles = [R.PipelineOracle(w, **cfg) for _ in range(S)]
    acts = np.zeros((nf, S), bool)
    for i in range(nf):
        out = pipe.step(pcm[:, i * 320:(i + 1) * 320], raw[:, i])
        sp, ac = out["is_speech"].cpu().numpy().astype(bool), out["is_active"].cpu().numpy().astype(bool)
        acts[i] = ac
        for s in range(S):
            o = oracles[s]
            before = len(o.trig.posteriors)
            want_sp, want_ac = o(pcm[s, i * 320:(i + 1) * 320], raw[s, i])
            new = np.array(o.trig.posteriors[before:], np.float32)
            near = new.size and np.abs(new - 0.5).min() <= POST_ATOL
            assert sp[s] == want_sp, (i, s)
            assert int(out["n_post"][s]) == new.size, (i, s)
            if new.size:
                assert np.abs(out["post"][s, :new.size].cpu().numpy() - new).max() < POST_ATOL
            if not near:
                assert ac[s] == want_ac, (i, s)
    np.testing.assert_array_equal(acts[:, 0], g["pipe_%s_active" % name])      # the reference's own run
    assert acts[:, 0].any() and not acts[-1, 0] or name == "crnn"
    pipe.reset()
    out = pipe.step(pcm[:, :320], raw[:, 0])
    assert not out["is_active"].any()
    pipe.close()


def test_keyword_recognizer_dropin_replays_reference_run():
    """SURVEY 8f row 4: the KeywordRecognizer drop-in (mel frames from the CUDA filter kernel with pre-emphasis 0.97,
    the reference's window / state / event logic) against the golden run of the reference's own class with the same
    stand-in keyword model pair (the reference ships no keyword model), and the constructor's error behaviour."""
    import os
    import sys
    from conftest import GOLDEN, WEIGHTS
    sys.path.insert(0, GOLDEN)
    import keyword_stub as KS
    from wakeword_detection_b200.context import SpeechContext
    from wakeword_detection_b200.keyword import KeywordRecognizer
    g = np.load(os.path.join(GOLDEN, "reference_keyword.npz"))
    d = os.path.join(WEIGHTS, "CRNN")
    classes = ["up", "down", "stop"]
    rec = KeywordRecognizer(classes=classes, model_dir=d, posterior_threshold=float(g["kw_threshold"]),
                            encode_model=KS.Encode(), detect_model=KS.Detect())
    assert (rec.mel_length, rec.mel_width, rec.encode_length, rec.encode_width) == (12, 40, 5, 6)
    ctx = SpeechContext()
    events = []
    ctx.add_handler("recognize", lambda c: events.append(("recognize", c.transcript, float(c.confidence))))
    ctx.add_handler("timeout", lambda c: events.append(("timeout", "", 0.0)))
    pcm, active = g["kw_pcm"], g["kw_active"]
    frames = []
    for i in range(len(active)):
        ctx.is_active = bool(active[i])
        n0 = len(events)
        rec(ctx, pcm[i * 320:(i + 1) * 320])
        frames += [i] * (len(events) - n0)
        assert np.abs(rec._encoded - g["kw_enc_window"][i]).max() < 1e-3, i
    assert frames == list(g["kw_event_frame"])
    assert [e[0] for e in events] == list(g["kw_event_kind"]) and [e[1] for e in events] == list(g["kw_event_class"])
    assert np.abs(np.array([e[2] for e in events]) - g["kw_event_conf"]).max() < 1e-3
    with pytest.raises(ValueError):
        KeywordRecognizer(classes=classes, model_dir=d)                     # no keyword encoder family in the library
    with pytest.raises(ValueError):
        KeywordRecognizer(classes=["a", "b"], model_dir=d, encode_model=KS.Encode(), detect_model=KS.Detect())
    with pytest.raises(ValueError):
        KeywordRecognizer(classes=classes, model_dir=d, fft_window_type="hamming", encode_model=KS.Encode(), detect_model=KS.Detect())
    rec.close()


def test_tflite_model_and_filter_dropins(golden, w_crnn):
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200.models import TFLiteModel
    from wakeword_detection_b200.filter import Filter
    d = os.path.join(WEIGHTS, "CRNN")
    f, e, dt = (TFLiteModel(os.path.join(d, n + ".tflite")) for n in ("filter", "encode", "detect"))
    assert list(f.input_details[0]["shape"]) == [1, 257] and list(e.input_details[0]["shape"]) == [1, 40, 151, 1]
    assert list(dt.input_details[0]["shape"]) == [1, 64] and list(dt.output_details[0]["shape"]) == [1, 1]
    x = np.zeros((1, 40, 151, 1), np.float32)
    post = dt(e(x)[0])[0]
    assert post.shape == (1, 1) and abs(float(post[0][0]) - 0.00343328) < 1e-5
    with pytest.raises(ValueError):
        e(np.zeros((1, 151, 40, 1), np.float32))
    with pytest.raises(ValueError):
        f(np.zeros((1, 257), np.float64))
    wd = os.path.join(WEIGHTS, "Wavenet")
    we, wdt = TFLiteModel(os.path.join(wd, "encode.tflite")), TFLiteModel(os.path.join(wd, "detect.tflite"))
    assert list(we.input_details[0]["shape"]) == [1, 182, 40]
    out = wdt(we(np.zeros((1, 182, 40), np.float32))[0])[0]
    np.testing.assert_allclose(out[0], [0.87389916, 0.12610082], atol=1e-5)

    # Filter.filter_frame over the ragged chunks of the golden run
    for tag, a in (("pe0", 0.0), ("pe97", 0.97)):
        flt = Filter(pre_emphasis=a, model_dir=d)
        assert flt.num_outputs() == 40
        xin = golden["filter_in"].copy()
        pos, mels, counts = 0, [], []
        for n in [320, 320, 7, 1000, 1, 512, 160, 159, 3000] + [320] * 40:
            chunk = xin[pos:pos + n].copy()
            pos += n
            if chunk.size == 0:
                break
            got = flt.filter_frame(chunk)
            counts.append(len(got))
            mels += got
        np.testing.assert_array_equal(counts, golden["filter_counts_" + tag])
        check_mel(np.stack(mels), golden["filter_mel_" + tag])
    with pytest.raises(ValueError):
        Filter(fft_window_type="hamming", model_dir=d)


@pytest.mark.parametrize("wname,name", [("CRNN_arik_original", "crnn"), ("Wavenet", "wavenet")])
def test_get_posterior_and_sweep_dropin(wname, name, golden):
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200 import evaluate_models as EM, _cabi
    d = os.path.join(WEIGHTS, wname)
    typ = "CRNN" if name == "crnn" else "Wavenet"
    clips = [golden["gp_%s_clip%d" % (name, i)] for i in range(3)]
    fn = np.array(EM.get_posterior(d, typ, "false_negatives", clips, 20, 16000))
    fa = np.array(EM.get_posterior(d, typ, "false_accepts", clips, 20, 16000))
    assert np.abs(fn - golden["gp_%s_frr_max" % name]).max() < POST_ATOL
    assert fa.shape == golden["gp_%s_far_traj" % name].shape
    assert np.abs(fa - golden["gp_%s_far_traj" % name]).max() < POST_ATOL
    # batching must not change anything (carry across clips is reproduced)
    fa1 = np.array(EM.get_posterior(d, typ, "false_accepts", clips, 20, 16000, batch_clips=1))
    np.testing.assert_array_equal(fa, fa1)
    # the sweep on the reference's own posteriors gives the reference's own numbers
    thr, FRR, FAR = EM.plot_FRR_FAR(golden["gp_%s_frr_max" % name], golden["gp_%s_far_traj" % name], 3, 0.5, typ,
                                    engine=_cabi.engine_for_dir(d, typ), show=False)
    np.testing.assert_array_equal(thr, golden["sweep_%s_thr" % name])
    np.testing.assert_array_equal(FRR, golden["sweep_%s_frr" % name])
    np.testing.assert_array_equal(FAR, golden["sweep_%s_far" % name])


@pytest.mark.parametrize("wname", ["CRNN_arik_original", "Wavenet"])
def test_sharded_evaluation_sums_to_single_process(wname, wake_pcm):
    """utils/evaluate_models.py:280-327 sharded over 1 / 2 / 4 / 8 (virtual) ranks on the CUDA path: contiguous runs of
    wake-word clips with the carried window + time chunks of the long false-accept clip with the (L-1)*160+352-sample
    PCM halo; the per-rank counters add up EXACTLY to the single-process sweep (the all-reduce itself is covered by
    the gloo world-2 test on CPU and by bench.py under torchrun)."""
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200 import evaluate_models as EM, _cabi
    typ = "Wavenet" if wname == "Wavenet" else "CRNN"
    d = os.path.join(WEIGHTS, wname)
    eng = _cabi.engine_for_dir(d, typ)
    wake = wake_pcm["wavenet" if typ == "Wavenet" else "crnn"].astype(np.float32) / 32768.0
    noise = lambda n, c, k: np.clip(synth.stream_float(n, c, 9, k), -1, 1).astype(np.float32)
    pos = [wake, noise(20321, 2, 1), wake[3000:30000], noise(16777, 0, 2), wake[:33001], noise(30000, 5, 3), wake[100:]]
    far = np.concatenate([noise(140000, 5, 4), wake, noise(252345, 2, 5), wake[:30000], noise(99999, 0, 6)])
    thr = R.thresholds_eval()
    kp = EM.get_posterior(d, typ, "false_negatives", pos, 20, 16000, engine=eng)
    nk = EM.get_posterior(d, typ, "false_accepts", [far], 20, 16000, engine=eng)
    acc1, edg1 = EM.sweep_counts(kp, nk, thr, eng)
    assert acc1[0] >= 2 and edg1[0] >= 1
    for world in (1, 2, 4, 8):
        acc, edg = np.zeros_like(acc1), np.zeros_like(edg1)
        for r in range(world):
            a, e = EM.evaluate_sharded(d, typ, pos, far, 20, 16000, thr, rank=r, world=world, engine=eng, reduce_over_ranks=False)
            acc += a
            edg += e
        np.testing.assert_array_equal(acc, acc1)
        np.testing.assert_array_equal(edg, edg1)


@pytest.mark.gpu
@pytest.mark.parametrize("wname", ["CRNN", "Wavenet"])
def test_encoders_are_deterministic(wname):
    """The tensor-core kernels hand tiles between warps through mbarriers / TMEM / shared memory; a missed
    dependency shows up as run-to-run differences.  Same input -> bit-identical posteriors, ragged sizes included."""
    import torch
    eng = get_engine(wname)
    for S, n in ((37, 52800), (3, 40000), (1, 32000)):
        pcm = synth.device_pcm(S, n, seed=100 + S, device=eng.device)
        mel = eng.filter(pcm)
        ref = eng.posteriors(mel, 2).clone()
        for _ in range(6):
            assert torch.equal(eng.posteriors(mel, 2), ref)


@pytest.mark.parametrize("S,F,hop", [(2, 411, 2), (5, 998, 2), (2, 700, 1), (3, 600, 4), (2, 1200, 8), (1, 153, 2), (40, 998, 2),
                                     (2, 1015, 2), (2, 1015, 1), (2, 1021, 2), (3, 151 + 2 * 72, 2),   # 1015: column t = 18 of the last windows is the strip's last row
                                     (4, 389, 2), (4, 391, 2), (5, 393, 2), (5, 395, 2), (3, 403, 2)])   # 120..127 windows per stream: position-ring tiles
                                                                                                          # that start 0..3 windows before a stream's end
def test_crnn_shared_columns_bit_identical_to_per_window_path(S, F, hop):
    """Sliding-window batches compute every conv / GRU-1 projection column once per stream position (crnn_tc.cu,
    CrnnShare); WWB_CRNN_NO_SHARE=1 forces the per-window tiles.  Same MMAs on the same operands: identical bits."""
    import os
    import torch
    tc, f32 = get_engine("CRNN", "tc"), get_engine("CRNN", "f32")
    torch.manual_seed(S * 1000 + F)
    X = torch.rand((S, F, 40), device=tc.device) * 5
    os.environ["WWB_CRNN_NO_SHARE"] = "1"
    try:
        a = tc.posteriors(X, hop=hop).clone()
    finally:
        os.environ["WWB_CRNN_NO_SHARE"] = "0"
    b = tc.posteriors(X, hop=hop).clone()
    assert bool((a == b).all())
    assert float((b - f32.posteriors(X, hop=hop)).abs().max()) < 1e-4


@pytest.mark.parametrize("S,F,hop", [(2, 411, 2), (5, 998, 2), (2, 700, 1), (3, 640, 4), (2, 1200, 8), (1, 196, 2), (40, 998, 2),
                                     (3, 641, 2), (2, 1100, 2), (2, 1101, 1), (1, 1561, 3)])   # 640 / 1100 / 1560: chunk boundaries of the stream pass
def test_wavenet_shared_activations_bit_identical_to_per_window_path(S, F, hop):
    """Sliding-window batches take every activation outside the causal-padding cone from a stream-level pass
    (wavenet_tc.cu, header); WWB_WN_NO_SHARE=1 computes every window on its own.  Same MMAs on the same operand values:
    identical bits; and both agree with the fp32 CUDA-core path."""
    import os
    import torch
    tc, f32 = get_engine("Wavenet", "tc"), get_engine("Wavenet", "f32")
    torch.manual_seed(S * 1000 + F)
    X = torch.rand((S, F, 40), device=tc.device) * 5
    os.environ["WWB_WN_NO_SHARE"] = "1"
    try:
        a = tc.posteriors(X, hop=hop).clone()
    finally:
        os.environ["WWB_WN_NO_SHARE"] = "0"
    b = tc.posteriors(X, hop=hop).clone()
    assert float((a - f32.posteriors(X, hop=hop)).abs().max()) < 1e-4
    assert bool((a == b).all())


@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_tf_lite_opts_models_predict_dropin(wname, name):
    """utils/evaluate_tf_lite_opts.py:49-67: clips -> posterior -> non-strict `>= threshold`, here as one batch."""
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200 import evaluate_tf_lite_opts as ETO
    w = load_weights(wname)
    X = _windows(name, w)
    ref = R.posterior(X, w)
    enc, det = ETO.load_tf_models(os.path.join(WEIGHTS, wname))
    post = ETO.posteriors(enc, det, X, wname)
    assert post.shape == (X.shape[0],) and np.abs(post - ref).max() < POST_ATOL
    for thr in (0.5, 0.9):
        preds = ETO.models_predict(enc, det, X, wname, threshold=thr)
        want = [1 if p >= thr else 0 for p in ref]
        flips = [i for i, (a, b) in enumerate(zip(preds, want)) if a != b]
        assert all(abs(ref[i] - thr) < POST_ATOL for i in flips)       # only inside the tolerance band
        assert 0 < sum(preds) < len(preds)
    assert ETO.models_predict(enc, det, X, wname, threshold=float(post[0]))[0] == 1     # `>=`, not `>`
    with pytest.raises(ValueError):
        ETO.models_predict(enc, det, X[:, :-1], wname)
    with pytest.raises(ValueError):
        ETO.models_predict(enc, det, X.astype(np.float64), wname)
    with pytest.raises(ValueError):
        ETO.models_predict(enc, det, X, "Wavenet" if wname == "CRNN" else "CRNN")


@pytest.mark.parametrize("wname,name", [("CRNN", "crnn"), ("Wavenet", "wavenet")])
def test_fp16_weight_variant_vs_oracle(wname, name):
    """SURVEY 8(f) row 3 / utils/evaluate_tf_lite_opts.py:103-131: the float16-weight variant (constants rounded to
    float16, float32 arithmetic) through the CUDA path against the oracle run on the SAME rounded weights (1e-3), plus the
    accuracy report the reference's script is after: how far the variant's posteriors / decisions are from float32."""
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200 import _cabi, weights as W, evaluate_tf_lite_opts as ETO
    w = load_weights(wname)
    wq = W.load_model_dir(os.path.join(WEIGHTS, wname), wname, quant=True)
    X = _windows(name, w)
    ref_q, ref_32 = R.posterior(X, wq), R.posterior(X, w)
    eng = _cabi.engine_for_dir(os.path.join(WEIGHTS, wname), wname, quant=True)
    post = eng.posteriors(X, hop=1).cpu().numpy()[:, 0]
    assert np.abs(post - ref_q).max() < POST_ATOL
    band = np.abs(ref_q - 0.5) <= POST_ATOL
    assert np.array_equal((post > 0.5)[~band], (ref_q > 0.5)[~band])
    drift = np.abs(ref_q - ref_32).max()
    flips = int(((ref_q >= 0.5) != (ref_32 >= 0.5)).sum())
    print("%s float16-weight variant: max |p16 - p32| = %.3e over %d windows, %d decision changes; CUDA vs oracle %.3e"
          % (wname, drift, X.shape[0], flips, np.abs(post - ref_q).max()))
    assert 1e-6 < drift < 5e-2                    # a different model (not the float32 one), but a close one
    # the drop-in entry points: -quant files are not shipped, so the variant is derived on request only
    enc, det = ETO.load_tf_models(os.path.join(WEIGHTS, wname), quant=True, derive_quant=True)
    assert enc.quant and det.quant
    p2 = ETO.posteriors(enc, det, X, wname)
    np.testing.assert_array_equal(p2, post)
    enc32, det32 = ETO.load_tf_models(os.path.join(WEIGHTS, wname))
    assert np.abs(ETO.posteriors(enc32, det32, X, wname) - ref_32).max() < POST_ATOL      # the float32 pair is a different engine


def test_dataset_filter_dropin(tmp_path, w_crnn):
    """utils/filter_dataset_to_h5.py:65-143: clips padded to whole 20 ms frames, ONE filter window carried across clips,
    empty clips dropped, features + attributes per clip; batched through the CUDA filter kernel."""
    import json
    import os
    from conftest import WEIGHTS
    from wakeword_detection_b200 import evaluate_tf_lite_opts as ETO
    from wakeword_detection_b200.filter_dataset import Dataset_Filter
    clips = [np.clip(synth.stream_float(n, c, 3, c), -1, 1).astype(np.float32) if n else np.zeros((0,), np.float32)
             for c, n in enumerate((16000, 9001, 333, 0, 24000))]
    meta = [{"audio_file_path": "audio/c%d.wav" % i, "is_hotword": i % 2, "worker_id": "w%d" % (i % 3)} for i in range(len(clips))]
    js = str(tmp_path / "test.json")
    json.dump(meta, open(js, "w"))
    df = Dataset_Filter(js, None, wake_word="hey-snips", sample_rate=16000, frame_width=20, hop_width=10,
                        out_dir=str(tmp_path / "out"), data_dir=str(tmp_path), models_dir=os.path.join(WEIGHTS, "CRNN"),
                        vad=lambda frame_bytes, sr: np.abs(np.frombuffer(frame_bytes, np.int16)).max() > 2000)
    recs = df.filter_clips(clips, [m["is_hotword"] for m in meta], [m["audio_file_path"] for m in meta])
    assert recs[3] is None and [r["file_name"] for r in recs if r] == ["c0", "c1", "c2", "c4"]
    # oracle: the padded clips back to back through one window (the reference's single Filter instance)
    padded = [np.pad(c, (0, -len(c) % 320)) for c in clips if len(c)]
    ref = R.mel_stream(np.concatenate(padded), w_crnn)
    rows = [(len(padded[0]) - 512) // 160 + 1] + [len(p) // 160 for p in padded[1:]]
    assert [r["features"].shape[0] for r in recs if r] == rows and sum(rows) == ref.shape[0]
    got = np.concatenate([r["features"] for r in recs if r])
    check_mel(got, ref)
    assert recs[0]["speech_start_ts"] >= 0 and recs[0]["speech_end_ts"] > recs[0]["speech_start_ts"]
    # whole-dataset path with array clips: write the npz twin and read it back with the evaluation loader
    df2 = Dataset_Filter(js, None, out_dir=str(tmp_path / "out"), data_dir="", models_dir=os.path.join(WEIGHTS, "CRNN"), vad=None)
    recs2 = [r for r in df2.filter_clips(clips, [m["is_hotword"] for m in meta], [m["audio_file_path"] for m in meta]) if r]
    for r, m in zip(recs2, [m for m, c in zip(meta, clips) if len(c)]):
        r["speaker"] = df2.speakers_dict[m["worker_id"]]
    path = df2.write_npz(recs2)
    X, y = ETO.load_data(path, 151, 40)
    assert X.shape == (4, 151, 40) and list(y) == [0, 1, 0, 0]
    assert np.array_equal(X[0, :rows[0]], recs2[0]["features"][:151]) and recs2[0]["speech_start_ts"] == -1
    assert df2.speakers_dict == {"w0": 0, "w1": 1, "w2": 2}
