"""The places where a batch call cuts its batch into pieces, each piece computed from offsets a single-piece call never
uses:

- the CRNN chunk loop (crnn_simt_posteriors): per-window batches cut every WWB_CRNN_CHUNK windows, shared-column
  batches cut into whole streams;
- the host-buffer pipeline (wwb_pipeline_host, wwb_sweep_submit / wwb_sweep_wait): the 1/8, 2/8, 5/8 stream slices,
  several models with different window counts in one sweep, two jobs in flight, refused jobs and the caller's buffers;
- the FAR / FRR counters at evaluation length, where the FAR kernel's grid-stride loop makes several passes.

The truth is the oracle in float64 (posteriors within 1e-3, decisions exact outside the band), the unsplit call bit
for bit wherever a split must be invisible, and the oracle's smoothing and edge loops for the counts."""
import ctypes
import math

import numpy as np
import pytest

from conftest import load_weights
from crnn_models import calibrate, mel_windows, shared_launches, synth_crnn
from oracle import restated as R
from streaming_helpers import wake_clip

F64 = np.float64
POST_ATOL = 1e-3
PRECISIONS = ["f32", "tc", "tc_fast"]
CHUNK_MODELS = ["crnn", "crnn97", "crnn17"]
STATS = []


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for line in STATS:
        print("\n[batch splits] " + line)


# ------------------------------------------------------------------------------------ models and engines
_WEIGHTS = {}


def weights(name):
    """the shipped CRNN (L = 151) and WaveNet (L = 182), and synthetic CRNNs at L = 97 (four conv variants, no position
    ring) and L = 17 (no interior column)"""
    if name not in _WEIGHTS:
        if name == "crnn":
            _WEIGHTS[name] = load_weights("CRNN")
        elif name == "wavenet":
            _WEIGHTS[name] = load_weights("Wavenet")
        else:
            L = int(name[4:])
            _WEIGHTS[name] = calibrate(synth_crnn(0, L), mel_windows(L))
    return _WEIGHTS[name]


@pytest.fixture(scope="module")
def engine():
    from wakeword_detection_b200 import _cabi
    made = {}

    def get(name, precision="tc"):
        if (name, precision) not in made:
            made[name, precision] = _cabi.Engine(weights(name), 0, precision)
        return made[name, precision]

    yield get
    for e in made.values():
        e.close()


def _pcm(S, N, dtype, seed):
    """[S, N] PCM: per-stream gain noise plus a tone, int16 over most of the int16 range or float32 in [-1, 1]"""
    r = np.random.default_rng(seed)
    t = np.arange(N) / 16000.0
    x = r.standard_normal((S, N)) * r.uniform(0.005, 0.3, (S, 1))
    x += 0.2 * np.sin(2 * np.pi * r.uniform(100, 3100, (S, 1)) * t[None, :])
    x = np.clip(x, -1, 1)
    if dtype == "float32":
        return x.astype(np.float32)
    return np.rint(x * 32767).astype(np.int16)


def _oracle_posteriors(pcm_row, w, hop, a, j):
    """float64 posteriors of windows j of one stream"""
    x = R.int16_to_float(pcm_row) if pcm_row.dtype == np.int16 else pcm_row.astype(np.float32)
    mel = R.mel_stream(x, w, a)
    L = int(w["mel_length"])
    return R.posterior(mel[(hop * np.asarray(j))[:, None] + np.arange(L)[None, :]], w, F64)


def _check_vs_float64(post, ref, what):
    err = float(np.abs(np.asarray(post, F64) - ref).max())
    assert err < POST_ATOL, (what, err)
    band = np.abs(ref - 0.5) <= POST_ATOL
    assert np.array_equal((post > 0.5)[~band], (ref > 0.5)[~band]), what
    return err


# ------------------------------------------------------------------------------------ A. CRNN chunks
def _chunked(eng, monkeypatch, chunk, fn):
    """fn() with WWB_CRNN_CHUNK = chunk (None: unset); returns (result, kernel launches)"""
    if chunk is None:
        monkeypatch.delenv("WWB_CRNN_CHUNK", raising=False)
    else:
        monkeypatch.setenv("WWB_CRNN_CHUNK", str(chunk))
    try:
        n0 = eng.launch_count()
        out = fn()
        return out, eng.launch_count() - n0
    finally:
        monkeypatch.delenv("WWB_CRNN_CHUNK", raising=False)


def _mel(eng, S, F, seed):
    """[S, F, 40] device mel of seeded synthetic PCM"""
    from wakeword_detection_b200 import synth
    return eng.filter(synth.device_pcm(S, 512 + 160 * (F - 1), seed, eng.device))


def _same(a, b):
    import torch
    return a.shape == b.shape and bool(torch.equal(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", CHUNK_MODELS)
def test_crnn_chunks_independent_windows(name, precision, engine, monkeypatch):
    """700 independent windows at chunks of 128, 129, 300 and 699 windows: posteriors and encoder outputs equal the
    unsplit call bit for bit, and the call ran ceil(700 / chunk) chunks"""
    import torch
    eng = engine(name, precision)
    L = eng.L
    mel = _mel(eng, 4, 400, 11)
    g = torch.Generator(device=eng.device)
    g.manual_seed(L)
    s = torch.randint(0, 4, (700,), device=eng.device, generator=g)
    t0 = torch.randint(0, 400 - L + 1, (700,), device=eng.device, generator=g)
    X = mel[s[:, None], t0[:, None] + torch.arange(L, device=eng.device)[None, :]].contiguous()
    run = lambda: (eng.posteriors(X, hop=1), eng.encode(X))
    (p0, e0), n0 = _chunked(eng, monkeypatch, None, run)
    assert p0.shape == (700, 1) and e0.shape == (700, 64)
    for chunk in (128, 129, 300, 699):
        (p, e), n = _chunked(eng, monkeypatch, chunk, run)
        assert n == math.ceil(700 / chunk) * n0, (chunk, n, n0)
        assert _same(p, p0) and _same(e, e0), chunk


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", CHUNK_MODELS)
def test_crnn_chunks_per_window_sliding(name, precision, engine, monkeypatch):
    """3 streams x 700 frames at hop 2 on the per-window path (WWB_CRNN_NO_SHARE=1; f32 always takes it) at chunks of
    128 and 300 windows, which cut streams in the middle: posteriors equal the unsplit call bit for bit"""
    eng = engine(name, precision)
    monkeypatch.setenv("WWB_CRNN_NO_SHARE", "1")
    mel = _mel(eng, 3, 700, 12)
    wps = eng.num_windows(700, 2)
    B = 3 * wps
    run = lambda: eng.posteriors(mel, hop=2)
    p0, n0 = _chunked(eng, monkeypatch, None, run)
    for chunk in (128, 300):
        assert chunk % wps, chunk                    # the first cut falls inside a stream
        p, n = _chunked(eng, monkeypatch, chunk, run)
        assert n == math.ceil(B / chunk) * n0, (chunk, n, n0)
        assert _same(p, p0), chunk


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", CHUNK_MODELS)
def test_crnn_chunks_shared_columns(name, precision, engine, monkeypatch):
    """7 streams x 998 frames at hops 1, 2, 4 and 8, chunks of 1, 2, 3 and 6 streams and of 3 wps - 1 windows (2 streams;
    wps = windows per stream): the shared-column path (tc, tc_fast) cuts whole streams and shifts the mel of every chunk
    after the first; f32 cuts the same batches into chunks of windows.  Posteriors equal the unsplit call bit for bit."""
    eng = engine(name, precision)
    monkeypatch.setenv("WWB_CRNN_NO_SHARE", "0")
    mel = _mel(eng, 7, 998, 13)
    shared = precision != "f32"
    for hop in (1, 2, 4, 8):
        wps = eng.num_windows(998, hop)
        run = lambda: eng.posteriors(mel, hop=hop)
        p0, n0 = _chunked(eng, monkeypatch, None, run)
        if shared:
            assert n0 == shared_launches(eng.L), (hop, n0)
        for chunk in [k * wps for k in (1, 2, 3, 6)] + [3 * wps - 1]:
            c = max(128, chunk)                      # the library's smallest chunk
            want = math.ceil(7 / max(1, c // wps)) if shared else math.ceil(7 * wps / c)
            assert want > 1, (hop, chunk)
            p, n = _chunked(eng, monkeypatch, chunk, run)
            assert n == want * n0, (hop, chunk, n, n0)
            assert _same(p, p0), (hop, chunk)


@pytest.mark.gpu
def test_crnn_default_shared_chunk_size(engine, wake_pcm):
    """The shipped CRNN at tc through `pipeline` over 1300 streams x 10 s at hop 2: two shared chunks of 1236 and 64
    streams (424 windows per stream, 524 288 windows per chunk at most).  The wake clip is spliced into streams 1236 (the
    first of the second chunk) and 1299 (the last).  Streams 0, 1235, 1236 and 1299 equal float64 and equal the same
    four streams run as their own batch bit for bit."""
    import torch
    from wakeword_detection_b200 import synth
    eng = engine("crnn", "tc")
    w = weights("crnn")
    S, N = 1300, 160000
    pcm = synth.device_pcm(S, N, 21, eng.device)
    clip = torch.from_numpy(wake_pcm["crnn"]).to(eng.device)
    for s, off in ((1236, 40000), (1299, 100000)):
        pcm[s, off:off + clip.numel()] = clip
    n0 = eng.launch_count()
    post = eng.pipeline(pcm, hop=2)
    n_big = eng.launch_count() - n0
    assert post.shape == (S, 424)
    pick = [0, 1235, 1236, 1299]
    n0 = eng.launch_count()
    alone = eng.pipeline(pcm[pick].contiguous(), hop=2)
    n_small = eng.launch_count() - n0
    assert n_big - n_small == shared_launches(151), (n_big, n_small)   # exactly one more chunk
    assert _same(post[pick], alone)
    host = pcm[pick].cpu().numpy()
    got = post[pick].cpu().numpy()
    j = np.arange(0, 424, 3)
    worst = max(_check_vs_float64(got[i, j], _oracle_posteriors(host[i], w, 2, 0.0, j), pick[i]) for i in range(4))
    assert got[2].max() > 0.9 and got[3].max() > 0.9
    STATS.append("1300 x 10 s shipped CRNN tc: max |err| vs float64 %.2e on streams %s" % (worst, pick))


# ------------------------------------------------------------------------------------ B. host pipeline
# (model, S, N, PCM dtype, pre-emphasis, hop); S >= 64 is cut into three slices of S/8, 2 (S/8) and the rest
GEOMETRY = [
    ("crnn", 1, 64000, "int16", 0.0, 2),
    ("wavenet", 7, 48123, "float32", 0.97, 1),
    ("crnn97", 63, 16037, "int16", 0.97, 1),
    ("crnn", 64, 40000, "float32", 0.0, 3),
    ("wavenet", 65, 36000, "int16", 0.0, 2),
    ("crnn", 71, 33117, "int16", 0.97, 2),
    ("wavenet", 71, 40000, "float32", 0.97, 3),
    ("crnn97", 64, 16037, "float32", 0.0, 2),
    ("crnn", 65, 511, "int16", 0.0, 2),
    ("wavenet", 7, 512, "float32", 0.97, 1),
    ("crnn", 7, 16037, "int16", 0.0, 1),
    ("crnn", 130, 64000, "float32", 0.0, 1),
]
FLOAT64_CASES = {3, 4}   # first stream of each slice against float64


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(GEOMETRY)))
def test_host_pipeline_geometry(case, engine):
    """wwb_pipeline_host (pageable buffers) and wwb_sweep_submit (page-locked buffers) equal the device-buffer
    wwb_pipeline bit for bit, over S = 1..130 streams (one slice below 64 streams, three above), 511, 512 and 16 037
    samples (no frame, one frame, fewer or barely more frames than the window), int16 and float32 PCM, pre-emphasis 0
    and 0.97, hops 1, 2 and 3"""
    from wakeword_detection_b200 import _cabi
    name, S, N, dtype, a, hop = GEOMETRY[case]
    eng = engine(name)
    w = weights(name)
    pcm = _pcm(S, N, dtype, 100 + case)
    want = eng.pipeline(pcm, hop=hop, pre_emphasis=a).cpu().numpy()
    nw = eng.num_windows(eng.num_frames(N), hop)
    assert want.shape == (S, nw)
    host = eng.pipeline_host(pcm, hop=hop, pre_emphasis=a)
    np.testing.assert_array_equal(host, want)
    pinned = _cabi.pinned_empty(pcm.shape, pcm.dtype)
    pinned[:] = pcm
    rec = eng.sweep_submit(pinned, hop, pre_emphasis=a)
    eng.sweep_wait()
    np.testing.assert_array_equal(rec["post"][0], want)
    if case in FLOAT64_CASES:
        assert S >= 64 and nw > 0
        j = np.arange(nw)
        for s in (0, S // 8, 3 * (S // 8)):
            _check_vs_float64(want[s], _oracle_posteriors(pcm[s], w, hop, a, j), (case, s))


def _far_oracle(post, thr):
    """FAR counts of every stream as one trajectory: R.smooth_same and R.rising_edges"""
    sm = [R.smooth_same(p.astype(F64)) for p in post]
    return np.array([sum(R.rising_edges(x, t) for x in sm) for t in thr], np.int64), sm


def _frr_oracle(post, thr):
    m = post.max(axis=1).astype(F64)
    return np.array([int((m > t).sum()) for t in thr], np.int64)


def _margin(smoothed, thr):
    """least distance of a smoothed value to a threshold: the kernel sums the 30 taps in sequence and numpy does not,
    so the two may differ in the last bit; an exact count comparison needs every value clear of every threshold"""
    thr = np.sort(thr)
    x = np.concatenate([np.ravel(s) for s in smoothed])
    i = np.searchsorted(thr, x)
    lo, hi = thr[np.clip(i - 1, 0, thr.size - 1)], thr[np.clip(i, 0, thr.size - 1)]
    return float(min(np.abs(x - lo).min(), np.abs(x - hi).min()))


def _check_counts(rec, m, post, thr, what):
    far, sm = _far_oracle(post, thr)
    gap = _margin(sm, thr)
    STATS.append("%s: least |smoothed - threshold| %.3e" % (what, gap))
    assert gap > 1e-12, (what, gap)
    np.testing.assert_array_equal(rec["far"][m], far)
    np.testing.assert_array_equal(rec["frr"][m], _frr_oracle(post, thr))


def _sweep_pcm(S, N, seed):
    pcm = _pcm(S, N, "int16", seed)
    for s in range(0, S, 9):
        clip = wake_clip("crnn" if s % 2 else "wavenet")
        off = (s * 997) % (N - clip.size)
        pcm[s, off:off + clip.size] = clip
    return pcm


@pytest.mark.gpu
def test_sweep_three_models_and_two_jobs_in_flight(engine):
    """The shipped CRNN, the shipped WaveNet and the L = 97 CRNN in one sweep over 130 x 64 000 samples (124, 108 and 151
    windows per stream): posteriors equal wwb_pipeline bit for bit, and FAR / FRR counts equal the oracle's loops.  Then
    two jobs in flight with different S (130, then 90) and threshold grids (evaluate_models, then plot_eval_models):
    each job's results equal the same job run alone."""
    from wakeword_detection_b200 import _cabi
    names = ["crnn", "wavenet", "crnn97"]
    engs = [engine(n) for n in names]
    lead, others = engs[0], engs[1:]
    N = 64000
    jobs = []
    for S, seed, thr in ((130, 31, R.thresholds_eval()), (90, 32, R.thresholds_plot())):
        pcm = _cabi.pinned_empty((S, N), np.int16)
        pcm[:] = _sweep_pcm(S, N, seed)
        jobs.append((pcm, thr))
    alone = []
    for pcm, thr in jobs:
        alone.append(lead.sweep_submit(pcm, 2, thr, others=others))
        lead.sweep_wait()
    pcm, thr = jobs[0]
    nws = set()
    for m, e in enumerate(engs):
        post = e.pipeline(pcm, hop=2).cpu().numpy()
        nws.add(post.shape[1])
        np.testing.assert_array_equal(alone[0]["post"][m], post)
        _check_counts(alone[0], m, post, thr, "sweep %s" % names[m])
        assert alone[0]["frr"][m][0] > 0
    assert len(nws) == 3
    both = [lead.sweep_submit(p, 2, t, others=others) for p, t in jobs]
    lead.sweep_wait()
    lead.sweep_wait()
    for a, b in zip(alone, both):
        for k in ("post", "far", "frr"):
            for m in range(3):
                np.testing.assert_array_equal(a[k][m], b[k][m])


def _launches(engs):
    return [e.launch_count() for e in engs]


def _valid_job_after(crnn, wn, pcm, thr, what):
    """a valid two-model job submitted right after a refused one comes out correct"""
    rec = crnn.sweep_submit(pcm, 2, thr, others=[wn])
    crnn.sweep_wait()
    for m, e in enumerate((crnn, wn)):
        post = e.pipeline(pcm, hop=2).cpu().numpy()
        np.testing.assert_array_equal(rec["post"][m], post)
        _check_counts(rec, m, post, thr, "%s m=%d" % (what, m))


def _refused(engs, match, pcm, thr):
    """the sweep is refused with ValueError before any copy or launch: no ctx's launch count moves and no job is left
    in flight"""
    before = _launches(engs)
    with pytest.raises(ValueError, match=match):
        engs[0].sweep_submit(pcm, 2, thr, others=engs[1:])
    assert _launches(engs) == before
    with pytest.raises(IndexError):
        engs[0].sweep_wait()


@pytest.mark.gpu
def test_sweep_refuses_short_far_trajectory(engine):
    """FAR counts over trajectories of 1..29 posteriors (shorter than the 30-tap window) are refused before any work,
    for the first model of a sweep and for a later one"""
    crnn, wn, c97 = engine("crnn"), engine("wavenet"), engine("crnn97")
    thr = R.thresholds_eval()
    # 169 frames: 10 windows of the shipped CRNN at hop 2, 37 of the L = 97 CRNN
    short = _pcm(5, 512 + 160 * 168, "int16", 41)
    for engs in ([crnn], [c97, crnn]):
        assert [e.num_windows(169, 2) for e in engs][-1] == 10
        _refused(engs, "shorter than the 30-tap", short, thr)
    _valid_job_after(crnn, wn, _pcm(70, 64000, "int16", 42), thr, "after a short trajectory")


@pytest.mark.gpu
def test_sweep_refuses_models_with_other_filters(engine):
    """One filter pass feeds every model of a sweep, so models whose filters differ in any one field (mel_w, mel_b,
    floor, offset, scale) are refused before any work"""
    from wakeword_detection_b200 import _cabi
    crnn, wn = engine("crnn"), engine("wavenet")
    thr = R.thresholds_eval()
    base = weights("crnn")
    changed = {"mel_w": lambda v: v * np.float32(1.001), "mel_b": lambda v: v + np.float32(0.01),
               "mel_floor": lambda v: v * np.float32(2), "mel_log_offset": lambda v: v + np.float32(0.5),
               "mel_scale": lambda v: v * np.float32(1.01)}
    pcm = _pcm(70, 64000, "int16", 43)
    for key, f in changed.items():
        w = dict(base)
        w[key] = np.asarray(f(np.asarray(base[key], np.float32)), np.float32)
        other = _cabi.Engine(w, 0, "tc")
        try:
            _refused([crnn, other], "filter fields", pcm, thr)
        finally:
            other.close()
    _valid_job_after(crnn, wn, pcm, thr, "after other filters")


@pytest.mark.gpu
def test_sweep_refuses_unsorted_thresholds(engine):
    crnn, wn = engine("crnn"), engine("wavenet")
    thr = R.thresholds_eval()
    pcm = _pcm(70, 64000, "int16", 44)
    _refused([crnn, wn], "ascending", pcm, thr[::-1].copy())
    _valid_job_after(crnn, wn, pcm, thr, "after unsorted thresholds")


def _page_locked(arr):
    """whether the driver takes the start of `arr` for page-locked host memory (CU_POINTER_ATTRIBUTE_MEMORY_TYPE is
    CU_MEMORYTYPE_HOST; pageable memory is unknown to the driver and the query fails)"""
    cuda = ctypes.CDLL("libcuda.so.1")
    cuda.cuPointerGetAttribute.argtypes = [ctypes.POINTER(ctypes.c_uint), ctypes.c_int, ctypes.c_uint64]
    t = ctypes.c_uint(0)
    rc = cuda.cuPointerGetAttribute(ctypes.byref(t), 2, ctypes.c_uint64(arr.ctypes.data))
    return rc == 0 and t.value == 1


@pytest.mark.gpu
def test_caller_buffers_not_left_page_locked(engine):
    """After wwb_pipeline_host returns, and after wwb_sweep_wait returns, none of the caller's pageable buffers is still
    page-locked: CUDA requires page-locked memory to be unregistered before it is freed, and a later buffer at the same
    address would be taken as registered.  Memory from wwb_host_alloc reads as page-locked (the query works)."""
    from wakeword_detection_b200 import _cabi
    crnn, wn = engine("crnn"), engine("wavenet")
    assert _page_locked(_cabi.pinned_empty((1024,), np.float32))
    pcm = _pcm(80, 64000, "int16", 51)                      # 10 MB in, 79 KB / 69 KB of posteriors out per model
    out = np.empty((80, crnn.num_windows(crnn.num_frames(64000), 1)), np.float32)
    assert out.nbytes >= 1 << 16
    crnn.pipeline_host(pcm, hop=1, out=out)
    assert not _page_locked(pcm) and not _page_locked(out)
    np.testing.assert_array_equal(out, crnn.pipeline(pcm, hop=1).cpu().numpy())
    rec = {k: [None, None] for k in ("post", "far", "frr")}
    rec["post"] = [np.empty((80, e.num_windows(e.num_frames(64000), 1)), np.float32) for e in (crnn, wn)]
    crnn.sweep_submit(pcm, 1, R.thresholds_eval(), others=[wn], out=rec)
    crnn.sweep_wait()
    for a in [pcm] + rec["post"] + rec["far"] + rec["frr"]:
        assert not _page_locked(a)
    for m, e in enumerate((crnn, wn)):
        np.testing.assert_array_equal(rec["post"][m], e.pipeline(pcm, hop=1).cpu().numpy())


# ------------------------------------------------------------------------------------ C. counters at length
N_FAR = 1_000_003


def _trajectory():
    """a clipped random walk (AR(1), mean 0.5) with saturated stretches of exactly 0.0 and 1.0"""
    from scipy.signal import lfilter
    r = np.random.default_rng(7)
    x = 0.5 + lfilter([0.045], [1, -0.999], r.standard_normal(N_FAR))
    p = np.clip(x, 0.0, 1.0).astype(np.float32)
    assert (p == 0).mean() > 0.02 and (p == 1).mean() > 0.02
    return p


def _grid_8192():
    return np.linspace(0.0001, 0.9999, 8192)


def _edges_all(sm, thr):
    """rising edges of (sm > t) for every t at once: position i rises for exactly the thresholds prev <= t < sm[i]"""
    prev = np.concatenate([[-np.inf], sm[:-1]])
    up = prev < sm
    a, b = np.sort(prev[up]), np.sort(sm[up])
    return (np.searchsorted(a, thr, "right") - np.searchsorted(b, thr, "right")).astype(np.int64)


@pytest.mark.gpu
def test_far_counts_at_evaluation_length(engine):
    """FAR edges of one trajectory of 1 000 003 posteriors (four grid-stride passes of the kernel) against R.smooth_same
    and R.rising_edges, for the evaluate_models grid, the plot_eval_models grid and 8192 thresholds (the maximum; 8193
    are refused).  The same trajectory as 2..8 time chunks with halos (dist.time_chunks) adds up to the whole."""
    from wakeword_detection_b200 import dist
    eng = engine("crnn")
    p = _trajectory()
    sm = R.smooth_same(p.astype(F64))
    grids = {"eval": R.thresholds_eval(), "plot": R.thresholds_plot(), "8192": _grid_8192()}
    whole = {}
    for k, thr in grids.items():
        gap = _margin([sm], thr)
        STATS.append("FAR %d posteriors, %s grid: least |smoothed - threshold| %.3e" % (N_FAR, k, gap))
        assert gap > 1e-12, (k, gap)
        got = eng.eval_counts(p, [0, N_FAR], thr, "far_edges").cpu().numpy()
        want = _edges_all(sm, thr)
        idx = range(thr.size) if thr.size < 1000 else range(0, thr.size, 61)
        assert [R.rising_edges(sm, thr[i]) for i in idx] == [int(want[i]) for i in idx]
        np.testing.assert_array_equal(got, want)
        assert want.min() > 0
        whole[k] = got
    with pytest.raises(ValueError, match="n_thr"):
        eng.eval_counts(p, [0, N_FAR], np.linspace(0.0001, 0.9999, 8193), "far_edges")
    for world in range(2, 9):
        for k, thr in grids.items():
            total = np.zeros(thr.size, np.int64)
            for b, e, lo, hi in dist.time_chunks(N_FAR, world):
                part = p[b - lo:e + hi]
                total += eng.eval_counts(part, [0, part.size], thr, "far_edges", halo_lo=[lo], halo_hi=[hi]).cpu().numpy()
            np.testing.assert_array_equal(total, whole[k], err_msg="world %d %s" % (world, k))


@pytest.mark.gpu
def test_frr_counts_many_segments(engine):
    """FRR over 100 003 segments of 1..20 posteriors against max > t, for the evaluate_models grid and a grid of
    float32 values; one segment in eight has its maximum exactly on a threshold, which does not count"""
    eng = engine("crnn")
    r = np.random.default_rng(8)
    lens = r.integers(1, 21, 100_003)
    seg = np.concatenate([[0], np.cumsum(lens)])
    p = r.random(int(seg[-1])).astype(np.float32)
    f32_grid = np.unique(np.linspace(0.3, 0.99, 2000).astype(np.float32)).astype(F64)
    for thr in (R.thresholds_eval(), f32_grid):
        exact = thr[np.float32(thr).astype(F64) == thr]
        q = p.copy()
        hit = r.random(lens.size) < 0.125
        for i in np.nonzero(hit)[0]:
            v = np.float32(exact[r.integers(exact.size)])
            a, b = seg[i], seg[i + 1]
            q[a:b] = np.minimum(q[a:b], v)
            q[a + r.integers(b - a)] = v
        m = np.maximum.reduceat(q, seg[:-1]).astype(F64)
        assert np.isin(m, thr).sum() >= hit.sum()
        want = np.array([int((m > t).sum()) for t in thr], np.int64)
        got = eng.eval_counts(q, seg, thr, "frr_max").cpu().numpy()
        np.testing.assert_array_equal(got, want)
