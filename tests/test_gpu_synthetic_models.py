"""The kernels against the oracle in float64 on synthetic models: weight layouts, window lengths, dilation schedules,
BatchNorm scales and filter fields the shipped models never exercise.

The shipped weights hide several classes of bug: their GRU input and recurrent biases are equal on the z and r gates,
mel_b is zero and every mel row is one contiguous triangle, the WaveNet runs one dilation schedule at one window length
with BatchNorm scales in [3.9, 69.5].  The models here are drawn from a seeded generator in the layout
weights.load_model_dir returns, each tensor at the per-tensor std of a shipped model, with knobs for what the shipped
weights fix.  The truth is the oracle in float64 (oracle.restated, dtype=np.float64); every comparison also records the
float32 oracle's own error, so each tolerance can be read against what fp32 arithmetic achieves.

Tolerances as in test_gpu_parity.py: encoder output, detect output and posteriors 1e-3 absolute (2e-2 for tc_fast),
decisions exact outside the band around the threshold.  The sensitivity and scale-invariance tests run without a GPU.
"""
import os

import numpy as np
import pytest

from conftest import load_weights
from oracle import restated as R
from streaming_helpers import CHUNKS, MAX_CHUNK, Push, Schedule, assert_same_rows, check_mel, host, stream_pcm
from wakeword_detection_b200 import synth

F64 = np.float64
POST_ATOL = 1e-3
FAST_ATOL = 2e-2
FILTER_KEYS = ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")
SHIPPED_DIL = np.tile(np.array([1, 2, 4, 8], np.int32), 6)
DILATIONS = {
    "shipped": SHIPPED_DIL,
    "reversed": np.tile(np.array([8, 4, 2, 1], np.int32), 6),
    "ones": np.ones(24, np.int32),
    "eights": np.full(24, 8, np.int32),           # D(23) = 384: more than any window
    "drawn": np.random.default_rng(11).permutation(np.concatenate([[3, 5, 6, 7], np.random.default_rng(12).integers(1, 9, 20)])).astype(np.int32),
}
SCALES = [2.0 ** k for k in range(-12, 13, 2)]
STATS = []


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for line in STATS:
        print("\n[synthetic] " + line)


# ------------------------------------------------------------------------------------ the generator
def _std(ref):
    return {k: float(np.std(v)) for k, v in ref.items() if isinstance(v, np.ndarray) and v.dtype == np.float32 and v.ndim}


_REF_STD = {}


def _ref_std(kind):
    if kind not in _REF_STD:
        _REF_STD[kind] = _std(load_weights("CRNN_arik_original" if kind == "crnn" else "Wavenet"))
    return _REF_STD[kind]


def synth_filter(seed=0, rows=False, bias=False, consts=False):
    """the shipped filter, or with `rows`: mel rows with gaps, runs longer than the 8-tap segments, a dense 257-bin
    row, an all-zero row and negative entries; `bias`: non-zero mel_b with one band pushed below the floor; `consts`:
    a non-default floor, log offset and scale.  The rows come to 125 segments (runs of up to 8 consecutive non-zero
    bins) of the 128 the filter kernels hold"""
    base = load_weights("CRNN")
    f = {k: np.array(base[k], copy=True) for k in FILTER_KEYS}
    r = np.random.default_rng(seed)
    mw = f["mel_w"]
    peak = float(mw.max())
    if rows:
        mw[3] = 0.0                                                       # all-zero row
        mw[7] = r.uniform(0.05, 1.0, 257).astype(np.float32) * peak * 0.2  # dense
        mw[12] = 0.0
        mw[12, 40:56:2] = peak * r.uniform(0.3, 1.0, 8)                   # every other bin: 8 one-tap segments
        mw[12, 90:93] = peak
        mw[20, 100:131] = peak * r.uniform(0.3, 1.0, 31)                  # a run of 31 bins: 4 segments
        mw[25, 150:170] = peak * np.linspace(1.0, 0.1, 20)                # overlaps the triangle already there
        neg = np.nonzero(mw[30])[0]
        mw[30, neg[::3]] *= -0.25                                         # negative entries inside a triangle
        gap = np.nonzero(mw[31])[0]
        mw[31, gap[len(gap) // 2 - 1: len(gap) // 2 + 1]] = 0.0           # a triangle with a gap
    if bias:
        f["mel_b"] = r.uniform(1e-3, 2e-2, 40).astype(np.float32)
        f["mel_b"][5] = -1e4                                              # below the floor in every frame
    if consts:
        f["mel_floor"] = np.float32(3e-5)
        f["mel_log_offset"] = np.float32(-9.25)
        f["mel_scale"] = np.float32(0.37)
    return f


def synth_model(kind, seed, n_out=2, dilation="shipped", L=182, bn="shipped", filt=None):
    """A model of `kind` ("crnn" | "wavenet") in the layout of weights.load_model_dir.  Every tensor is drawn at the
    per-tensor std of a shipped model, so the GRU biases differ on all three gates and det2_b and the gate biases are
    non-zero.  bn: "shipped" draws the BatchNorm scales from the shipped range [3.9, 69.5]; "mixed" makes a third of
    them negative and a sixth of them smaller than 1.  det2 is still to be calibrated (calibrate)."""
    r = np.random.default_rng(1000 * seed + (7 if kind == "crnn" else 13))
    sd = _ref_std(kind)
    ref = load_weights("CRNN_arik_original" if kind == "crnn" else "Wavenet")
    w = dict(filt if filt is not None else synth_filter())

    def draw(k, shape=None):
        return (r.standard_normal(ref[k].shape if shape is None else shape) * sd[k]).astype(np.float32)

    for k, v in ref.items():
        if k in FILTER_KEYS or not isinstance(v, np.ndarray) or v.dtype != np.float32:
            continue
        w[k] = draw(k)
    w["det2_w"] = draw("det2_w", (n_out, ref["det2_w"].shape[1]))
    w["det2_b"] = draw("det2_b", (n_out,))
    if kind == "crnn":
        w["mel_length"] = np.int32(151)
        return w
    w["mel_length"] = np.int32(L)
    w["dilation"] = np.array(DILATIONS[dilation] if isinstance(dilation, str) else dilation, np.int32)
    w["bn_mul"] = r.uniform(3.9, 69.5, (24, 16)).astype(np.float32)
    if bn == "mixed":
        m = w["bn_mul"].reshape(-1)
        idx = r.permutation(m.size)
        m[idx[: m.size // 3]] *= -1
        m[idx[m.size // 3: m.size // 2]] = r.uniform(0.05, 0.9, m.size // 2 - m.size // 3) * np.sign(m[idx[m.size // 3: m.size // 2]])
    return w


def mel_windows(L, n=16, filt=None):
    """n mel windows of length L from seeded synthetic audio of every class, plus an all-zero window"""
    f = filt if filt is not None else synth_filter()
    mels = [R.mel_stream(np.clip(synth.stream_float(16000 * 3, c, 5, c), -1, 1).astype(np.float32), f)
            for c in range(synth.N_CLASSES)]
    step = max(1, (mels[0].shape[0] - L) // 4)
    wins = [m[j:j + L] for m in mels for j in range(0, m.shape[0] - L, step)]
    idx = np.random.default_rng(L).permutation(len(wins))[: n - 1]
    return np.concatenate([np.stack([wins[i] for i in sorted(idx)]), np.zeros((1, L, 40), np.float32)]).astype(np.float32)


def calibrate(w, X):
    """Scale det2 so that the float64 posteriors of the windows X spread over (0, 1): the wake logit (the logit
    difference for a softmax head, a max over time for the WaveNet head) is linear in a positive scale of det2_w, so
    it is set to an inter-quartile range of 3 centred on 0.  det2_b stays non-zero.  Returns w."""
    w = dict(w)
    b0 = w["det2_b"].copy()
    w["det2_b"] = np.zeros_like(b0)
    w["det2_w"] = (w["det2_w"] * np.float32(1e-3)).astype(np.float32)   # no saturation while measuring
    p = R.posterior(X, w, F64)
    p = np.clip(p, 1e-300, 1 - 1e-16)
    d = np.log(p) - np.log1p(-p)
    iqr = float(np.percentile(d, 75) - np.percentile(d, 25))
    g = 3.0 / max(iqr, 1e-30)
    w["det2_w"] = (w["det2_w"] * g).astype(np.float32)
    med = float(np.median(d)) * g
    if w["det2_w"].shape[0] == 1:
        w["det2_b"] = np.array([-med], np.float32)
    else:
        w["det2_b"] = np.array([b0[0], b0[0] - med], np.float32)
    return w


_MODELS = {}


def model(kind, seed=0, n_out=2, dilation="shipped", L=182, bn="shipped"):
    """(weights, windows, float64 encoder / detect / posteriors, float32 oracle's encoder / posteriors), cached"""
    key = (kind, seed, n_out, dilation, L, bn)
    if key not in _MODELS:
        L = 151 if kind == "crnn" else L
        X = mel_windows(L)
        w = calibrate(synth_model(kind, seed, n_out, dilation, L, bn), X)
        enc = R.encode(X, w, F64)
        det = R.detect(enc, w, F64)
        ref = det[:, -1]
        assert np.all(w["det2_b"] != 0)
        assert np.mean((ref >= 0.05) & (ref <= 0.95)) >= 0.5, "posteriors saturated: %s" % np.round(ref, 3)
        enc32 = R.encode(X, w)
        _MODELS[key] = (w, X, enc, det, ref, enc32, R.detect(enc32, w)[:, -1])
    return _MODELS[key]


def family(w, s):
    """the equivalence family of w at scale s (same float64 posteriors for every s > 0).  WaveNet: in_w, in_b, res_w
    and res_b times s, bn_mul / s (the residual stream x scales by s, u = bn_mul * x + bn_add does not).  CRNN: conv_w
    and conv_b times s, the layer-1 GRU input weights / s (ReLU is positively homogeneous; the GRU biases stay)."""
    w = dict(w)
    s32 = np.float32(s)
    if R.is_crnn(w):
        up, down = ("conv_w", "conv_b"), ("gru1_f_w", "gru1_b_w")
    else:
        up, down = ("in_w", "in_b", "res_w", "res_b"), ("bn_mul",)
    for k in up:
        w[k] = (w[k] * s32).astype(np.float32)
    for k in down:
        w[k] = (w[k] / s32).astype(np.float32)
    return w


# ------------------------------------------------------------------------------------ CPU: the tests below can see bugs
def _swap(a, i, j, axis):
    a = np.array(a, copy=True)
    idx_i = [slice(None)] * a.ndim
    idx_j = [slice(None)] * a.ndim
    idx_i[axis], idx_j[axis] = i, j
    a[tuple(idx_i)], a[tuple(idx_j)] = a[tuple(idx_j)].copy(), a[tuple(idx_i)].copy()
    return a


def _mutants(w):
    """the classic mistakes, one at a time.  A swap of bi and br on the z and r gates is not among them: only their sum
    enters those gates, so it is the identity.  Using one bias twice there is not, and neither is the swap on the
    candidate gate, where br sits inside r * (U h + br)."""
    m = {}
    if R.is_crnn(w):
        g = dict(w)
        for k in ("gru1_f", "gru1_b", "gru2_f", "gru2_b"):
            br = g[k + "_br"].copy()
            br[:64] = g[k + "_bi"][:64]
            g[k + "_br"] = br
        m["gru bi used twice on z/r"] = g
        g = dict(w)
        for k in ("gru1_f", "gru1_b", "gru2_f", "gru2_b"):
            bi, br = g[k + "_bi"].copy(), g[k + "_br"].copy()
            bi[64:], br[64:] = g[k + "_br"][64:], g[k + "_bi"][64:]
            g[k + "_bi"], g[k + "_br"] = bi, br
        m["gru bi/br swapped on the candidate gate"] = g
        g = dict(w)
        for k in ("gru1_f", "gru1_b", "gru2_f", "gru2_b"):
            g[k + "_u"] = np.ascontiguousarray(g[k + "_u"].reshape(3, 32, 32).transpose(0, 2, 1).reshape(96, 32))
        m["U transposed per gate"] = g
        m["conv time taps reversed"] = dict(w, conv_w=np.ascontiguousarray(w["conv_w"][:, :, ::-1]))
    else:
        m["taps 0 and 2 swapped"] = dict(w, sig_w=_swap(w["sig_w"], 0, 2, 2), tanh_w=_swap(w["tanh_w"], 0, 2, 2))
        m["tanh and sigmoid swapped"] = dict(w, sig_w=w["tanh_w"], tanh_w=w["sig_w"], sig_b=w["tanh_b"], tanh_b=w["sig_b"])
        d = w["dilation"].copy()
        d[5] += 1 if d[5] < 8 else -1
        m["one dilation off by one"] = dict(w, dilation=d)
    return m


SENS_FAMILIES = [("crnn", 1, "shipped", 182), ("crnn", 2, "shipped", 182), ("wavenet", 2, "shipped", 182),
                 ("wavenet", 2, "drawn", 182), ("wavenet", 2, "reversed", 64), ("wavenet", 2, "shipped", 17)]


@pytest.mark.parametrize("kind,n_out,dil,L", SENS_FAMILIES)
def test_mistakes_move_the_reference(kind, n_out, dil, L):
    """Each classic mistake moves the float64 posteriors of the test windows by at least 1e-2, so the device tests,
    which hold the kernels to 1e-3, would catch it.  Dropping mel_b is checked through the filter: the windows are
    computed from the same audio with and without it."""
    w, X, _, _, ref, _, _ = model(kind, 0, n_out, dil, L)
    for name, mw in _mutants(w).items():
        moved = float(np.abs(R.posterior(X, mw, F64) - ref).max())
        assert moved >= 1e-2, (name, moved)
    fb = synth_filter(bias=True)
    Xb = mel_windows(int(w["mel_length"]), filt=fb)
    Xn = mel_windows(int(w["mel_length"]), filt=dict(fb, mel_b=np.zeros(40, np.float32)))
    moved = float(np.abs(R.posterior(Xb, w, F64) - R.posterior(Xn, w, F64)).max())
    assert moved >= 1e-2, ("mel_b dropped", moved)


@pytest.mark.parametrize("kind", ["crnn", "wavenet"])
def test_scale_family_is_exact_in_float64(kind):
    """The scale families the device test runs: the float64 posteriors are the same to 1e-6 for every s = 2^k."""
    w, X, _, _, ref, _, _ = model(kind)
    for s in SCALES:
        assert np.abs(R.posterior(X, family(w, s), F64) - ref).max() < 1e-6, s


def test_float64_oracle_keeps_the_float32_default(w_crnn, w_wavenet):
    """dtype=float64 is a separate arithmetic; the default is still float32 throughout"""
    X = mel_windows(182, n=3)
    for w, x in ((w_crnn, X[:, :151]), (w_wavenet, X)):
        assert R.encode(x, w).dtype == np.float32 and R.posterior(x, w).dtype == np.float32
        p64 = R.posterior(x, w, F64)
        assert p64.dtype == np.float64 and np.abs(p64 - R.posterior(x, w)).max() < 1e-4


# ------------------------------------------------------------------------------------ GPU
def _engine(w, precision):
    from wakeword_detection_b200 import _cabi
    return _cabi.Engine(w, 0, precision)


def _np(t):
    return t.cpu().numpy()


def _err(a, b):
    return float(np.abs(np.asarray(a, F64) - np.asarray(b, F64)).max())


def _check_model(tag, w, X, enc64, det64, ref, enc32, post32, precision):
    """encoder output, detect output (on the kernel's and on the reference's encoder output) and posteriors against
    float64; decisions outside the band; the fp32 oracle's error recorded beside the kernel's"""
    tol = FAST_ATOL if precision == "tc_fast" else POST_ATOL
    eng = _engine(w, precision)
    try:
        enc_t = eng.encode(X)
        enc = _np(enc_t)
        det = _np(eng.detect(enc_t))
        det_ref = _np(eng.detect(enc64.astype(np.float32)))
        post = _np(eng.posteriors(X, hop=1))[:, 0]
    finally:
        eng.close()
    e_enc, e_det, e_det2, e_post = _err(enc, enc64), _err(det, det64), _err(det_ref, det64), _err(post, ref)
    STATS.append("%s %s: enc %.2e (fp32 oracle %.2e), detect %.2e / on the reference's enc %.2e, post %.2e (fp32 oracle %.2e)"
                 % (tag, precision, e_enc, _err(enc32, enc64), e_det, e_det2, e_post, _err(post32, ref)))
    assert det.shape == det64.shape
    assert np.isfinite(post).all()
    assert e_enc < tol and e_det < tol and e_det2 < tol and e_post < tol, (e_enc, e_det, e_det2, e_post)
    if precision != "tc_fast":
        band = np.abs(ref - 0.5) <= POST_ATOL
        assert np.array_equal((post > 0.5)[~band], (ref > 0.5)[~band])
    return post


def _no_share(var, eng, X, hop):
    os.environ[var] = "1"
    try:
        return eng.posteriors(X, hop=hop).clone()
    finally:
        os.environ[var] = "0"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "tc", "tc_fast"])
@pytest.mark.parametrize("n_out", [1, 2])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_crnn_vs_float64(seed, n_out, precision):
    w, X, enc64, det64, ref, enc32, post32 = model("crnn", seed, n_out)
    _check_model("CRNN seed %d n_out %d" % (seed, n_out), w, X, enc64, det64, ref, enc32, post32, precision)


@pytest.mark.gpu
@pytest.mark.parametrize("n_out", [1, 2])
def test_crnn_shared_columns_bit_identical(n_out):
    """sliding windows (hop 1 and 2) on the tensor cores: the shared-column path equals the per-window tiles bit for bit"""
    import torch
    w = model("crnn", 1, n_out)[0]
    tc, f32 = _engine(w, "tc"), _engine(w, "f32")
    torch.manual_seed(n_out)
    X = torch.rand((2, 411, 40), device=tc.device) * 5
    for hop in (1, 2):
        a = _no_share("WWB_CRNN_NO_SHARE", tc, X, hop)
        b = tc.posteriors(X, hop=hop).clone()
        assert bool((a == b).all())
        assert float((b - f32.posteriors(X, hop=hop)).abs().max()) < POST_ATOL


WN_CONFIGS = [("shipped", 182, "shipped"), ("reversed", 182, "shipped"), ("ones", 182, "shipped"),
              ("eights", 182, "shipped"), ("drawn", 182, "shipped"), ("shipped", 17, "shipped"),
              ("shipped", 32, "shipped"), ("shipped", 100, "shipped"), ("shipped", 181, "shipped"),
              ("drawn", 64, "shipped"), ("shipped", 182, "mixed")]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "tc"])
@pytest.mark.parametrize("dil,L,bn", WN_CONFIGS)
def test_wavenet_vs_float64(dil, L, bn, precision):
    """Dilation schedules, window lengths and BatchNorm scales: encoder, detect and posteriors within 1e-3 of float64;
    ragged groups of 1..9 windows equal the full batch bit for bit"""
    w, X, enc64, det64, ref, enc32, post32 = model("wavenet", 0, 2, dil, L, bn)
    full = _check_model("WaveNet %s L=%d bn=%s" % (dil, L, bn), w, X, enc64, det64, ref, enc32, post32, precision)
    eng = _engine(w, precision)
    try:
        for n in range(1, 10):
            assert np.array_equal(_np(eng.posteriors(X[:n], hop=1))[:, 0], full[:n]), n
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dil,L,bn", WN_CONFIGS)
def test_wavenet_shared_activations_bit_identical(dil, L, bn):
    """Sliding windows (hop 1 and 2; F = 1101 and 1561 cross the stream pass's chunk boundaries): the shared-activation
    path equals WWB_WN_NO_SHARE=1 bit for bit, for every schedule and length, and agrees with the fp32 path"""
    import torch
    w = model("wavenet", 0, 2, dil, L, bn)[0]
    tc, f32 = _engine(w, "tc"), _engine(w, "f32")
    try:
        for F, hop in ((1101, 1), (1561, 2)):
            torch.manual_seed(F + L)
            X = torch.rand((2, F, 40), device=tc.device) * 5
            a = _no_share("WWB_WN_NO_SHARE", tc, X, hop)
            b = tc.posteriors(X, hop=hop).clone()
            assert a.shape == (2, (F - L) // hop + 1)
            assert bool((a == b).all()), (F, hop)
            assert float((b - f32.posteriors(X, hop=hop)).abs().max()) < POST_ATOL
    finally:
        tc.close()
        f32.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["crnn", "wavenet"])
def test_scale_family(kind):
    """Every member s = 2^k (k = -12..12, step 2) of the model's equivalence family: f32 and tc within 1e-3 of float64
    and finite.  Both paths rescale the weights by a power of two when they load them (api.cu), so every member runs
    on the same weights: its posteriors are bit-identical to the s = 1 member's"""
    w, X, _, _, ref, _, _ = model(kind)
    first = {}
    for s in SCALES:
        errs = []
        for precision in ("f32", "tc"):
            eng = _engine(family(w, s), precision)
            try:
                post = _np(eng.posteriors(X, hop=1))[:, 0]
            finally:
                eng.close()
            assert np.isfinite(post).all(), (s, precision)
            errs.append(_err(post, ref))
            assert errs[-1] < POST_ATOL, (s, precision, errs[-1])
            if precision in first:
                assert np.array_equal(post, first[precision]), (s, precision)
            first.setdefault(precision, post)
        p32 = R.posterior(X, family(w, s))
        STATS.append("%s scale family s=2^%d: f32 %.2e, tc %.2e (fp32 oracle %.2e)"
                     % (kind, int(np.log2(s)), errs[0], errs[1], _err(p32, ref)))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,bias,consts", [(True, False, False), (False, True, False), (False, False, True),
                                              (True, True, True)])
def test_filter_fields(rows, bias, consts):
    """Synthetic filter fields through eng.filter (int16 and float PCM, pre-emphasis 0 and 0.97, ragged lengths) and
    eng.mel_from_magnitude, against the float64 mel of the reference's magnitudes"""
    f = synth_filter(3, rows, bias, consts)
    eng = _engine(f, "f32")
    worst = worst32 = 0.0
    try:
        for n in (512, 671, 3001, 16000 + 37):
            pcm = synth.batch_int16(3, n, seed=n)
            xf = np.stack([np.clip(synth.stream_float(n, c, 9, c), -1, 1) for c in (0, 2, 5)]).astype(np.float32)
            for src, x in (("int16", pcm), ("float", xf)):
                for a in (0.0, 0.97):
                    mel = _np(eng.filter(x, a))
                    for i in range(3):
                        xi = R.int16_to_float(x[i]) if src == "int16" else x[i]
                        y = R.pre_emphasis(xi, a)
                        nf = R.num_frames(y.shape[0])
                        frames = y[np.arange(nf)[:, None] * R.HOP + np.arange(R.FFT)[None, :]]
                        mag = R.stft_magnitude(frames)
                        ref = R.mel_from_magnitude(mag, f, F64)
                        worst = max(worst, check_mel(mel[i], ref))
                        worst32 = max(worst32, _err(R.mel_from_magnitude(mag, f), ref))
        rng = np.random.default_rng(4)
        mag = (rng.random((65, 257)) * 4).astype(np.float32)
        mag[0] = 0
        mag[1, ::2] = 0
        got = _np(eng.mel_from_magnitude(mag))
        ref = R.mel_from_magnitude(mag, f, F64)
        worst = max(worst, check_mel(got, ref))
    finally:
        eng.close()
    STATS.append("filter rows=%d bias=%d consts=%d: max |mel err| %.2e (fp32 oracle %.2e)" % (rows, bias, consts, worst, worst32))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "tc"])
def test_streaming_synthetic_wavenet(precision):
    """A 64-frame WaveNet with the reversed dilation schedule through stream_push in ragged chunks against
    TriggerOracle; its state record is 48 + 2048 + 160 * 64 bytes, and an export / import round trip into another
    context continues bit-exact"""
    from wakeword_detection_b200 import _cabi
    w = model("wavenet", 0, 2, "reversed", 64)[0]
    cap, thr = 4, 0.5
    ns = list(CHUNKS) * 2
    pcm = stream_pcm(cap, sum(ns) + 1, 3)
    sch = Schedule("synthetic", cap, MAX_CHUNK, 0.0, pcm,
                   [Push(n, cap - (i % 3 == 2), np.ones(cap), np.zeros(cap), thr) for i, n in enumerate(ns)])
    orc = [R.TriggerOracle(w, thr, 0.0) for _ in range(cap)]
    eng = _cabi.Engine(w, 0, precision)
    eng.stream_alloc(cap, MAX_CHUNK)
    assert eng.stream_state_bytes() == 48 + 2048 + 160 * 64

    def push(e, i):
        p = sch.pushes[i]
        S = p.n_streams
        return host(e.stream_push(sch.chunks[i], p.speech[:S].astype(np.uint8), p.active[:S].astype(np.uint8), 0.0, thr))

    outs, worst, n_win = [], 0.0, 0
    for i, p in enumerate(sch.pushes):
        post, npost, trig, _ = out = push(eng, i)
        outs.append(out)
        for s in range(p.n_streams):
            o = orc[s]
            o.active = False
            before = len(o.posteriors)
            o(sch.chunks[i][s], True)
            new = np.array(o.posteriors[before:], np.float32)
            assert npost[s] == new.size, (i, s)
            if new.size:
                err = _err(post[s, :new.size], new)
                assert err <= POST_ATOL, (i, s, err)
                worst, n_win = max(worst, err), n_win + new.size
                if np.abs(new - thr).min() > POST_ATOL:
                    assert bool(trig[s]) == bool((new > thr).any()), (i, s)
    assert n_win > 100
    STATS.append("stream WaveNet L=64 reversed %s: %d windows, max |err| vs TriggerOracle %.2e" % (precision, n_win, worst))
    # export after push 12, import into a fresh context, continue both
    half = 13
    eng2 = _cabi.Engine(w, 0, precision)
    eng2.stream_alloc(cap, MAX_CHUNK)
    eng3 = _cabi.Engine(w, 0, precision)
    eng3.stream_alloc(cap, MAX_CHUNK)
    for i in range(half):
        push(eng2, i)
    eng3.stream_import(np.arange(cap), eng2.stream_export(np.arange(cap)))
    assert_same_rows([push(eng3, i) for i in range(half, len(ns))], outs[half:])
    for e in (eng, eng2, eng3):
        e.close()


@pytest.mark.gpu
def test_rejections_and_precision_refusals():
    """A mel matrix of more than 128 segments and dilations 0 and 9 are refused.  A BatchNorm scale of 0 loads at f32 and matches float64, and is refused at tc and
    tc_fast by create and by set_precision; a refused set_precision leaves the ctx working at f32.  A padding row
    -bn_add / bn_mul outside fp16 is refused at tc the same way."""
    w, X, _, _, _, _, _ = model("wavenet")
    dense = synth_filter()
    dense["mel_w"][:4] = np.float32(1e-3)                  # 4 x 33 segments
    for f in (dense, dict(w, **dense)):
        with pytest.raises(ValueError, match="segments"):
            _engine(f, "f32")
    for d in (0, 9):
        dil = w["dilation"].copy()
        dil[7] = d
        with pytest.raises(ValueError, match="dilation"):
            _engine(dict(w, dilation=dil), "f32")
    zero = dict(w, bn_mul=w["bn_mul"].copy())
    zero["bn_mul"][6, 3] = 0.0
    big = dict(w, bn_mul=w["bn_mul"].copy(), bn_add=w["bn_add"].copy())
    big["bn_mul"][9, 2], big["bn_add"][9, 2] = 1e-3, 100.0          # -bn_add / bn_mul = -1e5
    for bad, why in ((zero, "BatchNorm scale of 0"), (big, "fp16 range")):
        ref = R.posterior(X, bad, F64)
        for precision in ("tc", "tc_fast"):
            with pytest.raises(ValueError, match=why):
                _engine(bad, precision)
        eng = _engine(bad, "f32")
        try:
            before = _np(eng.posteriors(X, hop=1))[:, 0]
            assert _err(before, ref) < POST_ATOL
            for precision in ("tc", "tc_fast"):
                with pytest.raises(ValueError, match=why):
                    eng.set_precision(precision)
            assert np.array_equal(_np(eng.posteriors(X, hop=1))[:, 0], before)
        finally:
            eng.close()
