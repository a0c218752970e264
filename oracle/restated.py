"""ORACLE (test infrastructure, not product): numpy restatement of the reference's
filter -> encode -> detect path in closed form, batched over windows.

PARITY STATUS: arithmetic *unpinned by the reference* (no tests/golden vectors in
the reference; TFLite 2.4 not importable here — see oracle/tflite_literal.py).
Pins that do exist and are checked in tests/: (1) this file == literal execution
of the shipped `.tflite` graphs; (2) the known-answer values of SURVEY.md
Appendix A4; (3) golden vectors produced by running the reference's *own Python
glue* (spokestack/wakeword/tflite.py, utils/tf_lite/filter.py,
utils/evaluate_models.py) on top of the literal interpreter
(tests/golden/make_golden.py).

Every function cites the reference lines it follows.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module.
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np

F32 = np.float32
HOP = 160
FFT = 512


# ----------------------------------------------------------------------------
# filter
def int16_to_float(pcm: np.ndarray) -> np.ndarray:
    """spokestack/wakeword/tflite.py:150-151 — /32767 then clip to [-1, 1]."""
    x = pcm.astype(F32) / F32(2 ** 15 - 1)
    return np.clip(x, F32(-1.0), F32(1.0))


def pre_emphasis(x: np.ndarray, a: float, prev: float = 0.0) -> np.ndarray:
    """wakeword/tflite.py:156-158, utils/tf_lite/filter.py:42-44:
    y[n] = x[n] - a*x[n-1], state carried across calls; applied over a whole
    stream at once here (f32 product and difference, as numpy does for every call
    after the first)."""
    if a == 0.0:
        return x.astype(F32, copy=True)
    shifted = np.concatenate([np.asarray([prev], F32), x[..., :-1].astype(F32)], axis=-1)
    return (x.astype(F32) - F32(a) * shifted).astype(F32)


def stft_magnitude(frames: np.ndarray) -> np.ndarray:
    """wakeword/tflite.py:174-176 == filter.py:63-65: f32 frame * np.hanning (f64)
    -> np.fft.rfft (f64) -> abs -> f32.  frames: [..., 512] f32."""
    win = np.hanning(frames.shape[-1])
    spec = np.fft.rfft(frames.astype(F32) * win, n=frames.shape[-1])
    return np.abs(spec).astype(F32)


def mel_from_magnitude(mag: np.ndarray, w: Dict[str, np.ndarray], dtype=F32) -> np.ndarray:
    """filter.tflite (SURVEY.md A1): FC -> max(.,1e-5) -> log -> -(-11.5129) -> *0.5.

    `dtype` is the arithmetic of this and every model function below: float32 follows the reference, float64 is the
    high-precision reference the kernels' error is measured against."""
    F = np.dtype(dtype).type
    y = mag.astype(F) @ w["mel_w"].T.astype(F) + w["mel_b"].astype(F)
    y = np.maximum(y.astype(F), F(w["mel_floor"]))
    y = np.log(y).astype(F)
    y = (y - F(w["mel_log_offset"])).astype(F)
    return (y * F(w["mel_scale"])).astype(F)


def num_frames(n_samples: int) -> int:
    """Frames emitted after n samples of a stream (filter.py:50-55): frame k covers
    samples [160k, 160k+512), no centring."""
    return 0 if n_samples < FFT else (n_samples - FFT) // HOP + 1


def mel_of_stream(y: np.ndarray, w: Dict[str, np.ndarray]) -> np.ndarray:
    """All mel frames of an already pre-emphasised float stream y[N] -> [F, 40]
    (filter.py:46-75: ring of 512, hop 160)."""
    y = np.asarray(y, F32)
    nf = num_frames(y.shape[0])
    if nf == 0:
        return np.zeros((0, w["mel_w"].shape[0]), F32)
    idx = np.arange(nf)[:, None] * HOP + np.arange(FFT)[None, :]
    return mel_from_magnitude(stft_magnitude(y[idx]), w)


def mel_stream(x: np.ndarray, w: Dict[str, np.ndarray], a: float = 0.0) -> np.ndarray:
    """pre-emphasis + mel_of_stream for one whole stream (filter.py:38-75)."""
    return mel_of_stream(pre_emphasis(np.asarray(x, F32), a), w)


# ----------------------------------------------------------------------------
# CRNN  (SURVEY.md Appendix A2; architecture cross-check wwdetect/CRNN/model.py:21-56)
def _sigmoid(x, dtype=F32):
    F = np.dtype(dtype).type
    with np.errstate(over="ignore"):
        return (F(1) / (F(1) + np.exp(-x.astype(F)))).astype(F)


def crnn_conv(mel: np.ndarray, w: Dict[str, np.ndarray], dtype=F32) -> np.ndarray:
    """mel [B, L=151, 40] (time, freq) -> [B, 19, 640] with feature = f*32 + c.
    CONV_2D 32@(5 freq x 20 time), stride (2 freq, 8 time), SAME (freq pad 1/2,
    time pad 6/7), fused ReLU, then TRANSPOSE/RESHAPE to [time, freq*chan]."""
    F = np.dtype(dtype).type
    B, L, M = mel.shape
    kf, kt = w["conv_w"].shape[1], w["conv_w"].shape[2]
    of, ot = -(-M // 2), -(-L // 8)
    pf = max((of - 1) * 2 + kf - M, 0)
    pt = max((ot - 1) * 8 + kt - L, 0)
    x = np.pad(mel.astype(F), ((0, 0), (pt // 2, pt - pt // 2), (pf // 2, pf - pf // 2)))
    fi = (np.arange(of) * 2)[:, None] + np.arange(kf)[None, :]          # [of, kf]
    ti = (np.arange(ot) * 8)[:, None] + np.arange(kt)[None, :]          # [ot, kt]
    # patches[b, t, f, kf, kt]
    patches = x[:, ti[:, None, None, :], fi[None, :, :, None]]
    cw = w["conv_w"].reshape(w["conv_w"].shape[0], kf * kt).astype(F)
    y = patches.reshape(B, ot, of, kf * kt) @ cw.T + w["conv_b"].astype(F)
    y = np.maximum(y.astype(F), F(0))
    return y.reshape(B, ot, of * cw.shape[0])


def _gru(seq: np.ndarray, W, U, bi, br, reverse: bool, dtype=F32) -> np.ndarray:
    """Keras GRU v2 (reset_after=True), gate order z|r|h, h0 = 0; returns the
    output sequence in *original* time order (CRNN/encode.tflite WHILE bodies)."""
    F = np.dtype(dtype).type
    B, T, _ = seq.shape
    H = U.shape[1]
    xw = (seq.astype(F) @ W.T.astype(F) + bi.astype(F)).astype(F)     # [B,T,3H]
    h = np.zeros((B, H), F)
    out = np.zeros((B, T, H), F)
    order = range(T - 1, -1, -1) if reverse else range(T)
    for t in order:
        hu = (h @ U.T.astype(F) + br.astype(F)).astype(F)
        z = _sigmoid(xw[:, t, :H] + hu[:, :H], F)
        r = _sigmoid(xw[:, t, H:2 * H] + hu[:, H:2 * H], F)
        c = np.tanh(xw[:, t, 2 * H:] + r * hu[:, 2 * H:]).astype(F)
        h = (z * h + (F(1) - z) * c).astype(F)
        out[:, t] = h
    return out


def crnn_encode(mel: np.ndarray, w: Dict[str, np.ndarray], dtype=F32) -> np.ndarray:
    """mel windows [B, 151, 40] -> encoder output [B, 64] = [fwd_last, bwd_last]."""
    x = crnn_conv(mel, w, dtype)
    f1 = _gru(x, w["gru1_f_w"], w["gru1_f_u"], w["gru1_f_bi"], w["gru1_f_br"], False, dtype)
    b1 = _gru(x, w["gru1_b_w"], w["gru1_b_u"], w["gru1_b_bi"], w["gru1_b_br"], True, dtype)
    s1 = np.concatenate([f1, b1], axis=2)
    f2 = _gru(s1, w["gru2_f_w"], w["gru2_f_u"], w["gru2_f_bi"], w["gru2_f_br"], False, dtype)
    b2 = _gru(s1, w["gru2_b_w"], w["gru2_b_u"], w["gru2_b_bi"], w["gru2_b_br"], True, dtype)
    return np.concatenate([f2[:, -1], b2[:, 0]], axis=1)


def crnn_detect(enc: np.ndarray, w: Dict[str, np.ndarray], dtype=F32) -> np.ndarray:
    """[B, 64] -> detect output [B, n] (n=1 sigmoid head | n=2 softmax head)."""
    F = np.dtype(dtype).type
    h = np.maximum(enc.astype(F) @ w["det1_w"].T + w["det1_b"], F(0)).astype(F)
    z = (h @ w["det2_w"].T + w["det2_b"]).astype(F)
    if z.shape[1] == 1:
        return _sigmoid(z, F)
    z = z - z.max(axis=1, keepdims=True)
    e = np.exp(z).astype(F)
    return (e / e.sum(axis=1, keepdims=True)).astype(F)


# ----------------------------------------------------------------------------
# WaveNet  (SURVEY.md Appendix A3; cross-check wwdetect/wavenet/wavenet_model.py:11-128)
def wavenet_encode(mel: np.ndarray, w: Dict[str, np.ndarray], dtype=F32) -> np.ndarray:
    """mel windows [B, L, 40] -> [B, L, 32] (sum of the 24 skip branches)."""
    F = np.dtype(dtype).type
    B, T, _ = mel.shape
    x = np.maximum(mel.astype(F) @ w["in_w"].T + w["in_b"], F(0)).astype(F)
    nb = w["sig_w"].shape[0]
    out = None
    for k in range(nb):
        d = int(w["dilation"][k])
        u = (x * w["bn_mul"][k] + w["bn_add"][k]).astype(F)
        up = np.pad(u, ((0, 0), (2 * d, 0), (0, 0)))            # zeros *after* the BN affine
        taps = np.concatenate([up[:, j * d:j * d + T] for j in range(3)], axis=2)   # [B,T,48]
        a_s = taps @ w["sig_w"][k].reshape(16, 48).T + w["sig_b"][k]
        a_t = taps @ w["tanh_w"][k].reshape(16, 48).T + w["tanh_b"][k]
        g = (np.tanh(a_t.astype(F)).astype(F) * _sigmoid(a_s, F)).astype(F)
        s = np.maximum(g @ w["skip_w"][k].T + w["skip_b"][k], F(0)).astype(F)
        out = s if out is None else (out + s).astype(F)
        if k < nb - 1:
            x = (np.maximum(g @ w["res_w"][k].T + w["res_b"][k], F(0)) + x).astype(F)
    return out


def wavenet_detect(enc: np.ndarray, w: Dict[str, np.ndarray], dtype=F32) -> np.ndarray:
    """[B, L, 32] -> softmax [B, 2]: ReLU -> 1x1 32->32 ReLU -> 1x1 32->2 -> max over
    time -> softmax (Wavenet/detect.tflite)."""
    F = np.dtype(dtype).type
    h = np.maximum(enc.astype(F), F(0))
    h = np.maximum(h @ w["det1_w"].T + w["det1_b"], F(0)).astype(F)
    z = (h @ w["det2_w"].T + w["det2_b"]).astype(F).max(axis=1)
    z = z - z.max(axis=1, keepdims=True)
    e = np.exp(z).astype(F)
    return (e / e.sum(axis=1, keepdims=True)).astype(F)


def is_crnn(w) -> bool:
    return "conv_w" in w


def encode(mel: np.ndarray, w, dtype=F32) -> np.ndarray:
    return crnn_encode(mel, w, dtype) if is_crnn(w) else wavenet_encode(mel, w, dtype)


def detect(enc: np.ndarray, w, dtype=F32) -> np.ndarray:
    return crnn_detect(enc, w, dtype) if is_crnn(w) else wavenet_detect(enc, w, dtype)


def posterior(mel: np.ndarray, w, dtype=F32) -> np.ndarray:
    """Wake-class probability per window: out[..., -1] covers both CRNN heads and the
    WaveNet head (SURVEY.md §8 note N1; wakeword/tflite.py:228-231,
    evaluate_models.py:80,86)."""
    return detect(encode(mel, w, dtype), w, dtype)[:, -1]


# ----------------------------------------------------------------------------
# glue
def eval_windows(n_frames: int, L: int, hop: int = 2) -> int:
    """Number of posteriors get_posterior yields for a clip with n_frames mel frames
    (evaluate_models.py:66-73)."""
    return 0 if n_frames < L else (n_frames - L) // hop + 1


def eval_clip_samples(samples: np.ndarray, sample_rate: int = 16000,
                      frame_length: int = 320) -> np.ndarray:
    """evaluate_models.py:52-61: sr//2 zeros each side, then whole 320-sample chunks
    (the last chunk zero-padded)."""
    x = np.pad(np.asarray(samples, F32), (sample_rate // 2, sample_rate // 2))
    n = -(-x.shape[0] // frame_length) * frame_length
    return np.pad(x, (0, n - x.shape[0]))


def get_posterior(clips: Sequence[np.ndarray], w, eval_type: str, a: float = 0.0,
                  batch: int = 256) -> List:
    """evaluate_models.py:26-108 for already-loaded float clips.  The Filter object is
    created once (:30), so its 512-sample ring and pre-emphasis state carry over from
    clip to clip: clip i's frame grid continues the cumulative stream, i.e. its stream
    is prefixed by the (already pre-emphasised) samples the ring still held."""
    L = int(w["mel_length"])
    carry = np.zeros((0,), F32)
    prev = 0.0
    allp: List = []
    for clip in clips:
        x = eval_clip_samples(clip)
        y = pre_emphasis(x, a, prev)
        prev = float(x[-1])
        s = np.concatenate([carry, y])
        mel = mel_of_stream(s, w)
        carry = s[mel.shape[0] * HOP:]
        nw = eval_windows(mel.shape[0], L)
        post = np.zeros((nw,), F32)
        for i in range(0, nw, batch):
            j = np.arange(i, min(nw, i + batch))
            win = mel[(2 * j)[:, None] + np.arange(L)[None, :]]
            post[i:i + len(j)] = posterior(win, w)
        if eval_type == "false_negatives":
            allp.append(np.max(post))
        else:
            allp.extend(list(post))
    return allp


def smooth_same(p: np.ndarray, n: int = 30) -> np.ndarray:
    """evaluate_models.py:188-189: np.convolve(p, ones(n)/n, 'same') (f64)."""
    return np.convolve(np.asarray(p), np.ones((n,)) / n, mode="same")


def rising_edges(p: np.ndarray, thr: float) -> int:
    """evaluate_models.py:207-216 == plot_eval_models.py:84-96."""
    above = np.asarray(p) > thr
    if above.size == 0:
        return 0
    return int(above[0]) + int(np.count_nonzero(above[1:] & ~above[:-1]))


def far_frr_counts(pos_max: np.ndarray, neg: np.ndarray, thresholds: np.ndarray,
                   window: int = 30) -> Tuple[np.ndarray, np.ndarray]:
    """Integer numerators of plot_FRR_FAR (evaluate_models.py:183-218):
    accepts_pos[t] = #(pos_max > t); edges_neg[t] = rising edges of smoothed negatives."""
    sm = smooth_same(neg, window)
    acc = np.array([int((np.asarray(pos_max) > t).sum()) for t in thresholds], np.int64)
    edg = np.array([rising_edges(sm, t) for t in thresholds], np.int64)
    return acc, edg


def thresholds_eval() -> np.ndarray:
    """evaluate_models.py:185."""
    return np.arange(0.5, 0.99999, 0.005)


def thresholds_plot() -> np.ndarray:
    """plot_eval_models.py:103."""
    return np.arange(0.5, 0.9905, 0.001)


class TriggerOracle:
    """State machine equivalent to WakewordTrigger (spokestack/wakeword/tflite.py:123-246)
    for one stream: int16 chunks in, list of posteriors out; `active` latches when a
    posterior exceeds the threshold (strict >, :235)."""

    def __init__(self, w, threshold: float = 0.5, a: float = 0.0) -> None:
        self.w, self.thr, self.a = w, threshold, a
        self.L = int(w["mel_length"])
        self.pending = np.zeros((0,), F32)            # the sample ring's unread content
        self.frames = np.zeros((self.L, w["mel_w"].shape[0]), F32)   # frame_window.fill(0.0) :102
        self.prev_sample = 0.0
        self.was_speech = False
        self.post_max = 0.0
        self.active = False
        self.posteriors: List[float] = []

    def reset(self) -> None:
        """:241-246"""
        self.pending = np.zeros((0,), F32)
        self.frames[:] = 0.0
        self.post_max = 0.0

    def __call__(self, chunk: np.ndarray, is_speech: bool) -> None:
        vad_fall = self.was_speech and not is_speech
        self.was_speech = is_speech
        if not self.active:
            x = int16_to_float(chunk)
            y = pre_emphasis(x, self.a, self.prev_sample)
            self.prev_sample = float(x[-1])
            self.pending = np.concatenate([self.pending, y])
            # the rest of the chunk is still analysed after activation (:163-168, :233-239)
            while self.pending.shape[0] >= FFT:
                if is_speech:
                    mel = mel_from_magnitude(stft_magnitude(self.pending[None, :FFT]), self.w)[0]
                    self.frames = np.concatenate([self.frames[1:], mel[None]])
                    p = float(posterior(self.frames[None], self.w)[0])
                    self.posteriors.append(p)
                    self.post_max = max(self.post_max, p)
                    if p > self.thr:
                        self.active = True
                self.pending = self.pending[HOP:]
        if vad_fall:
            self.reset()


# ----------------------------------------------------------------------------
# pipeline stages around the trigger (SURVEY.md 8f row 2)
class VadDebounceOracle:
    """Rise / fall debounce of VoiceActivityDetector (spokestack/vad/webrtc.py:34-77); the raw per-frame decision of
    the webrtcvad C extension is an input."""

    def __init__(self, frame_width=20, vad_rise_delay=0, vad_fall_delay=0):
        self.rise = vad_rise_delay // frame_width
        self.fall = vad_fall_delay // frame_width
        self.run_value, self.run_length = 0, 0

    def __call__(self, is_speech: bool, raw: bool) -> bool:
        raw = bool(raw)
        if raw == self.run_value:
            self.run_length += 1
        else:
            self.run_value, self.run_length = raw, 1
        if self.run_value != is_speech:
            if self.run_value and self.run_length >= self.rise:
                is_speech = True
            if not self.run_value and self.run_length >= self.fall:
                is_speech = False
        return is_speech


class ActivationTimeoutOracle:
    """spokestack/activation_timeout.py:16-38."""

    def __init__(self, frame_width=20, min_active=500, max_active=5000):
        self.min_active = min_active / frame_width
        self.max_active = max_active / frame_width
        self.is_speech, self.active_length = False, 0

    def __call__(self, is_speech: bool, is_active: bool) -> bool:
        vad_fall = self.is_speech and not is_speech
        self.is_speech = is_speech
        if is_active:
            self.active_length += 1
            if self.active_length > self.min_active:
                if vad_fall or self.active_length > self.max_active:
                    self.active_length = 0
                    is_active = False
        return is_active


class PipelineOracle:
    """One stream through vad -> wake-word trigger -> activation timeout, one call per frame
    (SpeechPipeline._dispatch, spokestack/pipeline.py:25-28)."""

    def __init__(self, w, threshold=0.5, a=0.0, frame_width=20, vad_rise_delay=0, vad_fall_delay=0, min_active=500,
                 max_active=5000):
        self.vad = VadDebounceOracle(frame_width, vad_rise_delay, vad_fall_delay)
        self.trig = TriggerOracle(w, threshold, a)
        self.tmo = ActivationTimeoutOracle(frame_width, min_active, max_active)
        self.is_speech = False

    @property
    def is_active(self):
        return self.trig.active

    def __call__(self, frame: np.ndarray, raw_vad: bool):
        self.is_speech = self.vad(self.is_speech, raw_vad)
        self.trig(frame, self.is_speech)
        self.trig.active = self.tmo(self.is_speech, self.trig.active)
        return self.is_speech, self.trig.active


class KeywordOracle:
    """spokestack/asr/keyword/tflite.py:15-191 for one stream, with the encoder / detector as callables (the reference
    ships no keyword model): returns the list of (kind, class index, confidence) events a frame produced."""

    def __init__(self, w, encode_model, detect_model, threshold=0.5, a=0.97):
        self.w, self.enc, self.det, self.thr, self.a = w, encode_model, detect_model, threshold, a
        self.L = int(encode_model.input_details[0]["shape"][1])
        self.EL, self.EW = (int(v) for v in detect_model.input_details[0]["shape"][1:])
        self.state = np.zeros(encode_model.input_details[1]["shape"], F32)
        self.prev_sample, self.was_active = 0.0, False
        self.reset()

    def reset(self):
        self.pending = np.zeros((0,), F32)
        self.frames = np.zeros((self.L, self.w["mel_w"].shape[0]), F32)
        self.encoded = np.full((self.EL, self.EW), -1.0, F32)
        self.state[:] = 0.0

    def __call__(self, chunk, is_active):
        x = int16_to_float(chunk)
        y = pre_emphasis(x, self.a, self.prev_sample)
        self.prev_sample = float(x[-1])
        self.pending = np.concatenate([self.pending, y])
        while self.pending.shape[0] >= FFT:
            if is_active:
                mel = mel_from_magnitude(stft_magnitude(self.pending[None, :FFT]), self.w)[0]
                self.frames = np.concatenate([self.frames[1:], mel[None]])
                enc, self.state = self.enc(self.frames[None], self.state)
                self.encoded = np.concatenate([self.encoded[1:], np.asarray(enc, F32).reshape(1, self.EW)])
            self.pending = self.pending[HOP:]
        events = []
        if not is_active and self.was_active:
            post = self.det(self.encoded[None])[0][0]
            k = int(np.argmax(post))
            events.append(("recognize", k, float(post[k])) if post[k] >= self.thr else ("timeout", -1, 0.0))
            self.reset()
        self.was_active = is_active
        return events
