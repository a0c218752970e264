"""Synthetic CRNN models of any window length L = 17..256 frames, shared by the GPU test modules: the conv geometry the
kernels derive, a generator drawing every tensor at the shipped models' weight stds, seeded mel windows and the
calibration of the detect head."""
import numpy as np

from conftest import load_weights
from oracle import restated as R
from wakeword_detection_b200 import synth

F64 = np.float64
FILTER_KEYS = ("mel_w", "mel_b", "mel_floor", "mel_log_offset", "mel_scale")


def geometry(L):
    """(T, pad_lo, padded columns) of the conv over L frames: kernel 20, stride 8, TF SAME"""
    T = -(-L // 8)
    pad_lo = (8 * T + 12 - L) // 2
    padded = [t for t in range(T) if 8 * t - pad_lo < 0 or 8 * t - pad_lo + 19 >= L]
    return T, pad_lo, padded


def shared_launches(L):
    """kernel launches of one sliding-window posteriors call on the shared-column path: one front kernel per conv-weight
    variant in use, the two recurrences and the detect head (the per-window path launches 4)"""
    T, _, padded = geometry(L)
    return len(padded) + (len(padded) < T) + 3


def synth_crnn(seed, L, n_out=2):
    """a CRNN of window length L in the layout of weights.load_model_dir, every tensor drawn at the per-tensor std of
    CRNN_arik_original, with the shipped filter; det2 still to be calibrated"""
    ref = load_weights("CRNN_arik_original")
    r = np.random.default_rng(1000 * seed + L)
    w = {k: np.array(v, copy=True) for k, v in load_weights("CRNN").items() if k in FILTER_KEYS}
    for k, v in ref.items():
        if k in FILTER_KEYS or not isinstance(v, np.ndarray) or v.dtype != np.float32 or not v.ndim:
            continue
        shape = (n_out, v.shape[1]) if k == "det2_w" else (n_out,) if k == "det2_b" else v.shape
        w[k] = (r.standard_normal(shape) * float(np.std(v))).astype(np.float32)
    w["mel_length"] = np.int32(L)
    return w


def mel_windows(L, n=16):
    """n mel windows of length L from seeded synthetic audio of every class, plus an all-zero window"""
    f = load_weights("CRNN")
    mels = [R.mel_stream(np.clip(synth.stream_float(16000 * 3, c, 5, c), -1, 1).astype(np.float32), f)
            for c in range(synth.N_CLASSES)]
    step = max(1, (mels[0].shape[0] - L) // 4)
    wins = [m[j:j + L] for m in mels for j in range(0, m.shape[0] - L, step)]
    idx = np.random.default_rng(L).permutation(len(wins))[: n - 1]
    return np.concatenate([np.stack([wins[i] for i in sorted(idx)]), np.zeros((1, L, 40), np.float32)]).astype(np.float32)


def calibrate(w, X):
    """det2 scaled so that the float64 posteriors of X spread over (0, 1): wake logit IQR 3 centred on 0"""
    w = dict(w)
    b0 = w["det2_b"].copy()
    w["det2_b"] = np.zeros_like(b0)
    w["det2_w"] = (w["det2_w"] * np.float32(1e-3)).astype(np.float32)
    p = np.clip(R.posterior(X, w, F64), 1e-300, 1 - 1e-16)
    d = np.log(p) - np.log1p(-p)
    g = 3.0 / max(float(np.percentile(d, 75) - np.percentile(d, 25)), 1e-30)
    w["det2_w"] = (w["det2_w"] * g).astype(np.float32)
    med = float(np.median(d)) * g
    w["det2_b"] = np.array([-med], np.float32) if w["det2_w"].shape[0] == 1 else np.array([b0[0], b0[0] - med], np.float32)
    return w
