"""ctypes binding of libwwb200.so (include/wwb200.h) and the `Engine` that hands torch
CUDA tensors to it.  PyTorch is plumbing only here: device memory, streams, dtype
conversion.  There is no CPU path: without the built library or without a CUDA device
every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WWB200_LIB") or os.path.join(_HERE, "libwwb200.so")   # override: A/B builds of the same ABI

WWB_MODEL_NONE, WWB_MODEL_CRNN, WWB_MODEL_WAVENET = -1, 0, 1
WWB_PCM_I16, WWB_PCM_F32 = 0, 1
WWB_PREC_F32, WWB_PREC_TC, WWB_PREC_TC_FAST = 0, 1, 2
WWB_COUNT_FRR_MAX, WWB_COUNT_FAR_EDGES = 0, 1
WWB_MAX_STAGES = 8   # trigger stages of one chain (wwb_context_step_chain)
PRECISIONS = {"f32": WWB_PREC_F32, "tc": WWB_PREC_TC, "tc_fast": WWB_PREC_TC_FAST}

_fp = C.POINTER(C.c_float)


class WwbWeights(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("mel_length", C.c_int32), ("n_out", C.c_int32),
        ("n_mel", C.c_int32), ("n_bins", C.c_int32),
        ("mel_w", _fp), ("mel_b", _fp),
        ("mel_floor", C.c_float), ("mel_log_offset", C.c_float), ("mel_scale", C.c_float),
        ("conv_w", _fp), ("conv_b", _fp),
        ("gru_w", _fp * 4), ("gru_u", _fp * 4), ("gru_bi", _fp * 4), ("gru_br", _fp * 4),
        ("in_w", _fp), ("in_b", _fp), ("bn_mul", _fp), ("bn_add", _fp),
        ("dilation", C.POINTER(C.c_int32)),
        ("sig_w", _fp), ("sig_b", _fp), ("tanh_w", _fp), ("tanh_b", _fp),
        ("res_w", _fp), ("res_b", _fp), ("skip_w", _fp), ("skip_b", _fp),
        ("det1_w", _fp), ("det1_b", _fp), ("det2_w", _fp), ("det2_b", _fp),
    ]


# every symbol include/wwb200.h declares: (restype, argtypes)
_vp, _i64, _i32 = C.c_void_p, C.c_int64, C.c_int
PROTOTYPES = {
    "wwb_version": (C.c_int, []),
    "wwb_last_error": (C.c_char_p, [_vp]),
    "wwb_create": (C.c_int, [C.c_int, C.POINTER(WwbWeights), C.c_int, C.POINTER(_vp)]),
    "wwb_destroy": (C.c_int, [_vp]),
    "wwb_set_precision": (C.c_int, [_vp, C.c_int]),
    "wwb_sync": (C.c_int, [_vp, _vp]),
    "wwb_num_frames": (_i64, [_i64]),
    "wwb_num_windows": (_i64, [_vp, _i64, C.c_int]),
    "wwb_stream_granule": (_i64, [_vp, _i64, C.c_int]),
    "wwb_filter": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _i64, C.c_float, _vp, _vp]),
    "wwb_mel_from_magnitude": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "wwb_encode": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "wwb_detect": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "wwb_posteriors": (C.c_int, [_vp, _vp, _i64, _i64, C.c_int, _vp, _vp]),
    "wwb_pipeline": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _i64, C.c_float, C.c_int, _vp, _vp]),
    "wwb_pipeline_host": (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, C.c_float, C.c_int, _vp]),
    "wwb_sweep_submit": (C.c_int, [C.POINTER(_vp), C.c_int, _vp, C.c_int, _i64, _i64, C.c_float, C.c_int, _vp, C.c_int,
                                   C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "wwb_sweep_wait": (C.c_int, [_vp]),
    "wwb_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "wwb_host_free": (C.c_int, [_vp]),
    "wwb_eval_counts": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    "wwb_stream_alloc": (C.c_int, [_vp, _i64, _i64]),
    "wwb_stream_push": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _vp, _vp, _vp]),
    "wwb_stream_push_indexed": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _vp, _vp,
                                          _vp]),
    "wwb_stream_max_frames": (C.c_int, [_vp]),
    "wwb_stream_reset": (C.c_int, [_vp, _vp, _i64, _vp]),
    "wwb_stream_set_options": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "wwb_context_alloc": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "wwb_context_step": (C.c_int, [_vp, _vp, _i64, _i64, _vp, C.c_float, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "wwb_context_step_indexed": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _vp, _vp, _vp,
                                           _vp, _vp, _vp]),
    "wwb_context_reset": (C.c_int, [_vp, _vp]),
    "wwb_context_step_chain": (C.c_int, [C.POINTER(_vp), C.c_int, _vp, _i64, _i64, _vp, _vp, _vp, C.POINTER(_vp),
                                         C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _vp, _vp, _vp, _vp]),
    "wwb_context_step_chain_indexed": (C.c_int, [C.POINTER(_vp), C.c_int, _vp, _i64, _vp, _vp, _vp, _vp, _vp,
                                                 C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _vp, _vp,
                                                 _vp, _vp]),
    "wwb_stream_state_bytes": (_i64, [_vp]),
    "wwb_stream_export": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "wwb_stream_import": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "wwb_stream_import_chain": (C.c_int, [C.POINTER(_vp), C.c_int, _vp, _i64, C.POINTER(_vp), _vp, _vp]),
    "wwb_launch_count": (_i64, [_vp]),
    "wwb_debug_buffer": (C.c_int, [_vp, _vp]),
}

# ---- stream state records (include/wwb200.h, wwb_stream_export / wwb_stream_import): the only Python code that knows
# the layout.  A record is the 48-byte header, the pending samples and the [L, 40] frame window, oldest row first.
STREAM_STATE_MAGIC = 0x53425757      # "WWBS"
STREAM_STATE_VERSION = 1
STREAM_STATE_PENDING = 512
STREAM_STATE_PIPELINE = 1            # flags bit 0: the pipeline fields hold state
STREAM_STATE_HEADER = np.dtype([
    ("magic", "<u4"), ("version", "<u2"), ("flags", "<u2"), ("kind", "<i4"), ("mel_length", "<i4"),
    ("n_pending", "<i4"), ("prev_sample", "<f4"), ("post_max", "<f4"),
    ("was_speech", "u1"), ("is_speech", "u1"), ("is_active", "u1"), ("t_is_speech", "u1"),
    ("run_value", "<i4"), ("run_length", "<i4"), ("active_length", "<i4"), ("reserved", "<u4"),
])
# wwb_stream_import's reason codes (WWB_RECORD_*)
RECORD_REASONS = {1: "bad magic", 2: "unsupported record version", 3: "unknown flag bits",
                  4: "written by a context of another model kind", 5: "mel_length does not match this context",
                  6: "n_pending outside [0, 511]"}


def stream_state_dtype(L: int) -> np.dtype:
    """numpy dtype of one whole record of a model with an L-frame window"""
    return np.dtype([("header", STREAM_STATE_HEADER), ("pending", "<f4", (STREAM_STATE_PENDING,)),
                     ("mel", "<f4", (int(L), 40))])


def decode_stream_state(records, L: int) -> Dict[str, np.ndarray]:
    """records (uint8 [n, bytes] or [bytes]; numpy or a torch tensor on any device) -> dict of per-entry arrays: every
    header field, `pending` [n, 512] and `mel` [n, L, 40]"""
    if not isinstance(records, np.ndarray):
        records = records.detach().cpu().numpy()
    dt = stream_state_dtype(L)
    raw = np.ascontiguousarray(records).view(np.uint8).reshape(-1)
    if raw.size % dt.itemsize:
        raise ValueError("%d bytes are not a whole number of %d-byte records" % (raw.size, dt.itemsize))
    rec = raw.view(dt)
    out = {k: rec["header"][k].copy() for k in STREAM_STATE_HEADER.names}
    out["pending"] = rec["pending"].copy()
    out["mel"] = rec["mel"].copy()
    return out


_lib = None


def load_library() -> C.CDLL:
    """Loads the in-tree library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "wwb200: %s is missing — build it with `python -m wakeword_detection_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    try:
        import torch  # noqa: F401  (brings libcudart into the process)
    except Exception:  # pragma: no cover
        pass
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class WwbError(RuntimeError):
    pass


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array over page-locked host memory from wwb_host_alloc (freed when the array is collected): the
    host-buffer entry points copy from / to such arrays without the driver's pageable staging."""
    import weakref
    lib = load_library()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = _vp()
    rc = lib.wwb_host_alloc(C.byref(p), max(n, 16))
    if rc:
        raise WwbError((lib.wwb_last_error(None) or b"").decode())
    buf = (C.c_char * max(n, 16)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    weakref.finalize(buf, lib.wwb_host_free, p.value)
    return arr


def _raise(code: int, msg: str):
    if code == -1:
        raise ValueError(msg)
    if code == -3:
        raise IndexError(msg)
    raise WwbError(msg)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a), dtype=np.float32)


def _pcm_dtype(dtype) -> int:
    """WWB_PCM_* of a numpy or torch PCM dtype"""
    code = {"int16": WWB_PCM_I16, "float32": WWB_PCM_F32}.get(str(dtype).replace("torch.", ""))
    if code is None:
        raise ValueError("PCM must be int16 or float32, got %s" % dtype)
    return code


def make_weights_struct(w: Optional[Dict[str, np.ndarray]], filt: Dict[str, np.ndarray]):
    """Packs host arrays into the C struct; returns (struct, keepalive list)."""
    keep = []

    def p(a):
        a = _f32(a)
        keep.append(a)
        return a.ctypes.data_as(_fp)

    s = WwbWeights()
    s.n_mel, s.n_bins = filt["mel_w"].shape
    s.mel_w, s.mel_b = p(filt["mel_w"]), p(filt["mel_b"])
    s.mel_floor = float(filt["mel_floor"])
    s.mel_log_offset = float(filt["mel_log_offset"])
    s.mel_scale = float(filt["mel_scale"])
    if w is None or ("conv_w" not in w and "in_w" not in w):
        s.kind, s.mel_length, s.n_out = WWB_MODEL_NONE, 0, 0
        return s, keep
    s.mel_length = int(w["mel_length"])
    s.n_out = int(w["det2_w"].shape[0])
    for k in ("det1_w", "det1_b", "det2_w", "det2_b"):
        setattr(s, k, p(w[k]))
    if "conv_w" in w:
        s.kind = WWB_MODEL_CRNN
        s.conv_w, s.conv_b = p(w["conv_w"]), p(w["conv_b"])
        for i, key in enumerate(("gru1_f", "gru1_b", "gru2_f", "gru2_b")):
            s.gru_w[i] = p(w[key + "_w"])
            s.gru_u[i] = p(w[key + "_u"])
            s.gru_bi[i] = p(w[key + "_bi"])
            s.gru_br[i] = p(w[key + "_br"])
    else:
        s.kind = WWB_MODEL_WAVENET
        for k in ("in_w", "in_b", "bn_mul", "bn_add", "sig_w", "sig_b", "tanh_w", "tanh_b",
                  "res_w", "res_b", "skip_w", "skip_b"):
            setattr(s, k, p(w[k]))
        d = np.ascontiguousarray(w["dilation"], dtype=np.int32)
        keep.append(d)
        s.dilation = d.ctypes.data_as(C.POINTER(C.c_int32))
    return s, keep


class Engine:
    """One wwb_ctx on one GPU.  All tensor arguments are torch CUDA tensors on that
    device (numpy arrays are uploaded); results are torch CUDA tensors."""

    def __init__(self, weights: Dict[str, np.ndarray], device: int = 0, precision: str = "tc") -> None:
        import torch

        self.lib = load_library()
        self.torch = torch
        if not torch.cuda.is_available():
            raise WwbError("wwb200: no CUDA device visible; this framework has no CPU fallback")
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.weights = weights
        st, keep = make_weights_struct(weights, weights)
        ctx = _vp()
        rc = self.lib.wwb_create(self.device_index, C.byref(st), PRECISIONS[precision], C.byref(ctx))
        if rc:
            _raise(rc, (self.lib.wwb_last_error(None) or b"").decode())
        self.ctx = ctx
        self.kind = st.kind
        self.L = st.mel_length
        self.n_out = st.n_out
        self.n_mel = st.n_mel
        self.n_bins = st.n_bins
        self._stream_cap = None
        del keep

    # -- helpers ------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "ctx", None):
            self.lib.wwb_destroy(self.ctx)
            self.ctx = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc:
            _raise(rc, (self.lib.wwb_last_error(self.ctx) or b"").decode())

    def _stream(self):
        return _vp(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, a, dtype):
        t = self.torch
        if isinstance(a, t.Tensor):
            x = a
            if x.device != self.device:
                x = x.to(self.device)
        else:
            x = t.from_numpy(np.ascontiguousarray(a)).to(self.device)
        if x.dtype != dtype:
            x = x.to(dtype)
        return x.contiguous()

    def set_precision(self, precision: str) -> None:
        self._check(self.lib.wwb_set_precision(self.ctx, PRECISIONS[precision]))

    def sync(self) -> None:
        self._check(self.lib.wwb_sync(self.ctx, self._stream()))

    def launch_count(self) -> int:
        return int(self.lib.wwb_launch_count(self.ctx))

    def num_frames(self, n_samples: int) -> int:
        return int(self.lib.wwb_num_frames(int(n_samples)))

    def num_windows(self, n_frames: int, hop: int) -> int:
        return int(self.lib.wwb_num_windows(self.ctx, int(n_frames), int(hop)))

    def stream_granule(self, n_frames: int, hop: int) -> int:
        """Stream-count granule for callers that slice a batch (whole waves of the persistent kernels)."""
        return int(self.lib.wwb_stream_granule(self.ctx, int(n_frames), int(hop)))

    # -- hot path -------------------------------------------------------------------
    def _pcm(self, pcm):
        t = self.torch
        if isinstance(pcm, np.ndarray):
            pcm = t.from_numpy(np.ascontiguousarray(pcm))
        dt = _pcm_dtype(pcm.dtype)
        if pcm.dim() == 1:
            pcm = pcm[None]
        if pcm.dim() != 2:
            raise ValueError("PCM must be [n_streams, n_samples]")
        if pcm.device != self.device:
            pcm = pcm.to(self.device)
        if pcm.stride(1) != 1:
            pcm = pcm.contiguous()
        return pcm, dt

    def filter(self, pcm, pre_emphasis: float = 0.0, out=None):
        """[S, N] int16|float32 -> mel [S, F, 40] float32."""
        t = self.torch
        pcm, dt = self._pcm(pcm)
        S, N = pcm.shape
        F = self.num_frames(N)
        mel = out if out is not None else t.empty((S, F, self.n_mel), dtype=t.float32, device=self.device)
        self._check(self.lib.wwb_filter(self.ctx, pcm.data_ptr(), dt, S, N, pcm.stride(0) if S > 1 else N, float(pre_emphasis),
                                        mel.data_ptr(), self._stream()))
        return mel

    def mel_from_magnitude(self, mag):
        t = self.torch
        mag = self._dev(mag, t.float32)
        if mag.dim() != 2 or mag.shape[1] != self.n_bins:
            raise ValueError("cannot set tensor: dimension mismatch, expected [B,%d] got %s"
                             % (self.n_bins, list(mag.shape)))
        mel = t.empty((mag.shape[0], self.n_mel), dtype=t.float32, device=self.device)
        self._check(self.lib.wwb_mel_from_magnitude(self.ctx, mag.data_ptr(), mag.shape[0], mel.data_ptr(),
                                                    self._stream()))
        return mel

    def encode(self, mel_windows):
        """[B, L, 40] -> CRNN [B, 64] | WaveNet [B, L, 32]."""
        t = self.torch
        x = self._dev(mel_windows, t.float32)
        if x.dim() != 3 or x.shape[1] != self.L or x.shape[2] != self.n_mel:
            raise ValueError("cannot set tensor: dimension mismatch, expected [B,%d,%d] got %s"
                             % (self.L, self.n_mel, list(x.shape)))
        B = x.shape[0]
        shape = (B, 64) if self.kind == WWB_MODEL_CRNN else (B, self.L, 32)
        enc = t.empty(shape, dtype=t.float32, device=self.device)
        self._check(self.lib.wwb_encode(self.ctx, x.data_ptr(), B, enc.data_ptr(), self._stream()))
        return enc

    def detect(self, enc):
        t = self.torch
        x = self._dev(enc, t.float32)
        want = [64] if self.kind == WWB_MODEL_CRNN else [self.L, 32]
        if list(x.shape[1:]) != want:
            raise ValueError("cannot set tensor: dimension mismatch, expected [B,%s] got %s"
                             % (",".join(map(str, want)), list(x.shape)))
        out = t.empty((x.shape[0], self.n_out), dtype=t.float32, device=self.device)
        self._check(self.lib.wwb_detect(self.ctx, x.data_ptr(), x.shape[0], out.data_ptr(), self._stream()))
        return out

    def posteriors(self, mel, hop: int = 2, out=None):
        """mel [S, F, 40] -> wake posteriors [S, n_win] over windows hopping `hop` frames."""
        t = self.torch
        x = self._dev(mel, t.float32)
        if x.dim() != 3 or x.shape[2] != self.n_mel:
            raise ValueError("mel must be [S, F, %d]" % self.n_mel)
        S, F = x.shape[0], x.shape[1]
        nw = self.num_windows(F, hop)
        post = out if out is not None else t.empty((S, nw), dtype=t.float32, device=self.device)
        self._check(self.lib.wwb_posteriors(self.ctx, x.data_ptr(), S, F, int(hop), post.data_ptr(), self._stream()))
        return post

    def pipeline(self, pcm, hop: int = 2, pre_emphasis: float = 0.0, out=None):
        """PCM [S, N] -> posteriors [S, n_win] (filter -> encode -> detect)."""
        t = self.torch
        pcm, dt = self._pcm(pcm)
        S, N = pcm.shape
        nw = self.num_windows(self.num_frames(N), hop)
        post = out if out is not None else t.empty((S, nw), dtype=t.float32, device=self.device)
        self._check(self.lib.wwb_pipeline(self.ctx, pcm.data_ptr(), dt, S, N, pcm.stride(0) if S > 1 else N, float(pre_emphasis),
                                          int(hop), post.data_ptr(), self._stream()))
        return post

    def pipeline_host(self, pcm: np.ndarray, hop: int = 2, pre_emphasis: float = 0.0,
                      out: Optional[np.ndarray] = None) -> np.ndarray:
        """Same through HOST buffers (numpy in, numpy out; copies inside the call)."""
        pcm = np.ascontiguousarray(pcm)
        if pcm.ndim == 1:
            pcm = pcm[None]
        dt = _pcm_dtype(pcm.dtype)
        S, N = pcm.shape
        nw = self.num_windows(self.num_frames(N), hop)
        post = out if out is not None else np.empty((S, nw), np.float32)
        self._check(self.lib.wwb_pipeline_host(self.ctx, pcm.ctypes.data, dt, S, N, float(pre_emphasis), int(hop),
                                               post.ctypes.data))
        return post

    def sweep_submit(self, pcm: np.ndarray, hop: int = 2, thresholds=None, others: Sequence["Engine"] = (),
                     pre_emphasis: float = 0.0, want_post: bool = True, out=None):
        """Asynchronous host-buffer pipeline (wwb_sweep_submit): `pcm` [S, N] numpy (ideally from `pinned_empty`) ->
        for this engine and every engine in `others` (same device; ONE copy and ONE filter pass feed all of them)
        posteriors [S, n_win] and, with `thresholds`, the FAR-edge / FRR-max counters, all in HOST memory once
        `sweep_wait()` returns.  Returns the result record (dict of numpy arrays) that the wait fills."""
        if pcm.ndim != 2 or not pcm.flags.c_contiguous:
            raise ValueError("PCM must be a C-contiguous [n_streams, n_samples] array")
        dt = _pcm_dtype(pcm.dtype)
        engines = [self] + list(others)
        S, N = pcm.shape
        F = self.num_frames(N)
        n = len(engines)
        rec = out if out is not None else {"post": [None] * n, "far": [None] * n, "frr": [None] * n}
        thr = None
        if thresholds is not None:
            thr = np.ascontiguousarray(thresholds, np.float64)
            if thr.ndim != 1 or thr.size == 0 or np.any(np.diff(thr) < 0):
                raise ValueError("thresholds must be a non-empty ascending 1-D array")
        for m, e in enumerate(engines):
            nw = e.num_windows(F, hop)
            if want_post and (rec["post"][m] is None or rec["post"][m].shape != (S, nw)):
                rec["post"][m] = pinned_empty((S, nw), np.float32)
            if thr is not None:
                for k in ("far", "frr"):
                    if rec[k][m] is None or rec[k][m].shape != (thr.size,):
                        rec[k][m] = np.zeros((thr.size,), np.int64)
        arr = lambda xs: (_vp * n)(*[(x.ctypes.data if x is not None else None) for x in xs])
        ctxs = (_vp * n)(*[e.ctx for e in engines])
        self._check(self.lib.wwb_sweep_submit(
            ctxs, n, pcm.ctypes.data, dt, S, N, float(pre_emphasis), int(hop),
            thr.ctypes.data if thr is not None else None, int(thr.size) if thr is not None else 0,
            arr(rec["post"]) if want_post else None, arr(rec["far"]) if thr is not None else None,
            arr(rec["frr"]) if thr is not None else None))
        rec["_keep"] = (pcm, thr)
        return rec

    def sweep_wait(self) -> None:
        """Blocks until the oldest submitted job's results are in host memory."""
        self._check(self.lib.wwb_sweep_wait(self.ctx))

    def _cached_const(self, kind: str, arr: np.ndarray):
        """Device copy of a small host array (segment offsets, threshold grids), reused while its content is unchanged:
        a sweep calls eval_counts with the same tables every step, and four pageable H2D copies per step were most of
        the 'counts' stage."""
        cache = self.__dict__.setdefault("_const_cache", {})
        key = (kind, arr.dtype.str, arr.shape, hash(arr.tobytes()))
        hit = cache.get(key)
        if hit is None:
            if len(cache) > 64:
                cache.clear()
            hit = cache[key] = self.torch.from_numpy(np.ascontiguousarray(arr)).to(self.device)
        return hit

    def eval_counts(self, post, seg_off: Sequence[int], thresholds, mode: str, smooth: int = 30,
                    halo_lo=None, halo_hi=None):
        """FAR/FRR numerators -> int64 tensor [n_thr] on the device."""
        t = self.torch
        thr = np.asarray(thresholds, np.float64)
        if thr.ndim != 1 or thr.size == 0 or np.any(np.diff(thr) < 0):
            raise ValueError("thresholds must be a non-empty ascending 1-D array")
        seg = np.asarray(seg_off, np.int64)
        if seg.ndim != 1 or seg.size < 1 or np.any(np.diff(seg) < 0):
            raise ValueError("seg_off must be ascending")
        nseg = seg.size - 1
        m = {"frr_max": WWB_COUNT_FRR_MAX, "far_edges": WWB_COUNT_FAR_EDGES}[mode]
        if m == WWB_COUNT_FRR_MAX and np.any(np.diff(seg) == 0):
            # np.max([]) in the reference (evaluate_models.py:99)
            raise ValueError("zero-size array to reduction operation maximum which has no identity")
        if m == WWB_COUNT_FAR_EDGES and nseg and smooth > 1 and np.any((np.diff(seg) < smooth) & (np.diff(seg) > 0)):
            # np.convolve(p, ones(w)/w, 'same') on a trajectory SHORTER than the window swaps its operands and returns
            # max(M, N) = w values (evaluate_models.py:188-189): rare, so those segments are smoothed here in float64
            # exactly like numpy and the whole batch goes through the kernel unsmoothed (smooth = 1)
            if halo_lo is not None or halo_hi is not None:
                raise ValueError("time-chunk halos need chunks of at least %d posteriors" % smooth)
            ph = (post.detach().cpu().numpy() if isinstance(post, t.Tensor) else np.asarray(post)).reshape(-1).astype(np.float64)
            parts = [np.convolve(ph[a:b], np.ones((smooth,)) / smooth, mode='same') for a, b in zip(seg[:-1], seg[1:])]
            seg = np.concatenate([[0], np.cumsum([x.size for x in parts])]).astype(np.int64)
            return self._far_edges_f64(np.concatenate(parts) if parts else np.zeros((0,)), seg, thr)
        p = self._dev(post, t.float32).reshape(-1)
        n_total = int(seg[-1])
        if n_total > p.numel():
            raise ValueError("seg_off exceeds the posterior buffer")
        d_seg = self._cached_const("seg", seg)
        d_thr = self._cached_const("thr", thr)
        d_lo = self._dev(np.asarray(halo_lo, np.int32), t.int32) if halo_lo is not None else None
        d_hi = self._dev(np.asarray(halo_hi, np.int32), t.int32) if halo_hi is not None else None
        counts = t.zeros((thr.size,), dtype=t.int64, device=self.device)
        self._check(self.lib.wwb_eval_counts(
            self.ctx, p.data_ptr(), d_seg.data_ptr(), nseg,
            d_lo.data_ptr() if d_lo is not None else None, d_hi.data_ptr() if d_hi is not None else None,
            n_total, d_thr.data_ptr(), int(thr.size), m, int(smooth), counts.data_ptr(), self._stream()))
        return counts

    def _far_edges_f64(self, smoothed: np.ndarray, seg: np.ndarray, thr: np.ndarray):
        """Rising-edge counts of already smoothed float64 trajectories (host; only for the short-trajectory corner of
        eval_counts - the values would lose their float64 smoothing if they went back through the float32 kernel)."""
        counts = np.zeros((thr.size,), np.int64)
        for a, b in zip(seg[:-1], seg[1:]):
            x = smoothed[a:b]
            above = x[None, :] > thr[:, None]
            counts += np.count_nonzero(above & ~np.concatenate([np.zeros((thr.size, 1), bool), above[:, :-1]], axis=1), axis=1)
        return self.torch.from_numpy(counts).to(self.device)

    # -- streaming ------------------------------------------------------------------------
    def stream_alloc(self, max_streams: int, max_chunk: int) -> None:
        self._check(self.lib.wwb_stream_alloc(self.ctx, int(max_streams), int(max_chunk)))
        self._stream_cap = (int(max_streams), int(max_chunk))
        self.stream_reset()

    def stream_max_frames(self) -> int:
        return int(self.lib.wwb_stream_max_frames(self.ctx))

    def stream_push(self, pcm, is_speech=None, is_active=None, pre_emphasis: float = 0.0,
                    threshold: float = 0.5):
        """pcm [S, n] int16 -> (post [S, max_frames] (NaN = none), n_post [S] int32,
        trigger [S] uint8, post_max [S] float32) device tensors."""
        x = self._dense(pcm)
        S, n = x.shape
        out = self._trigger_out(S)
        self._call(self.lib.wwb_stream_push, (x.data_ptr(), S, n), (is_speech, is_active), pre_emphasis, threshold, out)
        return out

    def _flags(self, a):
        """optional per-stream uint8 flags -> device tensor (or None)"""
        t = self.torch
        if a is None:
            return None
        return a.to(self.device, t.uint8) if isinstance(a, t.Tensor) else self._dev(np.asarray(a), t.uint8)

    def _dense(self, pcm):
        """the int16 PCM of a dense push or step on the device, [S, n]"""
        x = self._dev(pcm, self.torch.int16)
        return x[None] if x.dim() == 1 else x

    def _indexed(self, ids, pcm_packed, lengths):
        """host int32 id / length tables and the packed int16 PCM on the device, checked for shape (the library checks
        the values)"""
        ids = np.ascontiguousarray(ids, np.int32)
        lengths = np.ascontiguousarray(lengths, np.int32)
        if ids.ndim != 1 or lengths.shape != ids.shape:
            raise ValueError("ids and lengths must be 1-D and of the same length")
        x = self._dev(pcm_packed, self.torch.int16)
        if x.dim() != 1 or x.numel() != int(lengths.astype(np.int64).sum()):
            raise ValueError("pcm_packed must be 1-D with sum(lengths) = %d samples, got %s"
                             % (int(lengths.astype(np.int64).sum()), list(x.shape)))
        return ids, lengths, x

    def _trigger_out(self, S: int):
        """the outputs of a push over S entries: post [S, max_frames], n_post, trigger, post_max"""
        t = self.torch
        return (t.empty((S, self.stream_max_frames()), dtype=t.float32, device=self.device),
                t.empty((S,), dtype=t.int32, device=self.device), t.empty((S,), dtype=t.uint8, device=self.device),
                t.empty((S,), dtype=t.float32, device=self.device))

    def _step_out(self, S: int, engines=None):
        """the outputs of a step over S entries, by name in the C ABI's order: post [S, max_frames], n_post, post_max,
        is_speech, is_active, activated, deactivated; for the chain of `engines` post [K, S, max_frames], n_post [K, S]
        and post_max [K, S] per stage, then activated_by [S] int8"""
        t = self.torch
        K = () if engines is None else (len(engines),)
        mf = {e.stream_max_frames() for e in engines or [self]}
        if len(mf) != 1:
            raise ValueError("the stages take chunks of different max_frames %s; allocate them alike" % sorted(mf))
        out = {"post": t.empty(K + (S, mf.pop()), dtype=t.float32, device=self.device),
               "n_post": t.empty(K + (S,), dtype=t.int32, device=self.device),
               "post_max": t.empty(K + (S,), dtype=t.float32, device=self.device)}
        for k in ("is_speech", "is_active", "activated", "deactivated"):
            out[k] = t.empty((S,), dtype=t.uint8, device=self.device)
        if engines is not None:
            out["activated_by"] = t.empty((S,), dtype=t.int8, device=self.device)
        return out

    def _call(self, fn, streams, flags, pre_emphasis, threshold, outputs) -> None:
        """fn(ctx, *streams, *flags, pre_emphasis, threshold, *outputs, stream): the C call of every push and step;
        `streams` name the streams and their PCM, `flags` are the optional per-entry uint8 inputs"""
        flags = [self._flags(f) for f in flags]
        self._check(fn(self.ctx, *streams, *[None if f is None else f.data_ptr() for f in flags], float(pre_emphasis),
                       float(threshold), *[o.data_ptr() for o in outputs], self._stream()))

    def stream_push_indexed(self, ids, pcm_packed, lengths, is_speech=None, is_active=None, pre_emphasis: float = 0.0,
                            threshold: float = 0.5):
        """One chunk for each slot in `ids` (distinct, any order), chunk i of lengths[i] samples, packed back to back in
        `pcm_packed` (1-D int16) -> (post [n_ids, max_frames] (NaN = none), n_post [n_ids] int32, trigger [n_ids] uint8,
        post_max [n_ids] float32) device tensors, one row per entry of `ids`.  is_speech / is_active per entry."""
        ids, lengths, x = self._indexed(ids, pcm_packed, lengths)
        out = self._trigger_out(ids.size)
        self._call(self.lib.wwb_stream_push_indexed, (ids.ctypes.data, ids.size, lengths.ctypes.data, x.data_ptr()),
                   (is_speech, is_active), pre_emphasis, threshold, out)
        return out

    def context_alloc(self, frame_width: int = 20, vad_rise_delay: int = 0, vad_fall_delay: int = 0, min_active: int = 500,
                      max_active: int = 5000) -> None:
        """Per-stream VAD debounce + ActivationTimeout state next to the streaming trigger (wwb_context_alloc)."""
        self._check(self.lib.wwb_context_alloc(self.ctx, int(frame_width), int(vad_rise_delay), int(vad_fall_delay),
                                               int(min_active), int(max_active)))

    def context_step(self, pcm, vad_raw=None, pre_emphasis: float = 0.0, threshold: float = 0.5):
        """One SpeechPipeline dispatch for every stream: vad debounce -> wake-word trigger -> activation timeout.
        pcm [S, n] int16, vad_raw [S] (None = speech) -> dict of device tensors: post [S, max_frames] (NaN = none),
        n_post, post_max, is_speech, is_active, activated, deactivated."""
        x = self._dense(pcm)
        S, n = x.shape
        out = self._step_out(S)
        self._call(self.lib.wwb_context_step, (x.data_ptr(), S, n), (vad_raw,), pre_emphasis, threshold, out.values())
        return out

    def context_step_indexed(self, ids, pcm_packed, lengths, vad_raw=None, pre_emphasis: float = 0.0,
                             threshold: float = 0.5):
        """context_step for the slots in `ids` only, tables and packing as in stream_push_indexed; vad_raw per entry ->
        the dict of context_step with one row per entry of `ids`."""
        ids, lengths, x = self._indexed(ids, pcm_packed, lengths)
        out = self._step_out(ids.size)
        self._call(self.lib.wwb_context_step_indexed, (ids.ctypes.data, ids.size, lengths.ctypes.data, x.data_ptr()),
                   (vad_raw,), pre_emphasis, threshold, out.values())
        return out

    def context_reset(self) -> None:
        self._check(self.lib.wwb_context_reset(self.ctx, self._stream()))

    # -- trigger chains: this engine's trigger and pipeline state, then one trigger stage per engine in `others` ---------
    def _chain(self, others):
        """(engines, ctx array) of the chain [self] + others"""
        engines = [self] + list(others)
        return engines, (_vp * len(engines))(*[e.ctx for e in engines])

    @staticmethod
    def _per_stage(v, K: int) -> np.ndarray:
        """a scalar or K values -> float32 [K] host array"""
        return np.ascontiguousarray(np.broadcast_to(np.asarray(v, np.float32), (K,)))

    def _call_chain(self, fn, others, streams, vad_raw, pre_emphasis, thresholds, S: int):
        engines, ctxs = self._chain(others)
        K = len(engines)
        a, thr = self._per_stage(pre_emphasis, K), self._per_stage(thresholds, K)
        out = self._step_out(S, engines)
        rows = lambda x: (_vp * K)(*[x[k].data_ptr() for k in range(K)])
        vad = self._flags(vad_raw)
        self._check(fn(ctxs, K, *streams, None if vad is None else vad.data_ptr(), a.ctypes.data, thr.ctypes.data,
                       rows(out["post"]), rows(out["n_post"]), rows(out["post_max"]),
                       *[o.data_ptr() for o in list(out.values())[3:]], self._stream()))
        return out

    def context_step_chain(self, others: Sequence["Engine"], pcm, vad_raw=None, pre_emphasis=0.0, thresholds=0.5):
        """One SpeechPipeline dispatch with one wake-word stage per engine: vad debounce -> trigger of this engine ->
        trigger of each engine in `others` -> activation timeout (wwb_context_step_chain).  This engine holds the
        pipeline state (context_alloc); every engine has stream state of the same capacity on the same device.
        pre_emphasis / thresholds: one value per stage or one for all.  -> the dict of context_step with post
        [K, S, max_frames], n_post [K, S] and post_max [K, S] per stage, plus activated_by [S] int8 (-1: none)."""
        x = self._dense(pcm)
        S, n = x.shape
        return self._call_chain(self.lib.wwb_context_step_chain, others, (x.data_ptr(), S, n), vad_raw, pre_emphasis,
                                thresholds, S)

    def context_step_chain_indexed(self, others: Sequence["Engine"], ids, pcm_packed, lengths, vad_raw=None,
                                   pre_emphasis=0.0, thresholds=0.5):
        """context_step_chain for the slots in `ids` only, tables and packing as in stream_push_indexed."""
        ids, lengths, x = self._indexed(ids, pcm_packed, lengths)
        return self._call_chain(self.lib.wwb_context_step_chain_indexed, others,
                                (ids.ctypes.data, ids.size, lengths.ctypes.data, x.data_ptr()), vad_raw, pre_emphasis,
                                thresholds, ids.size)

    def stream_import_chain(self, others: Sequence["Engine"], ids, records) -> None:
        """stream_import into every stage of the chain [self] + others, all or nothing across the stages: records[k]
        (uint8 [n_ids, bytes of stage k]) from stream_export of a stage-k engine.  A bad record raises
        ValueError("stage <k> record <i>: <reason>") and no slot of any stage is touched."""
        t = self.torch
        engines, ctxs = self._chain(others)
        ids = self._state_ids(ids)
        if len(records) != len(engines):
            raise ValueError("%d record sets for %d stages" % (len(records), len(engines)))
        recs = [self._records(r, ids.size, e.stream_state_bytes(), "stage %d: " % k)
                for k, (e, r) in enumerate(zip(engines, records))]
        status = t.zeros((3,), dtype=t.int32, device=self.device)
        ptrs = (_vp * len(recs))(*[r.data_ptr() or None for r in recs])
        self._check(self.lib.wwb_stream_import_chain(ctxs, len(engines), ids.ctypes.data, ids.size, ptrs,
                                                     status.data_ptr(), self._stream()))
        bad, why, stage = (int(v) for v in status.cpu())
        if bad:
            raise ValueError("stage %d record %d: %s" % (stage, bad - 1, RECORD_REASONS.get(why, "reason %d" % why)))

    def stream_state_bytes(self) -> int:
        """size of one stream state record (0 without stream_alloc or on a filter-only context)"""
        return int(self.lib.wwb_stream_state_bytes(self.ctx))

    def _records(self, records, n_ids: int, nb: int, prefix: str = ""):
        """records of one stage (uint8 [n_ids, nb], a tensor on any device or a numpy array) -> a contiguous uint8
        tensor on this context's device; a wrong dtype or size raises ValueError starting with `prefix`"""
        t = self.torch
        if isinstance(records, np.ndarray):
            records = t.from_numpy(np.ascontiguousarray(records).view(np.uint8))
        if records.dtype != t.uint8:
            raise ValueError("%srecords must be uint8, got %s" % (prefix, records.dtype))
        rec = records.to(self.device).contiguous()
        if nb and rec.numel() != n_ids * nb:
            raise ValueError("%srecords hold %d bytes, %d entries need %d" % (prefix, rec.numel(), n_ids, n_ids * nb))
        return rec

    def _state_ids(self, ids) -> np.ndarray:
        ids = np.ascontiguousarray(ids, np.int32)
        if ids.ndim != 1:
            raise ValueError("ids must be 1-D")
        return ids

    def stream_export(self, ids):
        """The state of the slots in `ids` (distinct, any order) -> uint8 tensor [n_ids, stream_state_bytes()] on this
        context's device, one record per entry (decode_stream_state reads them).  Stream-ordered after the pushes."""
        t = self.torch
        ids = self._state_ids(ids)
        out = t.empty((ids.size, self.stream_state_bytes()), dtype=t.uint8, device=self.device)
        self._check(self.lib.wwb_stream_export(self.ctx, ids.ctypes.data, ids.size, out.data_ptr() or None,
                                               self._stream()))
        return out

    def stream_import(self, ids, records) -> None:
        """Puts records (from stream_export of any context of the same model: uint8 [n_ids, bytes], a tensor on any
        device or a numpy array) into the slots in `ids`, all or nothing.  Waits for the device's verdict: a bad record
        raises ValueError("record <i>: <reason>") and no slot is touched."""
        t = self.torch
        ids = self._state_ids(ids)
        rec = self._records(records, ids.size, self.stream_state_bytes())
        status = t.zeros((2,), dtype=t.int32, device=self.device)
        self._check(self.lib.wwb_stream_import(self.ctx, ids.ctypes.data, ids.size, rec.data_ptr() or None,
                                               status.data_ptr(), self._stream()))
        bad, why = (int(v) for v in status.cpu())
        if bad:
            raise ValueError("record %d: %s" % (bad - 1, RECORD_REASONS.get(why, "reason %d" % why)))

    def stream_reset(self, mask=None) -> None:
        t = self.torch
        if self._stream_cap is None:
            raise IndexError("stream state not allocated")
        S = self._stream_cap[0]
        m = None
        if mask is not None:
            m = self._dev(np.asarray(mask), t.uint8)
            S = m.numel()
        self._check(self.lib.wwb_stream_reset(self.ctx, m.data_ptr() if m is not None else None, S, self._stream()))

    def stream_set_options(self, ids, threshold=None, listening=None) -> None:
        """Per-slot trigger options of the slots in `ids` (distinct, any order), one value per entry or one for all;
        None leaves that option as it is.  threshold: NaN = the threshold each push or step passes, any other value
        replaces it for the slot.  listening: 0 pauses the slot (every push treats it as is_active: nothing consumed or
        analysed, no trigger), 1 lets it continue from its retained window.  Stream-ordered like the pushes; kept
        across stream_reset, context_reset and stream_import, and not part of the records."""
        ids = self._state_ids(ids)
        thr, lst = _stream_options(ids.size, threshold, listening)
        self._check(self.lib.wwb_stream_set_options(self.ctx, ids.ctypes.data, ids.size,
                                                    None if thr is None else thr.ctypes.data,
                                                    None if lst is None else lst.ctypes.data, self._stream()))


def _stream_options(n: int, threshold=None, listening=None):
    """threshold / listening (None, a scalar or n values) -> (float32 [n] or None, uint8 [n] or None) host arrays; a
    wrong shape, or a listening value that is not a whole number in [0, 255], raises ValueError (the library refuses
    values other than 0 and 1)"""
    def per_entry(v, name):
        a = np.asarray(v)
        if a.ndim > 1 or (a.ndim == 1 and a.size != n):
            raise ValueError("%s must be a scalar or %d values, got shape %s" % (name, n, list(a.shape)))
        return np.broadcast_to(a, (n,))
    thr = None if threshold is None else np.ascontiguousarray(per_entry(threshold, "threshold"), np.float32)
    lst = None
    if listening is not None:
        v = per_entry(listening, "listening")
        lst = np.ascontiguousarray(v, np.uint8)
        if not np.array_equal(lst, v):
            raise ValueError("listening values must be 0 or 1")
    return thr, lst


_ENGINES: Dict[Tuple, Engine] = {}


def engine_for_dir(model_dir: str, model_type: str, device: int = 0, precision: str = "tc", quant: bool = False) -> Engine:
    """One shared Engine per (model directory, kind, device, precision, variant) — the reference builds three
    interpreters per directory; here they share one context.  quant=True: the float16-weight variant
    (weights.load_model_dir)."""
    from . import weights as W

    key = (os.path.abspath(model_dir), W.model_kind(model_type), int(device), precision, bool(quant))
    eng = _ENGINES.get(key)
    if eng is None or eng.ctx is None:
        eng = Engine(W.load_model_dir(model_dir, model_type, quant=quant), device=device, precision=precision)
        _ENGINES[key] = eng
    return eng
