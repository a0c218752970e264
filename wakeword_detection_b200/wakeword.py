"""`WakewordTrigger` drop-in and its many-stream form.

Reference: spokestack/wakeword/tflite.py:20-250.  Same constructor arguments, stage
protocol `trigger(context, frame)`, `reset()` and `close()`; the per-stream state of the
reference (512-sample window, previous sample, mel frame window pre-filled with 0.0,
posterior maximum) lives in HBM and every call runs filter -> encode -> detect on the
GPU (csrc: stream_filter_kernel -> encoder -> stream_finish_kernel).  The spoken reply
on wake (pydub, :113-121,:238) is optional: it is skipped when pydub is not installed.
"""
from __future__ import annotations

import logging
import os

import numpy as np

from . import _cabi
from .ring_buffer import RingBuffer

_LOG = logging.getLogger(__name__)


def _pack(chunks):
    """list of 1-D int16 chunks (numpy arrays or torch tensors) -> (one packed 1-D array or tensor, lengths)"""
    if any(len(c.shape) != 1 for c in chunks):
        raise ValueError("every chunk must be 1-D")
    lengths = [int(c.shape[0]) for c in chunks]
    if all(isinstance(c, np.ndarray) for c in chunks):
        return np.concatenate([np.zeros(0, np.int16)] + [c.astype(np.int16, copy=False) for c in chunks]), lengths
    import torch
    dev = next(c.device for c in chunks if isinstance(c, torch.Tensor))
    return torch.cat([torch.as_tensor(c).to(dev, torch.int16) for c in chunks]), lengths


class MultiStreamTrigger:
    """S independent WakewordTrigger state machines advanced by one call.

    push(pcm[S, n] int16, is_speech[S], is_active[S]) -> dict of device tensors:
      post [S, max_frames] (NaN where no frame was analysed), n_post [S], trigger [S],
      post_max [S].  The caller owns the `is_active` latch exactly like
      SpeechContext.is_active in the reference (:139,:236-239).

    push_streams(ids, chunks, is_speech, is_active) advances only the slots in `ids` (distinct, any order), each
    by its own chunk (a list of 1-D int16 arrays or tensors, any lengths up to chunk_samples): the way a server
    receives audio.  Same dict, one row per entry of `ids`.

    export_streams(ids) -> uint8 device tensor [n_ids, record bytes]: the state of those slots, one record each.
    import_streams(ids, records) puts such records (from any context of the same model, any device) into the slots in
    `ids`: to park and resume a session, move it to another slot, context or GPU, or rewind it.

    set_stream_options(ids, threshold, listening) sets per-slot options, one value per entry of `ids` or one for all:
    a threshold that replaces posterior_threshold for that slot (NaN: back to posterior_threshold), and listening 0 to
    pause a slot (its pushes are treated as is_active: nothing is consumed or analysed) or 1 to resume it from its
    retained window.  Resets and imports keep the options."""

    def __init__(self, model_dir: str, model_type: str, n_streams: int, chunk_samples: int = 320,
                 pre_emphasis: float = 0.0, posterior_threshold: float = 0.5, device: int = 0,
                 precision: str = "tc") -> None:
        from . import weights as W
        self.engine = _cabi.Engine(W.load_model_dir(model_dir, model_type), device, precision)
        self.n_streams = int(n_streams)
        self.pre_emphasis = float(pre_emphasis)
        self.threshold = float(posterior_threshold)
        self.engine.stream_alloc(self.n_streams, int(chunk_samples))

    def push(self, pcm, is_speech=None, is_active=None):
        post, n_post, trig, pmax = self.engine.stream_push(pcm, is_speech, is_active, self.pre_emphasis,
                                                           self.threshold)
        return {"post": post, "n_post": n_post, "trigger": trig, "post_max": pmax}

    def push_streams(self, ids, chunks, is_speech=None, is_active=None):
        pcm, lengths = _pack(chunks)
        post, n_post, trig, pmax = self.engine.stream_push_indexed(ids, pcm, lengths, is_speech, is_active,
                                                                   self.pre_emphasis, self.threshold)
        return {"post": post, "n_post": n_post, "trigger": trig, "post_max": pmax}

    def export_streams(self, ids):
        return self.engine.stream_export(ids)

    def import_streams(self, ids, records) -> None:
        self.engine.stream_import(ids, records)

    def set_stream_options(self, ids, threshold=None, listening=None) -> None:
        self.engine.stream_set_options(ids, threshold, listening)

    def reset(self, mask=None) -> None:
        self.engine.stream_reset(mask)

    def close(self) -> None:
        self.engine.close()


class MultiStreamPipeline:
    """S independent speech pipelines [vad debounce -> WakewordTrigger -> ActivationTimeout] advanced by one call, all
    state on the device (reference: spokestack/pipeline.py:25-28 dispatching spokestack/vad/webrtc.py:52-77,
    spokestack/wakeword/tflite.py:123-246, spokestack/activation_timeout.py:25-38).  The raw per-frame VAD decision is an
    input (the webrtcvad C extension is outside the path).

    step(pcm[S, n] int16, vad_raw[S]) -> dict of device tensors: post, n_post, post_max, is_speech, is_active,
    activated, deactivated.  step_streams(ids, frames, vad_raw) dispatches only the slots in `ids`, each with its own
    frame (list of 1-D int16 arrays or tensors); same dict, one row per entry of `ids`.  export_streams /
    import_streams and set_stream_options as on MultiStreamTrigger; the records carry the VAD debounce and
    ActivationTimeout state too (the delays are the context's own).  A paused slot's VAD debounce and timeout go on."""

    def __init__(self, model_dir: str, model_type: str, n_streams: int, frame_width: int = 20, sample_rate: int = 16000,
                 pre_emphasis: float = 0.0, posterior_threshold: float = 0.5, vad_rise_delay: int = 0,
                 vad_fall_delay: int = 0, min_active: int = 500, max_active: int = 5000, device: int = 0,
                 precision: str = "tc") -> None:
        from . import weights as W
        self.engine = _cabi.Engine(W.load_model_dir(model_dir, model_type), device, precision)
        self.n_streams = int(n_streams)
        self.frame_samples = int(frame_width * sample_rate / 1000)
        self.pre_emphasis = float(pre_emphasis)
        self.threshold = float(posterior_threshold)
        self.engine.stream_alloc(self.n_streams, self.frame_samples)
        self.engine.context_alloc(frame_width, vad_rise_delay, vad_fall_delay, min_active, max_active)

    def step(self, pcm, vad_raw=None):
        return self.engine.context_step(pcm, vad_raw, self.pre_emphasis, self.threshold)

    def step_streams(self, ids, frames, vad_raw=None):
        pcm, lengths = _pack(frames)
        return self.engine.context_step_indexed(ids, pcm, lengths, vad_raw, self.pre_emphasis, self.threshold)

    def export_streams(self, ids):
        return self.engine.stream_export(ids)

    def import_streams(self, ids, records) -> None:
        self.engine.stream_import(ids, records)

    def set_stream_options(self, ids, threshold=None, listening=None) -> None:
        self.engine.stream_set_options(ids, threshold, listening)

    def reset(self) -> None:
        self.engine.context_reset()

    def close(self) -> None:
        self.engine.close()


class MultiWakewordPipeline:
    """S speech pipelines listening for several wake words, [vad debounce -> WakewordTrigger(model 0) -> ... ->
    WakewordTrigger(model K-1) -> ActivationTimeout], the reference's SpeechPipeline with one trigger stage per model
    (spokestack/pipeline.py:25-28), advanced by one call with all state on the device.  Stage k sees the is_active that
    the stages before it set in the same frame: once one stage triggers, the later ones skip that frame's chunk.

    models: list of (model_dir, model_type) or dicts with model_dir, model_type and optionally posterior_threshold (0.5)
    and pre_emphasis (0.0); each stage keeps its own filter and window state.
    step(pcm[S, n] int16, vad_raw[S]) / step_streams(ids, frames, vad_raw) -> the dict of MultiStreamPipeline with post
    [K, S, max_frames], n_post [K, S] and post_max [K, S] per stage, plus activated_by [S] (int8: the stage that
    triggered, -1 if none).  export_streams(ids) -> one record tensor per stage (stage 0's carries the pipeline state);
    import_streams(ids, records) puts them back, all or nothing across the stages.

    set_stream_options(ids, threshold, listening) sets the options of MultiStreamTrigger per slot and stage: arrays
    [n_ids, K], or [n_ids] / a scalar for every stage.  A slot that listens to stage k only runs no encoder windows in
    the other stages, and a paused stage does not change the is_active that later stages see."""

    def __init__(self, models, n_streams: int, frame_width: int = 20, sample_rate: int = 16000, vad_rise_delay: int = 0,
                 vad_fall_delay: int = 0, min_active: int = 500, max_active: int = 5000, device: int = 0,
                 precision: str = "tc") -> None:
        from . import weights as W
        stages = [dict(m) if isinstance(m, dict) else {"model_dir": m[0], "model_type": m[1]} for m in models]
        if not 1 <= len(stages) <= _cabi.WWB_MAX_STAGES:
            raise ValueError("%d stages outside [1, %d]" % (len(stages), _cabi.WWB_MAX_STAGES))
        self.n_streams = int(n_streams)
        self.frame_samples = int(frame_width * sample_rate / 1000)
        self.pre_emphasis = [float(m.get("pre_emphasis", 0.0)) for m in stages]
        self.thresholds = [float(m.get("posterior_threshold", 0.5)) for m in stages]
        self.engines = []
        try:
            for m in stages:
                e = _cabi.Engine(W.load_model_dir(m["model_dir"], m["model_type"]), device, precision)
                self.engines.append(e)
                e.stream_alloc(self.n_streams, self.frame_samples)
            self.engines[0].context_alloc(frame_width, vad_rise_delay, vad_fall_delay, min_active, max_active)
        except BaseException:
            self.close()
            raise

    def step(self, pcm, vad_raw=None):
        return self.engines[0].context_step_chain(self.engines[1:], pcm, vad_raw, self.pre_emphasis, self.thresholds)

    def step_streams(self, ids, frames, vad_raw=None):
        pcm, lengths = _pack(frames)
        return self.engines[0].context_step_chain_indexed(self.engines[1:], ids, pcm, lengths, vad_raw,
                                                          self.pre_emphasis, self.thresholds)

    def export_streams(self, ids):
        return [e.stream_export(ids) for e in self.engines]

    def import_streams(self, ids, records) -> None:
        self.engines[0].stream_import_chain(self.engines[1:], ids, records)

    def set_stream_options(self, ids, threshold=None, listening=None) -> None:
        ids = np.ascontiguousarray(ids, np.int32)
        if ids.ndim != 1:
            raise ValueError("ids must be 1-D")
        K = len(self.engines)

        def per_stage(v, name):
            """None, a scalar, [n_ids] or [n_ids, K] -> the K stages' values"""
            if v is None:
                return [None] * K
            a = np.asarray(v)
            if a.ndim == 1:
                a = a[:, None]
            if a.ndim > 2 or (a.ndim == 2 and a.shape not in ((ids.size, K), (ids.size, 1))):
                raise ValueError("%s must be a scalar, [%d] or [%d, %d], got shape %s"
                                 % (name, ids.size, ids.size, K, list(np.shape(v))))
            return [np.broadcast_to(a, (ids.size, K))[:, k] for k in range(K)]

        # every stage's values are checked before the first stage's call: a bad argument cannot apply to some stages only
        opts = [_cabi._stream_options(ids.size, t, l)
                for t, l in zip(per_stage(threshold, "threshold"), per_stage(listening, "listening"))]
        if any(l is not None and (l > 1).any() for _, l in opts):
            raise ValueError("listening values must be 0 or 1")
        for e, (t, l) in zip(self.engines, opts):
            e.stream_set_options(ids, t, l)

    def reset(self) -> None:
        self.engines[0].context_reset()
        for e in self.engines[1:]:
            e.stream_reset()

    def close(self) -> None:
        for e in self.engines:
            e.close()


class WakewordTrigger:
    """Detects the presence of a wakeword in the audio input (single stream)."""

    def __init__(self, pre_emphasis: float = 0.0, sample_rate: int = 16000, fft_window_type: str = "hann",
                 fft_hop_length: int = 10, model_dir: str = "", model_type: str = "",
                 posterior_threshold: float = 0.5, **kwargs) -> None:
        self.pre_emphasis: float = pre_emphasis
        self.hop_length: int = int(fft_hop_length * sample_rate / 1000)
        if fft_window_type != "hann":
            raise ValueError("Invalid fft_window_type")
        self.model_type = model_type.upper()
        device = int(kwargs.pop("device", 0))
        precision = kwargs.pop("precision", "tc")
        max_chunk = int(kwargs.pop("max_chunk_samples", 1600))
        self._multi_args = (model_dir, model_type, 1, max_chunk, pre_emphasis, posterior_threshold, device, precision)
        self._multi = MultiStreamTrigger(*self._multi_args)
        e = self._multi.engine
        self._window_size = (e.n_bins - 1) * 2
        if self.hop_length != 160:
            raise ValueError("the CUDA filter is built for a 160-sample hop")
        self.mel_length: int = e.L
        self.mel_width: int = e.n_mel
        crnn = e.kind == _cabi.WWB_MODEL_CRNN
        self.encode_length: int = 1 if crnn else e.L
        self.encode_width: int = 64 if crnn else 32
        # host mirrors of the reference's public ring attributes (:92-104); the live state is on the device
        self.sample_window = RingBuffer(shape=[self._window_size])
        self.frame_window = RingBuffer(shape=[self.mel_length, self.mel_width])
        self.encode_window = RingBuffer(shape=[1, self.encode_length, self.encode_width])
        self.frame_window.fill(0.0)
        self.encode_window.fill(-1.0)
        self._posterior_threshold: float = posterior_threshold
        self._posterior_max: float = 0.0
        self._is_speech: bool = False
        self.last_posteriors = np.zeros((0,), np.float32)
        self.audio_responses = np.array([], dtype=object)
        self.load_awake_responses(kwargs.pop("audio_responses", "audio_responses"))

    def load_awake_responses(self, audio_path) -> None:
        try:
            from pydub import AudioSegment  # type: ignore
        except Exception:
            return
        if not os.path.isdir(audio_path):
            return
        segs = []
        for f in os.listdir(audio_path):
            p = os.path.join(audio_path, f)
            if os.path.isfile(p) and ".mp3" in p:
                segs.append(AudioSegment.from_mp3(p))
        self.audio_responses = np.array(segs, dtype=object)

    def __call__(self, context, frame) -> None:
        # the VAD-edge bookkeeping and the reset on a fall happen on the device
        # (stream_finish_kernel); the host mirrors them for logging (:135-146)
        vad_fall = self._is_speech and not context.is_speech
        self._is_speech = context.is_speech
        was_active = bool(context.is_active)
        frame = np.ascontiguousarray(frame, dtype=np.int16)
        if self._multi is None:      # the stage is used again after close(): a fresh device context, like a fresh interpreter
            self._multi = MultiStreamTrigger(*self._multi_args)
        out = self._multi.push(frame[None, :], np.array([context.is_speech], np.uint8),
                               np.array([was_active], np.uint8))
        n = int(out["n_post"][0])
        self.last_posteriors = out["post"][0, :n].cpu().numpy() if n else np.zeros((0,), np.float32)
        if not was_active:
            self._posterior_max = float(out["post_max"][0])
            if int(out["trigger"][0]):
                _LOG.info(f"AWAKE!: {self._posterior_max}")
                self._play_response()
                context.is_active = True
        if vad_fall:
            if not context.is_active:
                _LOG.info(f"wake: {self._posterior_max}")
            self._posterior_max = 0.0

    def _play_response(self) -> None:
        if len(self.audio_responses) == 0:
            return
        try:
            from pydub.playback import play  # type: ignore
            play(np.random.choice(self.audio_responses))
        except Exception:  # pragma: no cover
            pass

    def reset(self) -> None:
        if self._multi is not None:
            self._multi.reset()
        self.sample_window.reset()
        self.frame_window.reset().fill(0.0)
        self.encode_window.reset().fill(-1.0)
        self._posterior_max = 0.0

    def close(self) -> None:
        """:248-250 resets the stage; here it also releases the device context (weights, stream state, workspaces)."""
        self.reset()
        if self._multi is not None:
            self._multi.close()
            self._multi = None
