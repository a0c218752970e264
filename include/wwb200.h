/*
 * wwb200 — C ABI of the B200-native filter -> encode -> detect wake-word path.
 *
 * The reference (MerlinPCarson/WakeWord-Detection) has no FFI layer: its hot path
 * calls `tflite.Interpreter.set_tensor / invoke / get_tensor` from Python
 * (reference: spokestack/models/tensorflow.py:43-51).  This header is the boundary a
 * maintainer binds instead (ctypes stub in INTEGRATION.md); every entry point names
 * the reference call site it replaces.
 *
 * Conventions
 *  - plain C, no torch types.  `*_dev` pointers are borrowed device pointers on the
 *    ctx's device, `*_host` pointers are host memory.  Nothing passed in is freed.
 *  - `stream` is a `cudaStream_t` passed as void* (NULL = the legacy default stream).
 *    Device-pointer entry points only enqueue work; call wwb_sync() (or synchronise
 *    the stream yourself) before reading results.  `*_host` entry points return after
 *    the results are in host memory.
 *  - every function returns 0 on success or a negative wwb_status; the message is
 *    available from wwb_last_error().  There is no CPU fallback: without a CUDA
 *    device wwb_create fails with WWB_ERR_CUDA.
 *  - a ctx is bound to one device and is not re-entrant (the reference's TFLite
 *    Interpreter is not thread-safe either); distinct ctxs are independent.  Its scratch
 *    workspaces (mel, encoder intermediates, counters) are per ctx, not per stream: all
 *    calls on one ctx must be STREAM-ORDERED on one CUDA stream (or separated by
 *    wwb_sync); growing a workspace synchronises the device.  The *_host entry points use
 *    three streams owned by the ctx and are ordered among themselves.
 */
#ifndef WWB200_H
#define WWB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WWB_VERSION 100 /* 0.1.0 */

typedef enum {
  WWB_OK = 0,
  WWB_ERR_ARG = -1,   /* bad argument (Python shim raises ValueError)        */
  WWB_ERR_CUDA = -2,  /* CUDA runtime error / no device (RuntimeError)       */
  WWB_ERR_STATE = -3, /* call order / capacity violation (IndexError)        */
  WWB_ERR_ALLOC = -4
} wwb_status;

/* WWB_MODEL_NONE: filter only (a directory that holds just filter.tflite) */
enum { WWB_MODEL_NONE = -1, WWB_MODEL_CRNN = 0, WWB_MODEL_WAVENET = 1 };
enum { WWB_PCM_I16 = 0, WWB_PCM_F32 = 1 };
/* arithmetic of the encoder GEMMs */
enum {
  WWB_PREC_F32 = 0, /* CUDA-core fp32 (validation path)                                   */
  WWB_PREC_TC = 1,  /* tcgen05 tensor cores, fp16 hi/lo split operands, fp32 accumulate   */
  WWB_PREC_TC_FAST = 2 /* tcgen05, single fp16 operands (outside the 1e-3 parity bound)  */
};
enum { WWB_COUNT_FRR_MAX = 0, WWB_COUNT_FAR_EDGES = 1 };

/* Trained tensors, host pointers, float32, layouts as in the .tflite files
 * (FC weights [out,in]; see wakeword_detection_b200/weights.py).  Unused family = NULL. */
typedef struct {
  int32_t kind;       /* WWB_MODEL_*                                              */
  int32_t mel_length; /* encoder window length in mel frames: 151 (CRNN) / 17..182 (WaveNet; shipped 182) */
  int32_t n_out;      /* detect outputs: CRNN 1 (sigmoid) or 2 (softmax); WaveNet 2 (softmax) */
  int32_t n_mel;      /* 40 */
  int32_t n_bins;     /* 257 */
  /* filter.tflite: FC -> max(floor) -> log -> -offset -> *scale */
  const float* mel_w; /* [n_mel, n_bins] */
  const float* mel_b; /* [n_mel] */
  float mel_floor, mel_log_offset, mel_scale;
  /* CRNN */
  const float* conv_w;    /* [32,5,20]  (out, freq tap, time tap) */
  const float* conv_b;    /* [32] */
  const float* gru_w[4];  /* [96,in]  order: L1 fwd, L1 bwd, L2 fwd, L2 bwd */
  const float* gru_u[4];  /* [96,32] */
  const float* gru_bi[4]; /* [96] input-projection bias */
  const float* gru_br[4]; /* [96] recurrent bias */
  /* WaveNet */
  const float* in_w;   /* [16,40] */
  const float* in_b;   /* [16] */
  const float* bn_mul; /* [24,16] */
  const float* bn_add; /* [24,16] */
  const int32_t* dilation; /* [24] */
  const float* sig_w;  /* [24,16,3,16] (out, tap, in) */
  const float* sig_b;  /* [24,16] */
  const float* tanh_w; /* [24,16,3,16] */
  const float* tanh_b; /* [24,16] */
  const float* res_w;  /* [23,16,16] */
  const float* res_b;  /* [23,16] */
  const float* skip_w; /* [24,32,16] */
  const float* skip_b; /* [24,32] */
  /* detect head (CRNN: 64->64->n_out ; WaveNet: 32->32->2) */
  const float* det1_w;
  const float* det1_b;
  const float* det2_w;
  const float* det2_b;
} wwb_weights;

typedef struct wwb_ctx wwb_ctx;

int wwb_version(void);
/* message of the last failing call on `ctx` (or of the last failing wwb_create when ctx is NULL) */
const char* wwb_last_error(const wwb_ctx* ctx);

/* Replaces the three TFLiteModel(...) constructions (spokestack/wakeword/tflite.py:51-59,
 * utils/evaluate_models.py:30-36): uploads the weights, builds twiddle/mel tables. */
int wwb_create(int device, const wwb_weights* w, int precision, wwb_ctx** out);
int wwb_destroy(wwb_ctx* ctx);
/* WWB_PREC_TC / TC_FAST are refused (WWB_ERR_ARG, the ctx keeps its precision) for a model whose weights cannot be
 * packed for the tensor cores: a WaveNet with a BatchNorm scale of 0 or an operand outside the fp16 range (DESIGN.md §4).
 * wwb_create refuses such a model at those precisions; it loads at WWB_PREC_F32. */
int wwb_set_precision(wwb_ctx* ctx, int precision);
int wwb_sync(wwb_ctx* ctx, void* stream);

/* frames a stream of n_samples yields: 0 if n < 512 else (n-512)/160+1
 * (utils/tf_lite/filter.py:50-55). */
int64_t wwb_num_frames(int64_t n_samples);
/* windows of length L hopping `hop` frames over n_frames (utils/evaluate_models.py:66-73) */
int64_t wwb_num_windows(const wwb_ctx* ctx, int64_t n_frames, int hop);
/* Scheduling hint for callers that feed wwb_posteriors / wwb_pipeline in slices of streams (e.g. to overlap host->device
 * copies with compute): slices whose stream count is a multiple of the returned granule fill whole waves of the
 * persistent kernels (CRNN: strip tiles per stream against the SM count).  1 if there is no preference.
 * No reference counterpart (the TFLite path is batch-1). */
int64_t wwb_stream_granule(const wwb_ctx* ctx, int64_t n_frames, int hop);

/* K1 filter.  Replaces Filter.filter_frame / WakewordTrigger._sample+_analyze+_filter
 * (utils/tf_lite/filter.py:38-75, spokestack/wakeword/tflite.py:148-191) for whole
 * streams: pcm[s, 0:n_samples] (row pitch `pitch_samples`) -> mel[s, f, 0:40],
 * f < wwb_num_frames(n_samples), frame f = samples [160f, 160f+512).
 * int16 input is scaled by 1/32767 and clipped (wakeword/tflite.py:150-151); float
 * input is taken as is (evaluate_models.py:46).  Pre-emphasis y[n]=x[n]-a*x[n-1] with
 * x[-1] = 0 (wakeword/tflite.py:156-158). */
int wwb_filter(wwb_ctx* ctx, const void* pcm_dev, int pcm_dtype, int64_t n_streams,
               int64_t n_samples, int64_t pitch_samples, float pre_emphasis,
               float* mel_dev, void* stream);

/* filter.tflite alone, as the reference invokes it (wakeword/tflite.py:181-184,
 * utils/tf_lite/filter.py:70-75): |rFFT| magnitudes [B,257] -> mel [B,40]. */
int wwb_mel_from_magnitude(wwb_ctx* ctx, const float* mag_dev, int64_t n_frames, float* mel_dev,
                           void* stream);

/* encode.tflite on a batch: mel windows [B, L, 40] -> CRNN [B,64] | WaveNet [B,L,32]
 * (wakeword/tflite.py:193-209, evaluate_models.py:76-79,83-85). */
int wwb_encode(wwb_ctx* ctx, const float* mel_windows_dev, int64_t n_windows,
               float* enc_dev, void* stream);
/* detect.tflite on a batch: enc -> [B, n_out] (wakeword/tflite.py:217-231). */
int wwb_detect(wwb_ctx* ctx, const float* enc_dev, int64_t n_windows, float* out_dev,
               void* stream);

/* Fused encode+detect over sliding windows of per-stream mel sequences:
 * window j of stream s = mel[s, j*hop : j*hop+L, :]; post[s, j] = wake-class
 * probability (out[...,-1]; SURVEY.md §8 N1).  n_win = wwb_num_windows(n_frames, hop).
 * hop=2 is get_posterior (evaluate_models.py:42,70-86), hop=1 the streaming trigger,
 * n_frames == L the batch-of-clips path (evaluate_tf_lite_opts.py:49-69). */
int wwb_posteriors(wwb_ctx* ctx, const float* mel_dev, int64_t n_streams, int64_t n_frames,
                   int hop, float* post_dev, void* stream);

/* filter -> encode -> detect in one call, device buffers (mel kept in ctx workspace). */
int wwb_pipeline(wwb_ctx* ctx, const void* pcm_dev, int pcm_dtype, int64_t n_streams,
                 int64_t n_samples, int64_t pitch_samples, float pre_emphasis, int hop,
                 float* post_dev, void* stream);
/* same through HOST buffers - the call that replaces TFLiteModel.__call__'s copy-in / invoke /
 * copy-out (spokestack/models/tensorflow.py:33-51) for a batch of streams: H2D of the PCM in
 * three slices overlapped with the kernels, D2H of the posteriors, sync.  Host buffers that
 * are not page-locked are registered on first use (cached per address range). */
int wwb_pipeline_host(wwb_ctx* ctx, const void* pcm_host, int pcm_dtype, int64_t n_streams,
                      int64_t n_samples, float pre_emphasis, int hop, float* post_host);
/* Asynchronous form for sweeps (utils/evaluate_models.py:280-327 runs both model types over
 * the same audio): ONE host->device copy and ONE filter pass feed n_ctx models (ctxs[0] runs
 * the filter and owns the pipeline; all ctxs on one device).  Per model m: posteriors
 * post_host[m] [n_streams, n_win_m] and, if thr_host != NULL, the FAR rising-edge counts
 * (every stream one trajectory, 30-tap smoothing) and the FRR per-stream-max counts
 * (evaluate_models.py:183-218) as int64 [n_thr] each; any output pointer may be NULL.
 * Returns once the work is enqueued; up to two jobs may be in flight (the copy of job k+1
 * overlaps the kernels of job k).  wwb_sweep_wait blocks until the OLDEST job's results
 * are in host memory.  Input and output buffers must stay valid until then. */
int wwb_sweep_submit(wwb_ctx* const* ctxs, int n_ctx, const void* pcm_host, int pcm_dtype,
                     int64_t n_streams, int64_t n_samples, float pre_emphasis, int hop,
                     const double* thr_host, int n_thr, float* const* post_host,
                     int64_t* const* far_counts_host, int64_t* const* frr_counts_host);
int wwb_sweep_wait(wwb_ctx* ctx0);
/* page-locked host memory for the *_host entry points (cudaHostAlloc / cudaFreeHost) */
int wwb_host_alloc(void** out, size_t bytes);
int wwb_host_free(void* p);

/* FAR/FRR numerators (evaluate_models.py:183-218, plot_eval_models.py:84-129).
 * post[seg_off[i] : seg_off[i+1]] is segment i (clip or trajectory).
 * WWB_COUNT_FRR_MAX  : counts[t] += #segments whose max posterior > thr[t]
 * WWB_COUNT_FAR_EDGES: each segment is smoothed by a `smooth`-tap mean ('same',
 *     zero-extended, fp64) and counts[t] += rising edges of (smoothed > thr[t]).
 * thresholds fp64 [n_thr], ascending (np.arange); counts int64 [n_thr] (overwritten);
 * n_total = seg_off[n_segments].  halo_lo/halo_hi (int32 [n_segments], may be NULL):
 * the first/last posteriors of a segment that are context only — used by the smoothing
 * and as "previous sample" but not counted — so one long trajectory can be sharded into
 * time chunks (>= 16 before, >= 14 after) and the per-chunk counts simply add up. */
int wwb_eval_counts(wwb_ctx* ctx, const float* post_dev, const int64_t* seg_off_dev,
                    int64_t n_segments, const int32_t* halo_lo_dev, const int32_t* halo_hi_dev,
                    int64_t n_total, const double* thr_dev, int n_thr, int mode, int smooth,
                    int64_t* counts_dev, void* stream);

/* ---- many-stream streaming trigger (WakewordTrigger.__call__, wakeword/tflite.py:123-246)
 * State per stream lives in HBM: unread PCM tail (<512+chunk), previous sample, mel
 * ring [L(+chunk frames),40] pre-filled with 0.0 (:102), posterior max, active latch,
 * previous is_speech.  */
int wwb_stream_alloc(wwb_ctx* ctx, int64_t max_streams, int64_t max_chunk_samples);
/* One chunk of `n` samples for each of n_streams streams (pcm_dev [n_streams, n], int16).
 * is_speech/is_active uint8 [n_streams] (context.is_speech / context.is_active as seen
 * by the trigger); post_out [n_streams, max_frames] receives the posteriors of the
 * frames analysed in this call (NaN where none), n_post_out[s] their count;
 * trigger_out[s]=1 if a posterior exceeded `threshold` (strict >, :235) while the
 * stream was inactive; post_max_out[s] the running maximum (:233-234). */
int wwb_stream_push(wwb_ctx* ctx, const int16_t* pcm_dev, int64_t n_streams, int64_t n,
                    const uint8_t* is_speech_dev, const uint8_t* is_active_dev, float pre_emphasis,
                    float threshold, float* post_out_dev, int32_t* n_post_out_dev,
                    uint8_t* trigger_out_dev, float* post_max_out_dev, void* stream);
/* The same for a server's traffic: one chunk for each of n_ids streams, named by slot id, each
 * chunk of its own length.  Only the named slots advance, and the work is proportional to n_ids,
 * not to max_streams.
 * ids_host int32 [n_ids] (host): distinct slots in [0, max_streams), any order.  A slot may appear
 *   once per call: to feed a stream more samples, push again.
 * len_host int32 [n_ids] (host): chunk lengths, each in [1, max_chunk_samples].
 * pcm_dev int16: the chunks packed back to back in ids order (chunk i starts at sum(len[:i])).
 * is_speech_dev / is_active_dev uint8 [n_ids], per entry (NULL = speech / inactive, as above).
 * Outputs are per ENTRY i, not per slot: post_out [n_ids, max_frames] (NaN tail), n_post_out,
 * trigger_out, post_max_out [n_ids].  Slots not named are not touched.
 * The tables are checked before any device work; a rejected call changes no state (WWB_ERR_STATE:
 * no wwb_stream_alloc, n_ids outside [1, max_streams], an id out of range or repeated, a length out
 * of range, a filter-only ctx; WWB_ERR_ARG: NULL tables or PCM).  The library turns the lengths
 * into offsets and copies ids and offsets to the device on `stream` through page-locked staging
 * owned by ctx, so the call does not wait for earlier pushes. */
int wwb_stream_push_indexed(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const int32_t* len_host,
                            const int16_t* pcm_dev, const uint8_t* is_speech_dev, const uint8_t* is_active_dev,
                            float pre_emphasis, float threshold, float* post_out_dev, int32_t* n_post_out_dev,
                            uint8_t* trigger_out_dev, float* post_max_out_dev, void* stream);
int wwb_stream_max_frames(const wwb_ctx* ctx);
/* WakewordTrigger.reset (:241-246) for the streams whose mask byte is non-zero (NULL = all). */
int wwb_stream_reset(wwb_ctx* ctx, const uint8_t* mask_dev, int64_t n_streams, void* stream);

/* ---- the pipeline stages around the trigger, per stream on the device (SpeechPipeline._dispatch,
 * spokestack/pipeline.py:25-28): VAD rise/fall debounce (spokestack/vad/webrtc.py:52-77; the raw
 * per-frame decision of the webrtcvad C extension is an input) -> wake-word trigger (is_speech /
 * is_active taken from this state; a trigger activates the stream) -> ActivationTimeout
 * (spokestack/activation_timeout.py:25-38).  Needs wwb_stream_alloc first; delays in ms as the
 * reference's constructors take them (rise/fall: integer division by frame_width; min/max_active:
 * true division). */
int wwb_context_alloc(wwb_ctx* ctx, int frame_width_ms, int vad_rise_delay_ms, int vad_fall_delay_ms,
                      int min_active_ms, int max_active_ms);
/* One dispatch for every stream: pcm_dev [n_streams, n] int16 (n = one pipeline frame, e.g. 320),
 * vad_raw_dev uint8 [n_streams] (NULL = speech).  Outputs (device, any may be NULL): posteriors
 * analysed in this call as in wwb_stream_push, and per stream context.is_speech / context.is_active
 * after the three stages plus the activation / deactivation events of this call. */
int wwb_context_step(wwb_ctx* ctx, const int16_t* pcm_dev, int64_t n_streams, int64_t n,
                     const uint8_t* vad_raw_dev, float pre_emphasis, float threshold,
                     float* post_out_dev, int32_t* n_post_out_dev, float* post_max_out_dev,
                     uint8_t* is_speech_out_dev, uint8_t* is_active_out_dev,
                     uint8_t* activated_out_dev, uint8_t* deactivated_out_dev, void* stream);
/* wwb_context_step for the slots named in ids_host, with the tables, their checks and the per-entry
 * outputs of wwb_stream_push_indexed: one SpeechPipeline dispatch for each named slot, vad_raw_dev
 * uint8 [n_ids] per entry (NULL = speech), every output per entry.  Slots not named are not
 * touched.  Needs wwb_context_alloc (else WWB_ERR_STATE). */
int wwb_context_step_indexed(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const int32_t* len_host,
                             const int16_t* pcm_dev, const uint8_t* vad_raw_dev, float pre_emphasis, float threshold,
                             float* post_out_dev, int32_t* n_post_out_dev, float* post_max_out_dev,
                             uint8_t* is_speech_out_dev, uint8_t* is_active_out_dev,
                             uint8_t* activated_out_dev, uint8_t* deactivated_out_dev, void* stream);
/* all stages of all streams back to their initial state */
int wwb_context_reset(wwb_ctx* ctx, void* stream);

/* ---- stream state records: a stream's state out of its slot and back, to park an idle session, move it to another
 * slot, context or GPU, or rewind it.  One record per stream, of wwb_stream_state_bytes(ctx) bytes; its layout does not
 * depend on the capacity, max_chunk, precision or device of the ctx that wrote it:
 *   wwb_stream_state_header                       48 bytes
 *   float pending[WWB_STREAM_STATE_PENDING]       the pre-emphasised samples not yet consumed (WakewordTrigger's sample
 *                                                 ring); entries n_pending and beyond are 0
 *   float mel[mel_length][40]                     the frame window (frame_window), oldest row first; all 0 for a stream
 *                                                 never pushed or just reset
 * Record size: 48 + 4*512 + 160*mel_length bytes (26 256 for CRNN, 31 216 for WaveNet). */
#define WWB_STREAM_STATE_MAGIC 0x53425757u /* "WWBS" */
#define WWB_STREAM_STATE_VERSION 1         /* of the record layout (not WWB_VERSION) */
#define WWB_STREAM_STATE_PENDING 512
#define WWB_STREAM_STATE_PIPELINE 1u /* flags bit 0: the pipeline fields hold state (wwb_context_alloc) */
typedef struct {
  uint32_t magic;       /* WWB_STREAM_STATE_MAGIC */
  uint16_t version;     /* WWB_STREAM_STATE_VERSION */
  uint16_t flags;       /* WWB_STREAM_STATE_PIPELINE or 0; other bits 0 */
  int32_t kind;         /* WWB_MODEL_* of the ctx that wrote it */
  int32_t mel_length;   /* L */
  int32_t n_pending;    /* [0, 511] */
  float prev_sample;    /* last sample consumed, raw (int16 / 32767, clipped): the pre-emphasis state */
  float post_max;       /* running posterior maximum */
  uint8_t was_speech;   /* is_speech of the stream's last push */
  uint8_t is_speech;    /* pipeline: SpeechContext.is_speech (VAD debounce output) */
  uint8_t is_active;    /* pipeline: SpeechContext.is_active */
  uint8_t t_is_speech;  /* pipeline: ActivationTimeout._is_speech */
  int32_t run_value;    /* pipeline: VoiceActivityDetector._run_value */
  int32_t run_length;   /* pipeline: VoiceActivityDetector._run_length */
  int32_t active_length;/* pipeline: ActivationTimeout._active_length */
  uint32_t reserved;    /* 0 */
} wwb_stream_state_header;
/* wwb_stream_import's reason codes (status_dev[1]) */
enum {
  WWB_RECORD_OK = 0,
  WWB_RECORD_BAD_MAGIC = 1,
  WWB_RECORD_BAD_VERSION = 2,
  WWB_RECORD_BAD_FLAGS = 3,   /* an unknown flag bit */
  WWB_RECORD_BAD_KIND = 4,    /* written by a ctx of another model kind */
  WWB_RECORD_BAD_LENGTH = 5,  /* mel_length differs from this ctx's */
  WWB_RECORD_BAD_PENDING = 6  /* n_pending outside [0, 511] */
};
/* record size in bytes; 0 without wwb_stream_alloc or on a filter-only ctx */
int64_t wwb_stream_state_bytes(const wwb_ctx* ctx);
/* Gathers the state of the slots named in ids_host (host table, the rules of wwb_stream_push_indexed: distinct, in
 * [0, max_streams), 1 <= n_ids <= max_streams) into records_dev (16-byte aligned): entry i's record at
 * records_dev + i * wwb_stream_state_bytes(ctx).  Stream-ordered like the pushes; the slots are not modified.  Without
 * wwb_context_alloc the flags are 0 and the pipeline fields 0.  A rejected call changes nothing (WWB_ERR_STATE: the id
 * checks of the pushes, no wwb_stream_alloc, a filter-only ctx; WWB_ERR_ARG: NULL or misaligned buffers). */
int wwb_stream_export(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, void* records_dev, void* stream);
/* Scatters n_ids records (as written by wwb_stream_export, on this ctx's device) into the slots named in ids_host, all or
 * nothing: every record's magic, version, flags, kind, mel_length and n_pending are checked on the device first, and
 * status_dev int32[2] receives {0, 0} when the records were applied, else {1 + the lowest bad entry, WWB_RECORD_*} and no
 * slot is touched.  An applied record's window becomes ring rows 0..L-1 of its slot (the rest of the ring is zeroed); the
 * pipeline fields are applied when the ctx has pipeline state, and set to their initial values there when the record has
 * none.  The pipeline's delays are per ctx and not carried.  Host-side checks as wwb_stream_export. */
int wwb_stream_import(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const void* records_dev, int32_t* status_dev,
                      void* stream);

/* number of kernels this library has launched on ctx since creation (bench accounting) */
int64_t wwb_launch_count(const wwb_ctx* ctx);
/* development aid: device buffer (>= 8 KB, zeroed) that instrumented kernels fill with
 * clock64() timelines of their first work item; NULL disables it (default). */
int wwb_debug_buffer(wwb_ctx* ctx, void* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* WWB200_H */
