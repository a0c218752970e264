// Per-stream pipeline state machine on the device (SURVEY.md 8f row 2): the stages the reference's SpeechPipeline
// dispatches around the wake-word trigger, for many streams at once, state in HBM.
//
//   vad debounce       spokestack/vad/webrtc.py:52-77   raw per-frame decision (input: the webrtcvad C extension is out of
//                                                       scope) -> run-length rise / fall delays -> context.is_speech
//   wake-word trigger  spokestack/wakeword/tflite.py:123-246   wwb_stream_push with is_speech / is_active taken from this
//                                                       state; a trigger sets context.is_active
//   activation timeout spokestack/activation_timeout.py:25-38  counts active frames; after min_active a VAD fall or
//                                                       max_active deactivates
// One step = one SpeechPipeline._dispatch (spokestack/pipeline.py:25-28) for every stream: two one-thread-per-stream
// kernels around the trigger stages.  Both run over the entries i of the push, with the state of slot ids[i] (ids NULL =
// i) and every per-entry input and output at i.  A step runs one streaming push per trigger stage, each on its own ctx,
// with context_chain_kernel after each; the pipeline state and this scratch are stage 0's.  wwb_context_step is a chain
// of one stage without activated_by, where context_chain_kernel would change no state and is not launched.
#include "common.cuh"

namespace wwb {

__global__ void context_vad_kernel(ContextState C, const int32_t* __restrict__ ids, const uint8_t* __restrict__ vad_raw,
                                   int64_t S) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S) return;
  const int64_t s = ids ? (int64_t)ids[i] : i;
  const int raw = vad_raw ? (vad_raw[i] != 0) : 1;
  int rv = C.run_value[s], rl = C.run_length[s];
  if (raw == rv) {
    ++rl;
  } else {
    rv = raw;
    rl = 1;
  }
  C.run_value[s] = rv;
  C.run_length[s] = rl;
  int sp = C.is_speech[s];
  if (rv != sp) {
    if (rv && rl >= C.rise_length) sp = 1;
    if (!rv && rl >= C.fall_length) sp = 0;
  }
  C.is_speech[s] = (uint8_t)sp;
  C.e_is_speech[i] = (uint8_t)sp;   // what the push of this step sees
  C.e_is_active[i] = C.is_active[s];
}

__global__ void context_timeout_kernel(ContextState C, const int32_t* __restrict__ ids, const uint8_t* __restrict__ trigger,
                                       int64_t S, uint8_t* __restrict__ is_speech_out, uint8_t* __restrict__ is_active_out,
                                       uint8_t* __restrict__ activated_out, uint8_t* __restrict__ deactivated_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S) return;
  const int64_t s = ids ? (int64_t)ids[i] : i;
  const int sp = C.is_speech[s];
  int act = C.is_active[s];
  const int activated = trigger[i] && !act;       // wakeword/tflite.py:235-239
  act |= activated;
  const int vad_fall = C.t_is_speech[s] && !sp;   // activation_timeout.py:32-33
  C.t_is_speech[s] = (uint8_t)sp;
  int deactivated = 0;
  if (act) {
    const int len = C.active_length[s] + 1;
    C.active_length[s] = len;
    if ((float)len > C.min_active && (vad_fall || (float)len > C.max_active)) {
      C.active_length[s] = 0;
      act = 0;
      deactivated = 1;
    }
  }
  C.is_active[s] = (uint8_t)act;
  if (is_speech_out) is_speech_out[i] = (uint8_t)sp;
  if (is_active_out) is_active_out[i] = (uint8_t)act;
  if (activated_out) activated_out[i] = (uint8_t)activated;
  if (deactivated_out) deactivated_out[i] = (uint8_t)deactivated;
}

// Between the trigger stages of wwb_context_step_chain, after stage k's push wrote its trigger into C.trigger: a trigger
// activates the stream for the stages after k (e_is_active is their is_active input) and names k as the stage that
// activated it.  A stage triggers only while its is_active input is 0, so at most one stage per step does.  After the last
// stage C.trigger holds the merged trigger that context_timeout_kernel reads.
__global__ void context_chain_kernel(ContextState C, int64_t S, int k, bool last, int8_t* __restrict__ activated_by_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S) return;
  const bool trig = C.trigger[i] != 0;
  int by = k == 0 ? -1 : C.activated_by[i];
  if (trig) {
    by = k;
    C.e_is_active[i] = 1;
  }
  if (last) {
    C.trigger[i] = by >= 0 ? 1 : 0;
    if (activated_by_out) activated_by_out[i] = (int8_t)by;
  } else {
    C.activated_by[i] = (int8_t)by;
  }
}

int launch_context_chain(wwb_ctx* ctx, int64_t S, int k, bool last, int8_t* activated_by_out, cudaStream_t st) {
  context_chain_kernel<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(ctx->cs, S, k, last, activated_by_out);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_context_vad(wwb_ctx* ctx, const int32_t* ids, const uint8_t* vad_raw, int64_t S, cudaStream_t st) {
  context_vad_kernel<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(ctx->cs, ids, vad_raw, S);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_context_timeout(wwb_ctx* ctx, const int32_t* ids, const uint8_t* trigger, int64_t S, uint8_t* is_speech_out,
                           uint8_t* is_active_out, uint8_t* activated_out, uint8_t* deactivated_out, cudaStream_t st) {
  context_timeout_kernel<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(ctx->cs, ids, trigger, S, is_speech_out, is_active_out,
                                                                      activated_out, deactivated_out);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb
