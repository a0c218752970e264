// Shared declarations of the wwb200 library (internal).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/wwb200.h"

namespace wwb {

constexpr int kFFT = 512;
constexpr int kHop = 160;
constexpr int kBins = 257;
constexpr int kMel = 40;

// ---- mel projection in CSR-by-segment form (built on the host from the dense matrix) ----
// A "segment" is up to kSegTaps consecutive non-zeros of one mel band; a band owns a
// contiguous range of segments so partial sums are combined in a fixed order.
constexpr int kSegTaps = 8;
constexpr int kMaxSeg = 128;   // segments the filter kernels hold in shared memory (wwb_create refuses more)
struct MelTables {
  int n_seg = 0;          // total segments
  int* seg_band = nullptr;   // [n_seg]
  int* seg_first = nullptr;  // [n_seg] index into tap arrays
  int* seg_count = nullptr;  // [n_seg]
  int* band_seg0 = nullptr;  // [kMel+1] first segment of each band
  int* tap_bin = nullptr;    // [n_tap]
  float* tap_w = nullptr;    // [n_tap]
  float* bias = nullptr;     // [kMel]
  int n_tap = 0;
};

struct CrnnWeights {   // device copies, fp32, layouts chosen for the kernels
  float* conv_w = nullptr;   // [100][32]  (tap = kf*20+kt, chan)   transposed for coalesced reads
  float* conv_b = nullptr;   // [32]
  float* gru_w[4] = {};      // [in][96]   transposed: k-major rows
  float* gru_u[4] = {};      // [32][96]
  float* gru_bi[4] = {};     // [96]
  float* gru_br[4] = {};     // [96]
  float* det1_w = nullptr;   // [64][64] transposed [in][out]
  float* det1_b = nullptr;
  float* det2_w = nullptr;   // [n_out][64]
  float* det2_b = nullptr;
  unsigned char* tc_conv = nullptr;   // crnn_tc.cu: packed conv weights
  unsigned char* tc_w1 = nullptr;     // crnn_tc.cu: 20 packed k-slices of the layer-1 input projection
  unsigned char* tc_u[2] = {};        // crnn_tc.cu: packed recurrent weights, both directions, per layer
  float* tc_bh[2] = {};               // [2][32] recurrent bias of the candidate gate, per layer
  float* tc_bi[2] = {};               // [192] b_in with the z/r parts of the recurrent bias folded in
  unsigned char* tc_w2 = nullptr;     // crnn_tc.cu: layer-2 input projection packed for the fused layer-2 kernel
  float* tc_bi2 = nullptr;            // [2][96] tc_bi[1] in that kernel's accumulator column order
};

struct WavenetWeights {
  float* in_w = nullptr;     // [40][16] transposed
  float* in_b = nullptr;     // [16]
  float* bn_mul = nullptr;   // [24][16]
  float* bn_add = nullptr;
  int dilation[24] = {};
  float* gate_w = nullptr;   // [24][48][32]: k = tap*16+in ; n<16 tanh, n>=16 sigmoid
  float* gate_b = nullptr;   // [24][32]
  float* rs_w = nullptr;     // [24][16][48]: n<16 residual (zeros for block 23), n>=16 skip
  float* rs_b = nullptr;     // [24][48]
  float* det1_w = nullptr;   // [32][32] transposed [in][out]
  float* det1_b = nullptr;
  float* det2_w = nullptr;   // [2][32]
  float* det2_b = nullptr;
  unsigned char* tc_blocks = nullptr;   // tensor-core path: per-block packed weights (wavenet_tc.cu)
  unsigned char* tc_head = nullptr;     // resident head blob
  float h_det1_b[32] = {}, h_det2_w[64] = {}, h_det2_b[2] = {};   // host copies: kernel parameters of the tensor-core path
};

struct StreamState {
  int64_t max_streams = 0;
  int64_t max_chunk = 0;
  int pend_cap = 0;      // samples of pending PCM kept per stream
  int max_frames = 0;    // frames a single push can complete
  int ring = 0;          // mel ring rows per stream (L + max_frames)
  float* pending = nullptr;     // [S, pend_cap]
  int32_t* n_pending = nullptr; // [S]
  float* prev_sample = nullptr; // [S]
  float* mel_ring = nullptr;    // [S, ring, 40]
  int32_t* ring_head = nullptr; // [S] index of the oldest row of the current window
  float* post_max = nullptr;    // [S]
  uint8_t* was_speech = nullptr;// [S]
  // per-push scratch
  int32_t* n_new = nullptr;     // [S] frames analysed this push
  int32_t* win_stream = nullptr;// [S*max_frames]
  int32_t* win_start = nullptr; // [S*max_frames]
  int32_t* win_slot = nullptr;  // [S] first window slot of the stream in this push
  int32_t* n_win = nullptr;     // [1]
  float* win_post = nullptr;    // [S*max_frames]
  // tables of a call over n entries: [0, n) slot of each entry, then for an indexed push [n, 2n] the exclusive prefix
  // sum of the chunk lengths, for wwb_stream_set_options [n, 2n) the thresholds' bits and [2n, 3n) the listening flags
  int32_t* tables = nullptr;    // [stage_words(S)]
  // wwb_stream_import's check: [0] the lowest bad entry and its reason, [1] finished blocks (both 0 between calls)
  unsigned long long* import_check = nullptr;
};

// per-stream state of the pipeline stages around the trigger (context.cu)
struct ContextState {
  int64_t max_streams = 0;
  int rise_length = 0, fall_length = 0;   // vad_rise_delay // frame_width, vad_fall_delay // frame_width (frames)
  float min_active = 0.f, max_active = 0.f;   // min_active / frame_width, max_active / frame_width (frames, fractional)
  int32_t* run_value = nullptr;   // [S] VoiceActivityDetector._run_value
  int32_t* run_length = nullptr;  // [S]
  uint8_t* is_speech = nullptr;   // [S] SpeechContext.is_speech
  uint8_t* is_active = nullptr;   // [S] SpeechContext.is_active
  int32_t* active_length = nullptr;  // [S] ActivationTimeout._active_length
  uint8_t* t_is_speech = nullptr;    // [S] ActivationTimeout._is_speech
  uint8_t* trigger = nullptr;        // [S] scratch: the push's trigger output
  uint8_t* e_is_speech = nullptr;    // [S] scratch: is_speech / is_active per entry of the push (context_vad_kernel)
  uint8_t* e_is_active = nullptr;
  int8_t* activated_by = nullptr;    // [S] scratch of a trigger chain: the stage that triggered so far, -1 if none
};

// words of st.tables and of each host staging slot for S slots: room for the largest table above
inline int64_t stage_words(int64_t S) { return 3 * S + 1; }

// Per-slot trigger options (wwb_stream_set_options), allocated with the stream state.  Slot configuration, not session
// state: resets, imports and records leave them alone.  Kept out of StreamState so that the kernels that take a
// StreamState by value and do not read the options keep their parameter layout.
struct SlotOptions {
  float* threshold = nullptr;   // [S] NaN: the threshold the push or step passes
  uint8_t* listening = nullptr; // [S] 0: every push treats the slot as is_active
};

}  // namespace wwb

struct wwb_ctx {
  int device = 0;
  int kind = 0;
  int L = 0;          // mel_length
  int n_out = 1;
  int precision = WWB_PREC_F32;
  std::string tc_refused;   // why the model has no tensor-core weights (empty: it has them)
  int sm_count = 148;
  float mel_floor = 1e-5f, mel_log_offset = 0.f, mel_scale = 0.5f;
  std::vector<float> mel_w_host, mel_b_host;   // the filter's mel_w [40][257] and mel_b [40] as given (a sweep's models share one filter pass)
  wwb::MelTables mel;
  double* hann = nullptr;      // [512] 0.5 * np.hanning(512), fp64 (fft64.cuh)
  double2* tw256 = nullptr;    // [256] W256^k
  double2* tw512 = nullptr;    // [256] W512^k
  wwb::CrnnWeights crnn;
  wwb::WavenetWeights wn;
  wwb::StreamState st;
  wwb::ContextState cs;
  wwb::SlotOptions opt;
  // growable workspaces
  void* ws[8] = {};
  size_t ws_bytes[8] = {};
  int64_t launches = 0;
  void* debug_buf = nullptr;   // optional device buffer for kernel timeline dumps (wwb_debug_buffer)
  void* host_pipe = nullptr;   // host-buffer pipeline state (host_pipeline.cu), created on first use
  // host side of st.tables (indexed pushes, records, slot options): two page-locked staging slots of stage_words(S)
  // words, each guarded by an event recorded after its copy, and the duplicate-id marks (all 0 between calls)
  int32_t* stage_host[2] = {};
  cudaEvent_t stage_done[2] = {};
  int stage_next = 0;
  std::vector<uint8_t> id_seen;
  std::string err;
  std::vector<void*> owned;    // device allocations to free
};

namespace wwb {

extern std::string g_create_error;

int fail(wwb_ctx* ctx, int code, const char* fmt, ...);
void host_pipe_destroy(wwb_ctx* ctx);

#define WWB_CUDA(ctx, expr)                                                               \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess)                                                                \
      return wwb::fail(ctx, WWB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                 \
                       cudaGetErrorString(_e), __FILE__, __LINE__);                       \
  } while (0)

#define WWB_CHECK_LAUNCH(ctx)                                                             \
  do {                                                                                    \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess)                                                                \
      return wwb::fail(ctx, WWB_ERR_CUDA, "kernel launch failed: %s (%s:%d)",             \
                       cudaGetErrorString(_e), __FILE__, __LINE__);                       \
    (ctx)->launches++;                                                                    \
  } while (0)

// workspace slot `i` of at least `bytes`
int workspace(wwb_ctx* ctx, int i, size_t bytes, void** out);

// kernels' host launchers (one translation unit each)
int launch_filter(wwb_ctx* ctx, const void* pcm, int dtype, int64_t S, int64_t N, int64_t pitch,
                  float a, float* mel, cudaStream_t st);
int launch_mel_from_mag(wwb_ctx* ctx, const float* mag, int64_t B, float* mel, cudaStream_t st);
// Streaming kernels run over the entries i of a push.  ids (device, NULL = identity) names entry i's stream slot; off
// (device, NULL = i * n) is where its chunk starts in pcm, of length off[i+1] - off[i].
int launch_stream_filter(wwb_ctx* ctx, const int16_t* pcm, int64_t S, int64_t n, const int32_t* ids, const int32_t* off,
                         const uint8_t* is_speech, const uint8_t* is_active, float a,
                         cudaStream_t st);
int launch_stream_finish(wwb_ctx* ctx, int64_t S, const int32_t* ids, const uint8_t* is_speech, const uint8_t* is_active,
                         float threshold, float* post_out, int32_t* n_post_out, uint8_t* trigger_out,
                         float* post_max_out, cudaStream_t st);
int launch_stream_reset(wwb_ctx* ctx, const uint8_t* mask, int64_t S, cudaStream_t st);
// wwb_stream_set_options' scatter of the n entries staged in st.tables (ids, thresholds, listening flags)
int launch_stream_options(wwb_ctx* ctx, int64_t n, bool threshold, bool listening, cudaStream_t st);
// stream state records (stream_state.cu): ids is the device id table of n entries
int64_t stream_state_bytes(int L);
int launch_stream_export(wwb_ctx* ctx, const int32_t* ids, int64_t n, void* records, cudaStream_t st);
// an import: the check of one ctx's records into status int32[2] (stage < 0), or for stage `stage` of a chain into
// status int32[3] (kept if an earlier stage's check failed), then the scatter, which does nothing unless status[0] is 0
int launch_stream_check_stage(wwb_ctx* ctx, int64_t n, const void* records, int32_t* status, int stage, cudaStream_t st);
int launch_stream_scatter(wwb_ctx* ctx, const int32_t* ids, int64_t n, const void* records, const int32_t* status,
                          cudaStream_t st);
int launch_context_vad(wwb_ctx* ctx, const int32_t* ids, const uint8_t* vad_raw, int64_t S, cudaStream_t st);
// after trigger stage k of a chain (its trigger in cs.trigger): see context_chain_kernel
int launch_context_chain(wwb_ctx* ctx, int64_t S, int k, bool last, int8_t* activated_by_out, cudaStream_t st);
int launch_context_timeout(wwb_ctx* ctx, const int32_t* ids, const uint8_t* trigger, int64_t S, uint8_t* is_speech_out,
                           uint8_t* is_active_out, uint8_t* activated_out, uint8_t* deactivated_out, cudaStream_t st);

// window addressing shared by the encoders: window b reads rows
//   mel + (stream(b)*ring + (start(b)+t) % ring) * 40,  t = 0..L-1
struct WinMap {
  const float* mel;
  const int32_t* win_stream;  // optional explicit lists
  const int32_t* win_start;
  const int32_t* n_win_dev;   // optional device-side window count (streaming)
  int64_t n_win;              // host-side count (upper bound when n_win_dev is set)
  int64_t b0;                 // added to the window index (batch chunking)
  int win_per_stream;         // regular grid: stream = b / wps, start = (b % wps)*hop
  int hop;
  int ring;                   // rows per stream
  int64_t n_streams;          // streams the windows name (x0 of the WaveNet tensor-core path has n_streams * ring rows)
  const int32_t* stream_slot; // optional: stream s of the windows is stream stream_slot[s] of `mel` (indexed pushes)
};

int crnn_simt_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out,
                         float* post, cudaStream_t st);
int crnn_simt_detect(wwb_ctx* ctx, const float* enc, int64_t B, float* out, cudaStream_t st);
// Time geometry of the CRNN conv (kernel 20, stride 8, TF SAME) over a window of L frames: T = ceil(L / 8) columns and
// 8T + 12 - L zero frames, pad_lo of them before the window.  Column t covers window frames 8t - pad_lo .. + 19; bit t
// of padmask is set if that touches the padding.  Columns 0 and T - 1 always do, column 1 too when pad_lo = 9
// (L = 1, 2 mod 8) and column T - 2 when pad_hi >= 9 (L = 1, 2, 3 mod 8).  For L = 151: T = 19, pad 6 / 7, columns 0, 18.
struct CrnnGeom {
  int T, pad_lo;
  uint32_t padmask;
};
constexpr int kCrnnMinL = 17, kCrnnMaxL = 256;   // T = 3 .. 32 (padmask holds one bit per column)
inline CrnnGeom crnn_geom(int L) {
  CrnnGeom g;
  g.T = (L + 7) / 8;
  g.pad_lo = (8 * g.T + 12 - L) / 2;
  g.padmask = 0;
  for (int t = 0; t < g.T; ++t)
    if (8 * t - g.pad_lo < 0 || 8 * t - g.pad_lo + 19 >= L) g.padmask |= 1u << t;
  return g;
}
// conv-weight variant of column t in the shared-column path: 0 = all taps (interior columns), 1.. = the padded columns
// in order, each with the taps that meet the padding zeroed
__host__ __device__ __forceinline__ int crnn_variant(uint32_t padmask, int t) {
#ifdef __CUDA_ARCH__
  return (padmask >> t) & 1u ? 1 + __popc(padmask & ((1u << t) - 1u)) : 0;
#else
  return (padmask >> t) & 1u ? 1 + __builtin_popcount(padmask & ((1u << t) - 1u)) : 0;
#endif
}
std::vector<unsigned char> crnn_pack_conv(const float* conv_w, int L);
std::vector<unsigned char> crnn_pack_w1(const float* w_nk);
// shared-column geometry of a sliding-window batch (crnn_tc.cu)
struct CrnnShare {
  int q, nsp, Mp, F, wps, tps;
  int64_t n_streams;
  int T;              // conv columns per window
  uint32_t padmask;   // padded columns (CrnnGeom); the variants are 0 (unless every column is padded) and 1 .. popc
};
bool crnn_share_plan(const WinMap& wm, int L, CrnnShare* out);
int crnn_share_first_variant(const CrnnShare& g);   // 1 if every column is padded (variant 0 unused), else 0
int crnn_share_launches(const CrnnShare& g);        // front-kernel launches: one per variant in use
size_t crnn_share_xws_bytes(const CrnnShare& g, int64_t n_streams);
int crnn_front_tc(wwb_ctx* ctx, const WinMap& wm, float* xw1, cudaStream_t st, int mode = 0, const CrnnShare* g = nullptr,
                  int variant = 0);
std::vector<unsigned char> crnn_pack_u(const float* u_f, const float* u_b);
int gru_rec_tc(wwb_ctx* ctx, int layer, const float* xw, float* seq_out, float* last_out, int64_t B,
               const int32_t* n_dev, cudaStream_t st, const float* xws = nullptr, const CrnnShare* g = nullptr,
               unsigned char* seq_packed = nullptr);
std::vector<unsigned char> crnn_pack_w2(const float* w_nk);
std::vector<float> crnn_reorder_bias2(const float* bf);
size_t crnn_seq_packed_bytes(int64_t B, int T);
int gru2_fused_tc(wwb_ctx* ctx, const unsigned char* seq_packed, float* last_out, int64_t B, const int32_t* n_dev,
                  cudaStream_t st);
int wavenet_simt_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out,
                            float* post, cudaStream_t st);
int wavenet_tc_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out,
                          float* post, cudaStream_t st);
// the tensor-core operand blobs; empty if a BatchNorm scale is 0 or a packed operand is outside the fp16 range
std::vector<unsigned char> wavenet_pack_blocks(const float* gate_w, const float* gate_b, const float* rs_w,
                                               const float* rs_b, const float* bn_mul, const float* bn_add,
                                               const int* dilation);
std::vector<unsigned char> wavenet_pack_head(const float* bn_mul0, const float* bn_add0, const float* det1_w_nk,
                                             const float* det1_b, const float* det2_w, const float* det2_b);
int wavenet_simt_detect(wwb_ctx* ctx, const float* enc, int64_t B, float* out, cudaStream_t st);

int launch_eval_counts(wwb_ctx* ctx, const float* post, const int64_t* seg_off, int64_t n_seg,
                       const int32_t* halo_lo, const int32_t* halo_hi, int64_t n_total,
                       const double* thr, int n_thr, int mode, int smooth, int64_t* counts,
                       cudaStream_t st);

// win_row split in two: the window's stream / first mel row, and a row of that stream (ring-wrapped).  win_origin
// returns the stream as the windows name it (the compact entry of an indexed push); stream_row maps it to its slot.
__device__ __forceinline__ void win_origin(const WinMap& wm, int64_t b, int64_t& s, int& start) {
  b += wm.b0;
  if (wm.win_stream) {
    s = wm.win_stream[b];
    start = wm.win_start[b];
  } else {
    s = b / wm.win_per_stream;
    start = (int)(b % wm.win_per_stream) * wm.hop;
  }
}
__device__ __forceinline__ const float* stream_row(const WinMap& wm, int64_t s, int r) {
  if (r >= wm.ring) r -= wm.ring;
  if (wm.stream_slot) s = wm.stream_slot[s];
  return wm.mel + (s * wm.ring + r) * (int64_t)kMel;
}

__device__ __forceinline__ const float* win_row(const WinMap& wm, int64_t b, int t) {
  int64_t s;
  int start;
  win_origin(wm, b, s, start);
  return stream_row(wm, s, start + t);
}

}  // namespace wwb
