// K1 - fused filter kernel: PCM -> (scale/clip) -> pre-emphasis -> frames of 512 @ hop 160
// -> Hann -> 512-point real FFT (fp64) -> |.| -> 257x40 mel (sparse) -> 0.5*(ln(max(.,1e-5))+11.5129).
//
// Replaces (reference): spokestack/wakeword/tflite.py:148-191, utils/tf_lite/filter.py:38-75
// and filter.tflite.  HBM traffic is the algorithmic minimum (each PCM sample read once per chunk of a stream + 3 %
// halo, each mel value written once); the limiter is the fp64 pipe (fft64.cuh explains why the FFT is fp64:
// ~8900 fp64 instructions per frame against 64 per clock and SM), so the layout keeps that pipe fed:
//   * every WARP is an independent pipeline over chunks of one stream, two frames at a time (one per 16-lane half);
//     it owns its shared memory (sample ring, transpose buffers, magnitudes) and synchronises with __syncwarp only,
//     so the warps of an SM drift apart and one warp's staging / mel phase overlaps another's butterflies;
//   * window and twiddle factors a lane needs are the same for every frame (lane j is fixed): they live in
//     registers (fft64.cuh LaneConsts), W512^k comes from shared memory (both halves read the same address);
//   * consecutive frames overlap by 352 samples: an iteration stages only the 320 new samples of its frame pair
//     into the warp's ring (int16 -> f32 exactly as the reference converts them), prefetched one iteration ahead;
//   * magnitudes go to shared memory, the mel projection is evaluated from a segment table (<= 8 non-zeros per
//     segment, fixed summation order => deterministic results, bit-identical to mel_from_mag_kernel).
#include "common.cuh"
#include "fft64.cuh"

namespace wwb {

constexpr int F_WARPS = 12;                // independent warp pipelines per CTA (3 per scheduler; 16 KB of shared memory each)
constexpr int F_THREADS = F_WARPS * 32;    // 384 (x 168 registers = one CTA per SM)
constexpr int F_RING = 1024;               // floats per warp ring (>= 672 live samples + 320 staged ahead)
constexpr int MAGP = 272;                  // magnitude entries per warp (257 bins + zeroed padding read by padded taps)

struct MelParams {
  MelTables mt;
  float mel_floor, mel_log_offset, mel_scale;
};

struct FilterParams {
  const void* pcm;
  int64_t n_streams, n_samples, pitch;
  int64_t n_frames;        // per stream
  int item_frames;         // frames per work item (even)
  int items_per_stream;
  int64_t n_items;
  float a;                 // pre-emphasis
  float* mel;              // [S, F, 40]
  const double* hann_half; // [512] 0.5*np.hanning(512)
  const double2* tw256;    // [256] W256^k
  const double2* tw512;    // [256] W512^k
  MelParams mp;
};

struct __align__(16) FilterWarpSmem {
  float ring[F_RING];
  double2 xch[2][16 * f64::XP];
  float2 mag[MAGP];          // [bin] = (frame of half 0, frame of half 1): one 8-byte load serves both frames
  float2 partial[kMaxSeg];
};

struct __align__(16) FilterSmem {
  FilterWarpSmem w[F_WARPS];
  double2 tw512[256];
  double2 hann2[256];        // window of sample pair n (fft64.cuh)
  double2 twj[256];          // W256^(j k2) at [16 j + k2]
  // mel tables: a segment = up to 8 CONSECUTIVE bins of one band (the non-zeros of a mel band are contiguous), padded to 8
  // taps with weight 0 (fma(0, x, acc) == acc: the padded taps read the following bins / the zeroed padding); band -> segments
  float seg_w[kMaxSeg][8];
  int seg_bin0[kMaxSeg];
  int band_seg0[kMel + 1];
  float band_bias[kMel];
};

__device__ __forceinline__ float pcm_to_float(int16_t s) {
  // frame.astype(np.float32) / (2**15 - 1), np.clip(-1, 1)   (wakeword/tflite.py:150-151)
  // The correctly rounded quotient without the division subroutine: q0 = s*r, one FMA residual, one FMA correction
  // (r = fl(1/32767)); equal to IEEE s/32767 for all 65536 inputs (checked exhaustively, tests/test_host.py).
  const float r = 3.0518509447574615e-05f, f = (float)s;
  const float q0 = __fmul_rn(f, r);
  const float x = __fmaf_rn(__fmaf_rn(-q0, 32767.0f, f), r, q0);
  return fminf(fmaxf(x, -1.0f), 1.0f);
}

template <typename T>
__device__ __forceinline__ float load_sample(const T* p, int64_t i);
template <>
__device__ __forceinline__ float load_sample<int16_t>(const int16_t* p, int64_t i) {
  return pcm_to_float(__ldg(p + i));
}
template <>
__device__ __forceinline__ float load_sample<float>(const float* p, int64_t i) {
  return __ldg(p + i);
}

__device__ __forceinline__ void load_tables(FilterSmem& sm, const double* __restrict__ hann_half, const double2* __restrict__ tw256,
                                            const double2* __restrict__ tw512, const MelTables& mt, int tid, int nthreads) {
  for (int i = tid; i < 256; i += nthreads) {
    sm.tw512[i] = tw512[i];
    sm.hann2[i] = make_double2(hann_half[2 * i], hann_half[2 * i + 1]);
    sm.twj[i] = tw256[((i >> 4) * (i & 15)) & 255];
  }
  for (int i = tid; i < mt.n_seg * 8; i += nthreads) {
    const int seg = i >> 3, t = i & 7;
    sm.seg_w[seg][t] = t < mt.seg_count[seg] ? mt.tap_w[mt.seg_first[seg] + t] : 0.0f;
    if (t == 0) sm.seg_bin0[seg] = mt.tap_bin[mt.seg_first[seg]];
  }
  for (int i = tid; i <= kMel; i += nthreads) sm.band_seg0[i] = mt.band_seg0[i];
  for (int i = tid; i < kMel; i += nthreads) sm.band_bias[i] = mt.bias[i];
  for (int w = 0; w < F_WARPS; ++w)
    for (int i = tid; i < MAGP; i += nthreads) sm.w[w].mag[i] = make_float2(0.f, 0.f);
}

// One frame per 16-lane half of the warp (both halves execute this together): samples from `load` (pair m of lane j =
// samples 2(j+16m), +1 of the frame) -> 257 magnitudes in mag[bin].x (half 0) / .y (half 1).  Contains two __syncwarp.
template <typename LoadFn>
__device__ __forceinline__ void frame_spectrum64(LoadFn load, const FilterSmem& sm, double2* __restrict__ xch,
                                                 float2* __restrict__ mag2, int lane) {
  const int j = lane & 15, h = lane >> 4;
  f64::pass1(load, sm.hann2, sm.twj, xch, j);
  __syncwarp();
  double2 v[16];
  f64::pass2(xch, j, v);
  __syncwarp();
  float* mag = reinterpret_cast<float*>(mag2) + h;   // this half's component, stride 2
  const int src = (lane & 16) | ((16 - j) & 15);
  // lane j handles the bin pairs (k, 256 - k), k = 16 k1 + j, k1 = 0..7; Z[256-k] is v[XI(15-k1)] of lane 16-j
  // (lane 0 pairs with itself: Z[16 (16-k1)], and Z[256] = Z[0])
#pragma unroll
  for (int k1 = 0; k1 < 8; ++k1) {
    const double2 up = v[f64::XI(15 - k1)], self = v[f64::XI(k1 == 0 ? 0 : 16 - k1)];
    const double sx = j == 0 ? self.x : up.x, sy = j == 0 ? self.y : up.y;
    const double2 zp = make_double2(__shfl_sync(0xffffffffu, sx, src), __shfl_sync(0xffffffffu, sy, src));
    float mk, mnk;
    f64::split_pair(v[f64::XI(k1)], zp, sm.tw512[16 * k1 + j], mk, mnk);
    mag[2 * (16 * k1 + j)] = mk;
    mag[2 * (256 - 16 * k1 - j)] = mnk;
  }
  if (j == 0) {   // bin 128 pairs with itself
    float mk, mnk;
    f64::split_pair(v[f64::XI(8)], v[f64::XI(8)], sm.tw512[128], mk, mnk);
    mag[2 * 128] = mk;
  }
}

__device__ __forceinline__ float mel_log(float acc, float bias, const MelParams& P) {
  acc += bias;
  acc = fmaxf(acc, P.mel_floor);
  return __fmul_rn(__fsub_rn(logf(acc), P.mel_log_offset), P.mel_scale);
}

// mel projection + log compression of the two frames of a warp whose magnitudes are in ws.mag.  Per segment an fma chain
// from 0, segments added in order, bias, floor, log: bit-identical to mel_from_mag_kernel.  The band sums of frame 0 / 1
// go to out0 / out1 (nullptr = frame not wanted).  Contains two __syncwarp.
__device__ __forceinline__ void mel_pair(const FilterSmem& sm, FilterWarpSmem& ws, const MelParams& P, int n_seg,
                                         float* __restrict__ out0, float* __restrict__ out1, int lane) {
  __syncwarp();
  for (int seg = lane; seg < n_seg; seg += 32) {
    const float4 w0 = *reinterpret_cast<const float4*>(&sm.seg_w[seg][0]), w1 = *reinterpret_cast<const float4*>(&sm.seg_w[seg][4]);
    const float2* m = ws.mag + sm.seg_bin0[seg];
    const float2 m0 = m[0], m1 = m[1], m2 = m[2], m3 = m[3], m4 = m[4], m5 = m[5], m6 = m[6], m7 = m[7];
    float a0 = 0.f, a1 = 0.f;
    a0 = fmaf(w0.x, m0.x, a0); a1 = fmaf(w0.x, m0.y, a1);
    a0 = fmaf(w0.y, m1.x, a0); a1 = fmaf(w0.y, m1.y, a1);
    a0 = fmaf(w0.z, m2.x, a0); a1 = fmaf(w0.z, m2.y, a1);
    a0 = fmaf(w0.w, m3.x, a0); a1 = fmaf(w0.w, m3.y, a1);
    a0 = fmaf(w1.x, m4.x, a0); a1 = fmaf(w1.x, m4.y, a1);
    a0 = fmaf(w1.y, m5.x, a0); a1 = fmaf(w1.y, m5.y, a1);
    a0 = fmaf(w1.z, m6.x, a0); a1 = fmaf(w1.z, m6.y, a1);
    a0 = fmaf(w1.w, m7.x, a0); a1 = fmaf(w1.w, m7.y, a1);
    ws.partial[seg] = make_float2(a0, a1);
  }
  __syncwarp();
  {   // bands 0..31: one lane each, both frames
    const int s0 = sm.band_seg0[lane], s1 = sm.band_seg0[lane + 1];
    float a0 = 0.f, a1 = 0.f;
    for (int s = s0; s < s1; ++s) {
      const float2 p = ws.partial[s];
      a0 += p.x; a1 += p.y;
    }
    const float bias = sm.band_bias[lane];
    if (out0) out0[lane] = mel_log(a0, bias, P);
    if (out1) out1[lane] = mel_log(a1, bias, P);
  }
  if (lane < 2 * (kMel - 32)) {   // bands 32..39: lanes 0..7 frame 0, lanes 8..15 frame 1
    const int band = 32 + (lane & 7), f = lane >> 3;
    const int s0 = sm.band_seg0[band], s1 = sm.band_seg0[band + 1];
    float a = 0.f;
    for (int s = s0; s < s1; ++s) {
      const float2 p = ws.partial[s];
      a += f ? p.y : p.x;
    }
    float* out = f ? out1 : out0;
    if (out) out[band] = mel_log(a, sm.band_bias[band], P);
  }
}

template <typename T>
__global__ void __launch_bounds__(F_THREADS, 1) filter_kernel(const FilterParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FilterSmem& sm = *reinterpret_cast<FilterSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int j = lane & 15, h = lane >> 4;
  FilterWarpSmem& ws = sm.w[warp];

  load_tables(sm, P.hann_half, P.tw256, P.tw512, P.mp.mt, tid, F_THREADS);
  __syncthreads();
  const int n_seg = P.mp.mt.n_seg;

  const T* pcm = reinterpret_cast<const T*>(P.pcm);
  // Fast path (int16, 4-byte aligned rows of even length, no pre-emphasis = the reference's default): 32-bit loads of
  // sample pairs, the next iteration's 320 samples prefetched into registers behind the butterflies.
  const bool fast = sizeof(T) == 2 && P.a == 0.0f && (reinterpret_cast<uintptr_t>(pcm) & 3) == 0 && (P.pitch & 1) == 0 &&
                    (P.n_samples & 1) == 0;

  for (int64_t item = (int64_t)blockIdx.x * F_WARPS + warp; item < P.n_items; item += (int64_t)gridDim.x * F_WARPS) {
    const int64_t s = item / P.items_per_stream;
    const int64_t f0 = (item - s * P.items_per_stream) * P.item_frames;
    const int nf = (int)min((int64_t)P.item_frames, P.n_frames - f0);
    const T* row = pcm + s * P.pitch;
    const int64_t base = f0 * kHop;              // stream sample at ring position 0
    const int64_t n_avail = P.n_samples - base;  // samples of the stream from `base` on

    // stage relative samples [r0, r0 + cnt) into the ring (cnt even, r0 even); generic path
    auto stage_generic = [&](int r0, int cnt) {
      for (int r = lane; r < cnt; r += 32) {
        const int64_t idx = base + r0 + r;
        float v = 0.f;
        if (idx < P.n_samples) {
          v = load_sample<T>(row, idx);
          if (P.a != 0.0f) {
            // y[n] = x[n] - a*x[n-1] with fp32 product and difference (numpy semantics after the first call)
            const float xp = idx > 0 ? load_sample<T>(row, idx - 1) : 0.0f;
            v = __fsub_rn(v, __fmul_rn(P.a, xp));
          }
        }
        ws.ring[(r0 + r) & (F_RING - 1)] = v;
      }
    };
    const uint32_t* row32 = reinterpret_cast<const uint32_t*>(row + base);   // (fast path only)
    auto stage_word = [&](int r0, int wi, uint32_t word) {   // word wi of the range that starts at relative sample r0
      *reinterpret_cast<float2*>(&ws.ring[(r0 + 2 * wi) & (F_RING - 1)]) =
          make_float2(pcm_to_float((int16_t)(word & 0xffff)), pcm_to_float((int16_t)(word >> 16)));
    };
    uint32_t pre[5];
    auto prefetch = [&](int r0) {   // 320 samples = 160 words from relative sample r0
#pragma unroll
      for (int c = 0; c < 5; ++c) {
        const int wi = lane + 32 * c;
        pre[c] = (r0 + 2 * wi < n_avail) ? __ldg(row32 + (r0 >> 1) + wi) : 0u;
      }
    };

    __syncwarp();   // the previous item's last reads of the ring are done
    if (fast) {
#pragma unroll
      for (int c = 0; c < 6; ++c) {   // first 352 samples = 176 words
        const int wi = lane + 32 * c;
        if (wi < 176) stage_word(0, wi, (2 * wi < n_avail) ? __ldg(row32 + wi) : 0u);
      }
      prefetch(352);
    } else {
      stage_generic(0, 352);
    }

    for (int i = 0; i < nf; i += 2) {
      // new samples of this frame pair: relative [160 i + 352, 160 i + 672)
      if (fast) {
#pragma unroll
        for (int c = 0; c < 5; ++c) stage_word(160 * i + 352, lane + 32 * c, pre[c]);
      } else {
        stage_generic(160 * i + 352, 320);
      }
      __syncwarp();
      if (fast && i + 2 < nf) prefetch(160 * (i + 2) + 352);   // latency hidden behind the FFTs
      const int rb = 160 * (i + h) + 2 * j;
      auto load = [&](int m) {
        const float2 x = *reinterpret_cast<const float2*>(&ws.ring[(rb + 32 * m) & (F_RING - 1)]);
        return make_double2((double)x.x, (double)x.y);
      };
      frame_spectrum64(load, sm, ws.xch[h], ws.mag, lane);
      float* out = P.mel + ((s * P.n_frames + f0 + i) * kMel);
      mel_pair(sm, ws, P.mp, n_seg, out, i + 1 < nf ? out + kMel : nullptr, lane);
    }
  }
}

static MelParams mel_params(const wwb_ctx* ctx) {
  MelParams mp;
  mp.mt = ctx->mel;
  mp.mel_floor = ctx->mel_floor; mp.mel_log_offset = ctx->mel_log_offset; mp.mel_scale = ctx->mel_scale;
  return mp;
}

int launch_filter(wwb_ctx* ctx, const void* pcm, int dtype, int64_t S, int64_t N, int64_t pitch,
                  float a, float* mel, cudaStream_t st) {
  if (dtype != WWB_PCM_I16 && dtype != WWB_PCM_F32) return fail(ctx, WWB_ERR_ARG, "bad pcm dtype %d", dtype);
  if (S < 0 || N < 0 || pitch < N) return fail(ctx, WWB_ERR_ARG, "bad filter geometry");
  int64_t F = wwb_num_frames(N);
  if (S == 0 || F == 0) return WWB_OK;
  FilterParams P;
  P.pcm = pcm; P.n_streams = S; P.n_samples = N; P.pitch = pitch;
  P.n_frames = F;
  // work items = chunks of a stream; 64 frames per item (352 / (64 * 160) = 3.4 % halo) unless that leaves warps idle
  const int64_t n_warps = (int64_t)ctx->sm_count * F_WARPS;
  int item_frames = 64;
  while (item_frames > 2 && S * ((F + item_frames - 1) / item_frames) < 4 * n_warps) item_frames /= 2;
  P.item_frames = item_frames;
  P.items_per_stream = (int)((F + item_frames - 1) / item_frames);
  P.n_items = S * P.items_per_stream;
  P.a = a; P.mel = mel; P.hann_half = ctx->hann; P.tw256 = ctx->tw256; P.tw512 = ctx->tw512;
  P.mp = mel_params(ctx);
  size_t smem = sizeof(FilterSmem);
  int64_t grid = std::min<int64_t>((P.n_items + F_WARPS - 1) / F_WARPS, (int64_t)ctx->sm_count);
  if (dtype == WWB_PCM_I16) {
    WWB_CUDA(ctx, cudaFuncSetAttribute(filter_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    filter_kernel<int16_t><<<(unsigned)grid, F_THREADS, smem, st>>>(P);
  } else {
    WWB_CUDA(ctx, cudaFuncSetAttribute(filter_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    filter_kernel<float><<<(unsigned)grid, F_THREADS, smem, st>>>(P);
  }
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

// ---------------------------------------------------------------------------------------
// Streaming front end (WakewordTrigger._sample, wakeword/tflite.py:148-168) for many streams, three small kernels:
//   plan   (one thread per stream)  how many frames the chunk completes; if they are analysed (is_speech, :166-167)
//          one encoder window per frame is recorded (win_stream / win_start) and the stream's slot reserved
//   frames (one 16-lane half-warp per (stream, frame))  pending samples + chunk -> frame -> fp64 FFT -> mel row pushed
//          into the stream's ring; with one new frame per stream and push (hop 1, BASELINE config 4) 16 streams share a
//          CTA instead of one CTA per stream
//   tail   (one CTA per stream)  unread PCM tail, previous sample, ring head
// Each kernel runs over the entries i of the push: per-stream state is at slot ids[i], the chunk at pcm + off[i], and the
// per-push scratch (n_new, win_slot, window lists) and every output at i.  A dense push passes ids = off = NULL.
struct StreamFilterParams {
  const int16_t* pcm;
  int64_t n;
  int64_t n_streams;      // entries
  const int32_t* ids;     // [n_streams] slot of entry i (NULL = i)
  const int32_t* off;     // [n_streams + 1] chunk offsets (NULL = i * n)
  const uint8_t* is_speech;
  const uint8_t* is_active;
  float a;
  StreamState st;
  int L;
  const double* hann_half;
  const double2* tw256;
  const double2* tw512;
  MelParams mp;
};

__device__ __forceinline__ int stream_total_frames(int total) { return total >= kFFT ? (total - kFFT) / kHop + 1 : 0; }

__device__ __forceinline__ int64_t entry_slot(const int32_t* ids, int64_t i) { return ids ? (int64_t)ids[i] : i; }

// entry i's chunk and its length
__device__ __forceinline__ const int16_t* entry_chunk(const StreamFilterParams& P, int64_t i, int& n) {
  if (P.off) {
    const int o = P.off[i];
    n = P.off[i + 1] - o;
    return P.pcm + o;
  }
  n = (int)P.n;
  return P.pcm + i * P.n;
}

__global__ void __launch_bounds__(128) stream_plan_kernel(const StreamFilterParams P) {
  const StreamState& S = P.st;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n_streams) return;
  const int64_t s = entry_slot(P.ids, i);
  int n_new = 0;
  const bool active = P.is_active && P.is_active[i];   // "if not context.is_active: self._sample(...)" (:139-140)
  const bool speech = P.is_speech ? (P.is_speech[i] != 0) : true;
  if (!active && speech) {
    int n;
    entry_chunk(P, i, n);
    const int n_frames = stream_total_frames(S.n_pending[s] + n);
    if (n_frames > 0) {
      const int head = S.ring_head[s];
      const int slot = atomicAdd(S.n_win, n_frames);
      for (int q = 0; q < n_frames; ++q) {
        S.win_stream[slot + q] = (int32_t)i;
        S.win_start[slot + q] = (head + 1 + q) % S.ring;
      }
      S.win_slot[i] = slot;
      n_new = n_frames;
    }
  }
  S.n_new[i] = n_new;
}

__global__ void __launch_bounds__(F_THREADS, 1) stream_frames_kernel(const StreamFilterParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FilterSmem& sm = *reinterpret_cast<FilterSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int j = lane & 15, h = lane >> 4;
  FilterWarpSmem& ws = sm.w[warp];
  const StreamState& S = P.st;

  load_tables(sm, P.hann_half, P.tw256, P.tw512, P.mp.mt, tid, F_THREADS);
  __syncthreads();
  const int n_seg = P.mp.mt.n_seg;
  const int64_t n_items = P.n_streams * S.max_frames;

  // a warp takes two items (stream, frame) per iteration, one per half
  for (int64_t it0 = ((int64_t)blockIdx.x * F_WARPS + warp) * 2; it0 < n_items; it0 += (int64_t)gridDim.x * F_WARPS * 2) {
    const int64_t it = it0 + h;
    const int64_t e = it < n_items ? it / S.max_frames : 0;   // entry
    const int q = (int)(it - e * S.max_frames);
    const bool live = it < n_items && q < S.n_new[e];
    const int64_t s = live ? entry_slot(P.ids, e) : 0;
    float* frame = ws.ring + h * kFFT;   // the ring doubles as two frame buffers
    __syncwarp();
    if (live) {
      const int np = S.n_pending[s];
      const float* pend = S.pending + s * S.pend_cap;
      int n;
      const int16_t* chunk = entry_chunk(P, e, n);
      const float prev = S.prev_sample[s];
      for (int i = j; i < kFFT; i += 16) {
        const int p = q * kHop + i;
        float v;
        if (p < np) {
          v = pend[p];   // already pre-emphasised
        } else {
          const int c = p - np;
          const float x = pcm_to_float(chunk[c]);
          const float xp = c > 0 ? pcm_to_float(chunk[c - 1]) : prev;
          v = (P.a != 0.0f) ? __fsub_rn(x, __fmul_rn(P.a, xp)) : x;
        }
        frame[i] = v;
      }
    }
    __syncwarp();
    auto load = [&](int m) {
      const float2 x = *reinterpret_cast<const float2*>(&frame[2 * (j + 16 * m)]);
      return make_double2((double)x.x, (double)x.y);
    };
    frame_spectrum64(load, sm, ws.xch[h], ws.mag, lane);
    // the two halves are different streams: each frame goes to its own stream's ring row; the window for new frame q
    // ends at ring row (head + L + q) % ring
    const bool live0 = __shfl_sync(0xffffffffu, live ? 1 : 0, 0) != 0, live1 = __shfl_sync(0xffffffffu, live ? 1 : 0, 16) != 0;
    const int64_t s0 = __shfl_sync(0xffffffffu, s, 0), s1 = __shfl_sync(0xffffffffu, s, 16);
    const int q0 = __shfl_sync(0xffffffffu, q, 0), q1 = __shfl_sync(0xffffffffu, q, 16);
    float* dst0 = live0 ? S.mel_ring + (s0 * S.ring + (S.ring_head[s0] + P.L + q0) % S.ring) * kMel : nullptr;
    float* dst1 = live1 ? S.mel_ring + (s1 * S.ring + (S.ring_head[s1] + P.L + q1) % S.ring) * kMel : nullptr;
    mel_pair(sm, ws, P.mp, n_seg, dst0, dst1, lane);
  }
}

__global__ void __launch_bounds__(128) stream_tail_kernel(const StreamFilterParams P) {
  const StreamState& S = P.st;
  const int64_t i = blockIdx.x;
  const int tid = threadIdx.x;
  if (P.is_active && P.is_active[i]) return;
  const int64_t s = entry_slot(P.ids, i);
  int n;
  const int16_t* chunk = entry_chunk(P, i, n);
  const int np = S.n_pending[s];
  const int total = np + n;
  const int n_frames = stream_total_frames(total);
  float* pend = S.pending + s * S.pend_cap;
  const float prev = S.prev_sample[s];
  // new pending tail = samples [n_frames*hop, total) (< 512 + 160); moved through registers (overlapping ranges)
  const int keep0 = n_frames * kHop;
  const int keep = total - keep0;
  float tmp[6];
  int c = 0;
  for (int i = tid; i < keep && c < 6; i += 128, ++c) {
    const int p = keep0 + i;
    float v;
    if (p < np) {
      v = pend[p];
    } else {
      const int cc = p - np;
      const float x = pcm_to_float(chunk[cc]);
      const float xp = cc > 0 ? pcm_to_float(chunk[cc - 1]) : prev;
      v = (P.a != 0.0f) ? __fsub_rn(x, __fmul_rn(P.a, xp)) : x;
    }
    tmp[c] = v;
  }
  __syncthreads();
  c = 0;
  for (int i = tid; i < keep && c < 6; i += 128, ++c) pend[i] = tmp[c];
  if (tid == 0) {
    S.n_pending[s] = keep;
    if (n > 0) S.prev_sample[s] = pcm_to_float(chunk[n - 1]);
    if (S.n_new[i] > 0) S.ring_head[s] = (S.ring_head[s] + S.n_new[i]) % S.ring;
  }
}

// After the encoder has produced win_post: per-stream trigger bookkeeping
// (wakeword/tflite.py:233-239) and the reset on a VAD fall (:135-146, :241-246).
struct StreamFinishParams {
  StreamState st;
  int L;
  const int32_t* ids;     // [n_streams] slot of entry i (NULL = i)
  const uint8_t* is_speech;
  const uint8_t* is_active;
  float threshold;
  float* post_out;        // [entries, max_frames]
  int32_t* n_post_out;    // [entries]
  uint8_t* trigger_out;   // [entries]
  float* post_max_out;    // [entries]
  int64_t n_streams;      // entries
};

__global__ void stream_finish_kernel(const StreamFinishParams P) {
  const StreamState& S = P.st;
  const int64_t i = blockIdx.x;
  if (i >= P.n_streams) return;
  const int64_t s = entry_slot(P.ids, i);
  __shared__ int do_reset;
  if (threadIdx.x == 0) {
    const int n = S.n_new[i];
    const int slot = n > 0 ? S.win_slot[i] : 0;
    float pm = S.post_max[s];
    bool trig = false;
    const bool active = P.is_active && P.is_active[i];
    for (int q = 0; q < S.max_frames; ++q) {
      float p = nanf("");
      if (q < n) {
        p = S.win_post[slot + q];
        if (p > pm) pm = p;
        if (p > P.threshold && !active) trig = true;
      }
      if (P.post_out) P.post_out[i * S.max_frames + q] = p;
    }
    if (P.n_post_out) P.n_post_out[i] = n;
    if (P.trigger_out) P.trigger_out[i] = trig ? 1 : 0;
    if (P.post_max_out) P.post_max_out[i] = pm;
    const bool speech = P.is_speech ? (P.is_speech[i] != 0) : true;
    const bool fall = S.was_speech[s] && !speech;
    S.was_speech[s] = speech ? 1 : 0;
    S.post_max[s] = fall ? 0.0f : pm;
    if (fall) {
      S.n_pending[s] = 0;
      S.ring_head[s] = 0;
    }
    do_reset = fall ? 1 : 0;
  }
  __syncthreads();
  if (do_reset) {
    float* ring = S.mel_ring + s * S.ring * kMel;
    for (int i = threadIdx.x; i < S.ring * kMel; i += blockDim.x) ring[i] = 0.0f;
  }
}

__global__ void stream_reset_kernel(StreamState S, const uint8_t* mask, int64_t n_streams) {
  const int64_t s = blockIdx.x;
  if (s >= n_streams || (mask && !mask[s])) return;
  float* ring = S.mel_ring + s * S.ring * kMel;
  for (int i = threadIdx.x; i < S.ring * kMel; i += blockDim.x) ring[i] = 0.0f;
  if (threadIdx.x == 0) {
    S.n_pending[s] = 0;
    S.ring_head[s] = 0;
    S.post_max[s] = 0.0f;
  }
}

// filter.tflite on magnitudes: one thread per (frame, band)
__global__ void mel_from_mag_kernel(const float* __restrict__ mag, int64_t B, MelParams P, float* __restrict__ mel) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= B * kMel) return;
  const int64_t f = o / kMel;
  const int band = (int)(o - f * kMel);
  const MelTables& mt = P.mt;
  const float* row = mag + f * kBins;
  float acc = 0.f;
  for (int s = mt.band_seg0[band]; s < mt.band_seg0[band + 1]; ++s) {
    float part = 0.f;
    const int first = mt.seg_first[s], cnt = mt.seg_count[s];
    for (int t = 0; t < cnt; ++t) part = fmaf(mt.tap_w[first + t], row[mt.tap_bin[first + t]], part);
    acc += part;
  }
  acc += mt.bias[band];
  acc = fmaxf(acc, P.mel_floor);
  mel[o] = __fmul_rn(__fsub_rn(logf(acc), P.mel_log_offset), P.mel_scale);
}

int launch_mel_from_mag(wwb_ctx* ctx, const float* mag, int64_t B, float* mel, cudaStream_t st) {
  if (B == 0) return WWB_OK;
  MelParams P;
  P.mt = ctx->mel;
  P.mel_floor = ctx->mel_floor; P.mel_log_offset = ctx->mel_log_offset; P.mel_scale = ctx->mel_scale;
  mel_from_mag_kernel<<<(unsigned)((B * kMel + 255) / 256), 256, 0, st>>>(mag, B, P, mel);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_stream_filter(wwb_ctx* ctx, const int16_t* pcm, int64_t S, int64_t n, const int32_t* ids, const int32_t* off,
                         const uint8_t* is_speech, const uint8_t* is_active, float a,
                         cudaStream_t st) {
  StreamFilterParams P;
  P.pcm = pcm; P.n = n; P.n_streams = S; P.ids = ids; P.off = off; P.is_speech = is_speech; P.is_active = is_active; P.a = a;
  P.st = ctx->st; P.L = ctx->L;
  P.hann_half = ctx->hann; P.tw256 = ctx->tw256; P.tw512 = ctx->tw512;
  P.mp = mel_params(ctx);
  WWB_CUDA(ctx, cudaMemsetAsync(ctx->st.n_win, 0, sizeof(int32_t), st));
  stream_plan_kernel<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  size_t smem = sizeof(FilterSmem);
  WWB_CUDA(ctx, cudaFuncSetAttribute(stream_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t pairs = (S * ctx->st.max_frames + 1) / 2;
  const int64_t grid = std::min<int64_t>((pairs + F_WARPS - 1) / F_WARPS, (int64_t)ctx->sm_count);
  stream_frames_kernel<<<(unsigned)grid, F_THREADS, smem, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  stream_tail_kernel<<<(unsigned)S, 128, 0, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_stream_finish(wwb_ctx* ctx, int64_t S, const int32_t* ids, const uint8_t* is_speech, const uint8_t* is_active,
                         float threshold, float* post_out, int32_t* n_post_out, uint8_t* trigger_out,
                         float* post_max_out, cudaStream_t st) {
  StreamFinishParams P;
  P.st = ctx->st; P.L = ctx->L; P.ids = ids; P.is_speech = is_speech; P.is_active = is_active;
  P.threshold = threshold; P.post_out = post_out; P.n_post_out = n_post_out;
  P.trigger_out = trigger_out; P.post_max_out = post_max_out; P.n_streams = S;
  stream_finish_kernel<<<(unsigned)S, 128, 0, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_stream_reset(wwb_ctx* ctx, const uint8_t* mask, int64_t S, cudaStream_t st) {
  stream_reset_kernel<<<(unsigned)S, 128, 0, st>>>(ctx->st, mask, S);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb
