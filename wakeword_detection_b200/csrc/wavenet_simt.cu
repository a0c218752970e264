// WaveNet encode + detect on CUDA cores in fp32 (precision WWB_PREC_F32).
//
// Validation path of wavenet_tc.cu: the arithmetic of Wavenet/encode.tflite +
// detect.tflite (SURVEY.md Appendix A3) with fp32 products and sums.  One CTA per
// window, one thread per time step; the 16-channel residual stream and the 32-channel
// skip sum stay in registers for all 24 blocks, only the BN-affined activations `u`
// go through shared memory (the dilated taps read rows t-d and t-2d; rows < 0 are the
// causal zero padding, applied after the BN affine as in the graph).
#include "common.cuh"

namespace wwb {

constexpr int W_T = 182, W_C = 16, W_S = 32, W_NB = 24;
constexpr int W_THREADS = 192;
constexpr int W_PAD = 16;      // rows of causal zero padding (max 2*dilation)
constexpr int W_UP = 20;       // row pitch of u in floats (conflict-free float4 reads)

__device__ __forceinline__ float sigmoid_w(float x) { return 1.0f / (1.0f + expf(-x)); }

struct WnParams {
  WinMap wm;
  WavenetWeights w;
  int L;
  float* enc_out;   // [B, L, 32] or null
  float* det_out;   // [B, 2] or null
  float* post;      // [B] or null
};

__global__ void __launch_bounds__(W_THREADS) wavenet_simt_kernel(const WnParams P) {
  __shared__ __align__(16) float us[(W_T + W_PAD + 2) * W_UP];
  __shared__ __align__(16) float gw[48 * 32];     // gate weights of the current block [k][n]
  __shared__ __align__(16) float rw[16 * 48];     // residual|skip weights [k][n]
  __shared__ float gb[32], rb[48], bnm[16], bna[16];
  __shared__ float red[2][W_THREADS / 32];
  const int64_t b = blockIdx.x;
  if (P.wm.n_win_dev && b >= *P.wm.n_win_dev) return;
  const int t = threadIdx.x;
  const bool live = t < P.L;
  const WavenetWeights& W = P.w;

  for (int i = t; i < W_PAD * W_UP; i += W_THREADS) us[i] = 0.f;

  // input layer: x = ReLU(in_w * mel + in_b)
  float x[W_C];
  {
    float m[kMel];
    const float* row = win_row(P.wm, b, live ? t : 0);
#pragma unroll
    for (int i = 0; i < kMel; i += 4) {
      float4 v = *reinterpret_cast<const float4*>(row + i);
      m[i] = v.x; m[i + 1] = v.y; m[i + 2] = v.z; m[i + 3] = v.w;
    }
#pragma unroll
    for (int c = 0; c < W_C; ++c) x[c] = __ldg(W.in_b + c);
#pragma unroll
    for (int k = 0; k < kMel; ++k)
#pragma unroll
      for (int c = 0; c < W_C; ++c) x[c] = fmaf(__ldg(W.in_w + k * W_C + c), m[k], x[c]);
#pragma unroll
    for (int c = 0; c < W_C; ++c) x[c] = fmaxf(x[c], 0.f);
  }
  float skip[W_S];
#pragma unroll
  for (int n = 0; n < W_S; ++n) skip[n] = 0.f;

  for (int blk = 0; blk < W_NB; ++blk) {
    __syncthreads();   // previous block finished reading us / weights
    for (int i = t; i < 48 * 32; i += W_THREADS) gw[i] = W.gate_w[blk * 48 * 32 + i];
    for (int i = t; i < 16 * 48; i += W_THREADS) rw[i] = W.rs_w[blk * 16 * 48 + i];
    if (t < 32) gb[t] = W.gate_b[blk * 32 + t];
    if (t < 48) rb[t] = W.rs_b[blk * 48 + t];
    if (t < 16) { bnm[t] = W.bn_mul[blk * 16 + t]; bna[t] = W.bn_add[blk * 16 + t]; }
    __syncthreads();
    const int d = W.dilation[blk];
    float u[W_C];
#pragma unroll
    for (int c = 0; c < W_C; ++c) u[c] = __fadd_rn(__fmul_rn(x[c], bnm[c]), bna[c]);
    if (live) {
      float4* dst = reinterpret_cast<float4*>(us + (t + W_PAD) * W_UP);
#pragma unroll
      for (int c = 0; c < W_C; c += 4) dst[c / 4] = make_float4(u[c], u[c + 1], u[c + 2], u[c + 3]);
    }
    __syncthreads();
    // gate pre-activations: n < 16 tanh, n >= 16 sigmoid ; k = tap*16 + channel, tap 0 = t-2d
    float acc[32];
#pragma unroll
    for (int n = 0; n < 32; ++n) acc[n] = gb[n];
#pragma unroll
    for (int tap = 0; tap < 3; ++tap) {
      float in[W_C];
      if (tap == 2) {
#pragma unroll
        for (int c = 0; c < W_C; ++c) in[c] = u[c];
      } else {
        const int r = (live ? t : 0) + W_PAD - (2 - tap) * d;
        const float4* src = reinterpret_cast<const float4*>(us + r * W_UP);
#pragma unroll
        for (int c = 0; c < W_C; c += 4) {
          float4 v = src[c / 4];
          in[c] = v.x; in[c + 1] = v.y; in[c + 2] = v.z; in[c + 3] = v.w;
        }
      }
#pragma unroll
      for (int c = 0; c < W_C; ++c) {
        const float4* wr = reinterpret_cast<const float4*>(gw + (tap * 16 + c) * 32);
#pragma unroll
        for (int n = 0; n < 32; n += 4) {
          float4 wv = wr[n / 4];
          acc[n] = fmaf(wv.x, in[c], acc[n]);
          acc[n + 1] = fmaf(wv.y, in[c], acc[n + 1]);
          acc[n + 2] = fmaf(wv.z, in[c], acc[n + 2]);
          acc[n + 3] = fmaf(wv.w, in[c], acc[n + 3]);
        }
      }
    }
    float g[W_C];
#pragma unroll
    for (int c = 0; c < W_C; ++c) g[c] = tanhf(acc[c]) * sigmoid_w(acc[16 + c]);
    // residual (n < 16) and skip (n >= 16) 1x1 convolutions
    float o[48];
#pragma unroll
    for (int n = 0; n < 48; ++n) o[n] = rb[n];
#pragma unroll
    for (int c = 0; c < W_C; ++c) {
      const float4* wr = reinterpret_cast<const float4*>(rw + c * 48);
#pragma unroll
      for (int n = 0; n < 48; n += 4) {
        float4 wv = wr[n / 4];
        o[n] = fmaf(wv.x, g[c], o[n]);
        o[n + 1] = fmaf(wv.y, g[c], o[n + 1]);
        o[n + 2] = fmaf(wv.z, g[c], o[n + 2]);
        o[n + 3] = fmaf(wv.w, g[c], o[n + 3]);
      }
    }
    if (blk < W_NB - 1) {
#pragma unroll
      for (int c = 0; c < W_C; ++c) x[c] = fmaxf(o[c], 0.f) + x[c];
    }
#pragma unroll
    for (int n = 0; n < W_S; ++n) skip[n] += fmaxf(o[16 + n], 0.f);
  }

  if (P.enc_out && live) {
    float4* dst = reinterpret_cast<float4*>(P.enc_out + (b * P.L + t) * W_S);
#pragma unroll
    for (int n = 0; n < W_S; n += 4) dst[n / 4] = make_float4(skip[n], skip[n + 1], skip[n + 2], skip[n + 3]);
  }
  if (!P.det_out && !P.post) return;

  // detect: ReLU -> 1x1 32->32 ReLU -> 1x1 32->2 -> max over time -> softmax
  float h[W_S];
#pragma unroll
  for (int n = 0; n < W_S; ++n) h[n] = __ldg(W.det1_b + n);
#pragma unroll
  for (int k = 0; k < W_S; ++k) {
    float e = fmaxf(skip[k], 0.f);
#pragma unroll
    for (int n = 0; n < W_S; ++n) h[n] = fmaf(__ldg(W.det1_w + k * W_S + n), e, h[n]);
  }
  float z0 = __ldg(W.det2_b), z1 = __ldg(W.det2_b + 1);
#pragma unroll
  for (int k = 0; k < W_S; ++k) {
    float e = fmaxf(h[k], 0.f);
    z0 = fmaf(__ldg(W.det2_w + k), e, z0);
    z1 = fmaf(__ldg(W.det2_w + W_S + k), e, z1);
  }
  if (!live) { z0 = -INFINITY; z1 = -INFINITY; }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    z0 = fmaxf(z0, __shfl_xor_sync(0xffffffffu, z0, s));
    z1 = fmaxf(z1, __shfl_xor_sync(0xffffffffu, z1, s));
  }
  if ((t & 31) == 0) { red[0][t >> 5] = z0; red[1][t >> 5] = z1; }
  __syncthreads();
  if (t == 0) {
    for (int i = 1; i < W_THREADS / 32; ++i) { z0 = fmaxf(z0, red[0][i]); z1 = fmaxf(z1, red[1][i]); }
    float m = fmaxf(z0, z1);
    float e0 = expf(z0 - m), e1 = expf(z1 - m), s = e0 + e1;
    if (P.det_out) { P.det_out[b * 2] = e0 / s; P.det_out[b * 2 + 1] = e1 / s; }
    if (P.post) P.post[b] = e1 / s;
  }
}

// detect.tflite alone on a materialised encoder output [B, L, 32]
__global__ void __launch_bounds__(W_THREADS) wavenet_detect_kernel(const float* __restrict__ enc, WavenetWeights W,
                                                                   int L, float* __restrict__ out) {
  __shared__ float red[2][W_THREADS / 32];
  const int64_t b = blockIdx.x;
  const int t = threadIdx.x;
  const bool live = t < L;
  float skip[W_S];
  const float* row = enc + (b * L + (live ? t : 0)) * W_S;
#pragma unroll
  for (int n = 0; n < W_S; ++n) skip[n] = row[n];
  float h[W_S];
#pragma unroll
  for (int n = 0; n < W_S; ++n) h[n] = __ldg(W.det1_b + n);
#pragma unroll
  for (int k = 0; k < W_S; ++k) {
    float e = fmaxf(skip[k], 0.f);
#pragma unroll
    for (int n = 0; n < W_S; ++n) h[n] = fmaf(__ldg(W.det1_w + k * W_S + n), e, h[n]);
  }
  float z0 = __ldg(W.det2_b), z1 = __ldg(W.det2_b + 1);
#pragma unroll
  for (int k = 0; k < W_S; ++k) {
    float e = fmaxf(h[k], 0.f);
    z0 = fmaf(__ldg(W.det2_w + k), e, z0);
    z1 = fmaf(__ldg(W.det2_w + W_S + k), e, z1);
  }
  if (!live) { z0 = -INFINITY; z1 = -INFINITY; }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    z0 = fmaxf(z0, __shfl_xor_sync(0xffffffffu, z0, s));
    z1 = fmaxf(z1, __shfl_xor_sync(0xffffffffu, z1, s));
  }
  if ((t & 31) == 0) { red[0][t >> 5] = z0; red[1][t >> 5] = z1; }
  __syncthreads();
  if (t == 0) {
    for (int i = 1; i < W_THREADS / 32; ++i) { z0 = fmaxf(z0, red[0][i]); z1 = fmaxf(z1, red[1][i]); }
    float m = fmaxf(z0, z1);
    float e0 = expf(z0 - m), e1 = expf(z1 - m), s = e0 + e1;
    out[b * 2] = e0 / s;
    out[b * 2 + 1] = e1 / s;
  }
}

int wavenet_simt_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out, float* post,
                            cudaStream_t st) {
  if (wm.n_win == 0) return WWB_OK;
  // `us` holds W_T + W_PAD + 2 rows: a longer window would write past it (wwb_create refuses one)
  if (ctx->L > W_T) return fail(ctx, WWB_ERR_ARG, "WaveNet window longer than %d frames", W_T);
  WnParams P;
  P.wm = wm; P.w = ctx->wn; P.L = ctx->L; P.enc_out = enc_out; P.det_out = det_out; P.post = post;
  wavenet_simt_kernel<<<(unsigned)wm.n_win, W_THREADS, 0, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int wavenet_simt_detect(wwb_ctx* ctx, const float* enc, int64_t B, float* out, cudaStream_t st) {
  if (B == 0) return WWB_OK;
  wavenet_detect_kernel<<<(unsigned)B, W_THREADS, 0, st>>>(enc, ctx->wn, ctx->L, out);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb
