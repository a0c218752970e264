// CRNN encode + detect on CUDA cores in fp32 (precision WWB_PREC_F32).
//
// This is the validation path of the tensor-core kernels (crnn_tc.cu): the same
// arithmetic as CRNN/encode.tflite + detect.tflite (SURVEY.md Appendix A2) with every
// product and sum in fp32.  Stages (global intermediates in ctx workspaces):
//   conv   : mel window [L,40] -> ReLU(conv 5x20, stride (2,8), SAME) -> [T, 640], T = ceil(L / 8) (CrnnGeom)
//   proj   : [B*T, in] x [in, 192] + b_in     (both directions side by side)
//   gru    : T recurrent steps per direction, gates z|r|h, reset_after
//   detect : 64 -> 64 ReLU -> n_out, sigmoid / softmax
#include <stdlib.h>

#include "common.cuh"

namespace wwb {

constexpr int C_F = 20, C_CH = 32, C_FEAT = 640, C_H = 32, C_G = 96;
constexpr int C_KF = 5, C_KT = 20, C_TAPS = 100;
constexpr int C_PF = 1;                        // SAME padding before (freq); in time it is CrnnGeom::pad_lo
constexpr int C_XF = 44;                       // padded window in shared memory: 8T + 12 rows of C_XF

__global__ void __launch_bounds__(256) crnn_conv_kernel(WinMap wm, const float* __restrict__ w,
                                                        const float* __restrict__ bias,
                                                        float* __restrict__ out, int L, int T, int pad_lo) {
  extern __shared__ float xs_raw[];
  float(*xs)[C_XF] = reinterpret_cast<float(*)[C_XF]>(xs_raw);
  __shared__ float ws[C_TAPS][C_CH];
  const int64_t b = blockIdx.x;
  if (wm.n_win_dev && b >= *wm.n_win_dev) return;
  const int tid = threadIdx.x;
  for (int i = tid; i < (8 * T + 12) * C_XF; i += 256) xs_raw[i] = 0.f;
  for (int i = tid; i < C_TAPS * C_CH; i += 256) (&ws[0][0])[i] = w[i];
  __syncthreads();
  for (int i = tid; i < L * kMel; i += 256) {
    int t = i / kMel, f = i - t * kMel;
    xs[t + pad_lo][f + C_PF] = win_row(wm, b, t)[f];
  }
  __syncthreads();
  const int c = tid & 31, grp = tid >> 5;
  const float bc = bias[c];
  float* o = out + b * (T * C_FEAT);
  for (int p = grp; p < T * C_F; p += 8) {
    const int t = p / C_F, f = p - t * C_F;
    float acc = 0.f;
#pragma unroll
    for (int kf = 0; kf < C_KF; ++kf)
#pragma unroll
      for (int kt = 0; kt < C_KT; ++kt)
        acc = fmaf(ws[kf * C_KT + kt][c], xs[8 * t + kt][2 * f + kf], acc);
    o[t * C_FEAT + f * C_CH + c] = fmaxf(acc + bc, 0.f);
  }
}

// C[M, N] = A[M, K] * Wt[K, N] + bias[N]; 64x64 tiles, 4x4 per thread.
__global__ void __launch_bounds__(256) sgemm_bias_kernel(const float* __restrict__ A, const float* __restrict__ Wt,
                                                         const float* __restrict__ bias, float* __restrict__ C,
                                                         int64_t M, int N, int K) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t m0 = (int64_t)blockIdx.x * 64;
  const int n0 = blockIdx.y * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      int r = i >> 4, kk = i & 15;
      int64_t m = m0 + r;
      As[kk][r] = (m < M && k0 + kk < K) ? A[m * K + k0 + kk] : 0.f;
    }
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      int kk = i >> 6, n = i & 63;
      Bs[kk][n] = (k0 + kk < K && n0 + n < N) ? Wt[(int64_t)(k0 + kk) * N + n0 + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bb[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n < N) C[m * N + n] = acc[i][j] + bias[n];
    }
  }
}

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// xw: [B, T, 192] (fwd gates | bwd gates).  4 windows x 2 directions x 32 units per block.
// seq_out [B,T,64] (layer 1) or last_out [B,64] (layer 2).
__global__ void __launch_bounds__(256) gru_rec_kernel(const float* __restrict__ xw, const float* __restrict__ u_f,
                                                      const float* __restrict__ br_f, const float* __restrict__ u_b,
                                                      const float* __restrict__ br_b, float* __restrict__ seq_out,
                                                      float* __restrict__ last_out, int64_t B,
                                                      const int32_t* __restrict__ n_dev, int T) {
  __shared__ float us[2][C_H][C_G];
  __shared__ float hs[8][C_H];
  const int tid = threadIdx.x;
  for (int i = tid; i < C_H * C_G; i += 256) {
    (&us[0][0][0])[i] = u_f[i];
    (&us[1][0][0])[i] = u_b[i];
  }
  const int i = tid & 31, dir = (tid >> 5) & 1, wl = tid >> 6;
  const int64_t b = (int64_t)blockIdx.x * 4 + wl;
  const int64_t nB = n_dev ? (int64_t)*n_dev : B;
  const bool live = b < nB;
  const float* br = dir ? br_b : br_f;
  const float bz = br[i], brr = br[32 + i], bh = br[64 + i];
  float h = 0.f;
  hs[tid >> 5][i] = 0.f;
  __syncthreads();
  for (int step = 0; step < T; ++step) {
    const int t = dir ? (T - 1 - step) : step;
    float az = bz, ar = brr, ah = bh;
    const float* hrow = hs[tid >> 5];
#pragma unroll
    for (int k = 0; k < C_H; ++k) {
      float hk = hrow[k];
      az = fmaf(us[dir][k][i], hk, az);
      ar = fmaf(us[dir][k][32 + i], hk, ar);
      ah = fmaf(us[dir][k][64 + i], hk, ah);
    }
    float xz = 0.f, xr = 0.f, xh = 0.f;
    if (live) {
      const float* x = xw + (b * T + t) * (2 * C_G) + dir * C_G;
      xz = x[i]; xr = x[32 + i]; xh = x[64 + i];
    }
    float z = sigmoid_f(xz + az);
    float r = sigmoid_f(xr + ar);
    float c = tanhf(xh + r * ah);
    h = z * h + (1.0f - z) * c;
    __syncwarp();
    hs[tid >> 5][i] = h;
    __syncwarp();
    if (live && seq_out) seq_out[(b * T + t) * 64 + dir * C_H + i] = h;
  }
  if (live && last_out) last_out[b * 64 + dir * C_H + i] = h;
}

// enc [B,64] -> out [B,n_out]; post[b] = out[b, n_out-1]
__global__ void __launch_bounds__(128) crnn_detect_kernel(const float* __restrict__ enc, const float* __restrict__ w1t,
                                                          const float* __restrict__ b1, const float* __restrict__ w2,
                                                          const float* __restrict__ b2, int n_out,
                                                          float* __restrict__ out, float* __restrict__ post,
                                                          int64_t B, const int32_t* __restrict__ n_dev) {
  __shared__ float w1s[64][64];
  __shared__ float4 es[4][64];      // [warp][k] = input k of the warp's FOUR windows
  __shared__ float hs[4][4][64];    // [warp][window][unit]
  for (int i = threadIdx.x; i < 64 * 64; i += 128) (&w1s[0][0])[i] = w1t[i];
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  const int64_t nB = n_dev ? (int64_t)*n_dev : B;
  __syncthreads();
  // FOUR windows per warp and iteration: the kernel is bound by shared-memory wavefronts (per input k one broadcast of the
  // inputs + two rows of W1), and four windows share them (one window per warp: 154 us per 217 088 windows).  The block keeps
  // the 16 KB of W1 in shared memory for all its windows (with one block per 4 windows, re-staging W1 was 0.9 GB of L2
  // traffic per bench step and most of the kernel's time).
  for (int64_t b4 = ((int64_t)blockIdx.x * 4 + wl) * 4; b4 < nB; b4 += (int64_t)gridDim.x * 16) {
    float e0[4], e1[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const bool live = b4 + w < nB;
      e0[w] = live ? enc[(b4 + w) * 64 + lane] : 0.f;
      e1[w] = live ? enc[(b4 + w) * 64 + 32 + lane] : 0.f;
    }
    es[wl][lane] = make_float4(e0[0], e0[1], e0[2], e0[3]);
    es[wl][lane + 32] = make_float4(e1[0], e1[1], e1[2], e1[3]);
    __syncwarp();
    float a0[4], a1[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) { a0[w] = b1[lane]; a1[w] = b1[lane + 32]; }
#pragma unroll 8
    for (int k = 0; k < 64; ++k) {
      const float4 e = es[wl][k];
      const float w0 = w1s[k][lane], w1 = w1s[k][lane + 32];
      a0[0] = fmaf(w0, e.x, a0[0]); a1[0] = fmaf(w1, e.x, a1[0]);
      a0[1] = fmaf(w0, e.y, a0[1]); a1[1] = fmaf(w1, e.y, a1[1]);
      a0[2] = fmaf(w0, e.z, a0[2]); a1[2] = fmaf(w1, e.z, a1[2]);
      a0[3] = fmaf(w0, e.w, a0[3]); a1[3] = fmaf(w1, e.w, a1[3]);
    }
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      hs[wl][w][lane] = fmaxf(a0[w], 0.f);
      hs[wl][w][lane + 32] = fmaxf(a1[w], 0.f);
    }
    __syncwarp();
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const int64_t b = b4 + w;
      float z[2] = {0.f, 0.f};
      for (int o = 0; o < n_out; ++o) {
        float p = w2[o * 64 + lane] * hs[wl][w][lane];
        p = fmaf(w2[o * 64 + 32 + lane], hs[wl][w][lane + 32], p);
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) p += __shfl_xor_sync(0xffffffffu, p, s);
        z[o] = p + b2[o];
      }
      if (lane == 0 && b < nB) {
        if (n_out == 1) {
          float p = sigmoid_f(z[0]);
          if (out) out[b] = p;
          if (post) post[b] = p;
        } else {
          float m = fmaxf(z[0], z[1]);
          float e0_ = expf(z[0] - m), e1_ = expf(z[1] - m);
          float sden = e0_ + e1_;
          if (out) { out[b * 2] = e0_ / sden; out[b * 2 + 1] = e1_ / sden; }
          if (post) post[b] = e1_ / sden;
        }
      }
    }
    __syncwarp();
  }
}

static unsigned detect_grid(const wwb_ctx* ctx, int64_t B) {
  return (unsigned)std::min<int64_t>((B + 15) / 16, (int64_t)ctx->sm_count * 16);   // 4 warps x 4 windows per block and iteration
}

int crnn_simt_detect(wwb_ctx* ctx, const float* enc, int64_t B, float* out, cudaStream_t st) {
  if (B == 0) return WWB_OK;
  const CrnnWeights& W = ctx->crnn;
  crnn_detect_kernel<<<detect_grid(ctx, B), 128, 0, st>>>(enc, W.det1_w, W.det1_b, W.det2_w, W.det2_b,
                                                             ctx->n_out, out, nullptr, B, nullptr);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int crnn_simt_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out, float* post,
                         cudaStream_t st) {
  const int64_t B = wm.n_win;
  if (B == 0) return WWB_OK;
  const CrnnWeights& W = ctx->crnn;
  const CrnnGeom geo = crnn_geom(ctx->L);
  const int T = geo.T;
  // chunk the batch so the intermediates stay bounded (xw: 768 T bytes per window, 14.6 KB at L = 151)
  // a multiple of 128 windows x 148 SMs (the recurrence kernel's wave)
  int64_t chunk = 37888;
  if (const char* e = getenv("WWB_CRNN_CHUNK")) chunk = std::max<int64_t>(128, atoll(e));
  // sliding-window batches on the tensor-core path share the conv / GRU-1 projection columns between windows
  // (crnn_tc.cu, CrnnShare); chunks are then whole streams
  CrnnShare sh;
  // (WWB_CRNN_NO_SHARE=1 forces the per-window path: used by the tests to check that both give identical bits)
  const char* no_share = getenv("WWB_CRNN_NO_SHARE");
  const bool shared = ctx->precision != WWB_PREC_F32 && !(no_share && no_share[0] == '1') && crnn_share_plan(wm, ctx->L, &sh);
  // streaming pushes (device-side window count): one chunk - the kernels clamp to *n_win_dev, which chunks would have to
  // offset; wwb_stream_alloc bounds streams x frames per push and sizes these workspaces up front
  if (wm.n_win_dev) chunk = std::max<int64_t>(chunk, (B + 127) / 128 * 128);
  int64_t chunk_streams = 0;
  if (shared) {
    // intermediates are ~7.6 KB per window here (xwS 2.7 KB + packed layer-1 output 4.9 KB): chunks of up to 512 K windows
    // (4 GB); measured on the bench shape, one chunk of 217 K windows is 15 % faster than six of 37 K (fewer ragged waves)
    if (!getenv("WWB_CRNN_CHUNK")) chunk = 524288;
    chunk_streams = std::min(std::max<int64_t>(1, chunk / sh.wps), sh.n_streams);
    chunk = chunk_streams * sh.wps;
  }
  void *conv = nullptr, *xw, *s1, *enc_ws, *xws = nullptr;
  int rc;
  // the 48.6 KB/window conv intermediate exists only on the fp32 validation path (1.8 GB per chunk)
  const int n_var = 1 + __builtin_popcount(geo.padmask);   // conv-weight variants of the shared-column path
  if (ctx->precision == WWB_PREC_F32 && (rc = workspace(ctx, 1, (size_t)std::min(B, chunk) * T * C_FEAT * 4, &conv))) return rc;
  if (shared && (rc = workspace(ctx, 1, n_var * crnn_share_xws_bytes(sh, chunk_streams), &xws))) return rc;
  if ((rc = workspace(ctx, 2, shared ? 16 : (size_t)((std::min(B, chunk) + 127) / 128 * 128) * T * 2 * C_G * 4, &xw))) return rc;
  // layer-1 output: fp32 [B, T, 64] (fp32 path) or the packed fp16 hi/lo operand of the fused layer-2 kernel (same bytes per value)
  if ((rc = workspace(ctx, 3, std::max((size_t)std::min(B, chunk) * T * 64 * 4, crnn_seq_packed_bytes(std::min(B, chunk), T)), &s1))) return rc;
  if ((rc = workspace(ctx, 4, (size_t)std::min(B, chunk) * 64 * 4, &enc_ws))) return rc;
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int64_t nb = std::min(chunk, B - b0);
    WinMap sub = wm;
    sub.n_win = nb;
    sub.b0 = wm.b0 + b0;
    if (shared) {   // the chunk's streams become streams 0.. of the sub-batch
      sub.mel = wm.mel + (b0 / sh.wps) * (int64_t)wm.ring * kMel;
      sub.b0 = 0;
    }
    float* enc = enc_out ? enc_out + b0 * 64 : (float*)enc_ws;
    const int64_t M = nb * T;
    // both directions of a layer share one GEMM: Wt = [in][192]
    const bool tc = ctx->precision != WWB_PREC_F32;
    if (shared) {
      // interior columns once per position, then each padded column (same strips, masked conv weights)
      const size_t vbytes = crnn_share_xws_bytes(sh, nb / sh.wps);
      for (int v = crnn_share_first_variant(sh); v < n_var; ++v)
        if ((rc = crnn_front_tc(ctx, sub, (float*)((unsigned char*)xws + v * vbytes), st, 1, &sh, v))) return rc;
    } else if (tc) {
      if ((rc = crnn_front_tc(ctx, sub, (float*)xw, st))) return rc;
    } else {
      const size_t xs_bytes = (size_t)(8 * T + 12) * C_XF * sizeof(float);
      WWB_CUDA(ctx, cudaFuncSetAttribute(crnn_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xs_bytes));
      crnn_conv_kernel<<<(unsigned)nb, 256, xs_bytes, st>>>(sub, W.conv_w, W.conv_b, (float*)conv, ctx->L, T, geo.pad_lo);
      WWB_CHECK_LAUNCH(ctx);
      sgemm_bias_kernel<<<dim3((unsigned)((M + 63) / 64), 3), 256, 0, st>>>((float*)conv, W.gru_w[0], W.gru_bi[0],
                                                                            (float*)xw, M, 2 * C_G, C_FEAT);
      WWB_CHECK_LAUNCH(ctx);
    }
    if (tc) {
      // layer 1 leaves its output as the packed A operand of layer 2's input projection, which the layer-2 kernel computes itself
      if ((rc = gru_rec_tc(ctx, 0, (float*)xw, nullptr, nullptr, nb, wm.n_win_dev, st, (float*)xws, &sh, (unsigned char*)s1))) return rc;
      if ((rc = gru2_fused_tc(ctx, (unsigned char*)s1, enc, nb, wm.n_win_dev, st))) return rc;
    } else {
      gru_rec_kernel<<<(unsigned)((nb + 3) / 4), 256, 0, st>>>((float*)xw, W.gru_u[0], W.gru_br[0], W.gru_u[1],
                                                              W.gru_br[1], (float*)s1, nullptr, nb, wm.n_win_dev, T);
      WWB_CHECK_LAUNCH(ctx);
      sgemm_bias_kernel<<<dim3((unsigned)((M + 63) / 64), 3), 256, 0, st>>>((float*)s1, W.gru_w[2], W.gru_bi[2],
                                                                            (float*)xw, M, 2 * C_G, 64);
      WWB_CHECK_LAUNCH(ctx);
      gru_rec_kernel<<<(unsigned)((nb + 3) / 4), 256, 0, st>>>((float*)xw, W.gru_u[2], W.gru_br[2], W.gru_u[3],
                                                              W.gru_br[3], nullptr, enc, nb, wm.n_win_dev, T);
      WWB_CHECK_LAUNCH(ctx);
    }
    if (det_out || post) {
      crnn_detect_kernel<<<detect_grid(ctx, nb), 128, 0, st>>>(
          enc, W.det1_w, W.det1_b, W.det2_w, W.det2_b, ctx->n_out,
          det_out ? det_out + b0 * ctx->n_out : nullptr, post ? post + b0 : nullptr, nb, wm.n_win_dev);
      WWB_CHECK_LAUNCH(ctx);
    }
  }
  return WWB_OK;
}

}  // namespace wwb
