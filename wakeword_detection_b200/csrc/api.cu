// C ABI of wwb200 (include/wwb200.h): context, weight upload, entry points.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace wwb {

std::string g_create_error;

int fail(wwb_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_error = buf;
  return code;
}

int workspace(wwb_ctx* ctx, int i, size_t bytes, void** out) {
  if (bytes == 0) bytes = 16;
  if (ctx->ws_bytes[i] < bytes) {
    if (ctx->ws[i]) {
      // the old buffer may still be in use by enqueued work
      WWB_CUDA(ctx, cudaDeviceSynchronize());
      WWB_CUDA(ctx, cudaFree(ctx->ws[i]));
      ctx->ws[i] = nullptr;
      ctx->ws_bytes[i] = 0;
    }
    size_t want = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&ctx->ws[i], want);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(ctx, WWB_ERR_ALLOC, "cudaMalloc of %zu bytes (workspace %d) failed: %s", want, i,
                  cudaGetErrorString(e));
    }
    ctx->ws_bytes[i] = want;
  }
  *out = ctx->ws[i];
  return WWB_OK;
}

template <typename T>
static int upload(wwb_ctx* ctx, const std::vector<T>& host, T** dev) {
  void* p = nullptr;
  size_t bytes = std::max<size_t>(host.size() * sizeof(T), 16);
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return fail(ctx, WWB_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  ctx->owned.push_back(p);
  if (!host.empty()) WWB_CUDA(ctx, cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
  *dev = (T*)p;
  return WWB_OK;
}

template <typename T>
static int dalloc(wwb_ctx* ctx, size_t n, T** dev) {
  void* p = nullptr;
  size_t bytes = std::max<size_t>(n * sizeof(T), 16);
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return fail(ctx, WWB_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  ctx->owned.push_back(p);
  WWB_CUDA(ctx, cudaMemset(p, 0, bytes));
  *dev = (T*)p;
  return WWB_OK;
}

// transposed copy: src [rows][cols] -> dst [cols][rows]
static std::vector<float> transposed(const float* src, int rows, int cols) {
  std::vector<float> d((size_t)rows * cols);
  for (int r = 0; r < rows; ++r)
    for (int c = 0; c < cols; ++c) d[(size_t)c * rows + r] = src[(size_t)r * cols + c];
  return d;
}

static int build_filter_tables(wwb_ctx* ctx, const wwb_weights* w) {
  const double PI = 3.14159265358979323846;
  // fp64 tables of the FFT (fft64.cuh): np.hanning(512) = 0.5 - 0.5 cos(2 pi n / 511) with the 1/2 of the real-FFT
  // split folded in; W256^k, W512^k
  std::vector<double> hann(kFFT);
  for (int n = 0; n < kFFT; ++n) hann[n] = 0.5 * (0.5 - 0.5 * cos(2.0 * PI * n / (kFFT - 1)));
  std::vector<double2> t256(256), t512(256);
  for (int k = 0; k < 256; ++k) t256[k] = make_double2(cos(2 * PI * k / 256), -sin(2 * PI * k / 256));
  for (int k = 0; k < 256; ++k) t512[k] = make_double2(cos(2 * PI * k / 512), -sin(2 * PI * k / 512));
  int rc;
  if ((rc = upload(ctx, hann, &ctx->hann))) return rc;
  if ((rc = upload(ctx, t256, &ctx->tw256))) return rc;
  if ((rc = upload(ctx, t512, &ctx->tw512))) return rc;

  // mel matrix -> segments of <= kSegTaps non-zeros, bands contiguous
  std::vector<int> seg_band, seg_first, seg_count, band_seg0(kMel + 1), tap_bin;
  std::vector<float> tap_w, bias(kMel);
  for (int m = 0; m < kMel; ++m) {
    band_seg0[m] = (int)seg_band.size();
    bias[m] = w->mel_b ? w->mel_b[m] : 0.f;
    int in_seg = 0, last = -2;
    for (int k = 0; k < kBins; ++k) {
      float v = w->mel_w[(size_t)m * kBins + k];
      if (v == 0.f) continue;
      // a segment is a run of CONSECUTIVE bins (filter.cu reads it as seg_bin0 + t): a gap in the row starts a new one
      if (in_seg == 0 || in_seg == kSegTaps || k != last + 1) {
        seg_band.push_back(m);
        seg_first.push_back((int)tap_bin.size());
        seg_count.push_back(0);
        in_seg = 0;
      }
      last = k;
      tap_bin.push_back(k);
      tap_w.push_back(v);
      seg_count.back()++;
      in_seg++;
    }
  }
  band_seg0[kMel] = (int)seg_band.size();
  if (seg_band.size() > (size_t)kMaxSeg)
    return fail(ctx, WWB_ERR_ARG, "mel matrix has %d segments (runs of up to %d consecutive non-zero bins); at most %d supported",
                (int)seg_band.size(), kSegTaps, kMaxSeg);
  MelTables& mt = ctx->mel;
  mt.n_seg = (int)seg_band.size();
  mt.n_tap = (int)tap_bin.size();
  if ((rc = upload(ctx, seg_band, &mt.seg_band))) return rc;
  if ((rc = upload(ctx, seg_first, &mt.seg_first))) return rc;
  if ((rc = upload(ctx, seg_count, &mt.seg_count))) return rc;
  if ((rc = upload(ctx, band_seg0, &mt.band_seg0))) return rc;
  if ((rc = upload(ctx, tap_bin, &mt.tap_bin))) return rc;
  if ((rc = upload(ctx, tap_w, &mt.tap_w))) return rc;
  if ((rc = upload(ctx, bias, &mt.bias))) return rc;
  return WWB_OK;
}

// floor(log2 x) for a finite x > 0
static int floor_log2(double x) {
  int e;
  frexp(x, &e);
  return e - 1;
}

static float max_abs(const float* p, size_t n) {
  float m = 0.f;
  for (size_t i = 0; i < n; ++i)
    if (std::isfinite(p[i])) m = std::max(m, fabsf(p[i]));
  return m;
}

static void scale(std::vector<float>& v, float s) {
  for (float& x : v) x *= s;
}

static int build_crnn(wwb_ctx* ctx, const wwb_weights* w) {
  CrnnWeights& C = ctx->crnn;
  int rc;
  if (!w->conv_w || !w->conv_b || !w->det1_w || !w->det2_w) return fail(ctx, WWB_ERR_ARG, "CRNN weights missing");
  for (int i = 0; i < 4; ++i)
    if (!w->gru_w[i] || !w->gru_u[i] || !w->gru_bi[i] || !w->gru_br[i]) return fail(ctx, WWB_ERR_ARG, "GRU weights missing");
  // Power-of-two rescale (DESIGN.md §4): conv weights and bias times sigma, layer-1 input weights over sigma.  Exact in
  // fp32 (ReLU is positively homogeneous), so both paths compute the same function.  sigma = 2^floor(log2(g / c) / 2)
  // balances the largest layer-1 weight g against the largest conv weight c, so that the conv activations and the
  // layer-1 weights, fp16 hi/lo operands on the tensor cores, stay in fp16's normal range for models trained at any
  // feature scale.  Every power-of-two member of the family (conv * s, layer-1 / s) gets the same weights here.
  std::vector<float> conv_w(w->conv_w, w->conv_w + 32 * 100), conv_b(w->conv_b, w->conv_b + 32);
  std::vector<float> w1[2] = {std::vector<float>(w->gru_w[0], w->gru_w[0] + 96 * 640),
                              std::vector<float>(w->gru_w[1], w->gru_w[1] + 96 * 640)};
  {
    const float c = max_abs(conv_w.data(), conv_w.size());
    const float g = std::max(max_abs(w1[0].data(), w1[0].size()), max_abs(w1[1].data(), w1[1].size()));
    if (c > 0.f && g > 0.f) {
      const int e = floor_log2((double)g / (double)c);
      const float sigma = ldexpf(1.f, e >= 0 ? e / 2 : -((1 - e) / 2));
      scale(conv_w, sigma);
      scale(conv_b, sigma);
      scale(w1[0], 1.f / sigma);
      scale(w1[1], 1.f / sigma);
    }
  }
  const float* gru_w[4] = {w1[0].data(), w1[1].data(), w->gru_w[2], w->gru_w[3]};
  // conv [32][100] -> [100][32]
  if ((rc = upload(ctx, transposed(conv_w.data(), 32, 100), &C.conv_w))) return rc;
  if ((rc = upload(ctx, conv_b, &C.conv_b))) return rc;
  if ((rc = upload(ctx, crnn_pack_conv(conv_w.data(), w->mel_length), &C.tc_conv))) return rc;
  for (int layer = 0; layer < 2; ++layer) {
    const int in = layer == 0 ? 640 : 64;
    // both directions side by side: Wt [in][192], bias [192]
    std::vector<float> wt((size_t)in * 192), bi(192);
    for (int dir = 0; dir < 2; ++dir) {
      const float* src = gru_w[layer * 2 + dir];   // [96][in]
      for (int n = 0; n < 96; ++n) {
        bi[dir * 96 + n] = w->gru_bi[layer * 2 + dir][n];
        for (int k = 0; k < in; ++k) wt[(size_t)k * 192 + dir * 96 + n] = src[(size_t)n * in + k];
      }
    }
    if ((rc = upload(ctx, wt, &C.gru_w[layer * 2]))) return rc;
    if ((rc = upload(ctx, bi, &C.gru_bi[layer * 2]))) return rc;
    {  // tensor-core path: [192][in] (fwd units then bwd units), split into fp16 hi/lo stages
      std::vector<float> w_nk((size_t)192 * in);
      for (int dir = 0; dir < 2; ++dir)
        memcpy(&w_nk[(size_t)dir * 96 * in], gru_w[layer * 2 + dir], sizeof(float) * 96 * in);
      if (layer == 0 && (rc = upload(ctx, crnn_pack_w1(w_nk.data()), &C.tc_w1))) return rc;
      if (layer == 1 && (rc = upload(ctx, crnn_pack_w2(w_nk.data()), &C.tc_w2))) return rc;
    }
    {  // tensor-core recurrence: packed U, candidate-gate bias, input bias with the z/r recurrent bias folded in
      if ((rc = upload(ctx, crnn_pack_u(w->gru_u[layer * 2], w->gru_u[layer * 2 + 1]), &C.tc_u[layer]))) return rc;
      std::vector<float> bh(64), bf(192);
      for (int dir = 0; dir < 2; ++dir)
        for (int n = 0; n < 96; ++n) {
          const float br = w->gru_br[layer * 2 + dir][n];
          if (n >= 64) bh[dir * 32 + n - 64] = br;
          bf[dir * 96 + n] = n < 64 ? bi[dir * 96 + n] + br : bi[dir * 96 + n];
        }
      if ((rc = upload(ctx, bh, &C.tc_bh[layer]))) return rc;
      if ((rc = upload(ctx, bf, &C.tc_bi[layer]))) return rc;
      if (layer == 1 && (rc = upload(ctx, crnn_reorder_bias2(bf.data()), &C.tc_bi2))) return rc;
    }
    for (int dir = 0; dir < 2; ++dir) {
      if ((rc = upload(ctx, transposed(w->gru_u[layer * 2 + dir], 96, 32), &C.gru_u[layer * 2 + dir]))) return rc;
      if ((rc = upload(ctx, std::vector<float>(w->gru_br[layer * 2 + dir], w->gru_br[layer * 2 + dir] + 96),
                       &C.gru_br[layer * 2 + dir]))) return rc;
    }
  }
  if ((rc = upload(ctx, transposed(w->det1_w, 64, 64), &C.det1_w))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->det1_b, w->det1_b + 64), &C.det1_b))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->det2_w, w->det2_w + 64 * ctx->n_out), &C.det2_w))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->det2_b, w->det2_b + ctx->n_out), &C.det2_b))) return rc;
  return WWB_OK;
}

static int build_wavenet(wwb_ctx* ctx, const wwb_weights* w) {
  WavenetWeights& N = ctx->wn;
  int rc;
  if (!w->in_w || !w->bn_mul || !w->sig_w || !w->tanh_w || !w->res_w || !w->skip_w || !w->dilation || !w->det1_w)
    return fail(ctx, WWB_ERR_ARG, "WaveNet weights missing");
  // Power-of-two rescale of the residual stream x (DESIGN.md §4): in_w, in_b, res_w and res_b times sigma, bn_mul over
  // sigma.  Exact in fp32, so both paths compute the same function.  The tensor-core path folds bn_mul into the gate
  // weights and feeds x itself as the fp16 hi/lo operand, so the split error depends on where the model sits in this
  // family.  sigma brings the largest |bn_mul| into [64, 128), the octave of the shipped model (sigma = 1 there), and
  // maps every power-of-two member of the family onto the same weights.
  std::vector<float> in_w(w->in_w, w->in_w + 16 * 40), in_b(w->in_b, w->in_b + 16), bn_mul(w->bn_mul, w->bn_mul + 24 * 16),
      res_w(w->res_w, w->res_w + 23 * 16 * 16), res_b(w->res_b, w->res_b + 23 * 16);
  const float bn_max = max_abs(bn_mul.data(), bn_mul.size());
  if (bn_max > 0.f) {
    const float sigma = ldexpf(1.f, floor_log2(bn_max) - 6);
    scale(in_w, sigma);
    scale(in_b, sigma);
    scale(res_w, sigma);
    scale(res_b, sigma);
    scale(bn_mul, 1.f / sigma);
  }
  if ((rc = upload(ctx, transposed(in_w.data(), 16, 40), &N.in_w))) return rc;
  if ((rc = upload(ctx, in_b, &N.in_b))) return rc;
  if ((rc = upload(ctx, bn_mul, &N.bn_mul))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->bn_add, w->bn_add + 24 * 16), &N.bn_add))) return rc;
  std::vector<float> gw(24 * 48 * 32), gb(24 * 32), rw(24 * 16 * 48, 0.f), rb(24 * 48, 0.f);
  for (int b = 0; b < 24; ++b) {
    N.dilation[b] = w->dilation[b];
    if (N.dilation[b] < 1 || N.dilation[b] > 8) return fail(ctx, WWB_ERR_ARG, "dilation %d unsupported", N.dilation[b]);
    for (int o = 0; o < 16; ++o) {
      gb[b * 32 + o] = w->tanh_b[b * 16 + o];
      gb[b * 32 + 16 + o] = w->sig_b[b * 16 + o];
      for (int tap = 0; tap < 3; ++tap)
        for (int i = 0; i < 16; ++i) {
          size_t src = (((size_t)b * 16 + o) * 3 + tap) * 16 + i;
          gw[((size_t)b * 48 + tap * 16 + i) * 32 + o] = w->tanh_w[src];
          gw[((size_t)b * 48 + tap * 16 + i) * 32 + 16 + o] = w->sig_w[src];
        }
    }
    for (int i = 0; i < 16; ++i) {
      if (b < 23)
        for (int o = 0; o < 16; ++o) rw[((size_t)b * 16 + i) * 48 + o] = res_w[((size_t)b * 16 + o) * 16 + i];
      for (int o = 0; o < 32; ++o) rw[((size_t)b * 16 + i) * 48 + 16 + o] = w->skip_w[((size_t)b * 32 + o) * 16 + i];
    }
    if (b < 23)
      for (int o = 0; o < 16; ++o) rb[b * 48 + o] = res_b[b * 16 + o];
    for (int o = 0; o < 32; ++o) rb[b * 48 + 16 + o] = w->skip_b[b * 32 + o];
  }
  {  // tensor-core blobs only when they can be packed; otherwise wwb_set_precision refuses tc / tc_fast
    std::vector<unsigned char> blocks = wavenet_pack_blocks(gw.data(), gb.data(), rw.data(), rb.data(), bn_mul.data(),
                                                            w->bn_add, N.dilation);
    std::vector<unsigned char> head = wavenet_pack_head(bn_mul.data(), w->bn_add, w->det1_w, w->det1_b, w->det2_w, w->det2_b);
    if (blocks.empty() || head.empty()) {
      const bool zero = std::find(bn_mul.begin(), bn_mul.end(), 0.f) != bn_mul.end();
      ctx->tc_refused = zero ? "WaveNet: a BatchNorm scale of 0 cannot be folded into the tensor-core weights; use precision f32"
                             : "WaveNet: a tensor-core operand (folded gate weight or bias, padding row -bn_add/bn_mul after "
                               "the rescale, or head weight) is outside the fp16 range; use precision f32";
    } else {
      if ((rc = upload(ctx, blocks, &N.tc_blocks))) return rc;
      if ((rc = upload(ctx, head, &N.tc_head))) return rc;
    }
  }
  if ((rc = upload(ctx, gw, &N.gate_w))) return rc;
  if ((rc = upload(ctx, gb, &N.gate_b))) return rc;
  if ((rc = upload(ctx, rw, &N.rs_w))) return rc;
  if ((rc = upload(ctx, rb, &N.rs_b))) return rc;
  memcpy(N.h_det1_b, w->det1_b, sizeof(N.h_det1_b));
  memcpy(N.h_det2_w, w->det2_w, sizeof(N.h_det2_w));
  memcpy(N.h_det2_b, w->det2_b, sizeof(N.h_det2_b));
  if ((rc = upload(ctx, transposed(w->det1_w, 32, 32), &N.det1_w))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->det1_b, w->det1_b + 32), &N.det1_b))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->det2_w, w->det2_w + 64), &N.det2_w))) return rc;
  if ((rc = upload(ctx, std::vector<float>(w->det2_b, w->det2_b + 2), &N.det2_b))) return rc;
  return WWB_OK;
}

static int run_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out, float* post,
                          cudaStream_t st) {
  if (ctx->kind == WWB_MODEL_NONE) return fail(ctx, WWB_ERR_STATE, "ctx holds a filter only (no encode/detect weights)");
  if (ctx->kind == WWB_MODEL_CRNN) return crnn_simt_posteriors(ctx, wm, enc_out, det_out, post, st);
  if (ctx->precision != WWB_PREC_F32) return wavenet_tc_posteriors(ctx, wm, enc_out, det_out, post, st);
  return wavenet_simt_posteriors(ctx, wm, enc_out, det_out, post, st);
}

}  // namespace wwb

using namespace wwb;

extern "C" {

int wwb_version(void) { return WWB_VERSION; }

const char* wwb_last_error(const wwb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int wwb_create(int device, const wwb_weights* w, int precision, wwb_ctx** out) {
  if (!out) return fail(nullptr, WWB_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (!w || !w->mel_w) return fail(nullptr, WWB_ERR_ARG, "weights missing");
  if (w->n_mel != kMel || w->n_bins != kBins)
    return fail(nullptr, WWB_ERR_ARG, "filter geometry %dx%d unsupported (expected %dx%d)", w->n_mel, w->n_bins, kMel, kBins);
  if (w->kind != WWB_MODEL_CRNN && w->kind != WWB_MODEL_WAVENET && w->kind != WWB_MODEL_NONE)
    return fail(nullptr, WWB_ERR_ARG, "bad model kind");
  if (w->kind == WWB_MODEL_CRNN && (w->mel_length < kCrnnMinL || w->mel_length > kCrnnMaxL))
    return fail(nullptr, WWB_ERR_ARG, "CRNN window of %d frames unsupported (expected %d..%d)", w->mel_length, kCrnnMinL, kCrnnMaxL);
  if (w->kind == WWB_MODEL_WAVENET && (w->mel_length < 17 || w->mel_length > 182))
    return fail(nullptr, WWB_ERR_ARG, "WaveNet window of %d frames unsupported (expected 17..182)", w->mel_length);
  if (w->kind == WWB_MODEL_CRNN && w->n_out != 1 && w->n_out != 2)
    return fail(nullptr, WWB_ERR_ARG, "CRNN n_out %d unsupported (expected 1 or 2)", w->n_out);
  if (w->kind == WWB_MODEL_WAVENET && w->n_out != 2)
    return fail(nullptr, WWB_ERR_ARG, "WaveNet n_out %d unsupported (expected 2: the head is a 2-way softmax)", w->n_out);
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    return fail(nullptr, WWB_ERR_CUDA, "no CUDA device available (%s); wwb200 has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  }
  if (device < 0 || device >= n_dev) return fail(nullptr, WWB_ERR_ARG, "device %d out of range (0..%d)", device, n_dev - 1);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, WWB_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, WWB_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, WWB_ERR_CUDA, "device %d is sm_%d%d; wwb200 is built for sm_100a (B200) only", device, prop.major, prop.minor);
  wwb_ctx* ctx = new wwb_ctx();
  ctx->device = device;
  ctx->kind = w->kind;
  ctx->L = w->mel_length;
  ctx->n_out = w->n_out;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->mel_floor = w->mel_floor;
  ctx->mel_log_offset = w->mel_log_offset;
  ctx->mel_scale = w->mel_scale;
  ctx->mel_w_host.assign(w->mel_w, w->mel_w + (size_t)kMel * kBins);
  ctx->mel_b_host.assign(kMel, 0.f);
  if (w->mel_b) ctx->mel_b_host.assign(w->mel_b, w->mel_b + kMel);
  int rc = build_filter_tables(ctx, w);
  if (!rc && w->kind == WWB_MODEL_CRNN) rc = build_crnn(ctx, w);
  if (!rc && w->kind == WWB_MODEL_WAVENET) rc = build_wavenet(ctx, w);
  if (!rc) rc = wwb_set_precision(ctx, precision);
  if (rc) {
    g_create_error = ctx->err;
    wwb_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return WWB_OK;
}

int wwb_destroy(wwb_ctx* ctx) {
  if (!ctx) return WWB_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  host_pipe_destroy(ctx);
  for (int k = 0; k < 2; ++k) {
    if (ctx->stage_host[k]) cudaFreeHost(ctx->stage_host[k]);
    if (ctx->stage_done[k]) cudaEventDestroy(ctx->stage_done[k]);
  }
  for (void* p : ctx->owned) cudaFree(p);
  for (int i = 0; i < 8; ++i)
    if (ctx->ws[i]) cudaFree(ctx->ws[i]);
  delete ctx;
  return WWB_OK;
}

int wwb_set_precision(wwb_ctx* ctx, int precision) {
  if (!ctx) return WWB_ERR_ARG;
  if (precision != WWB_PREC_F32 && precision != WWB_PREC_TC && precision != WWB_PREC_TC_FAST)
    return fail(ctx, WWB_ERR_ARG, "unknown precision %d", precision);
  if (precision != WWB_PREC_F32 && !ctx->tc_refused.empty()) return fail(ctx, WWB_ERR_ARG, "%s", ctx->tc_refused.c_str());
  ctx->precision = precision;
  return WWB_OK;
}

int wwb_sync(wwb_ctx* ctx, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  WWB_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream));
  return WWB_OK;
}

int64_t wwb_num_frames(int64_t n) { return n < kFFT ? 0 : (n - kFFT) / kHop + 1; }

int64_t wwb_num_windows(const wwb_ctx* ctx, int64_t n_frames, int hop) {
  if (!ctx || hop < 1) return 0;
  return n_frames < ctx->L ? 0 : (n_frames - ctx->L) / hop + 1;
}

int64_t wwb_stream_granule(const wwb_ctx* ctx, int64_t n_frames, int hop) {
  if (!ctx || ctx->kind != WWB_MODEL_CRNN || ctx->precision == WWB_PREC_F32) return 1;
  WinMap wm;
  memset(&wm, 0, sizeof(wm));
  wm.win_per_stream = (int)wwb_num_windows(ctx, n_frames, hop);
  wm.n_win = wm.win_per_stream;
  wm.hop = hop;
  wm.ring = (int)n_frames;
  CrnnShare g;
  if (wm.win_per_stream < 1 || !crnn_share_plan(wm, ctx->L, &g)) return 1;
  const int64_t per_stream = (int64_t)g.q * g.nsp;   // strip tiles per stream and conv-weight variant (crnn_tc.cu)
  return ctx->sm_count % per_stream == 0 ? ctx->sm_count / per_stream : 1;
}

int wwb_filter(wwb_ctx* ctx, const void* pcm, int dtype, int64_t S, int64_t N, int64_t pitch, float a, float* mel,
               void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  if ((!pcm || !mel) && S > 0 && wwb_num_frames(N) > 0) return fail(ctx, WWB_ERR_ARG, "NULL buffer");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  return launch_filter(ctx, pcm, dtype, S, N, pitch, a, mel, (cudaStream_t)stream);
}

static WinMap batch_map(const wwb_ctx* ctx, const float* mel, int64_t S, int64_t F, int hop) {
  WinMap wm;
  memset(&wm, 0, sizeof(wm));
  wm.mel = mel;
  wm.win_per_stream = (int)wwb_num_windows(ctx, F, hop);
  wm.n_win = S * wm.win_per_stream;
  wm.hop = hop;
  wm.ring = (int)F;
  wm.n_streams = S;
  return wm;
}

int wwb_encode(wwb_ctx* ctx, const float* mel_windows, int64_t B, float* enc, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  if (B < 0 || (B > 0 && (!mel_windows || !enc))) return fail(ctx, WWB_ERR_ARG, "bad encode arguments");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  WinMap wm = batch_map(ctx, mel_windows, B, ctx->L, 1);
  return run_posteriors(ctx, wm, enc, nullptr, nullptr, (cudaStream_t)stream);
}

int wwb_mel_from_magnitude(wwb_ctx* ctx, const float* mag, int64_t B, float* mel, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  if (B < 0 || (B > 0 && (!mag || !mel))) return fail(ctx, WWB_ERR_ARG, "bad arguments");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  return launch_mel_from_mag(ctx, mag, B, mel, (cudaStream_t)stream);
}

int wwb_detect(wwb_ctx* ctx, const float* enc, int64_t B, float* out, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  if (ctx->kind == WWB_MODEL_NONE) return fail(ctx, WWB_ERR_STATE, "ctx holds a filter only");
  if (B < 0 || (B > 0 && (!enc || !out))) return fail(ctx, WWB_ERR_ARG, "bad detect arguments");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->kind == WWB_MODEL_CRNN) return crnn_simt_detect(ctx, enc, B, out, (cudaStream_t)stream);
  return wavenet_simt_detect(ctx, enc, B, out, (cudaStream_t)stream);
}

int wwb_posteriors(wwb_ctx* ctx, const float* mel, int64_t S, int64_t F, int hop, float* post, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  if (S < 0 || F < 0 || hop < 1) return fail(ctx, WWB_ERR_ARG, "bad posteriors geometry");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  WinMap wm = batch_map(ctx, mel, S, F, hop);
  if (wm.n_win == 0) return WWB_OK;
  if (!mel || !post) return fail(ctx, WWB_ERR_ARG, "NULL buffer");
  return run_posteriors(ctx, wm, nullptr, nullptr, post, (cudaStream_t)stream);
}

int wwb_pipeline(wwb_ctx* ctx, const void* pcm, int dtype, int64_t S, int64_t N, int64_t pitch, float a, int hop,
                 float* post, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t F = wwb_num_frames(N);
  void* mel;
  int rc = workspace(ctx, 0, (size_t)S * F * kMel * sizeof(float), &mel);
  if (rc) return rc;
  if ((rc = wwb_filter(ctx, pcm, dtype, S, N, pitch, a, (float*)mel, stream))) return rc;
  return wwb_posteriors(ctx, (const float*)mel, S, F, hop, post, stream);
}

int wwb_eval_counts(wwb_ctx* ctx, const float* post, const int64_t* seg_off, int64_t n_seg, const int32_t* halo_lo,
                    const int32_t* halo_hi, int64_t n_total, const double* thr, int n_thr, int mode, int smooth,
                    int64_t* counts, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  if (!thr || !counts || (n_seg > 0 && (!seg_off || (n_total > 0 && !post)))) return fail(ctx, WWB_ERR_ARG, "NULL buffer");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  return launch_eval_counts(ctx, post, seg_off, n_seg, halo_lo, halo_hi, n_total, thr, n_thr, mode, smooth, counts,
                            (cudaStream_t)stream);
}

// the explicit window lists of a streaming push over S entries (filled by the plan kernel, filter.cu); entry i is stream
// ids[i] of the ring (device table, NULL = i)
static WinMap stream_map(const wwb_ctx* ctx, int64_t S, const int32_t* ids) {
  WinMap wm;
  memset(&wm, 0, sizeof(wm));
  wm.mel = ctx->st.mel_ring;
  wm.stream_slot = ids;
  wm.win_stream = ctx->st.win_stream;
  wm.win_start = ctx->st.win_start;
  wm.n_win_dev = ctx->st.n_win;
  wm.n_win = S * ctx->st.max_frames;
  wm.n_streams = S;
  wm.win_per_stream = 1;
  wm.hop = 1;
  wm.ring = ctx->st.ring;
  return wm;
}

int wwb_stream_alloc(wwb_ctx* ctx, int64_t max_streams, int64_t max_chunk) {
  if (!ctx) return WWB_ERR_ARG;
  if (max_streams < 1 || max_chunk < 1 || max_chunk > 16000) return fail(ctx, WWB_ERR_ARG, "bad stream geometry");
  if (ctx->st.max_streams) return fail(ctx, WWB_ERR_STATE, "stream state already allocated");
  if (max_streams * ((max_chunk - 1) / kHop + 1) > (1 << 20))
    return fail(ctx, WWB_ERR_ARG, "%lld streams x %lld frames per push exceed 2^20 windows per push: split the streams over several contexts",
                (long long)max_streams, (long long)((max_chunk - 1) / kHop + 1));
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  StreamState& s = ctx->st;
  s.max_chunk = max_chunk;
  s.pend_cap = kFFT;
  s.max_frames = (int)((max_chunk - 1) / kHop + 1);
  s.ring = ctx->L + s.max_frames;
  int rc;
  const size_t S = (size_t)max_streams;
  if ((rc = dalloc(ctx, S * s.pend_cap, &s.pending))) return rc;
  if ((rc = dalloc(ctx, S, &s.n_pending))) return rc;
  if ((rc = dalloc(ctx, S, &s.prev_sample))) return rc;
  if ((rc = dalloc(ctx, S * s.ring * kMel, &s.mel_ring))) return rc;
  if ((rc = dalloc(ctx, S, &s.ring_head))) return rc;
  if ((rc = dalloc(ctx, S, &s.post_max))) return rc;
  if ((rc = dalloc(ctx, S, &s.was_speech))) return rc;
  if ((rc = dalloc(ctx, S, &s.n_new))) return rc;
  if ((rc = dalloc(ctx, S * s.max_frames, &s.win_stream))) return rc;
  if ((rc = dalloc(ctx, S * s.max_frames, &s.win_start))) return rc;
  if ((rc = dalloc(ctx, S, &s.win_slot))) return rc;
  if ((rc = dalloc(ctx, 1, &s.n_win))) return rc;
  if ((rc = dalloc(ctx, S * s.max_frames, &s.win_post))) return rc;
  if ((rc = dalloc(ctx, stage_words(S), &s.tables))) return rc;
  if ((rc = dalloc(ctx, 2, &s.import_check))) return rc;
  // slot options: every threshold a quiet NaN (all bits set: the call's threshold), every slot listening
  if ((rc = dalloc(ctx, S, &ctx->opt.threshold))) return rc;
  if ((rc = dalloc(ctx, S, &ctx->opt.listening))) return rc;
  WWB_CUDA(ctx, cudaMemset(ctx->opt.threshold, 0xFF, S * sizeof(float)));
  WWB_CUDA(ctx, cudaMemset(ctx->opt.listening, 1, S));
  for (int k = 0; k < 2; ++k) {
    if (!ctx->stage_host[k]) WWB_CUDA(ctx, cudaHostAlloc((void**)&ctx->stage_host[k], stage_words(S) * sizeof(int32_t), cudaHostAllocDefault));
    if (!ctx->stage_done[k]) WWB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->stage_done[k], cudaEventDisableTiming));
  }
  ctx->id_seen.assign(S, 0);
  s.max_streams = max_streams;
  // Size the encoder's workspaces for the largest push now (a dry run over zero windows: n_win is 0 after dalloc), so that
  // wwb_stream_push cannot fail on an allocation AFTER its filter stage has consumed the chunk and advanced the
  // per-stream state.
  if (ctx->kind != WWB_MODEL_NONE) {
    WinMap wm = stream_map(ctx, max_streams, nullptr);
    if ((rc = run_posteriors(ctx, wm, nullptr, nullptr, s.win_post, 0))) { s.max_streams = 0; return rc; }
    WWB_CUDA(ctx, cudaStreamSynchronize(0));
  }
  return WWB_OK;
}

int wwb_stream_max_frames(const wwb_ctx* ctx) { return ctx ? ctx->st.max_frames : 0; }

// filter -> encoder -> trigger bookkeeping over S entries (ids / off as in launch_stream_filter; NULL = dense push)
static int stream_push(wwb_ctx* ctx, const int16_t* pcm, int64_t S, int64_t n, const int32_t* ids, const int32_t* off,
                       const uint8_t* is_speech, const uint8_t* is_active, float a, float threshold, float* post_out,
                       int32_t* n_post_out, uint8_t* trigger_out, float* post_max_out, cudaStream_t st) {
  int rc = launch_stream_filter(ctx, pcm, S, n, ids, off, is_speech, is_active, a, st);
  if (rc) return rc;
  WinMap wm = stream_map(ctx, S, ids);
  if ((rc = run_posteriors(ctx, wm, nullptr, nullptr, ctx->st.win_post, st))) return rc;
  return launch_stream_finish(ctx, S, ids, is_speech, is_active, threshold, post_out, n_post_out, trigger_out,
                              post_max_out, st);
}

// The state a streaming call needs: wwb_stream_alloc, with `pipeline` wwb_context_alloc too, and with `model` encoder
// weights (not a filter-only ctx).
static int check_state(wwb_ctx* ctx, bool pipeline, bool model) {
  if (!ctx->st.max_streams) return fail(ctx, WWB_ERR_STATE, "wwb_stream_alloc has not been called");
  if (pipeline && !ctx->cs.max_streams) return fail(ctx, WWB_ERR_STATE, "wwb_context_alloc has not been called");
  if (model && ctx->kind == WWB_MODEL_NONE) return fail(ctx, WWB_ERR_STATE, "ctx holds a filter only (no encode/detect weights)");
  return WWB_OK;
}

// The checks of a dense push (`pipeline`: a dense step): the state allocated, S in [1, max_streams], n in [1, max_chunk],
// pcm present, then a model (a NULL pcm is reported before a filter-only ctx).
static int check_dense(wwb_ctx* ctx, bool pipeline, int64_t S, int64_t n, const int16_t* pcm) {
  const int64_t cap = pipeline ? ctx->cs.max_streams : ctx->st.max_streams;
  if (!cap) return check_state(ctx, pipeline, true);
  if (S < 1 || S > cap) return fail(ctx, WWB_ERR_STATE, "n_streams %lld outside [1, %lld]", (long long)S, (long long)cap);
  if (n < 1 || n > ctx->st.max_chunk)
    return fail(ctx, WWB_ERR_STATE, "chunk of %lld samples outside [1, %lld]", (long long)n, (long long)ctx->st.max_chunk);
  if (!pcm) return fail(ctx, WWB_ERR_ARG, "NULL pcm");
  return check_state(ctx, pipeline, true);
}

// The table checks of every call that names slots by id (the indexed pushes and steps, wwb_stream_export /
// wwb_stream_import; a rejected call touches nothing): n_ids in [1, cap] (cap: max_streams of allocated state), the id
// table and the call's device buffer `buf` present (and for a push, `push` true, the length table), distinct ids in
// [0, cap) and for a push chunk lengths in [1, max_chunk].
static int check_tables(wwb_ctx* ctx, int64_t cap, const int32_t* ids, int64_t n_ids, const int32_t* len, bool push,
                        const void* buf) {
  StreamState& s = ctx->st;
  if (n_ids < 1 || n_ids > cap)
    return fail(ctx, WWB_ERR_STATE, "n_ids %lld outside [1, %lld]", (long long)n_ids, (long long)cap);
  if (!ids || (push && !len)) return fail(ctx, WWB_ERR_ARG, push ? "NULL id or length table" : "NULL id table");
  if (!buf) return fail(ctx, WWB_ERR_ARG, push ? "NULL pcm" : "NULL records");
  int64_t marked = 0;
  char why[160] = "";
  for (int64_t i = 0; i < n_ids; ++i) {
    const int32_t id = ids[i];
    if (id < 0 || id >= cap) {
      snprintf(why, sizeof(why), "id %d of entry %lld outside [0, %lld)", id, (long long)i, (long long)cap);
      break;
    }
    if (ctx->id_seen[id]) {
      snprintf(why, sizeof(why), push ? "id %d named twice (entry %lld): push again to feed a stream more samples"
                                      : "id %d named twice (entry %lld)", id, (long long)i);
      break;
    }
    ctx->id_seen[id] = 1;
    ++marked;
    if (push && (len[i] < 1 || len[i] > s.max_chunk)) {
      snprintf(why, sizeof(why), "chunk of %d samples (entry %lld) outside [1, %lld]", len[i], (long long)i,
               (long long)s.max_chunk);
      break;
    }
  }
  for (int64_t i = 0; i < marked; ++i) ctx->id_seen[ids[i]] = 0;
  if (why[0]) return fail(ctx, WWB_ERR_STATE, "%s", why);
  return WWB_OK;
}

// The next page-locked staging slot, once its previous copy has finished: waiting only for that slot keeps the host from
// blocking behind the call before.  stage_copy sends its first n words to st.tables on `st`.
static int stage_slot(wwb_ctx* ctx, int32_t** h) {
  WWB_CUDA(ctx, cudaEventSynchronize(ctx->stage_done[ctx->stage_next]));
  *h = ctx->stage_host[ctx->stage_next];
  return WWB_OK;
}

static int stage_copy(wwb_ctx* ctx, int64_t n, cudaStream_t st) {
  const int k = ctx->stage_next;
  WWB_CUDA(ctx, cudaMemcpyAsync(ctx->st.tables, ctx->stage_host[k], (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  WWB_CUDA(ctx, cudaEventRecord(ctx->stage_done[k], st));
  ctx->stage_next = 1 - k;
  return WWB_OK;
}

// Copies checked slot ids (and, with `len`, the chunk offsets) to st.tables on `st`.
static int stage_tables(wwb_ctx* ctx, const int32_t* ids, int64_t n_ids, const int32_t* len, cudaStream_t st) {
  int32_t* h;
  int rc = stage_slot(ctx, &h);
  if (rc) return rc;
  memcpy(h, ids, (size_t)n_ids * sizeof(int32_t));
  int64_t n = n_ids;
  if (len) {
    int32_t at = 0;
    for (int64_t i = 0; i < n_ids; ++i) {
      h[n_ids + i] = at;
      at += len[i];
    }
    h[2 * n_ids] = at;
    n = 2 * n_ids + 1;
  }
  return stage_copy(ctx, n, st);
}

// the checks of an indexed push (`pipeline`: step) in the order of check_dense
static int check_indexed(wwb_ctx* ctx, bool pipeline, const int32_t* ids, int64_t n_ids, const int32_t* len,
                         const int16_t* pcm) {
  const int64_t cap = pipeline ? ctx->cs.max_streams : ctx->st.max_streams;
  if (!cap) return check_state(ctx, pipeline, true);
  int rc = check_tables(ctx, cap, ids, n_ids, len, true, pcm);
  return rc ? rc : check_state(ctx, pipeline, true);
}

int wwb_stream_push(wwb_ctx* ctx, const int16_t* pcm, int64_t S, int64_t n, const uint8_t* is_speech,
                    const uint8_t* is_active, float a, float threshold, float* post_out, int32_t* n_post_out,
                    uint8_t* trigger_out, float* post_max_out, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  int rc = check_dense(ctx, false, S, n, pcm);
  if (rc) return rc;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  return stream_push(ctx, pcm, S, n, nullptr, nullptr, is_speech, is_active, a, threshold, post_out, n_post_out,
                     trigger_out, post_max_out, (cudaStream_t)stream);
}

int wwb_stream_push_indexed(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const int32_t* len_host,
                            const int16_t* pcm, const uint8_t* is_speech, const uint8_t* is_active, float a,
                            float threshold, float* post_out, int32_t* n_post_out, uint8_t* trigger_out,
                            float* post_max_out, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_indexed(ctx, false, ids_host, n_ids, len_host, pcm);
  if (rc) return rc;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = stage_tables(ctx, ids_host, n_ids, len_host, st))) return rc;
  const int32_t* ids = ctx->st.tables;
  return stream_push(ctx, pcm, n_ids, 0, ids, ids + n_ids, is_speech, is_active, a, threshold, post_out, n_post_out,
                     trigger_out, post_max_out, st);
}

int wwb_stream_reset(wwb_ctx* ctx, const uint8_t* mask, int64_t S, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  int rc = check_state(ctx, false, false);
  if (rc) return rc;
  if (S < 1 || S > ctx->st.max_streams) return fail(ctx, WWB_ERR_STATE, "n_streams out of range");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  return launch_stream_reset(ctx, mask, S, (cudaStream_t)stream);
}

int wwb_stream_set_options(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const float* threshold_host,
                           const uint8_t* listening_host, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  int rc = check_state(ctx, false, true);
  if (rc) return rc;
  if (!threshold_host && !listening_host) return fail(ctx, WWB_ERR_ARG, "threshold and listening arrays both NULL");
  const void* values = threshold_host ? (const void*)threshold_host : (const void*)listening_host;
  if ((rc = check_tables(ctx, ctx->st.max_streams, ids_host, n_ids, nullptr, false, values))) return rc;
  for (int64_t i = 0; listening_host && i < n_ids; ++i)
    if (listening_host[i] > 1)
      return fail(ctx, WWB_ERR_ARG, "listening value %d (entry %lld) is not 0 or 1", listening_host[i], (long long)i);
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  int32_t* h;
  if ((rc = stage_slot(ctx, &h))) return rc;
  memcpy(h, ids_host, (size_t)n_ids * sizeof(int32_t));
  if (threshold_host) memcpy(h + n_ids, threshold_host, (size_t)n_ids * sizeof(float));
  for (int64_t i = 0; listening_host && i < n_ids; ++i) h[2 * n_ids + i] = listening_host[i];
  if ((rc = stage_copy(ctx, (listening_host ? 3 : 2) * n_ids, st))) return rc;
  return launch_stream_options(ctx, n_ids, threshold_host != nullptr, listening_host != nullptr, st);
}

int wwb_context_alloc(wwb_ctx* ctx, int frame_width_ms, int vad_rise_delay_ms, int vad_fall_delay_ms, int min_active_ms,
                      int max_active_ms) {
  if (!ctx) return WWB_ERR_ARG;
  int rc = check_state(ctx, false, false);
  if (rc) return rc;
  if (ctx->cs.max_streams) return fail(ctx, WWB_ERR_STATE, "context state already allocated");
  if (frame_width_ms < 1 || vad_rise_delay_ms < 0 || vad_fall_delay_ms < 0 || min_active_ms < 0 || max_active_ms < 0)
    return fail(ctx, WWB_ERR_ARG, "bad pipeline timing");
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  ContextState& c = ctx->cs;
  const size_t S = (size_t)ctx->st.max_streams;
  c.rise_length = vad_rise_delay_ms / frame_width_ms;          // vad/webrtc.py:43-44 (integer division)
  c.fall_length = vad_fall_delay_ms / frame_width_ms;
  c.min_active = (float)min_active_ms / (float)frame_width_ms; // activation_timeout.py:20-21 (true division)
  c.max_active = (float)max_active_ms / (float)frame_width_ms;
  if ((rc = dalloc(ctx, S, &c.run_value))) return rc;
  if ((rc = dalloc(ctx, S, &c.run_length))) return rc;
  if ((rc = dalloc(ctx, S, &c.is_speech))) return rc;
  if ((rc = dalloc(ctx, S, &c.is_active))) return rc;
  if ((rc = dalloc(ctx, S, &c.active_length))) return rc;
  if ((rc = dalloc(ctx, S, &c.t_is_speech))) return rc;
  if ((rc = dalloc(ctx, S, &c.trigger))) return rc;
  if ((rc = dalloc(ctx, S, &c.e_is_speech))) return rc;
  if ((rc = dalloc(ctx, S, &c.e_is_active))) return rc;
  if ((rc = dalloc(ctx, S, &c.activated_by))) return rc;
  c.max_streams = (int64_t)S;
  return WWB_OK;
}

// stage k's failure rc, reported on ctxs[0]: stage 0's as it stands, a later stage's under its number
static int stage_fail(wwb_ctx* const* ctxs, int k, int rc) {
  return k == 0 ? rc : fail(ctxs[0], rc, "stage %d: %s", k, ctxs[k]->err.c_str());
}

// vad debounce -> trigger stages 0 .. K-1 -> activation timeout over S entries (ids / off as in stream_push), the
// pipeline state on ctxs[0].  Every stage reads is_speech / is_active from ctxs[0]'s per-entry scratch and writes its
// trigger to ctxs[0]'s cs.trigger, which context_chain_kernel folds into the is_active of the next stage.  With K = 1 and
// no activated_by_out that kernel would change no state (cs.trigger keeps its 0 / 1), so it is not launched.
static int context_step_chain(wwb_ctx* const* ctxs, int K, const int16_t* pcm, int64_t S, int64_t n, const int32_t* ids,
                              const int32_t* off, const uint8_t* vad_raw, const float* a, const float* threshold,
                              float* const* post_out, int32_t* const* n_post_out, float* const* post_max_out,
                              uint8_t* is_speech_out, uint8_t* is_active_out, uint8_t* activated_out,
                              uint8_t* deactivated_out, int8_t* activated_by_out, cudaStream_t st) {
  wwb_ctx* c0 = ctxs[0];
  ContextState& c = c0->cs;
  int rc = launch_context_vad(c0, ids, vad_raw, S, st);
  if (rc) return rc;
  for (int k = 0; k < K; ++k) {
    if ((rc = stream_push(ctxs[k], pcm, S, n, ids, off, c.e_is_speech, c.e_is_active, a[k], threshold[k],
                          post_out ? post_out[k] : nullptr, n_post_out ? n_post_out[k] : nullptr, c.trigger,
                          post_max_out ? post_max_out[k] : nullptr, st)))
      return stage_fail(ctxs, k, rc);
    if ((K > 1 || activated_by_out) && (rc = launch_context_chain(c0, S, k, k == K - 1, activated_by_out, st))) return rc;
  }
  return launch_context_timeout(c0, ids, c.trigger, S, is_speech_out, is_active_out, activated_out, deactivated_out, st);
}

// 1 <= K <= WWB_MAX_STAGES, reported on c0
static int check_count(wwb_ctx* c0, int K) {
  if (K < 1 || K > WWB_MAX_STAGES) return fail(c0, WWB_ERR_ARG, "%d stages outside [1, %d]", K, WWB_MAX_STAGES);
  return WWB_OK;
}

// Stages 1 .. K-1 of a trigger chain, reported on ctxs[0] (stage 0 is checked as a single-model call): distinct non-NULL
// ctxs on ctxs[0]'s device, each with a model and stream state of ctxs[0]'s max_streams.
static int check_chain(wwb_ctx* const* ctxs, int K) {
  wwb_ctx* c0 = ctxs[0];
  for (int k = 1; k < K; ++k) {
    wwb_ctx* ck = ctxs[k];
    if (!ck) return fail(c0, WWB_ERR_ARG, "stage %d: NULL ctx", k);
    for (int j = 0; j < k; ++j)
      if (ctxs[j] == ck) return fail(c0, WWB_ERR_ARG, "stage %d: the ctx of stage %d again (each stage needs its own)", k, j);
    if (ck->device != c0->device)
      return fail(c0, WWB_ERR_ARG, "stage %d: ctx on device %d, stage 0 on device %d", k, ck->device, c0->device);
    int rc = check_state(ck, false, true);
    if (rc) return stage_fail(ctxs, k, rc);
    if (ck->st.max_streams != c0->st.max_streams)
      return fail(c0, WWB_ERR_STATE, "stage %d: stream state for %lld streams, stage 0 for %lld", k,
                  (long long)ck->st.max_streams, (long long)c0->st.max_streams);
  }
  return WWB_OK;
}

// chunks of n samples (len == NULL) or of len[0 .. n_ids) samples within the max_chunk of every stage after the first
// (stage 0's is checked with its tables)
static int check_chain_chunks(wwb_ctx* const* ctxs, int K, int64_t n, const int32_t* len, int64_t n_ids) {
  for (int k = 1; k < K; ++k) {
    const int64_t cap = ctxs[k]->st.max_chunk;
    for (int64_t i = 0; i < (len ? n_ids : 1); ++i) {
      const int64_t m = len ? len[i] : n;
      if (m > cap)
        return fail(ctxs[0], WWB_ERR_STATE, "stage %d: chunk of %lld samples (entry %lld) outside [1, %lld]", k,
                    (long long)m, (long long)i, (long long)cap);
    }
  }
  return WWB_OK;
}

// The dense and the indexed step over the stages ctxs[0 .. K) (K = 1: wwb_context_step / _indexed).  Every check runs
// before any device work, in this order: K, the per-stage arrays, stage 0 as a single-model step, the later stages, their
// chunk lengths.  The id tables of an indexed step are staged once, on ctxs[0], and every stage reads that device copy.
static int step_dense(wwb_ctx* const* ctxs, int K, const int16_t* pcm, int64_t S, int64_t n, const uint8_t* vad_raw,
                      const float* a, const float* threshold, float* const* post_out, int32_t* const* n_post_out,
                      float* const* post_max_out, uint8_t* is_speech_out, uint8_t* is_active_out, uint8_t* activated_out,
                      uint8_t* deactivated_out, int8_t* activated_by_out, cudaStream_t st) {
  wwb_ctx* c0 = ctxs[0];
  int rc = check_count(c0, K);
  if (rc) return rc;
  if (!a || !threshold) return fail(c0, WWB_ERR_ARG, "NULL pre-emphasis or threshold array");
  if ((rc = check_dense(c0, true, S, n, pcm)) || (rc = check_chain(ctxs, K)) ||
      (rc = check_chain_chunks(ctxs, K, n, nullptr, 0)))
    return rc;
  WWB_CUDA(c0, cudaSetDevice(c0->device));
  return context_step_chain(ctxs, K, pcm, S, n, nullptr, nullptr, vad_raw, a, threshold, post_out, n_post_out,
                            post_max_out, is_speech_out, is_active_out, activated_out, deactivated_out, activated_by_out, st);
}

static int step_indexed(wwb_ctx* const* ctxs, int K, const int32_t* ids_host, int64_t n_ids, const int32_t* len_host,
                        const int16_t* pcm, const uint8_t* vad_raw, const float* a, const float* threshold,
                        float* const* post_out, int32_t* const* n_post_out, float* const* post_max_out,
                        uint8_t* is_speech_out, uint8_t* is_active_out, uint8_t* activated_out, uint8_t* deactivated_out,
                        int8_t* activated_by_out, cudaStream_t st) {
  wwb_ctx* c0 = ctxs[0];
  int rc = check_count(c0, K);
  if (rc) return rc;
  if (!a || !threshold) return fail(c0, WWB_ERR_ARG, "NULL pre-emphasis or threshold array");
  if ((rc = check_indexed(c0, true, ids_host, n_ids, len_host, pcm)) || (rc = check_chain(ctxs, K)) ||
      (rc = check_chain_chunks(ctxs, K, 0, len_host, n_ids)))
    return rc;
  WWB_CUDA(c0, cudaSetDevice(c0->device));
  if ((rc = stage_tables(c0, ids_host, n_ids, len_host, st))) return rc;
  const int32_t* ids = c0->st.tables;
  return context_step_chain(ctxs, K, pcm, n_ids, 0, ids, ids + n_ids, vad_raw, a, threshold, post_out, n_post_out,
                            post_max_out, is_speech_out, is_active_out, activated_out, deactivated_out, activated_by_out, st);
}

int wwb_context_step(wwb_ctx* ctx, const int16_t* pcm, int64_t S, int64_t n, const uint8_t* vad_raw, float a, float threshold,
                     float* post_out, int32_t* n_post_out, float* post_max_out, uint8_t* is_speech_out, uint8_t* is_active_out,
                     uint8_t* activated_out, uint8_t* deactivated_out, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  return step_dense(&ctx, 1, pcm, S, n, vad_raw, &a, &threshold, &post_out, &n_post_out, &post_max_out, is_speech_out,
                    is_active_out, activated_out, deactivated_out, nullptr, (cudaStream_t)stream);
}

int wwb_context_step_indexed(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const int32_t* len_host,
                             const int16_t* pcm, const uint8_t* vad_raw, float a, float threshold, float* post_out,
                             int32_t* n_post_out, float* post_max_out, uint8_t* is_speech_out, uint8_t* is_active_out,
                             uint8_t* activated_out, uint8_t* deactivated_out, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  return step_indexed(&ctx, 1, ids_host, n_ids, len_host, pcm, vad_raw, &a, &threshold, &post_out, &n_post_out,
                      &post_max_out, is_speech_out, is_active_out, activated_out, deactivated_out, nullptr,
                      (cudaStream_t)stream);
}

int wwb_context_step_chain(wwb_ctx* const* ctxs, int n_stages, const int16_t* pcm, int64_t S, int64_t n,
                           const uint8_t* vad_raw, const float* a, const float* threshold, float* const* post_out,
                           int32_t* const* n_post_out, float* const* post_max_out, uint8_t* is_speech_out,
                           uint8_t* is_active_out, uint8_t* activated_out, uint8_t* deactivated_out,
                           int8_t* activated_by_out, void* stream) {
  if (!ctxs || !ctxs[0]) return WWB_ERR_ARG;
  return step_dense(ctxs, n_stages, pcm, S, n, vad_raw, a, threshold, post_out, n_post_out, post_max_out, is_speech_out,
                    is_active_out, activated_out, deactivated_out, activated_by_out, (cudaStream_t)stream);
}

int wwb_context_step_chain_indexed(wwb_ctx* const* ctxs, int n_stages, const int32_t* ids_host, int64_t n_ids,
                                   const int32_t* len_host, const int16_t* pcm, const uint8_t* vad_raw, const float* a,
                                   const float* threshold, float* const* post_out, int32_t* const* n_post_out,
                                   float* const* post_max_out, uint8_t* is_speech_out, uint8_t* is_active_out,
                                   uint8_t* activated_out, uint8_t* deactivated_out, int8_t* activated_by_out,
                                   void* stream) {
  if (!ctxs || !ctxs[0]) return WWB_ERR_ARG;
  return step_indexed(ctxs, n_stages, ids_host, n_ids, len_host, pcm, vad_raw, a, threshold, post_out, n_post_out,
                      post_max_out, is_speech_out, is_active_out, activated_out, deactivated_out, activated_by_out,
                      (cudaStream_t)stream);
}

int wwb_context_reset(wwb_ctx* ctx, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  int rc = check_state(ctx, true, false);
  if (rc) return rc;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  ContextState& c = ctx->cs;
  const size_t S = (size_t)c.max_streams;
  WWB_CUDA(ctx, cudaMemsetAsync(c.run_value, 0, S * 4, st));
  WWB_CUDA(ctx, cudaMemsetAsync(c.run_length, 0, S * 4, st));
  WWB_CUDA(ctx, cudaMemsetAsync(c.is_speech, 0, S, st));
  WWB_CUDA(ctx, cudaMemsetAsync(c.is_active, 0, S, st));
  WWB_CUDA(ctx, cudaMemsetAsync(c.active_length, 0, S * 4, st));
  WWB_CUDA(ctx, cudaMemsetAsync(c.t_is_speech, 0, S, st));
  return launch_stream_reset(ctx, nullptr, c.max_streams, st);
}

int64_t wwb_stream_state_bytes(const wwb_ctx* ctx) {
  if (!ctx || !ctx->st.max_streams || ctx->kind == WWB_MODEL_NONE) return 0;
  return stream_state_bytes(ctx->L);
}

// the host-side checks of wwb_stream_export / wwb_stream_import
static int check_state_call(wwb_ctx* ctx, const int32_t* ids, int64_t n_ids, const void* records) {
  int rc = check_state(ctx, false, true);
  if (rc || (rc = check_tables(ctx, ctx->st.max_streams, ids, n_ids, nullptr, false, records))) return rc;
  if ((uintptr_t)records % 16) return fail(ctx, WWB_ERR_ARG, "records must be 16-byte aligned");
  return WWB_OK;
}

int wwb_stream_export(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, void* records, void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_state_call(ctx, ids_host, n_ids, records);
  if (rc) return rc;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  if ((rc = stage_tables(ctx, ids_host, n_ids, nullptr, st))) return rc;
  return launch_stream_export(ctx, ctx->st.tables, n_ids, records, st);
}

// records[k] (n_ids each) into the slots ids_host names of stage k's ctx, all or nothing: the ids staged once on
// ctxs[0], then every stage's check before any scatter, so that a bad record of any stage leaves status[0] != 0 and every
// scatter idle.  `chain`: status int32[3] with the stage (wwb_stream_import_chain), else int32[2] (wwb_stream_import).
static int import_records(wwb_ctx* const* ctxs, int K, bool chain, const int32_t* ids_host, int64_t n_ids,
                          const void* const* records, int32_t* status, cudaStream_t st) {
  wwb_ctx* c0 = ctxs[0];
  WWB_CUDA(c0, cudaSetDevice(c0->device));
  int rc = stage_tables(c0, ids_host, n_ids, nullptr, st);
  if (rc) return rc;
  for (int k = 0; k < K; ++k)
    if ((rc = launch_stream_check_stage(ctxs[k], n_ids, records[k], status, chain ? k : -1, st)))
      return stage_fail(ctxs, k, rc);
  for (int k = 0; k < K; ++k)
    if ((rc = launch_stream_scatter(ctxs[k], c0->st.tables, n_ids, records[k], status, st))) return stage_fail(ctxs, k, rc);
  return WWB_OK;
}

int wwb_stream_import(wwb_ctx* ctx, const int32_t* ids_host, int64_t n_ids, const void* records, int32_t* status,
                      void* stream) {
  if (!ctx) return WWB_ERR_ARG;
  int rc = check_state_call(ctx, ids_host, n_ids, records);
  if (rc) return rc;
  if (!status) return fail(ctx, WWB_ERR_ARG, "NULL status");
  return import_records(&ctx, 1, false, ids_host, n_ids, &records, status, (cudaStream_t)stream);
}

int wwb_stream_import_chain(wwb_ctx* const* ctxs, int n_stages, const int32_t* ids_host, int64_t n_ids,
                            const void* const* records, int32_t* status, void* stream) {
  if (!ctxs || !ctxs[0]) return WWB_ERR_ARG;
  wwb_ctx* c0 = ctxs[0];
  int rc = check_count(c0, n_stages);
  if (rc || (rc = check_state(c0, true, true)) || (rc = check_chain(ctxs, n_stages))) return rc;
  if (!records) return fail(c0, WWB_ERR_ARG, "NULL records array");
  if ((rc = check_state_call(c0, ids_host, n_ids, records[0]))) return rc;
  for (int k = 1; k < n_stages; ++k)
    if (!records[k] || (uintptr_t)records[k] % 16)
      return fail(c0, WWB_ERR_ARG, "stage %d: records NULL or not 16-byte aligned", k);
  if (!status) return fail(c0, WWB_ERR_ARG, "NULL status");
  return import_records(ctxs, n_stages, true, ids_host, n_ids, records, status, (cudaStream_t)stream);
}

int64_t wwb_launch_count(const wwb_ctx* ctx) { return ctx ? ctx->launches : 0; }

int wwb_debug_buffer(wwb_ctx* ctx, void* dev_buf) {
  if (!ctx) return WWB_ERR_ARG;
  ctx->debug_buf = dev_buf;
  return WWB_OK;
}

}  // extern "C"
