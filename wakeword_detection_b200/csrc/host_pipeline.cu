// Host-buffer entry points: the plugin call a maintainer binds in place of
// TFLiteModel.__call__ (spokestack/models/tensorflow.py:33-51: copy in, invoke, copy out), batched over streams.
//
//   wwb_sweep_submit / wwb_sweep_wait   PCM in HOST memory -> filter -> encode -> detect of one or several models
//                                       -> posteriors (+ optional FAR / FRR counters) back in HOST memory,
//                                       up to two jobs in flight
//   wwb_pipeline_host                   = submit + wait for one model
//
// Three CUDA streams owned by the first ctx: copy-in, compute, copy-out.  A job's PCM goes into one of two device
// staging buffers, so the H2D copy of job k+1 runs while the kernels of job k do; a job submitted into an idle pipe
// is cut into three slices of streams (1/8, 2/8, 5/8) so that only the first, small copy is exposed.  Caller buffers
// are never page-locked here: pageable memory takes the driver's staged copy, which blocks the calling thread, and
// callers that want the overlapped path pass memory from wwb_host_alloc.  Registering the caller's memory would leave
// it page-locked after the call returns, and CUDA requires it unregistered before it is freed.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace wwb {

static const int kPipeSlots = 2;

struct HostPipeSlot {
  bool busy = false;
  void* pcm = nullptr;   // device staging
  size_t pcm_bytes = 0;
  cudaEvent_t staged_free = nullptr;   // the filter has consumed this staging buffer
  cudaEvent_t done = nullptr;          // all results of the job are in host memory
  // per model (index = position in the ctx list of the job)
  std::vector<void*> post;     // device posteriors [S, n_win]
  std::vector<size_t> post_bytes;
  std::vector<void*> counts;   // device int64 [2][n_thr]
  std::vector<size_t> counts_bytes;
  // The counters come back through a page-locked bounce buffer owned by the slot and are handed to the caller's arrays
  // in wwb_sweep_wait: a device->host copy into pageable memory blocks the submitting thread until the job's kernels
  // have run, which would serialise the next job's host->device copy behind this job's compute.
  int64_t* counts_pinned = nullptr;   // [n_ctx][2][n_thr]
  size_t counts_pinned_bytes = 0;
  struct Deliver { int64_t* dst; const int64_t* src; size_t bytes; };
  std::vector<Deliver> deliver;
};

struct HostPipe {
  cudaStream_t copy_in = nullptr, compute = nullptr, copy_out = nullptr;
  cudaEvent_t slice_in[8] = {};
  cudaEvent_t computed = nullptr;
  HostPipeSlot slot[kPipeSlots];
  int next = 0, oldest = 0, in_flight = 0;
  void* mel = nullptr;
  size_t mel_bytes = 0;
  void* thr = nullptr;
  size_t thr_bytes = 0;
  void* seg = nullptr;
  size_t seg_bytes = 0;
  std::vector<double> thr_host;        // content of `thr` (re-uploaded only when it changes)
  std::vector<int64_t> seg_key;        // (S, n_win...) the segment table was built for
};

static int grow(wwb_ctx* ctx, void** p, size_t* have, size_t want) {
  if (*have >= want) return WWB_OK;
  if (*p) {
    WWB_CUDA(ctx, cudaDeviceSynchronize());
    WWB_CUDA(ctx, cudaFree(*p));
    *p = nullptr;
    *have = 0;
  }
  want += want / 8 + 256;
  cudaError_t e = cudaMalloc(p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, WWB_ERR_ALLOC, "cudaMalloc of %zu bytes (host pipeline) failed: %s", want, cudaGetErrorString(e));
  }
  *have = want;
  return WWB_OK;
}

static int pipe_get(wwb_ctx* ctx, HostPipe** out) {
  if (!ctx->host_pipe) {
    HostPipe* hp = new HostPipe();
    ctx->host_pipe = hp;
    WWB_CUDA(ctx, cudaStreamCreateWithFlags(&hp->copy_in, cudaStreamNonBlocking));
    WWB_CUDA(ctx, cudaStreamCreateWithFlags(&hp->compute, cudaStreamNonBlocking));
    WWB_CUDA(ctx, cudaStreamCreateWithFlags(&hp->copy_out, cudaStreamNonBlocking));
    for (auto& e : hp->slice_in) WWB_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    WWB_CUDA(ctx, cudaEventCreateWithFlags(&hp->computed, cudaEventDisableTiming));
    for (auto& s : hp->slot) {
      WWB_CUDA(ctx, cudaEventCreateWithFlags(&s.staged_free, cudaEventDisableTiming));
      WWB_CUDA(ctx, cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    }
  }
  *out = (HostPipe*)ctx->host_pipe;
  return WWB_OK;
}

void host_pipe_destroy(wwb_ctx* ctx) {
  HostPipe* hp = (HostPipe*)ctx->host_pipe;
  if (!hp) return;
  cudaDeviceSynchronize();
  for (auto& s : hp->slot) {
    if (s.pcm) cudaFree(s.pcm);
    for (void* p : s.post) if (p) cudaFree(p);
    for (void* p : s.counts) if (p) cudaFree(p);
    if (s.counts_pinned) cudaFreeHost(s.counts_pinned);
    if (s.staged_free) cudaEventDestroy(s.staged_free);
    if (s.done) cudaEventDestroy(s.done);
  }
  for (void* p : {hp->mel, hp->thr, hp->seg}) if (p) cudaFree(p);
  for (auto& e : hp->slice_in) if (e) cudaEventDestroy(e);
  if (hp->computed) cudaEventDestroy(hp->computed);
  for (cudaStream_t s : {hp->copy_in, hp->compute, hp->copy_out}) if (s) cudaStreamDestroy(s);
  cudaGetLastError();
  delete hp;
  ctx->host_pipe = nullptr;
}

static int sweep_wait(wwb_ctx* ctx) {
  HostPipe* hp = (HostPipe*)ctx->host_pipe;
  if (!hp || hp->in_flight == 0) return fail(ctx, WWB_ERR_STATE, "wwb_sweep_wait: no job in flight");
  HostPipeSlot& s = hp->slot[hp->oldest];
  WWB_CUDA(ctx, cudaEventSynchronize(s.done));
  for (const auto& d : s.deliver) memcpy(d.dst, d.src, d.bytes);
  s.deliver.clear();
  s.busy = false;
  hp->oldest = (hp->oldest + 1) % kPipeSlots;
  hp->in_flight--;
  return WWB_OK;
}

static int sweep_submit(wwb_ctx* const* ctxs, int n_ctx, const void* pcm_host, int dtype, int64_t S, int64_t N, float a,
                        int hop, const double* thr_host, int n_thr, float* const* post_host, int64_t* const* far_host,
                        int64_t* const* frr_host) {
  wwb_ctx* ctx = ctxs[0];
  if (dtype != WWB_PCM_I16 && dtype != WWB_PCM_F32) return fail(ctx, WWB_ERR_ARG, "bad pcm dtype");
  if (S < 0 || N < 0 || hop < 1) return fail(ctx, WWB_ERR_ARG, "bad pipeline geometry");
  if (S * N > 0 && !pcm_host) return fail(ctx, WWB_ERR_ARG, "NULL pcm");
  for (int m = 0; m < n_ctx; ++m) {
    if (!ctxs[m] || ctxs[m]->device != ctx->device) return fail(ctx, WWB_ERR_ARG, "all models of a sweep must live on one device");
    if (ctxs[m]->kind == WWB_MODEL_NONE) return fail(ctx, WWB_ERR_STATE, "ctx %d holds a filter only (no encode/detect weights)", m);
  }
  // ONE filter pass feeds every model: they must share the filter's fields
  for (int m = 1; m < n_ctx; ++m)
    if (ctxs[m]->mel_w_host != ctx->mel_w_host || ctxs[m]->mel_b_host != ctx->mel_b_host ||
        ctxs[m]->mel_floor != ctx->mel_floor || ctxs[m]->mel_log_offset != ctx->mel_log_offset ||
        ctxs[m]->mel_scale != ctx->mel_scale)
      return fail(ctx, WWB_ERR_ARG, "model %d has other filter fields (mel_w, mel_b, floor, offset, scale) than model 0", m);
  const bool want_counts = thr_host && n_thr > 0 && (far_host || frr_host);
  if (want_counts && n_thr > 8192) return fail(ctx, WWB_ERR_ARG, "n_thr out of range");
  if (want_counts)
    for (int i = 1; i < n_thr; ++i)
      if (thr_host[i] < thr_host[i - 1]) return fail(ctx, WWB_ERR_ARG, "thresholds must be ascending");
  const size_t esz = dtype == WWB_PCM_I16 ? 2 : 4;
  const int64_t F = wwb_num_frames(N);
  std::vector<int64_t> nwin(n_ctx);
  for (int m = 0; m < n_ctx; ++m) {
    nwin[m] = wwb_num_windows(ctxs[m], F, hop);
    if (want_counts && far_host && far_host[m] && nwin[m] > 0 && nwin[m] < 30)
      return fail(ctx, WWB_ERR_ARG, "FAR trajectory of %lld posteriors is shorter than the 30-tap smoothing window", (long long)nwin[m]);
  }
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  HostPipe* hp;
  int rc = pipe_get(ctx, &hp);
  if (rc) return rc;
  if (hp->in_flight == kPipeSlots) return fail(ctx, WWB_ERR_STATE, "two jobs are in flight already: call wwb_sweep_wait first");
  const bool overlapped = hp->in_flight > 0;
  HostPipeSlot& sl = hp->slot[hp->next];

  // ---- buffers ----
  if ((rc = grow(ctx, &sl.pcm, &sl.pcm_bytes, (size_t)S * N * esz))) return rc;
  if ((rc = grow(ctx, &hp->mel, &hp->mel_bytes, (size_t)S * F * kMel * sizeof(float)))) return rc;
  if ((int)sl.post.size() < n_ctx) {
    sl.post.resize(n_ctx, nullptr); sl.post_bytes.resize(n_ctx, 0);
    sl.counts.resize(n_ctx, nullptr); sl.counts_bytes.resize(n_ctx, 0);
  }
  for (int m = 0; m < n_ctx; ++m) {
    if ((rc = grow(ctx, &sl.post[m], &sl.post_bytes[m], (size_t)std::max<int64_t>(S * nwin[m], 1) * sizeof(float)))) return rc;
    if (want_counts && (rc = grow(ctx, &sl.counts[m], &sl.counts_bytes[m], (size_t)2 * n_thr * sizeof(int64_t)))) return rc;
  }
  if (want_counts && sl.counts_pinned_bytes < (size_t)n_ctx * 2 * n_thr * sizeof(int64_t)) {
    if (sl.counts_pinned) cudaFreeHost(sl.counts_pinned);
    sl.counts_pinned = nullptr;
    sl.counts_pinned_bytes = (size_t)n_ctx * 2 * n_thr * sizeof(int64_t);
    WWB_CUDA(ctx, cudaHostAlloc((void**)&sl.counts_pinned, sl.counts_pinned_bytes, cudaHostAllocDefault));
  }
  sl.deliver.clear();
  if (want_counts) {
    // thresholds and the segment tables (every stream is one clip / one trajectory) are constant across the steps of a
    // sweep: uploaded once, re-uploaded only when they change
    std::vector<int64_t> key = {S, (int64_t)n_ctx};
    for (int m = 0; m < n_ctx; ++m) key.push_back(nwin[m]);
    const bool thr_same = (int)hp->thr_host.size() == n_thr && !memcmp(hp->thr_host.data(), thr_host, n_thr * sizeof(double));
    if (!thr_same || key != hp->seg_key) {
      WWB_CUDA(ctx, cudaStreamSynchronize(hp->compute));
      if ((rc = grow(ctx, &hp->thr, &hp->thr_bytes, (size_t)n_thr * sizeof(double)))) return rc;
      if ((rc = grow(ctx, &hp->seg, &hp->seg_bytes, (size_t)n_ctx * (S + 1) * sizeof(int64_t)))) return rc;
      std::vector<int64_t> seg((size_t)n_ctx * (S + 1));
      for (int m = 0; m < n_ctx; ++m)
        for (int64_t s = 0; s <= S; ++s) seg[(size_t)m * (S + 1) + s] = s * nwin[m];
      WWB_CUDA(ctx, cudaMemcpy(hp->thr, thr_host, (size_t)n_thr * sizeof(double), cudaMemcpyHostToDevice));
      WWB_CUDA(ctx, cudaMemcpy(hp->seg, seg.data(), seg.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
      hp->thr_host.assign(thr_host, thr_host + n_thr);
      hp->seg_key = key;
    }
  }

  // ---- slices of streams: 1/8, 2/8, 5/8 when nothing hides the first copy, one slice otherwise ----
  int64_t bounds[4] = {0, S, S, S};
  int n_slices = 1;
  if (!overlapped && S >= 64) {
    bounds[1] = S / 8; bounds[2] = 3 * (S / 8); bounds[3] = S;
    n_slices = 3;
  }
  // the staging buffer is free once the filter of the job that used it last has run
  WWB_CUDA(ctx, cudaStreamWaitEvent(hp->copy_in, sl.staged_free, 0));
  for (int i = 0; i < n_slices; ++i) {
    const int64_t s0 = bounds[i], s1 = bounds[i + 1];
    static const bool skip_h2d = getenv("WWB_DEBUG_SKIP_H2D") != nullptr;   // development probe: how much of a job is the copy
    if (s1 > s0 && N > 0 && !skip_h2d)
      WWB_CUDA(ctx, cudaMemcpyAsync((char*)sl.pcm + (size_t)s0 * N * esz, (const char*)pcm_host + (size_t)s0 * N * esz,
                                    (size_t)(s1 - s0) * N * esz, cudaMemcpyHostToDevice, hp->copy_in));
    WWB_CUDA(ctx, cudaEventRecord(hp->slice_in[i], hp->copy_in));
  }
  for (int i = 0; i < n_slices; ++i) {
    const int64_t s0 = bounds[i], s1 = bounds[i + 1];
    WWB_CUDA(ctx, cudaStreamWaitEvent(hp->compute, hp->slice_in[i], 0));
    if (s1 == s0) continue;
    float* mel = (float*)hp->mel + (size_t)s0 * F * kMel;
    if ((rc = wwb_filter(ctx, (const char*)sl.pcm + (size_t)s0 * N * esz, dtype, s1 - s0, N, N, a, mel, hp->compute))) return rc;
    if (i == n_slices - 1) WWB_CUDA(ctx, cudaEventRecord(sl.staged_free, hp->compute));
    for (int m = 0; m < n_ctx; ++m) {
      if (nwin[m] == 0) continue;
      rc = wwb_posteriors(ctxs[m], mel, s1 - s0, F, hop, (float*)sl.post[m] + (size_t)s0 * nwin[m], hp->compute);
      if (rc) return m == 0 ? rc : fail(ctx, rc, "model %d: %s", m, wwb_last_error(ctxs[m]));
    }
  }
  if (n_slices == 1 && S == 0) WWB_CUDA(ctx, cudaEventRecord(sl.staged_free, hp->compute));
  if (want_counts)
    for (int m = 0; m < n_ctx; ++m) {
      int64_t* c = (int64_t*)sl.counts[m];
      const int64_t* seg = (const int64_t*)hp->seg + (size_t)m * (S + 1);
      const int64_t nseg = nwin[m] > 0 ? S : 0;
      if ((rc = wwb_eval_counts(ctxs[m], (const float*)sl.post[m], seg, nseg, nullptr, nullptr, S * nwin[m], (const double*)hp->thr,
                                n_thr, WWB_COUNT_FAR_EDGES, 30, c, hp->compute))) return rc;
      if ((rc = wwb_eval_counts(ctxs[m], (const float*)sl.post[m], seg, nseg, nullptr, nullptr, S * nwin[m], (const double*)hp->thr,
                                n_thr, WWB_COUNT_FRR_MAX, 30, c + n_thr, hp->compute))) return rc;
    }
  WWB_CUDA(ctx, cudaEventRecord(hp->computed, hp->compute));
  WWB_CUDA(ctx, cudaStreamWaitEvent(hp->copy_out, hp->computed, 0));
  for (int m = 0; m < n_ctx; ++m) {
    if (post_host && post_host[m] && S * nwin[m] > 0)
      WWB_CUDA(ctx, cudaMemcpyAsync(post_host[m], sl.post[m], (size_t)S * nwin[m] * sizeof(float), cudaMemcpyDeviceToHost, hp->copy_out));
    if (want_counts) {
      int64_t* bounce = sl.counts_pinned + (size_t)m * 2 * n_thr;
      WWB_CUDA(ctx, cudaMemcpyAsync(bounce, sl.counts[m], (size_t)2 * n_thr * sizeof(int64_t), cudaMemcpyDeviceToHost, hp->copy_out));
      if (far_host && far_host[m]) sl.deliver.push_back({far_host[m], bounce, (size_t)n_thr * sizeof(int64_t)});
      if (frr_host && frr_host[m]) sl.deliver.push_back({frr_host[m], bounce + n_thr, (size_t)n_thr * sizeof(int64_t)});
    }
  }
  WWB_CUDA(ctx, cudaEventRecord(sl.done, hp->copy_out));
  sl.busy = true;
  hp->next = (hp->next + 1) % kPipeSlots;
  hp->in_flight++;
  return WWB_OK;
}

}  // namespace wwb

using namespace wwb;

extern "C" {

int wwb_sweep_submit(wwb_ctx* const* ctxs, int n_ctx, const void* pcm_host, int pcm_dtype, int64_t n_streams, int64_t n_samples,
                     float pre_emphasis, int hop, const double* thr_host, int n_thr, float* const* post_host,
                     int64_t* const* far_counts_host, int64_t* const* frr_counts_host) {
  if (!ctxs || n_ctx < 1 || n_ctx > 8 || !ctxs[0]) return WWB_ERR_ARG;
  return sweep_submit(ctxs, n_ctx, pcm_host, pcm_dtype, n_streams, n_samples, pre_emphasis, hop, thr_host, n_thr, post_host,
                      far_counts_host, frr_counts_host);
}

int wwb_sweep_wait(wwb_ctx* ctx) {
  if (!ctx) return WWB_ERR_ARG;
  WWB_CUDA(ctx, cudaSetDevice(ctx->device));
  return sweep_wait(ctx);
}

int wwb_pipeline_host(wwb_ctx* ctx, const void* pcm_host, int dtype, int64_t S, int64_t N, float a, int hop,
                      float* post_host) {
  if (!ctx) return WWB_ERR_ARG;
  // drain earlier asynchronous jobs first: this call is synchronous and returns ITS results
  while (ctx->host_pipe && ((HostPipe*)ctx->host_pipe)->in_flight > 0) {
    int rc = sweep_wait(ctx);
    if (rc) return rc;
  }
  wwb_ctx* list[1] = {ctx};
  float* posts[1] = {post_host};
  int rc = sweep_submit(list, 1, pcm_host, dtype, S, N, a, hop, nullptr, 0, posts, nullptr, nullptr);
  if (rc) return rc;
  return sweep_wait(ctx);
}

int wwb_host_alloc(void** out, size_t bytes) {
  if (!out) return WWB_ERR_ARG;
  *out = nullptr;
  cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(nullptr, WWB_ERR_ALLOC, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  }
  return WWB_OK;
}

int wwb_host_free(void* p) {
  if (p && cudaFreeHost(p) != cudaSuccess) {
    cudaGetLastError();
    return WWB_ERR_CUDA;
  }
  return WWB_OK;
}

}  // extern "C"
