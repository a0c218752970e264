// Stream state records (include/wwb200.h, wwb_stream_export / wwb_stream_import): a stream's trigger and pipeline state
// gathered from its slot into one fixed-size record, and scattered back into any slot of any ctx of the same model.
//
// Both directions are plain copies, one CTA per entry, 16-byte accesses.  The window is at most two contiguous segments of
// the ring (rows head..ring-1, then 0..), so the gather needs one compare per float4, no modulo.  An import writes the
// window to ring rows 0..L-1 with ring_head = 0 and zeroes the rest of the ring, so the whole ring of the slot is one
// contiguous destination.
#include <stddef.h>

#include "common.cuh"

namespace wwb {

static_assert(sizeof(wwb_stream_state_header) == 48, "record header is 48 bytes");
static_assert(offsetof(wwb_stream_state_header, version) == 4 && offsetof(wwb_stream_state_header, flags) == 6 &&
                  offsetof(wwb_stream_state_header, kind) == 8 && offsetof(wwb_stream_state_header, mel_length) == 12 &&
                  offsetof(wwb_stream_state_header, n_pending) == 16 &&
                  offsetof(wwb_stream_state_header, prev_sample) == 20 &&
                  offsetof(wwb_stream_state_header, post_max) == 24 &&
                  offsetof(wwb_stream_state_header, was_speech) == 28 &&
                  offsetof(wwb_stream_state_header, t_is_speech) == 31 &&
                  offsetof(wwb_stream_state_header, run_value) == 32 &&
                  offsetof(wwb_stream_state_header, active_length) == 40 &&
                  offsetof(wwb_stream_state_header, reserved) == 44,
              "record header layout");
static_assert(WWB_STREAM_STATE_PENDING == kFFT, "the record carries the whole pending buffer (pend_cap)");

constexpr int kHdr4 = (int)sizeof(wwb_stream_state_header) / 16;   // float4s of the header
constexpr int kPend4 = WWB_STREAM_STATE_PENDING / 4;
constexpr int kRow4 = kMel / 4;                                     // float4s of a mel row
constexpr int kStateThreads = 256;
constexpr int kUnroll = 4;                                          // loads in flight per thread

union RecordHeader {
  uint4 v[kHdr4];
  wwb_stream_state_header h;
};

int64_t stream_state_bytes(int L) {
  return (int64_t)sizeof(wwb_stream_state_header) + 4 * WWB_STREAM_STATE_PENDING + 4 * kMel * (int64_t)L;
}

struct StateParams {
  StreamState st;
  ContextState cs;        // cs.max_streams == 0: the ctx has no pipeline state
  const int32_t* ids;     // [n] slot of entry i
  int64_t n;
  int64_t rec4;           // record size in float4
  int L;
  int kind;
};

// entry i's record: header, then the pending samples (zero from n_pending on), then the window oldest row first
__global__ void __launch_bounds__(kStateThreads) stream_export_kernel(const StateParams P, float4* __restrict__ records) {
  const StreamState& S = P.st;
  const int64_t i = blockIdx.x;
  const int64_t s = P.ids[i];
  float4* __restrict__ rec = records + i * P.rec4;
  const int np = S.n_pending[s];
  const int head = S.ring_head[s];
  if (threadIdx.x == 0) {
    RecordHeader r;
    wwb_stream_state_header& h = r.h;
    h.magic = WWB_STREAM_STATE_MAGIC;
    h.version = WWB_STREAM_STATE_VERSION;
    h.kind = P.kind;
    h.mel_length = P.L;
    h.n_pending = np;
    h.prev_sample = S.prev_sample[s];
    h.post_max = S.post_max[s];
    h.was_speech = S.was_speech[s];
    h.reserved = 0;
    const ContextState& C = P.cs;
    if (C.max_streams) {
      h.flags = WWB_STREAM_STATE_PIPELINE;
      h.is_speech = C.is_speech[s];
      h.is_active = C.is_active[s];
      h.t_is_speech = C.t_is_speech[s];
      h.run_value = C.run_value[s];
      h.run_length = C.run_length[s];
      h.active_length = C.active_length[s];
    } else {
      h.flags = 0;
      h.is_speech = h.is_active = h.t_is_speech = 0;
      h.run_value = h.run_length = h.active_length = 0;
    }
    uint4* dst = reinterpret_cast<uint4*>(rec);
#pragma unroll
    for (int k = 0; k < kHdr4; ++k) dst[k] = r.v[k];
  }
  const float4* __restrict__ pend = reinterpret_cast<const float4*>(S.pending + s * S.pend_cap);
  const float4* __restrict__ ring = reinterpret_cast<const float4*>(S.mel_ring + s * S.ring * kMel);
  const float4* __restrict__ seg0 = ring + head * kRow4;                 // rows head .. ring-1
  const int n_seg0 = min(P.L, S.ring - head) * kRow4;                    // then rows 0 .. from float4 n_seg0 on
  const int n4 = kPend4 + P.L * kRow4;
  float4* __restrict__ body = rec + kHdr4;
  for (int k0 = threadIdx.x; k0 < n4; k0 += kUnroll * kStateThreads) {
    float4 v[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int k = k0 + u * kStateThreads;
      if (k >= n4) continue;
      if (k < kPend4) {
        v[u] = pend[k];
        const int e = 4 * k;
        if (e + 0 >= np) v[u].x = 0.f;
        if (e + 1 >= np) v[u].y = 0.f;
        if (e + 2 >= np) v[u].z = 0.f;
        if (e + 3 >= np) v[u].w = 0.f;
      } else {
        const int m = k - kPend4;
        v[u] = m < n_seg0 ? seg0[m] : ring[m - n_seg0];
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int k = k0 + u * kStateThreads;
      if (k < n4) body[k] = v[u];
    }
  }
}

// One thread per record: the first failing check of the lowest bad entry lands in import_check[0] as
// (~entry << 32 | reason) through atomicMax; the last block to finish writes the status and clears the scratch.
// stage < 0: status int32[2] of wwb_stream_import.  stage >= 0 (wwb_stream_import_chain, stages checked in order):
// status int32[3] with the stage, left as it is when an earlier stage's check failed.
__global__ void __launch_bounds__(kStateThreads) stream_check_kernel(const float4* __restrict__ records, int64_t n,
                                                                      int64_t rec4, int kind, int L,
                                                                      unsigned long long* check, int32_t* status,
                                                                      int stage) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    RecordHeader r;
    const uint4* src = reinterpret_cast<const uint4*>(records + i * rec4);
    r.v[0] = src[0];   // magic .. mel_length
    r.v[1] = src[1];   // n_pending ..
    const wwb_stream_state_header& h = r.h;
    int why = WWB_RECORD_OK;
    if (h.magic != WWB_STREAM_STATE_MAGIC) why = WWB_RECORD_BAD_MAGIC;
    else if (h.version != WWB_STREAM_STATE_VERSION) why = WWB_RECORD_BAD_VERSION;
    else if (h.flags & ~WWB_STREAM_STATE_PIPELINE) why = WWB_RECORD_BAD_FLAGS;
    else if (h.kind != kind) why = WWB_RECORD_BAD_KIND;
    else if (h.mel_length != L) why = WWB_RECORD_BAD_LENGTH;
    else if (h.n_pending < 0 || h.n_pending >= WWB_STREAM_STATE_PENDING) why = WWB_RECORD_BAD_PENDING;
    if (why != WWB_RECORD_OK) {
      atomicMax(&check[0], ((0xffffffffull - (unsigned long long)i) << 32) | (unsigned)why);
      __threadfence();
    }
  }
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&check[1], 1ull) == gridDim.x - 1;
  __syncthreads();
  if (last && threadIdx.x == 0) {
    const unsigned long long key = atomicExch(&check[0], 0ull);
    check[1] = 0;
    if (stage <= 0 || status[0] == 0) {
      status[0] = key ? (int32_t)(0xffffffffull - (key >> 32)) + 1 : 0;
      status[1] = (int32_t)(key & 0xffffffffull);
      if (stage >= 0) status[2] = key ? stage : 0;
    }
  }
}

// entry i's record into slot ids[i]: pending buffer, ring rows 0..L-1 (the window), zeros for rows L..ring-1, scalars.
// Does nothing unless stream_check_kernel accepted every record.
__global__ void __launch_bounds__(kStateThreads) stream_import_kernel(const StateParams P, const float4* __restrict__ records,
                                                                      const int32_t* __restrict__ status) {
  if (status[0] != 0) return;
  const StreamState& S = P.st;
  const int64_t i = blockIdx.x;
  const int64_t s = P.ids[i];
  const float4* __restrict__ rec = records + i * P.rec4;
  if (threadIdx.x == 0) {
    RecordHeader r;
    const uint4* src = reinterpret_cast<const uint4*>(rec);
#pragma unroll
    for (int k = 0; k < kHdr4; ++k) r.v[k] = src[k];
    const wwb_stream_state_header& h = r.h;
    S.n_pending[s] = h.n_pending;
    S.prev_sample[s] = h.prev_sample;
    S.post_max[s] = h.post_max;
    S.was_speech[s] = h.was_speech;
    S.ring_head[s] = 0;
    const ContextState& C = P.cs;
    if (C.max_streams) {   // initial values (wwb_context_reset) when the record carries no pipeline state
      const bool p = (h.flags & WWB_STREAM_STATE_PIPELINE) != 0;
      C.is_speech[s] = p ? h.is_speech : 0;
      C.is_active[s] = p ? h.is_active : 0;
      C.t_is_speech[s] = p ? h.t_is_speech : 0;
      C.run_value[s] = p ? h.run_value : 0;
      C.run_length[s] = p ? h.run_length : 0;
      C.active_length[s] = p ? h.active_length : 0;
    }
  }
  const float4* __restrict__ body = rec + kHdr4;
  float4* __restrict__ pend = reinterpret_cast<float4*>(S.pending + s * S.pend_cap);
  float4* __restrict__ ring = reinterpret_cast<float4*>(S.mel_ring + s * S.ring * kMel);
  const int n_win4 = P.L * kRow4;
  const int n4 = kPend4 + S.ring * kRow4;
  for (int k0 = threadIdx.x; k0 < n4; k0 += kUnroll * kStateThreads) {
    float4 v[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int k = k0 + u * kStateThreads;
      if (k < n4) v[u] = k < kPend4 + n_win4 ? body[k] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int k = k0 + u * kStateThreads;
      if (k < kPend4) pend[k] = v[u];
      else if (k < n4) ring[k - kPend4] = v[u];
    }
  }
}

static StateParams state_params(const wwb_ctx* ctx, const int32_t* ids, int64_t n) {
  StateParams P;
  P.st = ctx->st;
  P.cs = ctx->cs;
  P.ids = ids;
  P.n = n;
  P.rec4 = stream_state_bytes(ctx->L) / 16;
  P.L = ctx->L;
  P.kind = ctx->kind;
  return P;
}

int launch_stream_export(wwb_ctx* ctx, const int32_t* ids, int64_t n, void* records, cudaStream_t st) {
  const StateParams P = state_params(ctx, ids, n);
  stream_export_kernel<<<(unsigned)n, kStateThreads, 0, st>>>(P, (float4*)records);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_stream_check_stage(wwb_ctx* ctx, int64_t n, const void* records, int32_t* status, int stage, cudaStream_t st) {
  stream_check_kernel<<<(unsigned)((n + kStateThreads - 1) / kStateThreads), kStateThreads, 0, st>>>(
      (const float4*)records, n, stream_state_bytes(ctx->L) / 16, ctx->kind, ctx->L, ctx->st.import_check, status, stage);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

int launch_stream_scatter(wwb_ctx* ctx, const int32_t* ids, int64_t n, const void* records, const int32_t* status,
                          cudaStream_t st) {
  const StateParams P = state_params(ctx, ids, n);
  stream_import_kernel<<<(unsigned)n, kStateThreads, 0, st>>>(P, (const float4*)records, status);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb
