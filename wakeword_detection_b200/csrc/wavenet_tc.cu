// K5/K6 — WaveNet encode + detect on the tensor cores (precision WWB_PREC_TC / TC_FAST).
//
// One persistent CTA per SM processes groups of WN_G = 4 windows.  The rows of a group are interleaved
// TIME-MAJOR: (time t, window w) -> o = t*4 + w form the M dimension of every GEMM (6 tiles of 128 rows, 728 of the
// 768 rows are real; the 64 rows in front of row 0 are the causal zero padding of all four windows).  A dilated tap
// is still a linear row shift (4*d rows).  Each of the 768 epilogue threads owns ONE row for the whole 24-block
// stack: its 16-channel residual stream never leaves registers, its 32-channel skip sum lives in the thread's own 128 bytes
// of shared memory.  (The first half of round 2 ran 3 windows on 5 tiles at 80 registers per thread; 4 on 6 - 832 threads,
// 72 registers, 80 instead of 96 tensor-memory columns per tile - pays the per-block dependency chain once per 4 windows
// instead of 3: 15.5 -> 13.5 ms per 512 x 10 s; -> 12.9 with the snapshots stored as column planes.)
//
// SHARED ACTIVATIONS (sliding-window batches).  Row t of block b depends on the window's zero padding only while
// t < D(b) = sum_{m<=b} 2*dilation[m] (2, 6, 14, 30, 32, ... 180): every other activation is a function of the
// stream's absolute frame and identical in all ~91 windows that cover it.  With time-major rows the window-dependent
// ("dirty") rows of a block are a PREFIX, so tile i only has to take part from block join[i] = min{b : D(b) > t_min(i)}
// on (0, 5, 9, 14, 18, 22 for the shipped model: 76 instead of 144 tile-blocks per group).  A tile joins from per-frame
// SNAPSHOTS (residual stream x and the skip prefix sum after block join[i]-1; 192 B per frame and level, stored as 12
// column planes of float4 so that a warp's consecutive frames are consecutive in memory) written by a
// stream-level pass of this same kernel (stream_mode: a group is a chunk of 768 consecutive frames of one stream,
// rows o >= 180 of a chunk are past every receptive field; +1.5 % work).  Same MMAs on the same operand values in the
// same order, so the posteriors are bit-identical to the per-window formulation (WWB_WN_NO_SHARE=1 forces it).
// Per block and tile:
//   gate GEMM   D[128,32] = sum_tap U[rows - (2-tap)*d, 16] * Wg_tap          (tcgen05, TMEM)
//               taps 0/1 (row-shifted) read A from shared memory: the operand layout is linear
//               in the row index, so a dilated tap is a start-address offset;
//               tap 2 (no shift) reads A straight from TENSOR MEMORY, where the row's owner
//               thread stored it (tcgen05.st): 15.5 clk per MMA instead of 39.4 (tools/tc_rate_probe.cu)
//   epilogue 1  g = tanh(.)*sigmoid(.) (2 ex2 per channel, 1 rcp per channel pair), fp16 hi/lo -> TMEM, over the
//               consumed gate accumulator (A operand of the next GEMM), half by half
//   res/skip    D[128,48] = g[128,16] * [Wres | Wskip]       (A from TMEM; res lands on the consumed second half of
//               the gate accumulator, skip on its own 32 columns)
//   epilogue 2a x += ReLU(res); u = BN_next(x) -> hi/lo -> shared memory + TMEM   (releases the next gate GEMM)
//   epilogue 2b skip += ReLU(.)                                                   (overlaps that GEMM)
// The input 1x1 conv depends only on the mel row, which ~91 overlapping windows share: wn_input_kernel computes it once
// per row (fp32) and a group starts by loading its rows' 16 values.  The detect head (32->32 with A from TMEM; then
// 32->2, max over time, softmax) is a tensor-core GEMM of the same kind as the blocks' at the end of a group.
// Biases are added by the tensor core too: one extra k-step whose A chunk is the constant (1, 1, 0, ...)
// and whose B rows hold (bias_hi, bias_lo, 0, ...) - broadcast loads of per-block constants from shared
// memory cost one wavefront per 4 bytes and were the largest shared-memory consumer (profiles/).
// The gate weights and biases are pre-scaled by -2*log2(e) (tanh half) / -log2(e) (sigmoid half).
// The per-block BatchNorm affine u = bn_mul * x + bn_add is FOLDED into the gate GEMM (weights * bn_mul, bias +
// W * bn_add), so the A operand is the residual stream x itself and the epilogue neither loads the 32 constants
// (8 broadcast LDS.128 = 32 shared-memory wavefronts per warp and block, 17 % of the shared-memory pipe) nor
// applies them.  The causal zero padding is of u, not x: the padding rows in front of row 0 therefore
// hold x_pad = -bn_add / bn_mul (so that u_pad = 0), rewritten for each block by the res/skip warp.
// fp16 hi/lo operand split (3 MMAs per product) keeps the result at fp32 accuracy
// (DESIGN.md §precision).  Epilogue arithmetic uses the packed fp32x2 instructions (FFMA2/FADD2).
// Per-block weights (12 KB incl. the bias operands) stream through a 5-stage cp.async.bulk ring.
//
// GEMM issue: one extra warp issues the gate GEMMs tile after tile (in order, so they run back to back and
// stagger the tiles: the tensor pipe, the SFU and the FMA/ALU pipes then work on different tiles at the
// same time); a second extra warp issues the small res/skip GEMMs, so they never queue behind a
// wait of the gate warp.  Both busy-poll their barriers (their wake-up latency is on every tile's chain).
// Epilogue 2 is split: 2a (residual -> u) releases the next gate GEMM, 2b (skip sum) overlaps it.
// Ordering rules:
//   gate(k,i) needs epilogue 2 of (k-1,i) and (k-1,i-1)      (its taps reach up to 64 rows into tile i-1)
//   rs(k,i)   needs epilogue 1 of (k,i) and gate(k,i+1) COMPLETE: epilogue 2 of (k,i) overwrites rows that
//             GEMM reads, and GEMMs issued by different threads have no implicit order.
// Measured and not kept (profiles/r2_notes.md, source under profiles/experiments/): U rows double-buffered by block
// parity (no rs -> gate coupling), detect GEMMs issued by the res/skip warp so that tile 0 enters the next group while
// the other tiles finish block 23, both accumulator halves loaded before one wait, 2^x on the FMA pipe for part of
// epilogue 1.
#include <string.h>

#include "wavenet_tc.cuh"

namespace wwb {


struct WnSmem {
  unsigned char U[WN_UBUF];                // [plane][chunk][row]
  float4 skip[8 * WN_ROWS];                // skip sums [channel quad][row]: each thread keeps its row's 32 sums HERE, not in registers (see the kernel)
  unsigned char W[WN_WST][WN_WBLK];
  WnHead head;
  uint64_t bar_gate[WN_NT], bar_rs[WN_NT], bar_det[WN_NT];   // GEMM completion (tcgen05.commit) -> the tile's four warps
  uint64_t bar_u[WN_NT];                     // the tile's four warps finished epilogue 2 (tile 0: + the padding rows, written by the res/skip warp) -> gate warp
  uint64_t bar_dq[WN_NT];                    // the tile's four warps stored the detect head's input -> gate warp
  uint64_t bar_g[WN_NT];                     // the tile's four warps finished epilogue 1 -> res/skip warp
  uint64_t wfull[WN_WST];
  uint32_t tmem_base;
  int zmax[2][WN_G][2];                      // per-window max of the two logits, double-buffered by group parity
  int zcnt[2];                               // warps that have added their rows to zmax[parity]: the last one finalises the group
};


// fine-grained chain stamps of tile 0 (first timed group): [24 blocks][16 events] behind the hang-report area
#ifdef WWB_WN_DBG2
#define WN_DBG2(k, ev) do { if (P.dbg && blockIdx.x == 0 && grp == (int64_t)gridDim.x) P.dbg[WN_DBG_ROLES * 48 * 4 + 64 + (k) * 16 + (ev)] = clock64(); } while (0)
#else
#define WN_DBG2(k, ev) do { } while (0)
#endif
#ifdef WWB_TIMELINE   // NVCC_EXTRA=-DWWB_TIMELINE python -m wakeword_detection_b200.build --force, for tools/wn_timeline*.py.
                          // Off by default: compiled in, the stamps kept `grp` and the debug pointer live through the block loop and
                          // cost 11 % of the kernel (86.5 -> 76.9 ms per 2560-stream step)
#define WN_DBG(role, k, ev) do { if (P.dbg && blockIdx.x == 0 && (grp == (int64_t)gridDim.x || grp == 2 * (int64_t)gridDim.x)) P.dbg[((role) * 48 + (k) + (grp == (int64_t)gridDim.x ? 0 : 24)) * 4 + (ev)] = clock64(); } while (0)
#else
#define WN_DBG(role, k, ev) do { } while (0)
#endif


__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(WN_EPI_THREADS) : "memory"); }

// ---- hang diagnosis (compile with -DWWB_HANG_DEBUG and pass a debug buffer, tools/wn_hang.py): every wait is bounded;
// a warp whose wait times out records where it stands ([block][warp]: wait id, block index k, tile, group count, extra)
// behind the timeline area of the debug buffer and exits, so the kernel ends and the host reads a snapshot of all
// stuck warps of the CTA.  hk / hi / hx are per-role locals that only exist in this build.
#ifdef WWB_HANG_DEBUG
#define WN_SPIN_LIMIT (1u << 21)
#define WN_HANG_BASE 4096
__device__ __noinline__ void wn_hang(long long* dbg, int warp, int id, int hk, int hi, uint32_t n_u, uint32_t hx) {
  if (dbg && (threadIdx.x & 31) == 0) {
    long long* base = dbg + WN_HANG_BASE + ((long long)blockIdx.x * 32 + warp) * 8;
    base[0] = id; base[1] = hk; base[2] = hi; base[3] = n_u; base[4] = hx; base[5] = clock64();
  }
  asm volatile("exit;");
}
#define WN_BOUNDED(cond, id) do { uint32_t sp_ = 0; while (!(cond)) if (++sp_ > WN_SPIN_LIMIT) wn_hang(P.dbg, warp, id, hk, hi, n_u, hx); } while (0)
#define WN_MBAR_WAIT(bar, par, id) WN_BOUNDED(mbar_try_wait(bar, par), id)
#define WN_SPIN(bar, par, id) WN_BOUNDED(mbar_test_wait(bar, par), id)
#define WN_HSET(var, val) var = (val)
#else
#define WN_MBAR_WAIT(bar, par, id) mbar_wait(bar, par)
#define WN_SPIN(bar, par, id) mbar_spin(bar, par)
#define WN_HSET(var, val) do { } while (0)
#endif
// busy-poll (no suspension): for the two issuing warps, whose wake-up latency is on every tile's chain
// Not bounded itself (a poll counter cost 0.7 % of the kernel, 12.96 -> 13.06 ms; checked once per 8 unrolled polls: 13.17):
// every wait of the two issuing warps is for an arrival that an epilogue warp produces or for a GEMM the other issuing warp
// issues after such an arrival, and the epilogue warps wait with mbar_wait, which traps after 2^24 retries - a broken
// protocol still ends as a launch failure, not as a hung GPU (that is how the deadlock of the res/skip-detect variant
// surfaced, profiles/r2_notes.md).
__device__ __forceinline__ void mbar_spin(uint64_t* bar, uint32_t parity) {
#pragma unroll 1
  while (!mbar_test_wait(bar, parity)) { }
}
// A/B switch (tools/build_variant.sh): -DWWB_WN_ISS_SUSPEND puts the two issuing warps back on the suspending try_wait
// (busy-polling them: 13.85 -> 13.39 ms per 512 x 10 s; busy-polling the epilogue warps too: 15.5 ms, and 13.7-14.1 ms when only
// their res/skip wait or only the blocks with few active tiles poll)
#define WN_WAIT_E(bar, par, id) WN_MBAR_WAIT(bar, par, id)
#ifndef WWB_WN_ISS_SUSPEND
#define WN_WAIT_I(bar, par, id) WN_SPIN(bar, par, id)
#else
#define WN_WAIT_I(bar, par, id) WN_MBAR_WAIT(bar, par, id)
#endif

__global__ void __launch_bounds__(WN_THREADS, 1) wavenet_tc_kernel(const WnTcParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  WnSmem& sm = *reinterpret_cast<WnSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler
  const int64_t n_win = P.wm.n_win_dev ? (int64_t)*P.wm.n_win_dev : P.wm.n_win;
  const int64_t n_groups = P.stream_mode ? P.wm.n_streams * (int64_t)P.chunks_per_stream : (n_win + WN_G - 1) / WN_G;
  const int L = P.L;

  // ---- one-time setup ----
  for (int i = tid; i < (int)(sizeof(sm.U) / 16); i += WN_THREADS) reinterpret_cast<uint4*>(sm.U)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < (int)(sizeof(WnHead) / 16); i += WN_THREADS)
    reinterpret_cast<uint4*>(&sm.head)[i] = reinterpret_cast<const uint4*>(P.head)[i];
  if (tid < 2 * WN_G * 2) (&sm.zmax[0][0][0])[tid] = WN_KEY_NEG_INF;
  if (tid < 2) sm.zcnt[tid] = 0;
  if (tid == 0) {
    for (int i = 0; i < WN_NT; ++i) {
      mbar_init(&sm.bar_u[i], i == 0 ? 5 : 4); mbar_init(&sm.bar_g[i], 4); mbar_init(&sm.bar_gate[i], 1); mbar_init(&sm.bar_rs[i], 1);
      mbar_init(&sm.bar_det[i], 1); mbar_init(&sm.bar_dq[i], 4);
    }
    for (int s = 0; s < WN_WST; ++s) mbar_init(&sm.wfull[s], 1);
    mbar_fence_init();
  }
  if (warp == WN_EPI_WARPS) tmem_alloc(&sm.tmem_base, 512);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = sm.tmem_base;
  const int nsplit = P.nsplit;
  const uint32_t idesc_gate = make_idesc_f16(128, 32), idesc_rs = make_idesc_f16(128, 48);

  if (warp < WN_EPI_WARPS) {
    // =========================== epilogue threads: one row each ===========================
    const int tile = warp >> 2, q = warp & 3;
    const int o = tile * 128 + q * 32 + lane;       // row within the group
    const int R = P.rstride;
    const int t = o / R, w = o - t * R;             // time step, window (stream mode: R = 1, t = frame offset in the chunk)
    const uint32_t tacc = tmem + tile * WN_TMEM_TILE;                 // this tile's TMEM columns (lane 0)
    const uint32_t tbase = tacc + ((uint32_t)(q * 32) << 16);         // ... seen from this warp's lane quadrant
    uint32_t n_gate = 0, n_rs = 0, n_u = 0;  // completed phases of bar_gate / bar_rs ; groups done
#ifdef WWB_HANG_DEBUG
    int hk = -1, hi = tile; uint32_t hx = 0;
#endif
    unsigned char* const Urow = sm.U + (WN_PAD + o) * 16;
    float4* const sk = sm.skip + o;           // this row's skip sums: sk[c4 * WN_ROWS], conflict-free 16-byte accesses
    // (keeping 8 / 16 / 24 / 32 of the 32 sums in registers instead: 14.15 / 14.28 / 13.93 / 13.96 ms against 13.50 - profiles/r2_notes.md)
    {
      uint32_t one[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) one[i] = 0u;
      one[0] = 0x3c003c00u;   // (1.0h, 1.0h)
      tmem_st16(tmem + ((uint32_t)(q * 32) << 16) + WN_C_ONE, one);
      tmem_st_wait();
    }
    const u64 ZERO2 = pk(0.f, 0.f), ONE2 = pk(1.f, 1.f);
    const int jn = P.join[tile];            // first block of this tile
    const int src_slot = P.src_slot[tile];  // where its rows start from
    const bool stream_mode = P.stream_mode != 0;

    // Start state of a row: the input layer x0 = ReLU(in_w * mel + in_b) (computed once per mel row by wn_input_kernel)
    // with an empty skip sum, or - for a tile that joins at block jn > 0 - the stream-level snapshot after block jn-1.
    // The state of the NEXT group is fetched straight into x / skip before this group's detect epilogue (both are dead
    // by then), so its global-memory latency is not on the group-boundary chain.
    u64 x[8];               // channel pairs
    bool valid = false, snap_out = false;
    int64_t b = 0;
    float* snap_dst = nullptr;
    auto fetch_state = [&](int64_t g) {
      bool vn = g < n_groups;
      int64_t row = 0;
      snap_out = false;
      if (stream_mode) {
        const int64_t s0 = g / P.chunks_per_stream;
        const int c = (int)(g - s0 * P.chunks_per_stream);
        const int f = c * WN_CHUNK_STEP + o;
        vn = vn && f < P.wm.ring;
        row = s0 * P.wm.ring + (vn ? f : 0);
        snap_out = vn && (c == 0 || o >= WN_CHUNK_WARM);
        snap_dst = P.snap + row * 4;   // float4 index `row` of plane 0 (planes are n_rows float4 apart)
      } else {
        b = g * WN_G + w;
        vn = vn && (t < L) && (b < n_win);
        int64_t s0 = 0;
        int start = 0;
        if (vn) win_origin(P.wm, b, s0, start);
        int rr = start + (vn ? t : 0);
        if (rr >= P.wm.ring) rr -= P.wm.ring;
        row = s0 * P.wm.ring + rr;
      }
      valid = vn;
      if (src_slot >= 0) {
        // snapshot planes: [slot][12 float4 columns: x 0-3, skip 4-11][n_rows] - the rows of a warp are a handful of consecutive
        // frames, so each of the 12 loads touches a few sectors (as [row][48 floats] the stream pass's stores were one sector per lane)
        const float4* p = reinterpret_cast<const float4*>(P.snap) + (int64_t)src_slot * (WN_SNAP_F / 4) * P.n_rows + row;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = vn ? __ldg(p + (int64_t)i * P.n_rows) : make_float4(0.f, 0.f, 0.f, 0.f);
          x[2 * i] = pk(v.x, v.y);
          x[2 * i + 1] = pk(v.z, v.w);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) sk[i * WN_ROWS] = vn ? __ldg(p + (int64_t)(4 + i) * P.n_rows) : make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        const float4* p = reinterpret_cast<const float4*>(P.x0) + row;   // column planes like the snapshots: [4][n_rows] float4
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = vn ? __ldg(p + (int64_t)i * P.n_rows) : make_float4(0.f, 0.f, 0.f, 0.f);
          x[2 * i] = pk(v.x, v.y);
          x[2 * i + 1] = pk(v.z, v.w);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) sk[i * WN_ROWS] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // ---- start state -> U row of buffer 0 (operand of the first gate GEMM); that block's BatchNorm is folded into its gate weights ----
    auto put_start_state = [&]() {
      uint32_t ur[16];
#pragma unroll
      for (int i = 0; i < 8; ++i) split2(x[i], ur[i], ur[8 + i]);
      if (valid) {
        *reinterpret_cast<uint4*>(Urow) = make_uint4(ur[0], ur[1], ur[2], ur[3]);
        *reinterpret_cast<uint4*>(Urow + WN_PU) = make_uint4(ur[4], ur[5], ur[6], ur[7]);
        *reinterpret_cast<uint4*>(Urow + 2 * WN_PU) = make_uint4(ur[8], ur[9], ur[10], ur[11]);
        *reinterpret_cast<uint4*>(Urow + 3 * WN_PU) = make_uint4(ur[12], ur[13], ur[14], ur[15]);
      }
      tmem_st16(tbase + WN_C_U, ur);
      tmem_st_wait();
      fence_before_sync();
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.bar_u[tile]);
    };
    fetch_state(blockIdx.x);
    if ((int64_t)blockIdx.x < n_groups) put_start_state();
    for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x, ++n_u) {
      const bool valid_g = valid;             // (fetch_state of the next group overwrites `valid` before the detect epilogue)
      const bool snap_g = snap_out;
      float* const snap_g_dst = snap_dst;
      for (int k = jn; k < 24; ++k) {
        WN_HSET(hk, k);
        // ---- epilogue 1: gated activation ----
        WN_WAIT_E(&sm.bar_gate[tile], n_gate & 1, 5);
        ++n_gate;
        fence_after_sync();
        if (q == 0 && lane == 0) WN_DBG(tile, k, 0);
        if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 0);
        {
          // The accumulator columns are ordered [tanh 0-7 | sigmoid 0-7 | tanh 8-15 | sigmoid 8-15] (wavenet_pack_blocks), so
          // each half is consumed by ONE load and its g hi/lo can be stored over it right away: 8 result registers
          // live instead of 16 (the kernel sits at the register limit of 832 threads)
#pragma unroll
          for (int h8 = 0; h8 < 2; ++h8) {
            float v[16];
            tmem_ld16(tbase + h8 * 16, v);
            tmem_ld_wait();
            if (h8 == 0 && tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 1);
            uint32_t gh[4], gl[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              // accumulators arrive as a2 = -2*log2(e)*(a + b_t), b2 = -log2(e)*(b + b_s) (scaled weights, bias GEMM)
              const float a0 = v[2 * p], a1 = v[2 * p + 1], b0 = v[8 + 2 * p], b1 = v[8 + 2 * p + 1];
              // exponents clamped at 30: tanh is -1 and sigmoid 0 to 1e-9 beyond, and both denominators stay below
              // 2^61, so ONE reciprocal serves the pair of channels (1/d0 = d1/(d0 d1)): 5 SFU ops per pair instead
              // of 6 - the SFU queue is what stretches this epilogue (profiles/r1_notes.md)
              const float ea0 = ex2_approx(fminf(a0, 30.f)), ea1 = ex2_approx(fminf(a1, 30.f));
              const float eb0 = ex2_approx(fminf(b0, 30.f)), eb1 = ex2_approx(fminf(b1, 30.f));
              const u64 tt = fadd2(pk(eb0, eb1), ONE2);
              float d0, d1;
              upk(ffma2(pk(ea0, ea1), tt, tt), d0, d1);                 // (1 + e^-2a)(1 + e^-b)
              const float rp = rcp_approx(d0 * d1);
              const float r0 = rp * d1, r1 = rp * d0;
              const u64 g = pk(fmaf(-ea0, r0, r0), fmaf(-ea1, r1, r1)); // tanh(a) * sigmoid(b)
              split2(g, gh[p], gl[p]);
            }
            tmem_st4(tbase + WN_C_G + h8 * 4, gh);
            tmem_st4(tbase + WN_C_G + 8 + h8 * 4, gl);
          }
          if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 2);
          tmem_st_wait();
          if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 3);
        }
        fence_before_sync();
        if (q == 0 && lane == 0) WN_DBG(tile, k, 1);
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.bar_g[tile]);
        if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 4);

        // ---- epilogue 2a: residual, next block's BN -> u (releases the next gate GEMM) ----
        WN_WAIT_E(&sm.bar_rs[tile], n_rs & 1, 6);
        ++n_rs;
        fence_after_sync();
        if (q == 0 && lane == 0) WN_DBG(tile, k, 2);
        if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 5);
        const bool last = (k == 23);
        if (!last) {
#pragma unroll
          for (int h8 = 0; h8 < 2; ++h8) {
            float r[8];
            tmem_ld8(tbase + WN_C_R + h8 * 8, r);
            tmem_ld_wait();
            uint32_t uh[4], ul[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              const int c = h8 * 4 + p;
              x[c] = add_relu2(x[c], pk(r[2 * p], r[2 * p + 1]));
              split2(x[c], uh[p], ul[p]);   // the next block's BN is folded into its gate weights
            }
            if (valid_g) {
              *reinterpret_cast<uint4*>(Urow + h8 * WN_PU) = make_uint4(uh[0], uh[1], uh[2], uh[3]);
              *reinterpret_cast<uint4*>(Urow + (2 + h8) * WN_PU) = make_uint4(ul[0], ul[1], ul[2], ul[3]);
            }
            tmem_st4(tbase + WN_C_U + h8 * 4, uh);
            tmem_st4(tbase + WN_C_U + 8 + h8 * 4, ul);
          }
          if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 6);
          tmem_st_wait();
          if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 8);
          fence_before_sync();
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.bar_u[tile]);
          if (q == 0 && lane == 0) WN_DBG(tile, k, 3);
          if (tile == 0 && q == 0 && lane == 0) WN_DBG2(k, 9);
        }
        // ---- epilogue 2b: skip sum (off the critical path: the next gate GEMM is already running) ----
        // The 32 sums of a row live in shared memory, not in registers: with 16 + 32 state registers per row the kernel
        // spilled inside this loop at the 72 registers 832 threads leave; 8 LDS.128 + 8 STS.128 per row and block that
        // nothing waits for are cheaper.  After the last block the sums in hand become the detect head's input
        // (ReLU, fp16 hi/lo; channels 0-15 -> the u columns, 16-31 -> the g columns).
#pragma unroll
        for (int h8 = 0; h8 < 4; ++h8) {
          float s[8];
          tmem_ld8(tbase + WN_C_R + 16 + h8 * 8, s);
          const float4 c0 = sk[(2 * h8) * WN_ROWS], c1 = sk[(2 * h8 + 1) * WN_ROWS];
          tmem_ld_wait();
          const u64 n0 = add_relu2(pk(c0.x, c0.y), pk(s[0], s[1])), n1 = add_relu2(pk(c0.z, c0.w), pk(s[2], s[3]));
          const u64 n2 = add_relu2(pk(c1.x, c1.y), pk(s[4], s[5])), n3 = add_relu2(pk(c1.z, c1.w), pk(s[6], s[7]));
          float4 o0, o1;
          upk(n0, o0.x, o0.y); upk(n1, o0.z, o0.w); upk(n2, o1.x, o1.y); upk(n3, o1.z, o1.w);
          sk[(2 * h8) * WN_ROWS] = o0;
          sk[(2 * h8 + 1) * WN_ROWS] = o1;
          if (last) {
            uint32_t eh[4], el[4];
            split2(relu2(n0), eh[0], el[0]); split2(relu2(n1), eh[1], el[1]);
            split2(relu2(n2), eh[2], el[2]); split2(relu2(n3), eh[3], el[3]);
            const uint32_t cx = tbase + (h8 < 2 ? WN_C_U : WN_C_G) + (h8 & 1) * 4;
            tmem_st4(cx, eh);
            tmem_st4(cx + 8, el);
          }
        }
        fence_before_sync();
        if (stream_mode) {
          // stream-level pass: x and the skip prefix sum after this block, for the window tiles that join at block k+1
          const int sl = P.snap_slot[k];
          if (sl >= 0 && snap_g) {
            float4* dst = reinterpret_cast<float4*>(snap_g_dst) + (int64_t)sl * (WN_SNAP_F / 4) * P.n_rows;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float a0, a1, a2, a3;
              upk(x[2 * i], a0, a1);
              upk(x[2 * i + 1], a2, a3);
              dst[(int64_t)i * P.n_rows] = make_float4(a0, a1, a2, a3);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) dst[(int64_t)(4 + i) * P.n_rows] = sk[i * WN_ROWS];
          }
        }
        if (last) {
          tmem_st_wait();
          fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.bar_dq[tile]);
          if (q == 0 && lane == 0) WN_DBG(tile, k, 3);
        }
      }

      if (P.enc_out && valid_g) {
        float4* dst = reinterpret_cast<float4*>(P.enc_out + ((grp * WN_G + w) * L + t) * 32);
#pragma unroll
        for (int n = 0; n < 8; ++n) dst[n] = sk[n * WN_ROWS];
      }
      if (tile == 0 && q == 0 && lane == 0) WN_DBG(WN_NT + 1, 20, 0);   // boundary timeline: e2b(23) done
      WN_HSET(hk, 24);
      fetch_state(grp + gridDim.x);   // next group's start state: in flight during the detect epilogue
      // ---- detect head epilogue: ReLU(D + b1) -> 32->2 -> max over time ----
      WN_MBAR_WAIT(&sm.bar_det[tile], n_u & 1, 8);
      fence_after_sync();
      if (tile == 0 && q == 0 && lane == 0) WN_DBG(WN_NT + 1, 20, 1);   // detect GEMM done
      // 32 -> 2 with 128-bit loads of the constants and four independent partial sums per logit (as 96 scalar loads
      // feeding two 32-long dependent FMA chains this epilogue took ~2500 clk on the group-boundary critical path)
      float z0, z1;
      {
        u64 acc0[2] = {pk(0.f, 0.f), pk(0.f, 0.f)}, acc1[2] = {pk(0.f, 0.f), pk(0.f, 0.f)};
#pragma unroll
        for (int h8 = 0; h8 < 4; ++h8) {
          float d[8];
          tmem_ld8(tbase + WN_C_R + h8 * 8, d);
          tmem_ld_wait();
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            const int c = h8 * 8 + 2 * p;
            const u64 e = relu2(fadd2(pk(d[2 * p], d[2 * p + 1]), pk(P.det1_b[c], P.det1_b[c + 1])));
            acc0[p & 1] = ffma2(pk(P.det2_w[c], P.det2_w[c + 1]), e, acc0[p & 1]);
            acc1[p & 1] = ffma2(pk(P.det2_w[32 + c], P.det2_w[32 + c + 1]), e, acc1[p & 1]);
          }
        }
        float fa, fb;
        upk(fadd2(acc0[0], acc0[1]), fa, fb);
        z0 = (fa + fb) + P.det2_b[0];
        upk(fadd2(acc1[0], acc1[1]), fa, fb);
        z1 = (fa + fb) + P.det2_b[1];
      }
      // the detect accumulator has been read: hand the NEXT group's start state to the gate warp before the reductions
      // below (they are ~1000 clk of shuffles and shared-memory atomics that the next gate GEMM does not depend on)
      const int zp = (int)(n_u & 1);
      if (!stream_mode) {
        // a warp's 32 rows are ~11 time steps of all three windows: one reduction + one atomic per window and logit
#pragma unroll
        for (int dw = 0; dw < WN_G; ++dw) {
          const bool mine = valid_g && (w == dw);
          const unsigned m = __ballot_sync(0xffffffffu, mine);
          if (m) {
            const int k0 = __reduce_max_sync(0xffffffffu, mine ? f2key(z0) : WN_KEY_NEG_INF);
            const int k1 = __reduce_max_sync(0xffffffffu, mine ? f2key(z1) : WN_KEY_NEG_INF);
            if (lane == 0) {
              atomicMax(&sm.zmax[zp][dw][0], k0);
              atomicMax(&sm.zmax[zp][dw][1], k1);
            }
          }
        }
        if (tile == 0 && q == 0 && lane == 0) WN_DBG(WN_NT + 1, 20, 2);   // detect epilogue done
        // No CTA barrier at the group boundary: the LAST of the 20 warps to add its rows turns the maxima into posteriors
        // and clears them.  zmax / zcnt are double-buffered by group parity; the tiles of a CTA are never more than a few
        // blocks apart (each gate GEMM needs the tile below one block back), so group g + 2 cannot reach this point before
        // group g has been finalised.
        if (lane == 0) {
          __threadfence_block();
          if (atomicAdd(&sm.zcnt[zp], 1) == WN_EPI_WARPS - 1) {
            __threadfence_block();
            for (int dw = 0; dw < WN_G; ++dw) {
              const int64_t bb = grp * WN_G + dw;
              const float a0 = key2f(sm.zmax[zp][dw][0]), a1 = key2f(sm.zmax[zp][dw][1]);
              sm.zmax[zp][dw][0] = WN_KEY_NEG_INF;
              sm.zmax[zp][dw][1] = WN_KEY_NEG_INF;
              if (bb < n_win) {
                const float m = fmaxf(a0, a1);
                const float e0 = expf(a0 - m), e1 = expf(a1 - m), sden = e0 + e1;
                if (P.det_out) { P.det_out[bb * 2] = e0 / sden; P.det_out[bb * 2 + 1] = e1 / sden; }
                if (P.post) P.post[bb] = e1 / sden;
              }
            }
            sm.zcnt[zp] = 0;
          }
        }
        __syncwarp();
      }
      put_start_state();
      if (tile == 0 && q == 0 && lane == 0) WN_DBG(WN_NT + 1, 20, 3);
    }
  } else if (warp == WN_EPI_WARPS) {
    // =========================== gate-GEMM warp + weight loader ===========================
    // Issues the gate GEMMs tile after tile, each as soon as the tile's epilogue 2 has arrived.  Because one
    // thread issues them, they execute back to back in tile order, which staggers the tiles: while tile i+1's
    // gate GEMM runs, tile i is in epilogue 1 (SFU), tile i-1 in its res/skip GEMM or epilogue 2 (FMA/ALU).
    // gate(k,i) also needs epilogue 2 of (k-1,i-1) (its taps reach 16 rows into tile i-1): awaited one step earlier.
    uint32_t n_u = 0;
#ifdef WWB_HANG_DEBUG
    int hk = -1, hi = -1; uint32_t hx = 0;
#endif
    const uint64_t dU = make_desc(smem_u32(sm.U), WN_PU, 128);                   // U row 0, hi plane
    const uint64_t dWg = make_desc(smem_u32(sm.W[0]), 512, 128);                 // gate B: stage 0, tap 0, hi plane
    const uint64_t dBg = make_desc(smem_u32(sm.W[0]) + WN_OFF_GBIAS, 512, 128);  // gate bias B: stage 0
    const uint64_t dH = make_desc(smem_u32(sm.head.det1_B), 512, 128);           // detect B: k-step 0, hi plane
    uint32_t my_groups = 0;
    for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) ++my_groups;
    const uint32_t total_loads = my_groups * 24;
    for (uint32_t n = 0; n < (uint32_t)WN_WST && n < total_loads; ++n)
      if (lane == 0) {
        mbar_arrive_expect_tx(&sm.wfull[n], WN_WBLK);
        bulk_g2s(sm.W[n], P.wblob + (size_t)n * WN_WBLK, WN_WBLK, &sm.wfull[n]);
      }
    uint32_t n_w = 0;         // global block index (24 per group)
    uint32_t cu[WN_NT];       // consumed phases of bar_u, per tile (a tile that joins at block j has 24 - j per group)
#pragma unroll
    for (int i = 0; i < WN_NT; ++i) cu[i] = 0;
    const uint32_t rs3 = (uint32_t)P.rstride;
    for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x, ++n_u) {
      for (int k = 0; k < 24; ++k, ++n_w) {
        WN_MBAR_WAIT(&sm.wfull[n_w % WN_WST], (n_w / WN_WST) & 1, 1);
        const uint32_t d = (uint32_t)P.dil[k] * rs3;     // tap distance in rows
        const uint64_t wofs = (uint64_t)((n_w % WN_WST) * (WN_WBLK >> 4));
        const uint64_t b0 = dWg + wofs, bb = dBg + wofs;
#pragma unroll
        for (int i = 0; i < WN_NT; ++i) {
          if (k < P.join[i]) continue;                   // the tile's rows are still shared (stream-level) activations
          WN_HSET(hk, k); WN_HSET(hi, i);
          if (i == 1) WN_DBG(WN_NT + 1, k, 0);
          if (i == 0 && lane == 0) WN_DBG2(k, 10);
          WN_WAIT_I(&sm.bar_u[i], cu[i] & 1, 2);
          ++cu[i];
          if (i == 0 && lane == 0) WN_DBG2(k, 11);
          if (i == 1) WN_DBG(WN_NT + 1, k, 1);
          fence_after_sync();
          if (elect_one()) {   // one lane issues the whole tile (uniform descriptors, no per-MMA election)
            const uint32_t tacc = tmem + i * WN_TMEM_TILE;
            const uint64_t a0 = dU + (uint64_t)(WN_PAD + i * 128 - 2 * d), a1 = dU + (uint64_t)(WN_PAD + i * 128 - d);
            const uint64_t lo_a = (uint64_t)((2 * WN_PU) >> 4), lo_b = (uint64_t)(3072 >> 4);
            mma_f16_ss(tacc, a0, b0, idesc_gate, false);
            if (nsplit == 3) {
              mma_f16_ss(tacc, a0 + lo_a, b0, idesc_gate, true);
              mma_f16_ss(tacc, a0, b0 + lo_b, idesc_gate, true);
            }
            mma_f16_ss(tacc, a1, b0 + 64, idesc_gate, true);
            if (nsplit == 3) {
              mma_f16_ss(tacc, a1 + lo_a, b0 + 64, idesc_gate, true);
              mma_f16_ss(tacc, a1, b0 + 64 + lo_b, idesc_gate, true);
            }
            mma_f16_ts(tacc, tacc + WN_C_U, b0 + 128, idesc_gate, true);
            if (nsplit == 3) {
              mma_f16_ts(tacc, tacc + WN_C_U + 8, b0 + 128, idesc_gate, true);
              mma_f16_ts(tacc, tacc + WN_C_U, b0 + 128 + lo_b, idesc_gate, true);
            }
            mma_f16_ts(tacc, tmem + WN_C_ONE, bb, idesc_gate, true);
            mma_commit(&sm.bar_gate[i]);
            if (i == 0) WN_DBG2(k, 12);
            if (i == 0) WN_DBG(WN_NT, k, 0);
            if (i == WN_NT - 1) WN_DBG(WN_NT, k, 1);
          }
          __syncwarp();
          if (i == 1) WN_DBG(WN_NT + 1, k, 2);
        }
        // every active tile has finished block n_w-1 (its epilogue 2 was awaited above; at k == 0 the detect loop below
        // waited for every tile's block 23): refill that stage
        auto refill = [&](uint32_t m) {   // block m is finished everywhere: load block m + WN_WST into its stage
          const uint32_t nl = m + WN_WST;
          if (nl < total_loads && lane == 0) {
            mbar_arrive_expect_tx(&sm.wfull[nl % WN_WST], WN_WBLK);
            bulk_g2s(sm.W[nl % WN_WST], P.wblob + (size_t)(nl % 24) * WN_WBLK, WN_WBLK, &sm.wfull[nl % WN_WST]);
          }
        };
        if (n_w >= 1) refill(n_w - 1);
      }
      // detect head: D[128,32] = ReLU(skip)[128,32] * W1^T ; k-step 0 from the u columns, k-step 1 from the g columns
#pragma unroll
      for (int i = 0; i < WN_NT; ++i) {
        WN_MBAR_WAIT(&sm.bar_dq[i], n_u & 1, 9);
        fence_after_sync();
        if (elect_one()) {
          const uint32_t tacc = tmem + i * WN_TMEM_TILE;
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint32_t ta = tacc + (kk == 0 ? WN_C_U : WN_C_G);
            const uint64_t bh = dH + (uint64_t)((kk * 2 * 512) >> 4), bl = bh + (uint64_t)(2048 >> 4);
            mma_f16_ts(tacc + WN_C_R, ta, bh, idesc_gate, kk != 0);
            if (nsplit == 3) {
              mma_f16_ts(tacc + WN_C_R, ta + 8, bh, idesc_gate, true);
              mma_f16_ts(tacc + WN_C_R, ta, bl, idesc_gate, true);
            }
          }
          mma_commit(&sm.bar_det[i]);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== res/skip-GEMM warp ===========================
    // Tile after tile: when the tile's four warps have stored g (epilogue 1), issue its res and skip GEMMs
    // (A = g from TMEM, + bias k-step).  Epilogue 2a of the tile will then overwrite rows that gate(k) of
    // tile+1 reads, so that GEMM must have COMPLETED first (it is issued by another thread: no implicit order).
    uint32_t n_u = 0, n_w = 0;
#ifdef WWB_HANG_DEBUG
    int hk = -1, hi = -1; uint32_t hx = 0;
#endif
    const uint64_t dWr = make_desc(smem_u32(sm.W[0]) + WN_GATE_B, 768, 128);     // res/skip B: stage 0, hi plane
    const uint64_t dBr = make_desc(smem_u32(sm.W[0]) + WN_OFF_RBIAS, 768, 128);  // res/skip bias B: stage 0
    const uint32_t ones = tmem + WN_C_ONE;
    uint32_t cg[WN_NT];       // consumed phases of bar_g[i]: one per block the tile takes part in
#pragma unroll
    for (int i = 0; i < WN_NT; ++i) cg[i] = 0;
    // This warp also owns the padding rows in front of row 0 (x_pad of the NEXT block, see the header): it writes them
    // right after issuing rs(k, 0); their reader, gate(k+1, 0), waits for this warp's
    // arrival on bar_u[0] - so the copy overlaps tile 0's res/skip GEMM and epilogue 2 instead of sitting inside it.
    auto store_pad = [&](const unsigned char* chunk) {   // chunk: 64 bytes (hi0, hi1, lo0, lo1)
      const uint4* c4 = reinterpret_cast<const uint4*>(chunk);
      const uint4 c0 = c4[0], c1 = c4[1], c2 = c4[2], c3 = c4[3];
#pragma unroll
      for (int r = lane; r < WN_PAD; r += 32) {
        unsigned char* up = sm.U + r * 16;
        *reinterpret_cast<uint4*>(up) = c0;
        *reinterpret_cast<uint4*>(up + WN_PU) = c1;
        *reinterpret_cast<uint4*>(up + 2 * WN_PU) = c2;
        *reinterpret_cast<uint4*>(up + 3 * WN_PU) = c3;
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.bar_u[0]);
    };
    if ((int64_t)blockIdx.x < n_groups) store_pad(sm.head.pad0);   // level 0 of the first group
    for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x, ++n_u) {
      for (int k = 0; k < 24; ++k, ++n_w) {
        const uint64_t wofs = (uint64_t)((n_w % WN_WST) * (WN_WBLK >> 4));
        const uint64_t bh = dWr + wofs, bb = dBr + wofs, lo_b = (uint64_t)(1536 >> 4);
        WN_MBAR_WAIT(&sm.wfull[n_w % WN_WST], (n_w / WN_WST) & 1, 11);   // (observe the weight load ourselves)
#pragma unroll
        for (int i = 0; i < WN_NT; ++i) {
          if (k < P.join[i]) continue;
          WN_HSET(hk, k); WN_HSET(hi, i);
          if (i == 3) WN_DBG(WN_NT + 2, k, 0);
          // busy-poll: this warp has nothing else to do and its wake-up latency is on every tile's chain
          WN_WAIT_I(&sm.bar_g[i], cg[i] & 1, 10);
          // gate(k, i+1) reads rows of tile i that epilogue 2a of (k, i) overwrites.  cg[i+1] has not been advanced for
          // block k yet (tile i+1 comes next in this loop), so it is the phase of gate(k, i+1)
          if (i < WN_NT - 1 && k >= P.join[i + 1]) WN_WAIT_I(&sm.bar_gate[i + 1], cg[i + 1] & 1, 3);
          ++cg[i];
          if (i == 0 && lane == 0) WN_DBG2(k, 13);
          if (i == 3) WN_DBG(WN_NT + 2, k, 1);
          fence_after_sync();
          if (elect_one()) {
            // res and skip in one N = 48 GEMM.  One commit: the next gate GEMM overwrites the g columns, so epilogue 2a
            // must not release it before this GEMM has read them
            const uint32_t tacc = tmem + i * WN_TMEM_TILE;
            mma_f16_ts(tacc + WN_C_R, tacc + WN_C_G, bh, idesc_rs, false);
            if (nsplit == 3) {
              mma_f16_ts(tacc + WN_C_R, tacc + WN_C_G + 8, bh, idesc_rs, true);
              mma_f16_ts(tacc + WN_C_R, tacc + WN_C_G, bh + lo_b, idesc_rs, true);
            }
            mma_f16_ts(tacc + WN_C_R, ones, bb, idesc_rs, true);
            mma_commit(&sm.bar_rs[i]);
            if (i == 0) WN_DBG2(k, 14);
            if (i == 0) WN_DBG(WN_NT, k, 2);
            if (i == WN_NT - 1) WN_DBG(WN_NT, k, 3);
          }
          __syncwarp();
          if (i == 0)    // padding rows of the next block (after block 23: level 0 of the next group)
            store_pad(k < 23 ? sm.W[n_w % WN_WST] + WN_OFF_F32 + 320 : sm.head.pad0);
          if (i == 3) WN_DBG(WN_NT + 2, k, 2);
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == WN_EPI_WARPS) tmem_dealloc(tmem, 512);
}

// the gate pre-activations are produced pre-scaled for ex2: tanh half by -2*log2(e), sigmoid half by -log2(e)
static double gate_scale(int n) { return n < 16 ? -2.8853900817779268 : -1.4426950408889634; }
// accumulator column of gate output n (0-15 tanh half, 16-31 sigmoid half): [tanh 0-7 | sigmoid 0-7 | tanh 8-15 | sigmoid 8-15],
// so that epilogue 1 consumes the accumulator in two self-contained halves
static int gate_col(int n) { const int c = n & 15; return (c >> 3) * 16 + (n >> 4) * 8 + (c & 7); }

// false if x is outside the fp16 range (hi rounds to infinity) or not finite
static bool put_split(std::vector<unsigned char>& buf, size_t hi_off, size_t lo_off, float x, bool split) {
  __half h = __float2half_rn(x);
  __half l = split ? __float2half_rn(x - __half2float(h)) : __float2half_rn(0.f);
  memcpy(&buf[hi_off], &h, 2);
  memcpy(&buf[lo_off], &l, 2);
  return isfinite(__half2float(h));
}

// gate_w [24][48][32] (k = tap*16+ch ; n), rs_w [24][16][48], biases, bn, dilation (fp32 device-layout copies
// made by api.cu on the host before upload)
// padding rows for a block whose BatchNorm is (mul, add): x_pad = -add / mul (=> u_pad = 0), as the 64-byte
// (hi chunk 0, hi chunk 1, lo chunk 0, lo chunk 1) image of one U row.  false if a scale is 0 (cannot be folded) or
// -add / mul is outside the fp16 range.
static bool put_pad_rows(std::vector<unsigned char>& out, size_t off, const float* mul, const float* add) {
  bool ok = true;
  for (int c = 0; c < 16; ++c) {
    if (mul[c] == 0.f) return false;
    const size_t o = off + (size_t)(c / 8) * 16 + (c % 8) * 2;
    ok &= put_split(out, o, o + 32, (float)(-(double)add[c] / (double)mul[c]), true);
  }
  return ok;
}

std::vector<unsigned char> wavenet_pack_blocks(const float* gate_w, const float* gate_b, const float* rs_w,
                                               const float* rs_b, const float* bn_mul, const float* bn_add,
                                               const int* dilation) {
  std::vector<unsigned char> out((size_t)24 * WN_WBLK, 0);
  bool ok = true;
  for (int b = 0; b < 24; ++b) {
    const size_t base = (size_t)b * WN_WBLK;
    for (int k = 0; k < 48; ++k)
      for (int n = 0; n < 32; ++n) {
        const int c = k / 8, e = k % 8;
        const size_t off = base + ((size_t)c * 32 + gate_col(n)) * 16 + e * 2;
        ok &= put_split(out, off, off + 3072, (float)((double)gate_w[((size_t)b * 48 + k) * 32 + n] * (double)bn_mul[b * 16 + k % 16] * gate_scale(n)), true);
      }
    for (int k = 0; k < 16; ++k)
      for (int n = 0; n < 48; ++n) {
        const int c = k / 8, e = k % 8;
        const size_t off = base + WN_GATE_B + ((size_t)c * 48 + n) * 16 + e * 2;
        ok &= put_split(out, off, off + 1536, rs_w[((size_t)b * 16 + k) * 48 + n], true);
      }
    float f[113] = {0};
    f[112] = (float)dilation[b];
    memcpy(&out[base + WN_OFF_F32], f, sizeof(f));
    if (b < 23) ok &= put_pad_rows(out, base + WN_OFF_F32 + 320, bn_mul + (b + 1) * 16, bn_add + (b + 1) * 16);
    // bias operands of the 'ones' GEMM: row n = (hi, lo, 0, ...); the second k-chunk stays zero
    for (int n = 0; n < 32; ++n) {
      const size_t off = base + WN_OFF_GBIAS + (size_t)gate_col(n) * 16;
      double bsum = gate_b[b * 32 + n];   // + W * bn_add (the folded BatchNorm shift)
      for (int k = 0; k < 48; ++k) bsum += (double)gate_w[((size_t)b * 48 + k) * 32 + n] * (double)bn_add[b * 16 + k % 16];
      ok &= put_split(out, off, off + 2, (float)(bsum * gate_scale(n)), true);
    }
    for (int n = 0; n < 48; ++n) {
      const size_t off = base + WN_OFF_RBIAS + (size_t)n * 16;
      ok &= put_split(out, off, off + 2, rs_b[b * 48 + n], true);
    }
  }
  return ok ? out : std::vector<unsigned char>();
}

std::vector<unsigned char> wavenet_pack_head(const float* bn_mul0, const float* bn_add0, const float* det1_w_nk,
                                             const float* det1_b, const float* det2_w, const float* det2_b) {
  std::vector<unsigned char> out(sizeof(WnHead), 0);
  WnHead* h = reinterpret_cast<WnHead*>(out.data());
  bool ok = put_pad_rows(out, offsetof(WnHead, pad0), bn_mul0, bn_add0);
  memcpy(h->det1_b, det1_b, sizeof(h->det1_b));
  memcpy(h->det2_w, det2_w, sizeof(h->det2_w));
  memcpy(h->det2_b, det2_b, sizeof(h->det2_b));
  const size_t boff = offsetof(WnHead, det1_B);
  for (int n = 0; n < 32; ++n)
    for (int k = 0; k < 32; ++k) {
      const int c = k / 8, e = k % 8;
      const size_t off = boff + ((size_t)c * 32 + n) * 16 + e * 2;
      ok &= put_split(out, off, off + 2048, det1_w_nk[n * 32 + k], true);
    }
  return ok ? out : std::vector<unsigned char>();
}

// Input layer (Wavenet/encode.tflite op 0: 1x1 conv 40 -> 16 + ReLU, SURVEY.md Appendix A3) once per mel row, fp32:
// x0[row, c] = ReLU(b[c] + sum_k w[k][c] * mel[row, k]).  4 threads per row, 4 channels each; stored as 4 column planes
// of n_rows float4 (the rows a warp of the main kernel reads are a handful of consecutive frames).  With a stream_slot
// table (indexed push), row s * ring + r of x0 is row r of stream stream_slot[s] of mel: x0 stays compact.
__global__ void __launch_bounds__(256) wn_input_kernel(const float* __restrict__ mel, const int32_t* __restrict__ stream_slot,
                                                       int ring, const float* __restrict__ w_kc, const float* __restrict__ b,
                                                       float* __restrict__ x0, int64_t n_rows) {
  __shared__ float ws[kMel * 16];
  __shared__ float bs[16];
  for (int i = threadIdx.x; i < kMel * 16; i += 256) ws[i] = w_kc[i];
  if (threadIdx.x < 16) bs[threadIdx.x] = b[threadIdx.x];
  __syncthreads();
  const int c4 = threadIdx.x & 3;
  for (int64_t row = (int64_t)blockIdx.x * 64 + (threadIdx.x >> 2); row < n_rows; row += (int64_t)gridDim.x * 64) {
    int64_t src = row;
    if (stream_slot) {   // streaming rings: n_rows < 2^31 (wwb_stream_alloc bounds streams x frames)
      const int s = (int)row / ring;
      src = (int64_t)stream_slot[s] * ring + ((int)row - s * ring);
    }
    const float4* m4 = reinterpret_cast<const float4*>(mel + src * kMel);
    float a0 = bs[4 * c4], a1 = bs[4 * c4 + 1], a2 = bs[4 * c4 + 2], a3 = bs[4 * c4 + 3];
#pragma unroll
    for (int k4 = 0; k4 < kMel / 4; ++k4) {
      const float4 m = __ldg(m4 + k4);
      const float mv[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float4 wv = *reinterpret_cast<const float4*>(ws + (4 * k4 + e) * 16 + 4 * c4);
        a0 = fmaf(wv.x, mv[e], a0); a1 = fmaf(wv.y, mv[e], a1); a2 = fmaf(wv.z, mv[e], a2); a3 = fmaf(wv.w, mv[e], a3);
      }
    }
    reinterpret_cast<float4*>(x0)[(int64_t)c4 * n_rows + row] = make_float4(fmaxf(a0, 0.f), fmaxf(a1, 0.f), fmaxf(a2, 0.f), fmaxf(a3, 0.f));   // plane c4
  }
}

// Sliding-window batches share every activation outside the causal-padding cone (header): the tile schedule.
// D(b) = rows of block b's output that depend on the window's zero padding; tile i (first time step 128*i / 3) joins
// at the first block whose dirty prefix reaches it, from the snapshot one level below.
struct WnSharePlan {
  int join[WN_NT], src_slot[WN_NT], snap_slot[24], n_slots;
};
static WnSharePlan wn_share_plan(const int* dil, int L) {
  WnSharePlan g;
  for (int k = 0; k < 24; ++k) g.snap_slot[k] = -1;
  g.n_slots = 0;
  int D[24], acc = 0;
  for (int k = 0; k < 24; ++k) { acc += 2 * dil[k]; D[k] = acc; }
  for (int i = 0; i < WN_NT; ++i) {
    const int tmin = (i * 128) / WN_G;
    int j = 23;
    for (int k = 0; k < 24; ++k)
      if (D[k] > tmin) { j = k; break; }
    if (tmin >= L) j = 23;          // no real rows in this tile: it only has to keep the barrier protocol going
    g.join[i] = j;
    g.src_slot[i] = -1;
    if (j > 0 && tmin < L) {
      if (g.snap_slot[j - 1] < 0) g.snap_slot[j - 1] = g.n_slots++;
      g.src_slot[i] = g.snap_slot[j - 1];
    }
  }
  return g;
}

int wavenet_tc_posteriors(wwb_ctx* ctx, const WinMap& wm, float* enc_out, float* det_out, float* post,
                          cudaStream_t st) {
  if (wm.n_win == 0) return WWB_OK;
  if (ctx->L > WN_MAXT) return fail(ctx, WWB_ERR_ARG, "tensor-core WaveNet path supports windows up to 182 frames");
  const int64_t n_rows = wm.n_streams * (int64_t)wm.ring;
  void* x0;
  int rc = workspace(ctx, 1, (size_t)std::max<int64_t>(n_rows, 1) * 16 * sizeof(float), &x0);
  if (rc) return rc;
  wn_input_kernel<<<(unsigned)std::min<int64_t>((n_rows + 63) / 64, (int64_t)ctx->sm_count * 8), 256, 0, st>>>(
      wm.mel, wm.stream_slot, wm.ring, ctx->wn.in_w, ctx->wn.in_b, (float*)x0, n_rows);
  WWB_CHECK_LAUNCH(ctx);
  WnTcParams P;
  memset(&P, 0, sizeof(P));
  P.x0 = (const float*)x0;
  P.wm = wm;
  P.wblob = ctx->wn.tc_blocks;
  P.head = reinterpret_cast<const WnHead*>(ctx->wn.tc_head);
  P.L = ctx->L;
  P.nsplit = ctx->precision == WWB_PREC_TC ? 3 : 1;
  for (int b = 0; b < 24; ++b) { P.dil[b] = ctx->wn.dilation[b]; P.snap_slot[b] = -1; }
  for (int i = 0; i < WN_NT; ++i) { P.join[i] = 0; P.src_slot[i] = -1; }
  memcpy(P.det1_b, ctx->wn.h_det1_b, sizeof(P.det1_b));
  memcpy(P.det2_w, ctx->wn.h_det2_w, sizeof(P.det2_w));
  memcpy(P.det2_b, ctx->wn.h_det2_b, sizeof(P.det2_b));
  P.n_rows = n_rows;
  P.dbg = reinterpret_cast<long long*>(ctx->debug_buf);
  const size_t smem = sizeof(WnSmem) + 128;
  WWB_CUDA(ctx, cudaFuncSetAttribute(wavenet_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

  // regular grid of >= 8 overlapping windows per stream (not the explicit lists / ring addressing of the streaming
  // path): one stream-level pass writes the snapshots, the window groups then skip the tile-blocks that only hold
  // shared activations
  const char* no_share = getenv("WWB_WN_NO_SHARE");
  const bool share = !wm.win_stream && !wm.n_win_dev && wm.b0 == 0 && wm.win_per_stream >= 8 && wm.hop < ctx->L &&
                     !(no_share && no_share[0] == '1');
  if (share) {
    const WnSharePlan g = wn_share_plan(ctx->wn.dilation, ctx->L);
    if (g.n_slots > 0) {
      void* snap;
      if ((rc = workspace(ctx, 2, (size_t)g.n_slots * n_rows * WN_SNAP_F * sizeof(float), &snap))) return rc;
      WnTcParams S = P;
      S.stream_mode = 1;
      S.rstride = 1;
      S.chunks_per_stream = wm.ring <= WN_ROWS ? 1 : 1 + (wm.ring - WN_ROWS + WN_CHUNK_STEP - 1) / WN_CHUNK_STEP;
      S.snap = (float*)snap;
      for (int b = 0; b < 24; ++b) S.snap_slot[b] = g.snap_slot[b];
      S.enc_out = S.det_out = S.post = nullptr;
#ifndef WWB_HANG_DEBUG
      S.dbg = nullptr;
#endif
      const int64_t n_chunks = wm.n_streams * (int64_t)S.chunks_per_stream;
      wavenet_tc_kernel<<<(unsigned)std::min<int64_t>(n_chunks, ctx->sm_count), WN_THREADS, smem, st>>>(S);
      WWB_CHECK_LAUNCH(ctx);
      P.snap = (float*)snap;
      for (int i = 0; i < WN_NT; ++i) { P.join[i] = g.join[i]; P.src_slot[i] = g.src_slot[i]; }
    }
  }
  P.rstride = WN_G;
  P.enc_out = enc_out; P.det_out = det_out; P.post = post;
  const int64_t n_groups = (wm.n_win + WN_G - 1) / WN_G;
  const unsigned grid = (unsigned)std::min<int64_t>(n_groups, ctx->sm_count);
  wavenet_tc_kernel<<<grid, WN_THREADS, smem, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb
