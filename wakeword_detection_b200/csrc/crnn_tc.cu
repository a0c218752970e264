// K2/K3 — CRNN conv + GRU-1 input projection fused on the tensor cores
// (precision WWB_PREC_TC / TC_FAST).  Replaces CRNN/encode.tflite op 0 (CONV_2D 5x20,
// stride (2,8), SAME, ReLU) and the x-side FULLY_CONNECTED of the two layer-1 WHILE
// bodies (SURVEY.md Appendix A2) for a batch of windows:
//     mel window [L,40]  ->  xw1[b, t, 0:192] = conv_out[b, t, 0:640] . W1^T + b_in,   t < T = ceil(L / 8)
// (fwd gates z|r|h then bwd gates z|r|h), L = 17..256 (CrnnGeom).  The conv output (48.6 KB per window at L = 151)
// never leaves the SM.
//
// One persistent CTA per SM works on tiles of 128 GEMM rows.  For independent windows a tile is floor(128 / (T + 2))
// windows: row r = wl*(T+2) + t (wl = window in the tile, t = conv time step; T of every T + 2 rows are real; 6 x 21
// rows at L = 151) is the M index of every GEMM, so one thread owns one (window, t) pair.  For sliding-window batches
// a tile is a STRIP of 126 consecutive conv steps of one stream (CA_MODE_STRIPS below): every column is computed once
// per stream position instead of once per window that contains it.  Everything between the producers (which frames an element holds) and the projection
// epilogue (where a row's xw goes) is the same code in both modes.
//
//  * The conv is an implicit GEMM per output frequency f: D[128,32] = A_f[128,128] . Wc^T with
//    k = (freq tap kf, time tap kt).  A_f is never materialised: the window is kept in shared
//    memory TRANSPOSED and fp16-split, XP[freq row p][element e] = 8 consecutive time samples
//    (16 bytes), e = wl*(T+2) + chunk: frames 8 chunk - pad_lo .. + 7 of window wl.  Because the
//    conv's time stride is 8 = one element, the operand "row r, k-chunk (kf, j)" is XP[2f+kf][r + j]:
//    linear in r (16 bytes per row) — the tcgen05 shared-memory descriptor reads it in place (SBO = 128, LBO = 16 or, for the chunk
//    pair that straddles two freq taps, row pitch - 32).
//  * XP streams through a ring of three 8-row groups (+ one mirror row so that "next row" is
//    always physically adjacent), filled by four producer warps from the mel windows in global
//    memory (sector-aligned 128-bit loads, register transpose, conflict-free 128-bit stores).
//  * The conv accumulator of frequency f is read by the epilogue warps (bias, ReLU, fp16
//    hi/lo split) and written to shared memory as the k-slice [32f, 32f+32) of the GRU input
//    projection, whose 128x192 accumulator stays in TMEM over the 20 slices; W1 slices
//    (24 KB, pre-packed on the host) stream through a 3-slot cp.async.bulk ring.
//  * Everything is fp16 hi/lo split with three MMAs per product (hi*hi + lo*hi + hi*lo), fp32
//    accumulation in TMEM: fp32-equivalent results (DESIGN.md, precision).
#include <string.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace wwb {

using namespace tc;

// Window geometry (CrnnGeom): T conv steps per window, T + 2 row slots per window and floor(128 / (T + 2)) windows per
// tile of independent windows (6 x 21 for T = 19, 3 x 34 for T = 32).  The kernels are compiled twice: with T = 19
// (L = 145..152, the shipped models) fixed at compile time, and with T read from the parameters for every other length.
constexpr int CA_T_SHIPPED = 19;
constexpr int CA_F = 20;
constexpr int CA_PITCH = 131 * 16;                // bytes per XP row (130 elements used; odd multiple of 16)
constexpr int CA_RING_ROWS = 25;                  // 3 groups of 8 + mirror of physical row 0
constexpr int CA_XP_PLANE = CA_RING_ROWS * CA_PITCH;
constexpr int CA_GROUPS = 7;                      // 8-row groups per tile (padded rows p = freq + 8, 0..55)
constexpr int CA_A1_PLANE = 4 * 128 * 16;         // one k-slice (32 values) of 128 rows
constexpr int CA_W1_SLICE = 2 * 4 * 192 * 16;     // hi + lo planes of one k-slice of W1
constexpr int CA_W1_SLOTS = 3;
constexpr int CA_CR = 3;                          // conv accumulator / A1 slice ring depth
constexpr int CA_CW_PLANE = 16 * 32 * 16;         // conv weights: 16 k-chunks x 32 channels
constexpr int CA_EPI_WARPS = 4, CA_PROD_WARPS = 4;                  // producer warps per set; two sets alternate groups
constexpr int CA_ROLE_WARPS = 3;                  // conv-GEMM issuer, W1 loader, projection-GEMM issuer
constexpr int CA_THREADS = (CA_EPI_WARPS + CA_ROLE_WARPS + 2 * CA_PROD_WARPS) * 32;   // 480

struct CaSmem {
  unsigned char xp[2 * CA_XP_PLANE];
  unsigned char w1[CA_W1_SLOTS][CA_W1_SLICE];
  unsigned char cw[2 * CA_CW_PLANE];
  unsigned char cbias_B[2 * 32 * 16];   // conv bias as the B operand of a 'ones' k-step: row n = (hi, lo, 0, ...); second chunk 0
  unsigned char pbias_B[2 * 192 * 16];  // GRU-1 input bias as the B operand of a 'ones' k-step (row n = (hi, lo, 0, ...))
  uint64_t xp_full[3], xp_empty[3], cacc_full[CA_CR], cacc_empty[CA_CR], a1_full[CA_CR], a1_empty[CA_CR];
  uint64_t w1_full[CA_W1_SLOTS], w1_empty[CA_W1_SLOTS], pacc_full[2], pacc_empty[2];
  uint32_t tmem_base;
};

// Sliding-window batches (regular grid, hop h in {1,2,4,8}) share conv columns between windows: the conv's time stride
// is 8 frames, so column t of window j covers frames h*j + 8t - pad_lo .. + 19 and depends only on the POSITION INDEX
// m = j + q*t (q = 8/h) as long as it does not touch the window's zero padding (at L = 151: t = 1..17).  Those columns
// (and their 192-wide GRU-1 input projection) are computed once per stream and position by tiles that are STRIPS of 126
// consecutive conv steps of one stream and phase (mode 1).  The padded columns of a window (CrnnGeom::padmask: two, three
// or four of them) are strips as well, with the padding moved from the data into the WEIGHTS: padded column t of window j
// is the conv at position m = j + q*t with the time taps that would meet padding frames zeroed (L = 151: column 0 with
// taps 0..5 zeroed, column 18 with taps 13..19).  Each column is the same MMA sequence as in mode 0 with zero products in
// the same places, so the results are bit-identical.  One launch per weight variant writes its own buffer
//   xwS[variant][stream][48 float4 columns][Mp positions]     variant 0: interior, crnn_variant(padmask, t): padded t
// and the layer-1 recurrence reads 128 consecutive positions m = j0 + q*t .. of the variant that step t needs.
enum { CA_MODE_WINDOWS = 0, CA_MODE_STRIPS = 1 };
constexpr int CA_STRIP_ROWS = 126;
// geometry: CrnnShare (common.cuh): q = position indices per conv step (8 / hop), nsp = strips per stream and phase,
// Mp = positions per xwS column row (q * 126 * nsp), F = frames of a stream covered by windows, wps = windows per
// stream, tps = recurrence tiles per stream
using CaShare = CrnnShare;

struct CaParams {
  WinMap wm;
  const unsigned char* cw;      // packed conv weights (2 planes)
  const unsigned char* w1;      // [20][CA_W1_SLICE]
  const float* conv_b;
  const float* b_in;            // [192]
  float* xw1;                   // mode 0: [ceil(n_win/128), T, 48, 128] float4 (see the projection epilogue); mode 1: see CaShare
  int L;
  int T, pad_lo;                // CrnnGeom
  int nsplit;
  int mode;                     // CA_MODE_*
  int64_t n_tiles;              // modes 1/2 (mode 0 derives it from the window count)
  CaShare sh;
  long long* dbg;               // optional issuer timeline of the CTA's second tile: [20 f][8 events]
};

#ifdef WWB_TIMELINE   // NVCC_EXTRA=-DWWB_TIMELINE python -m wakeword_detection_b200.build --force (tools/ca_timeline.py); off by default
#define CA_DBG(f, ev) do { if (P.dbg && blockIdx.x == 0 && tcount == 1 && lane == 0) P.dbg[(f) * 8 + (ev)] = clock64(); } while (0)
#else
#define CA_DBG(f, ev) do { } while (0)
#endif

__device__ __forceinline__ void split8v(const float (&x)[8], uint4& hi, uint4& lo) {
  split_pair(x[0], x[1], hi.x, lo.x);
  split_pair(x[2], x[3], hi.y, lo.y);
  split_pair(x[4], x[5], hi.z, lo.z);
  split_pair(x[6], x[7], hi.w, lo.w);
}

template <int kT>   // kT > 0: T fixed at compile time; 0: T = P.T
__global__ void __launch_bounds__(CA_THREADS, 1) crnn_front_tc_kernel(const CaParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  CaSmem& sm = *reinterpret_cast<CaSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler: role branches are uniform branches
  const int64_t n_win = P.wm.n_win_dev ? (int64_t)*P.wm.n_win_dev : P.wm.n_win;
  const int mode = P.mode;
  const int T = kT > 0 ? kT : P.T;
  const int TP = T + 2, WPT = 128 / TP;             // row slots per window, windows per tile (mode 0)
  const int64_t n_tiles = mode == CA_MODE_WINDOWS ? (n_win + WPT - 1) / WPT : P.n_tiles;

  // ---- one-time setup ----
  for (int i = tid; i < (int)(sizeof(sm.xp) / 16); i += CA_THREADS) reinterpret_cast<uint4*>(sm.xp)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < (int)(sizeof(sm.cw) / 16); i += CA_THREADS)
    reinterpret_cast<uint4*>(sm.cw)[i] = reinterpret_cast<const uint4*>(P.cw)[i];
  if (tid < 64) reinterpret_cast<uint4*>(sm.cbias_B)[tid] = make_uint4(0u, 0u, 0u, 0u);
  for (int i = tid; i < (int)(sizeof(sm.pbias_B) / 16); i += CA_THREADS) reinterpret_cast<uint4*>(sm.pbias_B)[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  if (tid < 32) {
    __half bh, bl;
    split_f16(P.conv_b[tid], bh, bl);
    reinterpret_cast<uint32_t*>(sm.cbias_B + tid * 16)[0] = pack_h2(bh, bl);
  }
  if (tid < 192) {
    __half bh, bl;
    split_f16(P.b_in[tid], bh, bl);
    reinterpret_cast<uint32_t*>(sm.pbias_B + tid * 16)[0] = pack_h2(bh, bl);
  }
  if (tid == 0) {
    for (int i = 0; i < 3; ++i) { mbar_init(&sm.xp_full[i], CA_PROD_WARPS); mbar_init(&sm.xp_empty[i], 1); }
    for (int i = 0; i < CA_CR; ++i) {
      mbar_init(&sm.cacc_full[i], 1); mbar_init(&sm.cacc_empty[i], CA_EPI_WARPS);
      mbar_init(&sm.a1_full[i], CA_EPI_WARPS); mbar_init(&sm.a1_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(&sm.pacc_full[i], 1); mbar_init(&sm.pacc_empty[i], CA_EPI_WARPS); }
    for (int i = 0; i < CA_W1_SLOTS; ++i) { mbar_init(&sm.w1_full[i], 1); mbar_init(&sm.w1_empty[i], 1); }
    mbar_fence_init();
  }
  if (warp == CA_EPI_WARPS) tmem_alloc(&sm.tmem_base, 512);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = sm.tmem_base;
  const uint32_t TM_CACC = 0, TM_ONE = 96, TM_PACC = 128;   // conv acc ring: 3 x 32 cols; constant A chunk (1, 1, 0, ...); projection acc: 2 x 192 cols
  if (warp < 4) {   // one warp per TMEM lane quadrant writes the constant chunk before anybody can issue an MMA
    uint32_t one[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) one[i] = 0u;
    one[0] = 0x3c003c00u;   // (1.0h, 1.0h): the conv bias is added on the tensor core (k-step with this A chunk)
    tmem_st16(tmem + ((uint32_t)(warp * 32) << 16) + TM_ONE, one);
    tmem_st_wait();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();

  if (warp < CA_EPI_WARPS) {
    // =========================== epilogue warps: one row each ===========================
    const int q = warp;
    const int r = q * 32 + lane;
    const int wl = r / TP, t = r - wl * TP;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    uint32_t tcount = 0;

    // Projection epilogue (+ b_in -> xw1), 16 columns at a time.  It is DEFERRED: the accumulator of
    // tile n is drained in 12 pieces during the first 12 conv steps of tile n+1 (the projection
    // accumulator is double-buffered), because its 48 scattered 16-byte stores per row would
    // otherwise stall the conv epilogue — and with it the tensor pipe — for ~10k cycles per tile.
    // xw layout: [tile of 128 windows][t][48 float4 columns][128 windows]: the recurrence kernel
    // (one thread per window) reads it fully coalesced.
    const int64_t cstride = mode == CA_MODE_STRIPS ? P.sh.Mp : 128;   // float4 between two columns of a row's xw
    auto proj_chunk = [&](int64_t pbase, bool pvalid, int pbuf, int c0) {
      float v[16];
      tmem_ld16(tlane + TM_PACC + pbuf * 192 + c0, v);
      tmem_ld_wait();
      if (pvalid) {
        float4* dst = reinterpret_cast<float4*>(P.xw1) + pbase + (c0 / 4) * cstride;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          dst[i * cstride] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);   // b_in was added by the tensor core
      }
    };
    int64_t prev_b = 0;
    bool prev_valid = false, have_prev = false;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      // where this row's 48 float4 of xw go (index of column 0) and whether the row is real
      int64_t b;
      bool valid;
      if (mode == CA_MODE_WINDOWS) {
        const int64_t w = tile * WPT + wl;
        valid = (wl < WPT) && (t < T) && (w < n_win);
        b = (((w >> 7) * T + t) * 48) * 128 + (w & 127);
      } else {
        const int per = P.sh.q * P.sh.nsp;
        const int64_t stream = tile / per;
        const int rem = (int)(tile - stream * per);
        const int k = rem / P.sh.q, phase = rem - k * P.sh.q;
        const int m = phase + P.sh.q * (CA_STRIP_ROWS * k + r);
        valid = r < CA_STRIP_ROWS;
        b = stream * 48 * P.sh.Mp + m;
      }
      for (int f = 0; f < CA_F; ++f) {
        const uint32_t ci = tcount * CA_F + f;
        const int cb = ci % CA_CR;
        const uint32_t cph = (ci / CA_CR) & 1;
        mbar_wait(&sm.cacc_full[cb], cph);
        fence_after_sync();
        float v0[16], v1[16];
        tmem_ld16(tlane + TM_CACC + cb * 32, v0);
        tmem_ld16(tlane + TM_CACC + cb * 32 + 16, v1);
        tmem_ld_wait();
        fence_before_sync();
        uint4 hi[4], lo[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t h[4], l[4];
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            const float a0 = (c < 2) ? v0[c * 8 + 2 * p] : v1[(c - 2) * 8 + 2 * p];
            const float a1 = (c < 2) ? v0[c * 8 + 2 * p + 1] : v1[(c - 2) * 8 + 2 * p + 1];
            split2(pk(fmaxf(a0, 0.f), fmaxf(a1, 0.f)), h[p], l[p]);   // bias already in the accumulator
          }
          hi[c] = make_uint4(h[0], h[1], h[2], h[3]);
          lo[c] = make_uint4(l[0], l[1], l[2], l[3]);
        }
        // the fp16 hi/lo operand of the projection GEMM goes back into the conv accumulator's own 32 TMEM columns
        // (hi: 16 columns = two k-steps, lo: 16 columns): the projection reads A from tensor memory (96 instead of
        // 105 clk per MMA, and no shared-memory round trip of the 128 x 32 slice)
        {
          const uint32_t hr[16] = {hi[0].x, hi[0].y, hi[0].z, hi[0].w, hi[1].x, hi[1].y, hi[1].z, hi[1].w,
                                   hi[2].x, hi[2].y, hi[2].z, hi[2].w, hi[3].x, hi[3].y, hi[3].z, hi[3].w};
          const uint32_t lr[16] = {lo[0].x, lo[0].y, lo[0].z, lo[0].w, lo[1].x, lo[1].y, lo[1].z, lo[1].w,
                                   lo[2].x, lo[2].y, lo[2].z, lo[2].w, lo[3].x, lo[3].y, lo[3].z, lo[3].w};
          tmem_st16(tlane + TM_CACC + cb * 32, hr);
          tmem_st16(tlane + TM_CACC + cb * 32 + 16, lr);
          tmem_st_wait();
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.a1_full[cb]);
        // one piece of the previous tile's projection accumulator
        if (have_prev && f < 12) {
          const uint32_t pt = tcount - 1;
          if (f == 0) {
            mbar_wait(&sm.pacc_full[pt & 1], (pt >> 1) & 1);
            fence_after_sync();
          }
          proj_chunk(prev_b, prev_valid, pt & 1, f * 16);
          if (f == 11) {
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.pacc_empty[pt & 1]);
          }
        }
      }
      prev_b = b; prev_valid = valid; have_prev = true;
    }
    if (have_prev) {   // drain the last tile
      const uint32_t pt = tcount - 1;
      mbar_wait(&sm.pacc_full[pt & 1], (pt >> 1) & 1);
      fence_after_sync();
#pragma unroll 1
      for (int c0 = 0; c0 < 192; c0 += 16) proj_chunk(prev_b, prev_valid, pt & 1, c0);
      fence_before_sync();
    }
  } else if (warp == CA_EPI_WARPS) {
    // =========================== conv-GEMM issuer ===========================
    // All MMAs of one step are issued by ONE elected lane inside a single branch (descriptors are
    // built there with integer adds); per-MMA election costs ~20 extra instructions on this warp,
    // which made the issue rate, not the tensor pipe, the limiter (profiles/r1_crnn_front.md).
    // The projection GEMMs have their own issuing warp: with one warp for both, the ~5 barrier waits per
    // slice (each >= 100 clk even when already complete) plus two blocking issue phases made the issuer
    // the bottleneck at ~2500 clk per slice against 1575 clk of tensor-pipe work (tools/ca_timeline.py).
    const uint32_t idesc_c = make_idesc_f16(128, 32);
    const uint32_t uXP = smem_u32(sm.xp), uCW = smem_u32(sm.cw);
    const int nsplit = P.nsplit;
    uint32_t tcount = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      const uint32_t gbase = tcount * CA_GROUPS;
      int groups_ready = 0;
      for (int f = 0; f < CA_F; ++f) {
        const uint32_t ci = tcount * CA_F + f;
        const int cb = ci % CA_CR;
        // conv accumulator ci % 3 was last used by slice ci-3 and then held that slice's projection operand:
        // free once the projection GEMM of ci-3 has completed (a1_empty)
        if (ci >= (uint32_t)CA_CR) mbar_wait(&sm.a1_empty[cb], (((ci - CA_CR) / CA_CR) & 1));
        const int g_hi = (2 * f + 12) >> 3;
        CA_DBG(f, 0);
        for (; groups_ready <= g_hi; ++groups_ready) {
          const uint32_t gg = gbase + groups_ready;
          mbar_wait(&sm.xp_full[gg % 3], (gg / 3) & 1);
        }
        CA_DBG(f, 1);
        fence_after_sync();
        uint32_t rowaddr[5];
#pragma unroll
        for (int kf = 0; kf < 5; ++kf) {
          const int rowp = 2 * f + 7 + kf;
          rowaddr[kf] = uXP + (((gbase + (rowp >> 3)) % 3) * 8 + (rowp & 7)) * CA_PITCH;
        }
        CA_DBG(f, 2);
        if (elect_one()) {
          const uint32_t cacc = tmem + TM_CACC + cb * 32;
          const uint64_t dbase = make_desc(uCW, 512, 128);
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const int q0 = 2 * m, kf0 = q0 / 3, j0 = q0 % 3;
            const uint32_t lbo = (j0 == 2 && m != 7) ? (uint32_t)(CA_PITCH - 32) : 16u;
            const uint64_t dah = make_desc(rowaddr[kf0] + j0 * 16, lbo, 128), dal = dah + (uint64_t)(CA_XP_PLANE >> 4);
            const uint64_t dbh = dbase + (uint64_t)((q0 * 512) >> 4), dbl = dbh + (uint64_t)(CA_CW_PLANE >> 4);
            mma_f16_ss(cacc, dah, dbh, idesc_c, m != 0);
            if (nsplit == 3) {
              mma_f16_ss(cacc, dal, dbh, idesc_c, true);
              mma_f16_ss(cacc, dah, dbl, idesc_c, true);
            }
          }
          mma_f16_ts(cacc, tmem + TM_ONE, make_desc(smem_u32(sm.cbias_B), 512, 128), idesc_c, true);   // + conv bias
          mma_commit(&sm.cacc_full[cb]);
          // group f/4 was last read by conv(f) when f = 4*(f/4)
          if ((f & 3) == 0) mma_commit(&sm.xp_empty[(gbase + (f >> 2)) % 3]);
          if (f == CA_F - 1) { mma_commit(&sm.xp_empty[(gbase + 5) % 3]); mma_commit(&sm.xp_empty[(gbase + 6) % 3]); }
        }
        __syncwarp();
        CA_DBG(f, 3);
      }
    }
  } else if (warp == CA_EPI_WARPS + 2) {
    // =========================== projection-GEMM issuer ===========================
    // slice f of the GRU-1 input projection: pacc[128,192] += A1_f[128,32] . W1_f^T as soon as the epilogue warps have
    // turned conv accumulator f into the fp16 hi/lo operand and the W1 slice has landed
    const uint32_t idesc_p = make_idesc_f16(128, 192);
    const int nsplit = P.nsplit;
    uint32_t tcount = 0, w1cnt = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      const int pb = tcount & 1;
      const uint32_t pacc = tmem + TM_PACC + pb * 192;
      mbar_wait(&sm.pacc_empty[pb], ((tcount >> 1) & 1) ^ 1);
      for (int f = 0; f < CA_F; ++f, ++w1cnt) {
        const uint32_t ci = tcount * CA_F + f;
        const int cb = ci % CA_CR;
        const int sl = w1cnt % CA_W1_SLOTS;
        CA_DBG(f, 4);
        mbar_wait(&sm.a1_full[cb], (ci / CA_CR) & 1);
        CA_DBG(f, 5);
        mbar_wait(&sm.w1_full[sl], (w1cnt / CA_W1_SLOTS) & 1);
        CA_DBG(f, 6);
        fence_after_sync();
        if (elect_one()) {
          const uint32_t ta = tmem + TM_CACC + cb * 32;   // hi k-steps at +0 / +8, lo at +16 / +24
          const uint64_t db = make_desc(smem_u32(sm.w1[sl]), 3072, 128);
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint64_t dbh = db + (uint64_t)(kk * (6144 >> 4)), dbl = dbh + (uint64_t)((CA_W1_SLICE / 2) >> 4);
            mma_f16_ts(pacc, ta + kk * 8, dbh, idesc_p, (f | kk) != 0);
            if (nsplit == 3) {
              mma_f16_ts(pacc, ta + 16 + kk * 8, dbh, idesc_p, true);
              mma_f16_ts(pacc, ta + kk * 8, dbl, idesc_p, true);
            }
          }
          mma_commit(&sm.a1_empty[cb]);
          mma_commit(&sm.w1_empty[sl]);
          if (f == CA_F - 1) {
            mma_f16_ts(pacc, tmem + TM_ONE, make_desc(smem_u32(sm.pbias_B), 192 * 16, 128), idesc_p, true);   // + b_in
            mma_commit(&sm.pacc_full[pb]);
          }
        }
        __syncwarp();
        CA_DBG(f, 7);
      }
    }
  } else if (warp == CA_EPI_WARPS + 1) {
    // =========================== W1 slice loader ===========================
    if (lane == 0) {
      uint32_t cnt = 0;
      for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
        for (int f = 0; f < CA_F; ++f, ++cnt) {
          const int sl = cnt % CA_W1_SLOTS;
          mbar_wait(&sm.w1_empty[sl], ((cnt / CA_W1_SLOTS) & 1) ^ 1);
          mbar_arrive_expect_tx(&sm.w1_full[sl], CA_W1_SLICE);
          bulk_g2s(sm.w1[sl], P.w1 + (size_t)f * CA_W1_SLICE, CA_W1_SLICE, &sm.w1_full[sl]);
        }
    }
  } else {
    // =========================== XP producers ===========================
    const int pset = (warp - (CA_EPI_WARPS + CA_ROLE_WARPS)) / CA_PROD_WARPS;       // this set fills the groups with gg % 2 == pset
    const int task = tid - (CA_EPI_WARPS + CA_ROLE_WARPS + pset * CA_PROD_WARPS) * 32;   // 0..127; element e = task
    const bool has_task = mode == CA_MODE_WINDOWS ? task < WPT * TP : true;
    uint32_t gg = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      // element `task` of the tile = 8 consecutive frames f0 .. f0+7 (relative to `start` of stream s), valid in [0, fhi)
      int64_t s = 0;
      int start = 0, f0, fhi;
      bool live;
      if (mode == CA_MODE_WINDOWS) {
        const int wl = task / TP, c = task - wl * TP;   // window in tile, time chunk (frames 8c - pad_lo .. + 7)
        const int64_t b = tile * WPT + wl;
        live = has_task && b < n_win;
        if (live) win_origin(P.wm, b, s, start);
        f0 = 8 * c - P.pad_lo;
        fhi = P.L;
      } else {
        const int per = P.sh.q * P.sh.nsp;
        s = tile / per;
        const int rem = (int)(tile - s * per);
        const int k = rem / P.sh.q, phase = rem - k * P.sh.q;
        live = true;
        f0 = (8 / P.sh.q) * phase + 8 * (CA_STRIP_ROWS * k + task) - P.pad_lo;
        fhi = P.sh.F;
      }
      for (int g = 0; g < CA_GROUPS; ++g, ++gg) {
        if ((int)(gg & 1) != pset) continue;
        const int slot = gg % 3;
        // issue the loads before waiting for the slot
        float4 v[8][2];
        const bool data = live && g >= 1 && g <= 5;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int frame = f0 + i;
          if (data && frame >= 0 && frame < fhi) {
            const float4* src = reinterpret_cast<const float4*>(stream_row(P.wm, s, start + frame) + 8 * (g - 1));
            v[i][0] = __ldg(src);
            v[i][1] = __ldg(src + 1);
          } else {
            v[i][0] = make_float4(0.f, 0.f, 0.f, 0.f);
            v[i][1] = v[i][0];
          }
        }
        mbar_wait(&sm.xp_empty[slot], ((gg / 3) & 1) ^ 1);
        if (has_task) {
          unsigned char* base = sm.xp + (slot * 8) * CA_PITCH + task * 16;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float x[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 s = v[i][k >> 2];
              x[i] = (k & 3) == 0 ? s.x : (k & 3) == 1 ? s.y : (k & 3) == 2 ? s.z : s.w;
            }
            uint4 hi, lo;
            split8v(x, hi, lo);
            *reinterpret_cast<uint4*>(base + k * CA_PITCH) = hi;
            *reinterpret_cast<uint4*>(base + k * CA_PITCH + CA_XP_PLANE) = lo;
            if (slot == 0 && k == 0) {   // mirror of physical row 0 after the last ring row
              *reinterpret_cast<uint4*>(sm.xp + 24 * CA_PITCH + task * 16) = hi;
              *reinterpret_cast<uint4*>(sm.xp + 24 * CA_PITCH + task * 16 + CA_XP_PLANE) = lo;
            }
          }
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.xp_full[slot]);
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == CA_EPI_WARPS) tmem_dealloc(tmem, 512);
}

// ---- host side ------------------------------------------------------------------------------
static void put_split16(std::vector<unsigned char>& buf, size_t hi_off, size_t lo_off, float x) {
  __half h = __float2half_rn(x);
  __half l = __float2half_rn(x - __half2float(h));
  memcpy(&buf[hi_off], &h, 2);
  memcpy(&buf[lo_off], &l, 2);
}

// conv_w [32][5][20] -> 1 + popc(padmask) variants x [plane][16 chunks][32 channels][8 halves]; chunk q = kf*3 + j holds
// time taps 8j..8j+7.  Variant 0: all taps; variant crnn_variant(padmask, t) of a padded column t: the taps kt whose
// window frame 8t - pad_lo + kt lies outside 0..L-1 zeroed (L = 151: variant 1 = column 0 with taps 0..5 zeroed,
// variant 2 = column 18 with taps 13..19 zeroed)
std::vector<unsigned char> crnn_pack_conv(const float* conv_w, int L) {
  const CrnnGeom geo = crnn_geom(L);
  const int n_var = 1 + __builtin_popcount(geo.padmask);
  std::vector<unsigned char> out((size_t)n_var * 2 * CA_CW_PLANE, 0);
  for (int v = 0; v < n_var; ++v) {
    int col = -1;   // the padded column of variant v (none for variant 0)
    for (int t = 0; t < geo.T; ++t)
      if (v && crnn_variant(geo.padmask, t) == v) col = t;
    for (int q = 0; q < 15; ++q)
      for (int n = 0; n < 32; ++n)
        for (int e = 0; e < 8; ++e) {
          const int kf = q / 3, kt = (q % 3) * 8 + e, frame = 8 * col - geo.pad_lo + kt;
          if (kt >= 20 || (col >= 0 && (frame < 0 || frame >= L))) continue;
          const size_t off = (size_t)v * 2 * CA_CW_PLANE + ((size_t)q * 32 + n) * 16 + e * 2;
          put_split16(out, off, off + CA_CW_PLANE, conv_w[(n * 5 + kf) * 20 + kt]);
        }
  }
  return out;
}

// W1 [192][640] (row = fwd gates then bwd gates) -> 20 slices [plane][4 chunks][192][8 halves]
std::vector<unsigned char> crnn_pack_w1(const float* w_nk) {
  std::vector<unsigned char> out((size_t)20 * CA_W1_SLICE, 0);
  for (int f = 0; f < 20; ++f)
    for (int c = 0; c < 4; ++c)
      for (int n = 0; n < 192; ++n)
        for (int e = 0; e < 8; ++e) {
          const size_t off = (size_t)f * CA_W1_SLICE + ((size_t)c * 192 + n) * 16 + e * 2;
          put_split16(out, off, off + CA_W1_SLICE / 2, w_nk[(size_t)n * 640 + f * 32 + c * 8 + e]);
        }
  return out;
}

// the front-kernel launches of the shared-column path: one per conv-weight variant in use (variant 0 is not when every
// column is padded, L = 17, 18)
int crnn_share_first_variant(const CrnnShare& g) { return g.padmask + 1 == (1ull << g.T) ? 1 : 0; }
int crnn_share_launches(const CrnnShare& g) { return 1 + __builtin_popcount(g.padmask) - crnn_share_first_variant(g); }

// geometry of the shared-column path for a regular window grid; false if the grid does not qualify
bool crnn_share_plan(const WinMap& wm, int L, CrnnShare* out) {
  if (wm.win_stream || wm.n_win_dev || wm.b0 != 0 || wm.win_per_stream < 2) return false;
  const int hop = wm.hop;
  if (hop != 1 && hop != 2 && hop != 4 && hop != 8) return false;
  const int wps = wm.win_per_stream;
  if (wm.n_win % wps) return false;
  if ((int64_t)(wps - 1) * hop + L > wm.ring) return false;   // a window would wrap around the ring
  const CrnnGeom geo = crnn_geom(L);
  CrnnShare g;
  g.q = 8 / hop;
  g.wps = wps;
  g.tps = (wps + 127) / 128;
  g.F = (wps - 1) * hop + L;
  g.T = geo.T;
  g.padmask = geo.padmask;
  const int m_max = wps - 1 + (geo.T - 1) * g.q;   // column T - 1 of the last window
  g.nsp = (m_max / g.q + 1 + CA_STRIP_ROWS - 1) / CA_STRIP_ROWS;
  g.Mp = g.q * CA_STRIP_ROWS * g.nsp;
  g.n_streams = wm.n_win / wps;
  // worth it only if it is fewer tiles than the per-window tiles (128 / (T + 2) windows each)
  const int64_t tiles_shared = crnn_share_launches(g) * g.n_streams * g.q * g.nsp;
  if (tiles_shared >= (wm.n_win + 128 / (geo.T + 2) - 1) / (128 / (geo.T + 2))) return false;
  *out = g;
  return true;
}
// one variant's buffer (+ slack: the recurrence reads 128 positions from j0 + q*t even where fewer windows are left)
size_t crnn_share_xws_bytes(const CrnnShare& g, int64_t n_streams) { return ((size_t)n_streams * 48 * g.Mp + 256) * 16; }

int crnn_front_tc(wwb_ctx* ctx, const WinMap& wm, float* xw1, cudaStream_t st, int mode, const CrnnShare* g, int variant) {
  if (wm.n_win == 0) return WWB_OK;
  CaParams P;
  memset(&P, 0, sizeof(P));
  const CrnnGeom geo = crnn_geom(ctx->L);
  P.mode = mode;
  P.T = geo.T;
  P.pad_lo = geo.pad_lo;
  const int wpt = 128 / (geo.T + 2);
  int64_t n_tiles = (wm.n_win + wpt - 1) / wpt;
  if (mode != CA_MODE_WINDOWS) {
    P.sh = *g;
    n_tiles = (wm.n_win / g->wps) * g->q * g->nsp;
  }
  P.n_tiles = n_tiles;
  P.wm = wm;
  P.cw = ctx->crnn.tc_conv + (size_t)variant * 2 * CA_CW_PLANE;
  P.w1 = ctx->crnn.tc_w1;
  P.conv_b = ctx->crnn.conv_b;
  P.b_in = ctx->crnn.tc_bi[0];
  P.xw1 = xw1;
  P.L = ctx->L;
  P.nsplit = ctx->precision == WWB_PREC_TC ? 3 : 1;
  P.dbg = reinterpret_cast<long long*>(ctx->debug_buf);
  const size_t smem = sizeof(CaSmem) + 128;
  auto kernel = geo.T == CA_T_SHIPPED ? crnn_front_tc_kernel<CA_T_SHIPPED> : crnn_front_tc_kernel<0>;
  WWB_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)std::min<int64_t>(n_tiles, ctx->sm_count);
  kernel<<<grid, CA_THREADS, smem, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb

// ---------------------------------------------------------------------------------------------
// K3 (recurrence) — one bidirectional GRU layer (Keras v2, reset_after, gates z|r|h; the four
// WHILE bodies of CRNN/encode.tflite, SURVEY.md Appendix A2) for 128 windows per CTA with the
// windows on the M axis of the tensor core:
//     per step   D_dir[128, 96] = h_dir[128, 32] . U_dir^T          (tcgen05, fp16 hi/lo split)
//                z = sig(xz + hz), r = sig(xr + hr), c = tanh(xh + r*(hh + b_h)), h = c + z*(h - c)
// xw (the input projection incl. b_in and the z/r parts of the recurrent bias) comes from global
// memory, one 384-byte row per (window, t, dir).  Warps 0-3 run the forward direction (t = s),
// warps 4-7 the backward one (t = T - 1 - s); each thread owns one window: its h[32] stays in
// registers, the fp16-split copy in shared memory is the A operand of the next step.
namespace wwb {

using namespace tc;

constexpr int GR_H_BYTES = 2 * 4 * 128 * 16;     // hi + lo planes, K = 32
constexpr int GR_U_BYTES = 2 * 4 * 96 * 16;
constexpr int GR_EPI_WARPS = 16;                 // 2 directions x 4 lane quadrants x 2 unit halves: TWO threads per (window, direction),
                                                 // units 0-15 and 16-31 (a warp reaches the tensor-memory lanes 32 (warp % 4) ..., so warps w and
                                                 // w + 8 share a quadrant): 96 instead of 168 registers per thread, four epilogue warps per
                                                 // scheduler instead of two.  Measured neutral (CRNN stage 2.70 -> 2.68 ms per 512 x 10 s): the
                                                 // recurrences are not bound by per-warp latency but by the operand traffic of a step
                                                 // (layer 1: 96 KB of xw slabs per CTA and step from L2 = 3.2 TB/s over the launch; layer 2: 2 GB of
                                                 // layer-1 output read back from HBM per 512 x 10 s)
constexpr int GR_THREADS = (GR_EPI_WARPS + 2) * 32;   // + the MMA issuer warp + the operand loader warp = 576

constexpr int G2_A_BYTES = 2 * 8 * 128 * 16;       // layer-1 output of 128 windows at one step as a packed fp16 hi/lo operand (K = 64): 32 KB
constexpr int GR_X_BYTES = 24 * 128 * 16;          // one direction's xw of one step: 24 float4 columns x 128 windows (contiguous in HBM)
constexpr int GR_XST = 2;                          // xw stages PER DIRECTION (a stage never changes its consumer warps)
constexpr int GR_TW = 120;                         // windows per tile in position-ring mode: 120 rows + 4 look-ahead rows for each of the (at most)
                                                   // two streams a tile touches fill the 128 rows of a stage buffer

// h (the A operand of the recurrent GEMM) lives in TENSOR MEMORY, fp16 hi (16 columns) + lo (16 columns) per
// direction; that frees the shared memory for a TMA-filled ring of xw slabs (2 steps x 2 directions x 48 KB).
struct GrSmem {
  unsigned char x[2][GR_XST][GR_X_BYTES];          // [direction][stage]
  unsigned char u[2][GR_U_BYTES];
  float bh[2][32];
  uint64_t acc_full[2], h_ready[2];
  uint64_t x_full[2][GR_XST], x_empty[2][GR_XST];
  uint32_t tmem_base;
};

struct GrParams {
  const float* xw;              // [ceil(B/128), T, 48, 128] float4
  const float* xws;             // shared-column mode (else null): [variant][stream][48][Mp] float4 by position (CrnnShare)
  size_t xws_variant;           // bytes between two variants
  int q, Mp, wps;               // shared-column geometry (CrnnShare)
  uint32_t padmask;             // padded columns: step t reads variant crnn_variant(padmask, t)
  int ring;                     // position-ring mode (see the kernel)
  int T;                        // steps (conv columns per window)
  const unsigned char* u;       // [2][GR_U_BYTES] packed
  const float* bh;              // [2][32]  recurrent bias of the candidate gate
  float* seq_out;               // [B, T, 64] or null
  unsigned char* seq_packed;    // or null: the layer's output sequence as the fp16 hi/lo A operand of the next layer's input
                                // projection, [ceil(B/128)][T][plane hi, lo][8 chunks][128 windows][8 halves] (gru2_fused_tc_kernel)
  float* last_out;              // [B, 64] or null
  int64_t n_win;
  const int32_t* n_win_dev;
  int nsplit;
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcpf(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// GRU gates of TWO units with 8 SFU operations instead of 12 (the recurrence kernels are bound by the SFU: 4 lanes per
// clock and scheduler): one reciprocal serves a pair of denominators, 1/d0 = d1 * rcp(d0 d1).  z and r of a unit share
// one, the candidates of the two units the other.  The exponents are clamped at 60 (2^120 stays finite in the
// products; sigmoid is 9e-19 and tanh 1 to 2e-18 there).  az / ar = pre-activations of z / r, hb = U_h h + b_h, xh = the
// candidate's input part; h is updated in place: h' = z h + (1 - z) c.
__device__ __forceinline__ void gru_gates2(float az0, float ar0, float hb0, float xh0, float az1, float ar1, float hb1, float xh1,
                                           float& h0, float& h1) {
  const float L2E = 1.4426950408889634f;
  const float dz0 = 1.f + ex2f(fminf(-L2E * az0, 60.f)), dr0 = 1.f + ex2f(fminf(-L2E * ar0, 60.f));
  const float dz1 = 1.f + ex2f(fminf(-L2E * az1, 60.f)), dr1 = 1.f + ex2f(fminf(-L2E * ar1, 60.f));
  const float p0 = rcpf(dz0 * dr0), p1 = rcpf(dz1 * dr1);
  const float z0 = dr0 * p0, r0 = dz0 * p0, z1 = dr1 * p1, r1 = dz1 * p1;
  const float dc0 = 1.f + ex2f(fminf(2.f * L2E * fmaf(r0, hb0, xh0), 60.f));
  const float dc1 = 1.f + ex2f(fminf(2.f * L2E * fmaf(r1, hb1, xh1), 60.f));
  const float pc = rcpf(dc0 * dc1);
  const float c0 = fmaf(-2.f, dc1 * pc, 1.f), c1 = fmaf(-2.f, dc0 * pc, 1.f);   // tanh(v) = 1 - 2 / (1 + e^(2v))
  h0 = fmaf(z0, h0 - c0, c0);
  h1 = fmaf(z1, h1 - c1, c1);
}

__device__ __forceinline__ void tmem_ld8f(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ldN(uint32_t taddr, float (&v)[8]) { tmem_ld8f(taddr, v); }
__device__ __forceinline__ void tmem_ldN(uint32_t taddr, float (&v)[16]) { tmem_ld16(taddr, v); }
// per-thread asynchronous 16-byte copy global -> shared (LDGSTS), and an mbarrier arrival that fires when all of the thread's
// earlier cp.async have landed (it first adds itself to the pending count of the barrier's current phase)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// (A polling wait that keeps calling load_next() so that slab requests go out earlier was measured: 2.53 -> 2.56 ms with the
// position ring, 2.68 -> 2.74 without - the suspending wait stays.)
// (busy-polling issuer: 2.127 vs 2.129 ms - no difference once the loader has its own warp)
#define GR_ISS_WAIT(bar, par) mbar_wait(bar, par)

template <int kT>   // kT > 0: T fixed at compile time; 0: T = P.T
__global__ void __launch_bounds__(GR_THREADS, 1) gru_rec_tc_kernel(const GrParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  GrSmem& sm = *reinterpret_cast<GrSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler: role branches are uniform branches
  const int64_t n_win = P.n_win_dev ? (int64_t)*P.n_win_dev : P.n_win;
  const bool shared = P.xws != nullptr;
  // POSITION RING (shared-column mode, streams of >= GR_TW windows).  At step t window j needs column t of its stream = position
  // m = j + q t of the interior variant: consecutive steps of a tile read position windows that are shifted by q = 8 / hop
  // (4 at hop 2), so 124 of 128 positions of a step's slab are the previous step's.  Reloading whole slabs was 3.1 GB of
  // L2 -> SM traffic per launch (probe: the same kernel without the reloads 2.19 instead of 2.68 ms CRNN stage; with the
  // ring 2.53 - the three whole-slab loads a tile still needs have one step of lead time each).  In ring mode
  // the interior steps t = 1..T-2 of a tile and direction share ONE stage buffer as a ring over positions: 128 positions are
  // loaded once, each later step adds q (row = position modulo the ring size; a tile that touches two streams keeps one
  // ring per stream: n_A + 4 and n_B + 4 rows of the buffer's 128, hence tiles of 120 windows).  The padded columns
  // t = 0 / T-1 come from their own variants and use the direction's other buffer, loaded while the ring steps run; the two
  // buffers swap roles from tile to tile so that every large load has a step of lead time.  The barrier protocol is
  // unchanged: load n may be issued once step n - 2 of the direction has been consumed.  The host sets P.ring only if the
  // padded columns are exactly t = 0 and T - 1: lengths with a third or fourth padded column (L = 1, 2, 3 mod 8) read
  // whole slabs per step instead, since a padded step 1 or T - 2 would need a third buffer role.
  const bool ring = P.ring != 0;
  const int TW = ring ? GR_TW : 128;
  const int T = kT > 0 ? kT : P.T;
  const int64_t n_tiles = (n_win + TW - 1) / TW;

  for (int i = tid; i < (int)(2 * GR_U_BYTES / 16); i += GR_THREADS)
    reinterpret_cast<uint4*>(&sm.u[0][0])[i] = reinterpret_cast<const uint4*>(P.u)[i];
  if (tid < 64) (&sm.bh[0][0])[tid] = P.bh[tid];
  if (tid == 0) {
    for (int d = 0; d < 2; ++d) {
      mbar_init(&sm.acc_full[d], 1); mbar_init(&sm.h_ready[d], 8);
      for (int i = 0; i < GR_XST; ++i) { mbar_init(&sm.x_full[d][i], 1); mbar_init(&sm.x_empty[d][i], 8); }
    }
    mbar_fence_init();
  }
  if (warp == GR_EPI_WARPS) tmem_alloc(&sm.tmem_base, 256);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = sm.tmem_base;

  if (warp < GR_EPI_WARPS) {
    const int d = (warp >> 2) & 1, q = warp & 3, half = warp >> 3;
    const int r = q * 32 + lane;
    const int ub = half * 16;                         // this thread's units: ub .. ub + 15
    const uint32_t tbase = tmem + ((uint32_t)(q * 32) << 16) + d * 96 + ub;
    const uint32_t th = tmem + ((uint32_t)(q * 32) << 16) + 192 + d * 32 + half * 8;   // this row's h: hi 16 columns, lo 16 columns (2 units per column)
    const float* bh = sm.bh[d] + ub;
    uint32_t n_acc = 0, n_x = 0, n_tl = 0;   // n_tl: tiles this CTA has started (its parity says which buffer holds the padded-column slabs)
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++n_tl) {
      const int64_t b = tile * TW + r;
      const bool valid = r < TW && b < n_win;
      // ring mode: this row's ring (base row, size) and its current row in it
      int rbase = 0, rsize = 128, ridx = 0;   // (rows past the tile's windows just stay inside the buffer)
      if (ring) {
        const int64_t b0 = tile * TW;
        const int nrows = (int)(n_win - b0 < TW ? n_win - b0 : TW);
        const int j0 = (int)(b0 % P.wps);
        const int nA = nrows < P.wps - j0 ? nrows : P.wps - j0;
        if (r < nA) { rbase = 0; rsize = nA + 4; ridx = r; }
        else if (r < nrows) { rbase = nA + 4; rsize = nrows - nA + 4; ridx = r - nA; }
      }
      float h[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) h[i] = 0.f;
      for (int s = 0; s < T; ++s, ++n_x) {
        const int t = d ? T - 1 - s : s;
        // this direction's xw slab of the step was fetched by the TMA engine one step ahead (per-thread loads could
        // prefetch only one 400-clock chunk ahead of ~1500 clocks of DRAM latency)
        const int xs = n_x % GR_XST;
        mbar_wait(&sm.x_full[d][xs], (n_x / GR_XST) & 1);
        const bool vstep = s == 0 || s == T - 1;
        const int xbuf = ring ? (int)((n_tl & 1) ^ (vstep ? 0u : 1u)) : xs;
        const int xrow = ring && !vstep ? rbase + ridx : r;
        const float4* xp = reinterpret_cast<const float4*>(sm.x[d][xbuf]) + xrow + (ub / 4) * 128;
        float x_last = 0.f;
        if (s > 0) {
          mbar_wait(&sm.acc_full[d], n_acc & 1);
          ++n_acc;
          fence_after_sync();
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {                 // two pieces of 8 units
          float4 xc[3][2];
#pragma unroll
          for (int g = 0; g < 3; ++g)
#pragma unroll
            for (int i = 0; i < 2; ++i) xc[g][i] = xp[(g * 8 + u * 2 + i) * 128];
          if (u == 1) x_last = xc[2][1].w;
          float hz[8], hr[8], hh[8];
          if (s > 0) {
            tmem_ld8f(tbase + u * 8, hz);
            tmem_ld8f(tbase + 32 + u * 8, hr);
            tmem_ld8f(tbase + 64 + u * 8, hh);
            tmem_ld_wait();
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) { hz[i] = 0.f; hr[i] = 0.f; hh[i] = 0.f; }
          }
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const float4 vz = xc[0][i >> 2], vr = xc[1][i >> 2], vh = xc[2][i >> 2];
            const bool lo = (i & 3) == 0;
            gru_gates2((lo ? vz.x : vz.z) + hz[i], (lo ? vr.x : vr.z) + hr[i], hh[i] + bh[u * 8 + i], lo ? vh.x : vh.z,
                       (lo ? vz.y : vz.w) + hz[i + 1], (lo ? vr.y : vr.w) + hr[i + 1], hh[i + 1] + bh[u * 8 + i + 1], lo ? vh.y : vh.w,
                       h[u * 8 + i], h[u * 8 + i + 1]);
          }
        }
        // hand the stage back once every lane's loads from it have completed (the arrive depends on the last loaded
        // value of all lanes through a warp reduction)
        {
          uint32_t tok;
          asm volatile("mov.b32 %0, %1;" : "=r"(tok) : "f"(x_last));
          tok = __reduce_or_sync(0xffffffffu, tok);
          if (lane == 0) mbar_arrive_after(&sm.x_empty[d][xs], tok);
        }
        if (ring && !vstep) {   // the next interior step reads q positions further (forward) / back (backward direction)
          ridx += d ? -4 : 4;
          if (ridx >= rsize) ridx -= rsize;
          if (ridx < 0) ridx += rsize;
        }
        uint32_t hr8[8], lr8[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) split_pair(h[2 * c], h[2 * c + 1], hr8[c], lr8[c]);
        if (s < T - 1) {
          fence_before_sync();
          tmem_st8(th, hr8);
          tmem_st8(th + 16, lr8);
          tmem_st_wait();
          fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.h_ready[d]);
        }
        if (valid && P.seq_out) {
          float4* dst = reinterpret_cast<float4*>(P.seq_out + (b * T + t) * 64 + d * 32 + ub);
#pragma unroll
          for (int i = 0; i < 4; ++i) dst[i] = make_float4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
        }
        if (valid && P.seq_packed) {   // the split computed for the recurrent GEMM is the next layer's A operand: 512 contiguous bytes per warp store
          unsigned char* dst = P.seq_packed + ((size_t)((b >> 7) * T + t) * G2_A_BYTES) + (size_t)((d * 4 + half * 2) * 128 + (int)(b & 127)) * 16;
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            *reinterpret_cast<uint4*>(dst + u * 2048) = make_uint4(hr8[4 * u], hr8[4 * u + 1], hr8[4 * u + 2], hr8[4 * u + 3]);
            *reinterpret_cast<uint4*>(dst + G2_A_BYTES / 2 + u * 2048) = make_uint4(lr8[4 * u], lr8[4 * u + 1], lr8[4 * u + 2], lr8[4 * u + 3]);
          }
        }
      }
      if (valid && P.last_out) {
        float4* dst = reinterpret_cast<float4*>(P.last_out + b * 64 + d * 32 + ub);
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[i] = make_float4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
      }
    }
  } else if (warp == GR_EPI_WARPS + 1) {
    // xw loader: its own warp - as part of the issuing warp the address arithmetic and the copies of a slab request sat
    // between an h_ready arrival and the step's GEMM issue
    uint32_t n_ld[2] = {0, 0};          // slabs requested per direction
    int64_t ld_tile[2] = {blockIdx.x, blockIdx.x};
    int ld_s[2] = {0, 0};
    uint32_t ld_tl[2] = {0, 0};         // tiles whose loads have been started, per direction
    auto load_next = [&](const int dd) {   // requests direction dd's next slab if its stage is free (never blocks)
      if (ld_tile[dd] >= n_tiles) return;
      const int xs = n_ld[dd] % GR_XST;
      if (n_ld[dd] >= (uint32_t)GR_XST) {
        uint32_t ok = 0;   // one lane probes, the result is broadcast (a per-lane probe could split the warp)
        if (lane == 0) ok = mbar_test_wait(&sm.x_empty[dd][xs], ((n_ld[dd] / GR_XST) & 1) ^ 1) ? 1u : 0u;
        if (!__shfl_sync(0xffffffffu, ok, 0)) return;
      }
      const int t = dd ? T - 1 - ld_s[dd] : ld_s[dd];
      if (ring) {
        const int s = ld_s[dd];
        const bool vstep = s == 0 || s == T - 1;
        unsigned char* const buf = sm.x[dd][(ld_tl[dd] & 1) ^ (vstep ? 0u : 1u)];
        const int64_t b0 = ld_tile[dd] * TW;
        const int nrows = (int)(n_win - b0 < TW ? n_win - b0 : TW);
        const int64_t stream0 = b0 / P.wps;
        const int j0 = (int)(b0 - stream0 * P.wps);
        const int nA = nrows < P.wps - j0 ? nrows : P.wps - j0;
        const int nseg = nrows > nA ? 2 : 1;
        const unsigned char* base = reinterpret_cast<const unsigned char*>(P.xws) + crnn_variant(P.padmask, t) * P.xws_variant;
        const bool full = vstep || s == 1;   // a whole slab: the padded column of the step, or the ring's first 128 positions
        if (full) {
          if (lane == 0) mbar_arrive_expect_tx(&sm.x_full[dd][xs], (uint32_t)nrows * 24 * 16);
          __syncwarp();
          if (lane < 24) {
            for (int sg = 0; sg < nseg; ++sg) {
              const int n = sg ? nrows - nA : nA;                 // windows of this stream in the tile
              const int j = sg ? 0 : j0;                          // the first one's index in its stream
              const int rb = vstep ? (sg ? nA : 0) : (sg ? nA + 4 : 0);   // first buffer row of the segment (ring: of its ring)
              bulk_g2s(buf + ((size_t)lane * 128 + rb) * 16, base + (((size_t)(stream0 + sg) * 48 + dd * 24 + lane) * P.Mp + j + 4 * t) * 16,
                       (uint32_t)n * 16, &sm.x_full[dd][xs]);
            }
          }
        } else {
          // Interior step i = s - 1 >= 1: the 4 positions that enter each stream's window, 24 columns each = 96 float4 per
          // stream, as per-thread 16-byte cp.async (3 per lane and stream) - NOT as bulk copies: the kernel was bound by
          // the NUMBER of bulk-copy requests (~100 per step at ~90 clk each), not by their bytes.  Virtual index
          // v = n + 4 (i - 1) + k (forward) or v = -4 i + k (backward), k = 0..3, holds position (first position of the
          // ring's step 0) + v and lives in row v mod (n + 4).  Each lane's cp.async.mbarrier.arrive adds itself to the
          // phase's pending count and arrives when the lane's copies have landed; lane 0's plain arrival closes the phase.
          for (int sg = 0; sg < nseg; ++sg) {
            const int n = sg ? nrows - nA : nA;
            const int j = sg ? 0 : j0;
            const int rb = sg ? nA + 4 : 0;
            const int i = s - 1, R = n + 4;
            const int v0 = dd ? -4 * i : n + 4 * (i - 1);
            const int row0 = ((v0 % R) + R) % R;
            const int p0 = j + 4 * t + (dd ? 0 : n - 4);          // forward: the last 4 positions of the step's window; backward: its first 4
#pragma unroll
            for (int e3 = 0; e3 < 3; ++e3) {
              const int e = lane + 32 * e3, col = e >> 2, k = e & 3;
              int row = row0 + k;
              if (row >= R) row -= R;
              cp_async16(buf + ((size_t)col * 128 + rb + row) * 16, base + (((size_t)(stream0 + sg) * 48 + dd * 24 + col) * P.Mp + p0 + k) * 16);
            }
          }
          cp_async_mbar_arrive(&sm.x_full[dd][xs]);
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.x_full[dd][xs]);
        }
      } else if (shared) {
        // the tile's windows b0.. are dense over (stream, j): at step t they sit at consecutive positions m = j + q*t of
        // their stream, so a slab is one run of positions per stream the tile touches, times 24 column rows; the padded
        // columns come from their own variants of the strip computation
        const int64_t b0 = ld_tile[dd] * 128;
        const int nrows = (int)(n_win - b0 < 128 ? n_win - b0 : 128);
        if (lane == 0) mbar_arrive_expect_tx(&sm.x_full[dd][xs], (uint32_t)nrows * 24 * 16);
        __syncwarp();
        int64_t stream = b0 / P.wps;
        int j = (int)(b0 - stream * P.wps);
        const unsigned char* base = reinterpret_cast<const unsigned char*>(P.xws) + crnn_variant(P.padmask, t) * P.xws_variant;
        for (int row = 0; row < nrows; ++stream, j = 0) {
          const int n = nrows - row < P.wps - j ? nrows - row : P.wps - j;
          if (lane < 24)
            bulk_g2s(sm.x[dd][xs] + (lane * 128 + row) * 16, base + (((size_t)stream * 48 + dd * 24 + lane) * P.Mp + j + P.q * t) * 16,
                     (uint32_t)n * 16, &sm.x_full[dd][xs]);
          row += n;
        }
      } else if (lane == 0) {
        mbar_arrive_expect_tx(&sm.x_full[dd][xs], GR_X_BYTES);
        bulk_g2s(sm.x[dd][xs], reinterpret_cast<const unsigned char*>(P.xw) + ((size_t)(ld_tile[dd] * T + t) * 48 + dd * 24) * 128 * 16,
                 GR_X_BYTES, &sm.x_full[dd][xs]);
      }
      ++n_ld[dd];
      if (++ld_s[dd] == T) { ld_s[dd] = 0; ld_tile[dd] += gridDim.x; ++ld_tl[dd]; }
    };
    while (ld_tile[0] < n_tiles || ld_tile[1] < n_tiles) {
      const uint32_t before = n_ld[0] + n_ld[1];
      load_next(0);
      load_next(1);
      if (n_ld[0] + n_ld[1] == before) __nanosleep(64);
    }
  } else {
    // MMA issuer
    const uint32_t idesc = make_idesc_f16(128, 96);
    const int nsplit = P.nsplit;
    uint32_t n_h = 0;
    const uint64_t db0 = make_desc(smem_u32(sm.u[0]), 1536, 128), db1 = make_desc(smem_u32(sm.u[1]), 1536, 128);
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int s = 1; s < T; ++s, ++n_h) {
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          GR_ISS_WAIT(&sm.h_ready[d], n_h & 1);
          fence_after_sync();
          if (elect_one()) {
            const uint32_t acc = tmem + d * 96, ta = tmem + 192 + d * 32;
            const uint64_t db = d ? db1 : db0;
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              const uint64_t dbh = db + (uint64_t)((kk * 3072) >> 4), dbl = dbh + (uint64_t)((GR_U_BYTES / 2) >> 4);
              mma_f16_ts(acc, ta + kk * 8, dbh, idesc, kk != 0);
              if (nsplit == 3) {
                mma_f16_ts(acc, ta + 16 + kk * 8, dbh, idesc, true);
                mma_f16_ts(acc, ta + kk * 8, dbl, idesc, true);
              }
            }
            mma_commit(&sm.acc_full[d]);
          }
          __syncwarp();
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == GR_EPI_WARPS) tmem_dealloc(tmem, 256);
}

// U [96][32] (gate-major rows z|r|h) -> [plane][4 chunks][96][8 halves]
std::vector<unsigned char> crnn_pack_u(const float* u_f, const float* u_b) {
  std::vector<unsigned char> out(2 * GR_U_BYTES, 0);
  for (int d = 0; d < 2; ++d) {
    const float* u = d ? u_b : u_f;
    for (int c = 0; c < 4; ++c)
      for (int n = 0; n < 96; ++n)
        for (int e = 0; e < 8; ++e) {
          const size_t off = (size_t)d * GR_U_BYTES + ((size_t)c * 96 + n) * 16 + e * 2;
          put_split16(out, off, off + GR_U_BYTES / 2, u[n * 32 + c * 8 + e]);
        }
  }
  return out;
}

int gru_rec_tc(wwb_ctx* ctx, int layer, const float* xw, float* seq_out, float* last_out, int64_t B,
               const int32_t* n_dev, cudaStream_t st, const float* xws, const CrnnShare* g, unsigned char* seq_packed) {
  if (B == 0) return WWB_OK;
  GrParams P;
  memset(&P, 0, sizeof(P));
  P.xw = xw;
  const int T = crnn_geom(ctx->L).T;
  P.T = T;
  int64_t n_tiles = (B + 127) / 128;
  if (xws) {
    P.xws = xws;
    P.q = g->q; P.Mp = g->Mp; P.wps = g->wps;
    P.padmask = g->padmask;
    P.xws_variant = crnn_share_xws_bytes(*g, B / g->wps);
    P.ring = g->wps >= GR_TW && g->q == 4 && g->padmask == (1u | 1u << (T - 1));
    if (P.ring) n_tiles = (B + GR_TW - 1) / GR_TW;   // position-ring mode (see the kernel)
  }
  P.u = ctx->crnn.tc_u[layer];
  P.bh = ctx->crnn.tc_bh[layer];
  P.seq_out = seq_out;
  P.seq_packed = seq_packed;
  P.last_out = last_out;
  P.n_win = B;
  P.n_win_dev = n_dev;
  P.nsplit = ctx->precision == WWB_PREC_TC ? 3 : 1;
  const size_t smem = sizeof(GrSmem) + 128;
  auto kernel = T == CA_T_SHIPPED ? gru_rec_tc_kernel<CA_T_SHIPPED> : gru_rec_tc_kernel<0>;
  WWB_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)std::min<int64_t>(n_tiles, (int64_t)ctx->sm_count);
  kernel<<<grid, GR_THREADS, smem, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

// ---------------------------------------------------------------------------------------------
// K3 (layer 2, fused) - GRU-2 input projection + recurrence in one kernel.  Layer 1 leaves its output sequence in HBM
// as a packed fp16 hi/lo operand (32 KB per 128 windows and step); here it is the A operand of
//     acc_dir[128, 0:96]  = seq1[t][128, 64] . W2_dir^T + b_in      columns  xh | z | r      (issued ahead of h)
//     acc_dir[128, 32:96] += h_dir[128, 32] . U_zr^T                                  z | r
//     acc_dir[128, 96:128] = h_dir[128, 32] . U_h^T                                   hh
// so the 14.6 KB/window xw2 tensor is never written to or read from HBM (it was 3.2 GB each way per bench step) and the
// separate projection GEMM kernel is gone.  z and r leave the tensor core already summed (x part + h part); only the
// candidate gate needs its two parts separately.  The slab of step s+1 streams in (cp.async.bulk) while step s runs.
constexpr int G2_W_BYTES = 2 * 8 * 96 * 16;        // per direction: hi + lo planes, K = 64, N = 96
constexpr int G2_BIAS_BYTES = 2 * 96 * 16;         // B operand of the 'ones' k-step
constexpr int G2_AST = 2;                          // A slab stages per direction

struct G2Smem {
  unsigned char a[2][G2_AST][G2_A_BYTES];
  unsigned char w[2][G2_W_BYTES];
  unsigned char u[2][GR_U_BYTES];
  unsigned char bias_B[2][G2_BIAS_BYTES];
  float bh[2][32];
  uint64_t acc_full[2], acc_free[2], h_ready[2];
  uint64_t a_full[2][G2_AST], a_empty[2][G2_AST];
  uint32_t tmem_base;
};

struct G2Params {
  const unsigned char* seq;     // packed layer-1 output (GrParams::seq_packed)
  const unsigned char* w2;      // [2][G2_W_BYTES]
  const unsigned char* u;       // [2][GR_U_BYTES]
  const float* b_in;            // [2][96] in accumulator column order xh | z | r
  const float* bh;              // [2][32]
  float* last_out;              // [B, 64]
  int64_t n_win;
  const int32_t* n_win_dev;
  int nsplit;
  int T;                        // steps
};

template <int kT>   // kT > 0: T fixed at compile time; 0: T = P.T
__global__ void __launch_bounds__(GR_THREADS, 1) gru2_fused_tc_kernel(const G2Params P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  G2Smem& sm = *reinterpret_cast<G2Smem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int64_t n_win = P.n_win_dev ? (int64_t)*P.n_win_dev : P.n_win;
  const int64_t n_tiles = (n_win + 127) / 128;
  const int T = kT > 0 ? kT : P.T;

  for (int i = tid; i < (int)(2 * G2_W_BYTES / 16); i += GR_THREADS)
    reinterpret_cast<uint4*>(&sm.w[0][0])[i] = reinterpret_cast<const uint4*>(P.w2)[i];
  for (int i = tid; i < (int)(2 * GR_U_BYTES / 16); i += GR_THREADS)
    reinterpret_cast<uint4*>(&sm.u[0][0])[i] = reinterpret_cast<const uint4*>(P.u)[i];
  for (int i = tid; i < (int)(2 * G2_BIAS_BYTES / 16); i += GR_THREADS) reinterpret_cast<uint4*>(&sm.bias_B[0][0])[i] = make_uint4(0u, 0u, 0u, 0u);
  if (tid < 64) (&sm.bh[0][0])[tid] = P.bh[tid];
  __syncthreads();
  if (tid < 192) {   // row n of direction d = (hi, lo, 0, ...); the second chunk stays 0
    __half bhi, blo;
    split_f16(P.b_in[tid], bhi, blo);
    reinterpret_cast<uint32_t*>(&sm.bias_B[tid / 96][(tid % 96) * 16])[0] = pack_h2(bhi, blo);
  }
  if (tid == 0) {
    for (int d = 0; d < 2; ++d) {
      mbar_init(&sm.acc_full[d], 1); mbar_init(&sm.acc_free[d], 8); mbar_init(&sm.h_ready[d], 8);
      for (int i = 0; i < G2_AST; ++i) { mbar_init(&sm.a_full[d][i], 1); mbar_init(&sm.a_empty[d][i], 1); }
    }
    mbar_fence_init();
  }
  if (warp == GR_EPI_WARPS) tmem_alloc(&sm.tmem_base, 512);
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = sm.tmem_base;
  const uint32_t TM_H = 256, TM_ONE = 320;   // accumulators: direction d at columns d*128; h operand: 256 + d*32; constant chunk (1, 1, 0, ...)
  if (warp < 4) {
    uint32_t one[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) one[i] = 0u;
    one[0] = 0x3c003c00u;
    tmem_st16(tmem + ((uint32_t)(warp * 32) << 16) + TM_ONE, one);
    tmem_st_wait();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();

  if (warp < GR_EPI_WARPS) {
    const int d = (warp >> 2) & 1, q = warp & 3, half = warp >> 3;
    const int r = q * 32 + lane;
    const int ub = half * 16;                         // this thread's units: ub .. ub + 15
    const uint32_t tbase = tmem + ((uint32_t)(q * 32) << 16) + d * 128 + ub;
    const uint32_t th = tmem + ((uint32_t)(q * 32) << 16) + TM_H + d * 32 + half * 8;
    const float* bh = sm.bh[d] + ub;
    uint32_t n_acc = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int64_t b = tile * 128 + r;
      const bool valid = b < n_win;
      float h[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) h[i] = 0.f;
      for (int s = 0; s < T; ++s, ++n_acc) {
        mbar_wait(&sm.acc_full[d], n_acc & 1);
        fence_after_sync();
#pragma unroll
        for (int u = 0; u < 2; ++u) {                 // two pieces of 8 units
          float xh[8], az[8], ar[8], hh[8];
          tmem_ld8f(tbase + u * 8, xh);
          tmem_ld8f(tbase + 32 + u * 8, az);
          tmem_ld8f(tbase + 64 + u * 8, ar);
          if (s > 0) {
            tmem_ld8f(tbase + 96 + u * 8, hh);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) hh[i] = 0.f;
          }
          tmem_ld_wait();
          if (u == 1) {   // the accumulator has been read: the next step's input projection may overwrite it
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.acc_free[d]);
          }
#pragma unroll
          for (int i = 0; i < 8; i += 2)
            gru_gates2(az[i], ar[i], hh[i] + bh[u * 8 + i], xh[i], az[i + 1], ar[i + 1], hh[i + 1] + bh[u * 8 + i + 1], xh[i + 1],
                       h[u * 8 + i], h[u * 8 + i + 1]);
        }
        if (s < T - 1) {
          uint32_t hr8[8], lr8[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) split_pair(h[2 * c], h[2 * c + 1], hr8[c], lr8[c]);
          fence_before_sync();
          tmem_st8(th, hr8);
          tmem_st8(th + 16, lr8);
          tmem_st_wait();
          fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.h_ready[d]);
        }
      }
      if (valid) {
        float4* dst = reinterpret_cast<float4*>(P.last_out + b * 64 + d * 32 + ub);
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[i] = make_float4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
      }
    }
  } else if (warp == GR_EPI_WARPS + 1) {
    // slab loader (its own warp, like in gru_rec_tc_kernel)
    uint32_t n_ld[2] = {0, 0};
    int64_t ld_tile[2] = {blockIdx.x, blockIdx.x};
    int ld_s[2] = {0, 0};
    auto load_next = [&](const int dd) {   // requests direction dd's next slab if its stage is free (never blocks)
      if (ld_tile[dd] >= n_tiles) return;
      const int xs = n_ld[dd] % G2_AST;
      if (n_ld[dd] >= (uint32_t)G2_AST) {
        uint32_t ok = 0;
        if (lane == 0) ok = mbar_test_wait(&sm.a_empty[dd][xs], ((n_ld[dd] / G2_AST) & 1) ^ 1) ? 1u : 0u;
        if (!__shfl_sync(0xffffffffu, ok, 0)) return;
      }
      const int t = dd ? T - 1 - ld_s[dd] : ld_s[dd];
      if (lane == 0) {
        mbar_arrive_expect_tx(&sm.a_full[dd][xs], G2_A_BYTES);
        bulk_g2s(sm.a[dd][xs], P.seq + (size_t)(ld_tile[dd] * T + t) * G2_A_BYTES, G2_A_BYTES, &sm.a_full[dd][xs]);
      }
      ++n_ld[dd];
      if (++ld_s[dd] == T) { ld_s[dd] = 0; ld_tile[dd] += gridDim.x; }
    };
    while (ld_tile[0] < n_tiles || ld_tile[1] < n_tiles) {
      const uint32_t before = n_ld[0] + n_ld[1];
      load_next(0);
      load_next(1);
      if (n_ld[0] + n_ld[1] == before) __nanosleep(64);
    }
  } else {
    // MMA issuer
    const uint32_t idesc_x = make_idesc_f16(128, 96), idesc_zr = make_idesc_f16(128, 64), idesc_h = make_idesc_f16(128, 32);
    const int nsplit = P.nsplit;
    uint32_t n_step = 0, n_h = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int s = 0; s < T; ++s, ++n_step) {
        // input projections of this step (do not depend on h): as soon as the slab is in and the accumulator has been read
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const int xs = n_step % G2_AST;
          mbar_wait(&sm.a_full[d][xs], (n_step / G2_AST) & 1);
          if (n_step > 0) GR_ISS_WAIT(&sm.acc_free[d], (n_step - 1) & 1);
          fence_after_sync();
          if (elect_one()) {
            const uint32_t acc = tmem + d * 128;
            const uint64_t da = make_desc(smem_u32(sm.a[d][xs]), 2048, 128), db = make_desc(smem_u32(sm.w[d]), 1536, 128);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              const uint64_t dah = da + (uint64_t)((kk * 4096) >> 4), dal = dah + (uint64_t)((G2_A_BYTES / 2) >> 4);
              const uint64_t dbh = db + (uint64_t)((kk * 3072) >> 4), dbl = dbh + (uint64_t)((G2_W_BYTES / 2) >> 4);
              mma_f16_ss(acc, dah, dbh, idesc_x, kk != 0);
              if (nsplit == 3) {
                mma_f16_ss(acc, dal, dbh, idesc_x, true);
                mma_f16_ss(acc, dah, dbl, idesc_x, true);
              }
            }
            mma_f16_ts(acc, tmem + TM_ONE, make_desc(smem_u32(sm.bias_B[d]), 1536, 128), idesc_x, true);   // + b_in
            mma_commit(&sm.a_empty[d][xs]);
            if (s == 0) mma_commit(&sm.acc_full[d]);   // h = 0: no recurrent part
          }
          __syncwarp();
        }
        if (s == 0) continue;
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          GR_ISS_WAIT(&sm.h_ready[d], n_h & 1);
          fence_after_sync();
          if (elect_one()) {
            const uint32_t acc = tmem + d * 128, ta = tmem + TM_H + d * 32;
            const uint64_t db = make_desc(smem_u32(sm.u[d]), 1536, 128);
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              const uint64_t dbh = db + (uint64_t)((kk * 3072) >> 4), dbl = dbh + (uint64_t)((GR_U_BYTES / 2) >> 4);
              const uint64_t hoff = (uint64_t)((64 * 16) >> 4);   // U rows 64..95: candidate gate
              mma_f16_ts(acc + 32, ta + kk * 8, dbh, idesc_zr, true);
              mma_f16_ts(acc + 96, ta + kk * 8, dbh + hoff, idesc_h, kk != 0);
              if (nsplit == 3) {
                mma_f16_ts(acc + 32, ta + 16 + kk * 8, dbh, idesc_zr, true);
                mma_f16_ts(acc + 32, ta + kk * 8, dbl, idesc_zr, true);
                mma_f16_ts(acc + 96, ta + 16 + kk * 8, dbh + hoff, idesc_h, true);
                mma_f16_ts(acc + 96, ta + kk * 8, dbl + hoff, idesc_h, true);
              }
            }
            mma_commit(&sm.acc_full[d]);
          }
          __syncwarp();
        }
        ++n_h;
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == GR_EPI_WARPS) tmem_dealloc(tmem, 512);
}

// W2 [192][64] (row = fwd gates z|r|h then bwd gates z|r|h) -> per direction [plane][8 chunks][96 rows xh|z|r][8 halves]
std::vector<unsigned char> crnn_pack_w2(const float* w_nk) {
  std::vector<unsigned char> out(2 * G2_W_BYTES, 0);
  for (int d = 0; d < 2; ++d)
    for (int c = 0; c < 8; ++c)
      for (int n = 0; n < 96; ++n) {
        const int src_row = d * 96 + (n < 32 ? 64 + n : n - 32);
        for (int e = 0; e < 8; ++e) {
          const size_t off = (size_t)d * G2_W_BYTES + ((size_t)c * 96 + n) * 16 + e * 2;
          put_split16(out, off, off + G2_W_BYTES / 2, w_nk[(size_t)src_row * 64 + c * 8 + e]);
        }
      }
  return out;
}
// input bias [2][96] (z|r|h, recurrent z/r bias folded in) -> accumulator column order xh|z|r
std::vector<float> crnn_reorder_bias2(const float* bf) {
  std::vector<float> out(192);
  for (int d = 0; d < 2; ++d)
    for (int n = 0; n < 96; ++n) out[d * 96 + n] = bf[d * 96 + (n < 32 ? 64 + n : n - 32)];
  return out;
}
size_t crnn_seq_packed_bytes(int64_t B, int T) { return (size_t)((B + 127) / 128) * T * G2_A_BYTES; }

int gru2_fused_tc(wwb_ctx* ctx, const unsigned char* seq_packed, float* last_out, int64_t B, const int32_t* n_dev,
                  cudaStream_t st) {
  if (B == 0) return WWB_OK;
  G2Params P;
  memset(&P, 0, sizeof(P));
  P.seq = seq_packed;
  P.w2 = ctx->crnn.tc_w2;
  P.u = ctx->crnn.tc_u[1];
  P.b_in = ctx->crnn.tc_bi2;
  P.bh = ctx->crnn.tc_bh[1];
  P.last_out = last_out;
  P.n_win = B;
  P.n_win_dev = n_dev;
  P.nsplit = ctx->precision == WWB_PREC_TC ? 3 : 1;
  P.T = crnn_geom(ctx->L).T;
  const size_t smem = sizeof(G2Smem) + 128;
  auto kernel = P.T == CA_T_SHIPPED ? gru2_fused_tc_kernel<CA_T_SHIPPED> : gru2_fused_tc_kernel<0>;
  WWB_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t n_tiles = (B + 127) / 128;
  const unsigned grid = (unsigned)std::min<int64_t>(n_tiles, (int64_t)ctx->sm_count);
  kernel<<<grid, GR_THREADS, smem, st>>>(P);
  WWB_CHECK_LAUNCH(ctx);
  return WWB_OK;
}

}  // namespace wwb
