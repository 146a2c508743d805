// flow_t4.cu -- forward / grid flow kernel with FOUR 128-rotation tiles in flight per SM (tcgen05 + TMEM), sm_100a.
//
// flow_row.cu keeps two tiles per SM: its activations go to the tensor core through 32 KB of shared memory per tile and
// fc_last needs 256 TMEM columns per tile.  ncu on that kernel: issue slots 58 % active, tensor pipe 29 %, the
// rest is exposed latency of the dependent GEMM round trips (15 % of the samples sit in the mbarrier wait) -- two tiles are not
// enough independent work.  This kernel makes a tile small enough for four:
//   * the A operand (ReLU'd activations, fp16 hi / lo planes) lives in TENSOR MEMORY: tcgen05.mma in its TS form reads row r
//     from lane r, K elements (2c, 2c+1) packed in column c.  A thread writes its own row with tcgen05.st -- no shared-memory
//     staging, no swizzle arithmetic, no proxy fence per GEMM.  64 columns per tile.
//   * fc_last is issued as four N = 64 chunks (16 mixture components each) into ONE 64-column accumulator that is drained into
//     registers before the next chunk is issued.  64 columns per tile; 4 x (64 + 64) = the 512 columns of an SM.
//   * fc_first (K = 3, flow/condition.py:25) and the residual  relu_last(x0 + x3)  (flow/condition.py:29) run on the tensor
//     core as well: every GEMM starts with one K = 16 MMA of a per-rotation block  Y = (1, 1, y_hi, y_lo, y_hi, 1, 1, 0, 0, 0)
//     against a per-layer block (b_hi, b_lo, W0_hi, W0_hi, W0_lo, b0_hi, b0_lo, ...) (engine._bias_block), which yields the
//     bias, W0.y (error-compensated) and, in the last hidden layer, x0 again -- no stash of x0, no FMA loop on the CUDA cores.
//     The per-image term  c = W_f.feature  (hoisted, rnf_flow_condition) enters through one more K = 16 MMA against a per-tile
//     block (c_hi, c_lo) in grid mode (a tile never straddles images); in row mode it is added in the epilogue.
// One WORKER thread owns one rotation (512 threads = 4 tiles x 128 rows): nothing is computed twice, nothing is exchanged.
//
// Warp specialisation (round 2): a fifth warpgroup holds one SERVICE warp per tile that does nothing but wait for the tile's
// hand-over (an mbarrier the four worker warps arrive on), issue the tile's MMAs and refill weight pieces; the workers watch the
// MMA mbarrier of a dependent GEMM themselves.  Before, one of the tile's own worker warps issued: tcgen05.mma issue blocks at the pace
// of the tensor pipe (13 MMAs = ~450 cycles per GEMM, eight GEMMs per layer), so that warp ran ~30 % behind its three siblings
// and every hand-over of the tile waited for it.  Registers: 640 threads launch with 96 each (the CTA's pool); the service warpgroup
// drops to 32 (setmaxnreg.dec) and the four worker warpgroups take 112 (setmaxnreg.inc): 512 x 112 + 128 x 32 = 640 x 96.
// The bisection of Flow.inverse needs its 256 prepared parameters resident per row and stays in flow_row.cu.
#include <cstdlib>

#include "mobius_pair.cuh"
#include "tc_common.cuh"
#include "ablation_layers.cuh"

namespace rnf {
namespace {

#ifndef RNF_TC_TRACE
#define RNF_TC_TRACE 0
#endif
#if RNF_TC_TRACE
#define TRACE(i) do { if (tr_on) tr[(i)] = clock64(); } while (0)
#else
#define TRACE(i) do { } while (0)
#endif

constexpr int kTiles = 4;            // tiles in flight per SM (TMEM: 4 x 128 columns)
constexpr int kWorkers = kTiles * 128;
constexpr int kThreads = kWorkers + kTiles * 32;   // + one service warp per tile (warpgroup 4)
constexpr int kRows = 128;
constexpr int kWorkerRegs = 112, kServiceRegs = 32;   // setmaxnreg targets of the worker / service warpgroups
// setmaxnreg moves registers inside the pool the CTA was LAUNCHED with (640 threads x 96, the largest multiple of 8 that fits the file)
static_assert(kWorkers * kWorkerRegs + kTiles * 32 * kServiceRegs <= kThreads * 96, "register pool of the CTA");
// Workers wait for a chain GEMM by polling its mbarrier with this suspend-time hint (ns).
constexpr int kDirectWaitNs = 2000;
// Variants that measured slower or equal (DESIGN.md section 8b, svc-x: half-epilogue hand-over, named-barrier wake-up of the
// workers, suspend hints / naps in the service warps, the convert-back fp16 split) were removed; their code is in commit d73682a.

// shared memory (bytes from a 1024-aligned base)
constexpr int kOffW = 0;                                  // W1 | W2 | W3 pieces
constexpr int kOffLastW = kHidW;                          // W4 piece
constexpr int kOffAux = kOffLastW + kLastW;               // aux piece, double buffered on the layer parity
constexpr int kOffY = kOffAux + 2 * kAuxStride;           // [tile] Y block [128 x 16] fp16, no swizzle (4 KB)
constexpr int kOffC = kOffY + kTiles * 4096;              // [tile] per-image block [64 x 16] fp16, no swizzle (2 KB)
constexpr int kOffRed = kOffC + kTiles * 2048;            // [tile] reduction scratch
constexpr int kOffBar = kOffRed + kTiles * 128;
constexpr int kOffMisc = kOffBar + 8 * 24;
constexpr int kSmemBytes = kOffMisc + 64 + 64 * 8;
constexpr int kSmemAlloc = kSmemBytes + 1024;
static_assert(kOffLastW % 1024 == 0 && kW1Bytes % 1024 == 0, "UMMA SW128 tiles need 1024 B alignment");
static_assert(kOffY % 16 == 0 && kOffC % 16 == 0 && kOffAux % 16 == 0, "no-swizzle blocks need 16 B alignment");

// READY: hand-overs of a tile's workers to its service warp.  Between two phases of it the workers always wait for a GEMM, i.e. for
// the service warp to have consumed the earlier phase, so a parity wait can never be lapped.  Nothing reads the READY2 barriers
// (they served the removed half-epilogue hand-over); they stay initialised because dropping them changes the kernel's code.
enum { BAR_W_FULL = 0 /* W1,W2,W3,W4 */, BAR_AUX_FULL = 4 /* [2] */, BAR_MMA = 6 /* [tile] */, BAR_READY = 6 + kTiles /* [tile] */,
       BAR_READY2 = 6 + 2 * kTiles /* [tile] */, BAR_COUNT = 6 + 3 * kTiles };
static_assert(BAR_COUNT <= 24, "mbarrier slots");

// TMEM columns of a tile
constexpr uint32_t kColAhi = 0, kColAlo = 32, kColD = 64, kColsPerTile = 128;

// D (+)= A[tmem] . B[smem desc]^T : TS form of tcgen05.mma (A: lane = row, 16-bit K elements packed two per column)
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo32, uint32_t desc_hi32, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 db;\n"
      "setp.ne.b32 p, %5, 0;\n"
      "mov.b64 db, {%2, %3};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b_lo32), "r"(desc_hi32), "r"(idesc), "r"(accumulate)
      : "memory");
}

// 3-product split GEMM on top of an initialised accumulator: D += Alo.Whi + Ahi.Wlo + Ahi.Whi   (K = 64 in four K = 16 steps;
// a step is 8 TMEM columns on the A side, 32 B = +2 descriptor units on the B side)
__device__ __forceinline__ void issue_split_ts(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, uint32_t idesc) {
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_f16_ts(d, a_lo + 8 * k, b_hi + 2 * k, kDescHi, idesc, 1);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_f16_ts(d, a_hi + 8 * k, b_lo + 2 * k, kDescHi, idesc, 1);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_f16_ts(d, a_hi + 8 * k, b_hi + 2 * k, kDescHi, idesc, 1);
}

// ... the K steps k0, k0 + 1 of the three products.  The service warp issues a chain GEMM as two of these in separate elect blocks:
// its first MMA then leaves sooner after the hand-over than from one block of all 13 (DESIGN.md section 8b, svc-x).
__device__ __forceinline__ void issue_split_ts_half(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, uint32_t idesc, int k0) {
#pragma unroll
  for (int k = k0; k < k0 + 2; ++k) umma_f16_ts(d, a_lo + 8 * k, b_hi + 2 * k, kDescHi, idesc, 1);
#pragma unroll
  for (int k = k0; k < k0 + 2; ++k) umma_f16_ts(d, a_hi + 8 * k, b_lo + 2 * k, kDescHi, idesc, 1);
#pragma unroll
  for (int k = k0; k < k0 + 2; ++k) umma_f16_ts(d, a_hi + 8 * k, b_hi + 2 * k, kDescHi, idesc, 1);
}

__device__ __forceinline__ uint32_t pack_h2(__half lo, __half hi) {
  const __half2 h = __halves2half2(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// mbarrier wait whose try_wait carries a suspend-time hint: the thread sleeps in hardware until the phase completes or the hint
// expires, instead of re-issuing the try_wait / branch pair every ~100 cycles
template <int NS>
__device__ __forceinline__ void mbar_wait_hint(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"((uint32_t)NS)
        : "memory");
  } while (!ok);
}

// ReLU + error-compensated fp16 split of two activations with the residual taken packed.
// (The mixed-precision FHFMA form of the residual, fma.rn.f32.f16, issues one instruction less but runs at a quarter of the
// FMA rate: tools/cvt_rate.cu.)
__device__ __forceinline__ void relu_split_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  // The fp16 truncation of x, back in fp32, is x with its low 13 mantissa bits cleared: two LOP3 on the (half idle) ALU pipe
  // instead of two HADD2.F32 on the FMA pipe, which is the busiest pipe of this kernel (tools/pipe_rate.cu: every one of these
  // instructions costs 2 cycles per warp on its pipe).  hi is that masked value converted exactly (cvt.rn without satfinite),
  // so hi + lo = x to 22 bits for 0.125 <= x < 65536 and to 2^-25 absolute below; x >= 65536 gives hi = +Inf, which the next
  // GEMM turns into Inf / NaN rows instead of a silently clipped activation (tests/test_weight_scales.py).  Negative x:
  // hi = 0 (relu) and x - (x & mask) <= 0 -> lo = 0.
  const float m0 = __uint_as_float(__float_as_uint(x0) & 0xFFFFE000u), m1 = __uint_as_float(__float_as_uint(x1) & 0xFFFFE000u);
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(m1), "f"(m0));
  float d0, d1;
  upk(sub2(pk(x0, x1), pk(m0, m1)), d0, d1);
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(d1), "f"(d0));
}

// Epilogue of one GEMM: my row of the accumulator -> (+ c) -> ReLU -> fp16 hi / lo -> A operand in TMEM (K element 2e in the
// low half of column e).  All four 16-column loads are in flight before the first wait; the whole A operand is handed over at once.
template <typename HandOver>
__device__ __forceinline__ void epilogue64(uint32_t tm, const float* cadd, HandOver&& hand_over) {
  float a0[16], a1[16], a2[16], a3[16];
  tmem_ld16_async(tm + kColD, a0);
  tmem_ld16_async(tm + kColD + 16, a1);
  tmem_ld16_async(tm + kColD + 32, a2);
  tmem_ld16_async(tm + kColD + 48, a3);
  tmem_ld_wait16(a0); tmem_ld_wait16(a1); tmem_ld_wait16(a2); tmem_ld_wait16(a3);
  float* q[4] = {a0, a1, a2, a3};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      float* acc = q[2 * h + g];
      if (cadd != nullptr) {
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 c = __ldg(reinterpret_cast<const float4*>(cadd + 32 * h + 16 * g) + j4);
          acc[4 * j4] += c.x; acc[4 * j4 + 1] += c.y; acc[4 * j4 + 2] += c.z; acc[4 * j4 + 3] += c.w;
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) relu_split_pair(acc[2 * e], acc[2 * e + 1], hi[8 * g + e], lo[8 * g + e]);
    }
    tmem_st16_nowait(tm + kColAhi + 16 * h, hi);
    tmem_st16_nowait(tm + kColAlo + 16 * h, lo);
  }
  tmem_st_wait();
  hand_over();
}

template <int N>
__device__ __forceinline__ void set_max_regs_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void set_max_regs_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

struct TileSched {            // which tiles / layer steps a tile slot of this CTA processes (same arithmetic in workers and service warp)
  int n_active;
  int my_items;               // < 2^31 / layers: a CTA's share of at most 2^31 tiles
  int total_steps;
};

// ------------------------------------------------ service warp of one tile --------------------------------------------------
// Mirrors the control flow of the tile's workers: per Mobius layer five hand-overs that end in a GEMM the workers WAIT for
// (fc_first, three hidden layers, fc_last chunk 0) and three whose GEMM runs under the workers' arithmetic (chunks 1..3).
template <bool GRID>
__device__ __forceinline__ void service_warp(const FlowArgs& a, uint8_t* smem, const uint32_t tmem_base, const int tile, const int lane,
                                             const TileSched sc, const int n_mob, const long long* s_moff, int* s_cnt) {
  const uint32_t bars = smem_u32(smem + kOffBar);
  const uint8_t* wbytes = reinterpret_cast<const uint8_t*>(a.weights);
  // piece 0..2 = W1..W3, 3 = W4, 4 = aux (into buffer abuf): one bulk copy each, signalled on the piece's mbarrier.
  // A piece is refilled for the next layer as soon as ALL tiles' MMAs that read it are done.  (W4 as ONE piece is dead only after
  // the last tile's chunk 3, so the leading tile's chunk 0 of the next layer waits for the last tile -- ~2.9 k cycles per layer in
  // the timeline.  Refilling it chunk by chunk removes that wait and was measured 3 % SLOWER, with and without the service warps
  // (14.18 vs 13.78 M cycles per image): the coupling through this piece is what keeps the four tiles in two anti-phase pairs;
  // without it they drift into lock step and queue for the tensor pipe at the same time.)
  auto load_piece = [&](int mob_idx, int piece, int abuf) {
    const uint8_t* src = wbytes + s_moff[mob_idx] * 4;
    uint32_t dst, bytes, bar;
    if (piece < 3) { src += piece * kW1Bytes; dst = kOffW + piece * kW1Bytes; bytes = kW1Bytes; bar = BAR_W_FULL + piece; }
    else if (piece == 3) { src += kHidW; dst = kOffLastW; bytes = kLastW; bar = BAR_W_FULL + 3; }
    else { src += kHidW + kLastW; dst = kOffAux + abuf * kAuxStride; bytes = kAuxBytes; bar = BAR_AUX_FULL + abuf; }
    mbar_expect_tx(bars + 8 * bar, bytes);
    bulk_g2s(smem_u32(smem + dst), src, bytes, bars + 8 * bar);
  };
  if (tile == 0 && lane == 0 && sc.total_steps > 0) {      // tile slot 0 is active whenever the CTA has work
    for (int piece = 0; piece < 4; ++piece) load_piece(0, piece, 0);
    load_piece(0, 4, 0);
    if (sc.total_steps > 1) load_piece(n_mob > 1 ? 1 : 0, 4, 1);
  }
  const uint32_t tm_tile = tmem_base + (uint32_t)tile * kColsPerTile;
  const uint32_t y_d = umma_desc_lo_ns(smem_u32(smem + kOffY + tile * 4096)), c_d = umma_desc_lo_ns(smem_u32(smem + kOffC + tile * 2048));
  const uint32_t w_hid_d = umma_desc_lo(smem_u32(smem + kOffW)), w_last_d = umma_desc_lo(smem_u32(smem + kOffLastW));
  const uint32_t bias_hid_d = umma_desc_lo_ns(smem_u32(smem + kOffW + 16384)), bias_last_d = umma_desc_lo_ns(smem_u32(smem + kOffLastW + 65536));
  const uint32_t aux_blk_d = umma_desc_lo_ns(smem_u32(smem + kOffAux + kAuxFirst));
  const uint32_t bar_mma = bars + 8 * (BAR_MMA + tile), bar_ready = bars + 8 * (BAR_READY + tile);
  constexpr uint32_t kIdesc = umma_idesc(128, 64);
  const uint32_t d = tm_tile + kColD;
  const int n_active = sc.n_active;
  uint32_t par_mma = 0, par_ready = 0, par_w = 0;
  int step = 0;
  int mob_cur = 0;

  auto wait_ready = [&]() {                          // the tile's four worker warps have handed over (Y block / A operand / drained D)
    mbar_wait(bar_ready, par_ready);
    par_ready ^= 1;
    tc_fence_after();
  };
  auto wait_gemm = [&]() {                           // the workers watch the mbarrier themselves; this wait only orders the refill bookkeeping
    mbar_wait(bar_mma, par_mma);
    par_mma ^= 1;
  };

  for (int item = 0; item < sc.my_items; ++item) {
#pragma unroll 1
    for (int li = 0; li < a.n_layers; ++li) {
      const LayerDev L = a.layers[li];
      if (L.kind != RNF_LAYER_MOBIUS) continue;
      const bool c_by_mma = GRID && L.cond_slot >= 0 && a.cond != nullptr;
      const int abuf = (int)(step & 1);
      const int mob_n1 = mob_cur + 1 >= n_mob ? mob_cur + 1 - n_mob : mob_cur + 1;
      const int mob_n2 = mob_n1 + 1 >= n_mob ? mob_n1 + 1 - n_mob : mob_n1 + 1;
      // ---- fc_first and three hidden layers: four dependent GEMM round trips ----
#pragma unroll 1
      for (int l = 0; l < 4; ++l) {
        if (l == 0) mbar_wait(bars + 8 * (BAR_AUX_FULL + abuf), (uint32_t)((step >> 1) & 1));
        else mbar_wait(bars + 8 * (BAR_W_FULL + l - 1), (par_w >> (l - 1)) & 1u);
        wait_ready();                                // l == 0: Y block written; l > 0: the A operand
        if (l == 0) {
          if (elect_one_sync()) {
            umma_f16(d, y_d, aux_blk_d + abuf * (kAuxStride >> 4), kDescHiNS, kIdesc, 0);
            if (c_by_mma) umma_f16(d, y_d, c_d, kDescHiNS, kIdesc, 1);
            umma_commit(bar_mma);
          }
          __syncwarp();
        } else {
          const uint32_t wb = w_hid_d + (l - 1) * (kW1Bytes >> 4);
          if (elect_one_sync()) {
            umma_f16(d, y_d, bias_hid_d + (l - 1) * (kW1Bytes >> 4), kDescHiNS, kIdesc, 0);
            issue_split_ts_half(d, tm_tile + kColAhi, tm_tile + kColAlo, wb, wb + (8192 >> 4), kIdesc, 0);
          }
          __syncwarp();
          if (elect_one_sync()) {
            issue_split_ts_half(d, tm_tile + kColAhi, tm_tile + kColAlo, wb, wb + (8192 >> 4), kIdesc, 2);
            if (c_by_mma && l == 3) umma_f16(d, y_d, c_d, kDescHiNS, kIdesc, 1);
            umma_commit(bar_mma);
          }
          __syncwarp();
        }
        wait_gemm();
        // a piece is dead once ALL tiles' GEMM that reads it has completed: the last tile to get here refills it
        if (lane == 0) {
          if (l == 0) { if ((atomicAdd(&s_cnt[4 + abuf], 1) % n_active) == n_active - 1 && step + 2 < sc.total_steps) load_piece(mob_n2, 4, abuf); }
          else if ((atomicAdd(&s_cnt[l - 1], 1) % n_active) == n_active - 1 && step + 1 < sc.total_steps) load_piece(mob_n1, l - 1, 0);
        }
        __syncwarp();
      }
      // ---- fc_last in four N = 64 chunks through the single accumulator ----
      mbar_wait(bars + 8 * (BAR_W_FULL + 3), (par_w >> 3) & 1u);
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const uint32_t wb = w_last_d + c * (8192 >> 4);                    // rows 64c .. 64c+63 of the hi plane
        if (c == 0) {
          wait_ready();                              // the last hidden epilogue
        } else {                                     // chunk c - 1 drained into registers; the workers have ~1.5 k cycles of arithmetic left
          mbar_wait(bar_ready, par_ready);
          par_ready ^= 1;
          tc_fence_after();
        }
        if (c == 0) {
          if (elect_one_sync()) {
            umma_f16(d, y_d, bias_last_d, kDescHiNS, kIdesc, 0);
            issue_split_ts_half(d, tm_tile + kColAhi, tm_tile + kColAlo, wb, wb + (32768 >> 4), kIdesc, 0);
          }
          __syncwarp();
          if (elect_one_sync()) {
            issue_split_ts_half(d, tm_tile + kColAhi, tm_tile + kColAlo, wb, wb + (32768 >> 4), kIdesc, 2);
            umma_commit(bar_mma);
          }
          __syncwarp();
        } else {
          if (elect_one_sync()) {
            umma_f16(d, y_d, bias_last_d + c * (2048 >> 4), kDescHiNS, kIdesc, 0);
            issue_split_ts(d, tm_tile + kColAhi, tm_tile + kColAlo, wb, wb + (32768 >> 4), kIdesc);
            umma_commit(bar_mma);
          }
          __syncwarp();
        }
        if (c == 0) {
          wait_gemm();
        } else if (c == 3) {
          // W4 is dead the moment the last chunk's MMAs have completed (not after the arithmetic on it): the last tile to see
          // that refills it.
          wait_gemm();
          if (lane == 0 && (atomicAdd(&s_cnt[3], 1) % n_active) == n_active - 1 && step + 1 < sc.total_steps) load_piece(mob_n1, 3, 0);
          __syncwarp();
        } else {
          par_mma ^= 1;                              // chunks 1, 2: the workers poll the mbarrier themselves
        }
      }
      par_w ^= 0xFu;
      ++step;
      mob_cur = mob_n1;
    }
  }
}

template <bool GRID>
__global__ void __launch_bounds__(kThreads, 1) flow_t4_kernel(const FlowArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const bool service = warp >= kTiles * 4;           // warpgroup 4: one service warp per tile
  const int tile = service ? warp - kTiles * 4 : warp >> 2;
  const int rowi = (warp & 3) * 32 + lane;           // worker: row inside the tile = TMEM lane
  const uint32_t bars = smem_u32(smem + kOffBar);

  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kOffMisc);
  int* s_cnt = reinterpret_cast<int*>(smem + kOffMisc + 4);                // tiles done with: [0..2] W1..W3, [3] W4, [4 + buf] aux
  long long* s_moff = reinterpret_cast<long long*>(smem + kOffMisc + 64);

  int n_mob = 0;
  for (int i = 0; i < a.n_layers; ++i)
    if (a.layers[i].kind == RNF_LAYER_MOBIUS) {
      if (tid == 0) s_moff[n_mob] = a.layers[i].w_off_tc;
      ++n_mob;
    }
  if (tid == 0) {
    for (int i = 0; i < BAR_COUNT; ++i) mbar_init(bars + 8 * i, (i >= BAR_READY) ? 4 : 1);     // ready: one arrival per worker warp
    for (int i = 0; i < 6; ++i) s_cnt[i] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // Y and per-image blocks start out as zeros (the unused K slots stay zero for the whole kernel)
  for (int i = tid; i < (kTiles * (4096 + 2048)) / 16; i += kThreads) reinterpret_cast<uint4*>(smem + kOffY)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  // Tiles in flight in this launch (launch_flow_t4): 4 for large launches; a launch of only a few tiles per SM balances better with
  // fewer (e.g. 5.3 tiles per SM as 2 rounds of 3 instead of a round of 4 and a round of 4 on a third of the SMs).  The warps of
  // the unused tile slots skip the work loop.
  TileSched sc;
  sc.n_active = a.t4_active > 0 && a.t4_active < kTiles ? a.t4_active : kTiles;
  const int n_active = sc.n_active;
  const int64_t n_groups = (a.n_tiles + n_active - 1) / n_active;
  sc.my_items = (blockIdx.x < n_groups && tile < n_active) ? (int)((n_groups - 1 - blockIdx.x) / gridDim.x + 1) : 0;
  sc.total_steps = sc.my_items * n_mob;

  if (service) {
    set_max_regs_dec<kServiceRegs>();
    service_warp<GRID>(a, smem, tmem_base, tile, lane, sc, n_mob, s_moff, s_cnt);
  } else {
    set_max_regs_inc<kWorkerRegs>();
    const uint32_t tm = tmem_base + (uint32_t)tile * kColsPerTile + ((uint32_t)((warp & 3) * 32) << 16);   // my warp's lane quarter
    uint8_t* y_blk = smem + kOffY + tile * 4096;
    uint8_t* c_blk = smem + kOffC + tile * 2048;
    const uint32_t bar_mma = bars + 8 * (BAR_MMA + tile), bar_ready = bars + 8 * (BAR_READY + tile);
    uint32_t par_mma = 0;
#if RNF_TC_TRACE
    int64_t step = 0;
#endif

    // Hand-over of the tile's accumulator / A operand / Y block to the service warp: every thread orders its TMEM accesses,
    // one lane per warp arrives on the tile's mbarrier.  Nobody waits here.
    auto hand_over = [&]() {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_ready);
    };
    // Wait for a GEMM that the tile cannot overlap with anything (the dependent round trips of the chain): every worker warp
    // watches the MMA's mbarrier itself (try_wait with a suspend hint).  Sleeping in a named barrier that the service warp
    // arrives on instead adds a second wake-up hop to the critical path (measured ~1 % slower in cycles, DESIGN.md svc-x).
    auto wait_mma_long = [&]() {
      mbar_wait_hint<kDirectWaitNs>(bar_mma, par_mma);
      par_mma ^= 1;
      tc_fence_after();
    };
    auto wait_mma = [&]() {                            // a GEMM that ran under the previous chunk's arithmetic: normally complete
      mbar_wait(bar_mma, par_mma);
      par_mma ^= 1;
      tc_fence_after();
    };

    for (int item = 0; item < sc.my_items; ++item) {
      const int64_t tile_idx = n_active * (blockIdx.x + item * (int64_t)gridDim.x) + tile;
      int64_t row = 0, img = 0, g = 0;
      bool valid = false;
      float R[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
      if (tile_idx < a.n_tiles) {
        if (GRID) {
          img = tile_idx / a.tiles_per_image;
          g = (tile_idx % a.tiles_per_image) * kRows + rowi;
          valid = g < a.G;
          row = img * a.G + g;
          if (valid) {
            float Gm[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) Gm[i] = __ldg(a.R_in + g * 9 + i);
            if (a.offset != nullptr) {                 // samples = grid @ random_rot (eval.py:439-440)
              float O[9];
#pragma unroll
              for (int i = 0; i < 9; ++i) O[i] = __ldg(a.offset + i);
#pragma unroll
              for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j)
                  R[3 * i + j] = fmaf(Gm[3 * i + 2], O[6 + j], fmaf(Gm[3 * i + 1], O[3 + j], Gm[3 * i] * O[j]));
            } else {
#pragma unroll
              for (int i = 0; i < 9; ++i) R[i] = Gm[i];
            }
          }
        } else {
          row = tile_idx * kRows + rowi;
          valid = row < a.N;
          if (valid) {
#pragma unroll
            for (int i = 0; i < 9; ++i) R[i] = __ldg(a.R_in + row * 9 + i);
            if (a.cond != nullptr) img = a.feat_index != nullptr ? (int64_t)__ldg(a.feat_index + row) : row / a.rows_per_image;
          }
        }
      }
      const float* cond_img = a.cond != nullptr ? a.cond + img * a.cond_stride : nullptr;
      float ldj = 0.0f;
      float dgt = 0.0f;                                  // spread metric: angle of the evaluation point to the image's ground truth
      if (GRID && a.gt != nullptr && valid) dgt = gt_distance(a.gt + img * a.gt_k * 9, a.gt_k, R);

#pragma unroll 1
      for (int li = 0; li < a.n_layers; ++li) {
        const LayerDev L = a.layers[li];
        if (L.kind != RNF_LAYER_MOBIUS) {
          const float* W = L.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)L.cond_slot * kAffFloats
                                            : a.weights + L.w_off;
          affine_family_layer<true>(L, W, R, ldj);
          continue;
        }
        // ================================ Mobius layer ================================
        const int p0 = L.perm, p1 = (L.perm + 1) % 3, p2 = (L.perm + 2) % 3;
        float x[3], y[3];
        Plane P;
        get_col(R, p0, x);
        get_col(R, p1, y);
        make_frame_fast(x, y, P);
        const float zr = dot3(x, P.r), zv = dot3(x, P.v);   // in-plane coordinates of the moving column
        const float* cimg = (L.cond_slot >= 0 && cond_img != nullptr) ? cond_img + (int64_t)L.cond_slot * kH : nullptr;
        const bool c_by_mma = GRID && cimg != nullptr;      // warp- and tile-uniform (the service warp derives the same flag)
        const float* cadd = GRID ? nullptr : cimg;
#if RNF_TC_TRACE
        const bool tr_on = a.trace != nullptr && blockIdx.x == 0 && (warp & 3) == 0 && lane == 0 && step >= 40 && step < 48;
        long long* tr = a.trace + ((tile * 8 + (step - 40)) * 32);
#endif
        TRACE(0);

        // ---- my row of the Y block: (1, 1, y_hi, y_lo | y_hi, 1, 1, 0, 0, 0); per-image block in grid mode ----
        {
          __half yh[3], yl[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            yh[i] = __float2half_rn(y[i]);
            yl[i] = __float2half_rn(y[i] - __half2float(yh[i]));
          }
          const __half one = __float2half_rn(1.0f), zero = __float2half_rn(0.0f);
          uint8_t* yrow = y_blk + (rowi >> 3) * 256 + (rowi & 7) * 16;
          *reinterpret_cast<uint4*>(yrow) = make_uint4(pack_h2(one, one), pack_h2(yh[0], yh[1]), pack_h2(yh[2], yl[0]), pack_h2(yl[1], yl[2]));
          *reinterpret_cast<uint4*>(yrow + 128) = make_uint4(pack_h2(yh[0], yh[1]), pack_h2(yh[2], one), pack_h2(one, zero), 0u);
          if (c_by_mma && rowi < 64) {
            const float cv = __ldg(cimg + rowi);
            const __half ch = __float2half_rn(cv);
            const __half cl = __float2half_rn(cv - __half2float(ch));
            *reinterpret_cast<uint32_t*>(c_blk + (rowi >> 3) * 256 + (rowi & 7) * 16) = pack_h2(ch, cl);
          }
        }
        fence_proxy_async();
        hand_over();
        TRACE(1);
        // ---- fc_first and three hidden layers: four dependent GEMM round trips ----
#pragma unroll 1
        for (int l = 0; l < 4; ++l) {
          wait_mma_long();
          TRACE(3 + 3 * l);
          const float* ca = (l == 0 || l == 3) ? cadd : nullptr;
          epilogue64(tm, ca, hand_over);
          TRACE(4 + 3 * l);
        }
        // ---- fc_last in four N = 64 chunks through the single accumulator; 16 mixture components per chunk ----
        f32x2 S_sp2 = 0ull, S_th2 = 0ull, S_f2 = 0ull;   // packed partial sums (even | odd components)
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          float buf0[16], buf1[16];
          if (c == 0) wait_mma_long(); else wait_mma();  // chunks 1..3 ran under the previous chunk's arithmetic: no spinning
          TRACE(14 + c);
          tmem_ld16_async(tm + kColD, buf0);
          tmem_ld16_async(tm + kColD + 16, buf1);
          tmem_ld_wait16(buf0);
          mixture_pairs<2, true>(P, zr, zv, buf0, S_sp2, S_th2, S_f2);
          tmem_ld16_async(tm + kColD + 32, buf0);
          tmem_ld_wait16(buf1);
          mixture_pairs<2, true>(P, zr, zv, buf1, S_sp2, S_th2, S_f2);
          tmem_ld16_async(tm + kColD + 48, buf1);
          tmem_ld_wait16(buf0);
          tmem_ld_wait16(buf1);
          if (c < 3) hand_over();                        // accumulator drained: the next chunk runs under the math below
          mixture_pairs<2, true>(P, zr, zv, buf0, S_sp2, S_th2, S_f2);
          mixture_pairs<2, true>(P, zr, zv, buf1, S_sp2, S_th2, S_f2);
        }
        TRACE(18);
        float nx[3], nz[3];
        const float S_sp = hsum(S_sp2), S_th = hsum(S_th2), S_f = hsum(S_f2);
        const float inv_sp = rcp_nr(S_sp);
        circle_point_fast(P.r, P.v, mixture_angle(S_th, inv_sp), nx);
        ldj += log_fast(S_f * inv_sp);
        cross3(nx, y, nz);
        normalize3_fast(nz);
        set_col(R, p0, nx);
        set_col(R, p2, nz);
        TRACE(19);
#if RNF_TC_TRACE
        ++step;
#endif
      }

      // ================================ outputs ================================
      if (!GRID) {
        if (valid) {
#pragma unroll
          for (int i = 0; i < 9; ++i) a.R_out[row * 9 + i] = R[i];
          a.ldj_out[row] = ldj;
        }
      } else if (tile_idx < a.n_tiles) {
        float lp = ldj;
        if (a.fisher_A != nullptr) {
          float tr = 0.0f;
#pragma unroll
          for (int i = 0; i < 9; ++i) tr = fmaf(__ldg(a.fisher_A + img * 9 + i), R[i], tr);
          lp += tr - __ldg(a.fisher_c + img);
        }
        if (!valid) lp = -INFINITY;
        if (a.logp_out != nullptr && valid) a.logp_out[row] = lp;
        float* s_v = reinterpret_cast<float*>(smem + kOffRed + tile * 128);
        long long* s_i = reinterpret_cast<long long*>(smem + kOffRed + tile * 128 + 32);
        const int w4 = warp & 3;
        const int bar_red = 5 + tile;
        float bv = lp;
        long long bi = valid ? (long long)g : 0x7fffffffffffffffLL;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (lane == 0) { s_v[w4] = bv; s_i[w4] = bi; }
        named_bar(bar_red, 128);
        bv = s_v[0]; bi = s_i[0];
#pragma unroll
        for (int w = 1; w < 4; ++w) {
          const float ov = s_v[w];
          const long long oi = s_i[w];
          if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        const float m = bv;
        float e = (valid && m != -INFINITY) ? expf(lp - m) : 0.0f;
        float ed = e * dgt;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          e += __shfl_xor_sync(0xffffffffu, e, o);
          ed += __shfl_xor_sync(0xffffffffu, ed, o);
        }
        named_bar(bar_red, 128);
        if (lane == 0) { s_v[w4] = e; s_v[4 + w4] = ed; }
        named_bar(bar_red, 128);
        if (rowi == 0) {
          const float s = (s_v[0] + s_v[1]) + (s_v[2] + s_v[3]);
          float* p = a.part + tile_idx * kPartStride;
          p[0] = m;
          p[1] = s;
          p[4] = (s_v[4] + s_v[5]) + (s_v[6] + s_v[7]);
          p[2] = __int_as_float((int)(bi & 0xffffffffLL));
          p[3] = __int_as_float((int)(bi >> 32));
        }
        named_bar(bar_red, 128);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

}  // namespace

// Tiles in flight per CTA for a launch of n_tiles over sm_count persistent CTAs: minimise rounds x (relative duration of a round
// with a tiles in flight).  Round durations measured with the RNF_T4_ACTIVE override on raw.yml, eight full rounds each
// (tools/active_tiles_probe.py, profiles/r02_active_tiles_service.txt): 112 / 171 / 238 / 264 M rot/s with 1 / 2 / 3 / 4 tiles in
// flight, i.e. a round of one tile lasts 0.59 of a round of four, two 0.77, three 0.83.
int pick_active_tiles(int64_t n_tiles, int sm_count) {
  static const float kRound[5] = {0.f, 0.589f, 0.772f, 0.834f, 1.0f};
  int best = kTiles;
  float best_cost = 1e30f;
  for (int act = kTiles; act >= 1; --act) {
    const int64_t groups = (n_tiles + act - 1) / act;
    const int64_t rounds = (groups + sm_count - 1) / sm_count;
    const float cost = (float)rounds * kRound[act];
    if (cost < best_cost - 1e-6f) { best_cost = cost; best = act; }
  }
  return best;
}

cudaError_t launch_flow_t4(const FlowArgs& a_in, int sm_count, cudaStream_t st) {
  FlowArgs a = a_in;
  const bool grid_mode = a.G > 0;
  void (*kern)(const FlowArgs) = grid_mode ? flow_t4_kernel<true> : flow_t4_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemAlloc);
  if (e != cudaSuccess) return e;
  if (a.n_tiles <= 0) return cudaSuccess;
  a.t4_active = pick_active_tiles(a.n_tiles, sm_count);
  if (const char* force = getenv("RNF_T4_ACTIVE")) {         // measurement override (tools/): tiles in flight, 1..4
    const int v = atoi(force);
    if (v >= 1 && v <= kTiles) a.t4_active = v;
  }
  const int64_t groups = (a.n_tiles + a.t4_active - 1) / a.t4_active;
  const int64_t grid = groups < sm_count ? groups : sm_count;
  kern<<<(unsigned)grid, kThreads, kSmemAlloc, st>>>(a);
  return cudaGetLastError();
}

}  // namespace rnf
