// flow_row.cu -- fused flow kernel with the conditioner GEMMs on the 5th-gen tensor cores (tcgen05 + TMEM), two tiles per SM,
// one thread per rotation: forward, inverse (bisection) and grid mode, sm_100a.
//
// One CTA (256 threads, one per SM, persistent) works on a PAIR of 128-rotation tiles.  A tile's 128 rows are the 128 TMEM
// lanes of its accumulator; a row's thread keeps the rotation's 3x3 matrix and running log|det J| in registers across the
// whole layer stack (flow/flow.py:53-72).  Per Mobius layer (flow/mobiusflow.py:46-125) and tile:
//   CUDA cores : frame (r, v), first conditioner layer  h0 = W0[:, :3].y + b0 + c_img  (flow/condition.py:25)
//                -> ReLU -> split into fp16 (hi, lo) -> K-major 128B-swizzled A operand in shared memory
//   tensor core: D[128 x 64] = bias + A . W^T as a K = 16 bias MMA plus three products  Alo.Whi + Ahi.Wlo + Ahi.Whi  (fp32
//                accumulate in TMEM; error-compensated split => fp32-level accuracy), three times (layers.1/3/5)
//   CUDA cores : tcgen05.ld -> ReLU (residual on the last) -> split -> A operand
//   tensor core: fc_last  D[128 x 256] in two N = 128 chunks, each committed to its own mbarrier
//   CUDA cores : the 64 mixture components straight out of TMEM, eight at a time in packed f32x2 arithmetic (mobius_pair.cuh).
// Inverse direction: the prepared parameters of the 64 components go back into the row's own TMEM lane (256 columns) and the
// 15 bisection probes of BinFind.forward (flow/mobiusflow.py:196-224) stream them from there -- which is why this kernel keeps
// two tiles per SM; the forward / grid direction has a four-tile kernel (flow_t4.cu) and uses this one as its cross-check.
// Weights: the host packs, per Mobius layer, the exact shared-memory image (engine.pack_mobius_tc); one cp.async.bulk per
// piece brings it in, signalled on an mbarrier, and is re-issued for the next layer as soon as both tiles' MMAs that read the
// piece have completed -- so weight traffic overlaps the mixture math.
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

#ifndef RNF_INV_NEWTON
#define RNF_INV_NEWTON 1         // inverse: locate the root with Newton steps, then replay the reference's 15 halvings (see below)
#endif
constexpr int kThreads = 256;
constexpr int kRows = 128;                        // rows per tile = TMEM lanes = threads per tile

// shared-memory image (bytes from a 1024-aligned base); weight pieces as in tc_common.cuh
constexpr int kOffW = 0;
constexpr int kOffLastW = kHidW;
constexpr int kOffAux = kOffLastW + kLastW;       // double buffered (layer parity)
constexpr int kOffA = kOffAux + 2 * kAuxStride;   // [tile][hi|lo] 128x64 fp16 (16 KB each)
constexpr int kOffOnes = kOffA + 4 * 16384;       // constant [128 x 16] fp16 ones tile (bias MMA)
constexpr int kOffRed = kOffOnes + 4096;          // [tile] reduction scratch
constexpr int kOffBar = kOffRed + 2 * 128;
constexpr int kOffMisc = kOffBar + 8 * 16;        // tmem base, counters, Mobius offset table
constexpr int kSmemBytes = kOffMisc + 32 + 64 * 8;
constexpr int kSmemAlloc = kSmemBytes + 1024;
static_assert(kOffA % 1024 == 0 && kOffLastW % 1024 == 0 && kW1Bytes % 1024 == 0, "UMMA SW128 tiles need 1024 B alignment");
static_assert(kSmemAlloc <= 232448, "exceeds the 227 KB shared-memory limit of an sm_100 CTA");

enum { BAR_W_FULL = 0 /* W1,W2,W3,W4 */, BAR_AUX_FULL = 4 /* [2] */, BAR_MMA = 6 /* [tile][2] */, BAR_COUNT = 10 };

// ReLU + split 32 pre-activations (hidden units 32h .. 32h+31 of row r) into the fp16 hi / lo planes of the K-major SW128 A
// operand: element (r, k) lives at (r/8)*1024 + (r%8)*128 + ((k/8) ^ (r%8))*16 + (k%8)*2.
__device__ __forceinline__ void store_a32(uint8_t* a_hi, uint8_t* a_lo, int r, int h, const float v[32]) {
  const int rbase = (r >> 3) * 1024 + (r & 7) * 128;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      // as in flow_t4.cu: truncation by mask + packed subtract (5 instructions per pair instead of 6 with two conversions back and
      // two scalar subtracts); this kernel runs at the per-warp issue cadence, so an instruction less is time less.  The masked
      // value converts exactly up to 65504 and to +Inf from 65536 on: overflow is loud, as in flow_t4.cu relu_split_pair.
      const float x0 = v[8 * c + 2 * e], x1 = v[8 * c + 2 * e + 1];
      const float m0 = __uint_as_float(__float_as_uint(x0) & 0xFFFFE000u), m1 = __uint_as_float(__float_as_uint(x1) & 0xFFFFE000u);
      asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi[e]) : "f"(m1), "f"(m0));
      float d0, d1;
      upk(sub2(pk(x0, x1), pk(m0, m1)), d0, d1);
      asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo[e]) : "f"(d1), "f"(d0));
    }
    const int off = rbase + (((4 * h + c) ^ (r & 7)) << 4);
    *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, float v[32]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
        "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
        "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait32(float v[32]) {
  tmem_ld_wait16(v);        // one tcgen05.wait::ld covers every outstanding load; name all 32 registers for the compiler
  uint32_t* u = reinterpret_cast<uint32_t*>(v + 16);
  asm volatile(""
               : "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7]), "+r"(u[8]),
                 "+r"(u[9]), "+r"(u[10]), "+r"(u[11]), "+r"(u[12]), "+r"(u[13]), "+r"(u[14]), "+r"(u[15])
               :
               : "memory");
}

template <bool INV, bool GRID>
__global__ void __launch_bounds__(kThreads, 1) flow_row_kernel(const FlowArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int tile = warp >> 2;                        // 0 / 1
  const int rowi = (warp & 3) * 32 + lane;           // row inside the tile = TMEM lane
  const bool elected = (tid & 127) == 0;             // refills weights for the tile pair
  const bool issuer_warp = __shfl_sync(0xffffffffu, (int)elected, 0) != 0;   // warp-uniform: issues this tile's MMAs
  const uint32_t bars = smem_u32(smem + kOffBar);

  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kOffMisc);
  int* s_cnt = reinterpret_cast<int*>(smem + kOffMisc + 4);                // consumers done: [0..2] W1..W3, [3] W4, [4] aux
  long long* s_moff = reinterpret_cast<long long*>(smem + kOffMisc + 32);

  int n_mob = 0;
  for (int i = 0; i < a.n_layers; ++i) {
    const int li = INV ? a.n_layers - 1 - i : i;
    if (a.layers[li].kind == RNF_LAYER_MOBIUS) {
      if (tid == 0) s_moff[n_mob] = a.layers[li].w_off_tc;
      ++n_mob;
    }
  }
  if (tid == 0) {
    for (int i = 0; i < BAR_COUNT; ++i) mbar_init(bars + 8 * i, 1);
    for (int i = 0; i < 5; ++i) s_cnt[i] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // constant ones tile (bias MMA): 4096 B, thread tid writes bytes 16 tid .. 16 tid + 15; ones in K columns 0 and 1
  reinterpret_cast<uint4*>(smem + kOffOnes)[tid] = make_uint4((tid & 15) < 8 ? 0x3C003C00u : 0u, 0u, 0u, 0u);
  fence_proxy_async();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t tm = tmem_base + (uint32_t)(tile * 256) + ((uint32_t)((warp & 3) * 32) << 16);   // my lane, my tile

  const int64_t n_pairs = (a.n_tiles + 1) / 2;
  const int64_t my_items = blockIdx.x < n_pairs ? (n_pairs - 1 - blockIdx.x) / gridDim.x + 1 : 0;
  const int64_t total_steps = my_items * n_mob;
  const uint8_t* wbytes = reinterpret_cast<const uint8_t*>(a.weights);
  auto load_piece = [&](int mob_idx, int piece, int abuf) {
    const uint8_t* src = wbytes + s_moff[mob_idx] * 4;
    uint32_t dst, bytes, bar;
    if (piece < 3) { src += piece * kW1Bytes; dst = kOffW + piece * kW1Bytes; bytes = kW1Bytes; bar = BAR_W_FULL + piece; }
    else if (piece == 3) { src += kHidW; dst = kOffLastW; bytes = kLastW; bar = BAR_W_FULL + 3; }
    else { src += kHidW + kLastW; dst = kOffAux + abuf * kAuxStride; bytes = kAuxBytes; bar = BAR_AUX_FULL + abuf; }
    mbar_expect_tx(bars + 8 * bar, bytes);
    bulk_g2s(smem_u32(smem + dst), src, bytes, bars + 8 * bar);
  };
  if (tid == 0 && total_steps > 0) {
    for (int piece = 0; piece < 4; ++piece) load_piece(0, piece, 0);
    load_piece(0, 4, 0);
    if (total_steps > 1) load_piece(n_mob > 1 ? 1 : 0, 4, 1);
  }

  uint8_t* a_hi = smem + kOffA + tile * 32768;
  uint8_t* a_lo = a_hi + 16384;
  const uint32_t a_hi_d = umma_desc_lo(smem_u32(a_hi)), a_lo_d = umma_desc_lo(smem_u32(a_lo));
  const uint32_t w_hid_d = umma_desc_lo(smem_u32(smem + kOffW)), w_last_d = umma_desc_lo(smem_u32(smem + kOffLastW));
  const uint32_t ones_d = umma_desc_lo_ns(smem_u32(smem + kOffOnes));
  const uint32_t bias_hid_d = umma_desc_lo_ns(smem_u32(smem + kOffW + 16384)), bias_last_d = umma_desc_lo_ns(smem_u32(smem + kOffLastW + 65536));
  const int bar_tile = 1 + tile;                     // named barrier of the tile's 128 threads
  const uint32_t bar_mma0 = bars + 8 * (BAR_MMA + 2 * tile), bar_mma1 = bar_mma0 + 8;   // hidden GEMMs + chunk A | chunk B
  uint32_t par_mma0 = 0, par_mma1 = 0, par_w = 0;
  int64_t step = 0;
  int mob_cur = 0;

  for (int64_t item = 0; item < my_items; ++item) {
    const int64_t tile_idx = 2 * (blockIdx.x + item * (int64_t)gridDim.x) + tile;
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
    for (int lstep = 0; lstep < a.n_layers; ++lstep) {
      const int li = INV ? a.n_layers - 1 - lstep : lstep;
      const LayerDev L = a.layers[li];
      if (L.kind != RNF_LAYER_MOBIUS) {
        const float* W = L.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)L.cond_slot * kAffFloats
                                          : a.weights + L.w_off;
        if (INV) W += kAffInv;
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
#if RNF_TC_TRACE
      const bool tr_on = a.trace != nullptr && blockIdx.x == 0 && elected && step >= 40 && step < 48;
      long long* tr = a.trace + ((tile * 8 + (step - 40)) * 32);
#endif
      TRACE(0);
      TRACE(1);
      const int abuf = (int)(step & 1);
      const int mob_n1 = mob_cur + 1 >= n_mob ? mob_cur + 1 - n_mob : mob_cur + 1;
      const int mob_n2 = mob_n1 + 1 >= n_mob ? mob_n1 + 1 - n_mob : mob_n1 + 1;
      mbar_wait(bars + 8 * (BAR_AUX_FULL + abuf), (uint32_t)((step >> 1) & 1));
      const float4* sFirst = reinterpret_cast<const float4*>(smem + kOffAux + abuf * kAuxStride);

      // ---- first conditioner layer, all 64 hidden units; pre-activations stashed in TMEM columns 64..127 ----
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float h0[32];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          float4 cf = make_float4(0.f, 0.f, 0.f, 0.f);
          if (cimg != nullptr) cf = __ldg(reinterpret_cast<const float4*>(cimg + 32 * h) + j4);
          const float cc[4] = {cf.x, cf.y, cf.z, cf.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float4 f = sFirst[32 * h + 4 * j4 + e];
            h0[4 * j4 + e] = fmaf(f.z, y[2], fmaf(f.y, y[1], fmaf(f.x, y[0], f.w))) + cc[e];
          }
        }
        tmem_st32(tm + 64 + 32 * h, h0);
        store_a32(a_hi, a_lo, rowi, h, h0);          // ReLU happens inside the fp16 split
      }
      TRACE(2);
      // ---- three hidden layers on the tensor core ----
#pragma unroll 1
      for (int l = 0; l < 3; ++l) {
        fence_proxy_async();
        tc_fence_before();
        named_bar(bar_tile, 128);
        TRACE(3 + 4 * l);
        if (issuer_warp) {
          mbar_wait(bars + 8 * (BAR_W_FULL + l), (par_w >> l) & 1u);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t wb = w_hid_d + l * (kW1Bytes >> 4);
            issue_split_gemm(tmem_base + tile * 256, a_hi_d, a_lo_d, wb, wb + (8192 >> 4), ones_d, bias_hid_d + l * (kW1Bytes >> 4),
                             umma_idesc(128, 64));
            umma_commit(bar_mma0);
          }
          __syncwarp();
        }
        TRACE(4 + 4 * l);
        mbar_wait(bar_mma0, par_mma0);
        par_mma0 ^= 1;
        tc_fence_after();
        TRACE(5 + 4 * l);
        // W_l is dead once BOTH tiles' GEMM l has completed: the second tile to get here refills it for the next layer
        if (elected && (atomicAdd(&s_cnt[l], 1) & 1) && step + 1 < total_steps) load_piece(mob_n1, l, 0);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float acc[32];
          tmem_ld32(tm + 32 * h, acc);
          if (l == 2) {                              // relu_last(x0 + x)   (flow/condition.py:29); biases come out of the GEMM
            float h0[32];
            tmem_ld32(tm + 64 + 32 * h, h0);
#pragma unroll
            for (int j = 0; j < 32; j += 2) upk(add2(pk(acc[j], acc[j + 1]), pk(h0[j], h0[j + 1])), acc[j], acc[j + 1]);
          }
          store_a32(a_hi, a_lo, rowi, h, acc);
        }
        TRACE(6 + 4 * l);
      }
      // ---- fc_last: two N = 128 chunks, own barrier each ----
      fence_proxy_async();
      tc_fence_before();
      named_bar(bar_tile, 128);
      TRACE(15);
      if (issuer_warp) {
        mbar_wait(bars + 8 * (BAR_W_FULL + 3), (par_w >> 3) & 1u);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t d = tmem_base + tile * 256;
          issue_split_gemm(d, a_hi_d, a_lo_d, w_last_d, w_last_d + (32768 >> 4), ones_d, bias_last_d, umma_idesc(128, 128));
          umma_commit(bar_mma0);
          issue_split_gemm(d + 128, a_hi_d, a_lo_d, w_last_d + (16384 >> 4), w_last_d + ((32768 + 16384) >> 4), ones_d,
                           bias_last_d + (4096 >> 4), umma_idesc(128, 128));
          umma_commit(bar_mma1);
        }
        __syncwarp();
        par_w ^= 0xFu;
      }

      // ---- mixture of all 64 components, 8 at a time straight from TMEM; next 32 columns in flight ----
      f32x2 S_sp2 = 0ull, S_th2 = 0ull, S_f2 = 0ull;   // packed partial sums (even | odd components)
      {
        float bufA[32], bufB[32];
        TRACE(16);
        mbar_wait(bar_mma0, par_mma0);               // chunk A: columns 0..127
        par_mma0 ^= 1;
        tc_fence_after();
        TRACE(17);
        tmem_ld32_async(tm, bufA);
        tmem_ld_wait32(bufA);
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
          tmem_ld32_async(tm + 64 * j + 32, bufB);
          __nanosleep(0);                            // scheduler yield: lets the other tile's short MLP-chain bursts in (+3 %)
          mixture_pairs<4, !INV>(P, zr, zv, bufA, S_sp2, S_th2, S_f2);
          if (INV) tmem_st32(tm + 64 * j, bufA);
          tmem_ld_wait32(bufB);
          if (j < 3) {
            if (j == 1) {                            // next bufA lives in chunk B: make sure it has landed before loading
              mbar_wait(bar_mma1, par_mma1);
              par_mma1 ^= 1;
              tc_fence_after();
            }
            tmem_ld32_async(tm + 64 * j + 64, bufA);
          }
          mixture_pairs<4, !INV>(P, zr, zv, bufB, S_sp2, S_th2, S_f2);
          if (INV) tmem_st32(tm + 64 * j + 32, bufB);
          if (j < 3) tmem_ld_wait32(bufA);
        }
      }
      TRACE(18);
      TRACE(19);
      // W4 is dead once both chunks of BOTH tiles have completed; the aux buffer once both tiles are past their first layer
      if (elected) {
        if ((atomicAdd(&s_cnt[3], 1) & 1) && step + 1 < total_steps) load_piece(mob_n1, 3, 0);
        if ((atomicAdd(&s_cnt[4], 1) & 1) && step + 2 < total_steps) load_piece(mob_n2, 4, abuf);
      }
      float nx[3], nz[3];
      const float S_sp = hsum(S_sp2);
      if (!INV) {
        const float S_th = hsum(S_th2), S_f = hsum(S_f2);
        const float inv_sp = rcp_nr(S_sp);
        circle_point_fast(P.r, P.v, mixture_angle(S_th, inv_sp), nx);
        ldj += log_fast(S_f * inv_sp);
      } else {
        // target angle of the given column in its own frame (flow/mobiusflow.py:157-167); ~pi by construction
        float ys = atan2f(zv, zr);
        ys = ys >= 0.0f ? ys : ys + kTwoPi;
        if (fabsf(ys - kTwoPi) < 1e-4f) ys = 0.0f;
        // BinFind.forward (flow/mobiusflow.py:196-224): bracket [pi/2, 3pi/2], 15 halvings, return the last probe.
        // One evaluation of  F(t) = sum_k weight_k theta_k(z(t)) / sum_k weight_k - ys  (and, DERIV, of F') streams the row's
        // 256 prepared parameters from its TMEM lane.
        auto probe = [&](float t, float& dF) -> float {
          float sn, cs;
          sincos_2pi(t, sn, cs);
          f32x2 Fs2 = 0ull, Sf2 = 0ull;
          float bufA[32], bufB[32];
          tmem_ld32_async(tm, bufA);
          tmem_ld_wait32(bufA);
#pragma unroll 1
          for (int j = 0; j < 4; ++j) {
            tmem_ld32_async(tm + 64 * j + 32, bufB);
            probe_delta_pairs<4, RNF_INV_NEWTON != 0>(cs, sn, bufA, Fs2, Sf2);
            tmem_ld_wait32(bufB);
            if (j < 3) tmem_ld32_async(tm + 64 * j + 64, bufA);
            probe_delta_pairs<4, RNF_INV_NEWTON != 0>(cs, sn, bufB, Fs2, Sf2);
            if (j < 3) tmem_ld_wait32(bufA);
          }
          dF = hsum(Sf2) / S_sp;
          return fmaf(2.0f, hsum(Fs2) / S_sp, t) - ys;  // sum_k pi_k theta_k = t + 2 sum_k pi_k delta_k
        };
        float lo = kPi / 2.0f, hi = 1.5f * kPi, x0 = 0.0f;
        int n_eval = 0;                               // evaluations of F by this warp in this layer (measurement hook)
#if RNF_INV_NEWTON
        // The 15 sign tests of the reference are tests of x0 against the root t* of F: every theta_k(t) is an increasing circle
        // map that stays within +-2 asin(0.7) of t (|w'| < 0.7), so on the bracket F is continuous and strictly increasing
        // (F' = sum_k weight_k f_k / sum_k weight_k in [0.17, 5.7]) and  F(x0) < 0  <=>  x0 < t*.  So: find t* with a safeguarded
        // Newton iteration (3-4 evaluations instead of 15), then replay the reference's halving arithmetic with the sign of
        // x0 - t*.  Where that sign is not certain -- the predicted |F(x0)| = F'(t*) |x0 - t*| is below 2e-6, i.e. within the
        // fp32 evaluation noise of F, a region where the reference's own decision is rounding noise too -- x0 is evaluated
        // explicitly with the reference's arithmetic, exactly as the plain bisection would.  At most one dyadic probe per row can be
        // that close (their spacing is pi / 2^15 = 9.6e-5 at the last level).
        constexpr float kAmbBand = 1e-6f;             // replay: |predicted F(x0)| below which the sign is taken from an explicit evaluation
        float ts = kPi, dFs = 1.0f;                   // root estimate and slope there
        bool newton_ok = false;
        {
          float a_ = lo, b_ = hi;
          bool conv = false;
          float prev = 0.0f;                          // |Newton step| of the previous iteration (0: none, or a bisection step)
#pragma unroll 1
          for (int it = 0; it < 10; ++it) {
            float dF;
            const float F = probe(ts, dF);
            ++n_eval;
            if (!conv) {
              if (F < 0.0f) a_ = ts; else b_ = ts;
              dFs = dF;
              const float step = F / dF;
              const float as = fabsf(step);
              conv = as < 1e-5f;                        // quadratic convergence: the error after this step is ~step^2
              // ... and how far "~" is can be read off the last two steps: e_{k+1} = C e_k^2 with C = |F''/2F'| ~ |s_k| / s_{k-1}^2
              // once the iteration contracts (s_k = e_k up to the much smaller e_{k+1}).  Stop as soon as the error PREDICTED after
              // this step is below 5e-8 -- the fp32 evaluation noise of F keeps t* from being better than ~1e-7 anyway, and the
              // replay below evaluates explicitly whenever a midpoint is within 2e-6 / F' >= 3.5e-7 of t*.  Saves the evaluation
              // whose only result would be "the step is now below 1e-5" (typically the fourth).
              if (prev > 0.0f && as < 1e-2f) conv = conv || fmaxf(as / (prev * prev), 2.0f) * as * as < 5e-8f;
              float tn = ts - step;
              prev = as;
              if (!conv && !(tn > a_ && tn < b_)) { tn = 0.5f * (a_ + b_); prev = 0.0f; }
              ts = tn;
            }
            if (__all_sync(0xffffffffu, conv)) { newton_ok = true; break; }
          }
        }
        if (newton_ok) {
#pragma unroll 1
          for (int it = 0; it < 15; ++it) {
            x0 = (lo + hi) / 2.0f;
            const float d = x0 - ts;
            const bool amb = fabsf(d) * dFs < kAmbBand;
            bool neg = d < 0.0f;
            if (__any_sync(0xffffffffu, amb)) {
              float dF;
              const float fx0 = probe(x0, dF);
              ++n_eval;
              if (amb) neg = fx0 < 0.0f;
            }
            const float half_w = (hi - lo) / 2.0f;
            if (neg) lo = lo + half_w;
            else hi = hi - half_w;
          }
        } else
#endif
        {
#pragma unroll 1
          for (int it = 0; it < 15; ++it) {
            x0 = (lo + hi) / 2.0f;
            float dF;
            const float fx0 = probe(x0, dF);
            ++n_eval;
            const float half_w = (hi - lo) / 2.0f;
            if (fx0 < 0.0f) lo = lo + half_w;
            else if (fx0 >= 0.0f) hi = hi - half_w;
          }
        }
        if (a.probe_counter != nullptr && lane == 0) atomicAdd(a.probe_counter, 32ull * (unsigned long long)n_eval);
        float sn, cs;
        sincos_2pi(x0, sn, cs);
        nx[0] = fmaf(P.v[0], sn, P.r[0] * cs);
        nx[1] = fmaf(P.v[1], sn, P.r[1] * cs);
        nx[2] = fmaf(P.v[2], sn, P.r[2] * cs);
        f32x2 Sf2 = 0ull;
#pragma unroll 1
        for (int q = 0; q < 8; ++q) {
          float prm[32];
          tmem_ld32(tm + 32 * q, prm);
          jacobian_pairs<4>(cs, sn, prm, Sf2);
        }
        ldj -= log_fast(hsum(Sf2) / S_sp);
      }
      cross3(nx, y, nz);
      normalize3_fast(nz);
      set_col(R, p0, nx);
      set_col(R, p2, nz);
      TRACE(20);
      tc_fence_before();                             // my TMEM reads of this layer are ordered before the next layer's barrier
      ++step;
      mob_cur = mob_n1;
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
      float bv = lp;
      long long bi = valid ? (long long)g : 0x7fffffffffffffffLL;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      if (lane == 0) { s_v[w4] = bv; s_i[w4] = bi; }
      named_bar(3 + tile, 128);
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
      named_bar(3 + tile, 128);
      if (lane == 0) { s_v[w4] = e; s_v[4 + w4] = ed; }
      named_bar(3 + tile, 128);
      if (rowi == 0) {
        const float s = (s_v[0] + s_v[1]) + (s_v[2] + s_v[3]);
        float* p = a.part + tile_idx * kPartStride;
        p[0] = m;
        p[1] = s;
        p[4] = (s_v[4] + s_v[5]) + (s_v[6] + s_v[7]);
        p[2] = __int_as_float((int)(bi & 0xffffffffLL));
        p[3] = __int_as_float((int)(bi >> 32));
      }
      named_bar(3 + tile, 128);
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

bool flow_tc_supported(const rnf_flow* f) {
  for (int i = 0; i < f->model.n_layers; ++i)
    if (f->layers_host[i].kind == RNF_LAYER_MOBIUS && f->layers_host[i].w_off_tc < 0) return false;
  return true;
}

cudaError_t launch_flow_row(const FlowArgs& a, bool inverse, int sm_count, cudaStream_t st) {
  const bool grid_mode = a.G > 0;
  void (*kern)(const FlowArgs) = grid_mode ? flow_row_kernel<false, true>
                                           : (inverse ? flow_row_kernel<true, false> : flow_row_kernel<false, false>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemAlloc);
  if (e != cudaSuccess) return e;
  if (a.n_tiles <= 0) return cudaSuccess;
  const int64_t pairs = (a.n_tiles + 1) / 2;
  const int64_t grid = pairs < sm_count ? pairs : sm_count;
  kern<<<(unsigned)grid, kThreads, kSmemAlloc, st>>>(a);
  return cudaGetLastError();
}

}  // namespace rnf
