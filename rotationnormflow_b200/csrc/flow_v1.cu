// flow_v1.cu -- the exact-precision (FP32 CUDA-core) fused flow kernel for sm_100a.
//
// One thread owns one rotation: its 3x3 matrix and running log|det J| stay in registers across the whole
// layer stack (Flow.forward flow/flow.py:53-72, Flow.inverse flow/flow.py:74-92).  One CTA = 256 rotations.
// Per Mobius layer the CTA stages that layer's conditioner (117.5 KB, packed layout in rnf_common.cuh) in shared
// memory once; every thread then runs the 4-layer MLP (flow/condition.py:24-30) for its own rotation with
// warp-broadcast LDS.128 weight reads and a private activation column in shared memory, consumes the 256
// outputs 16 mixture components at a time (never materialised), and applies the Mobius mixture
// (flow/mobiusflow.py:46-125) or, for the inverse, the 15-step bisection (flow/mobiusflow.py:127-224).
// Quaternion affine / rotation layers (flow/squeezetrans.py:33-38, flow/rottrans.py:8-66) are ~100 flops in
// registers.  HBM traffic: 36 B in + 40 B out per rotation (grid mode: 36 B per grid rotation per image tile).
//
// This is the precision reference of the library (mlp_mode = RNF_MLP_FP32); the tensor-core path lives in
// flow_t4.cu / flow_row.cu and is validated against this one and against the CPU oracle.
#include "mobius_math.cuh"
#include "rnf_common.cuh"
#include "ablation_layers.cuh"

namespace rnf {

namespace {

constexpr int T = kV1Threads;                      // rotations per CTA
constexpr int kSmemFloats = kMobFloats + kH * T;   // weights + private activation columns
constexpr int kScratchPerCta = 4 * kK * T;         // inverse: (w.x, w.y, w.z, softplus) per component per thread

// first conditioner layer for output j: W0[j,:3].y + b0[j] (+ hoisted per-image W_f.feature)
__device__ __forceinline__ float first_layer(const float4* sFirst, const float* cimg, int j, const float y[3]) {
  const float4 f = sFirst[j];
  float h = fmaf(f.z, y[2], fmaf(f.y, y[1], fmaf(f.x, y[0], f.w)));
  if (cimg != nullptr) h += __ldg(cimg + j);
  return h;
}

// acc[0..63] += sum_k act[k] * Wt[k][col0 + 0..63]   (Wt row stride = ld floats)
__device__ __forceinline__ void gemv64(float acc[64], const float* __restrict__ Wt, int ld, const float* __restrict__ act) {
#pragma unroll 2
  for (int k = 0; k < kH; ++k) {
    const float a = act[k * T];
    const float4* w4 = reinterpret_cast<const float4*>(Wt + k * ld);
#pragma unroll
    for (int j4 = 0; j4 < 16; ++j4) {
      const float4 w = w4[j4];
      acc[4 * j4 + 0] = fmaf(a, w.x, acc[4 * j4 + 0]);
      acc[4 * j4 + 1] = fmaf(a, w.y, acc[4 * j4 + 1]);
      acc[4 * j4 + 2] = fmaf(a, w.z, acc[4 * j4 + 2]);
      acc[4 * j4 + 3] = fmaf(a, w.w, acc[4 * j4 + 3]);
    }
  }
}

template <bool INV>
__device__ __forceinline__ void mobius_layer(const float* __restrict__ sW, float* __restrict__ sAct, int perm,
                                             const float* cimg, float* __restrict__ scratch, float R[9], float& ldj) {
  const int p0 = perm, p1 = (perm + 1) % 3, p2 = (perm + 2) % 3;
  float x[3], y[3], r[3], v[3];
  get_col(R, p0, x);
  get_col(R, p1, y);
  make_frame(x, y, r, v);

  float* act = sAct + threadIdx.x;
  const float4* sFirst = reinterpret_cast<const float4*>(sW + kMobFirst);

  // ---- conditioner MLP (flow/condition.py:24-30) ----
#pragma unroll 8
  for (int j = 0; j < kH; ++j) act[j * T] = fmaxf(first_layer(sFirst, cimg, j, y), 0.0f);

#pragma unroll 1
  for (int l = 0; l < 3; ++l) {
    const float* Wt = sW + kMobHid + l * kMobHidStride;
    const float* bias = Wt + kH * kH;
    float acc[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) acc[j] = bias[j];
    gemv64(acc, Wt, kH, act);
    if (l < 2) {
#pragma unroll
      for (int j = 0; j < 64; ++j) act[j * T] = fmaxf(acc[j], 0.0f);
    } else {
#pragma unroll
      for (int j = 0; j < 64; ++j) act[j * T] = fmaxf(acc[j] + first_layer(sFirst, cimg, j, y), 0.0f);  // relu(x0 + x)
    }
  }

  // ---- fc_last, 16 mixture components at a time; outputs are consumed from registers ----
  float S_sp = 0.0f, S_th = 0.0f, S_f = 0.0f;
  const float* Wl = sW + kMobLast;
  const float* bl = Wl + kH * 4 * kK;
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    float acc[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) acc[j] = bl[c * 64 + j];
    gemv64(acc, Wl + c * 64, 4 * kK, act);
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const float sp = softplus_torch(acc[4 * q]);
      float w[3] = {acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]};
      comp_prep(w, y);
      S_sp += sp;
      if (!INV) {
        float th, f;
        comp_eval(x, w, r, v, th, f);
        S_th = fmaf(sp, th, S_th);
        S_f = fmaf(sp, f, S_f);
      } else {
        float* s = scratch + (4 * (c * 16 + q)) * T;
        s[0] = w[0]; s[T] = w[1]; s[2 * T] = w[2]; s[3 * T] = sp;
      }
    }
  }

  float nx[3];
  if (!INV) {
    circle_point(r, v, S_th / S_sp, nx);                      // tx = r cos(theta') + v sin(theta')
    ldj += logf(S_f / S_sp);
  } else {
    // target angle of the given column in its own frame (flow/mobiusflow.py:157-167); ~pi by construction
    float ys = atan2f(dot3(x, v), dot3(x, r));
    ys = ys >= 0.0f ? ys : ys + kTwoPi;
    if (fabsf(ys - kTwoPi) < 1e-4f) ys = 0.0f;
    // BinFind.forward (flow/mobiusflow.py:196-224): bracket [pi/2, 3pi/2], 15 halvings, return the last probe
    float lo = kPi / 2.0f, hi = 1.5f * kPi, x0 = 0.0f;
#pragma unroll 1
    for (int it = 0; it < 15; ++it) {
      x0 = (lo + hi) / 2.0f;
      float z[3];
      circle_point(r, v, x0, z);
      float Fs = 0.0f;
#pragma unroll 4
      for (int k = 0; k < kK; ++k) {
        const float* s = scratch + 4 * k * T;
        const float w[3] = {s[0], s[T], s[2 * T]};
        float th, f;
        comp_eval(z, w, r, v, th, f);
        Fs = fmaf(s[3 * T], th, Fs);
      }
      const float fx0 = Fs / S_sp - ys;
      const float half = (hi - lo) / 2.0f;
      if (fx0 < 0.0f) lo = lo + half;
      else if (fx0 >= 0.0f) hi = hi - half;
    }
    circle_point(r, v, x0, nx);
#pragma unroll 4
    for (int k = 0; k < kK; ++k) {
      const float* s = scratch + 4 * k * T;
      const float w[3] = {s[0], s[T], s[2 * T]};
      float th, f;
      comp_eval(nx, w, r, v, th, f);
      S_f = fmaf(s[3 * T], f, S_f);
    }
    ldj -= logf(S_f / S_sp);
  }
  float nz[3];
  cross3(nx, y, nz);                                          // cyclic permutations only (SURVEY.md a4)
  normalize3(nz);
  set_col(R, p0, nx);
  set_col(R, p2, nz);
}

template <bool INV, bool GRID>
__global__ void __launch_bounds__(T, 1) flow_v1_kernel(const FlowArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* sW = smem;
  float* sAct = smem + kMobFloats;
  __shared__ float s_red_v[T / 32];
  __shared__ float s_red_d[T / 32];
  __shared__ long long s_red_i[T / 32];
  __shared__ float s_bcast;
  const int tid = threadIdx.x;
  float* scratch = INV ? a.scratch + (size_t)blockIdx.x * kScratchPerCta + tid : nullptr;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    int64_t row, img = 0, g = 0;
    bool valid;
    float R[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
    if (GRID) {
      img = tile / a.tiles_per_image;
      g = (tile % a.tiles_per_image) * T + tid;
      valid = g < a.G;
      row = img * a.G + g;
      if (valid) {
        float Gm[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) Gm[i] = __ldg(a.R_in + g * 9 + i);
        if (a.offset != nullptr) {                             // samples = grid @ random_rot (eval.py:439-440)
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
      row = tile * T + tid;
      valid = row < a.N;
      if (valid) {
#pragma unroll
        for (int i = 0; i < 9; ++i) R[i] = __ldg(a.R_in + row * 9 + i);
        if (a.cond != nullptr) img = a.feat_index != nullptr ? (int64_t)__ldg(a.feat_index + row) : row / a.rows_per_image;
      }
    }
    const float* cond_img = a.cond != nullptr ? a.cond + img * a.cond_stride : nullptr;
    float ldj = 0.0f;
    float dgt = 0.0f;                                  // spread metric: angle of the evaluation point to the image's ground truth
    if (GRID && a.gt != nullptr && valid) dgt = gt_distance(a.gt + img * a.gt_k * 9, a.gt_k, R);

#pragma unroll 1
    for (int step = 0; step < a.n_layers; ++step) {
      const int li = INV ? a.n_layers - 1 - step : step;
      const LayerDev L = a.layers[li];
      if (L.kind == RNF_LAYER_MOBIUS) {
        __syncthreads();                                      // previous users of sW are done
        const float4* src = reinterpret_cast<const float4*>(a.weights + L.w_off);
        float4* dst = reinterpret_cast<float4*>(sW);
        for (int i = tid; i < kMobFloats / 4; i += T) dst[i] = __ldg(src + i);
        __syncthreads();
        const float* cimg = (L.cond_slot >= 0 && cond_img != nullptr) ? cond_img + (int64_t)L.cond_slot * kH : nullptr;
        mobius_layer<INV>(sW, sAct, L.perm, cimg, scratch, R, ldj);
      } else {
        const float* W = L.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)L.cond_slot * kAffFloats
                                          : a.weights + L.w_off;
        if (INV) W += kAffInv;
        affine_family_layer<false>(L, W, R, ldj);
      }
    }

    if (!GRID) {
      if (valid) {
#pragma unroll
        for (int i = 0; i < 9; ++i) a.R_out[row * 9 + i] = R[i];
        a.ldj_out[row] = ldj;
      }
    } else {
      float lp = ldj;
      if (a.fisher_A != nullptr) {                             // MatrixFisherN._log_prob (utils/fisher.py:217-232)
        float tr = 0.0f;
#pragma unroll
        for (int i = 0; i < 9; ++i) tr = fmaf(__ldg(a.fisher_A + img * 9 + i), R[i], tr);
        lp += tr - __ldg(a.fisher_c + img);
      }
      if (!valid) lp = -INFINITY;
      if (a.logp_out != nullptr && valid) a.logp_out[row] = lp;
      if (a.R_out != nullptr && valid) {
#pragma unroll
        for (int i = 0; i < 9; ++i) a.R_out[row * 9 + i] = R[i];
      }
      // per-tile (max, first arg-max, sum exp(lp - max))
      float bv = lp;
      long long bi = valid ? (long long)g : 0x7fffffffffffffffLL;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      __syncthreads();
      if ((tid & 31) == 0) { s_red_v[tid >> 5] = bv; s_red_i[tid >> 5] = bi; }
      __syncthreads();
      if (tid < 32) {
        bv = tid < T / 32 ? s_red_v[tid] : -INFINITY;
        bi = tid < T / 32 ? s_red_i[tid] : 0x7fffffffffffffffLL;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (tid == 0) { s_bcast = bv; s_red_i[0] = bi; }
      }
      __syncthreads();
      const float m = s_bcast;
      const long long mi = s_red_i[0];
      float e = (valid && m != -INFINITY) ? expf(lp - m) : 0.0f;
      float ed = e * dgt;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        e += __shfl_xor_sync(0xffffffffu, e, o);
        ed += __shfl_xor_sync(0xffffffffu, ed, o);
      }
      __syncthreads();
      if ((tid & 31) == 0) { s_red_v[tid >> 5] = e; s_red_d[tid >> 5] = ed; }
      __syncthreads();
      if (tid == 0) {
        float s = 0.0f, sd = 0.0f;
#pragma unroll
        for (int w = 0; w < T / 32; ++w) { s += s_red_v[w]; sd += s_red_d[w]; }
        float* p = a.part + tile * kPartStride;
        p[0] = m;
        p[1] = s;
        p[4] = sd;
        p[2] = __int_as_float((int)(mi & 0xffffffffLL));
        p[3] = __int_as_float((int)(mi >> 32));
      }
    }
  }
}

// One CTA per image: fold the per-tile partials in tile (= increasing grid index) order.
__global__ void grid_combine_kernel(const float* __restrict__ part, int64_t tiles_per_image, int64_t g_index0,
                                    float* __restrict__ max_out, int64_t* __restrict__ argmax_out,
                                    float* __restrict__ sumexp_out, float* __restrict__ spread_num_out) {
  const int64_t b = blockIdx.x;
  const float* p = part + b * tiles_per_image * kPartStride;
  __shared__ float s_v[32];
  __shared__ long long s_i[32];
  __shared__ float s_m;
  const int tid = threadIdx.x;
  float bv = -INFINITY;
  long long bi = 0x7fffffffffffffffLL;
  for (int64_t t = tid; t < tiles_per_image; t += blockDim.x) {
    const float v = p[t * kPartStride];
    const long long i = ((long long)(unsigned)__float_as_int(p[t * kPartStride + 2])) | ((long long)__float_as_int(p[t * kPartStride + 3]) << 32);
    if (grid_red_better(v, i, bv, bi)) { bv = v; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
  }
  if ((tid & 31) == 0) { s_v[tid >> 5] = bv; s_i[tid >> 5] = bi; }
  __syncthreads();
  if (tid < 32) {
    const int nw = blockDim.x >> 5;
    bv = tid < nw ? s_v[tid] : -INFINITY;
    bi = tid < nw ? s_i[tid] : 0x7fffffffffffffffLL;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (tid == 0) { s_m = bv; s_i[0] = bi; }
  }
  __syncthreads();
  const float m = s_m;
  float s = 0.0f, sd = 0.0f;
  for (int64_t t = tid; t < tiles_per_image; t += blockDim.x) {
    const float v = p[t * kPartStride];
    if (v != -INFINITY) {                 // a NaN tile maximum makes the sum NaN
      const float w = expf(v - m);
      s += p[t * kPartStride + 1] * w;
      sd += p[t * kPartStride + 4] * w;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    sd += __shfl_xor_sync(0xffffffffu, sd, o);
  }
  __syncthreads();
  __shared__ float s_d[32];
  if ((tid & 31) == 0) { s_v[tid >> 5] = s; s_d[tid >> 5] = sd; }
  __syncthreads();
  if (tid == 0) {
    float tot = 0.0f, totd = 0.0f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { tot += s_v[w]; totd += s_d[w]; }
    max_out[b] = m;
    argmax_out[b] = (int64_t)s_i[0] + g_index0;
    sumexp_out[b] = tot;
    if (spread_num_out != nullptr) spread_num_out[b] = totd;       // sum_g exp(logp_g - max) d(R_g, R_gt)
  }
}

}  // namespace

cudaError_t launch_flow_v1(const FlowArgs& a, bool inverse, int sm_count, cudaStream_t st) {
  const size_t smem = (size_t)kSmemFloats * sizeof(float);
  const bool grid_mode = a.G > 0;
  void (*kern)(const FlowArgs) = nullptr;
  if (grid_mode) kern = flow_v1_kernel<false, true>;
  else kern = inverse ? flow_v1_kernel<true, false> : flow_v1_kernel<false, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (a.n_tiles <= 0) return cudaSuccess;
  const int64_t grid = a.n_tiles < sm_count ? a.n_tiles : sm_count;
  kern<<<(unsigned)grid, T, smem, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_grid_combine(const float* part, int64_t tiles_per_image, int64_t B, int64_t g_index0, float* max_out,
                                int64_t* argmax_out, float* sumexp_out, float* spread_num_out, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  grid_combine_kernel<<<(unsigned)B, 256, 0, st>>>(part, tiles_per_image, g_index0, max_out, argmax_out, sumexp_out, spread_num_out);
  return cudaGetLastError();
}

}  // namespace rnf
