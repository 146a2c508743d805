// flow_grad.cu -- log p(R) of the forward direction AND its tangential rotation gradient in one launch (FP32 CUDA cores, sm_100a).
//
// What it evaluates, per row n (the nll_grad refinement of eval.py:464-480 climbs this):
//   logp[n] = ldj(R_n) [+ sum(A_b * R'_n) - c_b]                    Flow.forward (flow/flow.py:53-72) + MatrixFisherN._log_prob
//   G[n]    = R_n [g]x / 2,  g = vee(R_n^T d logp / dR_n)           the tangential gradient, convention of train_ops.cu
//
// Layout: ONE WARP PER ROTATION, several warps per CTA.  The refinement batch is one row per image (tens to ~1 k rows): a warp
// per row spreads that over the machine where a thread per row would occupy a handful of SMs.  Lane j owns hidden units j and
// j + 32 of the conditioner MLP (flow/condition.py:24-30) and mixture components j and j + 32 (fc_last outputs 4j..4j+3 and
// 4(j+32)..; lane-contiguous float4 reads, conflict-free); sums over components are warp shuffles; frames and columns are
// computed redundantly by every lane.  Per Mobius layer the CTA stages the packed FP32 image (rnf_common.cuh, 117.5 KB, the one
// flow_v1.cu reads) in shared memory once, single-buffered.
//
// Two sweeps:
//   forward : layers 0..L-1 as flow_v1.cu does; each layer's input rotation goes to the warp's shared-memory history
//             (9 floats per layer), log-dets accumulate, the matrix-Fisher term is added at the end.
//   reverse : g = tangent_of(R_L, A_b) (0 without a base term), g_ldj = 1.  For l = L-1..0 the layer's forward is recomputed
//             from R_l (the lane keeps its pre-activations for the ReLU masks), then its vector-Jacobian product is applied:
//               Mobius : the forward-direction formulas of mobius_mixture_bwd_kernel<false> (train_ops.cu) give g <- M g' + c1 + c2
//                        and dL/d(conditioner output)[256] (per-warp shared memory); the MLP backward reads the same staged weights
//                        transposed (row-skewed so that the 32 lanes hit 32 banks), the residual relu(h0 + h3) feeds h0
//                        (flow/condition.py:29), and g_y = W0[:, :3]^T g_h0 enters through the conditioner input y = R[:, p1]
//                        as tangent_of(R_l, g_y e_p1^T) -- what autograd of the slice contributes in the composed path.  The
//                        feature part of fc_first gets no gradient (this is a rotation gradient).
//               affine : quat_affine_bwd_kernel (train_ops.cu) with g_loglen = -4 g_ldj (has_ldj) or 0 (rotation layers,
//                        flow/rottrans.py:21); W is the forward block of the packed or per-image affine block.
//           Finally G = gradient_from_tangent(R_0, g).
// No global scratch, no host synchronisation, one launch: capturable in a CUDA graph.
//
// Training (flow_train_kernel, Flow.log_prob): the same layer functions with TRAIN = true.  Forward mode writes R' and ldj.  Backward
// mode reruns the forward sweep with history and the reverse sweep seeded by the caller's dL/dR' and dL/dldj per row; it writes the
// tangential dL/dR and, per (layer, row), a training record (kTws* below; dL/dW of the 4x4 for an affine layer).  The weights come
// from a buffer passed per call, so a training step never re-packs on the host; the weight gradients are GEMMs over the records
// (engine.TrainProgram.backward).
#include "mobius_math.cuh"
#include "rnf_common.cuh"

namespace rnf {

namespace {

constexpr int kWarpFloats = kH + 4 * kK;            // per-warp activation / gradient vector [64] + conditioner-output gradient [256]

// Training record of one (Mobius layer, row), kTwsFloats floats, rows of a layer contiguous ([layer][row][kTwsFloats]):
//   kTwsY    (y, 1)                                    input of fc_first's y columns and bias
//   kTwsAct  relu(h0), relu(h1), relu(h2), relu(h0+h3)  inputs of layers.1, .3, .5 and fc_last
//   kTwsGrad gh0 (residual included), gp1, gp2, gp3     gradients of the pre-activations h0 .. h3
//   kTwsGout dL/d(fc_last output) [256]                 packed order (component c at 4c..4c+3)
constexpr int kTwsY = 0, kTwsAct = 4, kTwsGrad = kTwsAct + 4 * kH, kTwsGout = kTwsGrad + 4 * kH;
constexpr int kTwsFloats = kTwsGout + 4 * kK;       // 772

struct GradArgs {
  const float* weights;
  const LayerDev* layers;
  int n_layers;
  int n_mobius_slots;
  const float* R_in;
  int64_t N;
  const float* cond;
  int64_t cond_stride;
  const int32_t* feat_index;
  int64_t rows_per_image;
  const float* fisher_A;
  const float* fisher_c;
  float* logp_out;
  float* grad_out;
  int64_t n_tiles;
  int warp_floats;                                  // kWarpFloats + history, rounded up to a multiple of 4
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// column p of R as a loop over rows; so3_math.cuh's get_col gives these kernels different SASS, so they keep this form
__device__ __forceinline__ void col_of(const float R[9], int p, float o[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) o[i] = sel3(p, R[3 * i], R[3 * i + 1], R[3 * i + 2]);
}

// One Mobius layer for the warp's rotation: recomputes the conditioner with the lane's pre-activations kept (units lane, lane+32),
// the mixture, and -- if BWD -- applies the VJP to the tangent gradient g (at the layer's output) in place.
// TRAIN (with BWD): the log-det terms are scaled by gl = dL/dldj of the row, and the row's record of the five linear layers goes
// to tws (kTws* layout below): their inputs and the gradients of their pre-activations, from which the weight gradients are GEMMs.
template <bool BWD, bool TRAIN = false>
__device__ __forceinline__ void mobius_layer(const float* __restrict__ sW, float* __restrict__ wbuf, const float* cimg, int p0,
                                             float R[9], float& ldj, float g[3], float gl = 1.0f, float* __restrict__ tws = nullptr) {
  const int lane = threadIdx.x & 31;
  const int p1 = (p0 + 1) % 3, p2 = (p0 + 2) % 3;
  float x[3], y[3], z[3], r[3], v[3];
  col_of(R, p0, x);
  col_of(R, p1, y);
  col_of(R, p2, z);
  make_frame(x, y, r, v);
  float* act = wbuf;                                     // [64]
  float* gout = wbuf + kH;                               // [256], packed fc_last order
  const float4* sFirst = reinterpret_cast<const float4*>(sW + kMobFirst);

  // ---- conditioner MLP forward (flow/condition.py:24-30), pre-activations of the lane's two units kept ----
  float h0[2], h1[2], h2[2], h3[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int j = lane + 32 * u;
    const float4 f = sFirst[j];
    float h = fmaf(f.z, y[2], fmaf(f.y, y[1], fmaf(f.x, y[0], f.w)));
    if (cimg != nullptr) h += __ldg(cimg + j);
    h0[u] = h;
  }
  __syncwarp();
  act[lane] = fmaxf(h0[0], 0.0f);
  act[lane + 32] = fmaxf(h0[1], 0.0f);
  if (TRAIN) {
    if (lane < 4) tws[kTwsY + lane] = lane < 3 ? sel3(lane, y[0], y[1], y[2]) : 1.0f;      // (y, 1): fc_first's weights and bias
    tws[kTwsAct + lane] = act[lane];
    tws[kTwsAct + lane + 32] = act[lane + 32];
  }
  __syncwarp();
#pragma unroll                                               // (static indices keep h1..h3 in registers)
  for (int l = 0; l < 3; ++l) {
    const float* Wt = sW + kMobHid + l * kMobHidStride;        // [k][j]
    float a0 = Wt[kH * kH + lane], a1 = Wt[kH * kH + lane + 32];
#pragma unroll 8
    for (int k = 0; k < kH; ++k) {
      const float a = act[k];
      a0 = fmaf(Wt[k * kH + lane], a, a0);
      a1 = fmaf(Wt[k * kH + lane + 32], a, a1);
    }
    float* hl = l == 0 ? h1 : (l == 1 ? h2 : h3);
    hl[0] = a0;
    hl[1] = a1;
    __syncwarp();
    if (l < 2) { act[lane] = fmaxf(a0, 0.0f); act[lane + 32] = fmaxf(a1, 0.0f); }
    else { act[lane] = fmaxf(h0[0] + a0, 0.0f); act[lane + 32] = fmaxf(h0[1] + a1, 0.0f); }      // relu(x0 + x)
    if (TRAIN) {
      tws[kTwsAct + kH * (l + 1) + lane] = act[lane];
      tws[kTwsAct + kH * (l + 1) + lane + 32] = act[lane + 32];
    }
    __syncwarp();
  }

  // ---- fc_last for components lane and lane + 32 ----
  const float* Wl = sW + kMobLast;                             // [k][256]
  const float* bl = Wl + kH * 4 * kK;
  float o[2][4];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const float4 b = reinterpret_cast<const float4*>(bl)[lane + 32 * u];
    o[u][0] = b.x; o[u][1] = b.y; o[u][2] = b.z; o[u][3] = b.w;
  }
#pragma unroll 4
  for (int k = 0; k < kH; ++k) {
    const float a = act[k];
    const float4* w4 = reinterpret_cast<const float4*>(Wl + k * 4 * kK);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float4 w = w4[lane + 32 * u];
      o[u][0] = fmaf(w.x, a, o[u][0]);
      o[u][1] = fmaf(w.y, a, o[u][1]);
      o[u][2] = fmaf(w.z, a, o[u][2]);
      o[u][3] = fmaf(w.w, a, o[u][3]);
    }
  }

  // ---- Mobius mixture (flow/mobiusflow.py:58-85), the 2-D form of train_ops.cu ----
  const float cz = dot3(x, r), sz = dot3(x, v);
  float al[2], be[2], nn[2], sc[2], alp[2], bep[2], sp[2], th[2], f[2];
  float S = 0.0f, Sth = 0.0f, Sf = 0.0f;
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const float w[3] = {o[u][1], o[u][2], o[u][3]};
    al[u] = dot3(w, r);                                      // the projection (I - y y^T) w leaves these unchanged
    be[u] = dot3(w, v);
    nn[u] = sqrtf(fmaf(be[u], be[u], al[u] * al[u]));
    sc[u] = 0.7f / (1.0f + nn[u]);
    alp[u] = sc[u] * al[u];
    bep[u] = sc[u] * be[u];
    sp[u] = softplus_torch(o[u][0]);
    const float X = cz - alp[u], Y = sz - bep[u];
    const float D2 = fmaf(Y, Y, X * X);
    const float om = 1.0f - fmaf(bep[u], bep[u], alp[u] * alp[u]);
    f[u] = om / D2;
    const float t = atan2f(fmaf(f[u], Y, -bep[u]), fmaf(f[u], X, -alp[u]));
    th[u] = t >= 0.0f ? t : t + kTwoPi;
    S += sp[u];
    Sth = fmaf(sp[u], th[u], Sth);
    Sf = fmaf(sp[u], f[u], Sf);
  }
  S = warp_sum(S);
  Sth = warp_sum(Sth);
  Sf = warp_sum(Sf);
  const float Th = Sth / S, Fm = Sf / S;

  if (!BWD) {
    float nx[3], nz[3];
    circle_point(r, v, Th, nx);
    cross3(nx, y, nz);
    normalize3(nz);
    ldj += logf(Fm);
    set_col(R, p0, nx);
    set_col(R, p2, nz);
    return;
  }

  // ---- VJP of the mixture (mobius_mixture_bwd_kernel<false>, g_ldj = 1): R' = R Rot(e_p1, phi) ----
  float Rn[9];
  {
    float nx[3], nz[3];
    circle_point(r, v, Th, nx);
    cross3(nx, y, nz);
    normalize3(nz);
#pragma unroll
    for (int i = 0; i < 9; ++i) Rn[i] = R[i];
    set_col(Rn, p0, nx);
    set_col(Rn, p2, nz);
  }
  const float cG = sel3(p1, g[0], g[1], g[2]), cF = gl / Fm;
  float sA[3] = {0.f, 0.f, 0.f}, sB[3] = {0.f, 0.f, 0.f};
  __syncwarp();
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const float X = cz - alp[u], Y = sz - bep[u];
    const float D2 = fmaf(Y, Y, X * X);
    const float om = 1.0f - fmaf(bep[u], bep[u], alp[u] * alp[u]);
    const float th_ap = 2.0f * Y / D2, th_bp = -2.0f * X / D2;
    const float f_ap = (-2.0f * alp[u] * D2 + 2.0f * om * X) / (D2 * D2);
    const float f_bp = (-2.0f * bep[u] * D2 + 2.0f * om * Y) / (D2 * D2);
    const float t = nn[u] > 1e-30f ? sc[u] / (nn[u] * (1.0f + nn[u])) : 0.0f;
    const float J11 = sc[u] - t * al[u] * al[u], J12 = -t * al[u] * be[u], J22 = sc[u] - t * be[u] * be[u];
    const float th_a = th_ap * J11 + th_bp * J12, th_b = th_ap * J12 + th_bp * J22;
    const float f_a = f_ap * J11 + f_bp * J12, f_b = f_ap * J12 + f_bp * J22;
    const float pi = sp[u] / S;
    const float A = pi * (cG * th_a + cF * f_a);
    const float B = pi * (cG * th_b + cF * f_b);
    const float sig = 1.0f / (1.0f + expf(-o[u][0]));
    float4 go;
    go.x = sig / S * (cG * (th[u] - Th) + cF * (f[u] - Fm));
    go.y = fmaf(B, z[0], -A * x[0]);                           // alpha = w.r = -w.x, beta = w.v = w.z on the manifold
    go.z = fmaf(B, z[1], -A * x[1]);
    go.w = fmaf(B, z[2], -A * x[2]);
    reinterpret_cast<float4*>(gout)[lane + 32 * u] = go;
    if (TRAIN) reinterpret_cast<float4*>(tws + kTwsGout)[lane + 32 * u] = go;
#pragma unroll
    for (int i = 0; i < 3; ++i) { sA[i] = fmaf(A, o[u][1 + i], sA[i]); sB[i] = fmaf(B, o[u][1 + i], sB[i]); }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) { sA[i] = warp_sum(sA[i]); sB[i] = warp_sum(sB[i]); }
  float gn[3];
  {
    float uA[3], uB[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      uA[i] = R[i] * sA[0] + R[3 + i] * sA[1] + R[6 + i] * sA[2];
      uB[i] = R[i] * sB[0] + R[3 + i] * sB[1] + R[6 + i] * sB[2];
    }
    const float e0[3] = {p0 == 0 ? 1.f : 0.f, p0 == 1 ? 1.f : 0.f, p0 == 2 ? 1.f : 0.f};
    const float e2[3] = {p2 == 0 ? 1.f : 0.f, p2 == 1 ? 1.f : 0.f, p2 == 2 ? 1.f : 0.f};
    float nA[3] = {-uA[0], -uA[1], -uA[2]}, c1[3], c2[3];
    cross3(e0, nA, c1);
    cross3(e2, uB, c2);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float m = 0.0f;
#pragma unroll
      for (int j = 0; j < 3; ++j) m = fmaf(R[i] * Rn[j] + R[3 + i] * Rn[3 + j] + R[6 + i] * Rn[6 + j], g[j], m);
      gn[i] = m + c1[i] + c2[i];
    }
  }
  __syncwarp();

  // ---- MLP backward with transposed (row-skewed) reads of the staged weights ----
  float gh0[2], gp[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {                              // g_a3 = W4^T g_out, then the mask of relu(h0 + h3)
    const int k = lane + 32 * u;
    const float* row = Wl + k * 4 * kK;
    float s = 0.0f;
#pragma unroll 8
    for (int t = 0; t < 4 * kK; ++t) {
      const int j = (t + lane) & (4 * kK - 1);
      s = fmaf(row[j], gout[j], s);
    }
    gp[u] = h0[u] + h3[u] > 0.0f ? s : 0.0f;
    gh0[u] = gp[u];                                            // residual path into h0 (flow/condition.py:29)
  }
#pragma unroll
  for (int l = 2; l >= 0; --l) {                              // layers.5, .3, .1: g_in = W^T g_pre, masked by relu of the input
    __syncwarp();
    act[lane] = gp[0];
    act[lane + 32] = gp[1];
    if (TRAIN) {                                               // gradient of the output of layers.{2l+1}: h_{l+1}
      tws[kTwsGrad + kH * (l + 1) + lane] = gp[0];
      tws[kTwsGrad + kH * (l + 1) + lane + 32] = gp[1];
    }
    __syncwarp();
    const float* Wt = sW + kMobHid + l * kMobHidStride;        // Wt[k][j] = W[j][k]
    const float* hin0 = l == 2 ? h2 : (l == 1 ? h1 : h0);
    float s0 = 0.0f, s1 = 0.0f;
    const float* row0 = Wt + lane * kH;
    const float* row1 = Wt + (lane + 32) * kH;
#pragma unroll 8
    for (int t = 0; t < kH; ++t) {
      const int j = (t + lane) & (kH - 1);
      const float gj = act[j];
      s0 = fmaf(row0[j], gj, s0);
      s1 = fmaf(row1[j], gj, s1);
    }
    gp[0] = hin0[0] > 0.0f ? s0 : 0.0f;
    gp[1] = hin0[1] > 0.0f ? s1 : 0.0f;
  }
  gh0[0] += gp[0];
  gh0[1] += gp[1];
  if (TRAIN) {
    tws[kTwsGrad + lane] = gh0[0];
    tws[kTwsGrad + lane + 32] = gh0[1];
  }
  // g_y = W0[:, :3]^T g_h0; the conditioner input y = R[:, p1] adds tangent_of(R, g_y e_p1^T)
  float gy[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const float4 fw = sFirst[lane + 32 * u];
    gy[0] = fmaf(fw.x, gh0[u], gy[0]);
    gy[1] = fmaf(fw.y, gh0[u], gy[1]);
    gy[2] = fmaf(fw.z, gh0[u], gy[2]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) gy[i] = warp_sum(gy[i]);
  float Gy[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  set_col(Gy, p1, gy);
  float ty[3];
  tangent_of(R, Gy, ty);
#pragma unroll
  for (int i = 0; i < 3; ++i) g[i] = gn[i] + ty[i];
  __syncwarp();
}

// calculate_16 (flow/squeezetrans.py:33-38) forward, or its tangent VJP (quat_affine_bwd_kernel) with g_loglen = gL.
// TRAIN (with BWD): gL is scaled by gl = dL/dldj of the row, and lane 0 writes dL/dW = dp q^T (16 floats) to dW.
template <bool BWD, bool TRAIN = false>
__device__ __forceinline__ void affine_layer(const float* __restrict__ W, bool has_ldj, float R[9], float& ldj, float g[3],
                                             float gl = 1.0f, float* __restrict__ dW = nullptr) {
  float Wr[17];
#pragma unroll
  for (int i = 0; i < 17; ++i) Wr[i] = __ldg(W + i);
  if (!BWD) {
    const float loglen = quat_affine(Wr, R);
    if (has_ldj) ldj += Wr[16] - 4.0f * loglen;
    return;
  }
  float q[4], p[4];
  mat_to_quat(R, q);
#pragma unroll
  for (int a = 0; a < 4; ++a) p[a] = fmaf(Wr[4 * a + 3], q[3], fmaf(Wr[4 * a + 2], q[2], fmaf(Wr[4 * a + 1], q[1], Wr[4 * a] * q[0])));
  const float len = sqrtf(p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3]);
  float ph[4], Eg[4], dp[4], Wt[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) ph[a] = p[a] / len;
  E_mul(ph, g, Eg);
  const float gL = has_ldj ? -4.0f * gl : 0.0f;               // d ldj / d log|Wq| (rotation layers: no log-det)
#pragma unroll
  for (int a = 0; a < 4; ++a) dp[a] = (2.0f * Eg[a] + gL * ph[a]) / len;
  if (TRAIN && (threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) dW[4 * a + b] = dp[a] * q[b];
  }
#pragma unroll
  for (int b = 0; b < 4; ++b) Wt[b] = Wr[b] * dp[0] + Wr[4 + b] * dp[1] + Wr[8 + b] * dp[2] + Wr[12 + b] * dp[3];
  ET_mul(q, Wt, g);
#pragma unroll
  for (int i = 0; i < 3; ++i) g[i] *= 0.5f;
}

__global__ void __launch_bounds__(512, 1) flow_grad_kernel(const GradArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* sW = smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_warps = blockDim.x >> 5;
  float* wbuf = smem + kMobFloats + (size_t)warp * a.warp_floats;
  float* hist = wbuf + kWarpFloats;                          // R_0 .. R_L, 9 floats each
  const int L = a.n_layers;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t row = tile * n_warps + warp;
    const bool valid = row < a.N;
    float R[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
    int64_t img = 0;
    if (valid) {
#pragma unroll
      for (int i = 0; i < 9; ++i) R[i] = __ldg(a.R_in + row * 9 + i);
      img = a.feat_index != nullptr ? (int64_t)__ldg(a.feat_index + row) : row / a.rows_per_image;
    }
    const float* cond_img = a.cond != nullptr ? a.cond + img * a.cond_stride : nullptr;
    float ldj = 0.0f;
    float g[3] = {0.f, 0.f, 0.f};

    // ---- forward sweep ----
#pragma unroll 1
    for (int li = 0; li < L; ++li) {
      const LayerDev Ld = a.layers[li];
      if (valid && lane < 9) hist[9 * li + lane] = R[lane];
      if (Ld.kind == RNF_LAYER_MOBIUS) {
        __syncthreads();
        const float4* src = reinterpret_cast<const float4*>(a.weights + Ld.w_off);
        float4* dst = reinterpret_cast<float4*>(sW);
        for (int i = threadIdx.x; i < kMobFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
        __syncthreads();
        if (valid) {
          const float* cimg = (Ld.cond_slot >= 0 && cond_img != nullptr) ? cond_img + (int64_t)Ld.cond_slot * kH : nullptr;
          mobius_layer<false>(sW, wbuf, cimg, Ld.perm, R, ldj, g);
        }
      } else if (valid) {
        const float* W = Ld.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)Ld.cond_slot * kAffFloats
                                           : a.weights + Ld.w_off;
        affine_layer<false>(W, Ld.has_ldj != 0, R, ldj, g);
      }
    }
    if (valid && lane < 9) hist[9 * L + lane] = R[lane];
    float lp = ldj;
    if (a.fisher_A != nullptr && valid) {                   // MatrixFisherN._log_prob (utils/fisher.py:217-232) and its gradient A
      float A[9], tr = 0.0f;
#pragma unroll
      for (int i = 0; i < 9; ++i) { A[i] = __ldg(a.fisher_A + img * 9 + i); tr = fmaf(A[i], R[i], tr); }
      lp += tr - __ldg(a.fisher_c + img);
      tangent_of(R, A, g);
    }

    // ---- reverse sweep ----
#pragma unroll 1
    for (int li = L - 1; li >= 0; --li) {
      const LayerDev Ld = a.layers[li];
      __syncwarp();
      float Rl[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) Rl[i] = hist[9 * li + i];
      float dummy = 0.0f;
      if (Ld.kind == RNF_LAYER_MOBIUS) {
        __syncthreads();
        const float4* src = reinterpret_cast<const float4*>(a.weights + Ld.w_off);
        float4* dst = reinterpret_cast<float4*>(sW);
        for (int i = threadIdx.x; i < kMobFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
        __syncthreads();
        if (valid) {
          const float* cimg = (Ld.cond_slot >= 0 && cond_img != nullptr) ? cond_img + (int64_t)Ld.cond_slot * kH : nullptr;
          mobius_layer<true>(sW, wbuf, cimg, Ld.perm, Rl, dummy, g);
        }
      } else if (valid) {
        const float* W = Ld.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)Ld.cond_slot * kAffFloats
                                           : a.weights + Ld.w_off;
        affine_layer<true>(W, Ld.has_ldj != 0, Rl, dummy, g);
      }
    }

    if (valid) {
      __syncwarp();
      float R0[9], G[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) R0[i] = hist[i];
      gradient_from_tangent(R0, g, G);
      if (lane == 0) {
        a.logp_out[row] = lp;
#pragma unroll
        for (int i = 0; i < 9; ++i) a.grad_out[row * 9 + i] = G[i];
      }
    }
    __syncwarp();
  }
}

// ---- training: log p's forward and the full backward (rotation, weight-image and per-image-constant gradients) -----------------
struct TrainArgs {
  const float* weights;                             // the packed FP32 image (same offsets as the handle's buffer)
  const LayerDev* layers;
  int n_layers;
  int n_mobius_slots;
  int n_mob_layers;                                 // Mobius / affine layers in the stack (index of the training records)
  int n_aff_layers;
  const float* R_in;
  int64_t N;
  const float* cond;
  int64_t cond_stride;
  const int32_t* feat_index;
  int64_t rows_per_image;
  float* R_out;                                     // forward mode
  float* ldj_out;
  const float* G_Rout;                              // backward mode: seeds (null: 0 / 1), outputs
  const float* g_ldj;
  float* G_R;
  float* ws_mob;                                    // [n_mob_layers][N][kTwsFloats]
  float* ws_aff;                                    // [n_aff_layers][N][16]
  int64_t n_tiles;
  int warp_floats;
};

// Forward mode (BWD = false): R_out, ldj.  Backward mode: the forward sweep with history, then the reverse sweep of flow_grad_kernel
// seeded with g = tangent_of(R_L, G_Rout[n]) and g_ldj[n], writing G_R (tangential) and the training records of every layer.
template <bool BWD>
__global__ void __launch_bounds__(512, 1) flow_train_kernel(const TrainArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* sW = smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_warps = blockDim.x >> 5;
  float* wbuf = smem + kMobFloats + (size_t)warp * a.warp_floats;
  float* hist = wbuf + kWarpFloats;                          // backward: R_0 .. R_L, 9 floats each
  const int L = a.n_layers;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t row = tile * n_warps + warp;
    const bool valid = row < a.N;
    float R[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
    int64_t img = 0;
    if (valid) {
#pragma unroll
      for (int i = 0; i < 9; ++i) R[i] = __ldg(a.R_in + row * 9 + i);
      img = a.feat_index != nullptr ? (int64_t)__ldg(a.feat_index + row) : row / a.rows_per_image;
    }
    const float* cond_img = a.cond != nullptr ? a.cond + img * a.cond_stride : nullptr;
    float ldj = 0.0f;
    float g[3] = {0.f, 0.f, 0.f};

    // ---- forward sweep ----
#pragma unroll 1
    for (int li = 0; li < L; ++li) {
      const LayerDev Ld = a.layers[li];
      if (BWD && valid && lane < 9) hist[9 * li + lane] = R[lane];
      if (Ld.kind == RNF_LAYER_MOBIUS) {
        __syncthreads();
        const float4* src = reinterpret_cast<const float4*>(a.weights + Ld.w_off);
        float4* dst = reinterpret_cast<float4*>(sW);
        for (int i = threadIdx.x; i < kMobFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
        __syncthreads();
        if (valid) {
          const float* cimg = (Ld.cond_slot >= 0 && cond_img != nullptr) ? cond_img + (int64_t)Ld.cond_slot * kH : nullptr;
          mobius_layer<false>(sW, wbuf, cimg, Ld.perm, R, ldj, g);
        }
      } else if (valid) {
        const float* W = Ld.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)Ld.cond_slot * kAffFloats
                                           : a.weights + Ld.w_off;
        affine_layer<false>(W, Ld.has_ldj != 0, R, ldj, g);
      }
    }
    if (!BWD) {
      if (valid && lane == 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) a.R_out[row * 9 + i] = R[i];
        a.ldj_out[row] = ldj;
      }
      __syncwarp();
      continue;
    }
    float gl = 1.0f;
    if (valid) {
      if (a.G_Rout != nullptr) {
        float G[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) G[i] = __ldg(a.G_Rout + row * 9 + i);
        tangent_of(R, G, g);
      }
      if (a.g_ldj != nullptr) gl = __ldg(a.g_ldj + row);
    }

    // ---- reverse sweep ----
    int mi = a.n_mob_layers, ai = a.n_aff_layers;
#pragma unroll 1
    for (int li = L - 1; li >= 0; --li) {
      const LayerDev Ld = a.layers[li];
      __syncwarp();
      float Rl[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) Rl[i] = hist[9 * li + i];
      float dummy = 0.0f;
      if (Ld.kind == RNF_LAYER_MOBIUS) {
        --mi;
        __syncthreads();
        const float4* src = reinterpret_cast<const float4*>(a.weights + Ld.w_off);
        float4* dst = reinterpret_cast<float4*>(sW);
        for (int i = threadIdx.x; i < kMobFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
        __syncthreads();
        if (valid) {
          const float* cimg = (Ld.cond_slot >= 0 && cond_img != nullptr) ? cond_img + (int64_t)Ld.cond_slot * kH : nullptr;
          mobius_layer<true, true>(sW, wbuf, cimg, Ld.perm, Rl, dummy, g, gl, a.ws_mob + ((int64_t)mi * a.N + row) * kTwsFloats);
        }
      } else {
        --ai;
        if (valid) {
          const float* W = Ld.cond_slot >= 0 ? cond_img + (int64_t)a.n_mobius_slots * kH + (int64_t)Ld.cond_slot * kAffFloats
                                             : a.weights + Ld.w_off;
          affine_layer<true, true>(W, Ld.has_ldj != 0, Rl, dummy, g, gl, a.ws_aff + ((int64_t)ai * a.N + row) * 16);
        }
      }
    }

    if (valid) {
      __syncwarp();
      float R0[9], G[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) R0[i] = hist[i];
      gradient_from_tangent(R0, g, G);
      if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) a.G_R[row * 9 + i] = G[i];
      }
    }
    __syncwarp();
  }
}

}  // namespace

size_t flow_grad_smem_bytes(int n_layers, int warps) {
  const int wf = (kWarpFloats + 9 * (n_layers + 1) + 3) & ~3;
  return ((size_t)kMobFloats + (size_t)warps * wf) * sizeof(float);
}

cudaError_t launch_flow_grad(const rnf_flow* f, const float* R_in, int64_t N, const float* cond, const int32_t* feat_index,
                             int64_t rows_per_image, const float* fisher_A, const float* fisher_c, float* logp_out, float* grad_out,
                             cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  const int L = f->model.n_layers;
  // warps (rows) per CTA: enough to reach every SM first, up to 16 once the batch covers the machine; fewer if the per-warp
  // rotation history of a very deep flow would not fit next to the staged conditioner
  int warps = (int)((N + f->sm_count - 1) / f->sm_count);
  warps = warps < 1 ? 1 : (warps > 16 ? 16 : warps);
  while (warps > 1 && flow_grad_smem_bytes(L, warps) > 227 * 1024) --warps;
  const size_t smem = flow_grad_smem_bytes(L, warps);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  cudaError_t e = cudaFuncSetAttribute(flow_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  GradArgs a;
  a.weights = f->weights_dev;
  a.layers = f->layers_dev;
  a.n_layers = L;
  a.n_mobius_slots = f->model.n_mobius_slots;
  a.R_in = R_in;
  a.N = N;
  a.cond = f->cond_floats > 0 ? cond : nullptr;
  a.cond_stride = f->cond_floats;
  a.feat_index = feat_index;
  a.rows_per_image = rows_per_image > 0 ? rows_per_image : 1;
  a.fisher_A = fisher_A;
  a.fisher_c = fisher_c;
  a.logp_out = logp_out;
  a.grad_out = grad_out;
  a.n_tiles = (N + warps - 1) / warps;
  a.warp_floats = (kWarpFloats + 9 * (L + 1) + 3) & ~3;
  const int64_t grid = a.n_tiles < f->sm_count ? a.n_tiles : f->sm_count;
  flow_grad_kernel<<<(unsigned)grid, 32 * warps, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace rnf

namespace rnf {

int64_t flow_train_workspace_floats(const rnf_flow* f, int64_t N) {
  int64_t n_mob = 0, n_aff = 0;
  for (int i = 0; i < f->model.n_layers; ++i) (f->layers_host[i].kind == RNF_LAYER_MOBIUS ? n_mob : n_aff) += 1;
  return N * (n_mob * kTwsFloats + n_aff * 16);
}

cudaError_t launch_flow_train(const rnf_flow* f, bool backward, const float* weights, const float* R_in, int64_t N, const float* cond,
                              const int32_t* feat_index, int64_t rows_per_image, float* R_out, float* ldj_out, const float* G_Rout,
                              const float* g_ldj, float* G_R, float* workspace, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  const int L = f->model.n_layers;
  int n_mob = 0;
  for (int i = 0; i < L; ++i) n_mob += f->layers_host[i].kind == RNF_LAYER_MOBIUS;
  // the forward mode keeps no rotation history: its per-warp buffer is the activation / gradient vector alone
  auto smem_bytes = [&](int warps) {
    return backward ? flow_grad_smem_bytes(L, warps) : ((size_t)kMobFloats + (size_t)warps * kWarpFloats) * sizeof(float);
  };
  int warps = (int)((N + f->sm_count - 1) / f->sm_count);
  warps = warps < 1 ? 1 : (warps > 16 ? 16 : warps);
  while (warps > 1 && smem_bytes(warps) > 227 * 1024) --warps;
  const size_t smem = smem_bytes(warps);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  TrainArgs a;
  a.weights = weights;
  a.layers = f->layers_dev;
  a.n_layers = L;
  a.n_mobius_slots = f->model.n_mobius_slots;
  a.n_mob_layers = n_mob;
  a.n_aff_layers = L - n_mob;
  a.R_in = R_in;
  a.N = N;
  a.cond = f->cond_floats > 0 ? cond : nullptr;
  a.cond_stride = f->cond_floats;
  a.feat_index = feat_index;
  a.rows_per_image = rows_per_image > 0 ? rows_per_image : 1;
  a.R_out = R_out;
  a.ldj_out = ldj_out;
  a.G_Rout = G_Rout;
  a.g_ldj = g_ldj;
  a.G_R = G_R;
  a.ws_mob = workspace;
  a.ws_aff = workspace != nullptr ? workspace + N * (int64_t)n_mob * kTwsFloats : nullptr;
  a.n_tiles = (N + warps - 1) / warps;
  a.warp_floats = backward ? (kWarpFloats + 9 * (L + 1) + 3) & ~3 : kWarpFloats;
  const int64_t grid = a.n_tiles < f->sm_count ? a.n_tiles : f->sm_count;
  auto kern = backward ? flow_train_kernel<true> : flow_train_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)grid, 32 * warps, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace rnf
