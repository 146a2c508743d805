// train_ops.cu -- the DIFFERENTIABLE per-layer operators behind Flow.forward / Flow.inverse when autograd is on
// (training: agent.py:87 loss.backward(); eval.py:468-477 nll_grad) or when config.segments is not the 64 the fused tcgen05
// kernels are specialised for.  One thread per rotation, plain FP32 with the precise math functions, any number K of mixture
// components.  The conditioner MLP itself stays a sequence of library GEMMs on the Python side (torch autograd supplies its
// backward); these kernels are everything after it:
//   mobius_mixture  forward : (R, out[N,4K]) -> (R', ldj)            flow/mobiusflow.py:58-85 (forward) / :141-183 (inverse,
//                              with the 15 bisection halvings of BinFind.forward, :196-224)
//   mobius_mixture  backward: VJP in the TANGENT space of SO(3).  A layer maps R -> R' = R Rot(e_p1, phi) with
//                              phi = Theta(a, alpha, beta) - pi, alpha_k = -(R^T w_k)[p0], beta_k = (R^T w_k)[p2]; a body-frame
//                              perturbation omega of R gives omega' = M^T omega + (dphi) e_p1, so with g' = vee(R'^T G') the tangent
//                              gradient is g = M g' + e_p0 x (-R^T sum_k A_k w_k) + e_p2 x (R^T sum_k B_k w_k), A_k = dL/dalpha_k,
//                              B_k = dL/dbeta_k, and G_R = R [g]x / 2.  Only the tangential part of a rotation gradient reaches the
//                              parameters (every layer keeps R on the manifold), so parameter and feature gradients equal the
//                              reference's autograd; verified against autograd through the oracle (tests/test_gpu_train.py,
//                              tools/proto/tangent_vjp.py).  Inverse direction: implicit-function theorem at the returned root,
//                              which is what BinFind.backward (flow/mobiusflow.py:248-273) evaluates.
//   quat_affine     forward / backward: calculate_16 (flow/squeezetrans.py:33-38) with per-row W; returns log|Wq| (the caller adds
//                              log|det W| with torch.linalg.slogdet, which is differentiable on its own).
//   ablation        forward / backward: the ablation layers of csrc/ablation_layers.cuh with a per-row matrix M in the requested
//                              direction; the forward is ablation_layer() itself, the backward a hand-written reverse sweep
//                              (tools/proto/ablation_vjp.py).
#include <cuda_runtime.h>
#include <math.h>

#include "ablation_layers.cuh"
#include "mobius_math.cuh"
#include "rnf_common.cuh"

namespace rnf {
namespace {

constexpr int kMaxK = 256;          // prepared components of one rotation are kept in (L1-backed) local memory

struct Frame3 {
  float x[3], y[3], z[3];
};

__device__ __forceinline__ void load_cols(const float* __restrict__ R, int p0, Frame3& f, float Rm[9]) {
#pragma unroll
  for (int i = 0; i < 9; ++i) Rm[i] = R[i];
  const int p1 = (p0 + 1) % 3, p2 = (p0 + 2) % 3;
#pragma unroll
  for (int i = 0; i < 3; ++i) { f.x[i] = Rm[3 * i + p0]; f.y[i] = Rm[3 * i + p1]; f.z[i] = Rm[3 * i + p2]; }
}

// prepared component: in-plane squashed centre (alpha', beta'), softplus weight
struct Prep {
  float al, be, n, s, alp, bep, sp;
};

__device__ __forceinline__ Prep prepare(const float* __restrict__ out, int K, int k, const float r[3], const float v[3]) {
  Prep c;
  const float a = out[k];
  const float w0 = out[K + 3 * k], w1 = out[K + 3 * k + 1], w2 = out[K + 3 * k + 2];
  c.al = fmaf(w2, r[2], fmaf(w1, r[1], w0 * r[0]));       // the projection (I - y y^T) w leaves these two dot products unchanged
  c.be = fmaf(w2, v[2], fmaf(w1, v[1], w0 * v[0]));
  c.n = sqrtf(fmaf(c.be, c.be, c.al * c.al));
  c.s = 0.7f / (1.0f + c.n);
  c.alp = c.s * c.al;
  c.bep = c.s * c.be;
  c.sp = softplus_torch(a);
  return c;
}

// wrapped angle of h_w'(z) and f = (1 - |w'|^2) / |z - w'|^2 at the in-plane point z = (cz, sz)
__device__ __forceinline__ void eval_point(float cz, float sz, float alp, float bep, float& theta, float& f) {
  const float X = cz - alp, Y = sz - bep;
  const float D2 = fmaf(Y, Y, X * X);
  const float om = 1.0f - fmaf(bep, bep, alp * alp);
  f = om / D2;
  const float hr = fmaf(f, X, -alp), hv = fmaf(f, Y, -bep);
  const float th = atan2f(hv, hr);
  theta = th >= 0.0f ? th : th + kTwoPi;
}

template <bool INV>
__global__ void __launch_bounds__(128) mobius_mixture_fwd_kernel(const float* __restrict__ R, const float* __restrict__ out, int64_t N, int K,
                                                                 int p0, float* __restrict__ R_out, float* __restrict__ ldj_out,
                                                                 float* __restrict__ theta_out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  Frame3 F;
  float Rm[9];
  load_cols(R + n * 9, p0, F, Rm);
  float r[3], v[3];
  make_frame(F.x, F.y, r, v);                              // r = -x/|x|, v = (y x r)/|y x r|   (flow/mobiusflow.py:64-67)
  const float* o = out + n * 4 * (int64_t)K;
  const float zr = dot3(F.x, r), zv = dot3(F.x, v);        // the moving column in its own frame: (-|x|, ~0)
  float pal[INV ? kMaxK : 1], pbe[INV ? kMaxK : 1], psp[INV ? kMaxK : 1];
  float S = 0.0f, Sth = 0.0f, Sf = 0.0f;
  for (int k = 0; k < K; ++k) {
    const Prep c = prepare(o, K, k, r, v);
    S += c.sp;
    if (INV) { pal[k] = c.alp; pbe[k] = c.bep; psp[k] = c.sp; }
    else {
      float th, f;
      eval_point(zr, zv, c.alp, c.bep, th, f);
      Sth = fmaf(c.sp, th, Sth);
      Sf = fmaf(c.sp, f, Sf);
    }
  }
  float theta, ldj;
  if (!INV) {
    theta = Sth / S;
    ldj = logf(Sf / S);
  } else {
    // target angle of the given column in its own frame (flow/mobiusflow.py:157-167), then BinFind.forward (:196-224)
    float ys = atan2f(zv, zr);
    ys = ys >= 0.0f ? ys : ys + kTwoPi;
    if (fabsf(ys - kTwoPi) < 1e-4f) ys = 0.0f;
    float lo = kPi / 2.0f, hi = 1.5f * kPi, x0 = 0.0f;
    for (int it = 0; it < 15; ++it) {
      x0 = (lo + hi) / 2.0f;
      float sn, cs;
      sincosf(x0, &sn, &cs);
      float Fs = 0.0f;
      for (int k = 0; k < K; ++k) {
        float th, f;
        eval_point(cs, sn, pal[k], pbe[k], th, f);
        Fs = fmaf(psp[k], th, Fs);
      }
      const float fx0 = Fs / S - ys;
      const float half_w = (hi - lo) / 2.0f;
      if (fx0 < 0.0f) lo = lo + half_w;
      else if (fx0 >= 0.0f) hi = hi - half_w;
    }
    theta = x0;
    float sn, cs;
    sincosf(x0, &sn, &cs);
    for (int k = 0; k < K; ++k) {
      float th, f;
      eval_point(cs, sn, pal[k], pbe[k], th, f);
      Sf = fmaf(psp[k], f, Sf);
    }
    ldj = -logf(Sf / S);
  }
  float nx[3], nz[3];
  circle_point(r, v, theta, nx);                           // r cos(theta) + v sin(theta)   (flow/mobiusflow.py:102,169)
  cross3(nx, F.y, nz);
  normalize3(nz);
  const int p2 = (p0 + 2) % 3;
#pragma unroll
  for (int i = 0; i < 3; ++i) { Rm[3 * i + p0] = nx[i]; Rm[3 * i + p2] = nz[i]; }
#pragma unroll
  for (int i = 0; i < 9; ++i) R_out[n * 9 + i] = Rm[i];
  ldj_out[n] = ldj;
  theta_out[n] = theta;
}

template <bool INV>
__global__ void __launch_bounds__(128) mobius_mixture_bwd_kernel(const float* __restrict__ R, const float* __restrict__ out, int64_t N, int K,
                                                                 int p0, const float* __restrict__ theta_in, const float* __restrict__ R_out,
                                                                 const float* __restrict__ G_Rout, const float* __restrict__ g_ldj,
                                                                 float* __restrict__ G_R, float* __restrict__ G_out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  Frame3 F;
  float Rm[9], Rn[9];
  load_cols(R + n * 9, p0, F, Rm);
#pragma unroll
  for (int i = 0; i < 9; ++i) Rn[i] = R_out[n * 9 + i];
  float r[3], v[3];
  make_frame(F.x, F.y, r, v);
  const float* o = out + n * 4 * (int64_t)K;
  const int p1 = (p0 + 1) % 3, p2 = (p0 + 2) % 3;
  // evaluation point of the mixture map: the moving column (forward) or the returned root (inverse)
  float cz, sz;
  if (INV) sincosf(theta_in[n], &sz, &cz);
  else { cz = dot3(F.x, r); sz = dot3(F.x, v); }
  float gp[3];
  tangent_of(Rn, G_Rout + n * 9, gp);
  const float gL = g_ldj[n];
  // pass 1: S, Theta = sum pi theta, F = sum pi f, F_theta = sum pi df/dtheta
  float S = 0.0f, Sth = 0.0f, Sf = 0.0f, Sft = 0.0f;
  for (int k = 0; k < K; ++k) {
    const Prep c = prepare(o, K, k, r, v);
    float th, f;
    eval_point(cz, sz, c.alp, c.bep, th, f);
    S += c.sp;
    Sth = fmaf(c.sp, th, Sth);
    Sf = fmaf(c.sp, f, Sf);
    if (INV) {
      const float X = cz - c.alp, Y = sz - c.bep;
      const float D2 = fmaf(Y, Y, X * X);
      const float om = 1.0f - fmaf(c.bep, c.bep, c.alp * c.alp);
      Sft = fmaf(c.sp, -2.0f * om * (c.alp * sz - c.bep * cz) / (D2 * D2), Sft);
    }
  }
  const float Th = Sth / S, Fm = Sf / S, Ft = Sft / S;
  // coefficients of dTheta-like and dF-like parameter derivatives in dL
  //   forward: phi = Theta - pi, ldj = log F                 -> cG = g'[p1],                      cF = gL / F
  //   inverse: psi = theta* - pi with G(theta*, p) = Theta - pi = 0, ldj = -log F(theta*, p)
  //            dpsi/dp = -G_p / F, dldj/dp = -F_p / F + F_theta G_p / F^2   -> cG = -g'[p1]/F + gL F_theta / F^2, cF = -gL / F
  float cG, cF;
  if (!INV) { cG = gp[p1]; cF = gL / Fm; }
  else { cG = -gp[p1] / Fm + gL * Ft / (Fm * Fm); cF = -gL / Fm; }
  float sA[3] = {0.f, 0.f, 0.f}, sB[3] = {0.f, 0.f, 0.f};          // sum_k A_k w_k, sum_k B_k w_k (world frame)
  float* go = G_out + n * 4 * (int64_t)K;
  for (int k = 0; k < K; ++k) {
    const Prep c = prepare(o, K, k, r, v);
    float th, f;
    eval_point(cz, sz, c.alp, c.bep, th, f);
    const float X = cz - c.alp, Y = sz - c.bep;
    const float D2 = fmaf(Y, Y, X * X);
    const float om = 1.0f - fmaf(c.bep, c.bep, c.alp * c.alp);
    const float th_ap = 2.0f * Y / D2, th_bp = -2.0f * X / D2;
    const float f_ap = (-2.0f * c.alp * D2 + 2.0f * om * X) / (D2 * D2);
    const float f_bp = (-2.0f * c.bep * D2 + 2.0f * om * Y) / (D2 * D2);
    const float t = c.n > 1e-30f ? c.s / (c.n * (1.0f + c.n)) : 0.0f;     // squash Jacobian: d(alpha', beta') / d(alpha, beta)
    const float J11 = c.s - t * c.al * c.al, J12 = -t * c.al * c.be, J22 = c.s - t * c.be * c.be;
    const float th_a = th_ap * J11 + th_bp * J12, th_b = th_ap * J12 + th_bp * J22;
    const float f_a = f_ap * J11 + f_bp * J12, f_b = f_ap * J12 + f_bp * J22;
    const float pi = c.sp / S;
    const float A = pi * (cG * th_a + cF * f_a);
    const float B = pi * (cG * th_b + cF * f_b);
    const float a = o[k];
    const float sig = 1.0f / (1.0f + expf(-a));                           // d softplus / da (threshold 20: sigmoid(20) = 1 - 2e-9)
    go[k] = sig / S * (cG * (th - Th) + cF * (f - Fm));
    // alpha = w.r = -w.x, beta = w.v = w.z on the manifold
    const float w0 = o[K + 3 * k], w1 = o[K + 3 * k + 1], w2 = o[K + 3 * k + 2];
    go[K + 3 * k] = fmaf(B, F.z[0], -A * F.x[0]);
    go[K + 3 * k + 1] = fmaf(B, F.z[1], -A * F.x[1]);
    go[K + 3 * k + 2] = fmaf(B, F.z[2], -A * F.x[2]);
    sA[0] = fmaf(A, w0, sA[0]); sA[1] = fmaf(A, w1, sA[1]); sA[2] = fmaf(A, w2, sA[2]);
    sB[0] = fmaf(B, w0, sB[0]); sB[1] = fmaf(B, w1, sB[1]); sB[2] = fmaf(B, w2, sB[2]);
  }
  // body-frame versions u = R^T s, then c = e_p0 x (-uA) + e_p2 x (uB)
  float uA[3], uB[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    uA[i] = Rm[i] * sA[0] + Rm[3 + i] * sA[1] + Rm[6 + i] * sA[2];
    uB[i] = Rm[i] * sB[0] + Rm[3 + i] * sB[1] + Rm[6 + i] * sB[2];
  }
  float e0[3] = {0.f, 0.f, 0.f}, e2[3] = {0.f, 0.f, 0.f}, nA[3] = {-uA[0], -uA[1], -uA[2]}, c1[3], c2[3];
  e0[p0] = 1.0f;
  e2[p2] = 1.0f;
  cross3(e0, nA, c1);
  cross3(e2, uB, c2);
  // M = R^T R' (body rotation about e_p1); g = M g' + c
  float g[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    float m = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float Mij = Rm[i] * Rn[j] + Rm[3 + i] * Rn[3 + j] + Rm[6 + i] * Rn[6 + j];
      m = fmaf(Mij, gp[j], m);
    }
    g[i] = m + c1[i] + c2[i];
  }
  gradient_from_tangent(Rm, g, G_R + n * 9);
}

__global__ void __launch_bounds__(128) quat_affine_fwd_kernel(const float* __restrict__ R, const float* __restrict__ W, int64_t N,
                                                              float* __restrict__ R_out, float* __restrict__ loglen_out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float Rm[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) Rm[i] = R[n * 9 + i];
  const float loglen = quat_affine(W + n * 16, Rm);
#pragma unroll
  for (int i = 0; i < 9; ++i) R_out[n * 9 + i] = Rm[i];
  loglen_out[n] = loglen;
}

// d_p = (2 E(p^) g' + gL p^) / l ;  G_W = d_p q^T ;  g = E(q)^T W^T d_p / 2        (tangent-space VJP of calculate_16)
__global__ void __launch_bounds__(128) quat_affine_bwd_kernel(const float* __restrict__ R, const float* __restrict__ W, int64_t N,
                                                              const float* __restrict__ R_out, const float* __restrict__ G_Rout,
                                                              const float* __restrict__ g_loglen, float* __restrict__ G_R,
                                                              float* __restrict__ G_W) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float Rm[9], Rn[9], q[4], p[4];
#pragma unroll
  for (int i = 0; i < 9; ++i) { Rm[i] = R[n * 9 + i]; Rn[i] = R_out[n * 9 + i]; }
  mat_to_quat(Rm, q);
  const float* Wn = W + n * 16;
#pragma unroll
  for (int a = 0; a < 4; ++a) p[a] = fmaf(Wn[4 * a + 3], q[3], fmaf(Wn[4 * a + 2], q[2], fmaf(Wn[4 * a + 1], q[1], Wn[4 * a] * q[0])));
  const float len = sqrtf(p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3]);
  float ph[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) ph[a] = p[a] / len;
  float gp[3], Eg[4], dp[4];
  tangent_of(Rn, G_Rout + n * 9, gp);
  E_mul(ph, gp, Eg);
  const float gL = g_loglen[n];
#pragma unroll
  for (int a = 0; a < 4; ++a) dp[a] = (2.0f * Eg[a] + gL * ph[a]) / len;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) G_W[n * 16 + 4 * a + b] = dp[a] * q[b];
  float Wt[4];
#pragma unroll
  for (int b = 0; b < 4; ++b) Wt[b] = Wn[b] * dp[0] + Wn[4 + b] * dp[1] + Wn[8 + b] * dp[2] + Wn[12 + b] * dp[3];
  float g[3];
  ET_mul(q, Wt, g);
#pragma unroll
  for (int i = 0; i < 3; ++i) g[i] *= 0.5f;
  gradient_from_tangent(Rm, g, G_R + n * 9);
}

// ---- ablation layers (csrc/ablation_layers.cuh).  M is the n x n matrix the layer applies in the requested direction, one per row.
__global__ void __launch_bounds__(128) ablation_fwd_kernel(const float* __restrict__ R, const float* __restrict__ M, int64_t N, int kind,
                                                           float* __restrict__ R_out, float* __restrict__ ldj_out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int nn = kind == RNF_LAYER_SMITH36 ? 36 : 9;
  Rot9 io;
#pragma unroll
  for (int i = 0; i < 9; ++i) io.m[i] = R[n * 9 + i];
  io.ldj = 0.0f;
  io = ablation_layer(kind, M + nn * n, io);
#pragma unroll
  for (int i = 0; i < 9; ++i) R_out[n * 9 + i] = io.m[i];
  ldj_out[n] = io.ldj;
}

// VJP of ablation::normalize_with_tangents<3>: t = i v, dt_k = i d_k - i^3 s_k v with i = 1/|v|, s_k = v.d_k.  dt_k depends on v
// through i, i^3 and s_k: these second-order terms carry the log-det gradient.
__device__ __forceinline__ void normalize_bwd(const float v[3], const float d[3][3], const float Gt[3], const float Gdt[3][3], float Gv[3],
                                              float Gd[3][3]) {
  const float i = 1.0f / sqrtf(dot3(v, v));
  const float i3 = i * i * i, i5 = i3 * i * i;
  const float vGt = dot3(v, Gt);
  float cv = 0.0f;
#pragma unroll
  for (int j = 0; j < 3; ++j) Gv[j] = i * Gt[j] - i3 * vGt * v[j];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float s = dot3(v, d[k]), a = dot3(Gdt[k], d[k]), b = dot3(Gdt[k], v);
    cv += 3.0f * i5 * s * b - i3 * a;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Gv[j] -= i3 * (b * d[k][j] + s * Gdt[k][j]);
      Gd[k][j] = i * Gdt[k][j] - i3 * b * v[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) Gv[j] += cv * v[j];
}

// cross3 VJP, accumulating: z = a x b gives G_a += b x G_z, G_b += G_z x a
__device__ __forceinline__ void cross_bwd(const float a[3], const float b[3], const float Gz[3], float Ga[3], float Gb[3]) {
  float u[3], w[3];
  cross3(b, Gz, u);
  cross3(Gz, a, w);
#pragma unroll
  for (int j = 0; j < 3; ++j) { Ga[j] += u[j]; Gb[j] += w[j]; }
}

// Reverse sweep of ablation::smith_tail: (c0, dc0, c1, dc1) <- (G_T = dL/dT, gL = dL/dldj).  The forward is recomputed here; the
// formulas are those of tools/proto/ablation_vjp.py smith_tail_bwd.
__device__ __forceinline__ void smith_tail_bwd(const float c0[3], const float dc0[3][3], const float c1[3], const float dc1[3][3],
                                               const float GT[9], float gL, float Gc0[3], float Gdc0[3][3], float Gc1[3], float Gdc1[3][3]) {
  float t0[3], dt0[3][3], t1[3], dt1[3][3], t2[3], dt2[3][3], raw1[3], draw1[3][3], ddot[3];
  ablation::normalize_with_tangents<3>(c0, dc0, t0, dt0);
  const float dot = t0[0] * c1[0] + t0[1] * c1[1] + t0[2] * c1[2];
#pragma unroll
  for (int i = 0; i < 3; ++i) raw1[i] = c1[i] - dot * t0[i];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    ddot[k] = (dt0[k][0] * c1[0] + dt0[k][1] * c1[1] + dt0[k][2] * c1[2]) + (t0[0] * dc1[k][0] + t0[1] * dc1[k][1] + t0[2] * dc1[k][2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) draw1[k][i] = dc1[k][i] - (ddot[k] * t0[i] + dot * dt0[k][i]);
  }
  ablation::normalize_with_tangents<3>(raw1, draw1, t1, dt1);
  cross3(t0, t1, t2);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float a[3], b[3];
    cross3(t0, dt1[k], a);
    cross3(dt0[k], t1, b);
#pragma unroll
    for (int i = 0; i < 3; ++i) dt2[k][i] = a[i] + b[i];
  }
  // V[k] = ((delta_k)_01, (delta_k)_02, (delta_k)_12), delta_k[a][b] = sum_c dt_c,k[a] t_c[b];  dL/dV = gL V^{-T} = gL cof(V) / det V
  float V[9];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    V[3 * k] = dt0[k][0] * t0[1] + dt1[k][0] * t1[1] + dt2[k][0] * t2[1];
    V[3 * k + 1] = dt0[k][0] * t0[2] + dt1[k][0] * t1[2] + dt2[k][0] * t2[2];
    V[3 * k + 2] = dt0[k][1] * t0[2] + dt1[k][1] * t1[2] + dt2[k][1] * t2[2];
  }
  float GV[9];
  GV[0] = V[4] * V[8] - V[5] * V[7]; GV[1] = V[5] * V[6] - V[3] * V[8]; GV[2] = V[3] * V[7] - V[4] * V[6];
  GV[3] = V[2] * V[7] - V[1] * V[8]; GV[4] = V[0] * V[8] - V[2] * V[6]; GV[5] = V[1] * V[6] - V[0] * V[7];
  GV[6] = V[1] * V[5] - V[2] * V[4]; GV[7] = V[2] * V[3] - V[0] * V[5]; GV[8] = V[0] * V[4] - V[1] * V[3];
  const float s = gL / (V[0] * GV[0] + V[1] * GV[1] + V[2] * GV[2]);
#pragma unroll
  for (int i = 0; i < 9; ++i) GV[i] *= s;
  // delta_k reverse: G_dt_c,k = (GV01 t_c[1] + GV02 t_c[2], GV12 t_c[2], 0); G_t_c[1] += GV01 dt_c,k[0], G_t_c[2] += GV02 dt_c,k[0] + GV12 dt_c,k[1]
  float Gt0[3], Gt1[3], Gt2[3], Gdt0[3][3], Gdt1[3][3], Gdt2[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i) { Gt0[i] = GT[3 * i]; Gt1[i] = GT[3 * i + 1]; Gt2[i] = GT[3 * i + 2]; }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float e01 = GV[3 * k], e02 = GV[3 * k + 1], e12 = GV[3 * k + 2];
    Gdt0[k][0] = e01 * t0[1] + e02 * t0[2]; Gdt0[k][1] = e12 * t0[2]; Gdt0[k][2] = 0.0f;
    Gdt1[k][0] = e01 * t1[1] + e02 * t1[2]; Gdt1[k][1] = e12 * t1[2]; Gdt1[k][2] = 0.0f;
    Gdt2[k][0] = e01 * t2[1] + e02 * t2[2]; Gdt2[k][1] = e12 * t2[2]; Gdt2[k][2] = 0.0f;
    Gt0[1] += e01 * dt0[k][0]; Gt0[2] += e02 * dt0[k][0] + e12 * dt0[k][1];
    Gt1[1] += e01 * dt1[k][0]; Gt1[2] += e02 * dt1[k][0] + e12 * dt1[k][1];
    Gt2[1] += e01 * dt2[k][0]; Gt2[2] += e02 * dt2[k][0] + e12 * dt2[k][1];
  }
  // dt2_k = t0 x dt1_k + dt0_k x t1 ; t2 = t0 x t1
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    cross_bwd(t0, dt1[k], Gdt2[k], Gt0, Gdt1[k]);
    cross_bwd(dt0[k], t1, Gdt2[k], Gdt0[k], Gt1);
  }
  cross_bwd(t0, t1, Gt2, Gt0, Gt1);
  float Graw1[3], Gdraw1[3][3];
  normalize_bwd(raw1, draw1, Gt1, Gdt1, Graw1, Gdraw1);
  // draw1_k = dc1_k - ddot_k t0 - dot dt0_k ; ddot_k = dt0_k.c1 + t0.dc1_k ; raw1 = c1 - dot t0 ; dot = t0.c1
  float Gdot = -(Graw1[0] * t0[0] + Graw1[1] * t0[1] + Graw1[2] * t0[2]);
#pragma unroll
  for (int i = 0; i < 3; ++i) { Gc1[i] = Graw1[i]; Gt0[i] -= dot * Graw1[i]; }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float Gdd = -dot3(Gdraw1[k], t0);
    Gdot -= dot3(Gdraw1[k], dt0[k]);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      Gdc1[k][i] = Gdraw1[k][i] + Gdd * t0[i];
      Gt0[i] += Gdd * dc1[k][i] - ddot[k] * Gdraw1[k][i];
      Gdt0[k][i] += Gdd * c1[i] - dot * Gdraw1[k][i];
      Gc1[i] += Gdd * dt0[k][i];
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) { Gt0[i] += Gdot * c1[i]; Gc1[i] += Gdot * t0[i]; }
  normalize_bwd(c0, dc0, Gt0, Gdt0, Gc0, Gdc0);
}

// out = A^T B (3x3, row-major)
__device__ __forceinline__ void matmul3_tn(const float* __restrict__ A, const float* __restrict__ B, float out[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) out[3 * i + j] = A[i] * B[j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
}

// out = A B^T (3x3, row-major)
__device__ __forceinline__ void matmul3_nt(const float* __restrict__ A, const float* __restrict__ B, float out[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) out[3 * i + j] = A[3 * i] * B[3 * j] + A[3 * i + 1] * B[3 * j + 1] + A[3 * i + 2] * B[3 * j + 2];
}

// Tangent-space VJP of one ablation layer (tools/proto/ablation_vjp.py): G_R = R [g]x / 2 with g = vee(R^T dL/dR), G_M [N,n,n].
//   RIGHT9  R' = R Q            : dL/dR = G' Q^T, G_M = R^T G'
//   POLAR9L/R R' = polar(A), A = M R / R M : H = R'^T A, X = R'^T G', y = ((tr H) I - H)^{-1} vee(X - X^T), G_A = R' [y]x, then
//                                 G_M = G_A R^T, dL/dR = M^T G_A (left) or G_M = R^T G_A, dL/dR = G_A M^T (right)
//   SMITH9  A = M R             : reverse sweep of smith_tail to (a0, a1) and the tangents, which also carry a2
//   SMITH36 t = M6 v, dt_k = M6 dv_k : G_M6 = G_t v^T + sum_k G_dt_k dv_k^T, then back to columns 0, 1 of R through v and dv
template <int KIND>
__global__ void __launch_bounds__(128) ablation_bwd_kernel(const float* __restrict__ R, const float* __restrict__ M, int64_t N,
                                                           const float* __restrict__ R_out, const float* __restrict__ G_Rout,
                                                           const float* __restrict__ g_ldj, float* __restrict__ G_R, float* __restrict__ G_M) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  constexpr int nn = KIND == RNF_LAYER_SMITH36 ? 36 : 9;
  const float* Mn = M + nn * n;
  float* GMn = G_M + nn * n;
  float Rm[9], Gp[9], GRm[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) { Rm[i] = R[n * 9 + i]; Gp[i] = G_Rout[n * 9 + i]; }
  if (KIND == RNF_LAYER_RIGHT9) {
    float Q[9], GQ[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) Q[i] = Mn[i];
    matmul3_nt(Gp, Q, GRm);
    matmul3_tn(Rm, Gp, GQ);
#pragma unroll
    for (int i = 0; i < 9; ++i) GMn[i] = GQ[i];
  } else if (KIND == RNF_LAYER_POLAR9L || KIND == RNF_LAYER_POLAR9R) {
    constexpr bool kLeft = KIND == RNF_LAYER_POLAR9L;
    float Mm[9], Q[9], A[9], H[9], X[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) { Mm[i] = Mn[i]; Q[i] = R_out[n * 9 + i]; }
    if (kLeft) ablation::matmul3(Mm, Rm, A);
    else ablation::matmul3(Rm, Mm, A);
    matmul3_tn(Q, A, H);
    matmul3_tn(Q, Gp, X);
    const float x0 = X[7] - X[5], x1 = X[2] - X[6], x2 = X[3] - X[1];
    // K = (tr H) I - H with H symmetrised (R' is the polar factor to FP32 rounding); y = K^{-1} x by the adjugate
    const float tr = H[0] + H[4] + H[8];
    const float h01 = 0.5f * (H[1] + H[3]), h02 = 0.5f * (H[2] + H[6]), h12 = 0.5f * (H[5] + H[7]);
    const float k00 = tr - H[0], k11 = tr - H[4], k22 = tr - H[8];
    const float c00 = k11 * k22 - h12 * h12, c01 = h02 * h12 + h01 * k22, c02 = h01 * h12 + h02 * k11;
    const float c11 = k00 * k22 - h02 * h02, c12 = k00 * h12 + h01 * h02, c22 = k00 * k11 - h01 * h01;
    const float idet = 1.0f / (k00 * c00 - h01 * c01 - h02 * c02);
    const float y0 = idet * (c00 * x0 + c01 * x1 + c02 * x2);
    const float y1 = idet * (c01 * x0 + c11 * x1 + c12 * x2);
    const float y2 = idet * (c02 * x0 + c12 * x1 + c22 * x2);
    const float Y[9] = {0.0f, -y2, y1, y2, 0.0f, -y0, -y1, y0, 0.0f};
    float GA[9], GMm[9];
    ablation::matmul3(Q, Y, GA);
    if (kLeft) { matmul3_nt(GA, Rm, GMm); matmul3_tn(Mm, GA, GRm); }
    else { matmul3_tn(Rm, GA, GMm); matmul3_nt(GA, Mm, GRm); }
#pragma unroll
    for (int i = 0; i < 9; ++i) GMn[i] = GMm[i];
  } else if (KIND == RNF_LAYER_SMITH9) {
    float Mm[9], A[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) Mm[i] = Mn[i];
    ablation::matmul3(Mm, Rm, A);
    float a0[3], a1[3], dc0[3][3], dc1[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      a0[i] = A[3 * i]; a1[i] = A[3 * i + 1];
      dc0[0][i] = -a1[i]; dc0[1][i] = -A[3 * i + 2]; dc0[2][i] = 0.0f;
      dc1[0][i] = a0[i];  dc1[1][i] = 0.0f;          dc1[2][i] = -A[3 * i + 2];
    }
    float Gc0[3], Gdc0[3][3], Gc1[3], Gdc1[3][3], GA[9], GMm[9];
    smith_tail_bwd(a0, dc0, a1, dc1, Gp, g_ldj[n], Gc0, Gdc0, Gc1, Gdc1);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      GA[3 * i] = Gc0[i] + Gdc1[0][i];
      GA[3 * i + 1] = Gc1[i] - Gdc0[0][i];
      GA[3 * i + 2] = -Gdc0[1][i] - Gdc1[2][i];
    }
    matmul3_nt(GA, Rm, GMm);
    matmul3_tn(Mm, GA, GRm);
#pragma unroll
    for (int i = 0; i < 9; ++i) GMn[i] = GMm[i];
  } else {  // RNF_LAYER_SMITH36
    float v[6], dv[3][6];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float u0 = Rm[h], u1 = Rm[3 + h], u2 = Rm[6 + h];
      v[3 * h] = u0; v[3 * h + 1] = u1; v[3 * h + 2] = u2;
      dv[0][3 * h] = u1; dv[0][3 * h + 1] = -u0; dv[0][3 * h + 2] = 0.0f;
      dv[1][3 * h] = u2; dv[1][3 * h + 1] = 0.0f; dv[1][3 * h + 2] = -u0;
      dv[2][3 * h] = 0.0f; dv[2][3 * h + 1] = u2; dv[2][3 * h + 2] = -u1;
    }
    float c0[3], c1[3], dc0[3][3], dc1[3][3];
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      float s = 0.0f, s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
#pragma unroll
      for (int b = 0; b < 6; ++b) {
        const float w = __ldg(Mn + 6 * a + b);
        s = fmaf(w, v[b], s); s0 = fmaf(w, dv[0][b], s0); s1 = fmaf(w, dv[1][b], s1); s2 = fmaf(w, dv[2][b], s2);
      }
      if (a < 3) { c0[a] = s; dc0[0][a] = s0; dc0[1][a] = s1; dc0[2][a] = s2; }
      else { c1[a - 3] = s; dc1[0][a - 3] = s0; dc1[1][a - 3] = s1; dc1[2][a - 3] = s2; }
    }
    float Gt[6], Gdt[3][6];
    {
      float Gc0[3], Gdc0[3][3], Gc1[3], Gdc1[3][3];
      smith_tail_bwd(c0, dc0, c1, dc1, Gp, g_ldj[n], Gc0, Gdc0, Gc1, Gdc1);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        Gt[i] = Gc0[i]; Gt[3 + i] = Gc1[i];
#pragma unroll
        for (int k = 0; k < 3; ++k) { Gdt[k][i] = Gdc0[k][i]; Gdt[k][3 + i] = Gdc1[k][i]; }
      }
    }
    float Gv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, Gdv[3][6];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int b = 0; b < 6; ++b) Gdv[k][b] = 0.0f;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
      for (int b = 0; b < 6; ++b) {
        const float w = __ldg(Mn + 6 * a + b);
        GMn[6 * a + b] = Gt[a] * v[b] + Gdt[0][a] * dv[0][b] + Gdt[1][a] * dv[1][b] + Gdt[2][a] * dv[2][b];
        Gv[b] = fmaf(w, Gt[a], Gv[b]);
        Gdv[0][b] = fmaf(w, Gdt[0][a], Gdv[0][b]); Gdv[1][b] = fmaf(w, Gdt[1][a], Gdv[1][b]); Gdv[2][b] = fmaf(w, Gdt[2][a], Gdv[2][b]);
      }
    }
    // through v = (r0, r1) and dv_k = (G_k r0, G_k r1); column 2 of R does not enter calculate_36
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int o = 3 * h;
      GRm[h] = Gv[o] - Gdv[0][o + 1] - Gdv[1][o + 2];
      GRm[3 + h] = Gv[o + 1] + Gdv[0][o] - Gdv[2][o + 2];
      GRm[6 + h] = Gv[o + 2] + Gdv[1][o] + Gdv[2][o + 1];
    }
    GRm[2] = GRm[5] = GRm[8] = 0.0f;
  }
  float g[3];
  tangent_of(Rm, GRm, g);
  gradient_from_tangent(Rm, g, G_R + n * 9);
}

}  // namespace

cudaError_t launch_train_mobius_fwd(const float* R, const float* out, int64_t N, int K, int perm, bool inverse, float* R_out, float* ldj,
                                    float* theta, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((N + 127) / 128);
  if (inverse) mobius_mixture_fwd_kernel<true><<<blocks, 128, 0, st>>>(R, out, N, K, perm, R_out, ldj, theta);
  else mobius_mixture_fwd_kernel<false><<<blocks, 128, 0, st>>>(R, out, N, K, perm, R_out, ldj, theta);
  return cudaGetLastError();
}

cudaError_t launch_train_mobius_bwd(const float* R, const float* out, int64_t N, int K, int perm, bool inverse, const float* theta,
                                    const float* R_out, const float* G_Rout, const float* g_ldj, float* G_R, float* G_out, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((N + 127) / 128);
  if (inverse) mobius_mixture_bwd_kernel<true><<<blocks, 128, 0, st>>>(R, out, N, K, perm, theta, R_out, G_Rout, g_ldj, G_R, G_out);
  else mobius_mixture_bwd_kernel<false><<<blocks, 128, 0, st>>>(R, out, N, K, perm, theta, R_out, G_Rout, g_ldj, G_R, G_out);
  return cudaGetLastError();
}

cudaError_t launch_train_affine_fwd(const float* R, const float* W, int64_t N, float* R_out, float* loglen, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  quat_affine_fwd_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(R, W, N, R_out, loglen);
  return cudaGetLastError();
}

cudaError_t launch_train_affine_bwd(const float* R, const float* W, int64_t N, const float* R_out, const float* G_Rout, const float* g_loglen,
                                    float* G_R, float* G_W, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  quat_affine_bwd_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(R, W, N, R_out, G_Rout, g_loglen, G_R, G_W);
  return cudaGetLastError();
}

cudaError_t launch_train_ablation_fwd(const float* R, const float* M, int64_t N, int kind, float* R_out, float* ldj, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  ablation_fwd_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(R, M, N, kind, R_out, ldj);
  return cudaGetLastError();
}

cudaError_t launch_train_ablation_bwd(const float* R, const float* M, int64_t N, int kind, const float* R_out, const float* G_Rout,
                                      const float* g_ldj, float* G_R, float* G_M, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((N + 127) / 128);
  switch (kind) {
    case RNF_LAYER_SMITH9: ablation_bwd_kernel<RNF_LAYER_SMITH9><<<blocks, 128, 0, st>>>(R, M, N, R_out, G_Rout, g_ldj, G_R, G_M); break;
    case RNF_LAYER_SMITH36: ablation_bwd_kernel<RNF_LAYER_SMITH36><<<blocks, 128, 0, st>>>(R, M, N, R_out, G_Rout, g_ldj, G_R, G_M); break;
    case RNF_LAYER_POLAR9L: ablation_bwd_kernel<RNF_LAYER_POLAR9L><<<blocks, 128, 0, st>>>(R, M, N, R_out, G_Rout, g_ldj, G_R, G_M); break;
    case RNF_LAYER_POLAR9R: ablation_bwd_kernel<RNF_LAYER_POLAR9R><<<blocks, 128, 0, st>>>(R, M, N, R_out, G_Rout, g_ldj, G_R, G_M); break;
    default: ablation_bwd_kernel<RNF_LAYER_RIGHT9><<<blocks, 128, 0, st>>>(R, M, N, R_out, G_Rout, g_ldj, G_R, G_M); break;
  }
  return cudaGetLastError();
}

int train_max_components() { return kMaxK; }

}  // namespace rnf
