// so3_math.cuh -- per-rotation SO(3) / quaternion arithmetic kept entirely in registers.
//
// Follows (reference file:line, relative to the reference root):
//   pytorch3d.transforms.matrix_to_quaternion / quaternion_to_matrix  (public 0.7.x definitions; called at
//       flow/squeezetrans.py:34,37 and flow/rottrans.py:18-20)
//   calculate_16                      flow/squeezetrans.py:33-38
//   my_det_4_4 / my_det_3_3           flow/squeezetrans.py:10-22
#pragma once
#include <cuda_runtime.h>

namespace rnf {

__device__ __forceinline__ void cross3(const float a[3], const float b[3], float o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}

__device__ __forceinline__ float dot3(const float a[3], const float b[3]) {
  return fmaf(a[2], b[2], fmaf(a[1], b[1], a[0] * b[0]));
}

__device__ __forceinline__ void normalize3(float a[3]) {
  const float n = sqrtf(dot3(a, a));
  a[0] = a[0] / n;
  a[1] = a[1] / n;
  a[2] = a[2] / n;
}

// column p of R / write column p, by selects (a runtime index into a register array would put it in local memory)
__device__ __forceinline__ float sel3(int p, float a, float b, float c) { return p == 0 ? a : (p == 1 ? b : c); }
__device__ __forceinline__ void get_col(const float R[9], int p, float o[3]) {
  o[0] = sel3(p, R[0], R[1], R[2]);
  o[1] = sel3(p, R[3], R[4], R[5]);
  o[2] = sel3(p, R[6], R[7], R[8]);
}
__device__ __forceinline__ void set_col(float R[9], int p, const float c[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    R[3 * i + 0] = p == 0 ? c[i] : R[3 * i + 0];
    R[3 * i + 1] = p == 1 ? c[i] : R[3 * i + 1];
    R[3 * i + 2] = p == 2 ? c[i] : R[3 * i + 2];
  }
}

// vee(R^T G): tangent (body frame) vector of a matrix gradient G at R, g_i = <G, R [e_i]x>
__device__ __forceinline__ void tangent_of(const float R[9], const float G[9], float g[3]) {
  float H[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) H[3 * i + j] = R[i] * G[j] + R[3 + i] * G[3 + j] + R[6 + i] * G[6 + j];
  g[0] = H[7] - H[5];
  g[1] = H[2] - H[6];
  g[2] = H[3] - H[1];
}

// G_R = R [g]x / 2
__device__ __forceinline__ void gradient_from_tangent(const float R[9], const float g[3], float G[9]) {
  const float h[9] = {0.0f, -g[2], g[1], g[2], 0.0f, -g[0], -g[1], g[0], 0.0f};
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) G[3 * i + j] = 0.5f * (R[3 * i] * h[j] + R[3 * i + 1] * h[3 + j] + R[3 * i + 2] * h[6 + j]);
}

// E(q) omega = q (x) (0, omega): the 4x3 matrix of a body-frame perturbation of a unit quaternion (real first), and E(q)^T d
__device__ __forceinline__ void E_mul(const float q[4], const float w[3], float o[4]) {
  o[0] = -q[1] * w[0] - q[2] * w[1] - q[3] * w[2];
  o[1] = q[0] * w[0] - q[3] * w[1] + q[2] * w[2];
  o[2] = q[3] * w[0] + q[0] * w[1] - q[1] * w[2];
  o[3] = -q[2] * w[0] + q[1] * w[1] + q[0] * w[2];
}
__device__ __forceinline__ void ET_mul(const float q[4], const float d[4], float o[3]) {
  o[0] = -q[1] * d[0] + q[0] * d[1] + q[3] * d[2] - q[2] * d[3];
  o[1] = -q[2] * d[0] - q[3] * d[1] + q[0] * d[2] + q[1] * d[3];
  o[2] = -q[3] * d[0] + q[2] * d[1] - q[1] * d[2] + q[0] * d[3];
}

// R (row-major 3x3) -> quaternion (real first).  Only the winning candidate row of the public
// algorithm is evaluated: argmax_i q_abs_i == argmax_i (q_abs_i^2) and that maximum is >= 1 because the
// four radicands sum to 4, so the 0.1 floor of the public code can never be active on it.
__device__ __forceinline__ void mat_to_quat(const float m[9], float q[4]) {
  const float m00 = m[0], m01 = m[1], m02 = m[2], m10 = m[3], m11 = m[4], m12 = m[5], m20 = m[6], m21 = m[7], m22 = m[8];
  const float a0 = 1.0f + m00 + m11 + m22;
  const float a1 = 1.0f + m00 - m11 - m22;
  const float a2 = 1.0f - m00 + m11 - m22;
  const float a3 = 1.0f - m00 - m11 + m22;
  int best = 0;
  float am = a0;
  if (a1 > am) { am = a1; best = 1; }
  if (a2 > am) { am = a2; best = 2; }
  if (a3 > am) { am = a3; best = 3; }
  const float qa = sqrtf(fmaxf(am, 0.0f));
  const float d = 2.0f * fmaxf(qa, 0.1f);
  const float qq = qa * qa;
  float c0, c1, c2, c3;
  if (best == 0)      { c0 = qq;        c1 = m21 - m12; c2 = m02 - m20; c3 = m10 - m01; }
  else if (best == 1) { c0 = m21 - m12; c1 = qq;        c2 = m10 + m01; c3 = m02 + m20; }
  else if (best == 2) { c0 = m02 - m20; c1 = m10 + m01; c2 = qq;        c3 = m12 + m21; }
  else                { c0 = m10 - m01; c1 = m20 + m02; c2 = m21 + m12; c3 = qq; }
  q[0] = c0 / d; q[1] = c1 / d; q[2] = c2 / d; q[3] = c3 / d;
}

// quaternion (real first, any non-zero norm) -> R, two_s = 2/|q|^2 as in the public definition.
__device__ __forceinline__ void quat_to_mat(const float q[4], float m[9]) {
  const float r = q[0], i = q[1], j = q[2], k = q[3];
  const float two_s = 2.0f / (r * r + i * i + j * j + k * k);
  m[0] = 1.0f - two_s * (j * j + k * k);
  m[1] = two_s * (i * j - k * r);
  m[2] = two_s * (i * k + j * r);
  m[3] = two_s * (i * j + k * r);
  m[4] = 1.0f - two_s * (i * i + k * k);
  m[5] = two_s * (j * k - i * r);
  m[6] = two_s * (i * k - j * r);
  m[7] = two_s * (j * k + i * r);
  m[8] = 1.0f - two_s * (i * i + j * j);
}

// calculate_16: R <- q2m(Wq/|Wq|); returns log|Wq| (caller forms logabsdet - 4*log|Wq|).
// W is 16 floats row-major reachable through a generic pointer (shared, global or constant).
__device__ __forceinline__ float quat_affine(const float* __restrict__ W, float R[9]) {
  float q[4], p[4];
  mat_to_quat(R, q);
#pragma unroll
  for (int a = 0; a < 4; ++a)
    p[a] = fmaf(W[4 * a + 3], q[3], fmaf(W[4 * a + 2], q[2], fmaf(W[4 * a + 1], q[1], W[4 * a] * q[0])));
  const float len = sqrtf(p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3]);
#pragma unroll
  for (int a = 0; a < 4; ++a) p[a] = p[a] / len;
  quat_to_mat(p, R);
  return logf(len);
}


// ---- single-SFU-instruction variants used by the tensor-core kernels (flow_t4.cu, flow_row.cu) -------------------------------------
// rcp / rsqrt approximations (<= 1 ulp) followed by one Newton step: ~0.5-1 ulp, no IEEE slow path, no branches.
__device__ __forceinline__ float rcp_nr(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return fmaf(fmaf(-x, r, 1.0f), r, r);
}
__device__ __forceinline__ float rsqrt_nr(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  const float h = 0.5f * x * r;
  return fmaf(fmaf(-h, r, 0.5f), r, r);               // r (1.5 - 0.5 x r^2)
}
__device__ __forceinline__ void normalize3_fast(float a[3]) {
  const float inv = rsqrt_nr(dot3(a, a));
  a[0] *= inv; a[1] *= inv; a[2] *= inv;
}

// calculate_16 without the intermediate normalisations.  quaternion_to_matrix is scale invariant (two_s = 2/|q|^2), so
// the candidate row of matrix_to_quaternion can stay un-divided: q~ = 2 q_abs q with winning entry q_abs^2 = the radicand,
// p~ = W q~ = 2 q_abs p, R' = q2m(p~) and log|Wq| = 0.5 log(|p~|^2 / (4 q_abs^2)).  No sqrt, two reciprocals, one log.
__device__ __forceinline__ float quat_affine_fast(const float* __restrict__ W, float R[9]) {
  const float m00 = R[0], m01 = R[1], m02 = R[2], m10 = R[3], m11 = R[4], m12 = R[5], m20 = R[6], m21 = R[7], m22 = R[8];
  const float a0 = 1.0f + m00 + m11 + m22;
  const float a1 = 1.0f + m00 - m11 - m22;
  const float a2 = 1.0f - m00 + m11 - m22;
  const float a3 = 1.0f - m00 - m11 + m22;
  int best = 0;
  float am = a0;
  if (a1 > am) { am = a1; best = 1; }
  if (a2 > am) { am = a2; best = 2; }
  if (a3 > am) { am = a3; best = 3; }
  float q[4];
  if (best == 0)      { q[0] = am;        q[1] = m21 - m12; q[2] = m02 - m20; q[3] = m10 - m01; }
  else if (best == 1) { q[0] = m21 - m12; q[1] = am;        q[2] = m10 + m01; q[3] = m02 + m20; }
  else if (best == 2) { q[0] = m02 - m20; q[1] = m10 + m01; q[2] = am;        q[3] = m12 + m21; }
  else                { q[0] = m10 - m01; q[1] = m20 + m02; q[2] = m21 + m12; q[3] = am; }
  float p[4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
    p[a] = fmaf(W[4 * a + 3], q[3], fmaf(W[4 * a + 2], q[2], fmaf(W[4 * a + 1], q[1], W[4 * a] * q[0])));
  const float pp = fmaf(p[3], p[3], fmaf(p[2], p[2], fmaf(p[1], p[1], p[0] * p[0])));
  const float two_s = 2.0f * rcp_nr(pp);
  const float r = p[0], i = p[1], j = p[2], k = p[3];
  const float si = two_s * i, sj = two_s * j, sk = two_s * k;
  R[0] = 1.0f - fmaf(sj, j, sk * k);
  R[1] = fmaf(si, j, -sk * r);
  R[2] = fmaf(si, k, sj * r);
  R[3] = fmaf(si, j, sk * r);
  R[4] = 1.0f - fmaf(si, i, sk * k);
  R[5] = fmaf(sj, k, -si * r);
  R[6] = fmaf(si, k, -sj * r);
  R[7] = fmaf(sj, k, si * r);
  R[8] = 1.0f - fmaf(si, i, sj * j);
  float l2;                                          // log through the SFU (lg2.approx: absolute error <= 2^-22)
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(pp * rcp_nr(4.0f * am)));
  return 0.34657359027997264f * l2;                  // 0.5 ln 2
}

// Geodesic angle from R to the closest of K ground-truth rotations: acos(clip((max_k sum_ij R_ij GT_kij - 1) / 2, -1, 1))
// (min_geodesic_distance_rotmats, utils/utils.py:231-235).  Weight of the spread metric  sum_g p_g d(R_g, R_gt) / sum_g p_g.
__device__ __forceinline__ float gt_distance(const float* __restrict__ gt, int K, const float R[9]) {
  float best = -INFINITY;
  for (int k = 0; k < K; ++k) {
    float tr = 0.0f;
#pragma unroll
    for (int i = 0; i < 9; ++i) tr = fmaf(R[i], __ldg(gt + k * 9 + i), tr);
    best = fmaxf(best, tr);
  }
  return acosf(fminf(fmaxf((best - 1.0f) * 0.5f, -1.0f), 1.0f));
}

__host__ __device__ inline float det3f(float a00, float a01, float a02, float a10, float a11, float a12, float a20,
                                       float a21, float a22) {
  const float d00 = a11 * a22 - a12 * a21;
  const float d01 = a12 * a20 - a10 * a22;
  const float d02 = a10 * a21 - a11 * a20;
  return d00 * a00 + d01 * a01 + d02 * a02;
}

// cofactor expansion along row 0, the operation order of my_det_4_4 (flow/squeezetrans.py:17-22)
__host__ __device__ inline float det4f(const float* A) {
#define RNF_A(r, c) A[4 * (r) + (c)]
  const float d0 = RNF_A(0, 0) * det3f(RNF_A(1, 1), RNF_A(1, 2), RNF_A(1, 3), RNF_A(2, 1), RNF_A(2, 2), RNF_A(2, 3), RNF_A(3, 1), RNF_A(3, 2), RNF_A(3, 3));
  const float d1 = RNF_A(0, 1) * det3f(RNF_A(1, 0), RNF_A(1, 2), RNF_A(1, 3), RNF_A(2, 0), RNF_A(2, 2), RNF_A(2, 3), RNF_A(3, 0), RNF_A(3, 2), RNF_A(3, 3));
  const float d2 = RNF_A(0, 2) * det3f(RNF_A(1, 0), RNF_A(1, 1), RNF_A(1, 3), RNF_A(2, 0), RNF_A(2, 1), RNF_A(2, 3), RNF_A(3, 0), RNF_A(3, 1), RNF_A(3, 3));
  const float d3 = RNF_A(0, 3) * det3f(RNF_A(1, 0), RNF_A(1, 1), RNF_A(1, 2), RNF_A(2, 0), RNF_A(2, 1), RNF_A(2, 2), RNF_A(3, 0), RNF_A(3, 1), RNF_A(3, 2));
#undef RNF_A
  return d0 - d1 + d2 - d3;
}

}  // namespace rnf
