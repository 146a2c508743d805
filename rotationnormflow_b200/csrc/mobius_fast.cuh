// mobius_fast.cuh -- single-instruction SFU primitives and the per-row frame of the tensor-core flow kernels.
//
// Same mathematics as mobius_math.cuh (flow/mobiusflow.py:17-24,62-72,94-125,196-245), restated for the Mobius layers of
// flow_t4.cu and flow_row.cu, whose mixture arithmetic is in mobius_pair.cuh:
//   * every w_k is projected onto the plane orthogonal to y (flow/mobiusflow.py:62-63) and r, v span that plane, so the
//     projected centre is (alpha, beta) = (w.r, w.v): the projection, the 3-D norms and the two 3-D dot products of
//     h with (r, v) collapse to 2-D arithmetic (the reference's own frame is orthonormal to ~1e-7, the same order as one
//     fp32 rounding of these quantities);
//   * 1/x, sqrt, 2^x, log2 use the SFU approximations (rcp/sqrt.approx: <= 1 ulp; ex2/lg2.approx: ~2^-22), whose errors
//     enter theta' = sum_k pi_k theta_k and log sum_k pi_k f_k averaged over the 64 components.
// The scalar mixture that mobius_pair.cuh replaced (atan2 polynomial, softplus, four components stage by stage) was removed;
// its code is in commit d73682a.
// Accuracy against the float64 reference is asserted end-to-end by tests/test_gpu_parity.py in "tc" mode.
#pragma once
#include <cuda_runtime.h>

#include "mobius_math.cuh"

namespace rnf {

__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// log(x) through the SFU: lg2.approx (absolute error <= 2^-22 on the result) times ln 2.  Used for the log-det terms, which
// are O(1) per layer and checked at 1e-4 relative after 42-49 layers.
__device__ __forceinline__ float log_fast(float x) { return 0.6931471805599453f * lg2_approx(x); }

// sin and cos of t in [0, 2 pi] (mixture angles and bisection probes never leave that range): quadrant by the magic-number
// round of t * 2/pi, two-constant Cody-Waite reduction to [-pi/4, pi/4], degree-7 / degree-8 minimax polynomials (the
// classic single-precision kernels).  Max abs error 9e-8 (tests/test_fastmath.py); ~20 instructions, no slow path.
__device__ __forceinline__ void sincos_2pi(float t, float& sn, float& cs) {
  const float kbig = fmaf(t, 0.63661977236758134f, 12582912.0f);        // 1.5 * 2^23: the integer lands in the low mantissa bits
  const int q = __float_as_int(kbig);
  const float kf = kbig - 12582912.0f;
  float r = fmaf(kf, -1.5707963705062866f, t);
  r = fmaf(kf, 4.371138828673793e-08f, r);
  const float z = r * r;
  float ps = fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f);
  ps = fmaf(ps, z, -1.6666654611e-1f);
  const float s = fmaf(ps * z, r, r);
  float pc = fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f);
  pc = fmaf(pc, z, 4.166664568298827e-2f);
  const float c = fmaf(pc * z, z, fmaf(-0.5f, z, 1.0f));
  const float a = (q & 1) ? c : s, b = (q & 1) ? s : c;                  // odd quadrant: sin <-> cos
  sn = (q & 2) ? -a : a;
  cs = ((q + 1) & 2) ? -b : b;
}

// point on the circle: z = r cos(t) + v sin(t), t in [0, 2 pi]            (flow/mobiusflow.py:102,169,231)
__device__ __forceinline__ void circle_point_fast(const float r[3], const float v[3], float t, float z[3]) {
  float s, c;
  sincos_2pi(t, s, c);
  z[0] = fmaf(v[0], s, r[0] * c);
  z[1] = fmaf(v[1], s, r[1] * c);
  z[2] = fmaf(v[2], s, r[2] * c);
}

// Per-layer constants of a row: frame (r, v).
struct Plane {
  float r[3], v[3];
};

// r = -x/|x| ; v = (y x r)/|y x r|   (flow/mobiusflow.py:64-67) with Newton-refined rsqrt instead of sqrt + 3 divisions
__device__ __forceinline__ void make_frame_fast(const float x[3], const float y[3], Plane& P) {
  P.r[0] = -x[0]; P.r[1] = -x[1]; P.r[2] = -x[2];
  normalize3_fast(P.r);
  cross3(y, P.r, P.v);
  normalize3_fast(P.v);
}

}  // namespace rnf
