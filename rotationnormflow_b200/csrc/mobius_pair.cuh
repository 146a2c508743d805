// mobius_pair.cuh -- the Mobius mixture arithmetic of mobius_fast.cuh, two components per instruction.
//
// sm_100 has packed FP32 arithmetic (PTX add / mul / fma .f32x2 -> SASS FADD2 / FMUL2 / FFMA2: one issue slot, two IEEE
// fp32 results; the second and third source may be a broadcast scalar register or a broadcast immediate).  The tcgen05 flow
// kernels are bound by instruction issue (ncu: issue slots 75 % active, FMA + ALU + XU pipes 50 / 30 / 44 %), and 2/3 of their
// instructions are this mixture, so components are evaluated in PAIRS: everything that is a multiply / add runs packed, only
// the SFU operations (ex2, lg2, sqrt, rcp), min / max and the selects stay scalar.  56 -> ~37 instructions per component.
//
// Column layout of one pair (the host permutes the fc_last rows accordingly, engine._last_layer_perm_pairs): 8 consecutive
// accumulator columns  (t_a, t_b, wx_a, wx_b, wy_a, wy_b, wz_a, wz_b)  with t = logit * log2(e) and w = 0.7 * centre (both factors are
// folded into the weights), so that a tcgen05.ld vector delivers every packed operand as an aligned register pair.
// Prepared parameters of a pair (inverse direction, kept in TMEM for the root search):
//   (-alpha'_a, -alpha'_b, -beta'_a, -beta'_b, 1 - |w'_a|^2, 1 - |w'_b|^2, weight_a, weight_b).
// The variants that lost or were superseded (logit clamp instead of the softplus select, degree-5 asin, two reciprocals + atan
// in the forward mixture, the inverse's probes with the full-circle angle wrap; DESIGN.md section 8b) were removed; their code
// is in commit d73682a.
#pragma once
#include "mobius_fast.cuh"

namespace rnf {

typedef unsigned long long f32x2;   // two fp32 in a 64-bit register pair: low word = component a, high word = component b

__device__ __forceinline__ f32x2 pk(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ f32x2 bc(float x) { return pk(x, x); }
__device__ __forceinline__ void upk(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float hsum(f32x2 v) {
  float lo, hi;
  upk(v, lo, hi);
  return lo + hi;
}
#define RNF_MAP2(out, in, fn) do { float l_, h_; upk(in, l_, h_); out = pk(fn(l_), fn(h_)); } while (0)

// asin(m) for a pair, |m| <= 1/sqrt 2, with s = m^2 supplied by the caller.  The angles of the mixture are asin of a sine
// (|sin| <= 0.7, see mixture_pairs and probe_delta_pairs) instead of atan of a quotient: no reciprocal on the SFU -- the XU pipe
// (8 cycles per warp instruction, tools/mufu_rate.cu) is the tightest unit of the mixture -- and a shorter polynomial:
// asin(m) = m + m s P(s), P of degree 6 (minimax fit, max abs error 4.4e-8 in fp32 Horner form, tests/test_fastmath.py).
__device__ __forceinline__ f32x2 asin_unit2_s(f32x2 m, f32x2 s) {
  f32x2 p = bc(0.12371734529733658f);
  p = fma2(p, s, bc(-0.11529727280139923f));
  p = fma2(p, s, bc(0.09339626878499985f));
  p = fma2(p, s, bc(0.01043224148452282f));
  p = fma2(p, s, bc(0.04762402921915054f));
  p = fma2(p, s, bc(0.07478351145982742f));
  p = fma2(p, s, bc(0.16667234897613525f));
  return fma2(mul2(p, s), m, m);
}

// NP pairs of mixture components, stage by stage.  raw[8 NP]: accumulator columns in the pair layout above; the centre rows
// arrive PRE-SCALED by 0.7 (engine.pack_mobius_tc), so with (a', b') = 0.7 (w.r, w.v) and u = 1 + |w| = 1 + |(a', b')| / 0.7
// the squashed centre of flow/mobiusflow.py:72 is w' = (a', b') / u.
// Mixture weight of a component, in units of ln 2:  softplus(a) / ln 2 = log2(1 + 2^t),  t = a log2(e).  theta' and
// log sum_k w_k f_k / sum_k w_k are ratios, so the common factor ln 2 never has to be applied.  torch's softplus is the
// identity above a = 20 (threshold), i.e. t above 20 log2(e) = 28.85; for 2^t < 2^-7 the series e (1 - e/2) / ln 2 replaces
// log2(1 + e), whose argument would round away e (absolute error of the weight <= 2e-7 either way: what matters is the error
// relative to the sum of the 64 weights).
// FWD: the evaluation point is the moving column itself, z = (zr, 0) with zr = -|x|, a point of the unit circle, on which the
// map of flow/mobiusflow.py:17-24 is the disk automorphism h = (z - w') / (1 - conj(w') z) (complex notation), so that
//     arg h = 2 arg(z - w') - arg z = 2 arg(z - w') - pi.
// Scaled by u (no reciprocal of u):  D = u (z - w') = (zr u - a', -b') =: (-Dn, -b'),  Dn > 0.3 u,  arg(z - w') = pi + atan(b' / Dn):
//     theta = pi + 2 atan(q),  q = b' / Dn,  |q| < tan(asin 0.7);   sum_k w_k theta_k = pi sum_k w_k + 2 sum_k w_k atan(q_k)
// -- no octant selects, and the angle does not wait for f (atan(q) is taken as asin(b' / |D|), see below).  The log-det term needs
//     f = (1 - |w'|^2) / |z - w'|^2 = (u^2 - |(a',b')|^2) / |D|^2,   |D|^2 = Dn^2 + b'^2.
// Accumulates (sum w, sum w atan q, sum w f) as packed partial sums (a-components in the low, b in the high word).
// !FWD: accumulates sum w (S_sp) and overwrites raw with the prepared parameters (-alpha', -beta', 1 - |w'|^2, weight);
// S_at and S_f are left as they are.
template <int NP, bool FWD>
__device__ __forceinline__ void mixture_pairs(const Plane& P, float zr, float zv, float* raw, f32x2& S_sp, f32x2& S_at, f32x2& S_f) {
  f32x2 sp[NP], ap[NP], bp[NP], bb[NP], n2[NP], u[NP], rt[NP];
  {
    f32x2 t[NP], e[NP], big[NP], small[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      t[j] = pk(raw[8 * j], raw[8 * j + 1]);
      RNF_MAP2(e[j], t[j], ex2_approx);
    }
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const f32x2 wx = pk(raw[8 * j + 2], raw[8 * j + 3]), wy = pk(raw[8 * j + 4], raw[8 * j + 5]), wz = pk(raw[8 * j + 6], raw[8 * j + 7]);
      ap[j] = fma2(wz, bc(P.r[2]), fma2(wy, bc(P.r[1]), mul2(wx, bc(P.r[0]))));
      bp[j] = fma2(wz, bc(P.v[2]), fma2(wy, bc(P.v[1]), mul2(wx, bc(P.v[0]))));
      bb[j] = mul2(bp[j], bp[j]);
      n2[j] = fma2(ap[j], ap[j], bb[j]);
      RNF_MAP2(rt[j], n2[j], sqrt_approx);
    }
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const f32x2 ope = add2(e[j], bc(1.0f));
      RNF_MAP2(big[j], ope, lg2_approx);
      small[j] = mul2(e[j], fma2(e[j], bc(-0.7213475204444817f), bc(1.4426950408889634f)));
      u[j] = fma2(rt[j], bc(1.4285714285714286f), bc(1.0f));            // 1 + |w|
    }
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      float tl, th, el, eh, bl, bh, sl, sh;
      upk(t[j], tl, th); upk(e[j], el, eh); upk(big[j], bl, bh); upk(small[j], sl, sh);
      const float vl = el < 0.0078125f ? sl : bl, vh = eh < 0.0078125f ? sh : bh;
      sp[j] = pk(tl > 28.853900817779268f ? tl : vl, th > 28.853900817779268f ? th : vh);
    }
  }
  if (FWD) {
    f32x2 f[NP], q[NP], qs[NP];
    const f32x2 nzr = bc(-zr);
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      // written without a single negation of a packed value (ptxas turns those into two LOP3 each): Dn = -D_r > 0
      const f32x2 Dn = fma2(nzr, u[j], ap[j]);
      const f32x2 DD = fma2(Dn, Dn, bb[j]);
      // u^2 - |(a',b')|^2 with |(a',b')| = rt:  1 + (2 / 0.7) rt + (1 / 0.49 - 1) rt^2  -- all terms positive
      const f32x2 num = fma2(fma2(rt[j], bc(1.0408163265306123f), bc(2.857142857142857f)), rt[j], bc(1.0f));
      // ONE SFU operation per component instead of two reciprocals (the XU pipe, 8 cycles per warp instruction, is the tightest
      // unit of the mixture: 10 -> 8 MUFU per pair): with rs = 1 / |D|,  sin(arg) = b' rs  and  1 / |D|^2 = rs^2, and since
      // Dn > 0 the angle atan(b' / Dn) = asin(b' rs), |b' rs| <= 0.7 (the squashed centre stays inside the disk of radius 0.7).
      f32x2 rs;
      RNF_MAP2(rs, DD, rsqrt_approx);
      const f32x2 rs2 = mul2(rs, rs);
      f[j] = mul2(num, rs2);
      q[j] = mul2(bp[j], rs);
      qs[j] = mul2(bb[j], rs2);
    }
    f32x2 at[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) at[j] = asin_unit2_s(q[j], qs[j]);
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      S_sp = add2(S_sp, sp[j]);
      S_at = fma2(sp[j], at[j], S_at);
      S_f = fma2(sp[j], f[j], S_f);
    }
  } else {
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      // -1 / u from the reciprocal of -u (a packed sign flip costs two LOP3: ncu r02, 4 % of the inverse kernel's instructions)
      const f32x2 nu = fma2(rt[j], bc(-1.4285714285714286f), bc(-1.0f));
      f32x2 nrc;
      RNF_MAP2(nrc, nu, rcp_approx);
      const f32x2 nal = mul2(ap[j], nrc), nbe = mul2(bp[j], nrc);
      const f32x2 omw = fma2(fma2(nal, nal, mul2(nbe, nbe)), bc(-1.0f), bc(1.0f));      // 1 - |w'|^2
      S_sp = add2(S_sp, sp[j]);
      upk(nal, raw[8 * j], raw[8 * j + 1]);
      upk(nbe, raw[8 * j + 2], raw[8 * j + 3]);
      upk(omw, raw[8 * j + 4], raw[8 * j + 5]);
      upk(sp[j], raw[8 * j + 6], raw[8 * j + 7]);
    }
  }
}

// wrapped mixture angle theta' = sum_k w_k theta_k / sum_k w_k from the forward sums of mixture_pairs
__device__ __forceinline__ float mixture_angle(float S_at, float inv_sp) { return fmaf(2.0f * S_at, inv_sp, kPi); }

// The same evaluation without any quadrant logic.  On the unit circle the Mobius map is the disk automorphism
// h = (z - w') / (1 - conj(w') z), so  theta_k = arg h = 2 arg(z - w') - t  with z = e^{it}; and because |w'| < 0.7 the direction of
// z - w' deviates from the direction of z by  delta_k = asin( (z x (z - w')) / |z - w'| ),  |sin delta_k| <= 0.7:
//     theta_k = t + 2 delta_k,      sum_k weight_k theta_k = t sum_k weight_k + 2 sum_k weight_k delta_k
// -- one rsqrt gives both sin(delta) and f = (1 - |w'|^2) / |z - w'|^2, the asin polynomial needs no min / max / select / copysign,
// and for t in [pi/2, 3pi/2] the result lies in (0.02, 6.27): already wrapped.  Accumulates Ds += weight delta (and Sf += weight f).
template <int NP, bool DERIV>
__device__ __forceinline__ void probe_delta_pairs(float zr, float zv, const float* prm, f32x2& Ds, f32x2& Sf) {
  f32x2 m[NP], ms[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const f32x2 nal = pk(prm[8 * j], prm[8 * j + 1]), nbe = pk(prm[8 * j + 2], prm[8 * j + 3]);
    const f32x2 dr = add2(nal, bc(zr)), dv = add2(nbe, bc(zv));          // z - w'
    const f32x2 dd = fma2(dv, dv, mul2(dr, dr));
    const f32x2 cr = fma2(dr, bc(-zv), mul2(dv, bc(zr)));                // z x (z - w') = cos t dv - sin t dr
    f32x2 rs;
    RNF_MAP2(rs, dd, rsqrt_approx);
    const f32x2 rs2 = mul2(rs, rs);
    m[j] = mul2(cr, rs);
    ms[j] = mul2(m[j], m[j]);                                           // one multiply less than (cr^2) rs2; one step longer chain
    if (DERIV) Sf = fma2(pk(prm[8 * j + 6], prm[8 * j + 7]), mul2(pk(prm[8 * j + 4], prm[8 * j + 5]), rs2), Sf);
  }
#pragma unroll
  for (int j = 0; j < NP; ++j) Ds = fma2(pk(prm[8 * j + 6], prm[8 * j + 7]), asin_unit2_s(m[j], ms[j]), Ds);
}

// sum_k weight_k f_k(z) over NP prepared pairs (log-det of the inverse direction, flow/mobiusflow.py:169-181)
template <int NP>
__device__ __forceinline__ void jacobian_pairs(float zr, float zv, const float* prm, f32x2& Sf) {
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const f32x2 dr = add2(pk(prm[8 * j], prm[8 * j + 1]), bc(zr)), dv = add2(pk(prm[8 * j + 2], prm[8 * j + 3]), bc(zv));
    const f32x2 dd = fma2(dv, dv, mul2(dr, dr));
    f32x2 rc;
    RNF_MAP2(rc, dd, rcp_approx);
    Sf = fma2(pk(prm[8 * j + 6], prm[8 * j + 7]), mul2(pk(prm[8 * j + 4], prm[8 * j + 5]), rc), Sf);
  }
}

}  // namespace rnf
