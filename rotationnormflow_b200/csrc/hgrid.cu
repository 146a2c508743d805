// hgrid.cu -- coarse-to-fine search on the HEALPix SO(3) grids (DESIGN 4.8): the children of grid indices and a per-image top-K.
//
// Children.  Grid index idx = t * npix + p at level l (healpix_rot.cuh): nside = 2^l, npix = 12 nside^2, p the RING pixel, t the tilt.
// The 8 children at level l + 1 are, for k = 4 * dt + j (dt = 0, 1; j = 0..3),
//   t' = 2 t + dt,   p' = nest2ring(2 nside, 4 ring2nest(nside, p) + j)          (the public HEALPix NESTED subdivision)
// so every level-(l+1) index has exactly one parent and the children of all level-l indices partition the level-(l+1) grid.  A
// child's rotation is healpix_rotation at its index, times the offset by the fmaf chain of the grid kernels (flow_t4.cu), so it is
// bit for bit the rotation Flow.grid_log_prob scores at that index.  A parent outside [0, 72 * 8^l) (padding: -1) gives children -1
// and NaN rotations and reads nothing.
//
// Top-K.  values [B,C] with int64 indices (or the column number): per image the K best entries under the order of the grid arg-max
// (grid_red_better: NaN first, then the larger value, then the lower index), best first.  An entry with a negative index is padding:
// it ranks after every entry with an index >= 0 and comes out as (-inf, -1), as do the places past C when K > C.  A slice stage
// bitonic-sorts slices of W = max(4096, 2 Kp) entries (Kp = K rounded up to a power of two) in shared memory, one CTA per (image,
// slice), and keeps the Kp best of each; merge rounds then fold the sorted lists pairwise, in place, in a fixed tree.  No atomics
// and no host synchronisation: the result is bitwise reproducible and the launches can be captured in a CUDA graph.
#include <math.h>

#include "healpix_rot.cuh"
#include "rnf_common.cuh"

namespace rnf {
namespace {

// the base-pixel tables of HEALPix: jrll = {2,2,2,2,3,3,3,3,4,4,4,4}, jpll = {1,3,5,7,0,2,4,6,1,3,5,7}
__device__ __forceinline__ long long jrll(long long face) { return 2 + (face >> 2); }
__device__ __forceinline__ long long jpll(long long face) { return 2 * (face & 3) + ((face >> 2) == 1 ? 0 : 1); }

__device__ __forceinline__ long long spread_bits(long long v) {   // bit i -> bit 2i (v < 2^29)
  unsigned long long x = (unsigned long long)v;
  x = (x | (x << 16)) & 0x0000FFFF0000FFFFULL;
  x = (x | (x << 8)) & 0x00FF00FF00FF00FFULL;
  x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0FULL;
  x = (x | (x << 2)) & 0x3333333333333333ULL;
  x = (x | (x << 1)) & 0x5555555555555555ULL;
  return (long long)x;
}

__device__ __forceinline__ long long compress_bits(long long v) {  // bit 2i -> bit i
  unsigned long long x = (unsigned long long)v & 0x5555555555555555ULL;
  x = (x | (x >> 1)) & 0x3333333333333333ULL;
  x = (x | (x >> 2)) & 0x0F0F0F0F0F0F0F0FULL;
  x = (x | (x >> 4)) & 0x00FF00FF00FF00FFULL;
  x = (x | (x >> 8)) & 0x0000FFFF0000FFFFULL;
  x = (x | (x >> 16)) & 0x00000000FFFFFFFFULL;
  return (long long)x;
}

// RING pixel -> NESTED pixel (HEALPix ring2xyf + xyf2nest)
__device__ long long ring2nest(long long nside, long long pix) {
  const long long nl2 = 2 * nside, ncap = 2 * nside * (nside - 1), npix = 12 * nside * nside;
  long long iring, iphi, kshift, nr, face;
  if (pix < ncap) {
    iring = (1 + isqrt_ll(1 + 2 * pix)) >> 1;
    iphi = pix + 1 - 2 * iring * (iring - 1);
    kshift = 0;
    nr = iring;
    face = (iphi - 1) / nr;
  } else if (pix < npix - ncap) {
    const long long ip = pix - ncap, tmp = ip / (4 * nside);
    iring = tmp + nside;
    iphi = ip - tmp * 4 * nside + 1;
    kshift = (iring + nside) & 1;
    nr = nside;
    const long long ire = tmp + 1, irm = nl2 + 2 - ire;
    const long long ifm = (iphi - (ire >> 1) + nside - 1) / nside, ifp = (iphi - (irm >> 1) + nside - 1) / nside;
    face = (ifp == ifm) ? (ifp | 4) : ((ifp < ifm) ? ifp : (ifm + 8));
  } else {
    const long long ip = npix - pix;
    iring = (1 + isqrt_ll(2 * ip - 1)) >> 1;
    iphi = 4 * iring + 1 - (ip - 2 * iring * (iring - 1));
    kshift = 0;
    nr = iring;
    iring = 2 * nl2 - iring;
    face = 8 + (iphi - 1) / nr;
  }
  const long long irt = iring - jrll(face) * nside + 1;
  long long ipt = 2 * iphi - jpll(face) * nr - kshift - 1;
  if (ipt >= nl2) ipt -= 8 * nside;
  const long long ix = (ipt - irt) >> 1, iy = (-ipt - irt) >> 1;
  return face * nside * nside + spread_bits(ix) + (spread_bits(iy) << 1);
}

// NESTED pixel -> RING pixel (HEALPix nest2xyf + xyf2ring)
__device__ long long nest2ring(long long nside, long long pix) {
  const long long npface = nside * nside, npix = 12 * npface, ncap = 2 * nside * (nside - 1), nl4 = 4 * nside;
  const long long face = pix / npface, sub = pix % npface;
  const long long ix = compress_bits(sub), iy = compress_bits(sub >> 1);
  const long long jr = jrll(face) * nside - ix - iy - 1;
  long long nr, kshift, n_before;
  if (jr < nside) {
    nr = jr;
    n_before = 2 * nr * (nr - 1);
    kshift = 0;
  } else if (jr > 3 * nside) {
    nr = nl4 - jr;
    n_before = npix - 2 * (nr + 1) * nr;
    kshift = 0;
  } else {
    nr = nside;
    n_before = ncap + (jr - nside) * nl4;
    kshift = (jr - nside) & 1;
  }
  long long jp = (jpll(face) * nr + ix - iy + 1 + kshift) / 2;
  if (jp > nl4) jp -= nl4;
  else if (jp < 1) jp += nl4;
  return n_before + jp - 1;
}

// one thread per (parent, child k)
__global__ void __launch_bounds__(256) healpix_children_kernel(int level, const int64_t* __restrict__ parent, int64_t n,
                                                               const float* __restrict__ offset, int64_t* __restrict__ child_out,
                                                               float* __restrict__ R_out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * 8) return;
  const int64_t i = e >> 3;
  const int k = (int)(e & 7);
  const long long nside = 1LL << level, npix = 12 * nside * nside;
  const long long idx = parent[i];
  float* o = R_out + e * 9;
  if (idx < 0 || idx >= 6 * nside * npix) {
    child_out[e] = -1;
#pragma unroll
    for (int q = 0; q < 9; ++q) o[q] = __int_as_float(0x7fffffff);
    return;
  }
  const long long t = idx / npix, p = idx % npix;
  const long long pc = nest2ring(2 * nside, 4 * ring2nest(nside, p) + (k & 3));
  const long long c = (2 * t + (k >> 2)) * (4 * npix) + pc;
  child_out[e] = c;
  float Gm[9];
  healpix_rotation(level + 1, c, Gm);
  if (offset != nullptr) {            // grid @ offset, the fmaf chain of flow_t4.cu (grid mode)
    float O[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) O[q] = __ldg(offset + q);
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) o[3 * a + b] = fmaf(Gm[3 * a + 2], O[6 + b], fmaf(Gm[3 * a + 1], O[3 + b], Gm[3 * a] * O[b]));
  } else {
#pragma unroll
    for (int q = 0; q < 9; ++q) o[q] = Gm[q];
  }
}

// ---- top-K ----------------------------------------------------------------------------------------------------------------------
constexpr int kTopkThreads = 512;
constexpr int64_t kTopkMinSlice = 4096;

// a before b: padding (index < 0) never, else the order of the grid arg-max
__device__ __forceinline__ bool topk_better(float av, long long ai, float bv, long long bi) {
  if (ai < 0) return false;
  if (bi < 0) return true;
  return grid_red_better(av, ai, bv, bi);
}

// in-place bitonic network over n = 2^m entries of (s_v, s_i): best first.  `first_k` > 1 skips the merges of sub-sequences shorter
// than first_k (the input is made of sorted runs of that length, alternately best-first and worst-first: a bitonic merge input)
__device__ void bitonic(float* s_v, long long* s_i, int n, int first_k) {
  for (int k = first_k; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = i + j;
        const bool best_first = (i & k) == 0;
        const float vi = s_v[i], vl = s_v[l];
        const long long ii = s_i[i], il = s_i[l];
        const bool sw = best_first ? topk_better(vl, il, vi, ii) : topk_better(vi, ii, vl, il);
        if (sw) {
          s_v[i] = vl; s_v[l] = vi;
          s_i[i] = il; s_i[l] = ii;
        }
      }
      __syncthreads();
    }
  }
}

// write the first `count` sorted entries: to a workspace list (all Kp, as they are) or to the output (K, padding canonical)
__device__ __forceinline__ void topk_emit(const float* s_v, const long long* s_i, int count, float* v_out, int64_t* i_out, bool final) {
  for (int t = threadIdx.x; t < count; t += blockDim.x) {
    const long long ii = s_i[t];
    const bool pad = final && ii < 0;
    v_out[t] = pad ? -INFINITY : s_v[t];
    i_out[t] = pad ? -1 : ii;
  }
}

// grid (B, S): sort slice s of image b (W entries, padded), keep its Kp best in list s of the image (or the K best in the output
// when S == 1)
__global__ void __launch_bounds__(kTopkThreads) topk_slice_kernel(const float* __restrict__ values, const int64_t* __restrict__ index,
                                                                 int64_t C, int W, int Kp, int K, float* __restrict__ ws_v,
                                                                 int64_t* __restrict__ ws_i, float* __restrict__ v_out,
                                                                 int64_t* __restrict__ i_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  long long* s_i = reinterpret_cast<long long*>(smem);
  float* s_v = reinterpret_cast<float*>(smem + (size_t)W * sizeof(long long));
  const int64_t b = blockIdx.x, s = blockIdx.y, S = gridDim.y;
  const int64_t g0 = s * (int64_t)W;
  for (int t = threadIdx.x; t < W; t += blockDim.x) {
    const int64_t g = g0 + t;
    if (g < C) {
      s_v[t] = values[b * C + g];
      s_i[t] = index != nullptr ? (long long)index[b * C + g] : (long long)g;
    } else {
      s_v[t] = -INFINITY;
      s_i[t] = -1;
    }
  }
  __syncthreads();
  bitonic(s_v, s_i, W, 2);
  if (S == 1) topk_emit(s_v, s_i, K, v_out + b * K, i_out + b * K, true);
  else topk_emit(s_v, s_i, Kp, ws_v + (b * S + s) * Kp, ws_i + (b * S + s) * Kp, false);
}

// grid (B, pairs): merge list 2 p step and list (2 p + 1) step of image b into list 2 p step (in place: no other CTA of the round
// touches either list); the last round (one pair) writes the output
__global__ void __launch_bounds__(kTopkThreads) topk_merge_kernel(int64_t S, int64_t step, int Kp, int K, float* __restrict__ ws_v,
                                                                 int64_t* __restrict__ ws_i, float* __restrict__ v_out,
                                                                 int64_t* __restrict__ i_out, int final) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = 2 * Kp;
  long long* s_i = reinterpret_cast<long long*>(smem);
  float* s_v = reinterpret_cast<float*>(smem + (size_t)n * sizeof(long long));
  const int64_t b = blockIdx.x;
  const int64_t la = 2 * (int64_t)blockIdx.y * step, lb = la + step;
  const float* av = ws_v + (b * S + la) * Kp;
  const int64_t* ai = ws_i + (b * S + la) * Kp;
  for (int t = threadIdx.x; t < Kp; t += blockDim.x) {
    s_v[t] = av[t];
    s_i[t] = ai[t];
    // the second list reversed (worst first): the two together are a bitonic sequence
    if (lb < S) {
      s_v[n - 1 - t] = ws_v[(b * S + lb) * Kp + t];
      s_i[n - 1 - t] = ws_i[(b * S + lb) * Kp + t];
    } else {
      s_v[n - 1 - t] = -INFINITY;
      s_i[n - 1 - t] = -1;
    }
  }
  __syncthreads();
  bitonic(s_v, s_i, n, n);
  if (final) topk_emit(s_v, s_i, K, v_out + b * K, i_out + b * K, true);
  else topk_emit(s_v, s_i, Kp, ws_v + (b * S + la) * Kp, ws_i + (b * S + la) * Kp, false);
}

struct TopkShape {
  int Kp, W;
  int64_t S;
};

TopkShape topk_shape(int64_t C, int K) {
  TopkShape t;
  t.Kp = 1;
  while (t.Kp < K) t.Kp <<= 1;
  t.W = (int)(2 * (int64_t)t.Kp > kTopkMinSlice ? 2 * (int64_t)t.Kp : kTopkMinSlice);
  t.S = C > 0 ? (C + t.W - 1) / t.W : 1;
  return t;
}

}  // namespace

int64_t topk_slices(int64_t C, int K) { return topk_shape(C, K).S; }

// workspace: values [B][S][Kp] float, then indices [B][S][Kp] int64 (none when one slice covers the row)
int64_t topk_workspace_bytes(int64_t B, int64_t C, int K) {
  const TopkShape t = topk_shape(C, K);
  if (t.S == 1) return 0;
  const int64_t n = B * t.S * t.Kp;
  return ((n * 4 + 255) & ~(int64_t)255) + n * 8;
}

cudaError_t launch_healpix_children(int level, const int64_t* parent, int64_t n, const float* offset, int64_t* child_out, float* R_out,
                                    cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  const int64_t blocks = (n * 8 + 255) / 256;
  healpix_children_kernel<<<(unsigned)blocks, 256, 0, st>>>(level, parent, n, offset, child_out, R_out);
  return cudaGetLastError();
}

cudaError_t launch_topk(const float* values, const int64_t* index, int64_t B, int64_t C, int K, void* workspace, float* v_out,
                        int64_t* i_out, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  const TopkShape t = topk_shape(C, K);
  const size_t slice_smem = (size_t)t.W * 12, merge_smem = (size_t)t.Kp * 24;
  cudaError_t e = cudaFuncSetAttribute(topk_slice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slice_smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)merge_smem);
  if (e != cudaSuccess) return e;
  const int64_t n = B * t.S * t.Kp;
  float* ws_v = (float*)workspace;
  int64_t* ws_i = t.S > 1 ? (int64_t*)((char*)workspace + ((n * 4 + 255) & ~(int64_t)255)) : nullptr;
  topk_slice_kernel<<<dim3((unsigned)B, (unsigned)t.S), kTopkThreads, slice_smem, st>>>(values, index, C, t.W, t.Kp, K, ws_v, ws_i, v_out,
                                                                                        i_out);
  e = cudaGetLastError();
  for (int64_t step = 1; e == cudaSuccess && step < t.S; step <<= 1) {
    const int64_t pairs = (t.S + 2 * step - 1) / (2 * step);
    topk_merge_kernel<<<dim3((unsigned)B, (unsigned)pairs), kTopkThreads, merge_smem, st>>>(t.S, step, t.Kp, K, ws_v, ws_i, v_out, i_out,
                                                                                           2 * step >= t.S ? 1 : 0);
    e = cudaGetLastError();
  }
  return e;
}

}  // namespace rnf
