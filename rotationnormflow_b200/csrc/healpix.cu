// healpix.cu -- on-device HEALPix SO(3) grid (Yershova et al.), index -> rotation (healpix_rot.cuh), plus the matrix-Fisher
// log-density and the geodesic metric.
#include "healpix_rot.cuh"
#include "rnf_common.cuh"

namespace rnf {
namespace {

__global__ void healpix_grid_kernel(int level, int64_t begin, int64_t end, float* __restrict__ out) {
  const int64_t n = end - begin;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
    healpix_rotation(level, begin + k, out + k * 9);
}

// MatrixFisherN._log_prob (utils/fisher.py:217-232): out[i] = sum(A_b * R_i) - c_b, b = image of row i (image-major rows,
// `rows_per_image` rotations each, as inputs.reshape(B, -1, 3, 3) does).  HBM bound: 36 B in + 4 B out per rotation.
__global__ void fisher_logprob_kernel(const float* __restrict__ A9, const float* __restrict__ c, const float* __restrict__ R,
                                      int64_t N, int64_t rows_per_image, float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / rows_per_image;
    float tr = 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k) tr = fmaf(__ldg(A9 + b * 9 + k), __ldg(R + i * 9 + k), tr);
    out[i] = tr - __ldg(c + b);
  }
}

// min_geodesic_distance_rotmats (utils/utils.py:231-235): angle between est[b] and the closest of its K ground-truth rotations:
// acos(clip((max_k sum_ij est_ij gt_kij - 1)/2, -1, 1)).  K = 1 is geodesic_distance_rotmats (utils/utils.py:225-228).
__global__ void min_geodesic_kernel(const float* __restrict__ est, const float* __restrict__ gt, int64_t B, int64_t K,
                                    float* __restrict__ out) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float e[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) e[i] = __ldg(est + b * 9 + i);
  float best = -INFINITY;
  for (int64_t k = 0; k < K; ++k) {
    const float* g = gt + (b * K + k) * 9;
    float tr = 0.0f;
#pragma unroll
    for (int i = 0; i < 9; ++i) tr = fmaf(e[i], __ldg(g + i), tr);
    best = fmaxf(best, tr);
  }
  out[b] = acosf(fminf(fmaxf((best - 1.0f) * 0.5f, -1.0f), 1.0f));
}

}  // namespace

cudaError_t launch_min_geodesic(const float* est, const float* gt, int64_t B, int64_t K, float* out, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  min_geodesic_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(est, gt, B, K, out);
  return cudaGetLastError();
}

cudaError_t launch_fisher_logprob(const float* A9, const float* c, const float* R, int64_t N, int64_t rows_per_image, float* out,
                                  cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  int64_t blocks = (N + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  fisher_logprob_kernel<<<(unsigned)blocks, 256, 0, st>>>(A9, c, R, N, rows_per_image, out);
  return cudaGetLastError();
}

cudaError_t launch_healpix(int level, int64_t begin, int64_t end, float* out, cudaStream_t st) {
  const int64_t n = end - begin;
  if (n <= 0) return cudaSuccess;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  healpix_grid_kernel<<<(unsigned)blocks, 256, 0, st>>>(level, begin, end, out);
  return cudaGetLastError();
}

}  // namespace rnf
