// rnf_common.cuh -- shared definitions between the C ABI (rnf_abi.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rnf_abi.h"

namespace rnf {

constexpr int kK = 64;  // Mobius mixture components (config.segments in every settings/*.yml)
constexpr int kH = 64;  // conditioner hidden width (flow/condition.py:9)

// ---- packed FP32 image of one Mobius conditioner (float offsets inside the layer block) -------------------
//   first : [64][4]   (W0[j][0..2] = columns of fc_first acting on y, b0[j])
//   hid l : [64 k][64 j] transposed weights of layers.{1,3,5}, then bias[64]
//   last  : [64 k][256 j'] transposed fc_last with outputs permuted so component c owns j' = 4c..4c+3
//           = (mixture logit a_c, w_c.x, w_c.y, w_c.z), then the equally permuted bias[256]
constexpr int kMobFirst = 0;
constexpr int kMobHid = kMobFirst + kH * 4;
constexpr int kMobHidStride = kH * kH + kH;
constexpr int kMobLast = kMobHid + 3 * kMobHidStride;
constexpr int kMobFloats = kMobLast + kH * 4 * kK + 4 * kK;  // 29376 floats = 117504 B

// ---- affine block (unconditional in the weight buffer, conditional per image in the cond buffer) -----------
//   [0..15] W, [16] log|det W|, [20..35] W^-1 (or W^T for rotation layers), [36] log|det W^-1|
constexpr int kAffFloats = RNF_AFFINE_BLOCK_FLOATS;
constexpr int kAffInv = 40;

// ---- conditional-affine MLP tail block (per slot, at model.caff_off + slot*kCaffFloats) ---------------------
//   b_first[64], 3 x (W[64 out][64 in] row-major as in nn.Linear, b[64]), W_last[16][64], b_last[16]
constexpr int kCaffFloats = kH + 3 * (kH * kH + kH) + 16 * kH + 16;

struct LayerDev {
  int32_t kind;
  int32_t perm;
  int32_t cond_slot;
  int32_t has_ldj;
  int64_t w_off;
  int64_t w_off_tc;
};

constexpr int kPartStride = 8;

struct FlowArgs {
  const float* weights;
  const LayerDev* layers;
  int n_layers;
  int n_mobius_slots;
  // rows
  const float* R_in;
  int64_t N;
  const float* cond;
  int64_t cond_stride;
  const int32_t* feat_index;
  int64_t rows_per_image;
  float* R_out;
  float* ldj_out;
  float* scratch;  // inverse: per-CTA bisection parameters
  // grid mode (G > 0)
  int64_t G;
  int64_t g_index0;
  int64_t tiles_per_image;
  int64_t n_tiles;
  const float* offset;
  const float* fisher_A;
  const float* fisher_c;
  float* logp_out;
  float* part;        // [n_tiles][kPartStride]: (max, sum exp(lp - max), argmax lo, argmax hi, sum exp(lp - max) * d_gt, -, -, -)
  const float* gt;    // [B][gt_k][9] ground-truth rotations per image (spread metric), nullptr = not requested
  int gt_k;
  int t4_active;      // flow_t4: tiles in flight per CTA in this launch (set by launch_flow_t4; 0 = all four)
  unsigned long long* probe_counter;   // measurement hook (rnf_debug_set_probe_counter), normally null
  long long* trace;   // debug builds (-DRNF_TC_TRACE): per-phase clock64() stamps of CTA 0, else unused
};

}  // namespace rnf

struct rnf_flow {
  rnf_model_desc model;
  rnf::LayerDev* layers_dev;
  rnf_layer_desc* layers_host;
  const float* weights_dev;
  int device;
  int sm_count;
  int64_t cond_floats;
};

// kernel launchers (defined in the .cu files)
namespace rnf {
// Order of the grid reductions (max, first arg-max): a NaN log-density ranks above every number, ties and NaN against NaN go
// to the lower index, so an image with a non-finite row gets a NaN max / sumexp and the index of its first such row instead
// of a finite result taken over the remaining rows.
__device__ __forceinline__ bool grid_red_better(float ov, long long oi, float bv, long long bi) {
  const bool on = ov != ov, bn = bv != bv;
  return on ? (!bn || oi < bi) : (!bn && (ov > bv || (ov == bv && oi < bi)));
}
cudaError_t launch_flow_v1(const FlowArgs& a, bool inverse, int sm_count, cudaStream_t st);
cudaError_t launch_fisher_sample(const float* usv, int64_t B, int64_t n, unsigned long long seed, float* out, cudaStream_t st);
cudaError_t launch_grid_combine(const float* part, int64_t tiles_per_image, int64_t B, int64_t g_index0, float* max_out,
                                int64_t* argmax_out, float* sumexp_out, float* spread_num_out, cudaStream_t st);
cudaError_t launch_condition(const rnf_flow* f, const float* feat, int64_t B, float* cond, cudaStream_t st,
                             const int32_t* row_index = nullptr, const int32_t* count = nullptr);
size_t dedup_scan_bytes(int64_t N);
cudaError_t launch_dedup(const float* feat, int64_t N, int64_t F, int32_t* idx, int32_t* first, int64_t cap, int32_t* count, void* ws,
                         size_t ws_bytes, int sm_count, cudaStream_t st);
cudaError_t launch_poison(const int32_t* count, int64_t cap, float* ldj, int64_t N, cudaStream_t st);
cudaError_t launch_train_mobius_fwd(const float* R, const float* out, int64_t N, int K, int perm, bool inverse, float* R_out, float* ldj,
                                    float* theta, cudaStream_t st);
cudaError_t launch_train_mobius_bwd(const float* R, const float* out, int64_t N, int K, int perm, bool inverse, const float* theta,
                                    const float* R_out, const float* G_Rout, const float* g_ldj, float* G_R, float* G_out, cudaStream_t st);
cudaError_t launch_train_affine_fwd(const float* R, const float* W, int64_t N, float* R_out, float* loglen, cudaStream_t st);
cudaError_t launch_train_affine_bwd(const float* R, const float* W, int64_t N, const float* R_out, const float* G_Rout, const float* g_loglen,
                                    float* G_R, float* G_W, cudaStream_t st);
cudaError_t launch_train_ablation_fwd(const float* R, const float* M, int64_t N, int kind, float* R_out, float* ldj, cudaStream_t st);
cudaError_t launch_train_ablation_bwd(const float* R, const float* M, int64_t N, int kind, const float* R_out, const float* G_Rout,
                                      const float* g_ldj, float* G_R, float* G_M, cudaStream_t st);
int train_max_components();
cudaError_t launch_healpix(int level, int64_t begin, int64_t end, float* out, cudaStream_t st);
cudaError_t launch_min_geodesic(const float* est, const float* gt, int64_t B, int64_t K, float* out, cudaStream_t st);
cudaError_t launch_fisher_logprob(const float* A9, const float* c, const float* R, int64_t N, int64_t rows_per_image, float* out,
                                  cudaStream_t st);
cudaError_t launch_flow_grad(const rnf_flow* f, const float* R_in, int64_t N, const float* cond, const int32_t* feat_index,
                             int64_t rows_per_image, const float* fisher_A, const float* fisher_c, float* logp_out, float* grad_out,
                             cudaStream_t st);
int64_t flow_train_workspace_floats(const rnf_flow* f, int64_t N);
cudaError_t launch_flow_train(const rnf_flow* f, bool backward, const float* weights, const float* R_in, int64_t N, const float* cond,
                              const int32_t* feat_index, int64_t rows_per_image, float* R_out, float* ldj_out, const float* G_Rout,
                              const float* g_ldj, float* G_R, float* workspace, cudaStream_t st);
constexpr int kV1Threads = 256;
}  // namespace rnf
