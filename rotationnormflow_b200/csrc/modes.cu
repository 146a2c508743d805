// modes.cu -- separated posterior modes of a grid log-density: greedy non-maximum suppression on SO(3), per image, on the device.
//
// Definition (DESIGN 4.7; tests/test_modes.py holds the fp64 restatement).  values [B,G], rotations [G,3,3], M modes, thresholds
// cos_sep = cos(min_separation / 2) and cos_nb = cos(neighbour_radius / 2) on the quaternion dot |q_g . q_c|.  Per image, every
// point unlabelled at the start, for m = 0 .. M-1:
//   c_m       = best unlabelled point in the order of grid_red_better (NaN first, then larger value, then lower index); none -> stop
//   local_max = no point g != c_m with |q_g . q_c| >= cos_nb has v_g > v_c (NaN never higher; a NaN mode is no local max)
//   label m   = every unlabelled g with g == c_m or |q_g . q_c| > cos_sep
//   mass      = sum_{label m} exp(v_g - v_c0) / sum_all exp(v_g - v_c0)
//
// Layout: one quaternion pass ([G] float4 in the workspace), then M + 1 rounds of one (slice, image) CTA grid and one per-image
// combine.  Round r labels the points of mode r-1 and sums their mass (round 1 also sums the normaliser), tests whether mode r-1 is
// a local maximum, and takes the slice arg-max of mode r over the points still unlabelled; the combine folds the slice partials
// in a fixed order and writes the outputs.  No atomics and no host synchronisation: the results are bitwise reproducible and the
// 2M + 3 launches can be captured in a CUDA graph.  Labels are one byte per (image, point): only "labelled or not" is needed,
// because each mode's mass is summed in the round that labels it.
#include <math.h>

#include "rnf_common.cuh"

namespace rnf {

constexpr int kModesThreads = 256;
constexpr int kModesPerThread = 16;
constexpr int64_t kModesSlice = (int64_t)kModesThreads * kModesPerThread;   // points per CTA
constexpr long long kModesNone = 0x7fffffffffffffffLL;                       // "no point": loses to every real index

struct ModesPart {      // per (image, slice), written by round r
  float best_v;         // slice arg-max of mode r over unlabelled points (kModesNone index: nothing left in the slice)
  float mass;           // sum exp(v - v_c0) over the points labelled r-1 here
  float total;          // round 1: sum exp(v - v_c0) over the whole slice
  int disq;             // a point within the neighbour radius is higher than c_{r-1}
  long long best_i;     // local index
};

struct ModesState {     // per image, written by the combine
  long long center;     // local index of the last mode found
  float v_c;            // its value
  float v_c0;           // value of mode 0 (the reference of the exponentials)
  float total;          // sum_all exp(v - v_c0), from round 1
  int found;            // modes found so far
};

static int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }

int64_t modes_slices(int64_t G) { return (G + kModesSlice - 1) / kModesSlice; }

// workspace sections: quaternions [G] float4, labels [B][G] bytes, partials [B][slices], state [B]
int64_t modes_workspace_bytes(int64_t G, int64_t B) {
  return align256(G * 16) + align256(B * G) + align256(B * modes_slices(G) * (int64_t)sizeof(ModesPart)) +
         align256(B * (int64_t)sizeof(ModesState));
}

// the quaternion of a rotation matrix: best-conditioned of the four candidate rows, normalised (evalpath.matrix_to_quaternion)
__global__ void __launch_bounds__(kModesThreads) modes_quat_kernel(const float* __restrict__ rot, int64_t G, float4* __restrict__ q_out) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const float* m = rot + g * 9;
  const float m00 = m[0], m01 = m[1], m02 = m[2], m10 = m[3], m11 = m[4], m12 = m[5], m20 = m[6], m21 = m[7], m22 = m[8];
  const float a0 = sqrtf(fmaxf(1.f + m00 + m11 + m22, 0.f)), a1 = sqrtf(fmaxf(1.f + m00 - m11 - m22, 0.f));
  const float a2 = sqrtf(fmaxf(1.f - m00 + m11 - m22, 0.f)), a3 = sqrtf(fmaxf(1.f - m00 - m11 + m22, 0.f));
  float4 q;
  if (a0 >= a1 && a0 >= a2 && a0 >= a3) q = make_float4(a0 * a0, m21 - m12, m02 - m20, m10 - m01);
  else if (a1 >= a2 && a1 >= a3) q = make_float4(m21 - m12, a1 * a1, m10 + m01, m02 + m20);
  else if (a2 >= a3) q = make_float4(m02 - m20, m10 + m01, a2 * a2, m12 + m21);
  else q = make_float4(m10 - m01, m20 + m02, m21 + m12, a3 * a3);
  const float inv = rsqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
  q_out[g] = make_float4(q.x * inv, q.y * inv, q.z * inv, q.w * inv);
}

__device__ __forceinline__ float qdot_abs(float4 a, float4 b) { return fabsf(a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w); }

// Round r of one image slice (see the file comment).  Round 0 also clears the slice's labels.
__global__ void __launch_bounds__(kModesThreads) modes_round_kernel(const float* __restrict__ values, int64_t G, const float4* __restrict__ quat,
                                                                    unsigned char* __restrict__ labels, ModesPart* __restrict__ part,
                                                                    const ModesState* __restrict__ state, int r, int M, float cos_sep,
                                                                    float cos_nb) {
  const int64_t b = blockIdx.x, s = blockIdx.y;   // neighbouring CTAs: the same slice of different images (shared quaternions)
  const int tid = threadIdx.x;
  long long c = -1;
  float v_c = 0.f, v_c0 = 0.f;
  float4 q_c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r > 0) {
    const ModesState st = state[b];
    if (st.found < r) return;          // mode r-1 was not found: nothing left in this image, the combine reads no partial
    c = st.center;
    v_c = st.v_c;
    v_c0 = st.v_c0;
    q_c = quat[c];
  }
  const float* v_img = values + b * G;
  unsigned char* lab_img = labels + b * G;
  float bv = -INFINITY, mass = 0.f, total = 0.f;
  long long bi = kModesNone;
  bool disq = false;
  const int64_t g0 = s * kModesSlice + tid;
#pragma unroll 4
  for (int k = 0; k < kModesPerThread; ++k) {
    const int64_t g = g0 + (int64_t)k * kModesThreads;
    if (g >= G) break;
    const float v = v_img[g];
    bool labelled;
    if (r == 0) {
      lab_img[g] = 0;
      labelled = false;
    } else {
      labelled = lab_img[g] != 0;
      if (r == 1) total += expf(v - v_c0);
      const bool higher = v > v_c && g != c;        // NaN compares false on either side
      if (!labelled || higher) {
        const float d = qdot_abs(quat[g], q_c);
        if (!labelled && (g == c || d > cos_sep)) {
          labelled = true;
          lab_img[g] = 1;
          mass += expf(v - v_c0);
        }
        if (higher && d >= cos_nb) disq = true;
      }
    }
    if (r < M && !labelled && grid_red_better(v, g, bv, bi)) { bv = v; bi = g; }
  }
  // CTA reduction in a fixed order: shuffle tree per warp, then the warps in index order
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    mass += __shfl_xor_sync(0xffffffffu, mass, o);
    total += __shfl_xor_sync(0xffffffffu, total, o);
  }
  __shared__ float s_v[kModesThreads / 32], s_m[kModesThreads / 32], s_t[kModesThreads / 32];
  __shared__ long long s_i[kModesThreads / 32];
  const int any_disq = __syncthreads_or(disq);
  if ((tid & 31) == 0) { s_v[tid >> 5] = bv; s_i[tid >> 5] = bi; s_m[tid >> 5] = mass; s_t[tid >> 5] = total; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kModesThreads / 32; ++w) {
      if (grid_red_better(s_v[w], s_i[w], bv, bi)) { bv = s_v[w]; bi = s_i[w]; }
      mass += s_m[w];
      total += s_t[w];
    }
    ModesPart p;
    p.best_v = bv;
    p.best_i = bi;
    p.mass = mass;
    p.total = total;
    p.disq = any_disq;
    part[b * gridDim.y + s] = p;
  }
}

// One CTA per image: fold the slice partials of round r in slice order and write the outputs of modes r-1 (mass, local_max) and r
// (index, value), or padding (index -1, value -inf, local_max false, mass 0) when mode r does not exist.
__global__ void __launch_bounds__(kModesThreads) modes_combine_kernel(const ModesPart* __restrict__ part, int64_t n_slices, int64_t g_index0,
                                                                      ModesState* __restrict__ state, int r, int M,
                                                                      int64_t* __restrict__ index_out, float* __restrict__ value_out,
                                                                      unsigned char* __restrict__ local_max_out, float* __restrict__ mass_out,
                                                                      int32_t* __restrict__ count_out) {
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x;
  const ModesPart* p = part + b * n_slices;
  ModesState st;
  if (r == 0) { st.center = -1; st.v_c = 0.f; st.v_c0 = 0.f; st.total = 0.f; st.found = 0; }
  else st = state[b];
  const bool live = st.found == r;     // every mode before r was found, so this round's CTAs ran
  float bv = -INFINITY, mass = 0.f, total = 0.f;
  long long bi = kModesNone;
  int disq = 0;
  if (live) {
    for (int64_t t = tid; t < n_slices; t += blockDim.x) {
      const ModesPart q = p[t];
      if (grid_red_better(q.best_v, q.best_i, bv, bi)) { bv = q.best_v; bi = q.best_i; }
      mass += q.mass;
      total += q.total;
      disq |= q.disq;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    mass += __shfl_xor_sync(0xffffffffu, mass, o);
    total += __shfl_xor_sync(0xffffffffu, total, o);
  }
  __shared__ float s_v[kModesThreads / 32], s_m[kModesThreads / 32], s_t[kModesThreads / 32];
  __shared__ long long s_i[kModesThreads / 32];
  const int any_disq = __syncthreads_or(disq);
  if ((tid & 31) == 0) { s_v[tid >> 5] = bv; s_i[tid >> 5] = bi; s_m[tid >> 5] = mass; s_t[tid >> 5] = total; }
  __syncthreads();
  if (tid != 0) return;
  for (int w = 1; w < kModesThreads / 32; ++w) {
    if (grid_red_better(s_v[w], s_i[w], bv, bi)) { bv = s_v[w]; bi = s_i[w]; }
    mass += s_m[w];
    total += s_t[w];
  }
  const int64_t o = b * M;
  if (live && r > 0) {                 // finish mode r-1
    if (r == 1) st.total = total;
    mass_out[o + r - 1] = mass / st.total;
    local_max_out[o + r - 1] = (!any_disq && st.v_c == st.v_c) ? 1 : 0;
  }
  if (r < M) {
    if (live && bi != kModesNone) {    // mode r
      st.center = bi;
      st.v_c = bv;
      if (r == 0) st.v_c0 = bv;
      st.found = r + 1;
      index_out[o + r] = (int64_t)bi + g_index0;
      value_out[o + r] = bv;
    } else {
      index_out[o + r] = -1;
      value_out[o + r] = -INFINITY;
      local_max_out[o + r] = 0;
      mass_out[o + r] = 0.f;
    }
  }
  state[b] = st;
  count_out[b] = st.found;
}

cudaError_t launch_rotation_modes(const float* values, int64_t B, int64_t G, int64_t g_index0, const float* rot, int M, float cos_sep,
                                  float cos_nb, void* workspace, int64_t* index_out, float* value_out, unsigned char* local_max_out,
                                  float* mass_out, int32_t* count_out, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  char* ws = (char*)workspace;
  float4* quat = (float4*)ws;
  unsigned char* labels = (unsigned char*)(ws + align256(G * 16));
  ModesPart* part = (ModesPart*)(ws + align256(G * 16) + align256(B * G));
  const int64_t S = modes_slices(G);
  ModesState* state = (ModesState*)((char*)part + align256(B * S * (int64_t)sizeof(ModesPart)));
  if (G > 0) {
    modes_quat_kernel<<<(unsigned)((G + kModesThreads - 1) / kModesThreads), kModesThreads, 0, st>>>(rot, G, quat);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  for (int r = 0; r <= M; ++r) {
    if (S > 0) {
      modes_round_kernel<<<dim3((unsigned)B, (unsigned)S), kModesThreads, 0, st>>>(values, G, quat, labels, part, state, r, M, cos_sep, cos_nb);
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return e;
    }
    modes_combine_kernel<<<(unsigned)B, kModesThreads, 0, st>>>(part, S, g_index0, state, r, M, index_out, value_out, local_max_out, mass_out,
                                                               count_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// ---- Sharded modes (DESIGN 4.7, "Sharded"): the rounds above over one rank's contiguous slice [g_index0, g_index0 + G_r) of the grid.
// Per round, every rank runs modes_shard_round_kernel over its (image, slice) CTAs and modes_shard_fold_kernel, which writes one
// ModesRecord per image; the caller all-gathers the records to [W][B] (rank-major) and every rank runs modes_shard_merge_kernel on
// the same bytes, so every rank holds the same state and outputs.  Indices are global throughout; the centre's quaternion travels
// in the record from the rank that owns the point, so the dot products are those of launch_rotation_modes bit for bit.

struct ModesRecord {    // per (rank, image), written by the fold of round r, read by the merge of round r on every rank
  float4 q;             // quaternion of the proposal (this rank's quaternion pass)
  float rot[9];         // its rotation matrix as the rank was given it
  float best_v;         // proposal of mode r: best unlabelled point of the rank's slice (kModesNone index: none)
  long long best_i;     // global index
  float mass;           // sum exp(v - v_c0) over the rank's points labelled r-1
  float total;          // round 1: sum exp(v - v_c0) over the rank's slice
  int disq;             // a point of the rank within the neighbour radius is higher than c_{r-1}
  int pad;              // 0
};
static_assert(sizeof(ModesRecord) == RNF_MODES_RECORD_BYTES, "the record size is part of the ABI");

struct ModesShardState {  // per image, written by the merge: identical on every rank
  float4 q_c;           // quaternion of the last mode found
  long long center;     // its global index
  float v_c, v_c0, total;
  int found;
};

// workspace sections: state [B] first (the merge needs no slice size), quaternions [G_r] float4, labels [B][G_r], partials [B][slices]
int64_t modes_shard_workspace_bytes(int64_t G, int64_t B) {
  return align256(B * (int64_t)sizeof(ModesShardState)) + align256(G * 16) + align256(B * G) +
         align256(B * modes_slices(G) * (int64_t)sizeof(ModesPart));
}

int64_t modes_shard_state_bytes(int64_t B) { return align256(B * (int64_t)sizeof(ModesShardState)); }

// modes_round_kernel over a slice of the grid: g and the centre are global indices (gl = g_index0 + local), the centre's quaternion
// comes from the merged state.  Partials carry global indices.
__global__ void __launch_bounds__(kModesThreads) modes_shard_round_kernel(const float* __restrict__ values, int64_t G, int64_t g_index0,
                                                                          const float4* __restrict__ quat, unsigned char* __restrict__ labels,
                                                                          ModesPart* __restrict__ part, const ModesShardState* __restrict__ state,
                                                                          int r, int M, float cos_sep, float cos_nb) {
  const int64_t b = blockIdx.x, s = blockIdx.y;
  const int tid = threadIdx.x;
  long long c = -1;
  float v_c = 0.f, v_c0 = 0.f;
  float4 q_c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r > 0) {
    const ModesShardState st = state[b];
    if (st.found < r) return;          // mode r-1 was not found: the fold reads no partial
    c = st.center;
    v_c = st.v_c;
    v_c0 = st.v_c0;
    q_c = st.q_c;
  }
  const float* v_img = values + b * G;
  unsigned char* lab_img = labels + b * G;
  float bv = -INFINITY, mass = 0.f, total = 0.f;
  long long bi = kModesNone;
  bool disq = false;
  const int64_t g0 = s * kModesSlice + tid;
#pragma unroll 4
  for (int k = 0; k < kModesPerThread; ++k) {
    const int64_t g = g0 + (int64_t)k * kModesThreads;
    if (g >= G) break;
    const long long gl = g_index0 + g;
    const float v = v_img[g];
    bool labelled;
    if (r == 0) {
      lab_img[g] = 0;
      labelled = false;
    } else {
      labelled = lab_img[g] != 0;
      if (r == 1) total += expf(v - v_c0);
      const bool higher = v > v_c && gl != c;       // NaN compares false on either side
      if (!labelled || higher) {
        const float d = qdot_abs(quat[g], q_c);
        if (!labelled && (gl == c || d > cos_sep)) {
          labelled = true;
          lab_img[g] = 1;
          mass += expf(v - v_c0);
        }
        if (higher && d >= cos_nb) disq = true;
      }
    }
    if (r < M && !labelled && grid_red_better(v, gl, bv, bi)) { bv = v; bi = gl; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    mass += __shfl_xor_sync(0xffffffffu, mass, o);
    total += __shfl_xor_sync(0xffffffffu, total, o);
  }
  __shared__ float s_v[kModesThreads / 32], s_m[kModesThreads / 32], s_t[kModesThreads / 32];
  __shared__ long long s_i[kModesThreads / 32];
  const int any_disq = __syncthreads_or(disq);
  if ((tid & 31) == 0) { s_v[tid >> 5] = bv; s_i[tid >> 5] = bi; s_m[tid >> 5] = mass; s_t[tid >> 5] = total; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kModesThreads / 32; ++w) {
      if (grid_red_better(s_v[w], s_i[w], bv, bi)) { bv = s_v[w]; bi = s_i[w]; }
      mass += s_m[w];
      total += s_t[w];
    }
    ModesPart p;
    p.best_v = bv;
    p.best_i = bi;
    p.mass = mass;
    p.total = total;
    p.disq = any_disq;
    part[b * gridDim.y + s] = p;
  }
}

// One CTA per image: fold the rank's slice partials of round r in slice order into the image's record, with the quaternion and the
// rotation of the proposal.  An image whose previous round found nothing, and a rank with no points, write the neutral record.
__global__ void __launch_bounds__(kModesThreads) modes_shard_fold_kernel(const ModesPart* __restrict__ part, int64_t n_slices, int64_t g_index0,
                                                                         const float4* __restrict__ quat, const float* __restrict__ rot,
                                                                         const ModesShardState* __restrict__ state, int r,
                                                                         ModesRecord* __restrict__ rec_out) {
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x;
  const ModesPart* p = part + b * n_slices;
  const bool live = r == 0 || state[b].found == r;
  float bv = -INFINITY, mass = 0.f, total = 0.f;
  long long bi = kModesNone;
  int disq = 0;
  if (live) {
    for (int64_t t = tid; t < n_slices; t += blockDim.x) {
      const ModesPart q = p[t];
      if (grid_red_better(q.best_v, q.best_i, bv, bi)) { bv = q.best_v; bi = q.best_i; }
      mass += q.mass;
      total += q.total;
      disq |= q.disq;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (grid_red_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    mass += __shfl_xor_sync(0xffffffffu, mass, o);
    total += __shfl_xor_sync(0xffffffffu, total, o);
  }
  __shared__ float s_v[kModesThreads / 32], s_m[kModesThreads / 32], s_t[kModesThreads / 32];
  __shared__ long long s_i[kModesThreads / 32];
  const int any_disq = __syncthreads_or(disq);
  if ((tid & 31) == 0) { s_v[tid >> 5] = bv; s_i[tid >> 5] = bi; s_m[tid >> 5] = mass; s_t[tid >> 5] = total; }
  __syncthreads();
  if (tid != 0) return;
  for (int w = 1; w < kModesThreads / 32; ++w) {
    if (grid_red_better(s_v[w], s_i[w], bv, bi)) { bv = s_v[w]; bi = s_i[w]; }
    mass += s_m[w];
    total += s_t[w];
  }
  ModesRecord o;
  o.q = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < 9; ++k) o.rot[k] = 0.f;
  if (bi != kModesNone) {
    const int64_t l = bi - g_index0;
    o.q = quat[l];
    for (int k = 0; k < 9; ++k) o.rot[k] = rot[l * 9 + k];
  }
  o.best_v = bv;
  o.best_i = bi;
  o.mass = mass;
  o.total = total;
  o.disq = any_disq;
  o.pad = 0;
  rec_out[b] = o;
}

// One thread per image: fold the gathered records [W][B] of round r in rank order (the order of grid_red_better for the next centre,
// sums of the mass partials, OR of the flags) and write the outputs of modes r-1 and r as modes_combine_kernel does, plus mode r's
// rotation (NaN padding).  Every rank runs it on the same records.
__global__ void __launch_bounds__(128) modes_shard_merge_kernel(const ModesRecord* __restrict__ recs, int W, int64_t B,
                                                                ModesShardState* __restrict__ state, int r, int M,
                                                                int64_t* __restrict__ index_out, float* __restrict__ value_out,
                                                                unsigned char* __restrict__ local_max_out, float* __restrict__ mass_out,
                                                                int32_t* __restrict__ count_out, float* __restrict__ rot_out) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  ModesShardState st;
  if (r == 0) { st.q_c = make_float4(0.f, 0.f, 0.f, 0.f); st.center = -1; st.v_c = 0.f; st.v_c0 = 0.f; st.total = 0.f; st.found = 0; }
  else st = state[b];
  const bool live = st.found == r;
  float bv = -INFINITY, mass = 0.f, total = 0.f;
  long long bi = kModesNone;
  int disq = 0, owner = -1;
  if (live) {
    for (int w = 0; w < W; ++w) {
      const ModesRecord& q = recs[(int64_t)w * B + b];
      if (grid_red_better(q.best_v, q.best_i, bv, bi)) { bv = q.best_v; bi = q.best_i; owner = w; }
      mass += q.mass;
      total += q.total;
      disq |= q.disq;
    }
  }
  const int64_t o = b * M;
  if (live && r > 0) {                 // finish mode r-1
    if (r == 1) st.total = total;
    mass_out[o + r - 1] = mass / st.total;
    local_max_out[o + r - 1] = (!disq && st.v_c == st.v_c) ? 1 : 0;
  }
  if (r < M) {
    float* R = rot_out + (o + r) * 9;
    if (live && bi != kModesNone) {    // mode r
      const ModesRecord& q = recs[(int64_t)owner * B + b];
      st.q_c = q.q;
      st.center = bi;
      st.v_c = bv;
      if (r == 0) st.v_c0 = bv;
      st.found = r + 1;
      index_out[o + r] = (int64_t)bi;
      value_out[o + r] = bv;
      for (int k = 0; k < 9; ++k) R[k] = q.rot[k];
    } else {
      index_out[o + r] = -1;
      value_out[o + r] = -INFINITY;
      local_max_out[o + r] = 0;
      mass_out[o + r] = 0.f;
      for (int k = 0; k < 9; ++k) R[k] = __int_as_float(0x7fffffff);   // NaN
    }
  }
  state[b] = st;
  count_out[b] = st.found;
}

static ModesShardState* shard_state(void* ws) { return (ModesShardState*)ws; }
static float4* shard_quat(void* ws, int64_t B) { return (float4*)((char*)ws + modes_shard_state_bytes(B)); }
static unsigned char* shard_labels(void* ws, int64_t G, int64_t B) { return (unsigned char*)shard_quat(ws, B) + align256(G * 16); }
static ModesPart* shard_part(void* ws, int64_t G, int64_t B) { return (ModesPart*)(shard_labels(ws, G, B) + align256(B * G)); }

cudaError_t launch_modes_shard_setup(const float* rot, int64_t G, int64_t B, void* workspace, cudaStream_t st) {
  if (G <= 0 || B <= 0) return cudaSuccess;
  modes_quat_kernel<<<(unsigned)((G + kModesThreads - 1) / kModesThreads), kModesThreads, 0, st>>>(rot, G, shard_quat(workspace, B));
  return cudaGetLastError();
}

cudaError_t launch_modes_shard_round(const float* values, int64_t B, int64_t G, int64_t g_index0, const float* rot, int r, int M,
                                     float cos_sep, float cos_nb, void* workspace, void* rec_out, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  const int64_t S = modes_slices(G);
  ModesPart* part = shard_part(workspace, G, B);
  if (S > 0) {
    modes_shard_round_kernel<<<dim3((unsigned)B, (unsigned)S), kModesThreads, 0, st>>>(values, G, g_index0, shard_quat(workspace, B),
                                                                                      shard_labels(workspace, G, B), part,
                                                                                      shard_state(workspace), r, M, cos_sep, cos_nb);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  modes_shard_fold_kernel<<<(unsigned)B, kModesThreads, 0, st>>>(part, S, g_index0, shard_quat(workspace, B), rot, shard_state(workspace), r,
                                                                (ModesRecord*)rec_out);
  return cudaGetLastError();
}

cudaError_t launch_modes_shard_merge(const void* records, int W, int64_t B, int r, int M, void* workspace, int64_t* index_out,
                                     float* value_out, unsigned char* local_max_out, float* mass_out, int32_t* count_out, float* rot_out,
                                     cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  modes_shard_merge_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>((const ModesRecord*)records, W, B, shard_state(workspace), r, M,
                                                                        index_out, value_out, local_max_out, mass_out, count_out, rot_out);
  return cudaGetLastError();
}

}  // namespace rnf
