// rnf_abi.cu -- the extern "C" boundary declared in include/rnf_abi.h.  No torch types, no exceptions.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "rnf_common.cuh"

namespace rnf {
cudaError_t launch_flow_row(const FlowArgs& a, bool inverse, int sm_count, cudaStream_t st);
cudaError_t launch_flow_t4(const FlowArgs& a, int sm_count, cudaStream_t st);
bool flow_tc_supported(const rnf_flow* f);
int pick_active_tiles(int64_t n_tiles, int sm_count);
int64_t modes_workspace_bytes(int64_t G, int64_t B);
int64_t modes_slices(int64_t G);
cudaError_t launch_rotation_modes(const float* values, int64_t B, int64_t G, int64_t g_index0, const float* rot, int M, float cos_sep,
                                  float cos_nb, void* workspace, int64_t* index_out, float* value_out, unsigned char* local_max_out,
                                  float* mass_out, int32_t* count_out, cudaStream_t st);
int64_t modes_shard_workspace_bytes(int64_t G, int64_t B);
int64_t modes_shard_state_bytes(int64_t B);
cudaError_t launch_modes_shard_setup(const float* rot, int64_t G, int64_t B, void* workspace, cudaStream_t st);
cudaError_t launch_modes_shard_round(const float* values, int64_t B, int64_t G, int64_t g_index0, const float* rot, int r, int M,
                                     float cos_sep, float cos_nb, void* workspace, void* rec_out, cudaStream_t st);
cudaError_t launch_modes_shard_merge(const void* records, int W, int64_t B, int r, int M, void* workspace, int64_t* index_out,
                                     float* value_out, unsigned char* local_max_out, float* mass_out, int32_t* count_out, float* rot_out,
                                     cudaStream_t st);
cudaError_t launch_healpix_children(int level, const int64_t* parent, int64_t n, const float* offset, int64_t* child_out, float* R_out,
                                    cudaStream_t st);
int64_t topk_slices(int64_t C, int K);
int64_t topk_workspace_bytes(int64_t B, int64_t C, int K);
cudaError_t launch_topk(const float* values, const int64_t* index, int64_t B, int64_t C, int K, void* workspace, float* v_out,
                        int64_t* i_out, cudaStream_t st);
}  // namespace rnf

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return (int)e;
}

long long* g_trace = nullptr;
unsigned long long* g_probe_counter = nullptr;

bool valid_mode(int m) { return m == RNF_MLP_FP32 || m == RNF_MLP_TC || m == RNF_MLP_TC_ROW; }

// rows reach their image through feat_index, or image-major at rows_per_image rows per image: N rows must fit in B images
int row_map_ok(const char* who, int64_t N, int64_t B, const int32_t* feat_index, int64_t rows_per_image) {
  if (feat_index) return RNF_OK;
  if (rows_per_image <= 0) return fail(RNF_EINVAL, "%s: need feat_index or rows_per_image > 0", who);
  if ((N + rows_per_image - 1) / rows_per_image > B)
    return fail(RNF_EINVAL, "%s: N=%lld rows at %lld rows/image exceed B=%lld images", who, (long long)N, (long long)rows_per_image,
                (long long)B);
  return RNF_OK;
}

// the gradient kernels (csrc/flow_grad.cu) run Mobius layers of kK components and quaternion affine layers only
int gradient_stack_ok(const rnf_flow* f, const char* who) {
  if (f->model.K != rnf::kK) return fail(RNF_ESHAPE, "%s: the kernel is built for segments=%d (got K=%d)", who, rnf::kK, f->model.K);
  for (int i = 0; i < f->model.n_layers; ++i) {
    const int k = f->layers_host[i].kind;
    if (k != RNF_LAYER_MOBIUS && k != RNF_LAYER_AFFINE)
      return fail(RNF_ESHAPE, "%s: layer %d is an ablation layer (kind %d), which has no gradient here", who, i, k);
  }
  return RNF_OK;
}

// the fields of a launch of the flow kernels that every entry point sets the same way
rnf::FlowArgs flow_args(const rnf_flow* f, const float* R_in, int64_t N, const float* cond) {
  rnf::FlowArgs a;
  memset(&a, 0, sizeof(a));
  a.weights = f->weights_dev;
  a.layers = f->layers_dev;
  a.n_layers = f->model.n_layers;
  a.n_mobius_slots = f->model.n_mobius_slots;
  a.R_in = R_in;
  a.N = N;
  a.cond = f->cond_floats > 0 ? cond : nullptr;
  a.cond_stride = f->cond_floats;
  a.rows_per_image = 1;
  a.trace = g_trace;
  a.probe_counter = g_probe_counter;
  return a;
}

// Tiles and kernel of an mlp_mode: 128-row tiles on the tensor cores, kV1Threads rows in FP32.  A grid launch (a.G > 0) tiles each
// of its B images separately.  RNF_MLP_TC runs four tiles per SM in the forward direction (flow_t4.cu); the bisection of the
// inverse needs its prepared parameters resident in tensor memory and runs in the two-tile kernel (flow_row.cu), as does everything
// in RNF_MLP_TC_ROW.
int launch_flow(const rnf_flow* f, rnf::FlowArgs& a, int64_t B, bool inverse, int mlp_mode, void* stream, const char* who) {
  if (mlp_mode != RNF_MLP_FP32 && !rnf::flow_tc_supported(f))
    return fail(RNF_ESTATE, "%s: model was packed without the tensor-core weight image", who);
  const int64_t tile = mlp_mode == RNF_MLP_FP32 ? rnf::kV1Threads : 128;
  if (a.G > 0) {
    a.tiles_per_image = (a.G + tile - 1) / tile;
    a.n_tiles = a.tiles_per_image * B;
  } else {
    a.n_tiles = (a.N + tile - 1) / tile;
  }
  cudaError_t e;
  if (mlp_mode == RNF_MLP_FP32) e = rnf::launch_flow_v1(a, inverse, f->sm_count, (cudaStream_t)stream);
  else if (mlp_mode == RNF_MLP_TC && !inverse) e = rnf::launch_flow_t4(a, f->sm_count, (cudaStream_t)stream);
  else e = rnf::launch_flow_row(a, inverse, f->sm_count, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int modes_count_ok(const char* who, int M) { return M < 1 || M > 256 ? fail(RNF_EINVAL, "%s: M=%d modes outside 1..256", who, M) : RNF_OK; }

// The checks of num_modes and the two angles, and the thresholds the kernels test, |q_g . q_c| > cos(theta / 2) and
// >= cos(rho / 2), in double and rounded once: the single-GPU and the sharded calls get them here, so they test the same floats.
int modes_thresholds(const char* who, int M, float min_separation, float neighbour_radius, float* cos_sep, float* cos_nb) {
  const int rc = modes_count_ok(who, M);
  if (rc != RNF_OK) return rc;
  const float pi = 3.14159265358979323846f;
  if (!(neighbour_radius > 0.f) || !(neighbour_radius <= min_separation) || !(min_separation <= pi))
    return fail(RNF_EINVAL, "%s: need 0 < neighbour_radius <= min_separation <= pi (got %g, %g)", who, (double)neighbour_radius,
                (double)min_separation);
  *cos_sep = (float)cos(0.5 * (double)min_separation);
  *cos_nb = (float)cos(0.5 * (double)neighbour_radius);
  return RNF_OK;
}

int modes_slices_ok(const char* who, const char* name, int64_t G) {
  if (rnf::modes_slices(G) > 65535)
    return fail(RNF_EINVAL, "%s: %s=%lld rotations exceed the 65535 x 4096 points of one launch", who, name, (long long)G);
  return RNF_OK;
}

}  // namespace

extern "C" {

// debug hook (not part of the ABI header): device buffer that -DRNF_TC_TRACE builds fill with clock64() stamps
void rnf_debug_set_trace(long long* dev_ptr) { g_trace = dev_ptr; }
// measurement hook (not part of the ABI header; bench.py): device counter that the inverse kernel increments by 32 per warp,
// Mobius layer and evaluation of the mixture map F, i.e. by the number of (sample, layer, evaluation) triples executed
void rnf_debug_set_probe_counter(unsigned long long* dev_ptr) { g_probe_counter = dev_ptr; }

// test hook (not part of the ABI header; host logic only, no device needed): tile slots flow_t4 would use for a launch of n_tiles
int rnf_debug_pick_active_tiles(long long n_tiles, int sm_count) { return rnf::pick_active_tiles((int64_t)n_tiles, sm_count); }

int rnf_abi_version(void) { return RNF_ABI_VERSION; }

const char* rnf_last_error(void) { return g_err; }

int rnf_device_check(int* sm_count_out) {
  // cudaGetDeviceProperties costs milliseconds per call (it queries every attribute, clocks and PCIe state included): the three
  // attributes needed here are read once per device with cudaDeviceGetAttribute and remembered.
  static int cached_sm[64];                         // 0 = not queried yet, -1 = not an sm_100 device
  static int cached_cc[64];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(RNF_ENODEV, "cudaGetDevice: %s", cudaGetErrorString(e));
  const bool slot = dev >= 0 && dev < 64;
  int sm = slot ? cached_sm[dev] : 0, cc = slot ? cached_cc[dev] : 0;
  if (sm == 0) {
    int major = 0, minor = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return fail(RNF_ENODEV, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
    cc = 10 * major + minor;
    if (major != 10) sm = -1;
    if (slot) { cached_cc[dev] = cc; cached_sm[dev] = sm; }   // benign race: every thread writes the same values
  }
  if (sm < 0) return fail(RNF_ENODEV, "device %d is sm_%d; this library contains sm_100a code only", dev, cc);
  if (sm_count_out) *sm_count_out = sm;
  return RNF_OK;
}

int rnf_flow_create(const rnf_model_desc* model, const rnf_layer_desc* layers, const float* weights_dev, rnf_flow** out) {
  if (!model || !out || (model->n_layers > 0 && !layers)) return fail(RNF_EINVAL, "rnf_flow_create: null argument");
  if (model->abi_version != RNF_ABI_VERSION)
    return fail(RNF_EINVAL, "rnf_flow_create: ABI version %d, library is %d", model->abi_version, RNF_ABI_VERSION);
  if (model->n_layers < 0 || model->F < 0) return fail(RNF_EINVAL, "rnf_flow_create: negative size");
  if (model->K != rnf::kK || model->H != rnf::kH)
    return fail(RNF_ESHAPE, "rnf_flow_create: kernels are built for segments=64, hidden=64 (got K=%d H=%d)", model->K, model->H);
  if (model->n_floats > 0 && !weights_dev) return fail(RNF_EINVAL, "rnf_flow_create: null weights");
  int n_mob = 0, n_aff = 0, total_mobius = 0;
  for (int i = 0; i < model->n_layers; ++i) {
    const rnf_layer_desc& L = layers[i];
    if (L.kind < RNF_LAYER_MOBIUS || L.kind > RNF_LAYER_RIGHT9) return fail(RNF_EINVAL, "layer %d: bad kind %d", i, L.kind);
    if (L.kind == RNF_LAYER_MOBIUS && (L.perm < 0 || L.perm > 2)) return fail(RNF_EINVAL, "layer %d: bad perm %d", i, L.perm);
    if (L.w_off < 0 || (L.w_off & 3) || L.w_off > model->n_floats) return fail(RNF_EINVAL, "layer %d: bad weight offset", i);
    if (L.cond_slot >= 0) {
      if (model->F <= 0) return fail(RNF_EINVAL, "layer %d is conditional but F == 0", i);
      if (L.kind == RNF_LAYER_MOBIUS) { if (L.cond_slot != n_mob++) return fail(RNF_EINVAL, "layer %d: Mobius slots must be consecutive", i); }
      else { if (L.cond_slot != n_aff++) return fail(RNF_EINVAL, "layer %d: affine slots must be consecutive", i); }
    }
    total_mobius += L.kind == RNF_LAYER_MOBIUS;
  }
  if (total_mobius > 64)
    return fail(RNF_ESHAPE, "rnf_flow_create: %d Mobius layers; the kernels keep their weight-offset table in 64 shared-memory slots", total_mobius);
  if (n_mob != model->n_mobius_slots || n_aff != model->n_affine_slots)
    return fail(RNF_EINVAL, "slot counts (%d,%d) do not match the layer table (%d,%d)", model->n_mobius_slots,
                model->n_affine_slots, n_mob, n_aff);
  int sm = 0;
  int rc = rnf_device_check(&sm);
  if (rc != RNF_OK) return rc;
  rnf_flow* f = (rnf_flow*)calloc(1, sizeof(rnf_flow));
  if (!f) return fail(RNF_EINVAL, "out of host memory");
  f->model = *model;
  f->weights_dev = weights_dev;
  f->sm_count = sm;
  cudaGetDevice(&f->device);
  f->cond_floats = (int64_t)n_mob * rnf::kH + (int64_t)n_aff * (rnf::kAffFloats + rnf::kH);
  const size_t bytes = sizeof(rnf_layer_desc) * (size_t)(model->n_layers > 0 ? model->n_layers : 1);
  f->layers_host = (rnf_layer_desc*)malloc(bytes);
  if (model->n_layers > 0) memcpy(f->layers_host, layers, sizeof(rnf_layer_desc) * model->n_layers);
  static_assert(sizeof(rnf::LayerDev) == sizeof(rnf_layer_desc), "layer table layouts must agree");
  cudaError_t e = cudaMalloc((void**)&f->layers_dev, bytes);
  if (e == cudaSuccess && model->n_layers > 0)
    e = cudaMemcpy(f->layers_dev, layers, sizeof(rnf_layer_desc) * model->n_layers, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    free(f->layers_host);
    free(f);
    return cuda_fail(e, "rnf_flow_create");
  }
  *out = f;
  return RNF_OK;
}

void rnf_flow_destroy(rnf_flow* f) {
  if (!f) return;
  cudaFree(f->layers_dev);
  free(f->layers_host);
  free(f);
}

int64_t rnf_flow_cond_floats(const rnf_flow* f) { return f ? f->cond_floats : 0; }

int rnf_flow_condition(rnf_flow* f, const float* feat_dev, int64_t B, float* cond_dev, void* stream) {
  if (!f) return fail(RNF_EINVAL, "rnf_flow_condition: null handle");
  if (f->cond_floats == 0) return fail(RNF_ESTATE, "rnf_flow_condition: the flow is unconditional");
  if (B < 0 || (B > 0 && (!feat_dev || !cond_dev))) return fail(RNF_EINVAL, "rnf_flow_condition: bad arguments");
  cudaError_t e = rnf::launch_condition(f, feat_dev, B, cond_dev, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_flow_condition");
}

int64_t rnf_dedup_workspace_bytes(int64_t N) { return N > 0 ? (int64_t)rnf::dedup_scan_bytes(N) : 0; }

int rnf_dedup_rows(const float* feat_dev, int64_t N, int64_t F, int32_t* idx_out_dev, int32_t* first_out_dev, int64_t cap,
                   int32_t* count_out_dev, void* workspace_dev, int64_t workspace_bytes, void* stream) {
  if (N < 0 || F <= 0 || cap <= 0) return fail(RNF_EINVAL, "rnf_dedup_rows: bad sizes");
  if (N == 0) return RNF_OK;
  if (N > 0x7fffffffLL) return fail(RNF_EINVAL, "rnf_dedup_rows: N=%lld rows exceed the int32 row index", (long long)N);
  if (!feat_dev || !idx_out_dev || !first_out_dev || !count_out_dev || !workspace_dev) return fail(RNF_EINVAL, "rnf_dedup_rows: null buffer");
  if (workspace_bytes < rnf_dedup_workspace_bytes(N)) return fail(RNF_EINVAL, "rnf_dedup_rows: workspace too small");
  int sm = 148;
  int rc = rnf_device_check(&sm);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_dedup(feat_dev, N, F, idx_out_dev, first_out_dev, cap, count_out_dev, workspace_dev, (size_t)workspace_bytes,
                                    sm, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_dedup_rows");
}

int rnf_flow_condition_runs(rnf_flow* f, const float* feat_dev, const int32_t* first_dev, const int32_t* count_dev, int64_t cap,
                            float* cond_dev, void* stream) {
  if (!f) return fail(RNF_EINVAL, "rnf_flow_condition_runs: null handle");
  if (f->cond_floats == 0) return fail(RNF_ESTATE, "rnf_flow_condition_runs: the flow is unconditional");
  if (cap <= 0 || !feat_dev || !first_dev || !count_dev || !cond_dev) return fail(RNF_EINVAL, "rnf_flow_condition_runs: bad arguments");
  cudaError_t e = rnf::launch_condition(f, feat_dev, cap, cond_dev, (cudaStream_t)stream, first_dev, count_dev);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_flow_condition_runs");
}

int rnf_poison_if_overflow(const int32_t* count_dev, int64_t cap, float* ldj_dev, int64_t N, void* stream) {
  if (N < 0 || !count_dev || (N > 0 && !ldj_dev)) return fail(RNF_EINVAL, "rnf_poison_if_overflow: bad arguments");
  cudaError_t e = rnf::launch_poison(count_dev, cap, ldj_dev, N, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_poison_if_overflow");
}

static int run_rows(rnf_flow* f, bool inverse, const float* R_in, int64_t N, const float* cond, int64_t B,
                    const int32_t* feat_index, int64_t rows_per_image, float* R_out, float* ldj_out, float* scratch,
                    int mlp_mode, void* stream) {
  const char* who = inverse ? "rnf_flow_inverse" : "rnf_flow_forward";
  if (!f) return fail(RNF_EINVAL, "%s: null handle", who);
  if (N < 0) return fail(RNF_EINVAL, "%s: negative N", who);
  if (!valid_mode(mlp_mode)) return fail(RNF_EINVAL, "%s: bad mlp_mode %d", who, mlp_mode);
  if (N == 0) return RNF_OK;
  if (!R_in || !R_out || !ldj_out) return fail(RNF_EINVAL, "%s: null buffer", who);
  if (f->cond_floats > 0) {
    if (!cond || B <= 0) return fail(RNF_ESTATE, "%s: conditional flow needs the output of rnf_flow_condition", who);
    const int rc = row_map_ok(who, N, B, feat_index, rows_per_image);
    if (rc != RNF_OK) return rc;
  }
  if (inverse && !scratch) return fail(RNF_EINVAL, "%s: null scratch", who);
  rnf::FlowArgs a = flow_args(f, R_in, N, cond);
  a.feat_index = feat_index;
  a.rows_per_image = rows_per_image > 0 ? rows_per_image : 1;
  a.R_out = R_out;
  a.ldj_out = ldj_out;
  a.scratch = scratch;
  return launch_flow(f, a, 1, inverse, mlp_mode, stream, who);
}

int rnf_flow_forward(rnf_flow* f, const float* R_in, int64_t N, const float* cond, int64_t B, const int32_t* feat_index,
                     int64_t rows_per_image, float* R_out, float* ldj_out, int mlp_mode, void* stream) {
  return run_rows(f, false, R_in, N, cond, B, feat_index, rows_per_image, R_out, ldj_out, nullptr, mlp_mode, stream);
}

int64_t rnf_flow_inverse_scratch_floats(const rnf_flow* f, int64_t N) {
  if (!f || N <= 0) return 0;
  const int64_t tiles = (N + rnf::kV1Threads - 1) / rnf::kV1Threads;
  const int64_t ctas = tiles < f->sm_count ? tiles : f->sm_count;
  return ctas * 4 * rnf::kK * rnf::kV1Threads;
}

int rnf_flow_inverse(rnf_flow* f, const float* R_in, int64_t N, const float* cond, int64_t B, const int32_t* feat_index,
                     int64_t rows_per_image, float* R_out, float* ldj_out, float* scratch, int mlp_mode, void* stream) {
  return run_rows(f, true, R_in, N, cond, B, feat_index, rows_per_image, R_out, ldj_out, scratch, mlp_mode, stream);
}

int rnf_flow_logprob_grad(rnf_flow* f, const float* R_in, int64_t N, const float* cond, int64_t B, const int32_t* feat_index,
                          int64_t rows_per_image, const float* fisher_A, const float* fisher_c, float* logp_out, float* grad_out,
                          void* stream) {
  const char* who = "rnf_flow_logprob_grad";
  if (!f) return fail(RNF_EINVAL, "%s: null handle", who);
  if (N < 0) return fail(RNF_EINVAL, "%s: negative N", who);
  if ((fisher_A == nullptr) != (fisher_c == nullptr)) return fail(RNF_EINVAL, "%s: fisher_A and fisher_c must be given together", who);
  int rc = gradient_stack_ok(f, who);
  if (rc != RNF_OK || N == 0) return rc;
  if (!R_in || !logp_out || !grad_out) return fail(RNF_EINVAL, "%s: null buffer", who);
  const bool per_image = f->cond_floats > 0 || fisher_A != nullptr;
  if (f->cond_floats > 0 && !cond) return fail(RNF_ESTATE, "%s: conditional flow needs the output of rnf_flow_condition", who);
  if (per_image) {
    if (B <= 0) return fail(RNF_EINVAL, "%s: B must be > 0 for a conditional flow or a Fisher base term", who);
    rc = row_map_ok(who, N, B, feat_index, rows_per_image);
    if (rc != RNF_OK) return rc;
  }
  cudaError_t e = rnf::launch_flow_grad(f, R_in, N, cond, per_image ? feat_index : nullptr, per_image ? rows_per_image : 1, fisher_A,
                                        fisher_c, logp_out, grad_out, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

// shared argument checks of the training entry points
static int check_train_args(const rnf_flow* f, const char* who, const float* weights, const float* R_in, int64_t N, const float* cond,
                            int64_t B, const int32_t* feat_index, int64_t rows_per_image) {
  if (!f) return fail(RNF_EINVAL, "%s: null handle", who);
  if (N < 0) return fail(RNF_EINVAL, "%s: negative N", who);
  const int rc = gradient_stack_ok(f, who);
  if (rc != RNF_OK || N == 0) return rc;
  if (!weights || !R_in) return fail(RNF_EINVAL, "%s: null buffer", who);
  if (f->cond_floats > 0) {
    if (!cond) return fail(RNF_ESTATE, "%s: conditional flow needs its per-image constants", who);
    if (B <= 0) return fail(RNF_EINVAL, "%s: B must be > 0 for a conditional flow", who);
    return row_map_ok(who, N, B, feat_index, rows_per_image);
  }
  return RNF_OK;
}

int64_t rnf_flow_train_workspace_floats(const rnf_flow* f, int64_t N) { return f && N > 0 ? rnf::flow_train_workspace_floats(f, N) : 0; }

int rnf_flow_train_forward(rnf_flow* f, const float* weights_dev, const float* R_in, int64_t N, const float* cond, int64_t B,
                           const int32_t* feat_index, int64_t rows_per_image, float* R_out, float* ldj_out, void* stream) {
  const char* who = "rnf_flow_train_forward";
  const int rc = check_train_args(f, who, weights_dev, R_in, N, cond, B, feat_index, rows_per_image);
  if (rc != RNF_OK || N == 0) return rc;
  if (!R_out || !ldj_out) return fail(RNF_EINVAL, "%s: null buffer", who);
  const bool cnd = f->cond_floats > 0;
  cudaError_t e = rnf::launch_flow_train(f, false, weights_dev, R_in, N, cond, cnd ? feat_index : nullptr, cnd ? rows_per_image : 1,
                                         R_out, ldj_out, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int rnf_flow_train_backward(rnf_flow* f, const float* weights_dev, const float* R_in, int64_t N, const float* cond, int64_t B,
                            const int32_t* feat_index, int64_t rows_per_image, const float* G_Rout, const float* g_ldj, float* G_R,
                            float* workspace, int64_t workspace_floats, void* stream) {
  const char* who = "rnf_flow_train_backward";
  const int rc = check_train_args(f, who, weights_dev, R_in, N, cond, B, feat_index, rows_per_image);
  if (rc != RNF_OK || N == 0) return rc;
  if (!G_R || !workspace) return fail(RNF_EINVAL, "%s: null buffer", who);
  if (workspace_floats < rnf::flow_train_workspace_floats(f, N)) return fail(RNF_EINVAL, "%s: workspace too small", who);
  const bool cnd = f->cond_floats > 0;
  cudaError_t e = rnf::launch_flow_train(f, true, weights_dev, R_in, N, cond, cnd ? feat_index : nullptr, cnd ? rows_per_image : 1,
                                         nullptr, nullptr, G_Rout, g_ldj, G_R, workspace, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int64_t rnf_grid_partial_floats(int64_t G, int64_t B) {
  if (G <= 0 || B <= 0) return 0;
  const int64_t tpi = (G + 127) / 128;  // sized for the smaller (tensor-core) tile so either kernel fits
  return tpi * B * rnf::kPartStride;
}

int rnf_grid_logprob(rnf_flow* f, const float* grid_dev, int64_t G, int64_t g_index0, const float* offset_dev,
                     const float* cond_dev, int64_t B, const float* fisher_A_dev, const float* fisher_c_dev,
                     float* logp_out_dev, float* part_dev, float* max_out_dev, int64_t* argmax_out_dev,
                     float* sumexp_out_dev, int mlp_mode, void* stream) {
  return rnf_grid_logprob_spread(f, grid_dev, G, g_index0, offset_dev, cond_dev, B, fisher_A_dev, fisher_c_dev, nullptr, 0,
                                 logp_out_dev, part_dev, max_out_dev, argmax_out_dev, sumexp_out_dev, nullptr, mlp_mode, stream);
}

int rnf_grid_logprob_spread(rnf_flow* f, const float* grid_dev, int64_t G, int64_t g_index0, const float* offset_dev,
                            const float* cond_dev, int64_t B, const float* fisher_A_dev, const float* fisher_c_dev,
                            const float* gt_dev, int gt_k, float* logp_out_dev, float* part_dev, float* max_out_dev,
                            int64_t* argmax_out_dev, float* sumexp_out_dev, float* spread_num_out_dev, int mlp_mode,
                            void* stream) {
  if (!f) return fail(RNF_EINVAL, "rnf_grid_logprob: null handle");
  if (G < 0 || B < 0) return fail(RNF_EINVAL, "rnf_grid_logprob: negative size");
  if (!valid_mode(mlp_mode)) return fail(RNF_EINVAL, "rnf_grid_logprob: bad mlp_mode %d", mlp_mode);
  if (G == 0 || B == 0) return RNF_OK;
  if (!grid_dev || !part_dev || !max_out_dev || !argmax_out_dev || !sumexp_out_dev)
    return fail(RNF_EINVAL, "rnf_grid_logprob: null buffer");
  if ((fisher_A_dev == nullptr) != (fisher_c_dev == nullptr))
    return fail(RNF_EINVAL, "rnf_grid_logprob: fisher_A and fisher_c must be given together");
  if (f->cond_floats > 0 && !cond_dev) return fail(RNF_ESTATE, "rnf_grid_logprob: conditional flow needs rnf_flow_condition output");
  if ((gt_dev == nullptr) != (spread_num_out_dev == nullptr) || (gt_dev != nullptr && gt_k <= 0))
    return fail(RNF_EINVAL, "rnf_grid_logprob_spread: gt [B,K,3,3] (K >= 1) and spread_num_out go together");
  rnf::FlowArgs a = flow_args(f, grid_dev, G * B, cond_dev);
  a.G = G;
  a.g_index0 = g_index0;
  a.offset = offset_dev;
  a.fisher_A = fisher_A_dev;
  a.fisher_c = fisher_c_dev;
  a.logp_out = logp_out_dev;
  a.part = part_dev;
  a.gt = gt_dev;
  a.gt_k = gt_k;
  const int rc = launch_flow(f, a, B, false, mlp_mode, stream, "rnf_grid_logprob");
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_grid_combine(part_dev, a.tiles_per_image, B, g_index0, max_out_dev, argmax_out_dev, sumexp_out_dev,
                               spread_num_out_dev, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_grid_logprob (combine)");
}

int rnf_healpix_grid(int level, int64_t begin, int64_t end, float* R_out_dev, void* stream) {
  if (level < 0 || level > 8) return fail(RNF_EINVAL, "rnf_healpix_grid: level %d outside 0..8 (utils/sd.py:32)", level);
  int64_t total = 72;
  for (int i = 0; i < level; ++i) total *= 8;
  if (begin < 0 || end < begin || end > total) return fail(RNF_EINVAL, "rnf_healpix_grid: bad range");
  if (end == begin) return RNF_OK;
  if (!R_out_dev) return fail(RNF_EINVAL, "rnf_healpix_grid: null output");
  cudaError_t e = rnf::launch_healpix(level, begin, end, R_out_dev, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_healpix_grid");
}

int rnf_fisher_sample(const float* usv_dev, int64_t B, int64_t n_per_image, uint64_t seed, float* R_out_dev, void* stream) {
  if (B < 0 || n_per_image < 0) return fail(RNF_EINVAL, "rnf_fisher_sample: negative size");
  if (B == 0 || n_per_image == 0) return RNF_OK;
  if (!usv_dev || !R_out_dev) return fail(RNF_EINVAL, "rnf_fisher_sample: null buffer");
  cudaError_t e = rnf::launch_fisher_sample(usv_dev, B, n_per_image, (unsigned long long)seed, R_out_dev, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_fisher_sample");
}

int rnf_fisher_log_prob(const float* A9_dev, const float* c_dev, int64_t B, const float* R_dev, int64_t N, float* out_dev,
                        void* stream) {
  if (B <= 0 || N < 0) return fail(RNF_EINVAL, "rnf_fisher_log_prob: bad sizes");
  if (N == 0) return RNF_OK;
  if (N % B != 0) return fail(RNF_EINVAL, "rnf_fisher_log_prob: N=%lld rotations do not split evenly over B=%lld images "
                              "(utils/fisher.py:223 reshapes to (B, -1, 3, 3))", (long long)N, (long long)B);
  if (!A9_dev || !c_dev || !R_dev || !out_dev) return fail(RNF_EINVAL, "rnf_fisher_log_prob: null buffer");
  cudaError_t e = rnf::launch_fisher_logprob(A9_dev, c_dev, R_dev, N, N / B, out_dev, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_fisher_log_prob");
}

int rnf_min_geodesic(const float* est_dev, const float* gt_dev, int64_t B, int64_t K, float* out_dev, void* stream) {
  if (B < 0 || K <= 0) return fail(RNF_EINVAL, "rnf_min_geodesic: bad sizes");
  if (B == 0) return RNF_OK;
  if (!est_dev || !gt_dev || !out_dev) return fail(RNF_EINVAL, "rnf_min_geodesic: null buffer");
  cudaError_t e = rnf::launch_min_geodesic(est_dev, gt_dev, B, K, out_dev, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_min_geodesic");
}

int rnf_train_max_components(void) { return rnf::train_max_components(); }

static int train_args_ok(const char* who, int64_t N, int K, int perm) {
  if (N < 0) return fail(RNF_EINVAL, "%s: negative N", who);
  if (K < 1 || K > rnf::train_max_components()) return fail(RNF_ESHAPE, "%s: K=%d mixture components (1..%d supported)", who, K, rnf::train_max_components());
  if (perm < 0 || perm > 2) return fail(RNF_EINVAL, "%s: perm must be 0, 1 or 2", who);
  return rnf_device_check(nullptr);
}

int rnf_train_mobius_forward(const float* R, const float* out, int64_t N, int K, int perm, int inverse, float* R_out, float* ldj, float* theta,
                             void* stream) {
  int rc = train_args_ok("rnf_train_mobius_forward", N, K, perm);
  if (rc != RNF_OK) return rc;
  if (N > 0 && (!R || !out || !R_out || !ldj || !theta)) return fail(RNF_EINVAL, "rnf_train_mobius_forward: null buffer");
  cudaError_t e = rnf::launch_train_mobius_fwd(R, out, N, K, perm, inverse != 0, R_out, ldj, theta, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_train_mobius_forward");
}

int rnf_train_mobius_backward(const float* R, const float* out, int64_t N, int K, int perm, int inverse, const float* theta, const float* R_out,
                              const float* G_Rout, const float* g_ldj, float* G_R, float* G_out, void* stream) {
  int rc = train_args_ok("rnf_train_mobius_backward", N, K, perm);
  if (rc != RNF_OK) return rc;
  if (N > 0 && (!R || !out || !theta || !R_out || !G_Rout || !g_ldj || !G_R || !G_out)) return fail(RNF_EINVAL, "rnf_train_mobius_backward: null buffer");
  cudaError_t e = rnf::launch_train_mobius_bwd(R, out, N, K, perm, inverse != 0, theta, R_out, G_Rout, g_ldj, G_R, G_out, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_train_mobius_backward");
}

int rnf_train_affine_forward(const float* R, const float* W, int64_t N, float* R_out, float* loglen, void* stream) {
  int rc = train_args_ok("rnf_train_affine_forward", N, 1, 0);
  if (rc != RNF_OK) return rc;
  if (N > 0 && (!R || !W || !R_out || !loglen)) return fail(RNF_EINVAL, "rnf_train_affine_forward: null buffer");
  cudaError_t e = rnf::launch_train_affine_fwd(R, W, N, R_out, loglen, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_train_affine_forward");
}

int rnf_train_affine_backward(const float* R, const float* W, int64_t N, const float* R_out, const float* G_Rout, const float* g_loglen,
                              float* G_R, float* G_W, void* stream) {
  int rc = train_args_ok("rnf_train_affine_backward", N, 1, 0);
  if (rc != RNF_OK) return rc;
  if (N > 0 && (!R || !W || !R_out || !G_Rout || !g_loglen || !G_R || !G_W)) return fail(RNF_EINVAL, "rnf_train_affine_backward: null buffer");
  cudaError_t e = rnf::launch_train_affine_bwd(R, W, N, R_out, G_Rout, g_loglen, G_R, G_W, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_train_affine_backward");
}

// argument checks before the device check, so that a bad call is reported as such on any host; N == 0 is a no-op (the buffers of
// empty tensors may be null)
static int ablation_args_ok(const char* who, int64_t N, int kind, bool null_buffer) {
  if (N < 0) return fail(RNF_EINVAL, "%s: negative N", who);
  if (kind < RNF_LAYER_SMITH9 || kind > RNF_LAYER_RIGHT9) return fail(RNF_EINVAL, "%s: kind %d is not an ablation layer (%d..%d)", who, kind,
                                                                     RNF_LAYER_SMITH9, RNF_LAYER_RIGHT9);
  if (N == 0) return RNF_OK;
  if (null_buffer) return fail(RNF_EINVAL, "%s: null buffer", who);
  return rnf_device_check(nullptr);
}

int rnf_train_ablation_forward(const float* R, const float* M, int64_t N, int kind, float* R_out, float* ldj, void* stream) {
  int rc = ablation_args_ok("rnf_train_ablation_forward", N, kind, !R || !M || !R_out || !ldj);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_train_ablation_fwd(R, M, N, kind, R_out, ldj, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_train_ablation_forward");
}

int rnf_train_ablation_backward(const float* R, const float* M, int64_t N, int kind, const float* R_out, const float* G_Rout, const float* g_ldj,
                                float* G_R, float* G_M, void* stream) {
  int rc = ablation_args_ok("rnf_train_ablation_backward", N, kind, !R || !M || !R_out || !G_Rout || !g_ldj || !G_R || !G_M);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_train_ablation_bwd(R, M, N, kind, R_out, G_Rout, g_ldj, G_R, G_M, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, "rnf_train_ablation_backward");
}

int64_t rnf_rotation_modes_workspace_bytes(int64_t G, int64_t B, int M) {
  if (G < 0 || B <= 0 || M < 1) return 0;
  return rnf::modes_workspace_bytes(G, B);
}

int rnf_rotation_modes(const float* values, int64_t B, int64_t G, int64_t g_index0, const float* rot, int M, float min_separation,
                       float neighbour_radius, void* workspace, int64_t workspace_bytes, int64_t* index_out, float* value_out,
                       uint8_t* local_max_out, float* mass_out, int32_t* count_out, void* stream) {
  // argument checks before the device check, so that a bad call is reported as such on any host; B == 0 is a no-op and G == 0 reads
  // no input (the buffers of empty tensors may be null)
  const char* who = "rnf_rotation_modes";
  if (B < 0 || G < 0) return fail(RNF_EINVAL, "%s: negative size", who);
  float cos_sep, cos_nb;
  int rc = modes_thresholds(who, M, min_separation, neighbour_radius, &cos_sep, &cos_nb);
  if (rc == RNF_OK) rc = modes_slices_ok(who, "G", G);
  if (rc != RNF_OK || B == 0) return rc;
  if (!workspace || !index_out || !value_out || !local_max_out || !mass_out || !count_out || (G > 0 && (!values || !rot)))
    return fail(RNF_EINVAL, "%s: null pointer", who);
  if (workspace_bytes < rnf_rotation_modes_workspace_bytes(G, B, M)) return fail(RNF_EINVAL, "%s: workspace too small", who);
  rc = rnf_device_check(nullptr);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_rotation_modes(values, B, G, g_index0, rot, M, cos_sep, cos_nb, workspace, index_out, value_out, local_max_out,
                                             mass_out, count_out, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int64_t rnf_rotation_modes_shard_workspace_bytes(int64_t G_r, int64_t B) {
  if (G_r < 0 || B <= 0) return 0;
  return rnf::modes_shard_workspace_bytes(G_r, B);
}

int rnf_rotation_modes_shard_setup(const float* rot, int64_t G_r, int64_t B, void* workspace, int64_t workspace_bytes, void* stream) {
  const char* who = "rnf_rotation_modes_shard_setup";
  if (B < 0 || G_r < 0) return fail(RNF_EINVAL, "%s: negative size", who);
  int rc = modes_slices_ok(who, "G_r", G_r);
  if (rc != RNF_OK || B == 0 || G_r == 0) return rc;
  if (!rot || !workspace) return fail(RNF_EINVAL, "%s: null pointer", who);
  if (workspace_bytes < rnf_rotation_modes_shard_workspace_bytes(G_r, B)) return fail(RNF_EINVAL, "%s: workspace too small", who);
  rc = rnf_device_check(nullptr);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_modes_shard_setup(rot, G_r, B, workspace, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int rnf_rotation_modes_shard_round(const float* values, int64_t B, int64_t G_r, int64_t g_index0, const float* rot, int r, int M,
                                   float min_separation, float neighbour_radius, void* workspace, int64_t workspace_bytes, void* record_out,
                                   void* stream) {
  const char* who = "rnf_rotation_modes_shard_round";
  if (B < 0 || G_r < 0) return fail(RNF_EINVAL, "%s: negative size", who);
  if (g_index0 < 0) return fail(RNF_EINVAL, "%s: negative g_index0", who);
  float cos_sep, cos_nb;
  int rc = modes_thresholds(who, M, min_separation, neighbour_radius, &cos_sep, &cos_nb);
  if (rc != RNF_OK) return rc;
  if (r < 0 || r > M) return fail(RNF_EINVAL, "%s: round %d outside 0..M=%d", who, r, M);
  rc = modes_slices_ok(who, "G_r", G_r);
  if (rc != RNF_OK || B == 0) return rc;
  if (!workspace || !record_out || (G_r > 0 && (!values || !rot))) return fail(RNF_EINVAL, "%s: null pointer", who);
  if (((uintptr_t)record_out & 15) != 0) return fail(RNF_EINVAL, "%s: record buffer not 16-byte aligned", who);
  if (workspace_bytes < rnf_rotation_modes_shard_workspace_bytes(G_r, B)) return fail(RNF_EINVAL, "%s: workspace too small", who);
  rc = rnf_device_check(nullptr);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_modes_shard_round(values, B, G_r, g_index0, rot, r, M, cos_sep, cos_nb, workspace, record_out,
                                                (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int rnf_rotation_modes_shard_merge(const void* records, int W, int64_t B, int r, int M, void* workspace, int64_t workspace_bytes,
                                   int64_t* index_out, float* value_out, uint8_t* local_max_out, float* mass_out, int32_t* count_out,
                                   float* rot_out, void* stream) {
  const char* who = "rnf_rotation_modes_shard_merge";
  if (B < 0) return fail(RNF_EINVAL, "%s: negative size", who);
  if (W < 1) return fail(RNF_EINVAL, "%s: W=%d ranks, need at least 1", who, W);
  int rc = modes_count_ok(who, M);
  if (rc != RNF_OK) return rc;
  if (r < 0 || r > M) return fail(RNF_EINVAL, "%s: round %d outside 0..M=%d", who, r, M);
  if (B == 0) return RNF_OK;
  if (!records || !workspace || !index_out || !value_out || !local_max_out || !mass_out || !count_out || !rot_out)
    return fail(RNF_EINVAL, "%s: null pointer", who);
  if (((uintptr_t)records & 15) != 0) return fail(RNF_EINVAL, "%s: record buffer not 16-byte aligned", who);
  if (workspace_bytes < rnf::modes_shard_state_bytes(B)) return fail(RNF_EINVAL, "%s: workspace too small", who);
  rc = rnf_device_check(nullptr);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_modes_shard_merge(records, W, B, r, M, workspace, index_out, value_out, local_max_out, mass_out, count_out,
                                                rot_out, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

// argument checks before the device check, so that a bad call is reported as such on any host
int rnf_healpix_children(int level, const int64_t* parent, int64_t n, const float* offset, int64_t* child_out, float* R_out, void* stream) {
  const char* who = "rnf_healpix_children";
  if (level < 0 || level > 7) return fail(RNF_EINVAL, "%s: child level %d outside 1..8", who, level + 1);
  if (n < 0) return fail(RNF_EINVAL, "%s: negative n", who);
  if (n == 0) return RNF_OK;
  if (!parent || !child_out || !R_out) return fail(RNF_EINVAL, "%s: null buffer", who);
  // one thread per child, 256 per block: gridDim.x = n / 32 blocks must stay within 2^31 - 1
  if (n > (int64_t)0x7fffffff * 32) return fail(RNF_EINVAL, "%s: n=%lld parents exceed the (2^31 - 1) * 32 of one launch", who, (long long)n);
  const int rc = rnf_device_check(nullptr);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_healpix_children(level, parent, n, offset, child_out, R_out, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

int64_t rnf_topk_workspace_bytes(int64_t B, int64_t C, int K) {
  if (B <= 0 || C < 0 || K < 1 || K > 4096) return 0;
  return rnf::topk_workspace_bytes(B, C, K);
}

int rnf_topk(const float* values, const int64_t* index, int64_t B, int64_t C, int K, void* workspace, int64_t workspace_bytes, float* v_out,
             int64_t* i_out, void* stream) {
  const char* who = "rnf_topk";
  if (B < 0 || C < 0) return fail(RNF_EINVAL, "%s: negative size", who);
  if (K < 1 || K > 4096) return fail(RNF_EINVAL, "%s: K=%d outside 1..4096", who, K);
  if (B > 0x7fffffffLL) return fail(RNF_EINVAL, "%s: B=%lld images exceed one launch", who, (long long)B);
  if (rnf::topk_slices(C, K) > 65535) return fail(RNF_EINVAL, "%s: C=%lld entries exceed the 65535 slices of one launch", who, (long long)C);
  if (B == 0) return RNF_OK;
  const int64_t need = rnf_topk_workspace_bytes(B, C, K);
  if (!v_out || !i_out || (C > 0 && !values) || (need > 0 && !workspace)) return fail(RNF_EINVAL, "%s: null buffer", who);
  if (workspace_bytes < need) return fail(RNF_EINVAL, "%s: workspace too small", who);
  const int rc = rnf_device_check(nullptr);
  if (rc != RNF_OK) return rc;
  cudaError_t e = rnf::launch_topk(values, index, B, C, K, workspace, v_out, i_out, (cudaStream_t)stream);
  return e == cudaSuccess ? RNF_OK : cuda_fail(e, who);
}

}  // extern "C"
