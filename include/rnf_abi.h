/*
 * rnf_abi.h -- C ABI of librnf_b200.so: the B200 (sm_100a) hot path of RotationNormFlow.
 *
 * The reference (PKU-EPIC/RotationNormFlow) is 100 % Python and has no FFI; its boundary for this
 * path is the nn.Module protocol of flow/flow.py.  The entry points below are what a ctypes binding
 * for that path binds (INTEGRATION.md shows the stub); each cites the reference interface it replaces.
 * All file:line citations are relative to the reference repository root.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer named *_dev is DEVICE memory owned by the caller
 *     (PyTorch allocates it); nothing here allocates device memory except rnf_flow_create's small
 *     copy of the layer table.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default).
 *   - return 0 on success, negative RNF_E* on argument errors, positive = cudaError_t.
 *     rnf_last_error() returns a thread-local message for the last non-zero return.
 *   - rotations are float32 [N,3,3] row-major (the layout of the reference's `rotation` tensors).
 *   - re-entrant per (handle, stream); no global mutable state (nn.DataParallel-style concurrent
 *     callers on different devices each own a handle; agent.py:22,53-54).
 */
#ifndef RNF_ABI_H_
#define RNF_ABI_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RNF_ABI_VERSION 15

/* error codes */
#define RNF_OK 0
#define RNF_EINVAL (-1)   /* bad argument (null pointer, negative size, bad enum)   */
#define RNF_ESHAPE (-2)   /* model dimensions unsupported by the compiled kernels   */
#define RNF_ENODEV (-3)   /* no CUDA device / device is not sm_100                  */
#define RNF_ESTATE (-4)   /* handle is not usable for this call (e.g. no features)  */

/* layer kinds (flow/flow.py:36-51 builds a list of exactly these two families) */
#define RNF_LAYER_MOBIUS 0 /* flow/mobiusflow.py:27-183  MobiusFlow                                   */
#define RNF_LAYER_AFFINE 1 /* flow/squeezetrans.py:33-38 calculate_16, and flow/rottrans.py:8-66 (has_ldj=0) */
/* ablation replacements of the affine layer (flow/affineflow.py:27-41,55-70); parameter block per direction:           */
#define RNF_LAYER_SMITH9 2  /* calculate_9   squeezetrans.py:197-232: 3x3 M (forward) / inv(M); Gram-Schmidt + log-det   */
#define RNF_LAYER_SMITH36 3 /* calculate_36  squeezetrans.py:291-331: 6x6 M / inv(M) on the 6-D representation           */
#define RNF_LAYER_POLAR9L 4 /* calculate_9_l rottrans.py:69-72: polar factor of M R (inverse block: M^T); log-det 0       */
#define RNF_LAYER_POLAR9R 5 /* calculate_9_r rottrans.py:75-78: polar factor of R M (inverse block: M^T); log-det 0       */
#define RNF_LAYER_RIGHT9 6  /* calculate_9_r_smith rottrans.py:81-91: R Q, Q = Gram-Schmidt(M) (inverse block: Q^T)       */
#define RNF_AFFINE_BLOCK_FLOATS 80 /* per affine-family layer: forward block [0,40), inverse-direction block [40,80)     */

/* kernel selection for the conditioner MLP (flow/condition.py:24-30) */
#define RNF_MLP_FP32 0    /* FP32 CUDA-core FMA: the exact-precision path                             */
#define RNF_MLP_TC 1      /* tcgen05 tensor cores, error-compensated split operands, FP32 accumulate: forward / grid with four
                             tiles per SM and the activations in tensor memory (csrc/flow_t4.cu), inverse as RNF_MLP_TC_ROW */
#define RNF_MLP_TC_ROW 2  /* same arithmetic, two tiles per SM, activations through shared memory (csrc/flow_row.cu)   */

/*
 * One entry per layer, in module order (index i == `layers.{i}` of the reference state dict).
 *   perm      : row r of the cyclic table flow/flow.py:13-15 reduced mod 3; the layer acts on columns
 *               (r, r+1, r+2) mod 3 of R.  Ignored by affine layers.
 *   cond_slot : >= 0 -> this layer reads per-image data produced by rnf_flow_condition():
 *                 Mobius: 64 floats  W_f.feature  (first conditioner layer hoisted per image)
 *                 affine: the parameter block (RNF_AFFINE_BLOCK_FLOATS floats) of that image: the 4x4 matrix of Condition16Trans /
                         ConditionRot, or the 3x3 / 6x6 matrix of an ablation layer
 *               -1 -> unconditional.
 *   has_ldj   : affine only. 1 = log|det W| - 4 log|Wq| (squeezetrans.py:38); 0 = rotation layer (rottrans.py:21).
 *   w_off     : float offset of this layer's block inside the packed weight buffer (layout: DESIGN.md).
 */
typedef struct rnf_layer_desc {
  int32_t kind;
  int32_t perm;
  int32_t cond_slot;
  int32_t has_ldj;
  int64_t w_off;
  int64_t w_off_tc;   /* offset of the tensor-core (split fp16) image of the conditioner, -1 if absent */
} rnf_layer_desc;

typedef struct rnf_model_desc {
  int32_t abi_version;    /* RNF_ABI_VERSION                                                        */
  int32_t n_layers;
  int32_t K;              /* Mobius mixture components (config.segments); kernels are built for 64   */
  int32_t H;              /* conditioner hidden width (flow/condition.py:9 Nh); kernels built for 64 */
  int32_t F;              /* feature width seen by the flow (0 = unconditional)                      */
  int32_t n_mobius_slots; /* conditional Mobius layers                                               */
  int32_t n_affine_slots; /* conditional affine / rot layers                                         */
  int32_t affine_is_rot;  /* conditional affine slots: 0 = Condition16Trans (matrix, inverse and log-dets written by
                             rnf_flow_condition), 1 = ConditionRot (matrix written, the caller replaces it by its SVD polar
                             factor), 2 = ablation layers: the caller fills the slots' parameter blocks itself            */
  int64_t wf_off;         /* [n_mobius_slots + n_affine_slots][H][F] first-layer feature weights     */
  int64_t caff_off;       /* [n_affine_slots] blocks of the conditional-affine MLP tails             */
  int64_t n_floats;       /* total floats in the packed buffer                                       */
} rnf_model_desc;

typedef struct rnf_flow rnf_flow;

int rnf_abi_version(void);
const char* rnf_last_error(void);

/* Number of SMs / device check: 0 if the current device is sm_100, else RNF_ENODEV. */
int rnf_device_check(int* sm_count_out);

/*
 * Replaces Flow.__init__ / get_flow (flow/flow.py:9-51) for the device side: registers the layer table
 * and the packed weights (device pointer, caller-owned, must outlive the handle).
 */
int rnf_flow_create(const rnf_model_desc* model, const rnf_layer_desc* layers,
                    const float* weights_dev, rnf_flow** out);
void rnf_flow_destroy(rnf_flow* flow);

/* Floats per image in the buffer written by rnf_flow_condition (0 for an unconditional flow). */
int64_t rnf_flow_cond_floats(const rnf_flow* flow);

/*
 * Per-image part of the conditioners: replaces, for every conditional layer at once, the feature columns of
 * fc_first in ConditionalTransform.forward (flow/condition.py:25, input built at flow/mobiusflow.py:54) and the
 * whole Condition16Trans / ConditionRot matrix network (flow/squeezetrans.py:47-54, flow/rottrans.py:43-46),
 * including the inverse-direction matrices (torch.linalg.inv, squeezetrans.py:54 / transpose, rottrans.py:58).
 *   feat_dev [B,F] float32 row-major  ->  cond_dev [B, rnf_flow_cond_floats()]
 */
int rnf_flow_condition(rnf_flow* flow, const float* feat_dev, int64_t B, float* cond_dev, void* stream);

/*
 * The reference's calling convention: `feature [N,F]` row-aligned with the rotations, built by `.repeat` (agent.py:240-244,
 * eval.py:450), i.e. long runs of identical rows.  rnf_dedup_rows recovers the run structure on the device, asynchronously:
 *   idx_out_dev   [N]   int32: run number of every row (the feat_index_dev of rnf_flow_forward / _inverse), clamped to cap - 1
 *   first_out_dev [cap] int32: first row of run b (entries >= count are 0)
 *   count_out_dev [1]   int32: number of runs.  If it exceeds `cap` the per-image buffers sized by `cap` do not hold all
 *                       images: the caller either reads it back and retries with a larger cap, or (stream capture) calls
 *                       rnf_poison_if_overflow after the flow, which turns every log-det into NaN in that case.
 *   workspace_dev : rnf_dedup_workspace_bytes(N) bytes.
 * One streaming pass over the N x F floats (HBM-bound), a device-wide scan, a scatter: no host synchronisation.
 * rnf_flow_condition_runs is rnf_flow_condition for the images (feat row first[b], b < *count_dev) of that structure.
 */
int64_t rnf_dedup_workspace_bytes(int64_t N);
int rnf_dedup_rows(const float* feat_dev, int64_t N, int64_t F, int32_t* idx_out_dev, int32_t* first_out_dev, int64_t cap,
                   int32_t* count_out_dev, void* workspace_dev, int64_t workspace_bytes, void* stream);
int rnf_flow_condition_runs(rnf_flow* flow, const float* feat_dev, const int32_t* first_dev, const int32_t* count_dev,
                            int64_t cap, float* cond_dev, void* stream);
int rnf_poison_if_overflow(const int32_t* count_dev, int64_t cap, float* ldj_dev, int64_t N, void* stream);

/*
 * Flow.forward (flow/flow.py:53-72) and Flow.inverse (flow/flow.py:74-92).
 *   R_in_dev  [N,3,3]   rotations (not modified)
 *   cond_dev  [B,cond_floats] from rnf_flow_condition, NULL for an unconditional flow
 *   row -> image mapping (the reference takes a row-aligned `feature [N,F]`, built by .repeat at
 *   agent.py:240-244 / eval.py:450):  feat_index_dev[row] if non-NULL, else row / rows_per_image.
 *   R_out_dev [N,3,3], ldj_out_dev [N]
 *   scratch_dev : inverse only, rnf_flow_inverse_scratch_floats() floats (bisection parameters).
 */
int rnf_flow_forward(rnf_flow* flow, const float* R_in_dev, int64_t N, const float* cond_dev, int64_t B,
                     const int32_t* feat_index_dev, int64_t rows_per_image, float* R_out_dev,
                     float* ldj_out_dev, int mlp_mode, void* stream);
int64_t rnf_flow_inverse_scratch_floats(const rnf_flow* flow, int64_t N);
int rnf_flow_inverse(rnf_flow* flow, const float* R_in_dev, int64_t N, const float* cond_dev, int64_t B,
                     const int32_t* feat_index_dev, int64_t rows_per_image, float* R_out_dev,
                     float* ldj_out_dev, float* scratch_dev, int mlp_mode, void* stream);

/*
 * log p and its tangential rotation gradient (eval.py:464-480 nll_grad; the Riemannian gradient of the forward direction), one
 * launch, FP32 (csrc/flow_grad.cu, one warp per rotation).
 *   R_in_dev [N,3,3]; cond/B/feat_index/rows_per_image as rnf_flow_forward; fisher_A_dev [B,9], fisher_c_dev [B] or both NULL
 *   logp_out_dev [N] = ldj [+ sum(A_b * R') - c_b]; grad_out_dev [N,3,3] = R [g]x / 2 (the tangential part of d logp / dR)
 * K != 64 and ablation layers (kinds RNF_LAYER_SMITH9 .. RNF_LAYER_RIGHT9) return RNF_ESHAPE.
 */
int rnf_flow_logprob_grad(rnf_flow* flow, const float* R_in_dev, int64_t N, const float* cond_dev, int64_t B,
                          const int32_t* feat_index_dev, int64_t rows_per_image, const float* fisher_A_dev,
                          const float* fisher_c_dev, float* logp_out_dev, float* grad_out_dev, void* stream);

/*
 * Training (agent.py:49-87: the gradient of a loss on log p with respect to everything log p depends on), FP32, one warp per row
 * (csrc/flow_grad.cu).  Both calls read the FP32 Mobius images and the unconditional affine blocks from weights_dev, at the
 * handle's offsets (the packed-image sections of the tensor-core kernels are not read); cond/B/feat_index/rows_per_image as
 * rnf_flow_forward.  K != 64 and ablation layers return RNF_ESHAPE.
 *   forward : R_out_dev [N,3,3], ldj_out_dev [N] of the forward direction.
 *   backward: seeds G_Rout_dev [N,3,3] = dL/dR_out (NULL = 0) and g_ldj_dev [N] = dL/dldj (NULL = 1); writes
 *             G_R_dev [N,3,3] = dL/dR_in, tangential (R [g]x / 2), and the training records to workspace_dev
 *             (rnf_flow_train_workspace_floats(N) floats):
 *               [n_mobius_layers][N][772]: (y, 1) [4], relu(h0), relu(h1), relu(h2), relu(h0 + h3) [4 x 64],
 *                                          dL/dh0 (residual included), dL/dh1, dL/dh2, dL/dh3 [4 x 64], dL/d(fc_last out) [256]
 *                                          (fc_last outputs in the packed order: component c at 4c .. 4c+3)
 *               [n_affine_layers][N][16] : dL/dW of the forward 4x4 of the layer (per-image or unconditional block)
 *             Layer order is the stack order; the weight gradients are GEMMs over rows of these records and the
 *             log-det slot of an affine block (has_ldj) receives the sum of g_ldj over its rows.
 */
int64_t rnf_flow_train_workspace_floats(const rnf_flow* flow, int64_t N);
int rnf_flow_train_forward(rnf_flow* flow, const float* weights_dev, const float* R_in_dev, int64_t N, const float* cond_dev, int64_t B,
                           const int32_t* feat_index_dev, int64_t rows_per_image, float* R_out_dev, float* ldj_out_dev, void* stream);
int rnf_flow_train_backward(rnf_flow* flow, const float* weights_dev, const float* R_in_dev, int64_t N, const float* cond_dev, int64_t B,
                            const int32_t* feat_index_dev, int64_t rows_per_image, const float* G_Rout_dev, const float* g_ldj_dev,
                            float* G_R_dev, float* workspace_dev, int64_t workspace_floats, void* stream);

/*
 * Grid evaluation: the inner loops of eval.py:444-462 (gradient()) and agent.py:246-266 fused:
 * for every image b < B and every grid rotation g in [0,G):
 *     R = grid[g] @ offset            (eval.py:439-440; offset NULL = identity)
 *     (R', ldj) = Flow.forward(R, feature_b)
 *     logp[b,g] = ldj + [ sum(A_b * R') - sumS_b - logc_b ]     (utils/fisher.py:217-232, if fisher_A_dev != NULL)
 * and per image the running (max, first arg-max index, sum exp(logp - max)) over this call's grid slice.
 *   grid_dev      [G,3,3] this rank's slice of the grid;  g_index0 = global index of its first rotation
 *   fisher_A_dev  [B,9], fisher_c_dev [B] = sumS_b + logc_b   (both NULL for no base term)
 *   logp_out_dev  [B,G] or NULL
 *   part_dev      workspace, rnf_grid_partial_floats(G, B) floats
 *   max_out_dev [B] float, argmax_out_dev [B] int64 (global index), sumexp_out_dev [B] float (relative to max_out)
 */
int64_t rnf_grid_partial_floats(int64_t G, int64_t B);
int rnf_grid_logprob(rnf_flow* flow, const float* grid_dev, int64_t G, int64_t g_index0, const float* offset_dev,
                     const float* cond_dev, int64_t B, const float* fisher_A_dev, const float* fisher_c_dev,
                     float* logp_out_dev, float* part_dev, float* max_out_dev, int64_t* argmax_out_dev,
                     float* sumexp_out_dev, int mlp_mode, void* stream);

/*
 * The same with the spread metric of the north star fused into the reduction epilogue (SURVEY.md 8f N2; the reference has
 * no implementation of it -- it is the probability-weighted version of its own min_geodesic_distance_rotmats,
 * utils/utils.py:231-235):  per image  sum_g exp(logp[b,g] - max_b) * min_k angle(grid[g] @ offset, gt[b,k]).
 *   gt_dev             [B,gt_k,3,3] ground-truth rotations per image (gt_k >= 1 symmetric equivalents)
 *   spread_num_out_dev [B] float: the numerator above; spread_b = spread_num / sumexp (radians); partial sums of several
 *                      grid slices / ranks merge like sumexp (rescale by exp(max_r - max) and add).
 * gt_dev == NULL and spread_num_out_dev == NULL: identical to rnf_grid_logprob.
 */
int rnf_grid_logprob_spread(rnf_flow* flow, const float* grid_dev, int64_t G, int64_t g_index0, const float* offset_dev,
                            const float* cond_dev, int64_t B, const float* fisher_A_dev, const float* fisher_c_dev,
                            const float* gt_dev, int gt_k, float* logp_out_dev, float* part_dev, float* max_out_dev,
                            int64_t* argmax_out_dev, float* sumexp_out_dev, float* spread_num_out_dev, int mlp_mode,
                            void* stream);

/*
 * generate_healpix_grid (utils/sd.py:48-82): rotations [begin,end) of the level-`level` grid
 * (72*8^level rotations, index = tilt*npix + pixel, RING pixel order), float64 math -> float32.
 */
int rnf_healpix_grid(int level, int64_t begin, int64_t end, float* R_out_dev, void* stream);

/*
 * MatrixFisherN._sample / sample_matrix_fisher (utils/fisher.py:117-207,234-243): n_per_image rotations per image from the
 * matrix-Fisher distribution with parameter A_b = U_b diag(S_b) V_b^T (proper SVD, utils/fisher.py:48-64), by rejection from
 * the angular-central-Gaussian envelope of the equivalent Bingham distribution on quaternions (b = 1.5).
 *   usv_dev   [B,24]: U (9, row-major), proper S (3), V (9), 3 pad floats
 *   seed      selects the random stream (Philox4x32-10 keyed by seed, counter = sample index / attempt): reproducible
 *             per (seed, B, n_per_image), independent of torch's generator -- parity with the reference is distributional
 *   R_out_dev [B,n_per_image,3,3]
 */
int rnf_fisher_sample(const float* usv_dev, int64_t B, int64_t n_per_image, uint64_t seed, float* R_out_dev, void* stream);

/*
 * MatrixFisherN._log_prob (utils/fisher.py:217-232) for image-major rows: R_dev [N,3,3] with N = B * rows_per_image,
 * A9_dev [B,9], c_dev [B] = sum of proper singular values + log normaliser (rotationnormflow_b200.fisher.fisher_constants)
 *   out[i] = sum(A_b * R_i) - c_b
 */
int rnf_fisher_log_prob(const float* A9_dev, const float* c_dev, int64_t B, const float* R_dev, int64_t N, float* out_dev,
                        void* stream);

/*
 * min_geodesic_distance_rotmats (utils/utils.py:231-235; K = 1: geodesic_distance_rotmats, :225-228): est_dev [B,3,3],
 * gt_dev [B,K,3,3] -> out_dev [B] = angle (radians) to the closest ground-truth rotation.  Post-path metric (SURVEY 8f N2).
 */
int rnf_min_geodesic(const float* est_dev, const float* gt_dev, int64_t B, int64_t K, float* out_dev, void* stream);

/*
 * Differentiable per-layer operators (csrc/train_ops.cu): what Flow.forward / Flow.inverse run when autograd is on -- training,
 * agent.py:87; eval.py:468-477 -- or when config.segments != 64.  The conditioner MLP (flow/condition.py:24-30) stays a sequence of
 * library GEMMs on the caller's side (its backward is the autograd of those); these are the Mobius mixture (flow/mobiusflow.py:58-85
 * forward, :141-183 inverse with BinFind.forward, :196-224) and calculate_16 (flow/squeezetrans.py:33-38), forward and
 * vector-Jacobian product, any number K <= rnf_train_max_components() of mixture components, one rotation per thread, FP32.
 *   R_dev [N,3,3]; out_dev [N,4K] conditioner output (K logits, then K x 3 centres); perm = first column of the cyclic row.
 *   forward : R_out_dev [N,3,3], ldj_dev [N] (the layer's own log-det, inverse direction included), theta_dev [N] (mixture angle /
 *             returned bisection root, needed by the backward of the inverse direction)
 *   backward: G_Rout_dev [N,3,3], g_ldj_dev [N] incoming; G_R_dev [N,3,3], G_out_dev [N,4K] outgoing.  Rotation gradients are
 *             TANGENTIAL (R [g]x / 2): the component that reaches parameters and features; BinFind.backward's implicit-function
 *             rule (flow/mobiusflow.py:248-273) is the inverse-direction case.
 *   affine  : W_dev [N,4,4] per-row matrices; loglen = log|W q|; the caller adds log|det W| itself.
 */
int rnf_train_max_components(void);
int rnf_train_mobius_forward(const float* R_dev, const float* out_dev, int64_t N, int K, int perm, int inverse, float* R_out_dev,
                             float* ldj_dev, float* theta_dev, void* stream);
int rnf_train_mobius_backward(const float* R_dev, const float* out_dev, int64_t N, int K, int perm, int inverse, const float* theta_dev,
                              const float* R_out_dev, const float* G_Rout_dev, const float* g_ldj_dev, float* G_R_dev, float* G_out_dev,
                              void* stream);
int rnf_train_affine_forward(const float* R_dev, const float* W_dev, int64_t N, float* R_out_dev, float* loglen_dev, void* stream);
int rnf_train_affine_backward(const float* R_dev, const float* W_dev, int64_t N, const float* R_out_dev, const float* G_Rout_dev,
                              const float* g_loglen_dev, float* G_R_dev, float* G_W_dev, void* stream);

/*
 * Differentiable ablation layers (csrc/ablation_layers.cuh; flow/affineflow.py:27-41,55-70): the same per-row arithmetic as the fused
 * kernels, forward and vector-Jacobian product, one rotation per thread, FP32.
 *   kind : RNF_LAYER_SMITH9 .. RNF_LAYER_RIGHT9
 *   M_dev: [N,n,n] (n = 6 for RNF_LAYER_SMITH36, else 3), the matrix the layer applies IN THIS DIRECTION, one per row: inv(M) of the
 *          Smith layers and M^T of the SVD layers in the inverse direction, the Gram-Schmidt Q (or Q^T) of calculate_9_r_smith.
 *   forward : R_out_dev [N,3,3], ldj_dev [N] (log|det| of the Smith layers by tangent propagation; 0 for the others)
 *   backward: the saved R_dev, M_dev, R_out_dev and the incoming G_Rout_dev [N,3,3], g_ldj_dev [N]; writes the TANGENTIAL rotation
 *             gradient G_R_dev [N,3,3] (R [g]x / 2) and G_M_dev [N,n,n] per row.
 */
int rnf_train_ablation_forward(const float* R_dev, const float* M_dev, int64_t N, int kind, float* R_out_dev, float* ldj_dev, void* stream);
int rnf_train_ablation_backward(const float* R_dev, const float* M_dev, int64_t N, int kind, const float* R_out_dev, const float* G_Rout_dev,
                                const float* g_ldj_dev, float* G_R_dev, float* G_M_dev, void* stream);

/*
 * Separated posterior modes of a grid log-density (csrc/modes.cu; DESIGN 4.7): per image, M rounds of greedy non-maximum
 * suppression on SO(3).  Round m takes the best point not yet labelled (NaN first, then larger value, then lower index: the order
 * of the grid arg-max), reports whether it is a local maximum (no point within neighbour_radius is higher) and labels every
 * unlabelled point closer than min_separation with m.  Angles are tested on quaternions of the fp32 matrices:
 * angle < theta <=> |q_g . q_c| > cos(theta / 2), angle <= rho <=> |q_g . q_c| >= cos(rho / 2).
 *   values_dev [B,G] float32 (e.g. the logp of rnf_grid_logprob); rot_dev [G,3,3] any rotation set (the geodesic angle is
 *   right-invariant, so the grid without its offset gives the same labels); 1 <= M <= 256; 0 < neighbour_radius <= min_separation <= pi
 *   workspace_dev  rnf_rotation_modes_workspace_bytes(G, B, M) bytes
 *   index_out_dev [B,M] int64 global index (g_index0 + local), value_out_dev [B,M], local_max_out_dev [B,M] (0/1),
 *   mass_out_dev [B,M] = sum over the mode's points of exp(v - v_mode0) / sum over all points of the same, count_out_dev [B] int32.
 *   Entries at or after count are padding: index -1, value -inf, local_max 0, mass 0.  B == 0 does nothing; G == 0 writes padding.
 * 2M + 3 launches, no atomics, no host synchronisation: bitwise reproducible and CUDA-graph capturable.
 */
int64_t rnf_rotation_modes_workspace_bytes(int64_t G, int64_t B, int M);
int rnf_rotation_modes(const float* values_dev, int64_t B, int64_t G, int64_t g_index0, const float* rot_dev, int M, float min_separation,
                       float neighbour_radius, void* workspace_dev, int64_t workspace_bytes, int64_t* index_out_dev, float* value_out_dev,
                       uint8_t* local_max_out_dev, float* mass_out_dev, int32_t* count_out_dev, void* stream);

/*
 * The same modes over a grid split across ranks (csrc/modes.cu; DESIGN 4.7 "Sharded"): rank k holds values [B,G_r] and rotations
 * [G_r,3,3] of the contiguous global slice [g_index0, g_index0 + G_r); every rank ends with the outputs rnf_rotation_modes gives on
 * the whole [B,G] (index, value, local_max, count bit for bit; mass up to the order of its sums).  Per rank:
 *   rnf_rotation_modes_shard_setup  once (quaternions of the slice), then for r = 0 .. M:
 *     rnf_rotation_modes_shard_round  writes this rank's record of round r, record_out_dev [B] x RNF_MODES_RECORD_BYTES;
 *     the caller all-gathers the records of the W ranks, rank-major, to records_dev [W][B] x RNF_MODES_RECORD_BYTES;
 *     rnf_rotation_modes_shard_merge  folds them in rank order and writes mode r-1's mass / local_max and mode r's index / value /
 *                                     rotation (rot_out_dev [B,M,3,3], the owning rank's matrix; padding NaN) and count_out_dev.
 *   workspace_dev  rnf_rotation_modes_shard_workspace_bytes(G_r, B) bytes, the same buffer for every call of one rank (the merged
 *                  state lives in it); record buffers 16-byte aligned.
 * Argument rules as rnf_rotation_modes, plus 0 <= r <= M, g_index0 >= 0, W >= 1.  B == 0 does nothing; G_r == 0 (an empty slice) reads
 * no input: setup does nothing and the round writes this rank's empty records, so the rank still takes part in every gather.
 * 2 launches per round and 1 per merge, no atomics, no host synchronisation: bitwise reproducible and CUDA-graph capturable.
 */
#define RNF_MODES_RECORD_BYTES 80
int64_t rnf_rotation_modes_shard_workspace_bytes(int64_t G_r, int64_t B);
int rnf_rotation_modes_shard_setup(const float* rot_dev, int64_t G_r, int64_t B, void* workspace_dev, int64_t workspace_bytes, void* stream);
int rnf_rotation_modes_shard_round(const float* values_dev, int64_t B, int64_t G_r, int64_t g_index0, const float* rot_dev, int r, int M,
                                   float min_separation, float neighbour_radius, void* workspace_dev, int64_t workspace_bytes,
                                   void* record_out_dev, void* stream);
int rnf_rotation_modes_shard_merge(const void* records_dev, int W, int64_t B, int r, int M, void* workspace_dev, int64_t workspace_bytes,
                                   int64_t* index_out_dev, float* value_out_dev, uint8_t* local_max_out_dev, float* mass_out_dev,
                                   int32_t* count_out_dev, float* rot_out_dev, void* stream);

/*
 * Coarse-to-fine search on the HEALPix grids (csrc/hgrid.cu; DESIGN 4.8).
 *
 * rnf_healpix_children: the 8 level-(level+1) children of level-`level` grid indices (0 <= level <= 7).  For parent idx = t*npix + p
 * (nside = 2^level, npix = 12 nside^2, p the RING pixel) child k = 4*dt + j (dt = 0, 1; j = 0..3) is
 *   t' = 2t + dt,  p' = nest2ring(2 nside, 4 ring2nest(nside, p) + j),  index t' * 4 npix + p'
 * (the NESTED subdivision: the children of all level-l indices partition the level-(l+1) grid).
 *   parent_dev [n] int64; offset_dev [3,3] or NULL; child_out_dev [n,8] int64; R_out_dev [n,8,3,3] = rnf_healpix_grid's row of the
 *   child, times the offset by the fmaf chain of rnf_grid_logprob (bit for bit the rotation the grid pass scores at that index).
 *   A parent outside [0, 72*8^level) (padding -1) gives children -1 and NaN rotations.  n == 0 does nothing; n <= (2^31 - 1) * 32.
 *
 * rnf_topk: per image the K best of values_dev [B,C] under the order of the grid arg-max (NaN first, then the larger value, then the
 * lower index), best first.  index_dev [B,C] int64 gives each entry's index (NULL: the column number); an entry with a negative index
 * is padding, ranked after every other entry.  1 <= K <= 4096; v_out_dev [B,K], i_out_dev [B,K] int64; places past the real entries
 * (K > C, or padding) are (-inf, -1).  workspace_dev: rnf_topk_workspace_bytes(B, C, K) bytes (0 is a valid size: no buffer needed).
 * B == 0 does nothing; C == 0 writes padding.  1 + ceil(log2(ceil(C / max(4096, 2 Kp)))) launches (Kp = K rounded up to a power of
 * two), no atomics, no host synchronisation: bitwise reproducible and CUDA-graph capturable.
 */
int rnf_healpix_children(int level, const int64_t* parent_dev, int64_t n, const float* offset_dev, int64_t* child_out_dev, float* R_out_dev,
                         void* stream);
int64_t rnf_topk_workspace_bytes(int64_t B, int64_t C, int K);
int rnf_topk(const float* values_dev, const int64_t* index_dev, int64_t B, int64_t C, int K, void* workspace_dev, int64_t workspace_bytes,
             float* v_out_dev, int64_t* i_out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RNF_ABI_H_ */
