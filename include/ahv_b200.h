/* lib3dahv_b200 — C ABI of the B200-native 3DAHV hypothesis-and-verification path.
 *
 * The reference (sailor-z/3DAHV) is pure Python/PyTorch and has no FFI of its
 * own; the hot path is an idiom pasted at modules/model.py:131-146, :184-196,
 * test_co3d.py:106,137-146 and test_linemod.py:43-63.  Every entry point below
 * cites the reference code it replaces.  All pointers are DEVICE pointers to
 * contiguous, 16-byte-aligned buffers owned by the caller unless the name ends
 * in `_host`.  `stream` is a `cudaStream_t` passed as `void*`.  Calls are
 * asynchronous and stream-ordered, allocate nothing (the `_host` entries, whose
 * scratch lives in a caller-owned session, and the explicit ahv_peer_alloc aside),
 * keep no global state, read no environment variables, and are CUDA-graph
 * capturable.  Return value: 0 on success, negative `AHV_E*`.
 * There is NO CPU fallback: on a device that is not sm_100 the compute entry
 * points return AHV_ENOTSUP.
 *
 * Fixed sizes of the path (modules/modules.py:64,97-100): volume C=16, D=H=W=8;
 * tri-plane K=384; verification head 384->32->32; 64 positions.
 */
#ifndef AHV_B200_H_
#define AHV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define AHV_API __attribute__((visibility("default")))
#else
#define AHV_API
#endif

#define AHV_VERSION 200 /* 0.2.0 */

enum {
  AHV_OK = 0,
  AHV_EINVAL = -1,  /* bad shape / null pointer / misaligned pointer / bad enum */
  AHV_ENOTSUP = -2, /* device is not sm_100 (no fallback path exists) */
  AHV_ECUDA = -3,   /* a CUDA runtime call or kernel launch failed */
  AHV_EWORKSPACE = -4 /* workspace too small: see ahv_workspace_bytes */
};

/* volume element type of `vol_src` */
enum { AHV_VOL_F32 = 0, AHV_VOL_BF16 = 1 };

/* arithmetic of the two 1x1 convolutions inside ahv_score:
 *   AHV_MATH_TC   fp16 operands (10-bit mantissa, TF32-equivalent) on tcgen05
 *                 tensor cores with fp32 accumulation in TMEM — the fast path;
 *   AHV_MATH_FP32 plain fp32 FFMA on CUDA cores — the bit-tight verification
 *                 mode (about 1e-6 relative to the reference).
 *   AHV_MATH_TC_F16GATHER  opt-in fast mode: as AHV_MATH_TC, but the source volume is
 *                 staged in shared memory as (scaled) fp16 and interpolated with packed
 *                 HFMA2, halving the shared-memory gather traffic.  bf16 volumes always
 *                 take this path (their staging is exact).  About 2e-4 relative.
 * Normalisation, correlation and selection are fp32 in every mode; trilinear resampling is
 * fp32 except in the f16-gather path.
 * Weight range: the tensor-core modes pack W1 and W2 as fp16(W * 2^-e), powers of two chosen so that
 * the largest row L1 norm lies in [4, 8) for W1 and in [1, 2) for W2, and undo them with the pair
 * scale before the bias.  The scores therefore do not depend on the weights' magnitude: scaling W1,
 * W2 or b2 by a power of two along the score's symmetries (W1 and b2 together, or W2 and b2) gives
 * bit-identical scores, and weights far below or above fp16's range (down to 1e-7 times and up to
 * 2e7 times a default initialisation, entries above 65504 included) meet the gates below at the
 * errors of the default initialisation (scripts/weight_range.py, tests/test_gpu_weight_range.py).
 * What fp16 cannot absorb is the spread between W1's rows, which sets the precision of the fp16
 * conv1 output: one row 2^4 times the others stays within every gate; at 2^6 AHV_MATH_TC (8.8e-4)
 * and bf16 volumes (1.8e-3) still do and AHV_MATH_TC_F16GATHER (2.1e-3) does not; at 2^8 none does.
 * Dynamic range: each pair's volume is multiplied by a power of two that maps max|V| into (b/2, b],
 * b = 32768 / L1n with L1n the normalised W1's largest row L1 norm (so b is in (4096, 8192] for any
 * W1 and conv1's output stays below 2^15), and undone before the bias, so one large voxel pushes the
 * rest of the volume towards fp16's subnormals.  Measured on an NVIDIA B200 (1000 W) against fp64,
 * for a standard-normal volume with outlier voxels up to r times larger (scripts/dynamic_range.py,
 * tests/test_gpu_pair_scale.py), the scores meet their gates as follows, for any W1 magnitude:
 *   AHV_MATH_TC, fp32 volumes           1e-3 up to r = 1e8 (4.4e-4 there; 7.5e-3 at 1e9)
 *   AHV_MATH_TC_F16GATHER, fp32 volumes 1e-3 up to r = 1e8 (6.2e-4 there; 8.2e-3 at 1e9)
 *   bf16 volumes (either tensor-core mode) 2e-3 against the bf16-rounded volume and 1e-2 against the
 *                                       unrounded one up to r = 1e8 (6.0e-4 there; 8.6e-3 at 1e9)
 *   AHV_MATH_FP32                       2e-5 up to r = 3e5; beyond it fp32 rounding of the outlier's
 *                                       share (the reference's fp32 path too) reaches 1e-4 at r = 1e7. */
enum { AHV_MATH_TC = 0, AHV_MATH_FP32 = 1, AHV_MATH_TC_F16GATHER = 2 };

AHV_API int ahv_version(void);
AHV_API const char* ahv_status_string(int status);

/* pytorch3d.transforms.random_rotations arithmetic (call sites
 * modules/model.py:102,131,184; model_co3d.py:86; test_co3d.py:106):
 * normals [n,4] (drawn by the caller, e.g. torch's CPU generator as the
 * reference does) -> unit quaternion with real part >= 0 -> R [n,3,3] row-major.
 * Individually rounded IEEE fp32 ops, bit-exact with oracle/ahv_oracle.c. */
AHV_API int ahv_so3_from_normals(const float* normals, float* R, int64_t n, void* stream);

/* Native sampler (extension; the reference only has CPU i.i.d. sampling):
 * Philox-4x32-10 counter RNG + Box-Muller normals + the same quaternion map.
 * Hypothesis i depends only on (seed, first_index + i), so any shard of the set
 * can be generated independently on any GPU. */
AHV_API int ahv_so3_sample(uint64_t seed, int64_t first_index, float* R, int64_t n, void* stream);

/* Deterministic SO(3) grid (extension, BASELINE config 4 "dense SO(3) grid"): points
 * [first_index, first_index+count) of the n_total-point super-Fibonacci spiral, as rotation
 * matrices.  Evaluated in fp64, rounded once: bit-identical to oracle/ahv_oracle.c. */
AHV_API int ahv_so3_grid(int64_t n_total, int64_t first_index, float* R, int64_t count, void* stream);

/* Local refinement set (extension, BASELINE config 4 "top-k refinement pass"; the reference has none):
 * R_out[i,0] = R_center[i]; R_out[i,j] = dR(i,j) @ R_center[i] for 0 < j < m, dR a Haar rotation (Philox
 * counter i*m+j keyed by seed) whose angle is rescaled from [0,pi] to [0,max_angle_deg] about its axis.
 * R_center [n,3,3] -> R_out [n,m,3,3].  Restated (to rounding of the transcendental functions) in
 * oracle/ahv_oracle.c. */
AHV_API int ahv_so3_perturb(const float* R_center, int64_t n, int m, float max_angle_deg, uint64_t seed, float* R_out,
                            void* stream);

/* utils.rotate_volume (utils.py:113-131): F.affine_grid + F.grid_sample
 * (trilinear, zeros padding, align_corners=False), materialised.
 * vol: [16,8,8,8] when vol_per_rotation==0 (the stride-0 `expand` of
 * modules/model.py:186) or [n,16,8,8,8] when 1 (:137).  out: [n,16,8,8,8].
 * base: the 8 base coordinates of affine_grid for size 8 (see DESIGN.md). */
AHV_API int ahv_rotate_volume(const float* vol, int vol_per_rotation, const float* R, const float* base,
                      float* out, int64_t n, void* stream);

/* Gradient of ahv_rotate_volume with respect to the volume (training variant, the autograd path of
 * utils.py:113-131 inside infoNCE_loss, modules/model.py:53): grad_out [n,16,8,8,8] is scattered
 * through the same trilinear taps.  vol_per_rotation==0: contributions of all n rotations are ADDED
 * into grad_vol [16,8,8,8] (caller zeroes it); ==1: grad_vol [n,16,8,8,8] is overwritten. */
AHV_API int ahv_rotate_volume_backward(const float* grad_out, int vol_per_rotation, const float* R,
                                       const float* base, float* grad_vol, int64_t n, void* stream);

/* dS/dR of ahv_rotate_volume (utils.py:113-131 differentiated in its grid, as F.grid_sample's backward does):
 * grad_R [n,3,3] is overwritten.  vol as in ahv_rotate_volume, grad_out [n,16,8,8,8].  ATen's convention: corner =
 * floor (forward difference at an exact integer coordinate), out-of-range taps contribute zero, and the derivative
 * along an axis is zero unless -1 <= its un-normalised coordinate < 8. */
AHV_API int ahv_rotate_volume_grad_R(const float* vol, int vol_per_rotation, const float* R, const float* base,
                                     const float* grad_out, float* grad_R, int64_t n, void* stream);

/* Gradient of the verification scores (training variant: the autograd path of modules/model.py:53-56 inside
 * infoNCE_loss, :43-63) in one fused kernel: for every (pair b, hypothesis n) the forward is recomputed in
 * shared memory and grad_scores[b,n] is pushed back to the source volume, the target features, W1, W2 and
 * b2 (fp32).  vol_src [B,16,8,8,8], tgt_feat [B,32,64] = forward_3d2d(vol_tgt), R [N,3,3] or [B,N,3,3],
 * grad_scores [B,N].  Gradients are ADDED into grad_vol [B,16,8,8,8], grad_tgt [B,32,64], grad_W1 [32,384],
 * grad_W2 [32,32], grad_b2 [32] (caller zeroes them).  Nothing is materialised per hypothesis. */
AHV_API int ahv_score_backward(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                               const float* W1, const float* W2, const float* b2, const float* base,
                               const float* grad_scores, float* grad_vol, float* grad_tgt, float* grad_W1,
                               float* grad_W2, float* grad_b2, int B, int64_t N, void* stream);

/* ResNetBlock_3D(32 -> 16, BN=False, stride 1) of the lifting stage (modules/modules.py:9-47 as applied at
 * :100-101 inside Feature_Aligner.forward_2d3d) - the step immediately upstream of the path (SURVEY.md §8f-2):
 *   out = conv2(relu(conv1(x))) + downsample(x)
 * x [m,32,8,8,8] -> out [m,16,8,8,8]; conv1_w [16,32,3,3,3], conv2_w [16,16,3,3,3], down_w [16,32(,1,1,1)]
 * (state-dict feature_aligner.feature_embedding_3d.{conv1,conv2,downsample.0}.weight).  One launch: a cluster of
 * 8 CTAs per volume (one depth slab each), the intermediate exchanged through distributed shared memory.
 * fp32 FFMA.  Inference only. */
AHV_API int ahv_resblock3d(const float* x, const float* conv1_w, const float* conv2_w, const float* down_w, float* out,
                           int64_t m, void* stream);

/* Saved-activation form of the training step (the reference's autograd saves ~420 KB per hypothesis; this saves 4 KB):
 * ahv_score_train = ahv_score with AHV_MATH_TC, fp32 volumes, k = 0, that also keeps conv1's ReLU'd output of every
 * (pair, hypothesis) - h1_saved [B*N][64][32] fp16 in the kernel's units (pair scale s, normalised W1) - and per
 * pair the factor that turns it back into conv1's output, 2^e1 / s (pair_inv_scale [B]; 2^-e1 is W1's normaliser);
 * ahv_score_backward_saved = ahv_score_backward reading them instead of recomputing conv1
 * (786 k of the backward's 2.4 M FMA per item).  math_mode AHV_MATH_FP32: the remaining contractions in fp32 FFMA;
 * AHV_MATH_TC: dA = dH1 W1 and dW1 = dH1^T A on tcgen05 (fp16 operands under power-of-two scales, fp32 accumulation in
 * TMEM; csrc/ahv_score_bwd_tc.cu).  Workspace: ahv_workspace_bytes(B, N, 1). */
AHV_API int ahv_score_train(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair, const float* W1,
                            const float* W2, const float* b2, const float* base, float* scores, void* h1_saved,
                            float* pair_inv_scale, int B, int64_t N, void* workspace, size_t workspace_bytes,
                            void* stream);
AHV_API int ahv_score_backward_saved(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                                     const float* W1, const float* W2, const float* b2, const float* base,
                                     const float* grad_scores, const void* h1_saved, const float* pair_inv_scale,
                                     float* grad_vol, float* grad_tgt, float* grad_W1, float* grad_W2, float* grad_b2,
                                     int B, int64_t N, int math_mode, void* stream);
/* ahv_score_backward / ahv_score_backward_saved plus the rotation gradient: h1_saved/pair_inv_scale both NULL =
 * recompute conv1; each gradient output may be NULL (at least one not); grad_R [N,3,3] (summed over pairs) or
 * [B,N,3,3], ADDED like the others.  fp32 FFMA in both forms (the saved-activation form is the AHV_MATH_FP32 kernel of
 * ahv_score_backward_saved); the rotation gradient follows ahv_rotate_volume_grad_R's convention.  Outputs left NULL
 * cost nothing: grad_R alone skips the adjoint of the resampling and the dW1 contraction. */
AHV_API int ahv_score_backward_ex(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                                  const float* W1, const float* W2, const float* b2, const float* base,
                                  const float* grad_scores, const void* h1_saved, const float* pair_inv_scale,
                                  float* grad_vol, float* grad_tgt, float* grad_W1, float* grad_W2, float* grad_b2,
                                  float* grad_R, int B, int64_t N, void* stream);

/* Deterministic form of the three backward entries above: bit-identical gradients from run to run (what PyTorch's
 * torch.use_deterministic_algorithms asks for).  Arguments as ahv_score_backward_ex, plus:
 *   math_mode   AHV_MATH_FP32 or AHV_MATH_TC.  h1_saved/pair_inv_scale NULL = the recompute form (fp32 FFMA, as
 *               ahv_score_backward / _ex); with them, AHV_MATH_FP32 = the FFMA form and AHV_MATH_TC = the tcgen05 form
 *               of ahv_score_backward_saved.  AHV_MATH_TC needs all five of grad_vol .. grad_b2 and no grad_R.
 *   workspace   ahv_score_backward_det_workspace_bytes(B, N, r_per_pair, grad_R != NULL) bytes, 16-byte aligned.
 * Gradients are ADDED into the caller-zeroed outputs, as the other entries do, but no float atomics are used: each CTA
 * stores its partials in its own workspace slots - the weight gradients in slot c (CTA c), dV and dT of pair b in slot
 * c + b, a shared R's gradient per item - and a second kernel adds every output element's partials in increasing slot
 * order, then adds the sum into the output.  Inside a CTA, every input voxel's share of the resampling adjoint is
 * summed in increasing output-voxel order.  The grid is min(B*N, SMs, 160) CTAs, so the bits depend only on the
 * inputs and on min(SMs, 160): two devices with at least 160 SMs, or with the same SM count, give the same bits.
 * The function computed is that of the atomic entries; only the summation order differs (one-item calls run one CTA
 * and give the same bits for everything but grad_vol).  Graph-capturable; allocates nothing. */
AHV_API size_t ahv_score_backward_det_workspace_bytes(int B, int64_t N, int r_per_pair, int want_grad_R);
AHV_API int ahv_score_backward_det(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                                   const float* W1, const float* W2, const float* b2, const float* base,
                                   const float* grad_scores, const void* h1_saved, const float* pair_inv_scale,
                                   float* grad_vol, float* grad_tgt, float* grad_W1, float* grad_W2, float* grad_b2,
                                   float* grad_R, int B, int64_t N, int math_mode, void* workspace, size_t workspace_bytes,
                                   void* stream);

/* infoNCE_loss given the scores (training variant, modules/model.py:43-63 / model_co3d.py:41-61), one launch:
 * positives of pair b = hypotheses whose rotation lies within acc_thr_deg of gt_R[b] (:46-49);
 * loss[b] = -log(sum_pos exp(s/T) / max(sum_all exp(s/T), 1e-8)) (:58-61); grad_scores [B,N] (or NULL) receives
 * d loss[b] / d scores[b,n].  scores [B,N]; R [N,3,3] or [B,N,3,3] (the per-pair sets of :102-103); gt_R [B,3,3]. */
AHV_API int ahv_infonce(const float* scores, const float* R, int r_per_pair, const float* gt_R, float acc_thr_deg,
                        float temperature, float* loss, float* grad_scores, int B, int64_t N, void* stream);

/* Feature_Aligner.forward_3d2d (modules/modules.py:112-124): tri-plane fold,
 * conv1x1 384->32, ReLU, conv1x1 32->32 + bias, L2 normalise over channels.
 * vol [m,16,8,8,8] -> feat [m,32,64].  W1 [32,384], W2 [32,32], b2 [32]
 * (state-dict feature_embedding_2d.{0.weight,2.weight,2.bias}). fp32 FFMA. */
AHV_API int ahv_forward_3d2d(const float* vol, const float* W1, const float* W2, const float* b2,
                     float* feat, int64_t m, void* stream);

/* Bytes of scratch ahv_score / ahv_topk need for (B pairs, N hypotheses, k). */
AHV_API size_t ahv_workspace_bytes(int B, int64_t N, int k);

/* The fused hot path, modules/model.py:186-196 (shared rotation set) and
 * :53-56 / :137-143 (per-pair rotations):
 *   for every pair b and hypothesis n:
 *     scores[b,n] = mean_p < normalize(head(rotate(vol_src[b], R[n]))) , tgt_feat[b] >
 *   then per pair the k best (score desc, ties -> lowest index).
 * vol_src  [B,16,8,8,8] fp32 or bf16 (vol_dtype)
 * tgt_feat [B,32,64] fp32 = ahv_forward_3d2d(vol_tgt)
 * R        [N,3,3] (r_per_pair==0) or [B,N,3,3] (r_per_pair==1)
 * scores   [B,N] or NULL (then they live only in the workspace)
 * topk_val [B,k], topk_idx [B,k] int64 (global index = local + idx_offset) or
 *          both NULL with k==0 to skip selection.
 * 1 <= k <= 32. */
AHV_API int ahv_score(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R,
              int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
              float* scores, float* topk_val, int64_t* topk_idx, int k, int64_t idx_offset, int B,
              int64_t N, int math_mode, void* workspace, size_t workspace_bytes, void* stream);

/* The whole verification step of modules/model.py:186-196 / test_co3d.py:137-146 in one call:
 * target features of vol_tgt [B,16,8,8,8] (fp32), fused scoring of every (pair, hypothesis),
 * selection and sampled_R[pred_index].  With AHV_MATH_TC and k==1 (the reference's torch.max) this
 * is two launches — the target-feature prologue, and the fused scoring kernel (launched programmatically
 * dependent on it; packs the weights and derives the per-pair scales itself) with the arg-max folded
 * into its epilogue and the winners decoded by its last CTA.
 * scores [B,N] or NULL; topk_val/topk_idx [B,k]; R_best [B,k,3,3] or NULL. */
AHV_API int ahv_verify(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                       const float* W1, const float* W2, const float* b2, const float* base, float* scores,
                       float* topk_val, int64_t* topk_idx, float* R_best, int k, int64_t idx_offset, int B,
                       int64_t N, int math_mode, void* workspace, size_t workspace_bytes, void* stream);

/* Two-pass selection in one call (extension, BASELINE config 4 "dense SO(3) grid with top-k refinement pass";
 * the reference stops at torch.max over its random set, test_linemod.py:62-63): ahv_verify over the N
 * rotations keeping the top k (first_val/first_idx [B,k], first_R [B,k,3,3]); ahv_so3_perturb builds m local
 * candidates around every winner (cand [B,k*m,3,3], caller-provided, 16-byte aligned; candidate j*m is winner
 * j itself); ahv_verify over each pair's own k*m candidates keeping the best (best_val [B], best_idx [B] = index
 * into that pair's candidate set, R_best [B,3,3] or NULL).  No host synchronisation, no allocation:
 * CUDA-graph capturable.  k <= min(32, N).  Workspace: ahv_refine_workspace_bytes. */
AHV_API size_t ahv_refine_workspace_bytes(int B, int64_t N, int k, int m);
AHV_API int ahv_refine(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                       const float* W1, const float* W2, const float* b2, const float* base, int k, int m,
                       float max_angle_deg, uint64_t seed, float* first_val, int64_t* first_idx, float* first_R,
                       float* cand, float* best_val, int64_t* best_idx, float* R_best, int B, int64_t N,
                       int math_mode, void* workspace, size_t workspace_bytes, void* stream);

/* Gradient ascent of the AHV_MATH_FP32 score on SO(3) from given rotations (extension; the reference has none):
 * R_init [B,K,3,3] per-pair candidates, tgt_feat [B,32,64] = ahv_forward_3d2d(vol_tgt).  `steps` backtracking steps
 * starting at step_deg; R_out [B,K,3,3], score_out [B,K] = fp32 score of R_out, never below that of R_init.
 * Each step forms a trial exp(theta [u]x) R along the Riemannian gradient direction u (then one Newton step back to
 * SO(3)), keeps it only where it scores higher (theta *= 1.2 there, /= 2 elsewhere), and differentiates the score
 * again only at an accepted trial.  vol_src fp32 or bf16 (AHV_VOL_*; bf16 is staged exactly: the same result as its
 * fp32 copy).  The scores equal ahv_score(AHV_MATH_FP32) of R_out bit for bit, and the result is bit-deterministic.
 * 0 <= steps <= 1000, step_deg finite and > 0; R_init / R_out 16-byte aligned.
 * One launch, no host synchronisation, no allocation: CUDA-graph capturable. */
AHV_API int ahv_gradient_ascent(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R_init,
                                const float* W1, const float* W2, const float* b2, const float* base, int steps,
                                float step_deg, float* R_out, float* score_out, int B, int K, void* stream);

/* Grid -> top-k -> gradient ascent -> per-pair arg-max in one call (config 4's accurate path), like ahv_refine:
 * ahv_verify(math_mode) keeps the top k (first_val/idx/R); ahv_gradient_ascent from first_R (R_all [B,k,3,3],
 * score_all [B,k]); best_val [B], best_idx [B] (index into k, ties -> lowest), R_best [B,3,3] or NULL.
 * k <= min(32, N); rotation buffers 16-byte aligned.  Workspace: ahv_refine_gradient_workspace_bytes.
 * No host synchronisation, no allocation: CUDA-graph capturable. */
AHV_API size_t ahv_refine_gradient_workspace_bytes(int B, int64_t N, int k);
AHV_API int ahv_refine_gradient(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                                const float* W1, const float* W2, const float* b2, const float* base, int k, int steps,
                                float step_deg, float* first_val, int64_t* first_idx, float* first_R, float* R_all,
                                float* score_all, float* best_val, int64_t* best_idx, float* R_best, int B, int64_t N,
                                int math_mode, void* workspace, size_t workspace_bytes, void* stream);

/* ahv_refine_gradient that ascends from k DISTINCT basins (extension): the grid pass scores the whole set (target
 * features, then ahv_score with k = 0; no fused arg-max, whose scores are never written) and keeps the k winners of
 * ahv_topk_distinct(min_sep_deg) in first_val/idx/R.  Slots left empty there (fewer than k rotations pairwise more than
 * min_sep_deg apart) are not ascended: R_all NaN, score_all -inf, so the arg-max never picks one.  0 <= min_sep_deg
 * <= 180; with min_sep_deg == 0 every output equals ahv_refine_gradient's bit for bit.  Every other argument, rule and
 * the workspace (ahv_refine_gradient_workspace_bytes) are ahv_refine_gradient's. */
AHV_API int ahv_refine_gradient_distinct(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                                         int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
                                         int k, int steps, float step_deg, float min_sep_deg, float* first_val,
                                         int64_t* first_idx, float* first_R, float* R_all, float* score_all, float* best_val,
                                         int64_t* best_idx, float* R_best, int B, int64_t N, int math_mode, void* workspace,
                                         size_t workspace_bytes, void* stream);

/* Top-k of distinct rotations (extension): greedy geodesic non-maximum suppression on SO(3) over the score-sorted
 * hypotheses of each pair.  With key(n) = ahv_topk's order (score descending, ties -> lowest index, NaN as ahv_topk
 * orders it), t(a,b) = trace(R_a R_b^T) in fp32 (nine individually rounded products summed left to right, no FMA) and
 * c = fp32(1 + 2 cos(min_sep_deg * pi / 180)) evaluated in double:
 *   w_0 = the largest key;  w_j = the largest key(n) < key(w_{j-1}) with t(n, w_i) < c for every i < j,
 * stopping at k winners or when none qualifies; the later slots are empty (value -inf, index -1, rotation NaN).
 * min_sep_deg == 0 suppresses nothing (the result is ahv_topk's bit for bit); min_sep_deg == 180 keeps the top-1 alone.
 * scores [B,N]; R [N,3,3] (r_per_pair == 0) or [B,N,3,3]; topk_val [B,k], topk_idx [B,k] int64, R_best [B,k,3,3] or
 * NULL.  1 <= k <= 32, 0 <= min_sep_deg <= 180, N <= 2^31 - 1; R and R_best 16-byte aligned.  One launch (a cluster of
 * 8 CTAs per pair), no workspace, no allocation, no host synchronisation: deterministic and CUDA-graph capturable. */
AHV_API int ahv_topk_distinct(const float* scores, const float* R, int r_per_pair, int B, int64_t N, int k,
                              float min_sep_deg, float* topk_val, int64_t* topk_idx, float* R_best, void* stream);

/* torch.max / top-k over an existing score matrix (modules/model.py:195). */
AHV_API int ahv_topk(const float* scores, int B, int64_t N, int k, int64_t idx_offset, float* topk_val,
             int64_t* topk_idx, void* workspace, size_t workspace_bytes, void* stream);

/* Merge `parts` per-shard top-k lists (layout [parts,B,k], e.g. the result of
 * an NCCL all-gather over hypothesis shards) into one [B,k] list with the same
 * ordering rule, so every rank obtains bit-identical results. */
AHV_API int ahv_topk_merge(const float* vals, const int64_t* idx, int parts, int B, int k, float* out_val,
                   int64_t* out_idx, void* stream);

/* sampled_R[pred_index] (modules/model.py:196): R_out[b,j] = R[idx[b,j]-idx_offset]. */
AHV_API int ahv_gather_rotations(const float* R, int r_per_pair, const int64_t* idx, int64_t idx_offset,
                         int B, int64_t N, int k, float* R_out, void* stream);

/* Hypothesis set sharded over the GPUs of one NVSwitch node (SURVEY.md §8e; the reference is single GPU,
 * batch 1, test_co3d.py:133).  Every rank scores ITS slice of the rotation set (global index = local +
 * idx_offset) for all pairs; the per-shard winners are exchanged through NVLink peer memory by the kernels
 * themselves, so the step contains no NCCL call, no merge launch and no winner gather, is identical on every
 * rank bit for bit (score descending, ties -> lowest global index) and CUDA-graph capturable.
 *
 * Exchange buffers: one per rank, ahv_peer_alloc(max_pairs, max_k) (a zeroed cudaMalloc whose header records
 * the capacity; the entry stride depends on the capacity only, so calls with different B and k may follow one
 * another on one buffer); ahv_peer_export -> 64-byte CUDA IPC handle to send to the peers, ahv_peer_open on
 * their side; ahv_peer_close / ahv_peer_free to release.  peers[r] = rank r's buffer as mapped in this process
 * (peers[rank] = own); peer_max_pairs / peer_max_k = the capacity all buffers were allocated with (calls with
 * B > peer_max_pairs or k > peer_max_k are rejected with AHV_EINVAL).  Every rank must make the same sequence
 * of exchanging calls.  A peer that never reaches a step is waited for ~20 s (device clock); that step then
 * returns NaN scores, index -1 and NaN rotations, and ahv_peer_status reports it.
 *
 * ahv_verify_sharded = ahv_verify on this rank's slice + the exchange: topk_val/topk_idx [B,k], R_best
 * [B,k,3,3] (or NULL) are the result over the WHOLE set.  With k == 1 and tensor-core arithmetic the scoring
 * kernel's last CTA performs the exchange itself (two launches per step, as on one GPU); otherwise the
 * shard's top-k is followed by one exchange kernel (ahv_topk_exchange, also callable on its own: val/idx [B,k]
 * = this shard's list with global indices, -1 = empty slot; R = this shard's rotations).  An empty slice
 * (N == 0) is allowed when world > 1.  idx_offset + N must not exceed 2^32. */
AHV_API size_t ahv_peer_bytes(int max_pairs, int max_k);
AHV_API int ahv_peer_alloc(int max_pairs, int max_k, void** ptr);
AHV_API int ahv_peer_free(void* ptr);
AHV_API int ahv_peer_export(void* ptr, unsigned char* handle64);
AHV_API int ahv_peer_open(const unsigned char* handle64, void** ptr);
AHV_API int ahv_peer_close(void* ptr);
/* Synchronising read of this rank's exchange header: exchanges completed, and whether one of them timed out
 * waiting for a peer. */
AHV_API int ahv_peer_status(const void* own, unsigned* exchanges_done, unsigned* timed_out);
/* Synchronising read of the capacity recorded in a (own or mapped) exchange buffer. */
AHV_API int ahv_peer_capacity(const void* buf, int* max_pairs, int* max_k);
AHV_API int ahv_topk_exchange(const float* val, const int64_t* idx, const float* R, int r_per_pair, int64_t idx_offset,
                              int64_t N, int B, int k, float* out_val, int64_t* out_idx, float* R_best, int rank,
                              int world, void* const* peers, int peer_max_pairs, int peer_max_k, void* stream);
AHV_API int ahv_verify_sharded(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                               const float* W1, const float* W2, const float* b2, const float* base, float* topk_val,
                               int64_t* topk_idx, float* R_best, int k, int64_t idx_offset, int B, int64_t N,
                               int math_mode, void* workspace, size_t workspace_bytes, int rank, int world,
                               void* const* peers, int peer_max_pairs, int peer_max_k, void* stream);

/* Entries taking HOST buffers (pageable or pinned) - what a non-PyTorch host (ctypes / cgo / JNI) binds: copy
 * the inputs to the device, run the whole verification step (ahv_verify, or ahv_verify_sharded when world > 1)
 * and copy the selection back; `stream` is synchronised before returning.  vol_tgt_host [B,16,8,8,8] fp32;
 * R_host as R above; outputs as above (scores_host may be NULL and must be NULL when world > 1).
 *
 * ahv_predict_host_ex takes fp32 or bf16 source volumes (vol_dtype), an index offset and the sharding
 * arguments of ahv_verify_sharded (world == 1: peers may be NULL), and keeps its device scratch in a
 * caller-owned session (ahv_host_session_create on the current device; grown on demand, reused across calls,
 * one call at a time per session).  ahv_predict_host is the one-shot form: fp32, one GPU, a temporary session
 * per call.  Neither touches process-global state. */
typedef struct ahv_host_session ahv_host_session;
AHV_API int ahv_host_session_create(ahv_host_session** session);
AHV_API int ahv_host_session_destroy(ahv_host_session* session);
AHV_API int ahv_predict_host_ex(ahv_host_session* session, const void* vol_src_host, int vol_dtype,
                                const float* vol_tgt_host, const float* R_host, int r_per_pair, const float* W1_host,
                                const float* W2_host, const float* b2_host, const float* base_host, float* scores_host,
                                float* topk_val_host, int64_t* topk_idx_host, float* R_best_host, int k,
                                int64_t idx_offset, int B, int64_t N, int math_mode, int rank, int world,
                                void* const* peers, int peer_max_pairs, int peer_max_k, void* stream);
AHV_API int ahv_predict_host(const float* vol_src_host, const float* vol_tgt_host, const float* R_host,
                     int r_per_pair, const float* W1_host, const float* W2_host,
                     const float* b2_host, const float* base_host, float* scores_host,
                     float* topk_val_host, int64_t* topk_idx_host, float* R_best_host, int k, int B,
                     int64_t N, int math_mode, void* stream);

/* Diagnostic: conflict-free LDS.128 streaming read on `ctas` CTAs of 1024
 * threads (2 per SM); `*bytes` receives the shared-memory bytes read.  bench.py
 * times it to obtain the measured shared-memory peak the gather roofline uses. */
AHV_API int ahv_diag_smem_read(float* out, int ctas, int iters, unsigned long long* bytes,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AHV_B200_H_ */
