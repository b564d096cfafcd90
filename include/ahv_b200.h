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

/* Nested, equal-volume SO(3) grid (extension): the Hopf fibration, HEALPix on S^2 in NESTED order times a regular
 * grid on S^1 (Yershova et al. 2010).  Level L (0 <= L <= 16): Nside = 2^L, 12*4^L pixels p, 6*2^L psi-intervals j
 * with centres psi_j = 2*pi*(j + 1/2)/(6*2^L), 72*8^L cells of equal Haar volume.  Cell index i = 6*p0 + j0 at level
 * 0; the children of cell i at level L + 1 are 8i + 2a + b (a: the HEALPix nested child digit, p' = 4p + a; b: the
 * psi digit, j' = 2j + b), and lie inside it.  Point: (theta, phi) = HEALPix nested pix2ang(Nside, p) and
 * q = (cos(theta/2)cos(psi/2), cos(theta/2)sin(psi/2), sin(theta/2)cos(phi+psi/2), sin(theta/2)sin(phi+psi/2)),
 * evaluated in fp64, rounded once to fp32, then ahv_so3_from_normals' quaternion -> matrix map.
 * ahv_so3_hopf_grid: cells [first_index, first_index + count) of `level` as rotation matrices R [count,3,3]. */
AHV_API int ahv_so3_hopf_grid(int level, int64_t first_index, float* R, int64_t count, void* stream);
/* For each of the n cells parent_idx[i] of `level` (0 <= level < 16), its 8 children at level + 1 in child order:
 * child_idx [n,8] (= 8*parent_idx[i] + c) and R_child [n,8,3,3], bit-identical to ahv_so3_hopf_grid(level + 1) at
 * those indices.  A parent index outside [0, 72*8^level) gives children -1 with NaN rotations. */
AHV_API int ahv_so3_hopf_children(int level, const int64_t* parent_idx, int64_t n, int64_t* child_idx, float* R_child,
                                  void* stream);

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
 * Screened form: with fp32 volumes, AHV_MATH_TC, k == 1, scores == NULL and B*N >= 2^18 (and N >= about 37 000, so
 * that its lists fit the workspace ahv_workspace_bytes sizes) the step is seven launches: the 16-bit gather
 * (AHV_MATH_TC_F16GATHER's kernel, 1.6x the fp32 gather's rate) scores every hypothesis; per pair, the hypotheses
 * within 2 tau (tau = 2e-3 in score units) of its best 16-bit score, at most 224, and 32 strided probes are re-scored by
 * the fp32 gather; a pair whose realised |fp32 - 16-bit| difference on that list exceeds tau / 4, or which has more
 * than 224 contenders, is scored again in full by the fp32 gather (the number of such pairs is read on the device:
 * no host synchronisation, CUDA-graph capturable).  The result equals the single pass's bit for bit whenever every
 * hypothesis's 16-bit score lies within tau of its fp32 score; that is checked on every call on each pair's list,
 * with the per-pair fallback behind it - a checked margin, not a proof.  Every other call is the single pass.
 * scores [B,N] or NULL; topk_val/topk_idx [B,k]; R_best [B,k,3,3] or NULL. */
AHV_API int ahv_verify(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                       const float* W1, const float* W2, const float* b2, const float* base, float* scores,
                       float* topk_val, int64_t* topk_idx, float* R_best, int k, int64_t idx_offset, int B,
                       int64_t N, int math_mode, void* workspace, size_t workspace_bytes, void* stream);

/* Diagnostics of the screened form of ahv_verify (and ahv_verify_sharded, per rank with the rank's N): *is_screened =
 * whether a call with (B, N), fp32 volumes, AHV_MATH_TC, k == 1 and no scores takes it.  If so and any of the other
 * outputs is set, reads what the last such call over `workspace` left there (synchronising copies):
 * flagged_pairs = pairs scored again in full, contenders [B] = hypotheses within 2 tau of each pair's best 16-bit
 * score (more than 224: overflow), max_err [B] = the largest |fp32 - 16-bit| score difference on each pair's list. */
AHV_API int ahv_verify_screen_stats(const void* workspace, int B, int64_t N, int* is_screened, int* flagged_pairs,
                                    int* contenders, float* max_err);

/* Two-pass selection in one call (extension, BASELINE config 4 "dense SO(3) grid with top-k refinement pass";
 * the reference stops at torch.max over its random set, test_linemod.py:62-63): ahv_verify over the N
 * rotations keeping the top k (first_val/first_idx [B,k], first_R [B,k,3,3]); ahv_so3_perturb builds m local
 * candidates around every winner (cand [B,k*m,3,3], caller-provided, 16-byte aligned; candidate j*m is winner
 * j itself); ahv_verify over each pair's own k*m candidates keeping the best (best_val [B], best_idx [B] = index
 * into that pair's candidate set, R_best [B,3,3] or NULL).  No host synchronisation, no allocation:
 * CUDA-graph capturable.  k <= min(32, N), 0 <= max_angle_deg <= 180: every argument, max_angle_deg included, is
 * checked before the first pass is enqueued, so a rejected call writes nothing.  Workspace: ahv_refine_workspace_bytes. */
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

/* Coarse-to-fine search on the nested Hopf grid (extension; see ahv_so3_hopf_grid), one call:
 *   target features once (ahv_forward_3d2d); the whole grid of base_level (72*8^base_level cells, shared by the B
 *   pairs) is generated into the workspace and scored with ahv_score(math_mode), its top-k in first_val [B,k],
 *   first_idx [B,k] (grid indices of base_level) and first_R [B,k,3,3];
 *   then `levels` times: the 8 children of each pair's k cells, the cells taken in ascending index order, form a
 *   per-pair set [B,8k] (ascending grid indices of the next level), scored with ahv_score(math_mode) and cut to its
 *   top-k, whose cells are the next parents.
 * val [B,k], idx [B,k] (grid indices of level base_level + levels) and R_out [B,k,3,3] (= ahv_so3_hopf_grid of that
 * level at idx) are the top-k of the finest level, in ahv_topk's order: slot 0 is the answer, ties go to the lowest
 * index.  levels = 0 gives the base level's top-k.  0 <= base_level <= 6, base_level + levels <= 16, 1 <= k <= 32,
 * B >= 1; every buffer required, rotation buffers, volumes, W1, W2 and the workspace 16-byte aligned.  Workspace:
 * ahv_search_hierarchical_workspace_bytes(B, base_level, k) (0 for invalid sizes), which holds the base grid
 * (36 B * 72*8^base_level).  No allocation, no host synchronisation: CUDA-graph capturable. */
AHV_API size_t ahv_search_hierarchical_workspace_bytes(int B, int base_level, int k);
AHV_API int ahv_search_hierarchical(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* W1, const float* W2,
                                    const float* b2, const float* base, int base_level, int levels, int k, float* first_val,
                                    int64_t* first_idx, float* first_R, float* val, int64_t* idx, float* R_out, int B,
                                    int math_mode, void* workspace, size_t workspace_bytes, void* stream);

/* Coarse-to-fine search that keeps k DISTINCT modes (extension), one call.  ahv_search_hierarchical keeps the global
 * top-k of every level, whose cells can crowd around one peak; this search descends each mode with a beam of its own:
 *   target features once; the whole base_level grid (72*8^base_level cells) generated into the workspace and scored
 *   with ahv_score(k = 0, math_mode), giving S0 [B,n0];
 *   modes: first_val [B,k], first_idx [B,k], first_R [B,k,3,3] = ahv_topk_distinct(S0, grid, k, min_sep_deg) bit for bit
 *   (empty slots -inf / -1 / NaN);
 *   slots: base cell n goes to slot j when n = first_idx[j], else to the lowest non-empty slot j with
 *   t(n, first_R[j]) >= c (t and c are ahv_topk_distinct's, the rule of ahv_posterior_mass), so slot j holds its winner
 *   and the cells that winner suppressed; cells of no slot are dropped;
 *   beams: slot j's beam is the top-`beam` cells of the slot in ahv_topk's key order (the winner first), kept in
 *   ascending grid index and padded with -1 at the end;
 *   each of `levels` levels: the 8 children of every beam cell form a per-pair set [B, 8*k*beam], slot-major (slot j's
 *   children are the segment [8*beam*j, 8*beam*(j+1)), ascending in grid index), scored with ahv_score(k = 0,
 *   math_mode); a child inherits its parent's slot, the children of a -1 pad never qualify, and slot j's next beam is
 *   the top-`beam` of its segment (ties to the lowest grid index).
 * val [B,k], idx [B,k] (grid indices of level base_level + levels) and R_out [B,k,3,3] (= ahv_so3_hopf_grid of that level
 * at idx) are the best cell of each final beam, ordered by key (score descending, ties to the lower index; slot 0 is the
 * answer), empty modes last as -inf / -1 / NaN.  The final modes are not suppressed again: two may lie close together.
 * levels = 0 gives first_* bit for bit.  Each pair scores 72*8^base_level + levels*8*k*beam hypotheses.
 * Rules: ahv_search_hierarchical's (0 <= base_level <= 6, base_level + levels <= 16, 1 <= k <= 32, B >= 1, every buffer
 * required, rotation buffers, volumes, W1, W2 and the workspace 16-byte aligned), plus 1 <= beam <= 8 and a finite
 * 0 < min_sep_deg <= 180.  Workspace: ahv_search_modes_workspace_bytes(B, base_level, k, beam) (0 for invalid sizes),
 * which holds the base grid and one slot byte per base cell and pair.  No allocation, no host synchronisation: CUDA-graph
 * capturable. */
AHV_API size_t ahv_search_modes_workspace_bytes(int B, int base_level, int k, int beam);
AHV_API int ahv_search_modes(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* W1, const float* W2,
                             const float* b2, const float* base, int base_level, int levels, int k, int beam, float min_sep_deg,
                             float* first_val, int64_t* first_idx, float* first_R, float* val, int64_t* idx, float* R_out, int B,
                             int math_mode, void* workspace, size_t workspace_bytes, void* stream);

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

/* Posterior mass of selected rotations (extension): the verification scores are trained as the logits of a
 * distribution over SO(3) (InfoNCE, modules/model.py:43-63), p_b(n) = exp(s[b,n]/T) / Z_b.  With m = max_n s[b,n]:
 *   log_z[b]  = m/T + log sum_n exp((s[b,n] - m)/T)
 *   mass[b,j] = sum_{n -> j} exp((s[b,n] - m)/T) / sum_n exp((s[b,n] - m)/T)
 * where hypothesis n goes to the LOWEST slot j with t(n, c_j) >= c: t and c = fp32(1 + 2 cos(radius_deg * pi / 180))
 * are ahv_topk_distinct's (radius_deg == 180: every rotation qualifies).  With centers = ahv_topk_distinct's R_best and
 * radius_deg = its min_sep_deg, slot j's mass is its winner plus exactly the hypotheses that winner suppressed;
 * 1 - sum_j mass[b,j] is the mass no slot holds.  scores [B,N]; R [N,3,3] (r_per_pair == 0) or [B,N,3,3]; centers
 * [B,k,3,3], a NaN centre being an empty slot (mass 0); log_z [B], mass [B,k].  0 <= k <= 32 (k == 0: centers and
 * mass NULL, log_z alone), 1 <= N <= 2^31 - 1, 0 <= radius_deg <= 180, temperature finite and > 0; R, centers and the
 * workspace 16-byte aligned.  A -inf score contributes 0; a pair with a NaN or +inf score gets NaN outputs; a pair whose
 * scores are all -inf gets log_z = -inf and NaN masses.  Sums run in double in a fixed order and are cast to fp32
 * once: the bits depend on the inputs alone (not on B, the pair's place in the batch or the SM count).  Two launches,
 * workspace ahv_posterior_mass_workspace_bytes(B, N, k) (~B * ceil(N/2048) * (k+1) * 8 bytes), no allocation, no host
 * synchronisation: CUDA-graph capturable. */
AHV_API size_t ahv_posterior_mass_workspace_bytes(int B, int64_t N, int k);
AHV_API int ahv_posterior_mass(const float* scores, const float* R, int r_per_pair, const float* centers, int B, int64_t N,
                               int k, float radius_deg, float temperature, float* log_z, float* mass, void* workspace,
                               size_t workspace_bytes, void* stream);

/* First moment of the posterior over each slot (extension): where inside each selected mode the probability sits, and
 * how wide the mode is.  Slots, temperature, value rules and summation order are ahv_posterior_mass's; with
 * e_n = exp((s[b,n] - m)/T) and W_j = sum_{n -> j} e_n (the sum mass[b,j] is formed from):
 *   moment[b,j]   = M_j = sum_{n -> j} e_n R_n / W_j                       (3x3, row-major)
 *   mean_R[b,j]   = argmax_{R in SO(3)} tr(R^T M_j), a proper rotation (det +1); any maximiser where it is not unique
 *   mean_cos[b,j] = (tr(mean_R^T M_j) - 1) / 2 = E_j[cos theta(R_n, mean_R)], clamped to [-1, 1] (the hypotheses'
 *                   fp32 matrices are orthonormal only to rounding); arccos(mean_cos) is close to the RMS angle to
 *                   mean_R when the mode is concentrated
 *   log_z, mass   = bit for bit ahv_posterior_mass's on the same arguments.
 * A pair with a NaN or +inf score gets NaN everywhere.  A slot with W_j == 0 in double gets NaN moment, mean_R and
 * mean_cos: an empty (NaN) centre, a slot whose scores are all -inf, or exp((s - m)/T) underflowing, i.e.
 * (m - s)/T > ~745 for every hypothesis of the slot (with scores in [-1, 1] that needs T < 2.7e-3).  Sums run in
 * double: each thread's hypotheses in index order, the warp butterfly, the warps in order, the chunks of 2048 in a
 * fixed order; M_j is projected in double (q-method, cyclic Jacobi) and every output is cast to fp32 once, so
 * the bits depend on the pair's inputs alone (not on B, the pair's place in the batch or the SM count).  Arguments as
 * ahv_posterior_mass, except 1 <= k <= 32 and every output required for B > 0: mean_R and moment [B,k,3,3], mean_cos
 * [B,k].  Two launches, workspace ahv_posterior_moments_workspace_bytes(B, N, k) (the mass's plus
 * B * ceil(N/2048) * k * 72 bytes), no allocation, no host synchronisation: CUDA-graph capturable. */
AHV_API size_t ahv_posterior_moments_workspace_bytes(int B, int64_t N, int k);
AHV_API int ahv_posterior_moments(const float* scores, const float* R, int r_per_pair, const float* centers, int B,
                                  int64_t N, int k, float radius_deg, float temperature, float* log_z, float* mass,
                                  float* mean_R, float* mean_cos, float* moment, void* workspace,
                                  size_t workspace_bytes, void* stream);

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

/* Exchange buffers with a score region (extension): ahv_peer_alloc_ex(max_pairs, max_k, max_hyps) adds
 * 2 x max_pairs x max_hyps fp32 after the entries, for ahv_scores_exchange of up to max_pairs x max_hyps scores;
 * max_hyps == 0 is ahv_peer_alloc (same size, same layout), 0 <= max_hyps <= 2^31 - 1.  ahv_peer_bytes_ex gives the
 * size (0 for invalid capacities), ahv_peer_capacity_ex reads all three capacities back (synchronising).  A buffer
 * of either kind serves every other exchanging entry, with the same sequence counter. */
AHV_API size_t ahv_peer_bytes_ex(int max_pairs, int max_k, int64_t max_hyps);
AHV_API int ahv_peer_alloc_ex(int max_pairs, int max_k, int64_t max_hyps, void** ptr);
AHV_API int ahv_peer_capacity_ex(const void* buf, int* max_pairs, int* max_k, int64_t* max_hyps);

/* All-gather of a score matrix sliced by hypothesis, through the score region (extension): part [B, hi-lo] fp32 =
 * columns [lo, hi) of [B,N], where lo = min(N, rank*ceil(N/world)) and hi = min(N, lo + ceil(N/world)) (the
 * partition of dist.shard_bounds; part may be NULL when the slice is empty); scores [B,N] receives the whole matrix,
 * the same on every rank.  B <= peer_max_pairs, 1 <= N <= peer_max_hyps (the buffers' ahv_peer_alloc_ex capacity),
 * world >= 2.  Two launches: a grid that stores the slice into every rank's region, whose last CTA alone announces
 * the exchange and waits for the peers, then a copy into `scores`.  A peer that never arrives gives NaN scores after
 * ~20 s, as for the other exchanges.  No host synchronisation, no allocation: CUDA-graph capturable. */
AHV_API int ahv_scores_exchange(const float* part, int B, int64_t N, float* scores, int rank, int world, void* const* peers,
                                int peer_max_pairs, int peer_max_k, int64_t peer_max_hyps, void* stream);

/* ahv_refine_gradient_distinct over a hypothesis set sharded across the GPUs of one node (extension).  Every rank
 * passes the WHOLE rotation set R (and the same volumes and arguments) and receives the whole-set result: every
 * output equals ahv_refine_gradient_distinct's on one GPU over the same set, bit for bit, on every rank.  Rank r
 * scores hypotheses [lo, hi) (the partition of ahv_scores_exchange).
 *   min_sep_deg == 0: the slice's top-k, merged over the ranks by the top-k exchange (ahv_verify_sharded).
 *   min_sep_deg > 0:  the slice's scores, all-gathered by ahv_scores_exchange, then ahv_topk_distinct over the
 *                     whole [B,N] and R on EVERY rank.  This selection is replicated, not sharded: greedy
 *                     suppression does not compose from per-shard lists (a rotation that wins on its shard may
 *                     suppress a neighbour and then lose to another shard's winner, and the neighbour it suppressed
 *                     belonged to the global answer).  Needs N <= peer_max_hyps.
 * The rank then ascends items [ilo, ihi) of the B*k (pair, slot) items, the same partition over B*k (k < world and
 * ranks with no item are fine), and one exchange gives every rank every ascended slot; the per-pair arg-max and its
 * rotation are computed on every rank.  Empty distinct slots: R_all NaN, score_all -inf, as on one GPU.
 * k <= min(32, N), B <= peer_max_pairs, k <= peer_max_k; every rank must make the same call.  world == 1 is
 * ahv_refine_gradient(_distinct) (peers may be NULL).  Two exchanges per call for world > 1.  Workspace:
 * ahv_refine_gradient_sharded_workspace_bytes(B, N, k, world).  No host synchronisation, no allocation: CUDA-graph
 * capturable. */
AHV_API size_t ahv_refine_gradient_sharded_workspace_bytes(int B, int64_t N, int k, int world);
AHV_API int ahv_refine_gradient_sharded(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                                        int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
                                        int k, int steps, float step_deg, float min_sep_deg, float* first_val,
                                        int64_t* first_idx, float* first_R, float* R_all, float* score_all, float* best_val,
                                        int64_t* best_idx, float* R_best, int B, int64_t N, int math_mode, void* workspace,
                                        size_t workspace_bytes, int rank, int world, void* const* peers, int peer_max_pairs,
                                        int peer_max_k, int64_t peer_max_hyps, void* stream);

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
