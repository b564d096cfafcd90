// extern "C" surface of lib3dahv_b200 (see include/ahv_b200.h for the contract
// and the reference interface each entry replaces).
#include <cmath>
#include <cstring>
#include <new>

#include "ahv_peer.cuh"

using namespace ahv;

namespace {

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
template <class... P> bool all_aligned16(P... p) { return (aligned16(p) && ...); }
template <class... P> bool all_set(P... p) { return (... && (p != nullptr)); }

// Argument rules shared by the entries (each entry keeps its own order of checks).
bool vol_dtype_ok(int vol_dtype) { return vol_dtype == AHV_VOL_F32 || vol_dtype == AHV_VOL_BF16; }
bool math_mode_ok(int m) { return m == AHV_MATH_TC || m == AHV_MATH_FP32 || m == AHV_MATH_TC_F16GATHER; }
bool n_ok(int64_t N) { return N >= 0 && N <= 0x7fffffffLL; }  // hypotheses per pair: 31-bit indices
bool k_ok(int k) { return k >= 1 && k <= kMaxK; }

// The library contains sm_100a code only; refuse anything else loudly.
int check_device() {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return AHV_ECUDA;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
    return AHV_ECUDA;
  return major == 10 ? AHV_OK : AHV_ENOTSUP;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Workspace layouts: the offset of each region (each 256-byte aligned) and the size of the whole.
// The verification workspace: [scores B*N fp32 | top-k partials | tensor-core scratch | per-shard top-k lists].
// ahv_score needs the bytes up to `lists` only.
struct VerifyWs {
  size_t topk, tc, lists, total;
  VerifyWs(int B, int64_t N, int k)
      : topk(align_up((size_t)B * (size_t)N * sizeof(float), 256)),
        tc(topk + align_up(topk_workspace_bytes(B, N, k), 256)),
        lists(tc + align_up(score_tc_workspace_bytes(B, N), 256)),
        total(lists + align_up((size_t)B * (size_t)(k > 0 ? k : 1) * (sizeof(float) + sizeof(int64_t)), 256)) {}
};

// ahv_refine: [the grid pass's verification workspace | the candidate pass's ([B, k*m], arg-max)]
struct RefineWs {
  size_t cand, total;
  RefineWs(int B, int64_t N, int k, int m)
      : cand(VerifyWs(B, N, k).total), total(cand + VerifyWs(B, (int64_t)k * m, 1).total) {}
};

// ahv_refine_gradient: [the grid pass's verification workspace | target features B*32*64 fp32 | top-k partials over [B,k]]
struct RefineGradientWs {
  size_t tgt, top, total;
  RefineGradientWs(int B, int64_t N, int k)
      : tgt(VerifyWs(B, N, k).total),
        top(tgt + align_up((size_t)B * kO * kP * sizeof(float), 256)),
        total(top + align_up(topk_workspace_bytes(B, k, 1), 256)) {}
};

}  // namespace

extern "C" {

AHV_API int ahv_version(void) { return AHV_VERSION; }

AHV_API const char* ahv_status_string(int status) {
  switch (status) {
    case AHV_OK: return "ok";
    case AHV_EINVAL: return "invalid argument (shape, null or misaligned pointer, enum)";
    case AHV_ENOTSUP: return "unsupported device: lib3dahv_b200 holds sm_100a code only, no fallback";
    case AHV_ECUDA: return "CUDA runtime error (see cudaGetLastError)";
    case AHV_EWORKSPACE: return "workspace too small (see ahv_workspace_bytes)";
    default: return "unknown status";
  }
}

AHV_API int ahv_so3_from_normals(const float* normals, float* R, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!normals || !R)) || !aligned16(normals)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_so3_from_normals(normals, R, n, (cudaStream_t)stream);
}

AHV_API int ahv_so3_sample(uint64_t seed, int64_t first_index, float* R, int64_t n, void* stream) {
  if (n < 0 || first_index < 0 || (n > 0 && !R)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_so3_sample(seed, first_index, R, n, (cudaStream_t)stream);
}

AHV_API int ahv_so3_grid(int64_t n_total, int64_t first_index, float* R, int64_t count, void* stream) {
  if (n_total < 1 || first_index < 0 || count < 0 || first_index + count > n_total || (count > 0 && !R))
    return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_so3_grid(n_total, first_index, R, count, (cudaStream_t)stream);
}

AHV_API int ahv_so3_perturb(const float* R_center, int64_t n, int m, float max_angle_deg, uint64_t seed, float* R_out,
                            void* stream) {
  if (n < 0 || m < 1 || !(max_angle_deg >= 0.0f) || max_angle_deg > 180.0f || (n > 0 && (!R_center || !R_out))) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_so3_perturb(R_center, n, m, max_angle_deg, seed, R_out, (cudaStream_t)stream);
}

AHV_API int ahv_rotate_volume(const float* vol, int vol_per_rotation, const float* R, const float* base,
                      float* out, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!vol || !R || !base || !out))) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_rotate_volume(vol, vol_per_rotation != 0, R, base, out, n, (cudaStream_t)stream);
}

AHV_API int ahv_rotate_volume_backward(const float* grad_out, int vol_per_rotation, const float* R,
                                       const float* base, float* grad_vol, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!grad_out || !R || !base || !grad_vol))) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_rotate_volume_bwd(grad_out, vol_per_rotation != 0, R, base, grad_vol, n, (cudaStream_t)stream);
}

AHV_API int ahv_score_backward(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                               const float* W1, const float* W2, const float* b2, const float* base,
                               const float* grad_scores, float* grad_vol, float* grad_tgt, float* grad_W1,
                               float* grad_W2, float* grad_b2, int B, int64_t N, void* stream) {
  if (B < 0 || !n_ok(N)) return AHV_EINVAL;
  if ((int64_t)B * N > 0 &&
      !all_set(vol_src, tgt_feat, R, W1, W2, b2, base, grad_scores, grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2))
    return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_score_bwd(vol_src, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, grad_scores, grad_vol, grad_tgt,
                          grad_W1, grad_W2, grad_b2, B, N, (cudaStream_t)stream);
}

AHV_API int ahv_rotate_volume_grad_R(const float* vol, int vol_per_rotation, const float* R, const float* base,
                                     const float* grad_out, float* grad_R, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!vol || !R || !base || !grad_out || !grad_R))) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_rotate_volume_grad_R(vol, vol_per_rotation != 0, R, base, grad_out, grad_R, n, (cudaStream_t)stream);
}

AHV_API int ahv_score_backward_ex(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                                  const float* W1, const float* W2, const float* b2, const float* base,
                                  const float* grad_scores, const void* h1_saved, const float* pair_inv_scale,
                                  float* grad_vol, float* grad_tgt, float* grad_W1, float* grad_W2, float* grad_b2,
                                  float* grad_R, int B, int64_t N, void* stream) {
  if (B < 0 || !n_ok(N)) return AHV_EINVAL;
  if (!grad_vol && !grad_tgt && !grad_W1 && !grad_W2 && !grad_b2 && !grad_R) return AHV_EINVAL;
  if (!h1_saved != !pair_inv_scale || !aligned16(h1_saved)) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && !all_set(vol_src, tgt_feat, R, W1, W2, b2, base, grad_scores)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_score_bwd(vol_src, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, grad_scores, grad_vol, grad_tgt,
                          grad_W1, grad_W2, grad_b2, B, N, (cudaStream_t)stream, h1_saved, pair_inv_scale, grad_R);
}

AHV_API size_t ahv_score_backward_det_workspace_bytes(int B, int64_t N, int r_per_pair, int want_grad_R) {
  if (B < 0 || !n_ok(N)) return 0;
  return DetBwdWs(B, N, want_grad_R && !r_per_pair).total * sizeof(float);
}

AHV_API int ahv_score_backward_det(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                                   const float* W1, const float* W2, const float* b2, const float* base,
                                   const float* grad_scores, const void* h1_saved, const float* pair_inv_scale,
                                   float* grad_vol, float* grad_tgt, float* grad_W1, float* grad_W2, float* grad_b2,
                                   float* grad_R, int B, int64_t N, int math_mode, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (B < 0 || !n_ok(N)) return AHV_EINVAL;
  if (math_mode != AHV_MATH_TC && math_mode != AHV_MATH_FP32) return AHV_EINVAL;
  if (!grad_vol && !grad_tgt && !grad_W1 && !grad_W2 && !grad_b2 && !grad_R) return AHV_EINVAL;
  if (math_mode == AHV_MATH_TC && (grad_R || !all_set(grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2))) return AHV_EINVAL;
  if (!h1_saved != !pair_inv_scale) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && !all_set(vol_src, tgt_feat, R, W1, W2, b2, base, grad_scores)) return AHV_EINVAL;
  if (!all_aligned16(vol_src, tgt_feat, R, W1, W2, h1_saved, workspace)) return AHV_EINVAL;
  const DetBwdWs w(B, N, grad_R && !r_per_pair);
  if ((int64_t)B * N > 0 && (!workspace || workspace_bytes < w.total * sizeof(float))) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_score_bwd_det(vol_src, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, grad_scores, h1_saved,
                              pair_inv_scale, grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, grad_R, B, N,
                              h1_saved && math_mode == AHV_MATH_TC, static_cast<float*>(workspace), (cudaStream_t)stream);
}

AHV_API int ahv_infonce(const float* scores, const float* R, int r_per_pair, const float* gt_R, float acc_thr_deg,
                        float temperature, float* loss, float* grad_scores, int B, int64_t N, void* stream) {
  if (B < 0 || N < 1 || !(temperature > 0.0f)) return AHV_EINVAL;
  if (B > 0 && (!scores || !R || !gt_R || !loss)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_infonce(scores, R, r_per_pair != 0, gt_R, acc_thr_deg, temperature, loss, grad_scores, B, N, (cudaStream_t)stream);
}

AHV_API int ahv_resblock3d(const float* x, const float* conv1_w, const float* conv2_w, const float* down_w, float* out,
                           int64_t m, void* stream) {
  if (m < 0 || (m > 0 && (!x || !conv1_w || !conv2_w || !down_w || !out))) return AHV_EINVAL;
  if (!all_aligned16(x, out)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_resblock3d(x, conv1_w, conv2_w, down_w, out, m, (cudaStream_t)stream);
}

AHV_API int ahv_score_train(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair, const float* W1,
                            const float* W2, const float* b2, const float* base, float* scores, void* h1_saved,
                            float* pair_inv_scale, int B, int64_t N, void* workspace, size_t workspace_bytes,
                            void* stream) {
  if (B < 0 || !n_ok(N)) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && !all_set(vol_src, tgt_feat, R, W1, W2, b2, base, scores, h1_saved, pair_inv_scale, workspace))
    return AHV_EINVAL;
  if (!all_aligned16(vol_src, tgt_feat, R, W1, W2, h1_saved, workspace)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_score_tc_train(vol_src, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, scores, h1_saved, pair_inv_scale, B, N,
                               workspace, workspace_bytes, (cudaStream_t)stream);
}

AHV_API int ahv_score_backward_saved(const float* vol_src, const float* tgt_feat, const float* R, int r_per_pair,
                                     const float* W1, const float* W2, const float* b2, const float* base,
                                     const float* grad_scores, const void* h1_saved, const float* pair_inv_scale,
                                     float* grad_vol, float* grad_tgt, float* grad_W1, float* grad_W2, float* grad_b2,
                                     int B, int64_t N, int math_mode, void* stream) {
  if (B < 0 || !n_ok(N)) return AHV_EINVAL;
  if (math_mode != AHV_MATH_TC && math_mode != AHV_MATH_FP32) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && !all_set(vol_src, tgt_feat, R, W1, W2, b2, base, grad_scores, h1_saved, pair_inv_scale,
                                      grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2))
    return AHV_EINVAL;
  if (!aligned16(h1_saved)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  if (math_mode == AHV_MATH_TC)
    return launch_score_bwd_tc(vol_src, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, grad_scores, h1_saved,
                               pair_inv_scale, grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, B, N, (cudaStream_t)stream);
  return launch_score_bwd(vol_src, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, grad_scores, grad_vol, grad_tgt,
                          grad_W1, grad_W2, grad_b2, B, N, (cudaStream_t)stream, h1_saved, pair_inv_scale);
}

AHV_API int ahv_forward_3d2d(const float* vol, const float* W1, const float* W2, const float* b2,
                     float* feat, int64_t m, void* stream) {
  if (m < 0 || (m > 0 && (!vol || !W1 || !W2 || !b2 || !feat))) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_forward_3d2d(vol, W1, W2, b2, feat, m, (cudaStream_t)stream);
}

AHV_API size_t ahv_workspace_bytes(int B, int64_t N, int k) {
  return B < 0 || N < 0 ? 0 : VerifyWs(B, N, k).total;
}

AHV_API int ahv_topk(const float* scores, int B, int64_t N, int k, int64_t idx_offset, float* topk_val,
             int64_t* topk_idx, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 0 || !n_ok(N) || !k_ok(k)) return AHV_EINVAL;
  if (B > 0 && (!scores || !topk_val || !topk_idx || !workspace)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_topk(scores, B, N, k, idx_offset, topk_val, topk_idx, workspace, workspace_bytes,
                     (cudaStream_t)stream);
}

AHV_API int ahv_topk_merge(const float* vals, const int64_t* idx, int parts, int B, int k, float* out_val,
                   int64_t* out_idx, void* stream) {
  if (parts < 1 || B < 0 || !k_ok(k)) return AHV_EINVAL;
  if (B > 0 && (!vals || !idx || !out_val || !out_idx)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_topk_merge(vals, idx, parts, B, k, out_val, out_idx, (cudaStream_t)stream);
}

AHV_API int ahv_gather_rotations(const float* R, int r_per_pair, const int64_t* idx, int64_t idx_offset,
                         int B, int64_t N, int k, float* R_out, void* stream) {
  if (B < 0 || N < 0 || k < 1) return AHV_EINVAL;
  if (B > 0 && (!R || !idx || !R_out)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_gather_rotations(R, r_per_pair != 0, idx, idx_offset, B, N, k, R_out,
                                 (cudaStream_t)stream);
}

AHV_API int ahv_score(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R,
              int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
              float* scores, float* topk_val, int64_t* topk_idx, int k, int64_t idx_offset, int B,
              int64_t N, int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 0 || !n_ok(N) || !vol_dtype_ok(vol_dtype) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if (k != 0 && !k_ok(k)) return AHV_EINVAL;  // k = 0: scores only
  if (k > 0 && (!topk_val || !topk_idx)) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && !all_set(vol_src, tgt_feat, R, W1, W2, b2, base)) return AHV_EINVAL;
  if (!all_aligned16(vol_src, tgt_feat, R, W1, W2, workspace)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  if ((int64_t)B * N == 0) return AHV_OK;

  const VerifyWs w(B, N, k);
  if (!workspace || workspace_bytes < w.lists) return AHV_EWORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  float* sc = scores ? scores : reinterpret_cast<float*>(ws);

  cudaStream_t s = (cudaStream_t)stream;
  if (math_mode == AHV_MATH_FP32)
    st = launch_score_fp32(vol_src, vol_dtype, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, sc, B,
                           N, s);
  else
    st = launch_score_tc(vol_src, vol_dtype, tgt_feat, R, r_per_pair != 0, W1, W2, b2, base, sc, B, N,
                         ws + w.tc, w.lists - w.tc, s, math_mode == AHV_MATH_TC_F16GATHER);
  if (st != AHV_OK) return st;
  if (k > 0) st = launch_topk(sc, B, N, k, idx_offset, topk_val, topk_idx, ws + w.topk, w.tc - w.topk, s);
  return st;
}

AHV_API int ahv_verify(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                       const float* W1, const float* W2, const float* b2, const float* base, float* scores,
                       float* topk_val, int64_t* topk_idx, float* R_best, int k, int64_t idx_offset, int B,
                       int64_t N, int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 0 || !n_ok(N) || !k_ok(k) || !vol_dtype_ok(vol_dtype) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && !all_set(vol_src, vol_tgt, R, W1, W2, b2, base, topk_val, topk_idx)) return AHV_EINVAL;
  if (!all_aligned16(vol_src, vol_tgt, R, W1, W2, workspace)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  if ((int64_t)B * N == 0) return AHV_OK;
  const VerifyWs w(B, N, k);
  if (!workspace || workspace_bytes < w.total) return AHV_EWORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  void* ws_tc = static_cast<unsigned char*>(workspace) + w.tc;  // packed weights, target features, scales, keys
  if (math_mode != AHV_MATH_FP32 && k == 1)  // three launches, nothing but 40 B per hypothesis touches HBM
    return launch_verify_tc_argmax(vol_src, vol_dtype, vol_tgt, R, r_per_pair != 0, W1, W2, b2, base, scores,
                                   topk_val, topk_idx, R_best, idx_offset, B, N, ws_tc,
                                   workspace_bytes - w.tc, s, math_mode == AHV_MATH_TC_F16GATHER);
  float* tgt = scratch_tgt_feat(ws_tc, B);
  st = launch_forward_3d2d(vol_tgt, W1, W2, b2, tgt, B, s);
  if (st != AHV_OK) return st;
  st = ahv_score(vol_src, vol_dtype, tgt, R, r_per_pair, W1, W2, b2, base, scores, topk_val, topk_idx, k,
                 idx_offset, B, N, math_mode, workspace, workspace_bytes, stream);
  if (st != AHV_OK) return st;
  if (R_best)
    st = launch_gather_rotations(R, r_per_pair != 0, topk_idx, idx_offset, B, N, k, R_best, s);
  return st;
}

// ---- two-pass selection: dense set -> top-k -> local refinement (BASELINE config 4; extension) -----------
AHV_API size_t ahv_refine_workspace_bytes(int B, int64_t N, int k, int m) {
  return B < 0 || N < 0 || !k_ok(k) || m < 1 ? 0 : RefineWs(B, N, k, m).total;
}

AHV_API int ahv_refine(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                       const float* W1, const float* W2, const float* b2, const float* base, int k, int m,
                       float max_angle_deg, uint64_t seed, float* first_val, int64_t* first_idx, float* first_R,
                       float* cand, float* best_val, int64_t* best_idx, float* R_best, int B, int64_t N,
                       int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 1 || N < 1 || !k_ok(k) || k > N || m < 1 || !n_ok((int64_t)k * m)) return AHV_EINVAL;
  if (!all_set(first_val, first_idx, first_R, cand, best_val, best_idx, workspace)) return AHV_EINVAL;
  if (!aligned16(cand)) return AHV_EINVAL;
  const RefineWs w(B, N, k, m);
  if (workspace_bytes < w.total) return AHV_EWORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  // pass 1: the whole set, top-k and their rotations
  int st = ahv_verify(vol_src, vol_dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, nullptr, first_val, first_idx, first_R, k,
                      0, B, N, math_mode, ws, w.cand, stream);
  if (st != AHV_OK) return st;
  // candidates: m rotations within max_angle_deg of each of the B*k winners (index 0 = the winner itself)
  st = ahv_so3_perturb(first_R, (int64_t)B * k, m, max_angle_deg, seed, cand, stream);
  if (st != AHV_OK) return st;
  // pass 2: per-pair candidate sets [B, k*m], arg-max
  return ahv_verify(vol_src, vol_dtype, vol_tgt, cand, 1, W1, W2, b2, base, nullptr, best_val, best_idx, R_best, 1, 0, B,
                    (int64_t)k * m, math_mode, ws + w.cand, w.total - w.cand, stream);
}

// ---- gradient ascent of the fp32 score on SO(3), alone and after the grid pass (extension) ---------------
namespace {
bool ascent_args_ok(int vol_dtype, int steps, float step_deg) {
  return vol_dtype_ok(vol_dtype) && steps >= 0 && steps <= 1000 &&
         std::isfinite(step_deg) && step_deg > 0.0f;   // the step cap bounds the runtime of one launch
}
}  // namespace

AHV_API int ahv_gradient_ascent(const void* vol_src, int vol_dtype, const float* tgt_feat, const float* R_init,
                                const float* W1, const float* W2, const float* b2, const float* base, int steps,
                                float step_deg, float* R_out, float* score_out, int B, int K, void* stream) {
  if (B < 1 || K < 1 || !ascent_args_ok(vol_dtype, steps, step_deg)) return AHV_EINVAL;
  if (!all_set(vol_src, tgt_feat, R_init, W1, W2, b2, base, R_out, score_out)) return AHV_EINVAL;
  if (!all_aligned16(vol_src, tgt_feat, R_init, R_out, W1, W2)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_gradient_ascent(vol_src, vol_dtype, tgt_feat, R_init, W1, W2, b2, base, steps, step_deg, R_out, score_out,
                                B, K, (cudaStream_t)stream);
}

AHV_API size_t ahv_refine_gradient_workspace_bytes(int B, int64_t N, int k) {
  return B < 0 || N < 0 || !k_ok(k) ? 0 : RefineGradientWs(B, N, k).total;
}

namespace {
bool min_sep_ok(float min_sep_deg) { return std::isfinite(min_sep_deg) && min_sep_deg >= 0.0f && min_sep_deg <= 180.0f; }

// ahv_refine_gradient (min_sep_deg == 0) and ahv_refine_gradient_distinct: the same chain apart from its first pass
int refine_gradient(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair, const float* W1,
                    const float* W2, const float* b2, const float* base, int k, int steps, float step_deg, float min_sep_deg,
                    float* first_val, int64_t* first_idx, float* first_R, float* R_all, float* score_all, float* best_val,
                    int64_t* best_idx, float* R_best, int B, int64_t N, int math_mode, void* workspace,
                    size_t workspace_bytes, void* stream) {
  if (B < 1 || N < 1 || !n_ok(N) || !k_ok(k) || k > N) return AHV_EINVAL;
  if (!ascent_args_ok(vol_dtype, steps, step_deg) || !min_sep_ok(min_sep_deg) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if (!all_set(vol_src, vol_tgt, R, W1, W2, b2, base, first_val, first_idx, first_R, R_all, score_all, best_val, best_idx,
               workspace))
    return AHV_EINVAL;
  if (!all_aligned16(vol_src, vol_tgt, R, W1, W2, first_R, R_all, R_best, workspace)) return AHV_EINVAL;
  const RefineGradientWs w(B, N, k);
  if (workspace_bytes < w.total) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  float* tgt = reinterpret_cast<float*>(ws + w.tgt);
  const bool distinct = min_sep_deg > 0.0f;
  if (!distinct) {
    // pass 1: the whole set, top-k and their rotations
    st = ahv_verify(vol_src, vol_dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, nullptr, first_val, first_idx, first_R, k,
                    0, B, N, math_mode, ws, w.tgt, stream);
    if (st != AHV_OK) return st;
  }
  // the ascent scores in fp32 against fp32 target features (bit-equal to ahv_forward_3d2d), whatever math_mode is
  st = launch_forward_3d2d(vol_tgt, W1, W2, b2, tgt, B, s);
  if (st != AHV_OK) return st;
  if (distinct) {
    // pass 1: every score of the set (the fused k = 1 arg-max writes none), then the k distinct winners
    st = ahv_score(vol_src, vol_dtype, tgt, R, r_per_pair, W1, W2, b2, base, nullptr, nullptr, nullptr, 0, 0, B, N,
                   math_mode, ws, w.tgt, stream);
    if (st != AHV_OK) return st;
    st = launch_topk_distinct(reinterpret_cast<const float*>(ws), R, r_per_pair != 0, B, N, k, min_sep_deg, first_val,
                              first_idx, first_R, s);
    if (st != AHV_OK) return st;
  }
  // empty slots (fewer than k distinct winners) are not ascended: R_all NaN, score_all -inf
  st = launch_gradient_ascent(vol_src, vol_dtype, tgt, first_R, W1, W2, b2, base, steps, step_deg, R_all, score_all, B, k, s,
                              distinct ? first_idx : nullptr);
  if (st != AHV_OK) return st;
  // per-pair arg-max over the k ascended candidates
  st = launch_topk(score_all, B, k, 1, 0, best_val, best_idx, ws + w.top, w.total - w.top, s);
  if (st != AHV_OK || !R_best) return st;
  return launch_gather_rotations(R_all, 1, best_idx, 0, B, k, 1, R_best, s);
}
}  // namespace

AHV_API int ahv_refine_gradient(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                                const float* W1, const float* W2, const float* b2, const float* base, int k, int steps,
                                float step_deg, float* first_val, int64_t* first_idx, float* first_R, float* R_all,
                                float* score_all, float* best_val, int64_t* best_idx, float* R_best, int B, int64_t N,
                                int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  return refine_gradient(vol_src, vol_dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, k, steps, step_deg, 0.0f, first_val,
                         first_idx, first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math_mode, workspace,
                         workspace_bytes, stream);
}

AHV_API int ahv_refine_gradient_distinct(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                                         int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
                                         int k, int steps, float step_deg, float min_sep_deg, float* first_val,
                                         int64_t* first_idx, float* first_R, float* R_all, float* score_all, float* best_val,
                                         int64_t* best_idx, float* R_best, int B, int64_t N, int math_mode, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  return refine_gradient(vol_src, vol_dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, k, steps, step_deg, min_sep_deg,
                         first_val, first_idx, first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math_mode,
                         workspace, workspace_bytes, stream);
}

// ---- top-k of distinct rotations: greedy geodesic non-maximum suppression on SO(3) (extension) ------------
AHV_API int ahv_topk_distinct(const float* scores, const float* R, int r_per_pair, int B, int64_t N, int k,
                              float min_sep_deg, float* topk_val, int64_t* topk_idx, float* R_best, void* stream) {
  if (B < 0 || !n_ok(N) || !k_ok(k) || !min_sep_ok(min_sep_deg)) return AHV_EINVAL;
  if (B > 0 && (!topk_val || !topk_idx)) return AHV_EINVAL;
  if ((int64_t)B * N > 0 && (!scores || !R)) return AHV_EINVAL;
  if (!all_aligned16(R, R_best)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_topk_distinct(scores, R, r_per_pair != 0, B, N, k, min_sep_deg, topk_val, topk_idx, R_best,
                              (cudaStream_t)stream);
}

// ---- hypothesis set sharded over the GPUs of one node: winners exchanged through peer memory -------------
AHV_API size_t ahv_peer_bytes(int max_pairs, int max_k) {
  return (max_pairs < 1 || !k_ok(max_k)) ? 0 : peer::buffer_bytes(max_pairs, max_k);
}

AHV_API int ahv_peer_alloc(int max_pairs, int max_k, void** ptr) {
  if (!ptr || max_pairs < 1 || !k_ok(max_k)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  const size_t bytes = peer::buffer_bytes(max_pairs, max_k);
  if (cudaMalloc(ptr, bytes) != cudaSuccess) return AHV_ECUDA;
  const uint32_t hdr[4] = {0u, 0u, (uint32_t)max_pairs, (uint32_t)max_k};  // seq, err, capacity
  if (cudaMemset(*ptr, 0, bytes) != cudaSuccess || cudaMemcpy(*ptr, hdr, sizeof(hdr), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess) {
    cudaFree(*ptr);
    *ptr = nullptr;
    return AHV_ECUDA;
  }
  return AHV_OK;
}

AHV_API int ahv_peer_free(void* ptr) { return (!ptr || cudaFree(ptr) == cudaSuccess) ? AHV_OK : AHV_ECUDA; }

AHV_API int ahv_peer_export(void* ptr, unsigned char* handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (!ptr || !handle64) return AHV_EINVAL;
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, ptr) != cudaSuccess) return AHV_ECUDA;
  memcpy(handle64, &h, 64);
  return AHV_OK;
}

AHV_API int ahv_peer_open(const unsigned char* handle64, void** ptr) {
  if (!handle64 || !ptr) return AHV_EINVAL;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  if (cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) return AHV_ECUDA;
  return AHV_OK;
}

AHV_API int ahv_peer_status(const void* own, unsigned* exchanges_done, unsigned* timed_out) {
  if (!own || !exchanges_done || !timed_out) return AHV_EINVAL;
  unsigned hdr[2];
  if (cudaMemcpy(hdr, own, sizeof(hdr), cudaMemcpyDeviceToHost) != cudaSuccess) return AHV_ECUDA;  // synchronises
  *exchanges_done = hdr[0];
  *timed_out = hdr[1];
  return AHV_OK;
}

AHV_API int ahv_peer_capacity(const void* buf, int* max_pairs, int* max_k) {
  if (!buf || !max_pairs || !max_k) return AHV_EINVAL;
  unsigned hdr[4];
  if (cudaMemcpy(hdr, buf, sizeof(hdr), cudaMemcpyDeviceToHost) != cudaSuccess) return AHV_ECUDA;  // synchronises
  *max_pairs = (int)hdr[2];
  *max_k = (int)hdr[3];
  return AHV_OK;
}

AHV_API int ahv_peer_close(void* ptr) { return (!ptr || cudaIpcCloseMemHandle(ptr) == cudaSuccess) ? AHV_OK : AHV_ECUDA; }

namespace {
int make_peer_args(int rank, int world, void* const* peers, int peer_max_pairs, int peer_max_k, peer::Args* pa) {
  if (world < 1 || world > peer::kMaxPeers || rank < 0 || rank >= world) return AHV_EINVAL;
  pa->rank = rank;
  pa->world = world;
  pa->cap_pairs = peer_max_pairs;
  pa->cap_k = peer_max_k;
  if (world > 1) {
    if (!peers || peer_max_pairs < 1 || !k_ok(peer_max_k)) return AHV_EINVAL;
    for (int r = 0; r < world; ++r) {
      if (!peers[r]) return AHV_EINVAL;
      pa->bufs[r] = static_cast<unsigned char*>(peers[r]);
    }
  }
  return AHV_OK;
}
}  // namespace

AHV_API int ahv_topk_exchange(const float* val, const int64_t* idx, const float* R, int r_per_pair, int64_t idx_offset,
                              int64_t N, int B, int k, float* out_val, int64_t* out_idx, float* R_best, int rank,
                              int world, void* const* peers, int peer_max_pairs, int peer_max_k, void* stream) {
  if (B < 1 || !k_ok(k) || N < 0 || idx_offset < 0 || !val || !idx || !out_val || !out_idx || (N > 0 && !R))
    return AHV_EINVAL;
  if (idx_offset + N > 0x100000000LL) return AHV_EINVAL;  // keys carry 32 index bits
  peer::Args pa;
  int st = make_peer_args(rank, world, peers, peer_max_pairs, peer_max_k, &pa);
  if (st != AHV_OK) return st;
  if (world < 2) return AHV_EINVAL;
  st = check_device();
  if (st != AHV_OK) return st;
  return launch_topk_exchange(val, idx, R, r_per_pair != 0, idx_offset, N, B, k, out_val, out_idx, R_best, pa,
                              (cudaStream_t)stream);
}

AHV_API int ahv_verify_sharded(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                               const float* W1, const float* W2, const float* b2, const float* base, float* topk_val,
                               int64_t* topk_idx, float* R_best, int k, int64_t idx_offset, int B, int64_t N,
                               int math_mode, void* workspace, size_t workspace_bytes, int rank, int world,
                               void* const* peers, int peer_max_pairs, int peer_max_k, void* stream) {
  if (B < 1 || !n_ok(N) || !k_ok(k) || idx_offset < 0) return AHV_EINVAL;
  if (idx_offset + N > 0x100000000LL) return AHV_EINVAL;  // keys carry 32 index bits
  if (!vol_dtype_ok(vol_dtype) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if (!vol_src || !vol_tgt || (N > 0 && !R) || !W1 || !W2 || !b2 || !base || !topk_val || !topk_idx) return AHV_EINVAL;
  if (!all_aligned16(vol_src, vol_tgt, R, W1, W2, workspace)) return AHV_EINVAL;
  peer::Args pa;
  int st = make_peer_args(rank, world, peers, peer_max_pairs, peer_max_k, &pa);
  if (st != AHV_OK) return st;
  if (world > 1 && (B > peer_max_pairs || k > peer_max_k)) return AHV_EINVAL;  // exchange buffer too small for this call
  st = check_device();
  if (st != AHV_OK) return st;
  if (world == 1)
    return N == 0 ? AHV_EINVAL
                  : ahv_verify(vol_src, vol_dtype, vol_tgt, R, r_per_pair, W1, W2, b2, base, nullptr, topk_val, topk_idx,
                               R_best, k, idx_offset, B, N, math_mode, workspace, workspace_bytes, stream);
  const VerifyWs w(B, N, k);
  if (!workspace || workspace_bytes < w.total) return AHV_EWORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  cudaStream_t s = (cudaStream_t)stream;
  if (k == 1 && N > 0 && math_mode != AHV_MATH_FP32)  // the scoring kernel exchanges and merges the winners itself
    return launch_verify_tc_argmax(vol_src, vol_dtype, vol_tgt, R, r_per_pair != 0, W1, W2, b2, base, nullptr, topk_val,
                                   topk_idx, R_best, idx_offset, B, N, ws + w.tc, w.lists - w.tc, s,
                                   math_mode == AHV_MATH_TC_F16GATHER, &pa);
  // k > 1 (or an empty shard, or fp32 FFMA arithmetic): local top-k of the shard, then the exchange kernel
  float* l_val = reinterpret_cast<float*>(ws + w.lists);
  int64_t* l_idx = reinterpret_cast<int64_t*>(ws + w.lists + align_up((size_t)B * k * sizeof(float), 8));
  const int kl = N < k ? (int)N : k;
  if (kl < k) {  // pad with (-inf, -1), which the merge ignores
    AHV_CUDA_OK(cudaMemsetAsync(l_val, 0xff, (size_t)B * k * sizeof(float), s));
    AHV_CUDA_OK(cudaMemsetAsync(l_idx, 0xff, (size_t)B * k * sizeof(int64_t), s));
  }
  if (N > 0) {
    float* tgt = scratch_tgt_feat(ws + w.tc, B);
    st = launch_forward_3d2d(vol_tgt, W1, W2, b2, tgt, B, s);
    if (st != AHV_OK) return st;
    if (kl == k) {
      st = ahv_score(vol_src, vol_dtype, tgt, R, r_per_pair, W1, W2, b2, base, nullptr, l_val, l_idx, k, idx_offset, B, N,
                     math_mode, workspace, workspace_bytes, stream);
    } else {  // fewer hypotheses than k on this shard: compact [B,kl] lists (in the output buffers, which the
              // exchange overwrites afterwards), then spread into the padded [B,k]
      st = ahv_score(vol_src, vol_dtype, tgt, R, r_per_pair, W1, W2, b2, base, nullptr, topk_val, topk_idx, kl, idx_offset, B,
                     N, math_mode, workspace, workspace_bytes, stream);
      if (st != AHV_OK) return st;
      AHV_CUDA_OK(cudaMemcpy2DAsync(l_val, (size_t)k * sizeof(float), topk_val, (size_t)kl * sizeof(float),
                                    (size_t)kl * sizeof(float), B, cudaMemcpyDeviceToDevice, s));
      AHV_CUDA_OK(cudaMemcpy2DAsync(l_idx, (size_t)k * sizeof(int64_t), topk_idx, (size_t)kl * sizeof(int64_t),
                                    (size_t)kl * sizeof(int64_t), B, cudaMemcpyDeviceToDevice, s));
    }
    if (st != AHV_OK) return st;
  }
  return launch_topk_exchange(l_val, l_idx, R, r_per_pair != 0, idx_offset, N, B, k, topk_val, topk_idx, R_best, pa, s);
}

// ---- host-buffer entries -------------------------------------------------------------------------------
// A session owns the device scratch of the host-buffer entry, grown on demand and reused across calls
// (explicit caller-owned state; nothing process-global is touched).
struct ahv_host_session {
  unsigned char* d = nullptr;
  size_t bytes = 0;
  int device = -1;
};

AHV_API int ahv_host_session_create(ahv_host_session** session) {
  if (!session) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  ahv_host_session* hs = new (std::nothrow) ahv_host_session();
  if (!hs) return AHV_ECUDA;
  if (cudaGetDevice(&hs->device) != cudaSuccess) { delete hs; return AHV_ECUDA; }
  *session = hs;
  return AHV_OK;
}

AHV_API int ahv_host_session_destroy(ahv_host_session* session) {
  if (!session) return AHV_OK;
  const bool ok = !session->d || cudaFree(session->d) == cudaSuccess;
  delete session;
  return ok ? AHV_OK : AHV_ECUDA;
}

AHV_API int ahv_predict_host_ex(ahv_host_session* session, const void* vol_src_host, int vol_dtype,
                                const float* vol_tgt_host, const float* R_host, int r_per_pair, const float* W1_host,
                                const float* W2_host, const float* b2_host, const float* base_host, float* scores_host,
                                float* topk_val_host, int64_t* topk_idx_host, float* R_best_host, int k,
                                int64_t idx_offset, int B, int64_t N, int math_mode, int rank, int world,
                                void* const* peers, int peer_max_pairs, int peer_max_k, void* stream) {
  if (!session || B < 1 || N < 1 || !k_ok(k)) return AHV_EINVAL;
  if (!vol_dtype_ok(vol_dtype)) return AHV_EINVAL;
  if (!all_set(vol_src_host, vol_tgt_host, R_host, W1_host, W2_host, b2_host, base_host)) return AHV_EINVAL;
  if (!topk_val_host || !topk_idx_host) return AHV_EINVAL;
  if (world > 1 && scores_host) return AHV_EINVAL;  // a sharded step returns the selection only
  int st = check_device();
  if (st != AHV_OK) return st;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev != session->device) return AHV_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t src_b = (size_t)B * kC * kVox * (vol_dtype == AHV_VOL_BF16 ? 2 : 4);
  const size_t tgt_b = (size_t)B * kC * kVox * sizeof(float);
  const size_t r_b = (size_t)(r_per_pair ? B : 1) * N * 9 * sizeof(float);
  const size_t w_b = (size_t)(kO * kK + kO * kO + kO + 8) * sizeof(float);
  const size_t out_b = (size_t)B * k * (sizeof(float) + sizeof(int64_t) + 9 * sizeof(float));
  const size_t ws_b = VerifyWs(B, N, k).total;
  const size_t total = align_up(src_b, 256) + align_up(tgt_b, 256) + align_up(r_b, 256) + align_up(w_b, 256) +
                       align_up(out_b, 256) + ws_b;
  if (session->bytes < total) {  // grow (rare): the stream may still use the old block
    if (cudaStreamSynchronize(s) != cudaSuccess) return AHV_ECUDA;
    if (session->d && cudaFree(session->d) != cudaSuccess) return AHV_ECUDA;
    session->d = nullptr;
    session->bytes = 0;
    if (cudaMalloc((void**)&session->d, total) != cudaSuccess) return AHV_ECUDA;
    session->bytes = total;
  }
  unsigned char* p = session->d;
  auto take = [&](size_t bytes) { unsigned char* r = p; p += align_up(bytes, 256); return r; };
  void* d_src = take(src_b);
  float* d_tgt = (float*)take(tgt_b);
  float* d_R = (float*)take(r_b);
  float* d_w = (float*)take(w_b);
  unsigned char* d_out = take(out_b);
  void* d_ws = p;
  float* d_W1 = d_w; float* d_W2 = d_W1 + kO * kK; float* d_b2 = d_W2 + kO * kO; float* d_base = d_b2 + kO;
  // d_out: [idx int64 B*k | val fp32 B*k | R_best fp32 B*k*9]
  int64_t* d_idx = (int64_t*)d_out;
  float* d_val = (float*)(d_out + (size_t)B * k * sizeof(int64_t));
  float* d_Rb = d_val + (size_t)B * k;
  st = AHV_ECUDA;
  do {
    if (cudaMemcpyAsync(d_src, vol_src_host, src_b, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_tgt, vol_tgt_host, tgt_b, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_R, R_host, r_b, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_W1, W1_host, kO * kK * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_W2, W2_host, kO * kO * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_b2, b2_host, kO * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_base, base_host, 8 * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (world > 1)
      st = ahv_verify_sharded(d_src, vol_dtype, d_tgt, d_R, r_per_pair, d_W1, d_W2, d_b2, d_base, d_val, d_idx, d_Rb, k,
                              idx_offset, B, N, math_mode, d_ws, ws_b, rank, world, peers, peer_max_pairs, peer_max_k,
                              stream);
    else
      st = ahv_verify(d_src, vol_dtype, d_tgt, d_R, r_per_pair, d_W1, d_W2, d_b2, d_base,
                      scores_host ? (float*)d_ws : nullptr, d_val, d_idx, d_Rb, k, idx_offset, B, N, math_mode, d_ws, ws_b,
                      stream);
    if (st != AHV_OK) break;
    st = AHV_ECUDA;
    if (scores_host &&
        cudaMemcpyAsync(scores_host, d_ws, (size_t)B * N * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess)
      break;
    if (cudaMemcpyAsync(topk_idx_host, d_idx, (size_t)B * k * 8, cudaMemcpyDeviceToHost, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(topk_val_host, d_val, (size_t)B * k * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess) break;
    if (R_best_host &&
        cudaMemcpyAsync(R_best_host, d_Rb, (size_t)B * k * 36, cudaMemcpyDeviceToHost, s) != cudaSuccess)
      break;
    st = AHV_OK;
  } while (0);
  if (cudaStreamSynchronize(s) != cudaSuccess && st == AHV_OK) st = AHV_ECUDA;
  return st;
}

AHV_API int ahv_predict_host(const float* vol_src_host, const float* vol_tgt_host, const float* R_host,
                     int r_per_pair, const float* W1_host, const float* W2_host,
                     const float* b2_host, const float* base_host, float* scores_host,
                     float* topk_val_host, int64_t* topk_idx_host, float* R_best_host, int k, int B,
                     int64_t N, int math_mode, void* stream) {
  ahv_host_session* hs = nullptr;
  int st = ahv_host_session_create(&hs);
  if (st != AHV_OK) return st;
  st = ahv_predict_host_ex(hs, vol_src_host, AHV_VOL_F32, vol_tgt_host, R_host, r_per_pair, W1_host, W2_host, b2_host,
                           base_host, scores_host, topk_val_host, topk_idx_host, R_best_host, k, 0, B, N, math_mode, 0, 1,
                           nullptr, 0, 0, stream);
  const int st2 = ahv_host_session_destroy(hs);
  return st != AHV_OK ? st : st2;
}

}  // extern "C"
