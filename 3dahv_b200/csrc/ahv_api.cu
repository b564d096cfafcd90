// extern "C" surface of lib3dahv_b200 (see include/ahv_b200.h for the contract
// and the reference interface each entry replaces).
#include <algorithm>
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

// Workspace layouts.  Each is built from the workspace's base, or from nullptr when only its size `total` is wanted, and
// places its regions with a Carve, each 256-byte aligned.

// The verification workspace: [scores B*N fp32 | top-k partials | tensor-core scratch | a shard's top-k lists [B,k]].
// ahv_score needs the bytes before the lists, `score_bytes`.
struct VerifyWs {
  float* scores;        // where score_chain scores when it is given no output
  size_t topk_bytes;
  unsigned char* topk;
  ScreenLists screen;   // the screened arg-max's lists, inside the top-k partials, which it leaves unused
  TcScratch tc;         // tc.tgt_feat: where verify_chain computes the target features
  float* l_val;
  int64_t* l_idx;
  size_t score_bytes, total;
  VerifyWs(void* ws, int B, int64_t N, int k) {
    Carve c(ws);
    scores = c.take<float>((size_t)B * N, 256);
    topk_bytes = (topk_workspace_bytes(B, N, k) + 255) / 256 * 256;
    topk = c.take<unsigned char>(topk_bytes, 256);
    Carve in_topk(topk);
    screen = ScreenLists(in_topk, B);
    Carve in_tc(c.take<unsigned char>(bytes_of<TcScratch>(B), 256));
    tc = TcScratch(in_tc, B);
    score_bytes = c.off;
    Carve in_lists(c.take<unsigned char>((size_t)B * (k > 0 ? k : 1) * (sizeof(float) + sizeof(int64_t)), 256));
    l_val = in_lists.take<float>((size_t)B * k, 8);
    l_idx = in_lists.take<int64_t>((size_t)B * k, 8);
    total = c.off;
  }
};

// ahv_refine: [the grid pass's verification workspace | the candidate pass's ([B, k*m], arg-max)]
struct RefineWs {
  unsigned char *grid, *cand;
  size_t total;
  RefineWs(void* ws, int B, int64_t N, int k, int m) {
    Carve c(ws);
    grid = c.take<unsigned char>(VerifyWs(nullptr, B, N, k).total, 256);
    cand = c.take<unsigned char>(VerifyWs(nullptr, B, (int64_t)k * m, 1).total, 256);
    total = c.off;
  }
};

// ahv_refine_gradient(_distinct) (world == 1) and ahv_refine_gradient_sharded, per = ceil(N / world) hypotheses at most
// on a rank: [the slice's verification workspace | the slice's rotations B*per*9 | the whole score matrix B*N (distinct
// pass 1) | target features B*32*64 | top-k partials over [B,k]].  One GPU scores R in place and keeps the distinct
// pass's scores in the verification workspace, so its two middle regions are empty.
struct ShardedRefineWs {
  unsigned char* verify;
  float *rs, *full, *tgt;
  unsigned char* top;
  size_t top_bytes, total;
  ShardedRefineWs(void* ws, int B, int64_t N, int k, int world) {
    const int64_t per = (N + world - 1) / world;
    Carve c(ws);
    verify = c.take<unsigned char>(VerifyWs(nullptr, B, per, k).total, 256);
    rs = c.take<float>(world > 1 ? (size_t)B * (size_t)per * 9 : 0, 256);
    full = c.take<float>(world > 1 ? (size_t)B * (size_t)N : 0, 256);
    tgt = c.take<float>((size_t)B * kO * kP, 256);
    top_bytes = (topk_workspace_bytes(B, k, 1) + 255) / 256 * 256;
    top = c.take<unsigned char>(top_bytes, 256);
    total = c.off;
  }
};

// The screened arg-max (launch_verify_tc_screened, ahv_score_tc.cu) serves ahv_verify and ahv_verify_sharded for fp32
// volumes under AHV_MATH_TC with k == 1 and no scores returned, once a call has enough items to repay its five extra
// launches (the single-pair latency calls, B = 1 at N = 3 000 or 50 000, stay on the single pass).  Its buffers live in the
// verification workspace that the k == 1 path leaves unused - the scores (B*N fp32) and the top-k partials (B*N/16
// bytes and more) - so the workspace size is the same as before; that needs N of about 40 000 or more.
constexpr int64_t kScreenMinItems = 1 << 18;
bool screened(const VerifyWs& w, int vol_dtype, int math_mode, const float* scores, int k, int B, int64_t N) {
  return vol_dtype == AHV_VOL_F32 && math_mode == AHV_MATH_TC && k == 1 && !scores && (int64_t)B * N >= kScreenMinItems &&
         N * sizeof(float) >= kScreenList * 10 * sizeof(float) && w.topk_bytes >= bytes_of<ScreenLists>(B);
}

// ---- chains: the device work of the entries, once their arguments have been checked -------------------------------
// Each entry checks its arguments, then the device, then composes chains and launch_* functions; no entry calls
// another (the host-buffer entries aside).  `pa` == nullptr or a group of one is one GPU.

// ahv_score: the scores (into `scores`, else the workspace's score region) and, for k > 0, their top-k
int score_chain(const Scored& p, const float* tgt_feat, float* scores, float* topk_val, int64_t* topk_idx, int k,
                int64_t idx_offset, int math_mode, void* ws, cudaStream_t s) {
  const VerifyWs w(ws, p.B, p.N, k);
  float* sc = scores ? scores : w.scores;
  const int st = math_mode == AHV_MATH_FP32 ? launch_score_fp32(p, tgt_feat, sc, s)
                                            : launch_score_tc(p, tgt_feat, sc, w.tc, s, math_mode == AHV_MATH_TC_F16GATHER);
  if (st != AHV_OK || k == 0) return st;
  return launch_topk(sc, p.B, p.N, k, idx_offset, topk_val, topk_idx, w.topk, w.topk_bytes, s);
}

// ahv_verify (B*N > 0) and a shard's step of ahv_verify_sharded (N == 0: an empty shard, which still joins the exchange).
// A shard returns the whole set's selection only, so it passes no scores.
int verify_chain(const Scored& p, const float* vol_tgt, float* scores, float* topk_val, int64_t* topk_idx, float* R_best,
                 int k, int64_t idx_offset, int math_mode, void* ws, cudaStream_t s, const peer::Args* pa) {
  if (pa && pa->world == 1) pa = nullptr;
  const int B = p.B;
  const int64_t N = p.N;
  const VerifyWs w(ws, B, N, k);
  if (N > 0 && screened(w, p.vol_dtype, math_mode, scores, k, B, N))  // a shard's last pass exchanges and merges the winners
    return launch_verify_tc_screened(p, vol_tgt, topk_val, topk_idx, R_best, idx_offset, w.tc, w.scores, w.screen, s, pa);
  // three launches, nothing but 40 B per hypothesis touches HBM; a shard's scoring kernel exchanges and merges itself
  if (N > 0 && k == 1 && math_mode != AHV_MATH_FP32)
    return launch_verify_tc_argmax(p, vol_tgt, scores, topk_val, topk_idx, R_best, idx_offset, w.tc, s,
                                   math_mode == AHV_MATH_TC_F16GATHER, pa);
  float* tgt = w.tc.tgt_feat;
  int st;
  if (!pa) {  // target features, scores and top-k, winner gather
    st = launch_forward_3d2d(vol_tgt, p.W1, p.W2, p.b2, tgt, B, s);
    if (st != AHV_OK) return st;
    st = score_chain(p, tgt, scores, topk_val, topk_idx, k, idx_offset, math_mode, ws, s);
    if (st != AHV_OK || !R_best) return st;
    return launch_gather_rotations(p.R, p.r_per_pair, topk_idx, idx_offset, B, N, k, R_best, s);
  }
  // a shard with k > 1 (or empty, or fp32 FFMA arithmetic): its local top-k, then the exchange kernel.  The top-k of a
  // shard with fewer than k hypotheses ends in (-inf, -1), which the exchange ignores; an empty shard's list is all that.
  if (N == 0) {
    AHV_CUDA_OK(cudaMemsetAsync(w.l_val, 0xff, (size_t)B * k * sizeof(float), s));
    AHV_CUDA_OK(cudaMemsetAsync(w.l_idx, 0xff, (size_t)B * k * sizeof(int64_t), s));
  } else {
    st = launch_forward_3d2d(vol_tgt, p.W1, p.W2, p.b2, tgt, B, s);
    if (st != AHV_OK) return st;
    st = score_chain(p, tgt, nullptr, w.l_val, w.l_idx, k, idx_offset, math_mode, ws, s);
    if (st != AHV_OK) return st;
  }
  return launch_topk_exchange(w.l_val, w.l_idx, p.R, p.r_per_pair, idx_offset, N, B, k, topk_val, topk_idx, R_best, *pa, s);
}

// ahv_refine_gradient(_distinct) and ahv_refine_gradient_sharded: the first pass (top-k, or with min_sep_deg > 0 the
// distinct top-k of every score), target features, gradient ascent of each winner, per-pair arg-max.  A rank of a group
// scores its shard_bounds slice of R, exchanges the first pass, ascends its share of the B*k slots and gathers every
// ascended slot; every rank then holds the whole-set result.
int refine_gradient_chain(const Scored& p, const float* vol_tgt, int k, int steps, float step_deg, float min_sep_deg,
                          float* first_val, int64_t* first_idx, float* first_R, float* R_all, float* score_all,
                          float* best_val, int64_t* best_idx, float* R_best, int math_mode, void* ws, cudaStream_t s,
                          const peer::Args* pa, int64_t peer_max_hyps) {
  if (pa && pa->world == 1) pa = nullptr;
  const int B = p.B;
  const int64_t N = p.N;
  const ShardedRefineWs w(ws, B, N, k, pa ? pa->world : 1);
  const bool distinct = min_sep_deg > 0.0f;
  int64_t lo = 0, hi = N;
  if (pa) peer::shard_bounds(N, pa->rank, pa->world, &lo, &hi);
  const int64_t n = hi - lo;
  const Scored slice = p.with_R(pa ? w.rs : p.R, p.r_per_pair, n);
  if (pa && n > 0)  // this rank's rotations, 16-byte aligned for the scorers (a shared set: one row)
    AHV_CUDA_OK(cudaMemcpy2DAsync(w.rs, (size_t)n * 9 * sizeof(float), p.R + (size_t)lo * 9, (size_t)N * 9 * sizeof(float),
                                  (size_t)n * 9 * sizeof(float), p.r_per_pair ? B : 1, cudaMemcpyDeviceToDevice, s));
  int st;
  if (!distinct) {
    // pass 1: the top-k and their rotations (a shard's, exchanged and merged into the whole set's)
    st = verify_chain(slice, vol_tgt, nullptr, first_val, first_idx, first_R, k, lo, math_mode, w.verify, s, pa);
    if (st != AHV_OK) return st;
  }
  // the ascent scores in fp32 against fp32 target features (bit-equal to ahv_forward_3d2d), whatever math_mode is
  st = launch_forward_3d2d(vol_tgt, p.W1, p.W2, p.b2, w.tgt, B, s);
  if (st != AHV_OK) return st;
  if (distinct) {
    // pass 1: every score of the set (the fused k = 1 arg-max writes none), a shard's all-gathered into the whole [B,N]
    // on every rank, then the k distinct winners: the SAME greedy selection over the whole set on every rank (per-shard
    // NMS lists do not merge into the global one)
    const float* sc = VerifyWs(w.verify, B, n, 0).scores;
    if (n > 0) {
      st = score_chain(slice, w.tgt, nullptr, nullptr, nullptr, 0, 0, math_mode, w.verify, s);
      if (st != AHV_OK) return st;
    }
    if (pa) {
      st = launch_scores_exchange(sc, B, N, w.full, *pa, peer_max_hyps, s);
      if (st != AHV_OK) return st;
      sc = w.full;
    }
    st = launch_topk_distinct(sc, p.R, p.r_per_pair, B, N, k, min_sep_deg, first_val, first_idx, first_R, s);
    if (st != AHV_OK) return st;
  }
  // empty slots (fewer than k distinct winners) are not ascended: R_all NaN, score_all -inf.  One GPU ascends every
  // slot (item_hi < 0), a rank its share, after which every ascended slot goes to every rank.
  int64_t ilo = 0, ihi = -1;
  if (pa) peer::shard_bounds((int64_t)B * k, pa->rank, pa->world, &ilo, &ihi);
  st = launch_gradient_ascent(p.with_R(first_R, true, k), w.tgt, steps, step_deg, R_all, score_all, s,
                              distinct ? first_idx : nullptr, ilo, ihi);
  if (st == AHV_OK && pa) st = launch_slot_gather(R_all, score_all, ilo, ihi, B, k, *pa, s);
  if (st != AHV_OK) return st;
  // per-pair arg-max over the k ascended candidates (on every rank)
  st = launch_topk(score_all, B, k, 1, 0, best_val, best_idx, w.top, w.top_bytes, s);
  if (st != AHV_OK || !R_best) return st;
  return launch_gather_rotations(R_all, 1, best_idx, 0, B, k, 1, R_best, s);
}

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

AHV_API int ahv_so3_hopf_grid(int level, int64_t first_index, float* R, int64_t count, void* stream) {
  if (level < 0 || level > kHopfMaxLevel || first_index < 0 || count < 0) return AHV_EINVAL;
  if (first_index > hopf_cells(level) - count || (count > 0 && !R)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_so3_hopf_grid(level, first_index, R, count, (cudaStream_t)stream);
}

AHV_API int ahv_so3_hopf_children(int level, const int64_t* parent_idx, int64_t n, int64_t* child_idx, float* R_child,
                                  void* stream) {
  if (level < 0 || level >= kHopfMaxLevel || n < 0 || n > INT64_MAX / 8) return AHV_EINVAL;
  if (n > 0 && !all_set(parent_idx, child_idx, R_child)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_so3_hopf_children(level, parent_idx, n, child_idx, R_child, (cudaStream_t)stream);
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
  const Scored p{vol_src, AHV_VOL_F32, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return launch_score_bwd(p, tgt_feat, grad_scores, grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, (cudaStream_t)stream);
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
  const Scored p{vol_src, AHV_VOL_F32, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return launch_score_bwd(p, tgt_feat, grad_scores, grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, (cudaStream_t)stream,
                          h1_saved, pair_inv_scale, grad_R);
}

AHV_API size_t ahv_score_backward_det_workspace_bytes(int B, int64_t N, int r_per_pair, int want_grad_R) {
  if (B < 0 || !n_ok(N)) return 0;
  return bytes_of<DetBwdWs>(B, N, want_grad_R && !r_per_pair);
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
  Carve c(workspace);
  const DetBwdWs w(c, B, N, grad_R && !r_per_pair);
  if ((int64_t)B * N > 0 && (!workspace || workspace_bytes < c.off)) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  const Scored p{vol_src, AHV_VOL_F32, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return launch_score_bwd_det(p, tgt_feat, grad_scores, h1_saved, pair_inv_scale, grad_vol, grad_tgt, grad_W1, grad_W2,
                              grad_b2, grad_R, h1_saved && math_mode == AHV_MATH_TC, w, (cudaStream_t)stream);
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
  if ((int64_t)B * N == 0) return AHV_OK;
  if (workspace_bytes < bytes_of<TcScratch>(B)) return AHV_EWORKSPACE;
  Carve c(workspace);
  const Scored p{vol_src, AHV_VOL_F32, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return launch_score_tc_train(p, tgt_feat, scores, h1_saved, pair_inv_scale, TcScratch(c, B), (cudaStream_t)stream);
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
  const Scored p{vol_src, AHV_VOL_F32, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  if (math_mode == AHV_MATH_TC)
    return launch_score_bwd_tc(p, tgt_feat, grad_scores, h1_saved, pair_inv_scale, grad_vol, grad_tgt, grad_W1, grad_W2,
                               grad_b2, (cudaStream_t)stream);
  return launch_score_bwd(p, tgt_feat, grad_scores, grad_vol, grad_tgt, grad_W1, grad_W2, grad_b2, (cudaStream_t)stream,
                          h1_saved, pair_inv_scale);
}

AHV_API int ahv_forward_3d2d(const float* vol, const float* W1, const float* W2, const float* b2,
                     float* feat, int64_t m, void* stream) {
  if (m < 0 || (m > 0 && (!vol || !W1 || !W2 || !b2 || !feat))) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_forward_3d2d(vol, W1, W2, b2, feat, m, (cudaStream_t)stream);
}

AHV_API size_t ahv_workspace_bytes(int B, int64_t N, int k) {
  return B < 0 || N < 0 ? 0 : VerifyWs(nullptr, B, N, k).total;
}

AHV_API int ahv_verify_screen_stats(const void* workspace, int B, int64_t N, int* is_screened, int* flagged_pairs,
                                    int* contenders, float* max_err) {
  if (B < 0 || !n_ok(N) || !is_screened) return AHV_EINVAL;
  const VerifyWs w(const_cast<void*>(workspace), B, N, 1);
  *is_screened = screened(w, AHV_VOL_F32, AHV_MATH_TC, nullptr, 1, B, N);
  if (!*is_screened || (!flagged_pairs && !contenders && !max_err)) return AHV_OK;
  if (!workspace) return AHV_EINVAL;
  const ScreenLists& L = w.screen;
  if (flagged_pairs) AHV_CUDA_OK(cudaMemcpy(flagged_pairs, L.flagged, sizeof(int), cudaMemcpyDeviceToHost));
  if (contenders) AHV_CUDA_OK(cudaMemcpy(contenders, L.count, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost));
  if (max_err) AHV_CUDA_OK(cudaMemcpy(max_err, L.err, (size_t)B * sizeof(float), cudaMemcpyDeviceToHost));
  return AHV_OK;
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
  if (!workspace || workspace_bytes < VerifyWs(nullptr, B, N, k).score_bytes) return AHV_EWORKSPACE;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return score_chain(p, tgt_feat, scores, topk_val, topk_idx, k, idx_offset, math_mode, workspace, (cudaStream_t)stream);
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
  if (!workspace || workspace_bytes < VerifyWs(nullptr, B, N, k).total) return AHV_EWORKSPACE;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return verify_chain(p, vol_tgt, scores, topk_val, topk_idx, R_best, k, idx_offset, math_mode, workspace,
                      (cudaStream_t)stream, nullptr);
}

// ---- two-pass selection: dense set -> top-k -> local refinement (BASELINE config 4; extension) -----------
AHV_API size_t ahv_refine_workspace_bytes(int B, int64_t N, int k, int m) {
  return B < 0 || N < 0 || !k_ok(k) || m < 1 ? 0 : RefineWs(nullptr, B, N, k, m).total;
}

AHV_API int ahv_refine(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                       const float* W1, const float* W2, const float* b2, const float* base, int k, int m,
                       float max_angle_deg, uint64_t seed, float* first_val, int64_t* first_idx, float* first_R,
                       float* cand, float* best_val, int64_t* best_idx, float* R_best, int B, int64_t N,
                       int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 1 || N < 1 || !k_ok(k) || k > N || m < 1 || !n_ok((int64_t)k * m)) return AHV_EINVAL;
  if (!all_set(first_val, first_idx, first_R, cand, best_val, best_idx, workspace)) return AHV_EINVAL;
  if (!aligned16(cand)) return AHV_EINVAL;
  const RefineWs w(workspace, B, N, k, m);
  if (workspace_bytes < w.total) return AHV_EWORKSPACE;
  if (!n_ok(N) || !vol_dtype_ok(vol_dtype) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if (!all_set(vol_src, vol_tgt, R, W1, W2, b2, base)) return AHV_EINVAL;
  if (!all_aligned16(vol_src, vol_tgt, R, W1, W2, workspace)) return AHV_EINVAL;
  if (!(max_angle_deg >= 0.0f) || max_angle_deg > 180.0f) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  cudaStream_t s = (cudaStream_t)stream;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  // pass 1: the whole set, top-k and their rotations
  st = verify_chain(p, vol_tgt, nullptr, first_val, first_idx, first_R, k, 0, math_mode, w.grid, s, nullptr);
  if (st != AHV_OK) return st;
  // candidates: m rotations within max_angle_deg of each of the B*k winners (index 0 = the winner itself)
  st = launch_so3_perturb(first_R, (int64_t)B * k, m, max_angle_deg, seed, cand, s);
  if (st != AHV_OK) return st;
  // pass 2: per-pair candidate sets [B, k*m], arg-max
  return verify_chain(p.with_R(cand, true, (int64_t)k * m), vol_tgt, nullptr, best_val, best_idx, R_best, 1, 0, math_mode,
                      w.cand, s, nullptr);
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
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R_init, true, B, K};
  return launch_gradient_ascent(p, tgt_feat, steps, step_deg, R_out, score_out, (cudaStream_t)stream);
}

AHV_API size_t ahv_refine_gradient_workspace_bytes(int B, int64_t N, int k) {
  return B < 0 || N < 0 || !k_ok(k) ? 0 : ShardedRefineWs(nullptr, B, N, k, 1).total;
}

namespace {
bool min_sep_ok(float min_sep_deg) { return std::isfinite(min_sep_deg) && min_sep_deg >= 0.0f && min_sep_deg <= 180.0f; }

// the argument rules of the gradient-refinement entries (min_sep_deg == 0: ahv_refine_gradient's plain top-k)
bool refine_gradient_args_ok(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, const float* W1,
                             const float* W2, const float* b2, const float* base, int k, int steps, float step_deg,
                             float min_sep_deg, const float* first_val, const int64_t* first_idx, const float* first_R,
                             const float* R_all, const float* score_all, const float* best_val, const int64_t* best_idx,
                             const float* R_best, int B, int64_t N, int math_mode, const void* workspace) {
  if (B < 1 || N < 1 || !n_ok(N) || !k_ok(k) || k > N) return false;
  if (!ascent_args_ok(vol_dtype, steps, step_deg) || !min_sep_ok(min_sep_deg) || !math_mode_ok(math_mode)) return false;
  return all_set(vol_src, vol_tgt, R, W1, W2, b2, base, first_val, first_idx, first_R, R_all, score_all, best_val, best_idx,
                 workspace) &&
         all_aligned16(vol_src, vol_tgt, R, W1, W2, first_R, R_all, R_best, workspace);
}
}  // namespace

AHV_API int ahv_refine_gradient(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R, int r_per_pair,
                                const float* W1, const float* W2, const float* b2, const float* base, int k, int steps,
                                float step_deg, float* first_val, int64_t* first_idx, float* first_R, float* R_all,
                                float* score_all, float* best_val, int64_t* best_idx, float* R_best, int B, int64_t N,
                                int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (!refine_gradient_args_ok(vol_src, vol_dtype, vol_tgt, R, W1, W2, b2, base, k, steps, step_deg, 0.0f, first_val, first_idx,
                               first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math_mode, workspace))
    return AHV_EINVAL;
  if (workspace_bytes < ShardedRefineWs(nullptr, B, N, k, 1).total) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return refine_gradient_chain(p, vol_tgt, k, steps, step_deg, 0.0f, first_val, first_idx, first_R, R_all, score_all, best_val,
                               best_idx, R_best, math_mode, workspace, (cudaStream_t)stream, nullptr, 0);
}

AHV_API int ahv_refine_gradient_distinct(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                                         int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
                                         int k, int steps, float step_deg, float min_sep_deg, float* first_val,
                                         int64_t* first_idx, float* first_R, float* R_all, float* score_all, float* best_val,
                                         int64_t* best_idx, float* R_best, int B, int64_t N, int math_mode, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  if (!refine_gradient_args_ok(vol_src, vol_dtype, vol_tgt, R, W1, W2, b2, base, k, steps, step_deg, min_sep_deg, first_val,
                               first_idx, first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math_mode, workspace))
    return AHV_EINVAL;
  if (workspace_bytes < ShardedRefineWs(nullptr, B, N, k, 1).total) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return refine_gradient_chain(p, vol_tgt, k, steps, step_deg, min_sep_deg, first_val, first_idx, first_R, R_all, score_all,
                               best_val, best_idx, R_best, math_mode, workspace, (cudaStream_t)stream, nullptr, 0);
}

// ---- coarse-to-fine search on the nested Hopf grid (extension) --------------------------------------------
namespace {
constexpr int kHopfMaxBaseLevel = 6;

// the result of a search of zero levels: the base level's
int copy_base_level(const float* first_val, const int64_t* first_idx, const float* first_R, float* val, int64_t* idx,
                    float* R_out, int B, int k, cudaStream_t s) {
  AHV_CUDA_OK(cudaMemcpyAsync(val, first_val, (size_t)B * k * sizeof(float), cudaMemcpyDeviceToDevice, s));
  AHV_CUDA_OK(cudaMemcpyAsync(idx, first_idx, (size_t)B * k * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
  AHV_CUDA_OK(cudaMemcpyAsync(R_out, first_R, (size_t)B * k * 9 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return AHV_OK;
}

// ahv_search_hierarchical: [scoring workspace of the larger pass | target features B*32*64 fp32 | base grid n0*9 fp32
//  | children [B,8k] int64 | their rotations [B,8k,9] fp32 | a level's top-k [B,k] fp32 and int64 | parents [B,k] int64]
struct HierWs {
  float *tgt, *grid;
  int64_t* kids;
  float *kids_R, *lval;
  int64_t *lidx, *par;
  size_t total;
  HierWs(void* ws, int B, int base_level, int k) {
    Carve c(ws);
    c.take<unsigned char>(std::max(VerifyWs(nullptr, B, hopf_cells(base_level), k).score_bytes,
                                   VerifyWs(nullptr, B, 8 * (int64_t)k, k).score_bytes), 256);
    tgt = c.take<float>((size_t)B * kO * kP, 256);
    grid = c.take<float>((size_t)hopf_cells(base_level) * 9, 256);
    kids = c.take<int64_t>((size_t)B * 8 * k, 256);
    kids_R = c.take<float>((size_t)B * 8 * k * 9, 256);
    lval = c.take<float>((size_t)B * k, 256);
    lidx = c.take<int64_t>((size_t)B * k, 256);
    par = c.take<int64_t>((size_t)B * k, 256);
    total = c.off;
  }
};
}  // namespace

AHV_API size_t ahv_search_hierarchical_workspace_bytes(int B, int base_level, int k) {
  return B < 1 || base_level < 0 || base_level > kHopfMaxBaseLevel || !k_ok(k) ? 0 : HierWs(nullptr, B, base_level, k).total;
}

AHV_API int ahv_search_hierarchical(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* W1, const float* W2,
                                    const float* b2, const float* base, int base_level, int levels, int k, float* first_val,
                                    int64_t* first_idx, float* first_R, float* val, int64_t* idx, float* R_out, int B,
                                    int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 1 || !k_ok(k) || !vol_dtype_ok(vol_dtype) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if (base_level < 0 || base_level > kHopfMaxBaseLevel || levels < 0 || base_level + levels > kHopfMaxLevel) return AHV_EINVAL;
  if (!all_set(vol_src, vol_tgt, W1, W2, b2, base, first_val, first_idx, first_R, val, idx, R_out, workspace))
    return AHV_EINVAL;
  if (!all_aligned16(vol_src, vol_tgt, W1, W2, first_R, R_out, workspace)) return AHV_EINVAL;
  const HierWs w(workspace, B, base_level, k);
  if (workspace_bytes < w.total) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n0 = hopf_cells(base_level), nc = 8 * (int64_t)k;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, w.grid, false, B, n0};
  st = launch_forward_3d2d(vol_tgt, W1, W2, b2, w.tgt, B, s);
  if (st == AHV_OK) st = launch_so3_hopf_grid(base_level, 0, w.grid, n0, s);
  // the base level: one set shared by the B pairs; its local indices are grid indices
  if (st == AHV_OK) st = score_chain(p, w.tgt, nullptr, first_val, first_idx, k, 0, math_mode, workspace, s);
  if (st == AHV_OK) st = launch_gather_rotations(w.grid, 0, first_idx, 0, B, n0, k, first_R, s);
  if (st != AHV_OK) return st;
  if (levels == 0) return copy_base_level(first_val, first_idx, first_R, val, idx, R_out, B, k, s);
  // Each level scores the 8 children of the pair's k cells, the cells taken in ascending index order.  The candidate
  // list then ascends in grid index (the children of cell i are 8i .. 8i+7), so the top-k's tie rule (lowest local
  // index) is the lowest grid index.
  st = launch_hopf_pick(nullptr, 0, first_idx, B, k, true, w.par, s);
  for (int l = 0; l < levels && st == AHV_OK; ++l) {
    const bool last = l == levels - 1;
    st = launch_so3_hopf_children(base_level + l, w.par, (int64_t)B * k, w.kids, w.kids_R, s);
    if (st == AHV_OK)
      st = score_chain(p.with_R(w.kids_R, true, nc), w.tgt, nullptr, last ? val : w.lval, w.lidx, k, 0, math_mode, workspace,
                       s);
    if (st == AHV_OK) st = launch_hopf_pick(w.kids, nc, w.lidx, B, k, !last, last ? idx : w.par, s);
  }
  if (st != AHV_OK) return st;
  return launch_gather_rotations(w.kids_R, 1, w.lidx, 0, B, nc, k, R_out, s);
}

// ---- coarse-to-fine search that keeps k distinct modes (extension) ------------------------------------------------
namespace {
constexpr int kMaxBeam = 8;

// ahv_search_modes: [scoring workspace of the larger pass | target features B*32*64 fp32 | base grid n0*9 fp32 | base
//  slots B*n0 bytes | children [B,8kw] int64 | their rotations [B,8kw,9] fp32 | beams [B,k,w] int64 | the beams for the
//  children generator [B,k,w] int64].  `scores`, the scoring workspace's score region, holds the base scores until the
//  first level.
struct ModesWs {
  float *scores, *tgt, *grid;
  uint8_t* slot;
  int64_t* kids;
  float* kids_R;
  int64_t *par, *gen;
  size_t total;
  ModesWs(void* ws, int B, int base_level, int k, int w) {
    const int64_t n0 = hopf_cells(base_level), nc = 8 * (int64_t)k * w;
    Carve c(ws);
    scores = VerifyWs(ws, B, n0, 0).scores;
    c.take<unsigned char>(std::max(VerifyWs(nullptr, B, n0, 0).score_bytes, VerifyWs(nullptr, B, nc, 0).score_bytes), 256);
    tgt = c.take<float>((size_t)B * kO * kP, 256);
    grid = c.take<float>((size_t)n0 * 9, 256);
    slot = c.take<uint8_t>((size_t)B * n0, 256);
    kids = c.take<int64_t>((size_t)B * nc, 256);
    kids_R = c.take<float>((size_t)B * nc * 9, 256);
    par = c.take<int64_t>((size_t)B * k * w, 256);
    gen = c.take<int64_t>((size_t)B * k * w, 256);
    total = c.off;
  }
};

bool modes_sizes_ok(int B, int base_level, int k, int beam) {
  return B >= 1 && base_level >= 0 && base_level <= kHopfMaxBaseLevel && k_ok(k) && beam >= 1 && beam <= kMaxBeam;
}
}  // namespace

AHV_API size_t ahv_search_modes_workspace_bytes(int B, int base_level, int k, int beam) {
  return modes_sizes_ok(B, base_level, k, beam) ? ModesWs(nullptr, B, base_level, k, beam).total : 0;
}

AHV_API int ahv_search_modes(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* W1, const float* W2,
                             const float* b2, const float* base, int base_level, int levels, int k, int beam, float min_sep_deg,
                             float* first_val, int64_t* first_idx, float* first_R, float* val, int64_t* idx, float* R_out, int B,
                             int math_mode, void* workspace, size_t workspace_bytes, void* stream) {
  if (!modes_sizes_ok(B, base_level, k, beam) || !vol_dtype_ok(vol_dtype) || !math_mode_ok(math_mode)) return AHV_EINVAL;
  if (levels < 0 || base_level + levels > kHopfMaxLevel) return AHV_EINVAL;
  if (!std::isfinite(min_sep_deg) || !(min_sep_deg > 0.0f) || min_sep_deg > 180.0f) return AHV_EINVAL;
  if (!all_set(vol_src, vol_tgt, W1, W2, b2, base, first_val, first_idx, first_R, val, idx, R_out, workspace))
    return AHV_EINVAL;
  if (!all_aligned16(vol_src, vol_tgt, W1, W2, first_R, R_out, workspace)) return AHV_EINVAL;
  const ModesWs w(workspace, B, base_level, k, beam);
  if (workspace_bytes < w.total) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n0 = hopf_cells(base_level), nc = 8 * (int64_t)k * beam;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, w.grid, false, B, n0};
  st = launch_forward_3d2d(vol_tgt, W1, W2, b2, w.tgt, B, s);
  if (st == AHV_OK) st = launch_so3_hopf_grid(base_level, 0, w.grid, n0, s);
  // the base level (one set shared by the B pairs; local indices are grid indices) and its k distinct winners
  if (st == AHV_OK) st = score_chain(p, w.tgt, nullptr, nullptr, nullptr, 0, 0, math_mode, workspace, s);
  if (st == AHV_OK) st = launch_topk_distinct(w.scores, w.grid, 0, B, n0, k, min_sep_deg, first_val, first_idx, first_R, s);
  if (st != AHV_OK) return st;
  if (levels == 0) return copy_base_level(first_val, first_idx, first_R, val, idx, R_out, B, k, s);
  st = launch_modes_beams(w.scores, w.grid, n0, first_idx, first_R, B, k, beam, min_sep_deg, w.slot, w.par, w.gen, s);
  // each level scores the children of every beam as a per-pair set [B, 8kw] and keeps each slot's top-w
  for (int l = 0; l < levels && st == AHV_OK; ++l) {
    st = launch_so3_hopf_children(base_level + l, w.gen, (int64_t)B * k * beam, w.kids, w.kids_R, s);
    if (st == AHV_OK)
      st = score_chain(p.with_R(w.kids_R, true, nc), w.tgt, nullptr, nullptr, nullptr, 0, 0, math_mode, workspace, s);
    if (st == AHV_OK)
      st = launch_modes_level(w.scores, w.kids, w.kids_R, B, k, beam, l == levels - 1, w.par, w.gen, val, idx, R_out, s);
  }
  return st;
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

// ---- posterior mass of the selected rotations under the verifier's softmax (extension) -------------------
namespace {
bool posterior_sizes_ok(int B, int64_t N, int k) { return B >= 0 && N >= 1 && n_ok(N) && k >= 0 && k <= kMaxK; }
}  // namespace

AHV_API size_t ahv_posterior_mass_workspace_bytes(int B, int64_t N, int k) {
  return posterior_sizes_ok(B, N, k) ? posterior_workspace_bytes(B, N, k, false) : 0;
}

AHV_API int ahv_posterior_mass(const float* scores, const float* R, int r_per_pair, const float* centers, int B, int64_t N,
                               int k, float radius_deg, float temperature, float* log_z, float* mass, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!posterior_sizes_ok(B, N, k) || !min_sep_ok(radius_deg)) return AHV_EINVAL;
  if (!std::isfinite(temperature) || !(temperature > 0.0f)) return AHV_EINVAL;
  if (B > 0 && !all_set(scores, R, log_z, workspace)) return AHV_EINVAL;
  if (k > 0 ? (B > 0 && !all_set(centers, mass)) : (centers || mass)) return AHV_EINVAL;  // k == 0: log_z alone
  if (!all_aligned16(R, centers, workspace)) return AHV_EINVAL;
  if (B > 0 && workspace_bytes < posterior_workspace_bytes(B, N, k, false)) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_posterior(scores, R, r_per_pair != 0, centers, B, N, k, radius_deg, temperature, log_z, mass, nullptr,
                          nullptr, nullptr, workspace, (cudaStream_t)stream);
}

// ---- first moment of the posterior over each slot: mean rotation and spread (extension) ------------------
AHV_API size_t ahv_posterior_moments_workspace_bytes(int B, int64_t N, int k) {
  return posterior_sizes_ok(B, N, k) && k_ok(k) ? posterior_workspace_bytes(B, N, k, true) : 0;
}

AHV_API int ahv_posterior_moments(const float* scores, const float* R, int r_per_pair, const float* centers, int B,
                                  int64_t N, int k, float radius_deg, float temperature, float* log_z, float* mass,
                                  float* mean_R, float* mean_cos, float* moment, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  if (!posterior_sizes_ok(B, N, k) || !k_ok(k) || !min_sep_ok(radius_deg)) return AHV_EINVAL;
  if (!std::isfinite(temperature) || !(temperature > 0.0f)) return AHV_EINVAL;
  if (B > 0 && !all_set(scores, R, centers, log_z, mass, mean_R, mean_cos, moment, workspace)) return AHV_EINVAL;
  if (!all_aligned16(R, centers, workspace)) return AHV_EINVAL;
  if (B > 0 && workspace_bytes < posterior_workspace_bytes(B, N, k, true)) return AHV_EWORKSPACE;
  int st = check_device();
  if (st != AHV_OK) return st;
  return launch_posterior(scores, R, r_per_pair != 0, centers, B, N, k, radius_deg, temperature, log_z, mass, mean_R,
                          mean_cos, moment, workspace, (cudaStream_t)stream);
}

// ---- hypothesis set sharded over the GPUs of one node: winners exchanged through peer memory -------------
AHV_API size_t ahv_peer_bytes(int max_pairs, int max_k) {
  return (max_pairs < 1 || !k_ok(max_k)) ? 0 : peer::buffer_bytes(max_pairs, max_k);
}

AHV_API size_t ahv_peer_bytes_ex(int max_pairs, int max_k, int64_t max_hyps) {
  return (max_pairs < 1 || !k_ok(max_k) || !n_ok(max_hyps)) ? 0 : peer::buffer_bytes_ex(max_pairs, max_k, max_hyps);
}

AHV_API int ahv_peer_alloc_ex(int max_pairs, int max_k, int64_t max_hyps, void** ptr) {
  if (!ptr || max_pairs < 1 || !k_ok(max_k) || !n_ok(max_hyps)) return AHV_EINVAL;
  int st = check_device();
  if (st != AHV_OK) return st;
  st = preload_exchange_kernels();
  if (st != AHV_OK) return st;
  const size_t bytes = peer::buffer_bytes_ex(max_pairs, max_k, max_hyps);
  if (cudaMalloc(ptr, bytes) != cudaSuccess) return AHV_ECUDA;
  const uint32_t hdr[4] = {0u, 0u, (uint32_t)max_pairs, (uint32_t)max_k};  // seq, err, capacity (cap_hyps below)
  const uint32_t cap_hyps = (uint32_t)max_hyps;
  if (cudaMemset(*ptr, 0, bytes) != cudaSuccess || cudaMemcpy(*ptr, hdr, sizeof(hdr), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(static_cast<uint32_t*>(*ptr) + peer::kHdrCapHyps, &cap_hyps, sizeof(cap_hyps), cudaMemcpyHostToDevice) !=
          cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess) {
    cudaFree(*ptr);
    *ptr = nullptr;
    return AHV_ECUDA;
  }
  return AHV_OK;
}

AHV_API int ahv_peer_alloc(int max_pairs, int max_k, void** ptr) { return ahv_peer_alloc_ex(max_pairs, max_k, 0, ptr); }

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

AHV_API int ahv_peer_capacity_ex(const void* buf, int* max_pairs, int* max_k, int64_t* max_hyps) {
  if (!buf || !max_pairs || !max_k || !max_hyps) return AHV_EINVAL;
  unsigned hdr[5];
  if (cudaMemcpy(hdr, buf, sizeof(hdr), cudaMemcpyDeviceToHost) != cudaSuccess) return AHV_ECUDA;  // synchronises
  *max_pairs = (int)hdr[2];
  *max_k = (int)hdr[3];
  *max_hyps = (int64_t)hdr[peer::kHdrCapHyps];
  return AHV_OK;
}

AHV_API int ahv_peer_close(void* ptr) { return (!ptr || cudaIpcCloseMemHandle(ptr) == cudaSuccess) ? AHV_OK : AHV_ECUDA; }

namespace {
// The group an entry is given: one GPU (world 1, rank 0), or peer::Args::valid.
int make_peer_args(int rank, int world, void* const* peers, int peer_max_pairs, int peer_max_k, peer::Args* pa) {
  pa->rank = rank;
  pa->world = world;
  pa->cap_pairs = peer_max_pairs;
  pa->cap_k = peer_max_k;
  if (world == 1) return rank == 0 ? AHV_OK : AHV_EINVAL;
  if (peers && world <= peer::kMaxPeers)
    for (int r = 0; r < world; ++r) pa->bufs[r] = static_cast<unsigned char*>(peers[r]);
  return pa->valid() ? AHV_OK : AHV_EINVAL;
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
  if (world > 1 && !pa.fits(B, k)) return AHV_EINVAL;
  st = check_device();
  if (st != AHV_OK) return st;
  if (world == 1 && N == 0) return AHV_EINVAL;
  if (!workspace || workspace_bytes < VerifyWs(nullptr, B, N, k).total) return AHV_EWORKSPACE;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return verify_chain(p, vol_tgt, nullptr, topk_val, topk_idx, R_best, k, idx_offset, math_mode, workspace,
                      (cudaStream_t)stream, &pa);
}

AHV_API int ahv_scores_exchange(const float* part, int B, int64_t N, float* scores, int rank, int world, void* const* peers,
                                int peer_max_pairs, int peer_max_k, int64_t peer_max_hyps, void* stream) {
  if (B < 1 || N < 1 || !n_ok(N) || !scores) return AHV_EINVAL;
  peer::Args pa;
  int st = make_peer_args(rank, world, peers, peer_max_pairs, peer_max_k, &pa);
  if (st != AHV_OK) return st;
  if (world < 2 || !n_ok(peer_max_hyps) || !pa.fits(B, 0, N, peer_max_hyps)) return AHV_EINVAL;
  int64_t lo, hi;
  peer::shard_bounds(N, rank, world, &lo, &hi);
  if (hi > lo && !part) return AHV_EINVAL;
  st = check_device();
  if (st != AHV_OK) return st;
  return launch_scores_exchange(part, B, N, scores, pa, peer_max_hyps, (cudaStream_t)stream);
}

AHV_API size_t ahv_refine_gradient_sharded_workspace_bytes(int B, int64_t N, int k, int world) {
  if (B < 0 || N < 0 || !k_ok(k) || world < 1 || world > peer::kMaxPeers) return 0;
  return ShardedRefineWs(nullptr, B, N, k, world).total;
}

AHV_API int ahv_refine_gradient_sharded(const void* vol_src, int vol_dtype, const float* vol_tgt, const float* R,
                                        int r_per_pair, const float* W1, const float* W2, const float* b2, const float* base,
                                        int k, int steps, float step_deg, float min_sep_deg, float* first_val,
                                        int64_t* first_idx, float* first_R, float* R_all, float* score_all, float* best_val,
                                        int64_t* best_idx, float* R_best, int B, int64_t N, int math_mode, void* workspace,
                                        size_t workspace_bytes, int rank, int world, void* const* peers, int peer_max_pairs,
                                        int peer_max_k, int64_t peer_max_hyps, void* stream) {
  if (!refine_gradient_args_ok(vol_src, vol_dtype, vol_tgt, R, W1, W2, b2, base, k, steps, step_deg, min_sep_deg, first_val,
                               first_idx, first_R, R_all, score_all, best_val, best_idx, R_best, B, N, math_mode, workspace))
    return AHV_EINVAL;
  peer::Args pa;
  int st = make_peer_args(rank, world, peers, peer_max_pairs, peer_max_k, &pa);
  if (st != AHV_OK) return st;
  const int64_t hyps = min_sep_deg > 0.0f ? N : 0;  // the slot gather's entries; distinct winners: the score region too
  if (world > 1 && (!pa.fits(B, k, hyps, peer_max_hyps) || (hyps > 0 && !n_ok(peer_max_hyps)))) return AHV_EINVAL;
  if (workspace_bytes < ShardedRefineWs(nullptr, B, N, k, world).total) return AHV_EWORKSPACE;
  st = check_device();
  if (st != AHV_OK) return st;
  const Scored p{vol_src, vol_dtype, W1, W2, b2, base, R, r_per_pair != 0, B, N};
  return refine_gradient_chain(p, vol_tgt, k, steps, step_deg, min_sep_deg, first_val, first_idx, first_R, R_all, score_all,
                               best_val, best_idx, R_best, math_mode, workspace, (cudaStream_t)stream, &pa, peer_max_hyps);
}

// ---- host-buffer entries -------------------------------------------------------------------------------
// A session owns the device scratch of the host-buffer entry, grown on demand and reused across calls
// (explicit caller-owned state; nothing process-global is touched).
struct ahv_host_session {
  unsigned char* d = nullptr;
  size_t bytes = 0;
  int device = -1;
};

// The device block of a host-buffer call: [source volumes | target volumes | rotations | W1, W2, b2 and base (8 floats) |
// top-k indices, values and rotations | verification workspace]
struct HostBlock {
  void* src;
  float *tgt, *R, *W1;  // W1 [32,384], then W2 [32,32], b2 [32] and base [8]
  int64_t* idx;
  float *val, *R_best;
  void* ws;
  size_t ws_bytes, total;
  HostBlock(void* p, size_t src_b, size_t tgt_b, size_t r_b, int B, int64_t N, int k) {
    Carve c(p);
    src = c.take<unsigned char>(src_b, 256);
    tgt = c.take<float>(tgt_b / sizeof(float), 256);
    R = c.take<float>(r_b / sizeof(float), 256);
    W1 = c.take<float>(kO * kK + kO * kO + kO + 8, 256);
    Carve out(c.take<unsigned char>((size_t)B * k * (sizeof(int64_t) + sizeof(float) + 9 * sizeof(float)), 256));
    idx = out.take<int64_t>((size_t)B * k, 1);
    val = out.take<float>((size_t)B * k, 1);
    R_best = out.take<float>((size_t)B * k * 9, 1);
    ws_bytes = VerifyWs(nullptr, B, N, k).total;
    ws = c.take<unsigned char>(ws_bytes, 1);
    total = c.off;
  }
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
  const HostBlock nb(nullptr, src_b, tgt_b, r_b, B, N, k);
  if (session->bytes < nb.total) {  // grow (rare): the stream may still use the old block
    if (cudaStreamSynchronize(s) != cudaSuccess) return AHV_ECUDA;
    if (session->d && cudaFree(session->d) != cudaSuccess) return AHV_ECUDA;
    session->d = nullptr;
    session->bytes = 0;
    if (cudaMalloc((void**)&session->d, nb.total) != cudaSuccess) return AHV_ECUDA;
    session->bytes = nb.total;
  }
  const HostBlock d(session->d, src_b, tgt_b, r_b, B, N, k);
  float* d_W1 = d.W1; float* d_W2 = d_W1 + kO * kK; float* d_b2 = d_W2 + kO * kO; float* d_base = d_b2 + kO;
  st = AHV_ECUDA;
  do {
    if (cudaMemcpyAsync(d.src, vol_src_host, src_b, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d.tgt, vol_tgt_host, tgt_b, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d.R, R_host, r_b, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_W1, W1_host, kO * kK * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_W2, W2_host, kO * kO * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_b2, b2_host, kO * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(d_base, base_host, 8 * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) break;
    if (world > 1)
      st = ahv_verify_sharded(d.src, vol_dtype, d.tgt, d.R, r_per_pair, d_W1, d_W2, d_b2, d_base, d.val, d.idx, d.R_best, k,
                              idx_offset, B, N, math_mode, d.ws, d.ws_bytes, rank, world, peers, peer_max_pairs, peer_max_k,
                              stream);
    else
      st = ahv_verify(d.src, vol_dtype, d.tgt, d.R, r_per_pair, d_W1, d_W2, d_b2, d_base,
                      scores_host ? (float*)d.ws : nullptr, d.val, d.idx, d.R_best, k, idx_offset, B, N, math_mode, d.ws, d.ws_bytes,
                      stream);
    if (st != AHV_OK) break;
    st = AHV_ECUDA;
    if (scores_host &&
        cudaMemcpyAsync(scores_host, d.ws, (size_t)B * N * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess)
      break;
    if (cudaMemcpyAsync(topk_idx_host, d.idx, (size_t)B * k * 8, cudaMemcpyDeviceToHost, s) != cudaSuccess) break;
    if (cudaMemcpyAsync(topk_val_host, d.val, (size_t)B * k * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess) break;
    if (R_best_host &&
        cudaMemcpyAsync(R_best_host, d.R_best, (size_t)B * k * 36, cudaMemcpyDeviceToHost, s) != cudaSuccess)
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
