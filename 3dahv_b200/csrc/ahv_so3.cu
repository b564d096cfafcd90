// SO(3) hypothesis generation.
//
// ahv_so3_from_normals: the arithmetic of pytorch3d.transforms.random_rotations
// (call sites modules/model.py:102,131,184; model_co3d.py:86; test_co3d.py:106)
// applied to caller-supplied Gaussian draws, every operation an individually
// rounded IEEE fp32 op (no FMA contraction) so the result is bit-identical to
// oracle/ahv_oracle.c:ahv_oracle_so3_from_normals.
//
// ahv_so3_sample: native counter-based sampler (extension, SURVEY.md §8f-4).
#include <algorithm>

#include "ahv_common.cuh"

namespace ahv {

__device__ __forceinline__ void quat_to_matrix_exact(float a, float b, float c, float d,
                                                     float* __restrict__ m) {
  // s = ((a*a + b*b) + c*c) + d*d, sequential like torch's sum over 4 elements
  float s = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c)),
                      __fmul_rn(d, d));
  float den = copysignf(__fsqrt_rn(s), a);
  float r = __fdiv_rn(a, den), i = __fdiv_rn(b, den), j = __fdiv_rn(c, den), k = __fdiv_rn(d, den);
  float qq = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(r, r), __fmul_rn(i, i)), __fmul_rn(j, j)),
                       __fmul_rn(k, k));
  float two_s = __fdiv_rn(2.0f, qq);
  float ii = __fmul_rn(i, i), jj = __fmul_rn(j, j), kk = __fmul_rn(k, k);
  float ij = __fmul_rn(i, j), ik = __fmul_rn(i, k), jk = __fmul_rn(j, k);
  float ir = __fmul_rn(i, r), jr = __fmul_rn(j, r), kr = __fmul_rn(k, r);
  m[0] = __fsub_rn(1.0f, __fmul_rn(two_s, __fadd_rn(jj, kk)));
  m[1] = __fmul_rn(two_s, __fsub_rn(ij, kr));
  m[2] = __fmul_rn(two_s, __fadd_rn(ik, jr));
  m[3] = __fmul_rn(two_s, __fadd_rn(ij, kr));
  m[4] = __fsub_rn(1.0f, __fmul_rn(two_s, __fadd_rn(ii, kk)));
  m[5] = __fmul_rn(two_s, __fsub_rn(jk, ir));
  m[6] = __fmul_rn(two_s, __fsub_rn(ik, jr));
  m[7] = __fmul_rn(two_s, __fadd_rn(jk, ir));
  m[8] = __fsub_rn(1.0f, __fmul_rn(two_s, __fadd_rn(ii, jj)));
}

__global__ void __launch_bounds__(256) so3_from_normals_kernel(const float4* __restrict__ normals,
                                                               float* __restrict__ R, int64_t n) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  float4 o = normals[t];
  float m[9];
  quat_to_matrix_exact(o.x, o.y, o.z, o.w, m);
#pragma unroll
  for (int e = 0; e < 9; ++e) R[t * 9 + e] = m[e];
}

// Philox-4x32-10 (Salmon et al. 2011), keyed by seed, counter = hypothesis index.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}

__global__ void __launch_bounds__(256) so3_sample_kernel(uint64_t seed, int64_t first,
                                                         float* __restrict__ R, int64_t n) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  uint64_t g = (uint64_t)(first + t);
  uint4 u = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), 0x3d41u, 0x4856u),
                          make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  // two Box-Muller pairs -> four standard normals; (u+0.5)/2^32 lies in (0,1)
  const float inv = 2.3283064365386963e-10f;
  float u0 = ((float)(u.x >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = (float)u.y * inv;
  float u2 = ((float)(u.z >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = (float)u.w * inv;
  float r0 = sqrtf(-2.0f * logf(u0)), r1 = sqrtf(-2.0f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.0f * u1, &s0, &c0);
  sincospif(2.0f * u3, &s1, &c1);
  float m[9];
  quat_to_matrix_exact(r0 * c0, r0 * s0, r1 * c1, r1 * s1, m);
#pragma unroll
  for (int e = 0; e < 9; ++e) R[t * 9 + e] = m[e];
}

// Deterministic near-uniform SO(3) grid: super-Fibonacci spiral (Alexa, CVPR 2022).  Point i of an
// n-point set: s=i+1/2, t=s/n, r=sqrt(t), rr=sqrt(1-t), a=2*pi*s/sqrt(2), b=2*pi*s/psi, psi=1.5337511687...
// q=(r sin a, r cos a, rr sin b, rr cos b) -> matrix by the same map as random_rotations.  Evaluated in fp64
// and rounded once to fp32 so the CPU restatement (oracle/ahv_oracle.c) reproduces it bit for bit.
__global__ void __launch_bounds__(256) so3_grid_kernel(int64_t n_total, int64_t first, float* __restrict__ R,
                                                       int64_t count) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const double s = (double)(first + t) + 0.5;
  const double u = s / (double)n_total;
  const double r = sqrt(u), rr = sqrt(1.0 - u);
  // reduce the angle to [0,1) turns before sinpi/cospi: exact in fp64 for these magnitudes
  double ta = s * 0.70710678118654752440, tb = s * 0.65199624317913454;  // s/sqrt(2), s/psi
  ta -= floor(ta);
  tb -= floor(tb);
  double sa, ca, sb, cb;
  sincospi(2.0 * ta, &sa, &ca);
  sincospi(2.0 * tb, &sb, &cb);
  float m[9];
  quat_to_matrix_exact((float)(r * sa), (float)(r * ca), (float)(rr * sb), (float)(rr * cb), m);
#pragma unroll
  for (int e = 0; e < 9; ++e) R[t * 9 + e] = m[e];
}

// Nested, equal-volume SO(3) grid: the Hopf fibration with HEALPix on S^2 in NESTED order and a regular grid on S^1
// (Yershova et al. 2010).  Level L: Nside = 2^L, 12*4^L pixels p, 6*2^L psi-intervals j with centres
// psi_j = 2*pi*(j + 1/2) / (6*2^L), 72*8^L cells.  Cell i = 6*p0 + j0 at level 0; the children of cell i are 8i + 2a + b,
// with a the HEALPix nested child digit (p' = 4p + a) and b the psi digit (j' = 2j + b), so they lie inside it.  Point:
// (theta, phi) = the HEALPix nested pix2ang centre of p (Gorski et al. 2005) and
// q = (cos(theta/2) cos(psi/2), cos(theta/2) sin(psi/2), sin(theta/2) cos(phi + psi/2), sin(theta/2) sin(phi + psi/2)),
// in fp64, rounded once to fp32, then the same quaternion -> matrix map as the other generators.  Restated in numpy
// (tests/hopf_oracle.py) and plain C (tests/hopf_oracle.c).
__device__ __forceinline__ int64_t even_bits(uint64_t x) {  // bits 0, 2, 4, ... of x, packed
  x &= 0x5555555555555555ull;
  x = (x | (x >> 1)) & 0x3333333333333333ull;
  x = (x | (x >> 2)) & 0x0f0f0f0f0f0f0f0full;
  x = (x | (x >> 4)) & 0x00ff00ff00ff00ffull;
  x = (x | (x >> 8)) & 0x0000ffff0000ffffull;
  x = (x | (x >> 16)) & 0x00000000ffffffffull;
  return (int64_t)x;
}

__device__ void hopf_rotation(int level, int64_t index, float* __restrict__ m) {
  int64_t p = (index >> (3 * level)) / 6, j = (index >> (3 * level)) % 6;
  for (int l = level - 1; l >= 0; --l) {
    const int d = (int)(index >> (3 * l)) & 7;
    p = 4 * p + (d >> 1);
    j = 2 * j + (d & 1);
  }
  // pix2ang, nested: face, then the bits of the in-face index de-interleaved, then the cap and equatorial formulas
  const int64_t nside = (int64_t)1 << level, npface = nside * nside;
  const int face = (int)(p >> (2 * level));
  const int64_t ipf = p & (npface - 1), ix = even_bits((uint64_t)ipf), iy = even_bits((uint64_t)ipf >> 1);
  const int64_t jr = (int64_t)(face / 4 + 2) * nside - ix - iy - 1;  // ring number, 1 .. 4*nside - 1
  const int jpll = 2 * (face % 4) + (face / 4 != 1);                  // 1 3 5 7 | 0 2 4 6 | 1 3 5 7
  int64_t nr;
  double c2, s2;  // cos^2(theta/2) = (1 + z)/2, sin^2(theta/2) = (1 - z)/2
  if (jr < nside) {
    nr = jr;
    const double t = (double)(nr * nr) / (3.0 * (double)npface);  // 1 - z
    s2 = 0.5 * t;
    c2 = 1.0 - 0.5 * t;
  } else if (jr > 3 * nside) {
    nr = 4 * nside - jr;
    const double t = (double)(nr * nr) / (3.0 * (double)npface);  // 1 + z
    c2 = 0.5 * t;
    s2 = 1.0 - 0.5 * t;
  } else {
    nr = nside;
    const double hz = (double)(2 * nside - jr) / (3.0 * (double)nside);  // z / 2
    c2 = 0.5 + hz;
    s2 = 0.5 - hz;
  }
  int64_t tp = jpll * nr + ix - iy;  // phi = pi * tp / (4 nr)
  if (tp < 0) tp += 8 * nr;
  const double h = (double)(2 * j + 1) / (3.0 * (double)(nside << 2));  // psi / 2 in units of pi
  double a = (double)tp / (4.0 * (double)nr) + h;                         // phi + psi / 2 in units of pi
  if (a >= 2.0) a -= 2.0;
  const double c = sqrt(c2), s = sqrt(s2);
  double sh, ch, sa, ca;
  sincospi(h, &sh, &ch);
  sincospi(a, &sa, &ca);
  quat_to_matrix_exact((float)(c * ch), (float)(c * sh), (float)(s * ca), (float)(s * sa), m);
}

__global__ void __launch_bounds__(256) so3_hopf_grid_kernel(int level, int64_t first, float* __restrict__ R, int64_t count) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += (int64_t)gridDim.x * blockDim.x) {
    float m[9];
    hopf_rotation(level, first + t, m);
#pragma unroll
    for (int e = 0; e < 9; ++e) R[t * 9 + e] = m[e];
  }
}

// child t of parent t/8: index 8 * parent + t % 8 at level + 1; a parent outside the level gives -1 and NaN
__global__ void __launch_bounds__(256) so3_hopf_children_kernel(int level, const int64_t* __restrict__ parent, int64_t n,
                                                                int64_t* __restrict__ child, float* __restrict__ R) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < 8 * n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = __ldg(parent + (t >> 3));
    float m[9];
    if (p >= 0 && p < hopf_cells(level)) {
      child[t] = 8 * p + (t & 7);
      hopf_rotation(level + 1, 8 * p + (t & 7), m);
    } else {
      child[t] = -1;
#pragma unroll
      for (int e = 0; e < 9; ++e) m[e] = __int_as_float(0x7fffffff);
    }
#pragma unroll
    for (int e = 0; e < 9; ++e) R[t * 9 + e] = m[e];
  }
}

// one warp per pair; the cells of a pair are distinct, so the rank of each among them is its sorted position
__global__ void __launch_bounds__(128) hopf_pick_kernel(const int64_t* __restrict__ cand, int64_t n,
                                                        const int64_t* __restrict__ pick, int B, int k, bool sort,
                                                        int64_t* __restrict__ out) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  int64_t v = -1;
  if (lane < k) {
    v = pick[(int64_t)b * k + lane];
    if (cand) v = (v >= 0 && v < n) ? cand[(int64_t)b * n + v] : -1;
  }
  int pos = lane;
  if (sort) {
    pos = 0;
    for (int i = 0; i < k; ++i) {
      const int64_t u = __shfl_sync(0xffffffffu, v, i);
      pos += (u < v) || (u == v && i < lane);
    }
  }
  if (lane < k) out[(int64_t)b * k + pos] = v;
}

// Local refinement set around given rotations (extension, BASELINE config 4 "top-k refinement pass"; the
// reference has no refinement): out[i,0] = center[i]; out[i,j>0] = dR(i,j) @ center[i] where dR is a Haar
// rotation (Philox counter i*m+j, same normal -> quaternion map as the sampler) whose rotation ANGLE theta in
// [0,pi] is rescaled to theta/pi * max_angle about the same axis.  Restated in oracle/ahv_oracle.c.
__global__ void __launch_bounds__(256) so3_perturb_kernel(const float* __restrict__ centers, int64_t n, int m,
                                                          float max_angle_rad, uint64_t seed, float* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * m) return;
  const int64_t i = t / m;
  const int j = (int)(t - i * m);
  float c[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) c[e] = __ldg(centers + i * 9 + e);
  float* o = out + t * 9;
  if (j == 0) {
#pragma unroll
    for (int e = 0; e < 9; ++e) o[e] = c[e];
    return;
  }
  const uint4 u = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)((uint64_t)t >> 32), 0x7065u, 0x7274u),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float inv32 = 2.3283064365386963e-10f;
  const float u0 = ((float)(u.x >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = (float)u.y * inv32;
  const float u2 = ((float)(u.z >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = (float)u.w * inv32;
  const float r0 = sqrtf(-2.0f * logf(u0)), r1 = sqrtf(-2.0f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.0f * u1, &s0, &c0);
  sincospif(2.0f * u3, &s1, &c1);
  const float qa = r0 * c0, qb = r0 * s0, qc = r1 * c1, qd = r1 * s1;  // Haar quaternion, unnormalised
  const float vn = sqrtf(qb * qb + qc * qc + qd * qd);
  const float theta = 2.0f * atan2f(vn, fabsf(qa));                    // rotation angle in [0, pi]
  const float phi = theta * (max_angle_rad * 0.318309886183790672f);   // rescaled into the cone
  float sh, ch;
  sincosf(0.5f * phi, &sh, &ch);
  const float k = vn > 0.0f ? sh / vn : 0.0f;
  float d[9];
  quat_to_matrix_exact(ch, k * qb, k * qc, k * qd, d);
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int q = 0; q < 3; ++q)
      o[r * 3 + q] = fmaf(d[r * 3 + 2], c[6 + q], fmaf(d[r * 3 + 1], c[3 + q], d[r * 3] * c[q]));
}

int launch_so3_perturb(const float* centers, int64_t n, int m, float max_angle_deg, uint64_t seed, float* out,
                       cudaStream_t s) {
  if (n * m == 0) return AHV_OK;
  so3_perturb_kernel<<<(unsigned)((n * m + 255) / 256), 256, 0, s>>>(centers, n, m, max_angle_deg * 0.017453292519943295f,
                                                                    seed, out);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_so3_grid(int64_t n_total, int64_t first, float* R, int64_t count, cudaStream_t s) {
  if (count == 0) return AHV_OK;
  so3_grid_kernel<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(n_total, first, R, count);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

namespace {
unsigned stride_blocks(int64_t items) { return (unsigned)std::min<int64_t>((items + 255) / 256, 1 << 16); }
}  // namespace

int launch_so3_hopf_grid(int level, int64_t first, float* R, int64_t count, cudaStream_t s) {
  if (count == 0) return AHV_OK;
  so3_hopf_grid_kernel<<<stride_blocks(count), 256, 0, s>>>(level, first, R, count);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_so3_hopf_children(int level, const int64_t* parent, int64_t n, int64_t* child, float* R, cudaStream_t s) {
  if (n == 0) return AHV_OK;
  so3_hopf_children_kernel<<<stride_blocks(8 * n), 256, 0, s>>>(level, parent, n, child, R);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_hopf_pick(const int64_t* cand, int64_t n, const int64_t* pick, int B, int k, bool sort, int64_t* out,
                     cudaStream_t s) {
  if (B == 0) return AHV_OK;
  hopf_pick_kernel<<<(unsigned)((B + 3) / 4), 128, 0, s>>>(cand, n, pick, B, k, sort, out);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_so3_from_normals(const float* normals, float* R, int64_t n, cudaStream_t s) {
  if (n == 0) return AHV_OK;
  int64_t blocks = (n + 255) / 256;
  so3_from_normals_kernel<<<(unsigned)blocks, 256, 0, s>>>((const float4*)normals, R, n);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

int launch_so3_sample(uint64_t seed, int64_t first, float* R, int64_t n, cudaStream_t s) {
  if (n == 0) return AHV_OK;
  int64_t blocks = (n + 255) / 256;
  so3_sample_kernel<<<(unsigned)blocks, 256, 0, s>>>(seed, first, R, n);
  AHV_CUDA_OK(cudaGetLastError());
  return AHV_OK;
}

}  // namespace ahv
