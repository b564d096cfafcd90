/* Plain-C restatement of the nested Hopf x HEALPix SO(3) grid (ahv_so3_hopf_grid), written from Yershova et al. (2010)
 * and the HEALPix nested pix2ang / ang2pix of Gorski et al. (2005).  Test infrastructure only (tests/hopf_oracle.py
 * compiles it with -ffp-contract=off); every step is fp64, rounded once to fp32, then pytorch3d's quaternion -> matrix
 * map with individually rounded fp32 ops. */
#include <math.h>
#include <stdint.h>

static const int kJrll[12] = {2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4};
static const int kJpll[12] = {1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7};
static const double kPi = 3.141592653589793238462643383279;

static int64_t even_bits(uint64_t x) {
  int64_t out = 0;
  for (int b = 0; b < 32; ++b) out |= (int64_t)((x >> (2 * b)) & 1u) << b;
  return out;
}

static int64_t interleave(int64_t ix, int64_t iy) {
  int64_t out = 0;
  for (int b = 0; b < 32; ++b) out |= (((ix >> b) & 1) << (2 * b)) | (((iy >> b) & 1) << (2 * b + 1));
  return out;
}

static void quat_to_matrix(float a, float b, float c, float d, float *m) {
  float s = ((a * a + b * b) + c * c) + d * d;
  float den = copysignf(sqrtf(s), a);
  float r = a / den, i = b / den, j = c / den, k = d / den;
  float two_s = 2.0f / (((r * r + i * i) + j * j) + k * k);
  m[0] = 1.0f - two_s * (j * j + k * k);
  m[1] = two_s * (i * j - k * r);
  m[2] = two_s * (i * k + j * r);
  m[3] = two_s * (i * j + k * r);
  m[4] = 1.0f - two_s * (i * i + k * k);
  m[5] = two_s * (j * k - i * r);
  m[6] = two_s * (i * k - j * r);
  m[7] = two_s * (j * k + i * r);
  m[8] = 1.0f - two_s * (i * i + j * j);
}

/* cells [first, first + count) of `level` -> R [count][9] */
void hopf_oracle_grid(int level, int64_t first, int64_t count, float *R) {
  const int64_t nside = (int64_t)1 << level, npface = nside * nside;
  for (int64_t t = 0; t < count; ++t) {
    const int64_t i = first + t;
    int64_t p = (i >> (3 * level)) / 6, j = (i >> (3 * level)) % 6;
    for (int l = level - 1; l >= 0; --l) {
      const int d = (int)((i >> (3 * l)) & 7);
      p = 4 * p + (d >> 1);
      j = 2 * j + (d & 1);
    }
    const int face = (int)(p >> (2 * level));
    const int64_t ipf = p & (npface - 1), ix = even_bits((uint64_t)ipf), iy = even_bits((uint64_t)ipf >> 1);
    const int64_t jr = kJrll[face] * nside - ix - iy - 1;
    int64_t nr;
    double c2, s2;
    if (jr < nside) {
      nr = jr;
      const double u = (double)(nr * nr) / (3.0 * (double)npface);
      c2 = 1.0 - 0.5 * u;
      s2 = 0.5 * u;
    } else if (jr > 3 * nside) {
      nr = 4 * nside - jr;
      const double u = (double)(nr * nr) / (3.0 * (double)npface);
      c2 = 0.5 * u;
      s2 = 1.0 - 0.5 * u;
    } else {
      nr = nside;
      const double hz = (double)(2 * nside - jr) / (3.0 * (double)nside);
      c2 = 0.5 + hz;
      s2 = 0.5 - hz;
    }
    int64_t tp = kJpll[face] * nr + ix - iy;
    if (tp < 0) tp += 8 * nr;
    const double h = (double)(2 * j + 1) / (3.0 * (double)(4 * nside));
    double a = (double)tp / (4.0 * (double)nr) + h;
    if (a >= 2.0) a -= 2.0;
    const double c = sqrt(c2), s = sqrt(s2);
    quat_to_matrix((float)(c * cos(kPi * h)), (float)(c * sin(kPi * h)), (float)(s * cos(kPi * a)), (float)(s * sin(kPi * a)),
                   R + 9 * t);
  }
}

/* the nested pixel at Nside 2^level holding (z = cos theta, phi) */
int64_t hopf_oracle_ang2pix(int level, double z, double phi) {
  const int64_t nside = (int64_t)1 << level;
  const double za = fabs(z);
  double tt = fmod(phi * (2.0 / kPi), 4.0);
  if (tt < 0) tt += 4.0;
  int64_t face, ix, iy;
  if (za <= 2.0 / 3.0) {
    const double t1 = nside * (0.5 + tt), t2 = nside * (z * 0.75);
    const int64_t jp = (int64_t)(t1 - t2), jm = (int64_t)(t1 + t2);
    const int64_t ifp = jp >> level, ifm = jm >> level;
    face = ifp == ifm ? (ifp | 4) : (ifp < ifm ? ifp : ifm + 8);
    ix = jm & (nside - 1);
    iy = nside - (jp & (nside - 1)) - 1;
  } else {
    int64_t ntt = (int64_t)tt;
    if (ntt > 3) ntt = 3;
    const double tp = tt - (double)ntt, tmp = nside * sqrt(3.0 * (1.0 - za));
    int64_t jp = (int64_t)(tp * tmp), jm = (int64_t)((1.0 - tp) * tmp);
    if (jp > nside - 1) jp = nside - 1;
    if (jm > nside - 1) jm = nside - 1;
    if (z >= 0) {
      face = ntt;
      ix = nside - jm - 1;
      iy = nside - jp - 1;
    } else {
      face = ntt + 8;
      ix = jp;
      iy = jm;
    }
  }
  return face * nside * nside + interleave(ix, iy);
}
