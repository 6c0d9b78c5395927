// icet_b200/csrc/icet_math.cuh -- device-side geometry and small dense algebra for the ICET path.
//
// Point-wise geometry is fp32 and written operation-for-operation like the reference
// (src/utils.cpp:93-152) so that, given identical inputs, r, z/r and the transformed
// coordinates are bit-identical to a non-FMA-contracted CPU evaluation (this TU is built
// with -fmad=false; sqrt and division are IEEE-rounded by default).  atan2f/acosf/sinf/cosf are
// CUDA's fp32 libm (<= 2 ulp from glibc's; see DESIGN.md "numerics").
//
// Per-voxel and 6x6 algebra runs in double (the reference: float).
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace icet {

// theta of utils::cartesianToSpherical (src/utils.cpp:104-107): atan2f(y, x), plus 2*pi (double add) when negative.
// Own evaluation instead of CUDA's atan2f (about half the instructions): t = min/max by reciprocal + one Newton
// step, atan(t) = t + t^3 P(t^2) on [0,1] (degree-8 minimax, < 1 ulp), the octant fix-up pi/2 - a, pi - a in double
// and ONE rounding to fp32 -- within 1 ulp of the correctly rounded atan2 (glibc's and CUDA's are within 1-2 ulp).
// Zero / non-finite inputs take the library routine.
__device__ __forceinline__ float theta_of(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const bool steep = ay > ax;  // selects (not fmaxf / fminf) so that a NaN coordinate reaches t
  const float mx = steep ? ay : ax, mn = steep ? ax : ay;
  float rc;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(mx));
  const float t0 = mn * rc;
  const float t = fmaf(fmaf(-t0, mx, mn), rc, t0);
  float th;
  if (t <= 1.0f) {  // false for NaN (0/0, inf/inf, NaN input)
    const float s = t * t;
    float p = -0.0019267977913841605f;
    p = fmaf(p, s, 0.01150327268987894f);
    p = fmaf(p, s, -0.03226083889603615f);
    p = fmaf(p, s, 0.059030335396528244f);
    p = fmaf(p, s, -0.08465225994586945f);
    p = fmaf(p, s, 0.10972991585731506f);
    p = fmaf(p, s, -0.14268141984939575f);
    p = fmaf(p, s, 0.19998906552791595f);
    p = fmaf(p, s, -0.3333331048488617f);
    const float a = fmaf(t * s, p, t);
    double v = (double)a;
    v = steep ? (M_PI / 2 - v) : v;
    v = (x < 0.0f) ? (M_PI - v) : v;
    th = copysignf((float)v, y);
  } else {
    th = atan2f(y, x);
  }
  if (th < 0.0f) th = (float)((double)th + 2.0 * M_PI);  // theta(i) += 2.0 * M_PI    :105-107
  return th;
}

// phi of utils::cartesianToSpherical (src/utils.cpp:108): acosf(q), q = z / r.  For |q| <= 0.5 (elevations within
// +-30 degrees of the horizon: every ring of a spinning LiDAR) acos(q) = pi/2 - asin(q) with asin(q) = q + q^3 P(q^2)
// and the subtraction done in double with one rounding to fp32 (within 1 ulp of correctly rounded); NaN (0/0 of a
// dropped return) propagates.  Steeper rays take the library routine.
__device__ __forceinline__ float phi_of(float q) {
  if (!(fabsf(q) > 0.5f)) {
    const float s = q * q;
    float p = 0.0435001514852047f;
    p = fmaf(p, s, 0.023313719779253006f);
    p = fmaf(p, s, 0.045668356120586395f);
    p = fmaf(p, s, 0.07493448257446289f);
    p = fmaf(p, s, 0.166668102145195f);
    const float corr = (q * s) * p;
    return (float)((M_PI / 2 - (double)q) - (double)corr);
  }
  return acosf(q);
}

// utils::cartesianToSpherical, reference src/utils.cpp:93-119
__device__ __forceinline__ void c2s(float x, float y, float z, float& r, float& th, float& ph) {
  float s = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
  r = __fsqrt_rn(s);                                        // rowwise().norm()          :98
  th = theta_of(y, x);                                      //                           :104-107
  ph = phi_of(__fdiv_rn(z, r));                             //                           :108
  if (isnan(r)) r = 1000.0f;                                // isNaN().select(1000.0, .) :116
  if (isnan(th)) th = 1000.0f;
  if (isnan(ph)) ph = 1000.0f;
}

// utils::sphericalToCartesian, reference src/utils.cpp:121-142
__device__ __forceinline__ void s2c(float r, float th, float ph, float& x, float& y, float& z) {
  float sp, cp, st, ct;
  sincosf(ph, &sp, &cp);
  sincosf(th, &st, &ct);
  float rs = __fmul_rn(r, sp);
  x = __fmul_rn(rs, ct);
  y = __fmul_rn(rs, st);
  z = __fmul_rn(r, cp);
}

// bin indices, ICET::sortSphericalCoordinates reference src/icet.cpp:545-546:
//     int((theta / (2*M_PI)) * numBinsTheta) % numBinsTheta     (double math on the fp32 angle)
__device__ __forceinline__ int bin_formula(float a, double period, int nb) {
  return static_cast<int>(((double)a / period) * nb) % nb;
}
// Exact table form of the same function.  f(a) = int((double(a)/period)*nb) is a non-decreasing step
// function of the fp32 angle, so it is fully described by T[k] = the smallest fp32 a >= 0 with
// f(a) >= k (k = 0..nb, computed on the host with the very same double expression; T[nb+1] = +inf).
// An fp32 estimate of the bin is corrected by at most one step against T.  Angles beyond `amax`
// (only the NaN sentinel 1000.0) take the formula.
struct BinTable {
  const float* T;  // nb + 2 entries
  float scale;     // fp32(nb / period)
  float amax;      // fp32(period): the largest angle the table covers
  int nb;
  float acap;      // fp32 angle whose estimate lands in record nb + 1 (pass kernels: everything beyond the period)
  int sbin;        // bin of the NaN sentinel 1000.0 by the double formula
};
// T may point to global or shared memory (the call is inlined, the address space is known statically)
__device__ __forceinline__ int bin_lookup(float a, const float* T, float scale, float amax, int nb, double period) {
  if (!(a <= amax) || a < 0.f) return bin_formula(a, period, nb);
  int k = __float2int_rz(a * scale);
  k = min(max(k, 0), nb);
  if (a < T[k]) k--;
  else if (a >= T[k + 1]) k++;
  return k == nb ? 0 : k;
}
__device__ __forceinline__ int bin_lookup(float a, const BinTable& t, double period) {
  return bin_lookup(a, t.T, t.scale, t.amax, t.nb, period);
}

// utils::R, reference src/utils.cpp:144-152 (row-major, fp32 trig on fp32 angles)
// (the _sc forms take the six sines / cosines: the warp-parallel solve evaluates them once, on three lanes)
__device__ __forceinline__ void rotR_sc(float sph, float cph, float sth, float cth, float sps, float cps, float* R) {
  R[0] = cth * cps;
  R[1] = sps * cph + sph * sth * cps;
  R[2] = sph * sps - sth * cph * cps;
  R[3] = -sps * cth;
  R[4] = cph * cps - sph * sth * sps;
  R[5] = sph * cps + sth * sps * cph;
  R[6] = sth;
  R[7] = -sph * cth;
  R[8] = cph * cth;
}
__device__ inline void rotR(float phi, float theta, float psi, float* R) {
  float sph, cph, sth, cth, sps, cps;
  sincosf(phi, &sph, &cph);
  sincosf(theta, &sth, &cth);
  sincosf(psi, &sps, &cps);
  R[0] = cth * cps;
  R[1] = sps * cph + sph * sth * cps;
  R[2] = sph * sps - sth * cph * cps;
  R[3] = -sps * cth;
  R[4] = cph * cps - sph * sth * sps;
  R[5] = sph * cps + sth * sps * cph;
  R[6] = sth;
  R[7] = -sph * cth;
  R[8] = cph * cth;
}

// (p + t) * R with row vectors, reference src/icet.cpp:377-378
__device__ __forceinline__ void transform(float px, float py, float pz, const float* t, const float* R,
                                          float& x, float& y, float& z) {
  float ax = __fadd_rn(px, t[0]), ay = __fadd_rn(py, t[1]), az = __fadd_rn(pz, t[2]);
  x = __fadd_rn(__fadd_rn(__fmul_rn(ax, R[0]), __fmul_rn(ay, R[3])), __fmul_rn(az, R[6]));
  y = __fadd_rn(__fadd_rn(__fmul_rn(ax, R[1]), __fmul_rn(ay, R[4])), __fmul_rn(az, R[7]));
  z = __fadd_rn(__fadd_rn(__fmul_rn(ax, R[2]), __fmul_rn(ay, R[5])), __fmul_rn(az, R[8]));
}

// The three 3x3 derivative matrices of ICET::get_H, reference src/icet.cpp:507-527 (fp32 trig),
// J = [Jx | Jy | Jz], each row-major.
__device__ __forceinline__ void getH_J_sc(float sph, float cph, float sth, float cth, float sps, float cps, float* J) {
  float* Jx = J;
  float* Jy = J + 9;
  float* Jz = J + 18;
  Jx[0] = 0.f; Jx[1] = (-sps * sph + cph * sth * cps); Jx[2] = (cph * sps + sth * sph * cps);
  Jx[3] = 0.f; Jx[4] = (-sph * cps - cph * sth * sps); Jx[5] = (cph * cps - sth * sps * sph);
  Jx[6] = 0.f; Jx[7] = (-cph * cth);                   Jx[8] = (-sph * cth);
  Jy[0] = (-sth * cps); Jy[1] = (cth * sph * cps);  Jy[2] = (-cth * cph * cps);
  Jy[3] = (sps * sth);  Jy[4] = (-cth * sph * sps); Jy[5] = (cth * sps * cph);
  Jy[6] = (cth);        Jy[7] = (sph * sth);        Jy[8] = (-sth * cph);
  Jz[0] = (-cth * sps); Jz[1] = (cps * cph - sph * sth * sps);  Jz[2] = (cps * sph + sth * cph * sps);
  Jz[3] = (-cps * cth); Jz[4] = (-sps * cph - sph * sth * cps); Jz[5] = (-sph * sps + sth * cps * cph);
  Jz[6] = 0.f; Jz[7] = 0.f; Jz[8] = 0.f;
}
__device__ inline void getH_J(float phi, float theta, float psi, float* J) {
  float sph, cph, sth, cth, sps, cps;
  sincosf(phi, &sph, &cph);
  sincosf(theta, &sth, &cth);
  sincosf(psi, &sps, &cps);
  float* Jx = J;
  float* Jy = J + 9;
  float* Jz = J + 18;
  Jx[0] = 0.f; Jx[1] = (-sps * sph + cph * sth * cps); Jx[2] = (cph * sps + sth * sph * cps);
  Jx[3] = 0.f; Jx[4] = (-sph * cps - cph * sth * sps); Jx[5] = (cph * cps - sth * sps * sph);
  Jx[6] = 0.f; Jx[7] = (-cph * cth);                   Jx[8] = (-sph * cth);
  Jy[0] = (-sth * cps); Jy[1] = (cth * sph * cps);  Jy[2] = (-cth * cph * cps);
  Jy[3] = (sps * sth);  Jy[4] = (-cth * sph * sps); Jy[5] = (cth * sps * cph);
  Jy[6] = (cth);        Jy[7] = (sph * sth);        Jy[8] = (-sth * cph);
  Jz[0] = (-cth * sps); Jz[1] = (cps * cph - sph * sth * sps);  Jz[2] = (cps * sph + sth * cph * sps);
  Jz[3] = (-cps * cth); Jz[4] = (-sps * cph - sph * sth * cps); Jz[5] = (-sph * sps + sth * cps * cph);
  Jz[6] = 0.f; Jz[7] = 0.f; Jz[8] = 0.f;
}

// ---------------------------------------------------------------------------------------------
// Eigen::SelfAdjointEigenSolver<Matrix3f>::compute as called at reference src/icet.cpp:181-184:
// scaling, fixed 3x3 tridiagonalisation, implicit symmetric QR (Wilkinson shift), selection sort.
// fp32 and operation-ordered like Eigen 3.3.7 because the reference's L mask and projections
// depend on the eigenvector SIGNS this particular algorithm produces (SURVEY.md H2).
// V is row-major, columns = eigenvectors, eigenvalues ascending.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float eig_hypot(float x, float y) {
  x = fabsf(x);
  y = fabsf(y);
  float p = fmaxf(x, y);
  if (p == 0.f) return 0.f;
  float qp = fminf(y, x) / p;
  return p * sqrtf(1.f + qp * qp);
}
__device__ __forceinline__ void make_givens(float p, float q, float& c, float& s) {
  if (q == 0.f) {
    c = p < 0.f ? -1.f : 1.f;
    s = 0.f;
  } else if (p == 0.f) {
    c = 0.f;
    s = q < 0.f ? 1.f : -1.f;
  } else if (fabsf(p) > fabsf(q)) {
    float t = q / p;
    float u = sqrtf(1.f + t * t);
    if (p < 0.f) u = -u;
    c = 1.f / u;
    s = -t * c;
  } else {
    float t = p / q;
    float u = sqrtf(1.f + t * t);
    if (q < 0.f) u = -u;
    s = -1.f / u;
    c = -t * s;
  }
}

__device__ inline void eig3f(const float A[9], float evals[3], float V[9]) {
  float m00 = A[0], m10 = A[3], m11 = A[4], m20 = A[6], m21 = A[7], m22 = A[8];
  float scale = fmaxf(fmaxf(fmaxf(fabsf(m00), fabsf(m10)), fmaxf(fabsf(m11), fabsf(m20))),
                      fmaxf(fabsf(m21), fabsf(m22)));
  if (scale == 0.f) scale = 1.f;
  m00 /= scale; m10 /= scale; m11 /= scale; m20 /= scale; m21 /= scale; m22 /= scale;
  float diag[3], sub[2];
  diag[0] = m00;
  float v1norm2 = m20 * m20;
  if (v1norm2 <= FLT_MIN) {
    diag[1] = m11; diag[2] = m22; sub[0] = m10; sub[1] = m21;
#pragma unroll
    for (int i = 0; i < 9; i++) V[i] = 0.f;
    V[0] = V[4] = V[8] = 1.f;
  } else {
    float beta = sqrtf(m10 * m10 + v1norm2);
    float invBeta = 1.f / beta;
    float m01 = m10 * invBeta;
    float m02 = m20 * invBeta;
    float q = 2.f * m01 * m21 + m02 * (m22 - m11);
    diag[1] = m11 + m02 * q;
    diag[2] = m22 - m02 * q;
    sub[0] = beta;
    sub[1] = m21 - m01 * q;
    V[0] = 1.f; V[1] = 0.f; V[2] = 0.f;
    V[3] = 0.f; V[4] = m01; V[5] = m02;
    V[6] = 0.f; V[7] = m02; V[8] = -m01;
  }
  // computeFromTridiagonal_impl (n = 3)
  int end = 2, start = 0, iter = 0;
  const float precision = 2.f * FLT_EPSILON;
  while (end > 0) {
    for (int i = start; i < end; ++i)
      if (fabsf(sub[i]) <= (fabsf(diag[i]) + fabsf(diag[i + 1])) * precision || fabsf(sub[i]) <= FLT_MIN)
        sub[i] = 0.f;
    while (end > 0 && sub[end - 1] == 0.f) end--;
    if (end <= 0) break;
    iter++;
    if (iter > 30 * 3) break;
    start = end - 1;
    while (start > 0 && sub[start - 1] != 0.f) start--;
    // tridiagonal_qr_step
    float td = (diag[end - 1] - diag[end]) * 0.5f;
    float e = sub[end - 1];
    float mu = diag[end];
    if (td == 0.f) {
      mu -= fabsf(e);
    } else {
      float e2 = e * e;
      float h = eig_hypot(td, e);
      if (e2 == 0.f)
        mu -= (e / (td + (td > 0.f ? 1.f : -1.f))) * (e / h);
      else
        mu -= e2 / (td + (td > 0.f ? h : -h));
    }
    float x = diag[start] - mu;
    float z = sub[start];
    for (int k = start; k < end; ++k) {
      float c, s;
      make_givens(x, z, c, s);
      float sdk = s * diag[k] + c * sub[k];
      float dkp1 = s * sub[k] + c * diag[k + 1];
      diag[k] = c * (c * diag[k] - s * sub[k]) - s * (c * sub[k] - s * diag[k + 1]);
      diag[k + 1] = s * sdk + c * dkp1;
      sub[k] = c * sdk - s * dkp1;
      if (k > start) sub[k - 1] = c * sub[k - 1] - s * z;
      x = sub[k];
      if (k < end - 1) {
        z = -s * sub[k + 1];
        sub[k + 1] = c * sub[k + 1];
      }
      if (!(c == 1.f && s == 0.f)) {
#pragma unroll
        for (int i = 0; i < 3; i++) {
          float xi = V[i * 3 + k], yi = V[i * 3 + k + 1];
          V[i * 3 + k] = c * xi - s * yi;
          V[i * 3 + k + 1] = s * xi + c * yi;
        }
      }
    }
  }
  if (iter <= 30 * 3) {
    for (int i = 0; i < 2; ++i) {
      int k = 0;
      float m = diag[i];
      for (int j = 1; j < 3 - i; j++)
        if (diag[i + j] < m) {
          m = diag[i + j];
          k = j;
        }
      if (k > 0) {
        float t = diag[i]; diag[i] = diag[k + i]; diag[k + i] = t;
        for (int r = 0; r < 3; r++) {
          float u = V[r * 3 + i]; V[r * 3 + i] = V[r * 3 + k + i]; V[r * 3 + k + i] = u;
        }
      }
    }
  }
  for (int i = 0; i < 3; i++) evals[i] = diag[i] * scale;
}

// ---------------------------------------------------------------------------------------------
// Moore-Penrose inverse with the rank rule of Eigen::CompleteOrthogonalDecomposition
// (column-pivoted Householder QR; a pivot counts if |R_ii| > FLT_EPSILON * min(m,n) * max|R_ii|;
// Z reflectors for the rank-deficient case).  Reference call sites: src/icet.cpp:320-321 (3x3),
// :410-411 (6x6).  Row-major A (rows x cols, both <= 6) -> P (cols x rows).  Double arithmetic,
// the fp32 epsilon is kept in the rank rule so that rank decisions mean the same thing.
// ---------------------------------------------------------------------------------------------
__device__ inline void make_householder(double* v, int len, int stride, double& tau, double& beta) {
  double tail = 0.0;
  for (int i = 1; i < len; i++) tail += v[i * stride] * v[i * stride];
  double c0 = v[0];
  if (len == 1 || tail <= DBL_MIN) {
    tau = 0.0;
    beta = c0;
    for (int i = 1; i < len; i++) v[i * stride] = 0.0;
  } else {
    beta = sqrt(c0 * c0 + tail);
    if (c0 >= 0.0) beta = -beta;
    for (int i = 1; i < len; i++) v[i * stride] = v[i * stride] / (c0 - beta);
    tau = (beta - c0) / beta;
  }
}

__device__ __noinline__ int cod_pinv(const double* A, int rows, int cols, double* P) {
  const int size = rows < cols ? rows : cols;
  const double eps_rank = (double)FLT_EPSILON;
  double qr[36], hC[6], cnU[6], cnD[6], zC[6];
  int transp[6];
  for (int i = 0; i < rows * cols; i++) qr[i] = A[i];
#define QR(i, j) qr[(i) * cols + (j)]
  double maxnorm = 0.0;
  for (int k = 0; k < cols; k++) {
    double s = 0.0;
    for (int i = 0; i < rows; i++) s += QR(i, k) * QR(i, k);
    cnD[k] = cnU[k] = sqrt(s);
    if (cnU[k] > maxnorm) maxnorm = cnU[k];
  }
  double th = maxnorm * eps_rank;
  const double threshold_helper = (th * th) / (double)rows;
  const double downdate = sqrt(DBL_EPSILON);
  int nonzero_pivots = size;
  double maxpivot = 0.0;
  for (int k = 0; k < size; k++) {
    int biggest = k;
    double big = cnU[k];
    for (int j = k + 1; j < cols; j++)
      if (cnU[j] > big) {
        big = cnU[j];
        biggest = j;
      }
    if (nonzero_pivots == size && big * big < threshold_helper * (double)(rows - k)) nonzero_pivots = k;
    transp[k] = biggest;
    if (k != biggest) {
      for (int i = 0; i < rows; i++) {
        double t = QR(i, k); QR(i, k) = QR(i, biggest); QR(i, biggest) = t;
      }
      double t = cnU[k]; cnU[k] = cnU[biggest]; cnU[biggest] = t;
      t = cnD[k]; cnD[k] = cnD[biggest]; cnD[biggest] = t;
    }
    double beta;
    make_householder(&QR(k, k), rows - k, cols, hC[k], beta);
    QR(k, k) = beta;
    if (fabs(beta) > maxpivot) maxpivot = fabs(beta);
    if (rows - k == 1) {
      for (int j = k + 1; j < cols; j++) QR(k, j) *= (1.0 - hC[k]);
    } else if (hC[k] != 0.0) {
      for (int j = k + 1; j < cols; j++) {
        double t = QR(k, j);
        for (int i = k + 1; i < rows; i++) t += QR(i, k) * QR(i, j);
        QR(k, j) -= hC[k] * t;
        for (int i = k + 1; i < rows; i++) QR(i, j) -= (hC[k] * QR(i, k)) * t;
      }
    }
    for (int j = k + 1; j < cols; j++) {
      if (cnU[j] != 0.0) {
        double t = fabs(QR(k, j)) / cnU[j];
        t = (1.0 + t) * (1.0 - t);
        t = t < 0.0 ? 0.0 : t;
        double ratio = cnU[j] / cnD[j];
        double t2 = t * ratio * ratio;
        if (t2 <= downdate) {
          double s = 0.0;
          for (int i = k + 1; i < rows; i++) s += QR(i, j) * QR(i, j);
          cnD[j] = cnU[j] = sqrt(s);
        } else {
          cnU[j] *= sqrt(t);
        }
      }
    }
  }
  int rank = 0;
  {
    const double premult = fabs(maxpivot) * (eps_rank * (double)size);
    for (int i = 0; i < nonzero_pivots; i++)
      if (fabs(QR(i, i)) > premult) rank++;
  }
  for (int i = 0; i < rows * cols; i++) P[i] = 0.0;
  if (rank == 0) return 0;
  if (rank < cols) {
    for (int k = rank - 1; k >= 0; --k) {
      if (k != rank - 1)
        for (int i = 0; i <= k; i++) {
          double t = QR(i, k); QR(i, k) = QR(i, rank - 1); QR(i, rank - 1) = t;
        }
      double beta;
      make_householder(&QR(k, rank - 1), cols - rank + 1, 1, zC[k], beta);
      QR(k, rank - 1) = beta;
      if (k > 0 && zC[k] != 0.0) {
        for (int i = 0; i < k; i++) {
          double t = QR(i, rank - 1);
          for (int j = rank; j < cols; j++) t += QR(i, j) * QR(k, j);
          QR(i, rank - 1) -= zC[k] * t;
          for (int j = rank; j < cols; j++) QR(i, j) -= (zC[k] * t) * QR(k, j);
        }
      }
      if (k != rank - 1)
        for (int i = 0; i <= k; i++) {
          double t = QR(i, k); QR(i, k) = QR(i, rank - 1); QR(i, rank - 1) = t;
        }
    }
  }
  // c = Q^T, y = T^-1 c, Z^T, permutation -- one right-hand side (column of I) at a time
  int perm[6];
  for (int i = 0; i < cols; i++) perm[i] = i;
  for (int k = 0; k < size; k++) {
    int t = perm[k]; perm[k] = perm[transp[k]]; perm[transp[k]] = t;
  }
  for (int j = 0; j < rows; j++) {
    double c[6], y[6];
    for (int i = 0; i < rows; i++) c[i] = (i == j) ? 1.0 : 0.0;
    for (int k = 0; k < rank; k++) {
      if (rows - k == 1) {
        c[k] *= (1.0 - hC[k]);
      } else if (hC[k] != 0.0) {
        double t = c[k];
        for (int i = k + 1; i < rows; i++) t += QR(i, k) * c[i];
        c[k] -= hC[k] * t;
        for (int i = k + 1; i < rows; i++) c[i] -= (hC[k] * QR(i, k)) * t;
      }
    }
    for (int i = 0; i < cols; i++) y[i] = 0.0;
    for (int i = rank - 1; i >= 0; --i) {
      double s = c[i];
      for (int k = i + 1; k < rank; k++) s -= QR(i, k) * y[k];
      y[i] = s / QR(i, i);
    }
    if (rank < cols) {
      for (int k = 0; k < rank; k++) {
        if (k != rank - 1) { double t = y[k]; y[k] = y[rank - 1]; y[rank - 1] = t; }
        if (zC[k] != 0.0) {
          double t = y[rank - 1];
          for (int i = rank; i < cols; i++) t += QR(k, i) * y[i];
          y[rank - 1] -= zC[k] * t;
          for (int i = rank; i < cols; i++) y[i] -= (zC[k] * QR(k, i)) * t;
        }
        if (k != rank - 1) { double t = y[k]; y[k] = y[rank - 1]; y[rank - 1] = t; }
      }
    }
    for (int k = 0; k < cols; k++) P[perm[k] * rows + j] = y[k];
  }
#undef QR
  return rank;
}

// Inverse of the SPD block selected by `mask` (bit i = row/col i kept) of a symmetric 3x3,
// embedded in zeros -- the pseudo-inverse of L*A*L^T when the kept block is comfortably
// full rank.  Returns false (W untouched) when the block is not safely invertible; the caller
// then falls back to cod_pinv.
// (Every index is a compile-time constant -- the kept rows / columns are selected by a switch on the mask -- so that M
// and W stay in registers: with run-time indices they live in local memory and every access of the per-voxel algebra to
// them is a load / store on the critical path of an iteration.)
template <int I0, int I1>
__device__ __forceinline__ bool masked_inv3_2(const double M[9], double W[9]) {
  const double a = M[I0 * 3 + I0], b = M[I0 * 3 + I1], d = M[I1 * 3 + I1];
  const double det = a * d - b * b;
  if (!(a > 0.0) || !(d > 0.0) || !(det > 0.0)) return false;
  const double ia = d / det, ib = -b / det, id = a / det;
  const double tr = a + d;
  const double tri = ia + id;
  if (!(tr * tri < 5e5)) return false;  // cond < 5e5: far from the COD rank threshold (pivot ratio 3.6e-7)
  W[I0 * 3 + I0] = ia;
  W[I0 * 3 + I1] = ib;
  W[I1 * 3 + I0] = ib;
  W[I1 * 3 + I1] = id;
  return true;
}
template <int I0>
__device__ __forceinline__ bool masked_inv3_1(const double M[9], double W[9]) {
  const double a = M[I0 * 3 + I0];
  if (!(a > 0.0)) return false;
  W[I0 * 3 + I0] = 1.0 / a;
  return true;
}
__device__ __forceinline__ bool masked_inv3(const double M[9], int mask, double W[9]) {
#pragma unroll
  for (int i = 0; i < 9; i++) W[i] = 0.0;
  switch (mask & 7) {
    case 0: return true;
    case 1: return masked_inv3_1<0>(M, W);
    case 2: return masked_inv3_1<1>(M, W);
    case 4: return masked_inv3_1<2>(M, W);
    case 3: return masked_inv3_2<0, 1>(M, W);
    case 5: return masked_inv3_2<0, 2>(M, W);
    case 6: return masked_inv3_2<1, 2>(M, W);
    default: break;
  }
  const double a = M[0], b = M[1], c = M[2], d = M[4], e = M[5], f = M[8];
  const double c00 = d * f - e * e, c01 = c * e - b * f, c02 = b * e - c * d;
  const double det = a * c00 + b * c01 + c * c02;
  if (!(a > 0.0) || !(d > 0.0) || !(f > 0.0) || !(det > 0.0)) return false;
  const double c11 = a * f - c * c, c12 = b * c - a * e, c22 = a * d - b * b;
  const double id = 1.0 / det;
  const double tr = a + d + f;
  const double csum = c00 + c11 + c22;
  const double tri = csum * id;
  // csum = l1 l2 + l1 l3 + l2 l3 >= tr^2 / 9e5 whenever cond < 1e5.  Below that it is rounding noise (M of rank one:
  // every 2x2 minor vanishes), det is as well, and their ratio can pass the trace bound while M is singular.
  if (!(tr * tri < 1e5) || !(csum > 1e-6 * (tr * tr))) return false;
  W[0] = c00 * id; W[1] = c01 * id; W[2] = c02 * id;
  W[3] = c01 * id; W[4] = c11 * id; W[5] = c12 * id;
  W[6] = c02 * id; W[7] = c12 * id; W[8] = c22 * id;
  return true;
}

// Cyclic Jacobi eigen-decomposition of a symmetric 6x6 (row-major); eigenvalues ascending,
// U row-major with columns = eigenvectors.  Stands in for SelfAdjointEigenSolver<MatrixXf>
// at reference src/icet.cpp:455-458 (only eigenvalues and sign-independent combinations of the
// eigenvectors reach X; see DESIGN.md for the :479 inflation term).
// All matrix indices are compile-time constants after unrolling, so A and U live in registers;
// the routine is kept out of line because it runs only when the warp solve's condition bound fails.
__device__ __noinline__ void jacobi6(const double* __restrict__ Ain, double* __restrict__ ev_out,
                                     double* __restrict__ U_out) {
  double A[36], U[36];
#pragma unroll
  for (int i = 0; i < 36; i++) {
    A[i] = Ain[i];
    U[i] = 0.0;
  }
#pragma unroll
  for (int i = 0; i < 6; i++) U[i * 6 + i] = 1.0;
#pragma unroll 1
  for (int sweep = 0; sweep < 24; sweep++) {
    double off = 0.0, dg = 0.0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      dg += A[i * 6 + i] * A[i * 6 + i];
#pragma unroll
      for (int j = i + 1; j < 6; j++) off += A[i * 6 + j] * A[i * 6 + j];
    }
    if (!(off > 1e-34 * dg)) break;
#pragma unroll
    for (int p = 0; p < 5; p++) {
#pragma unroll
      for (int q = p + 1; q < 6; q++) {
        const double apq = A[p * 6 + q];
        if (apq != 0.0) {
          const double theta = (A[q * 6 + q] - A[p * 6 + p]) / (2.0 * apq);
          const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
          const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
#pragma unroll
          for (int k = 0; k < 6; k++) {
            const double akp = A[k * 6 + p], akq = A[k * 6 + q];
            A[k * 6 + p] = c * akp - sn * akq;
            A[k * 6 + q] = sn * akp + c * akq;
          }
#pragma unroll
          for (int k = 0; k < 6; k++) {
            const double apk = A[p * 6 + k], aqk = A[q * 6 + k];
            A[p * 6 + k] = c * apk - sn * aqk;
            A[q * 6 + k] = sn * apk + c * aqk;
          }
#pragma unroll
          for (int k = 0; k < 6; k++) {
            const double ukp = U[k * 6 + p], ukq = U[k * 6 + q];
            U[k * 6 + p] = c * ukp - sn * ukq;
            U[k * 6 + q] = sn * ukp + c * ukq;
          }
        }
      }
    }
  }
  double ev[6];
#pragma unroll
  for (int i = 0; i < 6; i++) ev[i] = A[i * 6 + i];
  // ascending selection sort (static indices: compare-exchange network over all pairs)
#pragma unroll
  for (int i = 0; i < 5; i++) {
#pragma unroll
    for (int j = i + 1; j < 6; j++) {
      if (ev[j] < ev[i]) {
        const double t = ev[i]; ev[i] = ev[j]; ev[j] = t;
#pragma unroll
        for (int r = 0; r < 6; r++) {
          const double u = U[r * 6 + i]; U[r * 6 + i] = U[r * 6 + j]; U[r * 6 + j] = u;
        }
      }
    }
  }
  // sign convention (the reference's is an artefact of Eigen's QR): largest component positive
#pragma unroll
  for (int c = 0; c < 6; c++) {
    double best = U[c], mag = fabs(U[c]);
#pragma unroll
    for (int r = 1; r < 6; r++)
      if (fabs(U[r * 6 + c]) > mag) {
        mag = fabs(U[r * 6 + c]);
        best = U[r * 6 + c];
      }
    if (best < 0.0) {
#pragma unroll
      for (int r = 0; r < 6; r++) U[r * 6 + c] = -U[r * 6 + c];
    }
  }
#pragma unroll
  for (int i = 0; i < 6; i++) ev_out[i] = ev[i];
#pragma unroll
  for (int i = 0; i < 36; i++) U_out[i] = U[i];
}

}  // namespace icet
