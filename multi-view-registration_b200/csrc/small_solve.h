// small_solve.h -- the tiny dense solves of the ICP path (host side; eig_sym3 also runs on device).
//
//   svd3 + umeyama_rigid : TransformationEstimationSVD / Eigen::umeyama(with_scaling=false), the
//                          estimator pcl::IterativeClosestPoint uses by default inside icp.align
//                          (mvr/src/registrator.cpp:569, 920, 1012; SURVEY.md A7)
//   cholesky_solve6      : normal equations of TransformationEstimationPointToPlaneLLS (A12)
//   eig_sym3             : smallest-eigenvector plane fit of pcl::NormalEstimation (A13)
// The reference links Eigen/LAPACK for these; neither is available here, so they are written out.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define MVR_HD __host__ __device__
#else
#define MVR_HD
#endif

namespace mvr {

// One rotation of the one-sided Jacobi SVD on columns P, Q (compile-time indices keep B and W in
// registers on the device).  Returns false when the two columns are already orthogonal.
template <int P, int Q>
MVR_HD inline bool svd3_rotate(double (&B)[3][3], double (&W)[3][3]) {
  const double al = B[0][P] * B[0][P] + B[1][P] * B[1][P] + B[2][P] * B[2][P];
  const double be = B[0][Q] * B[0][Q] + B[1][Q] * B[1][Q] + B[2][Q] * B[2][Q];
  const double ga = B[0][P] * B[0][Q] + B[1][P] * B[1][Q] + B[2][P] * B[2][Q];
  if (ga == 0.0 || ga * ga <= 1e-32 * (al * be)) return false;   // |cos angle| <= 1e-16: orthogonal to working precision
  const double zeta = (be - al) / (2.0 * ga);
  const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
  const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int k = 0; k < 3; ++k) {
    const double bp = B[k][P], bq = B[k][Q];
    B[k][P] = c * bp - sn * bq; B[k][Q] = sn * bp + c * bq;
    const double wp = W[k][P], wq = W[k][Q];
    W[k][P] = c * wp - sn * wq; W[k][Q] = sn * wp + c * wq;
  }
  return true;
}

// Exchange columns P and Q of B and W when column Q is the longer one (sorting network step).
template <int P, int Q>
MVR_HD inline void svd3_order(double (&B)[3][3], double (&W)[3][3], double (&nrm)[3]) {
  if (nrm[Q] > nrm[P]) {
    double t = nrm[P]; nrm[P] = nrm[Q]; nrm[Q] = t;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 3; ++k) {
      t = B[k][P]; B[k][P] = B[k][Q]; B[k][Q] = t;
      t = W[k][P]; W[k][P] = W[k][Q]; W[k][Q] = t;
    }
  }
}

// One-sided (Hestenes) Jacobi SVD of a 3x3 row-major matrix: A = U diag(s) V^T, s descending,
// U and V orthogonal.  Works on the columns of A directly, so small singular values keep full
// relative accuracy (no A^T A squaring).
MVR_HD inline void svd3(const double* A, double* U, double* s, double* V) {
  double B[3][3], W[3][3];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < 3; ++i) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 3; ++j) { B[i][j] = A[i * 3 + j]; W[i][j] = (i == j) ? 1.0 : 0.0; }
  }
  for (int sweep = 0; sweep < 40; ++sweep) {
    bool rotated = svd3_rotate<0, 1>(B, W);
    rotated = svd3_rotate<0, 2>(B, W) || rotated;
    rotated = svd3_rotate<1, 2>(B, W) || rotated;
    if (!rotated) break;
  }
  double nrm[3];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int j = 0; j < 3; ++j) nrm[j] = sqrt(B[0][j] * B[0][j] + B[1][j] * B[1][j] + B[2][j] * B[2][j]);
  svd3_order<0, 1>(B, W, nrm);
  svd3_order<0, 2>(B, W, nrm);
  svd3_order<1, 2>(B, W, nrm);
  double Uc[3][3];  // Uc[col][row]
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int c = 0; c < 3; ++c) {
    s[c] = nrm[c];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 3; ++r) { V[r * 3 + c] = W[r][c]; Uc[c][r] = B[r][c]; }
  }
  const double tiny = 1e-300 + 1e-14 * s[0];
  if (s[0] > tiny) { for (int r = 0; r < 3; ++r) Uc[0][r] /= s[0]; }
  else { Uc[0][0] = 1; Uc[0][1] = 0; Uc[0][2] = 0; }
  if (s[1] > tiny) { for (int r = 0; r < 3; ++r) Uc[1][r] /= s[1]; }
  else {
    // second direction: the coordinate axis least aligned with the first, orthogonalised
    const double a0 = fabs(Uc[0][0]), a1 = fabs(Uc[0][1]), a2 = fabs(Uc[0][2]);
    double e[3] = {0, 0, 0};
    double d;
    if (a2 < a0 && a2 < a1) { e[2] = 1; d = Uc[0][2]; }
    else if (a1 < a0) { e[1] = 1; d = Uc[0][1]; }
    else { e[0] = 1; d = Uc[0][0]; }
    double n2 = 0;
    for (int r = 0; r < 3; ++r) { Uc[1][r] = e[r] - d * Uc[0][r]; n2 += Uc[1][r] * Uc[1][r]; }
    n2 = sqrt(n2);
    for (int r = 0; r < 3; ++r) Uc[1][r] /= n2;
  }
  double cr[3] = {Uc[0][1] * Uc[1][2] - Uc[0][2] * Uc[1][1], Uc[0][2] * Uc[1][0] - Uc[0][0] * Uc[1][2],
                  Uc[0][0] * Uc[1][1] - Uc[0][1] * Uc[1][0]};
  if (s[2] > tiny) {
    double sg = Uc[2][0] * cr[0] + Uc[2][1] * cr[1] + Uc[2][2] * cr[2];
    for (int r = 0; r < 3; ++r) Uc[2][r] = sg < 0 ? -cr[r] : cr[r];
  } else {
    for (int r = 0; r < 3; ++r) Uc[2][r] = cr[r];
  }
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) U[r * 3 + c] = Uc[c][r];
}

MVR_HD inline double det3(const double* M) {
  return M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) + M[2] * (M[3] * M[7] - M[4] * M[6]);
}

// Rigid transform (no scaling) from centroids and the 3x3 cross-covariance Sigma = E[(d-mu_d)(s-mu_s)^T]
// (row-major).  T: column-major double 4x4 with dst ~ T * src.
MVR_HD inline void umeyama_rigid(const double* mu_s, const double* mu_d, const double* Sigma, double* T) {
  double U[9], V[9], sv[3];
  svd3(Sigma, U, sv, V);
  double S[3] = {1.0, 1.0, 1.0};
  if (det3(U) * det3(V) < 0) S[2] = -1.0;
  double R[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double x = 0;
      for (int k = 0; k < 3; ++k) x += U[i * 3 + k] * S[k] * V[j * 3 + k];
      R[i * 3 + j] = x;
    }
  for (int k = 0; k < 16; ++k) T[k] = (k % 5 == 0) ? 1.0 : 0.0;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T[j * 4 + i] = R[i * 3 + j];
    T[12 + i] = mu_d[i] - (R[i * 3] * mu_s[0] + R[i * 3 + 1] * mu_s[1] + R[i * 3 + 2] * mu_s[2]);
  }
}

// Solve the 6x6 SPD system A x = b by Cholesky (A row-major, full).  false if not positive definite.
MVR_HD inline bool cholesky_solve6(const double* A, const double* b, double* x) {
  double L[36];
  for (int k = 0; k < 36; ++k) L[k] = 0.0;
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j <= i; ++j) {
      double sum = A[i * 6 + j];
      for (int k = 0; k < j; ++k) sum -= L[i * 6 + k] * L[j * 6 + k];
      if (i == j) {
        if (!(sum > 0.0)) return false;
        L[i * 6 + i] = sqrt(sum);
      } else {
        L[i * 6 + j] = sum / L[j * 6 + j];
      }
    }
  double y[6];
  for (int i = 0; i < 6; ++i) {
    double sum = b[i];
    for (int k = 0; k < i; ++k) sum -= L[i * 6 + k] * y[k];
    y[i] = sum / L[i * 6 + i];
  }
  for (int i = 5; i >= 0; --i) {
    double sum = y[i];
    for (int k = i + 1; k < 6; ++k) sum -= L[k * 6 + i] * x[k];
    x[i] = sum / L[i * 6 + i];
  }
  return true;
}

// (alpha, beta, gamma, tx, ty, tz) -> column-major 4x4, R = Rz(gamma) Ry(beta) Rx(alpha).
MVR_HD inline void pose_from_6(const double* x, double* T) {
  double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
  double R[9] = {cg * cb, -sg * ca + cg * sb * sa, sg * sa + cg * sb * ca,
                 sg * cb, cg * ca + sg * sb * sa,  -cg * sa + sg * sb * ca,
                 -sb,     cb * sa,                 cb * ca};
  for (int k = 0; k < 16; ++k) T[k] = (k % 5 == 0) ? 1.0 : 0.0;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T[j * 4 + i] = R[i * 3 + j];
    T[12 + i] = x[3 + i];
  }
}

// The increment of the symmetric objective (TransformationEstimationSymmetricPointToPlaneLLS::constructTransformationMatrix):
// T = R Trans(x3, x4, x5) R with the R of pose_from_6, i.e. rotation R R and translation R t.  Column-major 4x4.
MVR_HD inline void pose_from_6_symmetric(const double* x, double* T) {
  double R[16];
  pose_from_6(x, R);   // R[c * 4 + r]; its translation column is t
  for (int k = 0; k < 16; ++k) T[k] = (k % 5 == 0) ? 1.0 : 0.0;
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) T[c * 4 + r] = (R[r] * R[c * 4] + R[4 + r] * R[c * 4 + 1]) + R[8 + r] * R[c * 4 + 2];
    T[12 + r] = (R[r] * x[3] + R[4 + r] * x[4]) + R[8 + r] * x[5];
  }
}

// Symmetric 3x3 eigen-decomposition by cyclic Jacobi (row-major C), eigenvalues ascending,
// eigenvectors in the columns of V (row-major).
MVR_HD inline void eig_sym3(const double* C, double* w, double* V) {
  double S[3][3], E[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { S[i][j] = C[i * 3 + j]; E[i][j] = (i == j) ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 40; ++sweep) {
    double off = S[0][1] * S[0][1] + S[0][2] * S[0][2] + S[1][2] * S[1][2];
    double dg = S[0][0] * S[0][0] + S[1][1] * S[1][1] + S[2][2] * S[2][2];
    if (off == 0.0 || off <= 1e-34 * dg) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (S[p][q] == 0.0) continue;
        double theta = (S[q][q] - S[p][p]) / (2.0 * S[p][q]);
        double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < 3; ++k) { double a = S[k][p], b = S[k][q]; S[k][p] = c * a - sn * b; S[k][q] = sn * a + c * b; }
        for (int k = 0; k < 3; ++k) { double a = S[p][k], b = S[q][k]; S[p][k] = c * a - sn * b; S[q][k] = sn * a + c * b; }
        for (int k = 0; k < 3; ++k) { double a = E[k][p], b = E[k][q]; E[k][p] = c * a - sn * b; E[k][q] = sn * a + c * b; }
      }
  }
  int ord[3] = {0, 1, 2};
  for (int a = 0; a < 2; ++a)
    for (int b = a + 1; b < 3; ++b)
      if (S[ord[b]][ord[b]] < S[ord[a]][ord[a]]) { int t = ord[a]; ord[a] = ord[b]; ord[b] = t; }
  for (int c = 0; c < 3; ++c) {
    w[c] = S[ord[c]][ord[c]];
    for (int r = 0; r < 3; ++r) V[r * 3 + c] = E[r][ord[c]];
  }
}

}  // namespace mvr
