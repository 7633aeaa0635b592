// symmetric_oracle.cpp -- CPU checker of symmetric point-to-plane ICP (MVR_SYMMETRIC).  TEST INFRASTRUCTURE ONLY:
// tests/test_symmetric_icp.py compiles it into a temporary directory; the product never links it.
//
// It includes the CPU oracle (oracle/mvr_oracle.cpp) as it stands and adds, next to its point-to-point and point-to-plane
// estimators, PCL's TransformationEstimationSymmetricPointToPlaneLLS with enforce_same_direction_normals
// (pcl::IterativeClosestPointWithNormals with setUseSymmetricObjective(true), PCL >= 1.11), and the ICP loop of orc_icp_align
// with source normals that move with the source (transformPointCloudWithNormals).  The correspondences, the pinned float
// transform, the Cholesky solve and the convergence criteria are the oracle's own.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -fno-fast-math -fPIC [-fopenmp] -shared (the flags of oracle/Makefile).
#include "../oracle/mvr_oracle.cpp"

namespace {

// R(x0, x1, x2) = Rz Ry Rx, the rotation of estimate_p2plane_impl, row-major.
void rot_zyx(const double x[3], double R[3][3]) {
  const double ca = std::cos(x[0]), sa = std::sin(x[0]), cb = std::cos(x[1]), sb = std::sin(x[1]), cg = std::cos(x[2]), sg = std::sin(x[2]);
  const double M[3][3] = {{cg * cb, -sg * ca + cg * sb * sa, sg * sa + cg * sb * ca},
                          {sg * cb, cg * ca + sg * sb * sa, -cg * sa + sg * sb * ca},
                          {-sb, cb * sa, cb * ca}};
  std::memcpy(R, M, sizeof(M));
}

// Source normals in src_n (by source index, current orientation), target normals in tgt_n.  For each pair n = n1 + n2 if
// n1.n2 >= 0 else n1 - n2, v = [(p + q) x n, n], r = (q - p).n; a pair whose n is not finite is skipped.  Sums in double
// (PCL: Scalar = float).  T = R(x) Trans(x3, x4, x5) R(x) (constructTransformationMatrix).  x (nullable) receives the solution.
bool estimate_symmetric_impl(const P4* src, const P4* src_n, const P4* tgt, const P4* tgt_n, const std::vector<Corr>& corr, double T[16],
                             double* x_out = nullptr) {
  double A[6][6] = {}, b[6] = {};
  for (const Corr& c : corr) {
    const double sx = src[c.q].x, sy = src[c.q].y, sz = src[c.q].z, tx = tgt[c.m].x, ty = tgt[c.m].y, tz = tgt[c.m].z;
    const double ax = src_n[c.q].x, ay = src_n[c.q].y, az = src_n[c.q].z, bx = tgt_n[c.m].x, by = tgt_n[c.m].y, bz = tgt_n[c.m].z;
    const bool same = (ax * bx + ay * by) + az * bz >= 0.0;
    const double nx = same ? ax + bx : ax - bx, ny = same ? ay + by : ay - by, nz = same ? az + bz : az - bz;
    if (!(std::isfinite(nx) && std::isfinite(ny) && std::isfinite(nz))) continue;
    const double px = sx + tx, py = sy + ty, pz = sz + tz;
    const double J[6] = {py * nz - pz * ny, pz * nx - px * nz, px * ny - py * nx, nx, ny, nz};
    const double r = (nx * (tx - sx) + ny * (ty - sy)) + nz * (tz - sz);
    for (int i = 0; i < 6; ++i) { for (int j = 0; j < 6; ++j) A[i][j] += J[i] * J[j]; b[i] += J[i] * r; }
  }
  double x[6];
  if (!cholesky_solve6(A, b, x)) return false;
  if (x_out) std::memcpy(x_out, x, sizeof(x));
  double R[3][3];
  rot_zyx(x, R);
  for (int c = 0; c < 4; ++c) for (int r = 0; r < 4; ++r) T[c * 4 + r] = (r == c);
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) T[j * 4 + i] = (R[i][0] * R[0][j] + R[i][1] * R[1][j]) + R[i][2] * R[2][j];
    T[12 + i] = (R[i][0] * x[3] + R[i][1] * x[4]) + R[i][2] * x[5];
  }
  return true;
}

// Pinned normal rotation (float32, no FMA): n' = ((m00*nx + m01*ny) + m02*nz), curvature carried.
inline P4 rotate_normal(const float M[16], const P4& n) {
  P4 r;
  r.x = (M[0] * n.x + M[4] * n.y) + M[8] * n.z;
  r.y = (M[1] * n.x + M[5] * n.y) + M[9] * n.z;
  r.z = (M[2] * n.x + M[6] * n.y) + M[10] * n.z;
  r.w = n.w;
  return r;
}

}  // namespace

extern "C" {

// One symmetric step over the given correspondences: T (column-major) and x = (alpha, beta, gamma, tx, ty, tz).  1: not SPD.
int sym_estimate(const float* src, const float* src_normals, const float* tgt, const float* tgt_normals, const int* q, const int* m,
                 int count, double* T, double* x) {
  std::vector<Corr> c(count);
  for (int k = 0; k < count; ++k) c[k] = Corr{q[k], m[k], 0.f};
  return estimate_symmetric_impl((const P4*)src, (const P4*)src_normals, (const P4*)tgt, (const P4*)tgt_normals, c, T, x) ? 0 : 1;
}

// orc_icp_align with the symmetric estimator (prm->estimator is not read): src_normals = n x {nx, ny, nz, curvature} of the input
// source; a copy is turned by the guess's rotation at the start and by each increment's rotation after it.
int sym_icp_align(const float* src_in, const float* src_normals, int n, const float* tgt_in, int m, const float* tgt_normals,
                  const orc_icp_params* prm, const float* guess, float* final_out, orc_icp_report* rep, orc_iter_record* log, int max_log,
                  int* n_log) {
  const P4* src0 = (const P4*)src_in; const P4* tgt = (const P4*)tgt_in;
  if (!src_normals || !tgt_normals) return 1;
  std::vector<P4> cur(n), curn(n);
  float g[16];
  static const float I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  std::memcpy(g, guess ? guess : I16, sizeof(g));
  const bool guess_is_identity = std::memcmp(g, I16, sizeof(g)) == 0;
  for (int i = 0; i < n; ++i) {
    cur[i] = (guess_is_identity || !finite3(src0[i])) ? src0[i] : xform(g, src0[i]);
    curn[i] = rotate_normal(g, ((const P4*)src_normals)[i]);
  }
  double fin[16];
  for (int k = 0; k < 16; ++k) fin[k] = g[k];

  KdTree ttree; ttree.init(tgt, m);
  std::vector<Corr> corr;
  int iter = 0, reason = 0, converged = 0;
  double prev_mse = DBL_MAX, cur_mse = 0;
  int nlog = 0;
  unsigned long long queries = 0;
  const double rot_thr = 1.0 - prm->transformation_epsilon, trans_thr = prm->transformation_epsilon;
  const int min_corr = prm->min_correspondences > 0 ? prm->min_correspondences : 3;
  if (prm->max_iterations <= 0) { reason = 1; converged = 1; }
  while (!converged) {
    correspondences_impl(cur.data(), n, tgt, ttree, prm->max_correspondence_distance, prm->use_reciprocal, corr, &queries);
    if ((int)corr.size() < min_corr) { reason = 5; converged = 0; break; }
    double T[16];
    if (!estimate_symmetric_impl(cur.data(), curn.data(), tgt, (const P4*)tgt_normals, corr, T)) { reason = 5; break; }
    float Tf[16];
    for (int k = 0; k < 16; ++k) Tf[k] = (float)T[k];
    Tf[3] = Tf[7] = Tf[11] = 0.f; Tf[15] = 1.f;
    for (int i = 0; i < n; ++i) {
      if (finite3(cur[i])) cur[i] = xform(Tf, cur[i]);
      curn[i] = rotate_normal(Tf, curn[i]);
    }
    double Td[16];
    for (int k = 0; k < 16; ++k) Td[k] = Tf[k];
    matmul4d(Td, fin, fin);
    ++iter;
    double s = 0; for (const Corr& c : corr) s += c.d2;
    cur_mse = s / (double)corr.size();
    if (log && nlog < max_log) {
      log[nlog].iteration = iter; log[nlog].n_corr = (int)corr.size(); log[nlog].mse = cur_mse;
      for (int k = 0; k < 16; ++k) log[nlog].delta[k] = Td[k];
      ++nlog;
    }
    if (iter >= prm->max_iterations) { converged = 1; reason = 1; break; }
    if (!prm->fixed_iterations) {
      const double cos_angle = 0.5 * (Td[0] + Td[5] + Td[10] - 1.0);
      const double t2 = Td[12] * Td[12] + Td[13] * Td[13] + Td[14] * Td[14];
      if (cos_angle >= rot_thr && t2 <= trans_thr) { converged = 1; reason = 2; break; }
      if (std::fabs(cur_mse - prev_mse) < 1e-12) { converged = 1; reason = 3; break; }
      if (std::fabs(cur_mse - prev_mse) / prev_mse < prm->euclidean_fitness_epsilon) { converged = 1; reason = 4; break; }
      prev_mse = cur_mse;
    }
  }
  if (final_out) for (int k = 0; k < 16; ++k) final_out[k] = (float)fin[k];
  if (rep) { rep->iterations = iter; rep->converged = converged; rep->reason = reason; rep->n_correspondences = (int)corr.size(); rep->mse = cur_mse; rep->nn_queries = queries; }
  if (n_log) *n_log = nlog;
  return reason == 5 ? 2 : 0;
}

}  // extern "C"
