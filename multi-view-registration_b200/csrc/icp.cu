// icp.cu -- per-iteration ICP kernels (the search itself is in pair_search.cuh): estimator sums (K6 point-to-point 3x3 cross-covariance, K9 point-to-plane and
// symmetric point-to-plane 6x6 normal equations)
// with the solve and the convergence test in the reduction's last block, fitness reduction (K8) and
// order-preserving correspondence compaction.
//
// Restates, for the GPU, what pcl::IterativeClosestPoint does per iteration inside icp.align()
// (reference call sites mvr/src/registrator.cpp:569, 920, 1012, 1024; semantics SURVEY.md A3-A8):
//   determine(Reciprocal)Correspondences -> TransformationEstimationSVD -> transformCloud ->
//   DefaultConvergenceCriteria.
// The whole loop state lives in an IcpState on the device, so an align needs no host round trip per
// iteration: the host only enqueues iterations and reads the state back when a batch has run.
#include <algorithm>

#include "launch.h"
#include "pair_search.cuh"
#ifdef MVR_TS_TILE
#include "tile_search.cuh"
#endif
#include "small_solve.h"

// candidates evaluated per trip of the flat scan = independent 16-byte loads in flight per thread (measured: 8 > 4 > 2)
// resident 256-thread blocks per SM the register allocation aims at (forward reciprocal half / reverse half);
// measured on B200, same box, 24 x 200k pairs: (4, 3) 37.5 ms, (5, 3) 36.5, (4, 4) 34.9, (5, 4) 33.9, (5, 5) 34.3, (6, 6) 36.4
#ifndef MVR_FWD_MINBLOCKS
#define MVR_FWD_MINBLOCKS 5
#endif
#ifndef MVR_FWD1_MINBLOCKS
#define MVR_FWD1_MINBLOCKS 3   // one-way forward kernel (search + estimator sums)
#endif
#ifndef MVR_REV_MINBLOCKS
#define MVR_REV_MINBLOCKS 4
#endif
#ifndef MVR_PG_UNROLL
#define MVR_PG_UNROLL 6
#endif

namespace mvr {

// ---------------------------------------------------------------------------------------------
// estimator sums: fixed topology (thread grid-stride over ORIGINAL indices -> warp shuffle tree ->
// 8 warps in order -> REDUCE_BLOCKS partials summed in block order by the last block to finish), so
// results are identical run to run and do not depend on the order of points inside grid cells.
// ---------------------------------------------------------------------------------------------
// WARPS = warps of the calling block (8 for the 256-thread utility kernels, FUSED_WARPS for the fused iteration).
template <int NV, int WARPS = 8>
__device__ __forceinline__ void block_reduce_store(double (&v)[NV], double* __restrict__ partials) {
  __shared__ double sm[WARPS][NV];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double x = v[a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) sm[warp][a] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double x = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) x += sm[w][threadIdx.x];
    partials[(size_t)blockIdx.x * REDUCE_MAX_VALS + threadIdx.x] = x;
  }
}

// True in exactly one block per launch: the one that finished last.  On return in that block every
// block's partials are visible.
__device__ __forceinline__ bool last_block_done(unsigned int* ticket, unsigned int nblk) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(ticket, 1u);
    is_last = (t == nblk - 1);
    if (is_last) *ticket = 0;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// Ordered sum of the blocks' partials: FUSED_WARPS chunks of consecutive blocks summed in parallel (each in block
// order, 8 loads in flight), then the chunk sums in chunk order.  Called by all threads of the last block.
template <int NV>
__device__ __forceinline__ void ordered_total(const double* __restrict__ partials, int nblk, double* __restrict__ out) {
  __shared__ double ch[FUSED_WARPS][REDUCE_MAX_VALS];
  const int a = threadIdx.x & 31, c = threadIdx.x >> 5;
  const int per = (nblk + FUSED_WARPS - 1) / FUSED_WARPS;
  if (a < NV) {
    const int b0 = c * per, b1 = min(b0 + per, nblk);
    double x = 0;
    int b = b0;
    for (; b + 8 <= b1; b += 8) {
      double t[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) t[u] = __ldcg(partials + (size_t)(b + u) * REDUCE_MAX_VALS + a);
#pragma unroll
      for (int u = 0; u < 8; ++u) x += t[u];
    }
    for (; b < b1; ++b) x += __ldcg(partials + (size_t)b * REDUCE_MAX_VALS + a);
    ch[c][a] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double x = 0;
#pragma unroll
    for (int k = 0; k < FUSED_WARPS; ++k) x += ch[k][threadIdx.x];
    out[threadIdx.x] = x;
  }
  __syncthreads();
}

// The source index is kept in the frame the source was binned in (pair_index.cu).  cum = the increments
// applied since then (including the one the next iteration will apply), cinv its affine inverse, stretch
// an upper bound of ||A^-1||_2 for its linear part A (1 for an exact rotation; float-rounded rotations
// drift by ~1e-7 per iteration).  With eta = ||A^T A - I||_F: lambda_min(A^T A) >= 1 - eta.
__device__ __forceinline__ void icp_advance_frame(IcpState* st, const double (&Td)[16]) {
  double C0[16], C[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) C0[k] = st->cum[k];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      double x = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) x += Td[k * 4 + r] * C0[c * 4 + k];
      C[c * 4 + r] = x;
    }
#pragma unroll
  for (int k = 0; k < 16; ++k) st->cum[k] = C[k];
  // A(r, c) = C[c * 4 + r]
  const double a00 = C[0], a10 = C[1], a20 = C[2], a01 = C[4], a11 = C[5], a21 = C[6], a02 = C[8], a12 = C[9], a22 = C[10];
  const double c00 = a11 * a22 - a12 * a21, c01 = a12 * a20 - a10 * a22, c02 = a10 * a21 - a11 * a20;
  const double det = a00 * c00 + a01 * c01 + a02 * c02;
  const double id = 1.0 / det;
  double I[9];   // row-major inverse
  I[0] = c00 * id; I[1] = (a02 * a21 - a01 * a22) * id; I[2] = (a01 * a12 - a02 * a11) * id;
  I[3] = c01 * id; I[4] = (a00 * a22 - a02 * a20) * id; I[5] = (a02 * a10 - a00 * a12) * id;
  I[6] = c02 * id; I[7] = (a01 * a20 - a00 * a21) * id; I[8] = (a00 * a11 - a01 * a10) * id;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    st->cinv[r * 4 + 0] = I[r * 3 + 0]; st->cinv[r * 4 + 1] = I[r * 3 + 1]; st->cinv[r * 4 + 2] = I[r * 3 + 2];
    st->cinv[r * 4 + 3] = -(I[r * 3 + 0] * C[12] + I[r * 3 + 1] * C[13] + I[r * 3 + 2] * C[14]);
  }
  double eta2 = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double g = C[i * 4 + 0] * C[j * 4 + 0] + C[i * 4 + 1] * C[j * 4 + 1] + C[i * 4 + 2] * C[j * 4 + 2] - ((i == j) ? 1.0 : 0.0);
      eta2 += g * g;
    }
  const double eta = sqrt(eta2);
  // not a rigid motion any more (cannot happen with the estimators here): make every bound vacuous
  st->stretch = (eta < 0.5 && det > 0) ? (float)(1.0 / sqrt(1.0 - eta)) * 1.000001f + 1.0e-7f : 1.0e6f;
  st->n_gate = 0u;

  // How far the chain of in-place float transforms can have drifted from cum * (binning-time position) once the
  // pending increment Td has been applied (k_icp_forward does that at the start of the next iteration):
  //   cur' = fl(Td cur) = Td cur + e,  cum' = Td cum   =>   cur' - cum' s0 = A_Td (cur - cum s0) + e,
  // so dev' <= ||A_Td||_2 dev + |e|.  One pinned transform rounds every term at most four times (xform_pinned: product,
  // three sums), so per axis |e_r| <= 4.1 u (sum_j |Td_rj| B_j + |Td_r3|) with u = 2^-24 and B_j >= |coordinate j| of
  // every point before the step; ||A_Td||_2 <= sqrt(1 + ||A_Td^T A_Td - I||_F).
  const double u4 = 4.1 * 5.9604644775390625e-8;
  double e2 = 0, etaT2 = 0;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const double er = u4 * (fabs(Td[r]) * st->babs[0] + fabs(Td[4 + r]) * st->babs[1] + fabs(Td[8 + r]) * st->babs[2] + fabs(Td[12 + r])) + 1.0e-30;
    e2 += er * er;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double g = Td[i * 4 + 0] * Td[j * 4 + 0] + Td[i * 4 + 1] * Td[j * 4 + 1] + Td[i * 4 + 2] * Td[j * 4 + 2] - ((i == j) ? 1.0 : 0.0);
      etaT2 += g * g;
    }
  const double devn = st->devd * sqrt(1.0 + sqrt(etaT2)) * (1.0 + 1.0e-9) + sqrt(e2) * (1.0 + 1.0e-9);
  st->devd = devn;
  st->dev = __double2float_ru(devn) * 1.000001f;
  // the moved cloud lies in cum' * (binning box) widened by dev'
  double bn[3] = {0, 0, 0};
#pragma unroll
  for (int c8 = 0; c8 < 8; ++c8) {
    const double px = st->box[(c8 & 1) ? 3 : 0], py = st->box[(c8 & 2) ? 4 : 1], pz = st->box[(c8 & 4) ? 5 : 2];
#pragma unroll
    for (int r = 0; r < 3; ++r) bn[r] = fmax(bn[r], fabs(C[r] * px + C[4 + r] * py + C[8 + r] * pz + C[12 + r]));
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) st->babs[r] = (bn[r] + devn) * (1.0 + 1.0e-6) + 1.0e-3;
}

// The tail of one ICP iteration, run by one thread: estimate the increment from the sums, compose it
// into the accumulated transform, log, and evaluate DefaultConvergenceCriteria (SURVEY.md A8).
// SYM: the symmetric objective's increment (a separate instance: the others compile as they did before it existed).
template <bool SYM>
__device__ __noinline__ void icp_finish_iteration(IcpState* st, IterRec* log) {
  // everything the step needs, fetched up front so the loads overlap (st lives in global memory)
  double S[REDUCE_MAX_VALS], F0[16];
#pragma unroll
  for (int k = 0; k < REDUCE_MAX_VALS; ++k) S[k] = st->sums[k];
#pragma unroll
  for (int k = 0; k < 16; ++k) F0[k] = st->fin[k];
  const bool p2l = st->p2l != 0;   // 0 point-to-point, 1 point-to-plane, 2 symmetric point-to-plane (SYM)
  const double ox = st->ox, oy = st->oy, oz = st->oz;
  const int min_corr = st->min_corr, max_iter = st->max_iter, fixed = st->fixed, iter0 = st->iter;
  const double prev_mse = st->prev_mse, rot_thr = st->rot_thr, trans_thr = st->trans_thr, fit_eps = st->fit_eps;
  const double cnt = p2l ? S[27] : S[0];
  const double d2sum = p2l ? S[28] : S[16];
  st->queries += (unsigned long long)st->n_src + (st->recip ? (unsigned long long)st->n_gate : 0ull);
  const int n_corr = (int)cnt;
  st->n_corr = n_corr;
  if (n_corr < min_corr) { st->reason = 5; st->status = 2; st->done = 1; return; }  // "Not enough correspondences"
  double T[16];
  if (p2l) {
    double A[36], b[6], x[6];
    int k = 0;
    for (int a = 0; a < 6; ++a)
      for (int c = a; c < 6; ++c) { A[a * 6 + c] = S[k]; A[c * 6 + a] = S[k]; ++k; }
    for (int a = 0; a < 6; ++a) b[a] = S[21 + a];
    if (!cholesky_solve6(A, b, x)) { st->reason = 5; st->status = 5; st->done = 1; return; }
    if constexpr (SYM) pose_from_6_symmetric(x, T);
    else pose_from_6(x, T);
  } else {
    const double inv = 1.0 / cnt;
    const double mu_a[3] = {S[1] * inv, S[2] * inv, S[3] * inv}, mu_b[3] = {S[4] * inv, S[5] * inv, S[6] * inv};
    double Sg[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) Sg[r * 3 + c] = S[7 + r * 3 + c] * inv - mu_b[r] * mu_a[c];
    const double mu_s[3] = {mu_a[0] + ox, mu_a[1] + oy, mu_a[2] + oz};
    const double mu_d[3] = {mu_b[0] + ox, mu_b[1] + oy, mu_b[2] + oz};
    umeyama_rigid(mu_s, mu_d, Sg, T);
  }
  float Tf[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) Tf[k] = (float)T[k];
  Tf[3] = Tf[7] = Tf[11] = 0.f; Tf[15] = 1.f;
  double Td[16], F[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) Td[k] = Tf[k];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      double x = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) x += Td[k * 4 + r] * F0[c * 4 + k];
      F[c * 4 + r] = x;
    }
#pragma unroll
  for (int k = 0; k < 16; ++k) { st->fin[k] = F[k]; st->delta[k] = Tf[k]; }
  icp_advance_frame(st, Td);
  const int iter = iter0 + 1;
  st->iter = iter;
  const double cur_mse = d2sum / cnt;
  st->cur_mse = cur_mse;
  if (iter <= ICP_MAX_LOG) {
    IterRec& r = log[iter - 1];
    r.iteration = iter; r.n_corr = n_corr; r.mse = cur_mse;
#pragma unroll
    for (int k = 0; k < 16; ++k) r.delta[k] = Tf[k];
  }
  if (iter >= max_iter) { st->done = 1; st->reason = 1; return; }
  if (!fixed) {
    const double cos_angle = 0.5 * (Td[0] + Td[5] + Td[10] - 1.0);
    const double t2 = Td[12] * Td[12] + Td[13] * Td[13] + Td[14] * Td[14];
    if (cos_angle >= rot_thr && t2 <= trans_thr) { st->done = 1; st->reason = 2; return; }
    if (fabs(cur_mse - prev_mse) < 1e-12) { st->done = 1; st->reason = 3; return; }
    if (fabs(cur_mse - prev_mse) / prev_mse < fit_eps) { st->done = 1; st->reason = 4; return; }
    st->prev_mse = cur_mse;
  }
}

// ---------------------------------------------------------------------------------------------
// The fused iteration.  Per iteration of pcl::IterativeClosestPoint::computeTransformation (SURVEY.md A3):
//   k_icp_forward : transformCloud (the pending increment, in place) + determineCorrespondences
//                   (exact 1-NN in the target, gate) for every source point; without reciprocal
//                   correspondences also the estimator sums, the solve and the criteria;
//   k_icp_reverse : the reciprocal half of determineReciprocalCorrespondences (A5) -- for every target
//                   point some source point chose, its nearest source point -- fused with the estimator
//                   sums over the mutual pairs, the solve and the criteria.
// Two launches per iteration, no host round trip.  Both kernels walk SORTED positions with a fixed
// grid, and sorted positions are reproducible (pair_index.cu), so the sums are identical run to run.
// ---------------------------------------------------------------------------------------------

// Point-to-point sums about the origin o (a = s - o, b = t - o, exact in double):
// [0] n, [1..3] sum a, [4..6] sum b, [7..15] sum b_r * a_c (row r, col c), [16] sum d2.
__device__ __forceinline__ void acc_p2p(double (&v)[REDUCE_P2P_VALS], float4 s, float4 t, float d2, double ox, double oy, double oz) {
  const double ax = (double)s.x - ox, ay = (double)s.y - oy, az = (double)s.z - oz;
  const double bx = (double)t.x - ox, by = (double)t.y - oy, bz = (double)t.z - oz;
  v[0] += 1.0;
  v[1] += ax; v[2] += ay; v[3] += az;
  v[4] += bx; v[5] += by; v[6] += bz;
  v[7] += bx * ax; v[8] += bx * ay; v[9] += bx * az;
  v[10] += by * ax; v[11] += by * ay; v[12] += by * az;
  v[13] += bz * ax; v[14] += bz * ay; v[15] += bz * az;
  v[16] += (double)d2;
}

// Second moments on top of the point-to-point sums (the edge statistics of the LUM relaxation, lum.cpp):
// [17..22] sum a a^T (xx, xy, xz, yy, yz, zz), [23..28] sum b b^T.
__device__ __forceinline__ void acc_mom(double (&v)[REDUCE_MOM_VALS], float4 s, float4 t, float d2, double ox, double oy, double oz) {
  const double ax = (double)s.x - ox, ay = (double)s.y - oy, az = (double)s.z - oz;
  const double bx = (double)t.x - ox, by = (double)t.y - oy, bz = (double)t.z - oz;
  v[0] += 1.0;
  v[1] += ax; v[2] += ay; v[3] += az;
  v[4] += bx; v[5] += by; v[6] += bz;
  v[7] += bx * ax; v[8] += bx * ay; v[9] += bx * az;
  v[10] += by * ax; v[11] += by * ay; v[12] += by * az;
  v[13] += bz * ax; v[14] += bz * ay; v[15] += bz * az;
  v[16] += (double)d2;
  v[17] += ax * ax; v[18] += ax * ay; v[19] += ax * az; v[20] += ay * ay; v[21] += ay * az; v[22] += az * az;
  v[23] += bx * bx; v[24] += bx * by; v[25] += bx * bz; v[26] += by * by; v[27] += by * bz; v[28] += bz * bz;
}

// Point-to-plane normal equations (SURVEY.md A12): J = [cross(s, n), n], r = n.(d - s).
// [0..20] upper triangle of J^T J row-major, [21..26] J^T r, [27] n, [28] sum d2.
__device__ __forceinline__ void acc_p2l(double (&v)[REDUCE_P2L_VALS], float4 s, float4 t, float4 nn, float d2) {
  const double sx = s.x, sy = s.y, sz = s.z, nx = nn.x, ny = nn.y, nz = nn.z;
  const double J[6] = {nz * sy - ny * sz, nx * sz - nz * sx, ny * sx - nx * sy, nx, ny, nz};
  const double r = nx * ((double)t.x - sx) + ny * ((double)t.y - sy) + nz * ((double)t.z - sz);
  int k = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = a; b < 6; ++b) v[k++] += J[a] * J[b];
#pragma unroll
  for (int a = 0; a < 6; ++a) v[21 + a] += J[a] * r;
  v[27] += 1.0;
  v[28] += (double)d2;
}

// Symmetric point-to-plane normal equations (TransformationEstimationSymmetricPointToPlaneLLS), the layout of acc_p2l:
// n = n1 + n2 when n1.n2 >= 0, else n1 - n2 (enforce_same_direction_normals), v = [cross(s + t, n), n], r = n.(t - s).
// A pair whose n is not finite adds nothing to the system but still counts (and its d2 still enters the mse).
__device__ __forceinline__ void acc_sym(double (&v)[REDUCE_P2L_VALS], float4 s, float4 t, float4 n1, float4 n2, float d2) {
  const double sx = s.x, sy = s.y, sz = s.z, tx = t.x, ty = t.y, tz = t.z;
  const double ax = n1.x, ay = n1.y, az = n1.z, bx = n2.x, by = n2.y, bz = n2.z;
  const bool same = (ax * bx + ay * by) + az * bz >= 0.0;
  const double nx = same ? ax + bx : ax - bx, ny = same ? ay + by : ay - by, nz = same ? az + bz : az - bz;
  v[27] += 1.0;
  v[28] += (double)d2;
  if (!(isfinite(nx) && isfinite(ny) && isfinite(nz))) return;
  const double px = sx + tx, py = sy + ty, pz = sz + tz;
  const double J[6] = {py * nz - pz * ny, pz * nx - px * nz, px * ny - py * nx, nx, ny, nz};
  const double r = (nx * (tx - sx) + ny * (ty - sy)) + nz * (tz - sz);
  int k = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = a; b < 6; ++b) v[k++] += J[a] * J[b];
#pragma unroll
  for (int a = 0; a < 6; ++a) v[21 + a] += J[a] * r;
}

// block_reduce_store + last_block_done in one: the block's partial is written, fenced and the ticket drawn by warp 0 alone
// (the threads that wrote are the ones that fence), so the block's tail is two barriers instead of three and seven warps
// skip the memory fence.  Same sums in the same order.
template <int NV>
__device__ __forceinline__ bool block_reduce_ticket(double (&v)[NV], double* __restrict__ partials, unsigned int* ticket, unsigned int nblk) {
  __shared__ double sm[FUSED_WARPS][NV];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double x = v[a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) sm[warp][a] = x;
  }
  __syncthreads();
  if (warp == 0) {
    static_assert(NV <= 32, "one warp writes the partial");
    if (lane < NV) {
      double x = 0;
#pragma unroll
      for (int w = 0; w < FUSED_WARPS; ++w) x += sm[w][lane];
      partials[(size_t)blockIdx.x * REDUCE_MAX_VALS + lane] = x;
      __threadfence();
    }
    __syncwarp();
    if (lane == 0) {
      const unsigned int t = atomicAdd(ticket, 1u);
      is_last = (t == nblk - 1);
      if (is_last) *ticket = 0;
    }
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// Block partials -> (last block) ordered total -> solve, compose, criteria.
template <int NV, bool SYM = false>
__device__ __forceinline__ void reduce_and_finish(double (&v)[NV], double* __restrict__ partials, IcpState* __restrict__ st,
                                                  IterRec* __restrict__ log, int nblk) {
  if (!block_reduce_ticket<NV>(v, partials, &st->ticket, (unsigned int)nblk)) return;
  ordered_total<NV>(partials, nblk, st->sums);
  if (threadIdx.x == 0) {
    const long long t0 = clock64();
    icp_finish_iteration<SYM>(st, log);
    st->dbg[0] += clock64() - t0; st->dbg[1] += 1;
  }
}

template <int EST> struct EstVals {
  static constexpr int value = (EST == EST_P2L || EST == EST_SYM) ? (int)REDUCE_P2L_VALS : (EST == EST_MOM ? (int)REDUCE_MOM_VALS : (int)REDUCE_P2P_VALS);
};

// ns: the source point's normal (symmetric only; read by nothing else)
template <int EST, int NV>
__device__ __forceinline__ void acc_pair(double (&v)[NV], float4 s, float4 t, const float4* __restrict__ nrm, const float4* ns, float d2, double ox, double oy, double oz) {
  if constexpr (EST == EST_SYM) acc_sym(v, s, t, *ns, __ldg(nrm + __float_as_int(t.w)), d2);
  else if constexpr (EST == EST_P2L) acc_p2l(v, s, t, __ldg(nrm + __float_as_int(t.w)), d2);
  else if constexpr (EST == EST_MOM) acc_mom(v, s, t, d2, ox, oy, oz);
  else acc_p2p(v, s, t, d2, ox, oy, oz);
}

// Phase A of both kernels is the search (registers: the query, the running best, grid geometry); phase B
// re-reads the matches and accumulates the estimator sums (registers: 18-30 doubles).  The two never overlap, so a
// kernel's register budget is the larger of the two, not their sum.
// The seed of source point i: last iteration's neighbour is a real candidate and usually still the answer.
__device__ __forceinline__ void fwd_seed(const FwdArgs& a, int i, const float4 p, NnBest& b) {
  b = NnBest{MVR_INF, 0x7fffffff, -1};
  const int j0 = a.corr_p[i];
  if (j0 >= 0) {
    const float4 t = __ldg(a.tgt + j0);
    b.d2 = d2_pinned(p.x, p.y, p.z, t.x, t.y, t.z); b.idx = __float_as_int(t.w); b.pos = j0;
  }
}

template <bool RECIP>
__device__ __forceinline__ void fwd_commit(const FwdArgs& a, int i, const NnBest& b, unsigned int& ngate) {
  const bool keep = b.pos >= 0 && !((double)b.d2 > a.max2);   // PCL: if (distance > max_dist_sqr) continue;
  a.corr_p[i] = keep ? b.pos : -1;
  if (keep) {
    ++ngate;
    if (RECIP) atomicMin(a.rmin + b.pos, __float_as_uint(b.d2));
  }
}

#ifdef MVR_TS_TILE
#include "icp_tile.cuh"
#else
template <bool RECIP, int EST>
__global__ void __launch_bounds__(FUSED_THREADS, (RECIP ? MVR_FWD_MINBLOCKS : MVR_FWD1_MINBLOCKS) * (256 / FUSED_THREADS)) k_icp_forward(const __grid_constant__ FwdBatch batch, int first) {
  // this pair's arguments: parameter space -> shared memory (a dynamically indexed parameter would be copied to
  // local memory and pin registers)
  __shared__ FwdArgs s_args;
  static_assert(sizeof(FwdArgs) % 4 == 0 && sizeof(FwdArgs) / 4 <= FUSED_THREADS, "argument block");
  if (threadIdx.x < sizeof(FwdArgs) / 4) ((uint32_t*)&s_args)[threadIdx.x] = ((const uint32_t*)&batch.a[blockIdx.y])[threadIdx.x];
  __syncthreads();
  const FwdArgs& a = s_args;
  if ((int)blockIdx.x >= a.grid) return;
  IcpState* __restrict__ st = a.st;
  if (st->done) return;
  const int stride = a.grid * FUSED_THREADS;
  __shared__ uint2 s_seg[PG_SEGS * PG_STRIDE];
  uint2* seg = s_seg + threadIdx.x;
  Mat4f M;
  if (!first) {
#pragma unroll
    for (int k = 0; k < 16; ++k) M.m[k] = st->delta[k];
  }
  unsigned int ngate = 0;
  for (int i = blockIdx.x * FUSED_THREADS + threadIdx.x; i < a.n_valid; i += stride) {
    float4 p = a.cur[i];
    if (!first) {
      const float w = p.w;
      p = xform_pinned(M, p);
      p.w = w;
      a.cur[i] = p;
      if constexpr (EST == EST_SYM) a.nsrc[i] = rotate_pinned(M, a.nsrc[i]);   // the source normals move with the source
    }
    NnBest b;
    fwd_seed(a, i, p, b);
    // no partner inside the gate so far: one bit says whether the target has anything within the gate of p's cell
    if (a.gmask && !(b.d2 <= a.max_d2f)) {
      const int cx = pg_cell(grid_t(p.x, a.gt.ox, a.gt.inv_cell_x), a.gt.nx), cy = pg_cell(grid_t(p.y, a.gt.oy, a.gt.inv_cell), a.gt.ny),
                cz = pg_cell(grid_t(p.z, a.gt.oz, a.gt.inv_cell), a.gt.nz);
      const uint32_t wd = __ldg(a.gmask + ((size_t)cz * a.gt.ny + cy) * a.gm_stride + (cx >> 5));
      if (!((wd >> (cx & 31)) & 1u)) { a.corr_p[i] = -1; continue; }
    }
    pg_search<MVR_PG_UNROLL>(a.gt, a.tstart, a.tgt, a.m_valid, p.x, p.y, p.z, p.x, p.y, p.z, 0.0f, 1.0f, a.max_d2f, b, seg);
    fwd_commit<RECIP>(a, i, b, ngate);
  }
  if (RECIP) {
    // warp-level: no block barrier, a warp that is done is done
    const unsigned int wg = __reduce_add_sync(0xffffffffu, ngate);
    if ((threadIdx.x & 31) == 0 && wg) atomicAdd(&st->n_gate, wg);
  } else {
    // phase B: every thread revisits exactly the points it searched (its own writes, no barrier needed)
    const double ox = st->ox, oy = st->oy, oz = st->oz;
    constexpr int NV = EstVals<EST>::value;
    double v[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = 0.0;
    for (int i = blockIdx.x * FUSED_THREADS + threadIdx.x; i < a.n_valid; i += stride) {
      const int j = a.corr_p[i];
      if (j < 0) continue;
      const float4 p = a.cur[i];
      const float4 t = __ldg(a.tgt + j);
      acc_pair<EST>(v, p, t, a.nrm, a.nsrc + i, d2_pinned(p.x, p.y, p.z, t.x, t.y, t.z), ox, oy, oz);
    }
    reduce_and_finish<NV, EST == EST_SYM>(v, a.partials, st, a.log, a.grid);
  }
}

// Reciprocal half.  Only the target points some source point chose are searched: a block compacts the chosen ones
// of its `per` chunks of 256 target points (in order, deterministic) into a list in shared memory, every thread then
// searches its entries of the list, and sums over its own mutual pairs afterwards (phase B needs no barrier: a thread
// revisits exactly the entries it searched, so a warp that is done does not wait for the slowest one of the block).
#ifndef MVR_REV_MAX_CHUNKS
#define MVR_REV_MAX_CHUNKS 4
#endif
constexpr int REV_MAX_CHUNKS = MVR_REV_MAX_CHUNKS;
template <int EST>
__global__ void __launch_bounds__(FUSED_THREADS, MVR_REV_MINBLOCKS * (256 / FUSED_THREADS)) k_icp_reverse(const __grid_constant__ RevBatch batch) {
  __shared__ RevArgs s_args;
  static_assert(sizeof(RevArgs) % 4 == 0 && sizeof(RevArgs) / 4 <= FUSED_THREADS, "argument block");
  if (threadIdx.x < sizeof(RevArgs) / 4) ((uint32_t*)&s_args)[threadIdx.x] = ((const uint32_t*)&batch.a[blockIdx.y])[threadIdx.x];
  __syncthreads();
  const RevArgs& a = s_args;
  if ((int)blockIdx.x >= a.grid) return;
  IcpState* __restrict__ st = a.st;
  if (st->done) return;
  __shared__ uint2 s_seg[PG_SEGS * PG_STRIDE];
  __shared__ int s_q[REV_MAX_CHUNKS * FUSED_THREADS];   // the block's chosen target points (sorted positions), in order
  __shared__ int s_p[REV_MAX_CHUNKS * FUSED_THREADS];   // in: bits of the nearest chooser's d2; out: the mutual partner (sorted source position), -1 none
  __shared__ int s_wcnt[FUSED_WARPS];
  uint2* seg = s_seg + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // ---- the block's list
  const int chunks = (a.m_valid + FUSED_THREADS - 1) / FUSED_THREADS;
  int qn = 0;   // the same in every thread
  for (int cc = 0; cc < a.per; ++cc) {
    const int c = blockIdx.x * a.per + cc;
    if (c >= chunks) break;
    const int j = c * FUSED_THREADS + threadIdx.x;
    uint32_t r = 0x7f800000u;
    if (j < a.m_valid) {
      r = a.rmin[j];
      if (r != 0x7f800000u) a.rmin[j] = 0x7f800000u;   // re-armed for the next iteration
    }
    const bool chosen = r != 0x7f800000u;
    const unsigned int bal = __ballot_sync(0xffffffffu, chosen);
    if (lane == 0) s_wcnt[warp] = __popc(bal);
    __syncthreads();
    int ofs = qn, tot = 0;
#pragma unroll
    for (int w = 0; w < FUSED_WARPS; ++w) { const int n = s_wcnt[w]; if (w < warp) ofs += n; tot += n; }
    if (chosen) { const int k = ofs + __popc(bal & ((1u << lane) - 1u)); s_q[k] = j; s_p[k] = (int)r; }
    qn += tot;
    __syncthreads();
  }

  // ---- phase A: the searches
  const float stretch = st->stretch;
  const float dev0 = st->dev;
  unsigned int missed = 0;
  for (int k = threadIdx.x; k < qn; k += FUSED_THREADS) {
    const int j = s_q[k];
    const float4 t = __ldg(a.tgt + j);
    // the query in the frame the source was binned in
    const float ux = (float)(st->cinv[0] * t.x + st->cinv[1] * t.y + st->cinv[2] * t.z + st->cinv[3]);
    const float uy = (float)(st->cinv[4] * t.x + st->cinv[5] * t.y + st->cinv[6] * t.z + st->cinv[7]);
    const float uz = (float)(st->cinv[8] * t.x + st->cinv[9] * t.y + st->cinv[10] * t.z + st->cinv[11]);
    const float dev = dev0 + 1.0e-6f * fmaxf(fabsf(ux), fmaxf(fabsf(uy), fabsf(uz)));
    // a chooser sits at exactly this distance: the lexicographic minimum (d2, index) over all source points is found
    NnBest b{__uint_as_float((uint32_t)s_p[k]), 0x7fffffff, -1};
    pg_search<MVR_PG_UNROLL>(a.gs, a.sstart, a.cur, a.n_valid, t.x, t.y, t.z, ux, uy, uz, dev, stretch, MVR_INF, b, seg);
    if (b.pos < 0) ++missed;
    const int mutual = (b.pos >= 0 && __ldg(a.corr_p + b.pos) == j) ? b.pos : -1;   // or the nearest source point chose another target
    s_p[k] = mutual;
    if (a.rnn) a.rnn[j] = mutual;
  }
  if (missed) atomicAdd((unsigned long long*)&st->dbg[2], (unsigned long long)missed);   // must stay 0: a chooser was not found again

  // ---- phase B: the sums over this thread's own mutual pairs
  const double ox = st->ox, oy = st->oy, oz = st->oz;
  constexpr int NV = EstVals<EST>::value;
  double v[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) v[k] = 0.0;
  for (int k = threadIdx.x; k < qn; k += FUSED_THREADS) {
    const int r = s_p[k];
    if (r < 0) continue;
    const float4 t = __ldg(a.tgt + s_q[k]);
    const float4 s = a.cur[r];
    acc_pair<EST>(v, s, t, a.nrm, a.nsrc + r, d2_pinned(t.x, t.y, t.z, s.x, s.y, s.z), ox, oy, oz);
  }
  reduce_and_finish<NV, EST == EST_SYM>(v, a.partials, st, a.log, a.grid);
}
#endif   // MVR_TS_TILE

// (Tried in round 2 and dropped, profiles/r02_dynamic_items_ab.log: resident blocks drawing their chunks from a counter instead of
// one block per chunk -- 12 % slower with 24 pairs per launch, no gain with 3.)
// Chunks of 256 target points per block of the reverse half: enough for its compacted list to fill whole rounds of
// 256 searches (about half of the target points are chosen).  Measured on B200 (same box; 24 x 200k pairs per launch /
// one 200k pair alone): 2 chunks 25.3 ms / 2.06 ms, 3 chunks 24.1 / 2.08, 4 chunks 24.0 / 2.23 -- three chunks, four once
// a cloud fills the GPU on its own.  A pure function of the cloud size, so that the block partition, and with it the
// order of the sums, does not depend on what else runs in the batch.
int fused_rev_chunks(int items) {
#ifdef MVR_REV_CHUNKS
  return MVR_REV_CHUNKS;
#else
#ifdef MVR_TS_TILE
  (void)items;
  return 2;   // about half of the target points are chosen: two chunks fill one tile of 256 searches
#else
  return items >= 400000 ? 4 : 3;
#endif
#endif
}
int fused_grid_rev(int items) {
  const int chunks = (items + FUSED_THREADS - 1) / FUSED_THREADS;
  const int per = fused_rev_chunks(items);
  const int blocks = (chunks + per - 1) / per;   // not capped: every block takes exactly `per` chunks
  return blocks < 1 ? 1 : blocks;
}

int fused_grid(int items) {
  const int blocks = (items + FUSED_THREADS - 1) / FUSED_THREADS;
  return blocks < 1 ? 1 : (blocks > FUSED_MAX_BLOCKS ? FUSED_MAX_BLOCKS : blocks);
}

#ifdef MVR_SMEM_CARVEOUT
static void set_carveout_once() {
  static bool done = false;
  if (done) return;
  done = true;
  cudaFuncSetAttribute(k_icp_forward<true, EST_P2P>, cudaFuncAttributePreferredSharedMemoryCarveout, MVR_SMEM_CARVEOUT);
  cudaFuncSetAttribute(k_icp_reverse<EST_P2P>, cudaFuncAttributePreferredSharedMemoryCarveout, MVR_SMEM_CARVEOUT);
}
#else
static void set_carveout_once() {}
#endif

cudaError_t launch_icp_forward(const FwdBatch& d_batch, int pairs, int max_grid, int first, bool reciprocal, int est, cudaStream_t s) {
  if (pairs <= 0 || pairs > FUSED_MAX_PAIRS) return pairs <= 0 ? cudaSuccess : cudaErrorInvalidValue;
  set_carveout_once();
  const dim3 grid((unsigned)max_grid, (unsigned)pairs);
  if (reciprocal) {
    // the reciprocal forward half accumulates nothing: one instantiation serves every estimator but the symmetric one, whose
    // source normals move with the source
    if (est == EST_SYM) k_icp_forward<true, EST_SYM><<<grid, FUSED_THREADS, 0, s>>>(d_batch, first);
    else k_icp_forward<true, EST_P2P><<<grid, FUSED_THREADS, 0, s>>>(d_batch, first);
  } else {
    if (est == EST_SYM) k_icp_forward<false, EST_SYM><<<grid, FUSED_THREADS, 0, s>>>(d_batch, first);
    else if (est == EST_P2L) k_icp_forward<false, EST_P2L><<<grid, FUSED_THREADS, 0, s>>>(d_batch, first);
    else if (est == EST_MOM) k_icp_forward<false, EST_MOM><<<grid, FUSED_THREADS, 0, s>>>(d_batch, first);
    else k_icp_forward<false, EST_P2P><<<grid, FUSED_THREADS, 0, s>>>(d_batch, first);
  }
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_icp_reverse(const RevBatch& d_batch, int pairs, int max_grid, int est, cudaStream_t s) {
  if (pairs <= 0 || pairs > FUSED_MAX_PAIRS) return pairs <= 0 ? cudaSuccess : cudaErrorInvalidValue;
  const dim3 grid((unsigned)max_grid, (unsigned)pairs);
  if (est == EST_SYM) k_icp_reverse<EST_SYM><<<grid, FUSED_THREADS, 0, s>>>(d_batch);
  else if (est == EST_P2L) k_icp_reverse<EST_P2L><<<grid, FUSED_THREADS, 0, s>>>(d_batch);
  else if (est == EST_MOM) k_icp_reverse<EST_MOM><<<grid, FUSED_THREADS, 0, s>>>(d_batch);
  else k_icp_reverse<EST_P2P><<<grid, FUSED_THREADS, 0, s>>>(d_batch);
  count_launch();
  return cudaGetLastError();
}

// Un-gated exact 1-NN of arbitrary (unsorted) queries in a per-align target index: Registration::getFitnessScore's pass
// (mvr/src/registrator.cpp:572, 923, 1015).  The aligned source of a turntable pair has a part the target does not cover;
// those queries are tens of cells away from the nearest target point, and the row walk of pair_search.cuh (two table
// loads decide a whole row of cells) gets through that empty space ~30x faster than a cell-by-cell ring expansion.
// BY_W: the queries were sorted by cell (locality for large batches) and carry their original index in .w.
template <bool BY_W>
__global__ void __launch_bounds__(FUSED_THREADS, 4) k_pair_nn(const float4* __restrict__ q, int n, const float4* __restrict__ tgt,
                                                              const uint32_t* __restrict__ tstart, PairGrid g, int m_valid,
                                                              int32_t* __restrict__ out_idx, float* __restrict__ out_d2) {
  __shared__ uint2 s_seg[PG_SEGS * PG_STRIDE];
  const int i = blockIdx.x * FUSED_THREADS + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(q + i);
  NnBest b{MVR_INF, 0x7fffffff, -1};
  if (finite3(p)) pg_search<MVR_PG_UNROLL>(g, tstart, tgt, m_valid, p.x, p.y, p.z, p.x, p.y, p.z, 0.0f, 1.0f, MVR_INF, b, s_seg + threadIdx.x);
  const int o = BY_W ? __float_as_int(p.w) : i;
  out_idx[o] = b.pos >= 0 ? b.idx : -1;
  out_d2[o] = b.pos >= 0 ? b.d2 : MVR_INF;
}

cudaError_t launch_pair_nn(const float4* q, int n, bool by_w, const float4* tgt_sorted, const uint32_t* tstart, PairGrid g, int m_valid,
                           int32_t* out_idx, float* out_d2, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int blocks = (n + FUSED_THREADS - 1) / FUSED_THREADS;
  if (by_w) k_pair_nn<true><<<blocks, FUSED_THREADS, 0, s>>>(q, n, tgt_sorted, tstart, g, m_valid, out_idx, out_d2);
  else k_pair_nn<false><<<blocks, FUSED_THREADS, 0, s>>>(q, n, tgt_sorted, tstart, g, m_valid, out_idx, out_d2);
  count_launch();
  return cudaGetLastError();
}

// ---- start / end of a batch of aligns (launch.h) ------------------------------------------------
__global__ void __launch_bounds__(256) k_align_init(const __grid_constant__ InitBatch b, const IcpState* __restrict__ stage) {
  const InitJob& j = b.j[blockIdx.y];
  int32_t* __restrict__ corr_p = j.corr_p;
  uint32_t* __restrict__ rmin = j.rmin;
  const int n = j.n, m = rmin ? j.m : 0;
  const int stride = gridDim.x * blockDim.x;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) corr_p[i] = -1;           // no seed yet
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) rmin[i] = 0x7f800000u;   // +inf: "chosen by nobody"
  if (j.nsrc) {   // symmetric: the source normals by sorted position, turned by the guess like the points were
    const int nv = j.n_valid;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride)
      j.nsrc[i] = rotate_pinned(j.M, __ldg(j.snrm + __float_as_int(__ldg(j.sorted + i).w)));
  }
  if (blockIdx.x == 0) {
    static_assert(sizeof(IcpState) % 4 == 0, "IcpState words");
    const uint32_t* src = reinterpret_cast<const uint32_t*>(stage + blockIdx.y);
    uint32_t* dst = reinterpret_cast<uint32_t*>(j.st);
    for (int k = threadIdx.x; k < (int)(sizeof(IcpState) / 4); k += blockDim.x) dst[k] = src[k];
  }
}

__global__ void __launch_bounds__(256) k_align_gather(const __grid_constant__ InitBatch b, IcpState* __restrict__ stage) {
  const InitJob& j = b.j[blockIdx.x];
  const uint32_t* src = reinterpret_cast<const uint32_t*>(j.st);
  uint32_t* dst = reinterpret_cast<uint32_t*>(stage + blockIdx.x);
  for (int k = threadIdx.x; k < (int)(sizeof(IcpState) / 4); k += blockDim.x) dst[k] = src[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    stage[blockIdx.x].dbg[3] = j.crowded ? (long long)*j.crowded : 0ll;
    if (j.crowded) *j.crowded = 0u;
  }
}

cudaError_t launch_align_init(const InitBatch& batch, int count, const IcpState* stage, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (count > BUILD_MAX_JOBS) return cudaErrorInvalidValue;
  int items = 1;
  for (int k = 0; k < count; ++k) items = std::max(items, std::max(batch.j[k].n, batch.j[k].rmin ? batch.j[k].m : 0));
  const int blocks = std::max(1, std::min((items + 1023) / 1024, (148 * 8 + count - 1) / count));
  k_align_init<<<dim3((unsigned)blocks, (unsigned)count), 256, 0, s>>>(batch, stage); count_launch();
  return cudaGetLastError();
}

cudaError_t launch_align_gather(const InitBatch& batch, int count, IcpState* stage, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (count > BUILD_MAX_JOBS) return cudaErrorInvalidValue;
  k_align_gather<<<(unsigned)count, 256, 0, s>>>(batch, stage); count_launch();
  return cudaGetLastError();
}

__global__ void k_reduce_final(const double* __restrict__ partials, int nblk, int nv, double* __restrict__ out) {
  int t = threadIdx.x;
  if (t >= nv) return;
  double x = 0;
#pragma unroll 8
  for (int b = 0; b < nblk; ++b) x += partials[(size_t)b * REDUCE_MAX_VALS + t];
  out[t] = x;
}

__global__ void __launch_bounds__(256) k_reduce_fitness(const int32_t* __restrict__ idx, const float* __restrict__ d2, int n,
                                                        double max_range, double* __restrict__ partials) {
  double v[2] = {0.0, 0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float d = __ldg(d2 + i);
    if (__ldg(idx + i) >= 0 && (double)d <= max_range) { v[0] += (double)d; v[1] += 1.0; }
  }
  block_reduce_store<2>(v, partials);
}

__global__ void __launch_bounds__(256) k_transform_final(const float4* __restrict__ in, float4* __restrict__ out, int n,
                                                         const IcpState* __restrict__ st) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Mat4f M;
#pragma unroll
  for (int k = 0; k < 16; ++k) M.m[k] = (float)st->fin[k];
  float4 p = __ldg(in + i);
  out[i] = finite3(p) ? xform_pinned(M, p) : p;
}

cudaError_t launch_transform_final(const float4* in, float4* out, int n, const IcpState* st, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_transform_final<<<(n + 255) / 256, 256, 0, s>>>(in, out, n, st); count_launch();
  return cudaGetLastError();
}

cudaError_t launch_reduce_fitness(const int32_t* idx, const float* d2, int n, double max_range, double* partials,
                                  double* out, cudaStream_t s) {
  k_reduce_fitness<<<REDUCE_BLOCKS, 256, 0, s>>>(idx, d2, n, max_range, partials); count_launch();
  k_reduce_final<<<1, 32, 0, s>>>(partials, REDUCE_BLOCKS, 2, out); count_launch();
  return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_resolve_pairs(const float4* __restrict__ src, int n_valid, const int32_t* __restrict__ corr_p,
                                                       const int32_t* __restrict__ rnn, const float4* __restrict__ tgt,
                                                       int32_t* __restrict__ corr_j, float* __restrict__ corr_d2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_valid) return;
  const int p = __ldg(corr_p + i);
  if (p < 0 || (rnn && __ldg(rnn + p) != i)) return;
  const float4 s = __ldg(src + i), t = __ldg(tgt + p);
  const int o = __float_as_int(s.w);
  corr_j[o] = __float_as_int(t.w);
  corr_d2[o] = d2_pinned(s.x, s.y, s.z, t.x, t.y, t.z);
}

cudaError_t launch_resolve_pairs(const float4* src_sorted, int n_valid, const int32_t* corr_p, const int32_t* rnn, const float4* tgt_sorted,
                                 int32_t* corr_j, float* corr_d2, cudaStream_t s) {
  if (n_valid <= 0) return cudaSuccess;
  k_resolve_pairs<<<(n_valid + 255) / 256, 256, 0, s>>>(src_sorted, n_valid, corr_p, rnn, tgt_sorted, corr_j, corr_d2); count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// order-preserving compaction (ascending source index, like PCL's correspondence vector)
// ---------------------------------------------------------------------------------------------
constexpr int CP_THREADS = 256;
constexpr int CP_ITEMS = 4;
constexpr int CP_TILE = CP_THREADS * CP_ITEMS;

size_t compact_scratch_elems(int n) { return (size_t)(n > 0 ? (n + CP_TILE - 1) / CP_TILE : 1) + 1; }

__device__ __forceinline__ uint32_t block_excl_scan_256(uint32_t v, uint32_t* total) {
  __shared__ uint32_t ws[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) ws[warp] = incl;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) { uint32_t c = ws[w]; if (w < warp) base += c; tot += c; }
  *total = tot;
  __syncthreads();
  return base + incl - v;
}

__global__ void __launch_bounds__(CP_THREADS) k_compact_count(const int32_t* __restrict__ corr_j, int n, uint32_t* __restrict__ counts) {
  int base = blockIdx.x * CP_TILE + threadIdx.x * CP_ITEMS;
  uint32_t c = 0;
#pragma unroll
  for (int a = 0; a < CP_ITEMS; ++a) if (base + a < n && __ldg(corr_j + base + a) >= 0) ++c;
  uint32_t tot;
  block_excl_scan_256(c, &tot);
  if (threadIdx.x == 0) counts[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(1024) k_compact_scan(uint32_t* __restrict__ counts, int nblk, uint32_t* __restrict__ total_out) {
  __shared__ uint32_t ws[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b0 = 0; b0 < nblk; b0 += 1024) {
    int i = b0 + threadIdx.x;
    uint32_t v = i < nblk ? counts[i] : 0, incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) ws[warp] = incl;
    __syncthreads();
    uint32_t base = carry;
    for (int w = 0; w < warp; ++w) base += ws[w];
    if (i < nblk) counts[i] = base + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = base + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) { counts[nblk] = carry; *total_out = carry; }
}

__global__ void __launch_bounds__(CP_THREADS) k_compact_write(const int32_t* __restrict__ corr_j, const float* __restrict__ corr_d2,
                                                              int n, const uint32_t* __restrict__ offsets, int32_t* __restrict__ out_q,
                                                              int32_t* __restrict__ out_m, float* __restrict__ out_d2) {
  int base = blockIdx.x * CP_TILE + threadIdx.x * CP_ITEMS;
  int32_t j[CP_ITEMS];
  uint32_t c = 0;
#pragma unroll
  for (int a = 0; a < CP_ITEMS; ++a) { j[a] = (base + a < n) ? __ldg(corr_j + base + a) : -1; if (j[a] >= 0) ++c; }
  uint32_t tot;
  uint32_t pos = offsets[blockIdx.x] + block_excl_scan_256(c, &tot);
#pragma unroll
  for (int a = 0; a < CP_ITEMS; ++a)
    if (j[a] >= 0) { out_q[pos] = base + a; out_m[pos] = j[a]; out_d2[pos] = __ldg(corr_d2 + base + a); ++pos; }
}

cudaError_t launch_compact_corr(const int32_t* corr_j, const float* corr_d2, int n, uint32_t* scratch, int32_t* out_q,
                                int32_t* out_m, float* out_d2, uint32_t* count_out, cudaStream_t s) {
  int nblk = n > 0 ? (n + CP_TILE - 1) / CP_TILE : 0;
  if (nblk > 0) { k_compact_count<<<nblk, CP_THREADS, 0, s>>>(corr_j, n, scratch); count_launch(); }
  k_compact_scan<<<1, 1024, 0, s>>>(scratch, nblk, count_out); count_launch();
  if (nblk > 0) { k_compact_write<<<nblk, CP_THREADS, 0, s>>>(corr_j, corr_d2, n, scratch, out_q, out_m, out_d2); count_launch(); }
  return cudaGetLastError();
}

}  // namespace mvr
