// features.cu -- FPFH descriptors of a cloud's keypoints and exact nearest-descriptor matching (mvr_compute_fpfh,
// mvr_match_features): the feature half of the global registration (host/global.cpp, DESIGN.md sections 4 and 6).
// pcl::FPFHEstimation semantics on kNN neighbourhoods; no reference counterpart (the reference always starts from the
// turntable's rotation).
//
// The keypoints are the finite points of original index i % stride == 0 (the scorer's samples), gathered in index order.
// Their normals and neighbour lists come from k_normals on an index of the keypoint cloud (normals.cu); these kernels only
// read them.  Everything below runs in a fixed order per thread, so the results do not depend on the launch shape or the GPU:
// the pair features and the histograms in double (-fmad=false), the descriptor distances in float without FMA.
#include <algorithm>

#include "launch.h"

namespace mvr {

constexpr int KP_THREADS = 1024;   // k_keypoints: one block, a contiguous run of slots per thread
constexpr int FH_THREADS = 128;
constexpr int MT_THREADS = 128;    // k_match: query rows per block = B rows per shared tile

// Compaction of the keypoint slots s < slots (original index s * stride) in index order: out[0 .. n_kp) = the finite ones,
// out[n_kp .. slots) = NaN (what the bounding-box launch that follows counts as non-finite: n_kp = slots - that count).
__global__ void __launch_bounds__(KP_THREADS) k_keypoints(const float4* __restrict__ pts, int stride, int slots, float4* __restrict__ out,
                                                          int32_t* __restrict__ index) {
  __shared__ int s_off[KP_THREADS];
  const int per = (slots + KP_THREADS - 1) / KP_THREADS;
  const int s0 = min(slots, (int)threadIdx.x * per), s1 = min(slots, s0 + per);
  int cnt = 0;
  for (int s = s0; s < s1; ++s) cnt += finite3(__ldg(pts + (size_t)s * stride)) ? 1 : 0;
  s_off[threadIdx.x] = cnt;
  __syncthreads();
  for (int d = 1; d < KP_THREADS; d <<= 1) {   // inclusive scan
    const int v = threadIdx.x >= (unsigned)d ? s_off[threadIdx.x - d] : 0;
    __syncthreads();
    s_off[threadIdx.x] += v;
    __syncthreads();
  }
  int o = s_off[threadIdx.x] - cnt;
  for (int s = s0; s < s1; ++s) {
    const float4 p = __ldg(pts + (size_t)s * stride);
    if (finite3(p)) { out[o] = p; index[o] = s * stride; ++o; }
  }
  const int n_kp = s_off[KP_THREADS - 1];
  for (int s = n_kp + (int)threadIdx.x; s < slots; s += KP_THREADS) { out[s] = make_float4(nanf(""), nanf(""), nanf(""), 0.f); index[s] = -1; }
}

struct Pair { double f1, f2, f3; bool ok; };

// pcl::computePairFeatures(p1, n1, p2, n2) in double; the roles swap when |a1| < |a2| (PCL: acos|a1| > acos|a2|).
__device__ __forceinline__ Pair pair_features(float4 p1, float4 n1, float4 p2, float4 n2) {
  Pair r{0, 0, 0, false};
  double dx = (double)p2.x - p1.x, dy = (double)p2.y - p1.y, dz = (double)p2.z - p1.z;
  const double f4 = sqrt((dx * dx + dy * dy) + dz * dz);
  if (f4 == 0.0) return r;
  double ax = n1.x, ay = n1.y, az = n1.z, bx = n2.x, by = n2.y, bz = n2.z;
  const double a1 = ((ax * dx + ay * dy) + az * dz) / f4, a2 = ((bx * dx + by * dy) + bz * dz) / f4;
  if (fabs(a1) < fabs(a2)) {
    double t;
    t = ax; ax = bx; bx = t; t = ay; ay = by; by = t; t = az; az = bz; bz = t;
    dx = -dx; dy = -dy; dz = -dz;
    r.f3 = -a2;
  } else {
    r.f3 = a1;
  }
  double vx = dy * az - dz * ay, vy = dz * ax - dx * az, vz = dx * ay - dy * ax;   // v = dp x n1
  const double vn = sqrt((vx * vx + vy * vy) + vz * vz);
  if (vn == 0.0) return r;
  vx = vx / vn; vy = vy / vn; vz = vz / vn;
  const double wx = ay * vz - az * vy, wy = az * vx - ax * vz, wz = ax * vy - ay * vx;   // w = n1 x v
  r.f2 = (vx * bx + vy * by) + vz * bz;
  r.f1 = atan2((wx * bx + wy * by) + wz * bz, (ax * bx + ay * by) + az * bz);
  r.ok = true;
  return r;
}

__device__ __forceinline__ int feature_bin(double t) {   // t = 11 (f + offset) / range, floored and clamped to 0..10
  const double b = floor(t);
  return b < 0.0 ? 0 : (b > 10.0 ? 10 : (int)b);
}

__device__ __forceinline__ bool finite_normal(float4 n) { return isfinite(n.x) && isfinite(n.y) && isfinite(n.z); }

// SPFH of keypoint i: its pairs with the first k - 1 entries of its list that are not itself, in list order.  A pair with a
// non-finite normal, f4 == 0 or |v| == 0 adds nothing; every other pair adds 100 / (k - 1) to one bin of each sub-histogram.
__global__ void __launch_bounds__(FH_THREADS) k_spfh(const float4* __restrict__ kp, const float4* __restrict__ nrm, const int32_t* __restrict__ nbr,
                                                     int n, int k, double* __restrict__ spfh) {
  __shared__ unsigned char s_cnt[33 * FH_THREADS];   // bin b of this thread at [b * FH_THREADS + tid]: at most 31 pairs per bin
  const int i = blockIdx.x * FH_THREADS + threadIdx.x;
  if (i >= n) return;
  unsigned char* cnt = s_cnt + threadIdx.x;
  for (int b = 0; b < 33; ++b) cnt[b * FH_THREADS] = 0;
  const float4 p = __ldg(kp + i), ni = __ldg(nrm + i);
  if (finite_normal(ni)) {
    const double PI = 3.141592653589793;
    int taken = 0;
    for (int a = 0; a < k && taken < k - 1; ++a) {
      const int j = __ldg(nbr + (size_t)i * k + a);
      if (j < 0 || j == i) continue;
      ++taken;
      const float4 nj = __ldg(nrm + j);
      if (!finite_normal(nj)) continue;
      const Pair f = pair_features(p, ni, __ldg(kp + j), nj);
      if (!f.ok) continue;
      cnt[feature_bin(11.0 * (f.f1 + PI) / (2.0 * PI)) * FH_THREADS]++;
      cnt[(11 + feature_bin(11.0 * (f.f2 + 1.0) / 2.0)) * FH_THREADS]++;
      cnt[(22 + feature_bin(11.0 * (f.f3 + 1.0) / 2.0)) * FH_THREADS]++;
    }
  }
  const double inc = 100.0 / (double)(k - 1);
  for (int b = 0; b < 33; ++b) {
    double h = 0.0;   // the sum of the bin's pairs in list order: all of them add the same increment
    for (int c = cnt[b * FH_THREADS]; c > 0; --c) h += inc;
    spfh[(size_t)i * 33 + b] = h;
  }
}

// FPFH of keypoint i = own SPFH + the list's weighted SPFH (pcl::FPFHEstimation::weightPointSPFHSignature): the same k - 1
// neighbours, weight 1 / d2 (d2 = the pinned float distance the list is ordered by; 0: skipped), summed in list order in double;
// each 11-bin sub-histogram of that sum is scaled to 100.  A keypoint with a non-finite normal gets zeros (it never matches).
__global__ void __launch_bounds__(FH_THREADS) k_fpfh(const float4* __restrict__ kp, const float4* __restrict__ nrm, const int32_t* __restrict__ nbr,
                                                     const double* __restrict__ spfh, int n, int k, float* __restrict__ out) {
  __shared__ double s_acc[33 * FH_THREADS];
  const int i = blockIdx.x * FH_THREADS + threadIdx.x;
  if (i >= n) return;
  float* o = out + (size_t)i * 33;
  if (!finite_normal(__ldg(nrm + i))) {
    for (int b = 0; b < 33; ++b) o[b] = 0.f;
    return;
  }
  double* acc = s_acc + threadIdx.x;
  for (int b = 0; b < 33; ++b) acc[b * FH_THREADS] = 0.0;
  const float4 p = __ldg(kp + i);
  int taken = 0;
  for (int a = 0; a < k && taken < k - 1; ++a) {
    const int j = __ldg(nbr + (size_t)i * k + a);
    if (j < 0 || j == i) continue;
    ++taken;
    const float4 q = __ldg(kp + j);
    const float d2 = d2_pinned(p.x, p.y, p.z, q.x, q.y, q.z);
    if (d2 == 0.f) continue;
    const double w = 1.0 / (double)d2;
    const double* h = spfh + (size_t)j * 33;
    for (int b = 0; b < 33; ++b) acc[b * FH_THREADS] += __ldg(h + b) * w;
  }
  const double* own = spfh + (size_t)i * 33;
  for (int s = 0; s < 3; ++s) {
    double sum = 0.0;
    for (int b = 11 * s; b < 11 * s + 11; ++b) sum += acc[b * FH_THREADS];
    const double scale = sum != 0.0 ? 100.0 / sum : 0.0;
    for (int b = 11 * s; b < 11 * s + 11; ++b) o[b] = (float)(__ldg(own + b) + acc[b * FH_THREADS] * scale);
  }
}

// out[i] = the row of b nearest to row i of a in squared L2 over the 33 bins (summed in bin order, no FMA), ties to the lowest
// row; -1 for an all-zero query or when no row of b qualifies.  All-zero rows of b are never chosen.  CUDA cores, exact floats:
// B travels through shared memory in tiles of MT_THREADS rows, every lane reads the same row (a broadcast).
__global__ void __launch_bounds__(MT_THREADS) k_match(const float* __restrict__ a, int na, const float* __restrict__ b, int nb, int32_t* __restrict__ out) {
  __shared__ float s_b[MT_THREADS * 33];
  __shared__ int s_zero[MT_THREADS];
  const int i = blockIdx.x * MT_THREADS + threadIdx.x;
  float q[33];
  bool qz = true;
#pragma unroll
  for (int c = 0; c < 33; ++c) { q[c] = i < na ? __ldg(a + (size_t)i * 33 + c) : 0.f; qz = qz && q[c] == 0.f; }
  float best = MVR_INF;
  int bi = -1;
  for (int t0 = 0; t0 < nb; t0 += MT_THREADS) {
    const int cnt = min(MT_THREADS, nb - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * 33; e += MT_THREADS) s_b[e] = __ldg(b + (size_t)t0 * 33 + e);
    __syncthreads();
    if (threadIdx.x < cnt) {
      bool z = true;
      for (int c = 0; c < 33; ++c) z = z && s_b[threadIdx.x * 33 + c] == 0.f;
      s_zero[threadIdx.x] = z;
    }
    __syncthreads();
    if (qz) continue;
    for (int r = 0; r < cnt; ++r) {
      if (s_zero[r]) continue;
      const float* br = s_b + r * 33;
      float d = 0.f;
#pragma unroll
      for (int c = 0; c < 33; ++c) {
        const float t = __fsub_rn(q[c], br[c]);
        d = __fadd_rn(d, __fmul_rn(t, t));
      }
      if (d < best) { best = d; bi = t0 + r; }
    }
  }
  if (i < na) out[i] = bi;
}

cudaError_t launch_keypoints(const float4* pts, int stride, int slots, float4* out, int32_t* index, cudaStream_t s) {
  if (slots <= 0) return cudaSuccess;
  k_keypoints<<<1, KP_THREADS, 0, s>>>(pts, stride, slots, out, index);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_fpfh(const float4* kp, const float4* nrm, const int32_t* nbr, int n, int k, double* spfh, float* out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  if (k < 2 || k > 32) return cudaErrorInvalidValue;
  const unsigned grid = (unsigned)((n + FH_THREADS - 1) / FH_THREADS);
  k_spfh<<<grid, FH_THREADS, 0, s>>>(kp, nrm, nbr, n, k, spfh);
  k_fpfh<<<grid, FH_THREADS, 0, s>>>(kp, nrm, nbr, spfh, n, k, out);
  count_launch(2);
  return cudaGetLastError();
}

cudaError_t launch_match(const float* a, int na, const float* b, int nb, int32_t* out, cudaStream_t s) {
  if (na <= 0) return cudaSuccess;
  k_match<<<(unsigned)((na + MT_THREADS - 1) / MT_THREADS), MT_THREADS, 0, s>>>(a, na, b, nb, out);
  count_launch();
  return cudaGetLastError();
}

}  // namespace mvr
