// normals.cu -- kNN-PCA normal estimation (K10), a north-star extension with pcl::NormalEstimation
// semantics (SURVEY.md A13); the reference itself never estimates normals (they arrive inside its
// PointXYZRGBNormal .pcd files, mvr/include/types.h:14-18).
//
// One thread per point of the cell-sorted cloud (row-major grid of pair_index.cu, cell edge ~1.25 x the expected k-th
// neighbour distance): exact k nearest neighbours (self included, ties to the lowest index) from the 3 x 3 x 3 cells around
// the point -- nine contiguous runs of the sorted array, shared through L1 by the neighbouring threads, which sit in the
// same cells -- and, only if the k-th distance does not yet beat everything outside that block, from the next shells.
// The running k-list lives in SHARED memory as an unsorted set with its worst member tracked (a rejected candidate costs
// one comparison, an accepted one a 16-entry rescan); round 1 kept a sorted list in local memory (504 bytes of stack per
// thread, every insertion a chain of local loads and stores: 4.9 ms for 2M points).  The list is sorted once at the end
// (neighbours are reported in ascending (d2, index)), then two-pass covariance in double, Jacobi eigen-solve,
// normal = eigenvector of the smallest eigenvalue flipped towards the viewpoint, curvature = l0 / (l0 + l1 + l2).
#include <algorithm>

#include "launch.h"
#include "pair_search.cuh"
#include "small_solve.h"

namespace mvr {

constexpr int KNN_MAX = 32;
constexpr int KN_THREADS = 128;

struct KnnEntry { float d; int id; int pos; };

// the thread's list: entry a at L[a * KN_THREADS] (bank = thread)
struct KnnList {
  float* d; int* id; int* pos;
  int n, k, worst;       // worst = slot of the lexicographically largest (d, id) once the list is full
  float wd; int wid;
  __device__ __forceinline__ void rescan() {
    worst = 0; wd = d[0]; wid = id[0];
    for (int a = 1; a < k; ++a) {
      const float da = d[a * KN_THREADS]; const int ia = id[a * KN_THREADS];
      if (lex_less(wd, wid, da, ia)) { worst = a; wd = da; wid = ia; }
    }
  }
  __device__ __forceinline__ void push(float d2, int i, int p) {
    if (n < k) {
      d[n * KN_THREADS] = d2; id[n * KN_THREADS] = i; pos[n * KN_THREADS] = p;
      if (++n == k) rescan();
      return;
    }
    if (!lex_less(d2, i, wd, wid)) return;
    d[worst * KN_THREADS] = d2; id[worst * KN_THREADS] = i; pos[worst * KN_THREADS] = p;
    rescan();
  }
  __device__ __forceinline__ float worst_d() const { return n < k ? MVR_INF : wd; }
};

// One launch serves every cloud of a NormalsBatch: blockIdx.y selects the job, blockIdx.x < ceil(n / KN_THREADS) of that job
// does its work (the jobs travel by value in the kernel's parameter space, as the builds of pair_index.cu do).  k <= 16 asks
// for eight blocks per SM: the single-cloud kernel this replaced got 64 registers (eight blocks) unasked; without the bound the
// job-indexed parameters take it to 72 (seven blocks).
template <int KMAX>
__global__ void __launch_bounds__(KN_THREADS, KMAX <= 16 ? 8 : 0) k_normals(const __grid_constant__ NormalsBatch b, int k) {
  __shared__ float s_d[KMAX * KN_THREADS];     // k <= KMAX: 24 KB per block for k <= 16 (nine blocks per SM), 48 KB above
  __shared__ int s_id[KMAX * KN_THREADS];
  __shared__ int s_pos[KMAX * KN_THREADS];
  const NormalsJob& j = b.j[blockIdx.y];
  const int sp = blockIdx.x * KN_THREADS + threadIdx.x;
  if (sp >= j.n) return;
  const float4* __restrict__ sorted = j.sorted;
  const uint32_t* __restrict__ start = j.start;
  const PairGrid& g = j.g;
  const int n_valid = j.n_valid;
  float4* __restrict__ out = j.out;
  int32_t* __restrict__ nbr = j.nbr;
  const float3 vp = j.viewpoint;
  const float4 q = __ldg(sorted + sp);
  const int self = __float_as_int(q.w);
  if (sp >= n_valid) {  // non-finite point
    out[self] = make_float4(nanf(""), nanf(""), nanf(""), nanf(""));
    if (nbr) for (int a = 0; a < k; ++a) nbr[(size_t)self * k + a] = -1;
    return;
  }
  const float tx = grid_t(q.x, g.ox, g.inv_cell), ty = grid_t(q.y, g.oy, g.inv_cell), tz = grid_t(q.z, g.oz, g.inv_cell);
  const int cx = pg_cell(tx, g.nx), cy = pg_cell(ty, g.ny), cz = pg_cell(tz, g.nz);
  const float margin = MVR_CELL_MARGIN + 1.0e-6f * fmaxf(fabsf(tx), fmaxf(fabsf(ty), fabsf(tz)));
  const float cell2 = g.cell_lo * g.cell_lo * MVR_REL_SHRINK;
  KnnList L;
  L.d = s_d + threadIdx.x; L.id = s_id + threadIdx.x; L.pos = s_pos + threadIdx.x;
  L.n = 0; L.k = k; L.worst = 0; L.wd = MVR_INF; L.wid = 0x7fffffff;
  auto scan = [&](uint32_t s, uint32_t e) {
    for (uint32_t a = s; a < e; ++a) {
      const float4 p = __ldg(sorted + a);
      L.push(d2_pinned(q.x, q.y, q.z, p.x, p.y, p.z), __float_as_int(p.w), (int)a);
    }
  };
  for (int h = 1;; ++h) {
    // the shell between the cubes of half-width h - 1 and h (h = 1: the whole 3 x 3 x 3 block)
    const int x0 = max(cx - h, 0), x1 = min(cx + h, g.nx - 1);
    for (int z = max(cz - h, 0); z <= min(cz + h, g.nz - 1); ++z)
      for (int y = max(cy - h, 0); y <= min(cy + h, g.ny - 1); ++y) {
        const uint32_t* row = start + ((size_t)z * g.ny + y) * g.nx;
        const bool face = h == 1 || z == cz - h || z == cz + h || y == cy - h || y == cy + h;
        if (face) {
          scan(__ldg(row + x0), __ldg(row + x1 + 1));
        } else {   // an inner row: only its two end cells are new
          if (cx - h >= 0) scan(__ldg(row + cx - h), __ldg(row + cx - h + 1));
          if (cx + h <= g.nx - 1) scan(__ldg(row + cx + h), __ldg(row + cx + h + 1));
        }
      }
    // everything outside the cube is farther than u cells along some axis (an axis the cube covers entirely does not count)
    float u = MVR_INF;
    if (cx - h > 0) u = fminf(u, tx - (float)(cx - h));
    if (cx + h < g.nx - 1) u = fminf(u, (float)(cx + h + 1) - tx);
    if (cy - h > 0) u = fminf(u, ty - (float)(cy - h));
    if (cy + h < g.ny - 1) u = fminf(u, (float)(cy + h + 1) - ty);
    if (cz - h > 0) u = fminf(u, tz - (float)(cz - h));
    if (cz + h < g.nz - 1) u = fminf(u, (float)(cz + h + 1) - tz);
    if (u == MVR_INF) break;
    const float bu = fmaxf(u - margin, 0.0f);
    if (L.worst_d() < bu * bu * cell2) break;
  }
  // ascending (d2, index): insertion sort of at most 32 entries in shared memory
  for (int a = 1; a < L.n; ++a) {
    const float da = L.d[a * KN_THREADS]; const int ia = L.id[a * KN_THREADS], pa = L.pos[a * KN_THREADS];
    int b = a;
    while (b > 0 && lex_less(da, ia, L.d[(b - 1) * KN_THREADS], L.id[(b - 1) * KN_THREADS])) {
      L.d[b * KN_THREADS] = L.d[(b - 1) * KN_THREADS]; L.id[b * KN_THREADS] = L.id[(b - 1) * KN_THREADS]; L.pos[b * KN_THREADS] = L.pos[(b - 1) * KN_THREADS];
      --b;
    }
    L.d[b * KN_THREADS] = da; L.id[b * KN_THREADS] = ia; L.pos[b * KN_THREADS] = pa;
  }
  if (nbr) for (int a = 0; a < k; ++a) nbr[(size_t)self * k + a] = a < L.n ? L.id[a * KN_THREADS] : -1;
  if (L.n < 3) { out[self] = make_float4(nanf(""), nanf(""), nanf(""), nanf("")); return; }
  // two-pass covariance in double over the neighbours (their coordinates from the cell-sorted array: cache-friendly)
  double c[3] = {0, 0, 0};
  for (int a = 0; a < L.n; ++a) { const float4 p = __ldg(sorted + L.pos[a * KN_THREADS]); c[0] += p.x; c[1] += p.y; c[2] += p.z; }
  const double inv = 1.0 / (double)L.n;
  c[0] *= inv; c[1] *= inv; c[2] *= inv;
  double C[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int a = 0; a < L.n; ++a) {
    const float4 p = __ldg(sorted + L.pos[a * KN_THREADS]);
    const double d[3] = {(double)p.x - c[0], (double)p.y - c[1], (double)p.z - c[2]};
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int s = 0; s < 3; ++s) C[r * 3 + s] += d[r] * d[s];
  }
#pragma unroll
  for (int a = 0; a < 9; ++a) C[a] *= inv;
  double w[3], V[9];
  eig_sym3(C, w, V);
  double nx = V[0], ny = V[3], nz = V[6];
  const double vx = (double)vp.x - q.x, vy = (double)vp.y - q.y, vz = (double)vp.z - q.z;
  if (nx * vx + ny * vy + nz * vz < 0) { nx = -nx; ny = -ny; nz = -nz; }
  const double tr = w[0] + w[1] + w[2];
  out[self] = make_float4((float)nx, (float)ny, (float)nz, (float)(tr > 0 ? fabs(w[0] / tr) : 0.0));
}

cudaError_t launch_normals(const NormalsBatch& batch, int count, int k, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (count > BUILD_MAX_JOBS || k < 1 || k > KNN_MAX) return cudaErrorInvalidValue;
  int max_n = 0;
  for (int a = 0; a < count; ++a) max_n = std::max(max_n, batch.j[a].n);
  if (max_n <= 0) return cudaSuccess;
  const dim3 grid((unsigned)((max_n + KN_THREADS - 1) / KN_THREADS), (unsigned)count);
  if (k <= 16) k_normals<16><<<grid, KN_THREADS, 0, s>>>(batch, k);
  else k_normals<KNN_MAX><<<grid, KN_THREADS, 0, s>>>(batch, k);
  count_launch();
  return cudaGetLastError();
}

}  // namespace mvr
