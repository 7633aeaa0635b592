// index.cu -- GPU spatial index build: bounding box, Morton keys, stable LSD radix sort, cell table.
//
// Replaces pcl::KdTreeFLANN::setInputCloud, which icp.align() runs on the target once per align and
// on the source once per iteration for reciprocal correspondences (call sites
// mvr/src/registrator.cpp:566-569, 776-777, 913-920; SURVEY.md section 3.4).
//
// Algorithmic bytes per indexed point (DESIGN.md section 4): 16 B read + 16 B sorted-point write +
// 4 B permutation write, plus 4 B per table entry.
#include "launch.h"

namespace mvr {

// ---------------------------------------------------------------------------------------------
// bounding box
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t f2ord(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f);
#else
  uint32_t u; memcpy(&u, &f, 4);
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

float bbox_decode(uint32_t e) {
  uint32_t u = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
  float f; memcpy(&f, &u, 4);
  return f;
}

__global__ void k_bbox_init(uint32_t* out) {
  int t = threadIdx.x;
  if (t < 3) out[t] = 0xffffffffu;          // running min
  else if (t < 6) out[t] = 0u;              // running max
  else if (t == 6) out[t] = 0u;             // non-finite count
}

__device__ __forceinline__ void bbox_body(const float4* __restrict__ pts, int n, uint32_t* out) {
  float lo[3] = {MVR_INF, MVR_INF, MVR_INF}, hi[3] = {-MVR_INF, -MVR_INF, -MVR_INF};
  uint32_t bad = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = __ldg(pts + i);
    if (finite3(p)) {
      lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
      hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
    } else {
      ++bad;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
      hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
    }
    bad += __shfl_xor_sync(0xffffffffu, bad, o);
  }
  // one set of atomics per block, not per warp: they all hit the same seven words
  __shared__ float s_lo[8][3], s_hi[8][3];
  __shared__ uint32_t s_bad[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { s_lo[warp][a] = lo[a]; s_hi[warp][a] = hi[a]; }
    s_bad[warp] = bad;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int a = threadIdx.x;
    float l = MVR_INF, h = -MVR_INF;
#pragma unroll
    for (int w = 0; w < 8; ++w) { l = fminf(l, s_lo[w][a]); h = fmaxf(h, s_hi[w][a]); }
    if (l <= h) { atomicMin(out + a, f2ord(l)); atomicMax(out + 3 + a, f2ord(h)); }
  } else if (threadIdx.x == 3) {
    uint32_t b = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) b += s_bad[w];
    if (b) atomicAdd(out + 6, b);
  }
}

__global__ void __launch_bounds__(256) k_bbox(const float4* __restrict__ pts, int n, uint32_t* out) { bbox_body(pts, n, out); }

// Every cloud of a batch in one launch (blockIdx.y = cloud); the seven words of each are initialised by k_bbox_init_batch.
__global__ void k_bbox_init_batch(uint32_t* out, int count) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < 7 * count) out[t] = (t % 7 < 3) ? 0xffffffffu : 0u;
}
__global__ void __launch_bounds__(256) k_bbox_batch(const __grid_constant__ BboxBatch b, uint32_t* out) {
  const BboxJob& j = b.j[blockIdx.y];
  bbox_body(j.pts, j.n, out + 7 * blockIdx.y);
}

cudaError_t launch_bbox_init(uint32_t* out7, cudaStream_t s) {
  k_bbox_init<<<1, 32, 0, s>>>(out7); count_launch();
  return cudaGetLastError();
}

cudaError_t launch_bbox_batch(const BboxBatch& batch, int count, uint32_t* out7, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (count > BBOX_MAX_JOBS) return cudaErrorInvalidValue;
  int max_n = 0;
  for (int k = 0; k < count; ++k) max_n = max(max_n, batch.j[k].n);
  k_bbox_init_batch<<<(7 * count + 255) / 256, 256, 0, s>>>(out7, count); count_launch();
  if (max_n > 0) {
    const int blocks = max(1, min((max_n + 1023) / 1024, (148 * 4 + count - 1) / count));
    k_bbox_batch<<<dim3((unsigned)blocks, (unsigned)count), 256, 0, s>>>(batch, out7); count_launch();
  }
  return cudaGetLastError();
}

cudaError_t launch_bbox(const float4* pts, int n, uint32_t* out7, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  int blocks = min((n + 1023) / 1024, 148 * 2);
  k_bbox<<<blocks, 256, 0, s>>>(pts, n, out7); count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Morton keys (K1)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_morton_keys(const float4* __restrict__ pts, int n, GridDev g,
                                                     uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = point_key(__ldg(pts + i), g);
  vals[i] = (uint32_t)i;
}

// PointCloud::getTransformedPoints (mvr/src/point_cloud.cpp:290-303): p' = pose * p evaluated in double and
// narrowed to float; the input records may be wider than 16 bytes (PointXYZRGBNormal = 48).
struct Mat4d { double m[16]; };
__global__ void __launch_bounds__(256) k_apply_pose(const char* __restrict__ in, size_t stride, int n, Mat4d M, float4* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = reinterpret_cast<const float*>(in + (size_t)i * stride);
  const double x = p[0], y = p[1], z = p[2];
  float4 r;
  r.x = (float)(M.m[0] * x + M.m[4] * y + M.m[8] * z + M.m[12]);
  r.y = (float)(M.m[1] * x + M.m[5] * y + M.m[9] * z + M.m[13]);
  r.z = (float)(M.m[2] * x + M.m[6] * y + M.m[10] * z + M.m[14]);
  r.w = 1.0f;
  out[i] = r;
}

// Registrator::saveRegisteredPoints (mvr/src/registrator.cpp:344-400) for one view: every 48-byte
// pcl::PointXYZRGBNormal record {xyz pad | normal pad | rgb curvature pad pad} gets p' = pose * p and, exactly like the
// reference (matrix.preMult(normal), :367-371), n' = pose * n with the TRANSLATION applied too (full_matrix_normals = 1);
// full_matrix_normals = 0 rotates the normal only.  Double arithmetic narrowed to float; colour and curvature copied.
__global__ void __launch_bounds__(256) k_merge_rich(const float4* __restrict__ in, int n, Mat4d M, int full_matrix_normals, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 a = __ldg(in + 3 * (size_t)i), b = __ldg(in + 3 * (size_t)i + 1), c = __ldg(in + 3 * (size_t)i + 2);
  float4 r;
  r.x = (float)(M.m[0] * a.x + M.m[4] * a.y + M.m[8] * a.z + M.m[12]);
  r.y = (float)(M.m[1] * a.x + M.m[5] * a.y + M.m[9] * a.z + M.m[13]);
  r.z = (float)(M.m[2] * a.x + M.m[6] * a.y + M.m[10] * a.z + M.m[14]);
  r.w = a.w;
  const double t = full_matrix_normals ? 1.0 : 0.0;
  float4 q;
  q.x = (float)(M.m[0] * b.x + M.m[4] * b.y + M.m[8] * b.z + t * M.m[12]);
  q.y = (float)(M.m[1] * b.x + M.m[5] * b.y + M.m[9] * b.z + t * M.m[13]);
  q.z = (float)(M.m[2] * b.x + M.m[6] * b.y + M.m[10] * b.z + t * M.m[14]);
  q.w = b.w;
  out[3 * (size_t)i] = r; out[3 * (size_t)i + 1] = q; out[3 * (size_t)i + 2] = c;
}

cudaError_t launch_merge_rich(const void* in48, int n, const double* M16, int full_matrix_normals, void* out48, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  Mat4d M;
  for (int k = 0; k < 16; ++k) M.m[k] = M16[k];
  k_merge_rich<<<(n + 255) / 256, 256, 0, s>>>((const float4*)in48, n, M, full_matrix_normals, (float4*)out48); count_launch();
  return cudaGetLastError();
}

cudaError_t launch_apply_pose(const void* in, size_t stride, int n, const double* M16, float4* out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  Mat4d M;
  for (int k = 0; k < 16; ++k) M.m[k] = M16[k];
  k_apply_pose<<<(n + 255) / 256, 256, 0, s>>>((const char*)in, stride, n, M, out); count_launch();
  return cudaGetLastError();
}

cudaError_t launch_morton_keys(const float4* pts, int n, GridDev g, uint32_t* keys, uint32_t* vals, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_morton_keys<<<(n + 255) / 256, 256, 0, s>>>(pts, n, g, keys, vals); count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Stable LSD radix sort (K2): 8-bit digits, per pass {tile histogram, scan, ranked scatter}.
// A tile is 4096 consecutive pairs; warp w of the block owns the w-th 512-pair slice of the tile
// and walks it 32 at a time, so (warp, round, lane) order IS input order and ranks are stable.
// ---------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ITEMS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;

int radix_num_blocks(int n) { return n > 0 ? (n + RS_TILE - 1) / RS_TILE : 1; }

__global__ void __launch_bounds__(RS_THREADS) k_radix_hist(const uint32_t* __restrict__ keys, int n, int shift,
                                                           uint32_t* __restrict__ hist, int nblk) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  int base = blockIdx.x * RS_TILE;
#pragma unroll 4
  for (int i = threadIdx.x; i < RS_TILE; i += RS_THREADS) {
    int idx = base + i;
    if (idx < n) atomicAdd(&h[(__ldg(keys + idx) >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of `total` counters laid out digit-major; one block of 1024 threads
__global__ void __launch_bounds__(1024) k_radix_scan(uint32_t* __restrict__ hist, int total) {
  __shared__ uint32_t warp_sums[32];
  int per = (total + 1023) / 1024;
  int b = threadIdx.x * per, e = min(b + per, total);
  uint32_t sum = 0;
  for (int i = b; i < e; ++i) sum += hist[i];
  // block exclusive scan of `sum`
  uint32_t incl = sum;
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = warp_sums[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t v = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += v;
    }
    warp_sums[lane] = wi - w;
  }
  __syncthreads();
  uint32_t run = warp_sums[warp] + incl - sum;
  for (int i = b; i < e; ++i) { uint32_t c = hist[i]; hist[i] = run; run += c; }
}

__global__ void __launch_bounds__(RS_THREADS) k_radix_scatter(const uint32_t* __restrict__ kin, const uint32_t* __restrict__ vin,
                                                              uint32_t* __restrict__ kout, uint32_t* __restrict__ vout, int n,
                                                              int shift, const uint32_t* __restrict__ scanned, int nblk) {
  __shared__ uint32_t wc[RS_WARPS][256];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int w = 0; w < RS_WARPS; ++w) wc[w][tid] = 0;
  __syncthreads();
  const int base = blockIdx.x * RS_TILE + warp * (RS_ITEMS * 32);
  uint32_t key[RS_ITEMS];
  uint32_t rank[RS_ITEMS];
#pragma unroll
  for (int r = 0; r < RS_ITEMS; ++r) {
    int idx = base + r * 32 + lane;
    bool valid = idx < n;
    uint32_t live = __ballot_sync(0xffffffffu, valid);
    key[r] = 0; rank[r] = 0;
    if (valid) {
      key[r] = __ldg(kin + idx);
      uint32_t d = (key[r] >> shift) & 255u;
      uint32_t peers = __match_any_sync(live, d);
      int leader = __ffs(peers) - 1;
      uint32_t old = 0;
      if (lane == leader) { old = wc[warp][d]; wc[warp][d] = old + __popc(peers); }
      old = __shfl_sync(peers, old, leader);
      rank[r] = old + __popc(peers & ((1u << lane) - 1u));
    }
    __syncwarp();
  }
  __syncthreads();
  {
    uint32_t run = scanned[tid * nblk + blockIdx.x];
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) { uint32_t c = wc[w][tid]; wc[w][tid] = run; run += c; }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RS_ITEMS; ++r) {
    int idx = base + r * 32 + lane;
    if (idx < n) {
      uint32_t d = (key[r] >> shift) & 255u;
      uint32_t pos = wc[warp][d] + rank[r];
      kout[pos] = key[r];
      vout[pos] = __ldg(vin + idx);
    }
  }
}

cudaError_t launch_radix_sort(uint32_t* keys, uint32_t* vals, int n, int key_bits, SortScratch sc, uint32_t** keys_out,
                              uint32_t** vals_out, cudaStream_t s) {
  *keys_out = keys; *vals_out = vals;
  if (n <= 0) return cudaSuccess;
  int passes = (key_bits + 7) / 8;
  if (passes < 1) passes = 1;
  int nblk = radix_num_blocks(n);
  uint32_t *kin = keys, *vin = vals, *kout = sc.keys_alt, *vout = sc.vals_alt;
  for (int p = 0; p < passes; ++p) {
    int shift = 8 * p;
    k_radix_hist<<<nblk, RS_THREADS, 0, s>>>(kin, n, shift, sc.hist, nblk); count_launch();
    k_radix_scan<<<1, 1024, 0, s>>>(sc.hist, 256 * nblk); count_launch();
    k_radix_scatter<<<nblk, RS_THREADS, 0, s>>>(kin, vin, kout, vout, n, shift, sc.hist, nblk); count_launch();
    uint32_t* t = kin; kin = kout; kout = t;
    t = vin; vin = vout; vout = t;
  }
  *keys_out = kin; *vals_out = vin;
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// sorted point gather + cell table (K3)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_gather_sorted(const float4* __restrict__ pts, const uint32_t* __restrict__ perm, int n,
                                                       float4* __restrict__ sorted) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t j = __ldg(perm + i);
  float4 p = __ldg(pts + j);
  p.w = __uint_as_float(j);
  sorted[i] = p;
}

cudaError_t launch_gather_sorted(const float4* pts, const uint32_t* perm, int n, float4* sorted, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_gather_sorted<<<(n + 255) / 256, 256, 0, s>>>(pts, perm, n, sorted); count_launch();
  return cudaGetLastError();
}

// One thread per boundary i in [0, n]; a warp fills the (possibly long) run of empty cells that
// precedes each occupied cell cooperatively so the stores stay coalesced.
__global__ void __launch_bounds__(256) k_cell_table(const uint32_t* __restrict__ keys, int n, uint32_t C,
                                                    uint32_t* __restrict__ start) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  long long prev = -1, cur = -1;
  if (i <= n) {
    prev = (i == 0) ? -1 : (long long)min(__ldg(keys + i - 1), C);
    cur = (i < n) ? (long long)min(__ldg(keys + i), C) : (long long)C;
  }
  uint32_t has = __ballot_sync(0xffffffffu, cur > prev);
  while (has) {
    int l = __ffs(has) - 1;
    has &= has - 1;
    long long p = __shfl_sync(0xffffffffu, prev, l), c = __shfl_sync(0xffffffffu, cur, l);
    long long ii = __shfl_sync(0xffffffffu, i, l);
    for (long long k = p + 1 + lane; k <= c; k += 32) start[k] = (uint32_t)ii;
  }
}

cudaError_t launch_cell_table(const uint32_t* sorted_keys, int n, int bits, uint32_t* start, cudaStream_t s) {
  uint32_t C = 1u << (3 * bits);
  long long threads = (long long)n + 1;
  int blocks = (int)((threads + 255) / 256);
  k_cell_table<<<blocks, 256, 0, s>>>(sorted_keys, n, C, start); count_launch();
  return cudaGetLastError();
}

}  // namespace mvr
