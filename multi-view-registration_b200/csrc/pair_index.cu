// pair_index.cu -- the per-align spatial index of the fused ICP loop: row-major uniform grid, built ONCE.
//
// pcl::IterativeClosestPoint builds the target kd-tree once per align and, with reciprocal
// correspondences, a source kd-tree in EVERY iteration (SURVEY.md A3/A5; enabled by the reference at
// mvr/src/registrator.cpp:552, 768, 901).  Here both clouds are binned once per align: the target in a
// grid over its own box, the source -- after the initial guess has been applied -- in a grid over the
// guessed source box.  The source then moves rigidly every iteration but keeps its cells: the search
// (pair_search.cuh) carries the query into the binning frame instead of re-sorting 200k points 30 times.
//
// The build is a counting sort made deterministic (four launches, no multi-pass radix sort):
//   k_pair_count   : p <- guess * p (pinned float transform, ICP's transformCloud, SURVEY.md A10) when a guess is
//                    given; key = row-major cell (z, y, x; x fastest), non-finite points get the sentinel key
//                    `cells`; rank = the point's arrival number in its cell (one atomicAdd on the cell counter)
//   k_scan_cells_batch : exclusive scan of the counters -> start[c] = first sorted position of cell c (decoupled
//                    look-back; the counters are zeroed on the way for the next build)
//   k_pair_scatter : tmp[start[key] + rank] = {moved point, bits(original index)} -- arrival order inside a cell
//   k_pair_rerank  : the final position of a point = start[key] + number of points of its cell with a SMALLER
//                    original index (its cell is ~10 contiguous records of tmp), so points of a cell end up in
//                    ascending original index whatever order the atomics ran in: every sorted position, and with
//                    it the order of every later reduction, is reproducible run to run.
//
// Algorithmic bytes per point: 16 read + 16 written, + 8 B per cell.
#include <algorithm>

#include "launch.h"
#include "pair_search.cuh"

namespace mvr {

// One launch per phase serves EVERY build of a batch (blockIdx.y = job; the jobs travel by value in the kernel's
// parameter space): a 24-pair registration builds 48 indices with 4 launches instead of 192.
__device__ __forceinline__ const BuildJob& load_job(const BuildBatch& b, BuildJob& s_job) {
  static_assert(sizeof(BuildJob) % 4 == 0 && sizeof(BuildJob) / 4 <= 256, "job block");
  if (threadIdx.x < sizeof(BuildJob) / 4) ((uint32_t*)&s_job)[threadIdx.x] = ((const uint32_t*)&b.j[blockIdx.y])[threadIdx.x];
  __syncthreads();
  return s_job;
}

__global__ void __launch_bounds__(256) k_pair_count(const __grid_constant__ BuildBatch b) {
  __shared__ BuildJob s_job;
  const BuildJob& j = load_job(b, s_job);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n) return;
  float4 p = __ldg(j.in + i);
  const bool ok = finite3(p);
  if (j.apply && ok) p = xform_pinned(j.M, p);
  const uint32_t key = ok ? pg_key(p, j.g) : j.cells;
  j.keys[i] = key;
  j.rank[i] = atomicAdd(j.counters + key, 1u);
}

// ---------------------------------------------------------------------------------------------
// single-pass exclusive scan (Merrill & Garland decoupled look-back), 8192 counters per tile.
// tile_state[t] = (epoch*4 + flag) << 32 | value, flag 1 = tile aggregate, 2 = inclusive prefix;
// words written under an older epoch read as "not ready", so the array never needs clearing.
// ---------------------------------------------------------------------------------------------
constexpr int SC_THREADS = 256;
constexpr int SC_ITEMS = 32;   // counters per thread: the prefix travels down the tiles 32 tiles per look-back round trip, so a
                               // tile is made large (8192 counters) -- with 2048 a 1.7M-cell table took 25 us, latency all of it
constexpr int SC_TILE = SC_THREADS * SC_ITEMS;

int scan_num_tiles(size_t len) { return (int)((len + SC_TILE - 1) / SC_TILE); }

__device__ __forceinline__ void scan_tiles(uint32_t* __restrict__ counters, uint32_t* __restrict__ start, uint32_t len,
                                           unsigned long long* __restrict__ tile_state, uint32_t epoch, uint32_t ntiles);

// The cell tables of every build of a batch in one launch (blockIdx.y = job).
__global__ void __launch_bounds__(SC_THREADS) k_scan_cells_batch(const __grid_constant__ BuildBatch b) {
  __shared__ uint32_t* s_counters;
  __shared__ uint32_t* s_start;
  __shared__ unsigned long long* s_tiles;
  __shared__ uint32_t s_len, s_epoch, s_ntiles;
  if (threadIdx.x == 0) {
    const BuildJob& j = b.j[blockIdx.y];
    s_counters = j.counters; s_start = j.start; s_tiles = j.tiles; s_len = j.cells + 1u; s_epoch = j.epoch; s_ntiles = (uint32_t)j.ntiles;
  }
  __syncthreads();
  scan_tiles(s_counters, s_start, s_len, s_tiles, s_epoch, s_ntiles);
}

// tile_state[0] is the ticket counter of the launch (tiles are handed out in the order blocks START, so a tile never waits
// for a predecessor that has not been scheduled yet; the block that draws the last ticket resets the counter for the next
// launch); tile t's state word lives at tile_state[1 + t].
// ntiles: tiles of this table; gridDim.x >= ntiles blocks draw tickets (a batched launch is as wide as its largest table).
__device__ __forceinline__ void scan_tiles(uint32_t* __restrict__ counters, uint32_t* __restrict__ start, uint32_t len,
                                           unsigned long long* __restrict__ tile_state, uint32_t epoch, uint32_t ntiles) {
  __shared__ uint32_t warp_sums[SC_THREADS / 32];
  __shared__ uint32_t s_prefix, s_tile;
  if (threadIdx.x == 0) {
    unsigned int* ticket = reinterpret_cast<unsigned int*>(tile_state);
    const unsigned int t = atomicAdd(ticket, 1u);
    if (t == gridDim.x - 1) *ticket = 0u;   // every ticket of this launch has been drawn
    s_tile = t;
  }
  __syncthreads();
  const uint32_t tile = s_tile;
  if (tile >= ntiles) return;
  volatile unsigned long long* st = tile_state + 1;
  const uint32_t base = tile * SC_TILE + threadIdx.x * SC_ITEMS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t v[SC_ITEMS];
  if (base + SC_ITEMS <= len) {
#pragma unroll
    for (int k = 0; k < SC_ITEMS; k += 4) {
      const uint4 a = *reinterpret_cast<const uint4*>(counters + base + k);
      v[k] = a.x; v[k + 1] = a.y; v[k + 2] = a.z; v[k + 3] = a.w;
      *reinterpret_cast<uint4*>(counters + base + k) = make_uint4(0, 0, 0, 0);
    }
  } else {
#pragma unroll
    for (int k = 0; k < SC_ITEMS; ++k) {
      v[k] = (base + k < len) ? counters[base + k] : 0u;
      if (base + k < len) counters[base + k] = 0u;
    }
  }
  uint32_t tsum = 0;
#pragma unroll
  for (int k = 0; k < SC_ITEMS; ++k) tsum += v[k];
  uint32_t incl = tsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  uint32_t wbase = 0, agg = 0;
#pragma unroll
  for (int w = 0; w < SC_THREADS / 32; ++w) { uint32_t c = warp_sums[w]; if (w < warp) wbase += c; agg += c; }
  const uint32_t texcl = wbase + incl - tsum;

  const unsigned long long tag = (unsigned long long)epoch << 34;
  if (warp == 0) {
    if (tile == 0) {
      if (lane == 0) { st[0] = tag | (2ull << 32) | agg; s_prefix = 0; }
    } else {
      if (lane == 0) st[tile] = tag | (1ull << 32) | agg;
      uint32_t excl = 0;
      int j = (int)tile - 1;
      while (true) {
        const int t = j - lane;
        unsigned long long w = 0;
        bool ready;
        do {
          w = (t >= 0) ? st[t] : (tag | (2ull << 32));
          ready = (w >> 34) == (unsigned long long)epoch && ((w >> 32) & 3ull) != 0;
        } while (!__all_sync(0xffffffffu, ready));
        const uint32_t flag = (uint32_t)(w >> 32) & 3u, val = (uint32_t)w;
        const uint32_t incl_mask = __ballot_sync(0xffffffffu, flag == 2u);
        if (incl_mask) {
          const int first = __ffs(incl_mask) - 1;   // nearest predecessor holding an inclusive prefix
          uint32_t c = (lane <= first) ? val : 0u;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
          excl += c;
          break;
        }
        uint32_t c = val;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        excl += c;
        j -= 32;
      }
      if (lane == 0) { st[tile] = tag | (2ull << 32) | (excl + agg); s_prefix = excl; }
    }
  }
  __syncthreads();
  uint32_t run = s_prefix + texcl;
  if (base + SC_ITEMS <= len) {
#pragma unroll
    for (int k = 0; k < SC_ITEMS; k += 4) {
      uint4 a;
      a.x = run; run += v[k]; a.y = run; run += v[k + 1]; a.z = run; run += v[k + 2]; a.w = run; run += v[k + 3];
      *reinterpret_cast<uint4*>(start + base + k) = a;
    }
  } else {
#pragma unroll
    for (int k = 0; k < SC_ITEMS; ++k) {
      if (base + k < len) start[base + k] = run;
      run += v[k];
    }
  }
  // total after the last counter
  if (tile == ntiles - 1 && threadIdx.x == SC_THREADS - 1) start[len] = s_prefix + agg;
}

__global__ void __launch_bounds__(256) k_pair_scatter(const __grid_constant__ BuildBatch b) {
  __shared__ BuildJob s_job;
  const BuildJob& j = load_job(b, s_job);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n) return;
  float4 p = __ldg(j.in + i);
  if (j.apply && finite3(p)) p = xform_pinned(j.M, p);   // the same pinned arithmetic as k_pair_count: the same point
  p.w = __uint_as_float((uint32_t)i);
  (j.ordered ? j.tmp : j.sorted)[__ldg(j.start + __ldg(j.keys + i)) + __ldg(j.rank + i)] = p;
}

// A cell that holds more than RERANK_LIMIT points (duplicated or invalid returns piled on one spot, outliers clamped into a
// boundary cell) would make the rank count below quadratic: its points keep their arrival order instead and the population is
// reported through *crowded (searches stay exact; only the run-to-run order of sums over that cell's points is lost).
constexpr uint32_t RERANK_LIMIT = 1024;
__global__ void __launch_bounds__(256) k_pair_rerank(const __grid_constant__ BuildBatch b) {
  __shared__ BuildJob s_job;
  const BuildJob& j = load_job(b, s_job);
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= j.n || !j.ordered) return;
  const float4* __restrict__ tmp = j.tmp;
  const float4 p = __ldg(tmp + k);
  const uint32_t idx = __float_as_uint(p.w);
  const uint32_t key = __ldg(j.keys + idx);
  const uint32_t s = __ldg(j.start + key), e = __ldg(j.start + key + 1);
  if (e - s > RERANK_LIMIT) {
    j.sorted[k] = p;
    if (j.crowded && (uint32_t)k == s) atomicMax(j.crowded, e - s);
    return;
  }
  uint32_t r = 0;
  for (uint32_t q = s; q < e; ++q) r += (__float_as_uint(__ldg(&tmp[q].w)) < idx) ? 1u : 0u;
  j.sorted[s + r] = p;
}

// ---------------------------------------------------------------------------------------------
// Gate mask of a target index: bit x of word [(z * ny + y) * wstride + x / 32] is set when some target point lies in a
// cell within D cells in y and z and Dx cells in x of cell (x, y, z).  Cells that differ by more than D in some axis are at least D cells
// apart along it, so with D cell >= gate a CLEAR bit proves that a query filed in that cell has no target point within the
// gate: pcl's "if (distance > max_dist_sqr) continue" (SURVEY.md A4) without a search.  The part of a turntable view the
// neighbouring view does not cover is settled by one load per point and iteration.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_gate_occ(const uint32_t* __restrict__ start, PairGrid g, int wstride, size_t words, uint32_t* __restrict__ occ) {
  const size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= words) return;
  const size_t row = w / (size_t)wstride;
  const int xw = (int)(w % (size_t)wstride);
  const uint32_t* r = start + row * (size_t)g.nx;
  uint32_t bits = 0;
  uint32_t prev = __ldg(r + xw * 32);
  for (int b = 0; b < 32; ++b) {
    const int x = xw * 32 + b;
    if (x >= g.nx) break;
    const uint32_t next = __ldg(r + x + 1);
    if (next > prev) bits |= 1u << b;
    prev = next;
  }
  occ[w] = bits;
}

__global__ void __launch_bounds__(256) k_gate_dilate(const uint32_t* __restrict__ occ, PairGrid g, int wstride, int D, int Dx, size_t words, uint32_t* __restrict__ out) {
  const size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= words) return;
  const int xw = (int)(w % (size_t)wstride);
  const size_t row = w / (size_t)wstride;
  const int y = (int)(row % (size_t)g.ny), z = (int)(row / (size_t)g.ny);
  uint32_t acc = 0;
  for (int zz = max(z - D, 0); zz <= min(z + D, g.nz - 1); ++zz)
    for (int yy = max(y - D, 0); yy <= min(y + D, g.ny - 1); ++yy) {
      const uint32_t* r = occ + ((size_t)zz * g.ny + yy) * wstride;
      const uint32_t cur = __ldg(r + xw), prev = xw > 0 ? __ldg(r + xw - 1) : 0u, next = xw + 1 < wstride ? __ldg(r + xw + 1) : 0u;
      uint32_t v = cur;
      for (int k = 1; k <= Dx; ++k) v |= (cur << k) | (cur >> k) | (prev >> (32 - k)) | (next << (32 - k));
      acc |= v;
    }
  out[w] = acc;
}

cudaError_t launch_gate_mask(const uint32_t* start, PairGrid g, int wstride, int D, int Dx, uint32_t* occ, uint32_t* mask, cudaStream_t s) {
  const size_t words = (size_t)g.ny * g.nz * wstride;
  if (words == 0 || D < 1 || Dx < 1 || Dx > 31) return cudaErrorInvalidValue;
  const unsigned blocks = (unsigned)((words + 255) / 256);
  k_gate_occ<<<blocks, 256, 0, s>>>(start, g, wstride, words, occ); count_launch();
  k_gate_dilate<<<blocks, 256, 0, s>>>(occ, g, wstride, D, Dx, words, mask); count_launch();
  return cudaGetLastError();
}

// The four phases of `count` index builds (<= BUILD_MAX_JOBS) on stream s.
cudaError_t launch_pair_builds(const BuildBatch& batch, int count, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (count > BUILD_MAX_JOBS) return cudaErrorInvalidValue;
  int max_n = 0, max_tiles = 0;
  bool any_ordered = false;
  for (int k = 0; k < count; ++k) {
    max_n = std::max(max_n, batch.j[k].n);
    max_tiles = std::max(max_tiles, batch.j[k].ntiles);
    any_ordered = any_ordered || batch.j[k].ordered;
  }
  const dim3 gp((unsigned)std::max((max_n + 255) / 256, 1), (unsigned)count);
  if (max_n > 0) { k_pair_count<<<gp, 256, 0, s>>>(batch); count_launch(); }
  if (max_tiles > 0) { k_scan_cells_batch<<<dim3((unsigned)max_tiles, (unsigned)count), SC_THREADS, 0, s>>>(batch); count_launch(); }
  if (max_n > 0) { k_pair_scatter<<<gp, 256, 0, s>>>(batch); count_launch(); }
  if (max_n > 0 && any_ordered) { k_pair_rerank<<<gp, 256, 0, s>>>(batch); count_launch(); }
  return cudaGetLastError();
}

}  // namespace mvr
