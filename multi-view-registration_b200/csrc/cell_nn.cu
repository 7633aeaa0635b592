// cell_nn.cu -- exact 1-NN for MANY queries per target point: warp-cooperative scan of staged cells.
//
// What pcl::KdTreeFLANN::nearestKSearch(k = 1) answers for the reference (getFitnessScore, the correspondence
// estimators; mvr/src/registrator.cpp:502, 572, 649, 923), for the regime of BASELINE.json's throughput sweep:
// up to 16 queries per target point.  There the per-thread ball walk of pair_search.cuh wastes most of a warp
// (every lane follows its own rows and cell lengths); here the lanes of a warp share their candidates instead.
//
//   * target and queries are counting-sorted by the cells of ONE row-major grid (pair_index.cu), cell edge chosen
//     for a handful of target points per occupied cell;
//   * a warp takes 32 consecutive sorted queries -- with many queries per cell they mostly sit in one cell -- and,
//     for each distinct cell among them, stages the target points of the cell's 3 x 3 x 3 neighbourhood (nine
//     contiguous x runs) in shared memory, 32 at a time with one coalesced load, after which every lane of that
//     cell compares ALL staged points against its query: uniform trip counts, broadcast shared-memory reads, no
//     divergence inside a cell;
//   * the neighbourhood holds the true neighbour whenever the best distance found is smaller than the distance
//     from the query to the neighbourhood's boundary (checked per query with the conservative cell geometry of
//     pair_search.cuh); the few queries that fail the test finish with the seeded general search of pair_search.cuh.
//
// Ties resolve to the lowest original index: the comparison key is (d2 bits, index) as one 64-bit integer.
// Algorithmic bytes: 16 B per query read + 8 B result, 16 B per target point, 8 B per cell-table entry.
#include "launch.h"
#include "pair_search.cuh"

namespace mvr {

constexpr int CN_THREADS = 256;
constexpr int CN_WARPS = CN_THREADS / 32;

struct CellNnArgs {
  const float4* q;          // queries sorted by cell, .w = bits(original index); finite ones first
  int nq;
  const uint32_t* q_valid;  // device: number of finite queries (= the query cell table's entry of the sentinel cell)
  const float4* tgt;        // target sorted by cell, .w = bits(original index)
  const uint32_t* tstart;
  PairGrid g;
  int m_valid;
  int32_t* out_idx;         // by ORIGINAL query index
  float* out_d2;
};

__device__ __forceinline__ void cn_eval(const float4 p, int pos, float qx, float qy, float qz, unsigned long long& bkey, int& bpos) {
  const float d = d2_pinned(qx, qy, qz, p.x, p.y, p.z);
  // d >= 0 or NaN: its bits order like the value, NaN sorts above +inf and never wins
  const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned long long)__float_as_uint(p.w);
  if (key < bkey) { bkey = key; bpos = pos; }
}

// Distance (cells) from scaled coordinate t in cell c to the nearest face of the block [c - h, c + h] that still has
// grid behind it (+inf if the block reaches both ends of the axis).
__device__ __forceinline__ float cn_face(float t, int c, int n, int h) {
  float u = MVR_INF;
  if (c - h > 0) u = fminf(u, t - (float)(c - h));
  if (c + h < n - 1) u = fminf(u, (float)(c + h + 1) - t);
  return u;
}

constexpr int CN_MINBLOCKS = 4;
__global__ void __launch_bounds__(CN_THREADS, CN_MINBLOCKS) k_cell_nn(CellNnArgs a) {
  __shared__ float4 s_pts[CN_WARPS][PG_SEGS * 32 / 2];   // 32 staged points per warp; the fallback's segment list (PG_SEGS x 32 uint2) reuses it
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const PairGrid g = a.g;
  const int rowlen = g.nx, slab = g.nx * g.ny;
  const int nwarps = gridDim.x * CN_WARPS;
  const int chunks = (a.nq + 31) / 32;
  const int nq_valid = (int)__ldg(a.q_valid);
  const float cell2 = g.cell_lo * g.cell_lo * MVR_REL_SHRINK;
  for (int chunk = blockIdx.x * CN_WARPS + warp; chunk < chunks; chunk += nwarps) {
    const int i = chunk * 32 + lane;
    const bool valid = i < nq_valid && a.m_valid > 0;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < a.nq) q = __ldg(a.q + i);
    float tx = 0.f, ty = 0.f, tz = 0.f;
    int cx = 0, cy = 0, cz = 0;
    uint32_t ckey = 0xffffffffu;
    if (valid) {
      tx = grid_t(q.x, g.ox, g.inv_cell); ty = grid_t(q.y, g.oy, g.inv_cell); tz = grid_t(q.z, g.oz, g.inv_cell);
      cx = pg_cell(tx, g.nx); cy = pg_cell(ty, g.ny); cz = pg_cell(tz, g.nz);
      ckey = (uint32_t)((cz * g.ny + cy) * g.nx + cx);
    }
    unsigned long long bkey = 0x7f8000007fffffffull;   // (+inf, INT_MAX)
    int bpos = -1;

    // ---- level 1: the 3 x 3 x 3 neighbourhood of every distinct cell of the chunk, shared by the lanes of that cell
    unsigned int todo = __ballot_sync(0xffffffffu, valid);
    while (todo) {
      const int leader = __ffs(todo) - 1;
      const uint32_t lkey = __shfl_sync(0xffffffffu, ckey, leader);
      const int lx = __shfl_sync(0xffffffffu, cx, leader), ly = __shfl_sync(0xffffffffu, cy, leader), lz = __shfl_sync(0xffffffffu, cz, leader);
      const bool mine = valid && ckey == lkey;
      todo &= ~__ballot_sync(0xffffffffu, mine);
      // the nine x runs of the neighbourhood: lane r < 9 fetches row (ly + r % 3 - 1, lz + r / 3 - 1)
      uint32_t rs = 0, re = 0;
      if (lane < 9) {
        const int y = ly + lane % 3 - 1, z = lz + lane / 3 - 1;
        if (y >= 0 && y < g.ny && z >= 0 && z < g.nz) {
          const uint32_t* row = a.tstart + (size_t)z * slab + (size_t)y * rowlen;
          rs = __ldg(row + max(lx - 1, 0));
          re = __ldg(row + min(lx + 1, g.nx - 1) + 1);
        }
      }
      // run by run, 32 points at a time: one coalesced load into the warp's staging area, then every lane of the cell
      // compares all of them (measured on B200: staging all nine runs at once with cp.async was slower)
#pragma unroll 1
      for (int r = 0; r < 9; ++r) {
        const uint32_t s = __shfl_sync(0xffffffffu, rs, r), e = __shfl_sync(0xffffffffu, re, r);
        for (uint32_t t0 = s; t0 < e; t0 += 32u) {
          const int cnt = (int)min(32u, e - t0);
          if (lane < cnt) s_pts[warp][lane] = __ldg(a.tgt + t0 + lane);
          __syncwarp();
          if (mine) {
            int c = 0;
            for (; c + 4 <= cnt; c += 4) {
              const float4 p0 = s_pts[warp][c], p1 = s_pts[warp][c + 1], p2 = s_pts[warp][c + 2], p3 = s_pts[warp][c + 3];
              cn_eval(p0, (int)t0 + c, q.x, q.y, q.z, bkey, bpos);
              cn_eval(p1, (int)t0 + c + 1, q.x, q.y, q.z, bkey, bpos);
              cn_eval(p2, (int)t0 + c + 2, q.x, q.y, q.z, bkey, bpos);
              cn_eval(p3, (int)t0 + c + 3, q.x, q.y, q.z, bkey, bpos);
            }
            for (; c < cnt; ++c) cn_eval(s_pts[warp][c], (int)t0 + c, q.x, q.y, q.z, bkey, bpos);
          }
          __syncwarp();
        }
      }
    }

    // Is a neighbourhood of half-width h enough?  Everything outside it is farther than cn_face cells away.
    const float margin = MVR_CELL_MARGIN + 1.0e-6f * fmaxf(fabsf(tx), fmaxf(fabsf(ty), fabsf(tz)));
    auto enough = [&](int h) {
      const float u = fminf(cn_face(tx, cx, g.nx, h), fminf(cn_face(ty, cy, g.ny, h), cn_face(tz, cz, g.nz, h)));
      const float bu = fmaxf(u - margin, 0.0f);
      return (u == MVR_INF) || (__uint_as_float((uint32_t)(bkey >> 32)) < bu * bu * cell2);
    };
    const bool open = valid && !enough(1);

    __syncwarp();
    if (valid) {
      NnBest b{__uint_as_float((uint32_t)(bkey >> 32)), (int)(uint32_t)bkey, bpos};
      // ---- the few queries the neighbourhood cannot settle (far from the cloud): the seeded general search
      //      (its segment list lives in the warp's staging area, which the warp is done with)
      if (open) pg_search<4, 32>(g, a.tstart, a.tgt, a.m_valid, q.x, q.y, q.z, q.x, q.y, q.z, 0.0f, 1.0f, MVR_INF, b,
                                 reinterpret_cast<uint2*>(&s_pts[warp][0]) + lane);
      const int oi = __float_as_int(q.w);
      a.out_idx[oi] = b.pos >= 0 ? b.idx : -1;
      a.out_d2[oi] = b.pos >= 0 ? b.d2 : MVR_INF;
    } else if (i < a.nq) {
      const int oi = __float_as_int(q.w);
      a.out_idx[oi] = -1;
      a.out_d2[oi] = MVR_INF;
    }
    __syncwarp();   // the staging area is reused by the next chunk
  }
}

// ---------------------------------------------------------------------------------------------
// One WARP per query: exact un-gated 1-NN of queries in any order, for batches too small (or too sparse) to be worth
// sorting.  A per-thread search is a serial chain of dependent loads (cell table -> points, row after row: ~100 us for a
// batch that fits one wave, whatever its size); here the 32 lanes of a warp share ONE query: each lane fetches the table
// entries of one row of the cube of cells [c - h, c + h]^3 around the query's cell, the lanes then split the candidates of
// all rows evenly among themselves, and a 64-bit shuffle reduction of (d2 bits, index) keys picks the lexicographic minimum.
// The cube doubles (h = 1, 2, 4, ...) until the best distance is provably smaller than anything outside it -- for a
// query near the surface the first cube settles it: two dependent load round trips per query instead of dozens.
// Getting through empty space (a query tens of cells from the cloud) costs two table loads per row, 32 rows at a time.
// ---------------------------------------------------------------------------------------------
constexpr int WN_THREADS = 256;
constexpr int WN_WARPS = WN_THREADS / 32;

__global__ void __launch_bounds__(WN_THREADS, 4) k_warp_nn(const float4* __restrict__ q, int n, const float4* __restrict__ tgt,
                                                           const uint32_t* __restrict__ tstart, PairGrid g, int m_valid,
                                                           int32_t* __restrict__ out_idx, float* __restrict__ out_d2) {
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * WN_WARPS;
  const float cell2 = g.cell_lo * g.cell_lo * MVR_REL_SHRINK;
  const int rowlen = g.nx, slab = g.nx * g.ny;
  for (int i = blockIdx.x * WN_WARPS + (threadIdx.x >> 5); i < n; i += nwarps) {
    const float4 p = __ldg(q + i);
    if (!finite3(p) || m_valid <= 0) {
      if (lane == 0) { out_idx[i] = -1; out_d2[i] = MVR_INF; }
      continue;
    }
    const float tx = grid_t(p.x, g.ox, g.inv_cell), ty = grid_t(p.y, g.oy, g.inv_cell), tz = grid_t(p.z, g.oz, g.inv_cell);
    const int cx = pg_cell(tx, g.nx), cy = pg_cell(ty, g.ny), cz = pg_cell(tz, g.nz);
    const float margin = MVR_CELL_MARGIN + 1.0e-6f * fmaxf(fabsf(tx), fmaxf(fabsf(ty), fabsf(tz)));
    unsigned long long bkey = 0x7f8000007fffffffull;   // (+inf, INT_MAX)
    for (int h = 1;; h <<= 1) {
      const int x0 = max(cx - h, 0), x1 = min(cx + h, g.nx - 1);
      const int y0 = max(cy - h, 0), y1 = min(cy + h, g.ny - 1);
      const int z0 = max(cz - h, 0), z1 = min(cz + h, g.nz - 1);
      const int ny_c = y1 - y0 + 1, rows = ny_c * (z1 - z0 + 1);
      for (int r0 = 0; r0 < rows; r0 += 32) {
        // lane -> row: its run of sorted positions
        uint32_t rs = 0, len = 0;
        const int r = r0 + lane;
        if (r < rows) {
          const int y = y0 + r % ny_c, z = z0 + r / ny_c;
          // (the inner cube is scanned again when h doubles: duplicates never win, and the work is a geometric series)
          const uint32_t* row = tstart + (size_t)z * slab + (size_t)y * rowlen;
          rs = __ldg(row + x0);
          len = __ldg(row + x1 + 1) - rs;
        }
        // the lanes split the candidates of the 32 runs evenly: candidate c of the concatenation belongs to the run whose
        // inclusive prefix first exceeds c
        uint32_t incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += t;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        for (uint32_t c0 = 0; c0 < total; c0 += 32u) {
          const uint32_t c = c0 + (uint32_t)lane;
          // run of candidate c: the number of runs whose inclusive prefix is <= c (binary search over the lanes' prefixes)
          int lo = 0;
#pragma unroll
          for (int step = 16; step > 0; step >>= 1) {
            const uint32_t pv = __shfl_sync(0xffffffffu, incl, lo + step - 1);
            if (pv <= c) lo += step;
          }
          const int src = min(lo, 31);
          const uint32_t s_rs = __shfl_sync(0xffffffffu, rs, src), s_in = __shfl_sync(0xffffffffu, incl, src), s_len = __shfl_sync(0xffffffffu, len, src);
          if (c < total) {
            const uint32_t k = s_rs + (c - (s_in - s_len));
            const float4 t = __ldg(tgt + k);
            const float d = d2_pinned(p.x, p.y, p.z, t.x, t.y, t.z);
            const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned long long)__float_as_uint(t.w);
            if (key < bkey) bkey = key;
          }
        }
      }
      // the warp's best so far
      unsigned long long wkey = bkey;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, wkey, o);
        if (other < wkey) wkey = other;
      }
      bkey = wkey;
      // is the cube enough?  Everything outside it is farther than u cells away along some axis.
      const float u = fminf(cn_face(tx, cx, g.nx, h), fminf(cn_face(ty, cy, g.ny, h), cn_face(tz, cz, g.nz, h)));
      if (u == MVR_INF) break;   // the cube is the whole grid
      const float bu = fmaxf(u - margin, 0.0f);
      if (__uint_as_float((uint32_t)(bkey >> 32)) < bu * bu * cell2) break;
    }
    if (lane == 0) {
      const int idx = (int)(uint32_t)bkey;
      out_idx[i] = idx == 0x7fffffff ? -1 : idx;
      out_d2[i] = idx == 0x7fffffff ? MVR_INF : __uint_as_float((uint32_t)(bkey >> 32));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Cell-sorted queries, one thread per query, SEEDED: the fused ICP iteration's search (pair_search.cuh) owes its speed to a
// seed -- a real candidate near the query, so that the ball that provably holds the answer is about a cell wide.  Un-gated
// queries have no previous iteration to take one from; sorted by cell they get one almost for free:
//   1. every query scans the target points of ITS OWN cell (one table load pair, a handful of candidates);
//   2. a query whose cell holds no target point (it sits beside the surface) borrows the best candidate of the nearest lane
//      of its warp that has one -- the lanes of a warp are neighbours in cell order, and ANY real candidate is a valid seed;
//   3. the seeded ball walk finishes the query exactly (lanes still without a seed start from the growing cube).
// Against the cell-cooperative pass above (which evaluates the whole 27-cell neighbourhood, ~100 candidates per query) a
// query evaluates ~30; against the unseeded per-thread walk it skips the 27-cell first cube.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(FUSED_THREADS, 4) k_seeded_nn(const float4* __restrict__ q, int nq, const uint32_t* __restrict__ q_valid,
                                                                const float4* __restrict__ tgt, const uint32_t* __restrict__ tstart, PairGrid g,
                                                                int m_valid, int32_t* __restrict__ out_idx, float* __restrict__ out_d2) {
  __shared__ uint2 s_seg[PG_SEGS * PG_STRIDE];
  const int i = blockIdx.x * FUSED_THREADS + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int nq_valid = (int)__ldg(q_valid);
  const float far2 = 4.0f / (g.inv_cell * g.inv_cell);   // (two cell edges)^2
  float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < nq) p = __ldg(q + i);
  const bool fin = i < nq_valid && m_valid > 0;
  NnBest b{MVR_INF, 0x7fffffff, -1};
  if (fin) {
    const int cx = pg_cell(grid_t(p.x, g.ox, g.inv_cell_x), g.nx), cy = pg_cell(grid_t(p.y, g.oy, g.inv_cell), g.ny),
              cz = pg_cell(grid_t(p.z, g.oz, g.inv_cell), g.nz);
    const uint32_t* row = tstart + ((size_t)cz * g.ny + cy) * g.nx;
    pg_scan(tgt, __ldg(row + cx), __ldg(row + cx + 1), p.x, p.y, p.z, b);
  }
  const unsigned int have = __ballot_sync(0xffffffffu, fin && b.pos >= 0);
  const unsigned int need = __ballot_sync(0xffffffffu, fin && b.pos < 0);
  if (need && have) {
    const unsigned int below = have & ((1u << lane) - 1u), above = lane < 31 ? (have & ~((2u << lane) - 1u)) : 0u;
    const int lo = below ? 31 - __clz((int)below) : -1, hi = above ? __ffs((int)above) - 1 : -1;
    const int src = lo < 0 ? hi : (hi < 0 ? lo : (lane - lo <= hi - lane ? lo : hi));
    const int spos = __shfl_sync(0xffffffffu, b.pos, src < 0 ? lane : src);
    if (fin && b.pos < 0 && spos >= 0) {
      const float4 t = __ldg(tgt + spos);
      const float d = d2_pinned(p.x, p.y, p.z, t.x, t.y, t.z);
      // a far seed is worse than none: the ball walk visits every row inside its radius, the growing cube stops at the first
      // cube that holds a point (lanes at the end of a row sit next to lanes of another row)
      if (d <= far2) { b.d2 = d; b.idx = __float_as_int(t.w); b.pos = spos; }
    }
  }
  if (fin) pg_search<8>(g, tstart, tgt, m_valid, p.x, p.y, p.z, p.x, p.y, p.z, 0.0f, 1.0f, MVR_INF, b, s_seg + threadIdx.x);
  if (i < nq) {
    const int o = __float_as_int(p.w);
    out_idx[o] = b.pos >= 0 ? b.idx : -1;
    out_d2[o] = b.pos >= 0 ? b.d2 : MVR_INF;
  }
}

cudaError_t launch_seeded_nn(const float4* q_sorted, int nq, const uint32_t* d_nq_valid, const float4* tgt_sorted, const uint32_t* tstart, PairGrid g,
                             int m_valid, int32_t* out_idx, float* out_d2, cudaStream_t s) {
  if (nq <= 0) return cudaSuccess;
  k_seeded_nn<<<(nq + FUSED_THREADS - 1) / FUSED_THREADS, FUSED_THREADS, 0, s>>>(q_sorted, nq, d_nq_valid, tgt_sorted, tstart, g, m_valid, out_idx, out_d2);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_warp_nn(const float4* q, int n, const float4* tgt_sorted, const uint32_t* tstart, PairGrid g, int m_valid, int32_t* out_idx,
                           float* out_d2, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int blocks = std::min((n + WN_WARPS - 1) / WN_WARPS, 148 * 8 * 16);
  k_warp_nn<<<blocks, WN_THREADS, 0, s>>>(q, n, tgt_sorted, tstart, g, m_valid, out_idx, out_d2); count_launch();
  return cudaGetLastError();
}

cudaError_t launch_cell_nn(const float4* q_sorted, int nq, const uint32_t* d_nq_valid, const float4* tgt_sorted, const uint32_t* tstart, PairGrid g,
                           int m_valid, int32_t* out_idx, float* out_d2, cudaStream_t s) {
  if (nq <= 0) return cudaSuccess;
  CellNnArgs a{q_sorted, nq, d_nq_valid, tgt_sorted, tstart, g, m_valid, out_idx, out_d2};
  const int chunks = (nq + 31) / 32;
  const int blocks = std::min((chunks + CN_WARPS - 1) / CN_WARPS, 148 * 4 * 8);
  k_cell_nn<<<blocks, CN_THREADS, 0, s>>>(a); count_launch();
  return cudaGetLastError();
}

}  // namespace mvr
