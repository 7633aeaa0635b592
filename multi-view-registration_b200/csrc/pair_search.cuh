// pair_search.cuh -- exact nearest neighbour of one query in a ROW-MAJOR uniform grid whose points may
// have MOVED rigidly since they were binned (device side of the fused ICP iteration, icp.cu).
//
// This is the 1-NN search pcl::KdTreeFLANN::nearestKSearch(k = 1) answers for the reference inside
// icp.align (mvr/src/registrator.cpp:569, 920, 1012, 1024; SURVEY.md A4-A6), laid out for the way ICP
// asks it:
//   * both clouds of an align are binned ONCE (pair_index.cu) in a grid of nx x ny x nz cells, points
//     sorted by cell in row-major order (x fastest), so the cells [x0, x1] of one (y, z) row are ONE
//     contiguous run of the sorted array: a ball query walks a few rows, two table loads per row;
//   * every search starts from a SEED -- the neighbour found in the previous iteration (forward half)
//     or the distance of the nearest chooser (reciprocal half).  The seed is a real candidate, so the
//     ball of radius sqrt(seed d2) around the query provably holds the answer and is usually 1-2 cells
//     wide once the alignment has settled;
//   * the source cloud moves every iteration, but rigidly: its cells are kept in the frame it was
//     binned in (positions s0), the query is carried into that frame (u = C^-1 t), and distances are
//     evaluated on the CURRENT coordinates, so results are bit-identical to a search over a freshly
//     built index.  What the stale cells cost is a slack on every geometric bound, see below.
//
// Exactness, first for points that have not moved (dev = 0, stretch = 1: the target of the forward half,
// every index but the moving source).  grid_t() rounds with |error| <= 2^-23 |t| per point;
// margin (cells) = MVR_CELL_MARGIN + 1e-6 |t| absorbs that on both the query and the indexed point.  A
// point whose pinned float d2 is <= lim has |p_a - q_a| <= sqrt(lim) (1 + 2^-22) on every axis, hence its
// cell coordinate lies in [floor(t_a - rc), floor(t_a + rc)] with rc = sqrt(lim) inv_cell (1 + 1e-6) +
// margin: the box of rows walked below cannot miss it.  Lower bounds of rows and cells shrink the
// geometric gap by margin, use cell_lo (a float strictly below the true cell edge) and a relative 1e-6
// (MVR_REL_SHRINK), so lb is a true lower bound on the float d2 of every point filed there; a row or cell
// is skipped only when lb exceeds the running limit (strictly), so equal-distance ties with a lower index
// are never cut off.
// Points that moved rigidly: let a candidate k have pinned float d2(t, cur_k) <= lim; then |t - cur_k| <= rho
// with rho = sqrt(lim) (1 + 2^-22).  With C x = A x + b the accumulated increment since binning and
// dev >= |cur_k - C s0_k| for every k (bounded analytically by the solve, icp.cu icp_advance_frame):
//     u - s0_k = A^-1 (t - C s0_k)   =>   |u - s0_k| <= stretch (rho + dev),   stretch >= ||A^-1||_2.
// Hence s0_k's cell lies inside the box of radius rc = (sqrt(lim) stretch inv_cell)(1 + 1e-6) + margin
// around u's scaled coordinate, where margin grows by dev stretch inv_cell.  Conversely a point whose cell
// is gamma away from u (per-axis gaps already shrunk by margin) has |t - cur_k| >= |gamma| cell / stretch,
// so the same strict test holds with cell_lo / stretch for the cell edge.  Boundary cells are unbounded
// outwards (cell_gap): points and queries outside the grid are filed in / start from the clamped cell.
#pragma once
#include "common.cuh"

namespace mvr {

struct NnBest {
  float d2;
  int idx;   // original index of the best point, INT_MAX if none
  int pos;   // its position in the sorted array (-1 for a seed)
};

// Gap (cells, >= 0) between scaled coordinate t and the slab of cell c, boundary cells unbounded outwards.
__device__ __forceinline__ float cell_gap(float t, int c, int G) {
  float lo = (c > 0) ? (float)c - t : 0.0f;
  float hi = (c < G - 1) ? t - (float)(c + 1) : 0.0f;
  return fmaxf(fmaxf(lo, hi), 0.0f);
}

__device__ __forceinline__ int pg_cell(float t, int n) { return (int)fminf(fmaxf(floorf(t), 0.0f), (float)(n - 1)); }

// Row-major cell of a finite point.
__device__ __forceinline__ uint32_t pg_key(float4 p, const PairGrid& g) {
  const int cx = pg_cell(grid_t(p.x, g.ox, g.inv_cell_x), g.nx);
  const int cy = pg_cell(grid_t(p.y, g.oy, g.inv_cell), g.ny);
  const int cz = pg_cell(grid_t(p.z, g.oz, g.inv_cell), g.nz);
  return (uint32_t)((cz * g.ny + cy) * g.nx + cx);
}

// Fold the points of sorted positions [s, e) into the running best; two independent loads per trip.
__device__ __forceinline__ void pg_scan(const float4* __restrict__ pts, uint32_t s, uint32_t e, float qx, float qy, float qz, NnBest& b) {
  uint32_t k = s;
  for (; k + 1 < e; k += 2) {
    const float4 p0 = __ldg(pts + k), p1 = __ldg(pts + k + 1);
    const float d0 = d2_pinned(qx, qy, qz, p0.x, p0.y, p0.z), d1 = d2_pinned(qx, qy, qz, p1.x, p1.y, p1.z);
    const int i0 = __float_as_int(p0.w), i1 = __float_as_int(p1.w);
    if (lex_less(d0, i0, b.d2, b.idx)) { b.d2 = d0; b.idx = i0; b.pos = (int)k; }
    if (lex_less(d1, i1, b.d2, b.idx)) { b.d2 = d1; b.idx = i1; b.pos = (int)k + 1; }
  }
  if (k < e) {
    const float4 p0 = __ldg(pts + k);
    const float d0 = d2_pinned(qx, qy, qz, p0.x, p0.y, p0.z);
    const int i0 = __float_as_int(p0.w);
    if (lex_less(d0, i0, b.d2, b.idx)) { b.d2 = d0; b.idx = i0; b.pos = (int)k; }
  }
}

// Segment list of one thread in shared memory: slot j of thread t lives at seg[j * PG_STRIDE + t] (bank = t).
constexpr int PG_SEGS = 8;   // row segments collected before a flat scan
constexpr int PG_STRIDE = FUSED_THREADS;

// Flat scan of the thread's collected segments: ONE loop over all candidates of all rows, UNROLL independent loads per
// trip, so the trip count of a warp is the maximum over its lanes of the TOTAL number of candidates (not the sum over
// rows of per-row maxima) and the loads of a trip overlap.  Past a segment's end the last point is simply evaluated
// again: a duplicate never wins a strict lexicographic comparison.  (Measured on B200, same box: testing min(d) of a group against the best first, to skip the comparisons, was 9 % slower -- in
// a warp some lane nearly always improves; handing a block's queries out again sorted by their candidate count, so that the
// lanes of a warp scan lists of equal length, was 14 % slower (profiles/r02_work_sort_ab.log: three more block barriers and the
// lanes no longer read neighbouring cells); 8 loads per trip
// beat 4 by 2.5 % and 2 by 20 %; reading whole groups past the segment end into the next cells' points -- also exact --
// was 3 % slower, as was dropping the per-row x narrowing for narrow boxes; guarding every candidate of a trip by its
// own range test instead of re-reading the last point turned into divergent branches and was 70 % slower.)
template <int UNROLL, int STRIDE = PG_STRIDE>
__device__ __forceinline__ void pg_flat_scan(const float4* __restrict__ pts, const uint2* __restrict__ seg, int nseg, float qx, float qy,
                                             float qz, NnBest& b) {
  int j = 0;
  uint32_t k = 0, e = 0;
  for (;;) {
    if (k >= e) {   // collected segments are never empty: one step always lands on a candidate
      if (j >= nseg) return;
      const uint2 s = seg[j * STRIDE];
      ++j;
      k = s.x; e = s.y;
    }
    float4 p[UNROLL];
    uint32_t kk[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) { kk[u] = min(k + (uint32_t)u, e - 1u); p[u] = __ldg(pts + kk[u]); }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const float d = d2_pinned(qx, qy, qz, p[u].x, p[u].y, p[u].z);
      const int id = __float_as_int(p[u].w);
      if (lex_less(d, id, b.d2, b.idx)) { b.d2 = d; b.idx = id; b.pos = (int)kk[u]; }
    }
    k += UNROLL;
  }
}

// Nearest point to q among `pts` (current coordinates, .w = original index) sorted by the row-major
// cell of the positions they were BINNED at.  (ux, uy, uz): the query carried into the binning frame
// (= q when the points have not moved).  dev / stretch: see the header (0 / 1 for a static cloud).
// gate: nothing farther than this (float d2, rounded up) is of interest, +inf for none.  b may be
// pre-seeded with a real candidate or with a bare distance bound (idx = INT_MAX).
// seg: this thread's slot column of a PG_SEGS x STRIDE shared-memory array (slot j at seg[j * STRIDE]).
//
// Two phases per batch of rows: (1) walk the rows of the ball's box, prune by their lower bounds, and
// collect the surviving x runs as (start, end) segments; (2) scan all collected candidates in one flat
// loop.  A loose bound (ball wider than a cell: first iterations, bare gates) is first tightened on the
// query's own row.
template <int UNROLL, int STRIDE = PG_STRIDE>
__device__ __forceinline__ void pg_search(const PairGrid& g, const uint32_t* __restrict__ start, const float4* __restrict__ pts,
                                          int n_valid, float qx, float qy, float qz, float ux, float uy, float uz, float dev,
                                          float stretch, float gate, NnBest& b, uint2* __restrict__ seg) {
  if (n_valid <= 0) return;
  const float tx = grid_t(ux, g.ox, g.inv_cell_x), ty = grid_t(uy, g.oy, g.inv_cell), tz = grid_t(uz, g.oz, g.inv_cell);
  const int cx = pg_cell(tx, g.nx), cy = pg_cell(ty, g.ny), cz = pg_cell(tz, g.nz);
  // margins in cells of the respective axis (x cells are xr times finer)
  const float margin = MVR_CELL_MARGIN + 1.0e-6f * fmaxf(fabsf(ty), fabsf(tz)) + dev * stretch * g.inv_cell * 1.000001f;
  const float margin_x = MVR_CELL_MARGIN + 1.0e-6f * fabsf(tx) + dev * stretch * g.inv_cell_x * 1.000001f;
  const float rscale_x = stretch * g.inv_cell_x * 1.000001f;
  const int xri = (int)g.xr;
  const float cell2 = g.cell_lo * g.cell_lo * MVR_REL_SHRINK / (stretch * stretch * 1.000001f);
  const float inv_cell2 = 1.000002f / cell2;
  const float rscale = stretch * g.inv_cell * 1.000001f;
  const float fx = (float)(g.nx - 1), fy = (float)(g.ny - 1), fz = (float)(g.nz - 1);
  const int rowlen = g.nx, slab = g.nx * g.ny;

  float lim = fminf(b.d2, gate);
  if (!(lim < MVR_INF)) {
    // no bound at all (un-gated first iteration): grow a cube of cells until it holds a point
    for (int R = 1;; R <<= 1) {
      const int x0 = max(cx - R * xri, 0), x1 = min(cx + R * xri, g.nx - 1);
      const int y0 = max(cy - R, 0), y1 = min(cy + R, g.ny - 1);
      const int z0 = max(cz - R, 0), z1 = min(cz + R, g.nz - 1);
      for (int z = z0; z <= z1; ++z)
        for (int y = y0; y <= y1; ++y) {
          const uint32_t* row = start + (size_t)z * slab + (size_t)y * rowlen;
          pg_scan(pts, __ldg(row + x0), __ldg(row + x1 + 1), qx, qy, qz, b);
        }
      if (b.d2 < MVR_INF) break;
      if (x0 == 0 && y0 == 0 && z0 == 0 && x1 == g.nx - 1 && y1 == g.ny - 1 && z1 == g.nz - 1) return;   // empty index
    }
    lim = b.d2;
  }

  bool own_done = false;
  float rc = sqrtf(lim) * rscale + margin;
  if (rc > 1.25f) {
    // loose bound: the own row usually tightens it for all the others
    const float rcx = sqrtf(lim) * rscale_x + margin_x;
    const int x0 = (int)fminf(fmaxf(floorf(tx - rcx), 0.0f), fx), x1 = (int)fminf(fmaxf(floorf(tx + rcx), 0.0f), fx);
    const uint32_t* row = start + (size_t)cz * slab + (size_t)cy * rowlen;
    pg_scan(pts, __ldg(row + x0), __ldg(row + x1 + 1), qx, qy, qz, b);
    lim = fminf(b.d2, gate);
    rc = sqrtf(lim) * rscale + margin;
    own_done = true;   // [x0, x1] of the own row covers whatever the tighter ball still needs there
  }
  const float rcx = sqrtf(lim) * rscale_x + margin_x;
  const int x0 = (int)fminf(fmaxf(floorf(tx - rcx), 0.0f), fx), x1 = (int)fminf(fmaxf(floorf(tx + rcx), 0.0f), fx);
  const int y0 = (int)fminf(fmaxf(floorf(ty - rc), 0.0f), fy), y1 = (int)fminf(fmaxf(floorf(ty + rc), 0.0f), fy);
  const int z0 = (int)fminf(fmaxf(floorf(tz - rc), 0.0f), fz), z1 = (int)fminf(fmaxf(floorf(tz + rc), 0.0f), fz);

  int y = y0, z = z0;
  while (z <= z1) {
    int nseg = 0;
    // phase 1: collect up to PG_SEGS surviving rows
    while (nseg < PG_SEGS && z <= z1) {
      const float ez = fmaxf(cell_gap(tz, z, g.nz) - margin, 0.0f);
      const float ey = fmaxf(cell_gap(ty, y, g.ny) - margin, 0.0f);
      const float eyz = ez * ez + ey * ey;
      if (!(eyz * cell2 > lim) && !(own_done && y == cy && z == cz)) {
        // x extent of the ball inside this row
        const float rem = fmaxf(lim * inv_cell2 - eyz, 0.0f);
        const float rx = sqrtf(rem) * 1.000001f * g.xr + margin_x + margin_x;   // sqrt(rem) is in y/z cells
        const int xa = max(x0, (int)fminf(fmaxf(floorf(tx - rx), 0.0f), fx));
        const int xb = min(x1, (int)fminf(fmaxf(floorf(tx + rx), 0.0f), fx));
        const uint32_t* row = start + (size_t)z * slab + (size_t)y * rowlen;
        const uint32_t s = __ldg(row + xa), e = __ldg(row + xb + 1);
        if (e > s) { seg[nseg * STRIDE] = make_uint2(s, e); ++nseg; }
      }
      if (++y > y1) { y = y0; ++z; }
    }
    // phase 2: every collected candidate in one flat loop
    pg_flat_scan<UNROLL, STRIDE>(pts, seg, nseg, qx, qy, qz, b);
    lim = fminf(b.d2, gate);
  }
}

}  // namespace mvr
