// common.cuh -- pinned arithmetic and grid geometry shared by every kernel of the ICP path.
//
// The arithmetic below is the device half of the determinism spec (SURVEY.md App. B): the CPU oracle
// evaluates exactly the same IEEE float32 expressions (built with -ffp-contract=off), so Morton keys,
// nearest-neighbour indices and squared distances are comparable bit for bit.  The _rn intrinsics are
// never contracted into FMAs by nvcc.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mvr {

// Uniform grid: cell_a = clamp(floor((p_a - o_a) * inv_cell), 0, G-1), G = 1 << bits.
// cell_lo is a float strictly below the true cell edge 1/inv_cell (used only for conservative bounds).
struct GridDev {
  float ox, oy, oz;
  float inv_cell;
  float cell_lo;
  int bits;
  int G;
};

// Row-major uniform grid of the per-align index (pair_index.cu): nx x ny x nz cells, x fastest,
// cell_a = clamp(floor((p_a - o_a) * inv_cell), 0, n_a - 1).
// Cells may be FINER along x (xr cells per y/z cell edge, xr = 1, 2, 4 or 8): the points of a (y, z) row are one contiguous run
// whatever the x resolution, so a finer x only narrows the run a ball query reads -- the same two table loads per row, fewer
// candidates (the fused ICP iteration uses xr = PG_XRATIO of api.cu; every other user of the grid builds it with xr = 1).
struct PairGrid {
  float ox, oy, oz;
  float inv_cell;     // y and z: cells per unit length
  float cell_lo;      // a float strictly below the true y/z cell edge
  int nx, ny, nz;
  float inv_cell_x;   // x: cells per unit length = inv_cell * xr (exact: xr is a power of two)
  float xr;
};

struct Mat4f { float m[16]; };  // column-major

#define MVR_INF __int_as_float(0x7f800000)

__device__ __forceinline__ float d2_pinned(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// x' = ((m00*x + m01*y) + m02*z) + m03, float32, no FMA (ICP's in-place transformCloud, SURVEY.md A10).
__device__ __forceinline__ float4 xform_pinned(const Mat4f& M, float4 p) {
  float4 r;
  r.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M.m[0], p.x), __fmul_rn(M.m[4], p.y)), __fmul_rn(M.m[8], p.z)), M.m[12]);
  r.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M.m[1], p.x), __fmul_rn(M.m[5], p.y)), __fmul_rn(M.m[9], p.z)), M.m[13]);
  r.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M.m[2], p.x), __fmul_rn(M.m[6], p.y)), __fmul_rn(M.m[10], p.z)), M.m[14]);
  r.w = 1.0f;
  return r;
}

// The same without the translation term, for a normal {nx, ny, nz, curvature}: the curvature lane is carried unchanged
// (transformPointCloudWithNormals).
__device__ __forceinline__ float4 rotate_pinned(const Mat4f& M, float4 n) {
  float4 r;
  r.x = __fadd_rn(__fadd_rn(__fmul_rn(M.m[0], n.x), __fmul_rn(M.m[4], n.y)), __fmul_rn(M.m[8], n.z));
  r.y = __fadd_rn(__fadd_rn(__fmul_rn(M.m[1], n.x), __fmul_rn(M.m[5], n.y)), __fmul_rn(M.m[9], n.z));
  r.z = __fadd_rn(__fadd_rn(__fmul_rn(M.m[2], n.x), __fmul_rn(M.m[6], n.y)), __fmul_rn(M.m[10], n.z));
  r.w = n.w;
  return r;
}

__device__ __forceinline__ bool finite3(float4 p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

__host__ __device__ __forceinline__ uint32_t part1by2(uint32_t v) {
  v &= 0x3ffu;
  v = (v | (v << 16)) & 0x030000ffu;
  v = (v | (v << 8)) & 0x0300f00fu;
  v = (v | (v << 4)) & 0x030c30c3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}

__host__ __device__ __forceinline__ uint32_t morton3(uint32_t x, uint32_t y, uint32_t z) {
  return part1by2(x) | (part1by2(y) << 1) | (part1by2(z) << 2);
}

// scaled coordinate t = (p - o) * inv_cell in pinned float arithmetic
__device__ __forceinline__ float grid_t(float p, float o, float inv) { return __fmul_rn(__fsub_rn(p, o), inv); }

__device__ __forceinline__ int grid_cell(float t, int G) {
  float f = fminf(fmaxf(floorf(t), 0.0f), (float)(G - 1));
  return (int)f;
}

__device__ __forceinline__ uint32_t point_key(float4 p, const GridDev& g) {
  if (!finite3(p)) return 1u << (3 * g.bits);
  int cx = grid_cell(grid_t(p.x, g.ox, g.inv_cell), g.G);
  int cy = grid_cell(grid_t(p.y, g.oy, g.inv_cell), g.G);
  int cz = grid_cell(grid_t(p.z, g.oz, g.inv_cell), g.G);
  return morton3((uint32_t)cx, (uint32_t)cy, (uint32_t)cz);
}

__device__ __forceinline__ bool lex_less(float d2, int idx, float bd2, int bidx) {
  return d2 < bd2 || (d2 == bd2 && idx < bidx);
}

// Safety margin, in cells, that absorbs the rounding of grid_t on both the query and the indexed
// point (each |error| <= 2^-23 * 1024 cells ~ 1.3e-4): bounds derived from cell geometry are shrunk
// by this much before they are trusted.
#define MVR_CELL_MARGIN 1.0e-3f
#define MVR_REL_SHRINK 0.999999f

}  // namespace mvr
