// api.cu -- context, host-side ICP loop and the extern "C" boundary declared in include/mvr_b200.h.
//
// Host logic mirrors pcl::IterativeClosestPoint::computeTransformation + DefaultConvergenceCriteria
// as configured by the reference (mvr/src/registrator.cpp:551-560, 768-771, 901-904; SURVEY.md A3, A8):
// the correspondence search, rejection and estimator sums run in CUDA kernels, the 3x3 SVD / 6x6
// Cholesky solve and the convergence test run here on 18-29 doubles per iteration.
// There is no CPU fallback for any device stage.
#include <cfloat>
#include <chrono>
#include <cstdlib>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/mvr_b200.h"
#include "launch.h"
#include "small_solve.h"

// x cells per y/z cell edge of the per-align indices of the fused ICP iteration (pair_search.cuh); measured in DESIGN.md section 7
#ifndef MVR_PG_XRATIO
#define MVR_PG_XRATIO 4
#endif

using namespace mvr;

#include <atomic>
namespace mvr {
static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }
// host/registrator.h
int estimate_normals_batch(mvr_ctx* const* ctxs, const int* which, int count, int k, const float* viewpoints, float* const* out_nxyzc,
                           int* statuses);
}  // namespace mvr

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return (T*)p; }
};

struct Cloud {
  const float4* pts = nullptr;
  DevBuf own;
  int n = 0;
  float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
  int n_bad = 0;
  uint64_t gen = 0;
  // index: `sorted` (cell-ordered points, .w = original index) + `table` (cell starts).  Built either by
  // the counting sort of bin.cu (order inside a cell unspecified) or by the stable radix sort of
  // index.cu (mvr_index_build; `exportable`, keys/perm kept for mvr_index_export).
  bool index_valid = false;
  bool exportable = false;
  uint64_t index_gen = 0;
  mvr_grid grid{};
  GridDev gd{};
  DevBuf keys, vals, keys_alt, vals_alt, hist, counters, sorted, table;
  uint32_t* sorted_keys = nullptr;
  uint32_t* perm = nullptr;
  IndexDev dev() const {
    IndexDev ix;
    ix.pts = sorted.as<float4>(); ix.start = table.as<uint32_t>(); ix.g = gd; ix.n_valid = n - n_bad;
    return ix;
  }
  void release() {
    own.release(); keys.release(); vals.release(); keys_alt.release(); vals_alt.release(); hist.release();
    counters.release(); sorted.release(); table.release();
  }
};

struct ProfRec { int kind; cudaEvent_t a, b; double bytes, units; int count; };

// Per-align row-major index of one cloud (pair_index.cu).
struct PairIndex {
  DevBuf sorted, start, s0;   // points by cell (the source's move in place), cell table, source binning-time copy
  DevBuf gocc, gmask;         // gate mask of a target index (pair_index.cu) and its undilated occupancy words
  float gm_gate = -1.f;       // the gate (float d2, rounded up) the mask was built for; < 0: none
  int gm_stride = 0;
  PairGrid g{};
  uint32_t cells = 0;
  int n_valid = 0;
  uint64_t gen = 0;
  bool valid = false;
  void release() { sorted.release(); start.release(); s0.release(); gocc.release(); gmask.release(); gm_gate = -1.f; valid = false; }
};

}  // namespace

struct mvr_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  Cloud tgt, src;
  // normals {nx, ny, nz, curvature} by original point index: tnrm / snrm point at the context's own buffer (normals / snormals)
  // or at another context's (mvr_normals_share); null: none.  A new cloud drops its normals.
  DevBuf normals, snormals;
  const float4* tnrm = nullptr;
  const float4* snrm = nullptr;
  DevBuf nsrc;                   // symmetric aligns: the source normals by sorted position, moved with the source
  Mat4f guess_m{};               // the guess of the prepared align (turns the source normals at its start)
  DevBuf cur, corr_p, corr_j, corr_d2, rmin, rnn, partials, sums, out_cloud, qtmp, itmp, ftmp, scratch, misc, tiles, state, log;
  PairIndex pt, ps;              // target / source index of the running align
  PairIndex nt, nq;              // target / query index of the dense NN pass (cell_nn.cu)
  double nn_ppc = 8.0;           // its target points per occupied cell
  double nn_dense_ratio = 8.0;   // kept for mvr_ctx_set_nn_options (unused: batches above nn_sorted_from are sorted and seeded)
  int nn_mode = MVR_NN_AUTO;     // mvr_ctx_set_nn_mode
  int nn_sorted_from = 262144;   // AUTO: batches larger than this are sorted by cell and answered by the seeded pass
  bool gate_mask = false;        // mvr_ctx_set_gate_mask
  FwdArgs fa{}; RevArgs ra{};    // kernel arguments of the prepared align
  bool want_rnn = false;         // the next prepared align also records the mutual partners (mvr_correspondences)
  int group_pairs = 0;           // pairs per launch of a batch led by this context (mvr_ctx_set_batch_group); 0 = automatic
  // build scratch of the per-align indices (keys, arrival ranks, arrival-order records, cell counters, scan tiles): two sets,
  // so that the target and the source index of an align can be built by the same batched launches
  struct BuildScratch { DevBuf keys, vals, moved, count, tiles; uint32_t epoch = 1; } bs[2];
  // batched aligns led by this context: the pairs' IcpStates travel together (one copy each way)
  DevBuf stage_dev;
  IcpState* h_stage = nullptr;   // pinned, stage_cap records
  int stage_cap = 0;
  DevBuf bbox_dev;               // 7 words per cloud of a batched mvr_set_clouds_device
  uint32_t* h_bbox = nullptr;    // pinned, BBOX_MAX_JOBS * 7 words
  int log_pending = 0;           // records of the device log not fetched yet (mvr_icp_get_iterations fetches them)
  bool out_pending = false;      // out_cloud has not been computed yet (materialize_out)
  DevBuf crowded;                        // one word: population of the most crowded cell an index build could not rank (0: none)
  uint32_t crowded_seen = 0;             // its value after the last align
  IcpState* h_state = nullptr;   // pinned staging copy of the device IcpState
  IterRec* h_log = nullptr;      // pinned, ICP_MAX_LOG records
  double* h_sums = nullptr;      // pinned, REDUCE_MAX_VALS
  uint32_t* h_small = nullptr;   // pinned, 16 words
  std::string err;
  bool profiling = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  mvr_kernel_stat stats[MVR_K_COUNT] = {};
  std::vector<mvr_icp_iteration> iters;
  bool have_out = false;         // out_cloud holds transform(source, final) of the last align
  float cell_edge_opt = 0.f;
  int max_bits_opt = 8;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
};

namespace {

#define CK(expr)                                                                                 \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      ctx->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                             \
      return MVR_ERR_CUDA;                                                                       \
    }                                                                                            \
  } while (0)

int fail(mvr_ctx* ctx, int code, const char* msg) {
  if (ctx) ctx->err = msg;
  return code;
}

cudaEvent_t get_event(mvr_ctx* ctx) {
  if (!ctx->ev_pool.empty()) { cudaEvent_t e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

struct ProfScope {
  mvr_ctx* ctx; int idx;
  // count: launches (of the kernel family) the scope brackets -- the iterations of an align share ONE pair of events, so the
  // measurement puts nothing between them
  cudaStream_t st;
  ProfScope(mvr_ctx* c, int kind, double bytes, double units, int count = 1, cudaStream_t stream = nullptr) : ctx(c), idx(-1), st(stream ? stream : c->stream) {
    if (!c->profiling) return;
    ProfRec r{kind, get_event(c), get_event(c), bytes, units, count};
    cudaEventRecord(r.a, st);
    c->prof.push_back(r);
    idx = (int)c->prof.size() - 1;
  }
  ~ProfScope() { if (idx >= 0) cudaEventRecord(ctx->prof[idx].b, st); }
};

void prof_flush(mvr_ctx* ctx) {
  for (ProfRec& r : ctx->prof) {
    cudaEventSynchronize(r.b);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      mvr_kernel_stat& s = ctx->stats[r.kind];
      s.launches += (uint64_t)r.count; s.ms += ms; s.bytes += r.bytes; s.units += r.units;
    }
    ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b);
  }
  ctx->prof.clear();
}

// ---- grid selection ---------------------------------------------------------------------------
// Surface-density heuristic: a scan is a 2-manifold, so the number of occupied cells of edge e is
// about 1.5 * area / e^2 with area ~ half the bounding-box surface; solve for `ppc` points per cell.
double density_cell_edge(const float lo[3], const float hi[3], int n, double ppc) {
  double ex = std::max(0.0, (double)hi[0] - lo[0]), ey = std::max(0.0, (double)hi[1] - lo[1]), ez = std::max(0.0, (double)hi[2] - lo[2]);
  double area = ex * ey + ey * ez + ex * ez;  // = 0.5 * box surface
  double ext = std::max(ex, std::max(ey, ez));
  if (n <= 0 || ext <= 0) return 1.0;
  if (area <= 0) return ext / std::min(1024.0, std::max(1.0, (double)n / ppc));
  return std::sqrt(1.5 * ppc * area / (double)n);
}

mvr_grid make_grid(const float lo[3], const float hi[3], double cell, int max_bits) {
  mvr_grid g{};
  double ext = 0;
  for (int a = 0; a < 3; ++a) ext = std::max(ext, (double)hi[a] - (double)lo[a]);
  if (!(ext > 0) || !std::isfinite(ext)) ext = 1.0;
  if (!(cell > 0) || !std::isfinite(cell)) cell = ext;
  if (max_bits > 10) max_bits = 10;
  if (max_bits < 1) max_bits = 1;
  int bits = std::min(3, max_bits);
  while (bits < max_bits && cell * (double)(1 << bits) < ext * 1.0001) ++bits;
  if (cell * (double)(1 << bits) < ext * 1.0001) cell = ext * 1.0001 / (double)(1 << bits);
  for (int a = 0; a < 3; ++a) g.origin[a] = lo[a];
  g.inv_cell = (float)(1.0 / cell);
  g.cell = (float)cell;
  g.bits = bits;
  return g;
}

GridDev to_dev(const mvr_grid& g) {
  GridDev d;
  d.ox = g.origin[0]; d.oy = g.origin[1]; d.oz = g.origin[2];
  d.inv_cell = g.inv_cell;
  double c = (1.0 / (double)g.inv_cell) * (1.0 - 1e-6);
  d.cell_lo = std::nextafterf((float)c, 0.0f);
  d.bits = g.bits;
  d.G = 1 << g.bits;
  return d;
}

bool same_grid(const mvr_grid& a, const mvr_grid& b) {
  return std::memcmp(a.origin, b.origin, sizeof(a.origin)) == 0 && a.inv_cell == b.inv_cell && a.bits == b.bits;
}

// ---- clouds -----------------------------------------------------------------------------------
int cloud_bbox(mvr_ctx* ctx, Cloud& c) {
  for (int a = 0; a < 3; ++a) { c.lo[a] = 0; c.hi[a] = 0; }
  c.n_bad = 0;
  if (c.n <= 0) return MVR_OK;
  CK(ctx->misc.ensure(64));
  uint32_t* d = ctx->misc.as<uint32_t>();
  CK(launch_bbox_init(d, ctx->stream));
  CK(launch_bbox(c.pts, c.n, d, ctx->stream));
  CK(cudaMemcpyAsync(ctx->h_small, d, 7 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  c.n_bad = (int)ctx->h_small[6];
  if (c.n_bad < c.n)
    for (int a = 0; a < 3; ++a) { c.lo[a] = bbox_decode(ctx->h_small[a]); c.hi[a] = bbox_decode(ctx->h_small[3 + a]); }
  return MVR_OK;
}

int cloud_set(mvr_ctx* ctx, Cloud& c, const float* xyzw, size_t n, bool device_ptr) {
  if (n > (size_t)INT_MAX / 2) return fail(ctx, MVR_ERR_BAD_ARG, "cloud too large");
  if (n > 0 && !xyzw) return fail(ctx, MVR_ERR_BAD_ARG, "null point pointer");
  c.index_valid = false;
  c.gen++;
  c.n = (int)n;
  if (device_ptr) {
    c.pts = (const float4*)xyzw;
  } else {
    CK(c.own.ensure(std::max<size_t>(n, 1) * sizeof(float4)));
    if (n) CK(cudaMemcpyAsync(c.own.p, xyzw, n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    c.pts = c.own.as<float4>();
  }
  return cloud_bbox(ctx, c);
}

// Build the Morton-sorted grid index of `pts` (n points of cloud c) with grid g.
int build_index(mvr_ctx* ctx, Cloud& c, const float4* pts, const mvr_grid& g) {
  const int n = c.n;
  const size_t cells = (size_t)1 << (3 * g.bits);
  CK(c.keys.ensure(std::max(n, 1) * sizeof(uint32_t)));
  CK(c.vals.ensure(std::max(n, 1) * sizeof(uint32_t)));
  CK(c.keys_alt.ensure(std::max(n, 1) * sizeof(uint32_t)));
  CK(c.vals_alt.ensure(std::max(n, 1) * sizeof(uint32_t)));
  CK(c.hist.ensure((size_t)256 * radix_num_blocks(n) * sizeof(uint32_t)));
  CK(c.sorted.ensure(std::max(n, 1) * sizeof(float4)));
  CK(c.table.ensure((cells + 2) * sizeof(uint32_t)));
  c.grid = g;
  c.gd = to_dev(g);
  {
    ProfScope ps(ctx, MVR_K_MORTON, 24.0 * n, n);
    CK(launch_morton_keys(pts, n, c.gd, c.keys.as<uint32_t>(), c.vals.as<uint32_t>(), ctx->stream));
  }
  int key_bits = 3 * g.bits + (c.n_bad > 0 ? 1 : 0);
  SortScratch sc{c.keys_alt.as<uint32_t>(), c.vals_alt.as<uint32_t>(), c.hist.as<uint32_t>()};
  {
    ProfScope ps(ctx, MVR_K_SORT, 16.0 * n, n);
    CK(launch_radix_sort(c.keys.as<uint32_t>(), c.vals.as<uint32_t>(), n, key_bits, sc, &c.sorted_keys, &c.perm, ctx->stream));
  }
  {
    ProfScope ps(ctx, MVR_K_TABLE, 36.0 * n + 4.0 * (double)cells, n);
    CK(launch_gather_sorted(pts, c.perm, n, c.sorted.as<float4>(), ctx->stream));
    CK(launch_cell_table(c.sorted_keys, n, g.bits, c.table.as<uint32_t>(), ctx->stream));
  }
  c.index_valid = true;
  c.exportable = true;
  c.index_gen = c.gen;
  return MVR_OK;
}

mvr_grid auto_grid(mvr_ctx* ctx, const Cloud& c) {
  double e = ctx->cell_edge_opt > 0 ? ctx->cell_edge_opt : density_cell_edge(c.lo, c.hi, c.n - c.n_bad, 6.0);
  return make_grid(c.lo, c.hi, e, ctx->max_bits_opt);
}

PairGrid make_pair_grid(const float lo[3], const float hi[3], double e, uint32_t* cells_out, int xr = 1);
bool same_pair_grid(const PairGrid& a, const PairGrid& b);
int build_pair_index(mvr_ctx* ctx, PairIndex& ix, const float4* pts, int n, int n_bad, const Mat4f* guess, const PairGrid& g,
                     uint32_t cells, bool keep_s0, bool ordered = true);
int plan_pair_index(mvr_ctx* ctx, PairIndex& ix, int slot, const float4* pts, int n, int n_bad, const Mat4f* guess, const PairGrid& g,
                    uint32_t cells, bool ordered, cudaStream_t stream, BuildJob* job);
int run_pair_builds(mvr_ctx* ctx, const BuildJob* jobs, int count, cudaStream_t stream);

double pair_cell_edge(mvr_ctx* ctx, const Cloud& c, double max_dist);

// Many queries per target point: target and queries counting-sorted by the cells of one row-major grid, then the
// warp-cooperative scan of cell_nn.cu.
int nn_pass_dense(mvr_ctx* ctx, const float4* q, int n, int32_t* d_idx, float* d_d2, bool seeded) {
  Cloud& t = ctx->tgt;
  const int mv = t.n - t.n_bad;
  const double e = ctx->cell_edge_opt > 0 ? ctx->cell_edge_opt : density_cell_edge(t.lo, t.hi, mv, ctx->nn_ppc);
  uint32_t cells = 0;
  const PairGrid g = make_pair_grid(t.lo, t.hi, e, &cells);
  int rc;
  if (!(ctx->nt.valid && ctx->nt.gen == t.gen && same_pair_grid(ctx->nt.g, g))) {
    if ((rc = build_pair_index(ctx, ctx->nt, t.pts, t.n, t.n_bad, nullptr, g, cells, false))) return rc;
    ctx->nt.gen = t.gen;
  }
  if ((rc = build_pair_index(ctx, ctx->nq, q, n, 0, nullptr, g, cells, false, false))) return rc;
  ProfScope ps(ctx, MVR_K_NN, 24.0 * n + 16.0 * t.n, (double)n);
  if (seeded)
    CK(launch_seeded_nn(ctx->nq.sorted.as<float4>(), n, ctx->nq.start.as<uint32_t>() + cells, ctx->nt.sorted.as<float4>(),
                        ctx->nt.start.as<uint32_t>(), g, mv, d_idx, d_d2, ctx->stream));
  else
    CK(launch_cell_nn(ctx->nq.sorted.as<float4>(), n, ctx->nq.start.as<uint32_t>() + cells, ctx->nt.sorted.as<float4>(),
                      ctx->nt.start.as<uint32_t>(), g, mv, d_idx, d_d2, ctx->stream));
  return MVR_OK;
}

// Exact un-gated NN of n device points in the target index; results at the queries' original index.
int nn_pass(mvr_ctx* ctx, const float4* q, int n, int32_t* d_idx, float* d_d2) {
  // queries sorted by the cells of the target's grid, then either every query seeded from its own cell (SEEDED; AUTO from
  // nn_sorted_from queries on) or the cell-cooperative scan of whole neighbourhoods (CELL)
  if (ctx->nn_mode == MVR_NN_CELL) return nn_pass_dense(ctx, q, n, d_idx, d_d2, false);
  if (ctx->nn_mode == MVR_NN_SEEDED || (ctx->nn_mode == MVR_NN_AUTO && n > ctx->nn_sorted_from)) return nn_pass_dense(ctx, q, n, d_idx, d_d2, true);
  // The row walk of pair_search.cuh on the target's per-align index: small batches as they come, large ones sorted by
  // cell first (locality).  It also gets through the empty space around far queries quickly, which a cell-by-cell ring
  // expansion does not.
  Cloud& t = ctx->tgt;
  PairIndex& pt = ctx->pt;
  int rc;
  if (!(pt.valid && pt.gen == t.gen && pt.g.xr == 1.0f)) {   // the NN kernels take isotropic cells
    uint32_t cells = 0;
    const PairGrid gt = make_pair_grid(t.lo, t.hi, pair_cell_edge(ctx, t, INFINITY), &cells);
    if ((rc = build_pair_index(ctx, pt, t.pts, t.n, t.n_bad, nullptr, gt, cells, false))) return rc;
    pt.gen = t.gen;
  }
  ProfScope ps(ctx, MVR_K_NN, 24.0 * n + 16.0 * t.n, (double)n);
  // Measured on B200 (1M-point target; profiles/r02_nn_kernels.log): one warp per query answers 10k queries in 20 us against 87 us
  // for the per-thread walk and wins up to ~130k queries; above that its 32 lanes per query cap it at 2 G queries/s and the
  // per-thread walk (queries sorted by cell from 256k on) takes over, until the cell-cooperative pass wins at >= 8 queries per
  // target point.
  if (ctx->nn_mode == MVR_NN_WARP || (ctx->nn_mode == MVR_NN_AUTO && n <= 131072)) {
    // one warp per query, queries as they come (cell_nn.cu): no serial chain of dependent loads per query
    CK(launch_warp_nn(q, n, pt.sorted.as<float4>(), pt.start.as<uint32_t>(), pt.g, pt.n_valid, d_idx, d_d2, ctx->stream));
    return MVR_OK;
  }
  const bool sorted = n > 262144;
  if (sorted && (rc = build_pair_index(ctx, ctx->nq, q, n, 0, nullptr, pt.g, pt.cells, false, false))) return rc;
  CK(launch_pair_nn(sorted ? ctx->nq.sorted.as<float4>() : q, n, sorted, pt.sorted.as<float4>(), pt.start.as<uint32_t>(), pt.g, pt.n_valid, d_idx,
                    d_d2, ctx->stream));
  return MVR_OK;
}

void mat_identity(float* m) { for (int k = 0; k < 16; ++k) m[k] = (k % 5 == 0) ? 1.f : 0.f; }

float gate_float(double max_dist) {
  double m2 = max_dist * max_dist;
  if (!(m2 < (double)FLT_MAX)) return INFINITY;
  float f = (float)m2;
  if ((double)f < m2) f = std::nextafterf(f, INFINITY);
  return std::nextafterf(f, INFINITY);
}

// ---- per-align row-major index (pair_index.cu) ---------------------------------------------------
// Cell edge of a cloud's pair grid: gate / 2 when the point density allows (a settled alignment then
// looks at 1-2 cells per axis), otherwise bounded to 2 .. 12 points per occupied cell.
double pair_cell_edge(mvr_ctx* ctx, const Cloud& c, double max_dist) {
  if (ctx->cell_edge_opt > 0) return ctx->cell_edge_opt;
  const int nv = c.n - c.n_bad;
  const double e_lo = density_cell_edge(c.lo, c.hi, nv, 2.0), e_hi = density_cell_edge(c.lo, c.hi, nv, 12.0);
  const double m2 = max_dist * max_dist;
  return (m2 < 1e30) ? std::min(std::max(0.5 * max_dist * 1.002, e_lo), e_hi) : density_cell_edge(c.lo, c.hi, nv, 6.0);
}

// Grid over the box [lo, hi] padded by one cell; the edge grows until the table fits max_cells.  xr (1, 2, 4 or 8): x cells
// per y/z cell edge.
PairGrid make_pair_grid(const float lo[3], const float hi[3], double e, uint32_t* cells_out, int xr) {
  const double max_cells = 16.0 * 1024 * 1024;
  if (xr != 1 && xr != 2 && xr != 4 && xr != 8) xr = 1;
  double ext[3];
  for (int a = 0; a < 3; ++a) {
    ext[a] = (double)hi[a] - (double)lo[a];
    if (!(ext[a] >= 0) || !std::isfinite(ext[a])) ext[a] = 0;
  }
  if (!(e > 0) || !std::isfinite(e)) e = std::max(1e-3, std::max(ext[0], std::max(ext[1], ext[2])));
  int n[3];
  for (;;) {
    double tot = 1;
    for (int a = 0; a < 3; ++a) {
      const int r = a == 0 ? xr : 1;
      n[a] = (int)std::min(4096.0 * r, std::floor(ext[a] / (e / r)) + 3.0 * r);
      tot *= n[a];
    }
    if (tot <= max_cells) break;
    if (xr > 1) { xr /= 2; continue; }   // a coarser x first, then larger cells
    e *= 1.25;
  }
  PairGrid g;
  g.ox = lo[0] - (float)e; g.oy = lo[1] - (float)e; g.oz = lo[2] - (float)e;
  if (!std::isfinite(g.ox)) g.ox = 0.f;
  if (!std::isfinite(g.oy)) g.oy = 0.f;
  if (!std::isfinite(g.oz)) g.oz = 0.f;
  g.inv_cell = (float)(1.0 / e);
  g.cell_lo = std::nextafterf((float)((1.0 / (double)g.inv_cell) * (1.0 - 1e-6)), 0.0f);
  g.nx = n[0]; g.ny = n[1]; g.nz = n[2];
  g.xr = (float)xr;
  g.inv_cell_x = g.inv_cell * g.xr;
  *cells_out = (uint32_t)n[0] * (uint32_t)n[1] * (uint32_t)n[2];
  return g;
}

bool same_pair_grid(const PairGrid& a, const PairGrid& b) { return std::memcmp(&a, &b, sizeof(PairGrid)) == 0; }

// Plan the index of `n` points (n_bad of them non-finite) in grid g: buffers of ix and of scratch set `slot` (0 or 1) are
// made ready (first-time zeroing on `stream`, the stream the build will run on) and the build is described in *job.
// guess (nullable) is applied first (pinned float transform).  ordered = false leaves the points of a cell in arrival order
// (queries: their results go out by original index).
int plan_pair_index(mvr_ctx* ctx, PairIndex& ix, int slot, const float4* pts, int n, int n_bad, const Mat4f* guess, const PairGrid& g,
                    uint32_t cells, bool ordered, cudaStream_t stream, BuildJob* job) {
  mvr_ctx::BuildScratch& bs = ctx->bs[slot];
  const size_t nn = (size_t)std::max(n, 1);
  CK(bs.keys.ensure(nn * sizeof(uint32_t)));
  CK(bs.vals.ensure(nn * sizeof(uint32_t)));
  if (ordered) CK(bs.moved.ensure(nn * sizeof(float4)));
  CK(ix.sorted.ensure(nn * sizeof(float4)));
  CK(ix.start.ensure(((size_t)cells + 2) * sizeof(uint32_t)));
  if (((size_t)cells + 1) * sizeof(uint32_t) > bs.count.cap) {
    CK(bs.count.ensure(((size_t)cells + 1) * sizeof(uint32_t)));
    CK(cudaMemsetAsync(bs.count.p, 0, bs.count.cap, stream));   // the scan keeps the counters zero afterwards
  }
  const int ntiles = scan_num_tiles((size_t)cells + 1);
  const size_t tiles = (size_t)ntiles + 1;   // + the ticket word
  if (tiles * sizeof(unsigned long long) > bs.tiles.cap) {
    CK(bs.tiles.ensure(tiles * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(bs.tiles.p, 0, bs.tiles.cap, stream));
  }
  if (!ctx->crowded.p) { CK(ctx->crowded.ensure(64)); CK(cudaMemsetAsync(ctx->crowded.p, 0, 64, stream)); }
  BuildJob& j = *job;
  j = BuildJob{};
  j.in = pts; j.n = n; j.apply = guess ? 1 : 0;
  if (guess) j.M = *guess;
  j.g = g; j.cells = cells;
  j.keys = bs.keys.as<uint32_t>(); j.rank = bs.vals.as<uint32_t>(); j.counters = bs.count.as<uint32_t>();
  j.tiles = bs.tiles.as<unsigned long long>(); j.epoch = bs.epoch; j.ntiles = ntiles;
  bs.epoch = (bs.epoch % 0x3fffffffu) + 1;
  j.tmp = ordered ? bs.moved.as<float4>() : nullptr; j.sorted = ix.sorted.as<float4>(); j.start = ix.start.as<uint32_t>();
  j.crowded = ctx->crowded.as<uint32_t>(); j.ordered = ordered ? 1 : 0;
  ix.g = g; ix.cells = cells; ix.n_valid = n - n_bad; ix.valid = true; ix.gm_gate = -1.f;
  return MVR_OK;
}

// The planned builds, four launches per BUILD_MAX_JOBS of them (pair_index.cu); ctx: where errors and the profile go.
int run_pair_builds(mvr_ctx* ctx, const BuildJob* jobs, int count, cudaStream_t stream) {
  for (int k0 = 0; k0 < count; k0 += BUILD_MAX_JOBS) {
    const int c = std::min(count - k0, (int)BUILD_MAX_JOBS);
    BuildBatch batch;
    double bytes = 0, pts = 0;
    for (int k = 0; k < c; ++k) { batch.j[k] = jobs[k0 + k]; bytes += 32.0 * jobs[k0 + k].n + 8.0 * jobs[k0 + k].cells; pts += jobs[k0 + k].n; }
    ProfScope ps(ctx, MVR_K_SORT, bytes, pts, 1, stream);
    CK(launch_pair_builds(batch, c, stream));
  }
  return MVR_OK;
}

int build_pair_index(mvr_ctx* ctx, PairIndex& ix, const float4* pts, int n, int n_bad, const Mat4f* guess, const PairGrid& g,
                     uint32_t cells, bool keep_s0, bool ordered) {
  (void)keep_s0;
  BuildJob job;
  ix.valid = false;
  int rc = plan_pair_index(ctx, ix, &ix == &ctx->pt || &ix == &ctx->nt ? 0 : 1, pts, n, n_bad, guess, g, cells, ordered, ctx->stream, &job);
  if (rc) { ix.valid = false; return rc; }
  return run_pair_builds(ctx, &job, 1, ctx->stream);
}

// The gate mask of target index ix for gate max_d2f (float d2, rounded up); without one (no gate, or a gate many cells
// wide) the forward half searches every point.  Cells more than D apart in an axis are >= D cells apart along it; the
// rounding of grid_t on the query and on the target point is absorbed by `slack` cells.
int ensure_gate_mask(mvr_ctx* ctx, PairIndex& ix, float max_d2f, cudaStream_t stream) {
  // Off unless asked for (mvr_ctx_set_gate_mask): on the bench workload (neighbouring views of a 24-view turntable, ~4 % of the
  // source points beyond the gate) the mask saves 0.03 ms over 22 iterations and costs 0.2 ms to build for 24 targets
  // (profiles/r02_iteration_ab.log); it pays when a large part of the source has no partner (little overlap).
  if (!ctx->gate_mask || !(max_d2f < 3.0e38f) || ix.n_valid <= 0) { ix.gm_gate = -1.f; return MVR_OK; }
  if (ix.gm_gate == max_d2f) return MVR_OK;
  const double slack = 2.0 * ((double)MVR_CELL_MARGIN + 1.0e-6 * (double)std::max(ix.g.nx, std::max(ix.g.ny, ix.g.nz)));
  const double need = std::sqrt((double)max_d2f) * (1.0 + 1.0e-5) / (double)ix.g.cell_lo + slack;
  const int D = (int)std::ceil(need);
  const int Dx = (int)std::ceil(need * (double)ix.g.xr);
  ix.gm_gate = -1.f;
  if (D < 1 || D > 6 || Dx > 31) return MVR_OK;
  const int wstride = (ix.g.nx + 31) / 32;
  const size_t words = (size_t)ix.g.ny * ix.g.nz * wstride;
  CK(ix.gocc.ensure(words * sizeof(uint32_t)));
  CK(ix.gmask.ensure(words * sizeof(uint32_t)));
  CK(launch_gate_mask(ix.start.as<uint32_t>(), ix.g, wstride, D, Dx, ix.gocc.as<uint32_t>(), ix.gmask.as<uint32_t>(), stream));
  ix.gm_stride = wstride;
  ix.gm_gate = max_d2f;
  return MVR_OK;
}

int ensure_pinned(mvr_ctx* ctx) {
  if (!ctx->h_sums) CK(cudaMallocHost((void**)&ctx->h_sums, REDUCE_MAX_VALS * sizeof(double)));
  if (!ctx->h_small) CK(cudaMallocHost((void**)&ctx->h_small, 64 * sizeof(uint32_t)));
  if (!ctx->h_state) CK(cudaMallocHost((void**)&ctx->h_state, sizeof(IcpState)));
  if (!ctx->h_log) CK(cudaMallocHost((void**)&ctx->h_log, ICP_MAX_LOG * sizeof(IterRec)));
  return MVR_OK;
}

// fn(k) for k in [0, n) on up to MVR_HOST_THREADS (environment, default 6) host threads; the calling thread takes part.
template <class F>
void parallel_for(int n, F fn) {
  static const int max_threads = [] { const char* e = std::getenv("MVR_HOST_THREADS"); const int v = e ? std::atoi(e) : 6; return v < 1 ? 1 : (v > 64 ? 64 : v); }();
  const int nt = std::min(max_threads, n);
  if (nt <= 1) { for (int k = 0; k < n; ++k) fn(k); return; }
  std::atomic<int> next{0};
  auto work = [&] { for (int k = next.fetch_add(1); k < n; k = next.fetch_add(1)) fn(k); };
  std::vector<std::thread> th;
  for (int t = 1; t < nt; ++t) th.emplace_back(work);
  work();
  for (std::thread& t : th) t.join();
}

// Grid of the index mvr_estimate_normals builds over cloud c: the cell edge is ~1.25 x the expected distance of the k-th
// neighbour on a surface of the cloud's density, so the 27 cells around a point hold its k neighbours and prove it (the k-th
// distance is below one cell) for nearly every point.
PairGrid normals_grid(const mvr_ctx* ctx, const Cloud& c, int k, uint32_t* cells) {
  const double e = ctx->cell_edge_opt > 0 ? ctx->cell_edge_opt : density_cell_edge(c.lo, c.hi, c.n - c.n_bad, std::max(2.0, k / 3.0));
  return make_pair_grid(c.lo, c.hi, e, cells);
}

// The normals of the n points indexed by ix: viewpoint NULL = the origin.
NormalsJob normals_job(const PairIndex& ix, int n, const float* viewpoint, float4* out, int32_t* nbr) {
  NormalsJob j{};
  j.sorted = ix.sorted.as<float4>(); j.start = ix.start.as<uint32_t>(); j.g = ix.g;
  j.n = n; j.n_valid = ix.n_valid;
  j.viewpoint = viewpoint ? make_float3(viewpoint[0], viewpoint[1], viewpoint[2]) : make_float3(0.f, 0.f, 0.f);
  j.out = out; j.nbr = nbr;
  return j;
}


}  // namespace

// =================================================================================================
extern "C" {

const char* mvr_version(void) { return "mvr_b200 0.1 (sm_100a)"; }

uint64_t mvr_kernel_launch_count(void) { return (uint64_t)launch_count(); }

void mvr_transfer_sizes(size_t* state_bytes, size_t* log_record_bytes) {
  if (state_bytes) *state_bytes = sizeof(IcpState);
  if (log_record_bytes) *log_record_bytes = sizeof(IterRec);
}

const char* mvr_status_string(int s) {
  switch (s) {
    case MVR_OK: return "ok";
    case MVR_ERR_BAD_ARG: return "bad argument";
    case MVR_ERR_TOO_FEW_CORRESPONDENCES: return "not enough correspondences";
    case MVR_ERR_CUDA: return "CUDA error";
    case MVR_ERR_NO_INPUT: return "input cloud not set";
    case MVR_ERR_NOT_SPD: return "normal equations not positive definite";
    case MVR_ERR_ALLOC: return "allocation failed";
    case MVR_ERR_NCCL: return "NCCL unavailable or a collective failed";
    default: return "unknown status";
  }
}

void mvr_icp_params_default(mvr_icp_params* p) {
  if (!p) return;
  p->max_iterations = 10;
  p->max_correspondence_distance = std::sqrt(DBL_MAX);
  p->transformation_epsilon = 0.0;
  p->euclidean_fitness_epsilon = -DBL_MAX;
  p->use_reciprocal_correspondences = 0;
  p->estimator = MVR_POINT_TO_POINT;
  p->fixed_iterations = 0;
  p->min_correspondences = 3;
}

int mvr_ctx_create(int device, mvr_ctx** out) {
  if (!out) return MVR_ERR_BAD_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return MVR_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return MVR_ERR_CUDA;
  mvr_ctx* ctx = new mvr_ctx();
  ctx->device = device;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return MVR_ERR_CUDA; }
  ctx->own_stream = true;
  cudaEventCreate(&ctx->ev_a);
  cudaEventCreate(&ctx->ev_b);
  if (ensure_pinned(ctx) != MVR_OK) { mvr_ctx_destroy(ctx); return MVR_ERR_CUDA; }
  *out = ctx;
  return MVR_OK;
}

int mvr_ctx_destroy(mvr_ctx* ctx) {
  if (!ctx) return MVR_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  prof_flush(ctx);
  for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
  if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
  if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
  ctx->tgt.release(); ctx->src.release(); ctx->normals.release(); ctx->snormals.release(); ctx->nsrc.release();
  ctx->pt.release(); ctx->ps.release(); ctx->nt.release(); ctx->nq.release();
  for (auto& b : ctx->bs) { b.keys.release(); b.vals.release(); b.moved.release(); b.count.release(); b.tiles.release(); }
  ctx->stage_dev.release(); ctx->bbox_dev.release();
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->h_bbox) cudaFreeHost(ctx->h_bbox);
  DevBuf* bufs[] = {&ctx->cur, &ctx->corr_p, &ctx->rmin, &ctx->rnn, &ctx->corr_j, &ctx->corr_d2, &ctx->partials, &ctx->sums, &ctx->out_cloud, &ctx->qtmp,
                    &ctx->itmp, &ctx->ftmp, &ctx->scratch, &ctx->misc, &ctx->tiles, &ctx->state, &ctx->log, &ctx->crowded};
  for (DevBuf* b : bufs) b->release();
  if (ctx->h_sums) cudaFreeHost(ctx->h_sums);
  if (ctx->h_small) cudaFreeHost(ctx->h_small);
  if (ctx->h_state) cudaFreeHost(ctx->h_state);
  if (ctx->h_log) cudaFreeHost(ctx->h_log);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return MVR_OK;
}

int mvr_ctx_set_stream(mvr_ctx* ctx, void* s) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)s;
  ctx->own_stream = false;
  return MVR_OK;
}

void* mvr_ctx_get_stream(mvr_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int mvr_ctx_synchronize(mvr_ctx* ctx) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

const char* mvr_last_error(mvr_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int mvr_ctx_set_profiling(mvr_ctx* ctx, int on) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  ctx->profiling = on != 0;
  return MVR_OK;
}

int mvr_ctx_get_kernel_stats(mvr_ctx* ctx, mvr_kernel_stat* out, int reset) {
  if (!ctx || !out) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaStreamSynchronize(ctx->stream));
  prof_flush(ctx);
  std::memcpy(out, ctx->stats, sizeof(ctx->stats));
  if (reset) std::memset(ctx->stats, 0, sizeof(ctx->stats));
  return MVR_OK;
}

int mvr_ctx_set_index_options(mvr_ctx* ctx, float cell_edge, int max_bits) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  if (max_bits < 1 || max_bits > 10) return fail(ctx, MVR_ERR_BAD_ARG, "max_bits must be in 1..10");
  ctx->cell_edge_opt = cell_edge > 0 ? cell_edge : 0.f;
  ctx->max_bits_opt = max_bits;
  ctx->tgt.index_valid = false;
  ctx->src.index_valid = false;
  return MVR_OK;
}

int mvr_ctx_set_nn_options(mvr_ctx* ctx, double points_per_cell, double dense_ratio) {
  if (!ctx || !(points_per_cell > 0) || !(dense_ratio >= 0)) return MVR_ERR_BAD_ARG;
  ctx->nn_ppc = points_per_cell;
  ctx->nn_dense_ratio = dense_ratio;
  ctx->nt.valid = false;
  return MVR_OK;
}

int mvr_ctx_set_gate_mask(mvr_ctx* ctx, int on) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  ctx->gate_mask = on != 0;
  ctx->pt.gm_gate = -1.f;
  return MVR_OK;
}

int mvr_ctx_set_nn_mode(mvr_ctx* ctx, int mode) {
  if (!ctx || mode < MVR_NN_AUTO || mode > MVR_NN_SEEDED) return MVR_ERR_BAD_ARG;
  ctx->nn_mode = mode;
  return MVR_OK;
}

int mvr_ctx_set_batch_group(mvr_ctx* ctx, int pairs) {
  if (!ctx || pairs < 0 || pairs > (int)FUSED_MAX_PAIRS) return MVR_ERR_BAD_ARG;
  ctx->group_pairs = pairs;
  return MVR_OK;
}

int mvr_set_target(mvr_ctx* ctx, const float* xyzw, size_t n) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  ctx->tnrm = nullptr;
  return cloud_set(ctx, ctx->tgt, xyzw, n, false);
}
int mvr_set_source(mvr_ctx* ctx, const float* xyzw, size_t n) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  ctx->have_out = false;
  ctx->snrm = nullptr;
  return cloud_set(ctx, ctx->src, xyzw, n, false);
}
int mvr_set_target_device(mvr_ctx* ctx, const float* d, size_t n) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  ctx->tnrm = nullptr;
  return cloud_set(ctx, ctx->tgt, d, n, true);
}
int mvr_set_source_device(mvr_ctx* ctx, const float* d, size_t n) {
  if (!ctx) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  ctx->have_out = false;
  ctx->snrm = nullptr;
  return cloud_set(ctx, ctx->src, d, n, true);
}

// Many clouds at once: their bounding boxes are measured by ONE launch and read back by one copy (mvr_set_*_device pays a
// stream round trip per cloud: ~25 us each, 0.6 ms for the 24 views of a turntable sequence).
int mvr_set_clouds_device(mvr_ctx* const* ctxs, const int* which, const float* const* d_xyzw, const size_t* n, int count) {
  if (count < 0 || (count && (!ctxs || !which || !d_xyzw || !n))) return MVR_ERR_BAD_ARG;
  if (count == 0) return MVR_OK;
  mvr_ctx* ctx = ctxs[0];
  if (!ctx) return MVR_ERR_BAD_ARG;
  for (int k = 0; k < count; ++k) {
    if (!ctxs[k] || (which[k] != MVR_CLOUD_TARGET && which[k] != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
    if (ctxs[k]->device != ctx->device) return fail(ctx, MVR_ERR_BAD_ARG, "the contexts of a batch must share a device");
    if (n[k] > (size_t)INT_MAX / 2) return fail(ctx, MVR_ERR_BAD_ARG, "cloud too large");
    if (n[k] > 0 && !d_xyzw[k]) return fail(ctx, MVR_ERR_BAD_ARG, "null point pointer");
  }
  cudaSetDevice(ctx->device);
  if (!ctx->h_bbox) CK(cudaMallocHost((void**)&ctx->h_bbox, (size_t)BBOX_MAX_JOBS * 7 * sizeof(uint32_t)));
  CK(ctx->bbox_dev.ensure((size_t)BBOX_MAX_JOBS * 7 * sizeof(uint32_t)));
  for (int k0 = 0; k0 < count; k0 += BBOX_MAX_JOBS) {
    const int c = std::min(count - k0, (int)BBOX_MAX_JOBS);
    BboxBatch bb;
    for (int k = 0; k < c; ++k) { bb.j[k].pts = (const float4*)d_xyzw[k0 + k]; bb.j[k].n = (int)n[k0 + k]; bb.j[k].pad_ = 0; }
    CK(launch_bbox_batch(bb, c, ctx->bbox_dev.as<uint32_t>(), ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_bbox, ctx->bbox_dev.p, (size_t)c * 7 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < c; ++k) {
      mvr_ctx* m = ctxs[k0 + k];
      Cloud& cl = which[k0 + k] == MVR_CLOUD_TARGET ? m->tgt : m->src;
      if (which[k0 + k] == MVR_CLOUD_TARGET) m->tnrm = nullptr; else { m->have_out = false; m->out_pending = false; m->snrm = nullptr; }
      cl.index_valid = false;
      cl.gen++;
      cl.n = (int)n[k0 + k];
      cl.pts = (const float4*)d_xyzw[k0 + k];
      const uint32_t* w = ctx->h_bbox + 7 * k;
      for (int a = 0; a < 3; ++a) { cl.lo[a] = 0; cl.hi[a] = 0; }
      cl.n_bad = cl.n > 0 ? (int)w[6] : 0;
      if (cl.n > 0 && cl.n_bad < cl.n)
        for (int a = 0; a < 3; ++a) { cl.lo[a] = bbox_decode(w[a]); cl.hi[a] = bbox_decode(w[3 + a]); }
    }
  }
  return MVR_OK;
}

int mvr_cloud_share(mvr_ctx* dst, int which_dst, mvr_ctx* src, int which_src) {
  if (!dst || !src || (which_dst != MVR_CLOUD_TARGET && which_dst != MVR_CLOUD_SOURCE) ||
      (which_src != MVR_CLOUD_TARGET && which_src != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
  if (dst->device != src->device) return fail(dst, MVR_ERR_BAD_ARG, "contexts on different devices");
  const Cloud& s = which_src == MVR_CLOUD_TARGET ? src->tgt : src->src;
  Cloud& d = which_dst == MVR_CLOUD_TARGET ? dst->tgt : dst->src;
  if (s.gen == 0) return fail(dst, MVR_ERR_NO_INPUT, "cloud not set");
  if (&s == &d) return MVR_OK;
  d.index_valid = false;
  d.gen++;
  d.pts = s.pts; d.n = s.n; d.n_bad = s.n_bad;
  for (int a = 0; a < 3; ++a) { d.lo[a] = s.lo[a]; d.hi[a] = s.hi[a]; }
  if (which_dst == MVR_CLOUD_TARGET) dst->tnrm = nullptr; else { dst->have_out = false; dst->snrm = nullptr; }
  return MVR_OK;
}

static int set_normals(mvr_ctx* ctx, int which, const float* nxyzc, size_t n) {
  if (!ctx || !nxyzc) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  const bool tgt = which == MVR_CLOUD_TARGET;
  if ((int)n != (tgt ? ctx->tgt.n : ctx->src.n)) return fail(ctx, MVR_ERR_BAD_ARG, tgt ? "normals count differs from target size" : "normals count differs from source size");
  DevBuf& b = tgt ? ctx->normals : ctx->snormals;
  CK(b.ensure(std::max<size_t>(n, 1) * sizeof(float4)));
  CK(cudaMemcpyAsync(b.p, nxyzc, n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  (tgt ? ctx->tnrm : ctx->snrm) = b.as<float4>();
  return MVR_OK;
}

int mvr_set_target_normals(mvr_ctx* ctx, const float* nxyzc, size_t n) { return set_normals(ctx, MVR_CLOUD_TARGET, nxyzc, n); }
int mvr_set_source_normals(mvr_ctx* ctx, const float* nxyzc, size_t n) { return set_normals(ctx, MVR_CLOUD_SOURCE, nxyzc, n); }

int mvr_normals_share(mvr_ctx* dst, int which_dst, mvr_ctx* src, int which_src) {
  if (!dst || !src || (which_dst != MVR_CLOUD_TARGET && which_dst != MVR_CLOUD_SOURCE) ||
      (which_src != MVR_CLOUD_TARGET && which_src != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
  if (dst->device != src->device) return fail(dst, MVR_ERR_BAD_ARG, "contexts on different devices");
  const float4* p = which_src == MVR_CLOUD_TARGET ? src->tnrm : src->snrm;
  if (!p) return fail(dst, MVR_ERR_NO_INPUT, which_src == MVR_CLOUD_TARGET ? "the other context holds no target normals" : "the other context holds no source normals");
  const Cloud& sc = which_src == MVR_CLOUD_TARGET ? src->tgt : src->src;
  const Cloud& dc = which_dst == MVR_CLOUD_TARGET ? dst->tgt : dst->src;
  if (sc.n != dc.n) return fail(dst, MVR_ERR_BAD_ARG, "normals count differs from the cloud size");
  (which_dst == MVR_CLOUD_TARGET ? dst->tnrm : dst->snrm) = p;
  return MVR_OK;
}

int mvr_get_bbox(mvr_ctx* ctx, int which, float lo[3], float hi[3]) {
  if (!ctx || !lo || !hi || (which != MVR_CLOUD_TARGET && which != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
  const Cloud& c = which == MVR_CLOUD_TARGET ? ctx->tgt : ctx->src;
  if (c.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "cloud not set");
  for (int a = 0; a < 3; ++a) { lo[a] = c.lo[a]; hi[a] = c.hi[a]; }
  return MVR_OK;
}

int mvr_index_build(mvr_ctx* ctx, int which, const mvr_grid* grid) {
  if (!ctx || (which != MVR_CLOUD_TARGET && which != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  Cloud& c = which == MVR_CLOUD_TARGET ? ctx->tgt : ctx->src;
  if (!c.pts && c.n == 0 && c.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "cloud not set");
  mvr_grid g;
  if (grid) {
    if (grid->bits < 1 || grid->bits > 10 || !(grid->inv_cell > 0)) return fail(ctx, MVR_ERR_BAD_ARG, "bad grid");
    g = *grid;
  } else {
    g = auto_grid(ctx, c);
  }
  return build_index(ctx, c, c.pts, g);
}

int mvr_index_export(mvr_ctx* ctx, int which, mvr_grid* grid, uint32_t* sorted_keys, int32_t* perm, uint32_t* cell_start) {
  if (!ctx || (which != MVR_CLOUD_TARGET && which != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  Cloud& c = which == MVR_CLOUD_TARGET ? ctx->tgt : ctx->src;
  if (!c.index_valid || !c.exportable) return fail(ctx, MVR_ERR_NO_INPUT, "index not built (call mvr_index_build first)");
  if (grid) *grid = c.grid;
  if (sorted_keys && c.n) CK(cudaMemcpyAsync(sorted_keys, c.sorted_keys, c.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (perm && c.n) CK(cudaMemcpyAsync(perm, c.perm, c.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (cell_start) CK(cudaMemcpyAsync(cell_start, c.table.p, (((size_t)1 << (3 * c.grid.bits)) + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

int mvr_nn_query_device(mvr_ctx* ctx, const float* d_q, size_t n, int32_t* d_idx, float* d_d2) {
  if (!ctx || (n && (!d_q || !d_idx || !d_d2))) return MVR_ERR_BAD_ARG;
  if (n > (size_t)INT_MAX / 2) return fail(ctx, MVR_ERR_BAD_ARG, "too many queries");
  cudaSetDevice(ctx->device);
  if (ctx->tgt.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "target not set");
  if (n == 0) return MVR_OK;
  return nn_pass(ctx, (const float4*)d_q, (int)n, d_idx, d_d2);
}

int mvr_nn_query(mvr_ctx* ctx, const float* q, size_t n, int32_t* idx, float* d2) {
  if (!ctx || (n && (!q || !idx || !d2))) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->tgt.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "target not set");
  if (n == 0) return MVR_OK;
  CK(ctx->qtmp.ensure(n * sizeof(float4)));
  CK(ctx->itmp.ensure(n * sizeof(int32_t)));
  CK(ctx->ftmp.ensure(n * sizeof(float)));
  CK(cudaMemcpyAsync(ctx->qtmp.p, q, n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
  int rc = mvr_nn_query_device(ctx, ctx->qtmp.as<float>(), n, ctx->itmp.as<int32_t>(), ctx->ftmp.as<float>());
  if (rc) return rc;
  CK(cudaMemcpyAsync(idx, ctx->itmp.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(d2, ctx->ftmp.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

static int align_prepare_batch(mvr_ctx* const* ctxs, int count, const mvr_icp_params* prm, const float* guesses, int est, int* statuses,
                               std::vector<mvr_ctx*>& ok, std::vector<int>& slot);
// mvr_estimator -> the kernels' estimator (an unknown value means point-to-point)
static int estimator_code(int estimator) {
  return estimator == MVR_SYMMETRIC ? EST_SYM : (estimator == MVR_POINT_TO_PLANE ? EST_P2L : EST_P2P);
}
static int align_prepare(mvr_ctx* ctx, const mvr_icp_params* prm, const float* guess, int est) {
  int st = MVR_OK;
  std::vector<mvr_ctx*> ok;
  std::vector<int> slot;
  const int rc = align_prepare_batch(&ctx, 1, prm, guess, est, &st, ok, slot);
  return rc ? rc : st;
}

static int align_run(mvr_ctx* const* ctxs, int count, const mvr_icp_params* prm, int est);

int mvr_correspondences(mvr_ctx* ctx, double max_dist, int reciprocal, int32_t* iq, int32_t* im, float* dist, size_t* count) {
  if (!ctx || !count) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  *count = 0;
  if (ctx->tgt.gen == 0 || ctx->src.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "source/target not set");
  if (!(max_dist >= 0)) return fail(ctx, MVR_ERR_BAD_ARG, "max_dist must be >= 0");
  const int n = ctx->src.n;
  if (n == 0 || ctx->tgt.n == 0) return MVR_OK;
  if (!iq || !im || !dist) return MVR_ERR_BAD_ARG;
  // one correspondence pass of the fused iteration (no guess: the source as it is), then its pairs by source index
  mvr_icp_params one;
  mvr_icp_params_default(&one);
  one.max_iterations = 1; one.fixed_iterations = 1;
  one.use_reciprocal_correspondences = reciprocal ? 1 : 0;
  one.max_correspondence_distance = max_dist;
  one.min_correspondences = 1;
  ctx->want_rnn = true;
  int rc = align_prepare(ctx, &one, nullptr, EST_P2P);
  ctx->want_rnn = false;
  if (rc) return rc;
  if ((rc = align_run(&ctx, 1, &one, EST_P2P))) return rc;
  if (ctx->h_state->dbg[2] != 0) return fail(ctx, MVR_ERR_CUDA, "internal error: a reciprocal search lost its chooser (search bound violated)");
  CK(ctx->corr_j.ensure((size_t)n * sizeof(int32_t)));
  CK(ctx->corr_d2.ensure((size_t)n * sizeof(float)));
  CK(ctx->scratch.ensure(compact_scratch_elems(n) * sizeof(uint32_t) + 64));
  CK(ctx->itmp.ensure((size_t)2 * n * sizeof(int32_t)));
  CK(ctx->ftmp.ensure((size_t)n * sizeof(float)));
  CK(ctx->misc.ensure(64));
  int32_t* dq = ctx->itmp.as<int32_t>();
  int32_t* dm = dq + n;
  CK(cudaMemsetAsync(ctx->corr_j.p, 0xff, (size_t)n * sizeof(int32_t), ctx->stream));   // -1: no correspondence
  CK(launch_resolve_pairs(ctx->fa.cur, ctx->fa.n_valid, ctx->fa.corr_p, ctx->ra.rnn, ctx->fa.tgt, ctx->corr_j.as<int32_t>(),
                          ctx->corr_d2.as<float>(), ctx->stream));
  CK(launch_compact_corr(ctx->corr_j.as<int32_t>(), ctx->corr_d2.as<float>(), n, ctx->scratch.as<uint32_t>(), dq, dm,
                         ctx->ftmp.as<float>(), ctx->misc.as<uint32_t>(), ctx->stream));
  CK(cudaMemcpyAsync(ctx->h_small, ctx->misc.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  size_t c = ctx->h_small[0];
  if (c) {
    CK(cudaMemcpyAsync(iq, dq, c * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(im, dm, c * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dist, ctx->ftmp.p, c * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  *count = c;
  return MVR_OK;
}

// ---- the align behind mvr_icp_align, mvr_icp_align_batch and mvr_pair_moments_compute ------------------------------
// An align is split in three so that many of them can advance in lock-step, ONE launch per iteration half for a
// group of pairs (a single 200k-point pair fills a fraction of a B200):
//   align_plan / align_prepare_batch : per context on the host -- grids, buffers, initial state, kernel arguments; then per
//                   group of pairs, on the group's stream -- every per-align index (four launches), the seeds, gates and
//                   initial states (one launch);
//   align_run     : the iterations of every context of the batch (groups of pairs, each group on the stream of its first context);
//   align_finish  : per context -- report; the aligned cloud and the iteration log are produced when asked for.
// est = EST_MOM accumulates second moments next to the point-to-point sums (those of the LAST iteration's pairs).
// S: the stream the pair's group prepares and runs on; jobs: receives the index builds this align needs.
static int align_plan(mvr_ctx* ctx, const mvr_icp_params* prm, const float* guess, int est, cudaStream_t S, std::vector<BuildJob>& jobs) {
  cudaSetDevice(ctx->device);
  if (ctx->tgt.gen == 0 || ctx->src.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "source/target not set");
  Cloud& s = ctx->src;
  const int n = s.n;
  if (n == 0 || ctx->tgt.n == 0) return fail(ctx, MVR_ERR_NO_INPUT, "empty source or target");
  if (prm->estimator == MVR_POINT_TO_PLANE && !ctx->tnrm)
    return fail(ctx, MVR_ERR_NO_INPUT, "point-to-plane needs target normals (mvr_set_target_normals / mvr_estimate_normals)");
  if (est == EST_SYM && !ctx->tnrm)
    return fail(ctx, MVR_ERR_NO_INPUT, "symmetric point-to-plane needs target normals (mvr_set_target_normals / mvr_estimate_normals / mvr_normals_share)");
  if (est == EST_SYM && !ctx->snrm)
    return fail(ctx, MVR_ERR_NO_INPUT, "symmetric point-to-plane needs source normals (mvr_set_source_normals / mvr_estimate_normals / mvr_normals_share)");
  if (!(prm->max_correspondence_distance >= 0)) return fail(ctx, MVR_ERR_BAD_ARG, "max_correspondence_distance");
  float G[16];
  if (guess) std::memcpy(G, guess, sizeof(G)); else mat_identity(G);
  const bool reciprocal = prm->use_reciprocal_correspondences != 0;
  const double max_dist = prm->max_correspondence_distance;
  const bool p2l = est == EST_P2L || est == EST_SYM;
  const bool sym = est == EST_SYM;

  // ---- per-align indices: target over its own box (reused while the target and the grid stay the same),
  //      source over the box of the guessed source
  const int m = ctx->tgt.n;
  int rc = MVR_OK;
  {
    uint32_t cells = 0;
    const PairGrid gt = make_pair_grid(ctx->tgt.lo, ctx->tgt.hi, pair_cell_edge(ctx, ctx->tgt, max_dist), &cells, MVR_PG_XRATIO);
    PairIndex& pt = ctx->pt;
    if (!(pt.valid && pt.gen == ctx->tgt.gen && same_pair_grid(pt.g, gt))) {
      BuildJob job;
      pt.valid = false;
      if ((rc = plan_pair_index(ctx, pt, 0, ctx->tgt.pts, m, ctx->tgt.n_bad, nullptr, gt, cells, true, S, &job))) { pt.valid = false; return rc; }
      jobs.push_back(job);
      pt.gen = ctx->tgt.gen;
    }
  }
  {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (s.n - s.n_bad > 0) {
      for (int corner = 0; corner < 8; ++corner) {
        const double p[3] = {(corner & 1) ? s.hi[0] : s.lo[0], (corner & 2) ? s.hi[1] : s.lo[1], (corner & 4) ? s.hi[2] : s.lo[2]};
        for (int a = 0; a < 3; ++a) {
          const double v = G[a] * p[0] + G[4 + a] * p[1] + G[8 + a] * p[2] + G[12 + a];
          if (std::isfinite(v)) { lo[a] = std::min(lo[a], (float)v); hi[a] = std::max(hi[a], (float)v); }
        }
      }
    }
    for (int a = 0; a < 3; ++a) if (!(lo[a] <= hi[a])) { lo[a] = 0.f; hi[a] = 0.f; }
    uint32_t cells = 0;
    // the cell edge follows the source's own density (its box as given: a rigid guess keeps the surface area)
    const PairGrid gs = make_pair_grid(lo, hi, pair_cell_edge(ctx, s, max_dist), &cells, MVR_PG_XRATIO);
    Mat4f Gm;
    std::memcpy(Gm.m, G, sizeof(Gm.m));
    ctx->guess_m = Gm;
    BuildJob job;
    ctx->ps.valid = false;
    if ((rc = plan_pair_index(ctx, ctx->ps, 1, s.pts, n, s.n_bad, &Gm, gs, cells, true, S, &job))) { ctx->ps.valid = false; return rc; }
    jobs.push_back(job);
    for (int a = 0; a < 3; ++a) { ctx->h_state->box[a] = lo[a]; ctx->h_state->box[3 + a] = hi[a]; }   // kept across the memset below
  }
  const PairIndex &pt = ctx->pt, &psx = ctx->ps;
  CK(ctx->corr_p.ensure((size_t)std::max(n, 1) * sizeof(int32_t)));   // seeds and gates are filled by launch_align_init
  if (reciprocal) CK(ctx->rmin.ensure((size_t)std::max(m, 1) * sizeof(uint32_t)));
  if (sym) CK(ctx->nsrc.ensure((size_t)std::max(n, 1) * sizeof(float4)));   // filled by launch_align_init
  CK(ctx->partials.ensure((size_t)std::max((int)FUSED_MAX_BLOCKS, fused_grid_rev(m)) * REDUCE_MAX_VALS * sizeof(double)));
  CK(ctx->state.ensure(sizeof(IcpState)));
  CK(ctx->log.ensure((size_t)ICP_MAX_LOG * sizeof(IterRec)));
  IcpState* d_st = ctx->state.as<IcpState>();
  IterRec* d_log = ctx->log.as<IterRec>();

  // initial state: the guess has been applied while binning the source; it is the start of `fin`
  IcpState& h = *ctx->h_state;
  double sbox[6];
  for (int a = 0; a < 6; ++a) sbox[a] = h.box[a];
  std::memset(&h, 0, sizeof(h));
  // frame bookkeeping of the static source index: the box the guessed source was binned in (the pinned float transform
  // rounds each coordinate by < 1e-3 of it), no drift yet
  for (int a = 0; a < 3; ++a) {
    const double pad = 1e-3 + 1e-5 * std::max(std::fabs(sbox[a]), std::fabs(sbox[3 + a]));
    h.box[a] = sbox[a] - pad; h.box[3 + a] = sbox[3 + a] + pad;
    h.babs[a] = std::max(std::fabs(h.box[a]), std::fabs(h.box[3 + a]));
  }
  h.devd = 0.0; h.dev = 0.0f;
  for (int k = 0; k < 16; ++k) { h.delta[k] = (k % 5 == 0) ? 1.f : 0.f; h.fin[k] = G[k]; h.cum[k] = (k % 5 == 0) ? 1.0 : 0.0; }
  for (int k = 0; k < 12; ++k) h.cinv[k] = (k % 5 == 0) ? 1.0 : 0.0;
  h.stretch = 1.0f;
  h.prev_mse = DBL_MAX;
  h.rot_thr = 1.0 - prm->transformation_epsilon;
  h.trans_thr = prm->transformation_epsilon;
  h.fit_eps = prm->euclidean_fitness_epsilon;
  // provisional origin for the sums: centre of the target box (keeps the double sums well scaled)
  h.ox = 0.5 * ((double)ctx->tgt.lo[0] + ctx->tgt.hi[0]);
  h.oy = 0.5 * ((double)ctx->tgt.lo[1] + ctx->tgt.hi[1]);
  h.oz = 0.5 * ((double)ctx->tgt.lo[2] + ctx->tgt.hi[2]);
  h.max_iter = prm->max_iterations;
  h.fixed = prm->fixed_iterations != 0;
  h.min_corr = prm->min_correspondences > 0 ? prm->min_correspondences : 3;
  h.p2l = sym ? 2 : (p2l ? 1 : 0); h.recip = reciprocal; h.n_src = n;
  if (prm->max_iterations <= 0) { h.done = 1; h.reason = MVR_REASON_ITERATIONS; }
  ctx->iters.clear();
  ctx->log_pending = 0;
  ctx->have_out = false; ctx->out_pending = false;

  FwdArgs& fa = ctx->fa;
  fa = FwdArgs{};
  fa.cur = psx.sorted.as<float4>(); fa.n_valid = psx.n_valid;
  fa.tgt = pt.sorted.as<float4>(); fa.tstart = pt.start.as<uint32_t>(); fa.gt = pt.g; fa.m_valid = pt.n_valid;
  fa.corr_p = ctx->corr_p.as<int32_t>(); fa.rmin = reciprocal ? ctx->rmin.as<uint32_t>() : nullptr;
  fa.max2 = max_dist * max_dist; fa.max_d2f = gate_float(max_dist);
  fa.gmask = nullptr; fa.gm_stride = 0;   // set by align_prepare_batch once the target index exists
  fa.nrm = p2l ? ctx->tnrm : nullptr;
  fa.nsrc = sym ? ctx->nsrc.as<float4>() : nullptr;
  fa.partials = ctx->partials.as<double>(); fa.st = d_st; fa.log = d_log; fa.grid = fused_grid(psx.n_valid);
  RevArgs& ra = ctx->ra;
  ra = RevArgs{};
  ra.tgt = fa.tgt; ra.m_valid = pt.n_valid; ra.rmin = fa.rmin; ra.cur = fa.cur; ra.sstart = psx.start.as<uint32_t>(); ra.gs = psx.g;
  ra.n_valid = psx.n_valid; ra.corr_p = fa.corr_p; ra.nrm = fa.nrm; ra.nsrc = fa.nsrc;
  ra.rnn = nullptr;
  if (reciprocal && ctx->want_rnn) { CK(ctx->rnn.ensure((size_t)std::max(m, 1) * sizeof(int32_t))); ra.rnn = ctx->rnn.as<int32_t>(); }
  ra.partials = fa.partials; ra.st = d_st; ra.log = d_log; ra.grid = fused_grid_rev(pt.n_valid); ra.per = fused_rev_chunks(pt.n_valid);
  return MVR_OK;
}

// The contexts' pinned staging of a batch led by `lead`: room for `count` IcpStates on both sides.
static int ensure_stage(mvr_ctx* lead, int count) {
  mvr_ctx* ctx = lead;
  if (count > lead->stage_cap) {
    if (lead->h_stage) cudaFreeHost(lead->h_stage);
    lead->h_stage = nullptr; lead->stage_cap = 0;
    const int want = std::max(count + count / 2, 8);
    CK(cudaMallocHost((void**)&lead->h_stage, (size_t)want * sizeof(IcpState)));
    lead->stage_cap = want;
  }
  CK(lead->stage_dev.ensure((size_t)lead->stage_cap * sizeof(IcpState)));
  return MVR_OK;
}

static InitJob init_job_of(mvr_ctx* c) {
  InitJob j{};
  j.corr_p = c->corr_p.as<int32_t>(); j.n = std::max(c->src.n, 1); j.m = std::max(c->tgt.n, 1);
  j.rmin = c->fa.rmin; j.st = c->state.as<IcpState>(); j.crowded = c->crowded.as<uint32_t>();
  if (c->fa.nsrc) { j.nsrc = c->fa.nsrc; j.snrm = c->snrm; j.sorted = c->fa.cur; j.n_valid = c->fa.n_valid; j.M = c->guess_m; }
  return j;
}

// Pairs per lock-step group of a batch of `count` aligns led by `lead` (see align_run): a quarter of the batch unless
// mvr_ctx_set_batch_group chose a size.
static int batch_group_size(const mvr_ctx* lead, int count) {
  return lead->group_pairs > 0 ? std::min(lead->group_pairs, (int)FUSED_MAX_PAIRS) : std::max(1, std::min((count + 3) / 4, (int)FUSED_MAX_PAIRS));
}

// Prepare `count` aligns (same device): statuses[k] = the plan's verdict for context k; ok / slot = the contexts that go on
// and their positions.  The device work -- index builds, seeds, gates, initial states -- of every lock-step GROUP of pairs
// (align_run) is enqueued on the group's stream with a handful of launches whatever the group size (24 ring pairs in four
// groups: 48 index builds in 16 launches; one thread spent ~50 us per pair on launch calls alone when every pair prepared
// itself), so one group's builds overlap the iterations of the groups that started before it.
static int align_prepare_batch(mvr_ctx* const* ctxs, int count, const mvr_icp_params* prm, const float* guesses, int est, int* statuses,
                               std::vector<mvr_ctx*>& ok, std::vector<int>& slot) {
  ok.clear(); slot.clear();
  if (count <= 0) return MVR_OK;
  const int gsz0 = batch_group_size(ctxs[0], count);
  std::vector<std::vector<BuildJob>> jobs((size_t)count);
  for (int k = 0; k < count; ++k) if (ensure_pinned(ctxs[k]) != MVR_OK) return MVR_ERR_CUDA;
  // host side of every pair (grids, buffer checks, initial state): a few threads, no launches (first-time zeroing of a
  // scratch buffer goes to the stream of the group the pair is expected in)
  parallel_for(count, [&](int k) {
    statuses[k] = align_plan(ctxs[k], prm, guesses ? guesses + 16 * k : nullptr, est, ctxs[(k / gsz0) * gsz0]->stream, jobs[(size_t)k]);
  });
  for (int k = 0; k < count; ++k)
    if (statuses[k] == MVR_OK) { ok.push_back(ctxs[k]); slot.push_back(k); }
  if (ok.empty()) return MVR_OK;
  mvr_ctx* ctx = ok[0];   // CK() reports into it
  const int P = (int)ok.size();
  const int gsz = batch_group_size(ctx, P);
  if (P != count || gsz != gsz0) {
    // a context dropped out: the groups are not the expected ones -- order every group's stream behind every stream a plan
    // may have used (rare; only first-time zeroing is ever enqueued by a plan)
    for (int k = 0; k < count; k += gsz0) {
      cudaEvent_t e = ctxs[k]->ev_b;
      CK(cudaEventRecord(e, ctxs[k]->stream));
      for (int g0 = 0; g0 < P; g0 += gsz) CK(cudaStreamWaitEvent(ok[(size_t)g0]->stream, e, 0));
    }
  }
  int rc = ensure_stage(ctx, P);
  if (rc) return rc;
  for (int g0 = 0; g0 < P; g0 += gsz) {
    const int gn = std::min(gsz, P - g0);
    cudaStream_t S = ok[(size_t)g0]->stream;
    std::vector<BuildJob> all;
    for (int k = 0; k < gn; ++k) { const std::vector<BuildJob>& j = jobs[(size_t)slot[(size_t)(g0 + k)]]; all.insert(all.end(), j.begin(), j.end()); }
    if ((rc = run_pair_builds(ctx, all.data(), (int)all.size(), S))) return rc;
    for (int k0 = 0; k0 < gn; k0 += BUILD_MAX_JOBS) {
      const int c = std::min(gn - k0, (int)BUILD_MAX_JOBS);
      InitBatch ib;
      for (int k = 0; k < c; ++k) {
        mvr_ctx* m = ok[(size_t)(g0 + k0 + k)];
        ib.j[k] = init_job_of(m);
        std::memcpy(ctx->h_stage + g0 + k0 + k, m->h_state, sizeof(IcpState));
      }
      CK(cudaMemcpyAsync(ctx->stage_dev.as<IcpState>() + g0 + k0, ctx->h_stage + g0 + k0, (size_t)c * sizeof(IcpState), cudaMemcpyHostToDevice, S));
      CK(launch_align_init(ib, c, ctx->stage_dev.as<IcpState>() + g0 + k0, S));
    }
    for (int k = 0; k < gn; ++k) {
      mvr_ctx* m = ok[(size_t)(g0 + k)];
      if ((rc = ensure_gate_mask(m, m->pt, m->fa.max_d2f, S))) { ctx->err = m->err; return rc; }
      m->fa.gmask = m->pt.gm_gate >= 0.f ? m->pt.gmask.as<uint32_t>() : nullptr; m->fa.gm_stride = m->pt.gm_stride;
    }
  }
  return MVR_OK;
}

// The iterations of `count` prepared contexts (same device, same params) on the first one's stream.  The pairs
// advance in lock-step in groups of ctx->group_pairs (<= FUSED_MAX_PAIRS = 24, the kernel parameter space): a group runs
// to completion before the next one starts.  Measured on B200 (24 x 200k pairs): groups of 6 / 8 / 12 / 24 pairs take
// 28.3 / 27.7 / 26.8 / 25.3 ms -- fewer launch tails outweigh the L2 misses of a working set of 24 x 20 MB.
static int align_run(mvr_ctx* const* ctxs, int count, const mvr_icp_params* prm, int est) {
  mvr_ctx* ctx = ctxs[0];   // the lead: CK() reports into it, its ev_a .. ev_b bracket the iterations of the whole batch
  cudaSetDevice(ctx->device);
  const bool reciprocal = prm->use_reciprocal_correspondences != 0;
  // Groups of pairs advance in lock-step (one launch per iteration half serves a group); the groups themselves run
  // CONCURRENTLY, each on the stream of its first context, so that one group's launch tails, its serial solve and the gaps
  // between its dependent launches are filled by the others.  Measured on B200 (scripts/gpu_streams_vs_batch.py,
  // profiles/r02_concurrent_groups.log): 24 pairs 22.5 ms as one group, 20.6-20.8 ms as 2 .. 8 groups; 12 pairs 12.1 -> 10.5 ms;
  // 3 pairs 4.05 -> 3.3 ms.  Default: four groups (a group size set with mvr_ctx_set_batch_group is kept).
  const int gsz = batch_group_size(ctx, count);
  struct Group {
    int g0, gn, gf, gr, enqueued, first, todo;
    bool done, fetched;
    long long n_tot, m_tot;
    mvr_ctx* lead;
    FwdBatch fb;
    RevBatch rb;
  };
  // Source points per thread of the reciprocal forward half.  Measured on B200 (registration of 24 / 12 / 6 / 3 pairs of 200k
  // points, ms): 1 point 21.4 / 10.84 / 5.75 / 3.85, 2 points 20.3 / 10.44 / 5.63 / 3.90, 4 points 19.85 / 10.26 / 5.77 / 4.37,
  // 8 points 19.85, 16 points 20.1 -- about one point per 600k source points of the batch, at most four.
  long long batch_points = 0;
  for (int k = 0; k < count; ++k) batch_points += ctxs[k]->fa.n_valid;
  static const int fwd_items_env = [] { const char* e = std::getenv("MVR_FWD_ITEMS"); return e ? std::atoi(e) : 0; }();
  const int fwd_items = fwd_items_env > 0 ? fwd_items_env : (int)std::min<long long>(4, std::max<long long>(1, (batch_points + 300000) / 600000));
  std::vector<Group> groups;
  for (int g0 = 0; g0 < count; g0 += gsz) {
    Group g{};
    g.g0 = g0; g.gn = std::min(gsz, count - g0); g.gf = 1; g.gr = 1; g.enqueued = 0; g.first = 1; g.done = true; g.fetched = true;
    g.lead = ctxs[g0];
    for (int k = 0; k < g.gn; ++k) {
      mvr_ctx* c = ctxs[g0 + k];
      g.fb.a[k] = c->fa; g.rb.a[k] = c->ra;
      // the reciprocal forward half sums nothing, so its block partition is free to follow the load: with enough pairs to fill
      // the GPU several times over a thread takes `fwd_items` source points (fewer blocks, the per-block set-up amortised)
      if (reciprocal && fwd_items > 1) g.fb.a[k].grid = std::max(1, (c->fa.n_valid + FUSED_THREADS * fwd_items - 1) / (FUSED_THREADS * fwd_items));
      g.gf = std::max(g.gf, g.fb.a[k].grid); g.gr = std::max(g.gr, c->ra.grid);
      if (!c->h_state->done) g.done = false;
      g.n_tot += c->src.n; g.m_tot += c->tgt.n;
    }
    groups.push_back(g);
  }
  // every group's preparation (index builds, initial states) was enqueued on the group's own stream (align_prepare_batch)
  int rc0 = ensure_stage(ctx, count);
  if (rc0) return rc0;
  if (ctx->profiling) {   // a clean bracket for the roofline measurement: no build inside ev_a .. ev_b
    for (Group& g : groups) CK(cudaStreamSynchronize(g.lead->stream));
    CK(cudaEventRecord(ctx->ev_a, ctx->stream));
    for (size_t gi = 1; gi < groups.size(); ++gi) CK(cudaStreamWaitEvent(groups[gi].lead->stream, ctx->ev_a, 0));
  } else {
    CK(cudaEventRecord(ctx->ev_a, ctx->stream));
  }
  // staged states of a group -> its contexts (after the group's stream has been synchronised)
  auto unpack = [&](Group& g) {
    if (g.fetched) return;
    g.fetched = true;
    for (int k = 0; k < g.gn; ++k) {
      mvr_ctx* c = ctxs[g.g0 + k];
      std::memcpy(c->h_state, ctx->h_stage + g.g0 + k, sizeof(IcpState));
      c->crowded_seen = std::max(c->crowded_seen, (uint32_t)c->h_state->dbg[3]);
      c->h_state->dbg[3] = 0;
    }
  };
  for (int k = 0; k < count; ++k) ctxs[k]->crowded_seen = 0;
  // Enqueue iterations in batches; after each batch read the states back.  Once a pair raises `done` its blocks of the
  // remaining launches return immediately.
  int batch = prm->fixed_iterations ? 64 : 2;
  for (;;) {
    bool any = false;
    // The launches of the groups are enqueued ROUND-ROBIN, one iteration of every group at a time: a launch call costs the host
    // ~5 us, so enqueueing one group's 60 launches first would start the next group 0.3 ms late (3 pairs on 3 streams: 105 us
    // per iteration instead of ~80).
    int todo_max = 0;
    std::vector<std::unique_ptr<ProfScope>> scopes;
    for (Group& g : groups) {
      g.todo = 0;
      if (g.done) continue;
      any = true;
      g.todo = std::min(batch, std::max(prm->max_iterations - g.enqueued, 1));
      todo_max = std::max(todo_max, g.todo);
      // one scope = `todo` iterations: forward search (+ transform), reciprocal search (+ sums, solve, criteria) each.
      // Bytes per iteration as SURVEY.md section 8d counts them: every source and target point once (16 B each); with
      // reciprocal correspondences the source re-index PCL performs per iteration (36 B per source point) and the reverse
      // pass (16 B per source point) -- cell-table entries not counted.
      const double per_it = 16.0 * g.n_tot + 16.0 * g.m_tot + (reciprocal ? 52.0 * g.n_tot : 0.0);
      scopes.emplace_back(new ProfScope(g.lead, MVR_K_CORR, per_it * g.todo, (double)g.n_tot * g.todo, g.todo));
    }
    for (int it = 0; it < todo_max; ++it)
      for (Group& g : groups) {
        if (it >= g.todo) continue;
        CK(launch_icp_forward(g.fb, g.gn, g.gf, g.first, reciprocal, est, g.lead->stream));
        g.first = 0;
        if (reciprocal) CK(launch_icp_reverse(g.rb, g.gn, g.gr, est, g.lead->stream));
      }
    scopes.clear();   // closes the brackets (each on its group's stream)
    for (Group& g : groups) {
      if (g.todo == 0) continue;
      g.enqueued += g.todo;
      // the group's states come back together: one gather launch, one copy
      for (int k0 = 0; k0 < g.gn; k0 += BUILD_MAX_JOBS) {
        const int c = std::min(g.gn - k0, (int)BUILD_MAX_JOBS);
        InitBatch ib;
        for (int k = 0; k < c; ++k) ib.j[k] = init_job_of(ctxs[g.g0 + k0 + k]);
        IcpState* d = ctx->stage_dev.as<IcpState>() + g.g0 + k0;
        CK(launch_align_gather(ib, c, d, g.lead->stream));
        CK(cudaMemcpyAsync(ctx->h_stage + g.g0 + k0, d, (size_t)c * sizeof(IcpState), cudaMemcpyDeviceToHost, g.lead->stream));
      }
      g.fetched = false;
    }
    if (!any) break;
    bool more = false;
    for (Group& g : groups) {
      if (g.done) continue;
      if (prm->fixed_iterations) {
        g.done = g.enqueued >= prm->max_iterations;
      } else {
        CK(cudaStreamSynchronize(g.lead->stream));
        unpack(g);
        g.done = true;
        for (int k = 0; k < g.gn; ++k) if (!ctxs[g.g0 + k]->h_state->done) g.done = false;
      }
      if (!g.done) more = true;
    }
    if (!more) break;
    batch = std::min(batch * 2, 64);
  }
  // the lead stream joins the groups: ev_b marks the end of every pair's iterations, and whatever follows on the lead stream
  // (aligned clouds, logs) is ordered after all of them
  for (size_t gi = 1; gi < groups.size(); ++gi) {
    CK(cudaEventRecord(groups[gi].lead->ev_a, groups[gi].lead->stream));
    CK(cudaStreamWaitEvent(ctx->stream, groups[gi].lead->ev_a, 0));
  }
  CK(cudaEventRecord(ctx->ev_b, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (Group& g : groups) unpack(g);
  return MVR_OK;
}

// The aligned cloud icp.align returns, out = float(final) * source: computed when somebody asks for it (a batch of ring pairs
// never does), on the context's own stream -- the iterations are complete by the time an align returns.
static int materialize_out(mvr_ctx* ctx) {
  if (!ctx->have_out || !ctx->out_pending) return MVR_OK;
  const int n = ctx->src.n;
  CK(ctx->out_cloud.ensure((size_t)std::max(n, 1) * sizeof(float4)));
  {
    ProfScope ps(ctx, MVR_K_TRANSFORM, 32.0 * n, n);
    CK(launch_transform_final(ctx->src.pts, ctx->out_cloud.as<float4>(), n, ctx->state.as<IcpState>(), ctx->stream));
  }
  ctx->out_pending = false;
  return MVR_OK;
}

// The iteration log of the last align, fetched from the device on first use.
static int fetch_log(mvr_ctx* ctx) {
  const int n_log = ctx->log_pending;
  if (n_log <= 0) return MVR_OK;
  ctx->log_pending = 0;
  CK(cudaMemcpyAsync(ctx->h_log, ctx->log.p, (size_t)n_log * sizeof(IterRec), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < n_log; ++k) {
    mvr_icp_iteration rec;
    rec.iteration = ctx->h_log[k].iteration; rec.n_correspondences = ctx->h_log[k].n_corr; rec.mse = ctx->h_log[k].mse;
    std::memcpy(rec.delta, ctx->h_log[k].delta, sizeof(rec.delta));
    ctx->iters.push_back(rec);
  }
  return MVR_OK;
}

// After align_run (which has synchronised): the report of one context.  lead: the context whose ev_a .. ev_b bracket the
// iterations of the batch.
static int align_finish_collect(mvr_ctx* ctx, mvr_ctx* lead, float* out_pose, mvr_icp_report* report, int batch_pairs = 1) {
  const IcpState& h = *ctx->h_state;
  if (h.dbg[2] != 0) return fail(ctx, MVR_ERR_CUDA, "internal error: a reciprocal search lost its chooser (search bound violated)");
  ctx->have_out = true; ctx->out_pending = true;
  ctx->log_pending = std::min(h.iter, (int)ICP_MAX_LOG);
  if (out_pose) for (int k = 0; k < 16; ++k) out_pose[k] = (float)h.fin[k];
  if (report) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, lead->ev_a, lead->ev_b);
    report->iterations = h.iter; report->converged = (h.done && h.status == 0) ? 1 : 0; report->reason = h.reason;
    report->n_correspondences = h.n_corr; report->mse = h.cur_mse; report->nn_queries = h.queries;
    // pairs of a batch advance in lock-step and are not separable: each is given its share of the batch's device time
    report->gpu_ms = (double)ms / (double)std::max(batch_pairs, 1);
  }
  if (ctx->crowded_seen)
    ctx->err = "warning: a grid cell holds " + std::to_string(ctx->crowded_seen) + " points (duplicates or clamped outliers?): index build and search slow down, sums over it lose their fixed order";
  if (h.status == MVR_ERR_TOO_FEW_CORRESPONDENCES) ctx->err = "not enough correspondences";
  if (h.status == MVR_ERR_NOT_SPD) ctx->err = h.p2l == 2 ? "symmetric point-to-plane normal equations not positive definite" : "point-to-plane normal equations not positive definite";
  return h.status;
}

static int align_finish(mvr_ctx* ctx, mvr_ctx* lead, float* out_pose, float* out_xyzw, mvr_icp_report* report) {
  const int status = align_finish_collect(ctx, lead, out_pose, report);
  if (out_xyzw && ctx->have_out) {
    int rc = materialize_out(ctx);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_xyzw, ctx->out_cloud.p, (size_t)ctx->src.n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return status;
}

static int icp_align_impl(mvr_ctx* ctx, const mvr_icp_params* prm, const float* guess, float* out_pose, float* out_xyzw,
                          mvr_icp_report* report, bool moments) {
  if (!ctx || !prm) return MVR_ERR_BAD_ARG;
  const int est = estimator_code(prm->estimator);
  if (moments && est != EST_P2P) return fail(ctx, MVR_ERR_BAD_ARG, "pair moments are point-to-point statistics");
  const int est_run = moments ? EST_MOM : est;
  int rc = align_prepare(ctx, prm, guess, est_run);
  if (rc) return rc;
  if ((rc = align_run(&ctx, 1, prm, est_run))) return rc;
  return align_finish(ctx, ctx, out_pose, out_xyzw, report);
}

int mvr_icp_align(mvr_ctx* ctx, const mvr_icp_params* prm, const float* guess, float* out_pose, float* out_xyzw,
                  mvr_icp_report* report) {
  return icp_align_impl(ctx, prm, guess, out_pose, out_xyzw, report, false);
}

int mvr_icp_align_batch(mvr_ctx* const* ctxs, int count, const mvr_icp_params* prm, const float* guesses, float* out_poses,
                        mvr_icp_report* reports, int* statuses) {
  if (count < 0 || (count && (!ctxs || !statuses)) || !prm) return MVR_ERR_BAD_ARG;
  if (count == 0) return MVR_OK;
  for (int k = 0; k < count; ++k) {
    if (!ctxs[k]) return MVR_ERR_BAD_ARG;
    for (int j = 0; j < k; ++j) if (ctxs[j] == ctxs[k]) return fail(ctxs[0], MVR_ERR_BAD_ARG, "a context appears twice in the batch");
    if (ctxs[k]->device != ctxs[0]->device) return fail(ctxs[0], MVR_ERR_BAD_ARG, "the contexts of a batch must share a device");
  }
  const int est = estimator_code(prm->estimator);
  std::vector<mvr_ctx*> ok;
  std::vector<int> slot;
  const bool timing = std::getenv("MVR_DEBUG_TIMING") != nullptr;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  int rc = align_prepare_batch(ctxs, count, prm, guesses, est, statuses, ok, slot);
  if (rc) { if (!ok.empty() && ok[0] != ctxs[0]) ctxs[0]->err = ok[0]->err; return rc; }
  if (ok.empty()) return MVR_OK;
  const double t1 = now();
  rc = align_run(ok.data(), (int)ok.size(), prm, est);
  if (timing) std::fprintf(stderr, "[timing]   prepare (host enqueue) %.3f ms, run %.3f ms\n", t1 - t0, now() - t1);
  if (rc) { if (ok[0] != ctxs[0]) ctxs[0]->err = ok[0]->err; return rc; }
  for (size_t j = 0; j < ok.size(); ++j) {
    const int k = slot[j];
    statuses[k] = align_finish_collect(ok[j], ok[0], out_poses ? out_poses + 16 * k : nullptr, reports ? reports + k : nullptr, (int)ok.size());
  }
  return MVR_OK;
}

int mvr_pair_moments_compute(mvr_ctx* ctx, double max_dist, int reciprocal, const float* guess, mvr_pair_moments* out) {
  if (!ctx || !out) return MVR_ERR_BAD_ARG;
  std::memset(out, 0, sizeof(*out));
  mvr_icp_params one;
  mvr_icp_params_default(&one);
  one.max_iterations = 1; one.fixed_iterations = 1;
  one.use_reciprocal_correspondences = reciprocal ? 1 : 0;
  one.max_correspondence_distance = max_dist;
  one.min_correspondences = 1;
  mvr_icp_report rep{};
  const int rc = icp_align_impl(ctx, &one, guess, nullptr, nullptr, &rep, true);
  if (rc != MVR_OK && rc != MVR_ERR_TOO_FEW_CORRESPONDENCES) return rc;
  const IcpState& h = *ctx->h_state;
  out->origin[0] = h.ox; out->origin[1] = h.oy; out->origin[2] = h.oz;
  if (rc == MVR_OK) {
    out->n = h.sums[0];
    for (int k = 0; k < 3; ++k) { out->sa[k] = h.sums[1 + k]; out->sb[k] = h.sums[4 + k]; }
    for (int k = 0; k < 9; ++k) out->sba[k] = h.sums[7 + k];
    out->d2 = h.sums[16];
    for (int k = 0; k < 6; ++k) { out->saa[k] = h.sums[17 + k]; out->sbb[k] = h.sums[23 + k]; }
  }
  return MVR_OK;
}

static void moments_from_state(const IcpState& h, bool have, mvr_pair_moments* out) {
  std::memset(out, 0, sizeof(*out));
  out->origin[0] = h.ox; out->origin[1] = h.oy; out->origin[2] = h.oz;
  if (!have) return;
  out->n = h.sums[0];
  for (int k = 0; k < 3; ++k) { out->sa[k] = h.sums[1 + k]; out->sb[k] = h.sums[4 + k]; }
  for (int k = 0; k < 9; ++k) out->sba[k] = h.sums[7 + k];
  out->d2 = h.sums[16];
  for (int k = 0; k < 6; ++k) { out->saa[k] = h.sums[17 + k]; out->sbb[k] = h.sums[23 + k]; }
}

int mvr_pair_moments_compute_batch(mvr_ctx* const* ctxs, int count, double max_dist, int reciprocal, const float* guesses,
                                   mvr_pair_moments* out, int* statuses) {
  if (count < 0 || (count && (!ctxs || !out || !statuses))) return MVR_ERR_BAD_ARG;
  if (count == 0) return MVR_OK;
  for (int k = 0; k < count; ++k) {
    if (!ctxs[k]) return MVR_ERR_BAD_ARG;
    for (int j = 0; j < k; ++j) if (ctxs[j] == ctxs[k]) return fail(ctxs[0], MVR_ERR_BAD_ARG, "a context appears twice in the batch");
    if (ctxs[k]->device != ctxs[0]->device) return fail(ctxs[0], MVR_ERR_BAD_ARG, "the contexts of a batch must share a device");
  }
  mvr_icp_params one;
  mvr_icp_params_default(&one);
  one.max_iterations = 1; one.fixed_iterations = 1;
  one.use_reciprocal_correspondences = reciprocal ? 1 : 0;
  one.max_correspondence_distance = max_dist;
  one.min_correspondences = 1;
  std::vector<mvr_ctx*> ok;
  std::vector<int> slot;
  for (int k = 0; k < count; ++k) std::memset(out + k, 0, sizeof(mvr_pair_moments));
  int rc = align_prepare_batch(ctxs, count, &one, guesses, EST_MOM, statuses, ok, slot);
  if (rc) { if (!ok.empty() && ok[0] != ctxs[0]) ctxs[0]->err = ok[0]->err; return rc; }
  if (ok.empty()) return MVR_OK;
  rc = align_run(ok.data(), (int)ok.size(), &one, EST_MOM);
  if (rc) { if (ok[0] != ctxs[0]) ctxs[0]->err = ok[0]->err; return rc; }
  for (size_t j = 0; j < ok.size(); ++j) {
    const IcpState& h = *ok[j]->h_state;
    const int k = slot[j];
    if (h.dbg[2] != 0) { statuses[k] = fail(ok[j], MVR_ERR_CUDA, "internal error: a reciprocal search lost its chooser (search bound violated)"); continue; }
    const bool have = h.status == MVR_OK;
    statuses[k] = (have || h.status == MVR_ERR_TOO_FEW_CORRESPONDENCES) ? MVR_OK : h.status;
    moments_from_state(h, have, out + k);
    ok[j]->have_out = false; ok[j]->out_pending = false;
  }
  return MVR_OK;
}

double mvr_debug_value(mvr_ctx* ctx, int k) {
  if (ctx && k == 8) return (double)ctx->crowded_seen;   // population of a cell too crowded to rank in the last align's index builds
  if (!ctx || !ctx->h_state || k < 0 || k >= 8) return 0.0;
  return (double)ctx->h_state->dbg[k];
}

int mvr_icp_get_iterations(mvr_ctx* ctx, mvr_icp_iteration* out, int max_records, int* count) {
  if (!ctx || !count) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  int rcl = fetch_log(ctx);
  if (rcl) return rcl;
  int c = (int)ctx->iters.size();
  if (out) {
    int m = std::min(c, std::max(max_records, 0));
    if (m) std::memcpy(out, ctx->iters.data(), (size_t)m * sizeof(mvr_icp_iteration));
    *count = m;
  } else {
    *count = c;
  }
  return MVR_OK;
}

int mvr_fitness_score(mvr_ctx* ctx, double max_range, double* score) {
  if (!ctx || !score) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->tgt.gen == 0 || ctx->src.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "source/target not set");
  const int n = ctx->src.n;
  *score = DBL_MAX;
  if (n == 0 || ctx->tgt.n == 0) return MVR_OK;
  int rc = materialize_out(ctx);
  if (rc) return rc;
  const float4* cloud = ctx->have_out ? ctx->out_cloud.as<float4>() : ctx->src.pts;
  CK(ctx->itmp.ensure((size_t)n * sizeof(int32_t)));
  CK(ctx->ftmp.ensure((size_t)n * sizeof(float)));
  CK(ctx->partials.ensure((size_t)REDUCE_BLOCKS * REDUCE_MAX_VALS * sizeof(double)));
  CK(ctx->sums.ensure(REDUCE_MAX_VALS * sizeof(double)));
  if ((rc = nn_pass(ctx, cloud, n, ctx->itmp.as<int32_t>(), ctx->ftmp.as<float>()))) return rc;
  CK(launch_reduce_fitness(ctx->itmp.as<int32_t>(), ctx->ftmp.as<float>(), n, max_range, ctx->partials.as<double>(),
                           ctx->sums.as<double>(), ctx->stream));
  CK(cudaMemcpyAsync(ctx->h_sums, ctx->sums.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (ctx->h_sums[1] > 0) *score = ctx->h_sums[0] / ctx->h_sums[1];
  return MVR_OK;
}

int mvr_apply_pose(mvr_ctx* ctx, const void* points, size_t n, size_t stride_bytes, const double* pose, float* out_xyzw) {
  if (!ctx || !pose || (n && (!points || !out_xyzw))) return MVR_ERR_BAD_ARG;
  if (stride_bytes < 12 || stride_bytes % 4 != 0) return fail(ctx, MVR_ERR_BAD_ARG, "stride must be a multiple of 4 and >= 12");
  if (n > (size_t)INT_MAX / 2) return fail(ctx, MVR_ERR_BAD_ARG, "cloud too large");
  cudaSetDevice(ctx->device);
  if (n == 0) return MVR_OK;
  CK(ctx->scratch.ensure(n * stride_bytes));
  CK(ctx->qtmp.ensure(n * sizeof(float4)));
  CK(cudaMemcpyAsync(ctx->scratch.p, points, n * stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(launch_apply_pose(ctx->scratch.p, stride_bytes, (int)n, pose, ctx->qtmp.as<float4>(), ctx->stream));
  CK(cudaMemcpyAsync(out_xyzw, ctx->qtmp.p, n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

int mvr_apply_pose_device(mvr_ctx* ctx, const void* d_points, size_t n, size_t stride_bytes, const double* pose, float* d_out) {
  if (!ctx || !pose || (n && (!d_points || !d_out))) return MVR_ERR_BAD_ARG;
  if (stride_bytes < 12 || stride_bytes % 4 != 0) return fail(ctx, MVR_ERR_BAD_ARG, "stride must be a multiple of 4 and >= 12");
  if (n > (size_t)INT_MAX / 2) return fail(ctx, MVR_ERR_BAD_ARG, "cloud too large");
  cudaSetDevice(ctx->device);
  if (n == 0) return MVR_OK;
  CK(launch_apply_pose(d_points, stride_bytes, (int)n, pose, (float4*)d_out, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

int mvr_merge_registered(mvr_ctx* ctx, const void* const* views, const size_t* counts, const double* poses, const int* registered,
                         int n_views, int full_matrix_normals, void* out, size_t* out_count) {
  if (!ctx || n_views < 0 || !out_count || (n_views && (!views || !counts || !poses))) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  size_t total = 0;
  for (int v = 0; v < n_views; ++v) {
    if (registered && !registered[v]) continue;
    if (counts[v] && !views[v]) return fail(ctx, MVR_ERR_BAD_ARG, "null view");
    if (counts[v] > (size_t)INT_MAX / 4) return fail(ctx, MVR_ERR_BAD_ARG, "view too large");
    total += counts[v];
  }
  *out_count = total;
  if (!out || total == 0) return MVR_OK;   // out == NULL: size query
  CK(ctx->scratch.ensure(total * 48));
  size_t biggest = 0;
  for (int v = 0; v < n_views; ++v) if (!registered || registered[v]) biggest = std::max(biggest, counts[v]);
  CK(ctx->qtmp.ensure(std::max<size_t>(biggest, 1) * 48));
  size_t at = 0;
  for (int v = 0; v < n_views; ++v) {
    if ((registered && !registered[v]) || counts[v] == 0) continue;
    CK(cudaMemcpyAsync(ctx->qtmp.p, views[v], counts[v] * 48, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_merge_rich(ctx->qtmp.p, (int)counts[v], poses + 16 * v, full_matrix_normals, (char*)ctx->scratch.p + at * 48, ctx->stream));
    at += counts[v];
  }
  CK(cudaMemcpyAsync(out, ctx->scratch.p, total * 48, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

int mvr_copy_aligned_device(mvr_ctx* ctx, float* d_out) {
  if (!ctx || !d_out) return MVR_ERR_BAD_ARG;
  cudaSetDevice(ctx->device);
  if (!ctx->have_out) return fail(ctx, MVR_ERR_NO_INPUT, "no align has run");
  int rcm = materialize_out(ctx);
  if (rcm) return rcm;
  if (ctx->src.n > 0) CK(cudaMemcpyAsync(d_out, ctx->out_cloud.p, (size_t)ctx->src.n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MVR_OK;
}

int mvr_denoise(mvr_ctx* ctx, const void* points, size_t n, size_t stride_bytes, int segment_threshold, double triangle_length,
                int32_t* kept_index, size_t* kept_count, size_t* noise_count) {
  if (!ctx || !kept_count || (n && (!points || !kept_index))) return MVR_ERR_BAD_ARG;
  if (stride_bytes < 12 || stride_bytes % 4 != 0) return fail(ctx, MVR_ERR_BAD_ARG, "stride must be a multiple of 4 and >= 12");
  if (!(triangle_length > 0) || !std::isfinite(triangle_length)) return fail(ctx, MVR_ERR_BAD_ARG, "triangle_length must be positive");
  if (n > (size_t)INT_MAX / 4) return fail(ctx, MVR_ERR_BAD_ARG, "cloud too large");
  cudaSetDevice(ctx->device);
  *kept_count = 0;
  if (noise_count) *noise_count = 0;
  if (n == 0) return MVR_OK;
  const int ni = (int)n;
  // the points as PointXYZ records on the device (identity pose: getTransformedPoints' narrowing of x, y, z only)
  CK(ctx->scratch.ensure(n * stride_bytes));
  CK(ctx->qtmp.ensure(n * sizeof(float4)));
  CK(cudaMemcpyAsync(ctx->scratch.p, points, n * stride_bytes, cudaMemcpyHostToDevice, ctx->stream));
  const double I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  CK(launch_apply_pose(ctx->scratch.p, stride_bytes, ni, I16, ctx->qtmp.as<float4>(), ctx->stream));
  // grid with cell edge = the edge threshold: every neighbour within it sits in the 27 cells around a point
  Cloud tmp;
  tmp.pts = ctx->qtmp.as<float4>(); tmp.n = ni;
  int rc = cloud_bbox(ctx, tmp);
  if (rc) return rc;
  uint32_t cells = 0;
  const PairGrid g = make_pair_grid(tmp.lo, tmp.hi, triangle_length * 1.0001, &cells);
  if ((double)g.cell_lo < triangle_length) return fail(ctx, MVR_ERR_BAD_ARG, "cloud too large for this edge length (grid capped)");
  PairIndex& ix = ctx->nq;
  if ((rc = build_pair_index(ctx, ix, tmp.pts, ni, tmp.n_bad, nullptr, g, cells, false, false))) return rc;
  // parent | count | keys | vals | keys_alt | vals_alt | hist | n_noise
  const size_t nb = (size_t)radix_num_blocks(ni) * 256;
  CK(ctx->itmp.ensure(((size_t)6 * n + nb + 16) * sizeof(uint32_t)));
  uint32_t* parent = ctx->itmp.as<uint32_t>();
  uint32_t *count = parent + n, *keys = count + n, *vals = keys + n, *keys_alt = vals + n, *vals_alt = keys_alt + n, *hist = vals_alt + n, *d_noise = hist + nb;
  CK(cudaMemsetAsync(d_noise, 0, sizeof(uint32_t), ctx->stream));
  CK(launch_denoise_components(ix.sorted.as<float4>(), ix.start.as<uint32_t>(), g, ni, ix.n_valid, triangle_length, parent, keys, count, ctx->stream));
  CK(launch_denoise_keys(count, ni, (uint32_t)std::max(segment_threshold, 0), keys, vals, d_noise, ctx->stream));
  uint32_t *ko = nullptr, *vo = nullptr;
  SortScratch sc{keys_alt, vals_alt, hist};
  CK(launch_radix_sort(keys, vals, ni, 32, sc, &ko, &vo, ctx->stream));   // stable: components by root, points by index
  CK(cudaMemcpyAsync(ctx->h_small, d_noise, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const size_t noise = ctx->h_small[0], kept = n - noise;
  if (kept) CK(cudaMemcpyAsync(kept_index, vo, kept * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *kept_count = kept;
  if (noise_count) *noise_count = noise;
  ctx->nq.valid = false;
  return MVR_OK;
}

int mvr_estimate_normals(mvr_ctx* ctx, int which, int k, const float viewpoint[3], float* out, int32_t* neighbours) {
  if (!ctx || !out || (which != MVR_CLOUD_TARGET && which != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
  if (k < 3 || k > 32) return fail(ctx, MVR_ERR_BAD_ARG, "k must be in 3..32");
  cudaSetDevice(ctx->device);
  Cloud& c = which == MVR_CLOUD_TARGET ? ctx->tgt : ctx->src;
  if (c.gen == 0) return fail(ctx, MVR_ERR_NO_INPUT, "cloud not set");
  const int n = c.n;
  if (n == 0) return MVR_OK;
  uint32_t cells = 0;
  const PairGrid g = normals_grid(ctx, c, k, &cells);
  PairIndex& ix = ctx->nq;
  int rc = build_pair_index(ctx, ix, c.pts, n, c.n_bad, nullptr, g, cells, false, false);
  if (rc) return rc;
  DevBuf& nb = which == MVR_CLOUD_TARGET ? ctx->normals : ctx->snormals;
  CK(nb.ensure((size_t)n * sizeof(float4)));
  int32_t* dn = nullptr;
  if (neighbours) { CK(ctx->itmp.ensure((size_t)n * k * sizeof(int32_t))); dn = ctx->itmp.as<int32_t>(); }
  NormalsBatch batch;
  batch.j[0] = normals_job(ix, n, viewpoint, nb.as<float4>(), dn);
  {
    ProfScope ps(ctx, MVR_K_NORMALS, 32.0 * n, n);
    CK(launch_normals(batch, 1, k, ctx->stream));
  }
  ix.valid = false;
  CK(cudaMemcpyAsync(out, nb.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  if (neighbours) CK(cudaMemcpyAsync(neighbours, dn, (size_t)n * k * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  (which == MVR_CLOUD_TARGET ? ctx->tnrm : ctx->snrm) = nb.as<float4>();   // kept as the cloud's normals
  return MVR_OK;
}

// The normals of many clouds of one device: every index is planned on the host, then the builds (four launches per BUILD_MAX_JOBS
// clouds, run_pair_builds) and the normals (one launch per BUILD_MAX_JOBS clouds) go to the LEAD's stream.  That stream first
// waits for the work already queued on every context's stream (their clouds and buffers), and every context's stream then
// waits for the normals, so whatever a context does next -- on its own stream or on the stream of the align group it joins --
// runs after them.  The grids and the kernel are those of mvr_estimate_normals: the same bits, whatever the batch.
// which (nullable: all targets): entry a estimates the target (MVR_CLOUD_TARGET) or the source normals of ctxs[a]; a context
// may appear once per cloud.  A target's index is built in the context's query index (nq), a source's in its dense-pass
// target index (nt, rebuilt by the next NN pass), so both clouds of one context fit in one batch.
}  // extern "C"

// Declared in host/registrator.h: the ring driver estimates a shard's last source with its targets.
int mvr::estimate_normals_batch(mvr_ctx* const* ctxs, const int* which, int count, int k, const float* viewpoints, float* const* out_nxyzc,
                                int* statuses) {
  if (count < 0 || (count && (!ctxs || !statuses))) return MVR_ERR_BAD_ARG;
  if (count == 0) return MVR_OK;
  auto which_of = [&](int a) { return which ? which[a] : (int)MVR_CLOUD_TARGET; };
  for (int a = 0; a < count; ++a) {
    if (!ctxs[a] || (which_of(a) != MVR_CLOUD_TARGET && which_of(a) != MVR_CLOUD_SOURCE)) return MVR_ERR_BAD_ARG;
    for (int b = 0; b < a; ++b)
      if (ctxs[b] == ctxs[a] && which_of(b) == which_of(a)) return fail(ctxs[0], MVR_ERR_BAD_ARG, "a context appears twice in the batch");
    if (ctxs[a]->device != ctxs[0]->device) return fail(ctxs[0], MVR_ERR_BAD_ARG, "the contexts of a batch must share a device");
  }
  mvr_ctx* ctx = ctxs[0];   // the lead: CK() reports into it, its stream runs the batch, its profile records the launches
  if (k < 3 || k > 32) return fail(ctx, MVR_ERR_BAD_ARG, "k must be in 3..32");
  cudaSetDevice(ctx->device);
  const cudaStream_t S = ctx->stream;
  cudaEvent_t ev = get_event(ctx);
  if (!ev) return fail(ctx, MVR_ERR_CUDA, "cudaEventCreate failed");
  struct Todo { mvr_ctx* m; int slot; bool tgt; NormalsJob job; };
  std::vector<Todo> todo;
  std::vector<BuildJob> builds;
  int rc = MVR_OK;
  for (int a = 0; a < count && rc == MVR_OK; ++a) {
    mvr_ctx* m = ctxs[a];
    if (m != ctx && m->stream != S) {
      if (cudaEventRecord(ev, m->stream) != cudaSuccess || cudaStreamWaitEvent(S, ev, 0) != cudaSuccess) rc = fail(ctx, MVR_ERR_CUDA, "stream ordering failed");
    }
    if (rc) break;
    const bool tgt = which_of(a) == MVR_CLOUD_TARGET;
    Cloud& t = tgt ? m->tgt : m->src;
    if (t.gen == 0) { statuses[a] = fail(m, MVR_ERR_NO_INPUT, tgt ? "target not set" : "source not set"); continue; }
    statuses[a] = MVR_OK;
    if (t.n == 0) continue;
    uint32_t cells = 0;
    const PairGrid g = normals_grid(m, t, k, &cells);
    BuildJob bj;
    PairIndex& ix = tgt ? m->nq : m->nt;
    ix.valid = false;
    if ((rc = plan_pair_index(m, ix, tgt ? 1 : 0, t.pts, t.n, t.n_bad, nullptr, g, cells, false, S, &bj))) { ctx->err = m->err; break; }
    DevBuf& nb = tgt ? m->normals : m->snormals;
    if (nb.ensure((size_t)t.n * sizeof(float4)) != cudaSuccess) { rc = fail(ctx, MVR_ERR_CUDA, "normals buffer allocation failed"); break; }
    builds.push_back(bj);
    todo.push_back(Todo{m, a, tgt, normals_job(ix, t.n, viewpoints ? viewpoints + 3 * a : nullptr, nb.as<float4>(), nullptr)});
  }
  if (rc == MVR_OK) rc = run_pair_builds(ctx, builds.data(), (int)builds.size(), S);
  for (size_t t0 = 0; rc == MVR_OK && t0 < todo.size(); t0 += BUILD_MAX_JOBS) {
    const int c = (int)std::min(todo.size() - t0, (size_t)BUILD_MAX_JOBS);
    NormalsBatch batch;
    double pts = 0;
    for (int a = 0; a < c; ++a) { batch.j[a] = todo[t0 + a].job; pts += todo[t0 + a].job.n; }
    ProfScope ps(ctx, MVR_K_NORMALS, 32.0 * pts, pts, 1, S);
    const cudaError_t e = launch_normals(batch, c, k, S);
    if (e != cudaSuccess) rc = fail(ctx, MVR_ERR_CUDA, (std::string("launch_normals: ") + cudaGetErrorString(e)).c_str());
  }
  bool copies = false;
  for (size_t a = 0; rc == MVR_OK && a < todo.size(); ++a) {
    mvr_ctx* m = todo[a].m;
    (todo[a].tgt ? m->nq : m->nt).valid = false;
    (todo[a].tgt ? m->tnrm : m->snrm) = todo[a].job.out;
    float* out = out_nxyzc ? out_nxyzc[todo[a].slot] : nullptr;
    if (!out) continue;
    if (cudaMemcpyAsync(out, todo[a].job.out, (size_t)todo[a].job.n * sizeof(float4), cudaMemcpyDeviceToHost, S) != cudaSuccess) rc = fail(ctx, MVR_ERR_CUDA, "normals copy failed");
    copies = true;
  }
  // every context's later work waits for the normals (also after a failure: nothing queued above may overlap it)
  if (cudaEventRecord(ev, S) == cudaSuccess) {
    for (int a = 0; a < count; ++a) if (ctxs[a]->stream != S) cudaStreamWaitEvent(ctxs[a]->stream, ev, 0);
  } else if (rc == MVR_OK) {
    rc = fail(ctx, MVR_ERR_CUDA, "stream ordering failed");
  }
  ctx->ev_pool.push_back(ev);
  if (rc == MVR_OK && copies) CK(cudaStreamSynchronize(S));
  return rc;
}

extern "C" {

int mvr_estimate_normals_batch(mvr_ctx* const* ctxs, int count, int k, const float* viewpoints, float* const* out_nxyzc, int* statuses) {
  return mvr::estimate_normals_batch(ctxs, nullptr, count, k, viewpoints, out_nxyzc, statuses);
}

}  // extern "C"
