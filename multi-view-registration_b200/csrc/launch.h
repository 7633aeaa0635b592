// launch.h -- host-callable launchers of the CUDA kernels (one per kernel family).
// Every launcher enqueues on the given stream and returns the last CUDA error; none synchronises.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace mvr {

// Process-wide count of kernel launches issued by this library (bench.py reports it as gpu_launches).
void count_launch(int n = 1);
unsigned long long launch_count();

// ---- index.cu ------------------------------------------------------------------------------
// bbox: out[0..2] = min xyz, out[3..5] = max xyz (as order-preserving uint encodings), out[6] = count
// of non-finite points.  `out` must be initialised with bbox_init().
cudaError_t launch_bbox_init(uint32_t* out7, cudaStream_t s);
cudaError_t launch_bbox(const float4* pts, int n, uint32_t* out7, cudaStream_t s);
float bbox_decode(uint32_t enc);
// The boxes of `count` clouds in one launch: out7[7 * k ..] of cloud k (initialised by the launcher).
struct BboxJob { const float4* pts; int n; int pad_; };
enum { BBOX_MAX_JOBS = 64 };
struct BboxBatch { BboxJob j[BBOX_MAX_JOBS]; };
cudaError_t launch_bbox_batch(const BboxBatch& batch, int count, uint32_t* out7, cudaStream_t s);

// out[i] = float(M * in[i]) in double arithmetic; `in` records are `stride` bytes apart (x, y, z first).
cudaError_t launch_apply_pose(const void* in, size_t stride, int n, const double* M16, float4* out, cudaStream_t s);

cudaError_t launch_morton_keys(const float4* pts, int n, GridDev g, uint32_t* keys, uint32_t* vals, cudaStream_t s);

struct SortScratch {
  uint32_t* keys_alt;   // n
  uint32_t* vals_alt;   // n
  uint32_t* hist;       // 256 * radix_num_blocks(n)
};
int radix_num_blocks(int n);
// Stable LSD radix sort of (key, value) pairs on the low `key_bits` bits.  On return the sorted
// pairs are in *keys_out / *vals_out (one of the two buffers, chosen by pass parity).
cudaError_t launch_radix_sort(uint32_t* keys, uint32_t* vals, int n, int key_bits, SortScratch sc, uint32_t** keys_out,
                              uint32_t** vals_out, cudaStream_t s);

cudaError_t launch_gather_sorted(const float4* pts, const uint32_t* perm, int n, float4* sorted, cudaStream_t s);
// start[c] = first sorted position with key >= c, for c in [0, 1 << 3*bits].
cudaError_t launch_cell_table(const uint32_t* sorted_keys, int n, int bits, uint32_t* start, cudaStream_t s);

// ---- icp.cu --------------------------------------------------------------------------------
enum { REDUCE_P2P_VALS = 18, REDUCE_P2L_VALS = 30, REDUCE_MOM_VALS = 30, REDUCE_MAX_VALS = 32, REDUCE_BLOCKS = 592, ICP_MAX_LOG = 1024 };

// Per-iteration record kept on the device (mirrors mvr_icp_iteration of the C ABI).
struct IterRec {
  int iteration;
  int n_corr;
  double mse;
  float delta[16];
};

// Device-resident state of one align: the loop of pcl::IterativeClosestPoint::computeTransformation
// (SURVEY.md A3) advances entirely on the GPU; k_reduce_* 's last block solves for the increment,
// applies DefaultConvergenceCriteria (A8) and raises `done`, after which queued launches are no-ops.
struct IcpState {
  float delta[16];        // increment to apply at the start of the next iteration (the guess at first)
  double fin[16];         // accumulated transform, column-major
  double sums[REDUCE_MAX_VALS];
  double prev_mse, cur_mse;
  double rot_thr, trans_thr, fit_eps;   // criteria thresholds
  double ox, oy, oz;      // origin the sums are taken about
  unsigned long long queries;
  int iter, done, reason, status, n_corr;
  int max_iter, fixed, min_corr, p2l, recip, n_src;   // p2l: estimator of the solve, 0 point-to-point, 1 point-to-plane, 2 symmetric
  unsigned int ticket;    // blocks of the running reduction that have finished
  long long dbg[8];       // diagnostics: [0] clock cycles spent in the serial solve, [1] solves, [2] reciprocal searches that lost their chooser (must be 0),
                          // [3] (staged copy only) the pair's crowded word, see InitJob, [4..7] unused
  // frame bookkeeping of the static source index (pair_index.cu / pair_search.cuh)
  double cum[16];         // increments applied since the source was binned, incl. the pending `delta`, column-major
  double cinv[12];        // its affine inverse, rows {A^-1 | -A^-1 b}
  float stretch;          // >= ||A^-1||_2
  float dev;              // >= |cur - cum * s0| for every source point (s0 = its binning-time position): a bound on the rounding
                          // of the chain of in-place float transforms, advanced analytically by the solve (icp_advance_frame)
  unsigned int n_gate;    // forward matches that passed the gate in the running iteration
  double devd;            // the same bound in double
  double box[6];          // box (lo xyz, hi xyz) that held the source when it was binned
  double babs[3];         // >= |coordinate| per axis of every CURRENT source point
};

// ---- fused iteration (icp.cu) + per-align index (pair_index.cu) ---------------------------------
// grid = min(ceil(items / FUSED_THREADS), FUSED_MAX_BLOCKS): a pure function of the cloud size
enum { FUSED_THREADS = 256, FUSED_WARPS = FUSED_THREADS / 32, FUSED_MAX_BLOCKS = 148 * 8 * (256 / FUSED_THREADS) };

// Deterministic counting sort of a cloud by row-major cell (pair_index.cu): count (keys + arrival ranks; counters
// has cells + 1 zeroed entries, the last one collects non-finite points), scan, scatter into tmp in arrival
// order, rerank into ascending original index inside every cell.  A BuildJob describes one build; one launch per
// phase serves every job of a BuildBatch (blockIdx.y = job).
struct BuildJob {
  const float4* in;              // n points; M is applied first when apply != 0 (pinned float transform)
  int n, apply;
  Mat4f M;
  PairGrid g;
  uint32_t cells;                // non-finite points get the sentinel key `cells`
  uint32_t* keys;                // scratch, n
  uint32_t* rank;                // scratch, n
  uint32_t* counters;            // scratch, cells + 1, zero on entry and on exit
  unsigned long long* tiles;     // scratch of the scan: ticket word + scan_num_tiles(cells + 1) state words
  uint32_t epoch;                // of the scan (a different one per launch over the same tiles)
  int ntiles;                    // scan_num_tiles(cells + 1)
  float4* tmp;                   // scratch, n records in arrival order (ordered builds)
  float4* sorted;                // out: {point, bits(original index)} by cell
  uint32_t* start;               // out: cells + 2 entries
  uint32_t* crowded;             // nullable device word: raised (atomicMax) to the population of a cell too crowded to be ranked
  int ordered;                   // 0: the points of a cell stay in arrival order (queries: results go out by original index)
  int pad_;
};
enum { BUILD_MAX_JOBS = 48 };
struct BuildBatch { BuildJob j[BUILD_MAX_JOBS]; };
cudaError_t launch_pair_builds(const BuildBatch& batch, int count, cudaStream_t s);
int scan_num_tiles(size_t len);   // tiles of the scan over a table of len counters
// Gate mask of an index (pair_index.cu): occ and mask hold ny * nz * wstride words, wstride = ceil(nx / 32); D / Dx = dilation in
// y-z / x cells.
cudaError_t launch_gate_mask(const uint32_t* start, PairGrid g, int wstride, int D, int Dx, uint32_t* occ, uint32_t* mask, cudaStream_t s);
struct FwdArgs {
  float4* cur;             // source, sorted by binning cell, current coordinates (updated in place), .w = original index
  int n_valid;             // finite source points = sorted positions [0, n_valid)
  const float4* tgt;       // target, sorted by cell
  const uint32_t* tstart;
  PairGrid gt;
  int m_valid;
  int32_t* corr_p;         // [source sorted position] matched target sorted position, -1 none (in: last iteration's = seed)
  uint32_t* rmin;          // [target sorted position] min d2 bits over its choosers (reciprocal only; +inf bits on entry)
  double max2;             // gate, exact (PCL compares in double)
  float max_d2f;           // gate rounded up to float: bounds the search
  const uint32_t* gmask;   // nullable: gate mask of the target grid, bit x of word [(z * ny + y) * gm_stride + x / 32] =
  int gm_stride;           //   "some target point lies within the gate of cell (x, y, z)" (pair_index.cu)
  const float4* nrm;       // target normals by ORIGINAL index (point-to-plane only)
  double* partials;        // max(grid of the forward half, grid of the reverse half) x REDUCE_MAX_VALS
  IcpState* st;
  IterRec* log;
  int grid;                // blocks that work on this pair (a pure function of the cloud size): fused_grid(n_valid)
  float4* nsrc;            // source normals by SORTED position, current orientation (updated in place; symmetric only)
};
struct RevArgs {
  const float4* tgt;
  int m_valid;
  uint32_t* rmin;
  const float4* cur;
  const uint32_t* sstart;
  PairGrid gs;
  int n_valid;
  const int32_t* corr_p;
  int32_t* rnn;            // nullable: [target sorted position] sorted position of its mutual source partner, -1 none (chosen targets only)
  const float4* nrm;
  double* partials;
  IcpState* st;
  IterRec* log;
  int grid;                // fused_grid_rev(m_valid)
  int per;                 // fused_rev_chunks(m_valid): chunks of 256 target points per block (<= 4)
  const float4* nsrc;      // = FwdArgs::nsrc
};
// est: which sums the iteration accumulates over its correspondences
enum { EST_P2P = 0, EST_P2L = 1, EST_MOM = 2 /* point-to-point + second moments (LUM edge statistics) */, EST_SYM = 3 /* symmetric point-to-plane */ };
// One launch advances EVERY pair of a group by one iteration half: blockIdx.y selects the pair, blockIdx.x < grid of
// that pair does its work.  The arguments of all pairs travel by value in the kernel's parameter (constant) space, so
// indexing them by pair costs no registers.  max_grid = the largest grid of the group.
// first: first iteration of the aligns (the guess is already applied, no increment pending).
enum { FUSED_MAX_PAIRS = 24 };
struct FwdBatch { FwdArgs a[FUSED_MAX_PAIRS]; };
struct RevBatch { RevArgs a[FUSED_MAX_PAIRS]; };
// kernel parameter space (sm_70 and later, CUDA >= 12.1): 32764 bytes
static_assert(sizeof(FwdBatch) + sizeof(int) <= 32764 && sizeof(RevBatch) <= 32764, "a group's arguments must fit the kernel parameters");
// Start of a batch of aligns in one launch: per pair, corr_p <- -1 (no seed), rmin <- +inf bits (chosen by nobody; nullable),
// *st <- stage[k] (the initial states, uploaded together).  End of a batch: stage[k] <- *st (dbg[3] of the copy = the pair's
// crowded word, which is reset).  Symmetric aligns (nsrc non-null) also get their source normals by sorted position:
// nsrc[i] <- R(M) snrm[sorted[i].w] for the n_valid finite source points (the guess's rotation, pinned; curvature kept).
struct InitJob {
  int32_t* corr_p; int n; int m; uint32_t* rmin; IcpState* st; uint32_t* crowded;
  float4* nsrc; const float4* snrm; const float4* sorted; int n_valid; int pad_;
  Mat4f M;
};
struct InitBatch { InitJob j[BUILD_MAX_JOBS]; };
static_assert(sizeof(InitBatch) + sizeof(void*) <= 32764, "the batch's jobs must fit the kernel parameters");
cudaError_t launch_align_init(const InitBatch& batch, int count, const IcpState* stage, cudaStream_t s);
cudaError_t launch_align_gather(const InitBatch& batch, int count, IcpState* stage, cudaStream_t s);
int fused_grid(int items);
int fused_grid_rev(int items);   // blocks of the reverse half (not capped)
int fused_rev_chunks(int items);
cudaError_t launch_icp_forward(const FwdBatch& batch, int pairs, int max_grid, int first, bool reciprocal, int est, cudaStream_t s);
cudaError_t launch_icp_reverse(const RevBatch& batch, int pairs, int max_grid, int est, cudaStream_t s);
// Un-gated exact 1-NN of n queries in a per-align (row-major) target index.  by_w = false: results in query order;
// by_w = true: the queries were sorted by cell and carry their original index in .w, results by original index.
cudaError_t launch_pair_nn(const float4* q, int n, bool by_w, const float4* tgt_sorted, const uint32_t* tstart, PairGrid g, int m_valid,
                           int32_t* out_idx, float* out_d2, cudaStream_t s);
// The correspondences of one fused iteration by ORIGINAL source index (what launch_compact_corr consumes): for every
// finite source point (sorted position i, .w = original index) matched to target position p = corr_p[i] and, when rnn
// is given, mutual (rnn[p] == i): corr_j[orig] = original index of the target point, corr_d2[orig] = their pinned
// distance.  corr_j must be pre-filled with -1.
cudaError_t launch_resolve_pairs(const float4* src_sorted, int n_valid, const int32_t* corr_p, const int32_t* rnn, const float4* tgt_sorted,
                                 int32_t* corr_j, float* corr_d2, cudaStream_t s);
// out = float(st->fin) * in   (the aligned cloud icp.align returns)
cudaError_t launch_transform_final(const float4* in, float4* out, int n, const IcpState* st, cudaStream_t s);
// sum and count of d2[i] with idx[i] >= 0 and d2 <= max_range  (getFitnessScore); out[0]=sum, out[1]=count
cudaError_t launch_reduce_fitness(const int32_t* idx, const float* d2, int n, double max_range, double* partials,
                                  double* out, cudaStream_t s);

// Order-preserving compaction of the correspondences (ascending source index).
// scratch: uint32[compact_scratch_elems(n)].  count_out: device uint32.
size_t compact_scratch_elems(int n);
cudaError_t launch_compact_corr(const int32_t* corr_j, const float* corr_d2, int n, uint32_t* scratch, int32_t* out_q,
                                int32_t* out_m, float* out_d2, uint32_t* count_out, cudaStream_t s);

// 48-byte PointXYZRGBNormal records: position and normal through pose (index.cu k_merge_rich).
cudaError_t launch_merge_rich(const void* in48, int n, const double* M16, int full_matrix_normals, void* out48, cudaStream_t s);

// ---- cell_nn.cu ----------------------------------------------------------------------------
// Exact un-gated 1-NN of queries sorted by the cells of the target's row-major grid g (warp-cooperative; for many
// queries per target point).  d_nq_valid: device count of finite queries (they come first).  Results by original index.
cudaError_t launch_cell_nn(const float4* q_sorted, int nq, const uint32_t* d_nq_valid, const float4* tgt_sorted, const uint32_t* tstart,
                           PairGrid g, int m_valid, int32_t* out_idx, float* out_d2, cudaStream_t s);

// The same queries (sorted by the cells of g, finite ones first), one thread per query, seeded from the query's own cell or a
// neighbouring lane (cell_nn.cu).  Results by original index.
cudaError_t launch_seeded_nn(const float4* q_sorted, int nq, const uint32_t* d_nq_valid, const float4* tgt_sorted, const uint32_t* tstart,
                             PairGrid g, int m_valid, int32_t* out_idx, float* out_d2, cudaStream_t s);

// Exact un-gated 1-NN of queries in ANY order, one warp per query (small or sparse batches).  Results in query order.
cudaError_t launch_warp_nn(const float4* q, int n, const float4* tgt_sorted, const uint32_t* tstart, PairGrid g, int m_valid, int32_t* out_idx,
                           float* out_d2, cudaStream_t s);

// ---- denoise.cu ----------------------------------------------------------------------------
// Connected components of the radius graph (edge iff distance <= threshold) over an index whose cell edge is >= threshold:
// root[i] = smallest point index of i's component, count[root] = its size (n entries each, original indices); parent = scratch.
cudaError_t launch_denoise_components(const float4* sorted, const uint32_t* start, PairGrid g, int n, int n_valid, double threshold,
                                      uint32_t* parent, uint32_t* root, uint32_t* count, cudaStream_t s);
// in: keys[i] = root[i].  out: keys[i] = root of a kept point (component size >= segment_threshold), 0xffffffff of a dropped one;
// vals[i] = i; *n_noise += dropped.
cudaError_t launch_denoise_keys(const uint32_t* count, int n, uint32_t segment_threshold, uint32_t* keys, uint32_t* vals,
                                uint32_t* n_noise, cudaStream_t s);

// ---- normals.cu ----------------------------------------------------------------------------
// One cloud: sorted / start / g: a row-major index of it (pair_index.cu; the order inside a cell does not matter), n points of
// which the first n_valid sorted positions are finite.  out (n x {nx, ny, nz, curvature}) and nbr (nullable, n x k) are indexed
// by ORIGINAL point index.
struct NormalsJob {
  const float4* sorted;
  const uint32_t* start;
  PairGrid g;
  int n, n_valid;
  float3 viewpoint;
  float4* out;
  int32_t* nbr;
};
struct NormalsBatch { NormalsJob j[BUILD_MAX_JOBS]; };
// kNN(k) PCA normals of `count` (<= BUILD_MAX_JOBS) clouds in one launch, all with the same k.
cudaError_t launch_normals(const NormalsBatch& batch, int count, int k, cudaStream_t s);

// ---- score.cu -----------------------------------------------------------------------------
// One context of mvr_score_guesses_batch: samples src[s * stride] (original order, s < slots; the finite ones count), nc candidate
// transforms cand[0 .. nc), the target's per-align index (sorted / start / g, m_valid finite points) and the align's gate (max2
// exact, gate = gate_float(max_dist), scale = float(2^24 / gate)).  Out (zeroed before the launch): cost[a] and inliers[a] per
// candidate, *scored = the finite samples.
struct ScoreJob {
  const float4* src;
  int slots, stride;
  const float4* tgt;
  const uint32_t* tstart;
  PairGrid g;
  int m_valid;
  float gate, scale;
  double max2;
  const Mat4f* cand;
  unsigned long long* cost;
  uint32_t* inliers;
  uint32_t* scored;
};
enum { SCORE_MAX_CANDIDATES = 1024 };
struct ScoreBatch { ScoreJob j[BUILD_MAX_JOBS]; };
static_assert(sizeof(ScoreBatch) + sizeof(int) <= 32764, "the batch's jobs must fit the kernel parameters");
// `count` (<= BUILD_MAX_JOBS) contexts, all with nc (<= SCORE_MAX_CANDIDATES) candidates, in one launch (blockIdx.y = context).
cudaError_t launch_score(const ScoreBatch& batch, int count, int nc, cudaStream_t s);

// ---- features.cu --------------------------------------------------------------------------------
// The keypoints of a cloud: the finite points of original index s * stride (s < slots) in index order go to out[0 .. n_kp) with
// index[] = their original index; out[n_kp .. slots) = NaN, index = -1.  One block.
cudaError_t launch_keypoints(const float4* pts, int stride, int slots, float4* out, int32_t* index, cudaStream_t s);
// FPFH (33 floats per keypoint) of n keypoints from their normals and k_normals neighbour lists (n x k, keypoint indices);
// spfh: scratch, n x 33 doubles.  Two launches.
cudaError_t launch_fpfh(const float4* kp, const float4* nrm, const int32_t* nbr, int n, int k, double* spfh, float* out, cudaStream_t s);
// out[i] = nearest row of b (nb x 33) to row i of a (na x 33), exact; -1: none (all-zero rows never match).
cudaError_t launch_match(const float* a, int na, const float* b, int nb, int32_t* out, cudaStream_t s);

}  // namespace mvr
