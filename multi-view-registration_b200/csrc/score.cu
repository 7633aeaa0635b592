// score.cu -- how well each of many candidate rigid transforms puts a sampled source onto its target (mvr_score_guesses_batch).
// An opt-in extension with no reference counterpart: the ring driver scores turns about the turntable axis around each pair's
// guess and starts the pair from the best one (host/registrator.cpp, DESIGN.md section 6).
//
// Per context (blockIdx.y) and candidate a: the finite source points of original index i % stride == 0 are carried by the
// candidate's pinned float transform (the align's own, xform_pinned) and looked up in the target's static per-align index
// (pair_search.cuh, dev = 0, stretch = 1) with the align's gate.  A sample whose exact gated neighbour passes the align's
// double gate test costs floor(d2 * 2^24 / gate), at most 2^24; any other sample costs 2^24.  The sums are integers, so the
// result does not depend on the launch shape, the order of the atomics or the GPU.
#include <algorithm>

#include "launch.h"
#include "pair_search.cuh"

namespace mvr {

constexpr int SC_THREADS = PG_STRIDE;   // pg_search's segment list has one column per thread of the block
constexpr int SC_UNROLL = 6;            // loads per trip of pg_search's flat scan, as the fused iteration's searches
constexpr int SC_ITEMS = 4;             // (sample, candidate) items per thread and launch: the block's flush of its per-candidate
                                        // sums is paid once per SC_THREADS * SC_ITEMS items
// Which items the 32 lanes of a warp take: true = consecutive candidates of one sample (item f = sample * nc + candidate),
// false = consecutive samples of one candidate (f = candidate * slots + sample).  Neighbouring turns of a 1-degree grid put a
// point ~1.7 mm apart, inside one cell, so the lanes of the first layout walk nearly the same rows; consecutive samples in
// original index order are scattered over the view.  Measured in DESIGN.md section 7.
constexpr bool SC_CANDIDATE_LANES = true;

__global__ void __launch_bounds__(SC_THREADS) k_score(const __grid_constant__ ScoreBatch b, int nc) {
  __shared__ uint2 s_seg[PG_SEGS * PG_STRIDE];
  __shared__ unsigned long long s_cost[SCORE_MAX_CANDIDATES];
  __shared__ unsigned int s_in[SCORE_MAX_CANDIDATES];
  __shared__ unsigned int s_scored;
  const ScoreJob& j = b.j[blockIdx.y];
  const long long items = (long long)j.slots * nc;
  if ((long long)blockIdx.x * SC_THREADS >= items) return;   // the whole block: this context has fewer items than the launch
  for (int a = threadIdx.x; a < nc; a += SC_THREADS) { s_cost[a] = 0ull; s_in[a] = 0u; }
  if (threadIdx.x == 0) s_scored = 0u;
  __syncthreads();
  const uint32_t miss = 1u << 24;
  for (long long f = (long long)blockIdx.x * SC_THREADS + threadIdx.x; f < items; f += (long long)gridDim.x * SC_THREADS) {
    const int s = SC_CANDIDATE_LANES ? (int)(f / nc) : (int)(f % j.slots);
    const int a = SC_CANDIDATE_LANES ? (int)(f % nc) : (int)(f / j.slots);
    const float4 p = __ldg(j.src + (size_t)s * (size_t)j.stride);
    if (!finite3(p)) continue;   // not a sample
    if (a == 0) atomicAdd(&s_scored, 1u);
    const float4 q = xform_pinned(j.cand[a], p);
    uint32_t c = miss;
    if (finite3(q)) {
      NnBest nb{MVR_INF, 0x7fffffff, -1};
      pg_search<SC_UNROLL>(j.g, j.tstart, j.tgt, j.m_valid, q.x, q.y, q.z, q.x, q.y, q.z, 0.0f, 1.0f, j.gate, nb, s_seg + threadIdx.x);
      if (nb.pos >= 0 && !((double)nb.d2 > j.max2)) {   // the align's gate test
        c = min((uint32_t)floorf(__fmul_rn(nb.d2, j.scale)), miss);
        atomicAdd(&s_in[a], 1u);
      }
    }
    atomicAdd(&s_cost[a], (unsigned long long)c);
  }
  __syncthreads();
  for (int a = threadIdx.x; a < nc; a += SC_THREADS) {
    if (s_cost[a]) atomicAdd(j.cost + a, s_cost[a]);
    if (s_in[a]) atomicAdd(j.inliers + a, s_in[a]);
  }
  if (threadIdx.x == 0 && s_scored) atomicAdd(j.scored, s_scored);
}

cudaError_t launch_score(const ScoreBatch& batch, int count, int nc, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (count > BUILD_MAX_JOBS || nc < 1 || nc > SCORE_MAX_CANDIDATES) return cudaErrorInvalidValue;
  long long max_items = 0;
  for (int k = 0; k < count; ++k) max_items = std::max(max_items, (long long)batch.j[k].slots * nc);
  if (max_items <= 0) return cudaSuccess;
  const long long per_block = (long long)SC_THREADS * SC_ITEMS;
  const dim3 grid((unsigned)std::min<long long>((max_items + per_block - 1) / per_block, 65535), (unsigned)count);
  k_score<<<grid, SC_THREADS, 0, s>>>(batch, nc);
  count_launch();
  return cudaGetLastError();
}

}  // namespace mvr
