// global.cpp -- registration of two clouds without an initial guess (mvr_global_align): the counterpart of PCL's
// FPFHEstimation + SampleConsensusPrerejective, built on the public calls as registrator.cpp is.
//
// FPFH of both clouds' keypoints (features.cu), mutual nearest descriptors, then triples of matches drawn from a splitmix64
// stream and pre-rejected on their edge lengths on the host; each accepted triple is fitted (Umeyama, double) and every
// hypothesis is scored on the GPU by the exact integer cost of mvr_score_guesses_batch.  The deviations from PCL (seeded draws,
// mutual matches, the integer score) are in DESIGN.md section 6.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "../csrc/small_solve.h"
#include "registrator.h"

namespace {

// the same stream as synth.splitmix64(seed, counter): state seed + (counter + 1) * golden
struct SplitMix64 {
  uint64_t seed, counter = 0;
  uint64_t next() {
    uint64_t z = seed + (++counter) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  uint32_t below(uint32_t m) { return (uint32_t)(((unsigned __int128)next() * m) >> 64); }   // multiply-shift into [0, m)
};

double dist3(const float* a, const float* b) {
  const double dx = (double)a[0] - b[0], dy = (double)a[1] - b[1], dz = (double)a[2] - b[2];
  return std::sqrt(dx * dx + dy * dy + dz * dz);
}

void identity16(float* out) {
  for (int k = 0; k < 16; ++k) out[k] = (k % 5 == 0) ? 1.f : 0.f;
}

}  // namespace

extern "C" {

void mvr_global_params_default(mvr_global_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->keypoints = 4096;
  p->k = 32;
  p->max_dist = 4.0;
  p->hypotheses = 2048;
  p->max_draws = 1000000;
  p->similarity = 0.9;
  p->min_edge = 0.05;
  p->samples = 4096;
  p->seed = 0;
}

int mvr_global_align(mvr_ctx* ctx, const mvr_global_params* prm, float* out_pose, mvr_global_report* report) {
  if (!ctx || !prm || !out_pose) return MVR_ERR_BAD_ARG;
  identity16(out_pose);
  mvr_global_report rep{};
  rep.best = -1;
  if (report) *report = rep;
  if (prm->keypoints < 1 || prm->keypoints > 65536 || prm->k < 8 || prm->k > 32 || !(prm->max_dist > 0) || prm->hypotheses < 1 ||
      prm->max_draws < 1 || !(prm->similarity >= 0 && prm->similarity <= 1) || !(prm->min_edge >= 0) || prm->samples < 1 ||
      prm->samples > 65536)
    return MVR_ERR_BAD_ARG;
  cudaStream_t S = (cudaStream_t)mvr_ctx_get_stream(ctx);
  cudaEvent_t ev[4] = {};
  for (cudaEvent_t& e : ev)
    if (cudaEventCreate(&e) != cudaSuccess) { for (cudaEvent_t& f : ev) if (f) cudaEventDestroy(f); return MVR_ERR_CUDA; }
  struct Guard { cudaEvent_t* ev; ~Guard() { for (int a = 0; a < 4; ++a) cudaEventDestroy(ev[a]); } } guard{ev};

  // features of both clouds (target first), then the mutual matches
  const int K = prm->keypoints;
  std::vector<int32_t> idx(K);
  std::vector<float> xyz[2], feat[2];
  int nk[2] = {0, 0};
  cudaEventRecord(ev[0], S);
  for (int w = 0; w < 2; ++w) {
    xyz[w].resize((size_t)K * 4);
    feat[w].resize((size_t)K * 33);
    const int which = w == 0 ? MVR_CLOUD_TARGET : MVR_CLOUD_SOURCE;
    const int rc = mvr::compute_fpfh(ctx, which, K, prm->k, nullptr, idx.data(), nullptr, feat[w].data(), &nk[w], xyz[w].data());
    if (rc) return rc;
  }
  std::vector<int32_t> t2s(nk[0] + 1), s2t(nk[1] + 1);
  int rc = mvr_match_features(ctx, feat[1].data(), nk[1], feat[0].data(), nk[0], s2t.data(), t2s.data());
  if (rc) return rc;
  cudaEventRecord(ev[1], S);
  std::vector<int32_t> ms, mt;   // mutual matches in ascending source keypoint order
  for (int i = 0; i < nk[1]; ++i) {
    const int j = s2t[i];
    if (j >= 0 && t2s[j] == i) { ms.push_back(i); mt.push_back(j); }
  }
  const int M = (int)ms.size();
  rep.matches = M;
  float cudams = 0.f;
  if (cudaEventSynchronize(ev[1]) == cudaSuccess && cudaEventElapsedTime(&cudams, ev[0], ev[1]) == cudaSuccess) rep.gpu_ms = cudams;
  if (M < 3) {
    if (report) *report = rep;
    return MVR_ERR_TOO_FEW_CORRESPONDENCES;
  }

  // draws: three distinct matches; rejected when a source edge is shorter than min_edge x the source keypoints' bbox diagonal
  // or an edge-length ratio is below similarity; the rest fitted in double and narrowed to float
  const float* A = xyz[1].data();
  const float* B = xyz[0].data();
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = 0; i < nk[1]; ++i)
    for (int a = 0; a < 3; ++a) { lo[a] = std::fmin(lo[a], A[4 * i + a]); hi[a] = std::fmax(hi[a], A[4 * i + a]); }
  const double diag = std::sqrt((hi[0] - lo[0]) * (hi[0] - lo[0]) + (hi[1] - lo[1]) * (hi[1] - lo[1]) + (hi[2] - lo[2]) * (hi[2] - lo[2]));
  const double min_edge = prm->min_edge * diag;
  SplitMix64 rng{prm->seed};
  std::vector<float> hyp;
  hyp.reserve((size_t)prm->hypotheses * 16);
  int draws = 0, accepted = 0;
  while (accepted < prm->hypotheses && draws < prm->max_draws) {
    ++draws;
    int d[3];
    d[0] = (int)rng.below((uint32_t)M);
    do d[1] = (int)rng.below((uint32_t)M); while (d[1] == d[0]);
    do d[2] = (int)rng.below((uint32_t)M); while (d[2] == d[0] || d[2] == d[1]);
    bool ok = true;
    for (int e = 0; e < 3 && ok; ++e) {
      const int u = d[e], v = d[(e + 1) % 3];
      const double ea = dist3(A + 4 * ms[u], A + 4 * ms[v]), eb = dist3(B + 4 * mt[u], B + 4 * mt[v]);
      ok = ea >= min_edge && std::fmin(ea, eb) / std::fmax(ea, eb) >= prm->similarity;
    }
    if (!ok) continue;
    double mu_s[3] = {0, 0, 0}, mu_d[3] = {0, 0, 0}, Sg[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int e = 0; e < 3; ++e)
      for (int a = 0; a < 3; ++a) { mu_s[a] += A[4 * ms[d[e]] + a] / 3.0; mu_d[a] += B[4 * mt[d[e]] + a] / 3.0; }
    for (int e = 0; e < 3; ++e)
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) Sg[r * 3 + c] += (B[4 * mt[d[e]] + r] - mu_d[r]) * (A[4 * ms[d[e]] + c] - mu_s[c]) / 3.0;
    double T[16];
    mvr::umeyama_rigid(mu_s, mu_d, Sg, T);
    for (int q = 0; q < 16; ++q) hyp.push_back((float)T[q]);
    float* h = hyp.data() + hyp.size() - 16;
    h[3] = h[7] = h[11] = 0.f; h[15] = 1.f;
    ++accepted;
  }
  rep.draws = draws;
  rep.hypotheses = accepted;
  if (accepted == 0) {
    if (report) *report = rep;
    return MVR_ERR_TOO_FEW_CORRESPONDENCES;
  }

  // scores, at most SCORE_MAX_CANDIDATES (1024) per call; the lowest cost wins, ties to the lower index
  std::vector<uint64_t> cost(1024);
  std::vector<int32_t> inl(1024);
  cudaEventRecord(ev[2], S);
  for (int h0 = 0; h0 < accepted; h0 += 1024) {
    const int nc = std::min(1024, accepted - h0);
    int st = MVR_OK, scored = 0;
    rc = mvr::score_guesses_batch(&ctx, 1, hyp.data() + (size_t)h0 * 16, nc, prm->max_dist, prm->samples, cost.data(), inl.data(), &st, &scored);
    if (rc == MVR_OK) rc = st;
    if (rc) return rc;
    rep.samples = scored;
    for (int a = 0; a < nc; ++a)
      if (rep.best < 0 || cost[a] < rep.cost) { rep.best = h0 + a; rep.cost = cost[a]; rep.inliers = inl[a]; }
  }
  cudaEventRecord(ev[3], S);
  if (cudaEventSynchronize(ev[3]) == cudaSuccess && cudaEventElapsedTime(&cudams, ev[2], ev[3]) == cudaSuccess) rep.gpu_ms += cudams;
  std::memcpy(out_pose, hyp.data() + (size_t)rep.best * 16, 16 * sizeof(float));
  if (report) *report = rep;
  return MVR_OK;
}

}  // extern "C"
