// registrator.cpp -- host orchestration of the registration path (see registrator.h).
//
// Mirrors the reference's Registrator workflows (mvr/src/registrator.cpp) with the PCL calls replaced by
// the C ABI of this library: view ordering, turntable initial guess, align, pose composition, model growth.
// Point clouds stay on the GPU between steps; only poses and reports come back to the host.
#include "registrator.h"

#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

namespace mvr {

// ---- small pose algebra ----------------------------------------------------------------------
Matrix4d identity4d() {
  Matrix4d r;
  for (int k = 0; k < 16; ++k) r.m[k] = (k % 5 == 0) ? 1.0 : 0.0;
  return r;
}

Matrix4d multiply(const Matrix4d& a, const Matrix4d& b) {
  Matrix4d r;
  for (int c = 0; c < 4; ++c)
    for (int row = 0; row < 4; ++row) {
      double s = 0;
      for (int k = 0; k < 4; ++k) s += a.m[k * 4 + row] * b.m[c * 4 + k];
      r.m[c * 4 + row] = s;
    }
  return r;
}

Matrix4d inverseRigid(const Matrix4d& a) {
  Matrix4d r = identity4d();
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) r.m[j * 4 + i] = a.m[i * 4 + j];
  for (int i = 0; i < 3; ++i) r.m[12 + i] = -(r.m[i] * a.m[12] + r.m[4 + i] * a.m[13] + r.m[8 + i] * a.m[14]);
  return r;
}

Matrix4d toDouble(const Matrix4f& a) {
  Matrix4d r;
  for (int k = 0; k < 16; ++k) r.m[k] = a.m[k];
  return r;
}

Matrix4f toFloat(const Matrix4d& a) {
  Matrix4f r;
  for (int k = 0; k < 16; ++k) r.m[k] = (float)a.m[k];
  return r;
}

Matrix4d transposeOsg(const Matrix4d& a) {
  Matrix4d r;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) r.m[j * 4 + i] = a.m[i * 4 + j];
  return r;
}

static bool isIdentity(const Matrix4d& a) {
  for (int k = 0; k < 16; ++k)
    if (a.m[k] != ((k % 5 == 0) ? 1.0 : 0.0)) return false;
  return true;
}

// ---- device scratch owned by the driver ----------------------------------------------------------
namespace {
struct DeviceCloud {
  float* p = nullptr;
  size_t cap = 0;   // points
  bool ensure(size_t n) {
    if (n <= cap) return true;
    float* q = nullptr;
    size_t want = n + n / 8 + 64;
    if (cudaMalloc((void**)&q, want * 16) != cudaSuccess) return false;
    if (p) cudaFree(p);
    p = q; cap = want;
    return true;
  }
  ~DeviceCloud() { if (p) cudaFree(p); }
};

void fill_report(mvr_pair_report& r, int src, int tgt, const AlignResult& a, int iterations, uint64_t queries, double ms,
                 const Matrix4f& pose) {
  r.source_view = src; r.target_view = tgt; r.status = a.status; r.iterations = iterations;
  r.n_correspondences = a.n_correspondences; r.mse = a.mse; r.fitness = a.fitness; r.gpu_ms = ms; r.nn_queries = queries;
  std::memcpy(r.pose, pose.m, sizeof(r.pose));
}
}  // namespace

// ---- Registrator -------------------------------------------------------------------------------------
Registrator::Registrator(int device, int streams) : device_(device) {
  if (streams < 1) streams = 1;
  for (int k = 0; k < streams; ++k) {
    mvr_ctx* c = nullptr;
    if (mvr_ctx_create(device, &c) != MVR_OK) {
      err_ = "mvr_ctx_create failed: no usable CUDA device (there is no CPU fallback)";
      for (mvr_ctx* x : ctx_) mvr_ctx_destroy(x);
      ctx_.clear();
      return;
    }
    ctx_.push_back(c);
  }
}

Registrator::~Registrator() {
  for (mvr_ctx* x : ctx_) mvr_ctx_destroy(x);
  cudaSetDevice(device_);
  for (DeviceBuffer& b : view_cache_) if (b.p) cudaFree(b.p);
}

bool Registrator::DeviceBuffer::ensure(size_t bytes) {
  if (bytes <= cap) return true;
  if (p) cudaFree(p);
  p = nullptr; cap = 0;
  const size_t want = bytes + bytes / 8 + 256;
  if (cudaMalloc(&p, want) != cudaSuccess) { p = nullptr; return false; }
  cap = want;
  return true;
}

int Registrator::ensureContexts(int n) {
  while ((int)ctx_.size() < n) {
    mvr_ctx* c = nullptr;
    if (mvr_ctx_create(device_, &c) != MVR_OK) return fail(MVR_ERR_CUDA, "mvr_ctx_create failed");
    ctx_.push_back(c);
  }
  return MVR_OK;
}

double Registrator::objectRadius(int slot) const {
  float lo[3], hi[3];
  mvr_ctx* c = context(slot);
  if (!c || mvr_get_bbox(c, MVR_CLOUD_TARGET, lo, hi) != MVR_OK) return 1.0;
  double e = 0;
  for (int k = 0; k < 3; ++k) e = std::max(e, (double)hi[k] - (double)lo[k]);
  return e > 0 ? 0.5 * e : 1.0;
}

Matrix4d Registrator::getRotationMatrix(double angle) const {
  Matrix4d r;
  mvr_turntable_rotation(pivot_, axis_, angle, r.m);
  return r;
}

void Registrator::initRotation(View& v, int n_views) const {
  if (!v.pose_is_identity && !isIdentity(v.pose)) return;   // reference: only an untouched pose gets the turntable guess
  if (v.view == 0) return;
  v.pose = getRotationMatrix(mvr_turntable_view_angle(v.view, n_views));
  v.pose_is_identity = false;
}

// ---- persistence (formats: see registrator.h) ---------------------------------------------------------------------
bool loadTransformation(const char* path, Matrix4d& pose) {
  FILE* f = std::fopen(path, "r");
  if (!f) return false;
  Matrix4d m = identity4d();
  int got = 0;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {   // file row i, column j = element (i, j) of the column-vector matrix
      double e;
      if (std::fscanf(f, "%lf", &e) == 1) { m.m[j * 4 + i] = e; ++got; }
    }
  std::fclose(f);
  if (got != 16) return false;
  pose = m;
  return true;
}

bool saveTransformation(const char* path, const Matrix4d& pose) {
  FILE* f = std::fopen(path, "w");
  if (!f) return false;
  for (int i = 0; i < 4; ++i) {
    for (int j = 0; j < 4; ++j) std::fprintf(f, "%lf ", pose.m[j * 4 + i]);
    std::fprintf(f, "\n");
  }
  return std::fclose(f) == 0;
}

bool loadAxis(const char* path, double pivot[3], double axis[3]) {
  FILE* f = std::fopen(path, "r");
  if (!f) return false;
  double v[6];
  int got = 0;
  for (int k = 0; k < 6; ++k) got += std::fscanf(f, "%lf", &v[k]) == 1;
  std::fclose(f);
  if (got != 6) return false;
  for (int k = 0; k < 3; ++k) { pivot[k] = v[k]; axis[k] = v[3 + k]; }
  return true;
}

bool saveAxis(const char* path, const double pivot[3], const double axis[3]) {
  FILE* f = std::fopen(path, "w");
  if (!f) return false;
  // the reference holds both as osg::Vec3 (float) and prints them with %f
  std::fprintf(f, "%f %f %f\n", (double)(float)pivot[0], (double)(float)pivot[1], (double)(float)pivot[2]);
  std::fprintf(f, "%f %f %f\n", (double)(float)axis[0], (double)(float)axis[1], (double)(float)axis[2]);
  return std::fclose(f) == 0;
}

bool savePointsAsc(const char* path, const void* rich_points48, size_t n) {
  FILE* f = std::fopen(path, "w");
  if (!f) return false;
  const unsigned char* p = static_cast<const unsigned char*>(rich_points48);
  for (size_t i = 0; i < n; ++i, p += 48) {
    float xyz[3];
    std::memcpy(xyz, p, sizeof(xyz));
    // pcl::PointXYZRGBNormal packs the colour as b, g, r, a at byte 32
    std::fprintf(f, "%f %f %f %d %d %d\n", xyz[0], xyz[1], xyz[2], (int)p[34], (int)p[33], (int)p[32]);
  }
  return std::fclose(f) == 0;
}

bool Registrator::load(const char* axis_txt) { return loadAxis(axis_txt, pivot_, axis_); }
bool Registrator::save(const char* axis_txt) const { return saveAxis(axis_txt, pivot_, axis_); }

int Registrator::getTransformedPoints(const View& v, PointCloudXYZ& out) {
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  out.resize(v.size);
  if (v.on_device) return fail(MVR_ERR_BAD_ARG, "getTransformedPoints: host views only (device views stay on the device)");
  int rc = mvr_apply_pose(ctx_[0], v.points, v.size, sizeof(PointXYZ), v.pose.m, v.size ? &out[0].x : nullptr);
  if (rc) err_ = mvr_last_error(ctx_[0]);
  return rc;
}

AlignResult Registrator::pairwiseAlign(const View& source, const View& target, const mvr_icp_params& icp, const Matrix4f* guess,
                                       bool want_fitness, int slot) {
  AlignResult a;
  for (int k = 0; k < 16; ++k) a.final_transformation.m[k] = (k % 5 == 0) ? 1.f : 0.f;
  if (!ok()) { a.status = MVR_ERR_CUDA; return a; }
  mvr_ctx* c = ctx_[(size_t)slot % ctx_.size()];
  int rc = target.on_device ? mvr_set_target_device(c, &target.points->x, target.size) : mvr_set_target(c, &target.points->x, target.size);
  if (!rc) rc = source.on_device ? mvr_set_source_device(c, &source.points->x, source.size) : mvr_set_source(c, &source.points->x, source.size);
  mvr_icp_report rep{};
  if (!rc) rc = mvr_icp_align(c, &icp, guess ? guess->m : nullptr, a.final_transformation.m, nullptr, &rep);
  a.status = rc;
  a.iterations = rep.iterations; a.n_correspondences = rep.n_correspondences; a.converged = rep.converged != 0;
  a.mse = rep.mse; a.gpu_ms = rep.gpu_ms; a.nn_queries = rep.nn_queries;
  a.target_radius = objectRadius((int)((size_t)slot % ctx_.size()));
  if ((rc == MVR_OK || rc == MVR_ERR_TOO_FEW_CORRESPONDENCES) && want_fitness) {
    double f = -1;
    if (mvr_fitness_score(c, DBL_MAX, &f) == MVR_OK) a.fitness = f;
  }
  if (rc && rc != MVR_ERR_TOO_FEW_CORRESPONDENCES) fail(rc, mvr_last_error(c));
  return a;
}

// The shared body of registrationICP / automaticRegistration: every view of `order` is aligned, `repeat_times`
// times, against the model accumulated so far; its pose is composed with each result; the aligned points join
// the model (mvr/src/registrator.cpp:562-577 and 909-983).
int Registrator::accumulate(std::vector<View>& views, const std::vector<int>& order, const mvr_icp_params& icp, int repeat_times,
                            bool want_fitness, std::vector<mvr_pair_report>* reports, bool per_view_axis) {
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  if (views.empty()) return MVR_OK;
  cudaSetDevice(device_);
  mvr_ctx* c = ctx_[0];
  // every copy the driver makes is ordered on the context's own (non-blocking) stream: the legacy stream
  // would not be ordered against the context's kernels
  cudaStream_t st = (cudaStream_t)mvr_ctx_get_stream(c);
  size_t total = views[0].size;
  for (int v : order) total += views[(size_t)v].size;
  DeviceCloud model, src, raw;
  if (!model.ensure(std::max<size_t>(total, 1))) return fail(MVR_ERR_ALLOC, "model buffer");
  size_t model_n = 0;
  auto upload_posed = [&](const View& v, float* dst) -> int {   // dst = getTransformedPoints(v) on the device
    if (v.size == 0) return MVR_OK;
    const float* in = &v.points->x;
    if (!v.on_device) {
      if (!raw.ensure(v.size)) return MVR_ERR_ALLOC;
      if (cudaMemcpyAsync(raw.p, in, v.size * 16, cudaMemcpyHostToDevice, st) != cudaSuccess) return MVR_ERR_CUDA;
      in = raw.p;
    }
    return mvr_apply_pose_device(c, in, v.size, 16, v.pose.m, dst);
  };
  int rc = upload_posed(views[0], model.p);
  if (rc) return fail(rc, "target upload");
  model_n = views[0].size;
  views[0].registered = true;
  if (reports) reports->clear();
  fitness_log_.clear();
  const int V = (int)views.size();
  for (int vi : order) {
    View& v = views[(size_t)vi];
    // automaticRegistration gives a view its turntable pose when its turn comes (initRotation, mvr/src/registrator.cpp:766), i.e.
    // about the axis as refined from the views registered so far (:986)
    if (per_view_axis) initRotation(v, V);
    if (!src.ensure(std::max<size_t>(v.size, 1))) return fail(MVR_ERR_ALLOC, "source buffer");
    if ((rc = upload_posed(v, src.p))) return fail(rc, "source upload");
    if ((rc = mvr_set_target_device(c, model.p, model_n))) return fail(rc, mvr_last_error(c));
    AlignResult last;
    int iterations = 0;
    uint64_t queries = 0;
    double ms = 0;
    for (int r = 0; r < std::max(repeat_times, 1); ++r) {
      // the reference aligns in place (icp_.align(*source_)): every repeat starts from the previous output
      if ((rc = mvr_set_source_device(c, src.p, v.size))) return fail(rc, mvr_last_error(c));
      mvr_icp_report rep{};
      Matrix4f fin;
      rc = mvr_icp_align(c, &icp, nullptr, fin.m, nullptr, &rep);
      if (rc && rc != MVR_ERR_TOO_FEW_CORRESPONDENCES) return fail(rc, mvr_last_error(c));
      last.status = rc; last.final_transformation = fin; last.n_correspondences = rep.n_correspondences; last.mse = rep.mse;
      iterations += rep.iterations; queries += rep.nn_queries; ms += rep.gpu_ms;
      // pose <- final * pose  (reference: setMatrix(getMatrix() * cast(final)) in row-vector order)
      v.pose = multiply(toDouble(fin), v.pose);
      v.pose_is_identity = false;
      if ((rc = mvr_copy_aligned_device(c, src.p))) return fail(rc, mvr_last_error(c));
      if (want_fitness) {
        // the reference prints / logs icp_.getFitnessScore() after EVERY repeat (mvr/src/registrator.cpp:923-925, 1015); the score
        // here is that of the aligned cloud (SURVEY.md A9 on the reference's double application of `final`)
        double f = -1;
        if (mvr_fitness_score(c, DBL_MAX, &f) == MVR_OK) { last.fitness = f; mvr_fitness_record fr{v.view, r, f}; fitness_log_.push_back(fr); }
      }
    }
    v.registered = true;
    if (per_view_axis) refineAxis(views);   // :836, 986: the axis follows every newly registered view
    // *target += transformed_source
    if (cudaMemcpyAsync(model.p + model_n * 4, src.p, v.size * 16, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return fail(MVR_ERR_CUDA, "model append");
    model_n += v.size;
    if (reports) {
      mvr_pair_report pr{};
      fill_report(pr, v.view, -1, last, iterations, queries, ms, toFloat(v.pose));
      reports->push_back(pr);
    }
  }
  return MVR_OK;
}

// View order of registrationICP (mvr/src/registrator.cpp:529-541): 1, V-1, 2, V-2, ..., then the middle view.
static std::vector<int> front_back_order(int V) {
  std::vector<int> o;
  for (int i = 1; 2 * i < V; ++i) { o.push_back(i); if (V - i != i) o.push_back(V - i); }
  if (V % 2 == 0 && V >= 2) o.push_back(V / 2);
  return o;
}

int Registrator::registrationICP(std::vector<View>& views, int max_iterations, double max_distance, int repeat_times,
                                 std::vector<mvr_pair_report>* reports) {
  const int V = (int)views.size();
  for (int v = 0; v < V; ++v) { views[(size_t)v].view = v; initRotation(views[(size_t)v], V); }
  mvr_icp_params icp;
  mvr_icp_params_default(&icp);
  icp.use_reciprocal_correspondences = 1;          // :552
  icp.max_correspondence_distance = max_distance;  // :554
  icp.max_iterations = max_iterations;             // :556
  icp.transformation_epsilon = 0.000001;           // :558
  icp.euclidean_fitness_epsilon = 64;              // :560
  int rc = MVR_OK;
  for (int r = 0; r < std::max(repeat_times, 1) && rc == MVR_OK; ++r)   // :517-524 repeats the whole pass
    rc = accumulate(views, front_back_order(V), icp, 1, false, reports);
  return rc;
}

int Registrator::automaticRegistration(std::vector<View>& views, int max_iterations, int repeat_times, double max_distance,
                                       double transformation_epsilon, double euclidean_fitness_epsilon,
                                       std::vector<mvr_pair_report>* reports) {
  // The reference collects transformation_epsilon but never applies it to icp_ (SURVEY.md App. C); kept so.
  (void)transformation_epsilon;
  const int V = (int)views.size();
  for (int v = 0; v < V; ++v) views[(size_t)v].view = v;       // initRotation when the view's turn comes (accumulate)
  mvr_icp_params icp;
  mvr_icp_params_default(&icp);
  icp.use_reciprocal_correspondences = 1;                       // :768, 901
  icp.max_correspondence_distance = max_distance;               // :769, 902
  icp.max_iterations = max_iterations;                          // :770, 903
  icp.euclidean_fitness_epsilon = euclidean_fitness_epsilon;    // :771, 904
  std::vector<int> order;
  for (int v = 1; v < V; ++v) order.push_back(v);               // views 1..V-1 against the growing model
  // What is kept of the reference's flow: every view aligned repeat_times against the model grown so far, the fitness score
  // after every repeat, refineAxis after every view (so later views start from the refined axis).  What is dropped: the
  // reference re-runs the whole prefix 1..k from scratch for every k (automaticRegistrationICP inside the while loop, :753-757,
  // O(V^2) aligns whose results the next pass overwrites) and then indexes point_clouds_ out of range (:760-766 after the
  // clear at :985); DESIGN.md section 6 lists this.
  return accumulate(views, order, icp, repeat_times, true, reports, true);
}

int Registrator::multiViewRegister(std::vector<View>& views, const mvr_turntable_params& prm, std::vector<mvr_pair_report>& reports) {
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  const int normal_k = prm.normal_k == 0 ? 16 : prm.normal_k;   // 0: a zero-filled struct gets the default
  if (normal_k < 3 || normal_k > 32) return fail(MVR_ERR_BAD_ARG, "normal_k must be in 3..32 (0: 16)");
  const int V = (int)views.size();
  reports.assign((size_t)std::max(V, 0), mvr_pair_report{});
  if (V < 2) return MVR_OK;
  for (int k = 0; k < 3; ++k) { pivot_[k] = prm.pivot[k]; axis_[k] = prm.axis[k]; }
  for (int v = 0; v < V; ++v) { views[(size_t)v].view = v; initRotation(views[(size_t)v], V); }
  int p0 = std::max(prm.pair_begin, 0), p1 = prm.pair_end <= 0 ? V : std::min(prm.pair_end, V);
  for (int p = 0; p < V; ++p) { reports[(size_t)p].source_view = (p + 1) % V; reports[(size_t)p].target_view = p; reports[(size_t)p].status = -1; reports[(size_t)p].fitness = -1; }
  // The pairs of this rank advance in lock-step: pair k lives in context k, one kernel launch per iteration half
  // serves them all (mvr_icp_align_batch).  Every distinct host view is uploaded once.
  const int P = p1 - p0;
  if (P <= 0) return MVR_OK;
  const bool timing = std::getenv("MVR_DEBUG_TIMING") != nullptr;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_begin = now();
  int rc = ensureContexts(P);
  if (rc) return rc;
  cudaSetDevice(device_);
  std::vector<double> radius((size_t)V, 1.0);
  std::vector<int> need;
  for (int k = 0; k < P; ++k) { need.push_back((p0 + k) % V); need.push_back((p0 + k + 1) % V); }
  std::vector<const float*> dview;
  if ((rc = uploadViews(views, need, dview))) return rc;
  std::vector<mvr_ctx*> cs((size_t)P);
  std::vector<float> guesses((size_t)P * 16), finals((size_t)P * 16);
  std::vector<int> st((size_t)P, 0), iterations((size_t)P, 0);
  std::vector<uint64_t> queries((size_t)P, 0);
  std::vector<double> ms((size_t)P, 0.0);
  std::vector<mvr_icp_report> rep((size_t)P);
  // every pair's target in one call: the bounding boxes of all views are measured by one launch and read back together
  std::vector<int> set_rc((size_t)P, MVR_OK);
  {
    std::vector<mvr_ctx*> cc((size_t)P);
    std::vector<int> which((size_t)P, MVR_CLOUD_TARGET);
    std::vector<const float*> ptr((size_t)P);
    std::vector<size_t> cnt((size_t)P);
    for (int k = 0; k < P; ++k) { cc[(size_t)k] = ctx_[(size_t)k]; ptr[(size_t)k] = dview[(size_t)((p0 + k) % V)]; cnt[(size_t)k] = views[(size_t)(p0 + k)].size; }
    if ((rc = mvr_set_clouds_device(cc.data(), which.data(), ptr.data(), cnt.data(), P))) return fail(rc, mvr_last_error(ctx_[0]));
  }
  for (int k = 0; k < P; ++k) {
    const int p = p0 + k;
    const View& tgt = views[(size_t)p];
    const View& src = views[(size_t)((p + 1) % V)];
    mvr_ctx* c = ctx_[(size_t)k];
    cs[(size_t)k] = c;
    if ((rc = set_rc[(size_t)k])) return fail(rc, mvr_last_error(c));
    radius[(size_t)p] = objectRadius(k);
    // initial guess: where the turntable says the source sits in the target's frame
    const Matrix4f g = toFloat(multiply(inverseRigid(tgt.pose), src.pose));
    std::memcpy(&guesses[(size_t)k * 16], g.m, sizeof(g.m));
  }
  const double t_set = now();
  // the source of pair p is the view that pair p + 1 has as its target: shared, not measured again
  std::vector<int> src_of((size_t)P);   // the context whose target is pair k's source view, if this rank has that pair (else >= P)
  for (int k = 0; k < P; ++k) {
    const int sv = (p0 + k + 1) % V;
    const int j = ((sv - p0) % V + V) % V;
    src_of[(size_t)k] = j;
    if (j < P) rc = mvr_cloud_share(ctx_[(size_t)k], MVR_CLOUD_SOURCE, ctx_[(size_t)j], MVR_CLOUD_TARGET);
    else rc = mvr_set_source_device(ctx_[(size_t)k], dview[(size_t)sv], views[(size_t)sv].size);
    if (rc) return fail(rc, mvr_last_error(ctx_[(size_t)k]));
  }
  // point-to-plane and symmetric: the target normals of every pair in one batch, each towards the origin of its view's own sensor
  // frame (PCL's default viewpoint); a pure function of the view, so pair poses do not depend on how the ring is sharded.  The
  // repeats reuse them.  Point-to-plane needs no source normals.  Symmetric: a source view that is a target here shares that
  // pair's normals; the one that is not (the last source of a pair range) is estimated in the same batch -- the same grid and
  // kernel, so the same bits as on the rank that has it as a target.
  const bool sym = prm.icp.estimator == MVR_SYMMETRIC;
  if (prm.icp.estimator == MVR_POINT_TO_PLANE || sym) {
    std::vector<mvr_ctx*> nc(cs);
    std::vector<int> nw((size_t)P, MVR_CLOUD_TARGET);
    if (sym)
      for (int k = 0; k < P; ++k)
        if (src_of[(size_t)k] >= P) { nc.push_back(cs[(size_t)k]); nw.push_back(MVR_CLOUD_SOURCE); }
    std::vector<int> nst(nc.size(), 0);
    if ((rc = estimate_normals_batch(nc.data(), nw.data(), (int)nc.size(), normal_k, nullptr, nullptr, nst.data()))) return fail(rc, mvr_last_error(cs[0]));
    for (size_t a = 0; a < nc.size(); ++a) if (nst[a]) return fail(nst[a], mvr_last_error(nc[a]));
    for (int k = 0; sym && k < P; ++k) {
      const int j = src_of[(size_t)k];
      if (j >= P || views[(size_t)((p0 + k + 1) % V)].size == 0) continue;   // an empty view has no normals; its pairs report MVR_ERR_NO_INPUT
      if ((rc = mvr_normals_share(cs[(size_t)k], MVR_CLOUD_SOURCE, cs[(size_t)j], MVR_CLOUD_TARGET))) return fail(rc, mvr_last_error(cs[(size_t)k]));
    }
  }
  const double t_share = now();
  const int repeats = std::max(prm.repeat_times, 1);
  for (int r = 0; r < repeats; ++r) {
    if ((rc = mvr_icp_align_batch(cs.data(), P, &prm.icp, guesses.data(), finals.data(), rep.data(), st.data()))) return fail(rc, mvr_last_error(cs[0]));
    bool any = false;
    for (int k = 0; k < P; ++k) {
      if (st[(size_t)k] != MVR_OK && st[(size_t)k] != MVR_ERR_TOO_FEW_CORRESPONDENCES && st[(size_t)k] != MVR_ERR_NO_INPUT)
        return fail(st[(size_t)k], mvr_last_error(cs[(size_t)k]));
      if (st[(size_t)k] == MVR_ERR_NO_INPUT) {   // an empty view: the pair keeps its guess
        std::memcpy(&finals[(size_t)k * 16], &guesses[(size_t)k * 16], 16 * sizeof(float));
        rep[(size_t)k] = mvr_icp_report{};
      }
      iterations[(size_t)k] += rep[(size_t)k].iterations; queries[(size_t)k] += rep[(size_t)k].nn_queries; ms[(size_t)k] += rep[(size_t)k].gpu_ms;
      any = true;
    }
    if (!any) break;
    guesses = finals;   // the next repeat continues from this result
  }
  for (int k = 0; k < P; ++k) {
    const int p = p0 + k;
    AlignResult a;
    a.status = st[(size_t)k];
    std::memcpy(a.final_transformation.m, &finals[(size_t)k * 16], sizeof(a.final_transformation.m));
    a.n_correspondences = rep[(size_t)k].n_correspondences; a.mse = rep[(size_t)k].mse; a.converged = rep[(size_t)k].converged != 0;
    if (prm.want_fitness && (a.status == MVR_OK || a.status == MVR_ERR_TOO_FEW_CORRESPONDENCES)) {
      double f = -1;
      if (mvr_fitness_score(cs[(size_t)k], DBL_MAX, &f) == MVR_OK) a.fitness = f;
    }
    fill_report(reports[(size_t)p], (p + 1) % V, p, a, iterations[(size_t)k], queries[(size_t)k], ms[(size_t)k], a.final_transformation);
  }
  const double t_align = now();
  if (timing) std::fprintf(stderr, "[timing] upload+set_target %.3f ms, share+normals %.3f ms, align_batch %.3f ms\n", t_set - t_begin, t_share - t_set, t_align - t_share);
  if (p0 == 0 && p1 == V) {
    std::vector<Matrix4d> rel((size_t)V), abs_pose;
    std::vector<double> w((size_t)V);
    for (int p = 0; p < V; ++p) {
      Matrix4f f;
      std::memcpy(f.m, reports[(size_t)p].pose, sizeof(f.m));
      rel[(size_t)p] = toDouble(f);
      w[(size_t)p] = reports[(size_t)p].status == MVR_OK ? (double)reports[(size_t)p].n_correspondences : 0.0;
    }
    rc = ringClose(rel, w, prm.loop_closure != 0, prm.lum_iterations > 0 ? prm.lum_iterations : 16, pivot_, radius[0], abs_pose);   // radius of view 0: the same whatever the stream count
    if (rc) return fail(rc, "loop closure failed");
    const Matrix4d base = views[0].pose;
    for (int v = 0; v < V; ++v) {
      views[(size_t)v].pose = multiply(base, abs_pose[(size_t)v]);
      views[(size_t)v].pose_is_identity = false;
      views[(size_t)v].registered = true;
    }
  }
  return MVR_OK;
}

int Registrator::edgeMoments(const View& source, const View& target, double max_distance, const Matrix4f& guess, int slot,
                             mvr_pair_moments& out) {
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  mvr_ctx* c = ctx_[(size_t)slot % ctx_.size()];
  int rc = target.on_device ? mvr_set_target_device(c, &target.points->x, target.size) : mvr_set_target(c, &target.points->x, target.size);
  if (!rc) rc = source.on_device ? mvr_set_source_device(c, &source.points->x, source.size) : mvr_set_source(c, &source.points->x, source.size);
  if (!rc) rc = mvr_pair_moments_compute(c, max_distance, 1, guess.m, &out);
  if (rc) fail(rc, mvr_last_error(c));
  return rc;
}

int Registrator::uploadViews(const std::vector<View>& views, const std::vector<int>& which, std::vector<const float*>& dview) {
  const int V = (int)views.size();
  dview.assign((size_t)V, nullptr);
  if (view_cache_.size() < (size_t)V) view_cache_.resize((size_t)V);
  cudaSetDevice(device_);
  cudaStream_t s0 = (cudaStream_t)mvr_ctx_get_stream(ctx_[0]);
  for (int v : which) {
    if (dview[(size_t)v] || views[(size_t)v].size == 0) continue;
    const View& w = views[(size_t)v];
    if (w.on_device) { dview[(size_t)v] = &w.points->x; continue; }
    DeviceBuffer& b = view_cache_[(size_t)v];
    if (!b.ensure(w.size * 16)) return fail(MVR_ERR_ALLOC, "view upload buffer");
    if (cudaMemcpyAsync(b.p, w.points, w.size * 16, cudaMemcpyHostToDevice, s0) != cudaSuccess) return fail(MVR_ERR_CUDA, "view upload");
    dview[(size_t)v] = (const float*)b.p;
  }
  if (cudaStreamSynchronize(s0) != cudaSuccess) return fail(MVR_ERR_CUDA, "view upload");
  return MVR_OK;
}

int Registrator::registrationLUM(std::vector<View>& views, int max_iterations, double max_distance) {
  // mvr/src/registrator.cpp:611-678: every view gets its turntable pose, then max(1, max_iterations / 16) outer
  // loops of { every view posed into the common frame (getTransformedPoints, :636-637), reciprocal correspondences of the
  // ring edges i -> (i + 1) % V between the POSED clouds (:640-651), lum.compute() with 16 sweeps (:630, 653),
  // pose <- lum_T * pose (:655-661) }.  The posing and the correspondences run on the GPU, every edge's pairs are reduced
  // there to their moments in one batch (edge k lives in context k; a posed view is shared between the two edges it
  // belongs to), and pcl::registration::LUM's sweeps run on those 30 doubles per edge (lumComputePcl, lum.cpp).
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  const int V = (int)views.size();
  if (V < 2) return MVR_OK;
  for (int v = 0; v < V; ++v) { views[(size_t)v].view = v; initRotation(views[(size_t)v], V); views[(size_t)v].registered = true; }
  const int lum_max_iterations = 16;
  const int outer = std::max(1, max_iterations / lum_max_iterations);
  const int E = (V == 2) ? 1 : V;   // two views: one edge, not the same pair twice
  std::vector<int> es((size_t)E), et((size_t)E);
  for (int i = 0; i < E; ++i) { es[(size_t)i] = i; et[(size_t)i] = (i + 1) % V; }
  int rc = ensureContexts(E);
  if (rc) return rc;
  std::vector<int> all;
  for (int v = 0; v < V; ++v) all.push_back(v);
  std::vector<const float*> dview;
  if ((rc = uploadViews(views, all, dview))) return rc;
  cudaSetDevice(device_);
  std::vector<DeviceCloud> posed((size_t)V);
  for (int v = 0; v < V; ++v) if (!posed[(size_t)v].ensure(std::max<size_t>(views[(size_t)v].size, 1))) return fail(MVR_ERR_ALLOC, "posed view buffer");
  std::vector<mvr_ctx*> cs((size_t)E);
  for (int i = 0; i < E; ++i) cs[(size_t)i] = ctx_[(size_t)i];
  std::vector<mvr_pair_moments> mom((size_t)E);
  std::vector<int> st((size_t)E, 0);
  for (int loop = 0; loop < outer; ++loop) {
    // transformed_cloud = getTransformedPoints(view): double math narrowed to float, in the common frame
    for (int v = 0; v < V; ++v)
      if (views[(size_t)v].size && (rc = mvr_apply_pose_device(ctx_[0], dview[(size_t)v], views[(size_t)v].size, 16, views[(size_t)v].pose.m, posed[(size_t)v].p)))
        return fail(rc, mvr_last_error(ctx_[0]));
    // edge i: target = posed view i + 1 (measured once), source = posed view i = the target of edge i - 1 (shared)
    for (int i = 0; i < E; ++i)
      if ((rc = mvr_set_target_device(cs[(size_t)i], posed[(size_t)et[(size_t)i]].p, views[(size_t)et[(size_t)i]].size))) return fail(rc, mvr_last_error(cs[(size_t)i]));
    for (int i = 0; i < E; ++i) {
      const int j = (i - 1 + E) % E;   // the edge whose target is view i
      if (E > 1 && et[(size_t)j] == es[(size_t)i]) rc = mvr_cloud_share(cs[(size_t)i], MVR_CLOUD_SOURCE, cs[(size_t)j], MVR_CLOUD_TARGET);
      else rc = mvr_set_source_device(cs[(size_t)i], posed[(size_t)es[(size_t)i]].p, views[(size_t)es[(size_t)i]].size);
      if (rc) return fail(rc, mvr_last_error(cs[(size_t)i]));
    }
    if ((rc = mvr_pair_moments_compute_batch(cs.data(), E, max_distance, 1, nullptr, mom.data(), st.data()))) return fail(rc, mvr_last_error(cs[0]));
    for (int i = 0; i < E; ++i) {
      if (st[(size_t)i] == MVR_ERR_NO_INPUT) { mom[(size_t)i] = mvr_pair_moments{}; continue; }   // an empty view: no information
      if (st[(size_t)i]) return fail(st[(size_t)i], mvr_last_error(cs[(size_t)i]));
    }
    std::vector<double> poses6;
    std::vector<Matrix4d> X;
    rc = lumComputePcl(mom, es.data(), et.data(), V, lum_max_iterations, 0.0, poses6, X);
    if (std::getenv("MVR_DEBUG_LUM")) {
      double c = 0, n = 0;
      for (const mvr_pair_moments& e : mom) { c += e.d2; n += e.n; }
      std::fprintf(stderr, "[lum] loop %d rc %d pairs %.0f mean d2 %.6f\n", loop, rc, n, n > 0 ? c / n : 0.0);
    }
    if (rc) return fail(rc, "LUM failed");
    for (int v = 0; v < V; ++v) views[(size_t)v].pose = multiply(X[(size_t)v], views[(size_t)v].pose);   // pose <- lum_T * pose
  }
  refineAxis(views);
  return MVR_OK;
}

int Registrator::registration(std::vector<View>& views, int segment_threshold, double triangle_length, std::vector<std::vector<int32_t> >& kept) {
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  const int V = (int)views.size();
  kept.assign((size_t)V, std::vector<int32_t>());
  for (int v = 0; v < V; ++v) {
    View& w = views[(size_t)v];
    w.view = v;
    if (w.on_device) return fail(MVR_ERR_BAD_ARG, "registration: host views only");
    kept[(size_t)v].resize(std::max<size_t>(w.size, 1));
    size_t cnt = 0;
    const int rc = mvr_denoise(ctx_[0], w.points, w.size, sizeof(PointXYZ), segment_threshold, triangle_length, kept[(size_t)v].data(), &cnt, nullptr);
    if (rc) return fail(rc, mvr_last_error(ctx_[0]));
    kept[(size_t)v].resize(cnt);
    initRotation(w, V);
    w.registered = true;
  }
  refineAxis(views);
  return MVR_OK;
}

int Registrator::refineAxis(const std::vector<View>& views) {
  std::vector<Matrix4d> poses;
  for (size_t i = 1; i < views.size(); ++i)
    if (views[i].registered) poses.push_back(views[i].pose);
  return refineAxisFromPoses(poses, pivot_, axis_);
}

int Registrator::computeError(std::vector<View>& views, double max_distance, std::vector<std::pair<size_t, double> >& out) {
  // mvr/src/registrator.cpp:466-515: neighbour pairs (i, i+1) and (0, V-1) of registered views
  if (!ok()) return fail(MVR_ERR_CUDA, "no GPU context");
  out.clear();
  const int V = (int)views.size();
  mvr_ctx* c = ctx_[0];
  for (int i = 0; i < V; ++i) {
    const int j = (i + 1) % V;
    if (V == 2 && i == 1) break;
    View &s = views[(size_t)i], &t = views[(size_t)j];
    if (!s.registered || !t.registered) continue;
    PointCloudXYZ ps, pt;
    int rc = getTransformedPoints(s, ps);
    if (!rc) rc = getTransformedPoints(t, pt);
    if (rc) return rc;
    if ((rc = mvr_set_source(c, ps.empty() ? nullptr : &ps[0].x, ps.size()))) return fail(rc, mvr_last_error(c));
    if ((rc = mvr_set_target(c, pt.empty() ? nullptr : &pt[0].x, pt.size()))) return fail(rc, mvr_last_error(c));
    std::vector<int32_t> q(std::max<size_t>(ps.size(), 1)), m(std::max<size_t>(ps.size(), 1));
    std::vector<float> d(std::max<size_t>(ps.size(), 1));
    size_t cnt = 0;
    if ((rc = mvr_correspondences(c, max_distance, 1, q.data(), m.data(), d.data(), &cnt))) return fail(rc, mvr_last_error(c));
    double sum = 0;
    for (size_t k = 0; k < cnt; ++k) sum += d[k];
    out.push_back(std::make_pair(cnt, cnt ? sum / (double)cnt : 0.0));
  }
  return MVR_OK;
}

}  // namespace mvr
