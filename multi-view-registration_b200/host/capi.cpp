// capi.cpp -- extern "C" face of the host driver (declared in include/mvr_b200.h): the entry points a
// maintainer binds under the reference's Registrator slots (INTEGRATION.md).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "registrator.h"

using namespace mvr;

struct mvr_registrator {
  Registrator* reg;
  std::string err;
};

namespace {
void fill_views(const mvr_view* in, int V, std::vector<View>& out) {
  out.resize((size_t)V);
  for (int v = 0; v < V; ++v) {
    View& o = out[(size_t)v];
    o.points = reinterpret_cast<const PointXYZ*>(in[v].xyzw);
    o.size = in[v].n;
    o.on_device = in[v].on_device != 0;
    o.view = v;
    if (in[v].init_pose) {
      std::memcpy(o.pose.m, in[v].init_pose, sizeof(o.pose.m));
      o.pose_is_identity = false;
    }
  }
}
}  // namespace

extern "C" {

void mvr_turntable_params_default(mvr_turntable_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->axis[1] = -1.0;                          // Registrator's default axis normal (mvr/src/registrator.cpp:86-87)
  mvr_icp_params_default(&p->icp);
  p->icp.use_reciprocal_correspondences = 1;  // mvr/src/registrator.cpp:552
  p->icp.max_correspondence_distance = 4.0;   // ParameterManager default (mvr/src/parameter_manager.cpp:14)
  p->icp.max_iterations = 2147483647;         // dialog default INT_MAX (:13)
  p->icp.transformation_epsilon = 0.000001;   // mvr/src/registrator.cpp:558
  p->icp.euclidean_fitness_epsilon = 64;      // :560
  p->repeat_times = 5;                        // mvr/src/parameter_manager.cpp:17
  p->mode = MVR_REGISTER_RING_PAIRS;
  p->loop_closure = 1;
  p->lum_iterations = 16;                     // mvr/src/registrator.cpp:623
  p->normal_k = 16;
}

void mvr_turntable_rotation(const double pivot[3], const double axis[3], double angle, double* out16) {
  // osg: I * translate(-pivot) * rotate(angle, axis) * translate(pivot) in row-vector order
  //  ==  T(pivot) R T(-pivot) for column vectors (mvr/src/registrator.cpp:331-342)
  double n[3] = {axis[0], axis[1], axis[2]};
  const double len = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
  for (int k = 0; k < 16; ++k) out16[k] = (k % 5 == 0) ? 1.0 : 0.0;
  if (!(len > 0)) return;
  for (int k = 0; k < 3; ++k) n[k] /= len;
  const double c = std::cos(angle), s = std::sin(angle), t = 1.0 - c;
  const double R[9] = {t * n[0] * n[0] + c,        t * n[0] * n[1] - s * n[2], t * n[0] * n[2] + s * n[1],
                       t * n[0] * n[1] + s * n[2], t * n[1] * n[1] + c,        t * n[1] * n[2] - s * n[0],
                       t * n[0] * n[2] - s * n[1], t * n[1] * n[2] + s * n[0], t * n[2] * n[2] + c};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) out16[j * 4 + i] = R[i * 3 + j];
    out16[12 + i] = pivot[i] - (R[i * 3] * pivot[0] + R[i * 3 + 1] * pivot[1] + R[i * 3 + 2] * pivot[2]);
  }
}

double mvr_turntable_view_angle(int view, int n_views) {
  // reference, 12 views: ((view < 7) ? -view : 12 - view) * pi / 6  (mvr/src/point_cloud.cpp:409)
  if (n_views <= 0) return 0.0;
  const int half = n_views / 2;
  const int k = (view <= half) ? -view : n_views - view;
  return (double)k * (2.0 * M_PI / (double)n_views);
}

int mvr_registrator_create(int device, int streams, mvr_registrator** out) {
  if (!out) return MVR_ERR_BAD_ARG;
  *out = nullptr;
  mvr_registrator* r = new (std::nothrow) mvr_registrator();
  if (!r) return MVR_ERR_ALLOC;
  r->reg = new (std::nothrow) Registrator(device, streams);
  if (!r->reg || !r->reg->ok()) {
    delete r->reg;
    delete r;
    return MVR_ERR_CUDA;
  }
  *out = r;
  return MVR_OK;
}

int mvr_registrator_destroy(mvr_registrator* r) {
  if (!r) return MVR_OK;
  delete r->reg;
  delete r;
  return MVR_OK;
}

const char* mvr_registrator_last_error(mvr_registrator* r) { return r ? r->reg->lastError().c_str() : "null registrator"; }

mvr_ctx* mvr_registrator_context(mvr_registrator* r, int slot) { return r ? r->reg->context(slot) : nullptr; }
int mvr_registrator_streams(mvr_registrator* r) { return r ? r->reg->streams() : 0; }

int mvr_pairwise_align(mvr_registrator* r, const mvr_view* source, const mvr_view* target, const mvr_icp_params* icp,
                       const float* guess, float* out_pose, mvr_icp_report* report) {
  if (!r || !source || !target || !icp) return MVR_ERR_BAD_ARG;
  std::vector<View> v;
  const mvr_view two[2] = {*source, *target};
  fill_views(two, 2, v);
  Matrix4f g;
  if (guess) std::memcpy(g.m, guess, sizeof(g.m));
  AlignResult a = r->reg->pairwiseAlign(v[0], v[1], *icp, guess ? &g : nullptr, false, 0);
  if (out_pose) std::memcpy(out_pose, a.final_transformation.m, sizeof(a.final_transformation.m));
  if (report) {
    report->iterations = a.iterations; report->converged = a.converged; report->reason = 0;
    report->n_correspondences = a.n_correspondences; report->mse = a.mse; report->gpu_ms = a.gpu_ms; report->nn_queries = a.nn_queries;
  }
  return a.status;
}

int mvr_register_turntable(mvr_registrator* r, const mvr_view* views, int n_views, const mvr_turntable_params* prm,
                           float* poses, mvr_pair_report* reports) {
  if (!r || !prm || n_views < 0 || (n_views && !views)) return MVR_ERR_BAD_ARG;
  std::vector<View> v;
  fill_views(views, n_views, v);
  Registrator& reg = *r->reg;
  reg.setPivotPoint(prm->pivot[0], prm->pivot[1], prm->pivot[2]);
  reg.setAxisNormal(prm->axis[0], prm->axis[1], prm->axis[2]);
  std::vector<mvr_pair_report> rep;
  int rc;
  if (prm->mode == MVR_REGISTER_ACCUMULATE) {
    mvr_icp_params icp = prm->icp;
    // automaticRegistration's shape: views 1..V-1 in order against the growing model, repeat_times aligns each
    rc = reg.automaticRegistration(v, icp.max_iterations, prm->repeat_times, icp.max_correspondence_distance,
                                   icp.transformation_epsilon, icp.euclidean_fitness_epsilon, &rep);
  } else if (prm->mode == MVR_REGISTER_ICP) {
    rc = reg.registrationICP(v, prm->icp.max_iterations, prm->icp.max_correspondence_distance, prm->repeat_times, &rep);
  } else if (prm->mode == MVR_REGISTER_LUM) {
    rc = reg.registrationLUM(v, prm->icp.max_iterations, prm->icp.max_correspondence_distance);
  } else {
    rc = reg.multiViewRegister(v, *prm, rep);
  }
  if (reports) for (size_t k = 0; k < rep.size(); ++k) reports[k] = rep[k];
  if (poses)
    for (int k = 0; k < n_views; ++k) {
      Matrix4f f = toFloat(v[(size_t)k].pose);
      std::memcpy(poses + 16 * k, f.m, sizeof(f.m));
    }
  return rc;
}

int mvr_registrator_get_fitness_log(mvr_registrator* r, mvr_fitness_record* out, int max_records, int* count) {
  if (!r || !count) return MVR_ERR_BAD_ARG;
  const std::vector<mvr_fitness_record>& log = r->reg->fitnessLog();
  int n = (int)log.size();
  if (out) {
    n = std::min(n, std::max(max_records, 0));
    if (n) std::memcpy(out, log.data(), (size_t)n * sizeof(mvr_fitness_record));
  }
  *count = n;
  return MVR_OK;
}

int mvr_compute_error(mvr_registrator* r, const mvr_view* views, int n_views, double max_distance, size_t* counts, double* mean_d2,
                      int* n_pairs) {
  if (!r || n_views < 0 || (n_views && !views) || !n_pairs) return MVR_ERR_BAD_ARG;
  std::vector<View> v;
  fill_views(views, n_views, v);
  for (int k = 0; k < n_views; ++k) v[(size_t)k].registered = true;   // the caller passes the registered views only
  std::vector<std::pair<size_t, double> > out;
  const int rc = r->reg->computeError(v, max_distance, out);
  *n_pairs = (int)out.size();
  for (size_t k = 0; k < out.size(); ++k) {
    if (counts) counts[k] = out[k].first;
    if (mean_d2) mean_d2[k] = out[k].second;
  }
  return rc;
}

int mvr_ring_close(const float* rel_poses, const double* weights, int n_views, int relax, int iterations, const double* centre,
                   double rot_scale, float* poses) {
  if (!rel_poses || !poses || n_views < 1) return MVR_ERR_BAD_ARG;
  std::vector<Matrix4d> rel((size_t)n_views), X;
  std::vector<double> w((size_t)n_views, 1.0);
  for (int p = 0; p < n_views; ++p) {
    Matrix4f f;
    std::memcpy(f.m, rel_poses + 16 * p, sizeof(f.m));
    rel[(size_t)p] = toDouble(f);
    if (weights) w[(size_t)p] = weights[p];
  }
  int rc = ringClose(rel, w, relax != 0, iterations > 0 ? iterations : 16, centre, rot_scale, X);
  if (rc) return rc;
  for (int p = 0; p < n_views; ++p) {
    Matrix4f f = toFloat(X[(size_t)p]);
    std::memcpy(poses + 16 * p, f.m, sizeof(f.m));
  }
  return MVR_OK;
}

int mvr_lum_relax(const mvr_pair_moments* edges, const int* src, const int* tgt, int n_edges, int n_views, int iterations,
                  double* poses) {
  if (n_edges < 0 || n_views < 1 || !poses || (n_edges && (!edges || !src || !tgt))) return MVR_ERR_BAD_ARG;
  std::vector<mvr_pair_moments> e(edges, edges + n_edges);
  std::vector<Matrix4d> X;
  int rc = lumRelax(e, src, tgt, n_views, iterations > 0 ? iterations : 16, X);
  if (rc) return rc;
  for (int v = 0; v < n_views; ++v) std::memcpy(poses + 16 * v, X[(size_t)v].m, sizeof(X[(size_t)v].m));
  return MVR_OK;
}

int mvr_lum_compute(const mvr_pair_moments* edges, const int* src, const int* tgt, int n_edges, int n_views, int iterations,
                    double convergence_threshold, double* poses6, double* transforms) {
  if (n_edges < 0 || n_views < 1 || (!poses6 && !transforms) || (n_edges && (!edges || !src || !tgt))) return MVR_ERR_BAD_ARG;
  std::vector<mvr_pair_moments> e(edges, edges + n_edges);
  std::vector<double> p6;
  std::vector<Matrix4d> X;
  const int rc = lumComputePcl(e, src, tgt, n_views, iterations > 0 ? iterations : 5, convergence_threshold, p6, X);   // PCL default: 5 sweeps
  if (rc) return rc;
  if (poses6) std::memcpy(poses6, p6.data(), (size_t)n_views * 6 * sizeof(double));
  if (transforms) for (int v = 0; v < n_views; ++v) std::memcpy(transforms + 16 * v, X[(size_t)v].m, sizeof(X[(size_t)v].m));
  return MVR_OK;
}

void mvr_pair_moments_transform(const mvr_pair_moments* in, const double* pose, const double* new_origin, mvr_pair_moments* out) {
  if (!in || !pose || !out) return;
  Matrix4d P;
  std::memcpy(P.m, pose, sizeof(P.m));
  mvr_pair_moments tmp;
  momentsTransform(*in, P, new_origin, tmp);
  *out = tmp;
}

// ---- persistence in the reference's text formats ---------------------------------------------------------------
int mvr_transformation_load(const char* path, double* pose) {
  if (!path || !pose) return MVR_ERR_BAD_ARG;
  Matrix4d m;
  if (!loadTransformation(path, m)) return MVR_ERR_NO_INPUT;
  std::memcpy(pose, m.m, sizeof(m.m));
  return MVR_OK;
}

int mvr_transformation_save(const char* path, const double* pose) {
  if (!path || !pose) return MVR_ERR_BAD_ARG;
  Matrix4d m;
  std::memcpy(m.m, pose, sizeof(m.m));
  return saveTransformation(path, m) ? MVR_OK : MVR_ERR_BAD_ARG;
}

int mvr_axis_load(const char* path, double pivot[3], double axis[3]) {
  if (!path || !pivot || !axis) return MVR_ERR_BAD_ARG;
  return loadAxis(path, pivot, axis) ? MVR_OK : MVR_ERR_NO_INPUT;
}

int mvr_axis_save(const char* path, const double pivot[3], const double axis[3]) {
  if (!path || !pivot || !axis) return MVR_ERR_BAD_ARG;
  return saveAxis(path, pivot, axis) ? MVR_OK : MVR_ERR_BAD_ARG;
}

int mvr_points_save_asc(const char* path, const void* rich_points, size_t n) {
  if (!path || (n && !rich_points)) return MVR_ERR_BAD_ARG;
  return savePointsAsc(path, rich_points, n) ? MVR_OK : MVR_ERR_BAD_ARG;
}

int mvr_refine_axis(const float* poses, int count, double pivot[3], double axis[3]) {
  if (count < 0 || (count && !poses) || !pivot || !axis) return MVR_ERR_BAD_ARG;
  std::vector<Matrix4d> P((size_t)count);
  for (int k = 0; k < count; ++k) {
    Matrix4f f;
    std::memcpy(f.m, poses + 16 * k, sizeof(f.m));
    P[(size_t)k] = toDouble(f);
  }
  return refineAxisFromPoses(P, pivot, axis);
}

}  // extern "C"
