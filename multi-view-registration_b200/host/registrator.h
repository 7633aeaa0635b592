// registrator.h -- C++ host driver of the registration path: the B200-native counterpart of the reference's
// Registrator (mvr/include/registrator.h:40-49, mvr/src/registrator.cpp) freed of Qt / OSG / PCL.
//
// Same entry points and argument meaning as the reference:
//   registrationICP(max_iterations, max_distance, repeat_times)      mvr/src/registrator.cpp:517-588
//   automaticRegistration(max_iterations, repeat_times, max_distance,
//                         transformation_epsilon, euclidean_fitness_epsilon)   :746-842, 877-990, 1008-1030
//   registrationLUM(max_iterations, max_distance)                    :611-678
//   refineAxis()                                                     :402-455
//   getRotationMatrix(angle)                                         :331-342
// plus the two calls the north star names: pairwiseAlign (one icp.align) and multiViewRegister (the ring
// of independent neighbour pairs + loop closure, the form that shards over GPUs).
//
// Types follow the reference's (mvr/include/types.h:14-50):
//   PointXYZ   = pcl::PointXYZ   (16-byte {x, y, z, pad})
//   Matrix4f   = Eigen::Matrix4f (column-major, p' = M p)
//   Matrix4d   = the double pose a view carries; the reference stores it as a row-vector osg::Matrix on the
//                scene node, PclMatrixCaster transposes between the two conventions -- here every pose is
//                column-vector / column-major, and fromOsg()/toOsg() are that transpose.
// All arithmetic on points runs on the GPU through the C ABI (include/mvr_b200.h); there is no CPU path.
#pragma once
#include <cstddef>
#include <cstdint>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mvr_b200.h"

namespace mvr {

struct PointXYZ { float x, y, z, pad; };
typedef std::vector<PointXYZ> PointCloudXYZ;

struct Matrix4f { float m[16]; };   // column-major
struct Matrix4d { double m[16]; };  // column-major

Matrix4d identity4d();
Matrix4d multiply(const Matrix4d& a, const Matrix4d& b);   // a * b
Matrix4d inverseRigid(const Matrix4d& a);
Matrix4d toDouble(const Matrix4f& a);
Matrix4f toFloat(const Matrix4d& a);
// PclMatrixCaster (mvr/include/types.h:20-50): osg row-vector matrix <-> column-vector matrix = transpose.
Matrix4d transposeOsg(const Matrix4d& a);

// One scan of the turntable sequence: the reference's PointCloud (mvr/include/point_cloud.h) reduced to what
// the registration path touches -- points, pose, registered flag, view index.
struct View {
  const PointXYZ* points = nullptr;   // sensor-frame points (host, or device when on_device)
  size_t size = 0;
  bool on_device = false;
  int view = 0;
  Matrix4d pose = identity4d();       // PointCloud::getMatrix(), column-vector convention
  bool pose_is_identity = true;
  bool registered = false;
};

struct AlignResult {
  int status = 0;
  Matrix4f final_transformation;      // icp.getFinalTransformation()
  int iterations = 0;
  int n_correspondences = 0;
  bool converged = false;
  double mse = 0, fitness = -1, gpu_ms = 0;
  double target_radius = 1.0;         // half the largest extent of the target cloud
  uint64_t nn_queries = 0;
};

class Registrator {
 public:
  // `streams` GPU contexts on `device`; independent aligns are spread over them.
  explicit Registrator(int device = 0, int streams = 1);
  ~Registrator();
  Registrator(const Registrator&) = delete;
  Registrator& operator=(const Registrator&) = delete;

  bool ok() const { return !ctx_.empty(); }
  const std::string& lastError() const { return err_; }
  int streams() const { return (int)ctx_.size(); }
  mvr_ctx* context(int slot) const { return (slot >= 0 && slot < (int)ctx_.size()) ? ctx_[(size_t)slot] : nullptr; }
  // half the largest extent of the target cloud last given to context 0 (pair 0's target = view 0 in the ring mode):
  // the length scale of the loop closure, the same whatever the sharding
  double lastTargetRadius() const { return objectRadius(0); }

  // axis.txt state (mvr/src/registrator.cpp:258-328): defaults pivot (0,0,0), normal (0,-1,0) as in :86-87.
  void setPivotPoint(double x, double y, double z) { pivot_[0] = x; pivot_[1] = y; pivot_[2] = z; }
  void setAxisNormal(double x, double y, double z) { axis_[0] = x; axis_[1] = y; axis_[2] = z; }
  const double* getPivotPoint() const { return pivot_; }
  const double* getAxisNormal() const { return axis_; }
  Matrix4d getRotationMatrix(double angle) const;
  // PointCloud::initRotation (mvr/src/point_cloud.cpp:400-413) generalised from 12 views to n_views.
  void initRotation(View& v, int n_views) const;
  bool load(const char* axis_txt);
  bool save(const char* axis_txt) const;

  // PointCloud::getTransformedPoints (mvr/src/point_cloud.cpp:290-303) on the GPU.
  int getTransformedPoints(const View& v, PointCloudXYZ& out);

  // icp.setInputSource/Target + align + getFinalTransformation (+ getFitnessScore).
  AlignResult pairwiseAlign(const View& source, const View& target, const mvr_icp_params& icp, const Matrix4f* guess,
                            bool want_fitness = false, int slot = 0);

  // Reference drivers.  `views[0]` is the fixed reference view; poses are updated in place
  // (pose <- final * pose, the column-vector form of the reference's pose * cast(final)).
  int registrationICP(std::vector<View>& views, int max_iterations, double max_distance, int repeat_times = 1,
                      std::vector<mvr_pair_report>* reports = nullptr);
  int automaticRegistration(std::vector<View>& views, int max_iterations, int repeat_times, double max_distance,
                            double transformation_epsilon, double euclidean_fitness_epsilon,
                            std::vector<mvr_pair_report>* reports = nullptr);
  int registrationLUM(std::vector<View>& views, int max_iterations, double max_distance);
  // registration(object, segment_threshold) (mvr/src/registrator.cpp:719-744): every view is denoised (PointCloud::denoise with
  // ParameterManager's triangle length, default 2.5), gets its turntable pose and counts as registered; then refineAxis.  The
  // views' buffers are the caller's: kept[v] receives the indices of view v's surviving points in the reference's output order.
  int registration(std::vector<View>& views, int segment_threshold, double triangle_length, std::vector<std::vector<int32_t> >& kept);
  // One LUM edge: reciprocal correspondences source -> target under `guess` (source in the target's frame),
  // reduced on the GPU to their moments (target frame).
  int edgeMoments(const View& source, const View& target, double max_distance, const Matrix4f& guess, int slot, mvr_pair_moments& out);
  int refineAxis(const std::vector<View>& views);
  // the fitness scores the reference logs to fitness_scores.txt (mvr/src/registrator.cpp:880-925): one per view and repeat
  const std::vector<mvr_fitness_record>& fitnessLog() const { return fitness_log_; }
  // computeError (mvr/src/registrator.cpp:466-515): reciprocal correspondences of neighbouring registered views;
  // returns per pair (count, mean squared distance).
  int computeError(std::vector<View>& views, double max_distance, std::vector<std::pair<size_t, double> >& out);

  // North-star form: ring pairs [pair_begin, pair_end) aligned independently (concurrently over the streams),
  // then (when the whole ring was computed here) chained / relaxed into absolute poses.
  int multiViewRegister(std::vector<View>& views, const mvr_turntable_params& prm, std::vector<mvr_pair_report>& reports);

 private:
  int accumulate(std::vector<View>& views, const std::vector<int>& order, const mvr_icp_params& icp, int repeat_times,
                 bool want_fitness, std::vector<mvr_pair_report>* reports, bool per_view_axis = false);
  std::vector<mvr_fitness_record> fitness_log_;   // getFitnessScore() after every repeat of the last accumulative registration
  int ensureContexts(int n);             // grow the context pool to n (batched aligns use one context per pair)
  // device pointers of the listed views: device views as given, host views uploaded once into view_cache_
  int uploadViews(const std::vector<View>& views, const std::vector<int>& which, std::vector<const float*>& dview);
  struct DeviceBuffer { void* p = nullptr; size_t cap = 0; bool ensure(size_t bytes); };
  std::vector<DeviceBuffer> view_cache_;   // device copies of host views, one upload per view and registration
  double objectRadius(int slot) const;   // half the largest extent of the target cloud last given to context `slot`
  int fail(int code, const std::string& msg) { std::lock_guard<std::mutex> g(err_mu_); err_ = msg; return code; }
  std::mutex err_mu_;
  std::vector<mvr_ctx*> ctx_;
  int device_ = 0;
  double pivot_[3] = {0, 0, 0};
  double axis_[3] = {0, -1, 0};
  std::string err_;
};

// Ring loop closure (host): see lum.cpp.
int ringClose(const std::vector<Matrix4d>& rel, const std::vector<double>& weight, bool relax, int iterations,
              const double* centre, double rot_scale, std::vector<Matrix4d>& abs_out);
// Persistence in the reference's text formats (host).
//   transformation.txt (PointCloud::load/saveTransformation, mvr/src/point_cloud.cpp:305-347): the pose of a view, four
//     lines of four "%lf " numbers; the reference writes matrix(j, i) of its row-vector osg::Matrix, i.e. the
//     column-vector matrix row by row.
//   axis.txt (Registrator::load/save, mvr/src/registrator.cpp:258-328): "px py pz\nnx ny nz\n", "%f".
//   points.asc (Registrator::saveRegisteredPoints, :385-395): "x y z r g b\n" per point, "%f %f %f %d %d %d".
bool loadTransformation(const char* path, Matrix4d& pose);
bool saveTransformation(const char* path, const Matrix4d& pose);
bool loadAxis(const char* path, double pivot[3], double axis[3]);
bool saveAxis(const char* path, const double pivot[3], const double axis[3]);
bool savePointsAsc(const char* path, const void* rich_points48, size_t n);
// LUM relaxation on correspondence moments (host): see lum.cpp.  edges[e] joins views src[e] -> tgt[e], sums in
// the common world frame; X = rigid corrections, X[0] = identity.
void momentsTransform(const mvr_pair_moments& in, const Matrix4d& pose, const double* new_origin, mvr_pair_moments& out);
// pcl::registration::LUM::compute() on moments (lum.cpp): `iterations` sweeps of PCL's linearised update, vertex 0 fixed.
// poses6: V x (x, y, z, roll, pitch, yaw); X: V transforms = lum.getTransformation(v).  Moments in ONE common frame.
int lumComputePcl(const std::vector<mvr_pair_moments>& edges, const int* src, const int* tgt, int n_views, int iterations,
                  double convergence_threshold, std::vector<double>& poses6, std::vector<Matrix4d>& X);
int lumRelax(const std::vector<mvr_pair_moments>& edges, const int* src, const int* tgt, int n_views, int iterations,
             std::vector<Matrix4d>& X);
// least squares min |A x - b| for a tall dense A (rows x cols, row-major): math_solvers::least_squares
// (mvr/src/math_solvers.cpp:24-39, LAPACK dgels there; Householder QR here).
bool leastSquares(const std::vector<double>& A, const std::vector<double>& b, int rows, int cols, std::vector<double>& x);
int refineAxisFromPoses(const std::vector<Matrix4d>& poses, double pivot[3], double axis[3]);

// mvr_estimate_normals_batch with a cloud per entry (api.cu; not part of the C ABI): which[k] (mvr_cloud) picks the target or
// the source normals of ctxs[k], kept as that cloud's normals; a context may appear once per cloud.  which = NULL: all targets.
int estimate_normals_batch(mvr_ctx* const* ctxs, const int* which, int count, int k, const float* viewpoints, float* const* out_nxyzc,
                           int* statuses);

}  // namespace mvr
