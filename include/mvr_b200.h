/* mvr_b200.h -- C ABI of the B200-native ICP alignment path (libmvr_b200.so).
 *
 * The reference (fanxiaochen/Multi-View-Registration) has no FFI of its own: its registration
 * driver (mvr/src/registrator.cpp) talks to PCL classes directly.  Each entry point below names the
 * reference / PCL call it replaces (paths relative to /root/reference); INTEGRATION.md shows the
 * shim a maintainer would put under those call sites.
 *
 * Conventions (identical to the reference's PCL types):
 *   points  : array of 16-byte records {float x, y, z, pad}  == pcl::PointXYZ (mvr/include/types.h:14)
 *   poses   : float[16] column-major, column-vector convention (p' = M p) == Eigen::Matrix4f,
 *             i.e. what icp.getFinalTransformation() returns (mvr/src/registrator.cpp:573)
 *   indices : int32, -1 = "no neighbour"
 *   distances are SQUARED float32 distances computed as ((dx*dx + dy*dy) + dz*dz) without FMA,
 *   nearest-neighbour ties resolve to the LOWEST original index.
 *
 * Every function returns an mvr_status (0 = ok) and never throws.  A context is bound to one CUDA
 * device and one stream and may be used by one thread at a time.  There is NO CPU fallback: without a
 * usable CUDA device mvr_ctx_create fails with MVR_ERR_CUDA.
 */
#ifndef MVR_B200_H
#define MVR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mvr_ctx mvr_ctx;

typedef enum {
  MVR_OK = 0,
  MVR_ERR_BAD_ARG = 1,
  MVR_ERR_TOO_FEW_CORRESPONDENCES = 2, /* < min_correspondences (PCL: "Not enough correspondences") */
  MVR_ERR_CUDA = 3,
  MVR_ERR_NO_INPUT = 4,                /* target/source not set */
  MVR_ERR_NOT_SPD = 5,                 /* point-to-plane normal equations not positive definite */
  MVR_ERR_ALLOC = 6,
  MVR_ERR_NCCL = 7                     /* NCCL missing or a collective failed (multi-GPU entry points) */
} mvr_status;

typedef enum { MVR_CLOUD_TARGET = 0, MVR_CLOUD_SOURCE = 1 } mvr_cloud;
/* SYMMETRIC: pcl::IterativeClosestPointWithNormals with setUseSymmetricObjective(true), i.e.
 * TransformationEstimationSymmetricPointToPlaneLLS (PCL >= 1.11) with enforce_same_direction_normals: needs target AND source
 * normals; the source normals move with the source.  (Other values mean point-to-point.) */
typedef enum { MVR_POINT_TO_POINT = 0, MVR_POINT_TO_PLANE = 1, MVR_SYMMETRIC = 2 } mvr_estimator;
typedef enum {
  MVR_REASON_NONE = 0,
  MVR_REASON_ITERATIONS = 1,
  MVR_REASON_TRANSFORM = 2,
  MVR_REASON_ABS_MSE = 3,
  MVR_REASON_REL_MSE = 4,
  MVR_REASON_NO_CORRESPONDENCES = 5
} mvr_reason;

/* The setters the reference calls on pcl::IterativeClosestPoint (mvr/src/registrator.cpp:551-560,
 * 768-771, 901-904).  mvr_icp_params_default() fills in PCL's own defaults. */
typedef struct {
  int max_iterations;                  /* setMaximumIterations          (PCL default 10)            */
  double max_correspondence_distance;  /* setMaxCorrespondenceDistance  (PCL default sqrt(DBL_MAX)) */
  double transformation_epsilon;       /* setTransformationEpsilon      (PCL default 0)             */
  double euclidean_fitness_epsilon;    /* setEuclideanFitnessEpsilon    (PCL default -DBL_MAX)      */
  int use_reciprocal_correspondences;  /* setUseReciprocalCorrespondences (reference: true)         */
  int estimator;                       /* mvr_estimator; the reference only uses point-to-point (point-to-plane needs
                                          target normals, symmetric needs target and source normals) */
  int fixed_iterations;                /* 1: run exactly max_iterations (bench mode, criteria 2-4 off) */
  int min_correspondences;             /* PCL min_number_correspondences_ = 3                       */
} mvr_icp_params;

typedef struct {
  int iterations;
  int converged;          /* hasConverged() */
  int reason;             /* mvr_reason */
  int n_correspondences;  /* size of the last correspondence set */
  double mse;             /* mean squared distance of the last correspondence set */
  double gpu_ms;          /* device time of the align (CUDA events on the context stream); in a batch: the batch's time / its pairs */
  uint64_t nn_queries;    /* nearest-neighbour queries answered (forward + reciprocal) */
} mvr_icp_report;

typedef struct {
  int iteration;          /* 1-based */
  int n_correspondences;
  double mse;
  float delta[16];        /* the float32 increment applied to the source in this iteration */
} mvr_icp_iteration;

/* Geometry of a uniform-grid index: cell c_a = clamp(floor((p_a - origin_a) * inv_cell), 0, 2^bits-1),
 * key = Morton interleave (x bit 0, y bit 1, z bit 2) of the three cell coordinates. */
typedef struct {
  float origin[3];
  float inv_cell;
  float cell;
  int bits;
} mvr_grid;

/* Per-kernel device timing accumulated while mvr_ctx_set_profiling(ctx, 1) is on. */
typedef struct {
  uint64_t launches;
  double ms;       /* sum of CUDA-event durations */
  double bytes;    /* algorithmic bytes (DESIGN.md section 4) summed over those launches */
  double units;    /* queries / points processed */
} mvr_kernel_stat;

enum { MVR_K_MORTON = 0, MVR_K_SORT = 1, MVR_K_TABLE = 2, MVR_K_NN = 3, MVR_K_CORR = 4, MVR_K_REDUCE = 5,
       MVR_K_TRANSFORM = 6, MVR_K_NORMALS = 7, MVR_K_COUNT = 8 };

const char* mvr_version(void);
/* Number of CUDA kernels this library has launched in the calling process (all contexts). */
uint64_t mvr_kernel_launch_count(void);
/* Bytes an align moves between host and device besides the clouds: the per-align loop state (copied in once, read back
 * once per batch of iterations) and one per-iteration log record (read back after the align). */
void mvr_transfer_sizes(size_t* state_bytes, size_t* log_record_bytes);
const char* mvr_status_string(int status);
void mvr_icp_params_default(mvr_icp_params* p);

/* -- context ---------------------------------------------------------------------------------- */
int mvr_ctx_create(int device, mvr_ctx** out);
int mvr_ctx_destroy(mvr_ctx* ctx);
/* Run on a caller-owned stream (e.g. torch's current stream) instead of the context's own. */
int mvr_ctx_set_stream(mvr_ctx* ctx, void* cuda_stream);
int mvr_ctx_synchronize(mvr_ctx* ctx);
/* The CUDA stream (cudaStream_t) the context enqueues on: callers that move data themselves order it here. */
void* mvr_ctx_get_stream(mvr_ctx* ctx);
const char* mvr_last_error(mvr_ctx* ctx);
int mvr_ctx_set_profiling(mvr_ctx* ctx, int on);
int mvr_ctx_get_kernel_stats(mvr_ctx* ctx, mvr_kernel_stat* out /* [MVR_K_COUNT] */, int reset);
/* Diagnostics of the last align (development aid): k = 0 clock cycles in the serial per-iteration solve, 1 solves, 2 reciprocal
 * searches that lost their chooser (must be 0), 8 population of a grid cell too crowded to be ordered (0: none; mvr_last_error then
 * carries a warning: thousands of duplicated or invalid points on one spot make the index build and the search crawl). */
double mvr_debug_value(mvr_ctx* ctx, int k);
/* Tuning knobs of the spatial index: cell edge (<= 0: automatic) and maximum bits per axis (1..10). */
int mvr_ctx_set_index_options(mvr_ctx* ctx, float cell_edge, int max_bits);

/* Tuning of mvr_nn_query / mvr_fitness_score: large batches are sorted by the cells of a target grid with about
 * `points_per_cell` target points per occupied cell (default 8).  dense_ratio is kept for compatibility (unused).
 * Results do not depend on either. */
int mvr_ctx_set_nn_options(mvr_ctx* ctx, double points_per_cell, double dense_ratio);
/* Which kernel answers mvr_nn_query / mvr_fitness_score (results are identical; a tuning and A/B aid):
 * AUTO = one warp per query up to 131072 queries, the per-thread row walk up to 262144, above that the queries are sorted by
 * cell and every query is seeded from its own cell (SEEDED); WARP / THREAD / CELL / SEEDED force one of them (CELL: the
 * cell-cooperative scan of whole 27-cell neighbourhoods). */
typedef enum { MVR_NN_AUTO = 0, MVR_NN_WARP = 1, MVR_NN_THREAD = 2, MVR_NN_CELL = 3, MVR_NN_SEEDED = 4 } mvr_nn_mode;
int mvr_ctx_set_nn_mode(mvr_ctx* ctx, int mode);
/* Gate mask of the target index (default off): one bit per grid cell, "some target point lies within the gate of this cell".
 * With it a source point without a partner inside the gate is settled by one load instead of a gate-wide search; worth its
 * build time (two small kernels per target) when a large part of the source has no partner.  Results are identical. */
int mvr_ctx_set_gate_mask(mvr_ctx* ctx, int on);

/* -- inputs: icp.setInputTarget / icp.setInputSource (mvr/src/registrator.cpp:566-567, 776-777,
 *    913-914) and CorrespondenceEstimation::setInputSource/Target (:497-498, 645-646).
 *    Host variants copy n*16 bytes to the device; *_device variants adopt a device pointer that the
 *    caller keeps alive (no copy).  The target's grid index is built lazily by the first consumer. */
int mvr_set_target(mvr_ctx* ctx, const float* xyzw, size_t n);
int mvr_set_source(mvr_ctx* ctx, const float* xyzw, size_t n);
int mvr_set_target_device(mvr_ctx* ctx, const float* d_xyzw, size_t n);
int mvr_set_source_device(mvr_ctx* ctx, const float* d_xyzw, size_t n);
/* `count` device clouds at once (contexts of one device; which[k]: mvr_cloud): the same as mvr_set_target_device /
 * mvr_set_source_device per cloud, but every bounding box is measured by one launch and read back by one copy. */
int mvr_set_clouds_device(mvr_ctx* const* ctxs, const int* which, const float* const* d_xyzw, const size_t* n, int count);
/* Give `dst` the cloud another context of the same device already holds (same device pointer, same bounding box:
 * nothing is copied or recomputed).  The points must stay alive and unchanged while `dst` uses them -- a view of a
 * turntable ring is the target of one pair and the source of the next. */
int mvr_cloud_share(mvr_ctx* dst, int which_dst /* mvr_cloud */, mvr_ctx* src, int which_src);
/* Optional per-target-point normals (n x {nx,ny,nz,curvature}) for point-to-plane ICP.  A new target drops them. */
int mvr_set_target_normals(mvr_ctx* ctx, const float* nxyzc, size_t n);
/* The same for the source (symmetric ICP): n must equal the source size.  A new source drops them; during an align they turn
 * with the source (the guess's rotation at its start, each increment's rotation after), on a copy -- these stay as given. */
int mvr_set_source_normals(mvr_ctx* ctx, const float* nxyzc, size_t n);
/* Give `dst` the normals another context of the same device holds for its target or source (same device pointer, nothing
 * copied), like mvr_cloud_share: `src` must keep them alive and unchanged while `dst` uses them.  The two clouds must have
 * the same number of points (else MVR_ERR_BAD_ARG); MVR_ERR_NO_INPUT if `src` holds no such normals.  A ring view is the
 * target of one pair and the source of the next: its normals are estimated once. */
int mvr_normals_share(mvr_ctx* dst, int which_dst /* mvr_cloud */, mvr_ctx* src, int which_src);

/* -- spatial index (replaces pcl::KdTreeFLANN::setInputCloud inside icp.align) ------------------- */
/* Build the Morton-sorted uniform grid over a cloud with an explicit grid; exported for parity tests. */
int mvr_index_build(mvr_ctx* ctx, int which /* mvr_cloud */, const mvr_grid* grid /* NULL: automatic */);
/* Copy out the index: sorted keys (n), permutation perm[sorted position] = original index (n),
 * cell_start ((1 << 3*bits) + 1 entries).  Any pointer may be NULL. */
int mvr_index_export(mvr_ctx* ctx, int which, mvr_grid* grid, uint32_t* sorted_keys, int32_t* perm,
                     uint32_t* cell_start);

/* -- queries ---------------------------------------------------------------------------------- */
/* Exact un-gated 1-NN of n query points in the target: pcl::KdTreeFLANN::nearestKSearch(k=1). */
int mvr_nn_query(mvr_ctx* ctx, const float* q_xyzw, size_t n, int32_t* idx, float* d2);
int mvr_nn_query_device(mvr_ctx* ctx, const float* d_q_xyzw, size_t n, int32_t* d_idx, float* d_d2);

/* CorrespondenceEstimation::determineCorrespondences / determineReciprocalCorrespondences
 * (mvr/src/registrator.cpp:502, 649): source -> target, gate d2 <= max_dist^2, output compacted in
 * ascending source index.  Arrays must hold source-size entries. */
int mvr_correspondences(mvr_ctx* ctx, double max_dist, int reciprocal, int32_t* index_query, int32_t* index_match,
                        float* distance, size_t* count);

/* -- ICP: icp.align(output, guess) + getFinalTransformation (mvr/src/registrator.cpp:569-573, 920-921,
 *    1012-1013).  guess may be NULL (identity).  out_xyzw (nullable, may alias the source host buffer)
 *    receives transform(source, final).  Returns MVR_ERR_TOO_FEW_CORRESPONDENCES when PCL would have
 *    logged "Not enough correspondences"; out_pose then holds the transform accumulated so far. */
int mvr_icp_align(mvr_ctx* ctx, const mvr_icp_params* params, const float* guess, float* out_pose, float* out_xyzw,
                  mvr_icp_report* report);
/* `count` aligns in lock-step: context k holds pair k's source and target, every pair advances one iteration per
 * kernel launch (one launch serves a group of pairs -- a single scan pair does not fill a B200; the groups of a batch,
 * by default a quarter of it each, run concurrently on the streams of their first contexts).  Results are those of
 * `count` separate mvr_icp_align calls, bit for bit, whatever the grouping.  guesses: count x float[16] (nullable:
 * identities), out_poses: count x float[16], statuses: count x mvr_status of the individual aligns; the return value
 * reports batch-level failures.  All contexts must live on one device.  Afterwards every context answers
 * mvr_icp_get_iterations, mvr_fitness_score and mvr_copy_aligned_device for its own align (the log is fetched and the
 * aligned cloud computed at that moment). */
int mvr_icp_align_batch(mvr_ctx* const* ctxs, int count, const mvr_icp_params* params, const float* guesses, float* out_poses,
                        mvr_icp_report* reports, int* statuses);
/* Pairs per kernel launch of the batches this context leads (1..24; 0 = automatic, the default: a quarter of the batch).  The
 * pairs of a group advance in lock-step, one launch per iteration half; the groups of a batch run concurrently, each on the
 * stream of its first context.  Results do not depend on the grouping. */
int mvr_ctx_set_batch_group(mvr_ctx* ctx, int pairs);
/* Per-iteration records of the last align (n_correspondences, mse, delta). */
int mvr_icp_get_iterations(mvr_ctx* ctx, mvr_icp_iteration* out, int max_records, int* count);
/* Registration::getFitnessScore(max_range) (mvr/src/registrator.cpp:572, 923, 1015): mean squared
 * un-gated NN distance of the last align's output cloud (or of the source if no align ran). */
int mvr_fitness_score(mvr_ctx* ctx, double max_range, double* score);

/* -- edge statistics of the LUM relaxation: what pcl::registration::LUM::computeEdge derives from the
 *    correspondences the reference hands it (lum.setCorrespondences, mvr/src/registrator.cpp:640-651).
 *    One correspondence pass source -> target (guess applied to the source first), gate d2 <= max_dist^2,
 *    reciprocal or not; over the kept pairs (a = posed source point, b = target point), about `origin`:
 *    every quantity a rigid least-squares cost  sum |X_a a - X_b b|^2  needs, for ANY rigid X_a, X_b. */
typedef struct {
  double n;               /* number of correspondences (0: the edge carries no information) */
  double origin[3];       /* the sums below are over a - origin, b - origin (target frame) */
  double sa[3], sb[3];    /* sum a, sum b */
  double sba[9];          /* sum b a^T, row-major (row = component of b) */
  double saa[6], sbb[6];  /* sum a a^T, sum b b^T: xx xy xz yy yz zz */
  double d2;              /* sum of the float32 squared distances */
} mvr_pair_moments;
int mvr_pair_moments_compute(mvr_ctx* ctx, double max_dist, int reciprocal, const float* guess, mvr_pair_moments* out);

/* The edges of a whole pose graph at once: context k holds edge k's source and target; one launch per search half
 * serves a group of edges (like mvr_icp_align_batch).  statuses[k] = 0 also for an edge without correspondences
 * (out[k].n = 0). */
int mvr_pair_moments_compute_batch(mvr_ctx* const* ctxs, int count, double max_dist, int reciprocal, const float* guesses,
                                   mvr_pair_moments* out, int* statuses);

/* -- extensions named by the north star (no reference call site) -------------------------------- */
/* pcl::NormalEstimation semantics: kNN(k) PCA normals of a cloud, flipped towards viewpoint.
 * out: n x {nx, ny, nz, curvature}.  neighbours (nullable): n x k int32, ascending (d2, index).  The result is also kept on the
 * device as the cloud's normals (target: point-to-plane and symmetric ICP; source: symmetric ICP). */
int mvr_estimate_normals(mvr_ctx* ctx, int which, int k, const float viewpoint[3], float* out_nxyzc,
                         int32_t* neighbours);
/* kNN(k) PCA normals of the TARGET cloud of `count` contexts of one device, as mvr_estimate_normals computes them (same
 * bits), kept on the device as each context's target normals (what point-to-plane ICP reads).  All indices are built by
 * one set of build launches and all normals by one launch per 48 contexts, on the first context's stream; every context's
 * later work is ordered after its normals.  viewpoints: count x 3 (NULL: the origin of every target's frame).  out_nxyzc
 * (nullable, entries nullable): host copies, n x {nx, ny, nz, curvature}.  statuses[k]: MVR_ERR_NO_INPUT if context k has
 * no target; an empty target is MVR_OK with nothing to do.  No context may appear twice; k in 3..32. */
int mvr_estimate_normals_batch(mvr_ctx* const* ctxs, int count, int k, const float* viewpoints, float* const* out_nxyzc,
                               int* statuses);
/* Score n_candidates rigid transforms of each context's source against its target (device of ctxs[0]).
 * candidates: count x n_candidates x float[16] column-major; costs: count x n_candidates; inliers nullable.
 * samples: 1..65536; n_candidates: 1..1024.  statuses[k]: MVR_ERR_NO_INPUT without source/target;
 * an empty source or target scores samples x 2^24 / 0 (no error).
 * The samples are the finite source points of original index i % stride == 0, stride = max(1, ceil(n / samples)), the same for
 * every candidate.  Each is moved by the candidate's float transform (the one an align applies to its guess) and its exact
 * nearest target point within the gate max_dist is looked up; it costs floor(d2 * 2^24 / g), at most 2^24, when that neighbour
 * passes the align's gate test (d2 <= max_dist^2, g = the gate as a float rounded up), 2^24 otherwise.  costs = the sum over the
 * samples, inliers = the samples within the gate: integers, exact whatever the GPU.  Each context's target index is the one an
 * align with the same max_dist uses: that align does not build it again, and a second call on unchanged targets builds none.
 * No context may appear twice; the call returns when the results are on the host. */
int mvr_score_guesses_batch(mvr_ctx* const* ctxs, int count, const float* candidates, int n_candidates, double max_dist, int samples,
                            uint64_t* costs, int32_t* inliers, int* statuses);

/* -- global registration without an initial guess (pcl::FPFHEstimation + pcl::SampleConsensusPrerejective) ------------ */
/* FPFH descriptors of a cloud's keypoints: the finite points of original index i % stride == 0, stride = max(1, ceil(n /
 * keypoints)), in index order (at most `keypoints` of them).  Their kNN(k) PCA normals and neighbour lists are those
 * mvr_estimate_normals gives for the keypoints set as a cloud of their own (same bits), flipped towards viewpoint (NULL: the
 * centre of the cloud's bounding box, (lo + hi) * 0.5f); they do not replace the cloud's normals.  Per keypoint, over the first
 * k - 1 entries of its list that are not itself: PCL's pair features in double, 11 bins each, every pair adding 100 / (k - 1)
 * (SPFH); then FPFH = SPFH + the neighbours' SPFH weighted by 1 / d2, each sub-histogram of that sum scaled to 100, narrowed
 * to float.  A keypoint whose normal is not finite gets an all-zero descriptor (it never matches).  index: keypoints int32
 * (original indices), nxyzc (nullable): keypoints x 4, features: keypoints x 33; *n_kp = the keypoints found.
 * keypoints: 1..65536, k: 8..32.  MVR_ERR_NO_INPUT if the cloud is not set; an empty cloud gives *n_kp = 0. */
int mvr_compute_fpfh(mvr_ctx* ctx, int which /* mvr_cloud */, int keypoints, int k, const float viewpoint[3], int32_t* index, float* nxyzc,
                     float* features, int* n_kp);
/* Exact nearest descriptor (33 floats per row, host arrays) both ways: a_to_b[i] = the row of b nearest to row i of a in squared
 * L2 summed over bins 0..32 in order without FMA, ties to the lowest row; b_to_a likewise.  All-zero rows never match (-1). */
int mvr_match_features(mvr_ctx* ctx, const float* a, int na, const float* b, int nb, int32_t* a_to_b, int32_t* b_to_a);
typedef struct {
  int keypoints;        /* per cloud, 1..65536 (4096) */
  int k;                /* neighbours of the normals and features, 8..32 (32) */
  double max_dist;      /* gate of the hypothesis score, > 0 (4) */
  int hypotheses;       /* accepted hypotheses to score, >= 1 (2048) */
  int max_draws;        /* draws before giving up, >= 1 (1000000) */
  double similarity;    /* edge-length similarity of a draw, 0..1 (0.9) */
  double min_edge;      /* shortest source edge of a draw, as a fraction of the source keypoints' bbox diagonal (0.05) */
  int samples;          /* source points per score, 1..65536 (4096) */
  uint64_t seed;        /* of the draws' splitmix64 stream (0) */
} mvr_global_params;
typedef struct {
  int matches;          /* mutual feature matches */
  int draws;            /* triples drawn */
  int hypotheses;       /* triples accepted and scored */
  int best;             /* index of the best hypothesis (-1: none) */
  uint64_t cost;        /* its mvr_score_guesses_batch cost */
  int inliers;          /* its samples within max_dist */
  int samples;          /* the source samples scored */
  double gpu_ms;        /* device time of the features, the matching and the scoring (CUDA events on the context's stream) */
} mvr_global_report;
void mvr_global_params_default(mvr_global_params* p);
/* The rigid pose (float[16] column-major) that maps the context's source onto its target, with no initial guess: FPFH of both
 * clouds, mutual matches, triples of matches drawn from a splitmix64 stream of `seed` (a draw is rejected when a source edge is
 * shorter than min_edge or an edge-length ratio is below similarity), each accepted triple fitted rigidly (Umeyama, double,
 * narrowed to float), every hypothesis scored by mvr_score_guesses_batch(max_dist, samples); the lowest cost wins (ties: the
 * lower index).  A pure function of the two clouds and the parameters.  Fewer than 3 mutual matches or no accepted draw:
 * MVR_ERR_TOO_FEW_CORRESPONDENCES with out_pose = identity.  Refine with mvr_icp_align from out_pose: the context serves it
 * as before (an align with the same max_dist reuses the scorer's target index). */
int mvr_global_align(mvr_ctx* ctx, const mvr_global_params* params, float* out_pose, mvr_global_report* report);

/* -- pose application: PointCloud::getTransformedPoints (mvr/src/point_cloud.cpp:290-303) ------------
 * out[i] = {float(pose * p_i), 1}: the multiply runs in double (osg::Matrix is double) and is narrowed to
 * float, RGB / normal lanes are dropped.  in: n records of `stride_bytes` bytes whose first three floats
 * are x, y, z (16 for PointXYZ, 48 for PointXYZRGBNormal).  pose: double[16] column-major, p' = M p (the
 * transpose of the reference's row-vector osg::Matrix, see PclMatrixCaster mvr/include/types.h:20-50). */
int mvr_apply_pose(mvr_ctx* ctx, const void* points, size_t n, size_t stride_bytes, const double* pose, float* out_xyzw);
/* Same with device pointers on both sides (returns after the work has completed). */
int mvr_apply_pose_device(mvr_ctx* ctx, const void* d_points, size_t n, size_t stride_bytes, const double* pose, float* d_out_xyzw);
/* Copy transform(source, final) of the last mvr_icp_align into a device buffer of source-size points
 * (the reference grows its model with it: *target += transformed_source, mvr/src/registrator.cpp:576). */
int mvr_copy_aligned_device(mvr_ctx* ctx, float* d_out_xyzw);

/* -- registration driver: the reference's Registrator entry points (mvr/include/registrator.h:40-49) -- */
typedef struct mvr_registrator mvr_registrator;

typedef struct {
  const float* xyzw;       /* n PointXYZ records in the view's own sensor frame */
  size_t n;
  int on_device;           /* non-zero: xyzw is a device pointer on the registrator's device */
  const double* init_pose; /* nullable double[16] column-major initial pose of the view in view 0's frame;
                              NULL = PointCloud::initRotation: ideal turntable rotation of view index v */
} mvr_view;

typedef enum {
  MVR_REGISTER_RING_PAIRS = 0,  /* independent neighbour pairs (v+1 -> v, closing pair 0 -> V-1), then loop closure:
                                   the shardable form (ring edges of registrationLUM, mvr/src/registrator.cpp:640-651).
                                   The only mode that honours icp.estimator (point-to-plane and symmetric: see normal_k); the
                                   others build their own point-to-point settings, as the reference does */
  MVR_REGISTER_ACCUMULATE = 1,  /* automaticRegistration: views 1..V-1 in order, each aligned repeat_times against
                                   the growing model, then refineAxis (mvr/src/registrator.cpp:746-842, 877-990) */
  MVR_REGISTER_ICP = 2,         /* registrationICP: views in the order 1, V-1, 2, V-2, .. against the growing model,
                                   the whole pass repeated repeat_times (mvr/src/registrator.cpp:517-588) */
  MVR_REGISTER_LUM = 3          /* registrationLUM: max(1, max_iterations / 16) outer loops of { pose every view, reciprocal
                                   correspondences of the ring edges, 16 sweeps of pcl::registration::LUM (mvr_lum_compute),
                                   pose <- T pose } (mvr/src/registrator.cpp:611-678) */
} mvr_register_mode;

typedef struct {
  double pivot[3];         /* turntable axis: Registrator::getPivotPoint / getAxisNormal (axis.txt) */
  double axis[3];
  mvr_icp_params icp;      /* per-align settings (reference: reciprocal, max_dist 4, transEps 1e-6, fitEps 64) */
  int repeat_times;        /* aligns per view/pair, each starting from the previous result (reference default 5) */
  int mode;                /* mvr_register_mode */
  int loop_closure;        /* ring mode: 0 = chain the pair poses, 1 = relax the ring (host, after the gather) */
  int lum_iterations;      /* relaxation sweeps (reference lum.setMaxIterations(16)) */
  int pair_begin, pair_end;/* ring mode: compute only pairs [begin, end) (multi-GPU sharding); end <= 0 = all V */
  int want_fitness;        /* also run getFitnessScore() after the last align of each pair/view */
  int normal_k;            /* ring mode with icp.estimator = MVR_POINT_TO_PLANE or MVR_SYMMETRIC: neighbours of the normals,
                              3..32 (0 = the default, 16).  Each pair's target normals are estimated on the GPU (all pairs in
                              one batch, mvr_estimate_normals_batch) in the view's own sensor frame, i.e. towards its origin.
                              Symmetric: each pair's source normals are those of the pair that has the same view as its target
                              (mvr_normals_share); the last source of a pair range is estimated in the same batch. */
} mvr_turntable_params;

typedef struct {
  int source_view, target_view;  /* target_view = -1: the accumulated model */
  int status;                    /* mvr_status of the (last) align */
  int iterations;                /* summed over the repeats */
  int n_correspondences;
  double mse;
  double fitness;                /* getFitnessScore() if requested, else -1 */
  double gpu_ms;
  uint64_t nn_queries;
  float pose[16];                /* ring mode: relative pose source -> target frame; accumulate: view -> model frame */
} mvr_pair_report;

/* One line of the reference's fitness_scores.txt (mvr/src/registrator.cpp:880-925): getFitnessScore() after repeat `repeat` of view `view`. */
typedef struct { int view; int repeat; double score; } mvr_fitness_record;

void mvr_turntable_params_default(mvr_turntable_params* p);
/* Registrator::getRotationMatrix (mvr/src/registrator.cpp:331-342): T(pivot) R(axis, angle) T(-pivot), double[16]
 * column-major; and the angle PointCloud::initRotation gives view v of V (mvr/src/point_cloud.cpp:400-413). */
void mvr_turntable_rotation(const double pivot[3], const double axis[3], double angle, double* out16);
double mvr_turntable_view_angle(int view, int n_views);

/* `streams` contexts on `device` run pairs concurrently (each pair is small next to a B200). */
int mvr_registrator_create(int device, int streams, mvr_registrator** out);
int mvr_registrator_destroy(mvr_registrator* r);
const char* mvr_registrator_last_error(mvr_registrator* r);
/* The GPU context behind stream `slot` (owned by the registrator): for profiling switches and kernel statistics. */
mvr_ctx* mvr_registrator_context(mvr_registrator* r, int slot);
int mvr_registrator_streams(mvr_registrator* r);
/* icp.setInputSource / setInputTarget / align / getFinalTransformation as one call
 * (mvr/src/registrator.cpp:565-573): the pairwise-align entry point. */
int mvr_pairwise_align(mvr_registrator* r, const mvr_view* source, const mvr_view* target, const mvr_icp_params* icp,
                       const float* guess, float* out_pose, mvr_icp_report* report);
/* The multi-view-register entry point.  poses: V x float[16] absolute poses in view 0's frame (ring mode
 * with a partial pair range: only the pair reports are meaningful; compose with mvr_ring_close after the
 * gather).  reports: one per pair (ring: V entries indexed by pair; accumulate: V-1 entries, views 1..V-1). */
int mvr_register_turntable(mvr_registrator* r, const mvr_view* views, int n_views, const mvr_turntable_params* prm,
                           float* poses, mvr_pair_report* reports);
/* Ring mode only (the other modes ignore it): search turns about the turntable axis around each pair's initial guess before the
 * first align, for tables that step unevenly, slip or are turned by hand.  The candidates of pair p (target view T = p, source
 * view S = p + 1) are H_j = inv(T.pose) R(delta_j) S.pose, R = the turntable rotation (mvr_turntable_rotation), j = -J..J;
 * all pairs are scored by one mvr_score_guesses_batch with icp.max_correspondence_distance and each pair starts from its
 * lowest-cost H_j (ties: the smallest |j|, then the smaller j; H_0 is the guess without the search).  The choice depends only
 * on the pair's views, their poses and this setting: pair poses stay the same whatever the streams, grouping, pair ranges or
 * GPU count.  Off by default. */
typedef struct {
  double range;  /* radians; candidate turns about the axis span [-range, +range] around each pair's guess; <= 0: off */
  double step;   /* radians, > 0; candidates delta_j = j * step, j = -J..J, J = lround(range / step), 2J + 1 <= 1024 */
  int samples;   /* source points scored per candidate (0: 4096) */
} mvr_angle_search;
void mvr_angle_search_default(mvr_angle_search* s);   /* 15 degrees, 1 degree, 4096 */
int mvr_registrator_set_angle_search(mvr_registrator* r, const mvr_angle_search* s);   /* NULL or range <= 0: off */
/* One record per pair of the last ring registration with the search on: choice = j, angle = delta_j, cost / inliers of H_j,
 * samples = the source points scored, guess_cost / guess_inliers = those of H_0. */
typedef struct { int pair; int choice; double angle; uint64_t cost; int inliers; int samples;
                 uint64_t guess_cost; int guess_inliers; } mvr_angle_pick;
int mvr_registrator_get_angle_search(mvr_registrator* r, mvr_angle_pick* out, int max_records, int* count);   /* out NULL: count only */
/* -- the same entry point over several GPUs of one node ----------------------------------------------------------
 * The reference is one process (its registration runs on one pool thread, mvr/src/registrator.cpp:606, 696); what shards
 * is the ring of neighbour pairs (the edges of :640-651 / :482-487).  One call, inside: one host thread per GPU aligns a
 * contiguous block of the ring's pairs on its GPU (it uploads only the views it needs; point data never crosses GPUs),
 * the ranks exchange their pair records with ONE ncclAllGather (96 bytes per pair, NVLink), the ring is closed on the
 * host.  Results do not depend on the number of GPUs (same pair poses, bit for bit).  NCCL is bound at run time
 * (libnccl.so.2; override with the environment variable MVR_NCCL_LIB): MVR_ERR_NCCL if it is missing or fails. */
typedef struct mvr_multi mvr_multi;
/* What a rank contributes to the exchange, one per pair (no padding: 96 bytes). */
typedef struct {
  float pose[16];          /* relative pose source -> target frame, column-major */
  int32_t n_correspondences, iterations, status, reserved;
  double mse;
  uint64_t nn_queries;
} mvr_pair_record;
/* devices: n_devices distinct CUDA device ordinals (NULL: 0 .. n_devices - 1).  Creates one registrator per GPU and,
 * for n_devices > 1, the NCCL communicators (ncclCommInitAll). */
int mvr_multi_create(const int* devices, int n_devices, mvr_multi** out);
int mvr_multi_destroy(mvr_multi* m);
const char* mvr_multi_last_error(mvr_multi* m);
int mvr_multi_devices(mvr_multi* m);
/* The GPU contexts of rank `rank` (owned by the handle): profiling switches and kernel statistics. */
int mvr_multi_contexts(mvr_multi* m, int rank);
mvr_ctx* mvr_multi_context(mvr_multi* m, int rank, int slot);
/* The block of ring pairs rank `rank` of `n_ranks` aligns: [begin, end) = [rank * n / n_ranks, (rank + 1) * n / n_ranks). */
void mvr_multi_pair_range(int rank, int n_ranks, int n_pairs, int* pair_begin, int* pair_end);
/* Make the (host) views resident: every GPU gets a copy of the views its block of pairs needs.  Later calls with
 * use_resident = 1 align those copies and skip the host-to-device transfer. */
int mvr_multi_upload(mvr_multi* m, const mvr_view* views, int n_views);
/* views: n_views host views (init_pose as for mvr_register_turntable); prm->mode must be MVR_REGISTER_RING_PAIRS,
 * pair_begin / pair_end are ignored.  poses: n_views x float[16] absolute poses after the loop closure; reports
 * (nullable): n_views pair reports; records (nullable): the n_views gathered pair records as exchanged; device_ms
 * (nullable): per GPU, the device time of its part including the exchange (CUDA events). */
int mvr_register_turntable_multi(mvr_multi* m, const mvr_view* views, int n_views, const mvr_turntable_params* prm, int use_resident,
                                 float* poses, mvr_pair_report* reports, mvr_pair_record* records, double* device_ms);
/* mvr_registrator_set_angle_search on every rank; the records of the last call, in pair order (out NULL: count only). */
int mvr_multi_set_angle_search(mvr_multi* m, const mvr_angle_search* s);
int mvr_multi_get_angle_search(mvr_multi* m, mvr_angle_pick* out, int max_records, int* count);

/* Registrator::computeError (mvr/src/registrator.cpp:466-515): reciprocal correspondences (gate max_distance) between
 * neighbouring registered views (i, i + 1) and (V - 1, 0), each view posed by its init_pose first (getTransformedPoints).
 * Pair k: counts[k] correspondences with mean squared distance mean_d2[k]; arrays hold n_views entries. */
/* The fitness scores of the last MVR_REGISTER_ACCUMULATE / MVR_REGISTER_ICP run, one per view and repeat (out nullable: count only). */
int mvr_registrator_get_fitness_log(mvr_registrator* r, mvr_fitness_record* out, int max_records, int* count);
int mvr_compute_error(mvr_registrator* r, const mvr_view* views, int n_views, double max_distance, size_t* counts, double* mean_d2,
                      int* n_pairs);
/* Host-side loop closure over gathered ring pairs: rel[p] = pose of view (p+1)%V in view p's frame, w[p] its
 * weight (e.g. n_correspondences; <= 0 drops the edge).  centre (nullable) = where the object sits in every
 * view's frame (the turntable pivot), rot_scale = its radius: residuals are point displacements of such an
 * object.  Output V absolute poses, view 0 = identity. */
int mvr_ring_close(const float* rel_poses, const double* weights, int n_views, int relax, int iterations, const double* centre,
                   double rot_scale, float* poses);
/* pcl::registration::LUM::compute() for a pose graph whose edges are mvr_pair_moments in ONE common (world)
 * frame: minimises  sum_edges sum_k |X_s a_k - X_t b_k|^2  over rigid corrections X_v, X_0 = identity, by
 * `iterations` Gauss-Newton sweeps (LUM: setMaxIterations(16), mvr/src/registrator.cpp:630) of the dense
 * 6 (V - 1) normal equations.  edges[e] joins views src[e] -> tgt[e]; its sums must already be expressed
 * in the world frame (mvr_pair_moments_transform).  poses: V x double[16] column-major corrections. */
int mvr_lum_relax(const mvr_pair_moments* edges, const int* src, const int* tgt, int n_edges, int n_views, int iterations,
                  double* poses);
/* pcl::registration::LUM::compute() as the reference runs it (lum.setMaxIterations(16); lum.compute(); lum.getTransformation(v),
 * mvr/src/registrator.cpp:630-656), on correspondence moments instead of point lists: vertex poses (x, y, z, roll, pitch,
 * yaw), vertex 0 fixed; per sweep PCL's computeEdge (M'M, M'Z, s^2 of the pairs compounded onto the current poses), the dense
 * 6 (V - 1) system G X = B, pose_v -= incidenceCorrection(pose_v)^-1 X_v; stops early when the summed update norm is
 * <= convergence_threshold (V - 1) (PCL default 0).  edges[e]: moments of edge src[e] -> tgt[e] with BOTH clouds in the
 * common frame the vertices were added in (a = source point, b = target point).  poses6 (nullable): V x 6;
 * transforms (nullable): V x double[16] column-major = pcl::getTransformation(pose_v). */
int mvr_lum_compute(const mvr_pair_moments* edges, const int* src, const int* tgt, int n_edges, int n_views, int iterations,
                    double convergence_threshold, double* poses6, double* transforms);
/* Re-express moments under the rigid map p -> pose * p (double[16] column-major); the new origin is
 * new_origin (nullable: keep pose * old origin). */
void mvr_pair_moments_transform(const mvr_pair_moments* in, const double* pose, const double* new_origin, mvr_pair_moments* out);
/* Bounding box of the finite points of a cloud given to the context. */
int mvr_get_bbox(mvr_ctx* ctx, int which, float lo[3], float hi[3]);
/* Registrator::refineAxis (mvr/src/registrator.cpp:402-455): least-squares turntable axis from registered
 * view poses (poses: count x float[16] column-major).  pivot/axis are in-out. */
int mvr_refine_axis(const float* poses, int count, double pivot[3], double axis[3]);

/* -- either side of the path (SURVEY.md section 8f ranks 2 and 3) -----------------------------------------------------
 * Persistence in the reference's text formats: transformation.txt of a view (PointCloud::loadTransformation /
 * saveTransformation, mvr/src/point_cloud.cpp:305-347; pose = double[16] column-major, p' = M p), axis.txt of an object
 * (Registrator::load / save, mvr/src/registrator.cpp:258-328), points.asc of the merged model (:385-395). */
int mvr_transformation_load(const char* path, double* pose);
int mvr_transformation_save(const char* path, const double* pose);
int mvr_axis_load(const char* path, double pivot[3], double axis[3]);
int mvr_axis_save(const char* path, const double pivot[3], const double axis[3]);
int mvr_points_save_asc(const char* path, const void* rich_points, size_t n);
/* Registrator::saveRegisteredPoints (mvr/src/registrator.cpp:344-383): the registered views, each posed on the GPU,
 * concatenated in view order.  views[v]: counts[v] host records of 48 bytes (pcl::PointXYZRGBNormal: xyz at byte 0,
 * normal at 16, packed colour at 32, curvature at 36); poses: n_views x double[16] column-major; registered
 * (nullable: all): PointCloud::isRegistered() per view.  full_matrix_normals = 1 reproduces the reference, which
 * runs the normals through the whole matrix, translation included (:367-371); 0 rotates them only.
 * out = NULL only reports the record count. */
int mvr_merge_registered(mvr_ctx* ctx, const void* const* views, const size_t* counts, const double* poses, const int* registered,
                         int n_views, int full_matrix_normals, void* out, size_t* out_count);

/* PointCloud::denoise(segment_threshold, triangle_length) (mvr/src/point_cloud.cpp:423-466, called per view by
 * Registrator::registration, mvr/src/registrator.cpp:719-744): the points whose connected component -- edges join points at most
 * triangle_length apart; the reference takes them from a Delaunay triangulation, whose short edges have the same components as
 * this radius graph -- has at least segment_threshold members.  points: n host records of stride_bytes (x, y, z first; 16 or
 * 48).  kept_index (n entries): the indices of the kept points in the reference's output order (components by their smallest
 * point index, points by index); non-finite points are singletons.  noise_count (nullable): the reference's noise_points_num_. */
int mvr_denoise(mvr_ctx* ctx, const void* points, size_t n, size_t stride_bytes, int segment_threshold, double triangle_length,
                int32_t* kept_index, size_t* kept_count, size_t* noise_count);

#ifdef __cplusplus
}
#endif
#endif /* MVR_B200_H */
