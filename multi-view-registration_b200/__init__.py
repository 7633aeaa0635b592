"""Python binding of libmvr_b200.so -- the B200-native ICP alignment path.

This package is a thin ctypes layer over the C ABI in include/mvr_b200.h (the drop-in boundary for
the PCL calls the reference makes in mvr/src/registrator.cpp).  It contains no arithmetic of its own
and NO fallback: if the CUDA library is missing or no CUDA device is usable, it raises.

The directory name contains '-', so import it through the `mvr_b200` shim at the repo root.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MVR_B200_LIB") or os.path.join(_HERE, "libmvr_b200.so")   # the override is a development aid (A/B builds)

K_NAMES = ["morton", "sort", "table", "nn", "corr", "reduce", "transform", "normals"]
K_COUNT = 8
(OK, ERR_BAD_ARG, ERR_TOO_FEW, ERR_CUDA, ERR_NO_INPUT, ERR_NOT_SPD, ERR_ALLOC, ERR_NCCL) = range(8)
TARGET, SOURCE = 0, 1
NN_AUTO, NN_WARP, NN_THREAD, NN_CELL, NN_SEEDED = 0, 1, 2, 3, 4
POINT_TO_POINT, POINT_TO_PLANE, SYMMETRIC = 0, 1, 2


class MvrError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("mvr status %d: %s" % (status, msg))
        self.status = status


class IcpParams(C.Structure):
    _fields_ = [
        ("max_iterations", C.c_int),
        ("max_correspondence_distance", C.c_double),
        ("transformation_epsilon", C.c_double),
        ("euclidean_fitness_epsilon", C.c_double),
        ("use_reciprocal_correspondences", C.c_int),
        ("estimator", C.c_int),
        ("fixed_iterations", C.c_int),
        ("min_correspondences", C.c_int),
    ]


class IcpReport(C.Structure):
    _fields_ = [
        ("iterations", C.c_int),
        ("converged", C.c_int),
        ("reason", C.c_int),
        ("n_correspondences", C.c_int),
        ("mse", C.c_double),
        ("gpu_ms", C.c_double),
        ("nn_queries", C.c_uint64),
    ]


class IcpIteration(C.Structure):
    _fields_ = [("iteration", C.c_int), ("n_correspondences", C.c_int), ("mse", C.c_double), ("delta", C.c_float * 16)]


class Grid(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("inv_cell", C.c_float), ("cell", C.c_float), ("bits", C.c_int)]


class KernelStat(C.Structure):
    _fields_ = [("launches", C.c_uint64), ("ms", C.c_double), ("bytes", C.c_double), ("units", C.c_double)]


class TurntableParams(C.Structure):
    _fields_ = [
        ("pivot", C.c_double * 3),
        ("axis", C.c_double * 3),
        ("icp", IcpParams),
        ("repeat_times", C.c_int),
        ("mode", C.c_int),
        ("loop_closure", C.c_int),
        ("lum_iterations", C.c_int),
        ("pair_begin", C.c_int),
        ("pair_end", C.c_int),
        ("want_fitness", C.c_int),
        ("normal_k", C.c_int),
    ]


class PairMoments(C.Structure):
    """mvr_pair_moments: first and second moments of one edge's correspondence pairs (a = source, b = target)."""
    _fields_ = [("n", C.c_double), ("origin", C.c_double * 3), ("sa", C.c_double * 3), ("sb", C.c_double * 3),
                ("sba", C.c_double * 9), ("saa", C.c_double * 6), ("sbb", C.c_double * 6), ("d2", C.c_double)]

    @classmethod
    def from_pairs(cls, a, b, origin=None):
        """Moments of explicit pairs (n x 3 arrays), numpy double: what the GPU reduction returns for them."""
        a = np.asarray(a, dtype=np.float64).reshape(-1, 3)
        b = np.asarray(b, dtype=np.float64).reshape(-1, 3)
        o = np.zeros(3) if origin is None else np.asarray(origin, dtype=np.float64)
        m = cls()
        m.n = float(len(a))
        m.origin[:] = o.tolist()
        if len(a):
            x, y = a - o, b - o
            m.sa[:] = x.sum(0).tolist(); m.sb[:] = y.sum(0).tolist()
            m.sba[:] = (y.T @ x).reshape(9).tolist()
            xx, yy = x.T @ x, y.T @ y
            m.saa[:] = [xx[0, 0], xx[0, 1], xx[0, 2], xx[1, 1], xx[1, 2], xx[2, 2]]
            m.sbb[:] = [yy[0, 0], yy[0, 1], yy[0, 2], yy[1, 1], yy[1, 2], yy[2, 2]]
            m.d2 = float(((a - b) ** 2).sum())
        return m

    def as_dict(self):
        return dict(n=self.n, origin=np.array(self.origin[:]), sa=np.array(self.sa[:]), sb=np.array(self.sb[:]),
                    sba=np.array(self.sba[:]).reshape(3, 3), saa=np.array(self.saa[:]), sbb=np.array(self.sbb[:]), d2=self.d2)


class AngleSearch(C.Structure):
    """mvr_angle_search: turns about the turntable axis the ring driver scores around each pair's guess (range <= 0: off)."""
    _fields_ = [("range", C.c_double), ("step", C.c_double), ("samples", C.c_int)]


class AnglePick(C.Structure):
    """mvr_angle_pick: the turn a ring pair started from (choice = j, angle = j * step) and its score against the guess's (j = 0)."""
    _fields_ = [("pair", C.c_int), ("choice", C.c_int), ("angle", C.c_double), ("cost", C.c_uint64), ("inliers", C.c_int),
                ("samples", C.c_int), ("guess_cost", C.c_uint64), ("guess_inliers", C.c_int)]

    def as_dict(self):
        return dict(pair=self.pair, choice=self.choice, angle=self.angle, cost=int(self.cost), inliers=self.inliers, samples=self.samples,
                    guess_cost=int(self.guess_cost), guess_inliers=self.guess_inliers)


class GlobalParams(C.Structure):
    """mvr_global_params: the settings of Context.global_align (mvr_global_params_default: PCL-style defaults)."""
    _fields_ = [("keypoints", C.c_int), ("k", C.c_int), ("max_dist", C.c_double), ("hypotheses", C.c_int), ("max_draws", C.c_int),
                ("similarity", C.c_double), ("min_edge", C.c_double), ("samples", C.c_int), ("seed", C.c_uint64)]


class GlobalReport(C.Structure):
    """mvr_global_report: what Context.global_align found (best = index of the winning hypothesis, -1: none)."""
    _fields_ = [("matches", C.c_int), ("draws", C.c_int), ("hypotheses", C.c_int), ("best", C.c_int), ("cost", C.c_uint64),
                ("inliers", C.c_int), ("samples", C.c_int), ("gpu_ms", C.c_double)]

    def as_dict(self):
        return dict(matches=self.matches, draws=self.draws, hypotheses=self.hypotheses, best=self.best, cost=int(self.cost),
                    inliers=self.inliers, samples=self.samples, gpu_ms=self.gpu_ms)


class ViewDesc(C.Structure):
    _fields_ = [("xyzw", C.c_void_p), ("n", C.c_size_t), ("on_device", C.c_int), ("init_pose", C.POINTER(C.c_double))]


class PairRecord(C.Structure):
    """mvr_pair_record: what a rank contributes to the all-gather (96 bytes)."""
    _fields_ = [("pose", C.c_float * 16), ("n_correspondences", C.c_int32), ("iterations", C.c_int32), ("status", C.c_int32),
                ("reserved", C.c_int32), ("mse", C.c_double), ("nn_queries", C.c_uint64)]


class FitnessRecord(C.Structure):
    _fields_ = [("view", C.c_int), ("repeat", C.c_int), ("score", C.c_double)]


class PairReport(C.Structure):
    _fields_ = [
        ("source_view", C.c_int),
        ("target_view", C.c_int),
        ("status", C.c_int),
        ("iterations", C.c_int),
        ("n_correspondences", C.c_int),
        ("mse", C.c_double),
        ("fitness", C.c_double),
        ("gpu_ms", C.c_double),
        ("nn_queries", C.c_uint64),
        ("pose", C.c_float * 16),
    ]


# numpy view of an array of PairReport
REPORT = np.dtype([("source_view", "<i4"), ("target_view", "<i4"), ("status", "<i4"), ("iterations", "<i4"), ("n_correspondences", "<i4"),
                   ("pad", "<i4"), ("mse", "<f8"), ("fitness", "<f8"), ("gpu_ms", "<f8"), ("nn_queries", "<u8"), ("pose", "<f4", (16,))])
assert REPORT.itemsize == C.sizeof(PairReport)


class BoundViews:
    """Marshalled view descriptors (Registrator.bind_views)."""

    def __init__(self, arr, keep, n, views):
        self.arr, self.keep, self.n, self.views = arr, keep, n, views


RING_PAIRS, ACCUMULATE, ICP_ORDER, LUM = 0, 1, 2, 3

_lib = None


def lib():
    """Load libmvr_b200.so; raises if it has not been built (there is no other implementation)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libmvr_b200.so is not built: run `python __graft_entry__.py build` "
                          "(the CUDA library is the only implementation; there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, fp, ip, up = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
    L.mvr_version.restype = C.c_char_p
    L.mvr_kernel_launch_count.restype = C.c_uint64
    L.mvr_status_string.restype = C.c_char_p
    L.mvr_transfer_sizes.argtypes = [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.mvr_transfer_sizes.restype = None
    L.mvr_status_string.argtypes = [C.c_int]
    L.mvr_icp_params_default.argtypes = [C.POINTER(IcpParams)]
    L.mvr_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.mvr_ctx_destroy.argtypes = [vp]
    L.mvr_ctx_set_stream.argtypes = [vp, vp]
    L.mvr_ctx_synchronize.argtypes = [vp]
    L.mvr_last_error.argtypes = [vp]
    L.mvr_last_error.restype = C.c_char_p
    L.mvr_ctx_set_profiling.argtypes = [vp, C.c_int]
    L.mvr_ctx_get_kernel_stats.argtypes = [vp, C.POINTER(KernelStat), C.c_int]
    L.mvr_debug_value.argtypes = [vp, C.c_int]
    L.mvr_debug_value.restype = C.c_double
    L.mvr_ctx_set_index_options.argtypes = [vp, C.c_float, C.c_int]
    L.mvr_ctx_set_batch_group.argtypes = [vp, C.c_int]
    L.mvr_ctx_set_nn_options.argtypes = [vp, C.c_double, C.c_double]
    L.mvr_ctx_set_nn_mode.argtypes = [vp, C.c_int]
    L.mvr_ctx_set_gate_mask.argtypes = [vp, C.c_int]
    for name in ("mvr_set_target", "mvr_set_source", "mvr_set_target_device", "mvr_set_source_device", "mvr_set_target_normals",
                 "mvr_set_source_normals"):
        getattr(L, name).argtypes = [vp, vp, C.c_size_t]
    L.mvr_normals_share.argtypes = [vp, C.c_int, vp, C.c_int]
    L.mvr_index_build.argtypes = [vp, C.c_int, C.POINTER(Grid)]
    L.mvr_index_export.argtypes = [vp, C.c_int, C.POINTER(Grid), up, ip, up]
    L.mvr_nn_query.argtypes = [vp, fp, C.c_size_t, ip, fp]
    L.mvr_nn_query_device.argtypes = [vp, vp, C.c_size_t, vp, vp]
    L.mvr_correspondences.argtypes = [vp, C.c_double, C.c_int, ip, ip, fp, C.POINTER(C.c_size_t)]
    L.mvr_icp_align.argtypes = [vp, C.POINTER(IcpParams), fp, fp, vp, C.POINTER(IcpReport)]
    L.mvr_icp_align_batch.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(IcpParams), fp, fp, C.POINTER(IcpReport), ip]
    L.mvr_icp_get_iterations.argtypes = [vp, C.POINTER(IcpIteration), C.c_int, C.POINTER(C.c_int)]
    L.mvr_fitness_score.argtypes = [vp, C.c_double, C.POINTER(C.c_double)]
    L.mvr_denoise.argtypes = [vp, vp, C.c_size_t, C.c_size_t, C.c_int, C.c_double, ip, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.mvr_estimate_normals.argtypes = [vp, C.c_int, C.c_int, fp, fp, ip]
    L.mvr_estimate_normals_batch.argtypes = [C.POINTER(vp), C.c_int, C.c_int, fp, C.POINTER(fp), ip]
    dp = C.POINTER(C.c_double)
    L.mvr_score_guesses_batch.argtypes = [C.POINTER(vp), C.c_int, fp, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_uint64), ip, ip]
    L.mvr_compute_fpfh.argtypes = [vp, C.c_int, C.c_int, C.c_int, fp, ip, fp, fp, C.POINTER(C.c_int)]
    L.mvr_match_features.argtypes = [vp, fp, C.c_int, fp, C.c_int, ip, ip]
    L.mvr_global_params_default.argtypes = [C.POINTER(GlobalParams)]
    L.mvr_global_params_default.restype = None
    L.mvr_global_align.argtypes = [vp, C.POINTER(GlobalParams), fp, C.POINTER(GlobalReport)]
    L.mvr_angle_search_default.argtypes = [C.POINTER(AngleSearch)]
    L.mvr_angle_search_default.restype = None
    L.mvr_registrator_set_angle_search.argtypes = [vp, C.POINTER(AngleSearch)]
    L.mvr_registrator_get_angle_search.argtypes = [vp, C.POINTER(AnglePick), C.c_int, C.POINTER(C.c_int)]
    L.mvr_multi_set_angle_search.argtypes = [vp, C.POINTER(AngleSearch)]
    L.mvr_multi_get_angle_search.argtypes = [vp, C.POINTER(AnglePick), C.c_int, C.POINTER(C.c_int)]
    L.mvr_apply_pose.argtypes = [vp, vp, C.c_size_t, C.c_size_t, dp, fp]
    L.mvr_apply_pose_device.argtypes = [vp, vp, C.c_size_t, C.c_size_t, dp, vp]
    L.mvr_copy_aligned_device.argtypes = [vp, vp]
    L.mvr_turntable_params_default.argtypes = [C.POINTER(TurntableParams)]
    L.mvr_turntable_rotation.argtypes = [dp, dp, C.c_double, dp]
    L.mvr_turntable_view_angle.argtypes = [C.c_int, C.c_int]
    L.mvr_turntable_view_angle.restype = C.c_double
    L.mvr_registrator_create.argtypes = [C.c_int, C.c_int, C.POINTER(vp)]
    L.mvr_registrator_destroy.argtypes = [vp]
    L.mvr_registrator_last_error.argtypes = [vp]
    L.mvr_registrator_last_error.restype = C.c_char_p
    L.mvr_registrator_context.argtypes = [vp, C.c_int]
    L.mvr_registrator_context.restype = vp
    L.mvr_registrator_streams.argtypes = [vp]
    L.mvr_pairwise_align.argtypes = [vp, C.POINTER(ViewDesc), C.POINTER(ViewDesc), C.POINTER(IcpParams), fp, fp, C.POINTER(IcpReport)]
    L.mvr_register_turntable.argtypes = [vp, C.POINTER(ViewDesc), C.c_int, C.POINTER(TurntableParams), fp, C.POINTER(PairReport)]
    L.mvr_multi_create.argtypes = [ip, C.c_int, C.POINTER(vp)]
    L.mvr_multi_destroy.argtypes = [vp]
    L.mvr_multi_last_error.argtypes = [vp]
    L.mvr_multi_last_error.restype = C.c_char_p
    L.mvr_multi_devices.argtypes = [vp]
    L.mvr_multi_contexts.argtypes = [vp, C.c_int]
    L.mvr_multi_context.argtypes = [vp, C.c_int, C.c_int]
    L.mvr_multi_context.restype = vp
    L.mvr_multi_pair_range.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.mvr_multi_pair_range.restype = None
    L.mvr_multi_upload.argtypes = [vp, C.POINTER(ViewDesc), C.c_int]
    L.mvr_register_turntable_multi.argtypes = [vp, C.POINTER(ViewDesc), C.c_int, C.POINTER(TurntableParams), C.c_int, fp, C.POINTER(PairReport),
                                               C.POINTER(PairRecord), dp]
    L.mvr_registrator_get_fitness_log.argtypes = [vp, C.POINTER(FitnessRecord), C.c_int, C.POINTER(C.c_int)]
    L.mvr_compute_error.argtypes = [vp, C.POINTER(ViewDesc), C.c_int, C.c_double, C.POINTER(C.c_size_t), dp, C.POINTER(C.c_int)]
    L.mvr_ring_close.argtypes = [fp, dp, C.c_int, C.c_int, C.c_int, dp, C.c_double, fp]
    L.mvr_get_bbox.argtypes = [vp, C.c_int, fp, fp]
    L.mvr_set_clouds_device.argtypes = [C.POINTER(vp), ip, C.POINTER(vp), C.POINTER(C.c_size_t), C.c_int]
    L.mvr_refine_axis.argtypes = [fp, C.c_int, dp, dp]
    L.mvr_transformation_load.argtypes = [C.c_char_p, dp]
    L.mvr_transformation_save.argtypes = [C.c_char_p, dp]
    L.mvr_axis_load.argtypes = [C.c_char_p, dp, dp]
    L.mvr_axis_save.argtypes = [C.c_char_p, dp, dp]
    L.mvr_points_save_asc.argtypes = [C.c_char_p, vp, C.c_size_t]
    L.mvr_merge_registered.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t), dp, ip, C.c_int, C.c_int, vp, C.POINTER(C.c_size_t)]
    L.mvr_pair_moments_compute.argtypes = [vp, C.c_double, C.c_int, fp, C.POINTER(PairMoments)]
    L.mvr_lum_relax.argtypes = [C.POINTER(PairMoments), ip, ip, C.c_int, C.c_int, C.c_int, dp]
    L.mvr_lum_compute.argtypes = [C.POINTER(PairMoments), ip, ip, C.c_int, C.c_int, C.c_int, C.c_double, dp, dp]
    L.mvr_pair_moments_transform.argtypes = [C.POINTER(PairMoments), dp, dp, C.POINTER(PairMoments)]
    L.mvr_pair_moments_transform.restype = None
    _lib = L
    return L


def kernel_launch_count():
    return int(lib().mvr_kernel_launch_count())


def _transfer_sizes():
    a, b = C.c_size_t(0), C.c_size_t(0)
    lib().mvr_transfer_sizes(C.byref(a), C.byref(b))
    return int(a.value), int(b.value)


def icp_state_bytes():
    """Bytes of the per-align loop state an align copies in and reads back."""
    return _transfer_sizes()[0]


def icp_log_record_bytes():
    """Bytes of one per-iteration log record read back after an align."""
    return _transfer_sizes()[1]


def default_params(**kw):
    """mvr_icp_params with PCL's defaults, overridden by keyword (reference settings:
    mvr/src/registrator.cpp:551-560)."""
    p = IcpParams()
    lib().mvr_icp_params_default(C.byref(p))
    alias = {"max_dist": "max_correspondence_distance", "reciprocal": "use_reciprocal_correspondences"}
    for k, v in kw.items():
        setattr(p, alias.get(k, k), v)
    return p


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError("points must be n x 4 float32 (pcl::PointXYZ layout)")
    return a


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _up(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint32))


def pose_to_numpy(flat16):
    """column-major float[16] (Eigen::Matrix4f) -> 4x4 numpy (row-major view of the same matrix)."""
    return np.asarray(flat16, dtype=np.float32).reshape(4, 4).T.copy()


def pose_from_numpy(M):
    return np.ascontiguousarray(np.asarray(M, dtype=np.float32).T).reshape(16)


class Context:
    """One CUDA device + stream; mirrors a pcl::IterativeClosestPoint instance holding its
    source/target (Registrator::icp_, mvr/include/registrator.h:91)."""

    def __init__(self, device=0, _borrowed=None):
        self._keep = {}
        self._tgt_n = None   # points of the target set through this object (sizes the host copies of estimate_normals_batch)
        self._owned = _borrowed is None
        if _borrowed is not None:
            self._h = C.c_void_p(_borrowed)
            return
        self._h = C.c_void_p()
        rc = lib().mvr_ctx_create(int(device), C.byref(self._h))
        if rc != OK:
            raise MvrError(rc, "mvr_ctx_create failed (no usable CUDA device %d; there is no CPU fallback)" % device)
        self._keep = {}

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            if self._owned:
                lib().mvr_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, allow=()):
        if rc != OK and rc not in allow:
            raise MvrError(rc, (lib().mvr_last_error(self._h) or b"").decode() or lib().mvr_status_string(rc).decode())
        return rc

    # -- plumbing ------------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(lib().mvr_ctx_set_stream(self._h, C.c_void_p(int(cuda_stream_ptr))))

    def synchronize(self):
        self._ck(lib().mvr_ctx_synchronize(self._h))

    def set_profiling(self, on):
        self._ck(lib().mvr_ctx_set_profiling(self._h, int(bool(on))))

    def kernel_stats(self, reset=False):
        arr = (KernelStat * K_COUNT)()
        self._ck(lib().mvr_ctx_get_kernel_stats(self._h, arr, int(bool(reset))))
        return {K_NAMES[i]: dict(launches=int(arr[i].launches), ms=arr[i].ms, bytes=arr[i].bytes, units=arr[i].units)
                for i in range(K_COUNT)}

    def last_error(self):
        return (lib().mvr_last_error(self._h) or b"").decode()

    def debug_value(self, k):
        return float(lib().mvr_debug_value(self._h, int(k)))

    def set_index_options(self, cell_edge=0.0, max_bits=8):
        self._ck(lib().mvr_ctx_set_index_options(self._h, C.c_float(cell_edge), int(max_bits)))

    # -- inputs --------------------------------------------------------------------------------
    def set_nn_options(self, points_per_cell=8.0, dense_ratio=8.0):
        """NN-query tuning: dense_ratio = queries per target point from which the warp-cooperative pass runs (0: never)."""
        self._ck(lib().mvr_ctx_set_nn_options(self._h, float(points_per_cell), float(dense_ratio)))

    def set_nn_mode(self, mode):
        """NN_AUTO / NN_WARP / NN_THREAD / NN_CELL / NN_SEEDED: which kernel answers nn_query (identical results)."""
        self._ck(lib().mvr_ctx_set_nn_mode(self._h, int(mode)))

    def set_gate_mask(self, on):
        self._ck(lib().mvr_ctx_set_gate_mask(self._h, 1 if on else 0))

    def set_batch_group(self, pairs):
        """Pairs per kernel launch of the batches this context leads (1..24)."""
        self._ck(lib().mvr_ctx_set_batch_group(self._h, int(pairs)))

    def set_target(self, pts):
        pts = _pts(pts)
        self._ck(lib().mvr_set_target(self._h, pts.ctypes.data, len(pts)))
        self._tgt_n = len(pts)

    def set_source(self, pts):
        pts = _pts(pts)
        self._ck(lib().mvr_set_source(self._h, pts.ctypes.data, len(pts)))

    def set_target_device(self, ptr, n, keepalive=None):
        self._keep["tgt"] = keepalive
        self._ck(lib().mvr_set_target_device(self._h, C.c_void_p(int(ptr)), int(n)))
        self._tgt_n = int(n)

    def set_source_device(self, ptr, n, keepalive=None):
        self._keep["src"] = keepalive
        self._ck(lib().mvr_set_source_device(self._h, C.c_void_p(int(ptr)), int(n)))

    def set_target_normals(self, nrm):
        nrm = _pts(nrm)
        self._ck(lib().mvr_set_target_normals(self._h, nrm.ctypes.data, len(nrm)))

    def set_source_normals(self, nrm):
        """n x 4 {nx, ny, nz, curvature} of the source (symmetric ICP); n must equal the source size."""
        nrm = _pts(nrm)
        self._ck(lib().mvr_set_source_normals(self._h, nrm.ctypes.data, len(nrm)))

    def normals_share(self, which, other, other_which):
        """mvr_normals_share: this context's TARGET / SOURCE normals become the device normals `other` holds for its
        `other_which` cloud (no copy; `other` must keep them unchanged while this context uses them)."""
        self._ck(lib().mvr_normals_share(self._h, int(which), other._h, int(other_which)))

    # -- index ---------------------------------------------------------------------------------
    def index_build(self, which=TARGET, grid=None):
        g = None
        if grid is not None:
            g = Grid()
            g.origin[:] = [float(x) for x in grid["origin"]]
            g.inv_cell = float(grid["inv_cell"])
            g.cell = float(grid.get("cell", 1.0 / grid["inv_cell"]))
            g.bits = int(grid["bits"])
        self._ck(lib().mvr_index_build(self._h, int(which), C.byref(g) if g is not None else None))

    def index_export(self, which, n):
        g = Grid()
        self._ck(lib().mvr_index_export(self._h, int(which), C.byref(g), None, None, None))
        keys = np.empty(n, dtype=np.uint32)
        perm = np.empty(n, dtype=np.int32)
        start = np.empty((1 << (3 * g.bits)) + 1, dtype=np.uint32)
        self._ck(lib().mvr_index_export(self._h, int(which), C.byref(g), _up(keys), _ip(perm), _up(start)))
        grid = dict(origin=np.array(g.origin[:], dtype=np.float32), inv_cell=np.float32(g.inv_cell), cell=np.float32(g.cell), bits=g.bits)
        return grid, keys, perm, start

    # -- queries -------------------------------------------------------------------------------
    def nn_query(self, q):
        q = _pts(q)
        idx = np.empty(len(q), dtype=np.int32)
        d2 = np.empty(len(q), dtype=np.float32)
        self._ck(lib().mvr_nn_query(self._h, _fp(q), len(q), _ip(idx), _fp(d2)))
        return idx, d2

    def nn_query_device(self, q_ptr, n, idx_ptr, d2_ptr):
        self._ck(lib().mvr_nn_query_device(self._h, C.c_void_p(int(q_ptr)), int(n), C.c_void_p(int(idx_ptr)), C.c_void_p(int(d2_ptr))))

    def correspondences(self, n_source, max_dist, reciprocal):
        q = np.empty(max(n_source, 1), dtype=np.int32)
        m = np.empty(max(n_source, 1), dtype=np.int32)
        d = np.empty(max(n_source, 1), dtype=np.float32)
        cnt = C.c_size_t(0)
        self._ck(lib().mvr_correspondences(self._h, float(max_dist), int(bool(reciprocal)), _ip(q), _ip(m), _fp(d), C.byref(cnt)))
        c = cnt.value
        return q[:c].copy(), m[:c].copy(), d[:c].copy()

    # -- ICP -----------------------------------------------------------------------------------
    def icp_align(self, params, guess=None, n_source=None, want_cloud=False):
        """Returns dict(status, final 4x4, cloud or None, iterations, converged, reason, n_corr, mse,
        gpu_ms, nn_queries, log).  status MVR_ERR_TOO_FEW_CORRESPONDENCES is reported, not raised."""
        g = pose_from_numpy(guess) if guess is not None else None
        fin = np.empty(16, dtype=np.float32)
        cloud = np.empty((n_source, 4), dtype=np.float32) if want_cloud else None
        rep = IcpReport()
        rc = lib().mvr_icp_align(self._h, C.byref(params), _fp(g) if g is not None else None, _fp(fin),
                                 cloud.ctypes.data if cloud is not None else None, C.byref(rep))
        self._ck(rc, allow=(ERR_TOO_FEW, ERR_NOT_SPD))
        cnt = C.c_int(0)
        lib().mvr_icp_get_iterations(self._h, None, 0, C.byref(cnt))
        recs = (IcpIteration * max(cnt.value, 1))()
        lib().mvr_icp_get_iterations(self._h, recs, cnt.value, C.byref(cnt))
        log = [dict(iteration=recs[k].iteration, n_corr=recs[k].n_correspondences, mse=recs[k].mse,
                    delta=pose_to_numpy(recs[k].delta[:])) for k in range(cnt.value)]
        return dict(status=rc, final=pose_to_numpy(fin), cloud=cloud, iterations=rep.iterations, converged=rep.converged,
                    reason=rep.reason, n_corr=rep.n_correspondences, mse=rep.mse, gpu_ms=rep.gpu_ms,
                    nn_queries=int(rep.nn_queries), log=log)

    def pair_moments(self, max_dist, reciprocal=True, guess=None):
        """Moments of the (reciprocal) correspondences source -> target under `guess` (target frame)."""
        g = pose_from_numpy(guess) if guess is not None else None
        m = PairMoments()
        self._ck(lib().mvr_pair_moments_compute(self._h, float(max_dist), int(bool(reciprocal)), _fp(g) if g is not None else None, C.byref(m)))
        return m

    def merge_registered(self, views, poses, registered=None, full_matrix_normals=True):
        """Registrator::saveRegisteredPoints: views = list of RICH_POINT arrays, poses = list of 4x4; returns the merged array."""
        arrs = [np.ascontiguousarray(v, dtype=RICH_POINT) for v in views]
        V = len(arrs)
        ptrs = (C.c_void_p * max(V, 1))(*[a.ctypes.data for a in arrs])
        counts = (C.c_size_t * max(V, 1))(*[len(a) for a in arrs])
        P = np.ascontiguousarray(np.stack([np.asarray(T, dtype=np.float64).T.reshape(16) for T in poses])) if V else np.zeros((1, 16))
        reg = None if registered is None else np.ascontiguousarray(registered, dtype=np.int32)
        total = C.c_size_t(0)
        self._ck(lib().mvr_merge_registered(self._h, ptrs, counts, _dp(P), _ip(reg) if reg is not None else None, V, int(bool(full_matrix_normals)), None, C.byref(total)))
        out = np.empty(total.value, dtype=RICH_POINT)
        if total.value:
            self._ck(lib().mvr_merge_registered(self._h, ptrs, counts, _dp(P), _ip(reg) if reg is not None else None, V, int(bool(full_matrix_normals)),
                                                out.ctypes.data, C.byref(total)))
        return out

    def iterations(self):
        """Per-iteration records of the last align of this context (also after a batched align)."""
        cnt = C.c_int(0)
        self._ck(lib().mvr_icp_get_iterations(self._h, None, 0, C.byref(cnt)))
        recs = (IcpIteration * max(cnt.value, 1))()
        self._ck(lib().mvr_icp_get_iterations(self._h, recs, cnt.value, C.byref(cnt)))
        return [dict(iteration=recs[k].iteration, n_corr=recs[k].n_correspondences, mse=recs[k].mse,
                     delta=pose_to_numpy(recs[k].delta[:])) for k in range(cnt.value)]

    def fitness_score(self, max_range=None):
        import sys
        s = C.c_double(0)
        self._ck(lib().mvr_fitness_score(self._h, sys.float_info.max if max_range is None else float(max_range), C.byref(s)))
        return s.value

    def estimate_normals(self, which, n, k, viewpoint=(0.0, 0.0, 0.0), want_neighbours=False):
        vp = np.ascontiguousarray(viewpoint, dtype=np.float32)
        out = np.empty((n, 4), dtype=np.float32)
        nbr = np.empty((n, k), dtype=np.int32) if want_neighbours else None
        self._ck(lib().mvr_estimate_normals(self._h, int(which), int(k), _fp(vp), _fp(out), _ip(nbr) if nbr is not None else None))
        return (out, nbr) if want_neighbours else out


    def fpfh(self, which, keypoints, k, viewpoint=None):
        """mvr_compute_fpfh: (original indices of the keypoints int32, their normals n_kp x 4, FPFH n_kp x 33 float32).
        viewpoint None: the centre of the cloud's bounding box."""
        vp = None if viewpoint is None else np.ascontiguousarray(viewpoint, dtype=np.float32)
        idx = np.empty(int(keypoints), dtype=np.int32)
        nrm = np.empty((int(keypoints), 4), dtype=np.float32)
        feat = np.empty((int(keypoints), 33), dtype=np.float32)
        n = C.c_int(0)
        self._ck(lib().mvr_compute_fpfh(self._h, int(which), int(keypoints), int(k), _fp(vp) if vp is not None else None, _ip(idx), _fp(nrm),
                                        _fp(feat), C.byref(n)))
        m = n.value
        return idx[:m].copy(), nrm[:m].copy(), feat[:m].copy()

    def match_features(self, a, b):
        """mvr_match_features: (a_to_b, b_to_a) exact nearest rows of two n x 33 float32 descriptor tables (-1: none)."""
        a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1, 33)
        b = np.ascontiguousarray(b, dtype=np.float32).reshape(-1, 33)
        ab = np.empty(max(len(a), 1), dtype=np.int32)
        ba = np.empty(max(len(b), 1), dtype=np.int32)
        self._ck(lib().mvr_match_features(self._h, _fp(a), len(a), _fp(b), len(b), _ip(ab), _ip(ba)))
        return ab[:len(a)].copy(), ba[:len(b)].copy()

    def global_align(self, params=None):
        """mvr_global_align: (pose 4x4 float32 mapping the source onto the target, report dict with status).  A status of
        MVR_ERR_TOO_FEW_CORRESPONDENCES is reported (pose = identity), not raised."""
        p = params if params is not None else global_params()
        out = np.empty(16, dtype=np.float32)
        rep = GlobalReport()
        rc = lib().mvr_global_align(self._h, C.byref(p), _fp(out), C.byref(rep))
        self._ck(rc, allow=(ERR_TOO_FEW,))
        d = rep.as_dict()
        d["status"] = rc
        return pose_to_numpy(out), d

    def denoise(self, pts, segment_threshold=10, triangle_length=2.5):
        """PointCloud::denoise: (indices of the kept points in the reference's output order, number of noise points).
        pts: n x 4 float32 (PointXYZ) or a RICH_POINT array (48-byte records)."""
        a = np.ascontiguousarray(pts)
        n = len(a)
        stride = a.dtype.itemsize if a.dtype.fields else a.strides[0]
        keep = np.empty(max(n, 1), dtype=np.int32)
        cnt, noise = C.c_size_t(0), C.c_size_t(0)
        self._ck(lib().mvr_denoise(self._h, a.ctypes.data, n, stride, int(segment_threshold), float(triangle_length), _ip(keep), C.byref(cnt), C.byref(noise)))
        return keep[:cnt.value].copy(), int(noise.value)

    def apply_pose(self, pts, pose):
        """PointCloud::getTransformedPoints: pts (n x k float32, xyz first) -> n x 4 float32, pose 4x4 double."""
        pts = np.ascontiguousarray(pts, dtype=np.float32)
        M = np.ascontiguousarray(np.asarray(pose, dtype=np.float64).T).reshape(16)
        out = np.empty((len(pts), 4), dtype=np.float32)
        self._ck(lib().mvr_apply_pose(self._h, pts.ctypes.data, len(pts), pts.strides[0], M.ctypes.data_as(C.POINTER(C.c_double)), _fp(out)))
        return out


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def turntable_rotation(pivot, axis, angle):
    """Registrator::getRotationMatrix (mvr/src/registrator.cpp:331-342) as a 4x4 double (column-vector form)."""
    pv = np.ascontiguousarray(pivot, dtype=np.float64)
    ax = np.ascontiguousarray(axis, dtype=np.float64)
    out = np.empty(16, dtype=np.float64)
    lib().mvr_turntable_rotation(_dp(pv), _dp(ax), float(angle), _dp(out))
    return out.reshape(4, 4).T.copy()


def turntable_view_angle(view, n_views):
    return float(lib().mvr_turntable_view_angle(int(view), int(n_views)))


def turntable_params(**kw):
    p = TurntableParams()
    lib().mvr_turntable_params_default(C.byref(p))
    for k, v in kw.items():
        if k in ("pivot", "axis"):
            getattr(p, k)[:] = [float(x) for x in v]
        elif k == "icp":
            p.icp = v
        else:
            setattr(p, k, v)
    return p


def ring_close(rel_poses, weights=None, relax=True, iterations=16, centre=None, rot_scale=1.0):
    """Host loop closure: rel_poses V x 4x4 (view p+1 in view p's frame) -> V absolute 4x4 poses.
    centre = the turntable pivot, rot_scale = the object's radius (residuals become point displacements)."""
    V = len(rel_poses)
    rel = np.ascontiguousarray(np.stack([pose_from_numpy(T) for T in rel_poses]), dtype=np.float32)
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
    out = np.empty((V, 16), dtype=np.float32)
    cc = None if centre is None else np.ascontiguousarray(centre, dtype=np.float64)
    rc = lib().mvr_ring_close(_fp(rel), _dp(w) if w is not None else None, V, int(bool(relax)), int(iterations),
                              _dp(cc) if cc is not None else None, float(rot_scale), _fp(out))
    if rc != OK:
        raise MvrError(rc, lib().mvr_status_string(rc).decode())
    return [pose_to_numpy(out[k]) for k in range(V)]


def ring_close_flat(rel16, weights, relax=True, iterations=16, centre=None, rot_scale=1.0):
    """ring_close on V x 16 column-major float32 poses (as the pair records carry them); returns the V absolute poses as
    4x4 numpy matrices."""
    rel = np.ascontiguousarray(rel16, dtype=np.float32).reshape(-1, 16)
    V = len(rel)
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
    out = np.empty((V, 16), dtype=np.float32)
    cc = None if centre is None else np.ascontiguousarray(centre, dtype=np.float64)
    rc = lib().mvr_ring_close(_fp(rel), _dp(w) if w is not None else None, V, int(bool(relax)), int(iterations),
                              _dp(cc) if cc is not None else None, float(rot_scale), _fp(out))
    if rc != OK:
        raise MvrError(rc, lib().mvr_status_string(rc).decode())
    return list(out.reshape(V, 4, 4).transpose(0, 2, 1).copy())


# ---- persistence in the reference's text formats (transformation.txt, axis.txt, points.asc) ----------------------------
RICH_POINT = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("pad0", "<f4"),
                       ("normal_x", "<f4"), ("normal_y", "<f4"), ("normal_z", "<f4"), ("pad1", "<f4"),
                       ("b", "u1"), ("g", "u1"), ("r", "u1"), ("a", "u1"), ("curvature", "<f4"), ("pad2", "<f4", (2,))])   # pcl::PointXYZRGBNormal
assert RICH_POINT.itemsize == 48


def transformation_load(path):
    m = np.empty(16, dtype=np.float64)
    rc = lib().mvr_transformation_load(os.fsencode(path), _dp(m))
    if rc != OK:
        raise MvrError(rc, "cannot read " + str(path))
    return m.reshape(4, 4).T.copy()


def transformation_save(path, pose):
    m = np.ascontiguousarray(np.asarray(pose, dtype=np.float64).T).reshape(16)
    rc = lib().mvr_transformation_save(os.fsencode(path), _dp(m))
    if rc != OK:
        raise MvrError(rc, "cannot write " + str(path))


def axis_load(path):
    pv, ax = np.empty(3), np.empty(3)
    rc = lib().mvr_axis_load(os.fsencode(path), _dp(pv), _dp(ax))
    if rc != OK:
        raise MvrError(rc, "cannot read " + str(path))
    return pv, ax


def axis_save(path, pivot, axis):
    pv, ax = np.ascontiguousarray(pivot, dtype=np.float64), np.ascontiguousarray(axis, dtype=np.float64)
    rc = lib().mvr_axis_save(os.fsencode(path), _dp(pv), _dp(ax))
    if rc != OK:
        raise MvrError(rc, "cannot write " + str(path))


def points_save_asc(path, rich_points):
    a = np.ascontiguousarray(rich_points, dtype=RICH_POINT)
    rc = lib().mvr_points_save_asc(os.fsencode(path), a.ctypes.data, len(a))
    if rc != OK:
        raise MvrError(rc, "cannot write " + str(path))


def set_clouds_device(contexts, which, ptrs, counts, keepalive=None):
    """mvr_set_clouds_device: contexts[k] adopts the device cloud (ptrs[k], counts[k]) as its TARGET / SOURCE (which[k]); the
    bounding boxes of all clouds are measured by one launch."""
    n = len(contexts)
    hs = (C.c_void_p * n)(*[c._h for c in contexts])
    w = np.ascontiguousarray(which, dtype=np.int32)
    pp = (C.c_void_p * n)(*[int(p) for p in ptrs])
    cc = (C.c_size_t * n)(*[int(x) for x in counts])
    for k, c in enumerate(contexts):
        c._keep["tgt" if int(w[k]) == TARGET else "src"] = keepalive
    rc = lib().mvr_set_clouds_device(hs, _ip(w), pp, cc, n)
    if rc != OK:
        raise MvrError(rc, contexts[0].last_error() if n else "")
    for k, c in enumerate(contexts):
        if int(w[k]) == TARGET:
            c._tgt_n = int(counts[k])


def icp_align_batch(contexts, params, guesses=None):
    """mvr_icp_align_batch: the aligns of `contexts` (each with its own source/target) in lock-step, one kernel launch
    per iteration half for all of them.  Returns a list of dicts like Context.icp_align."""
    n = len(contexts)
    hs = (C.c_void_p * max(n, 1))(*[c._h for c in contexts])
    g = None
    if guesses is not None:
        g = np.ascontiguousarray(np.stack([pose_from_numpy(T) for T in guesses]), dtype=np.float32)
    fin = np.empty((max(n, 1), 16), dtype=np.float32)
    reps = (IcpReport * max(n, 1))()
    st = np.zeros(max(n, 1), dtype=np.int32)
    rc = lib().mvr_icp_align_batch(hs, n, C.byref(params), _fp(g) if g is not None else None, _fp(fin), reps, _ip(st))
    if rc != OK:
        raise MvrError(rc, (lib().mvr_last_error(contexts[0]._h) or b"").decode() if n else "bad batch")
    return [dict(status=int(st[k]), final=pose_to_numpy(fin[k]), iterations=reps[k].iterations, converged=bool(reps[k].converged),
                 reason=reps[k].reason, n_corr=reps[k].n_correspondences, mse=reps[k].mse, gpu_ms=reps[k].gpu_ms,
                 nn_queries=int(reps[k].nn_queries)) for k in range(n)]


def estimate_normals_batch(contexts, k, viewpoints=None, want=False):
    """mvr_estimate_normals_batch: kNN(k) PCA normals of every context's TARGET (the same bits as Context.estimate_normals),
    kept on the device for point-to-plane ICP.  viewpoints: len(contexts) x 3 (None: each target's origin).  Returns a list
    with, per context, its n x 4 float32 {nx, ny, nz, curvature} when want is true, else None.  Raises on a failed status."""
    n = len(contexts)
    hs = (C.c_void_p * max(n, 1))(*[c._h for c in contexts])
    vp = None if viewpoints is None else np.ascontiguousarray(np.asarray(viewpoints, dtype=np.float32).reshape(n, 3))
    outs = [None] * n
    ptrs = None
    if want:
        outs = [np.empty((c._tgt_n, 4), dtype=np.float32) if c._tgt_n is not None else None for c in contexts]
        ptrs = (C.POINTER(C.c_float) * max(n, 1))(*[_fp(o) if o is not None else C.POINTER(C.c_float)() for o in outs])
    st = np.zeros(max(n, 1), dtype=np.int32)
    rc = lib().mvr_estimate_normals_batch(hs, n, int(k), _fp(vp) if vp is not None else None, ptrs, _ip(st))
    if rc != OK:
        raise MvrError(rc, contexts[0].last_error() if n else lib().mvr_status_string(rc).decode())
    for i in range(n):
        if st[i] != OK:
            raise MvrError(int(st[i]), contexts[i].last_error() or lib().mvr_status_string(int(st[i])).decode())
    return outs


def score_guesses_batch(contexts, candidates, max_dist, samples=4096):
    """mvr_score_guesses_batch: candidates = len(contexts) x n_candidates 4x4 transforms (source -> target frame).  Returns
    (costs len(contexts) x n_candidates uint64, inliers the same shape int32, statuses int32 per context); raises on a failure
    of the batch itself (a context without input only sets its status)."""
    n = len(contexts)
    M = np.asarray(candidates, dtype=np.float32)
    if M.ndim != 4 or M.shape[0] != n or M.shape[2:] != (4, 4):
        raise ValueError("candidates must be len(contexts) x n_candidates x 4 x 4")
    nc = M.shape[1]
    flat = np.ascontiguousarray(M.transpose(0, 1, 3, 2)).reshape(-1)   # column-major per candidate
    hs = (C.c_void_p * max(n, 1))(*[c._h for c in contexts])
    costs = np.zeros((max(n, 1), nc), dtype=np.uint64)
    inl = np.zeros((max(n, 1), nc), dtype=np.int32)
    st = np.zeros(max(n, 1), dtype=np.int32)
    rc = lib().mvr_score_guesses_batch(hs, n, _fp(flat) if n else None, int(nc), float(max_dist), int(samples),
                                       costs.ctypes.data_as(C.POINTER(C.c_uint64)), _ip(inl), _ip(st))
    if rc != OK:
        raise MvrError(rc, contexts[0].last_error() if n else lib().mvr_status_string(rc).decode())
    return costs[:n], inl[:n], st[:n]


def global_params(**kw):
    """mvr_global_params with the library's defaults, overridden by keyword."""
    p = GlobalParams()
    lib().mvr_global_params_default(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def angle_search_default():
    s = AngleSearch()
    lib().mvr_angle_search_default(C.byref(s))
    return s


def _angle_search(range_, step, samples):
    if range_ is None or range_ <= 0:
        return None
    d = angle_search_default()
    return AngleSearch(float(range_), d.step if step is None else float(step), int(samples))


def _picks(getter, h):
    n = C.c_int(0)
    getter(h, None, 0, C.byref(n))
    arr = (AnglePick * max(n.value, 1))()
    getter(h, arr, n.value, C.byref(n))
    return [arr[k].as_dict() for k in range(n.value)]


def pair_moments_transform(m, pose, new_origin=None):
    """Moments of the pairs after the rigid map p -> pose * p (4x4), about new_origin (default pose * origin)."""
    P = np.ascontiguousarray(np.asarray(pose, dtype=np.float64).T).reshape(16)
    o = None if new_origin is None else np.ascontiguousarray(new_origin, dtype=np.float64)
    out = PairMoments()
    lib().mvr_pair_moments_transform(C.byref(m), _dp(P), _dp(o) if o is not None else None, C.byref(out))
    return out


def lum_relax(edges, src, tgt, n_views, iterations=16):
    """pcl::registration::LUM::compute on correspondence moments (world frame): V rigid corrections, X[0] = I (float64)."""
    E = len(edges)
    arr = (PairMoments * max(E, 1))(*edges)
    s = np.ascontiguousarray(src, dtype=np.int32)
    t = np.ascontiguousarray(tgt, dtype=np.int32)
    out = np.empty((max(n_views, 1), 16), dtype=np.float64)
    rc = lib().mvr_lum_relax(arr, _ip(s), _ip(t), E, int(n_views), int(iterations), _dp(out))
    if rc != OK:
        raise MvrError(rc, lib().mvr_status_string(rc).decode())
    return [out[k].reshape(4, 4).T.copy() for k in range(n_views)]


def lum_compute(edges, src, tgt, n_views, iterations=16, convergence_threshold=0.0):
    """pcl::registration::LUM::compute() on moments: returns (poses V x 6, transforms list of V 4x4 float64)."""
    E = len(edges)
    arr = (PairMoments * max(E, 1))(*edges)
    s = np.ascontiguousarray(np.asarray(src, dtype=np.int32))
    t = np.ascontiguousarray(np.asarray(tgt, dtype=np.int32))
    p6 = np.zeros((n_views, 6), dtype=np.float64)
    X = np.zeros((n_views, 16), dtype=np.float64)
    rc = lib().mvr_lum_compute(arr, _ip(s), _ip(t), E, int(n_views), int(iterations), float(convergence_threshold), _dp(p6), _dp(X))
    if rc != OK:
        raise MvrError(rc, "mvr_lum_compute failed")
    return p6, [X[v].reshape(4, 4).T.copy() for v in range(n_views)]


def refine_axis(poses, pivot, axis):
    """Registrator::refineAxis: poses = list of registered views' 4x4; returns (pivot, axis)."""
    P = np.ascontiguousarray(np.stack([pose_from_numpy(T) for T in poses]), dtype=np.float32) if len(poses) else np.zeros((0, 16), np.float32)
    pv = np.ascontiguousarray(pivot, dtype=np.float64).copy()
    ax = np.ascontiguousarray(axis, dtype=np.float64).copy()
    rc = lib().mvr_refine_axis(_fp(P), len(poses), _dp(pv), _dp(ax))
    if rc != OK:
        raise MvrError(rc, lib().mvr_status_string(rc).decode())
    return pv, ax


class Registrator:
    """The reference's Registrator entry points (mvr/include/registrator.h:40-49) over `streams` GPU contexts."""

    def __init__(self, device=0, streams=1):
        self._h = C.c_void_p()
        rc = lib().mvr_registrator_create(int(device), int(streams), C.byref(self._h))
        if rc != OK:
            raise MvrError(rc, "mvr_registrator_create failed (no usable CUDA device %d; there is no CPU fallback)" % device)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().mvr_registrator_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def streams(self):
        return int(lib().mvr_registrator_streams(self._h))

    def context(self, slot=0):
        """The Context behind stream `slot` (borrowed: stays owned by the registrator)."""
        return Context(_borrowed=lib().mvr_registrator_context(self._h, int(slot)))

    @staticmethod
    def _views(views, init_poses=None):
        """views: list of n x 4 float32 arrays, or of (device_ptr, n) tuples."""
        arr = (ViewDesc * len(views))()
        keep = []
        for k, v in enumerate(views):
            if v is None:
                arr[k].xyzw, arr[k].n, arr[k].on_device = None, 0, 0
            elif isinstance(v, tuple):
                arr[k].xyzw, arr[k].n, arr[k].on_device = int(v[0]), int(v[1]), 1
            else:
                a = _pts(v)
                keep.append(a)
                arr[k].xyzw, arr[k].n, arr[k].on_device = a.ctypes.data, len(a), 0
            if init_poses is not None and init_poses[k] is not None:
                m = np.ascontiguousarray(np.asarray(init_poses[k], dtype=np.float64).T).reshape(16)
                keep.append(m)
                arr[k].init_pose = _dp(m)
        return arr, keep

    def pairwise_align(self, source, target, params, guess=None):
        arr, keep = self._views([source, target])
        g = pose_from_numpy(guess) if guess is not None else None
        fin = np.empty(16, dtype=np.float32)
        rep = IcpReport()
        rc = lib().mvr_pairwise_align(self._h, C.byref(arr[0]), C.byref(arr[1]), C.byref(params), _fp(g) if g is not None else None, _fp(fin), C.byref(rep))
        if rc not in (OK, ERR_TOO_FEW):
            raise MvrError(rc, (lib().mvr_registrator_last_error(self._h) or b"").decode())
        return dict(status=rc, final=pose_to_numpy(fin), iterations=rep.iterations, n_corr=rep.n_correspondences, mse=rep.mse,
                    gpu_ms=rep.gpu_ms, nn_queries=int(rep.nn_queries))

    def set_angle_search(self, range=None, step=None, samples=0):
        """Ring mode: score turns about the axis, j * step for |j| <= lround(range / step) (radians; step None: 1 degree), around
        every pair's guess and start each pair from the best (mvr_registrator_set_angle_search).  range None or <= 0: off."""
        s = _angle_search(range, step, samples)
        rc = lib().mvr_registrator_set_angle_search(self._h, C.byref(s) if s is not None else None)
        if rc != OK:
            raise MvrError(rc, (lib().mvr_registrator_last_error(self._h) or b"").decode())

    def angle_search_log(self):
        """One dict per pair of the last ring registration with the search on (AnglePick fields)."""
        return _picks(lib().mvr_registrator_get_angle_search, self._h)

    def fitness_log(self):
        """[(view, repeat, getFitnessScore())] of the last accumulative registration (the reference's fitness_scores.txt)."""
        n = C.c_int(0)
        lib().mvr_registrator_get_fitness_log(self._h, None, 0, C.byref(n))
        arr = (FitnessRecord * max(n.value, 1))()
        lib().mvr_registrator_get_fitness_log(self._h, arr, n.value, C.byref(n))
        return [(arr[k].view, arr[k].repeat, arr[k].score) for k in range(n.value)]

    def compute_error(self, views, poses, max_distance):
        """Registrator::computeError: [(count, mean squared distance)] of the reciprocal correspondences of neighbouring views."""
        V = len(views)
        arr, keep = self._views(views, poses)
        counts = (C.c_size_t * max(V, 1))()
        msd = np.zeros(max(V, 1), dtype=np.float64)
        n = C.c_int(0)
        rc = lib().mvr_compute_error(self._h, arr, V, float(max_distance), counts, _dp(msd), C.byref(n))
        if rc != OK:
            raise MvrError(rc, (lib().mvr_registrator_last_error(self._h) or b"").decode())
        return [(int(counts[k]), float(msd[k])) for k in range(n.value)]

    def bind_views(self, views, init_poses=None):
        """The view descriptors of a sequence, marshalled once: pass the result to register_turntable instead of the
        lists when the same buffers are registered again and again (bench.py)."""
        arr, keep = self._views(views, init_poses)
        return BoundViews(arr, keep, len(views), views)

    def register_turntable(self, views, params, init_poses=None, raw=False):
        """Returns (poses: list of V 4x4 float32, reports: list of dict); raw = True: (poses V x 16 float32 column-major,
        reports as a numpy record array of REPORT) without per-pair Python objects."""
        if isinstance(views, BoundViews):
            V, arr, keep = views.n, views.arr, views.keep
        else:
            V = len(views)
            arr, keep = self._views(views, init_poses)
        poses = np.empty((max(V, 1), 16), dtype=np.float32)
        reps = (PairReport * max(V, 1))()
        rc = lib().mvr_register_turntable(self._h, arr, V, C.byref(params), _fp(poses), reps)
        if rc != OK:
            raise MvrError(rc, (lib().mvr_registrator_last_error(self._h) or b"").decode())
        if raw:
            return poses, np.frombuffer(reps, dtype=REPORT, count=max(V, 1))
        n_rep = V if params.mode == RING_PAIRS else (0 if params.mode == LUM else max(V - 1, 0))
        reports = [dict(source_view=reps[k].source_view, target_view=reps[k].target_view, status=reps[k].status,
                        iterations=reps[k].iterations, n_corr=reps[k].n_correspondences, mse=reps[k].mse, fitness=reps[k].fitness,
                        gpu_ms=reps[k].gpu_ms, nn_queries=int(reps[k].nn_queries), pose=pose_to_numpy(reps[k].pose[:]))
                   for k in range(n_rep)]
        return [pose_to_numpy(poses[k]) for k in range(V)], reports


class MultiRegistrator:
    """mvr_multi: the multi-view-register entry point over several GPUs of one node, inside the C ABI (one host thread per
    GPU, one ncclAllGather of the pair records, host loop closure)."""

    def __init__(self, devices):
        devs = np.ascontiguousarray(np.asarray(list(devices), dtype=np.int32))
        self._h = C.c_void_p()
        rc = lib().mvr_multi_create(_ip(devs), len(devs), C.byref(self._h))
        if rc != OK:
            raise MvrError(rc, "mvr_multi_create failed (%s)" % lib().mvr_status_string(rc).decode())
        self.n = len(devs)
        self._keep = None

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().mvr_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != OK:
            raise MvrError(rc, (lib().mvr_multi_last_error(self._h) or b"").decode())

    def contexts(self, rank):
        """The (borrowed) Contexts of one rank."""
        return [Context(_borrowed=lib().mvr_multi_context(self._h, int(rank), k)) for k in range(int(lib().mvr_multi_contexts(self._h, int(rank))))]

    def set_angle_search(self, range=None, step=None, samples=0):
        """Registrator.set_angle_search on every rank."""
        s = _angle_search(range, step, samples)
        self._ck(lib().mvr_multi_set_angle_search(self._h, C.byref(s) if s is not None else None))

    def angle_search_log(self):
        """The records of every rank's pairs, in pair order."""
        return _picks(lib().mvr_multi_get_angle_search, self._h)

    def upload(self, views, init_poses=None):
        arr, keep = Registrator._views(views, init_poses)
        self._ck(lib().mvr_multi_upload(self._h, arr, len(views)))

    def register_turntable(self, views, params, init_poses=None, use_resident=False):
        """Returns (poses, reports, records as a numpy array of ring.RECORD, per-device ms)."""
        from . import ring
        V = len(views)
        arr, keep = Registrator._views(views, init_poses)
        poses = np.empty((max(V, 1), 16), dtype=np.float32)
        reps = (PairReport * max(V, 1))()
        recs = (PairRecord * max(V, 1))()
        ms = np.zeros(self.n, dtype=np.float64)
        self._ck(lib().mvr_register_turntable_multi(self._h, arr, V, C.byref(params), 1 if use_resident else 0, _fp(poses), reps, recs, _dp(ms)))
        reports = [dict(source_view=reps[k].source_view, target_view=reps[k].target_view, status=reps[k].status,
                        iterations=reps[k].iterations, n_corr=reps[k].n_correspondences, mse=reps[k].mse,
                        nn_queries=int(reps[k].nn_queries), pose=pose_to_numpy(reps[k].pose[:])) for k in range(V)]
        records = np.frombuffer(bytes(recs), dtype=ring.RECORD, count=V).copy()
        return [pose_to_numpy(poses[k]) for k in range(V)], reports, records, ms
