"""cupoch.registration mirror: registration_icp / registration_generalized_icp / registration_colored_icp,
registration_fast_based_on_feature_matching, ICPConvergenceCriteria, TransformationEstimation*,
FastGlobalRegistrationOption, RegistrationResult.
Signatures follow src/python/cupoch_pybind/registration/registration.cpp:62-478.
"""
import ctypes as C

import numpy as np

from . import _lib
from .geometry import KDTreeSearchParamKNN, PointCloud
from .utility import DeviceArray, _DevicePool, as_f16


class ICPConvergenceCriteria:  # registration.h:35-49
    def __init__(self, relative_fitness=1e-6, relative_rmse=1e-6, max_iteration=30):
        self.relative_fitness = float(relative_fitness)
        self.relative_rmse = float(relative_rmse)
        self.max_iteration = int(max_iteration)

    def __repr__(self):
        return ("registration::ICPConvergenceCriteria class with relative_fitness=%e, relative_rmse=%e, "
                "and max_iteration=%d" % (self.relative_fitness, self.relative_rmse, self.max_iteration))


class TransformationEstimation:  # transformation_estimation.h:49-77
    _type = _lib.EST_UNSPECIFIED

    def get_transformation_estimation_type(self):
        return self._type

    def _corr_dev(self, corres):
        d = DeviceArray.wrap(np.ascontiguousarray(corres, np.int32).reshape(-1, 2), np.int32) if not isinstance(corres, DeviceArray) else corres
        return d, (len(d) if d is not None else 0)

    def compute_transformation(self, source, target, corres):
        """TransformationEstimation::ComputeTransformation on an explicit correspondence set (registration.cpp:115-118)."""
        _lib.require_gpu()
        d, n = self._corr_dev(corres)
        sc, tc = source._cloud(), target._cloud()
        p = _params(self, 0.0, ICPConvergenceCriteria())
        T = (C.c_float * 16)()
        _lib.check(_lib.lib().cphb_compute_transformation(self._type, C.byref(sc), C.byref(tc), d.ptr if n else None, n,
                                                          C.byref(p), T, None))
        return np.array(T, np.float32).reshape(4, 4)

    def compute_rmse(self, source, target, corres):
        """TransformationEstimation::ComputeRMSE (registration.cpp:111-114)."""
        _lib.require_gpu()
        d, n = self._corr_dev(corres)
        sc, tc = source._cloud(), target._cloud()
        p = _params(self, 0.0, ICPConvergenceCriteria())
        r = C.c_float(0)
        _lib.check(_lib.lib().cphb_compute_rmse(self._type, C.byref(sc), C.byref(tc), d.ptr if n else None, n, C.byref(p),
                                                C.byref(r), None))
        return float(r.value)


class TransformationEstimationPointToPoint(TransformationEstimation):
    _type = _lib.EST_POINT_TO_POINT

    def __repr__(self):
        return "TransformationEstimationPointToPoint"


class TransformationEstimationPointToPlane(TransformationEstimation):
    _type = _lib.EST_POINT_TO_PLANE

    def __init__(self, det_thresh=1e-6):
        self.det_thresh = float(det_thresh)

    def __repr__(self):
        return "TransformationEstimationPointToPlane"


class TransformationEstimationSymmetricMethod(TransformationEstimation):
    _type = _lib.EST_SYMMETRIC

    def __init__(self, det_thresh=1e-6):
        self.det_thresh = float(det_thresh)

    def __repr__(self):
        return "TransformationEstimationSymmetricMethod"


class TransformationEstimationForGeneralizedICP(TransformationEstimation):  # generalized_icp.h:14-52
    _type = _lib.EST_GENERALIZED_ICP

    def __init__(self, epsilon=1e-3):
        self.epsilon = float(epsilon)

    def __repr__(self):
        return "TransformationEstimationForGeneralizedICP with epsilon=%g" % self.epsilon


class TransformationEstimationForColoredICP(TransformationEstimation):  # colored_icp.cu:42-71
    _type = _lib.EST_COLORED_ICP

    def __init__(self, lambda_geometric=0.968, det_thresh=1e-6):
        if lambda_geometric < 0 or lambda_geometric > 1.0:
            lambda_geometric = 0.968
        self.lambda_geometric = float(lambda_geometric)
        self.det_thresh = float(det_thresh)


class RegistrationResult:  # registration.h:51-67
    """`correspondence_set` lives on the device like the reference's `correspondence_set_`; the host copy is
    made on first access, as the reference's pybind property does (registration.cpp:338-343)."""

    def __init__(self, transformation=None):
        self.transformation = np.eye(4, dtype=np.float32) if transformation is None else np.asarray(transformation, np.float32)
        self._corr_host = np.zeros((0, 2), np.int32)
        self._corr_dev, self._n_corr = None, 0
        self.inlier_rmse = 0.0
        self.fitness = 0.0
        self.iterations = 0
        self.converged = False

    @property
    def correspondence_set(self):
        if self._corr_dev is not None:
            self._corr_host = self._corr_dev.cpu(self._n_corr) if self._n_corr else np.zeros((0, 2), np.int32)
            _DevicePool.give(self._corr_dev)
            self._corr_dev = None
        return self._corr_host

    @correspondence_set.setter
    def correspondence_set(self, v):
        self._corr_dev = None
        self._corr_host = np.asarray(v, np.int32).reshape(-1, 2)

    def __del__(self):
        try:
            _DevicePool.give(self._corr_dev)
        except Exception:
            pass

    def __repr__(self):
        return ("registration::RegistrationResult with fitness=%f, inlier_rmse=%f, and correspondence_set size of %d"
                % (self.fitness, self.inlier_rmse, self._n_corr if self._corr_dev is not None else len(self._corr_host)))


ICP_NO_RETILE = 2   # CPHB_ICP_NO_RETILE
DEFAULT_FLAGS = 0   # OR of ICP_* flags applied to every registration (ablation / debugging)


def _params(estimation, max_distance, criteria, shard=None):
    p = _lib.IcpParams()
    p.shard_rank, p.shard_world = (int(shard[0]), int(shard[1])) if shard else (0, 0)
    p.estimation = estimation.get_transformation_estimation_type()
    p.max_correspondence_distance = float(max_distance)
    p.relative_fitness = criteria.relative_fitness
    p.relative_rmse = criteria.relative_rmse
    p.max_iteration = criteria.max_iteration
    p.det_thresh = getattr(estimation, "det_thresh", -1.0)
    p.lambda_geometric = getattr(estimation, "lambda_geometric", 0.968)
    p.flags = DEFAULT_FLAGS
    return p


def _result(res, corr, want_corr):
    out = RegistrationResult(np.array(res.transformation, np.float32).reshape(4, 4))
    out.fitness = float(res.fitness)
    out.inlier_rmse = float(res.inlier_rmse)
    out.iterations = int(res.iterations)
    out.converged = bool(res.converged)
    out.loop_ms = float(res.loop_ms)
    out.loop_launches = int(res.loop_launches)
    if want_corr:
        out._corr_dev, out._n_corr = corr, int(res.n_local_correspondences)
    return out


def registration_icp(source, target, max_correspondence_distance, init=None,
                     estimation_method=None, criteria=None, comm=None, return_correspondences=True, shard=None):
    """registration::RegistrationICP (registration.cu:121-173).
    Multi-GPU: pass `comm` (cupoch_b200.distributed.make_comm) and `shard=(rank, world)` with the FULL source on
    every rank; the library keeps this rank's Hilbert-contiguous block.  correspondence_set then holds this
    rank's pairs with global source indices."""
    estimation_method = estimation_method or TransformationEstimationPointToPoint()
    criteria = criteria or ICPConvergenceCriteria()
    init = np.eye(4, dtype=np.float32) if init is None else init
    if max_correspondence_distance <= 0.0:
        pass  # registration.cu:130-132 only logs; the search then yields no correspondences
    if estimation_method.get_transformation_estimation_type() == _lib.EST_UNSPECIFIED:
        if comm is not None or shard is not None:
            raise ValueError("user-defined TransformationEstimation runs the generic single-GPU loop")
        return _registration_icp_generic(source, target, max_correspondence_distance, init, estimation_method, criteria)
    _lib.require_gpu()
    sc, tc = source._cloud(), target._cloud()
    p = _params(estimation_method, max_correspondence_distance, criteria, shard)
    res = _lib.IcpResult()
    corr = _DevicePool.take((max(len(source), 1), 2), np.int32) if return_correspondences else None
    _lib.check(_lib.lib().cphb_registration_icp(C.byref(sc), C.byref(tc), as_f16(init), C.byref(p), comm,
                                                C.byref(res), corr.ptr if corr else None, None))
    return _result(res, corr, return_correspondences)


def _registration_icp_generic(source, target, max_correspondence_distance, init, estimation, criteria):
    """The reference's loop as written (registration.cu:145-172) for estimators the library has no fused path for:
    Python subclasses of TransformationEstimation that override compute_transformation(source, target, corres) -- what
    the reference's pybind trampoline PyTransformationEstimation (registration.cpp:36-60) makes possible.  Search and
    Transform run on the GPU through the same C ABI; only the user's estimator runs where the user wrote it.  `corres`
    is handed over as the host [n, 2] int32 array the reference's binding would convert it to."""
    _lib.require_gpu()
    T = np.array(np.asarray(init, np.float32).reshape(4, 4))
    pcd = source.clone()
    if not np.array_equal(T, np.eye(4, dtype=np.float32)):
        pcd.transform(T)
    result = evaluate_registration(pcd, target, max_correspondence_distance)
    result.transformation = T
    it = 0
    for it in range(1, max(criteria.max_iteration, 0) + 1):
        update = np.asarray(estimation.compute_transformation(pcd, target, result.correspondence_set), np.float32).reshape(4, 4)
        T = (update @ T).astype(np.float32)
        pcd.transform(update)
        backup_f, backup_r = result.fitness, result.inlier_rmse
        result = evaluate_registration(pcd, target, max_correspondence_distance)
        result.transformation = T
        if abs(backup_f - result.fitness) < criteria.relative_fitness and abs(backup_r - result.inlier_rmse) < criteria.relative_rmse:
            result.converged = True
            break
    result.iterations = it
    return result


def registration_icp_host(source_points, target_points, max_correspondence_distance, init=None, estimation_method=None,
                          criteria=None, source_normals=None, target_normals=None, source_colors=None, target_colors=None,
                          source_covariances=None, target_covariances=None, target_color_gradient=None, comm=None,
                          return_correspondences=False, shard=None, pairs_out=None):
    """registration::RegistrationICP straight from HOST arrays ([n,3] float32 numpy, ideally in pinned memory):
    one C-ABI call (cphb_registration_icp_host) uploads both clouds on a side stream, overlapping the copies with
    the index build and the source ordering, runs the loop and returns the result -- nothing stays on the device."""
    estimation_method = estimation_method or TransformationEstimationPointToPoint()
    criteria = criteria or ICPConvergenceCriteria()
    init = np.eye(4, dtype=np.float32) if init is None else init
    if estimation_method.get_transformation_estimation_type() == _lib.EST_UNSPECIFIED:
        # user-defined estimator (the reference's trampoline, registration.cpp:36-60): upload, then the generic loop
        if comm is not None or shard is not None:
            raise ValueError("user-defined TransformationEstimation runs the generic single-GPU loop")
        s_pc, t_pc = PointCloud(source_points), PointCloud(target_points)
        for pc, nrm, col, cov in ((s_pc, source_normals, source_colors, source_covariances),
                                  (t_pc, target_normals, target_colors, target_covariances)):
            if nrm is not None:
                pc.normals = nrm
            if col is not None:
                pc.colors = col
            if cov is not None:
                pc.covariances = cov
        out = _registration_icp_generic(s_pc, t_pc, max_correspondence_distance, init, estimation_method, criteria)
        if return_correspondences and pairs_out is not None:
            cs = out.correspondence_set
            pairs_out[:len(cs)] = cs
        return out
    _lib.require_gpu()

    def host(a, cols):
        if a is None:
            return None
        a = np.ascontiguousarray(a, np.float32)   # no copy for contiguous float32 input (keeps pinned memory pinned)
        if a.ndim < 2 or int(np.prod(a.shape[1:])) != cols:
            raise ValueError("expected [n, %d] float32" % cols)
        return a

    keep = [host(source_points, 3), host(target_points, 3), host(source_normals, 3), host(target_normals, 3),
            host(source_colors, 3), host(target_colors, 3), host(source_covariances, 9), host(target_covariances, 9),
            host(target_color_gradient, 3)]
    ptr = (lambda a: None if a is None else a.ctypes.data)
    sc, tc = _lib.Cloud(), _lib.Cloud()
    sc.points, sc.normals, sc.colors, sc.covariances, sc.n = ptr(keep[0]), ptr(keep[2]), ptr(keep[4]), ptr(keep[6]), len(keep[0])
    tc.points, tc.normals, tc.colors, tc.covariances, tc.n = ptr(keep[1]), ptr(keep[3]), ptr(keep[5]), ptr(keep[7]), len(keep[1])
    tc.color_gradient = ptr(keep[8])
    sc.cov_col_major = tc.cov_col_major = 0
    p = _params(estimation_method, max_correspondence_distance, criteria, shard)
    res = _lib.IcpResult()
    pairs = None
    if return_correspondences:
        # pairs_out: caller's [n, 2] int32 host array (pinned memory makes the D2H copy run at full PCIe speed)
        if pairs_out is not None and (pairs_out.dtype != np.int32 or not pairs_out.flags.c_contiguous or pairs_out.size < 2 * len(keep[0])):
            raise ValueError("pairs_out must be a C-contiguous int32 array of at least [n_source, 2]")
        pairs = pairs_out if pairs_out is not None else np.empty((max(len(keep[0]), 1), 2), np.int32)
    _lib.check(_lib.lib().cphb_registration_icp_host(C.byref(sc), C.byref(tc), as_f16(init), C.byref(p), comm, C.byref(res),
                                                     pairs.ctypes.data if pairs is not None else None, None))
    out = _result(res, None, False)
    if pairs is not None:
        out.correspondence_set = pairs[:int(res.n_local_correspondences)]
    return out


def evaluate_registration(source, target, max_correspondence_distance, transformation=None):
    """registration::EvaluateRegistration (registration.cu:106-119)."""
    T = np.eye(4, dtype=np.float32) if transformation is None else transformation
    _lib.require_gpu()
    sc, tc = source._cloud(False), target._cloud(False)
    res = _lib.IcpResult()
    corr = _DevicePool.take((max(len(source), 1), 2), np.int32)
    _lib.check(_lib.lib().cphb_evaluate_registration(C.byref(sc), C.byref(tc), float(max_correspondence_distance),
                                                     as_f16(T), C.byref(res), corr.ptr, None))
    return _result(res, corr, True)


def _with_covariances(pcd, epsilon):
    """InitializePointCloudForGeneralizedICP (generalized_icp.cu:37-61)."""
    if pcd.has_covariances():
        return pcd
    out = PointCloud()
    out._points, out._normals, out._colors = pcd._points, pcd._normals, pcd._colors
    if not out.has_normals():
        out.estimate_normals(KDTreeSearchParamKNN(20))
    n = len(out)
    cov = DeviceArray((n, 3, 3), np.float32)
    if n:
        _lib.check(_lib.lib().cphb_covariances_from_normals(out._normals.ptr, n, float(epsilon), cov.ptr, 0, None))
    out._covariances = cov
    return out


def registration_generalized_icp(source, target, max_correspondence_distance, init=None, estimation=None,
                                 criteria=None, comm=None, return_correspondences=True, shard=None):
    """registration::RegistrationGeneralizedICP (generalized_icp.cu:185-198)."""
    estimation = estimation or TransformationEstimationForGeneralizedICP()
    return registration_icp(_with_covariances(source, estimation.epsilon), _with_covariances(target, estimation.epsilon),
                            max_correspondence_distance, init, estimation, criteria, comm, return_correspondences, shard)


def initialize_pointcloud_for_colored_icp(target, radius, max_nn=30):
    """InitializePointCloudForColoredICP (colored_icp.cu:120-148)."""
    out = PointCloud()
    out._points, out._normals, out._colors = target._points, target._normals, target._colors
    n = len(out)
    grad = DeviceArray((n, 3), np.float32)
    if n:
        if not (out.has_normals() and out.has_colors()):
            _lib.check(_lib.lib().cphb_memset(grad.ptr, 0, grad.nbytes, None))
        else:
            _lib.check(_lib.lib().cphb_color_gradient(out._points.ptr, out._normals.ptr, out._colors.ptr, n,
                                                      float(radius), int(max_nn), grad.ptr, None))
    out._color_gradient = grad
    return out


def registration_colored_icp(source, target, max_correspondence_distance, init=None, criteria=None,
                             lambda_geometric=0.968, det_thresh=1e-6, comm=None, return_correspondences=True, shard=None):
    """registration::RegistrationColoredICP (colored_icp.cu:329-342)."""
    target_c = initialize_pointcloud_for_colored_icp(target, max_correspondence_distance * 2.0, 30)
    return registration_icp(source, target_c, max_correspondence_distance, init,
                            TransformationEstimationForColoredICP(lambda_geometric, det_thresh), criteria, comm,
                            return_correspondences, shard)


def kabsch(model, target, corres=None):
    """registration::Kabsch(model, target[, corres]) (kabsch.h:30-49) on device vectors / arrays."""
    _lib.require_gpu()
    m, t = DeviceArray.wrap(model), DeviceArray.wrap(target)
    T = (C.c_float * 16)()
    if corres is None:
        _lib.check(_lib.lib().cphb_kabsch(m.ptr, len(m), t.ptr, None, 0, T, None))
    else:
        d = DeviceArray.wrap(np.ascontiguousarray(corres, np.int32).reshape(-1, 2), np.int32)
        _lib.check(_lib.lib().cphb_kabsch(m.ptr, len(m), t.ptr, d.ptr, len(d), T, None))
    return np.array(T, np.float32).reshape(4, 4)


def kabsch_weighted(model, target, weight):
    """registration::KabschWeighted(model, target, weight) (kabsch.h:46-49) on device vectors / arrays."""
    _lib.require_gpu()
    m, t = DeviceArray.wrap(model), DeviceArray.wrap(target)
    w = DeviceArray.wrap(np.ascontiguousarray(weight, np.float32).reshape(-1) if not isinstance(weight, DeviceArray) else weight)
    if len(m) != len(t) or len(w) != len(m):
        raise ValueError("model, target and weight must have the same length")
    T = (C.c_float * 16)()
    _lib.check(_lib.lib().cphb_kabsch_weighted(m.ptr, t.ptr, w.ptr, len(m), T, None))
    return np.array(T, np.float32).reshape(4, 4)


class Feature:
    """registration::Feature<33> / Feature<352> (feature.h): `data` is [n, dim] float32 on the device; .cpu() downloads
    it.  (The reference stores it dimension-major for Python; here it is one row per point.)  Besides a DeviceArray,
    `data` may be anything DeviceArray.wrap accepts -- a numpy array, a torch tensor (CPU or CUDA) -- of shape
    [n, 33] or [n, 352], so that features computed elsewhere can be handed to the global registration."""

    def __init__(self, data):
        if not isinstance(data, DeviceArray):
            data = DeviceArray.wrap(data, np.float32)
            if len(data.shape) != 2 or data.shape[1] not in (33, 352):
                raise ValueError("Feature: expected [n, 33] or [n, 352], got %s" % (data.shape,))
        self.data = data

    def dimension(self):
        return self.data.shape[1]

    def num(self):
        return self.data.shape[0]

    def cpu(self):
        return self.data.cpu()


def compute_fpfh_feature(input, search_param):
    """registration::ComputeFPFHFeature (fpfh.cu:192-229)."""
    from .geometry import KDTreeSearchParamKNN, KDTreeSearchParamRadius
    _lib.require_gpu()
    n = len(input)
    out = DeviceArray((n, 33), np.float32)
    if n == 0:
        return Feature(out)
    if not input.has_normals():
        raise RuntimeError("[ComputeFPFHFeature] Failed because input point cloud has no normal.")
    if isinstance(search_param, KDTreeSearchParamKNN):
        knn, radius, max_nn = int(search_param.knn), 0.0, 0
    elif isinstance(search_param, KDTreeSearchParamRadius):
        knn, radius, max_nn = 0, float(search_param.radius), int(search_param.max_nn)
    else:
        raise RuntimeError("Unsupport search param type.")
    _lib.check(_lib.lib().cphb_compute_fpfh_feature(input._points.ptr, input._normals.ptr, n, knn, radius, max_nn, out.ptr, None))
    return Feature(out)


class FastGlobalRegistrationOption:  # fast_global_registration.h:43-104, registration.cpp:217-276
    """Options of registration_fast_based_on_feature_matching; defaults are the reference's."""

    def __init__(self, division_factor=1.4, use_absolute_scale=False, decrease_mu=True,
                 maximum_correspondence_distance=0.025, iteration_number=64, tuple_scale=0.95, maximum_tuple_count=1000):
        self.division_factor = float(division_factor)
        self.use_absolute_scale = bool(use_absolute_scale)
        self.decrease_mu = bool(decrease_mu)
        self.maximum_correspondence_distance = float(maximum_correspondence_distance)
        self.iteration_number = int(iteration_number)
        self.tuple_scale = float(tuple_scale)
        self.maximum_tuple_count = int(maximum_tuple_count)

    def _c(self):
        o = _lib.FgrOption()
        o.division_factor, o.use_absolute_scale, o.decrease_mu = self.division_factor, int(self.use_absolute_scale), int(self.decrease_mu)
        o.maximum_correspondence_distance, o.iteration_number = self.maximum_correspondence_distance, self.iteration_number
        o.tuple_scale, o.maximum_tuple_count = self.tuple_scale, self.maximum_tuple_count
        return o

    def __repr__(self):
        return ("registration::FastGlobalRegistrationOption with division_factor=%f use_absolute_scale=%d decrease_mu=%d "
                "maximum_correspondence_distance=%f iteration_number=%d tuple_scale=%f maximum_tuple_count=%d"
                % (self.division_factor, self.use_absolute_scale, self.decrease_mu, self.maximum_correspondence_distance,
                   self.iteration_number, self.tuple_scale, self.maximum_tuple_count))


def _features(f, n, what):
    if not isinstance(f, Feature):
        f = Feature(f)
    if f.num() != n:
        raise ValueError("%s: %d features for %d points" % (what, f.num(), n))
    return f


def registration_fast_based_on_feature_matching(source, target, source_feature, target_feature, option=None,
                                                return_trace=False):
    """registration::FastGlobalRegistration<33 | 352> (fast_global_registration.cu:391-431).  With return_trace the
    result also carries `trace` [iteration_number, 4, 4]: the pose in normalised coordinates after every iteration."""
    option = option or FastGlobalRegistrationOption()
    _lib.require_gpu()
    fs = _features(source_feature, len(source), "source_feature")
    ft = _features(target_feature, len(target), "target_feature")
    if fs.dimension() != ft.dimension():
        raise ValueError("source and target features differ in dimension")
    sc, tc = source._cloud(False), target._cloud(False)
    res = _lib.IcpResult()
    corr = _DevicePool.take((max(len(source), 1), 2), np.int32)
    tr = DeviceArray((max(option.iteration_number, 1), 16), np.float32) if return_trace else None
    _lib.check(_lib.lib().cphb_fast_global_registration(C.byref(sc), C.byref(tc), fs.data.ptr, fs.num(), ft.data.ptr, ft.num(),
                                                        fs.dimension(), C.byref(option._c()), C.byref(res), corr.ptr,
                                                        tr.ptr if tr is not None else None, None))
    out = _result(res, corr, True)
    if return_trace:
        out.trace = tr.cpu(max(option.iteration_number, 0)).reshape(-1, 4, 4)
    return out


def fgr_advanced_matching(source_points, target_points, source_feature, target_feature, option=None):
    """Test hook (cphb_fgr_advanced_matching): NormalizePointCloud + AdvancedMatching of the reference
    (fast_global_registration.cu:103-265) -> (pairs [m, 2] int32 (source, target), counts dict)."""
    option = option or FastGlobalRegistrationOption()
    _lib.require_gpu()
    sp, tp = DeviceArray.wrap(source_points), DeviceArray.wrap(target_points)
    fs, ft = _features(source_feature, len(sp), "source_feature"), _features(target_feature, len(tp), "target_feature")
    out = DeviceArray((max(option.maximum_tuple_count, 1), 2), np.int32)
    counts = (C.c_int64 * 4)()
    _lib.check(_lib.lib().cphb_fgr_advanced_matching(sp.ptr, len(sp), tp.ptr, len(tp), fs.data.ptr, fs.num(), ft.data.ptr,
                                                     ft.num(), fs.dimension(), C.byref(option._c()), out.ptr, counts, None))
    return out.cpu(counts[0]), {"pairs": counts[0], "mutual": counts[1], "trials": counts[2], "passing_pairs": counts[3]}


def bruteforce_nn(ref, query, both_directions=False):
    """knn::BruteForceNN<33 | 352>(ref, query, indices, distances) (bruteforce_nn.inl:101-135) on [n, dim] features:
    -> (indices [m] int32, squared distances [m] float32) of the nearest ref row for every query row.  With
    both_directions also (indices [n], squared distances [n]) of the nearest query row for every ref row, from the
    same distance evaluations (the two-way matcher of the global registration)."""
    _lib.require_gpu()
    r = ref if isinstance(ref, Feature) else Feature(ref)
    q = query if isinstance(query, Feature) else Feature(query)
    dim = r.dimension() if r.dimension() == q.dimension() else -1
    idx, d2 = DeviceArray((max(q.num(), 1),), np.int32), DeviceArray((max(q.num(), 1),), np.float32)
    ridx = DeviceArray((max(r.num(), 1),), np.int32) if both_directions else None
    rd2 = DeviceArray((max(r.num(), 1),), np.float32) if both_directions else None
    _lib.check(_lib.lib().cphb_feature_nn(r.data.ptr, r.num(), q.data.ptr, q.num(), dim, idx.ptr, d2.ptr,
                                          ridx.ptr if ridx else None, rd2.ptr if rd2 else None, None))
    out = (idx.cpu(q.num()), d2.cpu(q.num()))
    return out + (ridx.cpu(r.num()), rd2.cpu(r.num())) if both_directions else out


class IcpContext:
    """Reusable RegistrationICP state (index + Hilbert-ordered source), for repeated runs and
    the per-step test hook.  Thin wrapper over cphb_icp_create / _run / _step."""

    def __init__(self, source, target, max_correspondence_distance, estimation_method=None, criteria=None):
        _lib.require_gpu()
        self.source, self.target = source, target  # keep device buffers alive
        estimation_method = estimation_method or TransformationEstimationPointToPoint()
        criteria = criteria or ICPConvergenceCriteria()
        self._p = _params(estimation_method, max_correspondence_distance, criteria)
        sc, tc = source._cloud(), target._cloud()
        self._h = C.c_void_p()
        _lib.check(_lib.lib().cphb_icp_create(C.byref(sc), C.byref(tc), C.byref(self._p), None, C.byref(self._h)))
        self._corr = DeviceArray((max(len(source), 1), 2), np.int32)
        self._ci = DeviceArray((max(len(source), 1),), np.int32)

    def run(self, init=None, comm=None, return_correspondences=True):
        init = np.eye(4, dtype=np.float32) if init is None else init
        res = _lib.IcpResult()
        _lib.check(_lib.lib().cphb_icp_run(self._h, as_f16(init), comm, C.byref(res),
                                           self._corr.ptr if return_correspondences else None, None))
        out = _result(res, None, False)
        if return_correspondences:
            nl = int(res.n_local_correspondences)
            out.correspondence_set = self._corr.cpu(nl) if nl else np.zeros((0, 2), np.int32)
        return out

    def step(self, T):
        """-> (sums[32] float64, corr_index[n] int32) at pose T applied to the pristine source."""
        sums = (C.c_double * 32)()
        _lib.check(_lib.lib().cphb_icp_step(self._h, as_f16(T), sums, self._ci.ptr, None))
        return np.array(sums, np.float64), self._ci.cpu()[:len(self.source)]

    def close(self):
        if self._h:
            _lib.lib().cphb_stream_synchronize(None)
            _lib.lib().cphb_icp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
