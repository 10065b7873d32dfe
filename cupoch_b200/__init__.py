"""cupoch_b200 -- B200-native drop-in for cupoch's ICP / kNN / voxel-grid hot path.

    import cupoch_b200 as cph
    res = cph.registration.registration_icp(source, target, 0.02, init,
            cph.registration.TransformationEstimationPointToPlane())

Mirrors `import cupoch as cph` for: cph.geometry.{PointCloud, KDTreeFlann, KDTreeSearchParamKNN,
KDTreeSearchParamRadius, VoxelGrid, OccupancyGrid, OccupancyVoxel}, cph.registration.{registration_icp,
registration_generalized_icp, registration_colored_icp, registration_fast_based_on_feature_matching,
FastGlobalRegistrationOption, ICPConvergenceCriteria, TransformationEstimation*
(user subclasses run the generic loop), RegistrationResult, compute_fpfh_feature, kabsch, kabsch_weighted},
cph.utility.{Vector3fVector, compute_jtj_jtr, compute_weighted_jtj_jtr}; cupoch_b200.distributed holds the
multi-GPU orchestration (torch.distributed).  All computation runs in libcupoch_b200.so (hand-written sm_100a CUDA);
there is no CPU fallback.
"""
from . import _lib, geometry, registration, utility  # noqa: F401

__version__ = "0.1.0"


def initialize_allocator(mode=None, initial_pool_size=0, devices=None):
    """cupoch.initialize_allocator(mode, initial_pool_size, devices) (cupoch_pybind.cpp:47-50,
    utility/device_vector.cu:28-69).  The B200 engine always allocates from the CUDA stream-ordered pool
    with an unlimited release threshold; `initial_pool_size` bytes are reserved up front so that no
    registration call has to grow the pool (a growth step costs tens of milliseconds)."""
    if initial_pool_size and initial_pool_size > 0:
        _lib.require_gpu()
        _lib.check(_lib.lib().cphb_reserve_pool(int(initial_pool_size)))
    return None
