"""Counterpart of the reference's examples/python/advanced/fast_global_registration.py: FPFH features, then
FastGlobalRegistration from no initial pose, then point-to-plane ICP refinement.  The clouds are two overlapping
crops of a seeded non-periodic scene (cupoch_b200.testing.datagen.bumps_scene), the source moved by the 90-degree
permutation rotation of the reference's global_registration.py."""
import time

import numpy as np

import cupoch_b200 as cph
from cupoch_b200.testing import datagen


def prepare_dataset(voxel_size):
    pts = datagen.bumps_scene(200_000, 3)
    src, tgt = pts[pts[:, 0] < 0.7], pts[pts[:, 0] > 0.3]
    gt = np.array([[0, 0, 1, 0.4], [1, 0, 0, -0.2], [0, 1, 0, 0.3], [0, 0, 0, 1]], np.float64)
    gi = np.linalg.inv(gt)
    src = (src @ gi[:3, :3].T + gi[:3, 3]).astype(np.float32)
    out = []
    for p in (src, tgt):
        down = cph.geometry.PointCloud(p).voxel_down_sample(voxel_size)
        down.estimate_normals(cph.geometry.KDTreeSearchParamRadius(voxel_size * 2, 30))
        fpfh = cph.registration.compute_fpfh_feature(down, cph.geometry.KDTreeSearchParamRadius(voxel_size * 5, 100))
        out += [down, fpfh]
    return out + [gt]


if __name__ == "__main__":
    voxel_size = 0.02
    source_down, source_fpfh, target_down, target_fpfh, gt = prepare_dataset(voxel_size)
    start = time.time()
    result = cph.registration.registration_fast_based_on_feature_matching(
        source_down, target_down, source_fpfh, target_fpfh,
        cph.registration.FastGlobalRegistrationOption(maximum_correspondence_distance=voxel_size * 0.5))
    print("Fast global registration took %.3f sec." % (time.time() - start))
    print(result)
    print(result.transformation)
    refined = cph.registration.registration_icp(source_down, target_down, voxel_size, result.transformation,
                                                cph.registration.TransformationEstimationPointToPlane())
    print(refined)
    print("distance to the ground-truth pose (Frobenius):", float(np.linalg.norm(refined.transformation - gt)))
