"""FastGlobalRegistration and the fused feature matcher on the GPU against the CPU oracle (tests/fgr_oracle.c):
indices and d2 bits, pair lists, per-iteration poses and the final RegistrationResult at array_equal."""
import numpy as np
import pytest

import cupoch_b200 as cph
from cupoch_b200 import _lib
import fgr_oracle as F

R = cph.registration
pytestmark = pytest.mark.gpu


def _feat(n, dim, seed, levels=None):
    rng = np.random.default_rng(seed)
    if levels:
        return rng.integers(0, levels, (n, dim)).astype(np.float32)
    return rng.uniform(0, 100, (n, dim)).astype(np.float32)


def _pts(n, seed):
    return np.random.default_rng(seed).uniform(-1, 1, (n, 3)).astype(np.float32)


def _opt(o):
    return R.FastGlobalRegistrationOption(o.division_factor, bool(o.use_absolute_scale), bool(o.decrease_mu),
                                          o.maximum_correspondence_distance, o.iteration_number, o.tuple_scale,
                                          o.maximum_tuple_count)


@pytest.mark.parametrize("dim", [33, 352])
@pytest.mark.parametrize("nr,nq", [(1, 1), (17, 17), (3001, 4099), (4099, 3001)])
def test_feature_nn_equals_oracle(dim, nr, nq):
    ref, qry = _feat(nr, dim, 1), _feat(nq, dim, 2)
    idx, d2 = R.bruteforce_nn(ref, qry)
    oi, od = F.feature_nn(ref, qry)
    assert np.array_equal(idx, oi) and np.array_equal(d2.view(np.uint32), od.view(np.uint32))


@pytest.mark.parametrize("dim", [33, 352])
def test_feature_nn_ties(dim):
    ref = _feat(700, dim, 3, levels=2)
    ref[100:200] = 0.0
    ref[300:350] = ref[400:450]
    qry = np.concatenate([_feat(600, dim, 4, levels=2), np.zeros((5, dim), np.float32), ref[400:450]])
    idx, d2 = R.bruteforce_nn(ref, qry)
    oi, od = F.feature_nn(ref, qry)
    assert np.array_equal(idx, oi) and np.array_equal(d2.view(np.uint32), od.view(np.uint32))
    assert np.all(idx[-50:] == np.arange(300, 350))


@pytest.mark.parametrize("dim", [33, 352])
@pytest.mark.parametrize("nr,nq,levels", [(1, 1, None), (17, 17, None), (3001, 4099, None), (4099, 3001, None),
                                          (700, 650, 2)])
def test_feature_nn_two_way_equals_oracle(dim, nr, nq, levels):
    """the column direction of the two-way matcher (what the cross check of FastGlobalRegistration reads)"""
    ref, qry = _feat(nr, dim, 11, levels), _feat(nq, dim, 12, levels)
    if levels:
        ref[100:200] = 0.0
        qry[50:80] = 0.0
        ref[300:350] = ref[400:450]
        qry[500:550] = ref[400:450]
    idx, d2, ridx, rd2 = R.bruteforce_nn(ref, qry, both_directions=True)
    oi, od = F.feature_nn(ref, qry)
    ri, rd = F.feature_nn(qry, ref)
    assert np.array_equal(idx, oi) and np.array_equal(d2.view(np.uint32), od.view(np.uint32))
    assert np.array_equal(ridx, ri) and np.array_equal(rd2.view(np.uint32), rd.view(np.uint32))


def test_feature_nn_two_way_50k_by_60k_sampled():
    ref, qry = _feat(60000, 33, 15), _feat(50000, 33, 16)
    idx, d2, ridx, rd2 = R.bruteforce_nn(ref, qry, both_directions=True)
    rng = np.random.default_rng(17)
    rows, cols = rng.choice(len(qry), 300, replace=False), rng.choice(len(ref), 300, replace=False)
    oi, od = F.feature_nn(ref, qry[rows])
    ri, rd = F.feature_nn(qry, ref[cols])
    assert np.array_equal(idx[rows], oi) and np.array_equal(d2[rows].view(np.uint32), od.view(np.uint32))
    assert np.array_equal(ridx[cols], ri) and np.array_equal(rd2[cols].view(np.uint32), rd.view(np.uint32))


def test_gpu_fpfh_matches_reference_known_answer():
    """ComputeFPFHFeature on the GPU against the reference's known answer (feature.cpp:30-155) at its 1e-4"""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fpfh_ref.json")) as f:
        g = json.load(f)
    pc = cph.geometry.PointCloud(np.array(g["points"], np.float32))
    pc.normals = np.array(g["normals"], np.float32)
    got = R.compute_fpfh_feature(pc, cph.geometry.KDTreeSearchParamRadius(g["radius"], g["max_nn"])).cpu()
    np.testing.assert_allclose(got, np.array(g["expected"], np.float32), rtol=0, atol=g["tolerance"])


def test_feature_nn_50k_by_60k_sampled():
    ref, qry = _feat(60000, 33, 5), _feat(50000, 33, 6)
    idx, d2 = R.bruteforce_nn(ref, qry)
    rows = np.random.default_rng(7).choice(len(qry), 400, replace=False)
    oi, od = F.feature_nn(ref, qry[rows])
    assert np.array_equal(idx[rows], oi) and np.array_equal(d2[rows].view(np.uint32), od.view(np.uint32))


def _planted(ns, nt, seed, dim=33, n_true=400):
    src, tgt = _pts(ns, seed), _pts(nt, seed + 1)
    fs, ft = _feat(ns, dim, seed + 2), _feat(nt, dim, seed + 3)
    ft[:n_true] = fs[:n_true] + np.float32(0.5)
    tgt[:n_true] = src[:n_true] + np.float32(0.2)
    return src, tgt, fs, ft


@pytest.mark.parametrize("ns,nt,dim", [(2000, 1500, 33), (1500, 2000, 33), (1200, 1300, 352)])
@pytest.mark.parametrize("absolute,mu", [(False, True), (True, False)])
def test_advanced_matching_equals_oracle(ns, nt, dim, absolute, mu):
    src, tgt, fs, ft = _planted(ns, nt, 30, dim)
    o = F.option(use_absolute_scale=absolute, decrease_mu=mu)
    pairs, counts = R.fgr_advanced_matching(src, tgt, fs, ft, _opt(o))
    opairs, ocounts, _, _ = F.advanced_matching(src, tgt, fs, ft, o)
    assert counts == ocounts
    assert np.array_equal(pairs, opairs)
    assert counts["pairs"] == min(1000, counts["passing_pairs"]) > 10


@pytest.mark.parametrize("ns,nt", [(2000, 1500), (1500, 2000)])
@pytest.mark.parametrize("absolute,mu", [(False, True), (True, False), (False, False)])
def test_fgr_trace_and_result_equal_oracle(orc, ns, nt, absolute, mu):
    src, tgt, fs, ft = _planted(ns, nt, 40)
    o = F.option(use_absolute_scale=absolute, decrease_mu=mu, maximum_correspondence_distance=0.05, iteration_number=32)
    res = R.registration_fast_based_on_feature_matching(cph.geometry.PointCloud(src), cph.geometry.PointCloud(tgt),
                                                        R.Feature(fs), R.Feature(ft), _opt(o), return_trace=True)
    ref = F.fast_global_registration(orc, src, tgt, fs, ft, o)
    assert np.array_equal(res.trace, ref["trace"])
    assert float(np.abs(res.transformation.astype(np.float64) - ref["transformation"]).max()) == 0.0
    assert res.fitness == ref["fitness"] and res.inlier_rmse == ref["inlier_rmse"]
    assert np.array_equal(res.correspondence_set, ref["correspondence_set"])


def test_fgr_fewer_than_ten_pairs_gives_mean_translation(orc):
    src, tgt = _pts(300, 50), _pts(200, 51)
    fs, ft = _feat(300, 33, 52), _feat(200, 33, 53)
    o = F.option(maximum_tuple_count=6)
    res = R.registration_fast_based_on_feature_matching(cph.geometry.PointCloud(src), cph.geometry.PointCloud(tgt), fs, ft,
                                                        _opt(o))
    nrm = F.normalize(src, tgt)
    assert np.array_equal(res.transformation[:3, :3], np.eye(3, dtype=np.float32))
    assert np.array_equal(res.transformation[:3, 3], nrm["mean_target"] - nrm["mean_source"])
    ref = F.fast_global_registration(orc, src, tgt, fs, ft, o)
    assert np.array_equal(res.transformation, ref["transformation"]) and res.fitness == ref["fitness"]


def test_fgr_empty_inputs_give_default_result():
    empty = cph.geometry.PointCloud(np.zeros((0, 3), np.float32))
    full = cph.geometry.PointCloud(_pts(50, 60))
    for s, t, fs, ft in ((empty, full, np.zeros((0, 33), np.float32), _feat(50, 33, 61)),
                         (full, empty, _feat(50, 33, 61), np.zeros((0, 33), np.float32))):
        res = R.registration_fast_based_on_feature_matching(s, t, fs, ft)
        assert np.array_equal(res.transformation, np.eye(4, dtype=np.float32))
        assert res.fitness == 0.0 and res.inlier_rmse == 0.0 and len(res.correspondence_set) == 0


def test_fgr_bad_inputs_raise_before_any_launch():
    from cupoch_b200.utility import DeviceArray
    import ctypes as C
    L = _lib.lib()
    src, tgt = DeviceArray.from_numpy(_pts(50, 70)), DeviceArray.from_numpy(_pts(40, 71))
    fs, ft = DeviceArray.from_numpy(_feat(50, 33, 72)), DeviceArray.from_numpy(_feat(40, 33, 73))
    sc, tc = _lib.Cloud(), _lib.Cloud()
    sc.points, sc.n, tc.points, tc.n = src.ptr, 50, tgt.ptr, 40
    o = _lib.FgrOption()
    L.cphb_fgr_default_option(o)
    res = _lib.IcpResult()
    before = L.cphb_launch_count()
    for args in ((fs.ptr, 49, ft.ptr, 40, 33), (fs.ptr, 50, ft.ptr, 41, 33), (fs.ptr, 50, ft.ptr, 40, 32),
                 (fs.ptr, 50, ft.ptr, 40, 0)):
        rc = L.cphb_fast_global_registration(C.byref(sc), C.byref(tc), args[0], args[1], args[2], args[3], args[4],
                                             C.byref(o), C.byref(res), None, None, None)
        assert rc == -1  # CPHB_ERR_INVALID
    assert L.cphb_launch_count() == before
    with pytest.raises(ValueError):
        R.registration_fast_based_on_feature_matching(cph.geometry.PointCloud(_pts(50, 70)), cph.geometry.PointCloud(_pts(40, 71)),
                                                      _feat(49, 33, 72), _feat(40, 33, 73))
    bad = _feat(40, 33, 73)
    bad[7, 3] = np.nan
    before = L.cphb_launch_count()
    with pytest.raises(_lib.CphbError, match="non-finite"):
        R.registration_fast_based_on_feature_matching(cph.geometry.PointCloud(_pts(50, 70)), cph.geometry.PointCloud(_pts(40, 71)),
                                                      _feat(50, 33, 72), bad)
    # found by the matcher itself: the normalisation and the matcher ran, no later stage did
    assert L.cphb_launch_count() - before <= 2


def test_fgr_pipeline_recovers_pose_then_icp_refines():
    voxel = 0.02
    src, tgt, T_gt = F.fgr_scene(60000, 3, voxel)
    G = cph.geometry
    s, t = G.PointCloud(src).voxel_down_sample(voxel), G.PointCloud(tgt).voxel_down_sample(voxel)
    for pc in (s, t):
        pc.estimate_normals(G.KDTreeSearchParamRadius(2 * voxel, 30))
    fs = R.compute_fpfh_feature(s, G.KDTreeSearchParamRadius(5 * voxel, 100))
    ft = R.compute_fpfh_feature(t, G.KDTreeSearchParamRadius(5 * voxel, 100))
    res = R.registration_fast_based_on_feature_matching(s, t, fs, ft, R.FastGlobalRegistrationOption(
        maximum_correspondence_distance=0.5 * voxel))
    ang, dt = F.pose_error(res.transformation, T_gt)
    assert ang < 2.0 and dt < 0.01, (ang, dt)
    icp = R.registration_icp(s, t, voxel, res.transformation, R.TransformationEstimationPointToPlane())
    ang2, dt2 = F.pose_error(icp.transformation, T_gt)
    assert ang2 < 0.5 and dt2 < 0.005, (ang2, dt2)


def test_feature_nn_200k_scale_sampled():
    """the reference's distance matrix would be 160 GB here; the fused matcher keeps one key per row"""
    n = 200000
    ref, qry = _feat(n, 33, 80), _feat(n, 33, 81)
    src, tgt = _pts(n, 82), _pts(n, 83)
    pairs, counts = R.fgr_advanced_matching(src, tgt, ref, qry)
    assert counts["pairs"] <= 1000
    idx, d2 = R.bruteforce_nn(ref, qry)
    rows = np.random.default_rng(84).choice(n, 2000, replace=False)
    oi, od = F.feature_nn(ref, qry[rows])
    assert np.array_equal(idx[rows], oi) and np.array_equal(d2[rows].view(np.uint32), od.view(np.uint32))
