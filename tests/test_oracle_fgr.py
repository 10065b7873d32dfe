"""CPU checks of the FastGlobalRegistration oracle (tests/fgr_oracle.c): thrust's RNG bit for bit, the matching
properties of AdvancedMatching, the BruteForceNN tie rule, and pose recovery on a non-periodic scene."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import fgr_oracle as F

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

_THRUST_PROG = r"""
#include <cstdio>
#include <cstdlib>
#include <thrust/random.h>
int main(int argc, char **argv) {
    for (int a = 1; a + 1 < argc; a += 2) {
        size_t idx = strtoull(argv[a], 0, 10); int ncorr = atoi(argv[a + 1]);
        thrust::default_random_engine eng; thrust::uniform_int_distribution<int> dist(0, ncorr - 1);
        eng.discard(idx);
        int r0 = dist(eng), r1 = dist(eng), r2 = dist(eng);
        printf("%d %d %d\n", r0, r1, r2);
    }
}
"""


def test_minstd_draws_equal_thrust(tmp_path):
    """the tuple test's draws (compute_tuple_constraint_functor, fast_global_registration.cu:37-45) equal the toolkit's
    thrust::default_random_engine + uniform_int_distribution"""
    if not (os.path.exists(NVCC) or shutil.which("nvcc")):
        pytest.skip("nvcc not available")
    src = tmp_path / "draws.cu"
    src.write_text(_THRUST_PROG)
    exe = tmp_path / "draws"
    subprocess.check_call([NVCC if os.path.exists(NVCC) else "nvcc", "-O2", "-o", str(exe), str(src)])
    cases = [(0, 5000), (1, 5000), (2, 5000), (1000, 5000), (123456, 5000), (0, 1), (7, 3), (99999, 1000),
             (2 ** 31 + 5, 250000), (31415926, 77)]
    out = subprocess.check_output([str(exe)] + [str(v) for c in cases for v in c], text=True).split("\n")
    want = [tuple(int(x) for x in line.split()) for line in out if line.strip()]
    got = [F.minstd_draws(i, n) for i, n in cases]
    assert got == want
    assert got[0] == (0, 425, 3006) and got[1][0] == got[0][1]  # consecutive trials overlap


def _cloud_and_features(n, seed, dim=33, levels=None):
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    f = (rng.integers(0, levels, (n, dim)) if levels else rng.uniform(0, 100, (n, dim))).astype(np.float32)
    return pts, f


def _numpy_nn(ref, query):
    d = ((query.astype(np.float64)[:, None, :] - ref.astype(np.float64)[None]) ** 2).sum(-1)
    return d.argmin(1)


def test_feature_nn_matches_float64_and_tie_rule():
    ref, fr = _cloud_and_features(300, 1)
    _, fq = _cloud_and_features(200, 2)
    idx, d2 = F.feature_nn(fr, fq)
    assert np.array_equal(idx, _numpy_nn(fr, fq))  # continuous features: no near-ties at this size
    # duplicated rows and all-zero rows (FPFH on planes): the first index with the smallest distance wins
    fr2 = np.zeros((40, 33), np.float32)
    fr2[10:20] = fr[:10]
    fr2[20:30] = fr[:10]
    q = np.concatenate([np.zeros((3, 33), np.float32), fr[:10]])
    idx, d2 = F.feature_nn(fr2, q)
    assert list(idx[:3]) == [0, 0, 0] and np.all(d2[:3] == 0)
    assert list(idx[3:]) == list(range(10, 20)) and np.all(d2[3:] == 0)
    # integer features: many exact ties; the reference's strict-< scan keeps the smallest index
    _, fi = _cloud_and_features(120, 3, levels=2)
    _, fj = _cloud_and_features(90, 4, levels=2)
    idx, d2 = F.feature_nn(fi, fj)
    d = ((fj[:, None, :] - fi[None]) ** 2).sum(-1)
    assert np.array_equal(idx, d.argmin(1)) and np.array_equal(d2, d.min(1))


@pytest.mark.parametrize("ns,nt", [(700, 500), (500, 700)])
def test_advanced_matching_properties(ns, nt):
    src, fs = _cloud_and_features(ns, 10)
    tgt, ft = _cloud_and_features(nt, 11)
    # plant 300 true matches so that the tuple test has survivors
    ft[:300] = fs[:300] + np.float32(0.01)
    tgt[:300] = src[:300] + np.float32(0.1)
    opt = F.option(maximum_tuple_count=100)
    pairs, counts, mutual, swapped = F.advanced_matching(src, tgt, fs, ft, opt)
    assert swapped == (nt > ns)
    fi, fj = (ft, fs) if swapped else (fs, ft)
    nn_i, nn_j = _numpy_nn(fj, fi), _numpy_nn(fi, fj)
    want = np.array([(i, nn_i[i]) for i in range(len(fi)) if nn_j[nn_i[i]] == i], np.int32)
    assert np.array_equal(mutual, want)  # mutual nearest neighbours, in fi order
    assert counts["mutual"] == len(want) and counts["trials"] == 100 * len(want)
    assert counts["passing_pairs"] % 3 == 0 and counts["passing_pairs"] > counts["pairs"] == 100  # truncated at pairs
    # every whole kept triplet satisfies the scale test (recomputed in float64 with a margin for the float32 test)
    nrm = F.normalize(src, tgt)
    ps = (src - nrm["mean_source"]) / nrm["scale_global"]
    pt = (tgt - nrm["mean_target"]) / nrm["scale_global"]
    for t in range(len(pairs) // 3):
        a, b = ps[pairs[3 * t:3 * t + 3, 0]], pt[pairs[3 * t:3 * t + 3, 1]]
        for k in range(3):
            li = np.linalg.norm(a[k] - a[(k + 1) % 3])
            lj = np.linalg.norm(b[k] - b[(k + 1) % 3])
            assert li * 0.95 * (1 - 1e-5) < lj < li / 0.95 * (1 + 1e-5)
    # pairs are (source index, target index) and every pair is a mutual match
    mset = {(int(i), int(j)) for i, j in want}
    for s, t in pairs:
        assert ((int(t), int(s)) if swapped else (int(s), int(t))) in mset
    # without truncation the list holds every passing pair
    pairs_all, c2, _, _ = F.advanced_matching(src, tgt, fs, ft, F.option(maximum_tuple_count=10 ** 7))
    assert c2["pairs"] == c2["passing_pairs"] and np.array_equal(pairs_all[:100], pairs)


def test_fewer_than_ten_pairs_gives_mean_translation():
    src, _ = _cloud_and_features(50, 20)
    tgt, _ = _cloud_and_features(40, 21)
    T, trace = F.optimize(src, tgt, np.zeros((6, 2), np.int32))
    nrm = F.normalize(src, tgt)
    assert np.array_equal(T[:3, :3], np.eye(3, dtype=np.float32))
    assert np.array_equal(T[:3, 3], nrm["mean_target"] - nrm["mean_source"])
    assert np.array_equal(trace, np.broadcast_to(np.eye(4, dtype=np.float32), trace.shape))


# pose tolerance fixed by the CPU run of this scene: 0.96 deg / 4.8 mm at voxel 0.02
@pytest.mark.parametrize("voxel", [0.02])
def test_fgr_recovers_pose_on_bumps_scene(orc, voxel):
    src, tgt, T_gt = F.fgr_scene(60000, 3, voxel)
    s, _, _ = orc.voxel_down_sample(src, voxel)
    t, _, _ = orc.voxel_down_sample(tgt, voxel)
    sn, tn = orc.estimate_normals(s, 0, 2 * voxel, 30), orc.estimate_normals(t, 0, 2 * voxel, 30)
    fs, ft = orc.compute_fpfh_feature(s, sn, 0, 5 * voxel, 100), orc.compute_fpfh_feature(t, tn, 0, 5 * voxel, 100)
    r = F.fast_global_registration(orc, s, t, fs, ft, F.option(maximum_correspondence_distance=0.5 * voxel))
    ang, dt = F.pose_error(r["transformation"], T_gt)
    assert ang < 2.0 and dt < 0.01, (ang, dt)
    assert r["fitness"] > 0.5


def test_oracle_fpfh_matches_reference_known_answer(orc):
    """FGR's input: the reference's ComputeFPFHFeature known-answer test (feature.cpp:30-155) at its 1e-4"""
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fpfh_ref.json")) as f:
        g = json.load(f)
    got = orc.compute_fpfh_feature(np.array(g["points"]), np.array(g["normals"]), 0, g["radius"], g["max_nn"])
    assert got.shape == (20, 33)
    np.testing.assert_allclose(got, np.array(g["expected"], np.float32), rtol=0, atol=g["tolerance"])
