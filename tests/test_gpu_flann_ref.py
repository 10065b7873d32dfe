"""GPU parity against the REFERENCE'S OWN search engine: the FLANN CUDA kd-tree cupoch vendors
(third_party/flann/algorithms/kdtree_cuda_3d_index.cu), called exactly like cupoch::knn::KDTreeFlann calls it
(kdtree_flann.inl:70-144).  This pins the search row (SURVEY 8a R1/R1b) to reference CODE, not to a restatement:

  * which point is returned (index) and its d2 -- BIT-IDENTICAL: the product computes d2 in the operation order the
    reference's kernel has in SASS (FMUL dy,dy; FFMA dx,dx; FFMA dz,dz) -- on random clouds and on the ICP workload;
  * the tie rule (DESIGN.md hazard 1): FLANN keeps the first-visited of equal-distance points in kd order, the
    product keeps the smallest index -- measured here, asserted only through d2 (the distances must agree);
  * k > 1 radius results that are not full (R1b, result_set.h:405-473): same SET of neighbours.

The reference's answers are stored in tests/golden/flann_ref.npz (written by tools/make_flann_golden.py, which runs
the reference binary on the inputs defined here).  The full answers (tens of MB) are too large to keep, so the
golden file holds, per comparison:
  * 1-NN: SHA-256 digests of the found mask and of d2 over ALL queries (membership and d2 are compared bit for bit
    everywhere), and index + d2 of a seeded sample of the queries;
  * the tie lattice: the whole answer;
  * k > 1: a CRC-32 of each query's sorted neighbour set (sets are compared for every query), and for kNN a digest
    of the row-sorted d2 of all queries.
"""
import hashlib
import os
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cupoch_b200 as cph
from cupoch_b200.testing import datagen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "flann_ref.npz")
SAMPLE = 1024   # 1-NN queries whose reference index and d2 are stored


def _lattice():
    g = np.stack(np.meshgrid(*[np.arange(12, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.25
    tgt = np.concatenate([g, g[::3], g[::7]]).astype(np.float32)
    tgt = tgt[np.random.default_rng(3).permutation(len(tgt))]
    return tgt, np.concatenate([g + 0.125, g]).astype(np.float32)


def _config2():
    tgt, _ = datagen.surface(1_000_000, 11)
    return tgt, datagen.make_source(tgt, datagen.gt_transform(), 13, 14, 5e-4)


_UNIFORM = lambda: (datagen.uniform_cube(200_000, 101),
                    datagen.uniform_cube(100_000, 202, lo=(-0.05, -0.05, -0.05), hi=(1.05, 1.05, 1.05)))
_SMALL = lambda: (datagen.uniform_cube(20_000, 5), datagen.uniform_cube(5_000, 6))

# name: (clouds () -> (target, queries), search, radius, k).  tools/make_flann_golden.py runs the reference on these.
CASES = {
    "uniform_200k_r0.02": (_UNIFORM, "radius", 0.02, 1),
    "uniform_200k_r0.3": (_UNIFORM, "radius", 0.3, 1),
    # the first search of config 2 (misaligned surface), 1 M -> 1 M
    "config2_first_search_1M": (_config2, "radius", 0.02, 1),
    # lattice + duplicates, queries at cell centres / on lattice points: every query has several equidistant points
    "ties_lattice": (_lattice, "radius", 0.5, 1),
    "radius_k4_r0.05": (_SMALL, "radius", 0.05, 4),
    "radius_k15_r0.08": (_SMALL, "radius", 0.08, 15),
    "radius_k30_r0.1": (_SMALL, "radius", 0.1, 30),
    "knn30": (lambda: (datagen.uniform_cube(50_000, 7), datagen.uniform_cube(5_000, 8)), "knn", None, 30),
}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def set_crcs(idx):
    """CRC-32 of each row's sorted valid indices: equal CRCs <=> equal neighbour sets (up to a 2^-32 collision)"""
    return np.array([zlib.crc32(np.sort(r[r >= 0]).astype("<i4").tobytes()) for r in idx], np.uint32)


def sample_rows(name, n):
    return np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(n, min(SAMPLE, n), replace=False))


@pytest.fixture(scope="module")
def golden_flann():
    with np.load(GOLDEN, allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def _product(name):
    clouds, kind, r, k = CASES[name]
    tgt, qry = clouds()
    tree = cph.geometry.KDTreeFlann(cph.geometry.PointCloud(tgt))
    if kind == "knn":
        _, idx, d2 = tree.search_knn(qry, k)
    else:
        _, idx, d2 = tree.search_radius(qry, r, k)
    return tgt, qry, idx.cpu(), d2.cpu()


def _equidistant(qry, tgt, ia, ib):
    q = qry.astype(np.float64)
    da = ((q - tgt[ia].astype(np.float64)) ** 2).sum(1)
    db = ((q - tgt[ib].astype(np.float64)) ** 2).sum(1)
    return np.abs(da - db) <= 4e-7 * np.maximum(da, db) + 1e-30


def _compare_1nn(name, g):
    tgt, qry, idx, d2 = _product(name)
    idx, d2 = idx[:, 0], d2[:, 0]
    found = idx >= 0
    # membership and d2 over every query, bit for bit: d2 follows the operation order the reference's kernel has in
    # SASS (cphb_internal.cuh dist2)
    assert sha(found.astype(np.uint8)) == str(g[name + "/found_sha"]), "a query is found on one side only"
    assert sha(d2[found].astype(np.float32)) == str(g[name + "/d2_sha"]), "d2 differs from the reference binary's"
    # the product's point sits at that distance, so where its index is not FLANN's the two points tie
    d_own = ((qry[found].astype(np.float64) - tgt[idx[found]].astype(np.float64)) ** 2).sum(1)
    assert np.all(np.abs(d_own - d2[found]) <= 4e-7 * d_own + 1e-30), "returned point is not at the returned d2"
    # the sample: index and d2 of the reference
    rows = g[name + "/rows"]
    assert np.array_equal(rows, sample_rows(name, len(qry)))
    fi, fd = g[name + "/idx"], g[name + "/d2"]
    si, sd, sq = idx[rows], d2[rows], qry[rows]
    both = (si >= 0) & (fi >= 0)
    np.testing.assert_array_equal(sd[both], fd[both])
    idx_diff = both & (si != fi)
    # where the indices differ the two points must be (numerically) equidistant: a tie, not a wrong answer
    assert _equidistant(sq[idx_diff], tgt, si[idx_diff], fi[idx_diff]).all(), \
        "product and FLANN return different, non-equidistant points"
    return int(idx_diff.sum())


def test_flann_1nn_uniform(golden_flann):
    assert _compare_1nn("uniform_200k_r0.02", golden_flann) <= 5      # random floats: ties are essentially impossible
    _compare_1nn("uniform_200k_r0.3", golden_flann)


def test_flann_1nn_icp_workload(golden_flann):
    assert _compare_1nn("config2_first_search_1M", golden_flann) <= 20


def test_flann_ties(golden_flann):
    # d2 must agree bit for bit (all values are exact in float); the INDEX is the tie rule.
    tgt, qry, idx, d2 = _product("ties_lattice")
    fi, fd = golden_flann["ties_lattice/idx"], golden_flann["ties_lattice/d2"]
    np.testing.assert_array_equal(d2, fd)
    # both answers are nearest points; ours is the smallest index among them
    d_ours = ((qry - tgt[idx[:, 0]]) ** 2).sum(1)
    d_ref = ((qry - tgt[fi[:, 0]]) ** 2).sum(1)
    np.testing.assert_array_equal(d_ours, d_ref)
    assert (idx[:, 0] <= fi[:, 0]).all()


@pytest.mark.parametrize("k,r", [(4, 0.05), (15, 0.08), (30, 0.1)])
def test_flann_radius_k_not_full(golden_flann, k, r):
    # R1b: radius search with max_nn > 1 where most result lists are NOT full.  The reference heap-sorts an array it
    # only heapifies on the k-th insert (result_set.h:405-473): compare as sets
    name = "radius_k%d_r%g" % (k, r)
    _, _, idx, _ = _product(name)
    same_set = set_crcs(idx) == golden_flann[name + "/set_crc"]
    full = (idx >= 0).sum(1) == k
    # lists that are not full contain EVERY point inside the radius on both sides: the sets must be equal.  A full
    # list may differ only where the k-th and (k+1)-th neighbour tie.
    assert same_set[~full].all()
    assert same_set.mean() > 0.999


def test_flann_knn30(golden_flann):
    _, _, idx, d2 = _product("knn30")
    same_set = set_crcs(idx) == golden_flann["knn30/set_crc"]
    assert same_set.mean() > 0.999
    assert sha(np.sort(d2, 1).astype(np.float32)) == str(golden_flann["knn30/d2_sorted_sha"])
