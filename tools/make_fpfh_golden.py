"""Write tests/golden/fpfh_ref.json: the reference's known-answer test of ComputeFPFHFeature
(src/tests/registration/feature.cpp:30-155) as data -- 20 points, their normals, KDTreeSearchParamRadius(0.05 * 3, 5)
and the expected 33 x 20 feature matrix, stored as 20 rows of 33 (one row per point).

    python tools/make_fpfh_golden.py [path/to/reference/checkout]

Eigen's `mat << ...` fills a matrix row by row, so the k-th listed value is feature k // 20 of point k % 20."""
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main(ref_root):
    with open(os.path.join(ref_root, "src", "tests", "registration", "feature.cpp")) as f:
        src = f.read()
    body = src[src.index("TEST(Feature, ComputeFPFHFeature)"):]
    num = r"[-+]?[0-9]*\.?[0-9]+(?:[eE][-+]?[0-9]+)?"
    vec = re.compile(r"Vector3f\(\s*(%s),\s*(%s),\s*(%s)\)" % (num, num, num))
    pts_part = body[:body.index("thrust::host_vector<Vector3f> normals")]
    nrm_part = body[body.index("thrust::host_vector<Vector3f> normals"):body.index("geometry::PointCloud pc")]
    points = [[float(v) for v in m] for m in vec.findall(pts_part)]
    normals = [[float(v) for v in m] for m in vec.findall(nrm_part)]
    mat = body[body.index("mat_features <<") + len("mat_features <<"):]
    mat = mat[:mat.index(";")]
    vals = [float(v) for v in re.findall(num, mat)]
    assert len(points) == 20 and len(normals) == 20 and len(vals) == 33 * 20, (len(points), len(normals), len(vals))
    m = re.search(r"KDTreeSearchParamRadius\(\s*(%s)\s*\*\s*(%s),\s*(\d+)\)" % (num, num), body)
    radius, max_nn = float(m.group(1)) * float(m.group(2)), int(m.group(3))
    expected = [[vals[k * 20 + i] for k in range(33)] for i in range(20)]
    out = {"source": "src/tests/registration/feature.cpp:30-155 (TEST Feature.ComputeFPFHFeature)", "tolerance": 1e-4,
           "radius": radius, "max_nn": max_nn, "points": points, "normals": normals, "expected": expected}
    path = os.path.join(ROOT, "tests", "golden", "fpfh_ref.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "/root/reference")
