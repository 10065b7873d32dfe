"""bench.py's native arm at a small size: --steps sets the number of timed steps, and --dump-outputs writes what the
timed registration returns, bit for bit what registration_icp gives a caller for the same seeded workload."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_native_steps_and_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--points", "20000", "--steps", "2", "--warmup", "0",
                        "--no-extras", "--no-cpu", "--no-host-call", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and len(line["step_ms"]) == 2
    d = {f.name[:-4]: np.load(f) for f in tmp_path.iterdir()}
    assert sorted(d) == ["correspondence_set", "fitness", "inlier_rmse", "transformation"]
    assert all(a.dtype == np.float64 for a in d.values())

    import bench
    import cupoch_b200 as cph
    src, tgt, tn = bench.make_workload(20000)
    s, t = cph.geometry.PointCloud(src), cph.geometry.PointCloud(tgt)
    t.normals = tn
    R = cph.registration
    res = R.registration_icp(s, t, bench.MAX_DIST, np.eye(4, dtype=np.float32), R.TransformationEstimationPointToPlane(),
                             R.ICPConvergenceCriteria(0, 0, bench.ITERS))
    np.testing.assert_array_equal(d["transformation"], res.transformation)
    np.testing.assert_array_equal(d["correspondence_set"], res.correspondence_set)
    assert d["fitness"] == np.float64(res.fitness) and d["inlier_rmse"] == np.float64(res.inlier_rmse)
