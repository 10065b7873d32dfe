"""bench.py's reference arm on CPU (no GPU involved): the contract of the JSON line, and that under torchrun only rank 0
works and prints (the driver launches `--impl reference` the same way as the native arm, N > 1 included)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check_line(out):
    lines = [l for l in out.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "icp_iterations_per_sec" and d["unit"] == "iter/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["dtype"] == "f32" and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["points"] == 20000 and "workload" in d["config"]
    return d


def test_reference_arm_single_process():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--points", "20000", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    d = _check_line(r.stdout)
    assert d["n_gpus"] == 1


def test_reference_arm_under_torchrun_world_2():
    env = dict(os.environ, OMP_NUM_THREADS="1")   # what torchrun exports: the arm must ignore it and use every core it may
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29631", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--points", "20000",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = _check_line(r.stdout)
    assert d["n_gpus"] == 2
    import bench
    assert d["cpu_baseline"]["cores"] == bench.cpu_threads()   # not the single thread OMP_NUM_THREADS=1 would give


def test_reference_arm_steps_and_dump_outputs(tmp_path):
    """--steps sets the number of timed registrations; --dump-outputs writes the last one's RegistrationResult as float64
    arrays, the same on every run and equal to what the oracle returns for the same seeded workload"""
    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--points", "20000", "--steps", "2",
                            "--warmup", "0", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 0, r.stderr
        assert _check_line(r.stdout)["steps"] == 2
        dumps.append({f.name[:-4]: np.load(f) for f in (tmp_path / run).iterdir()})
    a, b = dumps
    assert sorted(a) == ["correspondence_set", "fitness", "inlier_rmse", "transformation"]
    for k in a:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k]), k
    import bench
    from oracle import oracle_py as orc
    src, tgt, tn = bench.make_workload(20000)
    ref = orc.registration_icp(orc.P2PLANE, src, tgt, bench.MAX_DIST, tgt_nrm=tn, relative_fitness=0, relative_rmse=0,
                               max_iteration=bench.ITERS)
    np.testing.assert_array_equal(a["transformation"], ref["transformation"])
    np.testing.assert_array_equal(a["correspondence_set"], ref["correspondence_set"])
    assert a["fitness"] == np.float32(ref["fitness"]) and a["inlier_rmse"] == np.float32(ref["inlier_rmse"])
