"""FastGlobalRegistration / BruteForceNN through the header-compatible C++ facade (include/cupoch/...): the facade
compiles against the C ABI with plain g++ (CPU check), and on the GPU box its results equal the oracle's."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import fgr_oracle as F
import test_facade_cpp as facade


def test_facade_fgr_compiles_and_links():
    exe = facade.build_facade("facade_fgr")
    out = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "libcupoch_b200.so" in out and "not found" not in out


@pytest.mark.gpu
def test_facade_fgr_matches_oracle(orc):
    exe = facade.build_facade("facade_fgr")
    rng = np.random.default_rng(90)
    src = rng.uniform(-1, 1, (1500, 3)).astype(np.float32)
    tgt = rng.uniform(-1, 1, (1300, 3)).astype(np.float32)
    fs = rng.uniform(0, 100, (1500, 33)).astype(np.float32)
    ft = rng.uniform(0, 100, (1300, 33)).astype(np.float32)
    ft[:400] = fs[:400] + np.float32(0.5)
    tgt[:400] = src[:400] + np.float32(0.2)
    with tempfile.TemporaryDirectory() as d:
        for name, a in (("src", src), ("tgt", tgt), ("fs", fs), ("ft", ft)):
            a.tofile(os.path.join(d, name + ".f32"))
        r = subprocess.run([exe, d], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        T = np.fromfile(os.path.join(d, "T.f32"), np.float32).reshape(4, 4)
        fit = np.fromfile(os.path.join(d, "fit.f32"), np.float32)
        corr = np.fromfile(os.path.join(d, "corr.i32"), np.int32).reshape(-1, 2)
        nn = np.fromfile(os.path.join(d, "nn.i32"), np.int32)
    ref = F.fast_global_registration(orc, src, tgt, fs, ft, F.option(maximum_correspondence_distance=0.05,
                                                                     iteration_number=32))
    assert np.array_equal(T, ref["transformation"])
    assert fit[0] == np.float32(ref["fitness"]) and fit[1] == np.float32(ref["inlier_rmse"])
    assert np.array_equal(corr, ref["correspondence_set"])
    assert np.array_equal(nn, F.feature_nn(fs, ft)[0])
