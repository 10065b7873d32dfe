"""ctypes loader for tests/fgr_oracle.c, the CPU restatement of FastGlobalRegistration and knn::BruteForceNN.

Test infrastructure only.  The library is compiled on first use into a temporary directory (the tree is never
written), together with oracle/oracle.c, whose LDLT / se(3) / composition routines it reuses."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
CFLAGS = ["-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-w"]
_lib = None
_tmp = None


class Option(C.Structure):  # cphb_fgr_option
    _fields_ = [("division_factor", C.c_float), ("use_absolute_scale", C.c_int), ("decrease_mu", C.c_int),
                ("maximum_correspondence_distance", C.c_float), ("iteration_number", C.c_int),
                ("tuple_scale", C.c_float), ("maximum_tuple_count", C.c_int)]


def option(division_factor=1.4, use_absolute_scale=False, decrease_mu=True, maximum_correspondence_distance=0.025,
           iteration_number=64, tuple_scale=0.95, maximum_tuple_count=1000):
    return Option(division_factor, int(use_absolute_scale), int(decrease_mu), maximum_correspondence_distance,
                  iteration_number, tuple_scale, maximum_tuple_count)


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="fgr_oracle_")
        so = os.path.join(_tmp.name, "libfgr_oracle.so")
        subprocess.check_call(["gcc"] + CFLAGS + ["-I", _ORACLE, "-shared", "-o", so, os.path.join(_HERE, "fgr_oracle.c"), "-lm"])
        _lib = C.CDLL(so)
        _lib.orc_fgr_advanced_matching.restype = C.c_int
    return _lib


def _f(a, cols=None):
    a = np.ascontiguousarray(a, np.float32)
    return a if cols is None else a.reshape(-1, cols)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def feature_nn(ref, query):
    """knn::BruteForceNN -> (idx int32 [m], d2 float32 [m])"""
    ref, query = _f(ref), _f(query)
    dim = ref.shape[1]
    idx, d2 = np.empty(len(query), np.int32), np.empty(len(query), np.float32)
    lib().orc_feature_nn(_p(ref), C.c_int(len(ref)), _p(query), C.c_int(len(query)), C.c_int(dim), _p(idx), _p(d2))
    return idx, d2


def minstd_draws(idx, ncorr):
    out = (C.c_int * 3)()
    lib().orc_minstd_draws(C.c_ulonglong(idx), C.c_longlong(ncorr), out)
    return tuple(out)


def normalize(src, tgt, use_absolute_scale=False):
    src, tgt = _f(src, 3), _f(tgt, 3)
    out = np.zeros(8, np.float32)
    lib().orc_fgr_normalize(_p(src), C.c_int(len(src)), _p(tgt), C.c_int(len(tgt)), C.c_int(int(use_absolute_scale)), _p(out))
    return {"mean_source": out[:3], "mean_target": out[3:6], "scale": out[6], "scale_global": out[7]}


def advanced_matching(src, tgt, fs, ft, opt=None):
    """-> (pairs [m,2] (source, target), counts dict, mutual [k,2] (fi, fj) in fi order, swapped)"""
    opt = opt or option()
    src, tgt, fs, ft = _f(src, 3), _f(tgt, 3), _f(fs), _f(ft)
    pairs = np.empty((max(opt.maximum_tuple_count, 1), 2), np.int32)
    mutual = np.empty((max(len(src), len(tgt), 1), 2), np.int32)
    counts = (C.c_longlong * 4)()
    sw = lib().orc_fgr_advanced_matching(_p(src), C.c_int(len(src)), _p(tgt), C.c_int(len(tgt)), _p(fs), _p(ft),
                                         C.c_int(fs.shape[1]), C.byref(opt), _p(pairs), counts, _p(mutual))
    c = {"pairs": counts[0], "mutual": counts[1], "trials": counts[2], "passing_pairs": counts[3]}
    return pairs[:counts[0]].copy(), c, mutual[:counts[1]].copy(), bool(sw)


def optimize(src, tgt, pairs, opt=None):
    """-> (T [4,4] source -> target in original units, trace [iteration_number, 4, 4])"""
    opt = opt or option()
    src, tgt = _f(src, 3), _f(tgt, 3)
    pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
    T = np.zeros(16, np.float32)
    tr = np.zeros((max(opt.iteration_number, 1), 16), np.float32)
    lib().orc_fgr_optimize(_p(src), C.c_int(len(src)), _p(tgt), C.c_int(len(tgt)), _p(pairs), C.c_int(len(pairs)),
                           C.byref(opt), _p(T), _p(tr))
    return T.reshape(4, 4), tr[:max(opt.iteration_number, 0)].reshape(-1, 4, 4)


def fast_global_registration(orc, src, tgt, fs, ft, opt=None):
    """FastGlobalRegistration (fast_global_registration.cu:391-431): matching, pose loop, then EvaluateRegistration
    through the ICP oracle `orc` (oracle_py) with zero iterations -> dict like oracle_py.registration_icp + trace"""
    opt = opt or option()
    pairs, counts, _, _ = advanced_matching(src, tgt, fs, ft, opt)
    T, trace = optimize(src, tgt, pairs, opt)
    out = orc.registration_icp(orc.P2P, src, tgt, opt.maximum_correspondence_distance, init=T, max_iteration=0)
    out["trace"], out["pairs"], out["counts"] = trace, pairs, counts
    return out


def permutation_T():
    """the initial misalignment of the reference's examples/python/advanced/global_registration.py"""
    return np.array([[0, 0, 1, 0], [1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 0, 1]], np.float64)


def fgr_scene(n, seed, voxel, overlap=(0.3, 0.7)):
    """two overlapping crops of datagen.bumps_scene; the source is moved by inv(T_gt), so T_gt aligns it with the
    target -> (source, target, T_gt)"""
    from cupoch_b200.testing import datagen
    pts = datagen.bumps_scene(n, seed)
    src = pts[pts[:, 0] < overlap[1]]
    tgt = pts[pts[:, 0] > overlap[0]]
    T = permutation_T()
    T[:3, 3] = (0.4, -0.2, 0.3)
    Ti = np.linalg.inv(T)
    src = (src.astype(np.float64) @ Ti[:3, :3].T + Ti[:3, 3]).astype(np.float32)
    return src, tgt, T


def pose_error(T, T_gt):
    """(rotation angle in degrees, translation error) of T against T_gt"""
    D = np.linalg.inv(T_gt) @ np.asarray(T, np.float64)
    ang = np.degrees(np.arccos(np.clip((np.trace(D[:3, :3]) - 1) / 2, -1, 1)))
    return float(ang), float(np.linalg.norm(np.asarray(T, np.float64)[:3, 3] - T_gt[:3, 3]))
