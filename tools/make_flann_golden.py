#!/usr/bin/env python3
"""Write tests/golden/flann_ref.npz: the reference's FLANN CUDA kd-tree answers for the comparisons of
tests/test_gpu_flann_ref.py (its CASES, same seeded inputs).

Needs a GPU and oracle/_ref/libflann_ref.so, which `__graft_entry__.build()` compiles (oracle/ref_flann/Makefile)
where the reference's sources are available.

    python tools/make_flann_golden.py [OUT.npz]
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_gpu_flann_ref as T  # noqa: E402

SO = os.path.join(ROOT, "oracle", "_ref", "libflann_ref.so")


def load():
    L = C.CDLL(SO)
    L.fref_build.restype = C.c_void_p
    L.fref_build.argtypes = [C.c_void_p, C.c_int]
    L.fref_free.argtypes = [C.c_void_p]
    L.fref_knn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.fref_radius.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p]
    return L


def flann(L, tgt, qry, kind, r, k):
    tgt = np.ascontiguousarray(tgt, np.float32)
    qry = np.ascontiguousarray(qry, np.float32)
    h = L.fref_build(tgt.ctypes.data, len(tgt))
    assert h, "the reference's FLANN index failed to build"
    idx = np.empty((len(qry), k), np.int32)
    d2 = np.empty((len(qry), k), np.float32)
    if kind == "knn":
        rc = L.fref_knn(h, qry.ctypes.data, len(qry), k, idx.ctypes.data, d2.ctypes.data)
    else:
        rc = L.fref_radius(h, qry.ctypes.data, len(qry), C.c_float(r), k, idx.ctypes.data, d2.ctypes.data)
    L.fref_free(h)
    assert rc == 0
    return idx, d2


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else T.GOLDEN
    L = load()
    out = {}
    for name, (clouds, kind, r, k) in T.CASES.items():
        tgt, qry = clouds()
        idx, d2 = flann(L, tgt, qry, kind, r, k)
        if name == "ties_lattice":
            out[name + "/idx"], out[name + "/d2"] = idx, d2
        elif k == 1:
            idx, d2 = idx[:, 0], d2[:, 0]
            found = idx >= 0
            rows = T.sample_rows(name, len(qry))
            out[name + "/found_sha"] = np.array(T.sha(found.astype(np.uint8)))
            out[name + "/d2_sha"] = np.array(T.sha(d2[found]))
            out[name + "/rows"], out[name + "/idx"], out[name + "/d2"] = rows.astype(np.int32), idx[rows], d2[rows]
        else:
            out[name + "/set_crc"] = T.set_crcs(idx)
            if kind == "knn":
                out[name + "/d2_sorted_sha"] = np.array(T.sha(np.sort(d2, 1)))
        print(name, "queries", len(qry), "found", int((idx >= 0).any(axis=-1).sum()) if idx.ndim > 1 else int((idx >= 0).sum()))
    np.savez_compressed(out_path, **out)
    print("wrote", out_path, os.path.getsize(out_path), "bytes")


if __name__ == "__main__":
    main()
