"""Build libcupoch_b200.so (sm_100a only) in-tree with nvcc.

    python -m cupoch_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
-fmad=false: the arithmetic contract (DESIGN.md) spells out every fused
multiply-add with an explicit intrinsic, so results do not depend on the
compiler's contraction choices.
"""
import hashlib
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(SRC, "_build")
LIB = os.path.join(HERE, "lib", "libcupoch_b200.so")
SOURCES = ["index.cu", "sort.cu", "search.cu", "icp.cu", "voxel.cu", "features.cu", "filters.cu", "voxelgrid.cu", "comm.cu",
           "reduce.cu", "fpfh.cu", "cluster.cu", "occgrid.cu", "fgr.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + SRC]


HEADERS = ["cphb_internal.cuh", "cphb_searchk.cuh", "cphb_eigen3.cuh", "icp_types.cuh", "icp_solve.cuh", "icp_rows.cuh", "icp_kernels.cuh",
           "icp_estimate.cuh", "icp_aux.cuh"]
MANIFEST = os.path.join(OBJ, "manifest.json")


def _sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def _signature(src):
    """content hash of a source + the headers it can include + the flags: staleness must not depend on file
    mtimes (the snapshot on the GPU box does not preserve them)"""
    parts = [_sha(os.path.join(SRC, src))] + [_sha(os.path.join(SRC, h)) for h in HEADERS]
    parts.append(_sha(os.path.join(ROOT, "include", "cupoch_b200.h")))
    parts.append(" ".join(FLAGS))
    return hashlib.sha256("|".join(parts).encode()).hexdigest()


def _load_manifest():
    try:
        with open(MANIFEST) as f:
            return json.load(f)
    except Exception:
        return {}


def _compile(src, manifest):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    sig = _signature(src)
    if manifest.get(src) != sig or not os.path.exists(obj):
        cmd = [NVCC] + FLAGS + ["-c", os.path.join(SRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj, sig, True
    return obj, sig, False


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(SRC, s))]
    if force:
        for s in srcs:
            o = os.path.join(OBJ, s.replace(".cu", ".o"))
            if os.path.exists(o):
                os.remove(o)
    manifest = {} if force else _load_manifest()
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        res = list(ex.map(lambda x: _compile(x, manifest), srcs))
    objs = [o for o, _, _ in res]
    if any(ch for _, _, ch in res) or not os.path.exists(LIB):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-cudart", "static", "-ldl", "-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
        if verbose:
            print("linked", LIB)
    with open(MANIFEST, "w") as f:
        json.dump({s_: sig for s_, (_, sig, _) in zip(srcs, res)}, f, indent=0)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
