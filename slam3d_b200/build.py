"""Builds libs3d_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.  No GPU is needed to build."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libs3d_b200.so")
SOURCES = ["voxel.cu", "grid.cu", "knn.cu", "gicp.cu", "ndt.cu", "map.cu", "ransac.cu", "api.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# -fmad=false: every float/double expression keeps its written operation order (PCL parity; see DESIGN.md)
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC,-O2"]


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "s3d_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdr_time = _deps()
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_time):
            jobs.append([NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])
    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            for r in ex.map(lambda c: subprocess.run(c, capture_output=True, text=True), jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed: " + " ".join(r.args))
    if jobs or not os.path.exists(LIB):
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs + ["-lcudart"])
    build_host(force or bool(jobs))
    return LIB


HOST_LIB = os.path.join(HERE, "libs3d_host.so")


def build_host(force=False):
    """C++ host mirror of slam3d::PointCloudSensor (slam3d_b200/host) on top of the C-ABI library."""
    hdir = os.path.join(HERE, "host")
    srcs = [os.path.join(hdir, f) for f in ("PointCloudSensor.cpp", "host_capi.cpp")]
    newest = max(os.path.getmtime(os.path.join(hdir, f)) for f in os.listdir(hdir))
    if force or not os.path.exists(HOST_LIB) or os.path.getmtime(HOST_LIB) < newest:
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", HOST_LIB] + srcs +
                              ["-L" + HERE, "-ls3d_b200", "-Wl,-rpath,$ORIGIN"])
    return HOST_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
