"""Python loader of the CPU oracle of NDT_OMP with pclomp's DIRECT7 neighbour search (oracle/ndt_omp_oracle.cpp).

TEST INFRASTRUCTURE: may be imported by tests/ and scripts/ only; the product package slam3d_b200 never imports it.
PARITY UNPINNED: see the header of ndt_omp_oracle.cpp.  The library is compiled with the oracle's flags on first use into a
private temporary directory (mode 0700, unpredictable name) that is removed once it is loaded, so nothing is written to the
source tree, which may be read-only.

gicp_align() stands for align() of a slam3d build with pclomp: NDT_OMP runs the neighbour search set_ndt_omp_search() names
("kdtree": pclomp's KDTREE mode, i.e. PCL's NDT — the main oracle's NDT branch; "direct7": pclomp's default).  Every other
algorithm goes to the main oracle (oracle/__init__.py) unchanged.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle
from slam3d_b200 import _abi
from slam3d_b200._abi import RegistrationParameters, Result

_HERE = os.path.dirname(os.path.abspath(__file__))
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared"]
_lib = None
_search = "kdtree"


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="s3d_ndt_omp_oracle_")
        try:
            out = os.path.join(tmp, "libs3d_ndt_omp_oracle.so")
            subprocess.check_call([os.environ.get("CXX", "g++")] + _FLAGS + ["-o", out, os.path.join(_HERE, "ndt_omp_oracle.cpp")])
            L = C.CDLL(out)  # stays mapped after the file is removed
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        L.s3d_oracle_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def set_ndt_omp_search(which):
    """Neighbour search of NDT_OMP in gicp_align: "kdtree" (default) or "direct7".  Process-wide; returns the previous setting."""
    global _search
    if which not in ("kdtree", "direct7"):
        raise ValueError(f"unknown NDT_OMP search {which!r}")
    old, _search = _search, which
    return old


def gicp_align(source, target, guess=None, params=None):
    """align(source, target, guess, config) of a slam3d build with pclomp.  Returns slam3d_b200._abi.Result."""
    p = params if params is not None else RegistrationParameters.defaults()
    if p.registration_algorithm != _abi.ALG_NDT_OMP:
        return oracle.gicp_align(source, target, guess, p)
    if _search == "kdtree":
        q = RegistrationParameters.from_buffer_copy(p)
        q.registration_algorithm = _abi.ALG_NDT
        return oracle.gicp_align(source, target, guess, q)
    s, sc = oracle._cloud(source)
    t, tc = oracle._cloud(target)
    g = oracle._guess_ptr(guess)
    res = Result()
    lib().s3d_oracle_ndt_omp_align(sc, tc, g.ctypes.data_as(C.c_void_p), C.byref(p), C.byref(res))
    return res


def last_error():
    """Message of the last gicp_align that ran NDT_OMP with DIRECT7 (other calls: oracle.last_error())."""
    return lib().s3d_oracle_last_error().decode()


def ndt_direct7_keys(target, resolution, queries):
    """DIRECT7 neighbourhoods (test hook): for each query, PCL's linear voxel indices of the kept leaves of the VoxelGridCovariance of
    `target` at `resolution`, in pclomp's offset order.  Returns (keys (n, 7) uint32 padded with 0xFFFFFFFF, counts (n,), centroids)."""
    t, tc = oracle._cloud(target)
    q, qc = oracle._cloud(queries)
    keys = np.empty((max(q.shape[0], 1), 7), np.uint32)
    counts = np.empty(max(q.shape[0], 1), np.int32)
    n_c = lib().s3d_oracle_ndt_direct7_keys(tc, C.c_float(resolution), qc, keys.ctypes.data_as(C.c_void_p), counts.ctypes.data_as(C.c_void_p))
    return keys[: q.shape[0]].copy(), counts[: q.shape[0]].copy(), n_c
