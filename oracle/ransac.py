"""Python loader of the CPU oracle of fillGroundPlane (oracle/ransac_oracle.cpp): PCL's RANSAC plane fit and the ring fill.

TEST INFRASTRUCTURE: may be imported by tests/ and scripts/ only; the product package slam3d_b200 never imports it.
PARITY UNPINNED: see the header of ransac_oracle.cpp.  The library is compiled with the oracle's flags on first use into a
private temporary directory (mode 0700, unpredictable name) that is removed once it is loaded, so nothing is written to the
source tree, which may be read-only.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from slam3d_b200._abi import Cloud

_HERE = os.path.dirname(os.path.abspath(__file__))
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="s3d_ransac_oracle_")
        try:
            out = os.path.join(tmp, "libs3d_ransac_oracle.so")
            subprocess.check_call([os.environ.get("CXX", "g++")] + _FLAGS + ["-o", out, os.path.join(_HERE, "ransac_oracle.cpp")])
            L = C.CDLL(out)  # stays mapped after the file is removed
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        L.s3d_oracle_ground_fill_size.restype = C.c_uint64
        L.s3d_oracle_ground_fill_size.argtypes = [C.c_double, C.c_double]
        _lib = L
    return _lib


def as_xyzw(a):
    """(n,3) or (n,4) array -> C-contiguous float32 (n,4) with w = 1 (pcl::PointXYZ memory)."""
    a = np.asarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("cloud must be (n,3) or (n,4)")
    if a.shape[1] == 3:
        out = np.ones((a.shape[0], 4), np.float32)
        out[:, :3] = a
        return out
    return np.ascontiguousarray(a)


def _cloud(a):
    a = as_xyzw(a)
    return a, Cloud(a.ctypes.data, a.shape[0])


def fit_plane_ransac(cloud, threshold, max_iterations=10000, probability=0.99):
    """RANSAC plane fit of fillGroundPlane.  Returns (ok, coefficients float32[4], iterations, inliers uint32)."""
    a, c = _cloud(cloud)
    coeff = np.zeros(4, np.float32)
    it = C.c_int32(0)
    m = C.c_uint64(0)
    inl = np.empty(max(a.shape[0], 1), np.uint32)
    st = lib().s3d_oracle_fit_plane_ransac(c, C.c_double(threshold), int(max_iterations), C.c_double(probability),
                                           coeff.ctypes.data_as(C.c_void_p), C.byref(it), C.byref(m), inl.ctypes.data_as(C.c_void_p))
    return st == 0, coeff, it.value, inl[: m.value].copy()


def ground_fill_size(map_resolution, radius):
    return lib().s3d_oracle_ground_fill_size(map_resolution, radius)


def fill_ground_plane(cloud, radius, map_resolution=0.1):
    """PointCloudSensor::fillGroundPlane: the points it appends (n,4) float32 and the plane, or (None, None) when RANSAC fails."""
    a, c = _cloud(cloud)
    out = np.empty((max(ground_fill_size(map_resolution, radius), 1), 4), np.float32)
    coeff = np.zeros(4, np.float32)
    m = C.c_uint64(0)
    st = lib().s3d_oracle_fill_ground_plane(c, C.c_double(map_resolution), C.c_double(radius), out.ctypes.data_as(C.c_void_p), C.byref(m),
                                            coeff.ctypes.data_as(C.c_void_p))
    if st != 0:
        return None, None
    return out[: m.value].copy(), coeff


def rng_stream(seed, n):
    """First n outputs of the oracle's mt19937(seed) and of its rnd() on a fresh engine with the same seed."""
    mt = np.empty(n, np.uint32)
    rnd = np.empty(n, np.int32)
    lib().s3d_oracle_test_rng(C.c_uint32(seed), int(n), mt.ctypes.data_as(C.c_void_p), rnd.ctypes.data_as(C.c_void_p))
    return mt, rnd
