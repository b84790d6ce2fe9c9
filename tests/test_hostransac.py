"""slam3d_b200/csrc/ransac_math.h (sampler, distance, replay and ring fill of the GPU path) compiled for the host and run in the GPU
path's block order (tests/hostransac.cpp), checked bit for bit against the oracle's fillGroundPlane (oracle/ransac_oracle.cpp):
coefficients, iterations, inliers and fill points, for several block sizes.  The harness is built in a temporary directory."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_oracle_ransac import THRESHOLD, degenerate_clouds, ground_cloud

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


@pytest.fixture(scope="module")
def ransac_oracle():
    from oracle import ransac
    ransac.lib()
    return ransac


@pytest.fixture(scope="module")
def hr():
    tmp = tempfile.mkdtemp(prefix="s3d_hostransac_")
    try:
        out = os.path.join(tmp, "hostransac.so")
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                               "-shared", "-I" + CUDA_INC, "-o", out, os.path.join(ROOT, "tests", "hostransac.cpp")])
        lib = C.CDLL(out)  # stays mapped after the directory is removed
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return lib


def xyzw(cloud):
    a = np.ones((len(cloud), 4), np.float32)
    a[:, :3] = cloud
    return a


def host_fit(hr, cloud, threshold, max_it, B, probability=0.99):
    a = xyzw(cloud)
    coeff = np.zeros(4, np.float32)
    it, m, blocks = C.c_int32(0), C.c_uint64(0), C.c_int32(0)
    inl = np.empty(max(len(a), 1), np.uint32)
    st = hr.hr_fit(a.ctypes.data_as(C.c_void_p), C.c_uint32(len(a)), C.c_double(threshold), max_it, C.c_double(probability), B,
                   coeff.ctypes.data_as(C.c_void_p), C.byref(it), C.byref(m), inl.ctypes.data_as(C.c_void_p), C.byref(blocks))
    return st == 0, coeff, it.value, inl[: m.value].copy(), blocks.value


CLOUDS = {
    "ground": (ground_cloud(11, 5000), 10000),
    "ground_nan": (ground_cloud(12, 3000, nan_frac=0.03), 10000),
    "sparse_ground": (ground_cloud(13, 2000, ground=0.08), 10000),
    "max_it_1": (ground_cloud(14, 1000), 1),
    **{k: (v, 10000) for k, v in degenerate_clouds().items()},
}


@pytest.mark.parametrize("B", [1, 7, 256])
@pytest.mark.parametrize("name", sorted(CLOUDS))
def test_host_fit_reproduces_oracle(hr, ransac_oracle, name, B):
    cloud, max_it = CLOUDS[name]
    ok, coeff, it, inl = ransac_oracle.fit_plane_ransac(cloud, THRESHOLD, max_it)
    ok2, coeff2, it2, inl2, blocks = host_fit(hr, cloud, THRESHOLD, max_it, B)
    assert ok == ok2 and it == it2
    if ok:
        assert np.array_equal(coeff.view(np.uint32), coeff2.view(np.uint32))
        assert np.array_equal(inl, inl2)
    assert blocks >= 1


def test_threshold_promotion(hr, ransac_oracle):
    """Thresholds that are not floats: the float comparison of the GPU path is the double comparison of PCL."""
    cloud = ground_cloud(15, 2000)
    for thr in (0.01, 0.0123456789, 0.02, 1.0 / 3.0):
        ok, coeff, it, inl = ransac_oracle.fit_plane_ransac(cloud, thr)
        ok2, coeff2, it2, inl2, _ = host_fit(hr, cloud, thr, 10000, 64)
        assert ok and ok2 and it == it2 and np.array_equal(coeff, coeff2) and np.array_equal(inl, inl2)


def test_mt_matches_oracle(hr, ransac_oracle):
    for seed in (5489, 12345):
        mt, _ = ransac_oracle.rng_stream(seed, 3000)
        out = np.empty(3000, np.uint32)
        hr.hr_mt(C.c_uint32(seed), 3000, out.ctypes.data_as(C.c_void_p))
        assert np.array_equal(out, mt)


@pytest.mark.parametrize("res,radius", [(0.1, 2.0), (0.1, 7.5), (0.25, 3.0), (0.05, 1.0)])
@pytest.mark.parametrize("name", ["ground", "identical"])
def test_host_fill_reproduces_oracle(hr, ransac_oracle, name, res, radius):
    cloud = CLOUDS[name][0]
    want, coeff = ransac_oracle.fill_ground_plane(cloud, radius, res)
    n = C.c_uint64(0)
    out = np.empty((max(len(want), 1), 4), np.float32)
    assert hr.hr_fill(coeff.ctypes.data_as(C.c_void_p), C.c_double(res), C.c_double(radius), out.ctypes.data_as(C.c_void_p), C.byref(n)) == 0
    assert n.value == len(want)
    assert np.array_equal(out[: n.value].view(np.uint32), want.view(np.uint32))
