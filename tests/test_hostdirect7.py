"""The DIRECT7 path of slam3d_b200/csrc/ndt_math.h (what ndt_eval_kernel<true> runs for NDT_OMP with S3D_NDT_OMP_DIRECT7)
compiled for the host (tests/hostdirect7.cpp) and held bit for bit to the oracle's DIRECT7 restatement
(oracle/ndt_omp_oracle.cpp): neighbour keys, then whole registrations (outer and line-search iterations, pair counts, float
pose).  The harness is built in a temporary directory."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from slam3d_b200 import _abi, synth
from slam3d_b200._abi import RegistrationParameters
from test_oracle_ndt_omp import query_points, with_degenerate_voxels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hd():
    tmp = tempfile.mkdtemp(prefix="s3d_hostdirect7_")
    try:
        out = os.path.join(tmp, "hostdirect7.so")
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                               "-shared", "-o", out, os.path.join(ROOT, "tests", "hostdirect7.cpp")])
        lib = C.CDLL(out)  # stays mapped after the directory is removed
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return lib


@pytest.fixture
def direct7(oracle_mod):
    from oracle import ndt_omp
    old = ndt_omp.set_ndt_omp_search("direct7")
    yield ndt_omp
    ndt_omp.set_ndt_omp_search(old)


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("res", [0.3, 0.7, 1.0])
def test_host_direct7_keys_equal_oracle(hd, oracle_mod, direct7, res):
    src, _, _ = synth.scan_pair(seed=11)
    target, centres = with_degenerate_voxels(oracle_mod.voxel_downsample(src, 0.1)[0], res)
    t = oracle_mod.as_xyzw(target)
    q = oracle_mod.as_xyzw(np.concatenate([query_points(target, res, np.random.default_rng(3)), centres]))
    keys = np.empty((len(q), 7), np.uint32); counts = np.empty(len(q), np.int32)
    assert hd.hd_direct7_keys(ptr(t), len(t), C.c_float(res), ptr(q), len(q), ptr(keys), ptr(counts)) > 0
    want_keys, want_counts, _ = direct7.ndt_direct7_keys(target, res, q)
    assert np.array_equal(counts, want_counts) and np.array_equal(keys, want_keys)


def ndt_omp(**kw):
    kw.setdefault("point_cloud_density", 0.2)
    return RegistrationParameters.defaults(registration_algorithm=_abi.ALG_NDT_OMP, **kw)


def run_host(hd, oracle_mod, src, tgt, guess, p):
    """The GPU's DIRECT7 NDT on the host, on the oracle's voxel-filtered clouds (PCL source = slam3d target)."""
    d = p.point_cloud_density
    fs = oracle_mod.voxel_downsample(src, d)[0] if d > 0 else oracle_mod.as_xyzw(src)
    ft = oracle_mod.voxel_downsample(tgt, d)[0] if d > 0 else oracle_mod.as_xyzw(tgt)
    g = np.eye(4) if guess is None else np.asarray(guess, np.float64)
    gf = np.ascontiguousarray(g.T.astype(np.float32))
    T = np.zeros(16, np.float32); info = np.zeros(6, np.int32)
    hd.hd_ndt_register(ptr(ft), ft.shape[0], ptr(fs), fs.shape[0], ptr(gf), C.c_float(p.resolution), C.c_double(p.step_size),
                       C.c_double(p.outlier_ratio), C.c_double(p.transformation_epsilon), p.maximum_iterations, ptr(T), ptr(info))
    return T.reshape(4, 4).T.astype(np.float64), info


CASES = [
    dict(seed=11, loop=False, guess=None, kw=dict(point_cloud_density=0.2)),
    dict(seed=11, loop=False, guess="noisy", kw=dict(point_cloud_density=0.2, resolution=0.7)),
    dict(seed=3, loop=False, guess=None, kw=dict(point_cloud_density=0.3, resolution=2.0, step_size=0.1)),
    dict(seed=5, loop=True, guess=None, kw=dict(point_cloud_density=0.5, resolution=2.0, step_size=0.2, max_translation=5.0)),
    dict(seed=5, loop=True, guess="truth", kw=dict(point_cloud_density=0.2, resolution=0.5, outlier_ratio=0.55)),
    dict(seed=7, loop=False, guess=None, kw=dict(point_cloud_density=0.2, resolution=0.3, transformation_epsilon=1e-9, maximum_iterations=12)),
]


def check(hd, oracle_mod, omp_oracle, src, tgt, guess, p):
    want = omp_oracle.gicp_align(src, tgt, guess, p)
    T, info = run_host(hd, oracle_mod, src, tgt, guess, p)
    assert want.status != _abi.S3D_UNKNOWN_ALGORITHM
    assert (info[0], info[1], info[2], info[3]) == (want.converged, want.outer_iterations, want.inner_iterations, want.n_correspondences)
    assert np.abs(T - want.pose()).max() == 0.0
    assert info[4] >= info[1] + 1


@pytest.mark.parametrize("case", CASES)
def test_host_direct7_reproduces_oracle(hd, oracle_mod, direct7, case):
    src, tgt, truth = synth.scan_pair(seed=case["seed"], loop=case["loop"])
    guess = None
    if case["guess"] == "truth":
        guess = truth
    elif case["guess"] == "noisy":
        guess = synth.make_pose([0.05, -0.03, 0.01], [0.002, -0.003, 0.004]) @ truth
    check(hd, oracle_mod, direct7, src, tgt, guess, ndt_omp(**case["kw"]))


@pytest.mark.parametrize("density", [0.1, 0.2])
def test_host_direct7_on_kitti(hd, oracle_mod, direct7, kitti, density):
    check(hd, oracle_mod, direct7, kitti[0], kitti[1], None, ndt_omp(point_cloud_density=density))
