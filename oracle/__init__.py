"""Python loader of the CPU oracle (oracle/s3d_oracle.cpp).

TEST INFRASTRUCTURE: may be imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs only.  The product package slam3d_b200 never imports this module.
PARITY UNPINNED: see the header of s3d_oracle.cpp.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from slam3d_b200._abi import Cloud, RegistrationParameters, Result

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libs3d_oracle.so")
_lib = None


def build(force=False):
    newest = max(os.path.getmtime(os.path.join(_HERE, f)) for f in ("s3d_oracle.cpp", "ndt_oracle.inc", "bfgs_oracle.inc"))
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < newest:
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.s3d_oracle_last_error.restype = C.c_char_p
    return _lib


_NATIVE_FLAGS = ["-O3", "-march=native", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared"]
_native = None


def use_native():
    """bench.py legs only (cpu_baseline, --impl reference): switch to a build made ON THIS MACHINE with g++ -O3 -march=native
    (BASELINE.md 3).  The portable -O2 library is built in the tree by build(); a -march=native one is specific to the host, so
    each process compiles its own into a private directory (tempfile.mkdtemp: mode 0700, unpredictable name) and deletes the
    directory once the library is loaded.  Nothing is written to the source tree, which may be read-only, and nothing is loaded
    that another user could have placed.  Returns a one-line description of what is loaded."""
    global _lib, _native
    if _native is None:
        src = os.path.join(_HERE, "s3d_oracle.cpp")
        tmp = tempfile.mkdtemp(prefix="s3d_oracle_native_")
        try:
            out = os.path.join(tmp, "libs3d_oracle_native.so")
            subprocess.check_call([os.environ.get("CXX", "g++")] + _NATIVE_FLAGS + ["-o", out, src],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            _native = C.CDLL(out)  # stays mapped after the file is removed
            _native.s3d_oracle_last_error.restype = C.c_char_p
        except Exception:
            lib()
            return "portable g++ -O2 build (the -march=native build failed on this host)"
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    _lib = _native
    return "g++ -O3 -march=native -ffp-contract=off, built on this host"


def _cloud(a):
    a = as_xyzw(a)
    return a, Cloud(a.ctypes.data, a.shape[0])


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


def voxel_downsample(cloud, leaf):
    a, c = _cloud(cloud)
    out = np.empty((max(a.shape[0], 1), 4), np.float32)
    leaf_index = np.empty(max(a.shape[0], 1), np.uint32)
    n_out = C.c_uint64(0)
    overflow = C.c_int32(0)
    lib().s3d_oracle_voxel_downsample(c, C.c_float(leaf), out.ctypes.data_as(C.c_void_p), C.byref(n_out),
                                      leaf_index.ctypes.data_as(C.c_void_p), C.byref(overflow))
    return out[: n_out.value].copy(), leaf_index[: a.shape[0]].copy(), bool(overflow.value)


def knn_covariances(cloud, k):
    a, c = _cloud(cloud)
    n = a.shape[0]
    idx = np.empty((n, k), np.uint32)
    d2 = np.empty((n, k), np.float32)
    cov = np.empty((n, 9), np.float64)
    st = lib().s3d_oracle_knn_covariances(c, k, idx.ctypes.data_as(C.c_void_p), d2.ctypes.data_as(C.c_void_p),
                                          cov.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError(lib().s3d_oracle_last_error().decode())
    return idx, d2, cov.reshape(n, 3, 3).transpose(0, 2, 1).copy()  # column-major -> [row, col]


def knn_bruteforce(reference, queries, k):
    r, rc = _cloud(reference)
    q, qc = _cloud(queries)
    idx = np.empty((q.shape[0], k), np.uint32)
    d2 = np.empty((q.shape[0], k), np.float32)
    st = lib().s3d_oracle_knn_bruteforce(rc, qc, k, idx.ctypes.data_as(C.c_void_p), d2.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError("knn_bruteforce failed")
    return idx, d2


def nearest_neighbors(reference, queries, transform=None):
    r, rc = _cloud(reference)
    q, qc = _cloud(queries)
    idx = np.empty(q.shape[0], np.uint32)
    d2 = np.empty(q.shape[0], np.float32)
    tp = None
    if transform is not None:
        t = np.ascontiguousarray(np.asarray(transform, np.float64).T)  # -> column-major
        tp = t.ctypes.data_as(C.c_void_p)
    st = lib().s3d_oracle_nearest_neighbors(rc, qc, tp, idx.ctypes.data_as(C.c_void_p), d2.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError("nearest_neighbors failed")
    return idx, d2


def set_gicp_optimizer(which):
    """Inner optimiser of gicp_align: "newton" (PCL >= 1.14 default, what the CUDA path mirrors; default) or "bfgs" (PCL <= 1.13 and
    `useBFGS()`: pcl/registration/bfgs.h, bfgs_oracle.inc).  Process-wide; returns the previous setting."""
    names = {"newton": 0, "bfgs": 1}
    old = lib().s3d_oracle_set_gicp_optimizer(names[which])
    return "bfgs" if old == 1 else "newton"


def test_bfgs(pts_moved, pts_fixed, mahal, T, max_inner=20):
    """estimateRigidTransformationBFGS on explicit correspondences (test hook). T: 4x4 float start; returns (T_out, inner, status)."""
    a = np.ascontiguousarray(pts_moved, np.float32); b = np.ascontiguousarray(pts_fixed, np.float32)
    M = np.ascontiguousarray(mahal, np.float64)
    Tm = np.ascontiguousarray(np.asarray(T, np.float32).T)
    done = C.c_int(0)
    st = lib().s3d_oracle_test_bfgs(a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), M.ctypes.data_as(C.c_void_p), a.shape[0],
                                    Tm.ctypes.data_as(C.c_void_p), max_inner, C.byref(done))
    return Tm.T.copy(), done.value, st


def _guess_ptr(guess):
    g = np.eye(4) if guess is None else np.asarray(guess, np.float64)
    return np.ascontiguousarray(g.T)  # column-major


def gicp_align(source, target, guess=None, params=None):
    """slam3d align(source, target, guess, config) on the CPU oracle. Returns slam3d_b200._abi.Result."""
    s, sc = _cloud(source)
    t, tc = _cloud(target)
    g = _guess_ptr(guess)
    p = params if params is not None else RegistrationParameters.defaults()
    res = Result()
    lib().s3d_oracle_gicp_align(sc, tc, g.ctypes.data_as(C.c_void_p), C.byref(p), C.byref(res))
    return res


def gicp_align_batch(sources, targets, guesses=None, params=None, n_threads=0):
    n = len(sources)
    keep = []
    sc = (Cloud * n)()
    tc = (Cloud * n)()
    for i in range(n):
        a, c = _cloud(sources[i]); keep.append(a); sc[i] = c
        a, c = _cloud(targets[i]); keep.append(a); tc[i] = c
    g = np.stack([_guess_ptr(None if guesses is None else guesses[i]) for i in range(n)])
    g = np.ascontiguousarray(g)
    p = params if params is not None else RegistrationParameters.defaults()
    res = (Result * n)()
    lib().s3d_oracle_gicp_align_batch(sc, tc, g.ctypes.data_as(C.c_void_p), C.byref(p), n, n_threads, res)
    return list(res)


def transform_cloud(cloud, T):
    a, c = _cloud(cloud)
    t = np.ascontiguousarray(np.asarray(T, np.float64).T)
    out = np.empty_like(a)
    lib().s3d_oracle_transform_cloud(c, t.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


def combined_measurement(clouds, poses, patch_pose):
    """createCombinedMeasurement (PointCloudSensor.cpp:258-266) on explicit lists; poses[i] = correctedPose_i * sensorPose_i."""
    n = len(clouds)
    keep = []
    cc = (Cloud * max(n, 1))()
    total = 0
    for i in range(n):
        a, c = _cloud(clouds[i]); keep.append(a); cc[i] = c; total += a.shape[0]
    P = np.ascontiguousarray(np.stack([np.asarray(p, np.float64).T for p in poses])) if n else np.zeros((1, 4, 4))
    inv = np.ascontiguousarray(isometry_inverse(patch_pose).T)
    out = np.empty((max(total, 1), 4), np.float32)
    m = C.c_uint64(0)
    lib().s3d_oracle_combined_measurement(cc, P.ctypes.data_as(C.c_void_p), n, inv.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.byref(m))
    return out[: m.value].copy()


def isometry_inverse(T):
    """Eigen::Isometry3d::inverse(): [R^T | -R^T t], in double."""
    T = np.asarray(T, np.float64)
    out = np.eye(4)
    out[:3, :3] = T[:3, :3].T
    out[:3, 3] = -(T[:3, :3].T @ T[:3, 3])
    return out


def remove_outliers(cloud, radius, min_neighbors):
    a, c = _cloud(cloud)
    out = np.empty((max(a.shape[0], 1), 4), np.float32)
    keep = np.zeros(max(a.shape[0], 1), np.uint8)
    n = C.c_uint64(0)
    lib().s3d_oracle_remove_outliers(c, C.c_double(radius), C.c_uint(min_neighbors), out.ctypes.data_as(C.c_void_p), C.byref(n),
                                     keep.ctypes.data_as(C.c_void_p))
    return out[: n.value].copy(), keep[: a.shape[0]].astype(bool)


def build_map(clouds, poses, outlier_radius, outlier_neighbors, resolution):
    n = len(clouds)
    keep = []
    cc = (Cloud * n)()
    total = 0
    for i in range(n):
        a, c = _cloud(clouds[i]); keep.append(a); cc[i] = c; total += a.shape[0]
    P = np.ascontiguousarray(np.stack([np.asarray(p, np.float64).T for p in poses])) if n else np.zeros((0, 4, 4))
    out = np.empty((max(total, 1), 4), np.float32)
    m = C.c_uint64(0)
    lib().s3d_oracle_build_map(cc, P.ctypes.data_as(C.c_void_p), n, C.c_double(outlier_radius), C.c_uint(outlier_neighbors),
                               C.c_double(resolution), out.ctypes.data_as(C.c_void_p), C.byref(m))
    return out[: m.value].copy()


def fnv1a(array):
    """FNV-1a over the raw bytes of a numpy array, as baseline/doicp_driver.cpp hashes PCL's outputs."""
    a = np.ascontiguousarray(array)
    lib().s3d_oracle_fnv1a.restype = C.c_uint64
    lib().s3d_oracle_fnv1a.argtypes = [C.c_void_p, C.c_uint64]
    return "%016x" % lib().s3d_oracle_fnv1a(a.ctypes.data, a.nbytes)


def max_threads():
    return lib().s3d_oracle_max_threads()


def last_error():
    return lib().s3d_oracle_last_error().decode()
