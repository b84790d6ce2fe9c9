"""slam3d_b200 — B200-native (sm_100a) scan matching behind slam3d::PointCloudSensor.

This package is a thin ctypes layer over libs3d_b200.so (hand-written CUDA, C-ABI in include/s3d_b200.h).
There is NO CPU fallback and the package never imports the test oracle: if the CUDA library is missing or no
device is present, calls fail loudly.
"""
import ctypes as C
import os

import numpy as np

from . import _abi
from ._abi import Cloud, Counters, PrepareSpec, RegistrationParameters, Result  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("S3D_LIB_PATH", os.path.join(_HERE, "libs3d_b200.so"))  # override: kernel-variant experiments only
_lib = None


class S3DError(RuntimeError):
    pass


def lib():
    """Loads libs3d_b200.so (built in-tree by slam3d_b200/build.py or __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise S3DError(f"{LIB_PATH} is missing: run `python slam3d_b200/build.py` (nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.s3d_last_error.restype = C.c_char_p
        L.s3d_version.restype = C.c_char_p
        L.s3d_context_stream.restype = C.c_void_p
        L.s3d_context_stream.argtypes = [C.c_void_p, C.c_int]
        L.s3d_create_context.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.s3d_destroy_context.argtypes = [C.c_void_p]
        L.s3d_get_counters.argtypes = [C.c_void_p, C.POINTER(Counters)]
        L.s3d_set_input_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.s3d_get_loop_stats.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int]
        L.s3d_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.s3d_set_gicp_optimizer.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.s3d_set_ndt_omp_search.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.s3d_get_stage_times.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.s3d_voxel_downsample.argtypes = [C.c_void_p, Cloud, C.c_float, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_int32)]
        L.s3d_knn_covariances.argtypes = [C.c_void_p, Cloud, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.s3d_nearest_neighbors.argtypes = [C.c_void_p, Cloud, Cloud, C.c_void_p, C.c_void_p, C.c_void_p]
        L.s3d_gicp_align.argtypes = [C.c_void_p, Cloud, Cloud, C.c_void_p, C.POINTER(RegistrationParameters), C.POINTER(Result)]
        L.s3d_gicp_align_batch.argtypes = [C.c_void_p, C.POINTER(Cloud), C.POINTER(Cloud), C.c_void_p, C.POINTER(RegistrationParameters),
                                           C.c_int, C.POINTER(Result)]
        L.s3d_gicp_align_loop_batch.argtypes = [C.c_void_p, C.POINTER(Cloud), C.POINTER(Cloud), C.c_void_p, C.POINTER(RegistrationParameters),
                                                C.POINTER(RegistrationParameters), C.c_int, C.POINTER(Result), C.POINTER(Result)]
        L.s3d_transform_cloud.argtypes = [C.c_void_p, Cloud, C.c_void_p, C.c_void_p]
        L.s3d_remove_outliers.argtypes = [C.c_void_p, Cloud, C.c_double, C.c_uint, C.c_void_p, C.POINTER(C.c_uint64)]
        L.s3d_build_map.argtypes = [C.c_void_p, C.POINTER(Cloud), C.c_void_p, C.c_int, C.c_double, C.c_uint, C.c_double, C.c_void_p,
                                    C.POINTER(C.c_uint64)]
        L.s3d_create_combined_measurement.argtypes = [C.c_void_p, C.POINTER(Cloud), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
        L.s3d_fit_plane_ransac.argtypes = [C.c_void_p, Cloud, C.c_double, C.c_int, C.c_double, C.c_void_p, C.POINTER(C.c_int32),
                                           C.POINTER(C.c_uint64), C.c_void_p]
        L.s3d_ground_fill_size.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_uint64)]
        L.s3d_fill_ground_plane.argtypes = [C.c_void_p, Cloud, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
        L.s3d_prepare_cloud.argtypes = [C.c_void_p, C.c_int, Cloud, C.c_double, C.c_int, C.POINTER(C.c_void_p)]
        L.s3d_prepare_clouds.argtypes = [C.c_void_p, C.c_int, C.POINTER(Cloud), C.c_int, C.c_double, C.c_int, C.POINTER(C.c_void_p)]
        L.s3d_prepare_cloud_ndt.argtypes = [C.c_void_p, C.c_int, Cloud, C.c_double, C.c_float, C.POINTER(C.c_void_p)]
        L.s3d_prepare_clouds_ndt.argtypes = [C.c_void_p, C.c_int, C.POINTER(Cloud), C.c_int, C.c_double, C.c_float, C.POINTER(C.c_void_p)]
        L.s3d_release_cloud.argtypes = [C.c_void_p, C.c_void_p]
        L.s3d_prepared_cloud_size.restype = C.c_uint64
        L.s3d_get_prepared_block_stats.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.s3d_prepared_cloud_size.argtypes = [C.c_void_p]
        L.s3d_gicp_align_prepared.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RegistrationParameters), C.POINTER(Result)]
        L.s3d_gicp_align_prepared_batch.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p,
                                                    C.POINTER(RegistrationParameters), C.c_int, C.POINTER(Result)]
        L.s3d_prepare_combined_measurements.argtypes = [C.c_void_p, C.c_int, C.POINTER(Cloud), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                        C.c_void_p, C.c_int, C.POINTER(PrepareSpec), C.c_int, C.POINTER(C.c_void_p)]
        L.s3d_upload_scans.argtypes = [C.c_void_p, C.c_int, C.POINTER(Cloud), C.c_int, C.POINTER(C.c_void_p)]
        L.s3d_release_scan.argtypes = [C.c_void_p, C.c_void_p]
        L.s3d_resident_scan_cloud.argtypes = [C.c_void_p]
        L.s3d_resident_scan_cloud.restype = Cloud
        L.s3d_gicp_align_loop_batch_prepared.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                                         C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(RegistrationParameters),
                                                         C.POINTER(RegistrationParameters), C.c_int, C.POINTER(Result), C.POINTER(Result)]
        _lib = L
    return _lib


def as_xyzw(a):
    """(n,3)/(n,4) numpy array -> C-contiguous float32 (n,4), w = 1 (pcl::PointXYZ memory). Torch tensors pass through."""
    if _is_torch(a):
        if a.dtype.__str__() != "torch.float32" or a.dim() != 2 or a.shape[1] != 4 or not a.is_contiguous():
            raise ValueError("torch clouds must be contiguous float32 (n,4)")
        return a
    a = np.asarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("cloud must be (n,3) or (n,4)")
    if a.shape[1] == 3:
        out = np.ones((a.shape[0], 4), np.float32)
        out[:, :3] = a
        return out
    return np.ascontiguousarray(a)


def _is_torch(a):
    return type(a).__module__.startswith("torch")


def _cloud(ctx, a):
    if isinstance(a, ResidentScan):  # a device cloud: the library reads it in place (or copies it to the GPU a call runs on)
        if not a._h:
            raise ValueError("ResidentScan was released")
        return a, lib().s3d_resident_scan_cloud(a._h)
    a = as_xyzw(a)
    if _is_torch(a):
        if a.is_cuda:
            # the library reads device inputs on its own streams: order them after the torch stream that produced the tensor
            import torch
            lib().s3d_set_input_stream(ctx._h, C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream), 1)
        return a, Cloud(a.data_ptr(), a.shape[0])
    return a, Cloud(a.ctypes.data, a.shape[0])


def _colmajor(T):
    return np.ascontiguousarray(np.asarray(np.eye(4) if T is None else T, np.float64).T)


class Context:
    """Owns the per-device workspaces/streams (s3d_create_context). One per process is enough; calls are re-entrant."""

    def __init__(self, devices=None):
        self._h = C.c_void_p()
        if devices:
            arr = (C.c_int * len(devices))(*devices)
            st = lib().s3d_create_context(arr, len(devices), C.byref(self._h))
        else:
            st = lib().s3d_create_context(None, 0, C.byref(self._h))
        if st != _abi.S3D_OK:
            raise S3DError(f"s3d_create_context failed ({st}): {last_error()}")

    def close(self):
        if self._h:
            lib().s3d_destroy_context(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, what):
        if st not in (_abi.S3D_OK,):
            raise S3DError(f"{what} failed ({st}): {last_error()}")

    def stream_handle(self, slot=0):
        return lib().s3d_context_stream(self._h, slot)

    STAGES = ("voxel", "grid", "knn_cov", "gicp_iter", "gicp_solve", "fitness")

    def set_profiling(self, enabled):
        lib().s3d_set_profiling(self._h, int(bool(enabled)))

    def stage_times(self, reset=True):
        ms = (C.c_double * 6)()
        n = (C.c_uint64 * 6)()
        lib().s3d_get_stage_times(self._h, ms, n, int(reset))
        return {k: {"ms": ms[i], "launches": int(n[i])} for i, k in enumerate(self.STAGES)}

    def set_gicp_optimizer(self, which):
        """Inner optimiser of every GICP registration on this context: "newton" (estimateRigidTransformationNewton, PCL >= 1.14's
        default; the default here) or "bfgs" (estimateRigidTransformationBFGS, the only one of PCL 1.8.1 ... 1.13).  NDT ignores
        it.  Change it while no call is running on the context.  Returns the previous setting."""
        if which not in _abi.GICP_OPTIMIZERS:
            raise ValueError(f"GICP optimizer must be one of {sorted(_abi.GICP_OPTIMIZERS)}, not {which!r}")
        prev = C.c_int(0)
        self._check(lib().s3d_set_gicp_optimizer(self._h, _abi.GICP_OPTIMIZERS[which], C.byref(prev)), "s3d_set_gicp_optimizer")
        return "bfgs" if prev.value == _abi.GICP_BFGS else "newton"

    def set_ndt_omp_search(self, which):
        """Neighbour search of every NDT_OMP registration on this context: "kdtree" (PCL's radius search, so NDT_OMP returns what NDT
        returns; the default here) or "direct7" (pclomp's default: the query's voxel and its 6 face neighbours).  NDT, GICP and
        GICP_OMP ignore it.  Change it while no call is running on the context.  Returns the previous setting."""
        if which not in _abi.NDT_OMP_SEARCHES:
            raise ValueError(f"NDT_OMP search must be one of {sorted(_abi.NDT_OMP_SEARCHES)}, not {which!r}")
        prev = C.c_int(0)
        self._check(lib().s3d_set_ndt_omp_search(self._h, _abi.NDT_OMP_SEARCHES[which], C.byref(prev)), "s3d_set_ndt_omp_search")
        return "direct7" if prev.value == _abi.NDT_OMP_DIRECT7 else "kdtree"

    def loop_stats(self, reset=False):
        t, c = C.c_uint64(0), C.c_uint64(0)
        lib().s3d_get_loop_stats(self._h, C.byref(t), C.byref(c), int(reset))
        return {"tiles": t.value, "control_steps": c.value}

    def prepared_block_stats(self):
        """Device blocks of prepared clouds since context creation: from cudaMalloc, and reused from released handles."""
        a, r = C.c_uint64(0), C.c_uint64(0)
        self._check(lib().s3d_get_prepared_block_stats(self._h, C.byref(a), C.byref(r)), "s3d_get_prepared_block_stats")
        return {"allocated": a.value, "reused": r.value}

    def counters(self):
        c = Counters()
        lib().s3d_get_counters(self._h, C.byref(c))
        return {"kernel_launches": c.kernel_launches, "h2d_bytes": c.h2d_bytes, "d2h_bytes": c.d2h_bytes}

    # PointCloudSensor::downsample (PointCloudSensor.cpp:190-201)
    def voxel_downsample(self, cloud, leaf, want_leaf_index=True):
        a, c = _cloud(self, cloud)
        n = a.shape[0]
        out = np.empty((max(n, 1), 4), np.float32)
        leaf_index = np.empty(max(n, 1), np.uint32) if want_leaf_index else None
        n_out = C.c_uint64(0)
        ov = C.c_int32(0)
        st = lib().s3d_voxel_downsample(self._h, c, leaf, out.ctypes.data, C.byref(n_out), leaf_index.ctypes.data if want_leaf_index else None, C.byref(ov))
        self._check(st, "s3d_voxel_downsample")
        return out[: n_out.value].copy(), (leaf_index[:n].copy() if want_leaf_index else None), bool(ov.value)

    def knn_covariances(self, cloud, k):
        a, c = _cloud(self, cloud)
        n = a.shape[0]
        idx = np.empty((n, k), np.uint32)
        d2 = np.empty((n, k), np.float32)
        cov = np.empty((n, 9), np.float64)
        st = lib().s3d_knn_covariances(self._h, c, k, idx.ctypes.data, d2.ctypes.data, cov.ctypes.data)
        self._check(st, "s3d_knn_covariances")
        return idx, d2, cov.reshape(n, 3, 3).transpose(0, 2, 1).copy()

    def nearest_neighbors(self, reference, queries, transform=None):
        r, rc = _cloud(self, reference)
        q, qc = _cloud(self, queries)
        idx = np.empty(q.shape[0], np.uint32)
        d2 = np.empty(q.shape[0], np.float32)
        t = _colmajor(transform) if transform is not None else None
        st = lib().s3d_nearest_neighbors(self._h, rc, qc, t.ctypes.data if t is not None else None, idx.ctypes.data, d2.ctypes.data)
        self._check(st, "s3d_nearest_neighbors")
        return idx, d2

    # align() (PointCloudSensor.cpp:119-174); returns the Result struct, status inside (0 ok, 1..3 = NoMatch reasons)
    def gicp_align(self, source, target, guess=None, params=None):
        s, sc = _cloud(self, source)
        t, tc = _cloud(self, target)
        g = _colmajor(guess)
        p = params if params is not None else RegistrationParameters.defaults()
        res = Result()
        st = lib().s3d_gicp_align(self._h, sc, tc, g.ctypes.data, C.byref(p), C.byref(res))
        if st in (_abi.S3D_INTERNAL_ERROR, _abi.S3D_INVALID_ARGUMENT):
            raise S3DError(f"s3d_gicp_align failed ({st}): {last_error()}")
        return res

    def gicp_align_batch(self, sources, targets, guesses=None, params=None):
        n = len(sources)
        keep = []
        sc = (Cloud * n)()
        tc = (Cloud * n)()
        for i in range(n):
            a, c = _cloud(self, sources[i]); keep.append(a); sc[i] = c
            a, c = _cloud(self, targets[i]); keep.append(a); tc[i] = c
        g = np.ascontiguousarray(np.stack([_colmajor(None if guesses is None else guesses[i]) for i in range(n)]))
        p = params if params is not None else RegistrationParameters.defaults()
        res = (Result * n)()
        st = lib().s3d_gicp_align_batch(self._h, sc, tc, g.ctypes.data, C.byref(p), n, res)
        self._check(st, "s3d_gicp_align_batch")
        return list(res)

    def gicp_align_loop_batch(self, sources, targets, guesses, coarse, fine):
        """createConstraint(loop=true) for a batch: coarse align, then fine align from the coarse pose. Returns (coarse, fine)."""
        n = len(sources)
        keep = []
        sc = (Cloud * n)()
        tc = (Cloud * n)()
        for i in range(n):
            a, c = _cloud(self, sources[i]); keep.append(a); sc[i] = c
            a, c = _cloud(self, targets[i]); keep.append(a); tc[i] = c
        g = np.ascontiguousarray(np.stack([_colmajor(None if guesses is None else guesses[i]) for i in range(n)]))
        rc = (Result * n)()
        rf = (Result * n)()
        st = lib().s3d_gicp_align_loop_batch(self._h, sc, tc, g.ctypes.data, C.byref(coarse), C.byref(fine), n, rc, rf)
        self._check(st, "s3d_gicp_align_loop_batch")
        return list(rc), list(rf)


class PreparedCloud:
    """Device-resident, preprocessed scan: voxel filter + NN grid + covariances (s3d_prepare_cloud, `k` set, `resolution` None)
    or + NDT voxel Gaussians (s3d_prepare_cloud_ndt, `k` 0, `resolution` the grid's) done once."""

    def __init__(self, ctx, handle, density, k, resolution=None):
        self._ctx, self._h, self.density, self.k, self.resolution = ctx, handle, density, k, resolution

    @property
    def size(self):
        return int(lib().s3d_prepared_cloud_size(self._h))

    def release(self):
        if self._h:
            lib().s3d_release_cloud(self._ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            if self._ctx._h:
                self.release()
        except Exception:
            pass


class ResidentScan:
    """A scan copied once into library-owned device memory of one device slot (s3d_upload_scans).  Every Context method that takes a
    cloud takes a ResidentScan in its place, with the same result as the host cloud and without uploading it again.  release()
    hands the memory back to the context's block pool."""

    def __init__(self, ctx, handle, size):
        self._ctx, self._h, self.size = ctx, handle, size

    @property
    def shape(self):
        return (self.size, 4)

    def release(self):
        if self._h:
            lib().s3d_release_scan(self._ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            if self._ctx._h:
                self.release()
        except Exception:
            pass


def _upload_scans(self, clouds, device_slot=0):
    """Copies each cloud (numpy array, torch tensor on the host or a GPU) verbatim to device memory of `device_slot`; returns one
    ResidentScan per cloud (all-or-nothing)."""
    n = len(clouds)
    keep = []
    cc = (Cloud * max(n, 1))()
    for i in range(n):
        a, c = _cloud(self, clouds[i]); keep.append(a); cc[i] = c
    hh = (C.c_void_p * max(n, 1))()
    self._check(lib().s3d_upload_scans(self._h, int(device_slot), cc, n, hh), "s3d_upload_scans")
    return [ResidentScan(self, C.c_void_p(hh[i]), int(cc[i].n)) for i in range(n)]


def _prepare_cloud(self, cloud, density, k=20, device_slot=0):
    a, c = _cloud(self, cloud)
    h = C.c_void_p()
    st = lib().s3d_prepare_cloud(self._h, device_slot, c, float(density), int(k), C.byref(h))
    self._check(st, "s3d_prepare_cloud")
    return PreparedCloud(self, h, float(density), int(k))


def _prepare_clouds(self, clouds, density, k=20, device_slot=0):
    n = len(clouds)
    keep = []
    cc = (Cloud * n)()
    for i in range(n):
        a, c = _cloud(self, clouds[i]); keep.append(a); cc[i] = c
    hh = (C.c_void_p * n)()
    st = lib().s3d_prepare_clouds(self._h, device_slot, cc, n, float(density), int(k), hh)
    self._check(st, "s3d_prepare_clouds")
    return [PreparedCloud(self, C.c_void_p(hh[i]), float(density), int(k)) for i in range(n)]


def _prepare_cloud_ndt(self, cloud, density, resolution, device_slot=0):
    """NDT handle: voxel filter at `density`, NN grid and the VoxelGridCovariance at `resolution` (what doNDT builds for its target)."""
    a, c = _cloud(self, cloud)
    h = C.c_void_p()
    st = lib().s3d_prepare_cloud_ndt(self._h, device_slot, c, float(density), float(resolution), C.byref(h))
    self._check(st, "s3d_prepare_cloud_ndt")
    return PreparedCloud(self, h, float(density), 0, float(C.c_float(resolution).value))


def _prepare_clouds_ndt(self, clouds, density, resolution, device_slot=0):
    n = len(clouds)
    keep = []
    cc = (Cloud * n)()
    for i in range(n):
        a, c = _cloud(self, clouds[i]); keep.append(a); cc[i] = c
    hh = (C.c_void_p * n)()
    st = lib().s3d_prepare_clouds_ndt(self._h, device_slot, cc, n, float(density), float(resolution), hh)
    self._check(st, "s3d_prepare_clouds_ndt")
    r = float(C.c_float(resolution).value)
    return [PreparedCloud(self, C.c_void_p(hh[i]), float(density), 0, r) for i in range(n)]


def _gicp_align_prepared(self, source, target, guess=None, params=None):
    g = _colmajor(guess)
    p = params if params is not None else RegistrationParameters.defaults()
    res = Result()
    st = lib().s3d_gicp_align_prepared(self._h, source._h, target._h, g.ctypes.data, C.byref(p), C.byref(res))
    if st in (_abi.S3D_INTERNAL_ERROR, _abi.S3D_INVALID_ARGUMENT):
        raise S3DError(f"s3d_gicp_align_prepared failed ({st}): {last_error()}")
    return res


def _gicp_align_prepared_batch(self, sources, targets, guesses=None, params=None):
    n = len(sources)
    sp = (C.c_void_p * n)(*[s._h for s in sources])
    tp = (C.c_void_p * n)(*[t._h for t in targets])
    g = np.ascontiguousarray(np.stack([_colmajor(None if guesses is None else guesses[i]) for i in range(n)]))
    p = params if params is not None else RegistrationParameters.defaults()
    res = (Result * n)()
    st = lib().s3d_gicp_align_prepared_batch(self._h, sp, tp, g.ctypes.data, C.byref(p), n, res)
    self._check(st, "s3d_gicp_align_prepared_batch")
    return list(res)


def _prepare_combined_measurements(self, scans, patches, specs, device_slot=0):
    """createCombinedMeasurement of every patch, built on the device from `scans` (each uploaded once) and prepared under every
    spec without a copy to the host (s3d_prepare_combined_measurements).  patches: list of (member scan indices, member poses,
    patch_pose); patch_pose None for all patches stops after the accumulation (getAccumulatedCloud).  specs: list of
    (density, k, resolution): k set and resolution None / 0 for a GICP handle, k 0 and resolution set for an NDT handle.
    Returns PreparedClouds as [patch][spec]."""
    n_scans, n_patches, n_specs = len(scans), len(patches), len(specs)
    keep = []
    cc = (Cloud * max(n_scans, 1))()
    for i in range(n_scans):
        a, c = _cloud(self, scans[i]); keep.append(a); cc[i] = c
    with_pose = [p[2] is not None for p in patches]
    if any(with_pose) and not all(with_pose):
        raise ValueError("patch_pose must be given for every patch or for none")
    members = [int(s) for p in patches for s in p[0]]
    first = np.cumsum([0] + [len(p[0]) for p in patches]).astype(np.int32)
    if any(len(p[0]) != len(p[1]) for p in patches):
        raise ValueError("every member scan needs its pose")
    ms = np.ascontiguousarray(np.asarray(members if members else [0], np.int32))
    mp = np.ascontiguousarray(np.stack([_colmajor(T) for p in patches for T in p[1]])) if members else np.zeros((1, 4, 4))
    pp = np.ascontiguousarray(np.stack([_colmajor(p[2]) for p in patches])) if n_patches and all(with_pose) else None
    sp = (PrepareSpec * max(n_specs, 1))()
    meta = []
    for i, (density, k, resolution) in enumerate(specs):
        r = float(resolution or 0.0)
        sp[i] = PrepareSpec(float(density), int(k), r)
        meta.append((float(density), int(k), float(C.c_float(r).value) if r else None))
    hh = (C.c_void_p * max(n_patches * n_specs, 1))()
    st = lib().s3d_prepare_combined_measurements(self._h, device_slot, cc, n_scans, ms.ctypes.data, mp.ctypes.data, first.ctypes.data,
                                                  pp.ctypes.data if pp is not None else None, n_patches, sp, n_specs, hh)
    self._check(st, "s3d_prepare_combined_measurements")
    return [[PreparedCloud(self, C.c_void_p(hh[p * n_specs + s]), *meta[s]) for s in range(n_specs)] for p in range(n_patches)]


def _gicp_align_loop_batch_prepared(self, coarse_sources, coarse_targets, fine_sources, fine_targets, guesses, coarse, fine):
    """createConstraint(loop=true) on prepared clouds: coarse align on the coarse handles, then fine align on the fine handles from
    the coarse pose (s3d_gicp_align_loop_batch_prepared).  Returns (coarse, fine) result lists."""
    n = len(coarse_sources)
    hs = [(C.c_void_p * max(n, 1))(*[h._h for h in x]) for x in (coarse_sources, coarse_targets, fine_sources, fine_targets)]
    g = np.ascontiguousarray(np.stack([_colmajor(None if guesses is None else guesses[i]) for i in range(n)])) if n else np.zeros((1, 4, 4))
    rc = (Result * max(n, 1))()
    rf = (Result * max(n, 1))()
    st = lib().s3d_gicp_align_loop_batch_prepared(self._h, hs[0], hs[1], hs[2], hs[3], g.ctypes.data, C.byref(coarse), C.byref(fine), n, rc, rf)
    self._check(st, "s3d_gicp_align_loop_batch_prepared")
    return list(rc)[:n], list(rf)[:n]


def _transform_cloud(self, cloud, T):
    a, c = _cloud(self, cloud)
    t = _colmajor(T)
    out = np.empty((a.shape[0], 4), np.float32)
    self._check(lib().s3d_transform_cloud(self._h, c, t.ctypes.data, out.ctypes.data), "s3d_transform_cloud")
    return out


def _remove_outliers(self, cloud, radius, min_neighbors):
    a, c = _cloud(self, cloud)
    out = np.empty((max(a.shape[0], 1), 4), np.float32)
    n = C.c_uint64(0)
    self._check(lib().s3d_remove_outliers(self._h, c, float(radius), int(min_neighbors), out.ctypes.data, C.byref(n)), "s3d_remove_outliers")
    return out[: n.value].copy()


def _build_map(self, clouds, poses, outlier_radius=0.2, outlier_neighbors=3, resolution=0.1):
    """PointCloudSensor::buildMap on explicit (cloud, pose) lists; defaults = the sensor's defaults (PointCloudSensor.cpp:179-183)."""
    n = len(clouds)
    keep = []
    cc = (Cloud * max(n, 1))()
    total = 0
    for i in range(n):
        a, c = _cloud(self, clouds[i]); keep.append(a); cc[i] = c; total += a.shape[0]
    P = np.ascontiguousarray(np.stack([_colmajor(p) for p in poses])) if n else np.zeros((1, 4, 4))
    out = np.empty((max(total, 1), 4), np.float32)
    m = C.c_uint64(0)
    self._check(lib().s3d_build_map(self._h, cc, P.ctypes.data, n, float(outlier_radius), int(outlier_neighbors), float(resolution),
                                    out.ctypes.data, C.byref(m)), "s3d_build_map")
    return out[: m.value].copy()


def _combined_measurement(self, clouds, poses, patch_pose):
    """createCombinedMeasurement (PointCloudSensor.cpp:258-266) on explicit (cloud, pose) lists."""
    n = len(clouds)
    keep = []
    cc = (Cloud * max(n, 1))()
    total = 0
    for i in range(n):
        a, c = _cloud(self, clouds[i]); keep.append(a); cc[i] = c; total += a.shape[0]
    P = np.ascontiguousarray(np.stack([_colmajor(p) for p in poses])) if n else np.zeros((1, 4, 4))
    pp = _colmajor(patch_pose)
    out = np.empty((max(total, 1), 4), np.float32)
    m = C.c_uint64(0)
    self._check(lib().s3d_create_combined_measurement(self._h, cc, P.ctypes.data, n, pp.ctypes.data, out.ctypes.data, C.byref(m)),
                "s3d_create_combined_measurement")
    return out[: m.value].copy()


def _fit_plane_ransac(self, cloud, threshold, max_iterations=10000, probability=0.99, want_inliers=False):
    """pcl::RandomSampleConsensus + SampleConsensusModelPlane (seeded as PCL seeds it, so the result is PCL's).  Returns
    (coefficients float32[4] = (a, b, c, d) with a unit normal, iterations, n_inliers, inliers): inliers are the ascending indices
    of the points with |a x + b y + c z + d| < threshold when want_inliers, else None."""
    a, c = _cloud(self, cloud)
    coeff = np.zeros(4, np.float32)
    it = C.c_int32(0)
    m = C.c_uint64(0)
    inl = np.empty(max(a.shape[0], 1), np.uint32) if want_inliers else None
    st = lib().s3d_fit_plane_ransac(self._h, c, float(threshold), int(max_iterations), float(probability), coeff.ctypes.data, C.byref(it),
                                    C.byref(m), inl.ctypes.data if want_inliers else None)
    self._check(st, "s3d_fit_plane_ransac")
    return coeff, it.value, m.value, (inl[: m.value].copy() if want_inliers else None)


def ground_fill_size(map_resolution, radius):
    """Number of points fill_ground_plane returns for (map_resolution, radius)."""
    n = C.c_uint64(0)
    st = lib().s3d_ground_fill_size(float(map_resolution), float(radius), C.byref(n))
    if st != _abi.S3D_OK:
        raise S3DError(f"s3d_ground_fill_size failed ({st}): {last_error()}")
    return n.value


def _fill_ground_plane(self, cloud, radius, map_resolution=0.1):
    """PointCloudSensor::fillGroundPlane: RANSAC plane of `cloud` (threshold 0.01), then rings of points every map_resolution up to
    `radius` laid into it.  Returns the new points (n,4) float32; the reference appends them to `cloud`."""
    a, c = _cloud(self, cloud)
    n = ground_fill_size(map_resolution, radius)
    out = np.empty((max(n, 1), 4), np.float32)
    self._check(lib().s3d_fill_ground_plane(self._h, c, float(map_resolution), float(radius), out.ctypes.data, None), "s3d_fill_ground_plane")
    return out[:n].copy()


Context.upload_scans = _upload_scans
Context.fit_plane_ransac = _fit_plane_ransac
Context.fill_ground_plane = _fill_ground_plane
Context.combined_measurement = _combined_measurement
Context.transform_cloud = _transform_cloud
Context.remove_outliers = _remove_outliers
Context.build_map = _build_map
Context.prepare_cloud = _prepare_cloud
Context.prepare_clouds = _prepare_clouds
Context.prepare_cloud_ndt = _prepare_cloud_ndt
Context.prepare_clouds_ndt = _prepare_clouds_ndt
Context.gicp_align_prepared = _gicp_align_prepared
Context.gicp_align_prepared_batch = _gicp_align_prepared_batch
Context.prepare_combined_measurements = _prepare_combined_measurements
Context.gicp_align_loop_batch_prepared = _gicp_align_loop_batch_prepared


def last_error():
    return lib().s3d_last_error().decode()
