"""Resident scans: s3d_upload_scans copies scans once into library-owned device memory, and the device view of a handle
(s3d_resident_scan_cloud) stands in for the host cloud in every entry point, with bit-identical results and no further upload.
The host mirror's store (setResidentScanBudget) keeps the clouds of measurements resident across calls without changing an edge."""
import ctypes as C
import math

import numpy as np
import pytest

from slam3d_b200 import _abi
from slam3d_b200._abi import Cloud, RegistrationParameters

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import slam3d_b200
    c = slam3d_b200.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def scans(kitti):
    """the four KITTI clouds with w = 1, and one whose w holds arbitrary values (a verbatim copy keeps them)"""
    import slam3d_b200
    out = [slam3d_b200.as_xyzw(k) for k in kitti]
    odd = slam3d_b200.as_xyzw(kitti[0][::3]).copy()
    odd[:, 3] = np.random.default_rng(5).standard_normal(len(odd)).astype(np.float32)
    return out + [odd]


@pytest.fixture(scope="module")
def views(ctx, scans):
    v = ctx.upload_scans(scans)
    yield v
    for s in v:
        s.release()


def h2d(ctx):
    return ctx.counters()["h2d_bytes"]


def same(a, b):
    assert bytes(a) == bytes(b), (a.status, b.status, a.fitness, b.fitness, a.outer_iterations, b.outer_iterations)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def pose(i):
    a = 0.01 * i
    T = np.eye(4)
    T[:2, :2] = [[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]]
    T[:3, 3] = [0.7 * i, 0.05 * i, 0.01 * i]
    return T


def test_upload_is_verbatim_and_counted(ctx, scans):
    before = h2d(ctx)
    v = ctx.upload_scans(scans)
    assert h2d(ctx) - before == sum(16 * s.shape[0] for s in scans)
    assert [x.size for x in v] == [s.shape[0] for s in scans] and v[0].shape == (scans[0].shape[0], 4)
    for x, s in zip(v, scans):  # removeOutliers with radius 0 hands its input back unchanged: the device copy, byte for byte
        assert np.array_equal(bits(ctx.remove_outliers(x, 0.0, 0)), bits(s))
    # device inputs are copied device to device and count no host bytes
    import torch
    t = torch.from_numpy(scans[1]).cuda()
    torch.cuda.synchronize()
    before = h2d(ctx)
    (d,) = ctx.upload_scans([t])
    assert h2d(ctx) == before
    assert np.array_equal(bits(ctx.remove_outliers(d, 0.0, 0)), bits(scans[1]))
    for x in v + [d]:
        x.release()


def test_empty_scan(ctx):
    import slam3d_b200
    (e,) = ctx.upload_scans([np.zeros((0, 4), np.float32)])
    assert e.size == 0
    c = slam3d_b200.lib().s3d_resident_scan_cloud(e._h)
    assert c.n == 0 and not c.xyzw
    assert ctx.voxel_downsample(e, 0.1)[0].shape == (0, 4)
    e.release()
    with pytest.raises(ValueError, match="released"):
        ctx.voxel_downsample(e, 0.1)


CONFIGS = {
    "gicp": dict(point_cloud_density=0.2),
    "ndt": dict(point_cloud_density=0.2, registration_algorithm=_abi.ALG_NDT, resolution=1.0),
    "ndt_omp": dict(point_cloud_density=0.2, registration_algorithm=_abi.ALG_NDT_OMP, resolution=1.0),
}


@pytest.mark.parametrize("optimizer", ["newton", "bfgs"])
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_align_on_views(ctx, scans, views, config, optimizer):
    """s3d_gicp_align, _batch, _loop_batch, prepare (GICP or NDT) and the prepared batch: every result field equal, no H2D"""
    params = RegistrationParameters.defaults(**CONFIGS[config])
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0)
    guess = np.eye(4); guess[0, 3] = 0.6
    prev_opt = ctx.set_gicp_optimizer(optimizer)
    prev_search = ctx.set_ndt_omp_search("direct7" if config == "ndt_omp" else "kdtree")
    try:
        pairs = [(0, 1), (1, 2), (2, 3), (4, 0)]
        before = h2d(ctx)
        got = [ctx.gicp_align(views[i], views[j], guess, params) for i, j in pairs]
        got_b = ctx.gicp_align_batch([views[i] for i, _ in pairs], [views[j] for _, j in pairs], [guess] * 4, params)
        got_lc, got_lf = ctx.gicp_align_loop_batch([views[i] for i, _ in pairs], [views[j] for _, j in pairs], [guess] * 4, coarse, params)
        if config == "gicp":
            hv = ctx.prepare_clouds(views, params.point_cloud_density, params.correspondence_randomness)
        else:
            hv = ctx.prepare_clouds_ndt(views, params.point_cloud_density, params.resolution)
        got_p = ctx.gicp_align_prepared_batch([hv[i] for i, _ in pairs], [hv[j] for _, j in pairs], [guess] * 4, params)
        assert h2d(ctx) == before  # no point data crossed the link
        want = [ctx.gicp_align(scans[i], scans[j], guess, params) for i, j in pairs]
        want_b = ctx.gicp_align_batch([scans[i] for i, _ in pairs], [scans[j] for _, j in pairs], [guess] * 4, params)
        want_lc, want_lf = ctx.gicp_align_loop_batch([scans[i] for i, _ in pairs], [scans[j] for _, j in pairs], [guess] * 4, coarse, params)
        if config == "gicp":
            hs = ctx.prepare_clouds(scans, params.point_cloud_density, params.correspondence_randomness)
        else:
            hs = ctx.prepare_clouds_ndt(scans, params.point_cloud_density, params.resolution)
        want_p = ctx.gicp_align_prepared_batch([hs[i] for i, _ in pairs], [hs[j] for _, j in pairs], [guess] * 4, params)
    finally:
        ctx.set_gicp_optimizer(prev_opt)
        ctx.set_ndt_omp_search(prev_search)
    assert [h.size for h in hv] == [h.size for h in hs]
    for a, b in zip(got + got_b + got_lc + got_lf + got_p, want + want_b + want_lc + want_lf + want_p):
        same(a, b)
    assert all(r.status == _abi.S3D_OK for r in want[:3])
    for h in hv + hs:
        h.release()


def test_stages_and_maps_on_views(ctx, scans, views):
    """downsample, kNN covariances, 1-NN, transform, removeOutliers, buildMap, createCombinedMeasurement, RANSAC and the ground fill"""
    before = h2d(ctx)
    T = pose(3)
    got = {
        "voxel": ctx.voxel_downsample(views[2], 0.1),
        "knn": ctx.knn_covariances(views[3], 20),
        "nn": ctx.nearest_neighbors(views[0], views[1], T),
        "transform": ctx.transform_cloud(views[4], T),
        "outliers": ctx.remove_outliers(views[1], 0.3, 3),
        "map": ctx.build_map(views, [pose(i) for i in range(5)]),
        "patch": ctx.combined_measurement(views[:4], [pose(i) for i in range(4)], pose(1)),
        "ransac": ctx.fit_plane_ransac(views[2], 0.05, want_inliers=True),
    }
    assert h2d(ctx) == before
    got["fill"] = ctx.fill_ground_plane(views[2], 3.0, 0.25)
    want = {
        "voxel": ctx.voxel_downsample(scans[2], 0.1),
        "knn": ctx.knn_covariances(scans[3], 20),
        "nn": ctx.nearest_neighbors(scans[0], scans[1], T),
        "transform": ctx.transform_cloud(scans[4], T),
        "outliers": ctx.remove_outliers(scans[1], 0.3, 3),
        "map": ctx.build_map(scans, [pose(i) for i in range(5)]),
        "patch": ctx.combined_measurement(scans[:4], [pose(i) for i in range(4)], pose(1)),
        "ransac": ctx.fit_plane_ransac(scans[2], 0.05, want_inliers=True),
        "fill": ctx.fill_ground_plane(scans[2], 3.0, 0.25),
    }
    for k in want:
        g, w = got[k], want[k]
        g, w = (g if isinstance(g, tuple) else (g,)), (w if isinstance(w, tuple) else (w,))
        assert len(g) == len(w), k
        for a, b in zip(g, w):
            if isinstance(b, np.ndarray):
                assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
            else:
                assert a == b, k
    assert got["map"].shape[0] > 1000 and got["ransac"][2] > 1000


@pytest.mark.parametrize("bfgs", [False, True])
def test_combined_measurements_on_views(ctx, scans, views, bfgs):
    """s3d_prepare_combined_measurements from views feeds s3d_gicp_align_loop_batch_prepared with the results of host scans; the
    views add only the member tables to h2d_bytes"""
    patches = [([1, 2, 3], [pose(1), pose(2), pose(3)], pose(2)), ([0, 1, 2], [pose(0), pose(1), pose(2)], pose(1)),
               ([2, 3, 4], [pose(2), pose(3), pose(4)], pose(3)), ([3], [pose(3)], pose(3))]
    specs = [(0.5, 20, None), (0.2, 20, None)]
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0)
    fine = RegistrationParameters.defaults(point_cloud_density=0.2)
    pairs = [(1, 0), (2, 0), (3, 0)]
    guesses = [np.linalg.inv(pose(1)) @ pose(2), np.linalg.inv(pose(3)) @ pose(2), np.linalg.inv(pose(3)) @ pose(2)]
    prev = ctx.set_gicp_optimizer("bfgs" if bfgs else "newton")
    try:
        out = {}
        for name, src in (("views", views), ("host", scans)):
            before = h2d(ctx)
            h = ctx.prepare_combined_measurements(src, patches, specs)
            up = h2d(ctx) - before
            out[name] = (up, [x.size for row in h for x in row],
                         ctx.gicp_align_loop_batch_prepared([h[i][0] for i, _ in pairs], [h[j][0] for _, j in pairs], [h[i][1] for i, _ in pairs],
                                                            [h[j][1] for _, j in pairs], guesses, coarse, fine))
            for row in h:
                for x in row:
                    x.release()
    finally:
        ctx.set_gicp_optimizer(prev)
    (up_v, sz_v, (c_v, f_v)), (up_h, sz_h, (c_h, f_h)) = out["views"], out["host"]
    assert sz_v == sz_h
    for a, b in zip(c_v + f_v, c_h + f_h):
        same(a, b)
    assert up_h - up_v == sum(16 * scans[i].shape[0] for i in range(5))  # the host call uploads every distinct scan once, the views none
    assert up_v < 64 * 1024


def test_block_pool_reuse(ctx, scans):
    before = ctx.prepared_block_stats()
    v = ctx.upload_scans(scans[:3])
    mid = ctx.prepared_block_stats()
    for x in v:
        x.release()
    w = ctx.upload_scans(scans[:3])
    after = ctx.prepared_block_stats()
    assert after["allocated"] == mid["allocated"] and after["reused"] - mid["reused"] == 3
    assert mid["allocated"] + mid["reused"] - before["allocated"] - before["reused"] == 3
    for x in w:
        x.release()


def test_invalid_arguments(ctx, scans):
    import slam3d_b200
    L = slam3d_b200.lib()
    s = scans[0]
    good = Cloud(s.ctypes.data, s.shape[0])

    def call(clouds, n=None, slot=0, ctx_h=None, out=True):
        n = len(clouds) if n is None else n
        cc = (Cloud * max(len(clouds), 1))(*clouds)
        hh = (C.c_void_p * 4)(*[C.c_void_p(1)] * 4)  # poisoned: every slot must come back NULL
        st = L.s3d_upload_scans(ctx._h if ctx_h is None else ctx_h, slot, cc if clouds else None, n, hh if out else None)
        return st, [hh[i] for i in range(min(max(n, 0), 4))]

    before = ctx.prepared_block_stats()
    cases = {
        "bad slot": dict(clouds=[good], slot=1),
        "negative slot": dict(clouds=[good], slot=-1),
        "NULL clouds": dict(clouds=[], n=2),
        "n < 0": dict(clouds=[good], n=-1),
        "2^31 points": dict(clouds=[good, Cloud(s.ctypes.data, 1 << 31)]),
        "NULL points": dict(clouds=[good, Cloud(None, 5)]),
        "NULL output": dict(clouds=[good], out=False),
    }
    for name, kw in cases.items():
        st, hh = call(**kw)
        assert st == _abi.S3D_INVALID_ARGUMENT, name
        assert name == "NULL output" or all(h is None for h in hh), name
    assert L.s3d_upload_scans(None, 0, None, 0, None) == _abi.S3D_INVALID_ARGUMENT
    assert ctx.prepared_block_stats() == before  # no block was taken
    assert L.s3d_release_scan(ctx._h, None) == _abi.S3D_OK
    assert L.s3d_resident_scan_cloud(None).n == 0
    st, hh = call([good, Cloud(None, 0)])
    assert st == _abi.S3D_OK and all(hh[:2])
    assert L.s3d_resident_scan_cloud(hh[1]).n == 0 and L.s3d_resident_scan_cloud(hh[0]).n == s.shape[0]
    for h in hh[:2]:
        assert L.s3d_release_scan(ctx._h, h) == _abi.S3D_OK


def test_cross_device_batch(scans):
    """a view resident on slot 0 inside a raw batch sharded over two devices: the pairs of device 1 copy it device to device and
    every result equals the single-device one"""
    import torch
    import slam3d_b200
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: only one is visible")
    two = slam3d_b200.Context(devices=[0, 1])
    one = slam3d_b200.Context(devices=[0])
    try:
        v = two.upload_scans(scans[:4])
        params = RegistrationParameters.defaults(point_cloud_density=0.2)
        guess = np.eye(4); guess[0, 3] = 0.6
        pairs = [(0, 1), (1, 2), (2, 3), (3, 0), (1, 0), (2, 1)]
        before = two.counters()["h2d_bytes"]
        got = two.gicp_align_batch([v[i] for i, _ in pairs], [v[j] for _, j in pairs], [guess] * len(pairs), params)
        assert two.counters()["h2d_bytes"] == before
        want = one.gicp_align_batch([scans[i] for i, _ in pairs], [scans[j] for _, j in pairs], [guess] * len(pairs), params)
        for a, b in zip(got, want):
            same(a, b)
        h1 = two.prepare_clouds(v[:2], 0.2, 20, device_slot=1)  # a prepare on the other device reads the slot-0 views
        h0 = one.prepare_clouds(scans[:2], 0.2, 20)
        same(two.gicp_align_prepared(h1[0], h1[1], guess, params), one.gicp_align_prepared(h0[0], h0[1], guess, params))
        for h in h1 + h0 + v:
            h.release()
    finally:
        two.close()
        one.close()


# ---- host mirror ---------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def host():
    from test_gpu_host import load_host
    lib = load_host()
    lib.s3dhost_set_resident_budget.argtypes = [C.c_uint64]
    lib.s3dhost_resident_stats.argtypes = [C.POINTER(C.c_uint64)] * 3
    lib.s3dhost_map_stats.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int)]
    lib.s3dhost_context.restype = C.c_void_p
    lib.s3dhost_run_trajectory_maps.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int,
                                                C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.POINTER(C.c_int)]
    yield lib
    lib.s3dhost_set_resident_budget(0)


def stats(host):
    u, h, b = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    host.s3dhost_resident_stats(C.byref(u), C.byref(h), C.byref(b))
    return u.value, h.value, b.value


def host_h2d(host):
    import slam3d_b200
    c = _abi.Counters()
    slam3d_b200.lib().s3d_get_counters(C.c_void_p(host.s3dhost_context()), C.byref(c))
    return c.h2d_bytes


def run_maps(host, sensor, scans, odoms, budget, map_every=0, batched=2):
    """the patch-range-2 figure-eight (3 links per vertex) with the store at `budget`: (edges, T, warnings, last message, map sizes,
    map hashes, uploads, h2d bytes)"""
    n = len(scans)
    ptrs = (C.c_void_p * n)(*[s.ctypes.data for s in scans])
    sizes = (C.c_uint64 * n)(*[s.shape[0] for s in scans])
    od = np.ascontiguousarray(np.stack([o.T for o in odoms]))
    edges = np.zeros((6 * n, 3), np.int32); T = np.zeros((6 * n, 16)); nw = C.c_int(0)
    ms = np.zeros(n, np.uint64); mh = np.zeros(n, np.uint64)
    host.s3dhost_set_resident_budget(budget)
    u0, h0 = stats(host)[0], host_h2d(host)
    ne = host.s3dhost_run_trajectory_maps(sensor, ptrs, sizes, n, od.ctypes.data, 1.7, 3, 10, 2, batched, map_every, n, ms.ctypes.data,
                                          mh.ctypes.data, 6 * n, edges.ctypes.data, T.ctypes.data, None, C.byref(nw))
    assert ne >= n - 1, host.s3dhost_last_message()
    ms_s, mc = C.c_double(0), C.c_int(0)
    host.s3dhost_map_stats(C.byref(ms_s), C.byref(mc))
    u1, h1 = stats(host)[0], host_h2d(host)
    host.s3dhost_set_resident_budget(0)
    return (edges[:ne].copy(), T[:ne].copy(), nw.value, host.s3dhost_last_message(), ms[: mc.value].copy(), mh[: mc.value].copy(),
            u1 - u0, h1 - h0)


@pytest.fixture(scope="module")
def trajectory(host):
    from test_gpu_host import _figure_eight
    n, truth, scans, odoms = _figure_eight()
    sensor = host.s3dhost_sensor_create(b"velodyne")
    fine = RegistrationParameters.defaults(point_cloud_density=0.2)
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0)
    host.s3dhost_sensor_set_params(sensor, C.byref(fine), 0)
    host.s3dhost_sensor_set_params(sensor, C.byref(coarse), 1)
    off = run_maps(host, sensor, scans, odoms, 0, map_every=6)
    yield host, sensor, scans, odoms, off
    host.s3dhost_sensor_destroy(sensor)


def test_mirror_store_keeps_edges_and_uploads_once(trajectory):
    host, sensor, scans, odoms, off = trajectory
    on = run_maps(host, sensor, scans, odoms, 1 << 34, map_every=6)
    for a, b in zip(on[:4], off[:4]):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    assert len(off[0][off[0][:, 2] == 1]) >= 2  # loop edges were matched
    # periodic buildMap over the growing graph: the same maps from stored and from host scans
    assert len(off[4]) == len(scans) // 6 and np.array_equal(on[4], off[4]) and np.array_equal(on[5], off[5])
    points = sum(16 * s.shape[0] for s in scans)
    assert on[6] == len(scans)  # every scan uploaded once, on its first use
    assert points <= on[7] < points + points // 20  # 16 n per scan plus the patch tables
    assert off[7] > 2 * on[7]
    assert stats(host)[2] == 0  # the measurements are gone, and their scans with them


def test_mirror_store_under_a_small_budget(trajectory):
    host, sensor, scans, odoms, off = trajectory
    budget = sum(16 * s.shape[0] for s in scans) // 4
    small = run_maps(host, sensor, scans, odoms, budget, map_every=6)
    for a, b in zip(small[:6], off[:6]):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    assert small[6] > len(scans)  # evicted scans were uploaded again


def test_mirror_store_host_patches(trajectory):
    """the host-patch path (createConstraints on createCombinedMeasurement patches) with the store on gives the same edges"""
    host, sensor, scans, odoms, off = trajectory
    ref = run_maps(host, sensor, scans, odoms, 0, batched=1)
    on = run_maps(host, sensor, scans, odoms, 1 << 34, batched=1)
    for a, b in zip(on[:4], ref[:4]):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b
    assert np.array_equal(ref[0], off[0]) and np.array_equal(ref[1], off[1])


def test_mirror_store_two_threads(host, kitti):
    """two threads run createConstraint concurrently on one sensor with the store on: identical edges in both, equal to the store off"""
    import slam3d_b200
    sensor = host.s3dhost_sensor_create(b"velodyne")
    fine = RegistrationParameters.defaults(point_cloud_density=0.5)
    host.s3dhost_sensor_set_params(sensor, C.byref(fine), 0)
    scans = [slam3d_b200.as_xyzw(k[::2]) for k in kitti]
    ptrs = (C.c_void_p * 4)(*[s.ctypes.data for s in scans])
    sizes = (C.c_uint64 * 4)(*[s.shape[0] for s in scans])
    odoms = np.zeros((4, 4, 4))
    for i in range(4):
        o = np.eye(4); o[0, 3] = 0.65 * i
        odoms[i] = o.T
    out = {}
    for cache in (0, 32):  # raw align() path and prepared-cache misses
        host.s3dhost_set_cache_capacity(cache)
        for budget in (0, 1 << 34):
            host.s3dhost_set_resident_budget(budget)
            T = np.zeros((3, 16)); nw = C.c_int(0)
            assert host.s3dhost_run_odometry(sensor, ptrs, sizes, 4, odoms.ctypes.data, 2, T.ctypes.data, C.byref(nw)) == 3
            out[cache, budget] = T
    host.s3dhost_set_resident_budget(0)
    host.s3dhost_set_cache_capacity(32)
    first = out[0, 0]
    assert all(np.array_equal(first, T) for T in out.values())
    host.s3dhost_sensor_destroy(sensor)
