"""NDT on prepared clouds: s3d_prepare_cloud(s)_ndt builds each scan's voxel filter, NN grid and NDT voxel Gaussians once, and
s3d_gicp_align_prepared(_batch) with NDT parameters must give exactly what s3d_gicp_align gives on the raw clouds."""
import ctypes as C
import math

import numpy as np
import pytest

from slam3d_b200 import _abi
from slam3d_b200._abi import RegistrationParameters

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import slam3d_b200
    c = slam3d_b200.Context()
    yield c
    c.close()


def ndt(**kw):
    kw.setdefault("point_cloud_density", 0.2)
    kw.setdefault("registration_algorithm", _abi.ALG_NDT)
    return RegistrationParameters.defaults(**kw)


def same(a, b):
    """bit-identical in every field of the result"""
    assert (a.status, a.converged) == (b.status, b.converged)
    assert (a.n_source, a.n_target, a.n_correspondences, a.outer_iterations, a.inner_iterations) == \
           (b.n_source, b.n_target, b.n_correspondences, b.outer_iterations, b.inner_iterations)
    assert np.array_equal(a.pose(), b.pose()) and a.fitness == b.fitness


@pytest.mark.parametrize("resolution", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("density", [0.1, 0.2, 0.3])
def test_parity_with_raw(ctx, kitti, density, resolution):
    p = ndt(point_cloud_density=density, resolution=resolution)
    h = ctx.prepare_clouds_ndt(kitti, density, resolution)
    assert all(x.resolution == resolution and x.k == 0 and x.density == density for x in h)
    for i in range(3):
        raw = ctx.gicp_align(kitti[i], kitti[i + 1], None, p)
        assert raw.status in (_abi.S3D_OK, _abi.S3D_NOT_CONVERGED, _abi.S3D_TOO_FAR_FROM_GUESS)
        same(ctx.gicp_align_prepared(h[i], h[i + 1], None, p), raw)
    for x in h:
        x.release()


def test_batches_reuse_handles(ctx, kitti):
    p = ndt(point_cloud_density=0.2, resolution=1.0)
    h = ctx.prepare_clouds_ndt(kitti, 0.2, 1.0)
    guess = np.eye(4); guess[0, 3] = 0.5
    raw = {(i, j): ctx.gicp_align(kitti[i], kitti[j], guess, p) for i, j in ((1, 0), (1, 2), (1, 3), (0, 1), (2, 3))}
    # one source against several targets, then an odometry chain in which handle 1 and 2 are first target, then source
    pairs = [(1, 0), (1, 2), (1, 3), (0, 1), (1, 2), (2, 3)]
    got = ctx.gicp_align_prepared_batch([h[i] for i, _ in pairs], [h[j] for _, j in pairs], [guess] * len(pairs), p)
    for (i, j), r in zip(pairs, got):
        same(r, raw[(i, j)])
    omp = ctx.gicp_align_prepared_batch([h[i] for i, _ in pairs], [h[j] for _, j in pairs], [guess] * len(pairs),
                                        ndt(point_cloud_density=0.2, resolution=1.0, registration_algorithm=_abi.ALG_NDT_OMP))
    for a, b in zip(omp, got):
        same(a, b)
    for x in h:
        x.release()


def test_gicp_handle_serves_as_target(ctx, kitti):
    p = ndt(point_cloud_density=0.3, resolution=1.0)
    src = ctx.prepare_cloud_ndt(kitti[0], 0.3, 1.0)
    tgt_gicp = ctx.prepare_cloud(kitti[1], 0.3, 20)
    tgt_ndt = ctx.prepare_cloud_ndt(kitti[1], 0.3, 1.0)
    raw = ctx.gicp_align(kitti[0], kitti[1], None, p)
    same(ctx.gicp_align_prepared(src, tgt_gicp, None, p), raw)
    same(ctx.gicp_align_prepared(src, tgt_ndt, None, p), raw)
    mixed = ctx.gicp_align_prepared_batch([src, src], [tgt_gicp, tgt_ndt], None, p)
    same(mixed[0], raw)
    same(mixed[1], raw)


def test_edges(ctx, kitti):
    import slam3d_b200
    p = ndt(point_cloud_density=0.2, resolution=1.0)
    a = ctx.prepare_cloud_ndt(kitti[0][::2], 0.2, 1.0)
    b = ctx.prepare_cloud_ndt(kitti[1][::2], 0.2, 1.0)
    empty = ctx.prepare_cloud_ndt(np.zeros((0, 3), np.float32), 0.2, 1.0)
    assert empty.size == 0
    assert ctx.gicp_align_prepared(empty, b, None, p).status == _abi.S3D_TOO_FEW_POINTS
    assert ctx.gicp_align_prepared(a, empty, None, p).status == _abi.S3D_TOO_FEW_POINTS
    small = ctx.prepare_cloud_ndt(kitti[0][:60], 0.2, 1.0)
    same(ctx.gicp_align_prepared(small, b, None, p), ctx.gicp_align(kitti[0][:60], kitti[1][::2], None, p))
    assert ctx.gicp_align_prepared(small, b, None, p).status == _abi.S3D_TOO_FEW_POINTS
    # int32 voxel-count guard: "Voxel grid is not searchable", same fields as the raw call
    p_tiny = ndt(point_cloud_density=0.2, resolution=0.01)
    fine = ctx.prepare_cloud_ndt(kitti[0][::2], 0.2, 0.01)
    raw = ctx.gicp_align(kitti[0][::2], kitti[1][::2], None, p_tiny)
    assert raw.status == _abi.S3D_NOT_CONVERGED and raw.outer_iterations == 0
    same(ctx.gicp_align_prepared(fine, b, None, p_tiny), raw)
    # call-level argument errors
    with pytest.raises(slam3d_b200.S3DError, match="resolution"):
        ctx.gicp_align_prepared(a, b, None, ndt(point_cloud_density=0.2, resolution=0.5))
    with pytest.raises(slam3d_b200.S3DError, match="another point_cloud_density"):
        ctx.gicp_align_prepared(a, b, None, ndt(point_cloud_density=0.3, resolution=1.0))
    with pytest.raises(slam3d_b200.S3DError, match="NDT data"):
        ctx.gicp_align_prepared(a, b, None, RegistrationParameters.defaults(point_cloud_density=0.2))
    for bad in (0.0, -1.0, math.nan):
        with pytest.raises(slam3d_b200.S3DError, match="resolution"):
            ctx.prepare_cloud_ndt(kitti[0][::2], 0.2, bad)
        with pytest.raises(slam3d_b200.S3DError, match="resolution"):
            ctx.prepare_clouds_ndt([kitti[0][::2], kitti[1][::2]], 0.2, bad)
    # a GICP handle as the NDT source: the per-pair result of before
    g = ctx.prepare_cloud(kitti[0][::2], 0.2, 20)
    assert ctx.gicp_align_prepared(g, b, None, p).status == _abi.S3D_UNKNOWN_ALGORITHM
    r = ctx.gicp_align_prepared_batch([g, a], [b, b], None, p)
    assert r[0].status == _abi.S3D_UNKNOWN_ALGORITHM
    same(r[1], ctx.gicp_align(kitti[0][::2], kitti[1][::2], None, p))


def test_released_blocks_are_recycled(ctx, kitti):
    p = ndt(point_cloud_density=0.2, resolution=1.0)
    h = ctx.prepare_clouds_ndt(kitti[:2], 0.2, 1.0)
    first = ctx.gicp_align_prepared(h[0], h[1], None, p)
    for x in h:
        x.release()
    b0 = ctx.prepared_block_stats()
    h = ctx.prepare_clouds_ndt(kitti[:2], 0.2, 1.0)          # the released blocks fit and are handed out again
    b1 = ctx.prepared_block_stats()
    assert b1["reused"] - b0["reused"] == 2 and b1["allocated"] == b0["allocated"]
    same(ctx.gicp_align_prepared(h[0], h[1], None, p), first)
    q = ctx.prepare_clouds_ndt(kitti[2:], 0.2, 1.0)
    same(ctx.gicp_align_prepared(q[0], q[1], None, p), ctx.gicp_align(kitti[2], kitti[3], None, p))
    same(ctx.gicp_align_prepared(h[0], h[1], None, p), ctx.gicp_align(kitti[0], kitti[1], None, p))


def test_device_inputs(ctx, kitti):
    import torch
    import slam3d_b200
    p = ndt(point_cloud_density=0.2, resolution=1.0)
    dev = [torch.from_numpy(slam3d_b200.as_xyzw(k)).cuda() for k in kitti[:2]]
    hd = ctx.prepare_clouds_ndt(dev, 0.2, 1.0)
    hh = ctx.prepare_clouds_ndt(kitti[:2], 0.2, 1.0)
    assert [x.size for x in hd] == [x.size for x in hh]
    same(ctx.gicp_align_prepared(hd[0], hd[1], None, p), ctx.gicp_align_prepared(hh[0], hh[1], None, p))
    torch.cuda.synchronize()


def test_no_reupload(ctx, kitti):
    p = ndt(point_cloud_density=0.2, resolution=1.0)
    h = ctx.prepare_clouds_ndt(kitti, 0.2, 1.0)
    c0 = ctx.counters()
    raw = ctx.gicp_align_batch(kitti[:-1], kitti[1:], None, p)
    c1 = ctx.counters()
    prep = ctx.gicp_align_prepared_batch(h[:-1], h[1:], None, p)
    c2 = ctx.counters()
    for a, b in zip(prep, raw):
        same(a, b)
    raw_h2d, prep_h2d = c1["h2d_bytes"] - c0["h2d_bytes"], c2["h2d_bytes"] - c1["h2d_bytes"]
    assert raw_h2d > 0 and prep_h2d < 0.01 * raw_h2d
    assert c2["kernel_launches"] - c1["kernel_launches"] < c1["kernel_launches"] - c0["kernel_launches"]


def test_host_mirror_cache(kitti):
    import slam3d_b200
    from test_gpu_host import create_constraint, load_host
    host = load_host()
    sensor = host.s3dhost_sensor_create(b"velodyne")
    fine = ndt(point_cloud_density=0.5, resolution=1.0)
    host.s3dhost_sensor_set_params(sensor, C.byref(fine), 0)
    I = np.eye(4)
    odom = np.eye(4); odom[0, 3] = 0.65
    try:
        runs = []
        for cap in (0, 32):
            host.s3dhost_set_cache_capacity(cap)
            runs.append([create_constraint(host, sensor, kitti[i][::2], kitti[i + 1][::2], I, I, odom) for i in range(3)])
        for (st0, T0, _, m0), (st1, T1, _, m1) in zip(*runs):
            assert st0 == st1 and (st0 == 0 or m0 == m1)
            assert np.array_equal(T0, T1)
        assert any(st == 0 for st, _, _, _ in runs[0])
        # a scan reused under NDT (target of one edge, source of the next) is prepared once
        scans = [slam3d_b200.as_xyzw(k[::2]) for k in kitti]
        ptrs = (C.c_void_p * 4)(*[s.ctypes.data for s in scans])
        sizes = (C.c_uint64 * 4)(*[s.shape[0] for s in scans])
        odoms = np.zeros((4, 4, 4))
        for i in range(4):
            o = np.eye(4); o[0, 3] = 0.65 * i
            odoms[i] = o.T
        out = np.zeros((3, 16)); nw = C.c_int(0)
        host.s3dhost_set_cache_capacity(0)
        n0 = host.s3dhost_run_odometry(sensor, ptrs, sizes, 4, odoms.ctypes.data, 1, out.ctypes.data, C.byref(nw))
        uncached, w0 = out.copy(), nw.value
        n_ok = sum(st == 0 for st, _, _, _ in runs[0])       # the same three registrations as the create_constraint calls above
        assert n0 == n_ok and w0 == 3 - n_ok and all(uncached[e].any() for e in range(n0))
        host.s3dhost_set_cache_capacity(32)
        hits0 = host.s3dhost_cache_hits()
        n1 = host.s3dhost_run_odometry(sensor, ptrs, sizes, 4, odoms.ctypes.data, 1, out.ctypes.data, C.byref(nw))
        assert host.s3dhost_cache_hits() - hits0 == 2
        assert n1 == n0 and nw.value == w0 and np.array_equal(out, uncached)
    finally:
        host.s3dhost_set_cache_capacity(32)
        host.s3dhost_sensor_destroy(sensor)
