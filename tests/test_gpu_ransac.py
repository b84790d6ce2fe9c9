"""GPU RANSAC plane fit and ground fill (ransac.cu) against the CPU oracle (oracle/ransac_oracle.cpp): equal float coefficients,
iterations, inlier counts and indices, bit-identical fill points; block size, device inputs and the host mirror change nothing."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_oracle_ransac import THRESHOLD, degenerate_clouds, ground_cloud

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ransac_oracle():
    from oracle import ransac
    ransac.lib()
    return ransac


@pytest.fixture(scope="module")
def ctx():
    import slam3d_b200
    c = slam3d_b200.Context()
    yield c
    c.close()


def synth_scan(seed):
    from slam3d_b200 import synth
    scene = synth.Scene(seed)
    return synth.scan(scene, synth.make_pose([0.0, 0.0, 0.0], [0.0, 0.0, 0.0]), np.random.default_rng(seed))


def check_fit(ctx, ransac_oracle, cloud, threshold=THRESHOLD, max_it=10000):
    ok, coeff, it, inl = ransac_oracle.fit_plane_ransac(cloud, threshold, max_it)
    assert ok
    g_coeff, g_it, g_n, g_inl = ctx.fit_plane_ransac(cloud, threshold, max_it, want_inliers=True)
    assert np.array_equal(g_coeff.view(np.uint32), coeff.view(np.uint32)), (g_coeff, coeff)
    assert g_it == it and g_n == len(inl)
    assert np.array_equal(g_inl, inl)
    return it


@pytest.mark.parametrize("i", range(4))
def test_golden_clouds(ctx, ransac_oracle, kitti, i):
    check_fit(ctx, ransac_oracle, kitti[i])


@pytest.mark.parametrize("seed", [3, 17])
def test_synthetic_scans(ctx, ransac_oracle, seed):
    check_fit(ctx, ransac_oracle, synth_scan(seed))


def test_nan_points(ctx, ransac_oracle):
    cloud = synth_scan(5).copy()
    rng = np.random.default_rng(5)
    cloud[rng.choice(len(cloud), len(cloud) // 10, replace=False)] = np.nan
    cloud[rng.choice(len(cloud), 100, replace=False), 1] = np.inf
    check_fit(ctx, ransac_oracle, cloud)
    check_fit(ctx, ransac_oracle, ground_cloud(6, 4000, nan_frac=0.2))


def test_map_2m_points(ctx, ransac_oracle):
    from slam3d_b200 import synth
    cloud = synth.map_cloud(n_scans=16)
    assert len(cloud) == 2097152
    check_fit(ctx, ransac_oracle, cloud)


@pytest.mark.parametrize("max_it", [1, 2, 10000])
def test_max_iterations(ctx, ransac_oracle, kitti, max_it):
    it = check_fit(ctx, ransac_oracle, ground_cloud(9, 20000, ground=0.05), max_it=max_it)
    assert it <= max_it + 1
    check_fit(ctx, ransac_oracle, kitti[0], max_it=max_it)


def test_thresholds(ctx, ransac_oracle, kitti):
    for thr in (0.0123456789, 0.05, 0.3):
        check_fit(ctx, ransac_oracle, kitti[1], threshold=thr)


def test_degenerate(ctx, ransac_oracle):
    import slam3d_b200
    d = degenerate_clouds()
    check_fit(ctx, ransac_oracle, d["three"])
    check_fit(ctx, ransac_oracle, d["identical"])
    for bad in (d["collinear"], d["three"][:2], np.zeros((0, 3), np.float32)):
        assert not ransac_oracle.fit_plane_ransac(bad, THRESHOLD)[0]
        with pytest.raises(slam3d_b200.S3DError):
            ctx.fit_plane_ransac(bad, THRESHOLD)
        with pytest.raises(slam3d_b200.S3DError):
            ctx.fill_ground_plane(bad, 2.0)
    with pytest.raises(slam3d_b200.S3DError):  # every point NaN: no plane has an inlier
        ctx.fit_plane_ransac(np.full((50, 3), np.nan, np.float32), THRESHOLD)


def test_bad_arguments(ctx):
    import slam3d_b200
    cloud = ground_cloud(1, 300)
    for thr, it, p in [(0.0, 10, 0.99), (-1.0, 10, 0.99), (float("nan"), 10, 0.99), (float("inf"), 10, 0.99), (0.01, 0, 0.99),
                       (0.01, 10, 0.0), (0.01, 10, 1.0), (0.01, 10, float("nan"))]:
        with pytest.raises(slam3d_b200.S3DError):
            ctx.fit_plane_ransac(cloud, thr, it, p)
    for res, radius in [(0.0, 1.0), (0.1, -1.0), (1e-6, 100.0)]:
        with pytest.raises(slam3d_b200.S3DError):
            ctx.fill_ground_plane(cloud, radius, res)


@pytest.mark.parametrize("res,radius", [(0.1, 2.0), (0.1, 10.0), (0.25, 3.0), (0.3, 0.2)])
def test_fill_bit_exact(ctx, ransac_oracle, kitti, res, radius):
    want, _ = ransac_oracle.fill_ground_plane(kitti[2], radius, res)
    got = ctx.fill_ground_plane(kitti[2], radius, res)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_fill_degenerate_planes(ctx, ransac_oracle):
    for cloud in (degenerate_clouds()["identical"], degenerate_clouds()["three"]):
        want, _ = ransac_oracle.fill_ground_plane(cloud, 1.0, 0.1)
        got = ctx.fill_ground_plane(cloud, 1.0, 0.1)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


_BLOCK_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import slam3d_b200
from conftest import load_kitti
from test_oracle_ransac import ground_cloud
ctx = slam3d_b200.Context()
out = []
for cloud, max_it in ((load_kitti(1), 10000), (load_kitti(3), 3), (ground_cloud(21, 20000, ground=0.05), 10000)):
    c, it, n, inl = ctx.fit_plane_ransac(cloud, 0.01, max_it, want_inliers=True)
    f = ctx.fill_ground_plane(cloud, 3.0, 0.1)
    out.append([c.view(np.uint32).tolist(), it, n, int(inl.sum()), f.view(np.uint32).sum(dtype=np.uint64).item()])
ctx.close()
print(json.dumps(out))
"""


def test_block_size_is_invisible():
    """S3D_RANSAC_BLOCK = 1, 7 and the default give identical results (the variable is read once per process)."""
    res = {}
    for b in ("1", "7", None):
        env = dict(os.environ)
        env.pop("S3D_RANSAC_BLOCK", None)
        if b:
            env["S3D_RANSAC_BLOCK"] = b
        r = subprocess.run([sys.executable, "-c", _BLOCK_SCRIPT, ROOT], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        res[b] = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["1"] == res["7"] == res[None]


def test_device_inputs(ctx, ransac_oracle, kitti):
    import torch
    cloud = kitti[0]
    t = torch.ones((len(cloud), 4), dtype=torch.float32, device="cuda")
    t[:, :3] = torch.from_numpy(cloud).cuda()
    host = ctx.fit_plane_ransac(cloud, THRESHOLD, want_inliers=True)
    dev = ctx.fit_plane_ransac(t, THRESHOLD, want_inliers=True)
    assert np.array_equal(host[0], dev[0]) and host[1:3] == dev[1:3] and np.array_equal(host[3], dev[3])
    assert np.array_equal(ctx.fill_ground_plane(t, 4.0), ctx.fill_ground_plane(cloud, 4.0))
    # device output buffers through the C-ABI
    import slam3d_b200
    from slam3d_b200._abi import Cloud
    n = slam3d_b200.ground_fill_size(0.1, 4.0)
    out = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    inl = torch.empty(len(cloud), dtype=torch.int32, device="cuda")
    coeff = np.zeros(4, np.float32)
    it, m = C.c_int32(0), C.c_uint64(0)
    L = slam3d_b200.lib()
    assert L.s3d_fill_ground_plane(ctx._h, Cloud(t.data_ptr(), len(cloud)), 0.1, 4.0, C.c_void_p(out.data_ptr()), coeff.ctypes.data) == 0
    assert np.array_equal(out.cpu().numpy(), ctx.fill_ground_plane(cloud, 4.0)) and np.array_equal(coeff, host[0])
    assert L.s3d_fit_plane_ransac(ctx._h, Cloud(t.data_ptr(), len(cloud)), THRESHOLD, 10000, 0.99, coeff.ctypes.data, C.byref(it), C.byref(m),
                                  C.c_void_p(inl.data_ptr())) == 0
    assert m.value == host[2] and np.array_equal(inl[: m.value].cpu().numpy().astype(np.uint32), host[3])


def test_host_mirror_fill_ground_plane(ransac_oracle, kitti):
    import slam3d_b200
    lib = C.CDLL(os.path.join(ROOT, "slam3d_b200", "libs3d_host.so"))
    lib.s3dhost_sensor_create.restype = C.c_void_p
    lib.s3dhost_sensor_destroy.argtypes = [C.c_void_p]
    lib.s3dhost_fill_ground_plane.restype = C.c_int64
    lib.s3dhost_fill_ground_plane.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_void_p]
    s = lib.s3dhost_sensor_create(b"lidar")
    try:
        for cloud, res, radius in ((kitti[3], 0.1, 5.0), (synth_scan(8), 0.2, 8.0)):
            a = ransac_oracle.as_xyzw(cloud)
            want, _ = ransac_oracle.fill_ground_plane(cloud, radius, res)
            out = np.empty((len(a) + slam3d_b200.ground_fill_size(res, radius), 4), np.float32)
            m = lib.s3dhost_fill_ground_plane(s, a.ctypes.data, len(a), res, radius, out.ctypes.data)
            assert m == len(a) + len(want)
            assert np.array_equal(out[: len(a)].view(np.uint32), a.view(np.uint32))
            assert np.array_equal(out[len(a): m].view(np.uint32), want.view(np.uint32))
    finally:
        lib.s3dhost_sensor_destroy(s)
