"""Loop closures on device-built patches: s3d_prepare_combined_measurements builds every patch of a call on the device from its
distinct scans and prepares it under every spec; s3d_gicp_align_loop_batch_prepared runs createConstraint's coarse -> fine sequence
on the handles.  Both must give exactly what the host path gives: s3d_create_combined_measurement, s3d_prepare_clouds(_ndt) and
s3d_gicp_align_loop_batch on the host patches."""
import ctypes as C
import math

import numpy as np
import pytest

from slam3d_b200 import _abi
from slam3d_b200._abi import Cloud, PrepareSpec, RegistrationParameters, Result

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import slam3d_b200
    c = slam3d_b200.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def scans(kitti):
    """five distinct scans: the four KITTI clouds and every other point of the first one"""
    import slam3d_b200
    return [slam3d_b200.as_xyzw(k) for k in kitti] + [slam3d_b200.as_xyzw(kitti[0][1::2])]


def pose(i):
    a = 0.01 * i
    T = np.eye(4)
    T[:2, :2] = [[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]]
    T[:3, 3] = [0.7 * i, 0.05 * i, 0.01 * i]
    return T


def patch(members, centre):
    """(member scan indices, member poses, patch_pose) of the patch around scan `centre`"""
    return list(members), [pose(i) for i in members], pose(centre)


def host_patch(ctx, scans, p, with_pose=True):
    """the patch s3d_create_combined_measurement returns (patch_pose NULL without a pose: getAccumulatedCloud)"""
    import slam3d_b200
    if with_pose:
        return ctx.combined_measurement([scans[i] for i in p[0]], p[1], p[2])
    n = len(p[0])
    cc = (Cloud * n)(*[Cloud(scans[i].ctypes.data, scans[i].shape[0]) for i in p[0]])
    P = np.ascontiguousarray(np.stack([np.asarray(T, np.float64).T for T in p[1]]))
    out = np.empty((sum(scans[i].shape[0] for i in p[0]), 4), np.float32)
    m = C.c_uint64(0)
    assert slam3d_b200.lib().s3d_create_combined_measurement(ctx._h, cc, P.ctypes.data, n, None, out.ctypes.data, C.byref(m)) == 0
    return out[: m.value].copy()


def same(a, b):
    """bit-identical in every field of the result"""
    assert bytes(a) == bytes(b), (a.status, b.status, a.fitness, b.fitness, a.outer_iterations, b.outer_iterations)


def release(*hs):
    for h in hs:
        if isinstance(h, list):
            release(*h)
        else:
            h.release()


SPECS = [(0.1, 20, None), (0.2, 20, None), (0.5, 20, None), (0.2, 0, 1.0), (0.2, 0, 2.0)]


@pytest.mark.parametrize("with_pose", [True, False])
def test_patches_equal_host_patches(ctx, scans, with_pose):
    """patches of 1, 3 and 5 scans (one scan twice at two poses in the last): the handles of the device-built patches have the sizes
    and give the align results of the handles of the host patches, for GICP at three densities and NDT at two resolutions"""
    patches = [patch([2], 2), patch([0, 1, 2], 1), patch([0, 1, 2, 3, 4], 2), ([1, 3, 1], [pose(1), pose(3), pose(5)], pose(3))]
    if not with_pose:
        patches = [(m, p, None) for m, p, _ in patches]
    dev = ctx.prepare_combined_measurements(scans, patches, SPECS)
    assert len(dev) == len(patches) and all(len(row) == len(SPECS) for row in dev)
    clouds = [host_patch(ctx, scans, p, with_pose) for p in patches]
    assert [c.shape[0] for c in clouds] == [sum(scans[i].shape[0] for i in p[0]) for p in patches]
    guess = np.eye(4); guess[0, 3] = 0.3
    for s, (density, k, resolution) in enumerate(SPECS):
        if resolution is None:
            host = ctx.prepare_clouds(clouds, density, k)
            params = RegistrationParameters.defaults(point_cloud_density=density, correspondence_randomness=k)
        else:
            host = ctx.prepare_clouds_ndt(clouds, density, resolution)
            params = RegistrationParameters.defaults(point_cloud_density=density, registration_algorithm=_abi.ALG_NDT, resolution=resolution)
        d = [row[s] for row in dev]
        assert [h.size for h in d] == [h.size for h in host]
        assert all(h.size > 0 for h in d)
        assert all((h.density, h.k, h.resolution) == (x.density, x.k, x.resolution) for h, x in zip(d, host))
        # every patch as source and as target of the 3-scan patch
        pairs = [(p, 1) for p in range(len(patches))] + [(1, p) for p in range(len(patches)) if p != 1]
        got = ctx.gicp_align_prepared_batch([d[i] for i, _ in pairs], [d[j] for _, j in pairs], [guess] * len(pairs), params)
        want = ctx.gicp_align_prepared_batch([host[i] for i, _ in pairs], [host[j] for _, j in pairs], [guess] * len(pairs), params)
        for a, b in zip(got, want):
            same(a, b)
        release(host)
    release(dev)


def gicp(density, **kw):
    return RegistrationParameters.defaults(point_cloud_density=density, **kw)


def ndt(density, resolution=1.0, **kw):
    kw.setdefault("registration_algorithm", _abi.ALG_NDT)
    return RegistrationParameters.defaults(point_cloud_density=density, resolution=resolution, **kw)


def spec_of(p):
    if p.registration_algorithm in (_abi.ALG_NDT, _abi.ALG_NDT_OMP):
        return (p.point_cloud_density, 0, p.resolution)
    return (p.point_cloud_density, p.correspondence_randomness, None)


COMBOS = {
    "gicp/gicp": (gicp(0.5, max_correspondence_distance=5.0), gicp(0.2)),
    "ndt/gicp": (ndt(0.5, 2.0), gicp(0.2)),
    "gicp_omp/ndt_omp": (gicp(0.5, registration_algorithm=_abi.ALG_GICP_OMP, max_correspondence_distance=5.0),
                         ndt(0.2, 1.0, registration_algorithm=_abi.ALG_NDT_OMP)),
}


def loop_both_ways(ctx, scans, patches, pairs, guesses, coarse, fine):
    """(raw coarse, raw fine, prepared coarse, prepared fine) of the loop batch over `pairs` of patch indices"""
    clouds = [host_patch(ctx, scans, p) for p in patches]
    rc, rf = ctx.gicp_align_loop_batch([clouds[i] for i, _ in pairs], [clouds[j] for _, j in pairs], guesses, coarse, fine)
    specs = [spec_of(coarse)] + ([spec_of(fine)] if spec_of(fine) != spec_of(coarse) else [])
    h = ctx.prepare_combined_measurements(scans, patches, specs)
    c, f = 0, len(specs) - 1
    pc, pf = ctx.gicp_align_loop_batch_prepared([h[i][c] for i, _ in pairs], [h[j][c] for _, j in pairs], [h[i][f] for i, _ in pairs],
                                                [h[j][f] for _, j in pairs], guesses, coarse, fine)
    release(h)
    return rc, rf, pc, pf


@pytest.mark.parametrize("direct7", [False, True])
@pytest.mark.parametrize("bfgs", [False, True])
@pytest.mark.parametrize("combo", sorted(COMBOS))
def test_loop_batch_equals_raw_loop_batch(ctx, scans, combo, bfgs, direct7):
    """three candidates against one shared target patch, and a candidate of 60 points whose coarse align fails"""
    coarse, fine = COMBOS[combo]
    tiny = scans[0][:60].copy()
    all_scans = scans + [tiny]
    patches = [patch([1, 2, 3], 2), patch([0, 1, 2], 1), patch([2, 3, 4], 3), patch([3], 3), ([5], [pose(4)], pose(4))]
    pairs = [(1, 0), (2, 0), (3, 0), (4, 0)]
    guesses = [np.linalg.inv(pose(1)) @ pose(2), np.linalg.inv(pose(3)) @ pose(2), np.linalg.inv(pose(3)) @ pose(2), np.eye(4)]
    prev_opt = ctx.set_gicp_optimizer("bfgs" if bfgs else "newton")
    prev_search = ctx.set_ndt_omp_search("direct7" if direct7 else "kdtree")
    try:
        rc, rf, pc, pf = loop_both_ways(ctx, all_scans, patches, pairs, guesses, coarse, fine)
    finally:
        ctx.set_gicp_optimizer(prev_opt)
        ctx.set_ndt_omp_search(prev_search)
    for a, b in zip(pc, rc):
        same(a, b)
    for a, b in zip(pf, rf):
        same(a, b)
    assert pc[3].status == _abi.S3D_TOO_FEW_POINTS and bytes(pf[3]) == bytes(pc[3])
    assert any(r.status in (_abi.S3D_OK, _abi.S3D_NOT_CONVERGED, _abi.S3D_TOO_FAR_FROM_GUESS) for r in pc[:3])  # the optimiser ran


@pytest.mark.parametrize("failure", ["fitness", "translation"])
def test_coarse_failure_keeps_coarse_result(ctx, scans, failure):
    """a patch matched with itself from 0.4 m away: the coarse align fails its fitness gate, or finds the patch and fails the
    distance-from-guess gate; the fine align does not run and out_fine is the coarse result"""
    gate = {"max_fitness_score": -1.0} if failure == "fitness" else {"max_translation": 1e-12}
    coarse, fine = gicp(0.5, max_correspondence_distance=5.0, **gate), gicp(0.2)
    patches = [patch([0, 1], 1), patch([0, 1], 1)]
    guess = np.eye(4); guess[0, 3] = 0.4
    rc, rf, pc, pf = loop_both_ways(ctx, scans, patches, [(1, 0)], [guess], coarse, fine)
    assert pc[0].status == (_abi.S3D_NOT_CONVERGED if failure == "fitness" else _abi.S3D_TOO_FAR_FROM_GUESS)
    same(pc[0], rc[0])
    same(pf[0], rf[0])
    assert bytes(pf[0]) == bytes(pc[0])


def test_scans_are_uploaded_once(ctx, scans):
    """patches that share scans: the device path uploads each distinct scan once plus small tables, downloads no point data,
    and moves far fewer bytes than building the patches on the host and preparing those"""
    patches = [patch([0, 1, 2], 1), patch([1, 2, 3], 2), patch([2, 3, 0], 3), patch([1, 2, 3], 2)]
    c0 = ctx.counters()
    h = ctx.prepare_combined_measurements(scans, patches, [(0.2, 20, None)])
    c1 = ctx.counters()
    distinct = sum(16 * scans[i].shape[0] for i in (0, 1, 2, 3))
    members = sum(len(p[0]) for p in patches)
    tiles = sum((scans[i].shape[0] + 2047) // 2048 for p in patches for i in p[0])
    tables = members * (128 + 16) + len(patches) * 128 + 8 * tiles
    dev_h2d, dev_d2h = c1["h2d_bytes"] - c0["h2d_bytes"], c1["d2h_bytes"] - c0["d2h_bytes"]
    assert dev_h2d <= distinct + tables
    assert dev_d2h < 64 * 1024
    clouds = [host_patch(ctx, scans, p) for p in patches]
    host = ctx.prepare_clouds(clouds, 0.2, 20)
    c2 = ctx.counters()
    raw_h2d, raw_d2h = c2["h2d_bytes"] - c1["h2d_bytes"], c2["d2h_bytes"] - c1["d2h_bytes"]
    assert dev_h2d < 0.3 * raw_h2d
    assert raw_d2h > sum(16 * c.shape[0] for c in clouds)
    assert [x[0].size for x in h] == [x.size for x in host]
    release(h, host)


def raw_prepare(ctx, scans, member_scan, first, specs, n_patches=None, slot=0, with_pose=True):
    """s3d_prepare_combined_measurements through ctypes: (status, handles)"""
    import slam3d_b200
    n_patches = len(first) - 1 if n_patches is None else n_patches
    cc = (Cloud * max(len(scans), 1))(*scans)
    ms = np.ascontiguousarray(np.asarray(member_scan or [0], np.int32))
    mp = np.ascontiguousarray(np.stack([np.eye(4)] * max(len(member_scan), 1)))
    fm = np.ascontiguousarray(np.asarray(first, np.int32))
    pp = np.ascontiguousarray(np.stack([np.eye(4)] * max(n_patches, 1)))
    sp = (PrepareSpec * max(len(specs), 1))(*[PrepareSpec(*s) for s in specs])
    hh = (C.c_void_p * max(n_patches * len(specs), 1))()
    st = slam3d_b200.lib().s3d_prepare_combined_measurements(ctx._h, slot, cc, len(scans), ms.ctypes.data, mp.ctypes.data, fm.ctypes.data,
                                                             pp.ctypes.data if with_pose else None, n_patches, sp, len(specs), hh)
    return st, [hh[i] for i in range(n_patches * len(specs))]


def test_invalid_arguments(ctx, scans):
    cl = [Cloud(s.ctypes.data, s.shape[0]) for s in scans[:2]]
    good = (0.2, 20, 0.0)
    before = ctx.prepared_block_stats()
    cases = {
        "bad slot": dict(slot=1),
        "negative slot": dict(slot=-1),
        "NaN density": dict(specs=[good, (float("nan"), 20, 0.0)]),
        "k = 0": dict(specs=[(0.2, 0, 0.0)]),
        "k > 4096": dict(specs=[good, (0.2, 4097, 0.0)]),
        "k and resolution": dict(specs=[(0.2, 20, 1.0)]),
        "NaN resolution": dict(specs=[(0.2, 0, float("nan"))]),
        "infinite resolution": dict(specs=[good, (0.2, 0, float("inf"))]),
        "negative resolution": dict(specs=[(0.2, 0, -1.0)]),
        "member index too large": dict(member_scan=[0, 2]),
        "negative member index": dict(member_scan=[-1, 1]),
        "first member not 0": dict(first=[1, 2]),
        "decreasing members": dict(first=[0, 2, 1]),
        "2^31 points": dict(scans=[Cloud(scans[0].ctypes.data, 1 << 30)], member_scan=[0, 0], first=[0, 2]),
    }
    for name, kw in cases.items():
        args = dict(scans=cl, member_scan=[0, 1], first=[0, 2], specs=[good])
        args.update(kw)
        st, hh = raw_prepare(ctx, **args)
        assert st == _abi.S3D_INVALID_ARGUMENT, name
        assert all(h is None for h in hh), name
    assert ctx.prepared_block_stats() == before
    st, hh = raw_prepare(ctx, cl, [0, 1], [0, 2], [good, (0.5, 0, 1.0)])
    assert st == _abi.S3D_OK and all(hh)
    import slam3d_b200
    for h in hh:
        slam3d_b200.lib().s3d_release_cloud(ctx._h, h)
    st, hh = raw_prepare(ctx, cl, [], [0], [good], n_patches=0)
    assert st == _abi.S3D_OK and hh == []


def test_loop_batch_checks_handles(ctx, scans):
    patches = [patch([0, 1], 1), patch([1, 2], 2)]
    h = ctx.prepare_combined_measurements(scans, patches, [(0.5, 20, None), (0.2, 20, None), (0.2, 0, 1.0)])
    g5, g2, n1 = [x[0] for x in h], [x[1] for x in h], [x[2] for x in h]
    coarse, fine = gicp(0.5), gicp(0.2)
    import slam3d_b200
    with pytest.raises(slam3d_b200.S3DError, match=r"\(6\)"):  # fine handles of the coarse density
        ctx.gicp_align_loop_batch_prepared([g5[0]], [g5[1]], [g5[0]], [g5[1]], None, coarse, fine)
    with pytest.raises(slam3d_b200.S3DError, match=r"\(6\)"):  # coarse handles of another density
        ctx.gicp_align_loop_batch_prepared([g2[0]], [g2[1]], [g2[0]], [g2[1]], None, coarse, fine)
    with pytest.raises(slam3d_b200.S3DError, match=r"\(6\)"):  # GICP on NDT handles
        ctx.gicp_align_loop_batch_prepared([g5[0]], [g5[1]], [n1[0]], [n1[1]], None, coarse, fine)
    with pytest.raises(slam3d_b200.S3DError, match=r"\(6\)"):  # NDT grid of another resolution
        ctx.gicp_align_loop_batch_prepared([g5[0]], [g5[1]], [n1[0]], [n1[1]], None, coarse, ndt(0.2, 2.0))
    with pytest.raises(slam3d_b200.S3DError, match=r"\(6\)"):  # k of the fine pass
        ctx.gicp_align_loop_batch_prepared([g5[0]], [g5[1]], [g2[0]], [g2[1]], None, coarse, gicp(0.2, correspondence_randomness=10))
    rc, rf = ctx.gicp_align_loop_batch_prepared([g5[0]], [g5[1]], [n1[0]], [n1[1]], None, coarse, ndt(0.2, 1.0))
    assert rc[0].status in (0, 2, 3) and rf[0].status in (0, 2, 3)
    assert ctx.gicp_align_loop_batch_prepared([], [], [], [], None, coarse, fine) == ([], [])
    release(h)


def test_minihost_device_patches():
    """MiniHost with patch range 2 and three links per vertex: device-built patches give the edges (bit for bit) and the warnings
    of the batched host-patch path"""
    from test_gpu_host import _figure_eight, _run_trajectory2, load_host
    host = load_host()
    n, truth, scans, odoms = _figure_eight()
    sensor = host.s3dhost_sensor_create(b"velodyne")
    fine = RegistrationParameters.defaults(point_cloud_density=0.2)
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0)
    host.s3dhost_sensor_set_params(sensor, C.byref(fine), 0)
    host.s3dhost_sensor_set_params(sensor, C.byref(coarse), 1)
    runs = {}
    for mode in (1, 2):
        e, T, w = _run_trajectory2(host, sensor, scans, odoms, n, patch_range=2, batched=mode, max_links=3, radius=1.7)
        runs[mode] = (e, T, w, host.s3dhost_last_message())
    (e1, T1, w1, m1), (e2, T2, w2, m2) = runs[1], runs[2]
    assert np.array_equal(e1, e2) and np.array_equal(T1, T2) and (w1, m1) == (w2, m2)
    assert len(e1[e1[:, 2] == 1]) >= 2
    # NDT coarse pass through the same host path
    host.s3dhost_sensor_set_params(sensor, C.byref(ndt(0.5, 2.0)), 1)
    ra = _run_trajectory2(host, sensor, scans, odoms, n, patch_range=2, batched=1, max_links=3, radius=1.7)
    rb = _run_trajectory2(host, sensor, scans, odoms, n, patch_range=2, batched=2, max_links=3, radius=1.7)
    assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1]) and ra[2] == rb[2]
    host.s3dhost_sensor_destroy(sensor)
