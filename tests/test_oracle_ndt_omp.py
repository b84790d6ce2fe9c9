"""NDT_OMP with pclomp's default DIRECT7 neighbour search (oracle/ndt_omp_oracle.cpp through oracle/ndt_omp.py) on the CPU.

The oracle's DIRECT7 neighbourhoods are checked against an independent numpy restatement of
VoxelGridCovariance::getNeighborhoodAtPoint7: float32 division by the leaf size, floor, the min_b / max_b bounds, leaves with
>= 6 points, invalid leaves dropped, pclomp's offset order.  Then the DIRECT7 registration is run end to end, and the setting
is shown to leave NDT and GICP untouched, with the KDTREE mode equal to NDT."""
import numpy as np
import pytest

from conftest import pose_delta
from slam3d_b200 import _abi, synth
from slam3d_b200._abi import RegistrationParameters

OFFSETS = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]


@pytest.fixture(scope="module")
def omp_oracle(oracle_mod):
    from oracle import ndt_omp
    ndt_omp.lib()
    return ndt_omp


@pytest.fixture
def direct7(omp_oracle):
    old = omp_oracle.set_ndt_omp_search("direct7")
    yield omp_oracle
    omp_oracle.set_ndt_omp_search(old)


def numpy_grid(target, res):
    """VoxelGridCovariance<PointXYZ>::applyFilter in numpy: min_b / max_b / divb_mul and the set of keys of usable leaves
    (>= 6 points, not marked invalid by the eigenvalue test)."""
    t = np.asarray(target, np.float32)[:, :3]
    t = t[np.isfinite(t).all(axis=1)]
    inv = np.float32(1.0) / np.float32(res)
    min_b = np.floor(t.min(axis=0) * inv).astype(np.int64)
    max_b = np.floor(t.max(axis=0) * inv).astype(np.int64)
    div = max_b - min_b + 1
    mul = np.array([1, div[0], div[0] * div[1]], np.int64)
    ijk = np.floor(t * inv).astype(np.int64) - min_b  # applyFilter keys the points with the multiplication
    keys = ijk @ mul
    usable = set()
    order = np.argsort(keys, kind="stable")
    uk, start, cnt = np.unique(keys[order], return_index=True, return_counts=True)
    for k, s, n in zip(uk, start, cnt):
        if n < 6:
            continue
        p = t[order[s:s + n]].astype(np.float64)
        ms = p.sum(axis=0)
        cs = p.T @ p
        mean = ms / n
        cov = ((cs - 2.0 * np.outer(ms, mean)) / n + np.outer(mean, mean)) * ((n - 1.0) / n)
        ev = np.linalg.eigvalsh(cov)
        if ev[0] < -1e-12 or ev[1] < -1e-12 or ev[2] <= 0:
            continue  # nr_points = -1
        usable.add(int(k))
    return dict(min_b=min_b, max_b=max_b, mul=mul, usable=usable)


def numpy_direct7(grid, queries, res):
    out = []
    for q in np.asarray(queries, np.float32)[:, :3]:
        row = []
        if np.isfinite(q).all():
            ijk = np.floor(q / np.float32(res)).astype(np.int64)  # getNeighborhoodAtPoint: float division
            for d in OFFSETS:
                c = ijk + np.array(d)
                if (c < grid["min_b"]).any() or (c > grid["max_b"]).any():
                    continue
                key = int((c - grid["min_b"]) @ grid["mul"])
                if key in grid["usable"]:
                    row.append(key)
        out.append(row)
    return out


def query_points(target, res, rng, n=4000):
    """Random points over the grid and past its bounds, cell-face points k * res (and their float neighbours), NaN / inf."""
    t = np.asarray(target, np.float32)[:, :3]
    lo, hi = t.min(axis=0), t.max(axis=0)
    span = hi - lo
    q = [rng.uniform(lo - 0.2 * span - 2 * res, hi + 0.2 * span + 2 * res, size=(n, 3)).astype(np.float32)]
    base = t[rng.integers(0, len(t), size=n)]
    faces = (np.round(base / np.float32(res)) * np.float32(res)).astype(np.float32)  # exactly on cell faces (per axis)
    q += [faces, np.nextafter(faces, np.float32(np.inf)), np.nextafter(faces, np.float32(-np.inf)), base]
    q.append(np.array([[np.nan, 0, 0], [np.inf, 1, 1], [0, -np.inf, 0]], np.float32))
    return np.concatenate(q).astype(np.float32)


def with_degenerate_voxels(target, res):
    """Adds voxels of 7 identical points: their covariance is exactly 0, so applyFilter marks them invalid (nr_points = -1)."""
    t = np.asarray(target, np.float32)[:, :3]
    c = t[:: max(1, len(t) // 8)][:8] + np.float32(3 * res)
    c = (np.floor(c / np.float32(res)) + np.float32(0.5)) * np.float32(res)
    return np.concatenate([t, np.repeat(c.astype(np.float32), 7, axis=0)]), c.astype(np.float32)


def compare(omp_oracle, target, res, queries):
    keys, counts, n_c = omp_oracle.ndt_direct7_keys(target, res, queries)
    assert n_c > 0
    want = numpy_direct7(numpy_grid(target, res), queries, res)
    for i, w in enumerate(want):
        assert list(keys[i, :counts[i]]) == w, (i, queries[i], list(keys[i, :counts[i]]), w)
    assert (keys[np.arange(7)[None, :] >= counts[:, None]] == 0xFFFFFFFF).all()
    return counts


@pytest.mark.parametrize("res", [0.3, 0.5, 0.7, 1.0, 2.0])
def test_direct7_neighbourhoods_synthetic(oracle_mod, omp_oracle, res):
    src, tgt, _ = synth.scan_pair(seed=11)
    target, centres = with_degenerate_voxels(oracle_mod.voxel_downsample(src, 0.1)[0], res)
    rng = np.random.default_rng(int(res * 100))
    q = np.concatenate([query_points(target, res, rng), centres])
    counts = compare(omp_oracle, target, res, q)
    assert counts.max() >= 4 and (counts == 0).any()
    assert (counts[-len(centres):] < 7).all()  # the invalid leaf under each degenerate centre is never returned
    # the division of getNeighborhoodAtPoint and applyFilter's multiplication disagree on some of these queries unless the
    # leaf size is a power of two (then 1 / res is exact and the two agree everywhere)
    qf = q[np.isfinite(q).all(axis=1)]
    inv = np.float32(1.0) / np.float32(res)
    assert (np.floor(qf / np.float32(res)) != np.floor(qf * inv)).any() == (res not in (0.5, 1.0, 2.0))


@pytest.mark.parametrize("res", [0.5, 1.0, 2.0])
def test_direct7_neighbourhoods_kitti(oracle_mod, omp_oracle, kitti, res):
    target = oracle_mod.voxel_downsample(kitti[0], 0.2)[0]
    rng = np.random.default_rng(7)
    compare(omp_oracle, target, res, np.concatenate([query_points(target, res, rng, 2000), kitti[1][::50]]))


def ndt_omp(**kw):
    kw.setdefault("point_cloud_density", 0.1)
    kw.setdefault("registration_algorithm", _abi.ALG_NDT_OMP)
    return RegistrationParameters.defaults(**kw)


def test_direct7_registration_converges(direct7):
    """Same pair, density and 2 cm / 2 mrad bound as test_oracle_ndt.py's radius-search run.  Measured: DIRECT7 ends 1.9 mm and
    0.0 mrad (below what pose_delta resolves on a float pose) from the ground truth after 21 outer iterations with 203 438
    (point, voxel) pairs; the radius search ends 1.8 mm / 0.22 mrad away after 18 with 142 858 pairs."""
    src, tgt, truth = synth.scan_pair(seed=11)
    r = direct7.gicp_align(src, tgt, None, ndt_omp())
    assert r.status == _abi.S3D_OK and r.converged == 1 and 2 <= r.outer_iterations < 50
    dt, dr = pose_delta(r.pose(), truth)
    assert dt < 0.02 and dr < 2e-3, (dt, dr)
    ndt = direct7.gicp_align(src, tgt, None, ndt_omp(registration_algorithm=_abi.ALG_NDT))
    assert r.n_correspondences != ndt.n_correspondences  # another neighbourhood, another iterate sequence


def same(a, b):
    assert (a.status, a.converged, a.outer_iterations, a.inner_iterations, a.n_correspondences, a.fitness) == (
        b.status, b.converged, b.outer_iterations, b.inner_iterations, b.n_correspondences, b.fitness)
    assert np.array_equal(a.pose(), b.pose())


def test_setting_leaves_other_algorithms_unchanged(oracle_mod, omp_oracle, kitti):
    """NDT and GICP ignore the setting; the KDTREE mode of NDT_OMP is PCL's NDT bit for bit."""
    src, tgt = kitti[0], kitti[1]
    ndt_p = RegistrationParameters.defaults(point_cloud_density=0.3, registration_algorithm=_abi.ALG_NDT)
    cases = [ndt_p, RegistrationParameters.defaults(point_cloud_density=0.5)]
    before = [oracle_mod.gicp_align(src, tgt, None, p) for p in cases]
    assert omp_oracle.set_ndt_omp_search("kdtree") == "kdtree"
    same(omp_oracle.gicp_align(src, tgt, None, ndt_omp(point_cloud_density=0.3)), before[0])
    assert omp_oracle.set_ndt_omp_search("direct7") == "kdtree"
    try:
        for p, b in zip(cases, before):
            same(omp_oracle.gicp_align(src, tgt, None, p), b)
        d7 = omp_oracle.gicp_align(src, tgt, None, ndt_omp(point_cloud_density=0.3))
        assert d7.status == _abi.S3D_OK and d7.n_correspondences != before[0].n_correspondences
    finally:
        assert omp_oracle.set_ndt_omp_search("kdtree") == "direct7"
    with pytest.raises(ValueError):
        omp_oracle.set_ndt_omp_search("direct26")


def test_direct7_gates(direct7, kitti):
    """align()'s gates around the DIRECT7 registration: fitness, distance from the guess, < 100 points, unsearchable grid."""
    src, tgt = kitti[0][::2], kitti[1][::2]
    r = direct7.gicp_align(src, tgt, None, ndt_omp(point_cloud_density=0.2, max_fitness_score=1e-6))
    assert r.status == _abi.S3D_NOT_CONVERGED and "NDT failed with Fitness-Score" in direct7.last_error()
    r = direct7.gicp_align(src, tgt, None, ndt_omp(point_cloud_density=0.2, max_translation=0.01))
    assert r.status == _abi.S3D_TOO_FAR_FROM_GUESS
    r = direct7.gicp_align(src[:500], tgt[:500], None, ndt_omp(point_cloud_density=20.0))
    assert r.status == _abi.S3D_TOO_FEW_POINTS
    r = direct7.gicp_align(src, tgt, None, ndt_omp(point_cloud_density=0.2, resolution=0.01))  # "Voxel grid is not searchable"
    assert r.status == _abi.S3D_NOT_CONVERGED and r.outer_iterations == 0 and np.array_equal(r.pose(), np.eye(4))
