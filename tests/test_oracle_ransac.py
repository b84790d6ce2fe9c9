"""The RANSAC plane fit and ring fill of fillGroundPlane in the CPU oracle (oracle/ransac_oracle.cpp), pinned against an
independent numpy restatement of the definitions in that file's header, numpy's MT19937 and a known plane."""
import math
import sys

import numpy as np
import pytest

THRESHOLD = 0.01


@pytest.fixture(scope="module")
def ransac_oracle():
    from oracle import ransac
    ransac.lib()
    return ransac


def ground_cloud(seed, n=3000, ground=0.6, nan_frac=0.0):
    """A tilted ground plane (3 mm noise) under uniform clutter; optionally some NaN points."""
    rng = np.random.default_rng(seed)
    m = int(n * ground)
    xy = rng.uniform(-15, 15, (m, 2))
    z = 0.02 * xy[:, 0] - 0.01 * xy[:, 1] - 1.7 + rng.normal(0, 0.003, m)
    pts = np.concatenate([np.column_stack([xy, z]), rng.uniform([-15, -15, -1.7], [15, 15, 3], (n - m, 3))])
    pts = pts[rng.permutation(n)].astype(np.float32)
    if nan_frac:
        pts[rng.choice(n, int(n * nan_frac), replace=False)] = np.nan
    return pts


def degenerate_clouds():
    t = np.arange(40, dtype=np.float32)
    return {
        "collinear": np.column_stack([t, 2 * t, 3 * t]).astype(np.float32),   # every ratio test rejects: no sample
        "identical": np.tile(np.float32([1.5, -2.0, 0.25]), (30, 1)),       # 0/0 ratios pass: zero normal, every point an inlier
        "three": np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0.1]]),
    }


class _Raw:
    """boost::mt19937(12345) outputs from numpy's MT19937 with the reference generator's seeding."""

    def __init__(self, seed):
        self.bg = np.random.MT19937()
        self.bg._legacy_seeding(seed)
        self.buf, self.pos = np.empty(0, np.uint64), 0

    def __call__(self):
        if self.pos == len(self.buf):
            self.buf, self.pos = self.bg.random_raw(4096), 0
        self.pos += 1
        return int(self.buf[self.pos - 1])


def numpy_ransac(cloud, threshold, max_iterations=10000, probability=0.99):
    """Independent restatement: (ok, coefficients, iterations, inliers)."""
    P = np.asarray(cloud, np.float32)[:, :3]
    n = len(P)
    f32 = np.float32
    rnd = _Raw(12345)
    shuffled = list(range(n))
    k, skipped, best, it, model = sys.float_info.max, 0, 0, 0, None
    log_p, one_over = math.log(1.0 - probability), 1.0 / n
    eps = sys.float_info.epsilon

    def good(s):
        p0, p1, p2 = P[s[0]], P[s[1]], P[s[2]]
        with np.errstate(all="ignore"):
            d = (p1 - p0) / (p2 - p0)
        return not (d[0] == d[1] and d[2] == d[1])

    def distances(c):
        with np.errstate(all="ignore"):
            return np.abs(((c[0] * P[:, 0] + c[1] * P[:, 1]) + c[2] * P[:, 2]) + c[3]).astype(np.float64)

    while it < k and skipped < 10 * max_iterations:
        sel = None
        if n >= 3:
            for _ in range(1000):
                for i in range(3):
                    j = i + (rnd() >> 1) % (n - i)
                    shuffled[i], shuffled[j] = shuffled[j], shuffled[i]
                if good(shuffled[:3]):
                    sel = shuffled[:3]
                    break
        if sel is None:
            break
        p0, p1, p2 = P[sel[0]], P[sel[1]], P[sel[2]]
        with np.errstate(all="ignore"):
            ax, ay, az = p1 - p0
            bx, by, bz = p2 - p0
            a, b, c = ay * bz - az * by, az * bx - ax * bz, ax * by - ay * bx
            n2 = ((a * a + b * b) + c * c) + f32(0) * f32(0)
            if n2 > 0:
                s = np.sqrt(n2)
                a, b, c = a / s, b / s, c / s
            d = -(((a * p0[0] + b * p0[1]) + c * p0[2]) + f32(0) * f32(1))
        coeff = np.array([a, b, c, d], np.float32)
        count = int(np.count_nonzero(distances(coeff) < threshold))
        if count > best:
            best, model = count, coeff
            w = count * one_over
            p = min(1.0 - eps, max(eps, 1.0 - math.pow(w, 3.0)))
            k = log_p / math.log(p)
        it += 1
        if it > max_iterations:
            break
    if model is None:
        return False, np.zeros(4, np.float32), it, np.zeros(0, np.uint32)
    return True, model, it, np.flatnonzero(distances(model) < threshold).astype(np.uint32)


def test_mt19937_check_value(ransac_oracle):
    """C++ standard [rand.predef]: the 10000th output of a default-constructed mt19937 is 4123659995."""
    mt, _ = ransac_oracle.rng_stream(5489, 10000)
    assert int(mt[-1]) == 4123659995


def test_rnd_is_mt_shifted(ransac_oracle):
    mt, rnd = ransac_oracle.rng_stream(12345, 5000)
    raw = _Raw(12345)
    expect = np.array([raw() for _ in range(5000)], np.uint64)
    assert np.array_equal(mt.astype(np.uint64), expect)
    assert np.array_equal(rnd.astype(np.uint64), expect >> 1)


CASES = {
    "ground": (ground_cloud(1, 600), 10000),
    "ground_nan": (ground_cloud(2, 600, nan_frac=0.05), 10000),
    "clutter": (ground_cloud(3, 300, ground=0.0), 10000),
    "max_it_1": (ground_cloud(4, 400), 1),
    "max_it_5": (ground_cloud(5, 400, ground=0.1), 5),
    **{k: (v, 10000) for k, v in degenerate_clouds().items()},
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_numpy_restatement(ransac_oracle, name):
    cloud, max_it = CASES[name]
    ok, coeff, it, inl = ransac_oracle.fit_plane_ransac(cloud, THRESHOLD, max_it)
    ok2, coeff2, it2, inl2 = numpy_ransac(cloud, THRESHOLD, max_it)
    assert ok == ok2 and it == it2
    if ok:
        assert np.array_equal(coeff.view(np.uint32), coeff2.view(np.uint32))
        assert np.array_equal(inl, inl2)
    if name == "collinear":
        assert not ok and it == 0
    if name == "identical":
        assert ok and len(inl) == len(cloud)


def test_oracle_recovers_plane_under_clutter(ransac_oracle):
    cloud = ground_cloud(7, 20000, ground=0.4)
    ok, coeff, it, inl = ransac_oracle.fit_plane_ransac(cloud, THRESHOLD)
    assert ok and 0 < it <= 10001
    truth = np.array([0.02, -0.01, -1.0]); d_truth = -1.7
    scale = np.linalg.norm(truth)
    n_true, d_true = truth / scale, d_truth / scale
    sign = np.sign(np.dot(coeff[:3], n_true))
    assert abs(np.dot(coeff[:3], n_true)) > 0.9999
    assert abs(sign * coeff[3] - d_true) < 0.01
    on_plane = np.abs(cloud.astype(np.float64) @ n_true + d_true) < 0.005
    assert np.mean(np.isin(np.flatnonzero(on_plane), inl)) > 0.9


@pytest.fixture(scope="module")
def product():
    import __graft_entry__
    __graft_entry__.build()
    import slam3d_b200
    return slam3d_b200


@pytest.mark.parametrize("res,radius", [(0.1, 2.0), (0.1, 5.0), (0.25, 3.0), (0.3, 0.2), (0.05, 1.0), (0.07, 10.0)])
def test_fill_count_matches_library(ransac_oracle, product, res, radius):
    n = product.ground_fill_size(res, radius)
    assert n == ransac_oracle.ground_fill_size(res, radius)
    pts, coeff = ransac_oracle.fill_ground_plane(ground_cloud(8, 500), radius, res)
    assert len(pts) == n
    if n:
        assert np.all(pts[:, 3] == 1) and np.all(np.abs(pts[:, :3] @ coeff[:3].astype(np.float64) + coeff[3]) < 1e-4 * max(1.0, radius))


@pytest.mark.parametrize("res,radius", [(0.0, 1.0), (-0.1, 1.0), (0.1, 0.0), (float("nan"), 1.0), (0.1, float("inf")), (1e-6, 100.0)])
def test_fill_size_rejects_bad_arguments(product, res, radius):
    with pytest.raises(product.S3DError):
        product.ground_fill_size(res, radius)
