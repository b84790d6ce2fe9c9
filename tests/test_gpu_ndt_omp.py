"""NDT_OMP with pclomp's DIRECT7 neighbour search on the GPU (ndt_eval_kernel<true>; s3d_set_ndt_omp_search) against the
CPU oracle's DIRECT7 restatement (oracle/ndt_omp_oracle.cpp through oracle/ndt_omp.py).

Gate as in test_gpu_ndt.py: same status, converged flag, outer and line-search iterations and (point, voxel) pairs, pose
within 1e-4 m / 1e-4 rad, fitness within 1e-4 relative.  The device runs the ndt_math.h code that test_hostdirect7.py holds
bit for bit to the oracle on the host; only the order of the double sums differs."""
import ctypes as C

import numpy as np
import pytest

from conftest import pose_delta
from slam3d_b200 import _abi, synth
from slam3d_b200._abi import RegistrationParameters

pytestmark = pytest.mark.gpu
TOL_T, TOL_R, TOL_FIT = 1e-4, 1e-4, 1e-4


@pytest.fixture(scope="module")
def ctx():
    import slam3d_b200
    c = slam3d_b200.Context()
    assert c.set_ndt_omp_search("direct7") == "kdtree"
    yield c
    c.close()


@pytest.fixture
def direct7(oracle_mod):
    from oracle import ndt_omp
    old = ndt_omp.set_ndt_omp_search("direct7")
    yield ndt_omp
    ndt_omp.set_ndt_omp_search(old)


def omp(**kw):
    kw.setdefault("point_cloud_density", 0.2)
    kw.setdefault("registration_algorithm", _abi.ALG_NDT_OMP)
    return RegistrationParameters.defaults(**kw)


def check(got, want):
    assert got.status == want.status, (got.status, want.status)
    assert (got.n_source, got.n_target) == (want.n_source, want.n_target)
    if want.status == _abi.S3D_TOO_FEW_POINTS:
        return
    dt, dr = pose_delta(want.pose(), got.pose())
    assert dt < TOL_T and dr < TOL_R, (dt, dr)
    assert abs(got.fitness - want.fitness) <= TOL_FIT * max(abs(want.fitness), 1e-12)
    assert got.converged == want.converged
    assert (got.outer_iterations, got.inner_iterations, got.n_correspondences) == (want.outer_iterations, want.inner_iterations, want.n_correspondences)


def same(a, b):
    assert (a.status, a.converged, a.outer_iterations, a.inner_iterations, a.n_correspondences, a.n_source, a.n_target) == (
        b.status, b.converged, b.outer_iterations, b.inner_iterations, b.n_correspondences, b.n_source, b.n_target)
    assert np.array_equal(a.pose(), b.pose()) and a.fitness == b.fitness


@pytest.mark.parametrize("density", [0.1, 0.2])
def test_kitti_pairs_vs_oracle(ctx, direct7, kitti, density):
    p = omp(point_cloud_density=density)
    for i in range(3):
        want = direct7.gicp_align(kitti[i], kitti[i + 1], None, p)
        assert want.status != _abi.S3D_UNKNOWN_ALGORITHM
        check(ctx.gicp_align(kitti[i], kitti[i + 1], None, p), want)


@pytest.mark.parametrize("res", [0.5, 0.7, 1.0, 2.0])
def test_synthetic_pairs_vs_oracle(ctx, direct7, res):
    for seed, loop in ((11, False), (5, True)):
        src, tgt, truth = synth.scan_pair(seed=seed, loop=loop)
        noisy = synth.make_pose([0.05, -0.03, 0.01], [0.002, -0.003, 0.004]) @ truth
        kw = dict(point_cloud_density=0.2, resolution=res)
        if loop:
            kw.update(step_size=0.2, max_translation=5.0)
        p = omp(**kw)
        for guess in (None, noisy, truth):
            check(ctx.gicp_align(src, tgt, guess, p), direct7.gicp_align(src, tgt, guess, p))


def test_gates_match_oracle(ctx, direct7, kitti):
    src, tgt = kitti[0][::2], kitti[1][::2]
    for kw in (dict(max_fitness_score=1e-6), dict(max_translation=0.05), dict(maximum_iterations=1), dict(point_cloud_density=0.0),
               dict(resolution=0.01), dict(point_cloud_density=2.0, resolution=0.5), dict(point_cloud_density=20.0)):
        p = omp(**kw)
        check(ctx.gicp_align(src, tgt, None, p), direct7.gicp_align(src, tgt, None, p))


def test_batch_single_and_prepared_are_bit_identical(ctx, kitti):
    p = omp(point_cloud_density=0.3, resolution=1.0)
    srcs = [kitti[0], kitti[1], kitti[2], kitti[0][::3], kitti[2][:90]]
    tgts = [kitti[1], kitti[2], kitti[3], kitti[1][::3], kitti[3][:90]]
    batch = ctx.gicp_align_batch(srcs, tgts, None, p)
    singles = [ctx.gicp_align(s, t, None, p) for s, t in zip(srcs, tgts)]
    for a, b in zip(batch, singles):
        same(a, b)
    assert batch[4].status == _abi.S3D_TOO_FEW_POINTS
    h = ctx.prepare_clouds_ndt(kitti, 0.3, 1.0)
    chain = ctx.gicp_align_prepared_batch(h[:-1], h[1:], None, p)
    for i in range(3):
        same(chain[i], singles[i])
        same(ctx.gicp_align_prepared(h[i], h[i + 1], None, p), singles[i])
    for x in h:
        x.release()


def test_loop_batch_equals_two_batch_calls(ctx, kitti):
    srcs, tgts = [kitti[0], kitti[1], kitti[2]], [kitti[1], kitti[2], kitti[3]]
    coarse = omp(point_cloud_density=0.5, resolution=2.0, step_size=0.2)
    for fine in (omp(point_cloud_density=0.2, registration_algorithm=_abi.ALG_NDT), RegistrationParameters.defaults(point_cloud_density=0.2),
                 omp(point_cloud_density=0.2)):
        rc, rf = ctx.gicp_align_loop_batch(srcs, tgts, None, coarse, fine)
        want_c = ctx.gicp_align_batch(srcs, tgts, None, coarse)
        guesses = [r.pose() for r in want_c]
        want_f = ctx.gicp_align_batch(srcs, tgts, guesses, fine)
        for i in range(3):
            same(rc[i], want_c[i])
            same(rf[i], want_c[i] if want_c[i].status != _abi.S3D_OK else want_f[i])


def test_other_algorithms_ignore_the_setting(kitti):
    """GICP, GICP_OMP and NDT give the same bits with DIRECT7 selected and without; kdtree NDT_OMP equals NDT bit for bit."""
    import slam3d_b200
    src, tgt = kitti[0], kitti[1]
    cases = [RegistrationParameters.defaults(point_cloud_density=0.3),
             RegistrationParameters.defaults(point_cloud_density=0.3, registration_algorithm=_abi.ALG_GICP_OMP),
             omp(point_cloud_density=0.3, registration_algorithm=_abi.ALG_NDT),
             omp(point_cloud_density=0.3, resolution=0.7, registration_algorithm=_abi.ALG_NDT)]
    off, on = slam3d_b200.Context(), slam3d_b200.Context()
    try:
        on.set_ndt_omp_search("direct7")
        for p in cases:
            same(on.gicp_align(src, tgt, None, p), off.gicp_align(src, tgt, None, p))
            same(on.gicp_align_batch([src, tgt], [tgt, src], None, p)[1], off.gicp_align_batch([src, tgt], [tgt, src], None, p)[1])
        for res in (0.7, 1.0):
            ndt = off.gicp_align(src, tgt, None, omp(point_cloud_density=0.3, resolution=res, registration_algorithm=_abi.ALG_NDT))
            same(off.gicp_align(src, tgt, None, omp(point_cloud_density=0.3, resolution=res)), ndt)
            d7 = on.gicp_align(src, tgt, None, omp(point_cloud_density=0.3, resolution=res))
            assert d7.n_correspondences != ndt.n_correspondences  # the two contexts really run different searches
    finally:
        off.close()
        on.close()


def test_setter_and_wrapper():
    import slam3d_b200
    a, b = slam3d_b200.Context(), slam3d_b200.Context()
    try:
        L = slam3d_b200.lib()
        prev = C.c_int(-1)
        assert L.s3d_set_ndt_omp_search(a._h, _abi.NDT_OMP_DIRECT7, C.byref(prev)) == _abi.S3D_OK and prev.value == _abi.NDT_OMP_KDTREE
        for bad in (2, -1, 7):
            prev = C.c_int(-1)
            assert L.s3d_set_ndt_omp_search(a._h, bad, C.byref(prev)) == _abi.S3D_INVALID_ARGUMENT
            assert prev.value == -1 and "S3D_NDT_OMP_KDTREE" in slam3d_b200.last_error()
        assert L.s3d_set_ndt_omp_search(None, _abi.NDT_OMP_KDTREE, None) == _abi.S3D_INVALID_ARGUMENT
        assert L.s3d_set_ndt_omp_search(a._h, _abi.NDT_OMP_DIRECT7, None) == _abi.S3D_OK  # previous may be NULL
        # the refused calls changed nothing; the second context kept its own default
        assert a.set_ndt_omp_search("direct7") == "direct7"
        assert b.set_ndt_omp_search("kdtree") == "kdtree"
        for bad in ("DIRECT7", "direct26", 1, None):
            with pytest.raises(ValueError):
                a.set_ndt_omp_search(bad)
        assert a.set_ndt_omp_search("kdtree") == "direct7"
        assert a.set_ndt_omp_search("kdtree") == "kdtree"
    finally:
        a.close()
        b.close()
