"""GICP with PCL <= 1.13's BFGS inner optimiser on the GPU (Context.set_gicp_optimizer("bfgs"), s3d_set_gicp_optimizer) against the
CPU oracle in BFGS mode (oracle.set_gicp_optimizer("bfgs")), through every GICP entry point and both loop schedulers.

Gates as for the Newton path: same status, convergence flag, outer and inner iteration counts and correspondence count; pose
within 1e-4 m / 1e-4 rad, fitness relative error <= 1e-4.  The synthetic odometry and loop-closure cases and the iteration-cap
gates meet them with bit-identical poses (one synthetic run from a perturbed guess excepted, see below).

Cases on the reference's KITTI clouds cannot: BFGS interpolates every trial step length from f and its slope along the search
direction, so on these clouds the last bits of the double sums — which depend on the order in which a reduction adds the
correspondences — change the sequence of trials.  The CPU oracle itself, with only the order of its point loops reversed, ends
those six pairs 1.5e-4 ... 5.1e-3 m, up to 2.8e-4 rad and up to 2.1e-3 relative fitness away, after other iteration counts
(DESIGN.md 2).  Those cases are held to the same status and convergence flag and to that spread: 1e-2 m, 1e-3 rad, 5e-3 relative
fitness, correspondence counts within 1e-3.  The oracle's process-wide switch is set and restored around every use."""
import ctypes as C
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import pose_delta
from slam3d_b200 import _abi
from slam3d_b200._abi import RegistrationParameters

pytestmark = pytest.mark.gpu
TOL_T, TOL_R, TOL_FIT = 1e-4, 1e-4, 1e-4
ORDER_T, ORDER_R, ORDER_FIT, ORDER_CORR = 1e-2, 1e-3, 5e-3, 1e-3   # cases whose BFGS path depends on the summation order
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    import slam3d_b200
    c = slam3d_b200.Context()
    assert c.set_gicp_optimizer("bfgs") == "newton"
    yield c
    c.close()


@contextlib.contextmanager
def oracle_bfgs(oracle_mod):
    old = oracle_mod.set_gicp_optimizer("bfgs")
    try:
        yield
    finally:
        oracle_mod.set_gicp_optimizer(old)


def check(got, want, order_sensitive=False):
    assert got.status == want.status
    assert (got.n_source, got.n_target) == (want.n_source, want.n_target)
    if want.status == _abi.S3D_TOO_FEW_POINTS:
        return
    assert got.converged == want.converged
    dt, dr = pose_delta(want.pose(), got.pose())
    if order_sensitive:
        assert dt < ORDER_T and dr < ORDER_R, (dt, dr)
        assert abs(got.fitness - want.fitness) <= ORDER_FIT * max(abs(want.fitness), 1e-12)
        assert abs(int(got.n_correspondences) - int(want.n_correspondences)) <= ORDER_CORR * want.n_correspondences
        assert got.inner_iterations >= got.outer_iterations
        return
    assert (got.outer_iterations, got.inner_iterations, got.n_correspondences) == (want.outer_iterations, want.inner_iterations, want.n_correspondences)
    assert dt < TOL_T and dr < TOL_R, (dt, dr)
    assert abs(got.fitness - want.fitness) <= TOL_FIT * max(abs(want.fitness), 1e-12)


def same(a, b):
    assert (a.status, a.converged, a.outer_iterations, a.inner_iterations, a.n_correspondences, a.n_source, a.n_target) == \
           (b.status, b.converged, b.outer_iterations, b.inner_iterations, b.n_correspondences, b.n_source, b.n_target)
    assert np.array_equal(a.pose(), b.pose()) and a.fitness == b.fitness


@pytest.mark.parametrize("density", [0.1, 0.2])
def test_kitti_pairs_vs_oracle(ctx, oracle_mod, kitti, density):
    p = RegistrationParameters.defaults(point_cloud_density=density)
    with oracle_bfgs(oracle_mod):
        for a, b in ((0, 1), (1, 2), (2, 3)):
            got = ctx.gicp_align(kitti[a], kitti[b], None, p)
            want = oracle_mod.gicp_align(kitti[a], kitti[b], None, p)
            check(got, want, order_sensitive=True)
            assert got.status == _abi.S3D_OK and got.inner_iterations > got.outer_iterations


def test_synthetic_odometry_pairs_vs_oracle(ctx, oracle_mod):
    """From the identity and from a perturbed true pose.  One of the four runs (seed 20260117 from the perturbed pose) is
    order-sensitive like the KITTI pairs: held to the spread, the other three to the exact gates."""
    from slam3d_b200 import synth
    p = RegistrationParameters.defaults(point_cloud_density=0.1)
    with oracle_bfgs(oracle_mod):
        for seed in (100, 20260117):
            src, tgt, truth = synth.scan_pair(seed=seed)
            check(ctx.gicp_align(src, tgt, None, p), oracle_mod.gicp_align(src, tgt, None, p))
            guess = truth.copy(); guess[:3, 3] += [0.05, -0.03, 0.01]
            got = ctx.gicp_align(src, tgt, guess, p)
            check(got, oracle_mod.gicp_align(src, tgt, guess, p), order_sensitive=seed == 20260117)
            dt, dr = pose_delta(truth, got.pose())
            assert dt < 0.02 and dr < 3e-3


def test_loop_closure_coarse_fine_vs_oracle(ctx, oracle_mod):
    """s3d_gicp_align_loop_batch (createConstraint, loop = true): both the coarse and the fine align run BFGS."""
    from slam3d_b200 import synth
    pairs = [synth.scan_pair(seed=100 + i, loop=True) for i in range(2)]
    srcs = [s[::2] for s, _, _ in pairs]
    tgts = [t[::2] for _, t, _ in pairs]
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0, max_translation=5.0)
    fine = RegistrationParameters.defaults(point_cloud_density=0.2, max_translation=5.0)
    lc, lf = ctx.gicp_align_loop_batch(srcs, tgts, None, coarse, fine)
    with oracle_bfgs(oracle_mod):
        for i in range(2):
            oc = oracle_mod.gicp_align(srcs[i], tgts[i], None, coarse)
            check(lc[i], oc)
            if oc.status == _abi.S3D_OK:
                check(lf[i], oracle_mod.gicp_align(srcs[i], tgts[i], lc[i].pose(), fine))
    assert lc[0].status == _abi.S3D_OK


def test_gates_vs_oracle(ctx, oracle_mod, kitti):
    src, tgt = kitti[0][::4], kitti[1][::4]
    cases = [  # (parameters, order-sensitive: the KITTI scans again, see the module docstring)
        (dict(point_cloud_density=0.5), True),
        (dict(point_cloud_density=0.5, max_fitness_score=1e-6), True),              # fitness gate
        (dict(point_cloud_density=0.5, max_translation=0.1), True),                  # too far from the guess
        (dict(point_cloud_density=0.5, maximum_optimizer_iterations=1), False),
        (dict(point_cloud_density=0.5, maximum_iterations=1), False),
        (dict(point_cloud_density=0.5, maximum_iterations=3, max_correspondence_distance=1.0), True),
    ]
    with oracle_bfgs(oracle_mod):
        for kw, sensitive in cases:
            p = RegistrationParameters.defaults(**kw)
            check(ctx.gicp_align(src, tgt, None, p), oracle_mod.gicp_align(src, tgt, None, p), order_sensitive=sensitive)
        p = RegistrationParameters.defaults(point_cloud_density=20.0)                # fewer than 100 points
        got, want = ctx.gicp_align(src[:500], tgt[:500], None, p), oracle_mod.gicp_align(src[:500], tgt[:500], None, p)
        assert got.status == want.status == _abi.S3D_TOO_FEW_POINTS
    r = ctx.gicp_align(src, tgt, None, RegistrationParameters.defaults(point_cloud_density=0.5, max_fitness_score=1e-6))
    assert r.status == _abi.S3D_NOT_CONVERGED
    r = ctx.gicp_align(src, tgt, None, RegistrationParameters.defaults(point_cloud_density=0.5, max_translation=0.1))
    assert r.status == _abi.S3D_TOO_FAR_FROM_GUESS
    # GICP_OMP selects the same branch, so the same optimiser
    omp = ctx.gicp_align(src, tgt, None, RegistrationParameters.defaults(point_cloud_density=0.5, registration_algorithm=_abi.ALG_GICP_OMP))
    same(omp, ctx.gicp_align(src, tgt, None, RegistrationParameters.defaults(point_cloud_density=0.5)))


def test_batch_prepared_and_loop_modes_are_bit_identical(ctx, kitti, monkeypatch):
    """batch == single, prepared == raw, and the three loop schedulers (persistent kernel, graph replay, host-driven rounds) give
    the same bits: the BFGS line search runs in the shared control step, whatever launches it."""
    p = RegistrationParameters.defaults(point_cloud_density=0.2)
    srcs = [kitti[0], kitti[1], kitti[2], kitti[0][:50]]
    tgts = [kitti[1], kitti[2], kitti[3], kitti[1]]
    batch = ctx.gicp_align_batch(srcs, tgts, None, p)
    singles = [ctx.gicp_align(s, t, None, p) for s, t in zip(srcs, tgts)]
    for a, b in zip(batch, singles):
        same(a, b)
    assert batch[3].status == _abi.S3D_TOO_FEW_POINTS
    prepared = ctx.prepare_clouds(kitti, 0.2, 20)
    chain = ctx.gicp_align_prepared_batch(prepared[:-1], prepared[1:], None, p)
    for i in range(3):
        same(chain[i], singles[i])
        same(ctx.gicp_align_prepared(prepared[i], prepared[i + 1], None, p), singles[i])
    for h in prepared:
        h.release()
    for mode in ("1", "2", "3"):  # read per call
        monkeypatch.setenv("S3D_LOOP_MODE", mode)
        got = ctx.gicp_align_batch(srcs[:3], tgts[:3], None, p)
        one = ctx.gicp_align(srcs[0], tgts[0], None, p)
        monkeypatch.delenv("S3D_LOOP_MODE")
        for a, b in zip(got, singles):
            same(a, b)
        same(one, singles[0])


def test_results_do_not_depend_on_the_launch_grid():
    """A launch grid of 3 % of the raw-size bound and the full grid give the same bits in BFGS mode (batch path)."""
    code = (
        "import numpy as np, hashlib, slam3d_b200\n"
        "from slam3d_b200 import synth\n"
        "from slam3d_b200._abi import RegistrationParameters\n"
        "pairs = [synth.scan_pair(seed=30 + i) for i in range(3)]\n"
        "ctx = slam3d_b200.Context()\n"
        "ctx.set_gicp_optimizer('bfgs')\n"
        "p = RegistrationParameters.defaults(point_cloud_density=0.2)\n"
        "h = hashlib.sha256()\n"
        "for rep in range(2):\n"
        "    rs = ctx.gicp_align_batch([a for a, _, _ in pairs], [b for _, b, _ in pairs], None, p)\n"
        "    for r in rs:\n"
        "        h.update(np.asarray(r.T, np.float64).tobytes()); h.update(np.float64(r.fitness).tobytes())\n"
        "        h.update(bytes([r.status, r.outer_iterations % 256, r.inner_iterations % 256]))\n"
        "print('HASH', h.hexdigest())\n")
    got = {}
    for frac in ("1", "0.03"):
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, S3D_GRID_FRAC=frac), cwd=ROOT, timeout=600)
        lines = [l for l in out.stdout.splitlines() if l.startswith("HASH")]
        assert lines, out.stdout + out.stderr
        got[frac] = lines[0]
    assert got["1"] == got["0.03"]


def test_switching_back_and_refusals(kitti):
    """Back to "newton" gives exactly what a fresh context gives; an unknown optimiser is refused and changes nothing; NDT
    ignores the setting."""
    import slam3d_b200
    src, tgt = kitti[0][::2], kitti[1][::2]
    p = RegistrationParameters.defaults(point_cloud_density=0.3)
    fresh = slam3d_b200.Context()
    ref = fresh.gicp_align(src, tgt, None, p)
    ndt_p = RegistrationParameters.defaults(point_cloud_density=0.3, registration_algorithm=_abi.ALG_NDT, resolution=1.0)
    ndt_ref = fresh.gicp_align(src, tgt, None, ndt_p)
    fresh.close()
    c = slam3d_b200.Context()
    try:
        assert c.set_gicp_optimizer("bfgs") == "newton"
        bf = c.gicp_align(src, tgt, None, p)
        assert bf.status == _abi.S3D_OK and not np.array_equal(bf.pose(), ref.pose())
        same(c.gicp_align(src, tgt, None, ndt_p), ndt_ref)
        prev = C.c_int(-1)
        for bad in (2, -1, 7):
            assert slam3d_b200.lib().s3d_set_gicp_optimizer(c._h, bad, C.byref(prev)) == _abi.S3D_INVALID_ARGUMENT
            assert prev.value == -1
        with pytest.raises(ValueError):
            c.set_gicp_optimizer("lbfgs")
        same(c.gicp_align(src, tgt, None, p), bf)       # the refused calls changed nothing
        assert c.set_gicp_optimizer("newton") == "bfgs"
        same(c.gicp_align(src, tgt, None, p), ref)
        assert slam3d_b200.lib().s3d_set_gicp_optimizer(c._h, _abi.GICP_NEWTON, None) == _abi.S3D_OK
    finally:
        c.close()
