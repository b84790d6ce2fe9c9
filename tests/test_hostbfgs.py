"""slam3d_b200/csrc/gicp_bfgs.h (PCL <= 1.13's BFGS inner optimiser as the resumable state machine the GPU runs) compiled for the
host and checked decision for decision against the oracle's estimateRigidTransformationBFGS (oracle/bfgs_oracle.inc) on the
problems of test_oracle_bfgs.py: bit-identical float transform, same inner iteration count, same status.  The harness is built
in a temporary directory, never in the tree."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_oracle_bfgs import _problem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# s3d::BfgsBranch
BRANCHES = ["bracket_rho", "bracket_slope", "bracket_wolfe", "section_wolfe", "roundoff", "cubic", "quadratic", "max_inner", "gradient",
            "degenerate", "line_search_cap"]
# every branch the line search can take on a GICP problem; the last two need a zero gradient / 100 line-search iterations
REQUIRED = BRANCHES[:9]

SEED_OFFSETS = {1: None, 2: None, 3: None, 7: (0.4, 0.3, -0.2, 0.05, 0.04, -0.06)}
CAPS = (1, 2, 3, 5, 20)


@pytest.fixture(scope="module")
def hb():
    tmp = tempfile.mkdtemp(prefix="s3d_hostbfgs_")
    try:
        out = os.path.join(tmp, "hostbfgs.so")
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                               "-shared", "-o", out, os.path.join(ROOT, "tests", "hostbfgs.cpp")])
        lib = C.CDLL(out)  # stays mapped after the directory is removed
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    lib.hb_bfgs.restype = C.c_int
    return lib


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _sym_problem(seed):
    kw = {} if SEED_OFFSETS[seed] is None else {"offset": SEED_OFFSETS[seed]}
    a, b, M, _ = _problem(seed, **kw)
    M = 0.5 * (M + M.transpose(0, 2, 1))  # exactly symmetric, so that the 6-entry form carries the same matrix
    return a, b, M


def _m6(M):
    return np.ascontiguousarray(np.stack([M[:, 0, 0], M[:, 0, 1], M[:, 0, 2], M[:, 1, 1], M[:, 1, 2], M[:, 2, 2]], 1))


def _run_both(oracle_mod, hb, a, b, M, T0, cap):
    """(oracle T, inner, status), (machine T, inner, status, evaluations) from the float start T0 (4x4, row-major view)"""
    Mc = np.ascontiguousarray(M.transpose(0, 2, 1))
    To, io, so = oracle_mod.test_bfgs(a, b, Mc, T0, max_inner=cap)
    Tm = np.ascontiguousarray(np.asarray(T0, np.float32).T)  # column-major
    inner, evals = C.c_int(0), C.c_int(0)
    sm = hb.hb_bfgs(ptr(a), ptr(b), ptr(_m6(M)), a.shape[0], ptr(Tm), cap, C.byref(inner), C.byref(evals))
    return (To, io, so), (Tm.T.copy(), inner.value, sm, evals.value)


def _hits(hb, reset=True):
    out = (C.c_longlong * 16)()
    n = hb.hb_hits(out, int(reset))
    return {BRANCHES[i]: out[i] for i in range(n)}


@pytest.mark.parametrize("seed", sorted(SEED_OFFSETS))
@pytest.mark.parametrize("cap", CAPS)
def test_bfgs_machine_reproduces_oracle(oracle_mod, hb, seed, cap):
    """From the identity and again from the result (the start at the minimum: the float-rounding regime), the machine ends on the
    oracle's float transform bit for bit, after the same number of BFGS iterations and with the same status."""
    a, b, M = _sym_problem(seed)
    T0 = np.eye(4, dtype=np.float32)
    for _ in range(2):
        (To, io, so), (Tm, im, sm, ev) = _run_both(oracle_mod, hb, a, b, M, T0, cap)
        assert (so, sm) == (0, 0)
        assert io == im and 1 <= im <= cap
        assert np.array_equal(To, Tm), np.abs(To.astype(np.float64) - Tm).max()
        assert ev >= im + 1  # the start plus at least one trial per iteration
        T0 = To


def test_bfgs_machine_refusals(oracle_mod, hb):
    """Fewer than 4 correspondences: PCL throws before the solve (nothing counted).  maximum_optimizer_iterations = 0: the first
    iteration runs and estimateRigidTransformationBFGS rejects the state it reaches (SolverDidntConvergeException)."""
    a, b, M = _sym_problem(7)
    (To, io, so), (Tm, im, sm, _) = _run_both(oracle_mod, hb, a[:3], b[:3], M[:3], np.eye(4, dtype=np.float32), 20)
    assert so == sm == 2 and io == im == 0
    assert np.array_equal(To, Tm)
    (To, io, so), (Tm, im, sm, _) = _run_both(oracle_mod, hb, a, b, M, np.eye(4, dtype=np.float32), 0)
    assert so == sm == 2 and io == im == 1
    assert np.array_equal(To, Tm) and np.array_equal(Tm, np.eye(4, dtype=np.float32))


def test_bfgs_cases_reach_every_branch(oracle_mod, hb):
    """The cases of test_bfgs_machine_reproduces_oracle, between them, take every decision of the line search and of the outer
    loop: both bracketing exits, Wolfe success in bracketing and in sectioning, the roundoff exit, both interpolations, the
    gradient test and the iteration cap."""
    _hits(hb, reset=True)
    for seed in sorted(SEED_OFFSETS):
        a, b, M = _sym_problem(seed)
        for cap in CAPS:
            T0 = np.eye(4, dtype=np.float32)
            for _ in range(2):
                (To, io, so), (Tm, im, sm, _) = _run_both(oracle_mod, hb, a, b, M, T0, cap)
                assert np.array_equal(To, Tm) and io == im and so == sm == 0
                T0 = To
    hits = _hits(hb)
    missing = [k for k in REQUIRED if hits[k] == 0]
    assert not missing, hits
