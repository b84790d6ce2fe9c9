"""NDT branch timing on the bench workload (synthetic 131k-point pairs, 0.1 m voxel, slam3d NDT defaults): batch of pairs
through s3d_gicp_align_batch with host scans (e2e) and per-stage device times; oracle on one host thread beside it.

--prepared adds the device cache for NDT (s3d_prepare_clouds_ndt + s3d_gicp_align_prepared_batch) on the same workload, in the
same process: prepare time per cloud, prepared and raw batch rates measured alternately, one pair's latency both ways, stage
times of both, the card's name and power limit, and a check that the prepared results equal the raw ones field for field.

--omp-search [kdtree] [direct7] times NDT_OMP with the listed neighbour searches (both when none is named) on the same workload,
one context per search, calls alternated in one process: registrations/s end to end, then the derivative-evaluation stage
(ndt_eval_kernel, stage gicp_iter) and the others of one profiled call each, with the card's name and power limit.  DIRECT7's
GPU results on the first --check-pairs distinct pairs are checked against the oracle's DIRECT7 restatement (same status,
converged flag and counts, pose within 1e-4 m / 1e-4 rad, fitness within 1e-4)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import slam3d_b200
from slam3d_b200 import _abi, synth
from slam3d_b200._abi import RegistrationParameters

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=32)
ap.add_argument("--distinct", type=int, default=4)
ap.add_argument("--steps", type=int, default=3)
ap.add_argument("--oracle", action="store_true")
ap.add_argument("--prepared", action="store_true", help="also time NDT on prepared clouds, alternating with the raw path")
ap.add_argument("--latency-reps", type=int, default=10, help="--prepared: single-pair calls per path")
ap.add_argument("--omp-search", nargs="*", choices=["kdtree", "direct7"], help="time NDT_OMP with these neighbour searches, alternated")
ap.add_argument("--check-pairs", type=int, default=2, help="--omp-search: distinct pairs checked against the oracle (DIRECT7)")
ap.add_argument("--out", help="also write the JSON to this file (--prepared: default profiles/r03_ndt_prepared.json)")
a = ap.parse_args()
if a.omp_search is not None and a.prepared:
    sys.exit("--omp-search and --prepared are separate measurements")
if a.prepared and not a.out:
    a.out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r03_ndt_prepared.json")
P = RegistrationParameters.defaults(point_cloud_density=0.1, registration_algorithm=_abi.ALG_NDT)
scenes = [synth.scan_pair(seed=100 + i) for i in range(a.distinct)]
srcs = [slam3d_b200.as_xyzw(scenes[i % a.distinct][0]) for i in range(a.pairs)]
tgts = [slam3d_b200.as_xyzw(scenes[i % a.distinct][1]) for i in range(a.pairs)]
ctx = slam3d_b200.Context()


def fields(r):
    return (r.status, r.converged, r.outer_iterations, r.inner_iterations, r.n_correspondences, r.n_source, r.n_target,
            r.fitness, tuple(r.T))


def pose_delta(A, B):
    """(translation [m], rotation angle [rad]) of inv(A) B."""
    D = np.linalg.inv(np.asarray(A, np.float64)) @ np.asarray(B, np.float64)
    return float(np.linalg.norm(D[:3, 3])), float(np.arccos(np.clip((np.trace(D[:3, :3]) - 1.0) / 2.0, -1.0, 1.0)))


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        out["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


res = ctx.gicp_align_batch(srcs, tgts, None, P)  # warm-up
omp_ok = True
if a.omp_search is not None:
    methods = list(dict.fromkeys(a.omp_search)) or ["kdtree", "direct7"]
    Pomp = RegistrationParameters.defaults(point_cloud_density=P.point_cloud_density, registration_algorithm=_abi.ALG_NDT_OMP)
    ctxs = {}
    for m in methods:
        ctxs[m] = slam3d_b200.Context()
        ctxs[m].set_ndt_omp_search(m)
        ctxs[m].gicp_align_batch(srcs, tgts, None, Pomp)  # warm-up
    t_step = {m: [] for m in methods}
    last = {}
    for _ in range(a.steps):  # alternate the searches, so that both see the same host and GPU conditions
        for m in methods:
            t0 = time.perf_counter()
            last[m] = ctxs[m].gicp_align_batch(srcs, tgts, None, Pomp)
            t_step[m].append(time.perf_counter() - t0)
    stages = {}
    for m in methods:  # profiled in calls of their own: the stage events are not part of the timed calls
        ctxs[m].set_profiling(True)
        ctxs[m].stage_times(reset=True)
        ctxs[m].gicp_align_batch(srcs, tgts, None, Pomp)
        stages[m] = {k: round(v["ms"], 3) for k, v in ctxs[m].stage_times(reset=True).items()}  # summed over the streams
        ctxs[m].set_profiling(False)
    out = {"workload": f"{a.pairs} pairs of synthetic {srcs[0].shape[0]}-point scans ({a.distinct} distinct), density {Pomp.point_cloud_density} m, "
                       f"NDT_OMP resolution {Pomp.resolution} m, step {Pomp.step_size}, outlier ratio {Pomp.outlier_ratio}",
           "card": card(), "steps": a.steps}
    for m in methods:
        med = float(np.median(t_step[m]))
        out[m] = {"ms_per_step": [t * 1e3 for t in t_step[m]], "registrations_per_s_e2e": a.pairs / med,
                  "derivative_eval_ms_one_call": stages[m]["gicp_iter"], "stage_ms_one_call": stages[m],
                  "ok": sum(r.status == 0 for r in last[m]),
                  "outer_iterations": [r.outer_iterations for r in last[m][: a.distinct]],
                  "line_iterations": [r.inner_iterations for r in last[m][: a.distinct]],
                  "pairs_last_evaluation": [r.n_correspondences for r in last[m][: a.distinct]]}
    if "direct7" in methods:
        from oracle import ndt_omp
        ndt_omp.set_ndt_omp_search("direct7")
        checked = []
        for i in range(min(a.check_pairs, a.distinct)):
            got, want = last["direct7"][i], ndt_omp.gicp_align(srcs[i], tgts[i], None, Pomp)
            dt, dr = pose_delta(want.pose(), got.pose())
            ok = ((got.status, got.converged, got.outer_iterations, got.inner_iterations, got.n_correspondences) ==
                  (want.status, want.converged, want.outer_iterations, want.inner_iterations, want.n_correspondences)
                  and dt < 1e-4 and dr < 1e-4 and abs(got.fitness - want.fitness) <= 1e-4 * abs(want.fitness))
            checked.append({"pair": i, "ok": bool(ok), "dt_m": dt, "dr_rad": dr})
            omp_ok = omp_ok and ok
        out["direct7_vs_oracle"] = checked
    if len(methods) == 2:
        out["direct7_over_kdtree_rate"] = out["direct7"]["registrations_per_s_e2e"] / out["kdtree"]["registrations_per_s_e2e"]
    for c in ctxs.values():
        c.close()
elif not a.prepared:
    ctx.set_profiling(True)
    ctx.stage_times(reset=True)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        res = ctx.gicp_align_batch(srcs, tgts, None, P)
    dt = (time.perf_counter() - t0) / a.steps
    out = {"pairs": a.pairs, "ms_per_step": dt * 1e3, "ndt_registrations_per_s_e2e": a.pairs / dt, "ok": sum(r.status == 0 for r in res),
           "outer_iterations": [r.outer_iterations for r in res[: a.distinct]], "line_iterations": [r.inner_iterations for r in res[: a.distinct]]}
    out["stage_ms_per_step"] = {k: round(v["ms"] / a.steps, 3) for k, v in ctx.stage_times(reset=True).items()}  # stage ids of s3d_b200.h (NDT: knn_cov = voxel Gaussians)
else:
    # every pair gets its own two handles, as every pair of the raw batch uploads and filters its own two scans
    clouds = srcs + tgts
    h = ctx.prepare_clouds_ndt(clouds, P.point_cloud_density, P.resolution)  # warm-up of the prepare pass
    for x in h:
        x.release()
    t0 = time.perf_counter()
    h = ctx.prepare_clouds_ndt(clouds, P.point_cloud_density, P.resolution)
    prep_ms = (time.perf_counter() - t0) * 1e3
    hs, ht = h[: a.pairs], h[a.pairs:]
    prep = ctx.gicp_align_prepared_batch(hs, ht, None, P)  # warm-up
    raw_t, prep_t = [], []
    for _ in range(a.steps):  # alternate the two paths, so that both see the same host and GPU conditions
        t0 = time.perf_counter()
        res = ctx.gicp_align_batch(srcs, tgts, None, P)
        raw_t.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        prep = ctx.gicp_align_prepared_batch(hs, ht, None, P)
        prep_t.append(time.perf_counter() - t0)
    equal = all(fields(x) == fields(y) for x, y in zip(res, prep))
    lat_raw, lat_prep = [], []
    for _ in range(a.latency_reps):
        t0 = time.perf_counter()
        r1 = ctx.gicp_align(srcs[0], tgts[0], None, P)
        lat_raw.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        r2 = ctx.gicp_align_prepared(hs[0], ht[0], None, P)
        lat_prep.append(time.perf_counter() - t0)
    equal = equal and fields(r1) == fields(r2)
    ctx.set_profiling(True)
    stages = {}
    for name, call in (("raw", lambda: ctx.gicp_align_batch(srcs, tgts, None, P)), ("prepared", lambda: ctx.gicp_align_prepared_batch(hs, ht, None, P)),
                       ("prepare", lambda: [x.release() for x in ctx.prepare_clouds_ndt(clouds, P.point_cloud_density, P.resolution)])):
        ctx.stage_times(reset=True)
        call()
        stages[name] = {k: round(v["ms"], 3) for k, v in ctx.stage_times(reset=True).items()}  # summed over the streams
    ctx.set_profiling(False)
    raw_med, prep_med = float(np.median(raw_t)), float(np.median(prep_t))
    out = {"workload": f"{a.pairs} pairs of synthetic {srcs[0].shape[0]}-point scans ({a.distinct} distinct), density {P.point_cloud_density} m, "
                       f"NDT resolution {P.resolution} m, step {P.step_size}, outlier ratio {P.outlier_ratio}",
           "card": card(), "steps": a.steps,
           "prepare_ms_per_cloud": prep_ms / len(clouds), "prepare_ms_total": prep_ms, "prepared_clouds": len(clouds),
           "raw_ms_per_step": [t * 1e3 for t in raw_t], "prepared_ms_per_step": [t * 1e3 for t in prep_t],
           "ndt_registrations_per_s_raw_e2e": a.pairs / raw_med, "ndt_registrations_per_s_prepared": a.pairs / prep_med,
           "prepared_over_raw_rate": raw_med / prep_med,
           "single_pair_ms_raw_median": float(np.median(lat_raw)) * 1e3, "single_pair_ms_prepared_median": float(np.median(lat_prep)) * 1e3,
           "stage_ms_one_call": stages, "ok": sum(r.status == 0 for r in prep), "prepared_equals_raw": bool(equal)}
    for x in h:
        x.release()
if a.oracle:
    import oracle
    t0 = time.perf_counter()
    r = oracle.gicp_align(srcs[0], tgts[0], None, P)
    out["oracle_ms_per_align_1thread"] = (time.perf_counter() - t0) * 1e3
    out["oracle_outer"] = r.outer_iterations
line = json.dumps(out)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(out, indent=1) + "\n")
if not omp_ok:
    sys.exit("DIRECT7 GPU results differ from the oracle")
if a.prepared and not out["prepared_equals_raw"]:
    sys.exit("prepared NDT results differ from the raw ones")
