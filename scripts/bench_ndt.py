"""NDT branch timing on the bench workload (synthetic 131k-point pairs, 0.1 m voxel, slam3d NDT defaults): batch of pairs
through s3d_gicp_align_batch with host scans (e2e) and per-stage device times; oracle on one host thread beside it.

--prepared adds the device cache for NDT (s3d_prepare_clouds_ndt + s3d_gicp_align_prepared_batch) on the same workload, in the
same process: prepare time per cloud, prepared and raw batch rates measured alternately, one pair's latency both ways, stage
times of both, the card's name and power limit, and a check that the prepared results equal the raw ones field for field."""
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
ap.add_argument("--out", help="also write the JSON to this file (--prepared: default profiles/r03_ndt_prepared.json)")
a = ap.parse_args()
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
if not a.prepared:
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
if a.prepared and not out["prepared_equals_raw"]:
    sys.exit("prepared NDT results differ from the raw ones")
