"""fillGroundPlane on the GPU (s3d_fit_plane_ransac / s3d_fill_ground_plane) against the CPU oracle on one host thread.

Workloads: a 131 072-point synthetic scan (synth.py), the 2 097 152-point accumulated map of 16 such scans (as in
test_gpu_map.py), and golden cloud 1 (a 124 668-point lidar scan on which the adaptive stop needs ~7 000 iterations).  For each:
  * GPU time of the plane fit (host clouds, inliers not requested) and of the whole fill (map resolution 0.1 m, radius 10 m):
    median and min over --reps calls after --warmup calls, host clock around the synchronous call;
  * PCL's iterations and the GPU's rounds: each round is one sampler and one counting launch, so
    rounds = (launches - 1 init - 3 inlier compaction) / 2;
  * the oracle's time for the same fit and fill, once (it is single-threaded);
  * equality: float coefficients, iterations, inlier count and indices, fill points bit for bit.
The GPU name and power limit are read in the same run.  S3D_RANSAC_BLOCK sets the round size (default 256).

    python scripts/bench_ransac.py [--reps 10] [--warmup 2] [--out bench_ransac.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

THRESHOLD, RES, RADIUS = 0.01, 0.1, 10.0


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        return {"gpu": "unknown", "power_limit": f"not read ({e.__class__.__name__})"}


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t))
    return {"median_ms": statistics.median(ts), "min_ms": min(ts)}


def workloads():
    from slam3d_b200 import synth
    from conftest import load_kitti
    scene = synth.Scene(3)
    yield "synthetic scan", synth.scan(scene, synth.make_pose([0.0, 0.0, 0.0], [0.0, 0.0, 0.0]), np.random.default_rng(3))
    yield "16-scan map", synth.map_cloud(n_scans=16)
    yield "golden cloud 1", load_kitti(1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import slam3d_b200
    from oracle import ransac as oracle
    oracle.lib()  # compiled on first use: keep that out of the timed oracle calls
    ctx = slam3d_b200.Context()
    report = {"info": gpu_info(), "block": os.environ.get("S3D_RANSAC_BLOCK", "256 (default)"), "threshold": THRESHOLD,
              "map_resolution": RES, "radius": RADIUS, "fill_points": slam3d_b200.ground_fill_size(RES, RADIUS), "workloads": []}
    all_equal = True
    for name, cloud in workloads():
        pts = oracle.as_xyzw(cloud)
        l0 = ctx.counters()["kernel_launches"]
        coeff, it, n_in, inl = ctx.fit_plane_ransac(pts, THRESHOLD, want_inliers=True)
        rounds = (ctx.counters()["kernel_launches"] - l0 - 1 - 3) // 2  # minus init and the three inlier-compaction launches
        fill = ctx.fill_ground_plane(pts, RADIUS, RES)
        t = time.perf_counter()
        ok, o_coeff, o_it, o_inl = oracle.fit_plane_ransac(pts, THRESHOLD)
        o_fit_ms = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        o_fill, _ = oracle.fill_ground_plane(pts, RADIUS, RES)
        o_fill_ms = 1e3 * (time.perf_counter() - t)
        equal = bool(ok and np.array_equal(coeff.view(np.uint32), o_coeff.view(np.uint32)) and it == o_it and n_in == len(o_inl)
                     and np.array_equal(inl, o_inl) and np.array_equal(fill.view(np.uint32), o_fill.view(np.uint32)))
        all_equal &= equal
        g_fit = timed(lambda: ctx.fit_plane_ransac(pts, THRESHOLD), a.reps, a.warmup)
        g_fill = timed(lambda: ctx.fill_ground_plane(pts, RADIUS, RES), a.reps, a.warmup)
        row = {"workload": name, "points": len(pts), "iterations": it, "rounds": rounds, "inliers": n_in, "gpu_fit": g_fit, "gpu_fill": g_fill,
               "oracle_fit_ms_1_thread": o_fit_ms, "oracle_fill_ms_1_thread": o_fill_ms,
               "speedup_fill_median": o_fill_ms / g_fill["median_ms"], "equal": equal}
        print(json.dumps(row), flush=True)
        report["workloads"].append(row)
    report["all_equal"] = all_equal
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)
    print(json.dumps({"info": report["info"], "all_equal": all_equal}))
    if not all_equal:
        sys.exit(1)


if __name__ == "__main__":
    main()
