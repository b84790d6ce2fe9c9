#!/usr/bin/env python
"""Config 5 with patches (SURVEY 8d: mPatchBuildingRange = 2, 3 links per vertex, candidates batched): the same figure-eight
trajectory as scripts/run_c5.py, through the MiniHost three times per repetition, alternating in one process:

  host    linkLastToNeighbors(true) builds every patch with createCombinedMeasurement (to the host) and matches the host patches
          with createConstraints (s3d_gicp_align_loop_batch: uploads and preprocesses every pair slot, coarse and fine pass)
  device  setDevicePatches(true): createLoopConstraints builds the distinct patches on the device from the distinct scans,
          prepares each once per pass setting and runs s3d_gicp_align_loop_batch_prepared
  resident  device patches with the host mirror's resident-scan store on (setResidentScanBudget): every scan is uploaded once,
          on its first use, and every later call (odometry prepares, patch builds) reads its device copy

All runs must record the same edges bit for bit and the same warnings.  Reported per mode: scans/s over the whole trajectory
(odometry included), H2D / D2H bytes and kernel launches of the library, and the mean time of one vertex's loop-closure call
(linkLastToNeighbors of a vertex that matched at least one candidate).  A last profiled run of each mode gives the device-time
split by stage (s3d_get_stage_times).  Last, one buildMap over the whole trajectory (s3d_build_map, the sensor's default map
settings) is timed from host scans and from resident scans (s3d_upload_scans), alternating.

    python scripts/bench_patches.py --scans 600 --reps 2 --out profiles/r04_bench_resident.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MODES = {"host": 1, "device": 2, "resident": 2}  # s3dhost_run_trajectory2's `batched`
RESIDENT_BUDGET = 1 << 36  # holds every scan of the trajectory: nothing is evicted


def workload(n):
    """run_c5.py's trajectory: scans, odometry (noisy), from its range cache"""
    from slam3d_b200 import synth
    import slam3d_b200
    radius, step = 1.5, 0.7
    lap = int(round(4 * np.pi * radius / step))
    step = 4 * np.pi * radius / lap
    cache = os.path.join(ROOT, ".cache_c5", "ranges.npy")
    if not os.path.exists(cache):
        subprocess.check_call([sys.executable, os.path.join(ROOT, "scripts", "run_c5.py"), "--build-cache-only"])
    rng_cache = np.load(cache)
    lanes = [0.0, 0.25]
    lane_poses = [synth.figure_eight_poses(lap, radius, step, lateral=l) for l in lanes]
    rng = np.random.default_rng(7)
    truth, scans = [], []
    for i in range(n):
        lane = (i // lap) % len(lanes)
        truth.append(lane_poses[lane][i % lap])
        scans.append(slam3d_b200.as_xyzw(synth.scan_from_ranges(rng_cache[lane, i % lap], rng)))
    odoms = [np.eye(4)]
    for i in range(1, n):
        rel = np.linalg.inv(truth[i - 1]) @ truth[i]
        rel = rel @ synth.make_pose(rng.normal(0, 0.014, 3) * [1, 1, 0.2], np.deg2rad(rng.normal(0, 0.2, 3) * [0.2, 0.2, 1]))
        odoms.append(odoms[-1] @ rel)
    return scans, odoms


def time_build_map(scans, poses, reps):
    """one s3d_build_map over every scan of the trajectory (outlier radius 0.2, 3 neighbours, 0.1 m: the sensor's defaults), from
    host scans and from resident scans, alternating; both maps must be equal bit for bit"""
    import slam3d_b200
    ctx = slam3d_b200.Context()
    t0 = time.perf_counter()
    views = ctx.upload_scans(scans)
    upload_s = time.perf_counter() - t0
    times = {"host": [], "resident": []}
    maps = {}
    for rep in range(reps + 1):  # repetition 0 warms up
        for mode in (("host", "resident") if rep % 2 == 0 else ("resident", "host")):
            h0 = ctx.counters()["h2d_bytes"]
            t0 = time.perf_counter()
            m = ctx.build_map(views if mode == "resident" else scans, poses)
            dt = time.perf_counter() - t0
            maps[mode] = (m.shape[0], m.tobytes())
            print(json.dumps({"build_map": mode, "rep": rep, "seconds": dt, "h2d_bytes": ctx.counters()["h2d_bytes"] - h0}), flush=True)
            if rep > 0:
                times[mode].append(dt)
    assert maps["host"] == maps["resident"], "maps differ"
    for v in views:
        v.release()
    ctx.close()
    return {"scans": len(scans), "map_points": maps["host"][0], "upload_once_s": upload_s,
            **{f"{m}_s": float(np.median(t)) for m, t in times.items()}, "runs": times}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=600)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--patch-range", type=int, default=2)
    ap.add_argument("--max-links", type=int, default=3)
    ap.add_argument("--radius", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import slam3d_b200
    import test_gpu_host as th
    from slam3d_b200._abi import Counters, RegistrationParameters
    L = slam3d_b200.lib()
    host = th.load_host()
    host.s3dhost_run_trajectory2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
    host.s3dhost_context.restype = C.c_void_p
    host.s3dhost_link_stats.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int)]
    host.s3dhost_set_resident_budget.argtypes = [C.c_uint64]
    host.s3dhost_resident_stats.argtypes = [C.POINTER(C.c_uint64)] * 3
    hctx = C.c_void_p(host.s3dhost_context())
    n = args.scans
    scans, odoms = workload(n)
    sensor = host.s3dhost_sensor_create(b"velodyne")
    fine = RegistrationParameters.defaults(point_cloud_density=0.1)
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0)
    host.s3dhost_sensor_set_params(sensor, C.byref(fine), 0)
    host.s3dhost_sensor_set_params(sensor, C.byref(coarse), 1)
    ptrs = (C.c_void_p * n)(*[s.ctypes.data for s in scans])
    sizes = (C.c_uint64 * n)(*[s.shape[0] for s in scans])
    od = np.ascontiguousarray(np.stack([o.T for o in odoms]))

    def counters():
        c = Counters()
        L.s3d_get_counters(hctx, C.byref(c))
        return np.array([c.kernel_launches, c.h2d_bytes, c.d2h_bytes], np.int64)

    def uploads():
        u, h, b = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        host.s3dhost_resident_stats(C.byref(u), C.byref(h), C.byref(b))
        return u.value

    def run(mode):
        edges = np.zeros((4 * n, 3), np.int32); T = np.zeros((4 * n, 16)); nw = C.c_int(0)
        host.s3dhost_set_resident_budget(RESIDENT_BUDGET if mode == "resident" else 0)
        c0, u0 = counters(), uploads()
        t0 = time.perf_counter()
        ne = host.s3dhost_run_trajectory2(sensor, ptrs, sizes, n, od.ctypes.data, args.radius, args.max_links, 10, args.patch_range,
                                          MODES[mode], 4 * n, edges.ctypes.data, T.ctypes.data, None, C.byref(nw))
        dt = time.perf_counter() - t0
        c1, u1 = counters(), uploads()
        host.s3dhost_set_resident_budget(0)
        assert ne >= 0, host.s3dhost_last_message()
        ls, lc = C.c_double(0), C.c_int(0)
        host.s3dhost_link_stats(C.byref(ls), C.byref(lc))
        d = c1 - c0
        return {"seconds": dt, "scans_per_s": n / dt, "kernel_launches": int(d[0]), "h2d_bytes": int(d[1]), "d2h_bytes": int(d[2]),
                "loop_calls": lc.value, "loop_call_ms": 1e3 * ls.value / max(lc.value, 1), "scans_uploaded_to_store": u1 - u0}, \
               (edges[:ne].copy(), T[:ne].copy(), nw.value, host.s3dhost_last_message().decode())

    gpu = {}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
        gpu = {"nvidia_smi": q.stdout.strip()}
    except OSError:
        pass
    runs = {m: [] for m in MODES}
    ref = {}
    order = list(MODES)
    for rep in range(args.reps + 1):  # repetition 0 warms up every mode (module load, workspace growth, loop graphs)
        for mode in order[rep % 3:] + order[:rep % 3]:
            r, out = run(mode)
            ref.setdefault(mode, out)
            for other in ref.values():
                assert np.array_equal(out[0], other[0]) and np.array_equal(out[1], other[1]) and out[2:] == other[2:], "edges differ"
            if rep > 0:
                runs[mode].append(r)
            print(json.dumps({"rep": rep, "mode": mode, **r}), flush=True)
    # stage split of one more run of each mode (profiling on: device time per stage, from CUDA events)
    stages = {}
    names = ("voxel", "grid", "knn_cov/ndt_grid", "loop", "loop_setup", "ndt_fitness")
    for mode in MODES:
        L.s3d_set_profiling(hctx, 1)
        ms, nl = (C.c_double * 6)(), (C.c_uint64 * 6)()
        L.s3d_get_stage_times(hctx, ms, nl, 1)
        r, _ = run(mode)
        L.s3d_get_stage_times(hctx, ms, nl, 1)
        L.s3d_set_profiling(hctx, 0)
        stages[mode] = {"wall_s": r["seconds"], **{k: {"ms": ms[i], "launches": int(nl[i])} for i, k in enumerate(names)}}
    build_map = time_build_map(scans, odoms, args.reps)
    e = ref["host"][0]
    summary = {
        "workload": f"config 5: {n}-scan figure-eight, patch range {args.patch_range}, {args.max_links} links per vertex, batched",
        "gpu": gpu, "edges": int(len(e)), "loop_edges": int(e[:, 2].sum()), "warnings": ref["host"][2], "edges_equal": True,
        "scan_bytes": int(sum(16 * s.shape[0] for s in scans)),
        **{m: {k: float(np.median([r[k] for r in runs[m]])) for k in runs[m][0]} for m in MODES},
        "runs": runs, "stages_profiled": stages, "build_map": build_map,
    }
    print(json.dumps(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    host.s3dhost_sensor_destroy(sensor)


if __name__ == "__main__":
    main()
