#!/usr/bin/env python
"""bench.py — GICP registrations/s on 131 072-point synthetic LiDAR scan pairs (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            our arm  (libs3d_b200.so, hand-written sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  reference arm (the CPU oracle, -O3 -march=native, all host threads)
    python bench.py --workload c3 | c4 [...]                 BASELINE.json configs[2] / configs[3] as the headline line
    python bench.py ... --dump-outputs DIR                   also writes what the last timed step returned as DIR/<name>.npy

One "step" of the default workload (c2) = one call of s3d_gicp_align_batch on `--pairs` independent scan pairs
(consecutive-scan odometry: voxel filter 0.1 m x2, NN grids, kNN-20 covariances x2, GICP loop, fitness, gates — the whole align()).
  value         whole-job registrations/s with the raw scans already resident in HBM (device pointers);
  e2e           the same call with HOST (pinned) scan buffers: H2D of both scans and D2H of the results inside the timing;
  e2e_pageable  the same from pageable host memory (what a std::vector / pcl::PointCloud is).
Multi-GPU (torchrun): every rank runs the same per-GPU batch on its own GPU (independent registrations, no data-path
collective; weak scaling: the same multiset of scan pairs on every GPU); elapsed = max over ranks.
The default line also carries, under `config`: the odometry chain through the device cache, config 3 (VoxelGrid on a 2M-point
cloud) and single-pair latency at N = 1, config 4 (256 loop-closure pairs, strong scaling over the ranks) at every N, and the
in-process multi-device context (ONE process driving all N GPUs) when N > 1.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "gicp_registrations_per_s_131k_pt_pairs"
UNIT = "registrations/s"
N_POINTS = 131072
VOXEL = 0.1
SEED0 = 20260117


def make_pairs(n_distinct, seed0=SEED0, loop=False):
    from slam3d_b200 import synth
    return [synth.scan_pair(seed=seed0 + i, loop=loop) for i in range(n_distinct)]


def params():
    from slam3d_b200._abi import RegistrationParameters
    return RegistrationParameters.defaults(point_cloud_density=VOXEL)  # 2.5 m corr. distance, 50 iterations, default epsilons


def dump_results(out_dir, results, prefix=""):
    """--dump-outputs: the fields of the Result structs a caller of the timed call receives, one float64 array per field
    (pose: (n, 4, 4), the others: (n,)), in the order of the pairs."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"pose": np.array([r.pose() for r in results], np.float64).reshape(-1, 4, 4)}
    for name in ("fitness", "status", "converged", "outer_iterations", "inner_iterations", "n_source", "n_target", "n_correspondences"):
        arrays[name] = np.array([getattr(r, name) for r in results], np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


DUMP_MAX_ROWS = 1 << 20  # per dumped cloud: 16 MB of float32 xyzw


def dump_cloud(out_dir, name, cloud):
    """--dump-outputs for a point cloud: all rows up to DUMP_MAX_ROWS, beyond that a fixed, seeded sample of them (in order)."""
    os.makedirs(out_dir, exist_ok=True)
    cloud = np.asarray(cloud, np.float32)
    if cloud.shape[0] > DUMP_MAX_ROWS:
        cloud = cloud[np.sort(np.random.default_rng(0).choice(cloud.shape[0], DUMP_MAX_ROWS, replace=False))]
    np.save(os.path.join(out_dir, name + ".npy"), cloud)


def loop_params():
    """createConstraint(loop = true), PointCloudSensor.cpp:286-292: coarse (0.5 m, 5 m) then fine (0.1 m) — SURVEY C4."""
    from slam3d_b200._abi import RegistrationParameters
    coarse = RegistrationParameters.defaults(point_cloud_density=0.5, max_correspondence_distance=5.0, max_translation=5.0)
    fine = RegistrationParameters.defaults(point_cloud_density=0.1, max_translation=5.0)
    return coarse, fine


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md): ONE `nvidia-smi -lms 200` process, started
    before and killed after, on rank 0 only.  (A fresh nvidia-smi every 200 ms on every rank — 8 processes that each enumerate all
    GPUs of the box — slowed the timed region of the 8-GPU run itself: 24.9 ms per step against 22.1 ms for the e2e pass that ran
    without a sampler, profiles/r02_summary.md.)"""

    def __init__(self, index, enabled=True):
        self.index = index
        self.enabled = enabled
        self.rows = []
        self.proc = None

    def __enter__(self):
        if self.enabled:
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            try:
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        try:
            self.proc.terminate()
            out, _ = self.proc.communicate(timeout=6)
        except Exception:
            self.proc.kill()
            out = ""
        if not out.strip():  # nothing came through the pipe: one query now, right behind the timed region
            try:
                q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                    "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout
            except Exception:
                out = ""
        self.rows = [[c.strip() for c in line.split(",")] for line in out.splitlines() if line.strip()]

    def summary(self):
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) >= 6 and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU arms: the oracle port built for THIS host (-O3 -march=native), one pair per host thread
# ---------------------------------------------------------------------------------------------------------------------------------
def _oracle_native():
    import oracle
    oracle.build()
    how = oracle.use_native()  # compiles a -march=native build in a private temporary directory; falls back to the portable build
    return oracle, how


def run_reference(args, rank, world):
    """Reference arm: the CPU implementation of the path (oracle port; real PCL is not installable, SURVEY 8c)."""
    if rank != 0:
        return
    oracle, how = _oracle_native()
    threads = oracle.max_threads()
    n = max(1, min(threads, 64))  # one pair per host thread: every core busy
    loop = args.workload == "c4"
    pairs = make_pairs(min(max(n, 16), 16), seed0=5000 if loop else SEED0, loop=loop)
    srcs = [pairs[i % len(pairs)][0] for i in range(n)]
    tgts = [pairs[i % len(pairs)][1] for i in range(n)]

    def step():
        if loop:
            coarse, fine = loop_params()
            rc = oracle.gicp_align_batch(srcs, tgts, None, coarse, n_threads=threads)
            return oracle.gicp_align_batch(srcs, tgts, [r.pose() for r in rc], fine, n_threads=threads)
        return oracle.gicp_align_batch(srcs, tgts, None, params(), n_threads=threads)

    warm = min(args.warmup, 3)
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    done = 0
    steps = args.steps
    for _ in range(steps):
        last = step()
        done += len(last)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_results(args.dump_outputs, last, "fine_" if loop else "")
    value = done / dt
    metric, unit = (METRIC, UNIT) if not loop else ("loop_closure_constraints_per_s_256_pairs", "constraints/s")
    wl = ("256 synthetic loop-closure candidate pairs (131072 points), coarse 0.5 m / 5 m then fine 0.1 m GICP (BASELINE.json configs[3])" if loop
          else "synthetic 64-beam LiDAR scan pair, 131072 points, 0.1 m voxel, GICP odometry (BASELINE.json configs[1])")
    sample = f"{n} pairs per step on {threads} host threads (one pair per thread), {steps} steps, {len(pairs)} distinct scenes, oracle port of PCL GICP, {how}"
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "strong" if loop else "weak", "vs_baseline": None, "dtype": "f32/f64",
        "data": "synthetic", "config": {"workload": wl, "pairs_per_step": n, "ms_per_align_per_thread": 1e3 * dt * min(threads, n) / done / (2 if loop else 1)},
        "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline_leg():
    """Bounded CPU sample of the default workload on the host cores (rank 0, N=1 only)."""
    oracle, how = _oracle_native()
    threads = oracle.max_threads()
    n = max(1, min(threads, 64))  # one pair per host thread: every core busy
    pairs = make_pairs(min(n, 16))
    srcs = [pairs[i % len(pairs)][0] for i in range(n)]
    tgts = [pairs[i % len(pairs)][1] for i in range(n)]
    p = params()
    t0 = time.perf_counter()
    one = oracle.gicp_align(srcs[0], tgts[0], None, p)
    t1 = time.perf_counter() - t0
    t0 = time.perf_counter()
    rounds = 0
    while True:
        oracle.gicp_align_batch(srcs, tgts, None, p, n_threads=threads)
        rounds += 1
        if time.perf_counter() - t0 > 8 or rounds >= 4:
            break
    dt = time.perf_counter() - t0
    return {"value": rounds * n / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{rounds} x {n} pairs ({len(pairs)} distinct scenes), one pair per host thread ({threads} threads), {how}; "
                      f"single-thread align = {1e3 * t1:.0f} ms ({one.outer_iterations} outer iterations)",
            "single_thread_ms_per_align": 1e3 * t1}


# ---------------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4"], help="headline workload: BASELINE.json configs[1] / [2] / [3]")
    ap.add_argument("--pairs", type=int, default=64, help="scan pairs per step and per GPU (c2)")
    ap.add_argument("--distinct", type=int, default=16, help="distinct synthetic scenes to cycle through")
    ap.add_argument("--in-process", action="store_true", help="ONE process drives all --gpus devices through one context (no torchrun)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-chain", action="store_true", help="skip the supplementary odometry-chain measurement (device cache)")
    ap.add_argument("--no-extras", action="store_true", help="skip the supplementary config 3 / config 4 / latency / in-process measurements")
    ap.add_argument("--scene-rank", type=int, default=-1, help="experiment: another set of scenes (seed offset 1000 R), to see the cost spread between scene sets")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0; inputs are seeded, so two builds compare output for output). "
                         "--impl reference runs min(host threads, 64) pairs per step, not --pairs: compare its dumps with reference dumps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import slam3d_b200
    from slam3d_b200 import _abi, sharding, synth

    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")  # host-side barrier for the in-process leg: an NCCL barrier keeps the waiting GPUs busy
    in_process = args.in_process and world == 1 and args.gpus > 1
    devices = list(range(args.gpus)) if in_process else [local_rank]
    n_dev = len(devices)
    ctx = slam3d_b200.Context(devices)
    p = params()
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"

    def barrier():
        for d in devices:
            torch.cuda.synchronize(d)
        if world > 1:
            dist.barrier()
        for d in devices:
            torch.cuda.synchronize(d)

    def timed_call(fn, steps):
        """K calls of fn between barriers; host wall clock around the (synchronous) calls, max over ranks."""
        barrier()
        c0 = ctx.counters()
        t0 = time.perf_counter()
        last = None
        for _ in range(steps):
            last = fn()
        barrier()
        wall = 1e3 * (time.perf_counter() - t0)
        c1 = ctx.counters()
        return sharding.max_over_ranks(wall, device="cuda"), {k: c1[k] - c0[k] for k in c0}, last

    def pin(a):
        return torch.from_numpy(slam3d_b200.as_xyzw(a)).pin_memory()

    # ==============================================================================================================================
    if args.workload == "c3":
        out = bench_c3(ctx, peak, peak_src, args, headline=True)
        if rank == 0:
            print(json.dumps(out))
        return
    if args.workload == "c4":
        out = bench_c4(ctx, args, rank, world, n_dev, headline=True, barrier=barrier)
        if rank == 0:
            print(json.dumps(out))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- synthetic input: `distinct` scenes, cycled to `pairs` per step and device --------------------------------------------------
    # Weak scaling needs the SAME work on every GPU: all ranks draw the same scenes (rank r starts the cycle at scene r), so
    # the per-GPU batch is the same multiset of pairs at every N.  (Rank-private scenes were measured in round 1: their cost
    # differs by up to 35 %, and the max over ranks then measures the slowest scene set, not the scaling.)
    pairs = make_pairs(args.distinct, seed0=SEED0 + (0 if args.scene_rank < 0 else 1000 * args.scene_rank))
    B = args.pairs * n_dev
    host_src, host_tgt, page_src, page_tgt, dev_src, dev_tgt = [], [], [], [], [], []
    for i in range(B):
        s, t, _ = pairs[(i + rank) % len(pairs)]
        hs, ht = pin(s), pin(t)
        host_src.append(hs); host_tgt.append(ht)
        page_src.append(slam3d_b200.as_xyzw(s).copy()); page_tgt.append(slam3d_b200.as_xyzw(t).copy())  # pageable numpy memory
        d = devices[min(i // args.pairs, n_dev - 1)]  # the shard of device d in an in-process run (contiguous shards, api.cu)
        dev_src.append(hs.cuda(d)); dev_tgt.append(ht.cuda(d))
    barrier()

    stream = torch.cuda.ExternalStream(ctx.stream_handle(0), device=torch.device("cuda", devices[0]))

    rank_ms = []

    def timed(srcs, tgts, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0 = ctx.counters()
        t0 = time.perf_counter()
        e0.record(stream)
        last = None
        for _ in range(steps):
            last = ctx.gicp_align_batch(srcs, tgts, None, p)
        e1.record(stream)
        local = 1e3 * (time.perf_counter() - t0)  # this rank alone, before the closing barrier (the calls are synchronous)
        barrier()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        if world > 1:  # the spread over ranks next to the max the contract asks for: GPU-to-GPU variation vs. contention
            g = [torch.zeros(1, device="cuda") for _ in range(world)]
            dist.all_gather(g, torch.tensor([local / steps], device="cuda"))
            rank_ms[:] = [round(float(x), 3) for x in g]
        c1 = ctx.counters()
        # the call is synchronous and uses several streams: the wall span covers the device span; max over ranks
        el = sharding.max_over_ranks(max(ms, 1e3 * wall), device="cuda")
        ev = sharding.max_over_ranks(ms, device="cuda")
        return ev, el, {k: c1[k] - c0[k] for k in c0}, last

    # ---- warm-up, then EXACTLY K timed steps with device-resident inputs --------------------------------------------------
    # the clock sampler runs from the warm-up on (same load), so that short timed regions still collect several samples
    with ClockSampler(devices[0], enabled=(rank == 0)) as clk:
        for _ in range(max(args.warmup, 3)):
            ctx.gicp_align_batch(dev_src, dev_tgt, None, p)
        ev_ms, wall_ms, cnt, last = timed(dev_src, dev_tgt, args.steps)
    if args.dump_outputs and rank == 0:
        dump_results(args.dump_outputs, last)
    value = world * B * args.steps / (wall_ms / 1e3)
    rank_ms_value = list(rank_ms)  # of the device-resident timed region (later timed() calls overwrite rank_ms)
    ok = sum(1 for r in last if r.status == _abi.S3D_OK)

    # per-kernel durations for the roofline: same workload, same process, right after the timed region, but on ONE stream
    # (with several concurrent streams an event pair also spans other streams' kernels, so a kernel's own duration is undefined)
    os.environ["S3D_STREAMS_PER_DEVICE"] = "1"
    os.environ["S3D_LOOP_MODE"] = "2"  # the per-pass kernels of the batch path (a single-stream call would otherwise take the persistent kernel)
    ctx_serial = slam3d_b200.Context([devices[0]])
    ser_src, ser_tgt = dev_src[:args.pairs], dev_tgt[:args.pairs]
    ctx_serial.gicp_align_batch(ser_src, ser_tgt, None, p)
    ctx_serial.set_profiling(True)
    ctx_serial.stage_times(reset=True)
    ctx_serial.loop_stats(reset=True)
    prof_steps = max(1, min(args.steps, 3))
    for _ in range(prof_steps):
        last_serial = ctx_serial.gicp_align_batch(ser_src, ser_tgt, None, p)
    stages = ctx_serial.stage_times(reset=True)
    loop_stats = ctx_serial.loop_stats(reset=True)
    ctx_serial.close()
    del os.environ["S3D_STREAMS_PER_DEVICE"]
    del os.environ["S3D_LOOP_MODE"]

    # ---- end to end: host buffers in, results out, same call ---------------------------------------------------------------------
    for _ in range(2):
        ctx.gicp_align_batch(host_src, host_tgt, None, p)
    e2e_ev, e2e_wall, e2e_cnt, _ = timed(host_src, host_tgt, args.steps)
    e2e_value = world * B * args.steps / (e2e_wall / 1e3)
    for _ in range(1):
        ctx.gicp_align_batch(page_src, page_tgt, None, p)
    pg_ev, pg_wall, pg_cnt, _ = timed(page_src, page_tgt, max(1, min(args.steps, 5)))
    pg_value = world * B * max(1, min(args.steps, 5)) / (pg_wall / 1e3)

    extras = {}
    # ---- supplementary: consecutive-scan odometry through the per-measurement device cache (SURVEY 8f rank 1) -----------------
    if world == 1 and n_dev == 1 and not args.no_chain:
        scans, _ = synth.trajectory(seed=SEED0, n_scans=9)
        order = list(range(9)) + list(range(7, 0, -1))            # 0..8..1: consecutive entries are neighbouring poses
        seq = [order[i % len(order)] for i in range(args.pairs + 1)]
        pinned = [pin(s) for s in scans]
        host_seq = [pinned[j] for j in seq]

        def chain_step():
            hh = ctx.prepare_clouds(host_seq, VOXEL, 20)
            rr = ctx.gicp_align_prepared_batch(hh[:-1], hh[1:], None, p)
            for h in hh:
                h.release()
            return rr

        for _ in range(2):
            chain_step()
        ms, _, rr = timed_call(chain_step, args.steps)
        extras["odometry_chain_device_cache"] = {
            "value": args.pairs * args.steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / args.steps, "scans_per_step": args.pairs + 1,
            "registrations_ok": sum(1 for r in rr if r.status == _abi.S3D_OK),
            "what": "e2e from pinned host scans: every scan uploaded and preprocessed once, used as target and as source"}

    if not args.no_extras:
        if world == 1 and n_dev == 1:
            # ---- one registration at a time: what an unchanged createConstraint caller sees (PointCloudSensor.cpp:269-299) ----
            s0, t0_, _ = pairs[0]
            hs, ht = pin(s0), pin(t0_)
            for _ in range(3):
                ctx.gicp_align(hs, ht, None, p)
            n_lat = 20
            ms, lc, _ = timed_call(lambda: ctx.gicp_align(hs, ht, None, p), n_lat)
            hh = ctx.prepare_clouds([hs, ht], VOXEL, 20)
            for _ in range(3):
                ctx.gicp_align_prepared(hh[0], hh[1], None, p)
            ms_p, _, _ = timed_call(lambda: ctx.gicp_align_prepared(hh[0], hh[1], None, p), n_lat)
            for h in hh:
                h.release()
            extras["single_pair_latency"] = {"ms_per_align_host_scans": ms / n_lat, "ms_per_align_prepared_clouds": ms_p / n_lat,
                                             "launches_per_align": lc["kernel_launches"] / n_lat,
                                             "what": "s3d_gicp_align on one pinned-host pair, synchronous, one call at a time"}
            extras["c3_voxelgrid_2m_points"] = bench_c3(ctx, peak, peak_src, args, headline=False)
        extras["c4_loop_closure_256_pairs"] = bench_c4(ctx, args, rank, world, n_dev, headline=False, barrier=barrier)
        if world > 1:
            # ---- the in-process multi-device path: ONE process (rank 0) shards a batch over all N GPUs through one context -------
            # (the other ranks wait on the HOST — gloo — so that their GPUs are really idle)
            barrier()
            dist.barrier(group=cpu_group)
            if rank == 0:
                ctx_all = slam3d_b200.Context(list(range(world)))
                bsrc = [host_src[i % len(host_src)] for i in range(args.pairs * world)]
                btgt = [host_tgt[i % len(host_tgt)] for i in range(args.pairs * world)]
                for _ in range(2):
                    ctx_all.gicp_align_batch(bsrc, btgt, None, p)
                n_ip = max(1, min(args.steps, 5))
                t0 = time.perf_counter()
                for _ in range(n_ip):
                    rr = ctx_all.gicp_align_batch(bsrc, btgt, None, p)
                dt = time.perf_counter() - t0
                extras["in_process_multi_device"] = {
                    "value": len(bsrc) * n_ip / dt, "unit": UNIT, "devices": world, "pairs_per_call": len(bsrc), "ms_per_call": 1e3 * dt / n_ip,
                    "registrations_ok": sum(1 for r in rr if r.status == _abi.S3D_OK),
                    "what": "s3d_create_context(devices = all N) in ONE process, pinned host scans in, results out; the other ranks idle"}
                ctx_all.close()
            dist.barrier(group=cpu_group)
            barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------------------------
    dom = max(stages, key=lambda k: stages[k]["ms"])
    m_tgt = float(np.mean([r.n_target for r in last]))
    m_src = float(np.mean([r.n_source for r in last]))
    n_ser = len(last_serial) * prof_steps
    outer_total = sum(r.outer_iterations for r in last_serial) * prof_steps           # search passes (pair-iterations)
    tiles_per_pass = float(np.mean([(r.n_target + 255) // 256 for r in last_serial]))
    passes_total = loop_stats["tiles"] / max(tiles_per_pass, 1.0)                         # search + trial + fitness passes
    eval_total = max(passes_total - outer_total - n_ser, 0.0)                            # trial passes
    # algorithmic bytes (DESIGN.md 4, SURVEY 8d with 24-byte normals instead of 48-byte covariances):
    bytes_by_stage = {
        "gicp_iter": 80.0 * m_tgt * outer_total,                        # search pass: 16+24 moving point/normal + 16+24 gathered fixed point/normal
        "knn_cov": 40.0 * (m_tgt + m_src) * n_ser,                      # 16 read + 24 written per point
        "voxel": (16.0 * 2 * N_POINTS + 16.0 * (m_tgt + m_src)) * n_ser,
        "grid": 36.0 * (m_tgt + m_src) * n_ser,
        "fitness": 32.0 * m_tgt * n_ser,
        "gicp_solve": 80.0 * m_tgt * eval_total,                        # trial pass: 16 + 16 + 48 (control kernels: a few KB)
    }
    kernel_of = {"gicp_iter": "gicp_search_kernel", "knn_cov": "knn_cov_kernel", "voxel": "voxel_*", "grid": "grid_*", "fitness": "gicp_fitness_kernel",
                 "gicp_solve": "gicp_trial_kernel + gicp_ctrl_kernel"}
    dom_ms = stages[dom]["ms"]
    dom_launches = max(stages[dom]["launches"], 1)
    achieved = bytes_by_stage[dom] / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else 0.0
    # DRAM traffic of the dominant kernel: per-unit figures of the committed ncu --set full capture (scripts/profile_round.sh writes
    # profiles/<tag>_traffic.json), scaled to this run's launch size; null when the file has no entry for the kernel.
    traffic, traffic_src = None, None
    tpaths = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_traffic.json")) if os.path.isdir(os.path.join(ROOT, "profiles")) else []
    if tpaths:
        tj = json.load(open(os.path.join(ROOT, "profiles", tpaths[-1])))
        ent = tj.get(kernel_of[dom])
        if ent:
            units = {"gicp_iter": m_tgt * outer_total, "knn_cov": (m_tgt + m_src) * n_ser}.get(dom)
            if units:
                traffic = ent["dram_bytes_per_unit"] * units / dom_launches
                traffic_src = f"profiles/{tpaths[-1]}: {ent['dram_bytes_per_unit']:.1f} B per {ent['unit']} ({ent.get('capture', '')})"
    roofline = {"bound": "hbm", "kernel": kernel_of[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "avg_launch_us": 1e3 * dom_ms / dom_launches, "launches": dom_launches,
                "algorithmic_bytes_per_launch": bytes_by_stage[dom] / dom_launches,
                "stage_ms_per_step": {k: v["ms"] / prof_steps for k, v in stages.items()},
                "stage_frac_of_peak": {k: (bytes_by_stage[k] / (v["ms"] / 1e3) / 1e9 / peak if v["ms"] > 0 else None) for k, v in stages.items()},
                "loop_kernel_passes_per_pair": {"search": outer_total / n_ser, "trial": eval_total / n_ser, "fitness": 1.0,
                                                "control_steps": loop_stats["control_steps"] / n_ser},
                "timing": f"CUDA events per stage on the launching stream, {prof_steps} single-stream steps of {args.pairs} pairs right after the timed region",
                "note": "not HBM bound: a pair's working set is L2 resident; the search kernels are instruction-issue / latency bound (DESIGN.md 4)"}
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world * n_dev, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": wall_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64",
        "data": "synthetic",
        "config": {"workload": "synthetic 64-beam LiDAR scan pair, 131072 points, 0.1 m voxel, GICP odometry (BASELINE.json configs[1])",
                   "rank_ms_per_step": rank_ms_value, "pairs_per_step_per_gpu": args.pairs, "distinct_scenes": args.distinct, "ms_per_align": wall_ms / args.steps / B,
                   "processes": "one process, one context over all devices (--in-process)" if in_process else "one process per GPU",
                   "l2": f"inputs larger than L2: {args.pairs} pairs x 4.2 MB raw + ~50 MB working set per pair per step",
                   "registrations_ok": ok, "mean_outer_iterations": float(np.mean([r.outer_iterations for r in last])),
                   "filtered_points": [int(m_src), int(m_tgt)], "device_event_ms_per_step": ev_ms / args.steps},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_cnt["h2d_bytes"] // args.steps,
                "d2h_bytes_per_step": e2e_cnt["d2h_bytes"] // args.steps, "ms_per_step": e2e_wall / args.steps, "host_memory": "pinned"},
        "e2e_pageable": {"value": pg_value, "unit": UNIT, "ms_per_step": pg_wall / max(1, min(args.steps, 5)),
                         "host_memory": "pageable (numpy arrays, like the std::vector behind a pcl::PointCloud)"},
        "gpu_launches": cnt["kernel_launches"],
        "clocks": clk.summary(),
        "roofline": roofline,
    }
    out["config"].update(extras)
    if world == 1 and n_dev == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_leg()
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------------------
def bench_c3(ctx, peak, peak_src, args, headline):
    """BASELINE.json configs[2]: VoxelGrid on the 2 097 152-point synthetic map cloud (device resident), leaf 0.05 / 0.1 / 0.2 m,
    plus kNN-20 covariances on the 0.1 m result."""
    import torch
    import slam3d_b200
    from slam3d_b200 import synth
    cloud = synth.map_cloud(n_scans=16)
    dev = torch.from_numpy(slam3d_b200.as_xyzw(cloud)).cuda()
    was = True
    ctx.set_profiling(True)
    res = {}
    n = args.steps if headline else 10
    for leaf in (0.05, 0.1, 0.2):
        for _ in range(3):
            out, _, _ = ctx.voxel_downsample(dev, leaf, want_leaf_index=False)
        ctx.stage_times(reset=True)
        for _ in range(n):
            out, _, _ = ctx.voxel_downsample(dev, leaf, want_leaf_index=False)
        st = ctx.stage_times(reset=True)
        if headline and args.dump_outputs:
            dump_cloud(args.dump_outputs, f"voxel_leaf_{leaf}", out)
        ms = st["voxel"]["ms"] / n
        m = out.shape[0]
        algo = 16.0 * cloud.shape[0] + 16.0 * m   # SURVEY 8d: 16 B per input point read + 16 B per voxel written
        res[f"leaf_{leaf}"] = {"ms": ms, "voxels": int(m), "launches": st["voxel"]["launches"] // n, "algorithmic_gb_s": algo / ms / 1e6,
                               "frac_of_hbm_peak": algo / ms / 1e6 / peak}
        if leaf == 0.1:
            fd = torch.from_numpy(out).cuda()
            for _ in range(2):
                ctx.knn_covariances(fd, 20)
            ctx.stage_times(reset=True)
            for _ in range(3):
                ctx.knn_covariances(fd, 20)
            st = ctx.stage_times(reset=True)
            res["knn20_cov_on_0.1m_result"] = {"grid_ms": st["grid"]["ms"] / 3, "knn_cov_ms": st["knn_cov"]["ms"] / 3,
                                               "mqueries_per_s": m / (st["knn_cov"]["ms"] / 3) / 1e3}
    ctx.set_profiling(False)
    res["peak_source"] = peak_src
    res["timing"] = "CUDA events around the voxel-filter kernels (s3d_set_profiling), input resident in HBM (33.5 MB, below L2: 126 MB)"
    if not headline:
        return res
    ms = res["leaf_0.1"]["ms"]
    traffic, traffic_src = None, None
    import glob
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_c3_traffic.json")))[-1:]:  # measured by ncu (scripts/profile_round.sh, c3_traffic_json.py)
        t = json.load(open(f))["leaf_0.1"]
        traffic = t["cold"]["dram_bytes"]
        traffic_src = (f"{os.path.basename(f)}: DRAM read + write of the 8 launches of one call, caches flushed before every launch "
                       f"(warm, input L2-resident: {t['warm']['dram_bytes'] / 1e6:.1f} MB)")
    return {"metric": "voxelgrid_mpoints_per_s_2m_cloud", "value": cloud.shape[0] / ms / 1e3, "unit": "Mpoints/s", "n_gpus": 1, "steps": n, "warmup": 3,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/u32", "data": "synthetic",
            "config": {"workload": "VoxelGrid downsample + covariance stress: 2M-point synthetic cloud, leaf sizes 0.05/0.1/0.2 m (BASELINE.json configs[2])",
                       "l2": "input 33.5 MB < L2: L2-resident stream", **res},
            "roofline": {"bound": "hbm", "kernel": "voxel filter (bbox, keys, 4 radix passes, centroids: 8 launches)", "achieved": res["leaf_0.1"]["algorithmic_gb_s"],
                         "peak": peak, "unit": "GB/s", "frac": res["leaf_0.1"]["frac_of_hbm_peak"], "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes": 16.0 * cloud.shape[0] + 16.0 * res["leaf_0.1"]["voxels"], "peak_source": peak_src}}


def bench_c4(ctx, args, rank, world, n_dev, headline, barrier):
    """BASELINE.json configs[3]: 256 loop-closure candidate pairs through s3d_gicp_align_loop_batch (coarse then fine, scans
    uploaded once), STRONG scaling: the 256 pairs are sharded over the ranks (or over the devices of an in-process context)."""
    import torch
    import slam3d_b200
    from slam3d_b200 import _abi, sharding
    total = 256
    lo, hi = sharding.shard_range(total, rank, world)
    scenes = make_pairs(min(args.distinct, 16), seed0=5000, loop=True)
    pinned = [(torch.from_numpy(slam3d_b200.as_xyzw(s)).pin_memory(), torch.from_numpy(slam3d_b200.as_xyzw(t)).pin_memory(), T) for s, t, T in scenes]
    srcs = [pinned[i % len(pinned)][0] for i in range(lo, hi)]
    tgts = [pinned[i % len(pinned)][1] for i in range(lo, hi)]
    truth = [pinned[i % len(pinned)][2] for i in range(lo, hi)]
    coarse, fine = loop_params()
    ctx.gicp_align_loop_batch(srcs, tgts, None, coarse, fine)
    steps = args.steps if headline else max(1, min(args.steps, 3))
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        rc, rf = ctx.gicp_align_loop_batch(srcs, tgts, None, coarse, fine)
    barrier()
    dt = sharding.max_over_ranks(time.perf_counter() - t0, device="cuda") / steps
    if headline and args.dump_outputs and rank == 0:
        dump_results(args.dump_outputs, rc, "coarse_")
        dump_results(args.dump_outputs, rf, "fine_")
    okf = [r.status == _abi.S3D_OK for r in rf]
    err = [float(np.linalg.norm((np.linalg.inv(T) @ r.pose())[:3, 3])) for r, T, good in zip(rf, truth, okf) if good]
    res = {"constraints_per_s": total / dt, "aligns_per_s": 2 * total / dt, "ms_per_256_pairs": 1e3 * dt, "pairs_this_rank": hi - lo,
           "accepted_this_rank": int(sum(okf)), "median_translation_error_m_vs_truth": float(np.median(err)) if err else None,
           "scaling": "strong: 256 pairs over all GPUs", "api": "s3d_gicp_align_loop_batch, pinned host scans in, results out"}
    if not headline:
        return res
    return {"metric": "loop_closure_constraints_per_s_256_pairs", "value": total / dt, "unit": "constraints/s", "n_gpus": world * n_dev, "steps": steps, "warmup": 1,
            "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": "batched loop-closure: 256 synthetic candidate scan pairs (131k pts), coarse + fine GICP (BASELINE.json configs[3])", **res},
            "e2e": {"value": total / dt, "unit": "constraints/s", "h2d_bytes_per_step": int(2 * 16 * N_POINTS * (hi - lo)), "d2h_bytes_per_step": 0, "ms_per_step": 1e3 * dt}}


if __name__ == "__main__":
    main()
