"""What the BFGS inner optimiser (PCL <= 1.13, s3d_set_gicp_optimizer(S3D_GICP_BFGS)) costs against the Newton one (PCL >= 1.14,
the default) on the headline workload of bench.py: synthetic 131 072-point scan pairs, 0.1 m voxel, 64 pairs per step.

Both optimisers run in the same process and are alternated round by round, so that clock and neighbour drift hit both alike:
  * registrations/s of s3d_gicp_align_batch with device-resident scans and with pinned host scans (end to end);
  * one-pair latency of s3d_gicp_align (pinned host scans) and of s3d_gicp_align_prepared (clouds prepared once);
  * 256-point tiles and control steps per registration (s3d_get_loop_stats): the passes the optimiser asks for.
The GPU name and power limit are read in the same run and written into the JSON (default profiles/r03_bfgs.json).

    python scripts/bench_bfgs.py [--pairs 64] [--steps 5] [--rounds 3] [--latency-reps 20] [--out profiles/r03_bfgs.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED0 = 20260117
VOXEL = 0.1


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers below still stand; say what is missing
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e.__class__.__name__})"}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--steps", type=int, default=5, help="timed batch calls per optimiser and round")
    ap.add_argument("--rounds", type=int, default=3, help="alternations newton / bfgs")
    ap.add_argument("--latency-reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bfgs.json"))
    args = ap.parse_args()

    import numpy as np
    import torch
    import slam3d_b200
    from slam3d_b200 import _abi, synth
    from slam3d_b200._abi import RegistrationParameters

    if not torch.cuda.is_available():
        raise SystemExit("bench_bfgs: no CUDA device (this measures the B200 path; there is no CPU fallback)")
    p = RegistrationParameters.defaults(point_cloud_density=VOXEL)
    scenes = [synth.scan_pair(seed=SEED0 + i) for i in range(args.distinct)]

    def pin(a):
        return torch.from_numpy(slam3d_b200.as_xyzw(a)).pin_memory()

    host_src = [pin(scenes[i % len(scenes)][0]) for i in range(args.pairs)]
    host_tgt = [pin(scenes[i % len(scenes)][1]) for i in range(args.pairs)]
    dev_src = [h.cuda() for h in host_src]
    dev_tgt = [h.cuda() for h in host_tgt]
    ctx = slam3d_b200.Context()
    prepared = ctx.prepare_clouds([host_src[0], host_tgt[0]], VOXEL, 20)
    opts = ("newton", "bfgs")

    def batch_rate(srcs, tgts):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            last = ctx.gicp_align_batch(srcs, tgts, None, p)
        dt = time.perf_counter() - t0  # the calls are synchronous
        return args.pairs * args.steps / dt, last

    def latency(fn):
        ms = []
        for _ in range(args.latency_reps):
            t0 = time.perf_counter()
            fn()
            ms.append(1e3 * (time.perf_counter() - t0))
        return statistics.median(ms)

    res = {o: {"device_resident": [], "host_e2e": [], "align_ms": [], "align_prepared_ms": []} for o in opts}
    work, last = {}, {}
    for o in opts:  # warm-up of every shape, and the work counts (deterministic) of one batch
        ctx.set_gicp_optimizer(o)
        ctx.gicp_align_batch(dev_src, dev_tgt, None, p)
        ctx.gicp_align_batch(host_src, host_tgt, None, p)
        ctx.gicp_align(host_src[0], host_tgt[0], None, p)
        ctx.gicp_align_prepared(prepared[0], prepared[1], None, p)
        ctx.loop_stats(reset=True)
        rs = ctx.gicp_align_batch(dev_src, dev_tgt, None, p)
        st = ctx.loop_stats(reset=True)
        last[o] = rs
        work[o] = {"tiles_per_registration": st["tiles"] / args.pairs, "control_steps_per_registration": st["control_steps"] / args.pairs,
                   "outer_iterations_mean": float(np.mean([r.outer_iterations for r in rs])),
                   "inner_iterations_mean": float(np.mean([r.inner_iterations for r in rs])),
                   "registrations_ok": sum(1 for r in rs if r.status == _abi.S3D_OK)}
    for rnd in range(args.rounds):
        for o in (opts if rnd % 2 == 0 else opts[::-1]):
            ctx.set_gicp_optimizer(o)
            res[o]["device_resident"].append(batch_rate(dev_src, dev_tgt)[0])
            res[o]["host_e2e"].append(batch_rate(host_src, host_tgt)[0])
            res[o]["align_ms"].append(latency(lambda: ctx.gicp_align(host_src[0], host_tgt[0], None, p)))
            res[o]["align_prepared_ms"].append(latency(lambda: ctx.gicp_align_prepared(prepared[0], prepared[1], None, p)))
    ctx.set_gicp_optimizer("newton")
    for h in prepared:
        h.release()
    ctx.close()

    def summary(v):
        return {"median": statistics.median(v), "min": min(v), "max": max(v), "runs": v}

    out = {"what": "BFGS (PCL <= 1.13) vs Newton (PCL >= 1.14) inner optimiser, same process, alternated",
           "workload": f"synthetic 64-beam LiDAR scan pairs, 131072 points, {VOXEL} m voxel, {args.pairs} pairs per step, {args.distinct} scenes",
           **gpu_info(), "steps": args.steps, "rounds": args.rounds, "latency_reps": args.latency_reps,
           "units": {"device_resident": "registrations/s", "host_e2e": "registrations/s", "align_ms": "ms (median)", "align_prepared_ms": "ms (median)"}}
    for o in opts:
        out[o] = {k: summary(v) for k, v in res[o].items()}
        out[o].update(work[o])
    out["bfgs_over_newton"] = {k: out["bfgs"][k]["median"] / out["newton"][k]["median"] for k in res["newton"]}
    out["bfgs_over_newton"]["tiles_per_registration"] = work["bfgs"]["tiles_per_registration"] / work["newton"]["tiles_per_registration"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "power_limit", "bfgs_over_newton")}))
    for o in opts:
        print(o, {k: round(out[o][k]["median"], 3) for k in res[o]}, {k: work[o][k] for k in work[o]})


if __name__ == "__main__":
    main()
