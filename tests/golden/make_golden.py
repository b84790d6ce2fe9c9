#!/usr/bin/env python
"""Regenerates tests/golden/ from the reference's test data:  python make_golden.py <slam3d checkout>/test

Inputs : <dir>/cloud{1..4}.bin                 (KITTI-format float32 x,y,z,intensity; SURVEY Appendix B).
Outputs: tests/golden/cloud{1..4}.xyz.f32.xz   xyz float32, lzma — the reference DATA travels with the repo,
                                               so that the tests need nothing outside it;
         tests/golden/golden.json              frozen outputs of the CPU oracle (oracle/s3d_oracle.cpp) on them.

The reference has no expected outputs for this path (SURVEY 8c), so golden.json pins the ORACLE (regression) and
gives the GPU tests fixed targets; it is not a PCL output.
"""
import hashlib
import json
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle  # noqa: E402
from slam3d_b200._abi import RegistrationParameters  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main(ref):
    clouds = []
    for i in range(1, 5):
        raw = np.fromfile(os.path.join(ref, f"cloud{i}.bin"), np.float32).reshape(-1, 4)
        xyz = np.ascontiguousarray(raw[:, :3])
        with open(os.path.join(HERE, f"cloud{i}.xyz.f32.xz"), "wb") as f:
            f.write(lzma.compress(xyz.tobytes(), preset=9))
        clouds.append(xyz)
    g = {"clouds": [int(c.shape[0]) for c in clouds], "voxel": {}, "knn": {}, "align": {}}
    for leaf in (0.05, 0.1, 0.2, 0.5, 1.0):
        rows = []
        for c in clouds:
            out, leaf_index, overflow = oracle.voxel_downsample(c, leaf)
            rows.append({"n_out": int(out.shape[0]), "overflow": bool(overflow), "leaf_sha": sha(leaf_index),
                         "out_sha": sha(out)})
        g["voxel"][str(leaf)] = rows
    f1, _, _ = oracle.voxel_downsample(clouds[0], 0.1)
    f2, _, _ = oracle.voxel_downsample(clouds[1], 0.1)
    idx, d2, cov = oracle.knn_covariances(f1, 20)
    g["knn"]["cloud1@0.1,k=20"] = {"index_sha": sha(idx), "dist2_sha": sha(d2), "cov_sum": float(cov.sum()),
                                   "cov_first": cov[0].tolist()}
    nn_i, nn_d = oracle.nearest_neighbors(f1, f2)
    g["knn"]["nn cloud2@0.1 -> cloud1@0.1"] = {"index_sha": sha(nn_i), "dist2_sha": sha(nn_d)}
    for density in (0.1, 0.2):
        p = RegistrationParameters.defaults(point_cloud_density=density)
        for a, b in ((0, 1), (1, 2), (2, 3)):
            r = oracle.gicp_align(clouds[a], clouds[b], None, p)
            g["align"][f"cloud{a+1}->cloud{b+1}@{density}"] = {
                "status": r.status, "converged": r.converged, "outer_iterations": r.outer_iterations,
                "inner_iterations": r.inner_iterations, "n_source": r.n_source, "n_target": r.n_target,
                "n_correspondences": r.n_correspondences, "fitness": r.fitness, "T": r.pose().tolist()}
    from slam3d_b200 import _abi  # noqa: E402
    g["align_ndt"] = {}
    for density in (0.1, 0.2):  # the NDT branch (PointCloudSensor.cpp:84-117) with slam3d's NDT defaults
        p = RegistrationParameters.defaults(point_cloud_density=density, registration_algorithm=_abi.ALG_NDT)
        for a, b in ((0, 1), (1, 2), (2, 3)):
            r = oracle.gicp_align(clouds[a], clouds[b], None, p)
            g["align_ndt"][f"cloud{a+1}->cloud{b+1}@{density}"] = {
                "status": r.status, "converged": r.converged, "outer_iterations": r.outer_iterations,
                "inner_iterations": r.inner_iterations, "n_source": r.n_source, "n_target": r.n_target,
                "n_correspondences": r.n_correspondences, "fitness": r.fitness, "T": r.pose().tolist()}
    g["map"] = map_golden(clouds)
    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(g, f, indent=1)
    print(json.dumps(g["align"], indent=1))


def pose(tx, ty, yaw):
    T = np.eye(4)
    T[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
    T[:3, 3] = [tx, ty, 0.01]
    return T


def map_golden(clouds):
    """patch / map building (PointCloudSensor.cpp:211-233, :301-318): frozen oracle outputs, same cases as tests/test_gpu_map.py"""
    m = {"transform cloud1": {"sha": sha(oracle.transform_cloud(clouds[0], pose(12.3, -4.5, 0.7)))}}
    out, keep = oracle.remove_outliers(clouds[1], 0.2, 3)
    m["remove_outliers cloud2 r=0.2 n=3"] = {"kept": int(keep.sum()), "sha": sha(out)}
    poses = [pose(0.69 * i, 0.004 * i, 0.0035 * i) for i in range(4)]
    mp = oracle.build_map(clouds, poses, 0.2, 3, 0.1)
    m["build_map 4 clouds"] = {"n_out": int(mp.shape[0]), "sha": sha(mp)}
    return m


def add_map_only():
    """python make_golden.py --map: adds the "map" entry to an existing golden.json without touching the other entries"""
    clouds = [np.frombuffer(lzma.decompress(open(os.path.join(HERE, f"cloud{i}.xyz.f32.xz"), "rb").read()), np.float32).reshape(-1, 3) for i in range(1, 5)]
    path = os.path.join(HERE, "golden.json")
    g = json.load(open(path))
    g["map"] = map_golden(clouds)
    with open(path, "w") as f:
        json.dump(g, f, indent=1)
    print(json.dumps(g["map"], indent=1))


if __name__ == "__main__":
    if "--map" in sys.argv:
        add_map_only()
    elif len(sys.argv) == 2:
        main(sys.argv[1])
    else:
        sys.exit(__doc__)
