"""CPU prototype: bounding boxes of 32 Morton-consecutive transformed queries in the fixed cloud's grid — what a shared-candidate 1-NN
tile would have to load.  Result: profiles/r02_summary.md."""
import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle
from slam3d_b200 import synth
from scipy.spatial import cKDTree

src, tgt, truth = synth.scan_pair(seed=20260117)
B, _, _ = oracle.voxel_downsample(src, 0.1)   # fixed cloud (slam3d source)
A, _, _ = oracle.voxel_downsample(tgt, 0.1)   # moving cloud
B = B[:, :3].astype(np.float64); A = A[:, :3].astype(np.float64)
print("truth\n", truth)
def spread(v):
    v = v & 0x3FF
    v = (v | (v << 16)) & 0x030000FF
    v = (v | (v << 8)) & 0x0300F00F
    v = (v | (v << 4)) & 0x030C30C3
    v = (v | (v << 2)) & 0x09249249
    return v
def morton_order(P, h0):
    lo = P.min(0)
    c = np.floor((P - lo) / h0).astype(np.int64)
    key = spread(c[:, 0]) | (spread(c[:, 1]) << 1) | (spread(c[:, 2]) << 2)
    return np.argsort(key, kind='stable'), key
h0 = 0.3
oa, keya = morton_order(A, h0)
A = A[oa]; keya = keya[oa]
treeB = cKDTree(B)
loB = B.min(0)
for name, T in (("iter1 identity", np.eye(4)), ("converged", truth)):
    Q = A @ T[:3, :3].T + T[:3, 3]
    d, j = treeB.query(Q)
    print(name, "NN dist pct 50/75/90/95/99", np.percentile(d, [50, 75, 90, 95, 99]), "frac > 2.5:", (d > 2.5).mean())
    for dil_cells in (1, 2):
      for maxcells in (96, 192):
        nwarps = (len(Q) + 31) // 32
        tot_slots = 0; cert = 0; nq = 0; big = 0; Cs = []
        for w in range(nwarps):
            q = Q[32 * w: 32 * w + 32]; dq = d[32 * w: 32 * w + 32]
            c = np.floor((q - loB) / h0).astype(np.int64)
            clo = c.min(0) - dil_cells; chi = c.max(0) + dil_cells
            ncell = np.prod(chi - clo + 1)
            if ncell > maxcells:
                big += len(q); continue
            rlo = loB + clo * h0; rhi = loB + (chi + 1) * h0
            cov = np.minimum(q - rlo, rhi - q).min(1)
            ok = np.minimum(dq, 2.5) <= cov * 0.999
            idx = treeB.query_ball_point((rlo + rhi) / 2, r=1.0, p=np.inf)  # placeholder
            # count points in box
            m = np.all((B >= rlo) & (B < rhi), axis=1).sum() if False else None
            cert += ok.sum(); nq += len(q)
        print(f"   dil {dil_cells} cells, max {maxcells} cells: warps too big: {big / len(Q):.3f} of queries; certified among tiled: {cert / max(nq,1):.3f}")
