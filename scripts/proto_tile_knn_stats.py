"""CPU prototype (numpy + cKDTree): what a warp-cooperative TILE kNN would have to scan on the bench clouds — group sizes, shared
candidate-set sizes and the share of queries whose k-th neighbour such a tile cannot certify.  Result: profiles/r02_summary.md."""
import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle
from slam3d_b200 import synth
from scipy.spatial import cKDTree

src, tgt, truth = synth.scan_pair(seed=20260117)
pts, _, _ = oracle.voxel_downsample(src, 0.1)
P = pts[:, :3].astype(np.float64)
n = len(P)
print("filtered", n)
tree = cKDTree(P)
d, _ = tree.query(P, k=20)
rk = d[:, -1]
print("kNN-20 radius pct 10/50/90/99/max", np.percentile(rk, [10, 50, 90, 99]), rk.max())

def spread(v):
    v = v & 0x3FF
    v = (v | (v << 16)) & 0x030000FF
    v = (v | (v << 8)) & 0x0300F00F
    v = (v | (v << 4)) & 0x030C30C3
    v = (v | (v << 2)) & 0x09249249
    return v

for h0 in (0.3,):
    lo = P.min(0)
    ext = (P.max(0) - lo).max()
    nlev = 1
    while nlev < 10 and h0 * (1 << nlev) <= ext * 1.001: nlev += 1
    c = np.floor((P - lo) / h0).astype(np.int64)
    key = spread(c[:, 0]) | (spread(c[:, 1]) << 1) | (spread(c[:, 2]) << 2)
    order = np.argsort(key, kind='stable')
    key = key[order]; Ps = P[order]; rks = rk[order]; cs = c[order]
    # population of each ancestor cell per point
    pops = []
    for L in range(nlev + 1):
        kl = key >> (3 * L)
        _, inv, cnt = np.unique(kl, return_inverse=True, return_counts=True)
        pops.append(cnt[inv])
    pops = np.stack(pops, 0)  # [L, n]
    for T in (16, 32, 64):
        # group level per point: largest L with pop[L] <= T (walk up while parent's pop <= T)
        gl = np.zeros(n, np.int64)
        for L in range(1, nlev + 1):
            ok = (pops[L] <= T) & (gl == L - 1)
            gl[ok] = L
        gpop = pops[gl, np.arange(n)]
        # a level-0 cell with > T points: chunks
        gkey = (key >> (3 * gl)) * 16 + gl
        ug, first, cnt = np.unique(gkey, return_index=True, return_counts=True)
        print(f"h0={h0} T={T}: groups {len(ug)} mean size {cnt.mean():.1f}  size hist", np.bincount(np.minimum(cnt, T + 1) * 8 // (T + 1), minlength=9)[:9])
        # per group: level L, cell coords; region options
        tot_slots_half = 0; tot_slots_full = 0; fail_half = 0; fail_full = 0; chosen_slots = 0; chosen_fail = 0; nq = 0
        Cs = []
        import collections
        stat = collections.Counter()
        for gi in range(len(ug)):
            s = first[gi]; q = cnt[gi]; L = gl[s]
            hL = h0 * (1 << L)
            cell = cs[s] >> L
            glo = lo + cell * hL; ghi = glo + hL
            Q = Ps[s:s + q]; R = rks[s:s + q]
            inner = np.minimum(Q - glo, ghi - Q).min(1)  # distance to own-cell faces
            res = {}
            for name, dil in (("half", 0.5 * hL), ("full", hL), ("two", 2 * hL)):
                if name == "half" and L == 0: continue
                idx = tree.query_ball_point((glo + ghi) / 2, r=(hL / 2 + dil) * 1.0000001, p=np.inf)
                C = len(idx)
                cert = R <= (dil + inner) * 0.9999
                res[name] = (C, int((~cert).sum()))
            # choose: half if q >= 0.6T and L>0 else full
            if L > 0 and q >= 0.6 * T: ch = "half"
            elif q >= 0.2 * T: ch = "full"
            else: ch = "two"
            C, nf = res[ch]
            teams_rounds = -(-q // T)
            chosen_slots += C * T * teams_rounds
            chosen_fail += nf; nq += q
            stat[ch] += q
            Cs.append(C)
        print(f"   chosen: lane-slots/query {chosen_slots / nq:.0f}  fallback frac {chosen_fail / nq:.3f}  C mean {np.mean(Cs):.0f} p90 {np.percentile(Cs, 90):.0f} max {max(Cs)}  by region {dict(stat)}")
