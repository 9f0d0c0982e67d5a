#!/usr/bin/env python
"""CPU census (scipy, no GPU) behind kernel 1t's ball-restricted tables: on the headline workload (Computers-shaped graph,
2-hop edge vicinities), how many vertices of S a root's shortest-path table leaves INVALID (the table path to the root
leaves S) and how many graph-row records those vertices cost (D_inv), for a table over the whole graph and for one over
the subgraph induced by the root's k-hop ball.  Counts, not times.
    python scripts/table_census.py [targets=240] [hop=2]
Ties: scipy's predecessor, not the kernel's smallest-id tree rule -- an estimate of the counts."""
import os
import sys

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import dijkstra

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tlc-gnn_b200"))
import bench  # noqa: E402

NT = int(sys.argv[1]) if len(sys.argv) > 1 else 240
HOP = int(sys.argv[2]) if len(sys.argv) > 2 else 2

c, labels, ne, csr, perm = bench.make_workload("computers")
rowptr, col, kap = [np.asarray(a) for a in csr]
N = len(rowptr) - 1
deg = np.diff(rowptr)
A = sp.csr_matrix((kap + 1.0, col, rowptr), shape=(N, N))
A01 = sp.csr_matrix((np.ones(len(col)), col, rowptr), shape=(N, N))


def ball(r):
    m = np.zeros(N, bool)
    m[r] = True
    f = m.copy()
    for _ in range(HOP):
        f = (A01.T @ f.astype(np.float64)) > 0
        m |= f
    return m


def invalid(root, S, sub):
    """(invalid vertices of S, their graph degrees) for the table of `root` built on the subgraph induced by mask `sub`"""
    idx = np.flatnonzero(sub)
    loc = -np.ones(N, int)
    loc[idx] = np.arange(len(idx))
    _, pred = dijkstra(A[idx][:, idx], indices=loc[root], return_predecessors=True)
    P = -np.ones(N, int)
    ok = pred >= 0
    P[idx[ok]] = idx[pred[ok]]
    cls = np.zeros(N, np.int8)  # 0 unknown, 1 valid, 2 invalid
    cls[root] = 1
    Sx = np.flatnonzero(S)
    for x in Sx:
        path, y = [], x
        while cls[y] == 0:
            path.append(y)
            p = P[y]
            if p < 0 or not S[p]:
                cls[y] = 2
                break
            y = p
        for z in path:
            cls[z] = cls[y]
    inv = Sx[cls[Sx] == 2]
    return len(inv), int(deg[inv].sum())


T = bench.batch_targets(ne, perm, 3, 0, 1, 4096)
pick = T[np.random.default_rng(1).choice(len(T), NT, replace=False)]
whole = np.ones(N, bool)
res = []
for u, v in pick:
    bu, bv = ball(u), ball(v)
    S = bu & bv
    a = [invalid(r, S, whole) for r in (u, v)]
    b = [invalid(r, S, br) for r, br in ((u, bu), (v, bv))]
    res.append((int(S.sum()), a[0][0] + a[1][0], a[0][1] + a[1][1], b[0][0] + b[1][0], b[0][1] + b[1][1]))
res = np.array(res, float)
res = res[np.argsort(-res[:, 0])]
print("%d targets, hop %d: invalid vertices per root and graph-row records they cost (D_inv) per target" % (NT, HOP))
for q in np.array_split(res, 4):
    print("n %6.0f..%6.0f | whole-graph table: invalid %4.1f%%  D_inv %8.0f | ball table: invalid %4.1f%%  D_inv %8.0f"
          % (q[:, 0].max(), q[:, 0].min(), 100 * q[:, 1].sum() / (2 * q[:, 0].sum()), q[:, 2].mean(),
             100 * q[:, 3].sum() / (2 * q[:, 0].sum()), q[:, 4].mean()))
print("all (mean n %.0f) | whole-graph table: invalid %4.1f%%  D_inv %8.0f | ball table: invalid %4.1f%%  D_inv %8.0f"
      % (res[:, 0].mean(), 100 * res[:, 1].sum() / (2 * res[:, 0].sum()), res[:, 2].mean(),
         100 * res[:, 3].sum() / (2 * res[:, 0].sum()), res[:, 4].mean()))
