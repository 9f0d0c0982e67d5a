import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tlc-gnn_b200"))
import numpy as np, bench
from tlc_b200 import _lib as L, api
c, labels, ne, csr, perm = bench.make_workload("computers")
g = api.VicinityGraph(*csr, device=0)
for s in range(4):
    tg = bench.batch_targets(ne, perm, s, 0, 1, 2048)
    t0 = time.perf_counter()
    g.vicinity_pi(tg, hop=2, flags=L.F_NORM)
    dt = time.perf_counter() - t0
    cn = g.last_counts()
    print("step", s, "ms %.1f" % (1e3*dt), "sum_n", cn["sum_n"], "sum_m(=invalid count in the debug build)", cn["sum_m"], "table", cn["table_route"], flush=True)
g.close()
