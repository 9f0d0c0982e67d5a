"""Persistence diagrams of caller-supplied graph batches (api.GraphBatch: tlc_graph_batch_diagrams_dev +
tlc_graph_batch_grad_dev) on seeded graph-classification-shaped batches: kernel 9's fused route against the staged
kernels 2 + 3 (+ 3b) forced by no_small, and against the C oracle (tlo_run_one_fval per graph, one thread per graph over
16 host threads).  The workloads are the dataloader batches of Knowledge_Distillation/data_utils_GC.py:
  zinc     : 4096 molecules of 15-31 atoms (~23), a spanning tree plus 0-3 ring bonds (~25 edges)
  proteins : 4096 graphs of 25-55 vertices (~40) with ~1.9 edges per vertex (~75)
each with and without extended persistence, and a staged-side set of 16 graphs of 5000 vertices / 7500 edges, which no
fused class takes.  Legs, alternated round by round: forward, and forward + backward (the sum of birth and death as the
loss), each timed with CUDA events over --calls calls per round, median of --rounds rounds; the oracle leg runs once.
Every set also checks that both routes give the same bits.  Writes graph_diagrams_bench.json with the GPU's name and
power limit, read in the same run, under --out.

    python scripts/graph_diagrams_bench.py --out profiles [--rounds 5 --calls 20]
"""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tlc-gnn_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "scripts")]


def random_graph(rng, n, extra):
    """a connected graph: a random spanning tree plus `extra` further edges, canonical order"""
    es = set()
    for i in range(1, n):
        j = int(rng.integers(0, i))
        es.add((j, i))
    while len(es) < n - 1 + extra:
        a, b = (int(x) for x in rng.integers(0, n, 2))
        if a != b:
            es.add((min(a, b), max(a, b)))
    return np.array(sorted(es), np.int64).reshape(-1, 2)


def workload(name, seed=0):
    rng = np.random.default_rng(seed)
    if name == "zinc":
        graphs = [random_graph(rng, n, int(rng.integers(0, 4))) for n in rng.integers(15, 32, 4096)]
    elif name == "proteins":
        graphs = [random_graph(rng, n, int(round(0.9 * n))) for n in rng.integers(25, 56, 4096)]
    else:  # staged
        graphs = [random_graph(rng, 5000, 2501) for _ in range(16)]
    sizes = [int(e.max()) + 1 if len(e) else 1 for e in graphs]
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    ei = np.concatenate([e + ptr[t] for t, e in enumerate(graphs)], 0).T
    f = rng.random(int(ptr[-1]))
    return ptr, ei, f, graphs


SETS = [("zinc", "zinc", False), ("zinc_ext", "zinc", True), ("proteins", "proteins", False),
        ("proteins_ext", "proteins", True), ("staged_16x5000", "staged", False), ("staged_16x5000_ext", "staged", True)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory (graph_diagrams_bench.json is written there)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20, help="calls per timed round")
    ap.add_argument("--threads", type=int, default=16, help="host threads of the oracle leg")
    args = ap.parse_args()
    import torch
    import oracle as orc
    from diagram_bench import gpu_info
    from tlc_b200 import api
    from tlc_b200 import graphgen as gg

    dev = torch.device("cuda", 0)
    result = dict(gpu=gpu_info(), rounds=args.rounds, calls=args.calls, oracle_threads=args.threads,
                  torch=torch.__version__, sets={})
    for key, wl, ext in SETS:
        ptr, ei, f, graphs = workload(wl)
        gb = api.GraphBatch(ptr, ei, device=0)
        x = torch.from_numpy(f).to(dev)
        xg = x.clone().requires_grad_(True)

        def fwd(ns):
            return gb.diagrams(x, extended=ext, no_small=ns)

        def fwd_bwd(ns):
            d = gb.diagrams(xg, extended=ext, no_small=ns)
            (d["birth"].sum() + d["death"].sum()).backward()
            xg.grad = None

        legs = {"fused_fwd": lambda: fwd(False), "staged_fwd": lambda: fwd(True),
                "fused_fwd_bwd": lambda: fwd_bwd(False), "staged_fwd_bwd": lambda: fwd_bwd(True)}
        for fn in legs.values():  # warm-up: every shape of the timed window
            fn()
        times = {k: [] for k in legs}
        for _ in range(args.rounds):
            for k, fn in legs.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.calls):
                    fn()
                b.record()
                b.synchronize()
                times[k].append(a.elapsed_time(b) / args.calls)
        d0, d1 = fwd(False), fwd(True)
        torch.cuda.synchronize()
        P = int(d0["poff"][-1])
        same = all(torch.equal(d0[k][:P] if k not in ("poff", "status") else d0[k],
                               d1[k][:P] if k not in ("poff", "status") else d1[k]) for k in d0)
        # the C oracle: one OracleGraph per graph, built before the clock starts
        ogs = []
        for e in graphs:
            n = int(e.max()) + 1 if len(e) else 1
            ogs.append((n, orc.OracleGraph(*gg.build_csr(n, e, np.zeros(len(e))))))
        fl = orc.F_EXTENDED if ext else 0

        def one(t):
            n, og = ogs[t]
            v0 = int(ptr[t])
            return og.run_one(0, 0, hop=n, mode=orc.MODE_NODE, flags=fl, fval=f[v0:v0 + n])["status"]

        with ThreadPoolExecutor(args.threads) as pool:
            t0 = time.perf_counter()
            st = list(pool.map(one, range(len(graphs))))
            oracle_ms = (time.perf_counter() - t0) * 1e3
        ok = bool(np.array_equal(np.array(st, np.uint8), d0["status"].cpu().numpy()))
        med = {k: float(np.median(v)) for k, v in times.items()}
        result["sets"][key] = dict(
            graphs=len(graphs), vertices=int(ptr[-1]), edges=int(ei.shape[1]), extended=ext, pairs=P,
            ms=med, ms_all={k: [round(t, 4) for t in v] for k, v in times.items()}, oracle_ms=oracle_ms,
            staged_over_fused_fwd=med["staged_fwd"] / med["fused_fwd"],
            staged_over_fused_fwd_bwd=med["staged_fwd_bwd"] / med["fused_fwd_bwd"],
            oracle_over_fused_fwd=oracle_ms / med["fused_fwd"], routes_identical=same, statuses_match_oracle=ok)
        print(key, json.dumps(result["sets"][key]["ms"]), "oracle %.2f ms" % oracle_ms, "same" if same else "DIFFER",
              flush=True)
        gb.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "graph_diagrams_bench.json"), "w") as fh:
        json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
