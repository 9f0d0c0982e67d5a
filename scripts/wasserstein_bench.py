"""Exact Wasserstein distances between device-resident diagrams (api.wasserstein_distances: tlc_wasserstein_batch_dev +
tlc_wasserstein_batch_grad_dev) against scipy's linear_sum_assignment on the host, on bench.py's seeded diagram sets
from vicinity_diagrams_dev: headline PD_zero (Computers hop 2) and C1 Cora hop 2 extended.  C4 PPI x24 node extended
is not a set here: one of its pairs (17.0 k against 29.5 k points) did not finish within 400 s (DESIGN.md section 7).
Pair t compares the diagram of target t with that of target
t + D/2 (two slices of one poff, so no copy).  Legs: op forward, op forward + backward (grad_out = 1), and the host
reference: the device-to-host copy of the diagrams, then the N x N expansion of tests/test_wasserstein_abi.py solved by
linear_sum_assignment, one pair per task over all host cores.  Order 1, internal_p inf (gudhi's defaults).  Reports ms
per call (median of --rounds), the max relative difference of the distances, and the GPU's name and power limit read
in the same run, as JSON under --out.

    python scripts/wasserstein_bench.py --out profiles [--rounds 3]
"""
import argparse
import json
import math
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tlc-gnn_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"),
                os.path.join(ROOT, "scripts")]

# (key, workload, hop, extended, mode, targets, host reference): bench.py's configurations
SETS = [
    ("headline_computers_hop2_pd_zero", "computers", 2, 0, "edge", 512, True),
    ("C1_cora_hop2_ext", "cora", 2, 1, "edge", 5278, True),
]


def _host_pair(args):
    from test_wasserstein_abi import ref_distance
    X, Y = args
    return ref_distance(X, Y, 1.0, math.inf)[0]


def diagram_set(torch, L, api, bench, dev, wl, hop, ext, mode, targets):
    c, labels, tt, csr, perm = bench.make_workload(wl, mode, 0)
    g = api.VicinityGraph(*csr, device=0)
    fl = L.F_NORM | (L.F_EXTENDED if ext else 0)
    if mode == "node":
        fl |= L.F_KEEP_ZERO | L.F_NORM_EPS
    E = min(targets, len(perm)) // 2 * 2
    tg = torch.from_numpy(bench.batch_targets(tt, perm, 0, 0, 1, E)).to(dev)
    d = g.vicinity_diagrams_dev(tg, hop=hop, mode=L.MODE_NODE if mode == "node" else L.MODE_EDGE, flags=fl)
    torch.cuda.synchronize(dev)
    g.close()
    h = E // 2
    return d["poff"][:h + 1].contiguous(), d["poff"][h:].contiguous(), d["birth"], d["death"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory (wasserstein_bench.json is written there)")
    ap.add_argument("--rounds", type=int, default=3, help="timed calls per leg (the legs alternate round by round)")
    ap.add_argument("--only", default=None, help="comma-separated set keys")
    args = ap.parse_args()
    import torch
    import bench
    from diagram_bench import gpu_info
    from tlc_b200 import _lib as L
    from tlc_b200 import api

    dev = torch.device("cuda", 0)
    cores = os.cpu_count() or 1
    pool = mp.get_context("spawn").Pool(cores)
    result = dict(gpu=gpu_info(), order=1.0, internal_p="inf", rounds=args.rounds, host_cores=cores,
                  torch=torch.__version__, sets={})
    try:
        for key, wl, hop, ext, mode, targets, host_ref in SETS:
            if args.only and key not in args.only.split(","):
                continue
            px, py, birth, death = diagram_set(torch, L, api, bench, dev, wl, hop, ext, mode, targets)
            D = px.numel() - 1
            nx = (px[1:] - px[:-1]).cpu().numpy()
            ny = (py[1:] - py[:-1]).cpu().numpy()
            G = torch.ones(D, dtype=torch.float64, device=dev)

            def op(backward):
                if not backward:
                    return api.wasserstein_distances(px, birth, death, py, birth, death)
                b, d = birth.detach().requires_grad_(True), death.detach().requires_grad_(True)
                out = api.wasserstein_distances(px, b, d, py, b, d)
                torch.autograd.grad(out, (b, d), G)
                return out.detach()

            def host():
                t0 = time.perf_counter()
                pxh, pyh, bh, dh = px.cpu().numpy(), py.cpu().numpy(), birth.cpu().numpy(), death.cpu().numpy()
                t_copy = time.perf_counter() - t0
                tasks = [(np.stack([bh[pxh[t]:pxh[t + 1]], dh[pxh[t]:pxh[t + 1]]], 1),
                          np.stack([bh[pyh[t]:pyh[t + 1]], dh[pyh[t]:pyh[t + 1]]], 1)) for t in range(D)]
                return np.array(pool.map(_host_pair, tasks, chunksize=1)), t_copy

            legs = ["op_fwd", "op_fwd_bwd"] + (["host_lsa"] if host_ref else [])
            times = {k: [] for k in legs}
            op(False)
            op(True)  # warm-up
            ref = None
            for _ in range(args.rounds):
                for leg in legs:
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    if leg == "host_lsa":
                        ref, _ = host()
                    else:
                        op(leg == "op_fwd_bwd")
                        torch.cuda.synchronize(dev)
                    times[leg].append(time.perf_counter() - t0)
            dist = op(False).cpu().numpy()
            entry = dict(pairs=D, points_x=int(nx.sum()), points_y=int(ny.sum()),
                         mean_points_per_diagram=float((nx.sum() + ny.sum()) / max(2 * D, 1)),
                         max_points_per_diagram=int(max(nx.max(initial=0), ny.max(initial=0))), legs={})
            for leg in legs:
                entry["legs"][leg] = dict(ms_per_call=1e3 * float(np.median(times[leg])),
                                          min_ms=1e3 * float(np.min(times[leg])), calls=len(times[leg]))
            if ref is not None:
                den = np.where(ref > 0, ref, 1.0)
                entry["max_rel_delta_vs_host"] = float(np.max(np.abs(dist - ref) / den, initial=0.0))
                entry["host_over_op_fwd"] = entry["legs"]["host_lsa"]["ms_per_call"] / entry["legs"]["op_fwd"]["ms_per_call"]
                entry["host_over_op_fwd_bwd"] = (entry["legs"]["host_lsa"]["ms_per_call"]
                                                 / entry["legs"]["op_fwd_bwd"]["ms_per_call"])
            entry["nan_pairs"] = int(np.isnan(dist).sum())
            result["sets"][key] = entry
            print(key, json.dumps(entry), flush=True)
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "wasserstein_bench.json"), "w") as f:  # after every set: a cut run keeps it
                json.dump(result, f, indent=1)
            del px, py, birth, death
            torch.cuda.empty_cache()
    finally:
        pool.terminate()
        pool.join()


if __name__ == "__main__":
    main()
