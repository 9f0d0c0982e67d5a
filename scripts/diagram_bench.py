"""Diagram output vs image output on the benchmark's seeded configurations: tlc_vicinity_pi_dev and
tlc_vicinity_diagrams_dev alternate on the same targets in one process.  Legs per configuration: the image call, the
diagrams with TLC_F_ASC_ONLY (PD_up + [min,max], non-extended configurations only), the full PD_zero and, where the
configuration is extended, PD_zero + PD_one.  Reports targets/s, pairs per target and bytes written per call, with the
GPU's name and power limit read in the same run, as JSON under --out.

    python scripts/diagram_bench.py --out profiles/diagrams [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tlc-gnn_b200")]

# (key, workload, hop, extended, mode, negatives, batch): bench.py's headline and secondary configurations
CONFIGS = [
    ("headline_computers_hop2", "computers", 2, 0, "edge", 0, 4096),
    ("C1_cora_hop2_ext", "cora", 2, 1, "edge", 0, 5278),
    ("C2_pubmed_hop2", "pubmed", 2, 0, "edge", 0, 8192),
    ("C3_computers_hop1_ext", "computers", 1, 1, "edge", 0, 8192),
    ("C3_computers_hop2_ext", "computers", 2, 1, "edge", 0, 256),
    ("C4_ppi24_node_ext", "ppi", 2, 1, "node", 0, 4096),
    ("C5_collab_neg_hop2", "collab", 2, 0, "edge", 1, 16384),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory (diagram_bench.json is written there)")
    ap.add_argument("--reps", type=int, default=5, help="timed calls per leg (alternating with the other legs)")
    ap.add_argument("--only", default=None, help="comma-separated configuration keys")
    args = ap.parse_args()
    import torch
    import bench
    from tlc_b200 import _lib as L
    from tlc_b200 import api

    dev = torch.device("cuda", 0)
    result = dict(gpu=gpu_info(), reps=args.reps, torch=torch.__version__, configs={})
    for key, wl, hop, ext, mode, negatives, batch in CONFIGS:
        if args.only and key not in args.only.split(","):
            continue
        c, labels, tt, csr, perm = bench.make_workload(wl, mode, negatives)
        g = api.VicinityGraph(*csr, device=0)
        fl = L.F_NORM | (L.F_EXTENDED if ext else 0)
        if mode == "node":
            fl |= L.F_KEEP_ZERO | L.F_NORM_EPS
        m = L.MODE_NODE if mode == "node" else L.MODE_EDGE
        E = min(batch, len(perm))
        legs = [("image", None)]
        if not ext:
            legs.append(("diagrams_asc_only", fl | L.F_ASC_ONLY))
        legs.append(("diagrams_pd_zero", fl & ~L.F_EXTENDED))
        if ext:
            legs.append(("diagrams_extended", fl))
        pi = torch.zeros((E, 25), dtype=torch.float64, device=dev)
        st = torch.zeros(E, dtype=torch.uint8, device=dev)
        times = {name: [] for name, _ in legs}
        stats = {}
        for rep in range(args.reps + 1):  # rep 0: warm-up (tables, arena, capacity guess)
            tg = torch.from_numpy(bench.batch_targets(tt, perm, rep, 0, 1, E)).to(dev)
            for name, leg_fl in legs:
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                if leg_fl is None:
                    g.vicinity_pi_dev(tg, pi, out_status=st, hop=hop, mode=m, flags=fl)
                    torch.cuda.synchronize(dev)
                    out = None
                else:
                    out = g.vicinity_diagrams_dev(tg, hop=hop, mode=m, flags=leg_fl, want_pi=True)
                    torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
                if rep == 0:
                    continue
                times[name].append(dt)
                if out is not None:
                    P = int(out["poff"][-1])
                    stats[name] = dict(pairs_per_target=P / E, bytes_written=P * 25 + (E + 1) * 8 + E * 25 * 8 + E)
        res = dict(workload=wl, hop=hop, extended=ext, mode=mode, negatives=negatives, targets=E, legs={})
        for name, _ in legs:
            ts = np.array(times[name])
            res["legs"][name] = dict(median_s=float(np.median(ts)), min_s=float(ts.min()), targets_per_s=E / float(np.median(ts)),
                                     **stats.get(name, dict(bytes_written=E * 25 * 8 + E)))
        img = res["legs"]["image"]["median_s"]
        for name, _ in legs[1:]:
            res["legs"][name]["time_vs_image"] = res["legs"][name]["median_s"] / img
        result["configs"][key] = res
        print(key, json.dumps(res["legs"]), flush=True)
        g.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "diagram_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
