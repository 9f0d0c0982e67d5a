"""Vicinities in graph-batch layout on the device (VicinityGraph.vicinity_batch_dev: tlc_vicinity_batch_dev, kernel 10)
against the route that existed before it, on bench.py's seeded workloads: C1 Cora hop 2 (edge mode), C2 PubMed hop 2,
C4 PPI x24 node mode with the generator's normalisation (512 targets: tlc_vicinity_detail copies every intermediate of
the whole batch to the host, and 4096 PPI vicinities would not fit its budget), and the headline Computers hop 2 at 512
targets (large vicinities).  Legs, alternated round by round after a warm-up, median over --rounds:
  structure      vicinity_batch_dev(fval=False): ptr, eptr, vert, edge_index, status
  structure_fval vicinity_batch_dev(): the same + the filtration values
  host_route     the same tensors on the device the old way: vicinity_detail, per-target assembly (the NaN rule
                 included) on the host, upload
  diagrams_dev   vicinity_diagrams_dev on the same targets (context: the whole pipeline to diagrams)
  step_dev       one learnable step: vicinity_batch_dev -> GraphBatch.from_device -> diagrams -> persistence_images ->
                 backward
  step_host      the same step from host_route's tensors and the host GraphBatch(ptr, edge_index)
  create_dev     GraphBatch.from_device alone on structure_fval's output
Also: bytes the call writes (offsets, vertices, edges, values, statuses) over its time against 7.7 TB/s (the HBM3e
figure of NVIDIA's B200 data sheet), and a byte-for-byte check that structure_fval and host_route give identical tensors.
Reads the GPU's name, power limit and max SM clock in the same run.  Writes JSON under --out.

    python scripts/vicinity_batch_bench.py --out profiles [--rounds 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tlc-gnn_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"),
                os.path.join(ROOT, "scripts")]

HBM_TBS = 7.7
# (key, workload, hop, mode, targets)
SETS = [
    ("C1_cora_hop2", "cora", 2, "edge", 5278),
    ("C2_pubmed_hop2", "pubmed", 2, "edge", 8192),
    ("C4_ppi24_node", "ppi", 2, "node", 512),
    ("headline_computers_hop2", "computers", 2, "edge", 512),
]


def host_route(torch, L, g, tgh, hop, mode, flags, dev):
    """today's route to the graph-batch tensors: every intermediate to the host, per-target assembly, upload"""
    det = g.vicinity_detail(tgh, hop=hop, mode=mode, flags=flags)
    E = len(tgh)
    verts, elo, ehi, fv, n, m = [], [], [], [], np.zeros(E, np.int64), np.zeros(E, np.int64)
    for i in range(E):
        a = g.per_target(det, i)
        n[i], m[i] = a["n"], a["m"]
        verts.append(a["vert"])
        elo.append(a["elo"])
        ehi.append(a["ehi"])
        fv.append(a["fval"] if det["status"][i] <= L.ST_TRIVIAL else np.full(a["n"], np.nan))
    ptr = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
    eptr = np.concatenate([[0], np.cumsum(m)]).astype(np.int64)
    first = np.repeat(ptr[:-1], m)
    ei = np.stack([np.concatenate(elo) + first, np.concatenate(ehi) + first]).astype(np.int32)
    out = dict(ptr=ptr, eptr=eptr, vert=np.concatenate(verts).astype(np.int32), edge_index=ei, fval=np.concatenate(fv),
               status=det["status"])
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in out.items()}, (ptr, ei)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory (vicinity_batch_bench.json is written there)")
    ap.add_argument("--rounds", type=int, default=5, help="timed calls per leg (the legs alternate round by round)")
    ap.add_argument("--only", default=None, help="comma-separated set keys")
    args = ap.parse_args()
    import torch
    import bench
    from diagram_bench import gpu_info
    from tlc_b200 import _lib as L
    from tlc_b200 import api

    dev = torch.device("cuda", 0)
    result = dict(gpu=gpu_info(), rounds=args.rounds, hbm_tbs=HBM_TBS, torch=torch.__version__, sets={})
    for key, wl, hop, mode_name, targets in SETS:
        if args.only and key not in args.only.split(","):
            continue
        c, labels, tt, csr, perm = bench.make_workload(wl, mode_name, 0)
        g = api.VicinityGraph(*csr, device=0)
        mode = L.MODE_NODE if mode_name == "node" else L.MODE_EDGE
        flags = L.F_NORM | (L.F_NORM_EPS if mode_name == "node" else 0)
        E = min(targets, len(perm))
        tgh = np.ascontiguousarray(bench.batch_targets(tt, perm, 0, 0, 1, E), dtype=np.int32)
        tg = torch.from_numpy(tgh).to(dev)
        keep = {}

        def step(ptr, ei, f0, host_gb):
            gb = api.GraphBatch(*host_gb) if host_gb is not None else api.GraphBatch.from_device(ptr, ei)
            f = f0.clone().requires_grad_(True)
            d = gb.diagrams(f)
            api.persistence_images(d["poff"], d["birth"], d["death"]).sum().backward()
            torch.cuda.synchronize(dev)
            gb.close()
            return f.grad

        def leg(name):
            if name == "structure":
                return g.vicinity_batch_dev(tg, hop=hop, mode=mode, flags=flags, fval=False)
            if name == "structure_fval":
                keep["dev"] = g.vicinity_batch_dev(tg, hop=hop, mode=mode, flags=flags)
                return keep["dev"]
            if name == "host_route":
                keep["host"], keep["host_np"] = host_route(torch, L, g, tgh, hop, mode, flags, dev)
                return keep["host"]
            if name == "diagrams_dev":
                return g.vicinity_diagrams_dev(tg, hop=hop, mode=mode, flags=flags)
            if name == "step_dev":
                vb = g.vicinity_batch_dev(tg, hop=hop, mode=mode, flags=flags)
                return step(vb["ptr"], vb["edge_index"], vb["fval"], None)
            if name == "step_host":
                h, hn = host_route(torch, L, g, tgh, hop, mode, flags, dev)
                return step(None, None, h["fval"], hn)
            if name == "create_dev":
                gb = api.GraphBatch.from_device(keep["dev"]["ptr"], keep["dev"]["edge_index"])
                gb.close()
                return None
            raise KeyError(name)

        legs = ["structure", "structure_fval", "host_route", "diagrams_dev", "step_dev", "step_host", "create_dev"]
        times = {k: [] for k in legs}
        for name in legs:  # warm-up: every shape the timed rounds use
            leg(name)
        torch.cuda.synchronize(dev)
        for _ in range(args.rounds):
            for name in legs:
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                leg(name)
                torch.cuda.synchronize(dev)
                times[name].append(time.perf_counter() - t0)
        a, b = keep["dev"], keep["host"]
        same = all(np.array_equal(a[k].cpu().numpy().view(np.uint8), b[k].cpu().numpy().view(np.uint8))
                   for k in ("ptr", "eptr", "vert", "edge_index", "fval"))
        ga = step(a["ptr"], a["edge_index"], a["fval"], None).cpu().numpy()
        gh = step(None, None, b["fval"], keep["host_np"]).cpu().numpy()
        V, M = int(a["vert"].numel()), int(a["edge_index"].shape[1])
        st = a["status"].cpu().numpy()
        written = 2 * (E + 1) * 8 + V * 4 + 2 * M * 4 + V * 8 + E
        entry = dict(targets=E, vertices=V, edges=M, live=int((st <= L.ST_TRIVIAL).sum()),
                     legs2_3_identical_bytes=bool(same),
                     step_grads_identical=bool(np.array_equal(np.nan_to_num(ga).view(np.int64),
                                                               np.nan_to_num(gh).view(np.int64))),
                     bytes_written=written, legs={})
        for name in legs:
            entry["legs"][name] = dict(ms=1e3 * float(np.median(times[name])), min_ms=1e3 * float(np.min(times[name])),
                                       calls=len(times[name]))
        ms2 = entry["legs"]["structure_fval"]["ms"]
        entry["structure_fval_hbm_share"] = written / (ms2 * 1e-3) / (HBM_TBS * 1e12)
        entry["host_route_over_structure_fval"] = entry["legs"]["host_route"]["ms"] / ms2
        entry["step_host_over_step_dev"] = entry["legs"]["step_host"]["ms"] / entry["legs"]["step_dev"]["ms"]
        result["sets"][key] = entry
        print(key, json.dumps(entry), flush=True)
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "vicinity_batch_bench.json"), "w") as f:  # after every set: a cut run keeps it
            json.dump(result, f, indent=1)
        g.close()
        del keep
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
