"""The batch imager of device-resident diagrams (api.persistence_images: tlc_pimg_batch_dev + tlc_pimg_batch_grad_dev) vs
the vectorised pure-torch restatement of the same image (tests/test_pimg_batch_abi.py, pinned there against the oracle),
on the same GPU.  Diagram sets: vicinity_diagrams_dev on bench.py's seeded workloads -- headline PD_zero (Computers hop 2,
4096 targets), C1 Cora hop 2 extended (5278), C4 PPI x24 node extended with the KD flags and the KD image mask (4096) --
plus 10^5 one-point diagrams.  Legs: forward, and forward + backward (grad_out uniform in [0, 1)), of each
implementation; the four legs alternate in one process after a warm-up, each timed over rounds of calls that end in a
device synchronise, at least --seconds per leg in all.  Reports ms per call, points/s, and max |delta| of the rows and of
both gradients against the restatement, with the GPU's name and power limit read in the same run, as JSON under --out.

    python scripts/pimg_grad_bench.py --out profiles/pimg_grad [--seconds 1.0] [--rounds 5]
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

# (key, workload, hop, extended, mode, batch): bench.py's configurations whose diagrams are imaged
SETS = [
    ("headline_computers_hop2_pd_zero", "computers", 2, 0, "edge", 4096),
    ("C1_cora_hop2_ext", "cora", 2, 1, "edge", 5278),
    ("C4_ppi24_node_ext_kd", "ppi", 2, 1, "node", 4096),
]


def diagram_sets(torch, L, api, bench, dev):
    for key, wl, hop, ext, mode, batch in SETS:
        c, labels, tt, csr, perm = bench.make_workload(wl, mode, 0)
        g = api.VicinityGraph(*csr, device=0)
        fl = L.F_NORM | (L.F_EXTENDED if ext else 0)
        if mode == "node":
            fl |= L.F_KEEP_ZERO | L.F_NORM_EPS
        E = min(batch, len(perm))
        tg = torch.from_numpy(bench.batch_targets(tt, perm, 0, 0, 1, E)).to(dev)
        d = g.vicinity_diagrams_dev(tg, hop=hop, mode=L.MODE_NODE if mode == "node" else L.MODE_EDGE, flags=fl)
        torch.cuda.synchronize(dev)
        g.close()
        yield key, (d["poff"], d["birth"], d["death"], d["kind"], L.default_img_mask(bool(ext), mode == "node"))
    rng = np.random.default_rng(0)
    n = 100000
    b = rng.uniform(0, 1, n)
    yield "single_point_1e5", (torch.arange(n + 1, dtype=torch.int64, device=dev),
                               torch.from_numpy(b).to(dev), torch.from_numpy(b + rng.uniform(0, 1, n)).to(dev), None, None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory (pimg_grad_bench.json is written there)")
    ap.add_argument("--seconds", type=float, default=1.0, help="least timed time per leg and set")
    ap.add_argument("--rounds", type=int, default=5, help="timed rounds per leg (the legs alternate round by round)")
    ap.add_argument("--resolution", type=int, default=5)
    args = ap.parse_args()
    import torch
    import bench
    from diagram_bench import gpu_info
    from test_pimg_batch_abi import torch_images
    from tlc_b200 import _lib as L
    from tlc_b200 import api

    dev = torch.device("cuda", 0)
    res = args.resolution
    result = dict(gpu=gpu_info(), resolution=res, seconds=args.seconds, rounds=args.rounds, torch=torch.__version__,
                  sets={})
    for key, (poff, birth, death, kind, mask) in diagram_sets(torch, L, api, bench, dev):
        D, P = poff.numel() - 1, int(poff[-1] - poff[0])
        G = torch.rand((D, res * res), dtype=torch.float64, device=dev)
        impls = dict(op=api.persistence_images, torch=torch_images)

        def run(impl, backward):
            if not backward:
                with torch.no_grad():
                    return impls[impl](poff, birth, death, kind, mask, res), None
            b, d = birth.detach().requires_grad_(True), death.detach().requires_grad_(True)
            out = impls[impl](poff, b, d, kind, mask, res)
            return out, torch.autograd.grad(out, (b, d), G)

        legs = [(impl + ("_fwd_bwd" if bw else "_fwd"), impl, bw) for impl in ("op", "torch") for bw in (0, 1)]
        calls = {}
        for name, impl, bw in legs:  # warm-up, then calls per round so that the rounds add up to --seconds
            run(impl, bw)
            n = 1
            while True:
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                for _ in range(n):
                    run(impl, bw)
                torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
                if dt > 0.05:
                    break
                n *= 2
            calls[name] = max(1, int(np.ceil(1.2 * args.seconds / args.rounds / (dt / n))))
        per_call = {name: [] for name, _, _ in legs}
        for _ in range(args.rounds):
            for name, impl, bw in legs:
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                for _ in range(calls[name]):
                    run(impl, bw)
                torch.cuda.synchronize(dev)
                per_call[name].append((time.perf_counter() - t0) / calls[name])
        out_op, (gb_op, gd_op) = run("op", 1)
        out_ref, (gb_ref, gd_ref) = run("torch", 1)
        out_op, out_ref = out_op.detach(), out_ref.detach()
        agree = dict(max_abs_delta_rows=float((out_op - out_ref).abs().max()),
                     max_abs_delta_grad_birth=float((gb_op - gb_ref).abs().max()),
                     max_abs_delta_grad_death=float((gd_op - gd_ref).abs().max()),
                     max_abs_rows=float(out_ref.abs().max()), max_abs_grad_birth=float(gb_ref.abs().max()),
                     max_abs_grad_death=float(gd_ref.abs().max()))
        entry = dict(diagrams=D, points=P, points_per_diagram=P / max(D, 1), legs={}, agreement=agree)
        for name, _, _ in legs:
            ts = np.array(per_call[name])
            med = float(np.median(ts))
            entry["legs"][name] = dict(ms_per_call=1e3 * med, min_ms=1e3 * float(ts.min()), points_per_s=P / med,
                                       calls_timed=calls[name] * args.rounds, timed_s=float(ts.sum() * calls[name]))
        for leg in ("fwd", "fwd_bwd"):
            entry["torch_over_op_" + leg] = entry["legs"]["torch_" + leg]["ms_per_call"] / entry["legs"]["op_" + leg]["ms_per_call"]
        result["sets"][key] = entry
        print(key, json.dumps(entry), flush=True)
        del out_op, out_ref, gb_op, gd_op, gb_ref, gd_ref
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "pimg_grad_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
