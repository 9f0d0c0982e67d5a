#!/usr/bin/env python
"""bench.py -- vicinity PDs + persistence images per second (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # CUDA path (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy

Workload (config.workload): Computers-shaped synthetic graph (13,752 nodes / 245,861 edges, seeded
Chung-Lu, curvature on a 1/1024 grid), target = graph edges, 2-hop vicinity, descriptor 'sum',
norm=True, 5x5 image -- BASELINE.json configs[2], the configuration the north_star target is quoted on.
One step = one pass of the hot path over a batch of `--batch` targets PER GPU (default 4096: the reference hands ALL
edges of a dataset to one call; measured on B200: 1024 per step -> 186 k, 4096 -> 217 k, 8192 -> 222 k targets/s,
larger batches amortise the tail waves of the per-vicinity CTAs) (weak scaling: every
rank takes its own disjoint batch of a seeded permutation of the edge list; a new batch every step, so
nothing is reused between steps and the per-step working set (GBs of per-vicinity arrays) >> L2).

value : targets/s, inputs (target ids) resident in HBM, CUDA events on the library's stream around the
        K timed steps, max over ranks.  N > 1 adds the NCCL all-gather of the fp32 image rows.
e2e   : the same through the reference-facing call (sg2dgm.riccidist2dgm.graph2pi.get_pimg_for_all_edges:
        host target list in, float64 pi_sg on the host out), host<->device copies inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tlc-gnn_b200"))

import numpy as np  # noqa: E402

METRIC = "vicinity_pd_pi_per_sec"
UNIT = "targets/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("TLC_BENCH_BATCH", "4096")))
    ap.add_argument("--workload", default=os.environ.get("TLC_BENCH_WORKLOAD", "computers"))
    ap.add_argument("--hop", type=int, default=2)
    ap.add_argument("--extended", type=int, default=int(os.environ.get("TLC_BENCH_EXTENDED", "0")))
    ap.add_argument("--mode", default="edge", choices=["edge", "node"],
                    help="node: PDGNN node-centred vicinities with the KD flags (Knowledge_Distillation/data_utils_NC.py shape)")
    ap.add_argument("--negatives", type=int, default=0, help="append an equal number of seeded non-adjacent pairs (collab config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--scaling", default=os.environ.get("TLC_BENCH_SCALING", "weak"), choices=["weak", "strong"],
                    help="weak: --batch targets per GPU and step (default); strong: --batch targets per step in total, split over the GPUs")
    ap.add_argument("--exchange", default=os.environ.get("TLC_EXCHANGE", "peer"), choices=["peer", "nccl"],
                    help="N > 1: peer = rows stored straight into every rank's table over NVLink (tlc_vicinity_pi_exchange); "
                         "nccl = pad + NCCL all-gather + un-permute (torch.distributed)")
    ap.add_argument("--secondary", type=int, default=int(os.environ.get("TLC_BENCH_SECONDARY", "1")),
                    help="1: also measure the other BASELINE.json configurations (a few steps each) into the `secondary` object")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed step as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB in all): the inputs are seeded, so two builds can be compared output "
                         "for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl cuda)")
    return args


def make_workload(name, mode="edge", negatives=0):
    """-> (config, labels, target table int64[*, 2], csr, seeded permutation of the target table).
    edge mode: targets = the graph's edges (+ an equal number of seeded non-adjacent pairs with --negatives 1);
    node mode: targets = every node, as (u, u); the PPI shape stacks 24 graphs block-diagonally (BASELINE.json configs[3])."""
    from tlc_b200 import graphgen as gg
    c = gg.make_config(name, n_graphs=24 if (name == "ppi" and mode == "node") else 1)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    tt = ne
    if mode == "node":
        ids = np.arange(len(labels), dtype=np.int64)
        tt = np.stack([ids, ids], 1)
    elif negatives:
        rng = np.random.default_rng(200 + gg.SHAPES[name][0])
        N = len(labels)
        key = set((np.minimum(ne[:, 0], ne[:, 1]) * N + np.maximum(ne[:, 0], ne[:, 1])).tolist())
        neg = np.zeros((0, 2), np.int64)
        while len(neg) < len(ne):
            cand = rng.integers(0, N, size=(len(ne) - len(neg) + 1024, 2))
            k = np.minimum(cand[:, 0], cand[:, 1]) * N + np.maximum(cand[:, 0], cand[:, 1])
            ok = (cand[:, 0] != cand[:, 1]) & ~np.isin(k, np.fromiter(key, dtype=np.int64, count=len(key)))
            neg = np.concatenate([neg, cand[ok]])[:len(ne)]
        tt = np.concatenate([ne, neg])
    perm = np.random.default_rng(300 + gg.SHAPES[name][0]).permutation(len(tt))
    return c, labels, tt, csr, perm


def path_flags(args, M):
    """(flags, mode) of the C-ABI / oracle call (the two share the flag values)."""
    fl = M.F_NORM | (M.F_EXTENDED if args.extended else 0)
    if args.mode == "node":
        fl |= M.F_KEEP_ZERO | M.F_NORM_EPS
    return fl, (M.MODE_NODE if args.mode == "node" else M.MODE_EDGE)


def batch_targets(ne, perm, step, rank, world, batch):
    """disjoint per (step, rank) slices of a seeded permutation of the edge list (wraps around)."""
    start = ((step * world + rank) * batch) % len(perm)
    idx = perm[np.arange(start, start + batch) % len(perm)]
    return np.ascontiguousarray(ne[idx].astype(np.int32))


DUMP_LIMIT = 64 << 20   # bytes of all dumped .npy files together


def dump_outputs(path, arrays, seed=0):
    """{name: array with one row per target} -> path/<name>.npy: float64 stays float64, everything else (fp32 rows,
    uint8 status) is written as float32.  If the rows do not fit DUMP_LIMIT, the same seeded sample of rows is kept
    in every array and the sampled row indices are written too (rows.npy)."""
    os.makedirs(path, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        out[name] = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
    rows = len(next(iter(out.values())))
    row_bytes = sum(a.nbytes for a in out.values()) / max(rows, 1)
    budget = DUMP_LIMIT - 4096 * (len(out) + 1)   # (.npy headers)
    if row_bytes * rows > budget:
        keep = np.sort(np.random.default_rng(seed).choice(rows, int(budget // (row_bytes + 8)), replace=False))
        out = {name: a[keep] for name, a in out.items()}
        out["rows"] = keep.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def config_dict(args, world):
    from tlc_b200 import graphgen as gg
    _, N, M, _, _ = gg.SHAPES[args.workload]
    kind = "edge vicinities" if args.mode == "edge" else "node-centred vicinities (PDGNN generator flags)"
    if args.mode == "node" and args.workload == "ppi":
        N, M = 24 * N, 24 * M
    return {"workload": "%s-shaped synthetic graph (%d nodes, %d edges), %d-hop %s%s, descriptor=sum, "
                        "norm=True, 5x5 image, extended_flag=%s" % (args.workload, N, M, args.hop, kind,
                                                                    " + equal negatives" if args.negatives else "",
                                                                    bool(args.extended)),
            "targets_per_gpu_per_step": args.batch if getattr(args, "scaling", "weak") == "weak" else args.batch / world,
            "global_targets_per_step": args.batch * world if getattr(args, "scaling", "weak") == "weak" else args.batch,
            "kappa": "U(-0.9,0.9) on a 1/1024 grid", "extended_flag": bool(args.extended),
            "l2": "new targets every step; per-step working set >> L2 (no flush needed)",
            "ball_cache": "warm: the k-hop ball bitmap of a node is expanded once per graph (13.7 k balls serve all 245,861 "
                          "targets) and the warm-up steps fill it; the timed steps reuse it, as every call after the first does",
            "sssp_tables": "warm where used (graph-row route, N <= 16384): the per-root shortest-path table rows (distance, tree "
                           "parent, path sum over the whole graph) are built once per root during the warm-up steps",
            "no_pair_certificate": "on (graph-row route): kernel 2v proves per target, from the step's own filtration values, that "
                                   "the ascending sweep emits no ordinary pair and then writes the essential pair without "
                                   "sorting (DESIGN.md section 5a); every target that fails the test is sorted and swept",
            "parallelism": "targets sharded over %d GPU(s), CSR replicated; N > 1: every rank stores its fp32 image rows "
                           "straight into every rank's table (peer stores over NVLink) or, --exchange nccl, NCCL all-gather" % world}


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  The timed region
    is tens of milliseconds, so NVML is polled in-process every ~2 ms (nvidia-smi -lms cannot sample that fast);
    falls back to a single `nvidia-smi --query-gpu` call when NVML is not importable."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        import threading
        self.idx = gpu_index
        self.sm, self.mask, self.max = [], 0, None
        self.h = None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu_index))
            self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
        self.th = threading.Thread(target=self._loop, daemon=True)

    def start(self):
        """begin polling (NVML was initialised in the constructor, outside the timed region: on rank 0 that takes
        ~10 ms, which the other ranks would otherwise spend waiting in the first all-gather of the timed region)"""
        self.th.start()

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v for v in vis.split(",") if v.strip() != ""]
        if ids and i < len(ids) and ids[i].strip().isdigit():
            return int(ids[i])
        return i

    def _sample(self):
        if self.h is not None:
            self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            try:
                self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                try:
                    self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass

    def _loop(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                pass
            self._stop.wait(0.002)

    def stop(self):
        try:
            self._sample()  # at least one sample taken before the region's closing synchronize returns
        except Exception:
            pass
        self._stop.set()
        self.th.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max, "reasons": []}
        if self.sm:
            out["sm_mhz"] = float(np.median(self.sm))
            out["samples"] = len(self.sm)
            out["reasons"] = sorted(k for k, bit in self.BAD.items() if self.mask & bit)
            out["source"] = "nvml, 2 ms poll during the timed region"
            return out
        try:  # no NVML: one nvidia-smi query (taken right after the region)
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            r = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=20).stdout.strip().split(", ")
            out["sm_mhz"], out["sm_max_mhz"] = float(r[0]), float(r[1])
            out["reasons"] = [n for n, v in zip(self.BAD, r[2:6]) if v.strip().lower().startswith("active")]
            out["samples"] = 1
            out["source"] = "nvidia-smi, one query at the end of the timed region"
        except Exception:
            pass
        return out


def cpu_baseline(csr, ne, perm, args, seconds, nthreads=0, offset=0):
    """the oracle port (oracle/tlc_oracle.c: the reference's algorithm restated in C, 2 shortest-path
    runs per vicinity instead of 2n) on the host cores, bounded sample of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    og = orc.OracleGraph(*csr)
    cores = orc.max_threads() if nthreads <= 0 else nthreads
    flags, omode = path_flags(args, orc)
    probe = batch_targets(ne, perm, 1000 + offset, 0, 1, max(2 * cores, 8))
    t0 = time.perf_counter()
    og.run_batch(probe, hop=args.hop, mode=omode, flags=flags, nthreads=cores)
    dt = time.perf_counter() - t0
    rate = len(probe) / dt
    sample = int(min(max(rate * seconds, len(probe)), 200000))
    tg = batch_targets(ne, perm, 2000 + offset, 0, 1, sample)
    t0 = time.perf_counter()
    r = og.run_batch(tg, hop=args.hop, mode=omode, flags=flags, nthreads=cores)
    dt = time.perf_counter() - t0
    return {"value": sample / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d targets of the same workload in %.1f s (C restatement of the reference algorithm, "
                      "pthreads over targets; fast-oracle filtration: 2 SSSP per vicinity)" % (sample, dt),
            "seconds": dt, "computed": int(r["cnt_compute"])}


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    c, labels, ne, csr, perm = make_workload(args.workload, args.mode, args.negatives)
    per_step = max(4.0, min(30.0, 150.0 / max(args.steps + args.warmup, 1)))
    res = []
    for s in range(args.warmup + args.steps):
        b = cpu_baseline(csr, ne, perm, args, per_step, offset=10 * s)
        if s >= args.warmup:
            res.append(b)
    value = float(np.mean([b["value"] for b in res]))
    secs = float(np.mean([b["seconds"] for b in res]))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * args.batch * world / value, "sample_ms": 1e3 * secs,
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": config_dict(args, world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": res[-1]["cores"], "kind": "port",
                             "sample": res[-1]["sample"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def stage_ms_of(g):
    """per-stage device ms of the last call: the staged kernels plus kernel S (the fused small-vicinity kernels)"""
    ms, _ = g.last_stage_ms()
    sm = g.last_small()
    ms["small"] = sm["ms_a"] + sm["ms_b"] + sm["ms_c"]
    ms["small_a"], ms["small_b"], ms["small_c"] = sm["ms_a"], sm["ms_b"], sm["ms_c"]
    return ms


# algorithmic bytes per target of each stage kernel (DESIGN.md section 4), from the vicinity's n, m and the
# SURVEY.md 8d compulsory read volume B_e of the extraction
def stage_alg_bytes(sum_n, sum_m, be_total, r2, live):
    adj = 24.0 * sum_m                       # induced adjacency, both directions: (4 B id + 8 B weight) * 2m
    return {"sizes": be_total - 16.0 * sum_m - 4.0 * r2 * live,      # expansion + induced-scan reads of the CSR
            "fill": (be_total - 4.0 * r2 * live) + adj + 16.0 * sum_n,  # same reads + kappa of the induced edges + adjacency write
            "filtration": 2.0 * adj + 40.0 * sum_n,                  # kernel 1b: every row read once per root + d1, d2, fval, tree
            "filtration_table": be_total,   # kernel 1t: charged the path's whole compulsory read volume B_e (SURVEY.md 8d), of which the
                                            # induced scan it replaces is > 90 % -- the table lookups avoid most of those reads
            "vorder": 48.0 * sum_n,                                  # sort keys/payload, rank tables, block table
            "sweep": 12.0 * sum_n,                                   # block table + rank order (+ rows only off the fast path)
            "image": 4.0 * r2 * live,
            "small": be_total}               # kernel S is the whole path: the compulsory bytes B_e of its targets


def measure_handoff(dev, peak_gbs):
    """SURVEY.md row N1 (kernel 5): gather + float64->float32 of the decoder's rows from the HBM-resident table, the
    shape of one training step of baselines/TLCGNN.py:35-53 on the Computers-shaped split (85 % of 245,861 positives +
    as many sampled negatives out of the train_neg slice).  HBM-bound: 12 B per element + 8 B per row index."""
    import torch
    from tlc_b200.table import PITable
    E = 2 * 245861
    tp = int(245861 * 0.85)
    tn = 245861
    table = PITable(torch.rand((E, 25), dtype=torch.float64, device=dev),
                    splits=[tp, tn, (E - tp - tn) // 4, (E - tp - tn) // 4, (E - tp - tn) // 4, E - tp - tn - 3 * ((E - tp - tn) // 4)])
    idx = torch.cat([torch.arange(tp, device=dev), tp + torch.randint(0, tn, (tp,), device=dev)])
    out = torch.empty((idx.numel(), 25), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > L2: the table is re-read from HBM every time
    ms = []
    for it in range(8):
        flush.fill_(it)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        table.gather(index=idx, out=out)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms[3:])) / 1e3
    nbytes = idx.numel() * (25 * 12 + 8)
    return {"kernel": "gather_rows (tlc_pi_gather)", "rows": int(idx.numel()), "ms": 1e3 * t, "rows_per_s": idx.numel() / t,
            "achieved_gbs": nbytes / 1e9 / t, "frac_of_hbm_peak": nbytes / 1e9 / t / peak_gbs,
            "note": "L2 flushed between repeats (256 MB write); time includes the call's own host sync"}


SECONDARY = [  # (key, BASELINE.json config it belongs to, bench arguments)
    ("C1_cora_hop2", "configs[0]", dict(workload="cora", hop=2, extended=0, mode="edge", negatives=0, batch=5278)),
    ("C1_cora_hop2_ext", "configs[0], extended_flag=True (the reference's shipped setting)", dict(workload="cora", hop=2, extended=1, mode="edge", negatives=0, batch=5278)),
    ("C2_pubmed_hop2", "configs[1]", dict(workload="pubmed", hop=2, extended=0, mode="edge", negatives=0, batch=8192)),
    ("C2_pubmed_hop2_ext", "configs[1], extended_flag=True", dict(workload="pubmed", hop=2, extended=1, mode="edge", negatives=0, batch=8192)),
    ("C3_computers_hop1_ext", "configs[2] at the reference's own hop for this dataset (baselines/TLCGNN.py:102), extended_flag=True",
     dict(workload="computers", hop=1, extended=1, mode="edge", negatives=0, batch=8192)),
    ("C3_computers_hop2_ext", "configs[2], extended_flag=True", dict(workload="computers", hop=2, extended=1, mode="edge", negatives=0, batch=256)),
    ("C4_ppi24_node_ext", "configs[3]", dict(workload="ppi", hop=2, extended=1, mode="node", negatives=0, batch=4096)),
    ("C5_collab_neg_hop2", "configs[4] (one GPU's share)", dict(workload="collab", hop=2, extended=0, mode="edge", negatives=1, batch=16384)),
]


def run_secondary(dev, local, peak, cache, steps=3, warmup=2, cpu_seconds=2.5, spot=64):
    """the other BASELINE.json configurations in the same run, each a short measurement (a few steps) with the same
    rules as the headline: device-timed value (inputs resident), e2e through the reference-facing call (host in / host
    out), the CPU port on a bounded sample, the dominant kernel with its roofline fraction, and an oracle spot check."""
    import torch
    from tlc_b200 import _lib as L
    from tlc_b200 import api
    import sg2dgm.riccidist2dgm as mirror
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    out = {}
    for key, what, kw in SECONDARY:
        a = argparse.Namespace(**kw)
        try:
            wkey = (a.workload, a.mode, a.negatives)
            if wkey not in cache:
                cache.clear()  # (one workload resident at a time)
                cache[wkey] = make_workload(a.workload, a.mode, a.negatives)
            c, labels, ne, csr, perm = cache[wkey]
            g = api.VicinityGraph(*csr, device=local)
            stream = torch.cuda.Stream(dev)
            flags, cmode = path_flags(a, L)
            B, r2 = a.batch, 25
            out_pi = torch.zeros((B, r2), dtype=torch.float64, device=dev)
            out_f32 = torch.zeros((B, r2), dtype=torch.float32, device=dev)
            out_st = torch.zeros((B,), dtype=torch.uint8, device=dev)
            batches = [torch.from_numpy(batch_targets(ne, perm, s0, 0, 1, B)).to(dev) for s0 in range(warmup + steps)]
            stage_acc, alg_bytes, sum_n, sum_m, live = {}, 0.0, 0, 0, 0
            with torch.cuda.stream(stream):
                g.set_stream(stream.cuda_stream)
                for s0 in range(warmup):
                    g.vicinity_pi_dev(batches[s0], out_pi, out_f32, out_st, hop=a.hop, mode=cmode, flags=flags)
                torch.cuda.synchronize()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for s0 in range(warmup, warmup + steps):
                    g.vicinity_pi_dev(batches[s0], out_pi, out_f32, out_st, hop=a.hop, mode=cmode, flags=flags)
                    for k, v in stage_ms_of(g).items():
                        stage_acc[k] = stage_acc.get(k, 0.0) + v
                    alg_bytes += g.last_algorithmic_bytes()
                    cn = g.last_counts()
                    sum_n += cn["sum_n"]; sum_m += cn["sum_m"]; live += cn["live"]
                ev1.record()
                torch.cuda.synchronize()
            value = B * steps / max(ev0.elapsed_time(ev1) / 1e3, 1e-9)
            sm = g.last_small()
            g.set_stream(None)
            g.close()
            # e2e: the reference-facing call, host buffers
            gm = mirror.graph2pi.from_csr(*csr, device=local)
            e2e_b = [batch_targets(ne, perm, 500 + s0, 0, 1, B) for s0 in range(steps + 1)]

            def call(tg):
                if a.mode == "node":
                    return gm._graph.vicinity_pi(tg, hop=a.hop, mode=cmode, flags=flags)
                gm.get_pimg_for_all_edges(tg, cores=16, hop=a.hop, norm=True, extended_flag=bool(a.extended), resolution=5, descriptor="sum")
                return gm.pi_sg, gm.status, gm.cnt_compute
            call(e2e_b[0])
            t0 = time.perf_counter()
            for s0 in range(steps):
                res = call(e2e_b[1 + s0])
            e2e = B * steps / (time.perf_counter() - t0)
            # oracle spot check on the last e2e batch
            og = orc.OracleGraph(*csr)
            oflags, omode = path_flags(a, orc)
            tg = e2e_b[steps][:spot]
            ref = og.run_batch(tg, hop=a.hop, mode=omode, flags=oflags, nthreads=orc.max_threads())
            pi_s, st_s = np.asarray(res[0])[:spot], np.asarray(res[1])[:spot]
            den = np.where(ref["pi"] != 0, np.abs(ref["pi"]), 1.0)
            err = float(np.max(np.abs(pi_s - ref["pi"]) / den)) if len(tg) else 0.0
            ok = bool(np.array_equal(st_s, ref["status"]) and err < 1e-5)
            gm._graph.close()
            cpu = cpu_baseline(csr, ne, perm, a, cpu_seconds)
            stages = {k: v for k, v in stage_acc.items() if k != "total" and not k.startswith("small_")}
            dom = max(stages, key=stages.get) if stages else "n/a"
            sab = stage_alg_bytes(float(sum_n), float(sum_m), alg_bytes, r2, float(live))
            dom_ms = stages.get(dom, 0.0)
            achieved = (sab.get(dom, alg_bytes) / 1e9) / max(dom_ms / 1e3, 1e-12)
            out[key] = {"config": what, "targets_per_step": B, "steps": steps, "value": value, "e2e": e2e, "unit": UNIT,
                        "cpu_port": {"value": cpu["value"], "cores": cpu["cores"], "sample": cpu["sample"]},
                        "value_over_port": value / max(cpu["value"], 1e-9), "e2e_over_port": e2e / max(cpu["value"], 1e-9),
                        "dominant_kernel": dom, "dominant_kernel_ms_per_step": dom_ms / steps,
                        "roofline_frac": achieved / peak, "achieved_gbs": achieved,
                        "stage_ms_per_step": {k: round(v / steps, 4) for k, v in stage_acc.items() if v > 0},
                        "kernel_S_rows_last_step": {"class_a": sm["rows_a"], "class_b": sm["rows_b"], "class_c": sm["rows_c"], "staged": sm["rows_staged"]},
                        "oracle_spot_check": {"targets": int(len(tg)), "status_equal_and_img_rel_err_lt_1e-5": ok, "max_rel_err": err}}
        except Exception as ex:  # a secondary line never fails the headline
            out[key] = {"config": what, "error": repr(ex)[:300]}
    return out


def run_cuda(args):
    import torch
    import torch.distributed as dist
    from tlc_b200 import _lib as L
    from tlc_b200 import api, multi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly ONE JSON line (rank 0): anything libraries print while starting up (e.g. NCCL's version
    # banner) is sent to stderr -- file descriptor 1 is pointed at stderr until the result line is written
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    os.environ["TLC_STAGE_TIMING"] = "1"

    c, labels, ne, csr, perm = make_workload(args.workload, args.mode, args.negatives)
    g = api.VicinityGraph(*csr, device=local)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)            # a real (non-default) stream: kernels, NCCL and the timing events share it
    g.set_stream(stream.cuda_stream)
    flags, cmode = path_flags(args, L)
    B, r2 = args.batch, 25

    out_pi = torch.zeros((B, r2), dtype=torch.float64, device=dev)
    out_f32 = torch.zeros((B, r2), dtype=torch.float32, device=dev)
    out_st = torch.zeros((B,), dtype=torch.uint8, device=dev)
    strong = args.scaling == "strong"
    G = B if strong else B * world   # targets per step over all ranks
    sv, exchange, exchange_note = None, None, None
    if world > 1:
        exchange = args.exchange
        if exchange == "peer":
            try:
                sv = multi.PeerShardedVicinity(g, csr[0], dev, max_rows=G, hop=args.hop, flags=flags, mode=cmode)
            except Exception as ex:  # (e.g. CUDA IPC not permitted between the ranks' containers): say so, use NCCL
                exchange, exchange_note = "nccl", "peer-store exchange unavailable: %s" % (repr(ex)[:160])
            ok = torch.tensor([1 if exchange == "peer" else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # all ranks take the same path
            if int(ok.item()) == 0 and exchange == "peer":
                exchange, exchange_note, sv = "nccl", "peer-store exchange unavailable on another rank", None
        if exchange == "nccl":
            sv = multi.ShardedVicinity(csr[0], multi.cuda_local_fn(g, dev, hop=args.hop, flags=flags, mode=cmode), dev)

    def global_targets(s):  # the step's targets of ALL ranks (weak: world * B per step; strong: B per step in total)
        if strong:
            return batch_targets(ne, perm, s, 0, 1, B)
        return np.concatenate([batch_targets(ne, perm, s, r, world, B) for r in range(world)])

    def step(s):  # inputs resident in HBM before the timed region
        if world > 1:
            return sv.prepare(global_targets(s))
        return torch.from_numpy(batch_targets(ne, perm, s, rank, world, B)).to(dev)

    def run(x):  # -> {name: device array} what the caller receives
        if world > 1:
            pi, st = sv.run(x)   # this rank's shard through the C-ABI, NCCL all-gather of the fp32 rows, un-permute
            return {"pi_f32": pi, "status": st}
        g.vicinity_pi_dev(x, out_pi, out_f32, out_st, hop=args.hop, mode=cmode, flags=flags)
        return {"pi": out_pi, "pi_f32": out_f32, "status": out_st}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    batches = [step(s) for s in range(args.warmup + args.steps)]
    for s in range(args.warmup):
        run(batches[s])
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    stage_acc = {}
    alg_bytes = 0.0
    handed_back = 0
    sum_n = sum_m = live = 0
    launches0 = api.launch_count()
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # library kernels, the all-gather and these events are all on torch's current stream
    ev0.record()
    t_wall0 = time.perf_counter()
    for s in range(args.warmup, args.warmup + args.steps):
        last = run(batches[s])
        for k, v in stage_ms_of(g).items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
        alg_bytes += g.last_algorithmic_bytes()
        cnts = g.last_counts()
        handed_back += cnts["handed_back"]
        sum_n += cnts["sum_n"]; sum_m += cnts["sum_m"]; live += cnts["live"]
    ev1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:   # (every rank holds the whole table of the step)
        dump_outputs(args.dump_outputs, last)
    launches = api.launch_count() - launches0
    ks_last = g.last_small()
    table_rows_last = g.last_counts().get("table_route", 0)
    table_build_ms = g.table_build_ms()
    census = None
    if table_rows_last > 0 and world == 1:
        # kernel 1t does not read all rows, so nobody counted the induced edges of those targets: an exact counting pass
        # over the timed steps' targets, OUTSIDE the timed region, supplies sum m and the 16 m term of the compulsory bytes
        cm = 0
        for s in range(args.warmup, args.warmup + args.steps):
            n_c, m_c, st_c = g.vicinity_sizes(batches[s].cpu().numpy(), hop=args.hop, mode=cmode)
            cm += int(m_c[st_c == 0].astype(np.int64).sum())
        census = {"sum_m": cm, "note": "kernel 1t (per-root shortest-path tables) served the filtration: the induced edges were "
                  "counted by a separate exact pass outside the timed region"}
        alg_bytes += 16.0 * (cm - sum_m)
        sum_m = cm
    # device time of the K steps (CUDA events on the launching stream), max over ranks
    dev_ms = float(ev0.elapsed_time(ev1))
    elapsed = max(dev_ms / 1e3, 1e-9)
    t = torch.tensor([elapsed], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_max = float(t.item())
    value = G * args.steps / elapsed_max

    # ---- e2e through the reference-facing API (host in, host out) ----
    import sg2dgm.riccidist2dgm as mirror

    g.set_stream(None)
    e2e_stage = {}
    if world == 1:
        gm = mirror.graph2pi.from_csr(*csr, device=local)
        e2e_batches = [batch_targets(ne, perm, 500 + s, rank, world, B) for s in range(args.steps + 1)]
        def e2e_call(tg):
            if args.mode == "node":  # the PDGNN generators have no batch driver: the C-ABI host-buffer call itself
                gm._graph.vicinity_pi(tg, hop=args.hop, mode=cmode, flags=flags)
            else:
                gm.get_pimg_for_all_edges(tg, cores=16, hop=args.hop, norm=True, extended_flag=bool(args.extended),
                                          resolution=5, descriptor="sum")
        e2e_call(e2e_batches[0])
        barrier()
        t0 = time.perf_counter()
        for s in range(args.steps):
            e2e_call(e2e_batches[1 + s])
            for k, v in stage_ms_of(gm._graph).items():
                e2e_stage[k] = e2e_stage.get(k, 0.0) + v
        te_local = time.perf_counter() - t0
        h2d, d2h = int(B * 8), int(B * (r2 * 8 + 1))
    else:
        # host target list in (every rank holds it, as the reference's caller would), full table back on the host
        e2e_lists = [global_targets(500 + s) for s in range(args.steps + 1)]
        sv.compute(e2e_lists[0])
        barrier()
        t0 = time.perf_counter()
        for s in range(args.steps):
            pi_all, st_all = sv.compute(e2e_lists[1 + s])
            if rank == 0:  # the caller's table on the host (one copy of it: rank 0; every rank holds it in HBM)
                pi_host = pi_all.cpu()
            else:
                torch.cuda.current_stream().synchronize()
        torch.cuda.synchronize()
        te_local = time.perf_counter() - t0
        h2d, d2h = int(G // world * 8), int(G * r2 * 4)
    te = torch.tensor([te_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = G * args.steps / float(te.item())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        # dominant kernel = the stage with the largest share of device time
        stages = {k: v for k, v in stage_acc.items() if k != "total" and not k.startswith("small_")}
        dom = max(stages, key=stages.get) if stages else "n/a"
        dom_ms = stages.get(dom, 0.0)
        sab = stage_alg_bytes(float(sum_n), float(sum_m), alg_bytes, r2, float(live))
        dom_key = "filtration_table" if (dom == "filtration" and table_rows_last > 0) else dom
        dom_bytes = sab.get(dom_key, alg_bytes)
        achieved = (dom_bytes / 1e9) / max(dom_ms / 1e3, 1e-12)
        traffic = None
        try:  # DRAM bytes per target of that kernel from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if dom_key in tj and args.workload == tj[dom_key].get("workload"):
                traffic = tj[dom_key]["dram_bytes_per_target"] * live / max(1, args.steps)
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": ("filtration_table_kernel (kernel 1t)" if dom_key == "filtration_table" else dom),
                    "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_step": dom_bytes / max(1, args.steps),
                    "kernel_ms_per_step": dom_ms / max(1, args.steps),
                    "note": "achieved = algorithmic bytes of the dominant stage kernel over the step's targets (DESIGN.md "
                            "section 4) / its device time (CUDA events on the library's stream); traffic = ncu dram bytes "
                            "of the same kernel scaled to the step's targets.  On the graph-row route the rows come from "
                            "the L2-resident CSR, so DRAM traffic is far below the algorithmic bytes: the HBM roof is the "
                            "contractual yardstick, the kernel itself is issue/latency bound (DESIGN.md section 6)",
                    "stage_ms_per_step": {k: v / args.steps for k, v in stage_acc.items()},
                    "stage_alg_gbytes_per_step": {k: v / 1e9 / args.steps for k, v in sab.items()},
                    "whole_path": {"compulsory_bytes_per_target": alg_bytes / max(1, live),
                                   "achieved_gbs": (alg_bytes / 1e9) / max(elapsed, 1e-12)}}
        # image kernel (kernel 4): diagram points per target from a small detail call outside the timed region, flops from
        # SURVEY.md section 8(d): 50 float64 FMA + 12 erfc per point with non-zero weight
        image_kernel = None
        if world == 1 and args.mode == "edge":
            try:
                smp = batch_targets(ne, perm, 900, rank, world, min(8, B))
                dd = g.vicinity_detail(smp, hop=args.hop, flags=flags)
                kk = []
                for i in range(len(smp)):
                    a = g.per_target(dd, i)
                    if a["status"] <= 1:
                        kk.append(int(np.count_nonzero(a["pdeath"] > a["pbirth"])))
                kbar = float(np.mean(kk)) if kk else 0.0
                img_ms = stage_acc.get("image", 0.0) / max(1, args.steps)
                pts = kbar * live / max(1, args.steps)
                image_kernel = {"points_per_target": kbar, "sample": len(kk), "fma_per_point": 50, "erfc_per_point": 12,
                                "ms_per_step": img_ms,
                                "fma_tflops": (2.0 * 50 * pts / 1e12) / max(img_ms / 1e3, 1e-12),
                                "erfc_per_s": (12 * pts) / max(img_ms / 1e3, 1e-12),
                                "note": "points = pairs with death > birth (weight > 0) in a detail call over a sample of the "
                                        "workload's targets; float64 CUDA-core work, 1 % of the step: no roofline claimed"}
            except Exception as ex:  # never fail the headline over the side measurement
                image_kernel = {"error": str(ex)[:200]}
        handoff = None
        if world == 1:
            try:
                handoff = measure_handoff(dev, peak)
            except Exception as ex:  # never fail the headline over the side measurement
                handoff = {"error": str(ex)[:200]}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(csr, ne, perm, args, args.cpu_seconds)
            cpu.pop("seconds", None)
        secondary = None
        if world == 1 and args.secondary:
            g.close()
            secondary = run_secondary(dev, local, peak, {(args.workload, args.mode, args.negatives): (c, labels, ne, csr, perm)})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * elapsed_max / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_dict(args, world), "exchange": exchange, "exchange_note": exchange_note,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "stage_ms_per_step": {k: v / args.steps for k, v in e2e_stage.items()}},
                "handed_back_per_step": handed_back / args.steps, "kernel_S_last_step": ks_last,
                "table_route_last_step": table_rows_last, "sssp_table_build_ms_one_time": table_build_ms, "edge_census": census,
                "gpu_launches": int(launches), "wall_ms_per_step": 1e3 * t_wall / args.steps,
                "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "handoff": handoff, "image_kernel": image_kernel,
                "secondary": secondary}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    g.close()
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(real_stdout, 1)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_cuda(a)
