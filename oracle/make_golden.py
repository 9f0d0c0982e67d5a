"""TEST INFRASTRUCTURE -- generates tests/golden/*.npz by running the REAL reference
(a checkout of pkuyzy/TLC-GNN at oracle/_ref/ or $TLC_REFERENCE_ROOT, imported in place through
oracle/ref_harness.py) on small seeded inputs; needs no GPU:
    python oracle/make_golden.py

Each fixture stores the inputs, the unmodified reference's batch output
(graph2pi.get_pimg_for_all_edges -> pi_sg, cnt_compute; riccidist2dgm.py:362-370) and, per target,
the reference's own stage functions run on the canonically ordered vicinity
(perturb_filter_function / Union_find / Accelerate_PD, accelerated_PD.py:6,26,115).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "tlc-gnn_b200"))

import ref_harness as rh  # noqa: E402
from tlc_b200 import graphgen as gg  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def ragged(list_of_arrays, dtype):
    off = np.zeros(len(list_of_arrays) + 1, dtype=np.int64)
    for i, a in enumerate(list_of_arrays):
        off[i + 1] = off[i] + len(a)
    flat = np.concatenate([np.asarray(a, dtype=dtype).reshape(-1) for a in list_of_arrays]) if list_of_arrays else np.zeros(0, dtype)
    return flat, off


def make_case(tag, edges, kappa, targets, hop, descriptor="sum", stage_targets=None):
    edges = np.asarray(edges, dtype=np.int64)
    targets = np.asarray(targets, dtype=np.int64)
    kl = [float(k) for k in kappa]
    out = dict(edges=edges, kappa=np.asarray(kappa, dtype=np.float64), targets=targets, hop=np.int64(hop),
               descriptor=np.array(descriptor))
    for ext in (False, True):
        pi, cnt, obj = rh.run_batch(edges, kl, targets, hop, ext, descriptor=descriptor)
        out["pi_ext%d" % ext] = pi
        out["cnt_ext%d" % ext] = np.int64(cnt)
    # per-target stages in canonical order, through the reference's own functions
    st_idx = list(range(len(targets))) if stage_targets is None else list(stage_targets)
    nodes, fvals, pd0, pos, neg, pd1, ncomp = [], [], [], [], [], [], []
    for i in st_idx:
        u, v = int(targets[i, 0]), int(targets[i, 1])
        if u not in obj.dict_node or v not in obj.dict_node:
            r = dict(nodes=[], ncomp=-1)
        else:
            try:
                r = rh.run_one_stages(obj, u, v, hop, descriptor=descriptor, norm=True, canonical=True)
            except BaseException:  # the batch driver swallows these too (riccidist2dgm.py:356-357)
                r = dict(nodes=[], ncomp=-2)
        ncomp.append(r["ncomp"])
        nodes.append(r["nodes"])
        ok = r["ncomp"] == 1 and "PD0" in r
        fvals.append([r["fval"][x] for x in r["nodes"]] if ok else [])
        pd0.append(np.asarray(r["PD0"], dtype=np.float64).reshape(-1) if ok else [])
        pos.append(np.asarray(r["Pos"], dtype=np.int64).reshape(-1) if ok else [])
        neg.append(np.asarray(r["Neg"], dtype=np.int64).reshape(-1) if ok else [])
        pd1.append(np.asarray(r["PD1"], dtype=np.float64).reshape(-1) if ok and r["PD1"] is not None else [])
    out["stage_idx"] = np.asarray(st_idx, dtype=np.int64)
    out["stage_ncomp"] = np.asarray(ncomp, dtype=np.int64)
    for name, lst, dt in (("nodes", nodes, np.int64), ("fval", fvals, np.float64), ("pd0", pd0, np.float64),
                          ("pos", pos, np.int64), ("neg", neg, np.int64), ("pd1", pd1, np.float64)):
        flat, off = ragged(lst, dt)
        out["stage_%s" % name] = flat
        out["stage_%s_off" % name] = off
    np.savez_compressed(os.path.join(OUT, tag + ".npz"), **out)
    print("wrote", tag, "targets", len(targets), "cnt", int(out["cnt_ext0"]), int(out["cnt_ext1"]))


def main():
    os.makedirs(OUT, exist_ok=True)
    if "--kd-only" in sys.argv:
        kd_cases()
        return
    if "--pimg-only" not in sys.argv:
        graph_cases()
        kd_cases()
    pimg_cases()


def graph_cases():
    # (1) SURVEY.md B.3 toy graph incl. every status class reachable on it
    toy = [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5), (1, 6), (2, 6)]
    make_case("toy7_hop2", toy, [0] * 7, [(1, 2), (0, 3), (0, 5), (0, 99), (2, 1), (6, 1), (3, 3)], 2)
    make_case("toy7_hop1", toy, [0] * 7, [(4, 5), (1, 2), (1, 6), (0, 1)], 1)
    # (2) Cora-shaped, hop-distance filtration (heavy ties)
    c = gg.make_config("cora", scale=0.25)
    rng = np.random.default_rng(11)
    idx = rng.choice(len(c["edges"]), 120, replace=False)
    neg = gg.negative_pairs(c["N"], c["edges"], 30, seed=201)
    make_case("cora_q_hop2", c["edges"], [0] * len(c["edges"]), np.concatenate([c["edges"][idx], neg]), 2)
    # (3) PubMed-shaped, dyadic Ricci
    c = gg.make_config("pubmed", scale=0.05)
    idx = np.random.default_rng(12).choice(len(c["edges"]), 80, replace=False)
    make_case("pubmed_s_hop2_dyadic", c["edges"], c["kappa"], c["edges"][idx], 2)
    # (4) PubMed-shaped, continuous Ricci (C2b: F4 / F5 territory)
    c = gg.make_config("pubmed", scale=0.05, continuous=True)
    make_case("pubmed_s_hop2_cont", c["edges"], c["kappa"], c["edges"][idx], 2)
    # (5) Computers-shaped (dense), hop 1 = the reference's own setting + a few hop 2
    c = gg.make_config("computers", scale=0.02)
    idx = np.random.default_rng(13).choice(len(c["edges"]), 60, replace=False)
    make_case("computers_s_hop1", c["edges"], c["kappa"], c["edges"][idx], 1)
    make_case("computers_s_hop2", c["edges"], c["kappa"], c["edges"][idx[:12]], 2)
    # (6) descriptors min / max
    c = gg.make_config("pubmed", scale=0.03)
    idx = np.random.default_rng(14).choice(len(c["edges"]), 30, replace=False)
    make_case("pubmed_s_min", c["edges"], c["kappa"], c["edges"][idx], 2, descriptor="min")
    make_case("pubmed_s_max", c["edges"], c["kappa"], c["edges"][idx], 2, descriptor="max")


def make_kd_case(tag, edges, kappa, nodes, hop, filt_name="ricci"):
    """PDGNN generator fixture (SURVEY.md row A9): the UNMODIFIED Knowledge_Distillation/data_utils_NC.py
    compute_persistence_image(g, u, filt='ricci', hop, ricci_curv, mode='PI') (:95-183) per node -> the 9-tuple
    (Ord0, Ext1, PI, filtration_val, edge_index, PI0, PI1, ...) in the reference's own (implementation-defined)
    vertex order, with the new-label -> graph-node map so that tests can canonicalise."""
    edges = np.asarray(edges, dtype=np.int64)
    g = rh.build_nx_graph(edges)
    ricci = rh.ricci_list(edges, [float(k) for k in kappa])
    out = dict(edges=edges, kappa=np.asarray(kappa, dtype=np.float64), nodes=np.asarray(nodes, dtype=np.int64),
               hop=np.int64(hop), filt_name=np.array(filt_name))
    none, old, filt, ord0, ext1, ei, pi, pi0, pi1 = [], [], [], [], [], [], [], [], []
    for u in nodes:
        r = rh.kd_run_node(g, ricci, int(u), hop, filt=filt_name)
        none.append(r is None)
        if r is None:
            r = dict(old_label=[], filt=[], ord0=[], ext1=[], edge_index=[], pi=np.zeros(25), pi0=np.zeros(25), pi1=np.zeros(25))
        old.append(r["old_label"]); filt.append(r["filt"]); ord0.append(r["ord0"]); ext1.append(r["ext1"])
        ei.append(np.asarray(r["edge_index"]).T if len(r["edge_index"]) else [])
        pi.append(r["pi"]); pi0.append(r["pi0"]); pi1.append(r["pi1"])
    out["none"] = np.asarray(none)
    for name, lst, dt in (("old_label", old, np.int64), ("filt", filt, np.float64), ("ord0", ord0, np.float64),
                          ("ext1", ext1, np.float64), ("edge_index", ei, np.int64)):
        flat, off = ragged(lst, dt)
        out["kd_%s" % name] = flat
        out["kd_%s_off" % name] = off
    out["pi"], out["pi0"], out["pi1"] = np.stack(pi), np.stack(pi0), np.stack(pi1)
    np.savez_compressed(os.path.join(OUT, tag + ".npz"), **out)
    print("wrote", tag, "nodes", len(nodes), "none", int(np.sum(none)))


def make_kd_lp_case(tag, edges, kappa, pairs, hop):
    """edge-centred PDGNN generator fixture: the UNMODIFIED Knowledge_Distillation/data_utils_LP.py
    compute_persistence_image(g, u, v, filt='ricci', hop, ricci_curv, mode='PI') (:105-196) per pair.
    kind: 0 = 9-tuple, 1 = `return None, None`, 2 = the reference raised."""
    edges = np.asarray(edges, dtype=np.int64)
    g = rh.build_nx_graph(edges)
    ricci = rh.ricci_list(edges, [float(k) for k in kappa])
    out = dict(edges=edges, kappa=np.asarray(kappa, dtype=np.float64), nodes=np.asarray(pairs, dtype=np.int64).reshape(-1, 2),
               hop=np.int64(hop))
    kind, old, filt, ord0, ext1, ei, pi, pi0, pi1 = [], [], [], [], [], [], [], [], []
    for u, v in out["nodes"]:
        r = rh.kd_lp_run_edge(g, ricci, int(u), int(v), hop)
        kind.append(1 if r is None else (2 if isinstance(r, str) else 0))
        if not isinstance(r, dict):
            r = dict(old_label=[], filt=[], ord0=[], ext1=[], edge_index=[], pi=np.zeros(25), pi0=np.zeros(25), pi1=np.zeros(25))
        old.append(r["old_label"]); filt.append(r["filt"]); ord0.append(r["ord0"]); ext1.append(r["ext1"])
        ei.append(np.asarray(r["edge_index"]).T if len(r["edge_index"]) else [])
        pi.append(r["pi"]); pi0.append(r["pi0"]); pi1.append(r["pi1"])
    out["kind"] = np.asarray(kind, dtype=np.int64)
    out["none"] = out["kind"] == 1
    for name, lst, dt in (("old_label", old, np.int64), ("filt", filt, np.float64), ("ord0", ord0, np.float64),
                          ("ext1", ext1, np.float64), ("edge_index", ei, np.int64)):
        flat, off = ragged(lst, dt)
        out["kd_%s" % name] = flat
        out["kd_%s_off" % name] = off
    out["pi"], out["pi0"], out["pi1"] = np.stack(pi), np.stack(pi0), np.stack(pi1)
    np.savez_compressed(os.path.join(OUT, tag + ".npz"), **out)
    print("wrote", tag, "pairs", len(out["nodes"]), "kinds", np.bincount(out["kind"], minlength=3).tolist())


def make_kd_gc_case(tag, graphs, filt_name="degree"):
    """graph-classification PDGNN generator fixture: the UNMODIFIED Knowledge_Distillation/data_utils_GC.py
    compute_persistence_image(g, filt, mode='PI') (:95-167) per whole graph.  graphs: list of (n, edges[m,2])."""
    none, filt, ord0, ext1, pi, pi0, pi1, sizes, elist = [], [], [], [], [], [], [], [], []
    for n, e in graphs:
        r = rh.kd_gc_run_graph(n, e, filt=filt_name)
        none.append(r is None)
        if r is None:
            r = dict(filt=[], ord0=[], ext1=[], pi=np.zeros(25), pi0=np.zeros(25), pi1=np.zeros(25))
        filt.append(r["filt"]); ord0.append(r["ord0"]); ext1.append(r["ext1"])
        pi.append(r["pi"]); pi0.append(r["pi0"]); pi1.append(r["pi1"])
        sizes.append(n); elist.append(np.asarray(e, dtype=np.int64).reshape(-1, 2))
    out = dict(none=np.asarray(none), sizes=np.asarray(sizes, dtype=np.int64), filt_name=np.array(filt_name),
               pi=np.stack(pi), pi0=np.stack(pi0), pi1=np.stack(pi1))
    for name, lst, dt in (("filt", filt, np.float64), ("ord0", ord0, np.float64), ("ext1", ext1, np.float64),
                          ("gedges", elist, np.int64)):
        flat, off = ragged(lst, dt)
        out["kd_%s" % name] = flat
        out["kd_%s_off" % name] = off
    np.savez_compressed(os.path.join(OUT, tag + ".npz"), **out)
    print("wrote", tag, "graphs", len(graphs), "none", int(np.sum(none)))


def gc_graphs(seed, count):
    """small random graphs of the TU-dataset size range: mostly connected, some disconnected, one edgeless"""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(count):
        n = int(rng.integers(6, 40))
        tree = [(int(rng.integers(0, i)), i) for i in range(1, n)]                     # random spanning tree: connected
        extra = [tuple(sorted(map(int, rng.choice(n, 2, replace=False)))) for _ in range(int(rng.integers(0, 2 * n)))]
        e = sorted(set(tuple(sorted(t)) for t in tree) | set(extra))
        if k % 5 == 3:                                                                  # drop a tree edge's endpoint: maybe disconnected
            e = [t for t in e if n - 1 not in t]
        if k == 7:
            e = []
        out.append((n, np.asarray(e, dtype=np.int64).reshape(-1, 2)))
    return out


def kd_cases():
    make_kd_gc_case("kd_gc_degree", gc_graphs(31, 24), "degree")
    c = gg.make_config("pubmed", scale=0.05, continuous=True)
    rng = np.random.default_rng(23)
    un = np.unique(c["edges"])
    pairs = np.concatenate([c["edges"][rng.choice(len(c["edges"]), 30, replace=False)],
                            rng.choice(un, size=(10, 2)), np.array([[un[3], un[3]]])])
    make_kd_lp_case("kd_lp_pubmed_s_hop2_cont", c["edges"], c["kappa"], pairs, 2)
    c = gg.make_config("ppi", scale=0.1)
    pairs = c["edges"][rng.choice(len(c["edges"]), 16, replace=False)]
    make_kd_lp_case("kd_lp_ppi_s_hop1", c["edges"], c["kappa"], pairs, 1)
    c = gg.make_config("ppi", scale=0.1)
    nodes = np.unique(c["edges"])[np.random.default_rng(21).choice(len(np.unique(c["edges"])), 20, replace=False)]
    make_kd_case("kd_ppi_s_hop1", c["edges"], c["kappa"], nodes, 1)
    make_kd_case("kd_ppi_s_hop1_degree", c["edges"], c["kappa"], nodes[:10], 1, filt_name="degree")          # :126-128
    make_kd_case("kd_ppi_s_hop1_centrality", c["edges"], c["kappa"], nodes[:10], 1, filt_name="centrality")  # :118-121
    make_kd_case("kd_ppi_s_hop1_clustering", c["edges"], c["kappa"], nodes[:8], 1, filt_name="clustering")   # :122-125
    c = gg.make_config("pubmed", scale=0.05, continuous=True)
    un = np.unique(c["edges"])
    nodes = un[np.random.default_rng(22).choice(len(un), 24, replace=False)]
    make_kd_case("kd_pubmed_s_hop2_cont", c["edges"], c["kappa"], nodes, 2)
    # hop 0: the ball is the lone centre -> `return None, None` (:103-104)
    make_kd_case("kd_pubmed_s_hop0", c["edges"], c["kappa"], nodes[:3], 0)


def pimg_cases():
    # (7) the reference tree's only PD->PI golden vector is a comment at KD/pimg.py:450-505; the
    # image of that diagram by the real sg2dgm PersistenceImager at full precision:
    ref = rh.load()
    PD = np.array([[0.0913, 0.0913], [0.1294, 0.1294], [0.1606, 0.1606], [0.1628, 0.1628], [0.0801, 0.1628],
                   [0.1993, 0.1993], [0.1186, 0.1993], [0.1189, 0.1993], [0.2081, 0.2081], [0.1294, 0.2081],
                   [0.0800, 0.2081], [0.3562, 0.3562]] + [[0.0784, 0.3562]] * 3 + [[0.0798, 0.3562], [1.0, 1.0]] +
                  [[0.0391, 1.0]] * 8 + [[0.0784, 1.0], [0.0913, 1.0], [0.0798, 0.2081]] + [[0.0784, 0.3562]] * 3 +
                  [[0.0391, 1.0]] * 15)
    gt4 = np.array([0.1209, 0.1381, 0.1520, 0.1610, 0.1642, 0.1173, 0.1340, 0.1474, 0.1561, 0.1592, 0.1093, 0.1249,
                    0.1374, 0.1455, 0.1483, 0.0979, 0.1119, 0.1230, 0.1303, 0.1328, 0.0843, 0.0963, 0.1059, 0.1121,
                    0.1143])
    img = ref.pimg.PersistenceImager(resolution=5).transform(PD).reshape(-1)
    assert PD.shape == (46, 2) and np.max(np.abs(img - gt4)) < 6e-5
    rng = np.random.default_rng(5)
    rnd = [rng.uniform(0, 1, size=(k, 2)) for k in (1, 7, 40)]
    rnd.append(rng.uniform(-0.5, 3.0, size=(25, 2)))  # outside [0,1]: legal, Gaussian tails
    res7 = ref.pimg.PersistenceImager(resolution=7).transform(rnd[2]).reshape(-1)
    np.savez_compressed(os.path.join(OUT, "pimg_vectors.npz"), PD=PD, gt4=gt4, img=img,
                        rnd0=rnd[0], rnd1=rnd[1], rnd2=rnd[2], rnd3=rnd[3],
                        img0=ref.pimg.PersistenceImager(resolution=5).transform(rnd[0]).reshape(-1),
                        img1=ref.pimg.PersistenceImager(resolution=5).transform(rnd[1]).reshape(-1),
                        img2=ref.pimg.PersistenceImager(resolution=5).transform(rnd[2]).reshape(-1),
                        img3=ref.pimg.PersistenceImager(resolution=5).transform(rnd[3]).reshape(-1), img2_res7=res7)
    print("wrote pimg_vectors")


# (8) tests/test_oracle_vs_reference.py: its inputs (seeded graphs and targets the other fixtures do not hold: self,
# repeated, reversed, unknown and far pairs, hop 3, min / max, the KD node generator on a PPI-shaped graph) and what the
# oracle computes on them.  The tests hold the oracle to these records everywhere and, where a checkout of the original
# exists, also compare it with the original live on the same inputs.  Written by `--vs-reference-pins` (no checkout
# needed: the records are the oracle's, not the original's).
VS_REF_FILE = os.path.join(OUT, "vs_reference_pins.npz")
VS_REF_BATCH = [("cora", 0.25, 2, False, True), ("pubmed", 0.04, 2, True, True), ("pubmed", 0.04, 2, False, False),
                ("computers", 0.02, 1, True, True)]
VS_REF_EDGE = [(3, "sum", True), (1, "max", True), (2, "min", False)]
VS_REF_STAGE_FIELDS = ("status", "vert", "fval", "pkind", "pbirth", "pdeath", "elo", "ehi", "pos", "neg")
VS_REF_KD_FIELDS = ("status", "vert", "fval", "pkind", "pbirth", "pdeath", "img")


def vs_ref_key(*parts):
    return "_".join(str(int(p) if isinstance(p, bool) else p) for p in parts)


def vs_ref_inputs():
    """{key: (graph key, graph config, targets or nodes in the graph's own labels)} of every test in
    test_oracle_vs_reference.py"""
    def case(name, scale, cont, seed, ntargets):
        c = gg.make_config(name, scale=scale, continuous=cont)
        rng = np.random.default_rng(seed)
        e = c["edges"]
        tg = e[rng.choice(len(e), ntargets, replace=False)]
        far = rng.integers(0, c["N"], size=(4, 2))
        return vs_ref_key("graph", name, scale, cont), c, np.concatenate([tg, far])
    out = {}
    for name, scale, hop, cont, ext in VS_REF_BATCH:
        out[vs_ref_key("batch", name, scale, hop, cont, ext)] = case(name, scale, cont, 11, 24)
    gk, c, tg = case("pubmed", 0.04, True, 5, 10)
    out["stages"] = (gk, c, tg[:10])
    c = gg.make_config("ppi", scale=0.06, continuous=True)
    labels, _ = gg.relabel_first_appearance(c["edges"])
    out["kd"] = (vs_ref_key("graph", "ppi", 0.06, True), c, np.random.default_rng(5).choice(labels, 6, replace=False))
    c = gg.make_config("pubmed", scale=0.04, continuous=True)
    e = c["edges"]
    rng = np.random.default_rng(23)
    pick = e[rng.choice(len(e), 10, replace=False)]
    un = np.unique(e)
    tg = np.concatenate([pick, pick[:3], pick[:3, ::-1], np.stack([un[:4], un[:4]], 1), rng.choice(un, size=(6, 2)),
                         np.array([[10 ** 7, int(un[0])], [int(un[1]), 10 ** 7 + 1]])])
    out["edge"] = (vs_ref_key("graph", "pubmed", 0.04, True), c, tg)
    return out


def vs_ref_graph(edges, kappa):
    """-> (oracle graph in first-appearance numbering, label -> id)"""
    import oracle as orc
    labels, ne = gg.relabel_first_appearance(edges)
    return orc.OracleGraph(*gg.build_csr(len(labels), ne, kappa)), {int(l): i for i, l in enumerate(labels)}


def vs_ref_map(lut, targets):
    return np.array([[lut.get(int(a), -1), lut.get(int(b), -1)] for a, b in targets], dtype=np.int32)


def vs_reference_pins():
    import oracle as orc
    out = {"source": np.array("oracle/tlc_oracle.c, not the original")}
    for key, (gk, c, tg) in vs_ref_inputs().items():
        out[gk + "__edges"], out[gk + "__kappa"] = c["edges"].astype(np.int32), c["kappa"]   # (graphs shared by cases: once)
        out[key + "__graph"], out[key + "__targets"] = np.array(gk), tg
        og, lut = vs_ref_graph(c["edges"], c["kappa"])
        if key.startswith("batch"):
            _, name, scale, hop, cont, ext = key.split("_")
            r = og.run_batch(vs_ref_map(lut, tg), hop=int(hop), flags=orc.F_NORM | (orc.F_EXTENDED if int(ext) else 0))
            out[key + "__pi"], out[key + "__cnt"] = r["pi"], np.int64(r["cnt_compute"])
        elif key == "edge":
            for hop, desc, ext in VS_REF_EDGE:
                r = og.run_batch(vs_ref_map(lut, tg), hop=hop, descriptor=desc, flags=orc.F_NORM | (orc.F_EXTENDED if ext else 0))
                kk = vs_ref_key("edge", hop, desc, ext)
                out[kk + "__pi"], out[kk + "__cnt"] = r["pi"], np.int64(r["cnt_compute"])
        elif key == "stages":
            for i, (a, b) in enumerate(tg):
                if int(a) in lut and int(b) in lut:
                    o = og.run_one(lut[int(a)], lut[int(b)], hop=2, flags=orc.F_NORM | orc.F_EXTENDED)
                    for f in VS_REF_STAGE_FIELDS:
                        out["stages__%d__%s" % (i, f)] = np.asarray(o[f])
        else:
            fl = orc.F_NORM | orc.F_EXTENDED | orc.F_KEEP_ZERO | orc.F_NORM_EPS
            for i, u in enumerate(tg):
                for hop in (1, 2):
                    o = og.run_one(lut[int(u)], lut[int(u)], hop=hop, mode=orc.MODE_NODE, flags=fl)
                    for f in VS_REF_KD_FIELDS:
                        out["kd__%d_%d__%s" % (i, hop, f)] = np.asarray(o[f])
    np.savez_compressed(VS_REF_FILE, **out)
    print("wrote", os.path.basename(VS_REF_FILE), len(out), "arrays")


if __name__ == "__main__":
    if "--vs-reference-pins" in sys.argv:
        vs_reference_pins()
    else:
        main()
