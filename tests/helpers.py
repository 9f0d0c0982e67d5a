"""shared test helpers: fixtures -> CSR in the reference's numbering, oracle drivers."""
import os

import numpy as np

import ricci_oracle as ro
from tlc_b200 import graphgen as gg

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GRAPH_CASES = ["toy7_hop2", "toy7_hop1", "cora_q_hop2", "pubmed_s_hop2_dyadic", "pubmed_s_hop2_cont",
               "computers_s_hop1", "computers_s_hop2", "pubmed_s_min", "pubmed_s_max"]


def load_case(tag):
    z = np.load(os.path.join(GOLDEN, tag + ".npz"))
    c = {k: z[k] for k in z.files}
    c["hop"] = int(c["hop"])
    c["descriptor"] = str(c["descriptor"])
    labels, ne = gg.relabel_first_appearance(c["edges"])
    c["labels"], c["new_edges"] = labels, ne
    c["csr"] = gg.build_csr(len(labels), ne, c["kappa"])
    lut = {int(l): i for i, l in enumerate(labels)}
    c["new_targets"] = np.array([[lut.get(int(a), -1), lut.get(int(b), -1)] for a, b in c["targets"]], dtype=np.int32)
    return c


def seg(c, name, i):
    off = c["stage_%s_off" % name]
    return c["stage_%s" % name][off[i]:off[i + 1]]


def rel_err(a, ref):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    den = np.where(ref != 0, np.abs(ref), 1.0)
    return float(np.max(np.abs(a - ref) / den)) if a.size else 0.0


KD_CASES = ["kd_ppi_s_hop1", "kd_pubmed_s_hop2_cont", "kd_pubmed_s_hop0", "kd_ppi_s_hop1_degree", "kd_ppi_s_hop1_centrality",
            "kd_ppi_s_hop1_clustering"]
KD_LP_CASES = ["kd_lp_pubmed_s_hop2_cont", "kd_lp_ppi_s_hop1"]  # edge-centred generator (data_utils_LP.py), nodes = [pairs, 2]


def load_kd_case(tag):
    """PDGNN generator fixture (oracle/make_golden.py: make_kd_case): per node the unmodified reference's 9-tuple."""
    z = np.load(os.path.join(GOLDEN, tag + ".npz"))
    c = {k: z[k] for k in z.files}
    c["hop"] = int(c["hop"])
    c["filt_name"] = str(c["filt_name"]) if "filt_name" in c else "ricci"
    labels, ne = gg.relabel_first_appearance(c["edges"])
    c["csr"] = gg.build_csr(len(labels), ne, c["kappa"])
    c["lut"] = {int(l): i for i, l in enumerate(labels)}
    c["new_nodes"] = np.array([c["lut"][int(u)] for u in c["nodes"].reshape(-1)], dtype=np.int32).reshape(c["nodes"].shape)
    return c


def kd_seg(c, name, k):
    off = c["kd_%s_off" % name]
    w = 2 if name in ("ord0", "ext1", "edge_index") else 1  # offsets count rows; these are [rows, 2] flattened
    return c["kd_%s" % name][w * off[k]:w * off[k + 1]]


def ricci_hub_graph():
    """graph for kernel 6's three launch classes (support = min(degree, 3000) + 1; an edge's class comes from its larger
    support: <= 120, <= 1024, <= 3001).  Deterministic, N = 3621 (not a multiple of 32).  Returns (rowptr, col, ids):
      h3500 = N - 1 (the last bitmap word; always the larger endpoint), h3001, h3000 (mid-range ids: the smaller endpoint
      of some edges, the larger of others), d1024, d1023, d120, d119: nodes of exactly that degree;
      boundary pairs h3500-h3001 and h3001-h3000 (3001 x 3001 codes), d1024-d1023, d120-d119;
      cut: a node adjacent to h3500 and to 8 of the 500 smallest neighbours of h3500 -- the ones the cut to 3000 drops;
    every other node is plain, adjacent to a random subset of the above plus a sparse random background (degree <= 30)."""
    N = 3621
    rs = np.random.RandomState(5)
    ids = dict(h3500=N - 1, h3001=1801, h3000=1200, d1024=2400, d1023=600, d120=3000, d119=300, cut=2999)
    deg = dict(h3500=3500, h3001=3001, h3000=3000, d1024=1024, d1023=1023, d120=120, d119=119)
    pairs = [("h3500", "h3001"), ("h3001", "h3000"), ("d1024", "d1023"), ("d120", "d119")]
    edges = [(ids[p], ids[q]) for p, q in pairs]
    plain = np.setdiff1d(np.arange(N), list(ids.values()))
    for name, d in deg.items():
        need = d - sum(name in pq for pq in pairs) - (name == "h3500")
        edges += [(ids[name], int(y)) for y in np.sort(rs.choice(plain, need, replace=False))]
    edges.append((ids["cut"], ids["h3500"]))
    h_nb = np.sort([y for x, y in edges if x == ids["h3500"]])
    edges += [(ids["cut"], int(y)) for y in h_nb[:8]]
    bg = rs.choice(plain, (2 * N, 2))
    edges += [(int(a), int(b)) for a, b in bg if a != b]
    e = np.asarray(edges, dtype=np.int64)
    e = np.unique(np.stack([e.min(1), e.max(1)], 1), axis=0)
    rp, col, _ = gg.build_csr(N, e, np.zeros(len(e)))
    dg = np.diff(rp)
    assert all(dg[ids[k]] == d for k, d in deg.items()) and dg[plain].max() <= 30 and dg[ids["cut"]] == 9
    assert np.all(np.isin(col[rp[ids["cut"]]:rp[ids["cut"] + 1]], np.append(h_nb[:8], ids["h3500"])))
    return rp, col, ids


def ricci_classes(rowptr, col):
    """(x < y) edges in CSR order and their kernel-6 launch class: 0 (larger support <= 120), 1 (<= 1024), 2 (the rest)"""
    deg = np.diff(np.asarray(rowptr, dtype=np.int64))
    src = np.repeat(np.arange(len(deg)), deg)
    keep = src < col
    e = np.stack([src[keep], np.asarray(col, dtype=np.int64)[keep]], 1)
    size = np.minimum(deg, ro.NBR_TOPK) + 1
    big = np.maximum(size[e[:, 0]], size[e[:, 1]])
    return e, np.where(big <= 120, 0, np.where(big <= 1024, 1, 2))


def sorted_rows(a):
    a = np.asarray(a, dtype=np.float64).reshape(-1, 2)
    return a[np.lexsort((a[:, 1], a[:, 0]))]


def kd_expected(c, k):
    """node k of a KD fixture in canonical form: graph ids (first-appearance numbering) ascending, the filtration
    values in that order, the induced edge set as sorted (lo, hi) graph-id pairs, Ord0 / Ext1 as sorted multisets
    (the reference's own vertex / pair order is implementation-defined, SURVEY.md F3)."""
    old = kd_seg(c, "old_label", k)
    newid = np.array([c["lut"][int(x)] for x in old], dtype=np.int64)
    order = np.argsort(newid)
    ei = kd_seg(c, "edge_index", k).reshape(-1, 2)
    eg = newid[ei] if len(ei) else np.zeros((0, 2), np.int64)
    eg = np.stack([eg.min(1), eg.max(1)], 1) if len(eg) else eg
    eg = eg[np.lexsort((eg[:, 1], eg[:, 0]))] if len(eg) else eg
    return dict(vert=newid[order], filt=kd_seg(c, "filt", k)[order], edges=eg,
                ord0=sorted_rows(kd_seg(c, "ord0", k)), ext1=sorted_rows(kd_seg(c, "ext1", k)),
                pi=c["pi"][k], pi0=c["pi0"][k], pi1=c["pi1"][k], none=bool(c["none"][k]))


def load_kd_gc_case(tag="kd_gc_degree"):
    """graph-classification generator fixture: list of (n, edges) + the unmodified reference's per-graph outputs."""
    z = np.load(os.path.join(GOLDEN, tag + ".npz"))
    c = {k: z[k] for k in z.files}
    graphs = []
    for k, n in enumerate(c["sizes"]):
        off = c["kd_gedges_off"]
        graphs.append((int(n), c["kd_gedges"][2 * off[k]:2 * off[k + 1]].reshape(-1, 2)))
    c["graphs"] = graphs
    c["filt_name"] = str(c["filt_name"])
    return c
