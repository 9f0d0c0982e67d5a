"""CUDA path (through the C-ABI) vs the oracle: bit-exact integers / float64 values, images 1e-5."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle as orc
from helpers import GRAPH_CASES, load_case, rel_err
from tlc_b200 import _lib as L
from tlc_b200 import api, graphgen as gg

IMG_TOL = 1e-5  # north_star: persistence images within 1e-5 relative


def compare_detail(g, og, targets, hop, descriptor, flags, oflags, mode=L.MODE_EDGE):
    d = g.vicinity_detail(targets, hop=hop, mode=mode, descriptor=descriptor, flags=flags)
    for i, (u, v) in enumerate(targets):
        a = g.per_target(d, i)
        o = og.run_one(int(u), int(v), hop=hop, mode=mode, descriptor=descriptor, flags=oflags)
        ctx = "target %d (%d,%d) status gpu %d oracle %d n %d m %d" % (i, u, v, a["status"], o["status"], o["n"], o["m"])
        assert a["status"] == o["status"], ctx
        assert a["n"] == o["n"] and a["m"] == o["m"], ctx
        if o["status"] in (5,):
            continue
        assert np.array_equal(a["vert"], o["vert"]), ctx              # kernel 1: vertex set, canonical order
        assert np.array_equal(a["elo"], o["elo"]) and np.array_equal(a["ehi"], o["ehi"]), ctx
        assert np.array_equal(a["ew"], o["ew"]), ctx
        if o["status"] > 1 and o["status"] != 7:
            continue
        assert (a["lu"], a["lv"]) == (o["lu"], o["lv"]), ctx
        assert np.array_equal(a["fval"], o["fval"]), ctx              # kernel 1b: bit-exact float64
        assert np.array_equal(a["ord_asc"], o["ord_asc"]), ctx        # kernel 2
        assert np.array_equal(a["ord_desc"], o["ord_desc"]), ctx
        k = len(o["pkind"])
        assert len(a["pkind"]) == k, ctx                              # kernel 3 / 3b: pairs bit-exact
        assert np.array_equal(a["pkind"], o["pkind"]), ctx
        assert np.array_equal(a["pbv"], o["pbv"]) and np.array_equal(a["pdv"], o["pdv"]), ctx
        assert np.array_equal(a["pbirth"], o["pbirth"]) and np.array_equal(a["pdeath"], o["pdeath"]), ctx
        assert np.array_equal(a["neg"], o["neg"]), ctx
        assert np.array_equal(a["pos"], o["pos"]), ctx
        assert rel_err(a["img"], o["img"]) < IMG_TOL, ctx             # kernel 4


# es = 1 forces the edge-sorted kernels 2+3 for the ascending sweep; es = 0 is the default vertex-ordered
# kernels 2v+3v (with hand-back to 2+3).  Both must reproduce the oracle's pair sequence bit for bit.
@pytest.mark.parametrize("tag", GRAPH_CASES)
@pytest.mark.parametrize("ext", [0, 1])
@pytest.mark.parametrize("es", [0, 1])
def test_golden_cases(tag, ext, es):
    c = load_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    og = orc.OracleGraph(*c["csr"])
    oflags = orc.F_NORM | (orc.F_EXTENDED if ext else 0)
    flags = L.F_NORM | (L.F_EXTENDED if ext else 0) | (L.F_EDGE_SORTED if es else 0)
    # batch call: images vs the REAL reference's pi_sg stored in the fixture, counts equal
    pi, status, cnt = g.vicinity_pi(c["new_targets"], hop=c["hop"], descriptor=c["descriptor"], flags=flags)
    ref = c["pi_ext%d" % ext]
    assert cnt == int(c["cnt_ext%d" % ext])
    assert np.array_equal(ref.any(axis=1), pi.any(axis=1))
    assert rel_err(pi, ref) < IMG_TOL
    o = og.run_batch(c["new_targets"], hop=c["hop"], descriptor=c["descriptor"], flags=oflags)
    assert np.array_equal(status, o["status"])
    compare_detail(g, og, c["new_targets"], c["hop"], c["descriptor"], flags, oflags)
    g.close()


@pytest.mark.parametrize("es", [0, 1])
@pytest.mark.parametrize("name,scale,hop,cont", [("cora", 1.0, 2, False), ("cora", 1.0, 3, False), ("pubmed", 0.3, 2, False),
                                                 ("pubmed", 0.3, 2, True), ("computers", 0.05, 2, False),
                                                 ("computers", 0.05, 2, True), ("ppi", 0.3, 1, False)])
def test_random_targets(name, scale, hop, cont, es):
    c = gg.make_config(name, scale=scale, continuous=cont)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(7)
    tg = ne[rng.choice(len(ne), 48, replace=False)].astype(np.int32)
    neg = rng.integers(0, len(labels), size=(16, 2)).astype(np.int32)
    tg = np.concatenate([tg, neg, np.array([[-1, 3], [0, 0]], np.int32)])
    oflags = orc.F_NORM | orc.F_EXTENDED
    flags = L.F_NORM | L.F_EXTENDED | (L.F_EDGE_SORTED if es else 0)
    compare_detail(g, og, tg, hop, "sum", flags, oflags)
    for ext in (1, 0):  # the batch call without `extended` runs the ascending sweep only (image needs no PD_down)
        fl = flags if ext else flags & ~L.F_EXTENDED
        ofl = oflags if ext else oflags & ~orc.F_EXTENDED
        pi, status, cnt = g.vicinity_pi(tg, hop=hop, flags=fl)
        o = og.run_batch(tg, hop=hop, flags=ofl)
        assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"]
        assert rel_err(pi, o["pi"]) < IMG_TOL
    g.close()


@pytest.mark.parametrize("es", [0, 1])
@pytest.mark.parametrize("eps", [1e-10, 3e-7, 0.0])
def test_near_tie_values(es, eps):
    """vertex values closer than a float ulp / than the 1e-6 key perturbation (SURVEY.md F4) and exact ties:
    exercises the equal-float run fix of kernel 2v, the near-tie ("distinct") blocks and the representative
    path of kernel 3v.  K common neighbours of an edge (u,v) with curvatures eps apart, some adjacent to each other,
    plus pendant paths that create local minima and component merges."""
    K = 40
    edges, kap = [(0, 1)], [0.25]
    for i in range(K):
        x = 2 + i
        edges += [(0, x), (1, x)]
        kap += [0.5 + ((i * 7) % K) * eps, 0.5 - ((i * 3) % K) * eps]
        if i % 3 == 0 and i + 1 < K:
            edges.append((x, x + 1)); kap.append(-0.5 + i * eps)
    base = 2 + K
    for i in range(6):   # short cycles hanging off the roots through cheap detours
        a, b = base + 2 * i, base + 2 * i + 1
        edges += [(0, a), (a, b), (b, 1), (b, 2 + i)]
        kap += [0.9 - i * eps, -0.8, 0.9 - 2 * i * eps, -0.7 + i * eps]
    e = np.array(edges, dtype=np.int64)
    labels, ne = gg.relabel_first_appearance(e)
    csr = gg.build_csr(len(labels), ne, np.array(kap))
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    tg = ne[:24].astype(np.int32)
    for hop in (1, 2):
        for ext in (0, 1):
            oflags = orc.F_NORM | (orc.F_EXTENDED if ext else 0)
            flags = L.F_NORM | (L.F_EXTENDED if ext else 0) | (L.F_EDGE_SORTED if es else 0)
            compare_detail(g, og, tg, hop, "sum", flags, oflags)
            pi, status, cnt = g.vicinity_pi(tg, hop=hop, flags=flags)
            o = og.run_batch(tg, hop=hop, flags=oflags)
            assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"]
            assert rel_err(pi, o["pi"]) < IMG_TOL
            if not ext and not es:  # the same through the graph-row route
                compare_asc(g, og, tg, hop, "sum", flags | L.F_DIRECT, oflags)
                pi_d, status_d, cnt_d = g.vicinity_pi(tg, hop=hop, flags=flags | L.F_DIRECT)
                assert g.last_counts()["graph_row_route"] > 0
                assert np.array_equal(pi, pi_d) and np.array_equal(status, status_d) and cnt == cnt_d
    g.close()


def test_node_mode_kd_flags():
    """PDGNN node-centred vicinities (Knowledge_Distillation/data_utils_NC.py:95-183 shape)."""
    c = gg.make_config("ppi", scale=0.25)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    nodes = np.random.default_rng(3).choice(len(labels), 24, replace=False)
    tg = np.stack([nodes, nodes], 1).astype(np.int32)
    flags = L.F_NORM | L.F_EXTENDED | L.F_KEEP_ZERO | L.F_NORM_EPS
    compare_detail(g, og, tg, 2, "sum", flags, flags, mode=L.MODE_NODE)
    g.close()


def test_pimg_transform_golden():
    import os
    from helpers import GOLDEN
    z = np.load(os.path.join(GOLDEN, "pimg_vectors.npz"))
    img = api.pimg_transform(z["PD"]).reshape(-1)
    assert np.max(np.abs(img - z["gt4"])) < 6e-5          # Knowledge_Distillation/pimg.py:450-505
    assert rel_err(img, z["img"]) < IMG_TOL
    for k in range(4):
        assert rel_err(api.pimg_transform(z["rnd%d" % k]).reshape(-1), z["img%d" % k]) < IMG_TOL
    assert rel_err(api.pimg_transform(z["rnd2"], 7).reshape(-1), z["img2_res7"]) < IMG_TOL


def test_union_find_api():
    """Union_find/Accelerate_PD entry point on a caller-supplied graph, order = tie-break."""
    c = load_case("pubmed_s_hop2_cont")
    og = orc.OracleGraph(*c["csr"])
    for ti in range(6):
        u, v = c["new_targets"][ti]
        o = og.run_one(int(u), int(v), hop=2, flags=orc.F_NORM | orc.F_EXTENDED)
        if o["status"] != 0:
            continue
        r = api.union_find(o["fval"], np.stack([o["elo"], o["ehi"]], 1), flags=L.F_EXTENDED)
        assert np.array_equal(r["pkind"], o["pkind"])
        assert np.array_equal(r["pbirth"], o["pbirth"]) and np.array_equal(r["pdeath"], o["pdeath"])
        assert np.array_equal(r["pos"], o["pos"]) and np.array_equal(r["neg"], o["neg"])


# ---------------------------------------------------------------------------------------------------------
# graph-row route (TLC_F_DIRECT): no adjacency in HBM, the filtration / vertex-order / sweep kernels read the
# graph's own CSR rows through the vicinity bitmap.  Serves ascending-sweep-only calls; must reproduce the
# oracle's vertex set, roots, filtration values, PD_up + [min,max] pairs (ids and values) and image bit for bit.
# ---------------------------------------------------------------------------------------------------------
def compare_asc(g, og, targets, hop, descriptor, flags, oflags, mode=L.MODE_EDGE):
    d = g.vicinity_detail(targets, hop=hop, mode=mode, descriptor=descriptor, flags=flags | L.F_ASC_ONLY)
    for i, (u, v) in enumerate(targets):
        a = g.per_target(d, i)
        o = og.run_one(int(u), int(v), hop=hop, mode=mode, descriptor=descriptor, flags=oflags)
        ctx = "target %d (%d,%d) status gpu %d oracle %d n %d m %d" % (i, u, v, a["status"], o["status"], o["n"], o["m"])
        assert a["status"] == o["status"], ctx
        assert a["n"] == o["n"], ctx
        if o["status"] in (5,):
            continue
        assert np.array_equal(a["vert"], o["vert"]), ctx
        if o["status"] > 1:
            continue
        assert (a["lu"], a["lv"]) == (o["lu"], o["lv"]), ctx
        assert np.array_equal(a["fval"], o["fval"]), ctx
        keep = np.isin(o["pkind"], (L.K_UP, L.K_ESS))
        assert np.array_equal(a["pkind"], o["pkind"][keep]), ctx
        assert np.array_equal(a["pbv"], o["pbv"][keep]) and np.array_equal(a["pdv"], o["pdv"][keep]), ctx
        assert np.array_equal(a["pbirth"], o["pbirth"][keep]) and np.array_equal(a["pdeath"], o["pdeath"][keep]), ctx
        assert rel_err(a["img"], o["img"]) < IMG_TOL, ctx


@pytest.mark.parametrize("tag", GRAPH_CASES)
def test_graph_row_route_golden(tag):
    c = load_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    og = orc.OracleGraph(*c["csr"])
    flags = L.F_NORM | L.F_DIRECT
    pi, status, cnt = g.vicinity_pi(c["new_targets"], hop=c["hop"], descriptor=c["descriptor"], flags=flags)
    assert g.last_counts()["graph_row_route"] > 0
    ref = c["pi_ext0"]  # the REAL reference's pi_sg
    assert cnt == int(c["cnt_ext0"])
    assert np.array_equal(ref.any(axis=1), pi.any(axis=1))
    assert rel_err(pi, ref) < IMG_TOL
    o = og.run_batch(c["new_targets"], hop=c["hop"], descriptor=c["descriptor"], flags=orc.F_NORM)
    assert np.array_equal(status, o["status"])
    pi2, status2, cnt2 = g.vicinity_pi(c["new_targets"], hop=c["hop"], descriptor=c["descriptor"], flags=L.F_NORM | L.F_NO_DIRECT)
    assert g.last_counts()["graph_row_route"] == 0
    assert np.array_equal(pi, pi2) and np.array_equal(status, status2) and cnt == cnt2  # the two routes agree bit for bit
    compare_asc(g, og, c["new_targets"], c["hop"], c["descriptor"], flags, orc.F_NORM)
    g.close()


@pytest.mark.parametrize("name,scale,hop,cont", [("cora", 1.0, 2, False), ("cora", 1.0, 3, False), ("pubmed", 0.3, 2, True),
                                                 ("computers", 0.05, 2, False), ("computers", 0.05, 2, True),
                                                 ("computers", 0.1, 1, True), ("ppi", 0.3, 1, False)])
def test_graph_row_route_random(name, scale, hop, cont):
    c = gg.make_config(name, scale=scale, continuous=cont)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(11)
    tg = ne[rng.choice(len(ne), 48, replace=False)].astype(np.int32)
    neg = rng.integers(0, len(labels), size=(16, 2)).astype(np.int32)
    tg = np.concatenate([tg, neg, np.array([[-1, 3], [0, 0]], np.int32)])
    compare_asc(g, og, tg, hop, "sum", L.F_NORM | L.F_DIRECT, orc.F_NORM)                  # kernel 1t (shortest-path tables)
    compare_asc(g, og, tg, hop, "sum", L.F_NORM | L.F_DIRECT | L.F_NO_TABLE, orc.F_NORM)   # kernel 1b on the graph rows
    o = og.run_batch(tg, hop=hop, flags=orc.F_NORM)
    # forced with / without the tables, default routing (kernel S first), staged + density-routed, materialised
    for fl in (L.F_DIRECT | L.F_NO_TABLE, L.F_DIRECT, 0, L.F_NO_SMALL, L.F_NO_DIRECT):
        pi, status, cnt = g.vicinity_pi(tg, hop=hop, flags=L.F_NORM | fl)
        assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"]
        assert rel_err(pi, o["pi"]) < IMG_TOL
        cn = g.last_counts()
        if fl == (L.F_DIRECT | L.F_NO_TABLE):
            pi_d, cn_d = pi, cn
            # (a target kernel 3v hands back needs the adjacency: the whole call is then redone on the materialised route)
            assert cn["graph_row_route"] > 0 or cn["handed_back"] > 0
            assert cn["table_route"] == 0
        else:
            assert np.array_equal(pi, pi_d)
            if fl == L.F_DIRECT:
                assert cn["table_route"] > 0 or cn["handed_back"] > 0
            if cn["table_route"] == 0:
                # the edge totals agree whether kernel 1's counting pass, kernel 1b (graph-row batch call) or kernel S counted them
                assert (cn["sum_n"], cn["sum_m"], cn["live"]) == (cn_d["sum_n"], cn_d["sum_m"], cn_d["live"])
            else:
                assert (cn["sum_n"], cn["live"]) == (cn_d["sum_n"], cn_d["live"])
    assert abs(g.last_algorithmic_bytes()) > 0
    g.close()


def test_graph_row_route_node_mode():
    c = gg.make_config("ppi", scale=0.25)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    nodes = np.random.default_rng(3).choice(len(labels), 24, replace=False)
    tg = np.stack([nodes, nodes], 1).astype(np.int32)
    fl = L.F_NORM | L.F_KEEP_ZERO | L.F_NORM_EPS
    for hop in (0, 1, 2):
        compare_asc(g, og, tg, hop, "sum", fl | L.F_DIRECT, fl, mode=L.MODE_NODE)
    g.close()


def test_edge_forced_mode_kd_flags():
    """PDGNN edge-centred vicinities, the two roots always members (Knowledge_Distillation/data_utils_LP.py:107-118)."""
    c = gg.make_config("pubmed", scale=0.3, continuous=True)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(4)
    tg = np.concatenate([ne[rng.choice(len(ne), 40, replace=False)], rng.integers(0, len(labels), size=(20, 2)),
                         np.array([[5, 5], [-1, 2]])]).astype(np.int32)
    flags = L.F_NORM | L.F_EXTENDED | L.F_KEEP_ZERO | L.F_NORM_EPS
    for hop in (1, 2):
        compare_detail(g, og, tg, hop, "sum", flags, flags, mode=L.MODE_EDGE_FORCED)
        pi, status, cnt = g.vicinity_pi(tg, hop=hop, mode=L.MODE_EDGE_FORCED, flags=flags)
        o = og.run_batch(tg, hop=hop, mode=orc.MODE_EDGE_FORCED, flags=flags)
        assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"] and rel_err(pi, o["pi"]) < IMG_TOL
    g.close()


@pytest.mark.parametrize("filt", ["degree", "centrality", "clustering"])
def test_structural_filtrations(filt):
    """PDGNN generators' filt='degree' / 'centrality' (Knowledge_Distillation/data_utils_NC.py:118-128), node and edge-forced modes."""
    c = gg.make_config("ppi", scale=0.25)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(8)
    nodes = rng.choice(len(labels), 16, replace=False)
    ff = {"degree": L.F_FILT_DEGREE, "centrality": L.F_FILT_CENTRALITY, "clustering": L.F_FILT_CLUSTERING}[filt]
    flags = L.F_NORM | L.F_EXTENDED | L.F_KEEP_ZERO | L.F_NORM_EPS | ff
    compare_detail(g, og, np.stack([nodes, nodes], 1).astype(np.int32), 1, "sum", flags, flags, mode=L.MODE_NODE)
    tg = ne[rng.choice(len(ne), 16, replace=False)].astype(np.int32)
    compare_detail(g, og, tg, 1, "sum", flags, flags, mode=L.MODE_EDGE_FORCED)
    pi, status, cnt = g.vicinity_pi(tg, hop=1, mode=L.MODE_EDGE_FORCED, flags=flags & ~L.F_EXTENDED)  # (never the graph-row route)
    o = og.run_batch(tg, hop=1, mode=orc.MODE_EDGE_FORCED, flags=flags & ~L.F_EXTENDED)
    assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"] and rel_err(pi, o["pi"]) < IMG_TOL
    g.close()


def test_handed_back_targets_on_the_graph_row_route(monkeypatch):
    """a near-tie block that needs more representatives than kernel 3v keeps (a clique of 24 common neighbours whose values
    differ by ~1e-10): the targets are handed back; on the graph-row batch call exactly those are redone on the
    materialised route and scattered back into the caller's rows."""
    K = 24
    edges, kap = [(0, 1)], [0.25]
    for i in range(K):
        x = 2 + i
        edges += [(0, x), (1, x)]
        kap += [0.5 + i * 1e-10, 0.5 - ((i * 5) % K) * 1e-10]
        for j in range(i):
            edges.append((2 + j, x)); kap.append(0.3 + (i * K + j) * 1e-9)
    # a second, ordinary part of the graph so that the call mixes handed-back and regular targets
    base = 2 + K
    for i in range(30):
        edges += [(base + i, base + (i + 1) % 30), (base + i, base + (i + 7) % 30)]
        kap += [0.1 * ((i % 5) - 2), 0.05 * ((i % 7) - 3)]
    edges.append((0, base)); kap.append(0.4)
    e = np.array(edges, dtype=np.int64)
    labels, ne = gg.relabel_first_appearance(e)
    csr = gg.build_csr(len(labels), ne, np.array(kap))
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    tg = np.concatenate([ne[:40], ne[-50:]]).astype(np.int32)
    o = og.run_batch(tg, hop=2, flags=orc.F_NORM)
    # (kernel 2v's no-pair certificate settles the clique targets before any sweep: every clique vertex has a root as a far
    #  lower neighbour.  Off for the hand-back check, on again below: the rows must not change.)
    monkeypatch.setenv("TLC_NO_FAST_DIAGRAM", "1")
    pi, status, cnt = g.vicinity_pi(tg, hop=2, flags=L.F_NORM | L.F_DIRECT)
    cn = g.last_counts()
    monkeypatch.delenv("TLC_NO_FAST_DIAGRAM")
    pi_c, status_c, cnt_c = g.vicinity_pi(tg, hop=2, flags=L.F_NORM | L.F_DIRECT)
    assert np.array_equal(pi_c, pi) and np.array_equal(status_c, status) and cnt_c == cnt
    assert cn["handed_back"] > 0 and 0 < cn["graph_row_route"] < cn["live"]      # some redone, the rest stayed on the route
    assert 0 < cn["table_route"] <= cn["graph_row_route"]                       # (the redone targets leave both counts)
    assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"] and rel_err(pi, o["pi"]) < IMG_TOL
    pi_m, status_m, cnt_m = g.vicinity_pi(tg, hop=2, flags=L.F_NORM | L.F_NO_DIRECT)
    assert np.array_equal(pi, pi_m) and np.array_equal(status, status_m) and cnt == cnt_m
    compare_asc(g, og, tg[:8], 2, "sum", L.F_NORM | L.F_DIRECT, orc.F_NORM)
    g.close()


def test_plain_path_sums_and_other_resolutions():
    """TLC_F_SUM_PLAIN: path sums added left to right as CPython <= 3.11's sum() does -- the interpreter the reference pins
    (3.7); default is the Neumaier-compensated sum() of CPython >= 3.12 (SURVEY.md F5).  Continuous curvature, so the
    two differ in the last bits.  Also batch calls at resolutions other than 5 (PersistenceImager(resolution), :207)."""
    c = gg.make_config("pubmed", scale=0.3, continuous=True)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(17)
    tg = ne[rng.choice(len(ne), 64, replace=False)].astype(np.int32)
    compare_detail(g, og, tg[:24], 2, "sum", L.F_NORM | L.F_EXTENDED | L.F_SUM_PLAIN, orc.F_NORM | orc.F_EXTENDED | orc.F_SUM_PLAIN)
    compare_asc(g, og, tg[:24], 2, "sum", L.F_NORM | L.F_SUM_PLAIN | L.F_DIRECT, orc.F_NORM | orc.F_SUM_PLAIN)
    d0 = g.vicinity_detail(tg[:24], hop=2, flags=L.F_NORM)
    d1 = g.vicinity_detail(tg[:24], hop=2, flags=L.F_NORM | L.F_SUM_PLAIN)
    assert not np.array_equal(d0["fval"], d1["fval"])          # the flag does change last bits on continuous weights
    for res in (3, 8):
        for fl in (0, L.F_DIRECT, L.F_EXTENDED):
            pi, status, cnt = g.vicinity_pi(tg, hop=2, resolution=res, flags=L.F_NORM | fl)
            o = og.run_batch(tg, hop=2, resolution=res, flags=orc.F_NORM | (orc.F_EXTENDED if fl == L.F_EXTENDED else 0))
            assert pi.shape == (len(tg), res * res)
            assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"] and rel_err(pi, o["pi"]) < IMG_TOL
    g.close()
