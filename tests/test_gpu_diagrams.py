"""The persistence diagrams of a batch (tlc_vicinity_diagrams / _dev) vs the oracle: every pair bit-exact in the reference's
order with graph vertex ids, on every route the batch call takes (kernel S, the staged pipeline on the materialised and the
graph-row route, the sub-calls that re-index targets); image rows and statuses equal to the image call's; the capacity
protocol; run-to-run determinism."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle as orc
from helpers import GRAPH_CASES, load_case
from tlc_b200 import _lib as L
from tlc_b200 import api, graphgen as gg


def make(name, scale=1.0, cont=False):
    c = gg.make_config(name, scale=scale, continuous=cont)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    return gg.build_csr(len(labels), ne, c["kappa"]), ne, len(labels)


def carries_pairs(status):
    return status <= L.ST_TRIVIAL or status == L.ST_NO_TREE_EDGES


def check_oracle(d, og, tg, hop, oflags, mode=L.MODE_EDGE, descriptor="sum", asc=False, rows=None):
    """target i's segment of the diagram call equals the oracle's pairs (kinds 0 / 1 only with asc), local ids mapped to
    graph ids through the oracle's vertex list"""
    for i in (range(len(tg)) if rows is None else rows):
        u, v = int(tg[i, 0]), int(tg[i, 1])
        o = og.run_one(u, v, hop=hop, mode=mode, descriptor=descriptor, flags=oflags)
        ctx = "target %d (%d,%d) status %d / %d" % (i, u, v, d["status"][i], o["status"])
        assert d["status"][i] == o["status"], ctx
        a, b = int(d["poff"][i]), int(d["poff"][i + 1])
        if not carries_pairs(o["status"]):
            assert a == b, ctx
            continue
        keep = np.isin(o["pkind"], (L.K_UP, L.K_ESS)) if asc else np.ones(len(o["pkind"]), bool)
        assert b - a == int(keep.sum()), ctx
        assert np.array_equal(d["kind"][a:b], o["pkind"][keep]), ctx
        assert np.array_equal(d["bv"][a:b], o["vert"][o["pbv"][keep]]), ctx
        assert np.array_equal(d["dv"][a:b], o["vert"][o["pdv"][keep]]), ctx
        assert np.array_equal(d["birth"][a:b], o["pbirth"][keep]), ctx
        assert np.array_equal(d["death"][a:b], o["pdeath"][keep]), ctx


PAIR_KEYS = ("poff", "kind", "bv", "dv", "birth", "death", "status")


def check_image(g, d, tg, **kw):
    pi, status, _ = g.vicinity_pi(tg, **kw)
    assert np.array_equal(d["status"], status)
    assert np.array_equal(d["pi"], pi)


@pytest.mark.parametrize("tag", GRAPH_CASES)
@pytest.mark.parametrize("ext", [0, 1])
def test_diagrams_golden_cases(tag, ext):
    c = load_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    og = orc.OracleGraph(*c["csr"])
    flags = L.F_NORM | (L.F_EXTENDED if ext else 0)
    tg = c["new_targets"]
    d = g.vicinity_diagrams(tg, hop=c["hop"], descriptor=c["descriptor"], flags=flags)
    check_oracle(d, og, tg, c["hop"], orc.F_NORM | (orc.F_EXTENDED if ext else 0), descriptor=c["descriptor"])
    check_image(g, d, tg, hop=c["hop"], descriptor=c["descriptor"], flags=flags)
    g.close()


@pytest.mark.parametrize("ext", [0, 1])
@pytest.mark.parametrize("name,scale,hop,cont", [("cora", 1.0, 2, False), ("pubmed", 0.3, 2, True), ("computers", 0.05, 2, True),
                                                 ("computers", 1.0, 1, False), ("ppi", 0.3, 1, False)])
def test_diagrams_random_targets_every_leg(name, scale, hop, cont, ext):
    csr, ne, N = make(name, scale, cont)
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(11)
    tg = ne[rng.choice(len(ne), 160, replace=False)].astype(np.int32)
    neg = rng.integers(0, N, size=(32, 2)).astype(np.int32)
    tg = np.concatenate([tg, neg, np.array([[-1, 3], [0, 0], [5, N + 7]], np.int32)])
    base = L.F_NORM | (L.F_EXTENDED if ext else 0)
    d0 = g.vicinity_diagrams(tg, hop=hop, flags=base)
    # the statistics of ONE call on a fresh graph (a call repeated for capacity may find kernel S paused by its own
    # heuristic: a call that hands most rows on pauses it for the next calls)
    g1 = api.VicinityGraph(*csr, device=0)
    d1 = g1.vicinity_diagrams(tg, hop=hop, flags=base, cap=int(d0["poff"][-1]))
    s = g1.last_small()
    g1.close()
    for k in PAIR_KEYS:
        assert np.array_equal(d1[k], d0[k]), k
    assert s["rows_a"] + s["rows_b"] + s["rows_c"] + s["rows_staged"] == len(tg)
    assert s["rows_a"] + s["rows_b"] + s["rows_c"] > 0
    check_oracle(d0, og, tg, hop, orc.F_NORM | (orc.F_EXTENDED if ext else 0))
    check_image(g, d0, tg, hop=hop, flags=base)
    for leg in (L.F_NO_SMALL, L.F_NO_TABLE, L.F_EDGE_SORTED, L.F_DIRECT, L.F_NO_DIRECT):
        d = g.vicinity_diagrams(tg, hop=hop, flags=base | leg)
        for k in PAIR_KEYS:
            assert np.array_equal(d[k], d0[k]), (leg, k)
        check_image(g, d, tg, hop=hop, flags=base | leg)
    if not ext:
        keep = np.isin(d0["kind"], (L.K_UP, L.K_ESS))
        seg = np.repeat(np.arange(len(tg)), np.diff(d0["poff"]))
        ref_poff = np.concatenate([[0], np.cumsum(np.bincount(seg[keep], minlength=len(tg)))])
        for leg in (0, L.F_NO_SMALL, L.F_DIRECT, L.F_NO_DIRECT):
            d = g.vicinity_diagrams(tg, hop=hop, flags=base | L.F_ASC_ONLY | leg)
            assert np.array_equal(d["poff"], ref_poff), leg
            for k in ("kind", "bv", "dv", "birth", "death"):
                assert np.array_equal(d[k], d0[k][keep]), (leg, k)
            assert np.array_equal(d["status"], d0["status"]), leg
            check_image(g, d, tg, hop=hop, flags=base | L.F_ASC_ONLY | leg)
    g.close()


def test_diagrams_kernel_s_and_staged_rows():
    """a call whose rows are split between kernel S and the staged pipeline: both halves land at their own rows"""
    csr, ne, N = make("computers", 1.0, False)
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    cand = ne[np.random.default_rng(5).choice(len(ne), 4096, replace=False)].astype(np.int32)
    n, m, _ = g.vicinity_sizes(cand, hop=2)
    small, big = np.flatnonzero(n <= 64)[:96], np.flatnonzero(n > 1024)[:24]
    assert len(small) > 0 and len(big) > 0
    tg = cand[np.random.default_rng(6).permutation(np.concatenate([small, big]))]
    n_, m_, _ = g.vicinity_sizes(tg, hop=2)
    d = g.vicinity_diagrams(tg, hop=2, flags=L.F_NORM, cap=int((n_.astype(np.int64) + m_ + 2).sum()))
    s = g.last_small()
    assert s["rows_a"] + s["rows_b"] + s["rows_c"] > 0 and s["rows_staged"] > 0, s
    check_image(g, d, tg, hop=2, flags=L.F_NORM)
    check_oracle(d, og, tg, 2, orc.F_NORM)
    g.close()


def test_asc_only_on_the_graph_row_route():
    csr, ne, N = make("computers", 0.05, False)
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(7)
    tg = ne[rng.choice(len(ne), 128, replace=False)].astype(np.int32)
    fl = L.F_NORM | L.F_ASC_ONLY | L.F_DIRECT
    d = g.vicinity_diagrams(tg, hop=2, flags=fl)
    cn = g.last_counts()
    assert cn["graph_row_route"] > 0 and cn["table_route"] > 0, cn
    check_oracle(d, og, tg, 2, orc.F_NORM, asc=True)
    check_image(g, d, tg, hop=2, flags=fl)
    g.close()


@pytest.mark.parametrize("case", ["node_kd", "forced", "union", "removeinter", "degree", "centrality", "clustering"])
def test_diagrams_modes_and_filtrations(case):
    csr, ne, N = make("pubmed", 0.3, True)
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(9)
    fl, ofl, mode, hop = L.F_NORM | L.F_EXTENDED, orc.F_NORM | orc.F_EXTENDED, L.MODE_EDGE, 2
    if case in ("node_kd", "degree", "centrality", "clustering"):
        ids = rng.choice(N, 64, replace=False).astype(np.int32)
        tg = np.stack([ids, ids], 1)
        mode = L.MODE_NODE
        fl |= L.F_KEEP_ZERO | L.F_NORM_EPS
        ofl |= orc.F_KEEP_ZERO | orc.F_NORM_EPS
        extra = {"degree": (L.F_FILT_DEGREE, orc.F_FILT_DEGREE), "centrality": (L.F_FILT_CENTRALITY, orc.F_FILT_CENTRALITY),
                 "clustering": (L.F_FILT_CLUSTERING, orc.F_FILT_CLUSTERING)}.get(case, (0, 0))
        fl |= extra[0]
        ofl |= extra[1]
    else:
        tg = np.concatenate([ne[rng.choice(len(ne), 64, replace=False)],
                             rng.integers(0, N, size=(16, 2))]).astype(np.int32)
        mode = {"forced": L.MODE_EDGE_FORCED, "union": L.MODE_EDGE_UNION, "removeinter": L.MODE_EDGE_REMOVEINTER}[case]
        hop = 1
    d = g.vicinity_diagrams(tg, hop=hop, mode=mode, flags=fl)
    check_oracle(d, og, tg, hop, ofl, mode=mode)
    check_image(g, d, tg, hop=hop, mode=mode, flags=fl)
    g.close()


def test_diagrams_hks():
    csr, ne, N = make("pubmed", 0.3, True)
    g = api.VicinityGraph(*csr, device=0)
    ids = np.random.default_rng(5).choice(N, 24, replace=False).astype(np.int32)
    tg = np.stack([ids, ids], 1)
    fl = L.F_NORM | L.F_EXTENDED | L.F_KEEP_ZERO | L.F_NORM_EPS | L.F_FILT_HKS
    d = g.vicinity_diagrams(tg, hop=2, mode=L.MODE_NODE, flags=fl)
    det = g.vicinity_detail(tg, hop=2, mode=L.MODE_NODE, flags=fl)
    checked = 0
    for i in range(len(tg)):
        a = g.per_target(det, i)
        assert d["status"][i] == a["status"]
        s, e = int(d["poff"][i]), int(d["poff"][i + 1])
        if not carries_pairs(a["status"]):
            assert s == e
            continue
        assert np.array_equal(d["kind"][s:e], a["pkind"])
        assert np.array_equal(d["bv"][s:e], a["vert"][a["pbv"]]) and np.array_equal(d["dv"][s:e], a["vert"][a["pdv"]])
        assert np.max(np.abs(d["birth"][s:e] - a["pbirth"]), initial=0) < 1e-9
        assert np.max(np.abs(d["death"][s:e] - a["pdeath"]), initial=0) < 1e-9
        checked += 1
    assert checked >= 12
    g.close()


@pytest.mark.parametrize("fast", [0, 1])
def test_handed_back_targets_keep_their_rows(monkeypatch, fast):
    """the hop-distance tie case of test_gpu_parity: kernel 3v hands targets back on the graph-row route, they are redone
    on the materialised route; their pairs sit at their own rows"""
    K = 24
    edges, kap = [(0, 1)], [0.25]
    for i in range(K):
        x = 2 + i
        edges += [(0, x), (1, x)]
        kap += [0.5 + i * 1e-10, 0.5 - ((i * 5) % K) * 1e-10]
        for j in range(i):
            edges.append((2 + j, x)); kap.append(0.3 + (i * K + j) * 1e-9)
    base = 2 + K
    for i in range(30):
        edges += [(base + i, base + (i + 1) % 30), (base + i, base + (i + 7) % 30)]
        kap += [0.1 * ((i % 5) - 2), 0.05 * ((i % 7) - 3)]
    edges.append((0, base)); kap.append(0.4)
    labels, ne = gg.relabel_first_appearance(np.array(edges, dtype=np.int64))
    csr = gg.build_csr(len(labels), ne, np.array(kap))
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    tg = np.concatenate([ne[:40], ne[-50:]]).astype(np.int32)
    if not fast:
        monkeypatch.setenv("TLC_NO_FAST_DIAGRAM", "1")
    fl = L.F_NORM | L.F_DIRECT | L.F_ASC_ONLY
    d = g.vicinity_diagrams(tg, hop=2, flags=fl)
    cn = g.last_counts()
    if not fast:
        assert cn["handed_back"] > 0 and 0 < cn["graph_row_route"] < cn["live"], cn
    check_oracle(d, og, tg, 2, orc.F_NORM, asc=True)
    check_image(g, d, tg, hop=2, flags=fl)
    g.close()


def test_capacity_protocol_and_determinism():
    import ctypes as C
    csr, ne, N = make("pubmed", 0.3, True)
    g = api.VicinityGraph(*csr, device=0)
    tg = ne[np.random.default_rng(2).choice(len(ne), 200, replace=False)].astype(np.int32)
    fl = L.F_NORM | L.F_EXTENDED
    full = g.vicinity_diagrams(tg, hop=2, flags=fl)
    total = int(full["poff"][-1])
    assert total > 0
    p = api.make_params(2, L.MODE_EDGE, "sum", 5, fl, None)
    E = len(tg)
    for cap in (0, total - 1):
        poff = np.full(E + 1, -7, np.int64)
        npairs = np.zeros(E, np.int32)
        bv = np.full(max(cap, 1), -3, np.int32)
        got = C.c_int64(0)
        d = L.Diagrams(cap, poff.ctypes.data, npairs.ctypes.data, None, bv.ctypes.data, None, None, None)
        rc = L.lib().tlc_vicinity_diagrams(g._h, tg.ctypes.data, E, C.byref(p), C.byref(d), None, None, C.byref(got))
        assert rc == L.E_CAPACITY and got.value == total
        assert np.array_equal(poff, full["poff"]) and np.array_equal(npairs, np.diff(full["poff"]))
        assert (bv == -3).all()  # the pair arrays are left untouched
    again = g.vicinity_diagrams(tg, hop=2, flags=fl)
    for k in PAIR_KEYS + ("pi",):
        assert np.array_equal(full[k], again[k]), k
    # the device entry point: the same output, bit for bit
    import torch
    dd = g.vicinity_diagrams_dev(torch.from_numpy(tg).cuda(), hop=2, flags=fl, want_pi=True)
    for k in ("poff", "kind", "bv", "dv", "birth", "death", "status", "pi"):
        assert np.array_equal(dd[k].cpu().numpy(), full[k]), k
    g.close()


def test_segments_reproduce_the_image_rows():
    csr, ne, N = make("cora", 1.0, False)
    g = api.VicinityGraph(*csr, device=0)
    tg = ne[np.random.default_rng(4).choice(len(ne), 64, replace=False)].astype(np.int32)
    d = g.vicinity_diagrams(tg, hop=2, flags=L.F_NORM | L.F_EXTENDED)
    checked = 0
    for i in range(len(tg)):
        if d["status"][i] != L.ST_OK:
            continue
        a, b = int(d["poff"][i]), int(d["poff"][i + 1])
        img = api.pimg_transform(np.stack([d["birth"][a:b], d["death"][a:b]], 1)).reshape(-1)
        den = np.where(d["pi"][i] != 0, np.abs(d["pi"][i]), 1.0)
        assert np.max(np.abs(img - d["pi"][i]) / den) < 1e-13, i
        checked += 1
    assert checked > 32
    g.close()


def test_full_size_computers_sampled():
    csr, ne, N = make("computers", 1.0, False)
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(42)
    tg = ne[rng.choice(len(ne), 4096, replace=False)].astype(np.int32)
    fl = L.F_NORM | L.F_ASC_ONLY
    d = g.vicinity_diagrams(tg, hop=2, flags=fl)
    check_oracle(d, og, tg, 2, orc.F_NORM, asc=True, rows=sorted(rng.choice(len(tg), 64, replace=False)))
    check_image(g, d, tg, hop=2, flags=fl)
    perm = rng.permutation(len(tg))
    dp = g.vicinity_diagrams(tg[perm], hop=2, flags=fl)
    assert np.array_equal(np.diff(dp["poff"]), np.diff(d["poff"])[perm])
    for j, i in enumerate(perm[:512]):
        a, b = int(d["poff"][i]), int(d["poff"][i + 1])
        c0, c1 = int(dp["poff"][j]), int(dp["poff"][j + 1])
        for k in ("kind", "bv", "dv", "birth", "death"):
            assert np.array_equal(dp[k][c0:c1], d[k][a:b]), (j, k)
    g.close()
