"""SURVEY.md row N4 on the GPU: kernel 6 (tlc_ollivier_ricci) against the CPU restatement oracle/ricci_oracle.py of the
published GraphRicciCurvature + POT algorithm (parity unpinned by the reference, see that file), and against closed forms
of the exact transport problem on toy graphs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import helpers as H
import ricci_oracle as ro
from tlc_b200 import api, graphgen as gg

TOL = 1e-9  # float64 Sinkhorn on both sides; only the summation order inside the matrix-vector products differs


def csr_of(n, edges):
    e = np.asarray(edges, dtype=np.int64)
    return gg.build_csr(n, e, np.zeros(len(e)))[:2]


def test_toy_graphs_closed_forms():
    for n in (4, 5, 8):
        rp, col = csr_of(n, [(i, j) for i in range(n) for j in range(i + 1, n)])
        k = api.ollivier_ricci(rp, col)
        assert np.allclose(k, 1.0 - abs(0.5 - 0.5 / (n - 1)), atol=1e-2)
    rp, col = csr_of(12, [(i, (i + 1) % 12) for i in range(12)])
    assert np.allclose(api.ollivier_ricci(rp, col), 0.0, atol=1e-2)


@pytest.mark.parametrize("name,scale", [("cora", 0.2), ("pubmed", 0.05), ("computers", 0.03)])
def test_random_graph_matches_restatement(name, scale):
    c = gg.make_config(name, scale=scale)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    rp, col, _ = gg.build_csr(len(labels), ne, c["kappa"])
    k, it = api.ollivier_ricci(rp, col, return_iters=True)
    rng = np.random.default_rng(1)
    # both directions of an edge carry the same value
    for x in rng.choice(len(labels), 20):
        for q in range(rp[x], rp[x + 1]):
            y = col[q]
            m = rp[y] + np.searchsorted(col[rp[y]:rp[y + 1]], x)
            assert k[q] == k[m]
    for x, y in ne[rng.choice(len(ne), 40, replace=False)]:
        q = rp[x] + np.searchsorted(col[rp[x]:rp[x + 1]], y)
        a, src = ro.support(rp, col, int(min(x, y)))
        b, tgt = ro.support(rp, col, int(max(x, y)))
        d = ro.hop_costs(rp, col, src, tgt)
        m, cpt = ro.sinkhorn2(a, b, d)
        assert abs(k[q] - (1.0 - m)) < TOL, (x, y, k[q], 1.0 - m)
        assert it[q] == cpt
    assert np.all(k <= 1.0 + 1e-12) and np.all(k >= -2.0)


def test_mirror_returns_the_reference_layout():
    from sg2dgm.feature_cache import compute_ricci_curvature
    ei = np.array([[10, 20, 30, 10, 20, 10], [20, 30, 10, 40, 10, 10]])   # a duplicate (20,10) and a self-loop (10,10)
    rl = compute_ricci_curvature(edge_index=ei)
    assert rl == sorted(rl) and len(rl) == 8                                   # 4 undirected edges, both directions
    d = {(a, b): k for a, b, k in rl}
    assert all(d[(a, b)] == d[(b, a)] for a, b in d)


# ---- the hub graph (tests/helpers.py): all three launch classes, the 3000-neighbour cut, both edge orientations ----

def oracle_edge(rp, col, x, y, alpha=0.5, keep_largest=True):
    """(curvature, Sinkhorn iterations) of edge (x, y) from the oracle, source side = the smaller id as in kernel 6;
    keep_largest=False keeps the 3000 SMALLEST neighbour ids instead (the wrong cut)"""
    x, y = min(int(x), int(y)), max(int(x), int(y))
    sup = []
    for z in (x, y):
        m, nodes = ro.support(rp, col, z, alpha)
        nb = col[rp[z]:rp[z + 1]]
        if not keep_largest and len(nb) > ro.NBR_TOPK:
            nodes = np.append(nb[:ro.NBR_TOPK], z)
        sup.append((m, nodes))
    m, cpt = ro.sinkhorn2(sup[0][0], sup[1][0], ro.support_costs(rp, col, sup[0][1], sup[1][1]))
    return 1.0 - m, cpt


def entry(rp, col, x, y):
    return int(rp[x] + np.searchsorted(col[rp[x]:rp[x + 1]], y))


def mirror(rp, col):
    N = len(rp) - 1
    src = np.repeat(np.arange(N, dtype=np.int64), np.diff(rp))
    return np.searchsorted(src * N + col, col.astype(np.int64) * N + src)


@pytest.fixture(scope="module")
def hub():
    rp, col, ids = H.ricci_hub_graph()
    k, it = api.ollivier_ricci(rp, col, return_iters=True)
    return rp, col, ids, k, it


def check_edges(rp, col, edges, k, it, alpha):
    for x, y in edges:
        q = entry(rp, col, x, y)
        ref, cpt = oracle_edge(rp, col, x, y, alpha)
        assert abs(k[q] - ref) < TOL and it[q] == cpt, (alpha, x, y, k[q], ref, it[q], cpt)


def test_hub_graph_every_class_against_the_oracle(hub):
    import torch
    rp, col, ids, k, it = hub
    e, cls = H.ricci_classes(rp, col)
    counts = np.bincount(cls, minlength=3)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    print("kernel 6 classes on the hub graph: %d / %d / %d edges, grids %d / %d / %d"
          % (counts[0], counts[1], counts[2], 8 * sms, 2 * sms, sms))
    assert counts[0] > 8 * sms and counts[1] > 2 * sms and counts[2] > sms   # every class loops over its slab / smem
    deg = np.diff(rp)
    assert deg.max() > ro.NBR_TOPK                                            # the cut runs
    assert np.all(it >= 1)                                                    # every entry was computed
    # the cut-sensitive edge: keeping the smallest ids of h3500, or all 3500, gives another curvature than the kernel's
    x, y = ids["cut"], ids["h3500"]
    right, cpt = oracle_edge(rp, col, x, y)
    wrong = oracle_edge(rp, col, x, y, keep_largest=False)[0]
    b, tgt = ro.support(rp, col, y, topk=3500)
    a, src = ro.support(rp, col, x)
    uncut = 1.0 - ro.sinkhorn2(a, b, ro.support_costs(rp, col, src, tgt))[0]
    assert abs(wrong - right) > 1e-6 and abs(uncut - right) > 1e-6, (right, wrong, uncut)
    q = entry(rp, col, x, y)
    assert abs(k[q] - right) < TOL and it[q] == cpt, ("cut", k[q], right, wrong, uncut)
    # boundary edges: the pairs that straddle each class limit, and every special node's edge to its smallest and largest
    # neighbour (the node is the larger endpoint of the one and the smaller of the other where it has neighbours on both
    # sides), then ~20 random edges per class
    edges = [(ids[p], ids[q]) for p, q in (("h3500", "h3001"), ("h3001", "h3000"), ("d1024", "d1023"), ("d120", "d119"))]
    for name in ("h3500", "h3001", "h3000", "d1024", "d1023", "d120", "d119"):
        nb = col[rp[ids[name]]:rp[ids[name] + 1]]
        edges += [(ids[name], nb[0]), (ids[name], nb[-1])]
    rng = np.random.default_rng(4)
    for c in range(3):
        edges += [tuple(p) for p in e[rng.choice(np.flatnonzero(cls == c), 20, replace=False)]]
    check_edges(rp, col, edges, k, it, 0.5)


@pytest.mark.parametrize("alpha", [0.0, 1.0, 0.25])
def test_hub_graph_other_alphas(alpha):
    """alpha = 0 puts no mass on the node itself, alpha = 1 none on its neighbours: a 1 / 0 = inf times a zero entry of v
    makes u NaN in the first iteration, and Sinkhorn reverts to its start (POT's "numerical errors" exit)"""
    rp, col, ids = H.ricci_hub_graph()
    k, it = api.ollivier_ricci(rp, col, alpha=alpha, return_iters=True)
    e, cls = H.ricci_classes(rp, col)
    rng = np.random.default_rng(5)
    edges = [(ids["h3001"], ids["h3000"]), (ids["d1024"], ids["d1023"]), (ids["d120"], ids["d119"]), (ids["cut"], ids["h3500"])]
    for c in range(3):
        edges += [tuple(p) for p in e[rng.choice(np.flatnonzero(cls == c), 5, replace=False)]]
    check_edges(rp, col, edges, k, it, alpha)
    if alpha in (0.0, 1.0):
        assert np.all(it == 0)
    else:
        assert np.all(it >= 1)


def test_hub_graph_bit_exact(hub):
    rp, col, ids, k, it = hub
    m = mirror(rp, col)
    assert np.array_equal(k[m], k) and np.array_equal(it[m], it)        # both directions of every entry
    k2, it2 = api.ollivier_ricci(rp, col, return_iters=True)
    assert np.array_equal(k2, k) and np.array_equal(it2, it)            # a second call
    # a disjoint component in front (ids 0 .. M-1): a star of degree 200 (class 1), one of degree 1100 (class 2) and a
    # sparse random part (class 0) shift every class's edge order, the CTA and slab each edge runs on, and all node ids
    M = 1700
    rs = np.random.RandomState(6)
    comp = [(0, i) for i in range(1, 201)] + [(201, i) for i in range(202, 1302)]
    comp += [(int(a), int(b)) for a, b in rs.randint(202, M, (2 * M, 2)) if a != b]
    comp = np.unique(np.sort(np.asarray(comp, dtype=np.int64), axis=1), axis=0)
    e, _ = H.ricci_classes(rp, col)
    rpc, colc, _ = gg.build_csr(M + len(rp) - 1, np.concatenate([comp, e + M]), np.zeros(len(comp) + len(e)))
    _, cls_c = H.ricci_classes(rpc, colc)
    assert np.all(np.bincount(cls_c[:len(comp)], minlength=3) > 0)
    kc, itc = api.ollivier_ricci(rpc, colc, return_iters=True)
    off = int(rpc[M])
    assert np.array_equal(kc[off:], k) and np.array_equal(itc[off:], it)
