"""Kernel 1t runs both roots of a target through the same passes when their two states fit its shared memory, and one
root at a time otherwise (larger vicinities, NODE mode, TLC_TABLE_ONE_ROOT=1).  Both give what kernel 1b
(TLC_F_NO_TABLE) gives, bit for bit, on every path of the kernel."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from tlc_b200 import _lib as L
from tlc_b200 import api, graphgen as gg

ROUTE = L.F_DIRECT | L.F_NO_SMALL  # graph-row route, no fused small-vicinity kernels: every vicinity reaches kernel 1t


def three_ways(g, tg, monkeypatch, flags, **kw):
    """the two-root path, the forced one-root path and kernel 1b give equal pi / status; returns the first's statistics"""
    out = []
    for one_root, extra in ((False, 0), (True, 0), (False, L.F_NO_TABLE)):
        if one_root:
            monkeypatch.setenv("TLC_TABLE_ONE_ROOT", "1")
        else:
            monkeypatch.delenv("TLC_TABLE_ONE_ROOT", raising=False)
        pi, st, cnt = g.vicinity_pi(tg, flags=flags | extra, **kw)
        out.append((pi, st, cnt, g.last_counts()))
    monkeypatch.delenv("TLC_TABLE_ONE_ROOT", raising=False)
    (pi2, st2, c2, n2), (pi1, st1, c1, n1), (pib, stb, cb, nb) = out
    assert np.array_equal(pi2, pi1) and np.array_equal(st2, st1) and c2 == c1
    assert np.array_equal(pi2, pib) and np.array_equal(st2, stb) and c2 == cb
    assert n1["table_route"] == n2["table_route"] > 0 and n1["table_two_root"] == 0
    assert nb["table_route"] == 0 and nb["table_two_root"] == 0
    return n2


def computers():
    c = gg.make_config("computers")
    labels, ne = gg.relabel_first_appearance(c["edges"])
    return ne, api.VicinityGraph(*gg.build_csr(len(labels), ne, c["kappa"]), device=0)


@pytest.mark.parametrize("plain", [0, L.F_SUM_PLAIN], ids=["neumaier", "plain"])
def test_headline_shaped_both_sides_of_the_fit_limit(monkeypatch, plain):
    # full-size Computers-shaped graph, 2-hop edge vicinities: most fit the two-root state, the largest (n above about
    # 10 000 of the 13 752 vertices) do not -- both kinds in one call
    ne, g = computers()
    rng = np.random.default_rng(11)
    tg = ne[rng.choice(len(ne), 768, replace=False)].astype(np.int32)
    cn = three_ways(g, tg, monkeypatch, hop=2, flags=L.F_NORM | plain | ROUTE)
    assert 0 < cn["table_two_root"] < cn["table_route"], cn
    # hop 1: every vicinity fits
    cn = three_ways(g, tg, monkeypatch, hop=1, flags=L.F_NORM | plain | ROUTE)
    assert cn["table_two_root"] > 0, cn
    g.close()


def test_node_mode_runs_one_root(monkeypatch):
    ne, g = computers()
    rng = np.random.default_rng(12)
    nodes = rng.choice(int(ne.max()) + 1, 256, replace=False)
    tg = np.stack([nodes, nodes], 1).astype(np.int32)
    cn = three_ways(g, tg, monkeypatch, hop=2, mode=L.MODE_NODE, flags=L.F_NORM | ROUTE)
    assert cn["table_two_root"] == 0, cn
    g.close()


def invalid_clique_graph(m=40):
    """Roots 0 and 1, a clique C of m vertices joined to both by heavy edges.  Each root also reaches C cheaply through
    a vertex of its own that lies outside the other root's 2-hop ball (0 - a - h - C, 1 - b - h2 - C), so inside S =
    ball(0) & ball(1) = {0, 1, C, h, h2} every vertex of C is invalid for both roots, and their m (m - 1) / 2 clique
    edges overflow the 4 n slots of the invalid-invalid list: the rescan path."""
    C = list(range(2, 2 + m))
    a, h, b, h2 = 2 + m, 3 + m, 4 + m, 5 + m
    edges, kappa = [], []
    def add(x, y, k):
        edges.append((x, y)); kappa.append(k)
    for i, x in enumerate(C):
        add(0, x, 0.8); add(1, x, 0.85); add(h, x, -0.9 + 0.001 * i); add(h2, x, -0.88 + 0.001 * i)
        for y in C[i + 1:]:
            add(x, y, -0.5 + 0.01 * ((x * 7 + y * 3) % 11))
    add(0, a, -0.9); add(a, h, -0.9); add(1, b, -0.9); add(b, h2, -0.9)
    n = h2 + 1
    return n, np.array(edges, np.int64), np.array(kappa), a, b


@pytest.mark.parametrize("plain", [0, L.F_SUM_PLAIN], ids=["neumaier", "plain"])
def test_mostly_invalid_vicinities_root_outside_s_and_u_equal_v(monkeypatch, plain):
    n, edges, kappa, a, b = invalid_clique_graph()
    g = api.VicinityGraph(*gg.build_csr(n, edges, kappa), device=0)
    tg = np.array([[0, 1], [1, 0], [0, 5], [3, 1], [0, a], [a, b], [b, 1], [5, 5], [0, 0]] * 8, np.int32)
    cn = three_ways(g, tg, monkeypatch, hop=2, flags=L.F_NORM | plain | ROUTE)
    assert cn["table_two_root"] > 0, cn
    g.close()
