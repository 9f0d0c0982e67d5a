"""SURVEY.md row N4 -- the Ollivier-Ricci (Sinkhorn) curvature precompute.  PARITY UNPINNED by the reference (its two
third-party packages are neither vendored, pinned nor installed here): the CPU restatement oracle/ricci_oracle.py is
pinned against closed forms of the exact transport problem on toy graphs, to the accuracy the entropic regularisation
(reg = 0.1 against hop costs) leaves."""
import itertools

import numpy as np
import pytest

import helpers as H
import ricci_oracle as ro
from tlc_b200 import graphgen as gg


def csr_of(n, edges):
    e = np.asarray(edges, dtype=np.int64)
    return gg.build_csr(n, e, np.zeros(len(e)))[:2]


def cycle(n):
    return csr_of(n, [(i, (i + 1) % n) for i in range(n)])


def complete(n):
    return csr_of(n, [(i, j) for i in range(n) for j in range(i + 1, n)])


def test_long_cycle_is_flat():
    rp, col = cycle(12)
    k = ro.compute_ricci_curvature(rp, col)
    assert np.allclose(k, 0.0, atol=1e-2)          # W1 = 1 on a cycle of length >= 6: kappa = 0


def test_complete_graph_closed_form():
    for n in (4, 5, 8):
        rp, col = complete(n)
        k = ro.compute_ricci_curvature(rp, col)
        expect = 1.0 - abs(0.5 - 0.5 / (n - 1))    # move the excess alpha - (1-alpha)/(n-1) from x to y
        assert np.allclose(k, expect, atol=1e-2), (n, k[:3], expect)


def test_star_and_path_against_the_exact_lp():
    # leaf - centre edges of a star, and the edges of a short path: exact W1 from a linear programme
    star = csr_of(6, [(0, i) for i in range(1, 6)])
    path = csr_of(6, [(i, i + 1) for i in range(5)])
    for rp, col in (star, path):
        for x in range(len(rp) - 1):
            for e in range(rp[x], rp[x + 1]):
                y = int(col[e])
                a, src = ro.support(rp, col, x)
                b, tgt = ro.support(rp, col, y)
                d = ro.hop_costs(rp, col, src, tgt)
                assert abs(ro.sinkhorn2(a, b, d)[0] - ro.exact_w1(a, b, d)) < 1e-2
                assert abs(ro.edge_curvature(rp, col, x, y) - ro.edge_curvature(rp, col, y, x)) < 1e-9   # symmetric


def test_random_graph_against_the_exact_lp_and_mass_conservation():
    c = gg.make_config("cora", scale=0.05)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    rp, col, _ = gg.build_csr(len(labels), ne, c["kappa"])
    rng = np.random.default_rng(0)
    for x, y in ne[rng.choice(len(ne), 12, replace=False)]:
        a, src = ro.support(rp, col, int(x))
        b, tgt = ro.support(rp, col, int(y))
        assert abs(a.sum() - 1.0) < 1e-12 and abs(b.sum() - 1.0) < 1e-12
        d = ro.hop_costs(rp, col, src, tgt)
        assert d.max() <= 3 and d.min() >= 0           # supports of an edge are at most 3 hops apart
        m, it = ro.sinkhorn2(a, b, d)
        assert it <= ro.NUM_ITER_MAX
        assert abs(m - ro.exact_w1(a, b, d)) < 1e-2
        assert -2.0 <= 1.0 - m <= 1.0


def star(k):
    return csr_of(k + 1, [(0, i) for i in range(1, k + 1)])


def test_support_costs_equal_hop_costs():
    graphs = [cycle(12), complete(5), csr_of(6, [(0, i) for i in range(1, 6)]), csr_of(6, [(i, i + 1) for i in range(5)])]
    for rp, col in graphs:                                     # toy graphs: every directed entry
        for x in range(len(rp) - 1):
            for y in col[rp[x]:rp[x + 1]]:
                src, tgt = ro.support(rp, col, x)[1], ro.support(rp, col, int(y))[1]
                assert np.array_equal(ro.support_costs(rp, col, src, tgt), ro.hop_costs(rp, col, src, tgt))
    c = gg.make_config("cora", scale=0.2)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    rp, col, _ = gg.build_csr(len(labels), ne, c["kappa"])
    rng = np.random.default_rng(2)
    for x, y in ne[rng.choice(len(ne), 30, replace=False)]:
        src, tgt = ro.support(rp, col, int(x))[1], ro.support(rp, col, int(y))[1]
        d = ro.support_costs(rp, col, src, tgt)
        assert np.array_equal(d, ro.hop_costs(rp, col, src, tgt)) and set(np.unique(d)) <= {0.0, 1.0, 2.0, 3.0}
    # the hub graph, at edges whose source side (smaller id) has a small support: one BFS per source node
    rp, col, ids = H.ricci_hub_graph()
    e, cls = H.ricci_classes(rp, col)
    small = np.diff(rp)[e[:, 0]] <= 12
    picks = [rng.choice(np.flatnonzero(small & (cls == k)), 4, replace=False) for k in range(3)]
    picks.append(np.flatnonzero((e[:, 0] == ids["cut"]) & (e[:, 1] == ids["h3500"])))
    picks = np.concatenate(picks)
    assert len(picks) == 13
    seen = set()
    for x, y in e[picks]:
        src, tgt = ro.support(rp, col, int(x))[1], ro.support(rp, col, int(y))[1]
        d = ro.support_costs(rp, col, src, tgt)
        assert np.array_equal(d, ro.hop_costs(rp, col, src, tgt)), (x, y)
        seen |= set(np.unique(d))
    assert seen == {0.0, 1.0, 2.0, 3.0}


@pytest.mark.parametrize("alpha", [0.5, 0.3])
def test_neighbour_mass_is_normalised_by_a_left_to_right_sum(alpha):
    w = np.e ** (-1.0 ** 2)
    numpy_differs = False
    for k in (1, 120, 121, 1024, 3000):
        rp, col = star(k)
        m, nodes = ro.support(rp, col, 0, alpha)
        s = list(itertools.accumulate([w] * k))[-1]           # e^-1 added k times, one after the other
        assert np.array_equal(nodes, np.append(np.arange(1, k + 1), 0))
        assert np.all(m[:-1] == (1.0 - alpha) * w / s) and m[-1] == alpha, k
        numpy_differs |= bool((1.0 - alpha) * w / np.full(k, w).sum() != m[0])
    assert numpy_differs                                       # the summation rule shows in the masses


def test_truncation_keeps_the_3000_largest_ids():
    rp, col, ids = H.ricci_hub_graph()
    w = np.e ** (-1.0 ** 2)
    s3000 = list(itertools.accumulate([w] * 3000))[-1]
    for name, drop in (("h3500", 500), ("h3001", 1), ("h3000", 0)):
        x = ids[name]
        nb = col[rp[x]:rp[x + 1]]
        m, nodes = ro.support(rp, col, x)
        assert np.array_equal(nodes, np.append(np.sort(nb)[drop:], x)), name
        assert len(m) == 3001 and np.all(m[:-1] == 0.5 * w / s3000) and m[-1] == 0.5
    # the cut node's neighbours (other than h3500) are all among the dropped ones
    cut_nb = col[rp[ids["cut"]]:rp[ids["cut"] + 1]]
    kept = ro.support(rp, col, ids["h3500"])[1][:-1]
    assert cut_nb[-1] == ids["h3500"] and not np.isin(cut_nb[:-1], kept).any()


def test_hub_graph_reaches_every_launch_class():
    rp, col, ids = H.ricci_hub_graph()
    N = len(rp) - 1
    deg = np.diff(rp)
    e, cls = H.ricci_classes(rp, col)
    assert N % 32 != 0 and ids["h3500"] == N - 1 and deg.max() == 3500
    for name, d in (("h3500", 3500), ("h3001", 3001), ("h3000", 3000), ("d1024", 1024), ("d1023", 1023), ("d120", 120),
                    ("d119", 119)):
        assert deg[ids[name]] == d
    for name in ("h3001", "h3000"):                           # both orientations: smaller endpoint and larger endpoint
        assert (e[:, 0] == ids[name]).any() and (e[:, 1] == ids[name]).any()
    # more edges per class than a B200 (148 SMs) launches CTAs for it (8 / 2 / 1 per SM): every CTA loops
    counts = np.bincount(cls, minlength=3)
    assert counts[0] > 148 * 8 and counts[1] > 148 * 2 and counts[2] > 148 * 1, counts
    size = np.minimum(deg, 3000) + 1
    big = np.maximum(size[e[:, 0]], size[e[:, 1]])
    for s in (120, 121, 1024, 1025, 3001):                     # both sides of every class limit
        assert (big == s).any(), s
