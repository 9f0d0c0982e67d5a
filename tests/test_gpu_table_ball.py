"""Kernel 1t's tables are built per root over the subgraph induced by the root's k-hop ball.  They depend on the hop and
the summation rule, so one graph object that switches either must rebuild them; and a vertex of S whose whole-graph
shortest path leaves the ball must still get its distance inside S."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle as orc
from helpers import rel_err
from tlc_b200 import _lib as L
from tlc_b200 import api, graphgen as gg

ROUTE = L.F_DIRECT | L.F_NO_SMALL  # graph-row route, no fused small-vicinity kernels: every vicinity reaches kernel 1t


def test_table_rebuild_on_hop_sum_and_mode_switches():
    c = gg.make_config("computers", scale=0.05)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    rng = np.random.default_rng(5)
    edges = ne[rng.choice(len(ne), 256, replace=False)].astype(np.int32)
    nodes = rng.choice(len(labels), 128, replace=False)
    node_tg = np.stack([nodes, nodes], 1).astype(np.int32)
    seq = [(2, L.MODE_EDGE, 0), (1, L.MODE_EDGE, 0), (2, L.MODE_EDGE, 0), (2, L.MODE_EDGE, L.F_SUM_PLAIN),
           (2, L.MODE_NODE, L.F_SUM_PLAIN), (1, L.MODE_NODE, 0), (2, L.MODE_EDGE, 0)]
    for hop, mode, plain in seq:
        tg = edges if mode == L.MODE_EDGE else node_tg
        fl = L.F_NORM | plain | ROUTE
        pi, status, cnt = g.vicinity_pi(tg, hop=hop, mode=mode, flags=fl)
        ctx = "hop %d mode %d plain %d" % (hop, mode, plain)
        assert g.last_counts()["table_route"] > 0, ctx
        pi_b, status_b, cnt_b = g.vicinity_pi(tg, hop=hop, mode=mode, flags=fl | L.F_NO_TABLE)  # kernel 1b
        assert g.last_counts()["table_route"] == 0, ctx
        assert np.array_equal(pi, pi_b) and np.array_equal(status, status_b) and cnt == cnt_b, ctx
        o = og.run_batch(tg, hop=hop, mode=mode, flags=orc.F_NORM | (orc.F_SUM_PLAIN if plain else 0))
        assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"], ctx
        assert rel_err(pi, o["pi"]) < 1e-5, ctx
    g.close()


def test_whole_graph_path_through_a_vertex_outside_the_ball():
    # target (0, 1), hop 2: S = ball(0) & ball(1) = {0, 1, 2, 3, 4}.  From root 0 the whole graph's shortest path to 3
    # is 0-4-5-6-3 (0.4) through 6, three hops from 0; inside S it is 0-2-3 (3.8).  Weights are kappa + 1.
    edges = np.array([[0, 1], [0, 2], [1, 2], [2, 3], [0, 4], [4, 5], [5, 6], [6, 3], [1, 7], [7, 8], [8, 3]], np.int64)
    kappa = np.array([0.0, 0.9, 0.0, 0.9, -0.9, -0.9, -0.9, -0.9, -0.5, 0.3, 0.7])
    csr = gg.build_csr(9, edges, kappa)
    g = api.VicinityGraph(*csr, device=0)
    og = orc.OracleGraph(*csr)
    tg = np.array([[0, 1], [1, 0], [0, 2], [2, 3], [1, 7], [3, 6]], np.int32)
    for plain in (0, L.F_SUM_PLAIN):
        oflags = orc.F_NORM | (orc.F_SUM_PLAIN if plain else 0)
        d = g.vicinity_detail(tg, hop=2, flags=L.F_NORM | plain | ROUTE | L.F_ASC_ONLY)
        assert g.last_counts()["table_route"] > 0
        for i, (u, v) in enumerate(tg):
            a = g.per_target(d, i)
            o = og.run_one(int(u), int(v), hop=2, flags=oflags)
            ctx = "target (%d, %d)" % (u, v)
            assert a["status"] == o["status"] and np.array_equal(a["vert"], o["vert"]), ctx
            assert np.array_equal(a["fval"], o["fval"]), ctx
        pi, status, cnt = g.vicinity_pi(tg, hop=2, flags=L.F_NORM | plain | ROUTE)
        assert g.last_counts()["table_route"] > 0
        o = og.run_batch(tg, hop=2, flags=oflags)
        assert np.array_equal(status, o["status"]) and cnt == o["cnt_compute"]
        assert rel_err(pi, o["pi"]) < 1e-5
    g.close()
