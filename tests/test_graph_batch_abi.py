"""Graph batches without a GPU: tlc_graph_batch_create rejects every malformed structure with a message naming the
offending graph or edge, the diagram and gradient calls reject bad flags and NULL pointers before any CUDA call,
api.normalize_edge_index keeps the first occurrence of every undirected edge in input order, and the numpy restatement
of the gradient scatter that the GPU tests use as their reference is pinned to autograd of the plain gather."""
import ctypes as C

import numpy as np
import pytest
import torch

from tlc_b200 import _lib as L
from tlc_b200 import api


def scatter_grad(poff, bv, dv, grad_birth, grad_death, N):
    """tlc_graph_batch_grad_dev restated: grad_f[v] = sum over points k in [poff[0], poff[D]) of grad_birth[k] where
    bv[k] == v and grad_death[k] where dv[k] == v, added in increasing k, birth term before death term, from 0.0.  A NULL
    gradient (None) counts as zeros."""
    g = np.zeros(N)
    for k in range(int(poff[0]), int(poff[-1])):
        if grad_birth is not None:
            g[bv[k]] += grad_birth[k]
        if grad_death is not None:
            g[dv[k]] += grad_death[k]
    return g


def create(noff, eoff, ea, eb, D=None):
    noff = np.ascontiguousarray(noff, np.int64)
    eoff = np.ascontiguousarray(eoff, np.int64)
    ea = np.ascontiguousarray(ea, np.int32)
    eb = np.ascontiguousarray(eb, np.int32)
    h = C.c_void_p()
    rc = L.lib().tlc_graph_batch_create(0, noff.size - 1 if D is None else D, noff.ctypes.data, eoff.ctypes.data,
                                        ea.ctypes.data if ea.size else None, eb.ctypes.data if eb.size else None,
                                        C.byref(h))
    return rc, L.lib().tlc_last_error().decode()


# two graphs: vertices 0..2 and 3..5, edges 0..1 and 2..3
GOOD = dict(noff=[0, 3, 6], eoff=[0, 2, 4], ea=[0, 1, 3, 4], eb=[1, 2, 4, 5])


@pytest.mark.parametrize("change, words", [
    (dict(ea=[0, 1, 3, 7]), ["edge 3", "graph 1", "outside"]),                 # out of the batch's range
    (dict(ea=[0, 1, 3, -1]), ["edge 3", "graph 1", "outside"]),
    (dict(ea=[0, 1, 3, 2]), ["edge 3 (2, 5)", "graph 1", "outside"]),           # an edge into the other graph
    (dict(ea=[0, 1, 1, 4], eb=[1, 2, 4, 5]), ["edge 2", "graph 1", "outside"]),
    (dict(ea=[0, 2, 3, 4], eb=[1, 2, 4, 5]), ["edge 1 (2, 2)", "graph 0", "self-loop"]),
    (dict(ea=[0, 0, 3, 4], eb=[1, 1, 4, 5]), ["edge 1 (0, 1)", "graph 0", "repeats edge 0"]),   # same direction
    (dict(ea=[0, 1, 3, 4], eb=[1, 0, 4, 5]), ["edge 1 (1, 0)", "graph 0", "repeats edge 0"]),   # reversed
    (dict(ea=[0, 1, 3, 4], eb=[1, 2, 4, 3]), ["edge 3 (4, 3)", "graph 1", "repeats edge 2"]),
    (dict(noff=[0, 4, 3]), ["noff is not monotone at graph 1"]),
    (dict(eoff=[0, 3, 2]), ["eoff is not monotone at graph 1"]),
    (dict(noff=[1, 3, 6]), ["noff[0] and eoff[0] must be 0"]),
    (dict(eoff=[1, 2, 4]), ["noff[0] and eoff[0] must be 0"]),
])
def test_create_rejects(change, words):
    a = dict(GOOD)
    a.update(change)
    rc, msg = create(**a)
    assert rc == L.E_INVALID
    for w in words:
        assert w in msg, (w, msg)


def test_create_rejects_sizes_and_pointers():
    rc, msg = create([0, 3], [0, 1], [], [])  # one edge, no edge arrays
    assert rc == L.E_INVALID and "ea and eb" in msg
    rc, msg = create([0, 3], [0, 0], [], [], D=-1)
    assert rc == L.E_INVALID and "D must be" in msg
    rc, msg = create([0, 1 << 31], [0, 0], [], [])
    assert rc == L.E_INVALID and "noff[D]" in msg
    h = C.c_void_p()
    assert L.lib().tlc_graph_batch_create(0, 0, None, None, None, None, C.byref(h)) == L.E_INVALID
    noff = np.zeros(1, np.int64)
    assert L.lib().tlc_graph_batch_create(0, 0, noff.ctypes.data, noff.ctypes.data, None, None, None) == L.E_INVALID


def test_repeated_edge_reports_the_earliest_repetition():
    # edges (0,1) (1,2) (2,0) (2,1) (1,0): the first repetition is edge 3, of edge 1
    rc, msg = create([0, 3], [0, 5], [0, 1, 2, 2, 1], [1, 2, 0, 1, 0])
    assert rc == L.E_INVALID and "edge 3 (2, 1)" in msg and "repeats edge 1" in msg


def test_diagram_and_grad_calls_check_before_cuda():
    lib = L.lib()
    poff = np.zeros(3, np.int64)
    d = L.Diagrams(100, poff.ctypes.data, None, None, None, None, None, None)
    f = np.zeros(4)
    for bad in (L.F_NORM, L.F_EDGE_SORTED, L.F_DIRECT, 1 << 20, L.F_EXTENDED | L.F_ASC_ONLY):
        assert lib.tlc_graph_batch_diagrams_dev(None, f.ctypes.data, bad, C.byref(d), None, None) == L.E_INVALID
        assert "TLC_F_" in lib.tlc_last_error().decode()
    assert lib.tlc_graph_batch_diagrams_dev(None, f.ctypes.data, 0, None, None, None) == L.E_INVALID
    assert "out and out->poff" in lib.tlc_last_error().decode()
    d0 = L.Diagrams(100, None, None, None, None, None, None, None)
    assert lib.tlc_graph_batch_diagrams_dev(None, f.ctypes.data, 0, C.byref(d0), None, None) == L.E_INVALID
    assert lib.tlc_graph_batch_diagrams_dev(None, f.ctypes.data, 0, C.byref(d), None, None) == L.E_INVALID
    assert "batch is NULL" in lib.tlc_last_error().decode()
    bv = np.zeros(4, np.int32)
    dg = L.Diagrams(100, poff.ctypes.data, None, None, bv.ctypes.data, None, None, None)
    assert lib.tlc_graph_batch_grad_dev(None, C.byref(dg), None, None, f.ctypes.data, None) == L.E_INVALID
    assert "d->dv" in lib.tlc_last_error().decode()
    assert lib.tlc_graph_batch_grad_dev(None, None, None, None, f.ctypes.data, None) == L.E_INVALID
    dg.dv = bv.ctypes.data
    assert lib.tlc_graph_batch_grad_dev(None, C.byref(dg), None, None, f.ctypes.data, None) == L.E_INVALID
    assert "batch is NULL" in lib.tlc_last_error().decode()
    b = C.c_int64(0)
    assert lib.tlc_graph_batch_pair_bound(None, C.byref(b)) == L.E_INVALID


def plain_dedup(ptr, edge_index):
    """first occurrence of every undirected edge, in input order, grouped by graph (stable)"""
    seen, kept = set(), []
    for a, b in zip(*[list(map(int, r)) for r in edge_index]):
        key = (min(a, b), max(a, b))
        if key not in seen:
            seen.add(key)
            kept.append((a, b))
    D = len(ptr) - 1
    graph = lambda v: max(0, min(D - 1, int(np.searchsorted(ptr, v, side="right")) - 1))
    kept.sort(key=lambda e: graph(e[0]))  # (Python's sort is stable)
    eoff = [0] * (D + 1)
    for a, _ in kept:
        eoff[graph(a) + 1] += 1
    return np.cumsum(eoff), [a for a, _ in kept], [b for _, b in kept]


@pytest.mark.parametrize("seed", range(12))
def test_normalize_matches_plain_dedup(seed):
    rng = np.random.default_rng(seed)
    D = int(rng.integers(1, 6))
    sizes = rng.integers(0, 9, D)
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    edges = []
    for t in range(D):
        n = int(sizes[t])
        if n < 2:
            continue
        for _ in range(int(rng.integers(0, 3 * n))):
            a, b = rng.choice(n, 2, replace=False) + ptr[t]
            edges.append((a, b))
            if seed % 2 == 0:
                edges.append((b, a))  # PyG lists both directions
    rng.shuffle(edges) if seed % 3 == 0 else None
    ei = np.array(edges, np.int64).T.reshape(2, -1)
    src = torch.from_numpy(ei) if seed % 4 == 1 else ei
    noff, eoff, ea, eb = api.normalize_edge_index(torch.from_numpy(ptr) if seed % 4 == 1 else ptr, src)
    r_eoff, r_a, r_b = plain_dedup(ptr, ei)
    assert np.array_equal(noff, ptr)
    assert np.array_equal(eoff, r_eoff)
    assert ea.tolist() == r_a and eb.tolist() == r_b
    assert ea.dtype == np.int32 and eb.dtype == np.int32


def test_normalize_keeps_self_loops_for_the_library_to_reject():
    noff, eoff, ea, eb = api.normalize_edge_index([0, 3], [[0, 1, 1, 2], [1, 1, 0, 2]])
    assert ea.tolist() == [0, 1, 2] and eb.tolist() == [1, 1, 2] and eoff.tolist() == [0, 3]
    rc, msg = create(noff, eoff, ea, eb)
    assert rc == L.E_INVALID and "self-loop" in msg
    with pytest.raises(ValueError):
        api.normalize_edge_index([0, 3], np.zeros((3, 2), np.int64))


@pytest.mark.parametrize("seed", range(4))
def test_scatter_restatement_is_the_gather_gradient(seed):
    rng = np.random.default_rng(seed)
    N, P = 30, 80
    bv, dv = rng.integers(0, N, P), rng.integers(0, N, P)
    poff = np.array([0, 17, 17, 60])  # points 60.. belong to no graph
    gb, gd = rng.standard_normal(P), rng.standard_normal(P)
    f = torch.zeros(N, dtype=torch.float64, requires_grad=True)
    k = slice(0, 60)
    (f[torch.from_numpy(bv[k])] * torch.from_numpy(gb[k])).sum().add(
        (f[torch.from_numpy(dv[k])] * torch.from_numpy(gd[k])).sum()).backward()
    assert np.allclose(scatter_grad(poff, bv, dv, gb, gd, N), f.grad.numpy(), rtol=0, atol=1e-13)
    only_b = scatter_grad(poff, bv, dv, gb, None, N)
    assert np.array_equal(only_b, scatter_grad(poff, bv, dv, gb, np.zeros(P), N))
    assert np.array_equal(scatter_grad(poff, bv, dv, None, None, N), np.zeros(N))
