"""Mirror of sg2dgm/riccidist2dgm.py (the accelerated path: riccidist2dgm.py:215-229, 310-329, 348-370).

`graph2pi(g, ricci_curv)` uploads the graph once; `get_pimg_for_all_edges` is ONE C-ABI call for the
whole batch (the reference maps a GIL-bound thread pool over edges, :367-370).  The legacy dionysus
half of the reference file (graph2dgm, sg2pimg, get_pimg) is out of scope (SURVEY.md section 2).
"""
import sys
import time

import numpy as np

from tlc_b200 import _lib as L
from tlc_b200 import api

__all__ = ["graph2pi", "filtration"]

_DESCRIPTORS = ("min", "max", "sum")


def default_plain_sum():
    """True when float sum() of the running interpreter adds left to right (CPython <= 3.11), False when it is
    Neumaier-compensated (CPython >= 3.12)."""
    return sys.version_info < (3, 12)


class graph2pi():
    def __init__(self, g, ricci_curv, device=0, plain_sum=None):
        """g: networkx-like graph (needs .nodes() and .edges()); ricci_curv: [[n1, n2, kappa], ...]
        (both directions, loaddatas.py:117-121).  Nodes are relabelled to integers in g.nodes() order
        exactly as nx.convert_node_labels_to_integers does (riccidist2dgm.py:217-220).
        plain_sum: how build_fv's `sum([...])` of the path weights (:30,35) is evaluated -- it is the ONE place where the
        reference's float64 results depend on the interpreter.  True: left to right, as sum() of CPython <= 3.11 does
        (the reference pins CPython 3.7: PersistenceImager.cpython-37m, requirements.txt).  False: the Neumaier-
        compensated sum() of CPython >= 3.12.  Default (None): whatever sum() of the RUNNING interpreter does, so the
        drop-in reproduces the reference executed in the caller's own environment; pass True to reproduce tables cached
        by the reference under its pinned 3.7.  The two differ in the last bits only, and only for curvatures whose
        path sums are not exactly representable (SURVEY.md F5)."""
        self.plain_sum = default_plain_sum() if plain_sum is None else bool(plain_sum)
        nodes = list(g.nodes())
        self.dict_node = {old: new for new, old in enumerate(nodes)}
        self.old_label = nodes
        N = len(nodes)
        dn = self.dict_node
        edges = np.array([(dn[a], dn[b]) for a, b in g.edges()], dtype=np.int64).reshape(-1, 2)
        edges = edges[edges[:, 0] != edges[:, 1]]
        lo = np.minimum(edges[:, 0], edges[:, 1])
        hi = np.maximum(edges[:, 0], edges[:, 1])
        # one entry per UNDIRECTED edge: a DiGraph listing both (a,b) and (b,a), or a MultiGraph, must not yield duplicate
        # CSR entries (nx.Graph semantics of the reference's subgraph views; tlc_graph_create rejects duplicate row entries)
        key = np.unique(lo * max(N, 1) + hi)
        lo, hi = key // max(N, 1), key % max(N, 1)
        # curvature per undirected edge; a later entry overwrites an earlier one (dict semantics, :222-226).
        # Edges without an entry have no 'weight' attribute: networkx then uses weight 1 for Dijkstra but
        # ricci_curv[...] raises KeyError -> dist = 100; such graphs are outside the contract (kappa given
        # for every edge, loaddatas.py:117-121) -- they get kappa = 0 here.
        order = np.argsort(key, kind="stable")
        key_sorted = key[order]
        kap = np.zeros(len(key), dtype=np.float64)
        if len(ricci_curv):
            rc = list(ricci_curv)
            ra = np.fromiter((dn[r[0]] for r in rc), dtype=np.int64, count=len(rc))
            rb = np.fromiter((dn[r[1]] for r in rc), dtype=np.int64, count=len(rc))
            rk = np.fromiter((float(r[2]) for r in rc), dtype=np.float64, count=len(rc))
            rkey = np.minimum(ra, rb) * max(N, 1) + np.maximum(ra, rb)
            idx = np.searchsorted(key_sorted, rkey)
            ok = (idx < len(key_sorted))
            ok[ok] &= key_sorted[idx[ok]] == rkey[ok]
            kap[order[idx[ok]]] = rk[ok]  # duplicates: last assignment wins, as in the reference's dict
        from tlc_b200.graphgen import build_csr
        self.csr = build_csr(N, np.stack([lo, hi], 1), kap)
        self._graph = api.VicinityGraph(*self.csr, device=device)
        self.N = N
        self.pi_sg = None
        self.cnt_compute = 0
        self.t1 = time.time()
        self.status = None
        self._int_labels = None
        if N and all(isinstance(x, (int, np.integer)) for x in nodes):  # vectorised dict_node for integer labels
            lab = np.asarray(nodes, dtype=np.int64)
            o = np.argsort(lab, kind="stable")
            self._int_labels = (lab[o], o.astype(np.int32))

    @classmethod
    def from_csr(cls, rowptr, col, kappa, device=0, plain_sum=None):
        """graph already in integer ids 0..N-1 (CSR, ascending rows): skips the networkx ingestion."""
        self = cls.__new__(cls)
        self.plain_sum = default_plain_sum() if plain_sum is None else bool(plain_sum)
        self.csr = (rowptr, col, kappa)
        self._graph = api.VicinityGraph(rowptr, col, kappa, device=device)
        self.N = self._graph.N
        self.dict_node = None
        self.old_label = None
        self.pi_sg, self.cnt_compute, self.t1, self.status = None, 0, time.time(), None
        self._int_labels = (np.arange(self.N, dtype=np.int64), np.arange(self.N, dtype=np.int32))
        return self

    # -- helpers ---------------------------------------------------------------------------------
    def _label_lut(self):
        """label -> id table for non-negative integer labels that are not much larger than N (a searchsorted over the
        call's 2E endpoints costs 0.7 - 1.5 ms per 4096 targets: as much as a tenth of the GPU step); else None"""
        lut = getattr(self, "_lut", None)
        if lut is None:
            lab, new = self._int_labels
            if len(lab) and lab[0] >= 0 and lab[-1] < 8 * len(lab) + 1024:
                lut = np.full(int(lab[-1]) + 1, -1, dtype=np.int32)
                lut[lab] = new
            else:
                lut = False
            self._lut = lut
        return None if lut is False else lut

    def _map_targets(self, total_edges):
        if self._int_labels is not None:
            try:
                t = np.asarray(total_edges)
                if t.ndim == 2 and t.shape[1] >= 2 and np.issubdtype(t.dtype, np.integer):
                    lab, new = self._int_labels
                    t = t[:, :2]
                    lut = self._label_lut()
                    if lut is not None:   # dense table label -> id (-1: not a node); ids 0..N-1 map to themselves
                        ok = (t >= 0) & (t < len(lut))
                        return np.where(ok, lut[np.where(ok, t, 0)], -1).astype(np.int32)
                    t = t.astype(np.int64)
                    idx = np.clip(np.searchsorted(lab, t), 0, len(lab) - 1)
                    return np.where(lab[idx] == t, new[idx], -1).astype(np.int32)
            except Exception:
                pass
        dn = self.dict_node
        out = np.empty((len(total_edges), 2), dtype=np.int32)
        for i, e in enumerate(total_edges):
            a, b = e[0], e[1]
            try:
                a = a.item() if hasattr(a, "item") else a
                b = b.item() if hasattr(b, "item") else b
            except Exception:
                pass
            out[i, 0] = dn.get(a, -1)   # KeyError -> zeros row   riccidist2dgm.py:353,356-357
            out[i, 1] = dn.get(b, -1)
        return out

    def _flags(self, norm, extended_flag):
        return ((L.F_NORM if norm else 0) | (L.F_EXTENDED if extended_flag else 0) |
                (L.F_SUM_PLAIN if getattr(self, "plain_sum", False) else 0))

    # -- reference surface -----------------------------------------------------------------------
    def sg2dgm_accelerate(self, u, v, hop, extended_flag=False, descriptor="seal", resolution=5, norm=False, cnt=0):
        """riccidist2dgm.py:310-329: u, v are NEW labels; returns the [res,res] image; raises where the
        reference raises (assert on connectivity, ZeroDivisionError, KeyError on a bad descriptor, ...)."""
        desc = descriptor if descriptor in _DESCRIPTORS else -1
        pi, status, _ = self._graph.vicinity_pi(np.array([[u, v]], dtype=np.int32), hop=hop, descriptor=desc,
                                                resolution=resolution, flags=self._flags(norm, extended_flag))
        st = int(status[0])
        if st == L.ST_EMPTY or st == L.ST_DISCONNECTED:
            raise AssertionError("vicinity is not one connected component")        # :318
        if st == L.ST_DEGENERATE:
            raise ZeroDivisionError("float division by zero")                      # :54-56
        if st == L.ST_UNKNOWN_NODE:
            raise KeyError((u, v))
        if st == L.ST_BAD_DESCRIPTOR:
            raise KeyError(descriptor)                                             # accelerated_PD.py:13
        if st == L.ST_NO_TREE_EDGES:
            raise IndexError("list index out of range")                            # accelerated_PD.py:122
        return pi[0].reshape(resolution, resolution)

    def sg2pimg(self, u, v, hop, weight_graph=True, norm=False, extended_flag=False, range='intersection',
                descriptor="seal", resolution=5):
        """riccidist2dgm.py:228-305 (u, v are NEW labels): the image of ONE target for a vicinity shape `range` in
        'intersection' | 'union' | 'removeinter'.  The reference computes these diagrams with dionysus (the legacy
        path); here they come from the same union-find kernels as sg2dgm_accelerate (the same extended persistence),
        including its connectivity assertion.  `weight_graph` is accepted for the signature (the path always uses the
        Ricci weights, as sg2dgm_accelerate hard-codes at :320)."""
        modes = {"intersection": L.MODE_EDGE, "union": L.MODE_EDGE_UNION, "removeinter": L.MODE_EDGE_REMOVEINTER}
        if range not in modes:
            raise SystemExit("Error: 'range' should be 'union' or 'intersection'! ")   # :303-305 (print + sys.exit())
        desc = descriptor if descriptor in _DESCRIPTORS else -1
        pi, status, _ = self._graph.vicinity_pi(np.array([[u, v]], dtype=np.int32), hop=hop, mode=modes[range], descriptor=desc,
                                                resolution=resolution, flags=self._flags(norm, extended_flag))
        st = int(status[0])
        if st in (L.ST_EMPTY, L.ST_DISCONNECTED):
            raise AssertionError("vicinity is not one connected component")
        if st == L.ST_DEGENERATE:
            raise ZeroDivisionError("float division by zero")
        if st == L.ST_UNKNOWN_NODE:
            raise KeyError((u, v))
        if st == L.ST_BAD_DESCRIPTOR:
            raise KeyError(descriptor)
        if st == L.ST_NO_TREE_EDGES:
            raise IndexError("list index out of range")
        return pi[0].reshape(resolution, resolution)

    def get_pimg_for_one_edge(self, u, v, hop=2, norm=True, extended_flag=False, resolution=5, descriptor='min', cnt=0):
        """riccidist2dgm.py:348-357 (note: the reference forces norm=True at :353)."""
        try:
            img = self.sg2dgm_accelerate(self.dict_node[u], self.dict_node[v], hop, norm=True,
                                         extended_flag=extended_flag, resolution=resolution,
                                         descriptor=descriptor).reshape(-1)
            if self.pi_sg is not None and 0 <= cnt < len(self.pi_sg):
                self.pi_sg[cnt] = img
            self.cnt_compute += 1
            return img
        except BaseException:
            return np.zeros([resolution * resolution])

    def get_pimg_for_all_edges(self, total_edges, cores, hop=2, norm=True, extended_flag=False, resolution=5,
                               descriptor='min'):
        """riccidist2dgm.py:362-370.  `cores` is accepted and ignored (one batched GPU call);
        as in the reference the per-edge call always normalises (:353)."""
        self.t1 = time.time()
        E = len(total_edges)
        self.pi_sg = np.zeros((E, resolution * resolution))
        self.cnt_compute = 0
        if E == 0:
            self.status = np.zeros(0, np.uint8)
            return
        desc = descriptor if descriptor in _DESCRIPTORS else -1
        tg = self._map_targets(total_edges)
        _, self.status, self.cnt_compute = self._graph.vicinity_pi(
            tg, hop=hop, descriptor=desc, resolution=resolution, flags=self._flags(True, extended_flag),
            out=self.pi_sg)

    def get_pdgm_for_all_edges(self, total_edges, cores, hop=2, norm=True, extended_flag=False, descriptor='min'):
        """The diagram counterpart of get_pimg_for_all_edges: self.pd_sg is a list with one float64 [K, 2] (birth,
        death) array per target -- np.array(PD0 + PD1) of riccidist2dgm.py:323-328, the array the reference hands to
        the imager -- empty for targets whose image the reference zeroes; self.pd_status holds the statuses."""
        self.t1 = time.time()
        E = len(total_edges)
        self.pd_sg = [np.zeros((0, 2)) for _ in range(E)]
        self.pd_status = np.zeros(E, np.uint8)
        if E == 0:
            return
        desc = descriptor if descriptor in _DESCRIPTORS else -1
        d = self._graph.vicinity_diagrams(self._map_targets(total_edges), hop=hop, descriptor=desc,
                                          flags=self._flags(True, extended_flag))
        bd = np.stack([d["birth"], d["death"]], axis=1)
        self.pd_sg = [bd[d["poff"][i]:d["poff"][i + 1]] for i in range(E)]
        self.pd_status = d["status"]

    def multi_wrapper_all_edges(self, args):
        return self.get_pimg_for_one_edge(*args)


class filtration():
    """riccidist2dgm.py:11-61 -- kept for callers that build the filtration of one vicinity themselves:
    build_fv returns the vicinity's filtration values computed by kernels 1 + 1b."""

    def __init__(self, g2pi, u, v, hop, ricci_curv=None):
        self.g2pi, self.root_1, self.root_2, self.hop = g2pi, u, v, hop

    def build_fv(self, weight_graph=True, norm=True, descriptor="sum"):
        d = self.g2pi._graph.vicinity_detail(np.array([[self.root_1, self.root_2]], np.int32), hop=self.hop,
                                             descriptor=descriptor, flags=L.F_NORM if norm else 0)
        a = self.g2pi._graph.per_target(d, 0)
        return {int(x): float(f) for x, f in zip(a["vert"], a["fval"])}
