"""TEST INFRASTRUCTURE ONLY -- in-container harness around the *real* reference.

Imports pkuyzy/TLC-GNN in place from a checkout of it (read-only): oracle/_ref/, which git ignores, or the
directory named by TLC_REFERENCE_ROOT, so that
  * the C restatement in oracle/tlc_oracle.c can be pinned against it, and
  * golden vectors under tests/golden/ can be generated (oracle/make_golden.py).

The reference is not part of this repository, so nothing in the `-m gpu`
tests, smoke() or bench.py imports this module; only `-m "not gpu"` tests that
skip when the reference tree is absent, and make_golden.py, do.

Two shims are needed (SURVEY.md section 8c):
  1. `import dionysus` (riccidist2dgm.py:3, dgformat.py:2) -- not installed, and
     not touched by the hot path -> an empty stub module.
  2. sg2dgm/PersistenceImager.pyx is untyped Python run through Cython
     (setup_PI.py:1-5; README.md:43 says a plain .py copy works) -> the .pyx is
     executed as Python source *where it lies*; nothing is copied into this repo.
"""
import importlib.machinery
import importlib.util
import os
import sys
import types

import numpy as np

REF_ROOT = os.environ.get("TLC_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available():
    return os.path.isfile(os.path.join(REF_ROOT, "sg2dgm", "riccidist2dgm.py"))


_loaded = {}


def _load_source(modname, path):
    loader = importlib.machinery.SourceFileLoader(modname, path)
    spec = importlib.util.spec_from_loader(modname, loader)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[modname] = mod
    loader.exec_module(mod)
    return mod


def load():
    """Returns a namespace with the reference's modules:
       .ricci (sg2dgm.riccidist2dgm), .apd (sg2dgm.accelerated_PD),
       .pimg (sg2dgm.PersistenceImager), .kd_apd (Knowledge_Distillation.accelerated_PD)."""
    if _loaded:
        return types.SimpleNamespace(**_loaded)
    if not available():
        raise RuntimeError("no checkout of pkuyzy/TLC-GNN at %s: clone it there or point TLC_REFERENCE_ROOT at one"
                           % REF_ROOT)
    # The reference's package is called `sg2dgm`, and so is our drop-in mirror.
    # Load the reference under a private package name so both can coexist.
    if "dionysus" not in sys.modules:
        sys.modules["dionysus"] = types.ModuleType("dionysus")  # shim 1
    saved = {k: sys.modules.get(k) for k in list(sys.modules) if k == "sg2dgm" or k.startswith("sg2dgm.")}
    for k in saved:
        del sys.modules[k]
    pkg = types.ModuleType("sg2dgm")
    pkg.__path__ = [os.path.join(REF_ROOT, "sg2dgm")]
    sys.modules["sg2dgm"] = pkg
    try:
        pimg = _load_source("sg2dgm.PersistenceImager",
                            os.path.join(REF_ROOT, "sg2dgm", "PersistenceImager.pyx"))  # shim 2
        pkg.PersistenceImager = pimg
        apd = _load_source("sg2dgm.accelerated_PD", os.path.join(REF_ROOT, "sg2dgm", "accelerated_PD.py"))
        dgf = _load_source("sg2dgm.dgformat", os.path.join(REF_ROOT, "sg2dgm", "dgformat.py"))
        ricci = _load_source("sg2dgm.riccidist2dgm", os.path.join(REF_ROOT, "sg2dgm", "riccidist2dgm.py"))
        kd_apd = _load_source("_ref_kd_accelerated_PD",
                              os.path.join(REF_ROOT, "Knowledge_Distillation", "accelerated_PD.py"))
    finally:
        # un-shadow: give `sg2dgm` back to whoever had it (our mirror), keep refs privately
        for k in [k for k in list(sys.modules) if k == "sg2dgm" or k.startswith("sg2dgm.")]:
            del sys.modules[k]
        for k, v in saved.items():
            sys.modules[k] = v
    _loaded.update(ricci=ricci, apd=apd, pimg=pimg, kd_apd=kd_apd, dgformat=dgf)
    return types.SimpleNamespace(**_loaded)


# ----------------------------------------------------------------------------------------------
# helpers that drive the reference exactly the way loaddatas.py:88-101 does
# ----------------------------------------------------------------------------------------------
def build_nx_graph(edges):
    """nx.Graph built by add_edges_from(edge list) -- loaddatas.py:88-92 (no isolated nodes)."""
    import networkx as nx
    g = nx.Graph()
    g.add_edges_from([(int(a), int(b)) for a, b in edges])
    return g


def ricci_list(edges, kappa):
    """sorted [[n1,n2,k],[n2,n1,k],...] -- loaddatas.py:117-121."""
    out = []
    for (a, b), k in zip(edges, kappa):
        out.append([int(a), int(b), k])
        out.append([int(b), int(a), k])
    return sorted(out)


def run_batch(edges, kappa, targets, hop, extended_flag, descriptor="sum", resolution=5, cores=1):
    """graph2pi(...).get_pimg_for_all_edges(...) unmodified -- riccidist2dgm.py:216,362.
    returns (pi_sg float64[E,res^2], cnt_compute)."""
    import contextlib
    import io
    ref = load()
    g = build_nx_graph(edges)
    pi = ref.ricci.graph2pi(g, ricci_curv=ricci_list(edges, kappa))
    with contextlib.redirect_stdout(io.StringIO()):
        pi.get_pimg_for_all_edges([list(map(int, t)) for t in targets], cores=cores, hop=hop, norm=True,
                                  extended_flag=extended_flag, resolution=resolution, descriptor=descriptor)
    return pi.pi_sg, pi.cnt_compute, pi


def run_one_stages(pi, u_old, v_old, hop, descriptor="sum", norm=True, canonical=True):
    """One target through the reference's own stage functions, returning every intermediate.
    riccidist2dgm.py:311-326.  With canonical=True the vicinity is rebuilt as a fresh nx.Graph
    whose dict insertion order is (vertices ascending, edges lexicographic (lo,hi)) so that the
    reference's stable sort yields the canonical tie-break of SURVEY.md section 8c (F3)."""
    import networkx as nx
    ref = load()
    u, v = pi.dict_node[u_old], pi.dict_node[v_old]
    nodes_u = [u] + [x for _, x in nx.bfs_edges(pi.graph, u, depth_limit=hop)]
    nodes_v = [v] + [x for _, x in nx.bfs_edges(pi.graph, v, depth_limit=hop)]
    nodes = sorted(set(nodes_u) & set(nodes_v))
    sub = pi.graph.subgraph(nodes)
    ncomp = len(list(nx.connected_components(sub)))
    out = dict(nodes=nodes, ncomp=ncomp)
    if ncomp != 1:
        return out
    if canonical:
        h = nx.Graph()
        h.add_nodes_from(nodes)
        es = sorted((min(a, b), max(a, b)) for a, b in sub.edges())
        for a, b in es:
            h.add_edge(a, b, weight=pi.graph[a][b]["weight"])
        sub = h
        out["edges"] = es
    fil = ref.ricci.filtration(sub, u, v, hop, ricci_curv=pi.ricci_curv)
    g = fil.build_fv(weight_graph=True, norm=norm)
    out["fval"] = {x: g.nodes[x][descriptor] for x in g.nodes()}
    sf = ref.apd.perturb_filter_function(g, descriptor=descriptor)
    PD0, Pos, Neg = ref.apd.Union_find(sf)
    out.update(PD0=PD0, Pos=Pos, Neg=Neg)
    out["PD1"] = ref.apd.Accelerate_PD(Pos, Neg, sf) if len(Neg) else None
    return out


# ----------------------------------------------------------------------------------------------
# PDGNN generator (SURVEY.md row A9): Knowledge_Distillation/data_utils_NC.py imported AS-IS.
# Its module header imports packages that are not installed here (matplotlib, gudhi, torch_geometric)
# and sibling modules absent from the tree (learnable_filter.loaddatas_LP, loaddatas_LP_arxiv); none of
# them is touched by compute_persistence_image(filt='ricci', mode='PI') (data_utils_NC.py:95-183),
# so empty stub modules satisfy the imports.  `sg2dgm.PersistenceImager` and
# `Knowledge_Distillation.accelerated_PD` resolve to the reference's own files.
# ----------------------------------------------------------------------------------------------
_kd_loaded = {}


def load_kd(which="NC"):
    """which = 'NC' (node-centred generator) or 'LP' (edge-centred generator, data_utils_LP.py)."""
    if which in _kd_loaded:
        return _kd_loaded[which]
    ref = load()
    stubs = {}

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        stubs[name] = m
        return m

    stub("matplotlib").pyplot = stub("matplotlib.pyplot")
    stub("gudhi")
    tg = stub("torch_geometric")
    tg.utils = stub("torch_geometric.utils", remove_self_loops=lambda ei, *a, **k: (ei, None))
    lf = stub("learnable_filter")
    lf.loaddatas_LP = stub("learnable_filter.loaddatas_LP")
    stub("loaddatas_LP_arxiv", get_edges_split=None)
    kd_pkg = stub("Knowledge_Distillation")
    kd_pkg.__path__ = [os.path.join(REF_ROOT, "Knowledge_Distillation")]
    kd_pkg.accelerated_PD = ref.kd_apd
    stubs["Knowledge_Distillation.accelerated_PD"] = ref.kd_apd
    kd_pkg.spectral = stub("Knowledge_Distillation.spectral", SpectralClustering=None)  # (absent sibling, data_utils_LP.py:18)
    kd_pkg.SBM_Model = stub("Knowledge_Distillation.SBM_Model", create_SBM_Model=None)  # (data_utils_GC.py:27)
    tg.datasets = stub("torch_geometric.datasets", TUDataset=None, ZINC=None)           # (data_utils_GC.py:24)
    stub("ogb").graphproppred = stub("ogb.graphproppred", PygGraphPropPredDataset=None)  # (data_utils_GC.py:26)
    sg = stub("sg2dgm")
    sg.__path__ = [os.path.join(REF_ROOT, "sg2dgm")]
    sg.PersistenceImager = ref.pimg
    stubs["sg2dgm.PersistenceImager"] = ref.pimg
    saved = {k: sys.modules.get(k) for k in stubs}
    saved.update({k: sys.modules[k] for k in list(sys.modules) if k.startswith("sg2dgm.")})
    for k in [k for k in list(sys.modules) if k == "sg2dgm" or k.startswith("sg2dgm.")]:
        del sys.modules[k]
    sys.modules.update(stubs)
    try:
        nc = _load_source("_ref_kd_data_utils_" + which,
                          os.path.join(REF_ROOT, "Knowledge_Distillation", "data_utils_%s.py" % which))
    finally:
        for k in stubs:
            sys.modules.pop(k, None)
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
    _kd_loaded[which] = nc
    return nc


def kd_run_node(g, ricci, u, hop, filt="ricci"):
    """data_utils_NC.compute_persistence_image(g, u, filt='ricci', hop, ricci_curv, mode='PI') unmodified
    (:95-183).  Returns None for the `return None, None` case (:103-104), else a dict with the 9-tuple's
    fields plus `old_label` (new label -> graph node, recovered by repeating the function's own first three
    statements, which are deterministic) so that per-vertex outputs can be put in canonical order."""
    import networkx as nx
    nc = load_kd()
    r = nc.compute_persistence_image(g, u, filt=filt, hop=hop, ricci_curv=ricci, mode="PI")
    if r[0] is None:
        return None
    nodes = [u] + [x for _, x in nx.bfs_edges(g, u, depth_limit=hop)]       # :97
    sub = nx.convert_node_labels_to_integers(g.subgraph(nodes), label_attribute="old_label")  # :98-99
    old = [sub.nodes[i]["old_label"] for i in range(len(sub))]
    ord0, ext1, pi, filt, edge_index, pi0, pi1, _, _ = r
    return dict(ord0=np.asarray(ord0, dtype=np.float64).reshape(-1, 2), ext1=np.asarray(ext1, dtype=np.float64).reshape(-1, 2),
                pi=np.asarray(pi, dtype=np.float64), pi0=np.asarray(pi0, dtype=np.float64), pi1=np.asarray(pi1, dtype=np.float64),
                filt=np.asarray(filt, dtype=np.float64), edge_index=np.asarray(edge_index.numpy(), dtype=np.int64),
                old_label=np.asarray(old, dtype=np.int64))


def kd_lp_run_edge(g, ricci, u, v, hop):
    """data_utils_LP.compute_persistence_image(g, u, v, filt='ricci', hop, ricci_curv, mode='PI') unmodified (:105-196):
    the edge-centred PDGNN generator, vicinity = (ball(u) & ball(v)) + [u] + [v].  Returns None for `return None, None`
    (:117-118), the string 'raised' when the reference itself raises (a disconnected vicinity: Accelerate_PD's BFS tree
    misses vertices -> KeyError, Knowledge_Distillation/accelerated_PD.py:124-137), else the fields of the 9-tuple."""
    import networkx as nx
    lp = load_kd("LP")
    try:
        r = lp.compute_persistence_image(g, u, v, filt="ricci", hop=hop, ricci_curv=ricci, mode="PI")
    except BaseException:
        return "raised"
    if r[0] is None:
        return None
    nodes_u = [u] + [x for _, x in nx.bfs_edges(g, u, depth_limit=hop)]      # :107-110
    nodes_v = [v] + [x for _, x in nx.bfs_edges(g, v, depth_limit=hop)]
    nodes = list(set(nodes_u) & set(nodes_v)) + [u] + [v]                    # :111
    sub = nx.convert_node_labels_to_integers(g.subgraph(nodes), label_attribute="old_label")
    old = [sub.nodes[i]["old_label"] for i in range(len(sub))]
    ord0, ext1, pi, filt, edge_index, pi0, pi1, _, _ = r
    return dict(ord0=np.asarray(ord0, dtype=np.float64).reshape(-1, 2), ext1=np.asarray(ext1, dtype=np.float64).reshape(-1, 2),
                pi=np.asarray(pi, dtype=np.float64), pi0=np.asarray(pi0, dtype=np.float64), pi1=np.asarray(pi1, dtype=np.float64),
                filt=np.asarray(filt, dtype=np.float64), edge_index=np.asarray(edge_index.numpy(), dtype=np.int64),
                old_label=np.asarray(old, dtype=np.int64))


def kd_gc_run_graph(n, edges, filt="degree"):
    """data_utils_GC.compute_persistence_image(g, filt, mode='PI') unmodified (:95-167): the graph-classification
    generator, the WHOLE graph is the vicinity (nodes 0..n-1 added in order, so subgraph.nodes() is 0..n-1).
    Returns None for `return None, None` (no edge, or not connected, :99-100)."""
    import networkx as nx
    gc = load_kd("GC")
    g = nx.Graph()
    g.add_nodes_from(range(n))
    g.add_edges_from([(int(a), int(b)) for a, b in edges])
    r = gc.compute_persistence_image(g, filt=filt, mode="PI")
    if r[0] is None:
        return None
    ord0, ext1, pi, fv, edge_index, pi0, pi1, _, _ = r
    return dict(ord0=np.asarray(ord0, dtype=np.float64).reshape(-1, 2), ext1=np.asarray(ext1, dtype=np.float64).reshape(-1, 2),
                pi=np.asarray(pi, dtype=np.float64), pi0=np.asarray(pi0, dtype=np.float64), pi1=np.asarray(pi1, dtype=np.float64),
                filt=np.asarray(fv, dtype=np.float64), edge_index=np.asarray(edge_index.numpy(), dtype=np.int64))
