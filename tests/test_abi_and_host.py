"""CPU-side checks: the C-ABI library loads without a GPU and exports every symbol include/tlc_b200.h declares
(no compute calls), constants of the Python binding equal the header's, argument errors are reported through the
rc / tlc_last_error convention, and the host-side mirror logic (label mapping, CSR ingestion) behaves like the
reference's graph2pi.__init__ (riccidist2dgm.py:216-226)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tlc_b200 import _lib as L
from tlc_b200 import graphgen as gg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "tlc_b200.h")).read()


def _declared_functions():
    names = re.findall(r"^\s*(?:const\s+)?[A-Za-z_0-9]+\s*\*?\s*(tlc_[a-z_0-9]+)\s*\(", HEADER, flags=re.M)
    return sorted(set(names))


def test_library_exports_every_declared_symbol():
    assert os.path.exists(L.SO_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = C.CDLL(L.SO_PATH)
    decl = _declared_functions()
    assert len(decl) >= 15
    for name in decl:
        assert hasattr(lib, name), name
    assert sorted(decl) == sorted(L.EXPORTS)          # the binding lists exactly the header's entry points


def test_binding_constants_match_header():
    macros = dict(re.findall(r"#define\s+(TLC_[A-Z_0-9]+)\s+\(?(-?\d+)u?\)?", HEADER))
    for k, v in [("TLC_F_NORM", L.F_NORM), ("TLC_F_EXTENDED", L.F_EXTENDED), ("TLC_F_KEEP_ZERO", L.F_KEEP_ZERO),
                 ("TLC_F_NORM_EPS", L.F_NORM_EPS), ("TLC_F_SUM_PLAIN", L.F_SUM_PLAIN), ("TLC_F_EDGE_SORTED", L.F_EDGE_SORTED),
                 ("TLC_MODE_EDGE", L.MODE_EDGE), ("TLC_MODE_NODE", L.MODE_NODE), ("TLC_K_UP", L.K_UP), ("TLC_K_ONE", L.K_ONE),
                 ("TLC_ST_OK", L.ST_OK), ("TLC_ST_NO_TREE_EDGES", L.ST_NO_TREE_EDGES), ("TLC_DESC_SUM", L.DESC["sum"]),
                 ("TLC_MODE_EDGE_FORCED", L.MODE_EDGE_FORCED), ("TLC_F_NO_DIRECT", L.F_NO_DIRECT), ("TLC_F_DIRECT", L.F_DIRECT),
                 ("TLC_F_ASC_ONLY", L.F_ASC_ONLY), ("TLC_F_FILT_DEGREE", L.F_FILT_DEGREE),
                 ("TLC_F_FILT_CENTRALITY", L.F_FILT_CENTRALITY), ("TLC_F_FILT_CLUSTERING", L.F_FILT_CLUSTERING),
                 ("TLC_F_NO_SMALL", L.F_NO_SMALL), ("TLC_F_NO_TABLE", L.F_NO_TABLE), ("TLC_ST_NOT_SMALL", L.ST_NOT_SMALL)]:
        assert int(macros[k]) == v, k
    assert C.sizeof(L.Params) == 24


def test_call_level_errors_without_gpu():
    lib = L.lib()
    h = C.c_void_p()
    rp = np.array([0, 1, 2], np.int32); col = np.array([1, 0], np.int32); kap = np.zeros(2)
    # bad arguments are rejected before any CUDA call
    assert lib.tlc_graph_create(0, 2, rp.ctypes.data, col.ctypes.data, kap.ctypes.data, 0, 0, C.byref(h)) == -1
    assert b"bad graph" in lib.tlc_last_error()
    bad = np.array([1, 1, 2], np.int32)
    assert lib.tlc_graph_create(2, 2, bad.ctypes.data, col.ctypes.data, kap.ctypes.data, 0, 0, C.byref(h)) == -1
    out = np.zeros(25)
    assert lib.tlc_pimg_transform(0, None, 3, 5, out.ctypes.data) == -1
    assert lib.tlc_pimg_transform(0, out.ctypes.data, 1, 99, out.ctypes.data) == -1
    import torch
    if not torch.cuda.is_available():   # no device: a well-formed call reports TLC_E_NODEVICE instead of crashing
        assert lib.tlc_graph_create(2, 2, rp.ctypes.data, col.ctypes.data, kap.ctypes.data, 0, 0, C.byref(h)) == -4


def test_graph_create_validates_the_csr():
    """a malformed CSR would mean out-of-bounds device accesses: every precondition is checked on the host, before any
    CUDA call (so this runs without a GPU), and reported through rc / tlc_last_error.  tlc_ollivier_ricci shares the
    validator; it takes no curvatures, so the curvature cases are tlc_graph_create's alone."""
    lib = L.lib()
    h = C.c_void_p()

    def create(rp, col, kap, entry="tlc_graph_create"):
        rp = np.asarray(rp, np.int32); col = np.asarray(col, np.int32); kap = np.asarray(kap, np.float64)
        if entry == "tlc_graph_create":
            rc = lib.tlc_graph_create(len(rp) - 1, len(col), rp.ctypes.data, col.ctypes.data, kap.ctypes.data, 0, 0, C.byref(h))
        else:
            out = np.zeros(len(col))
            rc = lib.tlc_ollivier_ricci(0, len(rp) - 1, len(col), rp.ctypes.data, col.ctypes.data, 0.5, out.ctypes.data, None)
        return rc, lib.tlc_last_error().decode()

    # path 0 - 1 - 2, well formed except for the one defect under test
    for e in ("tlc_graph_create", "tlc_ollivier_ricci"):
        rc, msg = create([0, 3, 1, 4], [1, 0, 2, 1], [0, 0, 0, 0], e);         assert rc == -1 and "monotone" in msg, e
        rc, msg = create([0, 1, 3, 4], [1, 0, 7, 1], [0, 0, 0, 0], e);         assert rc == -1 and "out of range" in msg, e
        rc, msg = create([0, 1, 3, 4], [0, 0, 2, 1], [0, 0, 0, 0], e);         assert rc == -1 and "self-loop" in msg, e
        rc, msg = create([0, 1, 3, 4], [1, 2, 0, 1], [0, 0, 0, 0], e);         assert rc == -1 and "ascending" in msg, e
        rc, msg = create([0, 2, 4, 4], [1, 1, 0, 0], [0, 0, 0, 0], e);         assert rc == -1 and "ascending" in msg, e  # duplicate entry
        rc, msg = create([0, 1, 2, 3], [1, 2, 1], [0, 0, 0], e);               assert rc == -1 and "symmetric" in msg, e
    rc, msg = create([0, 1, 3, 4], [1, 0, 2, 1], [0.5, 0.25, 0, 0]);       assert rc == -1 and "mirror" in msg      # kappa(0,1) != kappa(1,0)
    rc, msg = create([0, 1, 3, 4], [1, 0, 2, 1], [-1.0, -1.0, 0, 0]);      assert rc == -1 and "kappa + 1" in msg   # weight 0
    rc, msg = create([0, 1, 3, 4], [1, 0, 2, 1], [0, 0, np.nan, np.nan]);  assert rc == -1 and "kappa + 1" in msg
    rc, msg = create([0, 1, 3, 4], [1, 0, 2, 1], [0, 0, np.inf, np.inf]);  assert rc == -1 and "kappa + 1" in msg


def test_csr_ingestion_matches_reference_numbering():
    e = np.array([[7, 3], [3, 9], [9, 7], [2, 7]])
    labels, ne = gg.relabel_first_appearance(e)
    assert labels.tolist() == [7, 3, 9, 2]                      # first-appearance order, loaddatas.py:88-92
    assert ne.tolist() == [[0, 1], [1, 2], [2, 0], [3, 0]]
    rowptr, col, kap = gg.build_csr(4, ne, np.array([0.5, -0.25, 0.0, 0.125]))
    assert rowptr.tolist() == [0, 3, 5, 7, 8] and col.tolist() == [1, 2, 3, 0, 2, 0, 1, 0]
    assert kap.tolist() == [0.5, 0.0, 0.125, 0.5, -0.25, 0.0, -0.25, 0.125]   # kappa stored both directions :222-226


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(L, "_lib", None)
    monkeypatch.setattr(L, "SO_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError):
        L.lib()


def test_cache_filename_mapping():
    """loaddatas.py:57-62: photo -> Photo, computers -> Computers, others unchanged."""
    from tlc_b200.table import cache_filename
    assert cache_filename("photo") == "./data/TLCGNN/Photo.npy"
    assert cache_filename("computers") == "./data/TLCGNN/Computers.npy"
    assert cache_filename("PubMed", "/x") == "/x/PubMed.npy"


def test_oracle_and_binding_flag_values_agree():
    """tests pass one flag word to both sides: the oracle's TLO_* and the library's TLC_* values must coincide."""
    import oracle as orc
    for name in ("F_NORM", "F_EXTENDED", "F_KEEP_ZERO", "F_NORM_EPS", "F_SUM_PLAIN", "F_FILT_DEGREE", "F_FILT_CENTRALITY", "F_FILT_CLUSTERING",
                 "MODE_EDGE", "MODE_NODE", "MODE_EDGE_FORCED"):
        assert getattr(orc, name) == getattr(L, name), name


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the reference algorithm on the host cores) runs without a GPU and prints ONE JSON
    line with the contract's keys; a tiny workload keeps it to seconds."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cora",
                          "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_kd_emitter_batching_logic():
    """sg2dgm.kd._batches: consecutive batches, every target in exactly one, budget respected unless a single vicinity
    alone exceeds it (pure host logic; the C-ABI call is stubbed)."""
    import sg2dgm.kd as kd

    class FakeGraph:
        def __init__(self, n, m):
            self.n, self.m = np.asarray(n, np.int32), np.asarray(m, np.int32)

        def vicinity_sizes(self, tg, hop=2, mode=0):
            return self.n[:len(tg)], self.m[:len(tg)], np.zeros(len(tg), np.uint8)

    n = [10, 20, 5, 400, 7, 7, 7, 1000, 3]
    m = [30, 60, 9, 900, 8, 8, 8, 5000, 2]
    tg = np.zeros((len(n), 2), np.int32)
    b = kd._batches(FakeGraph(n, m), tg, 2, 0, budget=200)
    assert b[0][0] == 0 and b[-1][1] == len(n)
    assert all(b[i][1] == b[i + 1][0] for i in range(len(b) - 1))             # consecutive, no gaps
    cost = np.asarray(n) + np.asarray(m) + 1
    for lo, hi in b:
        assert hi > lo and (cost[lo:hi].sum() <= 200 or hi - lo == 1)          # an oversized vicinity travels alone
    assert kd._batches(FakeGraph(n, m), tg, 2, 0, budget=10 ** 9) == [(0, len(n))]


def test_mirror_label_mapping_paths():
    """graph2pi._map_targets: node label -> dense id as the reference's dict_node lookup (riccidist2dgm.py:353: a label that
    is not a node gives a zero row, here id -1) -- through the dense table (small non-negative labels), the searchsorted
    path (huge / negative labels) and the per-element dict path (non-integer labels); all three agree with a plain dict."""
    import sg2dgm.riccidist2dgm as mirror
    rng = np.random.default_rng(3)
    N = 500

    def make(labels):
        g = mirror.graph2pi.__new__(mirror.graph2pi)
        lab = np.asarray(labels, dtype=np.int64)
        o = np.argsort(lab, kind="stable")
        g._int_labels = (lab[o], o.astype(np.int32))
        g.N = N
        g.dict_node = {int(l): i for i, l in enumerate(labels)}
        return g

    for labels, lo, hi, want_lut in ((np.arange(N), -5, N + 5, True),                       # identity
                                     (rng.permutation(3 * N)[:N], -5, 3 * N + 5, True),       # small sparse labels
                                     (rng.permutation(10 ** 7)[:N] * 1000, 0, 10 ** 10, False),  # huge labels: no table
                                     (rng.permutation(4 * N)[:N] - 2 * N, -2 * N - 5, 2 * N + 5, False)):  # negative labels
        g = make(labels)
        assert (g._label_lut() is not None) == want_lut
        pool = np.concatenate([np.asarray(labels), rng.integers(lo, hi, size=200)])
        t = rng.choice(pool, size=(300, 2))
        got = g._map_targets(t)
        exp = np.array([[g.dict_node.get(int(a), -1), g.dict_node.get(int(b), -1)] for a, b in t], dtype=np.int32)
        assert got.dtype == np.int32 and np.array_equal(got, exp)
        assert np.array_equal(g._map_targets(t.astype(np.int32) if t.max() < 2 ** 31 and t.min() >= -2 ** 31 else t), exp)
    # non-integer labels: the dict path
    g = mirror.graph2pi.__new__(mirror.graph2pi)
    g._int_labels = None
    g.dict_node = {"a": 0, "b": 1, "c": 2}
    assert g._map_targets([("a", "c"), ("b", "zz")]).tolist() == [[0, 2], [1, -1]]
