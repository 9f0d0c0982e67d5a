"""ctypes binding of libtlc_b200.so (C-ABI declared in include/tlc_b200.h).

There is NO CPU fallback: if the shared object is missing the import of the compute entry points
fails loudly (build it with `python __graft_entry__.py build` or `make -C tlc-gnn_b200/csrc`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("TLC_LIB") or os.path.join(_HERE, "libtlc_b200.so")  # TLC_LIB: a differently tuned build (experiments)

# mirrors of the header's constants
MODE_EDGE, MODE_NODE, MODE_EDGE_FORCED, MODE_EDGE_UNION, MODE_EDGE_REMOVEINTER = 0, 1, 2, 3, 4
DESC = {"min": 0, "max": 1, "sum": 2}
F_NORM, F_EXTENDED, F_KEEP_ZERO, F_NORM_EPS, F_SUM_PLAIN, F_EDGE_SORTED = 1, 2, 4, 8, 16, 32
F_NO_DIRECT, F_DIRECT, F_ASC_ONLY = 64, 128, 256
F_FILT_DEGREE, F_FILT_CENTRALITY, F_FILT_CLUSTERING = 512, 1024, 2048
F_NO_SMALL = 4096
F_NO_TABLE = 8192
F_FILT_HKS = 16384
ST_NOT_SMALL = 255
E_INVALID, E_CUDA, E_NOMEM, E_NODEVICE, E_CAPACITY = -1, -2, -3, -4, -5
K_UP, K_ESS, K_DOWN, K_ESS_REV, K_ONE = 0, 1, 2, 3, 4
ST_OK, ST_TRIVIAL, ST_EMPTY, ST_DISCONNECTED, ST_DEGENERATE, ST_UNKNOWN_NODE, ST_BAD_DESCRIPTOR, ST_NO_TREE_EDGES = range(8)
ST_NONFINITE = 8
ST_NAMES = ["OK", "TRIVIAL", "EMPTY", "DISCONNECTED", "DEGENERATE", "UNKNOWN_NODE", "BAD_DESCRIPTOR", "NO_TREE_EDGES",
            "NONFINITE"]

EXPORTS = ["tlc_graph_create", "tlc_graph_destroy", "tlc_vicinity_pi", "tlc_vicinity_pi_dev", "tlc_vicinity_sizes",
           "tlc_vicinity_detail", "tlc_union_find", "tlc_pimg_transform", "tlc_last_error", "tlc_version",
           "tlc_launch_count", "tlc_last_stage_ms", "tlc_last_algorithmic_bytes", "tlc_graph_set_stream",
           "tlc_last_counts", "tlc_last_direct", "tlc_pi_gather", "tlc_last_small", "tlc_small_diagrams",
           "tlc_table_create", "tlc_table_attach", "tlc_vicinity_pi_exchange", "tlc_last_table",
           "tlc_last_table_two_root",
           "tlc_ollivier_ricci", "tlc_graph_set_hks_time", "tlc_table_build_ms", "tlc_vicinity_diagrams",
           "tlc_vicinity_diagrams_dev", "tlc_pimg_batch_dev", "tlc_pimg_batch_grad_dev",
           "tlc_wasserstein_workspace_bytes", "tlc_wasserstein_batch_dev", "tlc_wasserstein_batch_grad_dev",
           "tlc_graph_batch_create", "tlc_graph_batch_destroy", "tlc_graph_batch_pair_bound",
           "tlc_graph_batch_diagrams_dev", "tlc_graph_batch_grad_dev", "tlc_vicinity_batch_dev",
           "tlc_graph_batch_create_dev"]


class Params(C.Structure):
    _fields_ = [("hop", C.c_int32), ("mode", C.c_int32), ("descriptor", C.c_int32), ("resolution", C.c_int32),
                ("flags", C.c_uint32), ("img_mask", C.c_uint32)]


class Detail(C.Structure):
    _fields_ = [("cap_v", C.c_int64), ("cap_e", C.c_int64), ("cap_p", C.c_int64),
                ("voff", C.c_void_p), ("eoff", C.c_void_p), ("poff", C.c_void_p),
                ("n", C.c_void_p), ("m", C.c_void_p), ("lu", C.c_void_p), ("lv", C.c_void_p),
                ("npairs", C.c_void_p), ("npos", C.c_void_p), ("nneg", C.c_void_p),
                ("vert", C.c_void_p), ("elo", C.c_void_p), ("ehi", C.c_void_p),
                ("ew", C.c_void_p), ("fval", C.c_void_p),
                ("ord_asc", C.c_void_p), ("ord_desc", C.c_void_p),
                ("pkind", C.c_void_p), ("pbv", C.c_void_p), ("pdv", C.c_void_p),
                ("pbirth", C.c_void_p), ("pdeath", C.c_void_p),
                ("pos", C.c_void_p), ("neg", C.c_void_p),
                ("pi", C.c_void_p), ("status", C.c_void_p), ("pi_up", C.c_void_p), ("pi_one", C.c_void_p)]


class Diagrams(C.Structure):
    """tlc_diagrams: the pair arrays of tlc_vicinity_diagrams(_dev), host or device addresses"""
    _fields_ = [("cap", C.c_int64), ("poff", C.c_void_p), ("npairs", C.c_void_p), ("kind", C.c_void_p),
                ("bv", C.c_void_p), ("dv", C.c_void_p), ("birth", C.c_void_p), ("death", C.c_void_p)]


class VicinityBatch(C.Structure):
    """tlc_vicinity_batch: the graph-batch layout of tlc_vicinity_batch_dev, device addresses"""
    _fields_ = [("cap_v", C.c_int64), ("cap_e", C.c_int64), ("voff", C.c_void_p), ("eoff", C.c_void_p),
                ("vert", C.c_void_p), ("ea", C.c_void_p), ("eb", C.c_void_p), ("fval", C.c_void_p)]


class TlcError(RuntimeError):
    def __init__(self, rc, msg):
        super().__init__("libtlc_b200 rc=%d: %s" % (rc, msg))
        self.rc = rc


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError("libtlc_b200.so not built (%s). There is no CPU fallback; run "
                          "`make -C tlc-gnn_b200/csrc` or `python -c 'import __graft_entry__ as g; g.build()'`." % SO_PATH)
    L = C.CDLL(SO_PATH)
    vp, i32, i64, u64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_uint32
    L.tlc_graph_create.restype = C.c_int
    L.tlc_graph_create.argtypes = [i32, i64, vp, vp, vp, C.c_int, u64, C.POINTER(vp)]
    L.tlc_graph_destroy.restype = C.c_int
    L.tlc_graph_destroy.argtypes = [vp]
    L.tlc_vicinity_pi.restype = C.c_int
    L.tlc_vicinity_pi.argtypes = [vp, vp, i64, C.POINTER(Params), vp, vp, C.POINTER(i64)]
    L.tlc_vicinity_pi_dev.restype = C.c_int
    L.tlc_vicinity_pi_dev.argtypes = [vp, vp, i64, C.POINTER(Params), vp, vp, vp, C.POINTER(i64)]
    L.tlc_vicinity_sizes.restype = C.c_int
    L.tlc_vicinity_sizes.argtypes = [vp, vp, i64, C.POINTER(Params), vp, vp, vp]
    L.tlc_vicinity_detail.restype = C.c_int
    L.tlc_vicinity_detail.argtypes = [vp, vp, i64, C.POINTER(Params), C.POINTER(Detail)]
    L.tlc_union_find.restype = C.c_int
    L.tlc_union_find.argtypes = [C.c_int, i32, i32, vp, vp, vp, u32] + [vp] * 11
    L.tlc_pimg_transform.restype = C.c_int
    L.tlc_pimg_transform.argtypes = [C.c_int, vp, i64, i32, vp]
    L.tlc_pimg_batch_dev.restype = C.c_int
    L.tlc_pimg_batch_dev.argtypes = [C.c_int, i64, vp, vp, vp, vp, u32, i32, vp, vp]
    L.tlc_pimg_batch_grad_dev.restype = C.c_int
    L.tlc_pimg_batch_grad_dev.argtypes = [C.c_int, i64, vp, vp, vp, vp, u32, i32, vp, vp, vp, vp]
    L.tlc_wasserstein_workspace_bytes.restype = C.c_int
    L.tlc_wasserstein_workspace_bytes.argtypes = [i64, i64, i64, C.POINTER(u64)]
    L.tlc_wasserstein_batch_dev.restype = C.c_int
    L.tlc_wasserstein_batch_dev.argtypes = ([C.c_int, i64, i64, i64] + [vp] * 8 + [u32, C.c_double, C.c_double, vp, u64]
                                            + [vp] * 4)
    L.tlc_wasserstein_batch_grad_dev.restype = C.c_int
    L.tlc_wasserstein_batch_grad_dev.argtypes = [C.c_int, i64] + [vp] * 8 + [u32, C.c_double, C.c_double] + [vp] * 9
    L.tlc_graph_batch_create.restype = C.c_int
    L.tlc_graph_batch_create.argtypes = [C.c_int, i64, vp, vp, vp, vp, C.POINTER(vp)]
    L.tlc_graph_batch_destroy.restype = C.c_int
    L.tlc_graph_batch_destroy.argtypes = [vp]
    L.tlc_graph_batch_pair_bound.restype = C.c_int
    L.tlc_graph_batch_pair_bound.argtypes = [vp, C.POINTER(i64)]
    L.tlc_graph_batch_diagrams_dev.restype = C.c_int
    L.tlc_graph_batch_diagrams_dev.argtypes = [vp, vp, u32, C.POINTER(Diagrams), vp, vp]
    L.tlc_graph_batch_grad_dev.restype = C.c_int
    L.tlc_graph_batch_grad_dev.argtypes = [vp, C.POINTER(Diagrams), vp, vp, vp, vp]
    L.tlc_vicinity_batch_dev.restype = C.c_int
    L.tlc_vicinity_batch_dev.argtypes = [vp, vp, i64, C.POINTER(Params), C.POINTER(VicinityBatch), vp, C.POINTER(i64),
                                         C.POINTER(i64)]
    L.tlc_graph_batch_create_dev.restype = C.c_int
    L.tlc_graph_batch_create_dev.argtypes = [C.c_int, i64, vp, vp, vp, vp, vp, C.POINTER(vp)]
    L.tlc_last_error.restype = C.c_char_p
    L.tlc_version.restype = C.c_char_p
    L.tlc_launch_count.restype = i64
    L.tlc_last_stage_ms.restype = C.c_int
    L.tlc_last_stage_ms.argtypes = [vp, vp]
    L.tlc_last_algorithmic_bytes.restype = C.c_int
    L.tlc_last_algorithmic_bytes.argtypes = [vp, vp, vp, vp]
    L.tlc_graph_set_stream.restype = C.c_int
    L.tlc_graph_set_stream.argtypes = [vp, vp]
    L.tlc_last_counts.restype = C.c_int
    L.tlc_last_counts.argtypes = [vp, vp]
    L.tlc_pi_gather.restype = C.c_int
    L.tlc_pi_gather.argtypes = [C.c_int, vp, i64, i32, vp, i64, i64, vp, vp]
    L.tlc_last_direct.restype = i64
    L.tlc_last_direct.argtypes = [vp]
    L.tlc_ollivier_ricci.restype = C.c_int
    L.tlc_ollivier_ricci.argtypes = [C.c_int, i32, i64, vp, vp, C.c_double, vp, vp]
    L.tlc_graph_set_hks_time.restype = C.c_int
    L.tlc_graph_set_hks_time.argtypes = [vp, C.c_double]
    L.tlc_table_build_ms.restype = C.c_double
    L.tlc_table_build_ms.argtypes = [vp]
    L.tlc_last_table.restype = i64
    L.tlc_last_table.argtypes = [vp]
    L.tlc_last_table_two_root.restype = i64
    L.tlc_last_table_two_root.argtypes = [vp]
    L.tlc_last_small.restype = C.c_int
    L.tlc_last_small.argtypes = [vp, vp]
    L.tlc_table_create.restype = C.c_int
    L.tlc_table_create.argtypes = [vp, i64, i32, C.POINTER(vp), vp]
    L.tlc_table_attach.restype = C.c_int
    L.tlc_table_attach.argtypes = [vp, i32, i32, vp]
    L.tlc_vicinity_pi_exchange.restype = C.c_int
    L.tlc_vicinity_pi_exchange.argtypes = [vp, vp, vp, i64, C.POINTER(Params), C.POINTER(i64)]
    L.tlc_small_diagrams.restype = C.c_int
    L.tlc_small_diagrams.argtypes = [vp, vp, i64, C.POINTER(Params), vp] + [vp] * 10
    for name in ("tlc_vicinity_diagrams", "tlc_vicinity_diagrams_dev"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [vp, vp, i64, C.POINTER(Params), C.POINTER(Diagrams), vp, vp, C.POINTER(i64)]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise TlcError(rc, lib().tlc_last_error().decode("utf-8", "replace"))


def default_img_mask(extended, kd=False):
    """which pair kinds are rasterised: riccidist2dgm.py:327-328 (PD_zero + PD_one) or, for the KD
    generators, Ord0 u Ext1 only (Knowledge_Distillation/data_utils_NC.py:172-180)."""
    if kd:
        return (1 << K_UP) | (1 << K_ONE)
    return (1 << K_UP) | (1 << K_ESS) | (1 << K_DOWN) | (1 << K_ESS_REV) | ((1 << K_ONE) if extended else 0)
