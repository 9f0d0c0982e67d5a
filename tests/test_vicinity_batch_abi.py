"""tlc_vicinity_batch_dev and tlc_graph_batch_create_dev: the argument checks that need no GPU (they run before any CUDA
call) -- NULL required pointers, a disallowed flag, E out of range, bad tlc_params, negative capacities."""
import ctypes as C

import pytest

from tlc_b200 import _lib as L
from tlc_b200 import api

FAKE_GRAPH = C.create_string_buffer(64)  # never dereferenced: every check below fails first


def call_batch(g=FAKE_GRAPH, E=3, targets=True, p=None, out="good", status=None):
    voff = (C.c_int64 * 8)()
    eoff = (C.c_int64 * 8)()
    tg = (C.c_int32 * 8)()
    if out == "good":
        out = L.VicinityBatch(0, 0, C.addressof(voff), C.addressof(eoff), None, None, None, None)
    if p is None:
        p = api.make_params(2, L.MODE_EDGE, "sum", 5, L.F_NORM, None)
    tv, te = C.c_int64(-9), C.c_int64(-9)
    rc = L.lib().tlc_vicinity_batch_dev(C.addressof(g) if g is not None else None, C.addressof(tg) if targets else None,
                                        E, C.byref(p) if p is not False else None,
                                        C.byref(out) if out is not None else None, status, C.byref(tv), C.byref(te))
    return rc, L.lib().tlc_last_error().decode(), (tv.value, te.value)


def test_vicinity_batch_null_pointers():
    voff = (C.c_int64 * 8)()
    for kw, word in [(dict(g=None), "graph"), (dict(out=None), "voff"),
                     (dict(out=L.VicinityBatch(0, 0, None, C.addressof(voff), None, None, None, None)), "voff"),
                     (dict(out=L.VicinityBatch(0, 0, C.addressof(voff), None, None, None, None, None)), "eoff"),
                     (dict(targets=False), "targets"), (dict(p=False), "params")]:
        rc, msg, totals = call_batch(**kw)
        assert rc == L.E_INVALID and word in msg, (kw, msg)
        assert totals == (-9, -9)


@pytest.mark.parametrize("flag", [L.F_EXTENDED, L.F_KEEP_ZERO, L.F_EDGE_SORTED, L.F_NO_DIRECT, L.F_DIRECT, L.F_ASC_ONLY,
                                  L.F_NO_SMALL, L.F_NO_TABLE, 1 << 20])
def test_vicinity_batch_rejects_other_flags(flag):
    rc, msg, _ = call_batch(p=api.make_params(2, L.MODE_EDGE, "sum", 5, L.F_NORM | flag, None))
    assert rc == L.E_INVALID and "flags may only hold" in msg


def test_vicinity_batch_rejects_ranges_and_params():
    voff = (C.c_int64 * 8)()
    for kw, word in [(dict(E=-1), "E must be"), (dict(E=1 << 31), "E must be"),
                     (dict(out=L.VicinityBatch(-1, 0, C.addressof(voff), C.addressof(voff), None, None, None, None)), "cap"),
                     (dict(out=L.VicinityBatch(0, -1, C.addressof(voff), C.addressof(voff), None, None, None, None)), "cap"),
                     (dict(p=api.make_params(-1, L.MODE_EDGE, "sum", 5, L.F_NORM, None)), "hop"),
                     (dict(p=api.make_params(2, 7, "sum", 5, L.F_NORM, None)), "mode"),
                     (dict(p=api.make_params(2, -1, "sum", 5, L.F_NORM, None)), "mode")]:
        rc, msg, _ = call_batch(**kw)
        assert rc == L.E_INVALID and word in msg, (kw, msg)


def test_create_dev_rejects_before_cuda():
    lib = L.lib()
    off = (C.c_int64 * 4)()
    h = C.c_void_p()
    cases = [(dict(D=1, noff=off, eoff=off, out=None), "out"),
             (dict(D=-1, noff=off, eoff=off, out=h), "D must be"),
             (dict(D=1 << 31, noff=off, eoff=off, out=h), "D must be"),
             (dict(D=1, noff=None, eoff=off, out=h), "noff and eoff"),
             (dict(D=1, noff=off, eoff=None, out=h), "noff and eoff")]
    for a, word in cases:
        rc = lib.tlc_graph_batch_create_dev(0, a["D"], C.addressof(a["noff"]) if a["noff"] is not None else None,
                                            C.addressof(a["eoff"]) if a["eoff"] is not None else None, None, None, None,
                                            C.byref(a["out"]) if a["out"] is not None else None)
        assert rc == L.E_INVALID and word in lib.tlc_last_error().decode(), (a, word)


def test_from_device_rejects_bad_shapes():
    import torch
    with pytest.raises(ValueError, match="ptr"):
        api.GraphBatch.from_device(torch.zeros((2, 2), dtype=torch.int64), torch.zeros((2, 0), dtype=torch.int32))
    with pytest.raises(ValueError, match="edge_index"):
        api.GraphBatch.from_device(torch.zeros(2, dtype=torch.int64), torch.zeros((3, 1), dtype=torch.int32))
    with pytest.raises(ValueError, match="cuda"):  # host tensors are named before any CUDA call
        api.GraphBatch.from_device(torch.zeros(2, dtype=torch.int64), torch.zeros((2, 0), dtype=torch.int32))
