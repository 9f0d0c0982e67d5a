"""tlc_vicinity_diagrams / tlc_vicinity_diagrams_dev: argument checks that need no GPU (they run before any CUDA call)."""
import ctypes as C

import pytest

from tlc_b200 import _lib as L
from tlc_b200 import api


@pytest.mark.parametrize("name", ["tlc_vicinity_diagrams", "tlc_vicinity_diagrams_dev"])
def test_diagram_calls_reject_bad_arguments(name):
    fn = getattr(L.lib(), name)
    fake_graph = C.create_string_buffer(64)  # never dereferenced: every check below fails first
    poff = (C.c_int64 * 4)()
    tg = (C.c_int32 * 6)()
    good = L.Diagrams(0, C.addressof(poff), None, None, None, None, None, None)
    ok = api.make_params(2, L.MODE_EDGE, "sum", 5, L.F_NORM, None)
    cases = [
        (None, good, ok, "graph"),
        (fake_graph, None, ok, "poff"),
        (fake_graph, L.Diagrams(0, None, None, None, None, None, None, None), ok, "poff"),
        (fake_graph, L.Diagrams(-1, C.addressof(poff), None, None, None, None, None, None), ok, "cap"),
        (fake_graph, good, api.make_params(2, L.MODE_EDGE, "sum", 5, L.F_NORM | L.F_ASC_ONLY | L.F_EXTENDED, None), "ASC_ONLY"),
    ]
    for g, d, p, word in cases:
        total = C.c_int64(-9)
        rc = fn(C.addressof(g) if g is not None else None, C.addressof(tg), 3, C.byref(p),
                C.byref(d) if d is not None else None, None, None, C.byref(total))
        assert rc == L.E_INVALID, word
        assert word in L.lib().tlc_last_error().decode(), word
        assert total.value == -9
