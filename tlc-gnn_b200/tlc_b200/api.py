"""Host-side API over the C-ABI: device-resident graph handle + batched calls.

`VicinityGraph` is what sg2dgm.riccidist2dgm.graph2pi (the drop-in mirror) holds: the CSR graph and
curvature uploaded once (graph2pi.__init__, riccidist2dgm.py:216-226), then one C-ABI call per batch
of targets (get_pimg_for_all_edges, :362-370).
"""
import ctypes as C
import math

import numpy as np

from . import _lib as L


_CUDA_STREAM_LEGACY = 0x1  # cudaStreamLegacy (driver_types.h): an explicit handle of the legacy default stream


def _check_layout(t, dtype_name, shape, what):
    if str(t.dtype) != "torch." + dtype_name:
        raise TypeError("%s must be %s, got %s" % (what, dtype_name, t.dtype))
    if tuple(t.shape) != tuple(shape):
        raise ValueError("%s must have shape %s, got %s" % (what, tuple(shape), tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % what)


def _dev_ptr(t, dtype_name, shape, device_index, what):
    """data pointer of a torch CUDA tensor that crosses the C-ABI: dtype, shape, contiguity and device are checked here,
    because the library can only see a raw address."""
    if t is None:
        return None
    _check_layout(t, dtype_name, shape, what)
    if t.device.type != "cuda" or (t.device.index is not None and t.device.index != device_index):
        raise ValueError("%s must live on cuda:%d, got %s" % (what, device_index, t.device))
    return t.data_ptr()


def make_params(hop=2, mode=L.MODE_EDGE, descriptor="sum", resolution=5, flags=L.F_NORM, img_mask=None):
    d = L.DESC.get(descriptor, -1) if isinstance(descriptor, str) else int(descriptor)
    if img_mask is None:
        img_mask = L.default_img_mask(bool(flags & L.F_EXTENDED), bool(flags & L.F_KEEP_ZERO))
    return L.Params(int(hop), int(mode), d, int(resolution), int(flags), int(img_mask))


class VicinityGraph:
    """CSR (ascending neighbour ids per row) + per-directed-edge curvature, resident on one GPU."""

    def __init__(self, rowptr, col, kappa, device=0, arena_bytes=0):
        self.rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
        self.col = np.ascontiguousarray(col, dtype=np.int32)
        self.kappa = np.ascontiguousarray(kappa, dtype=np.float64)
        self.N = int(self.rowptr.size - 1)
        self.nnz = int(self.col.size)
        self.device = int(device)
        self._h = C.c_void_p()
        L.check(L.lib().tlc_graph_create(self.N, self.nnz, self.rowptr.ctypes.data, self.col.ctypes.data,
                                         self.kappa.ctypes.data, self.device, int(arena_bytes), C.byref(self._h)))

    @classmethod
    def from_edges(cls, N, edges, kappa, device=0, arena_bytes=0):
        from .graphgen import build_csr
        return cls(*build_csr(N, edges, kappa), device=device, arena_bytes=arena_bytes)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            L.lib().tlc_graph_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- whole path, host buffers (the reference-facing call) ----
    def vicinity_pi(self, targets, hop=2, mode=L.MODE_EDGE, descriptor="sum", resolution=5, flags=L.F_NORM,
                    img_mask=None, out=None):
        t = np.ascontiguousarray(targets, dtype=np.int32).reshape(-1, 2)
        E = t.shape[0]
        p = make_params(hop, mode, descriptor, resolution, flags, img_mask)
        r2 = resolution * resolution
        pi = out if out is not None else np.zeros((E, r2), dtype=np.float64)
        assert pi.dtype == np.float64 and pi.flags.c_contiguous and pi.shape == (E, r2)
        status = np.zeros(E, dtype=np.uint8)
        cnt = C.c_int64(0)
        L.check(L.lib().tlc_vicinity_pi(self._h, t.ctypes.data, E, C.byref(p), pi.ctypes.data, status.ctypes.data,
                                        C.byref(cnt)))
        return pi, status, int(cnt.value)

    # ---- whole path, device buffers (torch tensors on this graph's device) ----
    def vicinity_pi_dev(self, targets_dev, out_pi, out_pi_f32=None, out_status=None, hop=2, mode=L.MODE_EDGE,
                        descriptor="sum", resolution=5, flags=L.F_NORM, img_mask=None, want_count=False):
        """targets_dev int32[E,2], out_pi float64[E,res^2] (+ optional float32 copy, uint8 status):
        torch CUDA tensors; only their data pointers cross the C-ABI."""
        E = int(targets_dev.shape[0])
        p = make_params(hop, mode, descriptor, resolution, flags, img_mask)
        r2 = int(resolution) * int(resolution)
        cnt = C.c_int64(0)
        L.check(L.lib().tlc_vicinity_pi_dev(
            self._h, _dev_ptr(targets_dev, "int32", (E, 2), self.device, "targets_dev"), E, C.byref(p),
            _dev_ptr(out_pi, "float64", (E, r2), self.device, "out_pi"),
            _dev_ptr(out_pi_f32, "float32", (E, r2), self.device, "out_pi_f32"),
            _dev_ptr(out_status, "uint8", (E,), self.device, "out_status"),
            C.byref(cnt) if want_count else None))
        return int(cnt.value)

    def vicinity_sizes(self, targets, hop=2, mode=L.MODE_EDGE):
        t = np.ascontiguousarray(targets, dtype=np.int32).reshape(-1, 2)
        E = t.shape[0]
        p = make_params(hop, mode)
        n = np.zeros(E, np.int32)
        m = np.zeros(E, np.int32)
        st = np.zeros(E, np.uint8)
        L.check(L.lib().tlc_vicinity_sizes(self._h, t.ctypes.data, E, C.byref(p), n.ctypes.data, m.ctypes.data,
                                           st.ctypes.data))
        return n, m, st

    def vicinity_detail(self, targets, hop=2, mode=L.MODE_EDGE, descriptor="sum", resolution=5, flags=L.F_NORM,
                        img_mask=None):
        """every intermediate of the path for a small batch (stage-level parity tests)."""
        t = np.ascontiguousarray(targets, dtype=np.int32).reshape(-1, 2)
        E = t.shape[0]
        n, m, _ = self.vicinity_sizes(t, hop, mode)
        Nv, Ne = int(n.sum()), int(m.sum())
        Np = Nv + Ne + E
        p = make_params(hop, mode, descriptor, resolution, flags, img_mask)
        a = dict(voff=np.zeros(E + 1, np.int64), eoff=np.zeros(E + 1, np.int64), poff=np.zeros(E + 1, np.int64),
                 n=np.zeros(E, np.int32), m=np.zeros(E, np.int32), lu=np.zeros(E, np.int32), lv=np.zeros(E, np.int32),
                 npairs=np.zeros(E, np.int32), npos=np.zeros(E, np.int32), nneg=np.zeros(E, np.int32),
                 vert=np.zeros(Nv + 1, np.int32), elo=np.zeros(Ne + 1, np.int32), ehi=np.zeros(Ne + 1, np.int32),
                 ew=np.zeros(Ne + 1), fval=np.zeros(Nv + 1),
                 ord_asc=np.zeros(Ne + 1, np.int32), ord_desc=np.zeros(Ne + 1, np.int32),
                 pkind=np.zeros(Np + 1, np.int32), pbv=np.zeros(Np + 1, np.int32), pdv=np.zeros(Np + 1, np.int32),
                 pbirth=np.zeros(Np + 1), pdeath=np.zeros(Np + 1),
                 pos=np.zeros(Ne + 1, np.int32), neg=np.zeros(Nv + 1, np.int32),
                 pi=np.zeros((E, resolution * resolution)), status=np.zeros(E, np.uint8),
                 pi_up=np.zeros((E, resolution * resolution)), pi_one=np.zeros((E, resolution * resolution)))
        d = L.Detail()
        d.cap_v, d.cap_e, d.cap_p = Nv, Ne, Np
        for k, arr in a.items():
            setattr(d, k, arr.ctypes.data)
        L.check(L.lib().tlc_vicinity_detail(self._h, t.ctypes.data, E, C.byref(p), C.byref(d)))
        return a

    def per_target(self, a, i):
        """slice one target's segments out of a vicinity_detail() result."""
        vo, ve = a["voff"][i], a["voff"][i + 1]
        eo, ee = a["eoff"][i], a["eoff"][i + 1]
        po = a["poff"][i]
        np_ = a["npairs"][i]
        out = dict(status=int(a["status"][i]), n=int(a["n"][i]), m=int(a["m"][i]), lu=int(a["lu"][i]), lv=int(a["lv"][i]),
                   img=a["pi"][i], img_up=a["pi_up"][i], img_one=a["pi_one"][i])
        for k in ("vert", "fval"):
            out[k] = a[k][vo:ve]
        for k in ("elo", "ehi", "ew", "ord_asc", "ord_desc"):
            out[k] = a[k][eo:ee]
        for k in ("pkind", "pbv", "pdv", "pbirth", "pdeath"):
            out[k] = a[k][po:po + np_]
        out["pos"] = a["pos"][eo:eo + a["npos"][i]]
        out["neg"] = a["neg"][vo:vo + a["nneg"][i]]
        return out

    def small_diagrams(self, targets, hop=2, mode=L.MODE_EDGE, descriptor="sum", flags=L.F_NORM, img_mask=None):
        """diagrams straight from the fused small-vicinity kernels (kernel S): a list with one dict per target
        (status, n, m, img, pkind, pbv, pdv, pbirth, pdeath); targets kernel S cannot take have status ST_NOT_SMALL."""
        t = np.ascontiguousarray(targets, dtype=np.int32).reshape(-1, 2)
        E = t.shape[0]
        n, m, _ = self.vicinity_sizes(t, hop, mode)
        cap = n.astype(np.int64) + m.astype(np.int64) + 2
        poff = np.zeros(E + 1, np.int64)
        np.cumsum(cap, out=poff[1:])
        P = int(poff[-1])
        p = make_params(hop, mode, descriptor, 5, flags, img_mask)
        npairs = np.zeros(E, np.int32)
        pkind = np.zeros(P + 1, np.int32); pbv = np.zeros(P + 1, np.int32); pdv = np.zeros(P + 1, np.int32)
        pbirth = np.zeros(P + 1); pdeath = np.zeros(P + 1)
        pi = np.zeros((E, 25)); st = np.zeros(E, np.uint8)
        on = np.zeros(E, np.int32); om = np.zeros(E, np.int32)
        L.check(L.lib().tlc_small_diagrams(self._h, t.ctypes.data, E, C.byref(p), poff.ctypes.data, npairs.ctypes.data,
                                           pkind.ctypes.data, pbv.ctypes.data, pdv.ctypes.data, pbirth.ctypes.data,
                                           pdeath.ctypes.data, pi.ctypes.data, st.ctypes.data, on.ctypes.data, om.ctypes.data))
        out = []
        for i in range(E):
            a, b = int(poff[i]), int(poff[i]) + int(npairs[i])
            out.append(dict(status=int(st[i]), n=int(on[i]), m=int(om[i]), img=pi[i], pkind=pkind[a:b], pbv=pbv[a:b],
                            pdv=pdv[a:b], pbirth=pbirth[a:b], pdeath=pdeath[a:b]))
        return out

    # ---- persistence diagrams of a batch (include/tlc_b200.h: tlc_vicinity_diagrams*) ----
    _diagram_cap = 0  # grow-only guess of the pair arrays' capacity

    def _diagrams(self, fn, targets_ptr, E, p, alloc, pi_ptr, st_ptr, cap):
        """one diagram call with the capacity guess (or `cap` pairs), once more with the exact total on TLC_E_CAPACITY;
        alloc(cap) -> (arrays dict, Diagrams struct)"""
        total = C.c_int64(0)
        cap = max(self._diagram_cap, 8 * E) if cap is None else int(cap)
        for attempt in range(2):
            arrs, d = alloc(cap)
            rc = fn(self._h, targets_ptr, E, C.byref(p), C.byref(d), pi_ptr, st_ptr, C.byref(total))
            if rc == L.E_CAPACITY and attempt == 0:
                cap = int(total.value)
                continue
            L.check(rc)
            break
        self._diagram_cap = max(self._diagram_cap, cap)
        return arrs, int(total.value)

    def vicinity_diagrams(self, targets, hop=2, mode=L.MODE_EDGE, descriptor="sum", resolution=5, flags=L.F_NORM,
                          img_mask=None, cap=None):
        """the persistence diagrams of a batch, host buffers: dict of numpy arrays poff int64[E+1] (target t's pairs are
        [poff[t], poff[t+1])), kind uint8, bv / dv int32 (graph ids), birth / death float64, status uint8[E] and the image
        rows pi float64[E, res^2].  cap: capacity of the first attempt in pairs (default: a grow-only guess); a call that
        needs more is repeated once with the exact total"""
        t = np.ascontiguousarray(targets, dtype=np.int32).reshape(-1, 2)
        E = t.shape[0]
        p = make_params(hop, mode, descriptor, resolution, flags, img_mask)
        pi = np.zeros((E, int(resolution) * int(resolution)))
        status = np.zeros(E, np.uint8)
        poff = np.zeros(E + 1, np.int64)

        def alloc(cap):
            a = dict(poff=poff, kind=np.zeros(cap, np.uint8), bv=np.zeros(cap, np.int32), dv=np.zeros(cap, np.int32),
                     birth=np.zeros(cap), death=np.zeros(cap))
            d = L.Diagrams(cap, poff.ctypes.data, None, *(a[k].ctypes.data for k in ("kind", "bv", "dv", "birth", "death")))
            return a, d

        a, total = self._diagrams(L.lib().tlc_vicinity_diagrams, t.ctypes.data, E, p, alloc, pi.ctypes.data,
                                  status.ctypes.data, cap)
        out = {k: (v if k == "poff" else v[:total]) for k, v in a.items()}
        out.update(status=status, pi=pi)
        return out

    def vicinity_diagrams_dev(self, targets_dev, hop=2, mode=L.MODE_EDGE, descriptor="sum", resolution=5, flags=L.F_NORM,
                              img_mask=None, want_pi=False, cap=None):
        """the persistence diagrams of a batch, device buffers: targets_dev int32[E, 2] (torch, this graph's device) ->
        dict of CUDA tensors poff int64[E+1], kind uint8, bv / dv int32 (graph ids), birth / death float64, status uint8[E]
        and, with want_pi, the image rows pi float64[E, res^2] (else None); cap as in vicinity_diagrams"""
        import torch
        E = int(targets_dev.shape[0])
        dev = torch.device("cuda", self.device)
        tp = _dev_ptr(targets_dev, "int32", (E, 2), self.device, "targets_dev") if E else None
        p = make_params(hop, mode, descriptor, resolution, flags, img_mask)
        pi = torch.zeros((E, int(resolution) * int(resolution)), dtype=torch.float64, device=dev) if want_pi else None
        status = torch.zeros(E, dtype=torch.uint8, device=dev)
        poff = torch.zeros(E + 1, dtype=torch.int64, device=dev)
        torch.cuda.synchronize(dev)  # (the library works on its own stream)

        def alloc(cap):
            a = dict(poff=poff, kind=torch.empty(cap, dtype=torch.uint8, device=dev),
                     bv=torch.empty(cap, dtype=torch.int32, device=dev), dv=torch.empty(cap, dtype=torch.int32, device=dev),
                     birth=torch.empty(cap, dtype=torch.float64, device=dev),
                     death=torch.empty(cap, dtype=torch.float64, device=dev))
            torch.cuda.synchronize(dev)
            d = L.Diagrams(cap, poff.data_ptr(), None, *(a[k].data_ptr() for k in ("kind", "bv", "dv", "birth", "death")))
            return a, d

        a, total = self._diagrams(L.lib().tlc_vicinity_diagrams_dev, tp, E, p, alloc,
                                  pi.data_ptr() if pi is not None else None, status.data_ptr(), cap)
        out = {k: (v if k == "poff" else v[:total]) for k, v in a.items()}
        out.update(status=status, pi=pi)
        return out

    # ---- vicinities in graph-batch layout (include/tlc_b200.h: tlc_vicinity_batch_dev) ----
    _batch_cap = (0, 0)  # grow-only guess of the vertex / edge capacities

    def vicinity_batch_dev(self, targets_dev, hop=2, mode=L.MODE_EDGE, descriptor="sum", flags=L.F_NORM, fval=True):
        """the vicinities of a batch and their filtration in graph-batch (PyG Batch) layout, device buffers: targets_dev
        int32[E, 2] (torch, this graph's device) -> dict of CUDA tensors ptr / eptr int64[E+1] (target t's vertices are
        [ptr[t], ptr[t+1]), its edges [eptr[t], eptr[t+1])), vert int32 (graph ids, ascending inside a target),
        edge_index int32[2, M] (batch ids, row 0 < row 1, lexicographic inside a target: canonical form, ready for
        GraphBatch.from_device), fval float64 (the filtration tlc_vicinity_detail computes; NaN for every target whose
        status is neither OK nor TRIVIAL) or None with fval=False (no filtration is computed), and status uint8[E].
        flags: F_NORM, F_NORM_EPS, F_SUM_PLAIN and the F_FILT_* filtrations.  A call that needs more room than the
        grow-only guess is repeated once with the exact totals, as vicinity_diagrams_dev does."""
        import torch
        E = int(targets_dev.shape[0])
        dev = torch.device("cuda", self.device)
        tp = _dev_ptr(targets_dev, "int32", (E, 2), self.device, "targets_dev") if E else None
        p = make_params(hop, mode, descriptor, 5, flags, 0)
        ptr = torch.zeros(E + 1, dtype=torch.int64, device=dev)
        eptr = torch.zeros(E + 1, dtype=torch.int64, device=dev)
        status = torch.zeros(E, dtype=torch.uint8, device=dev)
        tv, te = C.c_int64(0), C.c_int64(0)
        cap_v, cap_e = self._batch_cap
        for attempt in range(2):
            vert = torch.empty(cap_v, dtype=torch.int32, device=dev)
            ei = torch.empty((2, cap_e), dtype=torch.int32, device=dev)
            fv = torch.empty(cap_v, dtype=torch.float64, device=dev) if fval else None
            torch.cuda.synchronize(dev)  # (the library works on its own stream)
            b = L.VicinityBatch(cap_v, cap_e, ptr.data_ptr(), eptr.data_ptr(), vert.data_ptr(), ei[0].data_ptr(),
                                ei[1].data_ptr(), fv.data_ptr() if fv is not None else None)
            rc = L.lib().tlc_vicinity_batch_dev(self._h, tp, E, C.byref(p), C.byref(b), status.data_ptr() if E else None,
                                                C.byref(tv), C.byref(te))
            if rc == L.E_CAPACITY and attempt == 0:
                cap_v, cap_e = int(tv.value), int(te.value)
                continue
            L.check(rc)
            break
        V, M = int(tv.value), int(te.value)
        self._batch_cap = (max(self._batch_cap[0], cap_v), max(self._batch_cap[1], cap_e))
        return dict(ptr=ptr, eptr=eptr, vert=vert[:V], edge_index=ei if M == cap_e else ei[:, :M].contiguous(),
                    fval=fv[:V] if fv is not None else None, status=status)

    # ---- multi-GPU exchange by peer stores (include/tlc_b200.h: tlc_table_*) ----
    def table_create(self, rows, resolution=5):
        """this rank's exchange table float32[rows][res^2 + 1]: -> (device address of row 0, 64-byte CUDA IPC handle)"""
        ptr = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        L.check(L.lib().tlc_table_create(self._h, int(rows), int(resolution) * int(resolution), C.byref(ptr), handle))
        return int(ptr.value), bytes(handle)

    def table_attach(self, handles, my_rank):
        """handles: the 64-byte IPC handles of ALL ranks, ordered by rank"""
        blob = b"".join(handles)
        assert len(blob) == 64 * len(handles)
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        L.check(L.lib().tlc_table_attach(self._h, len(handles), int(my_rank), buf))

    def vicinity_pi_exchange(self, targets_dev, row_index_dev, hop=2, mode=L.MODE_EDGE, descriptor="sum", resolution=5,
                             flags=L.F_NORM, img_mask=None):
        """this rank's shard (torch CUDA tensors int32[k,2], int64[k]) through the path, every row stored at its final
        index into the exchange table of every rank; asynchronous on the graph's stream"""
        k = int(targets_dev.shape[0])
        p = make_params(hop, mode, descriptor, resolution, flags, img_mask)
        L.check(L.lib().tlc_vicinity_pi_exchange(
            self._h, _dev_ptr(targets_dev, "int32", (k, 2), self.device, "targets_dev") if k else None,
            _dev_ptr(row_index_dev, "int64", (k,), self.device, "row_index_dev") if k else None, k, C.byref(p), None))

    def set_hks_time(self, t):
        """diffusion time of the heat-kernel-signature filtration (flag F_FILT_HKS; data_utils_NC: hks_time = 0.1)"""
        L.check(L.lib().tlc_graph_set_hks_time(self._h, float(t)))

    def table_build_ms(self):
        """device ms of the one-time build of the per-root shortest-path tables (kernel 1t), 0 if they are not in use"""
        return float(L.lib().tlc_table_build_ms(self._h))

    def last_small(self):
        """kernel S in the last call: device ms of its two launches (TLC_STAGE_TIMING=1), rows finished per class, rows
        handed on to the staged pipeline."""
        out = np.zeros(7)
        L.lib().tlc_last_small(self._h, out.ctypes.data)
        return dict(ms_a=float(out[0]), ms_b=float(out[1]), ms_c=float(out[2]), rows_a=int(out[3]), rows_b=int(out[4]),
                    rows_c=int(out[5]), rows_staged=int(out[6]))

    def last_stage_ms(self):
        out = np.zeros(10)
        nch = L.lib().tlc_last_stage_ms(self._h, out.ctypes.data)
        names = ["sizes", "fill", "filtration", "vorder", "sweep", "sort", "union_find", "loops", "image", "total"]
        return dict(zip(names, out.tolist())), int(nch)

    def set_stream(self, cuda_stream_ptr):
        """run on a caller-owned stream, e.g. torch.cuda.current_stream().cuda_stream.
        None restores the graph's own (non-blocking) stream.  0 -- what torch reports for its default stream -- selects the
        LEGACY default stream (cudaStreamLegacy), i.e. the stream the caller's default-stream work is ordered with; it is
        not silently replaced by the library's own stream."""
        if cuda_stream_ptr is None:
            ptr = None
        else:
            ptr = C.c_void_p(int(cuda_stream_ptr) if int(cuda_stream_ptr) != 0 else _CUDA_STREAM_LEGACY)
        L.check(L.lib().tlc_graph_set_stream(self._h, ptr))

    def last_counts(self):
        out = np.zeros(8, np.int64)
        L.lib().tlc_last_counts(self._h, out.ctypes.data)
        return dict(live=int(out[0]), sum_n=int(out[1]), sum_m=int(out[2]), chunks=int(out[3]), handed_back=int(out[4]),
                    blocks_general=int(out[5]), blocks_rowcheck=int(out[6]), blocks=int(out[7]),
                    graph_row_route=int(L.lib().tlc_last_direct(self._h)), table_route=int(L.lib().tlc_last_table(self._h)),
                    table_two_root=int(L.lib().tlc_last_table_two_root(self._h)))

    def last_algorithmic_bytes(self):
        tot = C.c_double(0)
        L.lib().tlc_last_algorithmic_bytes(self._h, C.byref(tot), None, None)
        return float(tot.value)


def union_find(fval, edges, flags=0, device=0):
    """Union_find + Accelerate_PD on one caller-supplied graph (accelerated_PD.py:26,115): edges in the
    caller's order (that order is the tie-break).  Returns a dict of pairs / pos / neg."""
    f = np.ascontiguousarray(fval, dtype=np.float64)
    e = np.ascontiguousarray(edges, dtype=np.int32).reshape(-1, 2)
    n, m = f.size, e.shape[0]
    a = np.ascontiguousarray(e[:, 0])
    b = np.ascontiguousarray(e[:, 1])
    cap = n + m + 2
    pkind = np.zeros(cap, np.int32); pbv = np.zeros(cap, np.int32); pdv = np.zeros(cap, np.int32)
    pbirth = np.zeros(cap); pdeath = np.zeros(cap)
    pos = np.zeros(m + 1, np.int32); neg = np.zeros(n + 1, np.int32)
    npairs = C.c_int32(0); npos = C.c_int32(0); nneg = C.c_int32(0); status = C.c_uint8(0)
    L.check(L.lib().tlc_union_find(device, n, m, f.ctypes.data, a.ctypes.data, b.ctypes.data, int(flags),
                                   C.addressof(npairs), pkind.ctypes.data, pbv.ctypes.data, pdv.ctypes.data,
                                   pbirth.ctypes.data, pdeath.ctypes.data, C.addressof(npos), pos.ctypes.data,
                                   C.addressof(nneg), neg.ctypes.data, C.addressof(status)))
    k = npairs.value
    return dict(status=int(status.value), pkind=pkind[:k], pbv=pbv[:k], pdv=pdv[:k], pbirth=pbirth[:k],
                pdeath=pdeath[:k], pos=pos[:npos.value], neg=neg[:nneg.value])


def pimg_transform(dgm, resolution=5, device=0):
    """PersistenceImager(resolution).transform(dgm) on the GPU (PersistenceImager.pyx:352-388)."""
    d = np.ascontiguousarray(dgm, dtype=np.float64).reshape(-1, 2)
    out = np.zeros(resolution * resolution)
    L.check(L.lib().tlc_pimg_transform(device, d.ctypes.data, d.shape[0], resolution, out.ctypes.data))
    return out.reshape(resolution, resolution)


_ImagesFn = None


def _images_fn():
    """the torch.autograd.Function over tlc_pimg_batch_dev / tlc_pimg_batch_grad_dev (built on first use: torch is only
    imported by the calls that take tensors)"""
    global _ImagesFn
    if _ImagesFn is not None:
        return _ImagesFn
    import torch
    from torch.autograd.function import once_differentiable

    def stream(dev):
        return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    class PersistenceImages(torch.autograd.Function):
        @staticmethod
        def forward(ctx, poff, birth, death, kind, img_mask, resolution):
            dev = birth.device
            D, r2 = poff.shape[0] - 1, resolution * resolution
            out = torch.empty((D, r2), dtype=torch.float64, device=dev)
            L.check(L.lib().tlc_pimg_batch_dev(dev.index, D, poff.data_ptr(), birth.data_ptr(), death.data_ptr(),
                                               kind.data_ptr() if kind is not None else None, img_mask, resolution,
                                               out.data_ptr(), stream(dev)))
            ctx.save_for_backward(poff, birth, death, kind)
            ctx.img_mask, ctx.resolution = img_mask, resolution
            return out

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_out):
            poff, birth, death, kind = ctx.saved_tensors
            dev = birth.device
            D, r2 = poff.shape[0] - 1, ctx.resolution * ctx.resolution
            g = grad_out.contiguous()
            _dev_ptr(g, "float64", (D, r2), dev.index, "grad_out")
            # the kernel writes [poff[0], poff[D]); the points outside every segment keep their zero
            gb = torch.zeros_like(birth) if ctx.needs_input_grad[1] else None
            gd = torch.zeros_like(death) if ctx.needs_input_grad[2] else None
            L.check(L.lib().tlc_pimg_batch_grad_dev(
                dev.index, D, poff.data_ptr(), birth.data_ptr(), death.data_ptr(),
                kind.data_ptr() if kind is not None else None, ctx.img_mask, ctx.resolution, g.data_ptr(),
                gb.data_ptr() if gb is not None else None, gd.data_ptr() if gd is not None else None, stream(dev)))
            return None, gb, gd, None, None, None

    _ImagesFn = PersistenceImages
    return _ImagesFn


def persistence_images(poff, birth, death, kind=None, img_mask=None, resolution=5):
    """persistence images of a batch of diagrams on the GPU, differentiable in birth and death: the batched
    Knowledge_Distillation/pimg.py `transform` (PersistenceImager(resolution).transform, PersistenceImager.pyx:352-388).
    poff int64[D+1], birth / death float64[P], kind uint8[P] (optional): CUDA tensors on one device; diagram t is the
    points poff[t] .. poff[t+1], which must be non-decreasing and lie in [0, P].  img_mask: bit k set -> points of kind k
    count (None: every kind; needs `kind`).  Returns float64[D, res^2], birth-major.  Forward and backward run on the
    current stream of the device.  The output of VicinityGraph.vicinity_diagrams_dev plugs in directly:
    persistence_images(d["poff"], d["birth"], d["death"], d["kind"], mask)."""
    if img_mask is not None and kind is None:
        raise ValueError("img_mask selects kinds: pass kind as well")
    resolution = int(resolution)
    if not 1 <= resolution <= 16:
        raise ValueError("resolution must be in 1..16, got %d" % resolution)
    if getattr(birth, "dim", lambda: 0)() != 1 or getattr(poff, "dim", lambda: 0)() != 1 or poff.shape[0] < 1:
        raise ValueError("poff must be 1-D with D + 1 >= 1 entries and birth 1-D")
    dev = birth.device.index if birth.device.type == "cuda" else 0
    P = int(birth.shape[0])
    specs = [(poff, "int64", (int(poff.shape[0]),), "poff"), (birth, "float64", (P,), "birth"),
             (death, "float64", (P,), "death"), (kind, "uint8", (P,), "kind")]
    for t, dtype_name, shape, what in specs:  # the layout of all of them first: a bad one is named wherever they live
        if t is not None:
            _check_layout(t, dtype_name, shape, what)
    for spec in specs:
        _dev_ptr(spec[0], spec[1], spec[2], dev, spec[3])
    mask = 0xFFFFFFFF if img_mask is None else int(img_mask) & 0xFFFFFFFF
    return _images_fn().apply(poff, birth, death, kind, mask, resolution)


_WassersteinFn = None


def _wasserstein_fn():
    """the torch.autograd.Function over tlc_wasserstein_batch_dev / tlc_wasserstein_batch_grad_dev (built on first use)"""
    global _WassersteinFn
    if _WassersteinFn is not None:
        return _WassersteinFn
    import torch
    from torch.autograd.function import once_differentiable

    def stream(dev):
        return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def ptr(t):
        return t.data_ptr() if t is not None else None

    class WassersteinDistances(torch.autograd.Function):
        @staticmethod
        def forward(ctx, poff_x, birth_x, death_x, kind_x, poff_y, birth_y, death_y, kind_y, mask, order, internal_p):
            dev = birth_x.device
            D, Px, Py = poff_x.shape[0] - 1, birth_x.shape[0], birth_y.shape[0]
            nbytes = C.c_uint64()
            L.check(L.lib().tlc_wasserstein_workspace_bytes(D, Px, Py, C.byref(nbytes)))
            ws = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=dev)
            dist = torch.empty(D, dtype=torch.float64, device=dev)
            # the kernel writes [poff[0], poff[D]); the points outside every segment keep -2 (not in any pair)
            mx = torch.full((Px,), -2, dtype=torch.int64, device=dev)
            my = torch.full((Py,), -2, dtype=torch.int64, device=dev)
            L.check(L.lib().tlc_wasserstein_batch_dev(
                dev.index, D, Px, Py, ptr(poff_x), ptr(birth_x), ptr(death_x), ptr(kind_x), ptr(poff_y), ptr(birth_y),
                ptr(death_y), ptr(kind_y), mask, order, internal_p, ws.data_ptr(), nbytes.value, dist.data_ptr(),
                mx.data_ptr(), my.data_ptr(), stream(dev)))
            ctx.save_for_backward(poff_x, birth_x, death_x, kind_x, poff_y, birth_y, death_y, kind_y, dist, mx, my)
            ctx.mask, ctx.order, ctx.internal_p = mask, order, internal_p
            ctx.mark_non_differentiable(mx, my)
            return dist, mx, my

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_dist, _gmx, _gmy):
            poff_x, birth_x, death_x, kind_x, poff_y, birth_y, death_y, kind_y, dist, mx, my = ctx.saved_tensors
            dev = birth_x.device
            D = poff_x.shape[0] - 1
            g = grad_dist.contiguous()
            _dev_ptr(g, "float64", (D,), dev.index, "grad_out")
            # the kernel writes [poff[0], poff[D]); the points outside every segment keep their zero
            need = ctx.needs_input_grad
            grads = [torch.zeros_like(t) if need[k] else None
                     for k, t in ((1, birth_x), (2, death_x), (5, birth_y), (6, death_y))]
            L.check(L.lib().tlc_wasserstein_batch_grad_dev(
                dev.index, D, ptr(poff_x), ptr(birth_x), ptr(death_x), ptr(kind_x), ptr(poff_y), ptr(birth_y),
                ptr(death_y), ptr(kind_y), ctx.mask, ctx.order, ctx.internal_p, dist.data_ptr(), mx.data_ptr(),
                my.data_ptr(), g.data_ptr(), *[ptr(t) for t in grads], stream(dev)))
            gbx, gdx, gby, gdy = grads
            return None, gbx, gdx, None, None, gby, gdy, None, None, None, None

    _WassersteinFn = WassersteinDistances
    return _WassersteinFn


def wasserstein_distances(poff_x, birth_x, death_x, poff_y, birth_y, death_y, kind_x=None, kind_y=None, kind_mask=None,
                          order=1.0, internal_p=math.inf, return_matching=False):
    """exact Wasserstein distances between D pairs of diagrams on the GPU, differentiable in the four point tensors:
    the batched gudhi wasserstein_distance(X, Y, order, internal_p, enable_autodiff=True) of
    Knowledge_Distillation/wasserstein.py.  Pair t is X = points poff_x[t] .. poff_x[t+1] of birth_x / death_x and
    Y = points poff_y[t] .. poff_y[t+1] of birth_y / death_y (poff int64[D+1], non-decreasing; birth / death float64;
    kind uint8, optional): CUDA tensors on one device.  kind_mask: bit k set -> points of kind k count (None: every
    kind); a side without `kind` counts all its points.  The defaults are gudhi's (order 1, internal_p inf).
    Returns float64[D], and with return_matching=True also (match_x int64[len(birth_x)], match_y int64[len(birth_y)]):
    the global index of the matched point of the other side, -1 the diagonal, -2 masked out or in no pair.  A pair with
    a non-finite selected point gives NaN.  Runs on the current stream of the device.  The output of
    VicinityGraph.vicinity_diagrams_dev plugs in directly: wasserstein_distances(a["poff"], a["birth"], a["death"],
    b["poff"], b["birth"], b["death"], a["kind"], b["kind"], mask)."""
    if kind_mask is not None and kind_x is None and kind_y is None:
        raise ValueError("kind_mask selects kinds: pass kind_x or kind_y as well")
    order, internal_p = float(order), float(internal_p)
    if not (order >= 1.0 and math.isfinite(order)):
        raise ValueError("order must be finite and >= 1, got %r" % order)
    if not internal_p >= 1.0:
        raise ValueError("internal_p must be >= 1 or inf, got %r" % internal_p)
    for po, b, what in ((poff_x, birth_x, "x"), (poff_y, birth_y, "y")):
        if getattr(b, "dim", lambda: 0)() != 1 or getattr(po, "dim", lambda: 0)() != 1 or po.shape[0] < 1:
            raise ValueError("poff_%s must be 1-D with D + 1 >= 1 entries and birth_%s 1-D" % (what, what))
    if poff_x.shape[0] != poff_y.shape[0]:
        raise ValueError("poff_x and poff_y must have the same length, got %d and %d"
                         % (poff_x.shape[0], poff_y.shape[0]))
    dev = birth_x.device.index if birth_x.device.type == "cuda" else 0
    Px, Py, D1 = int(birth_x.shape[0]), int(birth_y.shape[0]), int(poff_x.shape[0])
    specs = [(poff_x, "int64", (D1,), "poff_x"), (birth_x, "float64", (Px,), "birth_x"),
             (death_x, "float64", (Px,), "death_x"), (kind_x, "uint8", (Px,), "kind_x"),
             (poff_y, "int64", (D1,), "poff_y"), (birth_y, "float64", (Py,), "birth_y"),
             (death_y, "float64", (Py,), "death_y"), (kind_y, "uint8", (Py,), "kind_y")]
    for t, dtype_name, shape, what in specs:  # the layout of all of them first: a bad one is named wherever they live
        if t is not None:
            _check_layout(t, dtype_name, shape, what)
    for spec in specs:
        _dev_ptr(spec[0], spec[1], spec[2], dev, spec[3])
    mask = 0xFFFFFFFF if kind_mask is None else int(kind_mask) & 0xFFFFFFFF
    dist, mx, my = _wasserstein_fn().apply(poff_x, birth_x, death_x, kind_x, poff_y, birth_y, death_y, kind_y, mask,
                                           order, internal_p)
    return (dist, (mx, my)) if return_matching else dist


def _to_numpy(a, dtype):
    if hasattr(a, "detach"):  # a CPU torch tensor
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=dtype)


def normalize_edge_index(ptr, edge_index):
    """the C-ABI's edge lists from PyG's Batch.ptr int[D+1] and edge_index int[2, E] (numpy or CPU tensors): the first
    occurrence of every undirected edge is kept, as given, and later ones (either direction) are dropped; the kept edges
    are grouped by the graph of their first endpoint, in input order inside a graph (that order is the sweeps'
    tie-break).  Self-loops and out-of-range or cross-graph edges are kept for tlc_graph_batch_create to reject.
    Returns (noff int64[D+1], eoff int64[D+1], ea int32[M], eb int32[M])."""
    noff = _to_numpy(ptr, np.int64).reshape(-1)
    ei = _to_numpy(edge_index, np.int64)
    if noff.size < 1:
        raise ValueError("ptr must have D + 1 >= 1 entries")
    if ei.size == 0:
        ei = ei.reshape(2, 0)
    if ei.ndim != 2 or ei.shape[0] != 2:
        raise ValueError("edge_index must have shape [2, E], got %s" % (ei.shape,))
    a, b = ei[0], ei[1]
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    span = int(max(int(noff[-1]), int(hi.max(initial=0)) + 1, 1))
    _, first = np.unique((lo - int(lo.min(initial=0))) * span + hi, return_index=True)
    keep = np.sort(first)
    a, b = a[keep], b[keep]
    D = noff.size - 1
    g = np.clip(np.searchsorted(noff, a, side="right") - 1, 0, max(D - 1, 0))
    order = np.argsort(g, kind="stable")
    a, b, g = a[order], b[order], g[order]
    eoff = np.zeros(D + 1, np.int64)
    if D > 0:
        np.cumsum(np.bincount(g, minlength=D)[:D], out=eoff[1:])
    elif a.size:
        raise ValueError("edges given for a batch of no graphs")
    return noff, eoff, a.astype(np.int32), b.astype(np.int32)


_GraphDiagramsFn = None


def _graph_diagrams_fn():
    """the torch.autograd.Function over tlc_graph_batch_diagrams_dev / tlc_graph_batch_grad_dev (built on first use)"""
    global _GraphDiagramsFn
    if _GraphDiagramsFn is not None:
        return _GraphDiagramsFn
    import torch
    from torch.autograd.function import once_differentiable

    def stream(dev):
        return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    class GraphDiagrams(torch.autograd.Function):
        @staticmethod
        def forward(ctx, f, batch, flags):
            dev = f.device
            P = batch.pair_bound
            poff = torch.empty(batch.D + 1, dtype=torch.int64, device=dev)
            kind = torch.zeros(P, dtype=torch.uint8, device=dev)
            bv = torch.zeros(P, dtype=torch.int32, device=dev)
            dv = torch.zeros(P, dtype=torch.int32, device=dev)
            birth = torch.zeros(P, dtype=torch.float64, device=dev)
            death = torch.zeros(P, dtype=torch.float64, device=dev)
            status = torch.empty(batch.D, dtype=torch.uint8, device=dev)
            d = L.Diagrams(P, poff.data_ptr(), None, kind.data_ptr(), bv.data_ptr(), dv.data_ptr(), birth.data_ptr(),
                           death.data_ptr())
            L.check(L.lib().tlc_graph_batch_diagrams_dev(batch._h, f.data_ptr(), flags, C.byref(d),
                                                         status.data_ptr() if batch.D else None, stream(dev)))
            ctx.save_for_backward(poff, bv, dv)
            ctx.batch = batch
            ctx.set_materialize_grads(False)  # an unused birth / death gradient reaches the library as NULL
            ctx.mark_non_differentiable(poff, kind, bv, dv, status)
            return poff, kind, bv, dv, birth, death, status

        @staticmethod
        @once_differentiable
        def backward(ctx, _gp, _gk, _gbv, _gdv, grad_birth, grad_death, _gs):
            poff, bv, dv = ctx.saved_tensors
            batch = ctx.batch
            dev = bv.device
            gb = grad_birth.contiguous() if grad_birth is not None else None
            gd = grad_death.contiguous() if grad_death is not None else None
            for g, what in ((gb, "grad_birth"), (gd, "grad_death")):
                _dev_ptr(g, "float64", (batch.pair_bound,), dev.index, what)
            grad_f = torch.empty(batch.N, dtype=torch.float64, device=dev)
            d = L.Diagrams(batch.pair_bound, poff.data_ptr(), None, None, bv.data_ptr(), dv.data_ptr(), None, None)
            L.check(L.lib().tlc_graph_batch_grad_dev(batch._h, C.byref(d), gb.data_ptr() if gb is not None else None,
                                                     gd.data_ptr() if gd is not None else None, grad_f.data_ptr(),
                                                     stream(dev)))
            return grad_f, None, None

    _GraphDiagramsFn = GraphDiagrams
    return _GraphDiagramsFn


class GraphBatch:
    """A batch of graphs resident on one GPU, for persistence diagrams under a filtration that changes from call to
    call (a learnable filtration, or whole-graph persistence over a dataloader batch).  ptr int[D+1] and edge_index
    int[2, E] are PyG's Batch.ptr / edge_index (numpy or CPU tensors); edge_index may list both directions of an edge
    (see normalize_edge_index).  The structure is checked and uploaded once."""

    def __init__(self, ptr, edge_index, device=0):
        self.noff, self.eoff, self.ea, self.eb = normalize_edge_index(ptr, edge_index)
        self.D = int(self.noff.size - 1)
        self.N = int(self.noff[-1])
        self.M = int(self.eoff[-1])
        self.device = int(device)
        self._h = C.c_void_p()
        L.check(L.lib().tlc_graph_batch_create(self.device, self.D, self.noff.ctypes.data, self.eoff.ctypes.data,
                                               self.ea.ctypes.data, self.eb.ctypes.data, C.byref(self._h)))
        bound = C.c_int64(0)
        L.check(L.lib().tlc_graph_batch_pair_bound(self._h, C.byref(bound)))
        self.pair_bound = int(bound.value)

    @classmethod
    def from_device(cls, ptr, edge_index, device=0):
        """the same batch from structure already on the GPU: ptr int64[D+1] and edge_index int32 (or int64) [2, M], CUDA
        tensors on `device`, in CANONICAL FORM -- inside every graph edge_index[0] < edge_index[1] and the edges strictly
        ascending in (edge_index[0], edge_index[1]), graphs one after the other.  VicinityGraph.vicinity_batch_dev's ptr /
        edge_index are in this form.  A PyG batch (N = ptr[-1] vertices, graphs on consecutive vertex ranges) is
        canonicalised on the device with
            lo, hi = torch.minimum(edge_index[0], edge_index[1]), torch.maximum(edge_index[0], edge_index[1])
            key = torch.unique(lo * N + hi)              # sorted; drops repeats and the reverse directions
            edge_index = torch.stack([key // N, key % N]).to(torch.int32)
        (self-loops stay, and are rejected).  That order, not the input order, is then the sweeps' tie-break, whereas
        GraphBatch(ptr, edge_index) keeps the first occurrence of every edge in input order.  Input that is not in
        canonical form raises TlcError with the library's message naming the graph and the first offending edge.  The
        structure is checked on the device (O(M), no sort); the call synchronises with the current stream."""
        import torch
        device = int(device)
        if getattr(ptr, "dim", lambda: 0)() != 1 or ptr.shape[0] < 1:
            raise ValueError("ptr must be 1-D with D + 1 >= 1 entries")
        if getattr(edge_index, "dim", lambda: 0)() != 2 or edge_index.shape[0] != 2:
            raise ValueError("edge_index must have shape [2, M], got %s" % (tuple(getattr(edge_index, "shape", ())),))
        D, M = int(ptr.shape[0]) - 1, int(edge_index.shape[1])
        _dev_ptr(ptr, "int64", (D + 1,), device, "ptr")
        if edge_index.dtype == torch.int64:
            if M and bool(((edge_index < 0) | (edge_index >= 2 ** 31)).any()):
                raise ValueError("edge_index holds ids outside [0, 2^31)")
            edge_index = edge_index.to(torch.int32)
        _dev_ptr(edge_index.contiguous(), "int32", (2, M), device, "edge_index")
        ea, eb = edge_index[0].contiguous(), edge_index[1].contiguous()
        # graph t's edges start at the first edge whose ea reaches ptr[t] (ea is ascending in canonical form; the library
        # rejects edges that end up outside their graph or out of order otherwise)
        eoff = torch.searchsorted(ea.to(torch.int64), ptr).contiguous()
        if D >= 0:
            eoff[0] = 0
            eoff[D] = M
        self = cls.__new__(cls)
        self.noff, self.eoff, self.ea, self.eb = ptr, eoff, ea, eb
        self.D, self.device = D, device
        self._h = C.c_void_p()
        st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        L.check(L.lib().tlc_graph_batch_create_dev(device, D, ptr.data_ptr(), eoff.data_ptr(),
                                                   ea.data_ptr() if M else None, eb.data_ptr() if M else None, st,
                                                   C.byref(self._h)))
        self.N = int(ptr[-1].item())
        self.M = M
        bound = C.c_int64(0)
        L.check(L.lib().tlc_graph_batch_pair_bound(self._h, C.byref(bound)))
        self.pair_bound = int(bound.value)
        return self

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            L.lib().tlc_graph_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def diagrams(self, f, extended=False, keep_zero=False, asc_only=False, no_small=False):
        """persistence diagrams of every graph under the filtration f (float64 CUDA tensor [N] on the batch's device;
        may require grad).  Returns a dict of CUDA tensors: poff int64[D+1] (graph t's pairs are [poff[t], poff[t+1]),
        poff[D] the live length), kind uint8, bv / dv int32 (batch vertex ids), birth / death float64 -- all sized to
        the pair bound N + M + D, so that nothing waits for the device -- and status uint8[D].  birth and death are
        differentiable in f: the gradient of a pair value flows to the vertex that carries it.  Graph t's pairs are the
        pipeline's for a node-mode vicinity equal to that graph (Union_find + Accelerate_PD, accelerated_PD.py:26,115):
        PD_up, [min,max], PD_down, [max,min], then PD_one with extended; no pairs for a disconnected graph or one with a
        non-finite value (status ST_NONFINITE).  f is not normalised.  no_small: every graph through the staged kernels
        (same results).  Runs on the current stream.  The dict plugs into persistence_images(d["poff"], d["birth"],
        d["death"], d["kind"], mask) and wasserstein_distances."""
        if extended and asc_only:
            raise ValueError("asc_only excludes extended (the loops need the descending sweep)")
        _dev_ptr(f, "float64", (self.N,), self.device, "f")
        flags = ((L.F_EXTENDED if extended else 0) | (L.F_KEEP_ZERO if keep_zero else 0)
                 | (L.F_ASC_ONLY if asc_only else 0) | (L.F_NO_SMALL if no_small else 0))
        poff, kind, bv, dv, birth, death, status = _graph_diagrams_fn().apply(f, self, flags)
        return dict(poff=poff, kind=kind, bv=bv, dv=dv, birth=birth, death=death, status=status)


def launch_count():
    return int(L.lib().tlc_launch_count())


def ollivier_ricci(rowptr, col, alpha=0.5, device=0, return_iters=False):
    """Ollivier-Ricci curvature (Sinkhorn transport) of every directed CSR entry of an unweighted graph: what
    loaddatas.compute_ricci_curvature (OllivierRicci(alpha=0.5, method="Sinkhorn")) computes before the path."""
    rp = np.ascontiguousarray(rowptr, dtype=np.int32)
    cl = np.ascontiguousarray(col, dtype=np.int32)
    out = np.zeros(cl.size, dtype=np.float64)
    it = np.zeros(cl.size, dtype=np.int32)
    L.check(L.lib().tlc_ollivier_ricci(int(device), int(rp.size - 1), int(cl.size), rp.ctypes.data, cl.ctypes.data, float(alpha),
                                       out.ctypes.data, it.ctypes.data))
    return (out, it) if return_iters else out
