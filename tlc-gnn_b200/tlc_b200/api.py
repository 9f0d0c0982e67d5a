"""Host-side API over the C-ABI: device-resident graph handle + batched calls.

`VicinityGraph` is what sg2dgm.riccidist2dgm.graph2pi (the drop-in mirror) holds: the CSR graph and
curvature uploaded once (graph2pi.__init__, riccidist2dgm.py:216-226), then one C-ABI call per batch
of targets (get_pimg_for_all_edges, :362-370).
"""
import ctypes as C

import numpy as np

from . import _lib as L


_CUDA_STREAM_LEGACY = 0x1  # cudaStreamLegacy (driver_types.h): an explicit handle of the legacy default stream


def _dev_ptr(t, dtype_name, shape, device_index, what):
    """data pointer of a torch CUDA tensor that crosses the C-ABI: dtype, shape, contiguity and device are checked here,
    because the library can only see a raw address."""
    if t is None:
        return None
    if str(t.dtype) != "torch." + dtype_name:
        raise TypeError("%s must be %s, got %s" % (what, dtype_name, t.dtype))
    if tuple(t.shape) != tuple(shape):
        raise ValueError("%s must have shape %s, got %s" % (what, tuple(shape), tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % what)
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
                    graph_row_route=int(L.lib().tlc_last_direct(self._h)), table_route=int(L.lib().tlc_last_table(self._h)))

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
