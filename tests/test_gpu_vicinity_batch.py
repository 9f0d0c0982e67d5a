"""Vicinities in graph-batch layout on the GPU (VicinityGraph.vicinity_batch_dev, tlc_vicinity_batch_dev, kernel 10) and
graph batches created from device-resident structure (GraphBatch.from_device, tlc_graph_batch_create_dev): vertices,
edges and filtration values bit-exact against the unmodified reference's PDGNN tuples and against tlc_vicinity_detail;
statuses against tlc_vicinity_pi_dev; chunking; the capacity protocol; the whole device chain against the pipeline's own
diagrams and against the host route; rejections of input that is not in canonical form; reproducibility and streams."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import GRAPH_CASES, KD_CASES, KD_LP_CASES, kd_expected, load_case, load_kd_case
from test_gpu_graph_batch import connected_edges, make_batch, run, same_pairs, segment
from tlc_b200 import _lib as L
from tlc_b200 import api
from tlc_b200 import graphgen as gg

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def host(vb):
    return {k: (v.cpu().numpy() if v is not None else None) for k, v in vb.items()}


def bits(a):
    return np.asarray(a, np.float64).view(np.int64)


def random_graph(seed, N=600, deg=4):
    rng = np.random.default_rng(seed)
    e = rng.integers(0, N, (N * deg, 2))
    e = e[e[:, 0] != e[:, 1]]
    e = np.unique(np.stack([e.min(1), e.max(1)], 1), axis=0)
    kappa = np.round(rng.uniform(-0.9, 0.9, len(e)) * 64) / 64  # dyadic curvatures: ties in the path sums
    rp, col, kap = gg.build_csr(N + 5, e, kappa)  # five isolated nodes at the end
    return (rp, col, kap), rng


def targets_with_specials(rng, csr, E):
    rp, col, _ = csr
    N = len(rp) - 1
    src = np.repeat(np.arange(N), np.diff(rp))
    pick = rng.choice(len(col), E, replace=False)
    tg = np.stack([src[pick], col[pick]], 1).astype(np.int32)
    tg[3] = [-1, 5]          # a label unknown to dict_node
    tg[7] = [N - 1, 2]       # an isolated node
    tg[11] = [4, 4]          # u == v
    tg[13] = rng.integers(0, N - 5, 2)  # a non-adjacent pair
    return tg


def check_against_pipeline(g, tg, hop, mode, desc, flags):
    vb = host(g.vicinity_batch_dev(torch.from_numpy(tg).to(DEV), hop=hop, mode=mode, descriptor=desc, flags=flags))
    n, m, _ = g.vicinity_sizes(tg, hop, mode)
    assert np.array_equal(np.diff(vb["ptr"]), n) and np.array_equal(np.diff(vb["eptr"]), m)
    det = g.vicinity_detail(tg, hop=hop, mode=mode, descriptor=desc, flags=flags)
    st = torch.zeros(len(tg), dtype=torch.uint8, device=DEV)
    g.vicinity_pi_dev(torch.from_numpy(tg).to(DEV), torch.zeros((len(tg), 25), dtype=torch.float64, device=DEV),
                      out_status=st, hop=hop, mode=mode, descriptor=desc, flags=flags)
    torch.cuda.synchronize()
    st = st.cpu().numpy()
    assert np.array_equal(vb["status"], st), (vb["status"], st)
    V, M = int(n.sum()), int(m.sum())
    if desc == "bogus":  # (tlc_vicinity_detail stops after the counting pass: every target reports BAD_DESCRIPTOR)
        assert np.all(np.isnan(vb["fval"]))
        return vb, st
    assert np.array_equal(vb["vert"], det["vert"][:V])
    first = np.repeat(vb["ptr"][:-1], m)
    assert np.array_equal(vb["edge_index"][0] - first, det["elo"][:M])
    assert np.array_equal(vb["edge_index"][1] - first, det["ehi"][:M])
    live = np.repeat(st <= L.ST_TRIVIAL, n)
    assert np.array_equal(bits(vb["fval"][live]), bits(det["fval"][:V][live]))
    assert np.all(np.isnan(vb["fval"][~live]))
    return vb, st


@pytest.mark.parametrize("tag", KD_CASES + KD_LP_CASES)
def test_against_the_unmodified_reference(tag):
    c = load_kd_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    lp = tag in KD_LP_CASES
    tg = c["new_nodes"].astype(np.int32) if lp else np.repeat(c["new_nodes"].reshape(-1, 1), 2, 1).astype(np.int32)
    filt = {"ricci": 0, "degree": L.F_FILT_DEGREE, "centrality": L.F_FILT_CENTRALITY, "clustering": L.F_FILT_CLUSTERING}
    flags = L.F_NORM | L.F_NORM_EPS | filt[c["filt_name"]]
    vb = host(g.vicinity_batch_dev(torch.from_numpy(np.ascontiguousarray(tg)).to(DEV), hop=c["hop"],
                                   mode=L.MODE_EDGE_FORCED if lp else L.MODE_NODE, flags=flags))
    ok, live = 0, 0
    for k in range(len(tg)):
        e = kd_expected(c, k)
        live += not e["none"]
        if e["none"]:
            assert vb["status"][k] != L.ST_OK
            continue
        if lp and (int(c["kind"][k]) == 2 or vb["status"][k] == L.ST_DISCONNECTED):
            continue  # (a disconnected LP vicinity is outside the reference's contract: the reference has no check)
        a, b = int(vb["ptr"][k]), int(vb["ptr"][k + 1])
        vert = vb["vert"][a:b]
        assert np.array_equal(vert, e["vert"])
        assert np.array_equal(bits(vb["fval"][a:b]), bits(e["filt"]))
        ea, eb = (vb["edge_index"][:, int(vb["eptr"][k]):int(vb["eptr"][k + 1])] - a)
        assert np.array_equal(np.stack([vert[ea], vert[eb]], 1).reshape(-1, 2), e["edges"].reshape(-1, 2))
        ok += 1
    assert ok >= min(10, live)
    g.close()


@pytest.mark.parametrize("tag", GRAPH_CASES)
def test_against_the_pipeline_golden(tag):
    c = load_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    vb, st = check_against_pipeline(g, c["new_targets"], c["hop"], L.MODE_EDGE, c["descriptor"], L.F_NORM)
    assert np.any(st == L.ST_OK)
    g.close()


COVER = [(L.MODE_EDGE, 2, "sum", L.F_NORM), (L.MODE_EDGE, 1, "min", L.F_NORM | L.F_SUM_PLAIN),
         (L.MODE_EDGE, 0, "max", L.F_NORM), (L.MODE_EDGE, 2, "max", 0), (L.MODE_EDGE, 2, "bogus", L.F_NORM),
         (L.MODE_NODE, 2, "sum", L.F_NORM | L.F_NORM_EPS), (L.MODE_NODE, 1, "sum", L.F_NORM),
         (L.MODE_NODE, 0, "sum", L.F_NORM),
         (L.MODE_EDGE_FORCED, 2, "sum", L.F_NORM | L.F_NORM_EPS), (L.MODE_EDGE_FORCED, 1, "min", L.F_NORM),
         (L.MODE_EDGE_UNION, 1, "sum", L.F_NORM), (L.MODE_EDGE_UNION, 2, "min", L.F_NORM | L.F_SUM_PLAIN),
         (L.MODE_EDGE_REMOVEINTER, 1, "sum", L.F_NORM), (L.MODE_EDGE_REMOVEINTER, 2, "max", L.F_NORM),
         (L.MODE_NODE, 2, "sum", L.F_NORM | L.F_NORM_EPS | L.F_FILT_DEGREE),
         (L.MODE_NODE, 1, "sum", L.F_NORM | L.F_NORM_EPS | L.F_FILT_CENTRALITY),
         (L.MODE_NODE, 2, "sum", L.F_NORM | L.F_NORM_EPS | L.F_FILT_CLUSTERING),
         (L.MODE_NODE, 1, "sum", L.F_NORM | L.F_NORM_EPS | L.F_FILT_HKS),
         (L.MODE_EDGE_FORCED, 2, "sum", L.F_NORM | L.F_NORM_EPS | L.F_FILT_HKS),
         (L.MODE_EDGE, 2, "sum", L.F_FILT_DEGREE)]


@pytest.mark.parametrize("mode, hop, desc, flags", COVER)
def test_against_the_pipeline_random(mode, hop, desc, flags):
    csr, rng = random_graph(hop * 31 + mode * 7 + flags % 97)
    tg = targets_with_specials(rng, csr, 200)
    g = api.VicinityGraph(*csr, device=0)
    vb, st = check_against_pipeline(g, tg, hop, mode, desc, flags)
    assert st[3] == L.ST_UNKNOWN_NODE and st[7] == L.ST_UNKNOWN_NODE
    if desc == "bogus":
        assert np.all(np.isin(st, [L.ST_BAD_DESCRIPTOR, L.ST_EMPTY, L.ST_UNKNOWN_NODE]))
    g.close()


def test_chunking_gives_the_same_bytes():
    c = load_case("computers_s_hop2")
    tg = torch.from_numpy(c["new_targets"]).to(DEV)
    one = api.VicinityGraph(*c["csr"], device=0)
    a = host(one.vicinity_batch_dev(tg, hop=2))
    assert one.last_counts()["chunks"] == 1
    split = 0
    for mb in (64, 32, 16, 8, 4, 2, 1):  # the largest arena that splits the call, while one vicinity still fits
        small = api.VicinityGraph(*c["csr"], device=0, arena_bytes=mb << 20)
        try:
            b = host(small.vicinity_batch_dev(tg, hop=2))
        except L.TlcError:
            small.close()
            break
        split = small.last_counts()["chunks"]
        small.close()
        if split > 1:
            for k in a:
                assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), k
            break
    assert split > 1
    one.close()


def test_capacity_protocol():
    c = load_case("pubmed_s_hop2_cont")
    g = api.VicinityGraph(*c["csr"], device=0)
    tgh = c["new_targets"]
    E = len(tgh)
    tg = torch.from_numpy(tgh).to(DEV)
    n, m, sst = g.vicinity_sizes(tgh, 2, L.MODE_EDGE)
    V, M = int(n.sum()), int(m.sum())
    voff = torch.full((E + 1,), -7, dtype=torch.int64, device=DEV)
    eoff = torch.full((E + 1,), -7, dtype=torch.int64, device=DEV)
    st = torch.full((E,), 99, dtype=torch.uint8, device=DEV)
    vert = torch.full((V,), -3, dtype=torch.int32, device=DEV)
    ei = torch.full((2, M), -3, dtype=torch.int32, device=DEV)
    fv = torch.full((V,), 1.5, dtype=torch.float64, device=DEV)
    torch.cuda.synchronize()
    p = api.make_params(2, L.MODE_EDGE, "sum", 5, L.F_NORM, 0)
    for cap_v, cap_e in ((0, 0), (V, M - 1), (V - 1, M)):
        b = L.VicinityBatch(cap_v, cap_e, voff.data_ptr(), eoff.data_ptr(), vert.data_ptr(), ei[0].data_ptr(),
                            ei[1].data_ptr(), fv.data_ptr())
        tv, te = C.c_int64(0), C.c_int64(0)
        rc = L.lib().tlc_vicinity_batch_dev(g._h, tg.data_ptr(), E, C.byref(p), C.byref(b), st.data_ptr(), C.byref(tv),
                                            C.byref(te))
        assert rc == L.E_CAPACITY and (tv.value, te.value) == (V, M)
        assert np.array_equal(voff.cpu().numpy(), np.concatenate([[0], np.cumsum(n)]))
        assert np.array_equal(eoff.cpu().numpy(), np.concatenate([[0], np.cumsum(m)]))
        assert np.all(vert.cpu().numpy() == -3) and np.all(ei.cpu().numpy() == -3) and np.all(fv.cpu().numpy() == 1.5)
        assert not np.any(st.cpu().numpy() == 99)
    b = L.VicinityBatch(V, M, voff.data_ptr(), eoff.data_ptr(), vert.data_ptr(), ei[0].data_ptr(), ei[1].data_ptr(),
                        fv.data_ptr())
    L.check(L.lib().tlc_vicinity_batch_dev(g._h, tg.data_ptr(), E, C.byref(p), C.byref(b), st.data_ptr(), None, None))
    full = host(g.vicinity_batch_dev(tg, hop=2))
    assert np.array_equal(vert.cpu().numpy(), full["vert"]) and np.array_equal(ei.cpu().numpy(), full["edge_index"])
    assert np.array_equal(bits(fv.cpu().numpy()), bits(full["fval"]))
    nof = host(g.vicinity_batch_dev(tg, hop=2, fval=False))
    assert nof["fval"] is None
    for k in ("ptr", "eptr", "vert", "edge_index"):
        assert np.array_equal(nof[k], full[k]), k
    g.close()


@pytest.mark.parametrize("node", [False, True])
def test_chain_equals_the_pipeline(node):
    c = load_case("pubmed_s_hop2_cont" if not node else "cora_q_hop2")
    g = api.VicinityGraph(*c["csr"], device=0)
    tgh = c["new_targets"] if not node else np.repeat(c["new_targets"][:, :1], 2, 1)
    tg = torch.from_numpy(np.ascontiguousarray(tgh)).to(DEV)
    mode = L.MODE_NODE if node else L.MODE_EDGE
    flags = L.F_NORM | (L.F_NORM_EPS if node else 0)
    vb = g.vicinity_batch_dev(tg, hop=2, mode=mode, flags=flags)
    h = host(vb)
    gb = api.GraphBatch.from_device(vb["ptr"], vb["edge_index"])
    for ext in (False, True):
        for kz in (False, True):
            fl = flags | (L.F_EXTENDED if ext else 0) | (L.F_KEEP_ZERO if kz else 0)
            ref = g.vicinity_diagrams_dev(tg, hop=2, mode=mode, flags=fl)
            ref = {k: (v.cpu().numpy() if v is not None else None) for k, v in ref.items()}
            for ns in (False, True):
                d = run(gb, h["fval"], extended=ext, keep_zero=kz, no_small=ns)
                for t in range(len(tgh)):
                    a, b = int(h["ptr"][t]), int(h["ptr"][t + 1])
                    if h["status"][t] == L.ST_OK:
                        s = segment(d, t)
                        s["bv"] = h["vert"][s["bv"]]
                        s["dv"] = h["vert"][s["dv"]]
                        r0, r1 = int(ref["poff"][t]), int(ref["poff"][t + 1])
                        same_pairs(s, ref["kind"][r0:r1], ref["bv"][r0:r1], ref["dv"][r0:r1], ref["birth"][r0:r1],
                                   ref["death"][r0:r1], where=(t, ext, kz, ns))
                    elif b > a and h["status"][t] != L.ST_TRIVIAL:
                        assert d["status"][t] == L.ST_NONFINITE, t
    gb.close()
    g.close()


def canonical_batch(seed, D=40):
    rng = np.random.default_rng(seed)
    graphs = []
    for _ in range(D):
        n = int(rng.integers(1, 300))
        m = int(rng.integers(n - 1, min(3 * n, n * (n - 1) // 2) + 1)) if n > 1 else 0
        graphs.append((n, connected_edges(rng, n, m)))
    ptr, ei = make_batch(graphs)
    return ptr, ei, rng


def test_against_the_host_route():
    ptr, ei, rng = canonical_batch(3)
    f = rng.random(int(ptr[-1]))
    host_gb = api.GraphBatch(ptr, ei)
    dev_gb = api.GraphBatch.from_device(torch.from_numpy(ptr).to(DEV), torch.from_numpy(ei).to(DEV))
    assert (dev_gb.D, dev_gb.N, dev_gb.M, dev_gb.pair_bound) == (host_gb.D, host_gb.N, host_gb.M, host_gb.pair_bound)
    grads = []
    for gb in (host_gb, dev_gb):
        for kw in (dict(), dict(extended=True), dict(extended=True, keep_zero=True, no_small=True)):
            ft = torch.from_numpy(f).to(DEV).requires_grad_(True)
            d = gb.diagrams(ft, **kw)
            (d["birth"] * 1.5 + d["death"] * d["death"]).sum().backward()
            grads.append((host({k: v.detach() for k, v in d.items()}), ft.grad.cpu().numpy()))
    for (da, ga), (db, gbd) in zip(grads[:3], grads[3:]):
        for k in da:
            assert np.array_equal(da[k].view(np.uint8), db[k].view(np.uint8)), k
        assert np.array_equal(bits(ga), bits(gbd))
    # gradcheck through from_device on a small batch
    sp, se, srng = canonical_batch(4, D=4)
    sgb = api.GraphBatch.from_device(torch.from_numpy(sp).to(DEV), torch.from_numpy(se).to(DEV).to(torch.int32))
    x = torch.from_numpy(srng.random(int(sp[-1]))).to(DEV).requires_grad_(True)
    assert torch.autograd.gradcheck(lambda v: sgb.diagrams(v, extended=True)["death"] - sgb.diagrams(v, extended=True)["birth"],
                                    (x,), eps=1e-7, atol=1e-6)
    host_gb.close()
    dev_gb.close()
    sgb.close()


def test_full_step_equals_the_host_route():
    c = load_case("cora_q_hop2")
    g = api.VicinityGraph(*c["csr"], device=0)
    tgh = c["new_targets"]
    vb = g.vicinity_batch_dev(torch.from_numpy(tgh).to(DEV), hop=2)
    st = vb["status"].cpu().numpy()
    # the same step built from tlc_vicinity_detail, per-target assembly and the host GraphBatch
    det = g.vicinity_detail(tgh, hop=2)
    graphs, fs = [], []
    for i in range(len(tgh)):
        a = g.per_target(det, i)
        graphs.append((a["n"], np.stack([a["elo"], a["ehi"]], 1).astype(np.int64)))
        fs.append(a["fval"] if st[i] <= L.ST_TRIVIAL else np.full(a["n"], np.nan))
    ptr, ei = make_batch(graphs)
    out = []
    for gb, f0 in ((api.GraphBatch.from_device(vb["ptr"], vb["edge_index"]), vb["fval"]),
                   (api.GraphBatch(ptr, ei), torch.from_numpy(np.concatenate(fs)).to(DEV))):
        f = f0.clone().requires_grad_(True)
        d = gb.diagrams(f)
        img = api.persistence_images(d["poff"], d["birth"], d["death"])
        img.sum().backward()
        out.append((img.detach().cpu().numpy(), f.grad.cpu().numpy()))
        gb.close()
    assert np.array_equal(bits(out[0][0]), bits(out[1][0]))
    assert np.array_equal(bits(np.nan_to_num(out[0][1])), bits(np.nan_to_num(out[1][1])))
    g.close()


GOOD = dict(noff=[0, 3, 6, 6, 8], ea=[0, 0, 1, 3, 4, 6], eb=[1, 2, 2, 4, 5, 7])


@pytest.mark.parametrize("change, words", [
    (dict(ea=[0, 0, 2, 3, 4, 6], eb=[1, 2, 1, 4, 5, 7]), ["edge 2 (2, 1)", "graph 0", "ea > eb"]),
    (dict(ea=[0, 1, 0, 3, 4, 6], eb=[1, 2, 2, 4, 5, 7]), ["edge 2 (0, 2)", "graph 0", "not after edge 1"]),
    (dict(ea=[0, 0, 0, 3, 4, 6], eb=[1, 2, 2, 4, 5, 7]), ["edge 2 (0, 2)", "graph 0", "repeats edge 1"]),
    (dict(ea=[0, 0, 1, 3, 5, 6], eb=[1, 2, 2, 4, 5, 7]), ["edge 4 (5, 5)", "graph 1", "self-loop"]),
    (dict(ea=[0, 0, 1, 3, 4, 6], eb=[1, 2, 3, 4, 5, 7]), ["edge 2 (1, 3)", "graph 0", "outside"]),
    (dict(ea=[0, 0, 1, 3, 4, 6], eb=[1, 2, 2, 4, 5, 9]), ["edge 5 (6, 9)", "graph 3", "outside"]),
    (dict(noff=[0, 3, 2, 6, 8]), ["noff is not monotone at graph 1"]),
    (dict(noff=[1, 3, 6, 6, 8]), ["noff[0] and eoff[0] must be 0"]),
])
def test_create_dev_rejections(change, words):
    a = dict(GOOD)
    a.update(change)
    noff = torch.tensor(a["noff"], dtype=torch.int64, device=DEV)
    eoff = torch.tensor([0, 3, 5, 5, 6], dtype=torch.int64, device=DEV)
    ea = torch.tensor(a["ea"], dtype=torch.int32, device=DEV)
    eb = torch.tensor(a["eb"], dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    h = C.c_void_p()
    rc = L.lib().tlc_graph_batch_create_dev(0, 4, noff.data_ptr(), eoff.data_ptr(), ea.data_ptr(), eb.data_ptr(), None,
                                            C.byref(h))
    msg = L.lib().tlc_last_error().decode()
    assert rc == L.E_INVALID, msg
    for w in words:
        assert w in msg, (w, msg)
    with pytest.raises(L.TlcError):  # the Python wrapper raises with the library's message
        api.GraphBatch.from_device(noff, torch.stack([ea, eb]))


def test_create_dev_accepts_empty():
    gb = api.GraphBatch.from_device(torch.zeros(1, dtype=torch.int64, device=DEV), torch.zeros((2, 0), dtype=torch.int32, device=DEV))
    assert (gb.D, gb.N, gb.M) == (0, 0, 0)
    gb.close()
    ptr = torch.tensor([0, 1, 4, 4, 6], dtype=torch.int64, device=DEV)  # graphs without edges, one empty graph
    gb = api.GraphBatch.from_device(ptr, torch.zeros((2, 0), dtype=torch.int32, device=DEV))
    d = run(gb, np.arange(6, dtype=np.float64))
    assert d["status"][1] == L.ST_DISCONNECTED and d["status"][2] == L.ST_EMPTY and d["status"][3] == L.ST_DISCONNECTED
    gb.close()


def test_reproducible_and_side_stream():
    c = load_case("computers_s_hop2")
    g = api.VicinityGraph(*c["csr"], device=0)
    tg = torch.from_numpy(c["new_targets"]).to(DEV)
    a = host(g.vicinity_batch_dev(tg, hop=2, mode=L.MODE_NODE, flags=L.F_NORM | L.F_NORM_EPS | L.F_FILT_HKS))
    b = host(g.vicinity_batch_dev(tg, hop=2, mode=L.MODE_NODE, flags=L.F_NORM | L.F_NORM_EPS | L.F_FILT_HKS))
    s = torch.cuda.Stream(DEV)
    with torch.cuda.stream(s):
        g.set_stream(s.cuda_stream)
        tg2 = tg.clone()
        x = host(g.vicinity_batch_dev(tg2, hop=2, mode=L.MODE_NODE, flags=L.F_NORM | L.F_NORM_EPS | L.F_FILT_HKS))
        g.set_stream(None)
    for k in a:
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), k
        assert np.array_equal(a[k].view(np.uint8), x[k].view(np.uint8)), k
    g.close()
