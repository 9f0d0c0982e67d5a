"""Persistence diagrams of caller-supplied graph batches on the GPU (api.GraphBatch, tlc_graph_batch_*, kernel 9):
pairs bit-exact against the oracle and against tlc_union_find for arbitrary edge orders, on the fused route of every
size class and on the staged route; equality with the pipeline's own vicinities; statuses; compact output;
reproducibility; and the gradient against the numpy scatter, gradcheck and a whole f -> diagrams -> images / Wasserstein
chain."""
import numpy as np
import pytest
import torch

import oracle as orc
from helpers import load_case
from test_graph_batch_abi import scatter_grad
from test_pimg_batch_abi import torch_images
from test_wasserstein_abi import torch_wasserstein
from tlc_b200 import _lib as L
from tlc_b200 import api
from tlc_b200 import graphgen as gg

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)

# (n, m) across the fused classes' edges (warp: n <= 64 / m <= 256, 128 threads: <= 256 / <= 2048, 256 threads:
# <= 1024 / <= 4096) and the staged route beyond them
SIZES = [(1, 0), (2, 1), (5, 6), (23, 25), (40, 75), (64, 256), (64, 257), (65, 80), (256, 2048), (257, 400),
         (600, 900), (1024, 4096), (1024, 4097), (1025, 1500), (3000, 4500)]


def connected_edges(rng, n, m):
    """a random connected graph on n vertices with m edges, canonical lexicographic order"""
    es = set()
    perm = rng.permutation(n)
    for i in range(1, n):
        a, b = int(perm[i]), int(perm[rng.integers(0, i)])
        es.add((min(a, b), max(a, b)))
    while len(es) < m:
        a, b = (int(x) for x in rng.integers(0, n, 2))
        if a != b:
            es.add((min(a, b), max(a, b)))
    return np.array(sorted(es), np.int64).reshape(-1, 2)


def values(rng, n, kind):
    if kind == "plateau":   # few distinct values: exact ties everywhere
        return rng.integers(0, 4, n).astype(np.float64) / 4
    if kind == "cluster":   # clusters 2.5e-7 apart: the perturbed keys (F4) cross the lexicographic order
        return rng.integers(0, 3, n) * 0.5 + rng.integers(0, 4, n) * 2.5e-7
    return rng.random(n)


def make_batch(graphs, shuffle=None):
    """graphs: list of local edge arrays [m, 2] with n -> (ptr, edge_index [2, M]) batch-global"""
    ptr = np.zeros(len(graphs) + 1, np.int64)
    ei = []
    for t, (n, e) in enumerate(graphs):
        ptr[t + 1] = ptr[t] + n
        ei.append(e + ptr[t])
    return ptr, np.concatenate(ei, 0).T if ei else np.zeros((2, 0), np.int64)


def host(d):
    out = {k: v.detach().cpu().numpy() for k, v in d.items()}
    P = int(out["poff"][-1])
    for k in ("kind", "bv", "dv", "birth", "death"):
        out[k] = out[k][:P]
    return out


def segment(h, t):
    a, b = int(h["poff"][t]), int(h["poff"][t + 1])
    return {k: h[k][a:b] for k in ("kind", "bv", "dv", "birth", "death")}


def same_pairs(got, kind, bv, dv, birth, death, where=""):
    assert np.array_equal(got["kind"], np.asarray(kind, np.uint8)), where
    assert np.array_equal(got["bv"], np.asarray(bv)), where
    assert np.array_equal(got["dv"], np.asarray(dv)), where
    assert np.array_equal(got["birth"].view(np.int64), np.asarray(birth, np.float64).view(np.int64)), where
    assert np.array_equal(got["death"].view(np.int64), np.asarray(death, np.float64).view(np.int64)), where


def run(gb, f, **kw):
    d = gb.diagrams(torch.from_numpy(f).to(DEV), **kw)
    torch.cuda.synchronize()
    return host(d)


FLAGSETS = {"none": {}, "keep_zero": dict(keep_zero=True), "ext_keep_zero": dict(extended=True, keep_zero=True),
            "ext": dict(extended=True), "asc_only": dict(asc_only=True)}


@pytest.mark.parametrize("vals", ["plateau", "cluster", "random"])
@pytest.mark.parametrize("flagset", list(FLAGSETS))
def test_against_the_oracle(flagset, vals):
    rng = np.random.default_rng(hash((flagset, vals)) % 2**32)
    graphs = [(n, connected_edges(rng, n, m)) for n, m in SIZES + [(5000, 7500)]]
    ptr, ei = make_batch(graphs)
    f = np.concatenate([values(rng, n, vals) for n, _ in graphs])
    gb = api.GraphBatch(ptr, ei, device=0)
    kw = FLAGSETS[flagset]
    # the oracle on the block-diagonal CSR, node mode from each graph's first vertex, hop >= n, fval overridden
    N = int(ptr[-1])
    csr = gg.build_csr(N, ei.T, np.zeros(ei.shape[1]))
    og = orc.OracleGraph(*csr)
    oflags = (orc.F_EXTENDED if kw.get("extended") else 0) | (orc.F_KEEP_ZERO if kw.get("keep_zero") else 0)
    hs = [run(gb, f, **kw), run(gb, f, no_small=True, **kw)]
    for t, (n, _) in enumerate(graphs):
        if n == 1:  # (an isolated vertex is no oracle target; test_statuses_and_compact_output covers it)
            continue
        v0 = int(ptr[t])
        o = og.run_one(v0, v0, hop=n, mode=orc.MODE_NODE, flags=oflags, fval=f[v0:v0 + n])
        k = len(o["pkind"])
        if kw.get("asc_only"):  # PD_up and [min,max]: the pairs up to the first essential one
            k = int(np.flatnonzero(o["pkind"] == L.K_ESS)[0]) + 1
        for h in hs:
            assert h["status"][t] == o["status"], (t, n)
            same_pairs(segment(h, t), o["pkind"][:k], o["vert"][o["pbv"][:k]], o["vert"][o["pdv"][:k]],
                       o["pbirth"][:k], o["pdeath"][:k], where=(t, n))
    for h in hs:
        assert np.all(np.diff(h["poff"]) >= 0) and h["poff"][0] == 0 and h["poff"][-1] <= gb.pair_bound
    gb.close()


@pytest.mark.parametrize("flagset", ["none", "keep_zero", "ext"])
def test_arbitrary_edge_orders(flagset):
    rng = np.random.default_rng(7)
    graphs = []
    for n, m in SIZES[1:]:
        e = connected_edges(rng, n, m)[rng.permutation(m)]
        flip = rng.random(m) < 0.5
        e[flip] = e[flip][:, ::-1]
        graphs.append((n, e))
    ptr, ei = make_batch(graphs)
    f = np.concatenate([values(rng, n, "plateau" if t % 2 else "cluster") for t, (n, _) in enumerate(graphs)])
    gb = api.GraphBatch(ptr, ei, device=0)
    kw = FLAGSETS[flagset]
    fl = (L.F_EXTENDED if kw.get("extended") else 0) | (L.F_KEEP_ZERO if kw.get("keep_zero") else 0)
    hs = [run(gb, f, **kw), run(gb, f, no_small=True, **kw)]
    for t, (n, e) in enumerate(graphs):
        v0 = int(ptr[t])
        u = api.union_find(f[v0:v0 + n], e, flags=fl)
        for h in hs:
            assert h["status"][t] == u["status"]
            same_pairs(segment(h, t), u["pkind"], u["pbv"] + v0, u["pdv"] + v0, u["pbirth"], u["pdeath"], where=t)
    gb.close()


@pytest.mark.parametrize("ext", [False, True])
@pytest.mark.parametrize("tag", ["toy7_hop2", "cora_q_hop2", "pubmed_s_hop2_cont", "computers_s_hop1"])
def test_against_the_pipeline(tag, ext):
    c = load_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    flags = L.F_NORM | (L.F_EXTENDED if ext else 0)
    tg = c["new_targets"]
    det = g.vicinity_detail(tg, hop=c["hop"], descriptor=c["descriptor"], flags=flags)
    ref = g.vicinity_diagrams(tg, hop=c["hop"], descriptor=c["descriptor"], flags=flags)
    ok = [i for i in range(len(tg)) if det["status"][i] == L.ST_OK]
    assert ok
    graphs, fs, verts = [], [], []
    for i in ok:
        a = g.per_target(det, i)
        graphs.append((a["n"], np.stack([a["elo"], a["ehi"]], 1).astype(np.int64)))
        fs.append(a["fval"])
        verts.append(a["vert"])
    ptr, ei = make_batch(graphs)
    gb = api.GraphBatch(ptr, ei, device=0)
    f = np.concatenate(fs)
    for ns in (False, True):
        h = run(gb, f, extended=ext, no_small=ns)
        for t, i in enumerate(ok):
            assert h["status"][t] == L.ST_OK
            s = segment(h, t)
            a, b = int(ref["poff"][i]), int(ref["poff"][i + 1])
            v0 = int(ptr[t])
            s["bv"] = verts[t][s["bv"] - v0]
            s["dv"] = verts[t][s["dv"] - v0]
            same_pairs(s, ref["kind"][a:b], ref["bv"][a:b], ref["dv"][a:b], ref["birth"][a:b], ref["death"][a:b], where=i)
    gb.close()
    g.close()


def test_statuses_and_compact_output():
    # empty graph, single vertex, disconnected graph, NaN / inf values, and two ordinary graphs around them
    tri = np.array([[0, 1], [1, 2], [0, 2]])
    graphs = [(3, tri), (0, np.zeros((0, 2), np.int64)), (1, np.zeros((0, 2), np.int64)), (4, np.array([[0, 1], [2, 3]])),
              (3, tri), (3, tri), (2000, connected_edges(np.random.default_rng(1), 2000, 2100)), (3, tri)]
    ptr, ei = make_batch(graphs)
    f = np.random.default_rng(2).random(int(ptr[-1]))
    f[int(ptr[4]) + 1] = np.nan
    f[int(ptr[5])] = np.inf
    f[int(ptr[6]) + 1500] = -np.inf
    gb = api.GraphBatch(ptr, ei, device=0)
    assert gb.pair_bound == int(ptr[-1]) + ei.shape[1] + len(graphs)
    for ns in (False, True):
        h0 = run(gb, f, no_small=ns)
        h1 = run(gb, f, extended=True, no_small=ns)
        exp0 = [L.ST_OK, L.ST_EMPTY, L.ST_OK, L.ST_DISCONNECTED, L.ST_NONFINITE, L.ST_NONFINITE, L.ST_NONFINITE, L.ST_OK]
        exp1 = list(exp0)
        exp1[2] = L.ST_NO_TREE_EDGES
        assert h0["status"].tolist() == exp0 and h1["status"].tolist() == exp1
        for h in (h0, h1):
            cnt = np.diff(h["poff"])
            assert h["poff"][0] == 0 and h["poff"][-1] <= gb.pair_bound
            assert cnt[1] == 0 and cnt[3] == 0 and cnt[4] == cnt[5] == cnt[6] == 0
            v = int(ptr[2])  # the single vertex keeps [f, f] and [f, f] (its essential pairs)
            same_pairs(segment(h, 2), [L.K_ESS, L.K_ESS_REV], [v, v], [v, v], [f[v], f[v]], [f[v], f[v]])
            assert cnt[0] > 0 and cnt[7] > 0
    gb.close()


def test_capacity_and_flags_are_checked_before_any_work():
    ptr, ei = make_batch([(3, np.array([[0, 1], [1, 2]]))])
    gb = api.GraphBatch(ptr, ei, device=0)
    f = torch.rand(3, dtype=torch.float64, device=DEV)
    poff = torch.full((2,), -7, dtype=torch.int64, device=DEV)
    d = L.Diagrams(gb.pair_bound - 1, poff.data_ptr(), None, None, None, None, None, None)
    assert L.lib().tlc_graph_batch_diagrams_dev(gb._h, f.data_ptr(), 0, d, None, None) == L.E_CAPACITY
    d.cap = gb.pair_bound
    assert L.lib().tlc_graph_batch_diagrams_dev(gb._h, f.data_ptr(), L.F_NORM, d, None, None) == L.E_INVALID
    assert L.lib().tlc_graph_batch_diagrams_dev(gb._h, None, 0, d, None, None) == L.E_INVALID
    torch.cuda.synchronize()
    assert poff.tolist() == [-7, -7]
    with pytest.raises(TypeError):
        gb.diagrams(f.float())
    with pytest.raises(ValueError):
        gb.diagrams(f[:2])
    with pytest.raises(L.TlcError):
        api.GraphBatch([0, 3], [[0, 1], [1, 1]])
    gb.close()


def test_reproducible_and_independent_of_the_batch():
    rng = np.random.default_rng(3)
    graphs = [(n, connected_edges(rng, n, m)) for n, m in SIZES * 2]
    ptr, ei = make_batch(graphs)
    f = np.concatenate([values(rng, n, "cluster") for n, _ in graphs])
    gb = api.GraphBatch(ptr, ei, device=0)
    for kw in (dict(extended=True), dict(keep_zero=True, no_small=True)):
        a, b = run(gb, f, **kw), run(gb, f, **kw)
        for k in a:
            assert np.array_equal(a[k], b[k]), k
        h = len(graphs) // 3
        halves = [(0, h), (h, len(graphs))]
        for lo, hi in halves:
            p2, e2 = make_batch(graphs[lo:hi])
            g2 = api.GraphBatch(p2, e2, device=0)
            s = run(g2, f[int(ptr[lo]):int(ptr[hi])], **kw)
            for t in range(hi - lo):
                x, y = segment(a, lo + t), segment(s, t)
                y["bv"] = y["bv"] + int(ptr[lo]); y["dv"] = y["dv"] + int(ptr[lo])
                same_pairs(x, y["kind"], y["bv"], y["dv"], y["birth"], y["death"], where=t)
                assert a["status"][lo + t] == s["status"][t]
            g2.close()
    gb.close()


def tie_free_batch(rng, sizes):
    graphs = [(n, connected_edges(rng, n, m)) for n, m in sizes]
    ptr, ei = make_batch(graphs)
    N = int(ptr[-1])
    f = rng.permutation(N).astype(np.float64) * 1e-2 + 0.5  # values >= 1e-2 apart: eps << 1e-6 cannot reorder keys
    return ptr, ei, f


@pytest.mark.parametrize("ns", [False, True])
def test_gradcheck(ns):
    rng = np.random.default_rng(4)
    ptr, ei, f = tie_free_batch(rng, [(5, 6), (8, 10), (1, 0), (6, 5)])
    gb = api.GraphBatch(ptr, ei, device=0)
    x = torch.from_numpy(f).to(DEV).requires_grad_(True)

    def fn(x):
        d = gb.diagrams(x, extended=True, no_small=ns)
        return d["birth"], d["death"]

    assert torch.autograd.gradcheck(fn, (x,), eps=1e-9, atol=1e-6, rtol=1e-6)
    gb.close()


@pytest.mark.parametrize("ns", [False, True])
def test_gradient_equals_the_scatter(ns):
    rng = np.random.default_rng(5)
    ptr, ei, f = tie_free_batch(rng, [(n, m) for n, m in SIZES[:12]])
    gb = api.GraphBatch(ptr, ei, device=0)
    x = torch.from_numpy(f).to(DEV).requires_grad_(True)
    d = gb.diagrams(x, extended=True, keep_zero=True, no_small=ns)
    P = gb.pair_bound
    gbirth = torch.from_numpy(rng.standard_normal(P)).to(DEV)
    gdeath = torch.from_numpy(rng.standard_normal(P)).to(DEV)
    h = {k: v.detach().cpu().numpy() for k, v in d.items()}
    (g_both,) = torch.autograd.grad((d["birth"], d["death"]), x, (gbirth, gdeath), retain_graph=True)
    (g_b,) = torch.autograd.grad(d["birth"], x, gbirth, retain_graph=True)   # death's gradient: NULL
    (g_d,) = torch.autograd.grad(d["death"], x, gdeath, retain_graph=True)   # birth's gradient: NULL
    gbn, gdn = gbirth.cpu().numpy(), gdeath.cpu().numpy()
    N = int(ptr[-1])
    for got, b_, d_ in ((g_both, gbn, gdn), (g_b, gbn, None), (g_d, None, gdn)):
        ref = scatter_grad(h["poff"], h["bv"], h["dv"], b_, d_, N)
        assert np.array_equal(got.cpu().numpy().view(np.int64), ref.view(np.int64))
    # the raw entry point with both gradients NULL writes zeros everywhere
    out = torch.full((N,), 3.0, dtype=torch.float64, device=DEV)
    dd = L.Diagrams(P, d["poff"].data_ptr(), None, None, d["bv"].data_ptr(), d["dv"].data_ptr(), None, None)
    L.check(L.lib().tlc_graph_batch_grad_dev(gb._h, dd, None, None, out.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(out, torch.zeros_like(out))
    gb.close()


def test_chain_to_images_and_wasserstein():
    rng = np.random.default_rng(6)
    sizes = [(23, 25), (40, 75), (30, 29), (300, 500)]
    ptr, ei, f = tie_free_batch(rng, sizes + sizes)
    f = f / f.max()
    gb = api.GraphBatch(ptr, ei, device=0)
    D = len(sizes)
    x = torch.from_numpy(f).to(DEV).requires_grad_(True)
    d = gb.diagrams(x, extended=True)
    mask = (1 << L.K_UP) | (1 << L.K_ONE)
    img = api.persistence_images(d["poff"], d["birth"], d["death"], d["kind"], mask)
    px, py = d["poff"][:D + 1].contiguous(), d["poff"][D:].contiguous()
    w, (mx, my) = api.wasserstein_distances(px, d["birth"], d["death"], py, d["birth"], d["death"], d["kind"], d["kind"],
                                            mask, order=2.0, return_matching=True)
    loss = img.square().sum() + w.sum()
    loss.backward()
    # the same chain in CPU float64 at the op's own pairing: birth = f[bv], death = f[dv]
    h = {k: v.detach().cpu() for k, v in d.items()}
    P = int(h["poff"][-1])
    xc = torch.from_numpy(f).requires_grad_(True)
    bc = torch.zeros(gb.pair_bound, dtype=torch.float64)
    dc = torch.zeros(gb.pair_bound, dtype=torch.float64)
    bc = bc.index_put((torch.arange(P),), xc[h["bv"][:P].long()])
    dc = dc.index_put((torch.arange(P),), xc[h["dv"][:P].long()])
    img_c = torch_images(h["poff"], bc, dc, h["kind"], mask)
    mxc, myc = mx.cpu(), my.cpu()
    wc = []
    for t in range(D):
        a0, a1 = int(h["poff"][t]), int(h["poff"][t + 1])
        b0, b1 = int(h["poff"][D + t]), int(h["poff"][D + t + 1])
        lx = torch.where(mxc[a0:a1] >= 0, mxc[a0:a1] - b0, mxc[a0:a1])
        ly = torch.where(myc[b0:b1] >= 0, myc[b0:b1] - a0, myc[b0:b1])
        wc.append(torch_wasserstein(bc[a0:a1], dc[a0:a1], bc[b0:b1], dc[b0:b1], lx, ly, q=2.0))
    loss_c = img_c.square().sum() + torch.stack(wc).sum()
    loss_c.backward()
    assert torch.allclose(img.detach().cpu(), img_c.detach(), rtol=1e-12, atol=1e-13)
    assert torch.allclose(w.detach().cpu(), torch.stack(wc).detach(), rtol=1e-12, atol=1e-13)
    assert torch.allclose(x.grad.cpu(), xc.grad, rtol=1e-10, atol=1e-12)
    gb.close()


def test_side_stream():
    rng = np.random.default_rng(8)
    ptr, ei, f = tie_free_batch(rng, [(n, m) for n, m in SIZES[:10]] * 20)
    gb = api.GraphBatch(ptr, ei, device=0)
    ref = run(gb, f, extended=True)
    x0 = torch.from_numpy(f).to(DEV)
    gref = scatter_grad(ref["poff"], ref["bv"], ref["dv"], np.ones(gb.pair_bound), np.ones(gb.pair_bound), int(ptr[-1]))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x = x0.clone().requires_grad_(True)
        d = gb.diagrams(x, extended=True)
        (d["birth"].sum() + d["death"].sum()).backward()
        got = {k: v.clone() for k, v in d.items()}
        g = x.grad.clone()
    torch.cuda.current_stream().wait_stream(s)
    h = host(got)
    for k in ref:
        assert np.array_equal(ref[k], h[k]), k
    assert np.array_equal(g.cpu().numpy(), gref)
    gb.close()
