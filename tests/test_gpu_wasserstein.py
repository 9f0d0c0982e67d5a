"""Exact Wasserstein distances between device-resident diagrams (tlc_wasserstein_batch_dev /
tlc_wasserstein_batch_grad_dev, api.wasserstein_distances) on the GPU: distances against the scipy optimum of the
expansion pinned in test_wasserstein_abi.py, validity and cost of the returned matchings, the pipeline's own diagrams,
adversarial ties, bit-reproducibility, and gradients against torch's autograd of the restatement of gudhi's autodiff
branch at the op's own matching."""
import math
import multiprocessing as mp
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from helpers import GRAPH_CASES, load_case
from test_wasserstein_abi import (INF, QP, matching_cost, random_diagram, ref_distance, selected,
                                  torch_wasserstein)
from tlc_b200 import _lib as L
from tlc_b200 import api

DEV = torch.device("cuda", 0)
_POOL = None


def pool():
    """host worker processes for the scipy references (spawned: they never touch CUDA)"""
    global _POOL
    if _POOL is None:
        _POOL = mp.get_context("spawn").Pool(max(1, min(os.cpu_count() or 1, 32)))
    return _POOL


def teardown_module(module):
    if _POOL is not None:
        _POOL.terminate()
        _POOL.join()


def _ref_task(args):
    X, Y, q, p = args
    return ref_distance(X, Y, q, p)[0]


def cuda(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV, dtype)


def pack(dgms, kinds=None, pad=3):
    """[K_t, 2] diagrams -> poff, birth, death, kind on the device, `pad` points (0.25, 0.75) before and after"""
    sizes = [len(d) for d in dgms]
    poff = pad + np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    padp = np.tile([[0.25, 0.75]], (pad, 1))
    pts = np.concatenate([padp] + [np.reshape(d, (-1, 2)) for d in dgms] + [padp])
    kind = None
    if kinds is not None:
        kind = cuda(np.concatenate([np.zeros(pad)] + list(kinds) + [np.zeros(pad)]).astype(np.uint8), torch.uint8)
    return cuda(poff, torch.int64), cuda(pts[:, 0]), cuda(pts[:, 1]), kind


def host(d):
    po, b, dd = d["poff"].cpu().numpy(), d["birth"].cpu().numpy(), d["death"].cpu().numpy()
    k = d["kind"].cpu().numpy() if d.get("kind") is not None else None
    return po, b, dd, k


def check_batch(dx, dy, dist, mx, my, q, p, mask=None, refs=None):
    """every pair: distance = scipy optimum (rel 1e-12), matching valid (each selected point used once, zero
    persistence on the diagonal, masked -2), the matching's host cost = the distance"""
    (px, bx, ddx, kx), (py, by, ddy, ky) = host(dx), host(dy)
    dist, mx, my = dist.cpu().numpy(), mx.cpu().numpy(), my.cpu().numpy()
    D = len(px) - 1
    tasks = []
    for t in range(D):
        xs, ys = np.arange(px[t], px[t + 1]), np.arange(py[t], py[t + 1])
        sx = selected(kx[xs] if kx is not None else None, 0xFFFFFFFF if mask is None else mask, len(xs))
        sy = selected(ky[ys] if ky is not None else None, 0xFFFFFFFF if mask is None else mask, len(ys))
        assert np.all(mx[xs[~sx]] == -2) and np.all(my[ys[~sy]] == -2), t
        xs, ys = xs[sx], ys[sy]
        X, Y = np.stack([bx[xs], ddx[xs]], 1), np.stack([by[ys], ddy[ys]], 1)
        assert np.all(mx[xs[X[:, 0] == X[:, 1]]] == -1) and np.all(my[ys[Y[:, 0] == Y[:, 1]]] == -1), t
        m_loc = -np.ones(len(xs), np.int64)
        lut = {int(g): i for i, g in enumerate(ys)}
        for i, g in enumerate(mx[xs]):
            if g >= 0:
                j = lut[int(g)]
                assert my[g] == xs[i], t  # the two sides agree
                m_loc[i] = j
        taken = mx[xs][mx[xs] >= 0]
        assert len(np.unique(taken)) == len(taken), t
        assert np.all(np.isin(my[ys][my[ys] >= 0], xs)), t
        w = matching_cost(X, Y, m_loc, q, p)
        assert abs(w - dist[t]) <= 1e-12 * max(w, 1e-300), (t, w, dist[t])
        tasks.append((X, Y, q, p))
    ref = refs if refs is not None else pool().map(_ref_task, tasks, chunksize=4)
    ref = np.asarray(ref)
    err = np.abs(dist - ref) / np.where(ref > 0, ref, 1.0)
    assert err.max(initial=0.0) < 1e-12, (int(err.argmax()), dist[err.argmax()], ref[err.argmax()])


def run(dx, dy, mask=None, q=1.0, p=INF):
    return api.wasserstein_distances(dx["poff"], dx["birth"], dx["death"], dy["poff"], dy["birth"], dy["death"],
                                     dx.get("kind"), dy.get("kind"), mask, q, p, return_matching=True)


def random_pairs(rng, D=500, top=300, lattice=False):
    sx, sy = rng.integers(0, top + 1, D), rng.integers(0, top + 1, D)
    sx[:3], sy[:3] = [0, 0, 7], [0, 9, 0]  # empty / empty, empty / non-empty, non-empty / empty
    X = [random_diagram(rng, int(n), lattice=lattice) for n in sx]
    Y = [random_diagram(rng, int(n), lattice=lattice) for n in sy]
    kx = [rng.integers(0, 5, len(d)) for d in X]
    ky = [rng.integers(0, 5, len(d)) for d in Y]
    return [dict(zip(("poff", "birth", "death", "kind"), pack(a, k))) for a, k in ((X, kx), (Y, ky))]


MASK = (1 << L.K_UP) | (1 << L.K_ESS) | (1 << L.K_ONE)


@pytest.mark.parametrize("q,p", QP)
def test_random_batches_against_scipy(q, p):
    rng = np.random.default_rng(int(100 * q + (7 if math.isinf(p) else p)))
    dx, dy = random_pairs(rng)
    dist, (mx, my) = run(dx, dy, MASK, q, p)
    check_batch(dx, dy, dist, mx, my, q, p, MASK)
    P = dx["birth"].numel()
    assert torch.all(mx[:3] == -2) and torch.all(mx[P - 3:] == -2)  # the padding is in no pair


def small_targets(c, limit=600):
    """the case's targets whose 2-hop edge vicinity has at most `limit` vertices + edges (keeps the host reference
    quick)"""
    g = api.VicinityGraph(*c["csr"], device=0)
    n, m, _ = g.vicinity_sizes(c["new_targets"], hop=2)
    g.close()
    return c["new_targets"][n.astype(np.int64) + m <= limit]


def vicinity(c, tg, hop, ext, mode=L.MODE_EDGE):
    g = api.VicinityGraph(*c["csr"], device=0)
    flags = L.F_NORM | (L.F_EXTENDED if ext else 0)
    tg = tg if mode == L.MODE_EDGE else np.stack([tg[:, 0]] * 2, 1)  # node mode: (u, u)
    d = g.vicinity_diagrams_dev(cuda(tg, torch.int32), hop=hop, mode=mode, descriptor=c["descriptor"], flags=flags)
    torch.cuda.synchronize()
    g.close()
    return d


@pytest.mark.parametrize("tag", GRAPH_CASES[:5])
def test_pipeline_diagrams(tag):
    """the same targets at hop 1 against hop 2, and edge against node mode: every kind, PD_up + ESS, PD_one"""
    c = load_case(tag)
    tg = small_targets(c)
    assert len(tg) >= 4
    for (h1, m1), (h2, m2) in (((1, L.MODE_EDGE), (2, L.MODE_EDGE)), ((c["hop"], L.MODE_EDGE), (c["hop"], L.MODE_NODE))):
        dx, dy = vicinity(c, tg, h1, 1, m1), vicinity(c, tg, h2, 1, m2)
        for mask in (None, (1 << L.K_UP) | (1 << L.K_ESS), 1 << L.K_ONE):
            dist, (mx, my) = run(dx, dy, mask)
            check_batch(dx, dy, dist, mx, my, 1.0, INF, mask)
        dist, (mx, my) = run(dx, dy, None, 2.0, 2.0)
        check_batch(dx, dy, dist, mx, my, 2.0, 2.0)


def test_one_large_pair():
    rng = np.random.default_rng(11)
    X, Y = random_diagram(rng, 2500, zero=0.0), random_diagram(rng, 2000, zero=0.0)
    dx, dy = [dict(zip(("poff", "birth", "death", "kind"), pack([a]))) for a in (X, Y)]
    dist, (mx, my) = run(dx, dy)
    check_batch(dx, dy, dist, mx, my, 1.0, INF, refs=[ref_distance(X, Y, 1.0, INF)[0]])


@pytest.mark.parametrize("q,p", [(1.0, INF), (2.0, 2.0), (1.5, 1.0)])
def test_adversarial_ties(q, p):
    rng = np.random.default_rng(12)
    lat = [random_diagram(rng, int(n), lattice=True) for n in (200, 350, 400, 60)]
    same = [np.tile([[0.25, 0.75]], (n, 1)) for n in (300, 500)]
    base = random_diagram(rng, 300, zero=0.0)
    mirror = base[:, ::-1]  # reflected across the diagonal: every cost to the diagonal is the same
    X = lat[:2] + [same[0], base, lat[2]]
    Y = [lat[3], lat[1], same[1], mirror, lat[2] + 0.25]
    dx, dy = [dict(zip(("poff", "birth", "death", "kind"), pack(a))) for a in (X, Y)]
    dist, (mx, my) = run(dx, dy, None, q, p)
    check_batch(dx, dy, dist, mx, my, q, p)


def test_non_finite_pairs_are_reported_and_leave_the_others_alone():
    rng = np.random.default_rng(13)
    X = [random_diagram(rng, 30) for _ in range(5)]
    Y = [random_diagram(rng, 25) for _ in range(5)]
    X[1] = X[1].copy(); X[1][4, 1] = math.nan
    Y[3] = Y[3].copy(); Y[3][0, 0] = -math.inf
    dx, dy = [dict(zip(("poff", "birth", "death", "kind"), pack(a))) for a in (X, Y)]
    dist, (mx, my) = run(dx, dy)
    d = dist.cpu().numpy()
    assert np.isnan(d[1]) and np.isnan(d[3]) and np.isfinite(d[[0, 2, 4]]).all()
    px, py = dx["poff"].cpu().numpy(), dy["poff"].cpu().numpy()
    for t in (1, 3):
        assert torch.all(mx[px[t]:px[t + 1]] == -1) and torch.all(my[py[t]:py[t + 1]] == -1)
    for t in (0, 2, 4):
        assert abs(d[t] - ref_distance(X[t], Y[t])[0]) <= 1e-12 * d[t]
    # a non-finite point that is masked out does not count
    kx = [np.zeros(len(a)) for a in X]
    kx[1][4] = L.K_DOWN
    dxk = dict(dx, kind=pack(X, kx)[3])
    dist2 = run(dxk, dict(dy, kind=None), 1 << L.K_UP)[0].cpu().numpy()
    assert np.isfinite(dist2[1]) and np.isnan(dist2[3])
    # the gradient of an unsolved pair is NaN on its selected points, and the others' are finite
    bx = dx["birth"].clone().requires_grad_(True)
    api.wasserstein_distances(dx["poff"], bx, dx["death"], dy["poff"], dy["birth"], dy["death"]).sum().backward()
    g = bx.grad.cpu().numpy()
    assert np.isnan(g[px[1]:px[2]]).all() and np.isfinite(g[px[0]:px[1]]).all() and np.isfinite(g[px[2]:px[3]]).all()


def test_bit_reproducible_split_batches_and_padding():
    rng = np.random.default_rng(14)
    dx, dy = random_pairs(rng, D=200, top=200)
    one = run(dx, dy, MASK, 1.5, 2.0)
    two = run(dx, dy, MASK, 1.5, 2.0)
    assert torch.equal(one[0], two[0]) and torch.equal(one[1][0], two[1][0]) and torch.equal(one[1][1], two[1][1])
    h = 77
    parts = []
    for sl in (slice(0, h + 1), slice(h, None)):
        parts.append(run(dict(dx, poff=dx["poff"][sl].contiguous()), dict(dy, poff=dy["poff"][sl].contiguous()),
                         MASK, 1.5, 2.0))
    assert torch.equal(torch.cat([parts[0][0], parts[1][0]]), one[0])
    px, py = dx["poff"].cpu().numpy(), dy["poff"].cpu().numpy()
    assert torch.equal(parts[0][1][0][:px[h]], one[1][0][:px[h]]) and torch.equal(parts[1][1][0][px[h]:], one[1][0][px[h]:])
    assert torch.equal(parts[0][1][1][:py[h]], one[1][1][:py[h]]) and torch.equal(parts[1][1][1][py[h]:], one[1][1][py[h]:])
    # the raw call writes [poff[0], poff[D]) and nothing else, in the match and the gradient arrays
    D, Px, Py = len(px) - 1, dx["birth"].numel(), dy["birth"].numel()
    nb = 64 * (Px + Py)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    dist = torch.empty(D, dtype=torch.float64, device=DEV)
    mx = torch.full((Px,), 99, dtype=torch.int64, device=DEV)
    my = torch.full((Py,), 99, dtype=torch.int64, device=DEV)
    ins = [t.data_ptr() if t is not None else None for t in (dx["poff"], dx["birth"], dx["death"], dx["kind"],
                                                              dy["poff"], dy["birth"], dy["death"], dy["kind"])]
    L.check(L.lib().tlc_wasserstein_batch_dev(0, D, Px, Py, *ins, MASK, 1.5, 2.0, ws.data_ptr(), nb, dist.data_ptr(),
                                              mx.data_ptr(), my.data_ptr(), None))
    G = torch.randn(D, dtype=torch.float64, device=DEV)
    grads = [torch.full((n,), 7.0, dtype=torch.float64, device=DEV) for n in (Px, Px, Py, Py)]
    L.check(L.lib().tlc_wasserstein_batch_grad_dev(0, D, *ins, MASK, 1.5, 2.0, dist.data_ptr(), mx.data_ptr(),
                                                   my.data_ptr(), G.data_ptr(), *[g.data_ptr() for g in grads], None))
    torch.cuda.synchronize()
    assert torch.equal(dist, one[0])
    for arr, lo, hi, fill in ((mx, px[0], px[-1], 99), (my, py[0], py[-1], 99), (grads[0], px[0], px[-1], 7.0),
                              (grads[3], py[0], py[-1], 7.0)):
        assert torch.all(arr[:lo] == fill) and torch.all(arr[hi:] == fill)
    assert torch.equal(mx[px[0]:px[-1]], one[1][0][px[0]:px[-1]])


def pair_grads(fn_inputs, dist_fn, G):
    ts = [t.clone().requires_grad_(True) for t in fn_inputs]
    out = dist_fn(*ts)
    return out.detach(), torch.autograd.grad(out, ts, G, allow_unused=True)


def ref_grads(dx, dy, mx, my, G, q, p, mask=None):
    """torch autograd of the restatement of gudhi's autodiff branch, pair by pair, at the op's own matching"""
    (px, *_), (py, *_) = host(dx), host(dy)
    kx = dx.get("kind")
    ky = dy.get("kind")
    mxh, myh = mx.cpu(), my.cpu()
    ts = [t.detach().cpu().clone().requires_grad_(True) for t in (dx["birth"], dx["death"], dy["birth"], dy["death"])]
    tot = 0.0
    for t in range(len(px) - 1):
        xs, ys = slice(px[t], px[t + 1]), slice(py[t], py[t + 1])
        lx = mxh[xs].clone()
        ly = myh[ys].clone()
        lx[lx >= 0] -= py[t]
        ly[ly >= 0] -= px[t]
        W = torch_wasserstein(ts[0][xs], ts[1][xs], ts[2][ys], ts[3][ys], lx, ly, q, p)
        tot = tot + W * G[t].cpu()
    gs = torch.autograd.grad(tot, ts, allow_unused=True)
    return [torch.zeros_like(ts[k]) if g is None else g for k, g in enumerate(gs)]


def op_grads(dx, dy, G, q, p, mask=None):
    ts = [t.clone().requires_grad_(True) for t in (dx["birth"], dx["death"], dy["birth"], dy["death"])]
    dist, (mx, my) = api.wasserstein_distances(dx["poff"], ts[0], ts[1], dy["poff"], ts[2], ts[3], dx.get("kind"),
                                                dy.get("kind"), mask, q, p, return_matching=True)
    gs = torch.autograd.grad(dist, ts, G)
    return dist.detach(), mx, my, gs


def close(a, b, tol=1e-12):
    a, b = a.cpu().numpy(), b.cpu().numpy()
    den = np.maximum(np.abs(b), 1e-3 * max(np.abs(b).max(initial=0.0), 1e-300))
    return float(np.max(np.abs(a - b) / den, initial=0.0)) < tol


@pytest.mark.parametrize("q,p", QP)
def test_gradients_against_the_restatement(q, p):
    rng = np.random.default_rng(int(200 + 10 * q + (7 if math.isinf(p) else p)))
    dx, dy = random_pairs(rng, D=40, top=40)
    G = torch.randn(40, dtype=torch.float64, device=DEV)
    dist, mx, my, gs = op_grads(dx, dy, G, q, p, MASK)
    ref = ref_grads(dx, dy, mx, my, G, q, p, MASK)
    # masked points: the restatement does not see them (match -2), the op gives 0
    for got, want in zip(gs, ref):
        assert close(got, want), (q, p)


def test_gradcheck_tie_free():
    rng = np.random.default_rng(15)
    X = [rng.uniform(0, 1, (n, 2)) for n in (4, 0, 3)]
    Y = [rng.uniform(0, 1, (n, 2)) for n in (3, 2, 0)]
    dx, dy = [dict(zip(("poff", "birth", "death", "kind"), pack(a, pad=1))) for a in (X, Y)]
    for q, p in ((1.0, INF), (1.5, 2.0), (2.0, 1.0), (1.5, 3.0)):
        ins = [t.clone().requires_grad_(True) for t in (dx["birth"], dx["death"], dy["birth"], dy["death"])]
        f = lambda a, b, c, d: api.wasserstein_distances(dx["poff"], a, b, dy["poff"], c, d,  # noqa: E731
                                                         order=q, internal_p=p)
        assert torch.autograd.gradcheck(f, ins, eps=1e-7, atol=1e-6)


def test_gradient_conventions_and_null_pointers():
    f = lambda *a: np.array(a, dtype=np.float64).reshape(-1, 2)  # noqa: E731
    # pair 0: x0 == y0 (zero-length difference); pair 1: inf-norm tie; pair 2: S = 0 (all zero persistence);
    # pair 3: a masked point
    X = [f(0.0, 1.0), f(0.0, 1.0), f(0.5, 0.5), f(0.0, 1.0, 0.2, 0.9)]
    Y = [f(0.0, 1.0), f(2.0, 3.0), f(0.3, 0.3), f(0.1, 1.0)]
    kx = [np.zeros(1), np.zeros(1), np.zeros(1), np.array([0, L.K_DOWN])]
    ky = [np.zeros(1)] * 4
    dx = dict(zip(("poff", "birth", "death", "kind"), pack(X, kx, pad=2)))
    dy = dict(zip(("poff", "birth", "death", "kind"), pack(Y, ky, pad=2)))
    G = torch.tensor([1.0, 2.0, 3.0, 4.0], dtype=torch.float64, device=DEV)
    mask = 1 << L.K_UP
    dist, mx, my, gs = op_grads(dx, dy, G, 1.0, INF, mask)
    d = dist.cpu().numpy()
    assert d[0] == 0.0 and d[2] == 0.0
    gbx, gdx, gby, gdy = [g.cpu().numpy() for g in gs]
    assert gbx[2] == 0.0 and gdx[2] == 0.0 and gby[2] == 0.0 and gdy[2] == 0.0  # x0 == y0
    # pair 1: x = (0, 1), y = (2, 3): matched (cost 2) vs diagonal (0.5 + 0.5): the diagonal wins -> +-G/2 each
    assert gbx[3] == -1.0 and gdx[3] == 1.0
    assert gbx[4] == 0.0 and gdx[4] == 0.0 and gby[4] == 0.0 and gdy[4] == 0.0  # S = 0
    assert gbx[6] == 0.0 and gdx[6] == 0.0  # masked
    ref = ref_grads(dx, dy, mx, my, G, 1.0, INF)
    for got, want in zip(gs, ref):
        assert close(got, want)
    # a tie of the inf-norm: x = (0, 0.5), y = (0.25, 0.75): e = (-0.25, -0.25), cheaper than the diagonal (0.5)
    dx2 = dict(zip(("poff", "birth", "death", "kind"), pack([f(0.0, 0.5)], pad=0)))
    dy2 = dict(zip(("poff", "birth", "death", "kind"), pack([f(0.25, 0.75)], pad=0)))
    _, _, _, g2 = op_grads(dx2, dy2, torch.ones(1, dtype=torch.float64, device=DEV), 1.0, INF)
    assert [g.item() for g in g2] == [-0.5, -0.5, 0.5, 0.5]
    # NULL gradient pointers: each alone equals its part of the full gradient; autograd asks only for what it needs
    D, Px, Py = 4, dx["birth"].numel(), dy["birth"].numel()
    ins = [t.data_ptr() for t in (dx["poff"], dx["birth"], dx["death"], dx["kind"], dy["poff"], dy["birth"],
                                  dy["death"], dy["kind"])]
    for which in range(4):
        outs = [torch.full((n,), 7.0, dtype=torch.float64, device=DEV) if k == which else None
                for k, n in enumerate((Px, Px, Py, Py))]
        L.check(L.lib().tlc_wasserstein_batch_grad_dev(
            0, D, *ins, mask, 1.0, INF, dist.data_ptr(), mx.data_ptr(), my.data_ptr(), G.data_ptr(),
            *[o.data_ptr() if o is not None else None for o in outs], None))
        torch.cuda.synchronize()
        lo, hi = (int(dx["poff"][0]), int(dx["poff"][-1])) if which < 2 else (int(dy["poff"][0]), int(dy["poff"][-1]))
        assert torch.equal(outs[which][lo:hi], gs[which][lo:hi])
    dd = dy["death"].clone().requires_grad_(True)
    api.wasserstein_distances(dx["poff"], dx["birth"], dx["death"], dy["poff"], dy["birth"], dd, dx["kind"],
                              dy["kind"], mask).mul(G).sum().backward()
    assert torch.equal(dd.grad, gs[3])


def test_inputs_and_calls_on_a_side_stream():
    rng = np.random.default_rng(16)
    sizes = rng.integers(1, 120, 256)
    poff_h = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    P = int(poff_h[-1])
    s = torch.cuda.Stream(DEV)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        m = torch.rand((4096, 4096), dtype=torch.float64, device=DEV)
        for _ in range(4):  # work queued ahead of the inputs
            m = (m @ m).clamp_(0, 1)
        u = torch.rand((4, P), dtype=torch.float64, device=DEV) + 0 * m[0, 0]
        bx = u[0].clone().requires_grad_(True)
        dx = (u[0] + u[1] - 0.3).detach().requires_grad_(True)
        by = u[2].clone().requires_grad_(True)
        dy = (u[2] + u[3] - 0.3).detach().requires_grad_(True)
        poff = torch.as_tensor(poff_h).to(DEV)
        G = torch.rand(len(sizes), dtype=torch.float64, device=DEV)
        dist, (mx, my) = api.wasserstein_distances(poff, bx, dx, poff, by, dy, return_matching=True)
        (dist * G).sum().backward()
    s.synchronize()
    ax = dict(poff=poff, birth=bx.detach(), death=dx.detach(), kind=None)
    ay = dict(poff=poff, birth=by.detach(), death=dy.detach(), kind=None)
    check_batch(ax, ay, dist.detach(), mx, my, 1.0, INF)
    ref = ref_grads(ax, ay, mx, my, G, 1.0, INF)
    for got, want in zip((bx.grad, dx.grad, by.grad, dy.grad), ref):
        assert close(got, want)


def test_composition_with_persistence_images():
    rng = np.random.default_rng(17)
    X = [random_diagram(rng, n, zero=0.0) for n in (20, 35, 8)]
    Y = [random_diagram(rng, n, zero=0.0) for n in (25, 5, 12)]
    dx, dy = [dict(zip(("poff", "birth", "death", "kind"), pack(a))) for a in (X, Y)]
    b = dx["birth"].clone().requires_grad_(True)
    d = dx["death"].clone().requires_grad_(True)
    img = api.persistence_images(dx["poff"], b, d)
    w = api.wasserstein_distances(dx["poff"], b, d, dy["poff"], dy["birth"], dy["death"], order=2.0, internal_p=2.0)
    (img.sum() + w.sum()).backward()
    bi, di = b.detach().clone().requires_grad_(True), d.detach().clone().requires_grad_(True)
    gi = torch.autograd.grad(api.persistence_images(dx["poff"], bi, di).sum(), (bi, di))
    bw, dw = b.detach().clone().requires_grad_(True), d.detach().clone().requires_grad_(True)
    gw = torch.autograd.grad(api.wasserstein_distances(dx["poff"], bw, dw, dy["poff"], dy["birth"], dy["death"],
                                                       order=2.0, internal_p=2.0).sum(), (bw, dw))
    assert torch.allclose(b.grad, gi[0] + gw[0], rtol=1e-13, atol=1e-15)
    assert torch.allclose(d.grad, gi[1] + gw[1], rtol=1e-13, atol=1e-15)
