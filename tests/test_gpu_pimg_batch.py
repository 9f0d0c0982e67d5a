"""The batch imager of device-resident diagrams (tlc_pimg_batch_dev / tlc_pimg_batch_grad_dev, api.persistence_images) on
the GPU: the stored golden images, the pipeline's own image rows on every route, bit-reproducibility, and gradients
against torch's autograd of the restatement pinned in test_pimg_batch_abi.py."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from helpers import GOLDEN, GRAPH_CASES, load_case, rel_err
from test_pimg_batch_abi import golden_diagrams, torch_images
from tlc_b200 import _lib as L
from tlc_b200 import api, graphgen as gg

IMG_TOL = 1e-5
DEV = torch.device("cuda", 0)


def cuda(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV, dtype)


def pack(dgms, pad=0):
    """[K_t, 2] diagrams -> poff, birth, death on the device, `pad` points before and after the segments"""
    sizes = [len(d) for d in dgms]
    poff = pad + np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    pts = np.concatenate([np.full((pad, 2), 0.5)] + [np.reshape(d, (-1, 2)) for d in dgms] + [np.full((pad, 2), 0.5)])
    return cuda(poff, torch.int64), cuda(pts[:, 0]), cuda(pts[:, 1])


def pimg(d, mask, res=5):
    return api.persistence_images(d["poff"], d["birth"], d["death"], d["kind"], mask, res)


def check_rows(rows, d, ref):
    rows, ref = rows.cpu().numpy(), np.asarray(ref.cpu().numpy() if torch.is_tensor(ref) else ref)
    empty = np.diff(d["poff"].cpu().numpy()) == 0
    assert np.all(rows[empty] == 0.0)
    assert rel_err(rows, ref) < 1e-12


def test_golden_vectors_in_one_batch():
    cases, gt4 = golden_diagrams()
    res5 = [c for c in cases if c[1] == 5]
    empty = np.zeros((0, 2))
    dgms = [empty] + [c[0] for c in res5[:2]] + [empty] + [c[0] for c in res5[2:]] + [empty]
    imgs = [None] + [c[2] for c in res5[:2]] + [None] + [c[2] for c in res5[2:]] + [None]
    poff, b, dth = pack(dgms, pad=3)
    rows = api.persistence_images(poff, b, dth).cpu().numpy()
    for row, img in zip(rows, imgs):
        if img is None:
            assert np.all(row == 0.0)
        else:
            assert rel_err(row, img) < IMG_TOL
    assert np.max(np.abs(rows[1] - gt4)) < 6e-5
    (d7, _, img7), = [c for c in cases if c[1] == 7]
    poff, b, dth = pack([d7, empty])
    rows7 = api.persistence_images(poff, b, dth, resolution=7).cpu().numpy()
    assert rel_err(rows7[0], img7) < IMG_TOL and np.all(rows7[1] == 0.0)


def bad_targets(N):
    return np.array([[-1, 0], [0, 0], [0, N + 7]], np.int32)


@pytest.mark.parametrize("tag", GRAPH_CASES)
@pytest.mark.parametrize("ext", [0, 1])
def test_pipeline_rows_golden_cases(tag, ext):
    c = load_case(tag)
    g = api.VicinityGraph(*c["csr"], device=0)
    tg = np.concatenate([c["new_targets"], bad_targets(len(c["labels"]))])
    flags = L.F_NORM | (L.F_EXTENDED if ext else 0)
    d = g.vicinity_diagrams_dev(cuda(tg, torch.int32), hop=c["hop"], descriptor=c["descriptor"], flags=flags, want_pi=True)
    assert len(set(d["status"].cpu().numpy().tolist())) > 1
    check_rows(pimg(d, L.default_img_mask(ext)), d, d["pi"])
    g.close()


def make(name, scale=1.0, cont=False):
    c = gg.make_config(name, scale=scale, continuous=cont)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    return gg.build_csr(len(labels), ne, c["kappa"]), ne, len(labels)


def test_pipeline_rows_kernel_s_materialised_and_graph_row_routes():
    csr, ne, N = make("computers", 1.0, False)
    g = api.VicinityGraph(*csr, device=0)
    cand = ne[np.random.default_rng(5).choice(len(ne), 4096, replace=False)].astype(np.int32)
    n, m, _ = g.vicinity_sizes(cand, hop=2)
    small, big = np.flatnonzero(n <= 64)[:96], np.flatnonzero(n > 1024)[:24]
    tg = np.concatenate([cand[np.random.default_rng(6).permutation(np.concatenate([small, big]))], bad_targets(N)])
    n_, m_, _ = g.vicinity_sizes(tg, hop=2)
    cap = int((n_.astype(np.int64) + m_ + 2).sum())
    d = g.vicinity_diagrams_dev(cuda(tg, torch.int32), hop=2, flags=L.F_NORM, want_pi=True, cap=cap)
    s, cn = g.last_small(), g.last_counts()
    assert s["rows_a"] + s["rows_b"] + s["rows_c"] > 0 and s["rows_staged"] > 0 and cn["graph_row_route"] == 0, (s, cn)
    check_rows(pimg(d, L.default_img_mask(False)), d, d["pi"])
    fl = L.F_NORM | L.F_ASC_ONLY | L.F_DIRECT | L.F_NO_SMALL
    d = g.vicinity_diagrams_dev(cuda(tg, torch.int32), hop=2, flags=fl, want_pi=True, cap=cap)
    assert g.last_counts()["graph_row_route"] > 0
    check_rows(pimg(d, L.default_img_mask(False)), d, d["pi"])
    g.close()


def test_pipeline_rows_kd_masks():
    csr, ne, N = make("pubmed", 0.3, True)
    g = api.VicinityGraph(*csr, device=0)
    ids = np.random.default_rng(9).choice(N, 64, replace=False).astype(np.int32)
    tg = np.stack([ids, ids], 1)
    fl = L.F_NORM | L.F_EXTENDED | L.F_KEEP_ZERO | L.F_NORM_EPS
    d = g.vicinity_diagrams_dev(cuda(tg, torch.int32), hop=2, mode=L.MODE_NODE, flags=fl)
    det = g.vicinity_detail(tg, hop=2, mode=L.MODE_NODE, flags=fl)
    assert (d["death"] == d["birth"]).any()  # the keep-zero pairs
    for mask, key in (((1 << L.K_UP) | (1 << L.K_ONE), "pi"), (1 << L.K_UP, "pi_up"), (1 << L.K_ONE, "pi_one")):
        check_rows(pimg(d, mask), d, det[key])
    g.close()


@pytest.mark.parametrize("res", [1, 7, 16])
def test_pipeline_rows_resolutions(res):
    csr, ne, N = make("pubmed", 0.3, True)
    g = api.VicinityGraph(*csr, device=0)
    tg = np.concatenate([ne[np.random.default_rng(4).choice(len(ne), 128, replace=False)], bad_targets(N)]).astype(np.int32)
    fl = L.F_NORM | L.F_EXTENDED
    d = g.vicinity_diagrams_dev(cuda(tg, torch.int32), hop=2, flags=fl, resolution=res, want_pi=True)
    check_rows(pimg(d, L.default_img_mask(True), res), d, d["pi"])
    g.close()


def random_batch(rng, sizes, pad=5, special=False):
    """poff, birth, death, kind on the device: diagrams of the given sizes between `pad` points on either side"""
    P = int(sum(sizes)) + 2 * pad
    b = rng.uniform(-0.5, 1.5, P)
    p = rng.uniform(-0.5, 1.5, P)
    if special:  # p < 0, p == 0, p == 1 exactly (dyadic births), p > 1, values outside [0, 1]
        sel = rng.random(P)
        b = np.where(sel < 0.4, rng.integers(-8, 16, P) / 8.0, b)
        p = np.where(sel < 0.2, 0.0, np.where(sel < 0.4, 1.0, p))
    kind = rng.integers(0, 5, P).astype(np.uint8)
    kind[rng.random(P) < 0.02] = 40  # no bit of the mask covers it
    poff = pad + np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return cuda(poff, torch.int64), cuda(b), cuda(b + p), cuda(kind, torch.uint8)


MASK = (1 << L.K_UP) | (1 << L.K_ESS) | (1 << L.K_ONE)


def grads(fn, poff, b, d, kind, mask, res, G):
    bb, dd = b.clone().requires_grad_(True), d.clone().requires_grad_(True)
    out = fn(poff, bb, dd, kind, mask, res)
    gb, gd = torch.autograd.grad(out, (bb, dd), G)
    return out.detach(), gb, gd


def check_grads(mine, ref):
    (o, gb, gd), (ro, rgb, rgd) = [[t.cpu().numpy() for t in x] for x in (mine, ref)]
    assert rel_err(o, ro) < 1e-12
    # both gradients are sums over the pixels of terms of either sign (grad_out has either sign; grad_birth is moreover
    # a difference of two such sums): an element that cancels to near zero carries the absolute rounding error of its
    # terms, which are of the order of the largest element -- relative error, floored at 1 % of the largest element
    for got, ref in ((gb, rgb), (gd, rgd)):
        den = np.maximum(np.abs(ref), 1e-2 * np.abs(ref).max())
        assert np.max(np.abs(got - ref) / np.where(den > 0, den, 1.0)) < 1e-12
    assert np.array_equal(gb == 0, rgb == 0) and np.array_equal(gd == 0, rgd == 0)


@pytest.mark.parametrize("res", [1, 5, 16])
def test_gradcheck(res):
    rng = np.random.default_rng(res)
    sizes = [3, 0, 4, 1]
    poff, b, d, kind = random_batch(rng, sizes, pad=2)
    p = rng.uniform(-0.5, 1.5, b.numel())
    p = np.where(np.abs(p) < 1e-2, p + 0.05, np.where(np.abs(p - 1) < 1e-2, p + 0.05, p))  # >= 1e-3 from the kinks
    d = b + cuda(p)
    b.requires_grad_(True)
    d.requires_grad_(True)
    assert torch.autograd.gradcheck(lambda x, y: api.persistence_images(poff, x, y, kind, MASK, res), (b, d))


@pytest.mark.parametrize("res", [1, 5, 16])
def test_gradients_against_the_restatement(res):
    rng = np.random.default_rng(100 + res)
    sizes = rng.integers(0, 40, 64)
    sizes[[0, 31, 63]] = 0
    poff, b, d, kind = random_batch(rng, sizes, special=True)
    G = torch.randn((len(sizes), res * res), dtype=torch.float64, device=DEV)
    check_grads(grads(api.persistence_images, poff, b, d, kind, MASK, res, G),
                grads(torch_images, poff, b, d, kind, MASK, res, G))


@pytest.mark.parametrize("shape", ["one_large", "many_single"])
def test_gradients_large_and_single_point_diagrams(shape):
    rng = np.random.default_rng(7)
    sizes = [200000] if shape == "one_large" else [1] * 100000
    poff, b, d, kind = random_batch(rng, sizes, special=True)
    G = torch.rand((len(sizes), 25), dtype=torch.float64, device=DEV)
    check_grads(grads(api.persistence_images, poff, b, d, kind, MASK, 5, G),
                grads(torch_images, poff, b, d, kind, MASK, 5, G))


def test_a_million_point_diagram():
    rng = np.random.default_rng(8)
    poff, b, d, _ = random_batch(rng, [1000000, 3])
    ref = torch_images(poff, b, d)
    assert rel_err(api.persistence_images(poff, b, d).cpu().numpy(), ref.cpu().numpy()) < 1e-12


@pytest.mark.parametrize("res", [1, 5, 16])
def test_bit_reproducible_and_independent_of_the_batch(res):
    rng = np.random.default_rng(20 + res)
    sizes = np.concatenate([rng.integers(0, 3000, 40), [200000], rng.integers(0, 50, 40)])
    poff, b, d, kind = random_batch(rng, sizes, special=True)
    D = len(sizes)
    G = torch.randn((D, res * res), dtype=torch.float64, device=DEV)
    one = grads(api.persistence_images, poff, b, d, kind, MASK, res, G)
    two = grads(api.persistence_images, poff, b, d, kind, MASK, res, G)
    for x, y in zip(one, two):
        assert torch.equal(x, y)
    h = D // 2 + 3
    lo = grads(api.persistence_images, poff[:h + 1].contiguous(), b, d, kind, MASK, res, G[:h])
    hi = grads(api.persistence_images, poff[h:].contiguous(), b, d, kind, MASK, res, G[h:])
    assert torch.equal(torch.cat([lo[0], hi[0]]), one[0])
    assert torch.equal(lo[1] + hi[1], one[1]) and torch.equal(lo[2] + hi[2], one[2])  # each is zero outside its points


def test_null_gradient_pointer_and_the_written_range():
    rng = np.random.default_rng(30)
    poff, b, d, kind = random_batch(rng, [5, 0, 17, 3], pad=4)
    D, P = 4, b.numel()
    G = torch.randn((D, 25), dtype=torch.float64, device=DEV)
    _, rgb, rgd = grads(api.persistence_images, poff, b, d, kind, MASK, 5, G)
    lo, hi = int(poff[0]), int(poff[-1])
    for which in ("birth", "death"):
        gb = torch.full((P,), 7.0, dtype=torch.float64, device=DEV)
        gd = torch.full((P,), 7.0, dtype=torch.float64, device=DEV)
        L.check(L.lib().tlc_pimg_batch_grad_dev(
            0, D, poff.data_ptr(), b.data_ptr(), d.data_ptr(), kind.data_ptr(), MASK, 5, G.data_ptr(),
            gb.data_ptr() if which == "birth" else None, gd.data_ptr() if which == "death" else None, None))
        torch.cuda.synchronize()
        got, untouched, ref = (gb, gd, rgb) if which == "birth" else (gd, gb, rgd)
        assert torch.all(untouched == 7.0)
        assert torch.all(got[:lo] == 7.0) and torch.all(got[hi:] == 7.0)
        assert torch.equal(got[lo:hi], ref[lo:hi])
    # autograd asks only for what it needs
    dd = d.clone().requires_grad_(True)
    api.persistence_images(poff, b, dd, kind, MASK).mul(G).sum().backward()
    assert torch.equal(dd.grad, rgd)


def test_inputs_and_calls_on_a_side_stream():
    rng = np.random.default_rng(40)
    sizes = rng.integers(1, 2000, 512)
    poff_h = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    P = int(poff_h[-1])
    s = torch.cuda.Stream(DEV)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        m = torch.rand((4096, 4096), dtype=torch.float64, device=DEV)
        for _ in range(4):  # work queued ahead of the inputs
            m = (m @ m).clamp_(0, 1)
        u = torch.rand((2, P), dtype=torch.float64, device=DEV) + 0 * m[0, 0]
        b = (u[0] * 2 - 0.5).requires_grad_(True)
        d = (b.detach() + u[1] * 2 - 0.5).requires_grad_(True)
        poff = torch.as_tensor(poff_h).to(DEV, non_blocking=False)
        G = torch.rand((len(sizes), 25), dtype=torch.float64, device=DEV)
        out = api.persistence_images(poff, b, d)
        (out * G).sum().backward()
    s.synchronize()
    ref = grads(lambda po, x, y, k, msk, r: torch_images(po, x, y, resolution=r), poff, b.detach(), d.detach(), None,
                None, 5, G)
    check_grads((out.detach(), b.grad, d.grad), ref)
