"""Wasserstein distances between device-resident diagrams without a GPU: tlc_wasserstein_batch_dev /
tlc_wasserstein_batch_grad_dev reject bad arguments before any CUDA call, the workspace query follows its formula,
api.wasserstein_distances checks its tensors before touching CUDA, and the host restatements the GPU tests use as their
references are pinned here: the N x N assignment expansion (scipy's linear_sum_assignment) against gudhi's own
(n+1) x (m+1) mass-transport LP solved exactly (scipy's linprog, HiGHS), and the torch restatement of gudhi's autodiff
branch that serves as the gradient reference."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment, linprog

from tlc_b200 import _lib as L
from tlc_b200 import api

INF = math.inf


def kappa(p):
    """delta(x) = |d - b| * kappa: the p-norm distance of (b, d) to its projection on the diagonal"""
    return 0.5 if math.isinf(p) else 2.0 ** (1.0 / p - 1.0)


def ground(e, p):
    """||e||_p over the last axis of e[..., 2]"""
    return np.linalg.norm(e, ord=p, axis=-1)


def selected(kind, mask, n):
    if kind is None:
        return np.ones(n, bool)
    k = np.asarray(kind, np.int64)
    return (k < 32) & (((int(mask) >> np.minimum(k, 31)) & 1) == 1)


def expansion(X, Y, q, p):
    """the square N = n' + m' problem of k8_wasserstein.cu over the nonzero-persistence points X [n', 2], Y [m', 2]:
    rows X then m' diagonal slots, columns Y then n' diagonal slots"""
    n, m = len(X), len(Y)
    C_ = np.zeros((n + m, n + m))
    if n and m:
        C_[:n, :m] = ground(X[:, None, :] - Y[None, :, :], p) ** q
    C_[:n, m:] = (np.abs(X[:, 1] - X[:, 0]) * kappa(p))[:, None] ** q
    C_[n:, :m] = (np.abs(Y[:, 1] - Y[:, 0]) * kappa(p))[None, :] ** q
    return C_


def ref_distance(X, Y, q=1.0, p=INF):
    """(distance, match_x, match_y) of one pair by the expansion and linear_sum_assignment; matches are local indices
    into X / Y, -1 the diagonal.  Zero-persistence points go to the diagonal outside the solve."""
    X, Y = np.reshape(X, (-1, 2)).astype(np.float64), np.reshape(Y, (-1, 2)).astype(np.float64)
    ix, iy = np.flatnonzero(X[:, 0] != X[:, 1]), np.flatnonzero(Y[:, 0] != Y[:, 1])
    mx, my = -np.ones(len(X), np.int64), -np.ones(len(Y), np.int64)
    if len(ix) + len(iy) == 0:
        return 0.0, mx, my
    C_ = expansion(X[ix], Y[iy], q, p)
    r, c = linear_sum_assignment(C_)
    n, m = len(ix), len(iy)
    for i, j in zip(r, c):
        if i < n and j < m:
            mx[ix[i]], my[iy[j]] = iy[j], ix[i]
    return float(C_[r, c].sum()) ** (1.0 / q), mx, my


def gudhi_lp(X, Y, q=1.0, p=INF):
    """gudhi's wasserstein_distance as it states the problem (all points, zero persistence included): the
    (n+1) x (m+1) transport with the diagonal's mass m on X's side and n on Y's, solved exactly by HiGHS"""
    X, Y = np.reshape(X, (-1, 2)).astype(np.float64), np.reshape(Y, (-1, 2)).astype(np.float64)
    n, m = len(X), len(Y)
    if n + m == 0:
        return 0.0
    M = np.zeros((n + 1, m + 1))
    if n and m:
        M[:n, :m] = ground(X[:, None, :] - Y[None, :, :], p) ** q
    M[:n, m] = (np.abs(X[:, 1] - X[:, 0]) * kappa(p)) ** q
    M[n, :m] = (np.abs(Y[:, 1] - Y[:, 0]) * kappa(p)) ** q
    a = np.concatenate([np.ones(n), [m]])
    b = np.concatenate([np.ones(m), [n]])
    A = np.zeros((n + 1 + m + 1, (n + 1) * (m + 1)))
    for i in range(n + 1):
        A[i, i * (m + 1):(i + 1) * (m + 1)] = 1.0
    for j in range(m + 1):
        A[n + 1 + j, j::m + 1] = 1.0
    res = linprog(M.reshape(-1), A_eq=A, b_eq=np.concatenate([a, b]), bounds=(0, None), method="highs")
    assert res.status == 0, res.message
    return max(float(res.fun), 0.0) ** (1.0 / q)


def matching_cost(X, Y, mx, q, p):
    """W of a matching given from X's side (local indices, -1 the diagonal); the Y points no X point takes go to the
    diagonal"""
    X, Y = np.reshape(X, (-1, 2)), np.reshape(Y, (-1, 2))
    taken = np.zeros(len(Y), bool)
    s = 0.0
    for k, j in enumerate(mx):
        if j >= 0:
            s += ground(X[k] - Y[j], p) ** q
            taken[j] = True
        else:
            s += (abs(X[k, 1] - X[k, 0]) * kappa(p)) ** q
    s += float(np.sum((np.abs(Y[~taken, 1] - Y[~taken, 0]) * kappa(p)) ** q))
    return s ** (1.0 / q)


def torch_wasserstein(bx, dx, by, dy, mx, my, q=1.0, p=INF):
    """gudhi's enable_autodiff branch (wasserstein.py) restated in torch for ONE pair at a given matching (local
    indices, -1 the diagonal, -2 masked out): the matched pairs' ||x - y||_p, the diagonal points' (d - b) 2^(1/p - 1),
    all of them in one torch.linalg.vector_norm of order q.  Differentiable in the four tensors."""
    mx, my = torch.as_tensor(mx), torch.as_tensor(my)
    xs = torch.nonzero(mx >= 0).reshape(-1)
    X = torch.stack([bx, dx], -1)
    Y = torch.stack([by, dy], -1)
    parts = []
    if xs.numel():
        parts.append(torch.linalg.vector_norm(Y[mx[xs]] - X[xs], p, dim=-1))
    for P_, m_ in ((X, mx), (Y, my)):
        dg = torch.nonzero(m_ == -1).reshape(-1)
        if dg.numel():
            parts.append((P_[dg, 1] - P_[dg, 0]) * kappa(p))
    if not parts:
        return (bx.sum() + dx.sum() + by.sum() + dy.sum()) * 0.0
    return torch.linalg.vector_norm(torch.cat(parts), q)


def random_diagram(rng, n, below=0.3, zero=0.1, dup=0.1, lattice=False):
    """n points: some below the diagonal, some of zero persistence, some duplicated"""
    if lattice:
        b = rng.integers(0, 4, n) / 4.0
        d = b + rng.integers(-2, 4, n) / 4.0
    else:
        b = rng.uniform(0, 1, n)
        d = b + rng.uniform(0, 1, n) * np.where(rng.random(n) < below, -1.0, 1.0)
    d = np.where(rng.random(n) < zero, b, d)
    X = np.stack([b, d], 1)
    if n > 1:
        k = rng.random(n) < dup
        X[k] = X[rng.integers(0, n, int(k.sum()))]
    return X


QP = [(q, p) for q in (1.0, 1.5, 2.0) for p in (1.0, 2.0, INF)]


@pytest.mark.parametrize("q,p", QP)
def test_expansion_equals_the_gudhi_transport_lp(q, p):
    rng = np.random.default_rng(int(10 * q + (3 if math.isinf(p) else p)))
    sizes = [(0, 0), (0, 5), (4, 0), (1, 1), (3, 7), (8, 8), (12, 5)]
    for trial in range(3):
        for n, m in sizes:
            lat = trial == 2
            X, Y = random_diagram(rng, n, lattice=lat), random_diagram(rng, m, lattice=lat)
            w, mx, my = ref_distance(X, Y, q, p)
            assert abs(w - gudhi_lp(X, Y, q, p)) <= 1e-9 * max(1.0, w), (n, m, trial)
            assert abs(matching_cost(X, Y, mx, q, p) - w) <= 1e-12 * max(1.0, w)
            for k in np.flatnonzero(X[:, 0] == X[:, 1]):
                assert mx[k] == -1  # zero persistence: the diagonal
            for k, j in enumerate(mx):  # my mirrors mx
                if j >= 0:
                    assert my[j] == k


@pytest.mark.parametrize("q,p", QP)
def test_closed_forms(q, p):
    rng = np.random.default_rng(5)
    X = random_diagram(rng, 9, zero=0.0)
    assert ref_distance(X, X, q, p)[0] == 0.0
    dx = np.abs(X[:, 1] - X[:, 0]) * kappa(p)
    w = ref_distance(np.zeros((0, 2)), X, q, p)[0]
    assert abs(w - np.sum(dx ** q) ** (1 / q)) <= 1e-13 * w
    for _ in range(20):
        x, y = rng.uniform(-1, 2, 2), rng.uniform(-1, 2, 2)
        want = min(ground(x - y, p) ** q, (abs(x[1] - x[0]) * kappa(p)) ** q + (abs(y[1] - y[0]) * kappa(p)) ** q)
        got = ref_distance(x, y, q, p)[0]
        assert abs(got - want ** (1 / q)) <= 1e-13 * max(got, 1e-300)


@pytest.mark.parametrize("q,p", QP)
def test_torch_restatement_value_and_gradient(q, p):
    """at the optimal matching the torch restatement gives the optimum, and its gradient is the closed form
    G (n / W)^(q-1) dn/d(b, d) stated in include/tlc_b200.h"""
    rng = np.random.default_rng(7)
    X, Y = random_diagram(rng, 6, zero=0.0, dup=0.0), random_diagram(rng, 8, zero=0.0, dup=0.0)
    w, mx, my = ref_distance(X, Y, q, p)
    t = [torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (X[:, 0], X[:, 1], Y[:, 0], Y[:, 1])]
    W = torch_wasserstein(*t, mx, my, q, p)
    assert abs(W.item() - w) <= 1e-13 * w
    W.backward()
    for k in range(len(X)):
        j = mx[k]
        e = X[k] - Y[j] if j >= 0 else None
        if j >= 0:
            n = ground(e, p)
            if math.isinf(p):
                g = np.sign(e) * (np.abs(e) == n) / np.sum(np.abs(e) == n)
            else:
                g = np.sign(e) * np.abs(e) ** (p - 1) / n ** (p - 1)
        else:
            n = abs(X[k, 1] - X[k, 0]) * kappa(p)
            s = np.sign(X[k, 1] - X[k, 0]) * kappa(p)
            g = np.array([-s, s])
        g = g * (n / w) ** (q - 1)
        assert np.allclose([t[0].grad[k].item(), t[1].grad[k].item()], g, rtol=1e-12, atol=1e-15), k


def test_torch_restatement_conventions():
    """zero-length difference -> 0, inf-norm tie split evenly, S = 0 -> 0, masked points (-2) -> 0"""
    f = lambda *a: torch.tensor(a, dtype=torch.float64, requires_grad=True)  # noqa: E731
    bx, dx, by, dy = f(0.0, 1.0), f(1.0, 3.0), f(0.0, 5.0), f(1.0, 5.0)
    W = torch_wasserstein(bx, dx, by, dy, [0, -2], [0, -1], 1.0, INF)
    W.backward()
    assert bx.grad.tolist() == [0.0, 0.0] and dx.grad.tolist() == [0.0, 0.0]  # x0 == y0; x1 masked
    assert by.grad.tolist() == [0.0, 0.0] and dy.grad.tolist() == [0.0, 0.0]  # y1 has zero persistence
    bx, dx, by, dy = f(0.0), f(1.0), f(2.0), f(3.0)
    torch_wasserstein(bx, dx, by, dy, [0], [0], 1.0, INF).backward()  # e = (-2, -2): a tie
    assert bx.grad.item() == -0.5 and dx.grad.item() == -0.5 and by.grad.item() == 0.5 and dy.grad.item() == 0.5
    bx, dx, by, dy = f(0.5), f(0.5), f(0.2), f(0.2)
    torch_wasserstein(bx, dx, by, dy, [-1], [-1], 2.0, 2.0).backward()  # S = 0
    assert bx.grad.item() == 0.0 and dy.grad.item() == 0.0


def test_workspace_query_follows_its_formula():
    lib = L.lib()
    out = C.c_uint64(7)
    for D, Px, Py in ((0, 0, 0), (1, 0, 0), (5, 100, 3), (1 << 20, 123456789, 987654321)):
        assert lib.tlc_wasserstein_workspace_bytes(D, Px, Py, C.byref(out)) == 0
        assert out.value == 64 * (Px + Py)
    for D, Px, Py in ((-1, 0, 0), (1 << 31, 0, 0), (1, -1, 0), (1, 0, -1), (1, 1 << 56, 0)):
        assert lib.tlc_wasserstein_workspace_bytes(D, Px, Py, C.byref(out)) == L.E_INVALID
    assert lib.tlc_wasserstein_workspace_bytes(1, 1, 1, None) == L.E_INVALID


BAD = [  # (D, order, internal_p, index of the NULL pointer among the six inputs or None, word the message names)
    (-1, 1.0, INF, None, "D"),
    (1 << 31, 1.0, INF, None, "D"),
    (2, 0.5, INF, None, "order"),
    (2, math.nan, INF, None, "order"),
    (2, INF, INF, None, "order"),
    (2, 1.0, 0.5, None, "internal_p"),
    (2, 1.0, math.nan, None, "internal_p"),
    (2, 1.0, -INF, None, "internal_p"),
] + [(2, 1.0, INF, k, w) for k, w in enumerate(["dev_poff_x", "dev_birth_x", "dev_death_x", "dev_poff_y",
                                                   "dev_birth_y", "dev_death_y"])]


def test_entry_points_reject_bad_arguments():
    lib = L.lib()
    fake = C.create_string_buffer(4096)  # never dereferenced: every check below fails first
    ptr = C.addressof(fake)
    Px, Py = 10, 20
    need = 64 * (Px + Py)
    for D, q, p, null, word in BAD:
        ins = [None if k == null else ptr for k in range(6)]
        xs, ys = ins[:3] + [None], ins[3:] + [None]
        assert lib.tlc_wasserstein_batch_dev(0, D, Px, Py, *xs, *ys, 1, q, p, ptr, need, ptr, ptr, ptr,
                                             None) == L.E_INVALID, word
        assert word in lib.tlc_last_error().decode(), word
        assert lib.tlc_wasserstein_batch_grad_dev(0, D, *xs, *ys, 1, q, p, ptr, ptr, ptr, ptr, ptr, ptr, ptr, ptr,
                                                  None) == L.E_INVALID, word
        assert word in lib.tlc_last_error().decode(), word
    xs = [ptr, ptr, ptr, None]
    fwd = lambda D, Px, Py, ws, nb, dist: lib.tlc_wasserstein_batch_dev(  # noqa: E731
        0, D, Px, Py, *xs, *xs, 1, 1.0, INF, ws, nb, dist, None, None, None)
    assert fwd(2, Px, Py, ptr, need - 1, ptr) == L.E_INVALID  # one byte too small
    assert "workspace" in lib.tlc_last_error().decode()
    assert fwd(2, Px, Py, None, need, ptr) == L.E_INVALID
    assert "dev_workspace" in lib.tlc_last_error().decode()
    assert fwd(2, Px, Py, ptr, need, None) == L.E_INVALID
    assert "dev_dist" in lib.tlc_last_error().decode()
    assert fwd(2, -1, Py, ptr, need, ptr) == L.E_INVALID
    grad = lambda dist, mx, my, g: lib.tlc_wasserstein_batch_grad_dev(  # noqa: E731
        0, 2, *xs, *xs, 1, 1.0, INF, dist, mx, my, g, ptr, ptr, ptr, ptr, None)
    for args, word in (((None, ptr, ptr, ptr), "dev_dist"), ((ptr, None, ptr, ptr), "dev_match_x"),
                       ((ptr, ptr, None, ptr), "dev_match_y"), ((ptr, ptr, ptr, None), "dev_grad_out")):
        assert grad(*args) == L.E_INVALID, word
        assert word in lib.tlc_last_error().decode(), word
    # nothing to do: no CUDA call, so these succeed without a device
    n4 = [None] * 4
    assert lib.tlc_wasserstein_batch_dev(0, 0, 0, 0, *n4, *n4, 1, 1.0, INF, None, 0, None, None, None, None) == 0
    assert lib.tlc_wasserstein_batch_grad_dev(0, 0, *n4, *n4, 1, 1.0, INF, *[None] * 8, None) == 0
    assert lib.tlc_wasserstein_batch_grad_dev(0, 2, *xs, *xs, 1, 1.0, INF, ptr, ptr, ptr, ptr, None, None, None, None,
                                              None) == 0


def cpu_inputs(P=6):
    return (torch.tensor([0, 2, P]), torch.rand(P, dtype=torch.float64), torch.rand(P, dtype=torch.float64),
            torch.zeros(P, dtype=torch.uint8))


@pytest.mark.parametrize("case", ["cpu", "poff_dtype", "birth_dtype", "death_y_dtype", "kind_dtype", "death_shape",
                                  "kind_y_shape", "birth_2d", "poff_empty", "poff_lengths", "death_strided",
                                  "mask_without_kind", "order_half", "order_nan", "order_inf", "p_half", "p_nan"])
def test_wasserstein_distances_checks_its_tensors_before_cuda(case, monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("a CUDA call was made")
    monkeypatch.setattr(api, "_wasserstein_fn", no_cuda)
    px, bx, dx, kx = cpu_inputs()
    py, by, dy, ky = cpu_inputs(9)
    kw = dict(kind_x=kx, kind_y=ky, kind_mask=1)
    err = ValueError
    if case == "poff_dtype":
        px, err = px.to(torch.int32), TypeError
    elif case == "birth_dtype":
        bx, err = bx.float(), TypeError
    elif case == "death_y_dtype":
        dy, err = dy.float(), TypeError
    elif case == "kind_dtype":
        kw["kind_x"], err = kx.to(torch.int32), TypeError
    elif case == "death_shape":
        dx = dx[:5]
    elif case == "kind_y_shape":
        kw["kind_y"] = torch.zeros(7, dtype=torch.uint8)
    elif case == "birth_2d":
        bx = bx.reshape(2, 3)
    elif case == "poff_empty":
        px = torch.zeros(0, dtype=torch.int64)
    elif case == "poff_lengths":
        py = torch.tensor([0, 9])
    elif case == "death_strided":
        dx = torch.rand(12, dtype=torch.float64)[::2]
    elif case == "mask_without_kind":
        kw = dict(kind_mask=1)
    elif case.startswith("order"):
        kw["order"] = {"order_half": 0.5, "order_nan": math.nan, "order_inf": INF}[case]
    elif case.startswith("p_"):
        kw["internal_p"] = {"p_half": 0.5, "p_nan": math.nan}[case]
    with pytest.raises(err):
        api.wasserstein_distances(px, bx, dx, py, by, dy, **kw)
