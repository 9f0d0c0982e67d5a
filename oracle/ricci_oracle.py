"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the curvature precompute the reference calls before the path
(SURVEY.md row N4):

    /root/reference/loaddatas.py:105-123   compute_ricci_curvature(data):
        Gd_OT = OllivierRicci(Gd, alpha=0.5, method="Sinkhorn", verbose="INFO"); Gd_OT.compute_ricci_curvature()
        ricci_list = sorted([[n1, n2, k], [n2, n1, k] for every edge])

PARITY UNPINNED.  The arithmetic lives in two third-party packages that are neither vendored in /root/reference nor
pinned in its requirements.txt, and neither is installed here (no network): `GraphRicciCurvature` (OllivierRicci) and
`POT` (ot.sinkhorn2).  This file restates their PUBLISHED algorithm (GraphRicciCurvature 0.5.3 OllivierRicci.py,
POT 0.8 ot/bregman.py sinkhorn_knopp) for the reference's call -- an unweighted nx.Graph, so every edge weight is 1:

  * mass distribution of a node x (`_get_single_node_neighbors_distributions`): neighbour weights base ** (-w ** exp_power)
    = e ** -1 each, normalised by their python sum() -> (1 - alpha) * e^-1 / (e^-1 added k times) on each of the k
    kept neighbours, alpha on x itself; only the nbr_topk = 3000 neighbours with the largest (weight, id) are kept (a
    heap of that size);
  * cost matrix d = all-pairs shortest path lengths between the two supports (`_apsp[np.ix_(src, tgt)]`): hop counts,
    0..3 for the supports of an edge;
  * m = ot.sinkhorn2(x, y, d, 1e-1, method='sinkhorn'): K = exp(d / -reg); u = 1/dim_a, v = 1/dim_b; repeat
    v = b / (K^T u), u = 1 / (Kp v) with Kp = K / a[:, None]; every 10th iteration err = || u * (K v) ... ||: the right
    marginal sum_i u_i K_ij v_j against b, stop when err <= 1e-9 or after 1000 iterations; loss = sum(u K v * d);
  * curvature = 1 - m / weight(x, y) = 1 - m.

It is pinned instead by closed forms of the exact transport problem on toy graphs (tests/test_ricci_oracle.py): the
entropic regularisation 0.1 against hop costs 0..3 (Gibbs factors 1, 4.5e-5, 2e-9, 9e-14) leaves the loss within 1e-2
of the exact optimum (measured 3e-3 .. 7e-3 on complete graphs).  Only tests/ may import this module.
"""
import numpy as np

ALPHA = 0.5
REG = 1e-1
NBR_TOPK = 3000
NUM_ITER_MAX = 1000
STOP_THR = 1e-9


def _neighbours(rowptr, col, x):
    return col[rowptr[x]:rowptr[x + 1]]


def support(rowptr, col, x, alpha=ALPHA, topk=NBR_TOPK):
    """(masses, node ids) of x's distribution: its (at most topk) neighbours, then x itself"""
    nb = np.asarray(_neighbours(rowptr, col, x), dtype=np.int64)
    if nb.size == 0:
        return np.array([1.0]), np.array([x], dtype=np.int64)
    if nb.size > topk:  # the heap keeps the topk largest (weight, id) tuples; all weights are equal here
        nb = np.sort(nb)[-topk:]
    w = np.full(nb.size, np.e ** (-1.0 ** 2))
    # The weights are normalised by their sum added left to right, one weight at a time: GraphRicciCurvature adds them
    # with python's sum(), which does exactly that on CPython <= 3.11 (the reference pins 3.7).  Neither numpy's
    # pairwise w.sum() nor the compensated sum() of CPython >= 3.12 gives the same bits for k = 120, 121, 1024, 3000.
    s = 0.0
    for t in w.tolist():
        s += t
    dist = (1.0 - alpha) * w / s
    return np.concatenate([dist, [alpha]]), np.concatenate([nb, [x]])


def hop_costs(rowptr, col, src, tgt):
    """hop distances between two node lists (0..3 is all an edge's supports can produce; larger ones by BFS)"""
    N = len(rowptr) - 1
    d = np.zeros((len(src), len(tgt)))
    tpos = {}
    for j, b in enumerate(tgt):
        tpos.setdefault(int(b), []).append(j)
    for i, a in enumerate(src):
        dist = np.full(N, -1, dtype=np.int64)
        dist[a] = 0
        frontier = [int(a)]
        left = len(set(int(b) for b in tgt) - {int(a)})
        depth = 0
        while frontier and left > 0:
            depth += 1
            nxt = []
            for x in frontier:
                for y in _neighbours(rowptr, col, x):
                    if dist[y] < 0:
                        dist[y] = depth
                        nxt.append(int(y))
                        if int(y) in tpos:
                            left -= 1
            frontier = nxt
        for b, js in tpos.items():
            for j in js:
                d[i, j] = dist[b] if dist[b] >= 0 else np.inf
    return d


def support_costs(rowptr, col, src, tgt):
    """hop_costs for the two supports of an edge, built from the sparse adjacency instead of one BFS per source: with
    B = A + I, the distance is 0 on the diagonal, 1 where B[a, b] > 0, 2 where (B B)[a, b] > 0, else 3.  Valid only
    where every distance is at most 3 -- true for an edge's supports (neighbour - x - y - neighbour)."""
    import scipy.sparse as sp
    N = len(rowptr) - 1
    A = sp.csr_matrix((np.ones(len(col)), np.asarray(col), np.asarray(rowptr)), shape=(N, N))
    B = (A + sp.identity(N, format="csr")).tocsr()
    src = np.asarray(src, dtype=np.int64)
    tgt = np.asarray(tgt, dtype=np.int64)
    bs, bt = B[src], B[tgt]
    one = bs[:, tgt].toarray() > 0
    two = (bs @ bt.T).toarray() > 0                    # B is symmetric: (B B)[src][:, tgt] = B[src] B[tgt]^T
    same = src[:, None] == tgt[None, :]
    return 3.0 - one - two - same


def sinkhorn2(a, b, M, reg=REG, num_iter_max=NUM_ITER_MAX, stop_thr=STOP_THR):
    """POT's sinkhorn_knopp loss for one pair of histograms (ot/bregman.py)"""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    M = np.asarray(M, dtype=np.float64)
    u = np.ones(len(a)) / len(a)
    v = np.ones(len(b)) / len(b)
    K = np.exp(M / (-reg))
    cpt, err = 0, 1.0
    with np.errstate(divide="ignore", invalid="ignore"):   # a zero mass (alpha = 0 or 1) ends the loop through inf * 0
        Kp = (1.0 / a).reshape(-1, 1) * K
        while err > stop_thr and cpt < num_iter_max:
            uprev, vprev = u, v
            KtU = K.T @ u
            v = b / KtU
            u = 1.0 / (Kp @ v)
            if (np.any(KtU == 0) or np.any(np.isnan(u)) or np.any(np.isnan(v)) or np.any(np.isinf(u))
                    or np.any(np.isinf(v))):
                u, v = uprev, vprev
                break
            if cpt % 10 == 0:
                tmp2 = np.einsum("i,ij,j->j", u, K, v)
                err = np.linalg.norm(tmp2 - b)
            cpt += 1
    return float(np.sum(u.reshape(-1, 1) * K * v.reshape(1, -1) * M)), cpt


def edge_curvature(rowptr, col, x, y):
    a, src = support(rowptr, col, x)
    b, tgt = support(rowptr, col, y)
    d = support_costs(rowptr, col, src, tgt)
    m, _ = sinkhorn2(a, b, d)
    return 1.0 - m / 1.0


def compute_ricci_curvature(rowptr, col):
    """curvature of every directed CSR entry (both directions of an edge carry the same value, loaddatas.py:117-121)"""
    rowptr = np.asarray(rowptr)
    col = np.asarray(col)
    N = len(rowptr) - 1
    out = np.zeros(len(col))
    done = {}
    for x in range(N):
        for e in range(rowptr[x], rowptr[x + 1]):
            y = int(col[e])
            key = (min(x, y), max(x, y))
            if key not in done:
                done[key] = edge_curvature(rowptr, col, key[0], key[1])
            out[e] = done[key]
    return out


def exact_w1(a, b, M):
    """exact optimal transport cost (linear programme, scipy): the closed-form side of the pinning tests"""
    from scipy.optimize import linprog
    na, nb = len(a), len(b)
    A_eq = np.zeros((na + nb, na * nb))
    for i in range(na):
        A_eq[i, i * nb:(i + 1) * nb] = 1.0
    for j in range(nb):
        A_eq[na + j, j::nb] = 1.0
    r = linprog(np.asarray(M).reshape(-1), A_eq=A_eq, b_eq=np.concatenate([a, b]), bounds=(0, None), method="highs")
    return float(r.fun)
