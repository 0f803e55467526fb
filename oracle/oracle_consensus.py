"""NumPy restatement of the device consensus measures (vbnmf_consensus, csrc/consensus.cuh): the
moments S1, S2 of the co-clustering counts, the groups of cells with equal label tuples, their
integer cross-agreements IP and the greedy average-linkage merge list, once literally (O(G^3)) and
once with the per-row cache of the device loop (O(G^2) in practice).  Test infrastructure only.

L is nrun x m (one row of labels per run).  a_xy = runs in which cells x and y share a label."""
import numpy as np


def _choose2(x):
    x = np.asarray(x, dtype=np.int64)
    return int(np.sum(x * (x - 1) // 2))


def moments(L):
    """S1 = sum_{x<y} a_xy and S2 = sum_{x<y} a_xy^2, exact, from the label pairs of run pairs."""
    L = np.asarray(L, dtype=np.int64)
    nrun = L.shape[0]
    s1 = sum(_choose2(np.unique(L[t], return_counts=True)[1]) for t in range(nrun))
    cross = 0
    for t in range(nrun):
        for u in range(t + 1, nrun):
            cross += _choose2(np.unique(L[t] * (L[u].max() + 1) + L[u], return_counts=True)[1])
    return s1, s1 + 2 * cross


def moments_pairwise(L):
    """The same sums straight from the m(m-1)/2 pairs (small m)."""
    L = np.asarray(L)
    m = L.shape[1]
    iu = np.triu_indices(m, 1)
    a = sum((row[:, None] == row[None, :])[iu].astype(np.int64) for row in L)
    return int(a.sum()), int((a * a).sum())


def groups(L):
    """Distinct columns of L in the order of (L[0], L[1], ...): tuples (G x nrun), sizes (G)."""
    tup, cnt = np.unique(np.asarray(L).T, axis=0, return_counts=True)
    return tup, cnt.astype(np.int64)


def ip_matrix(tup, sizes):
    """IP_ab = n_a n_b #{t: T_at = T_bt} (G x G, int64; the diagonal is not used)."""
    agree = np.zeros((len(sizes), len(sizes)), dtype=np.int64)
    for t in range(tup.shape[1]):
        agree += tup[:, t][:, None] == tup[:, t][None, :]
    return sizes[:, None] * sizes[None, :] * agree


def _q(ip, nrun, na, nb):
    """q = IP / (nrun N_a N_b): both exact int64 values converted to fp64, one IEEE division."""
    return np.asarray(ip, dtype=np.int64).astype(np.float64) / \
        (np.int64(nrun) * np.asarray(na, dtype=np.int64) * np.asarray(nb, dtype=np.int64)).astype(np.float64)


def greedy_literal(ip, sizes, nrun):
    """G - 1 steps: the largest q over all active a < b (first of equals in row-major order, i.e.
    the smallest a, then the smallest b), merge b into a.  Returns merges ((G-1) x 5: a, b, IP_ab,
    N_a, N_b).  O(G^3)."""
    IP = np.array(ip, dtype=np.int64)
    N = np.array(sizes, dtype=np.int64)
    G = len(N)
    active = np.ones(G, dtype=bool)
    upper = np.triu(np.ones((G, G), dtype=bool), 1)
    out = []
    for _ in range(G - 1):
        Q = np.where(upper & active[:, None] & active[None, :], _q(IP, nrun, N[:, None], N[None, :]),
                     -np.inf)
        k = int(np.argmax(Q))
        a, b = divmod(k, G)
        out.append((a, b, int(IP[a, b]), int(N[a]), int(N[b])))
        IP[a, :] += IP[b, :]
        IP[:, a] = IP[a, :]
        N[a] += N[b]
        active[b] = False
    return np.array(out, dtype=np.int64).reshape(-1, 5)


def greedy_cached(ip, sizes, nrun):
    """The same merge list with the row cache of the device loop: best[k] = (q, b) over active
    b > k; after merging b into a only rows k < a (adopt a, or rescan when their best was a or b and
    q(k, a) fell below it), rows a < k < b whose best was b, and row a are touched.
    Returns (merges, rescans)."""
    IP = np.array(ip, dtype=np.int64)
    N = np.array(sizes, dtype=np.int64)
    G = len(N)
    active = np.ones(G, dtype=bool)
    bq = np.full(G, -1.0)
    bb = np.full(G, -1, dtype=np.int64)

    def scan(k):
        j = np.flatnonzero(active[k + 1:]) + k + 1
        if len(j) == 0:
            bq[k], bb[k] = -1.0, -1
            return
        q = _q(IP[k, j], nrun, N[k], N[j])
        i = int(np.argmax(q))
        bq[k], bb[k] = q[i], j[i]

    for k in range(G):
        scan(k)
    out, rescans = [], 0
    for _ in range(G - 1):
        rows = np.flatnonzero(active & (bb >= 0))
        a = int(rows[np.argmax(bq[rows])])        # first maximum: the smallest a
        b = int(bb[a])
        out.append((a, b, int(IP[a, b]), int(N[a]), int(N[b])))
        IP[a, :] += IP[b, :]
        IP[:, a] = IP[a, :]
        N[a] += N[b]
        active[b] = False
        bb[b] = -1
        ks = np.flatnonzero(active[:a])
        qn = _q(IP[ks, a], nrun, N[ks], N[a])
        was = (bb[ks] == a) | (bb[ks] == b)
        keep = qn >= bq[ks]
        adopt = (was & keep) | (~was & ((qn > bq[ks]) | ((qn == bq[ks]) & (a < bb[ks]))))
        bq[ks[adopt]], bb[ks[adopt]] = qn[adopt], a
        mid = np.flatnonzero(active[a + 1:b]) + a + 1
        redo = [a] + ks[was & ~keep].tolist() + mid[bb[mid] == b].tolist()
        for k in redo:
            scan(k)
        rescans += len(redo)
    return np.array(out, dtype=np.int64).reshape(-1, 5), rescans


def tree(L, cached=True):
    """(S1, S2, G, merges) of labels L."""
    L = np.asarray(L)
    s1, s2 = moments(L)
    tup, sz = groups(L)
    ip = ip_matrix(tup, sz)
    merges = greedy_cached(ip, sz, L.shape[0])[0] if cached else greedy_literal(ip, sz, L.shape[0])
    return s1, s2, len(sz), merges
