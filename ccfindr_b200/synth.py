"""Synthetic count matrices for tests and benchmarks.

simulate_whx() follows the recipe of the reference's simulate_whx (R/utils.R:826-846):
w ~ Gamma(shape=aw, scale=bw/aw), h ~ Gamma(shape=ah, scale=bh/ah), x ~ Poisson(w.h), empty
rows/columns dropped.  R's RNG stream cannot be reproduced without R, so the draws come from a
NumPy Philox generator keyed by `seed`.

tenx_like() is the 10x-shaped generator of SURVEY.md section 8(d): W, H ~ Gamma(0.3, mean 1),
per-cell depth ~ LogNormal(0, 0.5), x ~ Poisson(s * d_j * (W H)_ij) with the scalar s bisected to
hit a target nonzero fraction; sampling runs on the GPU in column chunks with one Philox stream
per chunk, so that a shard of cells generated on one GPU equals the same columns of the
single-GPU matrix.
"""
import numpy as np
import scipy.sparse as sp


def _rng(seed, stream=0):
    return np.random.Generator(np.random.Philox(key=[int(seed), int(stream)]))


def simulate_whx(nrow, ncol, rank, aw=0.1, bw=1.0, ah=0.1, bh=1.0, seed=1):
    """R/utils.R:826-846.  Returns dict(w, h, x) with x a dense float64 count matrix."""
    g = _rng(seed)
    # R fills matrix(rgamma(n*rank), nrow, rank) column-major; only the distribution matters here
    w = g.gamma(shape=aw, scale=bw / aw, size=(rank, nrow)).T.copy()
    h = g.gamma(shape=ah, scale=bh / ah, size=(ncol, rank)).T.copy()
    x = g.poisson(w @ h).astype(np.float64)
    i = x.sum(axis=1) > 0
    j = x.sum(axis=0) > 0
    return dict(w=w[i], h=h[:, j], x=x[i][:, j])


def random_init(nrow, ncol, rank, hyper, seed):
    """vb_init(initializer='random') (R/bayesian.R:111-115): w ~ Gamma(aw, scale bw/aw),
    h ~ Gamma(ah, scale bh/ah), from a NumPy Philox stream."""
    g = _rng(seed, stream=1)
    w = g.gamma(shape=hyper["aw"], scale=hyper["bw"] / hyper["aw"], size=(rank, nrow)).T.copy()
    h = g.gamma(shape=hyper["ah"], scale=hyper["bh"] / hyper["ah"], size=(ncol, rank)).T.copy()
    return w, h


def uniform_init(nrow, ncol, rank, seed):
    """init() of the ML path (R/factorize.R:30-38): w, h ~ U(0,1)."""
    g = _rng(seed, stream=2)
    return g.random(size=(rank, nrow)).T.copy(), g.random(size=(ncol, rank)).T.copy()


def fix_empty(csc, seed=0):
    """Give every empty row/column one count at a random position (the API rejects empties,
    R/bayesian.R:244-247)."""
    csc = csc.tocsc()
    n, m = csc.shape
    g = _rng(seed, stream=3)
    er = np.flatnonzero(np.asarray(csc.sum(axis=1)).ravel() == 0)
    ec = np.flatnonzero(np.asarray(csc.sum(axis=0)).ravel() == 0)
    if len(er) == 0 and len(ec) == 0:
        return csc
    rows = np.concatenate([er, g.integers(0, n, size=len(ec))])
    cols = np.concatenate([g.integers(0, m, size=len(er)), ec])
    add = sp.csc_matrix((np.ones(len(rows)), (rows, cols)), shape=(n, m))
    out = (csc + add).tocsc()
    out.sort_indices()
    return out


# ---- 10x-shaped generator (SURVEY.md section 8d), sampled on the GPU ------------------------
TENX_CHUNK = 4000  # cells per Philox stream; shard boundaries must be multiples of this


def tenx_factors(n, m, r_true, seed):
    """Host-side latent factors of the generator: W, H ~ Gamma(shape 0.3, mean 1) and per-cell
    depth ~ LogNormal(0, 0.5), all m cells (so that any shard slices the same draw)."""
    g = _rng(seed, stream=10)
    W = g.gamma(shape=0.3, scale=1.0 / 0.3, size=(n, r_true)).astype(np.float32)
    H = g.gamma(shape=0.3, scale=1.0 / 0.3, size=(m, r_true)).astype(np.float32)  # cell-major
    d = g.lognormal(mean=0.0, sigma=0.5, size=m).astype(np.float32)
    return W, H, d


def tenx_scale(W, H, d, density, seed, device):
    """Scalar s such that the nonzero fraction of Poisson(s d_j (W H)_ij) is `density`:
    bisection on mean(1 - exp(-s d_j (WH)_ij)) over a fixed sample of 2048 cells."""
    import torch
    g = _rng(seed, stream=11)
    m = H.shape[0]
    cols = np.sort(g.choice(m, size=min(2048, m), replace=False))
    Wt = torch.from_numpy(W).to(device=device, dtype=torch.float64)
    Ht = torch.from_numpy(H[cols]).to(device=device, dtype=torch.float64)
    dt = torch.from_numpy(d[cols]).to(device=device, dtype=torch.float64)
    lam = (Ht @ Wt.T) * dt[:, None]
    lo, hi = 0.0, 1.0
    while float((1.0 - torch.exp(-hi * lam)).mean()) < density:
        hi *= 2.0
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        if float((1.0 - torch.exp(-mid * lam)).mean()) < density:
            lo = mid
        else:
            hi = mid
    return 0.5 * (lo + hi)


def tenx_like_device(n, m, r_true, density, seed, device, col_start=0, col_end=None):
    """CSC arrays (torch CUDA tensors: colptr int64, rowidx int32, values float32) of columns
    [col_start, col_end) of the synthetic n x m matrix G(n, m, r_true, density, seed).
    col_start must be a multiple of TENX_CHUNK (one Philox stream per chunk of cells)."""
    import torch
    col_end = m if col_end is None else col_end
    assert col_start % TENX_CHUNK == 0
    W, H, d = tenx_factors(n, m, r_true, seed)
    s = tenx_scale(W, H, d, density, seed, device)
    Wt = torch.from_numpy(W).to(device)
    rows, vals, counts = [], [], []
    for c0 in range(col_start, col_end, TENX_CHUNK):
        c1 = min(c0 + TENX_CHUNK, col_end, m)
        Hc = torch.from_numpy(H[c0:c1]).to(device)
        dc = torch.from_numpy(d[c0:c1]).to(device) * float(s)
        lam = (Hc @ Wt.T) * dc[:, None]                      # cells x genes
        gen = torch.Generator(device=device)
        gen.manual_seed((int(seed) << 32) + c0 // TENX_CHUNK)
        x = torch.poisson(lam, generator=gen)
        # a cell without counts gets one (SURVEY.md 8d: the API rejects empty columns)
        empty = torch.nonzero(x.sum(dim=1) == 0).flatten()
        if empty.numel():
            x[empty, (empty + c0) % n] = 1.0
        nz = torch.nonzero(x)                                # sorted by (cell, gene) = CSC order
        rows.append(nz[:, 1].to(torch.int32))
        vals.append(x[nz[:, 0], nz[:, 1]].to(torch.float32))
        counts.append(torch.bincount(nz[:, 0], minlength=c1 - c0))
        del lam, x, nz
    rowidx = torch.cat(rows)
    values = torch.cat(vals)
    del rows, vals
    cnt = torch.cat(counts)
    colptr = torch.zeros(cnt.numel() + 1, dtype=torch.int64, device=device)
    colptr[1:] = torch.cumsum(cnt, 0)
    return colptr, rowidx, values, s


def tenx_expected_nnz(n, m, r_true, density, seed, device):
    """Expected number of nonzeros of every TENX_CHUNK-cell chunk of G(n, m, r_true, density,
    seed): sum_ij (1 - exp(-s d_j (W H)_ij)).  Cheap (no sampling) and identical on every rank:
    the basis of the nnz-balanced shard boundaries of a multi-GPU run."""
    import torch
    W, H, d = tenx_factors(n, m, r_true, seed)
    s = tenx_scale(W, H, d, density, seed, device)
    Wt = torch.from_numpy(W).to(device)
    out = []
    for c0 in range(0, m, TENX_CHUNK):
        c1 = min(c0 + TENX_CHUNK, m)
        Hc = torch.from_numpy(H[c0:c1]).to(device)
        dc = torch.from_numpy(d[c0:c1]).to(device) * float(s)
        lam = (Hc @ Wt.T) * dc[:, None]
        out.append(float((1.0 - torch.exp(-lam)).sum(dtype=torch.float64)))
    return np.array(out)


# ---- CPU restatement of the on-device 'random' initialiser (csrc/kernels_common.cuh) ---------
_M64 = (1 << 64) - 1


def _mix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


class _Stream:
    """splitmix64 counter stream of one matrix entry (VbStream)."""

    def __init__(self, seed, ident):
        self.s = _mix64(seed & _M64) ^ _mix64((ident + 0x632BE59BD9B4E019) & _M64)

    def next(self):
        self.s = (self.s + 0x9E3779B97F4A7C15) & _M64
        return _mix64(self.s)

    def uniform(self):
        return (float(self.next() >> 11) + 0.5) * (1.0 / 9007199254740992.0)

    def normal(self):
        u1, u2 = self.uniform(), self.uniform()
        return np.sqrt(-2.0 * np.log(u1)) * np.cos(6.283185307179586476925 * u2)

    def gamma(self, a):
        a1 = a + 1.0 if a < 1.0 else a
        d = a1 - 1.0 / 3.0
        c = 1.0 / np.sqrt(9.0 * d)
        g = 0.0
        for _ in range(1000):
            x = self.normal()
            v0 = 1.0 + c * x
            u = self.uniform()
            if v0 <= 0.0:
                continue
            v = v0 * v0 * v0
            if np.log(u) < 0.5 * x * x + d - d * v + d * np.log(v):
                g = d * v
                break
        if a < 1.0:
            g *= self.uniform() ** (1.0 / a)
        return g


def device_random_init_reference(nrow, ncol, rank, hyper, seed, cell_offset=0):
    """What Engine.init_random(rank, hyper, seed, cell_offset) puts on the device: w (nrow x rank),
    h (rank x ncol).  Pure-Python loops: small cases only."""
    w = np.zeros((nrow, rank))
    h = np.zeros((rank, ncol))
    for i in range(nrow):
        for k in range(rank):
            w[i, k] = hyper["bw"] / hyper["aw"] * _Stream(seed, (0 << 62) | (i << 6) | k).gamma(hyper["aw"])
    for j in range(ncol):
        for k in range(rank):
            ident = (1 << 62) | ((j + cell_offset) << 6) | k
            h[k, j] = hyper["bh"] / hyper["ah"] * _Stream(seed, ident).gamma(hyper["ah"])
    return w, h


def orient_svd_pairs(u, v):
    """The orientation Engine.init_svd applies before the 'svd' formula: for every k >= 1,
    (u_k, v_k) -> (-u_k, -v_k) when |u_k-| |v_k-| > |u_k+| |v_k+| (norms of the negative and
    positive parts); ties and component 0 are kept.  Returns new arrays."""
    u, v = np.array(u, dtype=np.float64), np.array(v, dtype=np.float64)
    for k in range(1, u.shape[1]):
        P = np.linalg.norm(np.maximum(u[:, k], 0)) * np.linalg.norm(np.maximum(v[:, k], 0))
        N = np.linalg.norm(np.minimum(u[:, k], 0)) * np.linalg.norm(np.minimum(v[:, k], 0))
        if N > P:
            u[:, k], v[:, k] = -u[:, k], -v[:, k]
    return u, v


def device_svd_init_reference(u, d, v):
    """What Engine.init_svd puts on the device for the truncated SVD (u n x r, d, v m x r):
    orient_svd_pairs, then the reference formula (api.svd_init_from).  Returns w, h."""
    from .api import svd_init_from
    u, v = orient_svd_pairs(u, v)
    return svd_init_from(u, np.asarray(d, dtype=np.float64), v)


# ---- CPU restatement of the on-device column shuffle (csrc/shuffle.cuh) ----------------------
_GOLDEN = np.uint64(0x9E3779B97F4A7C15)


def _mix64_np(z):
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _umulhi(u, n):
    """(u * n) >> 64 for a uint64 array u and 0 < n < 2^31, computed on the 32-bit halves of u
    (exact: hi * n + (lo * n >> 32) < 2^64)."""
    n = np.uint64(n)
    hi, lo = u >> np.uint64(32), u & np.uint64(0xFFFFFFFF)
    return (hi * n + ((lo * n) >> np.uint64(32))) >> np.uint64(32)


def _shuffle_draws(seed, j, count):
    """u_0 .. u_{count-1} of column j: the first `count` next() of VbStream(seed, 3 << 62 | j)."""
    s0 = np.uint64(_Stream(seed, (3 << 62) | int(j)).s)
    with np.errstate(over="ignore"):
        return _mix64_np(s0 + np.arange(1, count + 1, dtype=np.uint64) * _GOLDEN)


def shuffle_rows(seed, j, n, k):
    """s_0 .. s_{k-1}: the first k distinct rows umulhi(u_t, n) among the draws of column j."""
    if k > n:
        raise ValueError("a column holds more entries than there are rows")
    if k == 0:
        return np.zeros(0, dtype=np.int64)
    # expected draws for k distinct of n: n (H_n - H_{n-k}) <= k + k^2 / (n - k); the batch is
    # doubled until it holds k distinct rows (for k close to n the k^2 term is capped)
    nb = k + min(k * k // max(n - k, 1), 8 * k) + 64
    while True:
        with np.errstate(over="ignore"):
            r = _umulhi(_shuffle_draws(seed, j, nb), n)
        _, first = np.unique(r, return_index=True)
        if len(first) >= k:
            return r[np.sort(first)[:k]].astype(np.int64)
        nb *= 2


def shuffle_columns_reference(csc, seed):
    """What Engine.shuffle(seed) holds: each column of `csc` shuffled over the rows
    (factorize(randomize=TRUE), R/factorize.R:172-173).  indptr is kept; the t-th stored entry of
    column j (stored zeros included, ascending source row) goes to row
    shuffle_rows(seed, j, n, k)[t], and every column is sorted by row."""
    X = sp.csc_matrix(csc)
    if not X.has_sorted_indices:
        X = X.copy()
        X.sort_indices()
    n, m = X.shape
    rows = np.empty(X.nnz, dtype=np.int32)
    vals = np.empty(X.nnz, dtype=np.float64)
    for j in range(m):
        b, e = int(X.indptr[j]), int(X.indptr[j + 1])
        s = shuffle_rows(seed, j, n, e - b)
        o = np.argsort(s)
        rows[b:e] = s[o]
        vals[b:e] = X.data[b:e][o]
    return sp.csc_matrix((vals, rows, X.indptr.copy()), shape=(n, m))
