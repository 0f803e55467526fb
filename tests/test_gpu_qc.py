"""GPU tests of the cell / gene QC: Engine.qc_stats and Engine.subset (csrc/qc.cuh) against the
NumPy / scipy restatement in oracle/oracle_qc.py, and the front end (filter_cells, filter_genes,
calc_vmr, normalize_count) against the same oracle and the reference driver."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_counts, relerr
from oracle import oracle_qc as oq

pytestmark = pytest.mark.gpu

HYPER = dict(aw=1.0, bw=1.0, ah=1.0, bh=1.0)
STAT_KEYS = ("cell_sum", "gene_sum", "gene_sumsq")
COUNT_KEYS = ("gene_cells", "cell_genes")


def with_zeros(X):
    """X with an all-zero gene appended that stores explicit zeros in the first two cells."""
    n, m = X.shape
    C = sp.csc_matrix(X).tocoo()
    Y = sp.csc_matrix((np.concatenate([C.data, [0.0, 0.0]]),
                       (np.concatenate([C.row, [n, n]]), np.concatenate([C.col, [0, 1]]))),
                      shape=(n + 1, m))  # coo -> csc keeps stored zeros
    Y.sort_indices()
    return Y


def fp64_counts(X):
    """A few integer counts that fp32 cannot hold exactly (above 2^24): the handle keeps the counts
    in fp64.  Few enough that every gene's sum of squares stays below 2^53 (exact)."""
    Y = sp.csc_matrix(X, copy=True)
    Y.data[::997] += 16777216.0
    return Y


def real_counts(X, seed=4):
    Y = sp.csc_matrix(X, copy=True)
    Y.data = Y.data * np.random.default_rng(seed).uniform(0.1, 3.0, size=Y.nnz)
    return Y


def check_stats(st, ref, exact):
    for k in STAT_KEYS:
        if exact:
            assert np.array_equal(st[k], ref[k]), k
        else:
            assert relerr(st[k], ref[k]) <= 1e-12, k
    for k in COUNT_KEYS:
        assert st[k].dtype == np.int64 and np.array_equal(st[k], ref[k]), k


def check_csc_equal(A, B):
    assert A.shape == B.shape
    assert np.array_equal(A.indptr, B.indptr)
    assert np.array_equal(A.indices, B.indices)
    assert np.array_equal(A.data, B.data)


def host_subset(X, rows, cols, scale):
    Y = sp.csc_matrix(X)[np.flatnonzero(rows)][:, np.flatnonzero(cols)]
    if scale is not None:
        sc = scale[np.flatnonzero(cols)]
        Y = sp.csc_matrix((Y.data * sc[np.repeat(np.arange(Y.shape[1]), np.diff(Y.indptr))],
                           Y.indices, Y.indptr), shape=Y.shape)
    return Y


# ---- 1. statistics ------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["pbmc", "c1s1", "c1s2", "c1s3", "tiny"])
@pytest.mark.parametrize("kind", ["int", "int-fp64", "zeros", "real"])
def test_qc_stats_match_oracle(name, kind):
    from ccfindr_b200.engine import Engine
    X = load_counts(name)
    X = {"int": X, "int-fp64": fp64_counts(X), "zeros": with_zeros(X), "real": real_counts(X)}[kind]
    exact = kind != "real"
    with Engine(X) as eng:
        st = eng.qc_stats()
        check_stats(st, oq.stats(X), exact)
        if exact:  # repeatable bit for bit
            again = eng.qc_stats()
            assert all(np.array_equal(again[k], st[k]) for k in STAT_KEYS)


def c2_device_matrix():
    import torch
    from ccfindr_b200 import synth
    dev = torch.device("cuda", 0)
    colptr, rowidx, values, _ = synth.tenx_like_device(20000, 100000, 10, 0.08, 2, dev)
    X = sp.csc_matrix((values.cpu().numpy().astype(np.float64), rowidx.cpu().numpy(),
                       colptr.cpu().numpy()), shape=(20000, 100000))
    return (colptr, rowidx, values), X


def test_qc_stats_and_subset_at_c2_size():
    """20k genes x 100k cells (~1.6e8 nonzeros) generated on the device: sums bitwise equal to
    scipy's, counts exact; a ~90 % subset equals scipy's X[gi][:, ci]."""
    from ccfindr_b200.engine import Engine
    (colptr, rowidx, values), X = c2_device_matrix()
    n, m = X.shape
    with Engine.from_device_csc(n, m, X.nnz, colptr, rowidx, values) as eng:
        st = eng.qc_stats()
        check_stats(st, oq.stats(X), exact=True)
        rng = np.random.default_rng(9)
        rows, cols = rng.random(n) < 0.9, rng.random(m) < 0.9
        with eng.subset(rows, cols) as sub:
            check_csc_equal(sub.csc(), host_subset(X, rows, cols, None))
            check_stats(sub.qc_stats(), oq.stats(host_subset(X, rows, cols, None)), exact=True)


# ---- 2. subset ----------------------------------------------------------------------------------
def masks(X, seed=1):
    n, m = X.shape
    rng = np.random.default_rng(seed)
    D = X.toarray()
    one_col = np.zeros(m, bool); one_col[m // 2] = True
    one_row = np.zeros(n, bool); one_row[int(np.argmax((D > 0).sum(axis=1)))] = True
    # keep the genes of one cell only: other cells lose every entry (empty cells)
    few_rows = D[:, 0] > 0
    # keep a handful of cells: some genes are left without entries (empty genes)
    few_cols = np.zeros(m, bool); few_cols[:3] = True
    return {
        "all": (np.ones(n, bool), np.ones(m, bool)),
        "halves": (rng.random(n) < 0.5, rng.random(m) < 0.5),
        "one_row": (one_row, np.ones(m, bool)),
        "one_col": (np.ones(n, bool), one_col),
        "empty_cells": (few_rows, np.ones(m, bool)),
        "empty_genes": (np.ones(n, bool), few_cols),
    }


@pytest.mark.parametrize("name,kind", [("pbmc", "int"), ("c1s1", "zeros"), ("tiny", "int"),
                                       ("c1s3", "int-fp64"), ("c1s2", "real")])
@pytest.mark.parametrize("scaled", [False, True])
def test_subset_matches_scipy(name, kind, scaled):
    from ccfindr_b200._lib import VbnmfError
    from ccfindr_b200.engine import Engine
    X = load_counts(name)
    X = {"int": X, "int-fp64": fp64_counts(X), "zeros": with_zeros(X), "real": real_counts(X)}[kind]
    n, m = X.shape
    scale = np.random.default_rng(2).uniform(0.2, 5.0, size=m) if scaled else None
    with Engine(X) as eng:
        for label, (rows, cols) in masks(X).items():
            ref = host_subset(X, rows, cols, scale)
            with eng.subset(rows, cols, scale) as sub:
                assert (sub.n, sub.m, sub.nnz) == ref.shape + (ref.nnz,), label
                check_csc_equal(sub.csc(), ref)
                check_stats(sub.qc_stats(), oq.stats(ref), exact=kind != "real" and not scaled)
                D = ref.toarray()
                empty = ((D > 0).sum(axis=1) == 0).any() or ((D > 0).sum(axis=0) == 0).any()
                r = min(2, min(ref.shape))
                w0 = np.ones((ref.shape[0], r)); h0 = np.ones((r, ref.shape[1]))
                if empty:
                    with pytest.raises(VbnmfError, match="empty"):
                        sub.set_state(w0, h0)
                    continue
                sub.set_state(w0, h0)
                with Engine(ref) as host:
                    host.set_state(w0, h0)
                    assert sub.layout_info() == host.layout_info(), label
        check_csc_equal(eng.csc(), sp.csc_matrix(X))  # the source is left as it was


def test_subset_value_format_follows_the_kept_values():
    """fp64 source whose only non-fp32 values are dropped: the subset is fp32 / packed-16 like
    Engine(host subset); a scale that makes values inexact in fp32 gives fp64."""
    from ccfindr_b200.engine import Engine
    X = sp.csc_matrix(load_counts("tiny"), copy=True)
    n, m = X.shape
    nnz_gene = X.getnnz(axis=1)
    j = next(j for j in range(m) if (nnz_gene - (X[:, j].toarray().ravel() > 0)).min() > 0)
    X.data[X.indptr[j]:X.indptr[j + 1]] += 0.1
    cols = np.ones(m, bool); cols[j] = False
    rows = np.ones(n, bool)
    with Engine(X) as eng:
        for scale, fmt in ((None, "p16"), (np.full(m, 1.0 / 3.0), "f64"), (np.full(m, 0.5), "f32")):
            ref = host_subset(X, rows, cols, scale)
            r = 2
            w0 = np.ones((ref.shape[0], r)); h0 = np.ones((r, ref.shape[1]))
            with eng.subset(rows, cols, scale) as sub, Engine(ref) as host:
                sub.set_state(w0, h0); host.set_state(w0, h0)
                assert sub.layout_info()["format"] == host.layout_info()["format"]
                # (0.5 x small integers is exact in fp32 but not an integer: the 8-byte format)
                assert sub.layout_info()["format"] == fmt


# ---- 3. errors ----------------------------------------------------------------------------------
def test_subset_errors():
    from ccfindr_b200._lib import VbnmfError
    from ccfindr_b200.engine import Engine
    X = sp.csc_matrix(np.array([[1.0, 0.0, 2.0], [0.0, 3.0, 0.0]]))
    with Engine(X) as eng:
        t2, t3 = np.ones(2, bool), np.ones(3, bool)
        with pytest.raises(VbnmfError):
            eng.subset(np.zeros(2, bool), t3)
        with pytest.raises(VbnmfError):
            eng.subset(t2, np.zeros(3, bool))
        with pytest.raises(VbnmfError, match="no entries"):
            eng.subset(np.array([False, True]), np.array([True, False, True]))
        for bad in ((np.ones(3, bool), t3), (t2, np.ones(2, bool)), (t2.astype(int), t3)):
            with pytest.raises(ValueError):
                eng.subset(*bad)
        with pytest.raises(ValueError):
            eng.subset(t2, t3, np.ones(2))
        with pytest.raises(ValueError):
            eng.subset(t2, t3, np.array([1.0, np.inf, 1.0]))
        with eng.subset(t2, t3) as sub:  # the engine still works after the refusals
            check_csc_equal(sub.csc(), X)


# ---- 4. residency -------------------------------------------------------------------------------
def test_device_resident_subset_runs_bit_for_bit(tmp_path):
    from ccfindr_b200 import api
    from ccfindr_b200.engine import Engine
    X = load_counts("pbmc")
    api.write_10x(api.scNMFSet(X), str(tmp_path))
    n, m = X.shape
    rng = np.random.default_rng(3)
    rows, cols = rng.random(n) < 0.8, rng.random(m) < 0.8
    for _ in range(5):  # no empty genes or cells left: set_state accepts the subset
        rows &= X[:, np.flatnonzero(cols)].getnnz(axis=1) > 0
        cols &= X[np.flatnonzero(rows)].getnnz(axis=0) > 0
    ref = host_subset(X, rows, cols, None)
    assert ref.getnnz(axis=1).min() > 0 and ref.getnnz(axis=0).min() > 0

    def run(eng):
        eng.init_random(3, HYPER, seed=17)
        res = eng.run(HYPER, Itmax=40)
        return res, eng.get_state(("ew", "eh"))

    with Engine.from_mtx(tmp_path / "matrix.mtx") as src:
        before = run(src)
        with src.subset(rows, cols) as sub:
            got = run(sub)
        after = run(src)
    with Engine(ref) as host:
        want = run(host)
    for a, b in ((got, want), (after, before)):
        assert a[0]["lml"] == b[0]["lml"]
        assert np.array_equal(a[0]["lkh_trace"], b[0]["lkh_trace"])
        assert np.array_equal(a[1]["ew"], b[1]["ew"]) and np.array_equal(a[1]["eh"], b[1]["eh"])


# ---- 5. front end -------------------------------------------------------------------------------
def pbmc_object(tmp_path):
    from ccfindr_b200 import api
    X = load_counts("pbmc")
    n, m = X.shape
    obj = api.scNMFSet(X, rowData=[("ENSG%05d" % i, "SYM%d" % i) for i in range(n)],
                       colData=[("CELL%d-1" % j,) for j in range(m)])
    api.write_10x(obj, str(tmp_path))
    return api.read_10x(str(tmp_path))


def check_object(obj, ref):
    Y, rd, cd = ref
    check_csc_equal(obj.counts, sp.csc_matrix(Y))
    assert obj.rowData == rd and obj.colData == cd


def test_front_end_matches_oracle(tmp_path):
    from ccfindr_b200 import api
    obj = pbmc_object(tmp_path)
    X0 = obj.counts.copy()
    umi = oq.stats(obj.counts)["cell_sum"]
    lo, hi = float(np.sort(umi)[40]), float(np.sort(umi)[-30])   # boundaries at cells' totals
    check_object(api.filter_cells(obj, umi_min=lo, umi_max=hi), oq.filter_cells(obj, lo, hi))
    check_object(api.filter_cells(obj), oq.filter_cells(obj))
    vmr_ref = oq.calc_vmr(obj.counts)
    vmr = api.calc_vmr(obj)
    assert np.array_equal(np.isnan(vmr), np.isnan(vmr_ref))
    assert relerr(vmr[~np.isnan(vmr)], vmr_ref[~np.isnan(vmr_ref)]) < 1e-10
    s = np.sort(vmr_ref[~np.isnan(vmr_ref)])
    vmin = 0.5 * (s[len(s) // 2] + s[len(s) // 2 + 1])
    markers = [obj.rowData[0][0], obj.rowData[5][1], "NOT-A-GENE"]
    kw = dict(markers=markers, vmr_min=vmin, min_cells_expressed=5, max_cells_expressed=400)
    check_object(api.filter_genes(obj, **kw), oq.filter_genes(obj, **kw))
    check_object(api.normalize_count(obj), oq.normalize_count(obj))
    check_csc_equal(obj.counts, X0)  # the input is untouched


def test_vignette_chain_equals_oracle_filtered(tmp_path):
    from ccfindr_b200 import api, synth
    obj = pbmc_object(tmp_path)
    umi = oq.stats(obj.counts)["cell_sum"]
    lo = float(np.sort(umi)[60])
    vmr = oq.calc_vmr(obj.counts)
    s = np.sort(vmr[~np.isnan(vmr)])
    vmin = 0.5 * (s[len(s) // 3] + s[len(s) // 3 + 1])
    a = api.remove_zeros(api.filter_genes(api.filter_cells(obj, umi_min=lo), vmr_min=vmin,
                                          min_cells_expressed=3))
    Y, rd, cd = oq.filter_cells(obj, umi_min=lo)
    Y, rd, cd = oq.filter_genes(api.scNMFSet(Y, rd, cd), vmr_min=vmin, min_cells_expressed=3)
    b = api.remove_zeros(api.scNMFSet(Y, rd, cd))
    check_object(a, (b.counts, b.rowData, b.colData))
    n, m = a.counts.shape
    inits = {(1, r): synth.random_init(n, m, r, HYPER, 50 + r) for r in (2, 3)}
    ra = api.vb_factorize(a, ranks=[2, 3], nrun=1, verbose=0, inits=inits, Itmax=60)
    rb = api.vb_factorize(b, ranks=[2, 3], nrun=1, verbose=0, inits=inits, Itmax=60)
    assert np.array_equal(ra.measure["lml"], rb.measure["lml"])
    for k in range(2):
        assert np.array_equal(ra.basis[k], rb.basis[k])
        assert np.array_equal(ra.coeff[k], rb.coeff[k])


def test_vb_factorize_on_normalized_counts_matches_reference_driver(tmp_path):
    from ccfindr_b200 import api, synth
    from oracle import bindings as ob
    obj = api.normalize_count(pbmc_object(tmp_path))
    assert not np.all(obj.counts.data == np.round(obj.counts.data))
    n, m = obj.counts.shape
    w0, h0 = synth.random_init(n, m, 3, HYPER, 7)
    s = api.vb_factorize(obj, ranks=[3], nrun=1, verbose=0, inits={(1, 3): (w0, h0)}, Itmax=50)
    ref = ob.sparse_vb_run(obj.counts, w0, h0, HYPER, Itmax=50)
    assert relerr(s.measure["lml"], [ref["lml"]]) < 1e-9
    assert relerr(s.basis[0], ref["ew"]) < 1e-9 and relerr(s.coeff[0], ref["eh"]) < 1e-9
