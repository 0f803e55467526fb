"""CPU tests of the cell / gene QC: oracle/oracle_qc.py against a literal dense restatement of
filter_cells, filter_genes, calc_vmr and normalize_count (R/utils.R:78-95,134-218,318-327), and the
host-side selection helpers of the front end (thresholds, markers, median) against the oracle."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_counts
from ccfindr_b200 import api
from oracle import oracle_qc as oq

GOLDEN = ("pbmc", "c1s1", "c1s2", "c1s3", "tiny")


class Obj:
    def __init__(self, X, rowData=None, colData=None):
        self.counts = sp.csc_matrix(X)
        n, m = self.counts.shape
        self.rowData = list(rowData) if rowData is not None else ["g%d" % i for i in range(n)]
        self.colData = list(colData) if colData is not None else ["c%d" % j for j in range(m)]


def dense_vmr(D):
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = D.mean(axis=1)
        return np.where(mean == 0, np.nan, D.var(axis=1, ddof=1) / mean)


def same_nan(a, b, rtol):
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    assert np.allclose(a[ok], b[ok], rtol=rtol, atol=0)


def check_csc_equal(A, B):
    A, B = sp.csc_matrix(A), sp.csc_matrix(B)
    assert A.shape == B.shape
    assert np.array_equal(A.indptr, B.indptr)
    assert np.array_equal(A.indices, B.indices)
    assert np.array_equal(A.data, B.data)


def with_extras(X):
    """X with an all-zero gene appended, and two explicit zeros stored in columns 0 and 1."""
    X = sp.vstack([sp.csc_matrix(X), sp.csc_matrix((1, X.shape[1]))]).tocsc()
    X.sort_indices()
    n = X.shape[0]
    C = X.tocoo()
    rows, cols, vals = list(C.row), list(C.col), list(C.data)
    rows += [n - 1, n - 1]; cols += [0, 1]; vals += [0.0, 0.0]
    Y = sp.csc_matrix((vals, (rows, cols)), shape=X.shape)  # coo -> csc keeps stored zeros
    Y.sort_indices()
    assert (Y.data == 0).sum() == 2
    return Y


def cases():
    out = [(name, load_counts(name)) for name in GOLDEN]
    out.append(("pbmc+zeros", with_extras(load_counts("pbmc"))))
    rng = np.random.default_rng(5)
    Xf = load_counts("c1s1").copy()
    Xf.data = Xf.data * rng.uniform(0.1, 3.0, size=Xf.nnz)  # non-integer counts
    out.append(("c1s1-real", Xf))
    return out


@pytest.mark.parametrize("name,X", cases(), ids=[c[0] for c in cases()])
def test_oracle_stats_and_vmr_match_dense(name, X):
    D = X.toarray()
    st = oq.stats(X)
    integer = np.all(X.data == np.round(X.data))
    for key, ref in (("cell_sum", D.sum(axis=0)), ("gene_sum", D.sum(axis=1)),
                     ("gene_sumsq", (D * D).sum(axis=1))):
        if integer:
            assert np.array_equal(st[key], ref), key
        else:
            assert np.allclose(st[key], ref, rtol=1e-12, atol=0), key
    assert np.array_equal(st["gene_cells"], (D > 0).sum(axis=1))
    assert np.array_equal(st["cell_genes"], (D > 0).sum(axis=0))
    same_nan(oq.calc_vmr(X), dense_vmr(D), 1e-12)
    # the front end's one-pass formula from the sums
    same_nan(api.vmr_from_sums(st["gene_sum"], st["gene_sumsq"], X.shape[1]), dense_vmr(D), 1e-9)


@pytest.mark.parametrize("name,X", cases(), ids=[c[0] for c in cases()])
def test_oracle_filters_match_dense(name, X):
    D = X.toarray()
    obj = Obj(X)
    umi = D.sum(axis=0)
    lo, hi = np.quantile(umi, 0.2), np.quantile(umi, 0.9)
    Y, rd, cd = oq.filter_cells(obj, umi_min=lo, umi_max=hi)
    keep = (umi >= lo) & (umi <= hi)
    assert np.array_equal(Y.toarray(), D[:, keep])
    assert cd == [c for c, k in zip(obj.colData, keep) if k] and rd == obj.rowData
    check_csc_equal(Y, X[np.arange(X.shape[0])][:, np.flatnonzero(keep)])

    vmr = dense_vmr(D)
    ncell = (D > 0).sum(axis=1)
    vmin = float(np.nanmedian(vmr))
    vmin = 0.5 * (vmin + np.nanmin(vmr[vmr > vmin]))  # between two genes' values
    Y, rd, cd = oq.filter_genes(obj, vmr_min=vmin, min_cells_expressed=3,
                                max_cells_expressed=X.shape[1] - 2)
    with np.errstate(invalid="ignore"):
        keep = (vmr > vmin) & (ncell >= 3) & (ncell <= X.shape[1] - 2)
    assert np.array_equal(Y.toarray(), D[keep])
    assert rd == [g for g, k in zip(obj.rowData, keep) if k] and cd == obj.colData
    check_csc_equal(Y, X[np.flatnonzero(keep)][:, np.arange(X.shape[1])])

    Y, rd, cd = oq.normalize_count(obj)
    med = np.median(umi)
    assert np.allclose(Y.toarray(), D * (med / umi)[None, :], rtol=1e-15, atol=0)
    assert Y.nnz == X.nnz and rd == obj.rowData and cd == obj.colData


@pytest.mark.parametrize("name,X", cases(), ids=[c[0] for c in cases()])
def test_front_end_selection_matches_oracle(name, X):
    """The host half of filter_cells / filter_genes / normalize_count on the oracle's sums."""
    obj = Obj(X)
    st = oq.stats(X)
    umi = st["cell_sum"]
    lo = float(np.sort(umi)[len(umi) // 3])
    Y, _, cd = oq.filter_cells(obj, umi_min=lo)
    keep = api.cell_mask(umi, umi_min=lo)
    assert cd == [c for c, k in zip(obj.colData, keep) if k]
    vmr = oq.calc_vmr(X)
    vmin = float(np.nanmedian(vmr))
    vmin = 0.5 * (vmin + np.nanmin(vmr[vmr > vmin]))
    markers = [obj.rowData[0], obj.rowData[-1]]
    _, rd, _ = oq.filter_genes(obj, markers=markers, vmr_min=vmin, min_cells_expressed=2)
    rows = api.gene_mask(api.vmr_from_sums(st["gene_sum"], st["gene_sumsq"], X.shape[1]),
                         st["gene_cells"], obj.rowData, markers, vmr_min=vmin,
                         min_cells_expressed=2)
    assert rd == [g for g, k in zip(obj.rowData, rows) if k]
    Y, _, _ = oq.normalize_count(obj)
    scale = api.normalize_scale(umi)
    col = np.repeat(np.arange(X.shape[1]), np.diff(X.indptr))
    assert np.array_equal(Y.data, X.data * scale[col])  # bitwise: the device multiply is the same


def test_explicit_zeros_and_empty_gene():
    X = with_extras(load_counts("tiny"))
    n = X.shape[0]
    st = oq.stats(X)
    assert st["gene_cells"][n - 1] == 0 and st["gene_sum"][n - 1] == 0
    assert st["cell_genes"][0] == (X[:, 0].toarray() > 0).sum()
    vmr = oq.calc_vmr(X)
    assert np.isnan(vmr[n - 1])
    assert np.isnan(api.vmr_from_sums(st["gene_sum"], st["gene_sumsq"], X.shape[1])[n - 1])
    obj = Obj(X)
    _, rd, _ = oq.filter_genes(obj, vmr_min=-1.0)
    assert obj.rowData[n - 1] not in rd and len(rd) == n - 1  # NaN fails vmr > vmr_min
    _, rd, _ = oq.filter_genes(obj, markers=[obj.rowData[n - 1]], vmr_min=-1.0)
    assert rd == obj.rowData
    # the stored zeros of a kept column survive the subset, as in scipy
    Y, _, _ = oq.filter_cells(obj)
    assert (Y.data == 0).sum() == 2


def test_boundaries_are_as_specified():
    # cells with totals 3, 5, 7: umi_min = 5 keeps the cell at 5, umi_max = 5 too
    X = sp.csc_matrix(np.array([[1.0, 2.0, 3.0], [2.0, 3.0, 4.0]]))
    obj = Obj(X)
    _, _, cd = oq.filter_cells(obj, umi_min=5)
    assert cd == ["c1", "c2"]
    assert list(api.cell_mask([3.0, 5.0, 7.0], umi_min=5)) == [False, True, True]
    _, _, cd = oq.filter_cells(obj, umi_min=5, umi_max=5)
    assert cd == ["c1"]
    # a gene with vmr exactly vmr_min is dropped: gene (0, 2, 0, 2): mean 1, var 4/3
    X = sp.csc_matrix(np.array([[0.0, 2.0, 0.0, 2.0], [1.0, 1.0, 1.0, 2.0]]))
    vmr = oq.calc_vmr(X)
    assert vmr[0] == 4.0 / 3.0
    _, rd, _ = oq.filter_genes(Obj(X), vmr_min=4.0 / 3.0)
    assert rd == []
    st = oq.stats(X)
    v = api.vmr_from_sums(st["gene_sum"], st["gene_sumsq"], 4)
    assert v[0] == 4.0 / 3.0
    assert not api.gene_mask(v, st["gene_cells"], ["a", "b"], vmr_min=4.0 / 3.0).any()


def test_marker_matching_on_one_and_two_field_rowdata():
    X = sp.csc_matrix(np.array([[0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [0.0, 5.0, 0.0]]))
    # one field per gene (ids)
    obj = Obj(X, rowData=["ENSG1", "ENSG2", "ENSG3"])
    _, rd, _ = oq.filter_genes(obj, markers=["ENSG1"], vmr_min=0)
    assert rd == ["ENSG1", "ENSG3"]  # ENSG2 has vmr 0, ENSG1 none (NaN) but is a marker
    assert list(api.marker_mask(obj.rowData, ["ENSG1"])) == [True, False, False]
    assert list(api.marker_mask(obj.rowData, "ENSG2")) == [False, True, False]
    # two fields (id, symbol): either matches
    obj = Obj(X, rowData=[("ENSG1", "CD3E"), ("ENSG2", "MS4A1"), ("ENSG3", "LYZ")])
    _, rd, _ = oq.filter_genes(obj, markers=["MS4A1"], vmr_min=0)
    assert rd == [("ENSG2", "MS4A1"), ("ENSG3", "LYZ")]
    assert list(api.marker_mask(obj.rowData, ["ENSG1", "LYZ"])) == [True, False, True]
    assert not api.marker_mask(obj.rowData, None).any()
    assert not api.marker_mask(obj.rowData, ["CD3"]).any()


def test_median_even_and_odd():
    assert oq.median([3.0, 1.0, 2.0]) == 2.0
    assert oq.median([4.0, 1.0, 3.0, 2.0]) == 2.5
    assert oq.median([1.0, 2.0]) == 1.5
    rng = np.random.default_rng(1)
    for k in (1, 2, 7, 10, 451):
        x = rng.uniform(1, 100, size=k)
        assert oq.median(x) == np.median(x)
        s = api.normalize_scale(x)
        assert np.array_equal(s, oq.median(x) / x)
    with pytest.raises(ValueError, match="empty columns"):
        api.normalize_scale([1.0, 0.0, 2.0])
    with pytest.raises(ValueError, match="empty columns"):
        oq.normalize_count(Obj(sp.csc_matrix(np.array([[1.0, 0.0], [1.0, 0.0]]))))
