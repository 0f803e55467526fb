"""NumPy / scipy restatement of the cell and gene QC of ccfindR (R/utils.R:78-95,134-218,318-327):
filter_cells, filter_genes, calc_vmr and normalize_count, computed directly on the host (column and
row sums with scipy, a two-pass variance, scipy subsetting).  Test infrastructure: the GPU path is
compared against it; nothing under ccfindr_b200/ imports it.

Objects are anything with `counts` (scipy sparse, genes x cells), `rowData` and `colData` (lists);
the functions return (counts, rowData, colData) and leave their input untouched."""
import numpy as np
import scipy.sparse as sp


def stats(X):
    """cell_sum, gene_sum, gene_sumsq (fp64) and the entries with a non-zero value per gene and
    per cell (explicit stored zeros do not count, as R's counts > 0)."""
    X = sp.csc_matrix(X, dtype=np.float64)
    nz = X.copy()
    nz.data = (X.data != 0).astype(np.float64)
    return dict(cell_sum=np.asarray(X.sum(axis=0)).ravel(),
                gene_sum=np.asarray(X.sum(axis=1)).ravel(),
                gene_sumsq=np.asarray(X.multiply(X).sum(axis=1)).ravel(),
                gene_cells=np.asarray(nz.sum(axis=1)).ravel().astype(np.int64),
                cell_genes=np.asarray(nz.sum(axis=0)).ravel().astype(np.int64))


def median(x):
    """R's median: the middle value, or the mean of the two middle values for an even count."""
    s = np.sort(np.asarray(x, dtype=np.float64))
    k = len(s)
    return s[k // 2] if k % 2 else (s[k // 2 - 1] + s[k // 2]) / 2.0


def calc_vmr(X):
    """var / mean per gene over all m cells, zeros included; var with denominator m - 1, from the
    deviations of every cell (two passes); NaN where the mean is 0."""
    X = sp.csr_matrix(X, dtype=np.float64)
    n, m = X.shape
    out = np.empty(n)
    for i in range(n):
        vals = X.data[X.indptr[i]:X.indptr[i + 1]]
        mean = vals.sum() / m
        ss = ((vals - mean) ** 2).sum() + (m - len(vals)) * mean * mean
        out[i] = np.nan if mean == 0 else (ss / (m - 1)) / mean
    return out


def _subset(obj, gi, ci):
    X = sp.csc_matrix(obj.counts)
    return (X[gi][:, ci], [obj.rowData[i] for i in gi], [obj.colData[j] for j in ci])


def filter_cells(obj, umi_min=0, umi_max=np.inf):
    umi = stats(obj.counts)["cell_sum"]
    ci = np.flatnonzero((umi >= umi_min) & (umi <= umi_max))
    return _subset(obj, np.arange(obj.counts.shape[0]), ci)


def filter_genes(obj, markers=None, vmr_min=0, min_cells_expressed=0,
                 max_cells_expressed=np.inf):
    vmr = calc_vmr(obj.counts)
    ncells = stats(obj.counts)["gene_cells"]
    marks = set([markers] if isinstance(markers, str) else (markers or []))
    gi = []
    for i, g in enumerate(obj.rowData):
        fields = g if isinstance(g, (tuple, list)) else (g,)
        ok = (not np.isnan(vmr[i]) and vmr[i] > vmr_min
              and min_cells_expressed <= ncells[i] <= max_cells_expressed)
        if ok or any(f in marks for f in fields):
            gi.append(i)
    return _subset(obj, np.array(gi, dtype=np.int64), np.arange(obj.counts.shape[1]))


def normalize_count(obj):
    X = sp.csc_matrix(obj.counts, dtype=np.float64)
    umi = stats(X)["cell_sum"]
    if (umi == 0).any():
        raise ValueError("Input matrix contains empty columns")
    scale = median(umi) / umi
    col = np.repeat(np.arange(X.shape[1]), np.diff(X.indptr))
    Y = sp.csc_matrix((X.data * scale[col], X.indices.copy(), X.indptr.copy()), shape=X.shape)
    return (Y, list(obj.rowData), list(obj.colData))
