"""Host-side mirror of the ccfindR interface for the accelerated path.

The reference's host code is R; R is not installed here, so this mirror is Python with the same
function names, argument meaning and error behaviour (the R `.Call` shim that binds the same C ABI
ships as source in r-shim/).  What runs where:

    vb_factorize()   R/bayesian.R:229-301  validation, run/rank loops, best-run selection, slots:
                                           here;  the it-loop of vb_iterate (:336-352), the update
                                           (src/vbnmf_update.cpp) and hyper_update (:2-53): in
                                           libvbnmf.so on the GPU (Engine.run)
    factorize()      R/factorize.R:139-276 loops and measures here; the it-loop (:189-212) with
                                           nmf_updateR + likelihood on the GPU (Engine.ml_run);
                                           with device_shuffle=True the null matrices of
                                           randomize (:172-173) on the GPU too (Engine.shuffle);
                                           with device_consensus=True dispersion and the
                                           cophenetic correlation (:51-78) too (engine.consensus)
    cluster_id()     R/utils.R:903-909     first-maximum argmax per cell (GPU: Engine.cluster_id)
    optimal_rank()   R/utils2.R:59-95      host post-processing of measure (smoothing spline)
    filter_cells(), filter_genes(), calc_vmr(), normalize_count()
                     R/utils.R:78-95,134-218,318-327  thresholds, marker matching and the median
                                           here; the per-cell / per-gene sums and the subset /
                                           scale of the matrix on the GPU (Engine.qc_stats,
                                           Engine.subset)

There is no CPU fallback: every factorization needs libvbnmf.so and a CUDA device.
"""
import warnings

import numpy as np
import scipy.sparse as sp

from . import synth
from ._lib import ERR_HYPER, ERR_MEMORY, VbnmfError
from .engine import EPS, Engine


class scNMFSet:
    """The slots of the reference's scNMFSet that this path reads and fills
    (R/scNMF_class.R:66-71): counts (genes x cells), ranks, basis, dbasis, coeff, dcoeff, measure."""

    def __init__(self, count=None, rowData=None, colData=None):
        if count is None:
            raise ValueError("count matrix required")
        self.counts = sp.csc_matrix(count, dtype=np.float64)
        self.counts.sort_indices()
        self.rowData = list(rowData) if rowData is not None else list(range(1, self.counts.shape[0] + 1))
        self.colData = list(colData) if colData is not None else list(range(1, self.counts.shape[1] + 1))
        self.ranks = []
        self.basis, self.dbasis, self.coeff, self.dcoeff = [], [], [], []
        self.measure = None  # dict of columns, like the data.frame of R/bayesian.R:297-298
        self.metadata = {}

    def nrow(self):
        return self.counts.shape[0]

    def ncol(self):
        return self.counts.shape[1]

    def __repr__(self):
        return "scNMFSet(%d genes x %d cells, ranks=%s)" % (self.nrow(), self.ncol(), self.ranks)


def remove_zeros(object):
    """R/scNMF_class.R:636-656: drop genes and cells without any count."""
    mat = object.counts
    gi = np.flatnonzero(np.asarray(mat.sum(axis=1)).ravel() > 0)
    ci = np.flatnonzero(np.asarray(mat.sum(axis=0)).ravel() > 0)
    if len(gi) == mat.shape[0] and len(ci) == mat.shape[1]:
        return object
    out = scNMFSet(mat[gi][:, ci], rowData=[object.rowData[i] for i in gi],
                   colData=[object.colData[j] for j in ci])
    return out


# ---- cell / gene QC (R/utils.R:78-95,134-218,318-327): statistics and subsetting on the GPU -------
def vmr_from_sums(gene_sum, gene_sumsq, m):
    """Variance-to-mean ratio per gene over all m cells, zeros included: var is R's var
    (denominator m - 1), mean = S1 / m; a gene with mean 0 gets NaN (R's 0 / 0)."""
    s1 = np.asarray(gene_sum, dtype=np.float64)
    s2 = np.asarray(gene_sumsq, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = s1 / m
        var = (s2 - s1 * s1 / m) / (m - 1)
        return np.where(mean == 0, np.nan, var / mean)


def cell_mask(cell_sum, umi_min=0, umi_max=np.inf):
    """filter_cells: cells with umi_min <= total count <= umi_max."""
    cell_sum = np.asarray(cell_sum)
    return (cell_sum >= umi_min) & (cell_sum <= umi_max)


def marker_mask(rowData, markers):
    """Genes of which some field of rowData (the id or symbol of genes.tsv) is in markers."""
    if markers is None:
        return np.zeros(len(rowData), dtype=bool)
    mset = {markers} if isinstance(markers, str) else set(markers)
    return np.array([any(f in mset for f in (g if isinstance(g, (tuple, list)) else (g,)))
                     for g in rowData], dtype=bool)


def gene_mask(vmr, gene_cells, rowData, markers=None, vmr_min=0, min_cells_expressed=0,
              max_cells_expressed=np.inf):
    """filter_genes: vmr > vmr_min (NaN fails) with min <= cells expressed <= max, or a marker."""
    gene_cells = np.asarray(gene_cells)
    keep = (np.asarray(vmr) > vmr_min) & (gene_cells >= min_cells_expressed) \
        & (gene_cells <= max_cells_expressed)
    return keep | marker_mask(rowData, markers)


def normalize_scale(cell_sum):
    """normalize_count: the factor median(cell_sum) / cell_sum[j] of every cell, in fp64 (the
    median of an even number of cells is the mean of the two middle values, as R's)."""
    cell_sum = np.asarray(cell_sum, dtype=np.float64)
    if (cell_sum == 0).any():
        raise ValueError("Input matrix contains empty columns")
    return np.median(cell_sum) / cell_sum


def _qc_subset(object, device, select):
    """Statistics of object.counts on the GPU, select(stats) -> (keep_rows, keep_cols, col_scale),
    the subset built on the GPU and returned as a new scNMFSet (counts, rowData, colData)."""
    with Engine(object.counts, device=device) as eng:
        rows, cols, scale = select(eng.qc_stats())
        with eng.subset(rows, cols, scale) as sub:
            mat = sub.csc()
    return scNMFSet(mat, rowData=[g for g, k in zip(object.rowData, rows) if k],
                    colData=[c for c, k in zip(object.colData, cols) if k])


def calc_vmr(object, device=0):
    """calc_vmr (R/utils.R:134-218): variance-to-mean ratio of every gene over all cells (sums on
    the GPU).  NaN for a gene without counts."""
    with Engine(object.counts, device=device) as eng:
        st = eng.qc_stats()
    return vmr_from_sums(st["gene_sum"], st["gene_sumsq"], object.ncol())


def filter_cells(object, umi_min=0, umi_max=np.inf, device=0):
    """filter_cells (R/utils.R:78-95): a new scNMFSet with the cells whose total count lies in
    [umi_min, umi_max].  The defaults keep every cell (they are not the reference's defaults,
    which are not restated here).  Totals and the subset are computed on the GPU."""
    def select(st):
        return np.ones(object.nrow(), dtype=bool), cell_mask(st["cell_sum"], umi_min, umi_max), None
    return _qc_subset(object, device, select)


def filter_genes(object, markers=None, vmr_min=0, min_cells_expressed=0,
                 max_cells_expressed=np.inf, device=0):
    """filter_genes (R/utils.R:134-218, without rescue.genes): a new scNMFSet with the genes whose
    VMR exceeds vmr_min and which have a non-zero count in between min_cells_expressed and
    max_cells_expressed cells, plus every gene with a field of its rowData in `markers`.
    Statistics and the subset are computed on the GPU."""
    def select(st):
        vmr = vmr_from_sums(st["gene_sum"], st["gene_sumsq"], object.ncol())
        rows = gene_mask(vmr, st["gene_cells"], object.rowData, markers, vmr_min,
                         min_cells_expressed, max_cells_expressed)
        return rows, np.ones(object.ncol(), dtype=bool), None
    return _qc_subset(object, device, select)


def normalize_count(object, device=0):
    """normalize_count (R/utils.R:318-327): a new scNMFSet with every cell's counts scaled by
    median(cell totals) / its total.  The factors are computed in fp64 on the host from totals
    summed on the GPU; the scaled matrix is built on the GPU.  An empty cell raises ValueError."""
    def select(st):
        return (np.ones(object.nrow(), dtype=bool), np.ones(object.ncol(), dtype=bool),
                normalize_scale(st["cell_sum"]))
    return _qc_subset(object, device, select)


def read_10x(dir, count="matrix.mtx", genes="genes.tsv", barcodes="barcodes.tsv",
             remove_zeros_=True, device=None):
    """R/utils.R:28-54: MatrixMarket counts + gene / barcode tables -> scNMFSet whose counts are
    CSC (the dgCMatrix of :34), ready for the device upload without densification.
    device=<CUDA ordinal>: the text of matrix.mtx is parsed and sorted into CSC on the GPU
    (Engine.from_mtx) instead of by scipy on the host."""
    import os
    import scipy.io
    if not os.path.isdir(dir):
        raise FileNotFoundError("Input directory %s does not exist" % dir)
    for f in (count, genes, barcodes):
        if not os.path.exists(os.path.join(dir, f)):
            raise FileNotFoundError("Count file %s does not exist" % os.path.join(dir, f))
    if device is not None:
        with Engine.from_mtx(os.path.join(dir, count), device=device) as eng:
            mat = eng.csc()
    else:
        mat = sp.csc_matrix(scipy.io.mmread(os.path.join(dir, count)), dtype=np.float64)
    glist = [ln.split() for ln in open(os.path.join(dir, genes)) if ln.strip()]
    clist = [ln.split() for ln in open(os.path.join(dir, barcodes)) if ln.strip()]
    if len(glist) != mat.shape[0] or len(clist) != mat.shape[1]:
        raise ValueError("annotation tables do not match the matrix dimensions")
    x = scNMFSet(mat, rowData=[tuple(g) for g in glist], colData=[tuple(c) for c in clist])
    return remove_zeros(x) if remove_zeros_ else x


def write_10x(object, dir, count="matrix.mtx", genes="genes.tsv", barcodes="barcodes.tsv"):
    """R/utils.R:867-884."""
    import os
    import scipy.io
    scipy.io.mmwrite(os.path.join(dir, count), sp.coo_matrix(object.counts), field="integer"
                     if np.all(object.counts.data == np.round(object.counts.data)) else "real")
    with open(os.path.join(dir, genes), "w") as f:
        for g in object.rowData:
            f.write(" ".join(str(v) for v in (g if isinstance(g, (tuple, list)) else (g,))) + "\n")
    with open(os.path.join(dir, barcodes), "w") as f:
        for c in object.colData:
            f.write(" ".join(str(v) for v in (c if isinstance(c, (tuple, list)) else (c,))) + "\n")
    return object


def _check_no_empty(mat):
    """R/bayesian.R:242-247, R/factorize.R:147-150."""
    if int((np.asarray(mat.sum(axis=1)).ravel() == 0).sum()) > 0:
        raise ValueError("Input matrix contains empty rows")
    if int((np.asarray(mat.sum(axis=0)).ravel() == 0).sum()) > 0:
        raise ValueError("Input matrix contains empty columns")


def vb_init(nrow, ncol, mat, rank, hyper, initializer, seed):
    """R/bayesian.R:109-171.  'random' draws from NumPy's Philox stream (R's RNG stream cannot be
    reproduced without R); 'svd' and 'svd2' follow the reference formulas on a truncated SVD."""
    if initializer == "random":
        return synth.random_init(nrow, ncol, rank, hyper, seed)
    if initializer not in ("svd", "svd2"):
        raise ValueError("Unknown initializer")
    from scipy.sparse.linalg import svds
    if min(nrow, ncol) / 2 <= rank or min(nrow, ncol) - 1 <= rank:
        u, d, vt = np.linalg.svd(np.asarray(mat.todense()), full_matrices=False)
        u, d, vt = u[:, :rank], d[:rank], vt[:rank]
    else:
        u, d, vt = svds(mat.astype(np.float64), k=rank, random_state=np.random.default_rng(seed))
        o = np.argsort(-d)
        u, d, vt = u[:, o], d[o], vt[o]
    v = vt.T
    if initializer == "svd2":                                   # :150-159
        w = np.abs(u)
        h = np.abs(np.diag(d) @ v.T)
        scale = hyper["bh"] / h.mean()
        return w / scale, h * scale
    return svd_init_from(u, d, v)


def svd_init_from(u, d, v):
    """The 'svd' initializer (R/bayesian.R:116-149) from a truncated SVD: u n x r, d (r), v m x r.
    Returns w (n x r), h (r x m).  Literal, including the typo of :136-137."""
    nrow, ncol, rank = u.shape[0], v.shape[0], len(d)
    w = np.zeros((nrow, rank))
    h = np.zeros((rank, ncol))
    d1 = np.sqrt(d[0])
    w[:, 0] = d1 * u[:, 0]
    sgn = np.sign(w[0, 0])
    if sgn < 0:
        w = -w
    h[0, :] = sgn * d1 * v[:, 0]
    for k in range(1, rank):
        x, y = u[:, k], v[:, k]
        xp, yp = np.where(x > 0, x, 0.0), np.where(y > 0, y, 0.0)
        xn, yn = np.where(x < 0, -x, 0.0), np.where(y < 0, -y, 0.0)
        xpnrm, ypnrm = np.sqrt((xp ** 2).sum()), np.sqrt((yp ** 2).sum())
        mp = xpnrm * ypnrm
        xnnrm, ynnrm = np.sqrt((xp ** 2).sum()), np.sqrt((yp ** 2).sum())  # sic, :136-137 use xp, yp
        mn = xnnrm * ynnrm
        if mp >= mn:
            uu, vv, sig = xp / xpnrm, yp / ypnrm, mp
        else:
            uu, vv, sig = xn / xnnrm, yn / ynnrm, mn
        w[:, k] = np.sqrt(d[k] * sig) * uu
        h[k, :] = np.sqrt(d[k] * sig) * vv
    return w, h


def dispersion_from_labels(label_runs):
    """dispersion(conav/irun, ncol) of R/factorize.R:51-67 without the m(m-1)/2 connectivity vector:
    cells are grouped by their tuple of cluster labels over the runs; two cells are co-clustered in
    t runs iff their tuples agree in t positions.  Cost: (distinct tuples)^2, not cells^2."""
    L = np.stack([np.asarray(v) for v in label_runs], axis=1)
    nc, nrun = L.shape
    tup, cnt = np.unique(L, axis=0, return_counts=True)
    cnt = cnt.astype(np.float64)
    con = float(np.sum(cnt * (cnt - 1.0) / 2.0)) * 0.25        # same tuple: (1 - 0.5)^2
    G = len(tup)
    step = max(1, int(4e6 // max(G, 1)))
    for a0 in range(0, G, step):                                # blocks of rows of the G x G table
        blk = tup[a0:a0 + step]
        same = np.zeros((len(blk), G))
        for t in range(nrun):
            same += blk[:, t][:, None] == tup[:, t][None, :]
        wgt = cnt[a0:a0 + step][:, None] * cnt[None, :]
        mask = np.arange(a0, a0 + len(blk))[:, None] < np.arange(G)[None, :]   # pairs a < b once
        con += float(np.sum(np.where(mask, wgt * (same / nrun - 0.5) ** 2, 0.0)))
    return 1.0 / nc + 8.0 * con / nc ** 2


def lpt_schedule(costs, nworkers):
    """Longest-processing-time-first assignment of independent jobs to workers.
    Returns a list (one per worker) of job indices, each in decreasing cost order."""
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    load = [0.0] * nworkers
    out = [[] for _ in range(nworkers)]
    for i in order:
        w = min(range(nworkers), key=lambda k: (load[k], k))
        out[w].append(i)
        load[w] += costs[i]
    return out


def vb_factorize(object, ranks=2, nrun=1, verbose=2, progress_bar=True, initializer="random",
                 Itmax=10000, hyper_update=(True,) * 4, gamma_a=1, gamma_b=1, Tol=1e-5,
                 hyper_update_n0=10, hyper_update_dn=1, connectivity=True, fudge=None, ncores=1,
                 useC=True, unif_stop=True, seed=1, device=0, inits=None, precision=0,
                 parallel=False, device_init=False, shard_cells=False, device_consensus=False):
    """Bayesian NMF inference of a count matrix (R/bayesian.R:229-301).

    Arguments as in the reference (dots replaced by underscores).  Extras: `seed` keys the NumPy
    Philox streams of the 'random' initializer (run i, rank r uses seed*100003 + 1000*r + i);
    `inits[(irun, rank)] = (w0, h0)` overrides the draw; `device` is the CUDA ordinal.
    `ncores` and `useC` are accepted and ignored: the update always runs on the GPU.
    `precision`: 0 = fp64 (reference arithmetic), 1 = fp32-storage / fp64-accumulate.
    `device_init=True`: the 'random' initializer is drawn on the GPU (Engine.init_random, a counter
    RNG keyed by seed and matrix position) and the 'svd2' and 'svd' initializers are computed on
    the GPU (Engine.init_svd2, Engine.init_svd: randomized truncated SVD of the resident matrix)
    instead of on the host and uploaded.  'svd' on the GPU orients each pair of singular vectors
    k >= 1 before the reference formula (vbnmf_init_svd in include/vbnmf.h).
    `parallel=True` (inside an initialised torch.distributed job, one process per GPU): the
    nrun x len(ranks) independent factorizations are spread over the ranks (the role of
    Rmpi::mpi.applyLB, R/bayesian.R:263), every rank holds a full copy of the matrix, results are
    all-gathered and every rank returns the same object.
    `shard_cells=True` (same setting): ONE factorization at a time on all GPUs -- every rank keeps
    an nnz-balanced contiguous range of the cells on its GPU, the W-side statistics are all-reduced
    once per iteration (SURVEY.md 8e), and the coeff / dcoeff columns are gathered at the end, so
    every rank returns the same full object.  For matrices that do not fit one GPU, or to cut the
    time of one large factorization.
    `device_consensus=True`: the dispersion printed with `connectivity` is computed on the GPU from
    exact integer moments of the label runs (consensus_from_labels) instead of on the host.
    """
    if fudge is None:
        fudge = EPS                                             # :238
    mat = object.counts                                         # :239
    if initializer in ("svd", "svd2") and nrun > 1:
        raise ValueError("SVD initializer does not require nrun > 1")  # :241-242
    _check_no_empty(mat)                                        # :244-247
    nrow, ncol = mat.shape
    ranks = [int(r) for r in np.atleast_1d(ranks) if r <= ncol]  # :249
    nrank = len(ranks)
    ga = np.atleast_1d(np.asarray(gamma_a, dtype=np.float64))
    gb = np.atleast_1d(np.asarray(gamma_b, dtype=np.float64))

    if device_init and initializer not in ("random", "svd", "svd2"):
        raise ValueError("device_init applies to the 'random', 'svd' and 'svd2' initializers")
    if device_init:
        initializer += "_device"
    common = (ga, gb, initializer, Itmax, hyper_update, Tol, hyper_update_n0, hyper_update_dn,
              connectivity, fudge, device_consensus)
    vb = []
    if parallel and shard_cells:
        raise ValueError("parallel (independent jobs per GPU) and shard_cells (one job on all GPUs) "
                         "are alternatives")
    if shard_cells:
        vb = _vb_sharded(mat, ranks, nrun, common, unif_stop, verbose, seed, inits, device,
                         precision)
    elif parallel:
        vb = _vb_parallel(mat, ranks, nrun, common, unif_stop, verbose, seed, inits, device,
                          precision)
    else:
        with Engine(mat, device=device) as eng:
            eng.set_precision(precision)
            for irun in range(1, nrun + 1):                     # lapply over runs, :260-261
                vb.append(_vb_iterate(eng, irun, mat, ranks, *common, unif_stop, nrun, verbose,
                                      seed, inits, vb))

    basis = [None] * nrank
    coeff, dbasis, dcoeff = [None] * nrank, [None] * nrank, [None] * nrank
    cols = {k: [] for k in ("rank", "lml", "aw", "bw", "ah", "bh", "nunif")}
    for k in range(nrank):                                      # :268-292
        rmax, imax = -np.inf, None
        for i in range(nrun):
            if vb[i]["rdat"][k] > rmax:                         # strict >: the first of equals wins
                imax, rmax = i, vb[i]["rdat"][k]
        if rmax == -np.inf:
            continue
        cols["rank"].append(ranks[k]); cols["lml"].append(rmax)
        basis[k], coeff[k] = vb[imax]["wdat"][k], vb[imax]["hdat"][k]
        dbasis[k], dcoeff[k] = vb[imax]["dwdat"][k], vb[imax]["dhdat"][k]
        for key in ("aw", "bw", "ah", "bh"):
            cols[key].append(vb[imax]["hyperp"][k][key])
        cols["nunif"].append(vb[imax]["nunif"][k])
    # (extra, not in the reference: iterations each run took, for throughput accounting)
    object.metadata["niter"] = {(i + 1, ranks[k]): int(vb[i]["niter"][k]) for i in range(nrun)
                                for k in range(nrank) if vb[i]["hyperp"][k] is not None}
    object.ranks = cols["rank"]                                 # :293-299
    object.basis, object.dbasis = basis, dbasis
    object.coeff, object.dcoeff = coeff, dcoeff
    object.measure = {k: np.array(v) for k, v in cols.items()}
    return object


def dist_comm(device):
    """A libvbnmf NCCL communicator over the ranks of the initialised torch.distributed group:
    rank 0 makes the unique id, the group broadcasts it (the role Rmpi would play for the R shim)."""
    import torch
    import torch.distributed as dist
    from .engine import Comm
    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("needs an initialised torch.distributed process group")
    world, me = dist.get_world_size(), dist.get_rank()
    box = [Engine.nccl_unique_id() if me == 0 else None]
    dist.broadcast_object_list(box, src=0)
    return Comm(world, me, box[0], device=device)


def _vb_sharded(mat, ranks, nrun, common, unif_stop, verbose, seed, inits, device, precision):
    """vb_iterate for every run with the cells sharded over the ranks of torch.distributed."""
    import torch.distributed as dist
    from . import sharding
    from .engine import set_host_threads
    comm = dist_comm(device)
    world, me = comm.nranks, comm.rank
    b = sharding.balanced_bounds(mat.indptr, world)
    c0, c1 = b[me], b[me + 1]
    if c1 <= c0:
        raise ValueError("more GPUs than cells to shard")
    vb = []
    try:
        with Engine(sharding.shard_csc(mat, c0, c1), device=device) as eng:
            eng.set_precision(precision)
            eng.attach_comm(comm)
            for irun in range(1, nrun + 1):
                out = _vb_iterate(eng, irun, mat, ranks, *common, unif_stop, nrun,
                                  verbose if me == 0 else 0, seed, inits, vb, cols=(c0, c1))
                # coeff / dcoeff: this rank's columns -> all columns on every rank
                parts = [None] * world
                dist.all_gather_object(parts, (out["hdat"], out["dhdat"]))
                for k in range(len(ranks)):
                    if out["hdat"][k] is not None:
                        out["hdat"][k] = np.concatenate([p[0][k] for p in parts], axis=1)
                        out["dhdat"][k] = np.concatenate([p[1][k] for p in parts], axis=1)
                vb.append(out)
    finally:
        comm.close()
    return vb


def jobs_to_keep(scalars, nrun, nrank):
    """(irun, k) of the jobs whose factor matrices the aggregation can still ask for: the best run
    of every rank index k -- strict >, the first of equals (R/bayesian.R:271) -- or every job when
    one raised the uniform-column flag (the rank scan of that run then breaks, R/bayesian.R:370-378,
    and what is best depends on the run order).  scalars[(irun, k)] = dict(rdat=..., unif=...)."""
    if any(res["unif"] for res in scalars.values()):
        return set(scalars)
    keep = set()
    for k in range(nrank):
        rmax, imax = -np.inf, None
        for irun in range(1, nrun + 1):
            if scalars[(irun, k)]["rdat"] > rmax:
                imax, rmax = irun, scalars[(irun, k)]["rdat"]
        if imax is not None:
            keep.add((imax, k))
    return keep


def _vb_parallel(mat, ranks, nrun, common, unif_stop, verbose, seed, inits, device, precision):
    """Independent (run, rank) factorizations spread over the ranks of torch.distributed."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("parallel=True needs an initialised torch.distributed process group")
    world, me = dist.get_world_size(), dist.get_rank()
    jobs = [(irun, k) for irun in range(1, nrun + 1) for k in range(len(ranks))]
    # cost of a job ~ rank^2: both the time of an iteration and the number of iterations to
    # convergence grow about linearly with the rank (C4 sweep: r = 2: 36 iterations of 0.75 ms,
    # r = 30: 245 of 5 ms)
    mine = lpt_schedule([float(ranks[k]) ** 2 for _, k in jobs], world)[me]
    done = {}
    with Engine(mat, device=device) as eng:
        eng.set_precision(precision)
        for j in mine:
            irun, k = jobs[j]
            # one-rank call of the per-run routine; the uniform-column rule is applied afterwards
            out = _vb_iterate(eng, irun, mat, [ranks[k]], *common, False, nrun, 0, seed, inits, [])
            done[(irun, k)] = {key: out[key][0] for key in out}
            done[(irun, k)]["unif"] = out["unif_flag"][0]
    # Results back to every rank in two steps: the scalars of all jobs first, then the factor
    # matrices of the jobs that can still be chosen -- the best run of every rank (strict >, the
    # first of equals: the rule of the aggregation, R/bayesian.R:271).  Exchanging the matrices of
    # all 145 jobs of the C4 sweep (4.5 GB, pickled and padded per rank) took longer than the
    # factorizations on 8 GPUs.  If a job raised the uniform-column flag the run order matters
    # (R/bayesian.R:370-378 breaks the rank scan of that run), so everything is exchanged.
    big_keys = ("wdat", "hdat", "dwdat", "dhdat")
    small = {key: {f: v for f, v in res.items() if f not in big_keys} for key, res in done.items()}
    gathered = [None] * world
    dist.all_gather_object(gathered, small)
    allres = {}
    for d in gathered:
        allres.update(d)
    keep = jobs_to_keep(allres, nrun, len(ranks))
    big = {key: {f: done[key][f] for f in big_keys} for key in done if key in keep}
    dist.all_gather_object(gathered, big)
    for key in allres:
        allres[key].update({f: None for f in big_keys})
    for d in gathered:
        for key, mats in d.items():
            allres[key].update(mats)
    vb = []
    for irun in range(1, nrun + 1):
        out = dict(rdat=[-np.inf] * len(ranks), wdat=[None] * len(ranks), hdat=[None] * len(ranks),
                   dwdat=[None] * len(ranks), dhdat=[None] * len(ranks),
                   hyperp=[None] * len(ranks), nunif=[0] * len(ranks), niter=[0] * len(ranks))
        for k in range(len(ranks)):
            res = allres[(irun, k)]
            if res["unif"]:                                     # R/bayesian.R:370-378, post hoc
                warnings.warn("Rank %d row/column constant." % ranks[k])
                if unif_stop:
                    warnings.warn("Rank scan stopped for rank >= %d" % ranks[k])
                    if k == 0:
                        raise RuntimeError("Rerun with lower ranks")
                    break
            for key in ("rdat", "wdat", "hdat", "dwdat", "dhdat", "hyperp", "nunif", "niter"):
                out[key][k] = res[key]
        if verbose >= 2:
            for k in range(len(ranks)):
                if out["hyperp"][k] is not None:
                    print("Run %d Rank = %d: log(evidence) = %s" % (irun, ranks[k], out["rdat"][k]))
        vb.append(out)
    return vb


def _vb_iterate(eng, irun, mat, ranks, ga, gb, initializer, Itmax, hyper_update, Tol, n0, dn,
                connectivity, fudge, device_consensus, unif_stop, nrun, verbose, seed, inits,
                previous, cols=None):
    """R/bayesian.R:303-390 for one run; the it-loop runs on the GPU.  cols = (c0, c1): the engine
    holds the cells [c0, c1) of `mat` and the calls are collective over the shards."""
    nrow, ncol = mat.shape
    c0, c1 = cols if cols is not None else (0, ncol)
    if cols is not None:
        connectivity = False      # the dispersion print needs the labels of all cells
    nrank = len(ranks)
    out = dict(rdat=[-np.inf] * nrank, wdat=[None] * nrank, hdat=[None] * nrank,
               dwdat=[None] * nrank, dhdat=[None] * nrank, hyperp=[None] * nrank,
               nunif=[0] * nrank, labels=[None] * nrank, niter=[0] * nrank,
               unif_flag=[False] * nrank)
    if verbose >= 2 and nrun > 1:
        print("Run %d" % irun)
    for irank, rank in enumerate(ranks):
        if rank > min(nrow, ncol):
            raise ValueError("Rank exceeded min(nrow,ncol)")    # :319-320
        hyper = dict(aw=float(ga[0]), ah=float(ga[-1]), bw=float(gb[0]), bh=float(gb[-1]))  # :321-326
        if inits is not None and (irun, rank) in inits:
            w0, h0 = inits[(irun, rank)]
            eng.set_state(w0, h0[:, c0:c1])                     # lw = ew = w, lh = eh = h (:170)
        elif initializer == "random_device":
            eng.init_random(rank, hyper, seed * 100003 + 1000 * rank + irun, cell_offset=c0)
        elif initializer == "svd2_device":                      # :150-159 where the matrix lives
            eng.init_svd2(rank, hyper, seed * 100003 + 1000 * rank + irun, cell_offset=c0)
        elif initializer == "svd_device":                       # :116-149, pairs oriented
            eng.init_svd(rank, seed * 100003 + 1000 * rank + irun, cell_offset=c0)
        else:
            w0, h0 = vb_init(nrow, ncol, mat, rank, hyper, initializer,
                             seed * 100003 + 1000 * rank + irun)
            eng.set_state(w0, h0[:, c0:c1])
        try:
            res = eng.run(hyper, Itmax=Itmax, Tol=Tol, hyper_update=hyper_update, n0=n0, dn=dn,
                          fudge=fudge)
        except VbnmfError as e:
            if e.code == ERR_HYPER:
                raise RuntimeError("Hyper-parameter update failed to converge") from e  # :43
            raise
        hyper, lk0, it = res["hyper"], res["lml"], res["niter"]
        if verbose >= 3:
            for i in range(it):
                hv = res["hyper_trace"][i]
                print("%d, log(evidence) = %s, aw = %s, bw = %s, ah = %s, bh = %s"
                      % (i + 1, res["lkh_trace"][i], hv[0], hv[1], hv[2], hv[3]))
        disp = None
        if connectivity:                                        # :353-357 (only printed)
            out["labels"][irank] = eng.cluster_id()
            runs = [p["labels"][irank] for p in previous if p["labels"][irank] is not None]
            if device_consensus:
                disp = consensus_from_labels(runs + [out["labels"][irank]], tree=False,
                                             device=eng.device)[0]
            else:
                disp = dispersion_from_labels(runs + [out["labels"][irank]])
        if verbose >= 2:
            msg = "Rank = %d: Nsteps = %d, log(evidence) = %s, hyper = (%s,%s,%s,%s)" % (
                rank, it, lk0, hyper["aw"], hyper["bw"], hyper["ah"], hyper["bh"])
            print(msg + (", dispersion = %s" % disp if connectivity else ""))
        unif = eng.uniform_columns(Tol)                         # :368-369
        out["unif_flag"][irank] = bool(unif.sum() > 0)
        if unif.sum() > 0:
            warnings.warn("Rank %d row/column %s constant." % (
                rank, ",".join(str(i + 1) for i in np.flatnonzero(unif))))
            if unif_stop:
                warnings.warn("Rank scan stopped for rank >= %d" % rank)
                if irank == 0:
                    raise RuntimeError("Rerun with lower ranks")  # :375
                break
        st = eng.get_state(("ew", "eh", "dw", "dh"))
        out["rdat"][irank] = lk0                                # :379-384
        out["wdat"][irank], out["hdat"][irank] = st["ew"], st["eh"]
        out["dwdat"][irank], out["dhdat"][irank] = np.sqrt(st["dw"]), np.sqrt(st["dh"])
        out["hyperp"][irank] = hyper
        out["niter"][irank] = it
    return out


def factorize(object, ranks=2, nrun=20, randomize=False, nsmpl=1, verbose=2, progress_bar=True,
              Itmax=10000, ncnn_step=40, criterion="likelihood", linkage="average", Tol=1e-5,
              store_connectivity=False, seed=1, device=0, device_shuffle=False,
              device_consensus=False):
    """Maximum likelihood factorization (R/factorize.R:139-276); the it-loop (:189-212) runs on the
    GPU with either stopping criterion.  The consensus measures never form the m(m-1)/2
    connectivity vector of the reference (:51-78): dispersion and the cophenetic correlation are
    computed from the groups of cells that share their labels over the runs.

    `randomize=True` fits every rank on `nsmpl` null matrices, each column of the counts shuffled
    over the genes (:172-173).  By default the shuffle is a NumPy permutation of the dense column
    (Philox stream keyed by `seed`) and every null matrix is uploaded anew.
    `device_shuffle=True` (needs `randomize=True`): the counts are uploaded once and each null
    matrix is drawn on the GPU from the resident copy (Engine.shuffle; no dense matrix, no upload):
    sample `ismpl` of rank `r` is Engine.shuffle(seed * 100003 + 1000 * r + 37 * ismpl), closed
    after its `nrun` restarts.  Same distribution, different draw than the default.
    `device_consensus=True` (average linkage only): dispersion and the cophenetic correlation are
    computed on the GPU (consensus_from_labels) from exact integer moments and the merge list of
    the average-linkage tree, with no cap on the number of label groups below what device memory
    holds.  Equal distances are merged in a defined order (smallest group indices first), so the
    cophenetic value can differ from the default's, which breaks such ties differently."""
    if criterion not in ("likelihood", "connectivity"):
        raise ValueError("Unknown stopping criterion.")        # :212
    if device_shuffle and not randomize:
        raise ValueError("device_shuffle applies to randomize=True")
    if device_consensus and linkage != "average":
        raise ValueError("device_consensus supports linkage='average' only")
    mat0 = object.counts
    _check_no_empty(mat0)
    nrow, ncol = mat0.shape
    ranks = [int(r) for r in np.atleast_1d(ranks)]
    nrank = len(ranks)
    wdat, hdat = [None] * nrank, [None] * nrank
    rave, dave, coav = np.zeros(nrank), np.zeros(nrank), np.zeros(nrank)
    rste, dste, cste = np.full(nrank, np.nan), np.full(nrank, np.nan), np.full(nrank, np.nan)
    g = np.random.Generator(np.random.Philox(key=[int(seed), 77]))
    eng = Engine(mat0, device=device)
    sample = eng
    labels_last = None
    try:
        for irank, rank in enumerate(ranks):
            if verbose > 0:
                print("Rank %d" % rank)
            rdat, ddat, cdat = [], [], []
            for ismpl in range(1, nsmpl + 1):
                mat = mat0
                if randomize and not device_shuffle:             # :172-173 column-wise shuffle
                    dense = np.asarray(mat0.todense())
                    for j in range(ncol):
                        dense[:, j] = g.permutation(dense[:, j])
                    mat = sp.csc_matrix(dense)
                    eng.close()
                    eng = Engine(mat, device=device)
                if device_shuffle:                               # :172-173 on the GPU
                    sample = eng.shuffle(seed * 100003 + 1000 * rank + 37 * ismpl)
                else:
                    sample = eng
                rmax, labels = -np.inf, []
                for irun in range(1, nrun + 1):
                    w0, h0 = synth.uniform_init(nrow, ncol, rank,
                                                seed * 100003 + 1000 * rank + 37 * ismpl + irun)
                    res = sample.ml_run(w0, h0, Itmax=Itmax, Tol=Tol, criterion=criterion,
                                        ncnn_step=ncnn_step)
                    lk0 = res["lik"]
                    labels.append(np.argmax(res["h"], axis=0) + 1)  # connectivity(), :51-60
                    if device_consensus:
                        disp = consensus_from_labels(labels, tree=False, device=device)[0]
                    else:
                        disp = dispersion_from_labels(labels)
                    if verbose >= 2:
                        print("Nsteps = %d , likelihood = %s , dispersion = %s\n" % (
                            res["niter"], lk0, disp))
                    if (irun == 1 or lk0 > rmax) and not np.isnan(lk0):  # :219-223
                        rmax, wmax, hmax = lk0, res["w"], res["h"]
                if sample is not eng:
                    sample.close()
                if device_consensus:
                    coph = consensus_from_labels(labels, device=device)[1]
                else:
                    coph = _cophenet(labels, ncol, linkage)
                labels_last = labels
                if verbose >= 1:
                    print("Sample# %d : Max(likelihood) = %s , dispersion = %s , cophenetic = %s"
                          % (ismpl, rmax, disp, coph))
                if ismpl == 1:
                    wdat[irank], hdat[irank] = wmax.copy(), hmax.copy()
                else:
                    wdat[irank] += wmax
                    hdat[irank] += hmax
                rdat.append(rmax); ddat.append(disp); cdat.append(coph)
            wdat[irank] /= nsmpl
            hdat[irank] /= nsmpl
            if nsmpl > 1:
                den = np.sqrt(nsmpl - 1)
                rste[irank] = np.std(rdat, ddof=1) / den
                dste[irank] = np.std(ddat, ddof=1) / den
                cste[irank] = np.std(cdat, ddof=1) / den
            rave[irank], dave[irank], coav[irank] = np.mean(rdat), np.mean(ddat), np.mean(cdat)
    finally:
        sample.close()
        eng.close()
    object.ranks = ranks
    object.basis, object.coeff = wdat, hdat
    if randomize:
        object.measure = dict(rank=np.array(ranks), likelihood=rave, r_se=rste, dispersion=dave,
                              d_se=dste, cophenetic=coav, c_se=cste)
    else:
        object.measure = dict(rank=np.array(ranks), likelihood=rave, dispersion=dave,
                              cophenetic=coav)
    if store_connectivity:
        object.metadata = dict(nrun=nrun, labels=labels_last)
    return object


def label_groups(label_runs):
    """Cells grouped by their tuple of labels over the runs: (tuples G x nrun, sizes G).  Two cells
    of the same group are co-clustered in every run; cells of groups a, b in as many runs as their
    tuples agree in."""
    L = np.stack([np.asarray(v) for v in label_runs], axis=1)
    tup, cnt = np.unique(L, axis=0, return_counts=True)
    return tup, cnt.astype(np.float64)


def _linkage_weighted(D, sizes, method):
    """Agglomerative clustering of G groups of identical points (sizes = points per group) by the
    Lance-Williams recurrence, the same trees as stats::hclust / scipy on the expanded point set:
    identical points merge first at height 0, which leaves exactly the groups with their sizes.
    Returns the G x G matrix of cophenetic distances between groups.  O(G^3) worst case, G = number
    of distinct label tuples (hundreds to a few thousand), independent of the number of cells."""
    G = len(sizes)
    D = np.array(D, dtype=np.float64)
    np.fill_diagonal(D, np.inf)
    n = np.array(sizes, dtype=np.float64)
    active = np.ones(G, dtype=bool)
    members = [[g] for g in range(G)]
    coph = np.zeros((G, G))
    if method in ("centroid", "median", "ward.D2"):
        raise ValueError("linkage %r needs Euclidean squared distances" % method)
    for _ in range(G - 1):
        idx = np.flatnonzero(active)
        sub = D[np.ix_(idx, idx)]
        k = int(np.argmin(sub))
        i, j = idx[k // len(idx)], idx[k % len(idx)]
        if i > j:
            i, j = j, i
        dij = D[i, j]
        for a in members[i]:
            coph[a, members[j]] = dij
        for a in members[j]:
            coph[a, members[i]] = dij
        rest = idx[(idx != i) & (idx != j)]
        if method == "average":
            new = (n[i] * D[i, rest] + n[j] * D[j, rest]) / (n[i] + n[j])
        elif method == "single":
            new = np.minimum(D[i, rest], D[j, rest])
        elif method == "complete":
            new = np.maximum(D[i, rest], D[j, rest])
        elif method == "mcquitty":
            new = 0.5 * (D[i, rest] + D[j, rest])
        elif method in ("ward", "ward.D"):
            t = n[i] + n[j] + n[rest]
            new = ((n[i] + n[rest]) * D[i, rest] + (n[j] + n[rest]) * D[j, rest] - n[rest] * dij) / t
        else:
            raise ValueError("unknown linkage %r" % method)
        D[i, rest] = new
        D[rest, i] = new
        active[j] = False
        D[j, :] = np.inf
        D[:, j] = np.inf
        n[i] += n[j]
        members[i] += members[j]
    return coph


def cophenet_from_labels(label_runs, method="average", max_groups=6000):
    """cophenet(conav/nrun, ncol) of R/factorize.R:69-78 -- cor(d, cophenetic(hclust(d))) with
    d = 1 - average connectivity -- without the nc x nc matrix: hclust on the groups of cells with
    identical label tuples (weighted by their sizes) and the Pearson correlation accumulated over
    group pairs with multiplicity size_a * size_b (same-group pairs contribute (0, 0)).
    The cost depends on the number of distinct label tuples, not on the number of cells."""
    tup, sz = label_groups(label_runs)
    G, nrun = tup.shape
    if sz.sum() < 3:
        return np.nan
    if G > max_groups:
        return np.nan
    agree = np.zeros((G, G))
    for t in range(nrun):
        agree += tup[:, t][:, None] == tup[:, t][None, :]
    D = 1.0 - agree / nrun
    C = _linkage_weighted(D, sz, method)
    iu = np.triu_indices(G, 1)
    wgt = (sz[:, None] * sz[None, :])[iu]
    d, c = D[iu], C[iu]
    same = float(np.sum(sz * (sz - 1.0) / 2.0))              # pairs inside a group: d = coph = 0
    N = same + wgt.sum()
    md, mc = (wgt * d).sum() / N, (wgt * c).sum() / N
    vd = (wgt * (d - md) ** 2).sum() + same * md ** 2
    vc = (wgt * (c - mc) ** 2).sum() + same * mc ** 2
    cov = (wgt * (d - md) * (c - mc)).sum() + same * md * mc
    if vd <= 0 or vc <= 0:
        return np.nan
    return float(cov / np.sqrt(vd * vc))


def _cophenet(labels, nc, method="average"):
    return cophenet_from_labels(labels, method)


# ---- consensus measures from integer moments and the merge list (vbnmf_consensus) -------------
def dispersion_from_moments(s1, s2, m, nrun):
    """dispersion (R/factorize.R:62-67) from S1 = sum a and S2 = sum a^2 over the m(m-1)/2 cell
    pairs, a = runs in which both cells share a label: sum (a/nrun - 1/2)^2 = con4 / (4 nrun^2)
    with the integer con4 = 4 S2 - 4 nrun S1 + nrun^2 m(m-1)/2."""
    s1, s2, m, nrun = int(s1), int(s2), int(m), int(nrun)
    con4 = 4 * s2 - 4 * nrun * s1 + nrun * nrun * (m * (m - 1) // 2)
    return 1.0 / m + 8.0 * (con4 / (4.0 * nrun * nrun)) / m ** 2


def cophenet_from_merges(s1, s2, m, nrun, merges):
    """cophenet (R/factorize.R:69-78) under average linkage from S1, S2 and the merge list
    ((G-1) x 5: a, b, IP_ab, N_a, N_b; vbnmf_consensus).  A merge joins N_a N_b cell pairs at
    height h = 1 - IP_ab / (nrun N_a N_b), which is also their mean distance, so
    sum d c = sum c^2 and every moment of the correlation is a sum over the merges or an integer.
    NaN when m < 3 or either variance is not positive, as cophenet_from_labels."""
    s1, s2, m, nrun = int(s1), int(s2), int(m), int(nrun)
    if m < 3:
        return np.nan
    P = m * (m - 1) // 2
    mg = np.asarray(merges, dtype=np.int64).reshape(-1, 5)
    p = (mg[:, 3] * mg[:, 4]).astype(np.float64)
    h = 1.0 - mg[:, 2].astype(np.float64) / (np.int64(nrun) * mg[:, 3] * mg[:, 4]).astype(np.float64)
    hp = h * p
    sc = float(np.cumsum(hp)[-1]) if len(hp) else 0.0          # sequential sums, merge order
    sc2 = float(np.cumsum(h * hp)[-1]) if len(hp) else 0.0
    sd = (nrun * P - s1) / nrun
    sd2 = (nrun * nrun * P - 2 * nrun * s1 + s2) / (nrun * nrun)
    cov = sc2 - sd * sc / P
    vd = sd2 - sd * sd / P
    vc = sc2 - sc * sc / P
    if vd <= 0 or vc <= 0:
        return np.nan
    return float(cov / np.sqrt(vd * vc))


def consensus_from_labels(label_runs, tree=True, device=0, max_groups=0):
    """(dispersion, cophenetic) of label runs (1-based, as factorize makes them) computed on the
    GPU (engine.consensus): the moments always, the average-linkage tree when tree=True (else the
    cophenetic value is None).  More label groups than max_groups or device memory allow: a
    warning and a NaN cophenetic value, as cophenet_from_labels past its cap."""
    from . import engine
    L = np.stack([np.asarray(v) for v in label_runs]).astype(np.int64) - 1
    nrun, m = L.shape
    try:
        res = engine.consensus(L, device=device, tree=tree, max_groups=max_groups)
    except VbnmfError as e:
        if e.code != ERR_MEMORY:
            raise
        warnings.warn("cophenetic correlation not computed: %d label groups (%s)" % (e.ngroups, e))
        res = engine.consensus(L, device=device, tree=False)
        return dispersion_from_moments(res["s1"], res["s2"], m, nrun), np.nan
    disp = dispersion_from_moments(res["s1"], res["s2"], m, nrun)
    if not tree:
        return disp, None
    return disp, cophenet_from_merges(res["s1"], res["s2"], m, nrun, res["merges"])


def cluster_id(object, rank=2):
    """R/utils.R:903-909: apply(h, 2, which.max) on coeff for `rank` (1-based, first maximum)."""
    k = list(object.ranks).index(rank)
    return np.argmax(np.asarray(object.coeff[k]), axis=0).astype(np.int32) + 1


# ---- optimal_rank (R/utils2.R:59-111), host post-processing of ~30 numbers ----------------------
def _smooth_spline(x, y, df):
    """Natural cubic smoothing spline through (x, y) with `df` effective degrees of freedom
    (what stats::smooth.spline(x, y, df=df) fits when every x is a knot).  Returns fitted y."""
    x = np.asarray(x, float)
    y = np.asarray(y, float)
    n = len(x)
    if df >= n - 1e-9 or n < 4:
        return y.copy()
    hk = np.diff(x)
    Q = np.zeros((n, n - 2))
    R = np.zeros((n - 2, n - 2))
    for j in range(n - 2):
        Q[j, j], Q[j + 1, j], Q[j + 2, j] = 1 / hk[j], -1 / hk[j] - 1 / hk[j + 1], 1 / hk[j + 1]
        R[j, j] = (hk[j] + hk[j + 1]) / 3
        if j + 1 < n - 2:
            R[j, j + 1] = R[j + 1, j] = hk[j + 1] / 6
    K = Q @ np.linalg.solve(R, Q.T)
    ev, V = np.linalg.eigh(0.5 * (K + K.T))
    ev = np.clip(ev, 0, None)
    ev[:2] = 0.0  # the two zero eigenvalues: linear functions are not penalised
    lo, hi = -40.0, 40.0
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if (1.0 / (1.0 + np.exp(mid) * ev)).sum() > df:
            lo = mid
        else:
            hi = mid
    lam = np.exp(0.5 * (lo + hi))
    return V @ ((V.T @ y) / (1.0 + lam * ev))


def _slope(y, x):
    """R/utils2.R:97-111."""
    n = len(x)
    s = np.zeros(n)
    s[0] = (y[1] - y[0]) / (x[1] - x[0])
    for i in range(1, n - 1):
        s[i] = (y[i + 1] - y[i]) / (x[i + 1] - x[i])
    s[n - 1] = s[n - 2]
    return s


def optimal_rank(object, df=10, BF_threshold=3, type=None, m=None):
    """R/utils2.R:59-95.  object: scNMFSet after vb_factorize, or a dict with 'rank' and 'lml'."""
    if isinstance(object, scNMFSet):
        me_x, me_y = np.asarray(object.measure["rank"], float), np.asarray(object.measure["lml"])
        m = object.nrow()
    elif isinstance(object, dict):
        me_x, me_y = np.asarray(object["rank"], float), np.asarray(object["lml"], float)
        if m is None:
            raise ValueError("No. of rows unknown")
    else:
        raise TypeError("Inappropriate class of object")
    o = np.argsort(me_x)
    fx, fy = me_x[o], _smooth_spline(me_x[o], me_y[o], min(df, len(me_x)))
    rst = fx[int(np.argmax(fy))]
    bf = np.log(BF_threshold) / m
    if type is None:
        rng = fx[np.abs(fy - fy.max()) <= bf]
        type = 2 if me_x.max() in rng else 1
    if type == 1:
        ropt = rst
    else:
        sl = _slope(fy, fx)
        idx = int(np.flatnonzero(sl < bf)[0]) if (sl < bf).sum() > 0 else len(fx) - 1
        ropt = fx[idx]
    return dict(type=int(type), ropt=float(ropt))
