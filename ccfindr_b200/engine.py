"""Thin object wrapper over the C ABI: one Engine = one vbnmf_handle = one GPU holding the CSC
count matrix (or one shard of its cells).  Host code only; all arithmetic runs in libvbnmf.so."""
import ctypes as C

import numpy as np

from . import _lib

EPS = float(np.finfo(np.float64).eps)  # .Machine$double.eps (R/bayesian.R:238)
HKEYS = ("aw", "bw", "ah", "bh")


def _dp(a):
    return None if a is None else a.ctypes.data_as(_lib.c_dp)


def hyper_vec(hyper):
    if isinstance(hyper, dict):
        return np.array([float(hyper[k]) for k in HKEYS], dtype=np.float64)
    return np.array(hyper, dtype=np.float64)


def hyper_dict(v):
    return {k: float(x) for k, x in zip(HKEYS, v)}


class Engine:
    """Device-resident VB-NMF state for one count matrix.

    counts: scipy.sparse matrix (genes x cells) or anything scipy can convert to CSC -- the
    `counts(object)` of an scNMFSet (R/bayesian.R:239).
    """

    def __init__(self, counts=None, device=0):
        import scipy.sparse as sp
        csc = counts if sp.isspmatrix_csc(counts) else sp.csc_matrix(counts)
        if not csc.has_sorted_indices:
            csc = csc.copy()
            csc.sort_indices()
        n, m = csc.shape
        rowidx = np.ascontiguousarray(csc.indices, dtype=np.int32)
        values = np.ascontiguousarray(csc.data, dtype=np.float64)
        p32 = p64 = None
        if csc.indptr.dtype == np.int32:  # dgCMatrix @p is int32
            ptr = np.ascontiguousarray(csc.indptr)
            p32 = ptr.ctypes.data_as(_lib.c_i32p)
        else:
            ptr = np.ascontiguousarray(csc.indptr, dtype=np.int64)
            p64 = ptr.ctypes.data_as(_lib.c_i64p)
        self._open(lambda out: self.lib.vbnmf_create(out, n, m, csc.nnz, p32, p64,
                                                     rowidx.ctypes.data_as(_lib.c_i32p),
                                                     _dp(values), int(device)), device)

    def _open(self, create, device, keep=None):
        """Make this Engine the owner of the handle create(out) makes (out: where the library
        stores it); keep: objects that must outlive the handle."""
        self.lib = _lib.load()
        self.handle = C.c_void_p()
        self._keep = keep
        self.device = int(device)
        _lib.check(create(C.byref(self.handle)))
        info = self.info()
        self.n, self.m, self.nnz = int(info["n"]), int(info["m"]), int(info["nnz"])
        self.r = 0

    @classmethod
    def _create(cls, create, device, keep=None):
        """An Engine around the handle create(out) makes."""
        self = cls.__new__(cls)
        self._open(create, device, keep)
        return self

    @classmethod
    def from_device_csc(cls, n, m, nnz, colptr_i64, rowidx_i32, values_f32, device=0):
        """colptr/rowidx/values: torch CUDA tensors (int64, int32, float32) already on `device`.
        The library reads them on its own stream: whatever produced them (the caller's current
        torch stream) is waited for first -- without this the scan of the counts can overtake a
        still running torch.cat and miss the tail of the matrix (seen as a constant offset of the
        bound: the sum of lgamma(x + 1) came out short while the factors were right)."""
        import torch
        torch.cuda.current_stream(torch.device("cuda", int(device))).synchronize()
        lib = _lib.load()
        # the borrowed device arrays must outlive the handle
        return cls._create(lambda out: lib.vbnmf_create_from_device(
            out, int(n), int(m), int(nnz), C.c_void_p(colptr_i64.data_ptr()),
            C.c_void_p(rowidx_i32.data_ptr()), C.c_void_p(values_f32.data_ptr()), int(device)),
            device, keep=(colptr_i64, rowidx_i32, values_f32))

    @classmethod
    def from_mtx(cls, path, device=0):
        """MatrixMarket coordinate file (10x `matrix.mtx`) parsed and sorted into CSC on the GPU
        (readMM + as(., 'dgCMatrix') of read_10x, R/utils.R:34)."""
        lib = _lib.load()
        return cls._create(lambda out: lib.vbnmf_create_from_mtx(out, str(path).encode(), int(device),
                                                                 None), device)

    def csc(self):
        """The count matrix the handle holds, as a scipy CSC matrix."""
        import scipy.sparse as sp
        colptr = np.zeros(self.m + 1, dtype=np.int64)
        rowidx = np.zeros(self.nnz, dtype=np.int32)
        values = np.zeros(self.nnz, dtype=np.float64)
        self._ck(self.lib.vbnmf_get_csc(self.handle, colptr.ctypes.data_as(_lib.c_i64p),
                                        rowidx.ctypes.data_as(_lib.c_i32p), _dp(values)))
        return sp.csc_matrix((values, rowidx, colptr), shape=(self.n, self.m))

    # -- cell / gene QC, column shuffle -------------------------------------------------------
    def qc_stats(self):
        """Per-cell and per-gene statistics of the resident matrix, computed on the device (the
        inputs of filter_cells / filter_genes / calc_vmr, R/utils.R:78-95,134-218): cell_sum (m),
        gene_sum and gene_sumsq (n) as fp64 sums of x and x^2, gene_cells (n) and cell_genes (m)
        as numbers of entries with a non-zero value.  Exact for integer counts."""
        out = dict(cell_sum=np.zeros(self.m), gene_sum=np.zeros(self.n), gene_sumsq=np.zeros(self.n),
                   gene_cells=np.zeros(self.n, dtype=np.int64),
                   cell_genes=np.zeros(self.m, dtype=np.int64))
        self._ck(self.lib.vbnmf_qc_stats(self.handle, _dp(out["cell_sum"]), _dp(out["gene_sum"]),
                                         _dp(out["gene_sumsq"]),
                                         out["gene_cells"].ctypes.data_as(_lib.c_i64p),
                                         out["cell_genes"].ctypes.data_as(_lib.c_i64p)))
        return out

    def subset(self, keep_rows, keep_cols, col_scale=None):
        """A new Engine on the same device holding the genes where keep_rows is true and the cells
        where keep_cols is true (order kept), each entry of cell j multiplied by col_scale[j] when
        given (normalize_count, R/utils.R:318-327).  Built from this engine's device arrays: only
        the masks and the scales cross the bus.  This engine is left as it was."""
        keep_rows = np.asarray(keep_rows)
        keep_cols = np.asarray(keep_cols)
        if keep_rows.dtype != np.bool_ or keep_cols.dtype != np.bool_:
            raise ValueError("keep_rows and keep_cols must be boolean arrays")
        if keep_rows.shape != (self.n,):
            raise ValueError("keep_rows must have one entry per gene (%d)" % self.n)
        if keep_cols.shape != (self.m,):
            raise ValueError("keep_cols must have one entry per cell (%d)" % self.m)
        scale = None
        if col_scale is not None:
            scale = np.ascontiguousarray(col_scale, dtype=np.float64)
            if scale.shape != (self.m,):
                raise ValueError("col_scale must have one entry per cell (%d)" % self.m)
            if not np.isfinite(scale).all():
                raise ValueError("col_scale must be finite")
        rows = np.ascontiguousarray(keep_rows, dtype=np.uint8)
        cols = np.ascontiguousarray(keep_cols, dtype=np.uint8)
        return Engine._create(lambda out: self.lib.vbnmf_create_subset(
            out, self.handle, rows.ctypes.data_as(_lib.c_u8p), cols.ctypes.data_as(_lib.c_u8p),
            _dp(scale)), self.device)

    def shuffle(self, seed):
        """A new Engine on the same device holding this engine's matrix with every column shuffled
        over the genes: the null matrix of factorize(randomize=TRUE) (R/factorize.R:172-173).
        colptr and each column's values are kept and only the rows are drawn, from a counter RNG
        keyed by (seed, column); synth.shuffle_columns_reference is the CPU restatement.  Built
        from this engine's device arrays: nothing crosses the bus.  This engine is left as it
        was."""
        return Engine._create(lambda out: self.lib.vbnmf_create_shuffled(
            out, self.handle, int(seed) & 0xFFFFFFFFFFFFFFFF), self.device)

    # -- lifetime ------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "handle", None) and self.handle.value:
            self.lib.vbnmf_destroy(self.handle)
            self.handle = C.c_void_p()
        self._keep = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, rc):
        _lib.check(rc, self.handle)

    # -- configuration -------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(self.lib.vbnmf_set_stream(self.handle, C.c_void_p(int(cuda_stream_ptr))))

    def set_precision(self, precision):
        self._ck(self.lib.vbnmf_set_precision(self.handle, int(precision)))

    @staticmethod
    def nccl_unique_id():
        buf = (C.c_char * 128)()
        rc = _lib.load().vbnmf_nccl_unique_id(buf)
        if rc != 0:
            _lib.check(rc, None)
        return bytes(buf)

    def attach_comm(self, comm):
        """comm: a Comm (one NCCL communicator per process); cells are sharded over its ranks."""
        self._ck(self.lib.vbnmf_attach_comm(self.handle, comm.ptr))
        self._comm = comm

    def info(self):
        v = (C.c_int64 * 8)()
        self._ck(self.lib.vbnmf_info(self.handle, v))
        return dict(zip(("n", "m", "nnz", "r", "rs", "precision", "nranks", "m_global"), v))

    def layout_info(self):
        """Tiled device layout in use (after set_state): storage format of the nonzeros
        ('f32', 'f64' or 'p16'), tile rows, slab counts, stored entries per pass, bytes."""
        v = (C.c_int64 * 8)()
        self._ck(self.lib.vbnmf_layout_info(self.handle, v))
        d = dict(zip(("format", "tile_rows", "gene_slabs", "cell_slabs", "entries_cols",
                      "entries_rows", "nonzeros_per_group_step", "bytes"), v))
        d["format"] = ("f32", "f64", "p16")[d["format"]]
        return d

    # -- state ---------------------------------------------------------------------------------
    def set_state(self, lw, lh, ew=None, eh=None):
        """wh list of vbnmf_update (src/vbnmf_update.cpp:22-25): lw, ew n x r; lh, eh r x m."""
        lw = np.asfortranarray(lw, dtype=np.float64)
        lh = np.asfortranarray(lh, dtype=np.float64)
        r = lw.shape[1]
        if lw.shape != (self.n, r) or lh.shape != (r, self.m):
            raise ValueError("lw must be n x r and lh r x m")
        ew = None if ew is None else np.asfortranarray(ew, dtype=np.float64)
        eh = None if eh is None else np.asfortranarray(eh, dtype=np.float64)
        self._ck(self.lib.vbnmf_set_state(self.handle, r, _dp(lw), _dp(lh), _dp(ew), _dp(eh)))
        self.r = r

    def init_random(self, rank, hyper, seed, cell_offset=0):
        """vb_init(initializer='random') (R/bayesian.R:111-115) drawn on the device: no host
        matrices, no upload.  The draw is keyed by (seed, gene / global cell index, k); see
        synth.device_random_init_reference for the CPU restatement."""
        hy = hyper_vec(hyper)
        self._ck(self.lib.vbnmf_init_random(self.handle, int(rank), _dp(hy), int(seed),
                                            int(cell_offset)))
        self.r = int(rank)

    def init_svd2(self, rank, hyper, seed=1, cell_offset=0):
        """vb_init(initializer='svd2') (R/bayesian.R:150-159) computed on the device from the
        resident count matrix (randomized truncated SVD): no host SVD, no upload."""
        hy = hyper_vec(hyper)
        self._ck(self.lib.vbnmf_init_svd2(self.handle, int(rank), _dp(hy), int(seed),
                                          int(cell_offset)))
        self.r = int(rank)

    def init_svd(self, rank, seed=1, cell_offset=0):
        """vb_init(initializer='svd') (R/bayesian.R:116-149) computed on the device from the same
        truncated SVD as init_svd2, each pair of singular vectors k >= 1 oriented first (see
        vbnmf_init_svd in include/vbnmf.h; synth.device_svd_init_reference restates it)."""
        self._ck(self.lib.vbnmf_init_svd(self.handle, int(rank), int(seed), int(cell_offset)))
        self.r = int(rank)

    def get_state(self, which=("lw", "lh", "ew", "eh", "dw", "dh")):
        r = self.r
        out = {}
        for k in which:
            out[k] = np.zeros((self.n, r) if k[1] == "w" else (r, self.m), order="F")
        args = [_dp(out.get(k)) for k in ("lw", "lh", "ew", "eh", "dw", "dh")]
        self._ck(self.lib.vbnmf_get_state(self.handle, *args))
        return out

    def step(self, hyper, fudge=EPS):
        """One vbnmf_update (src/vbnmf_update.cpp:16-102).  Returns lkh."""
        hy = hyper_vec(hyper)
        lkh = C.c_double(0.0)
        self._ck(self.lib.vbnmf_step(self.handle, _dp(hy), float(fudge), C.byref(lkh)))
        return lkh.value

    def means(self):
        v = np.zeros(4)
        self._ck(self.lib.vbnmf_get_means(self.handle, _dp(v)))
        return v

    def run(self, hyper, Itmax=10000, Tol=1e-5, hyper_update=(True,) * 4, n0=10, dn=1, fudge=EPS):
        """The it-loop of vb_iterate (R/bayesian.R:336-352).  Returns a dict with the final hyper,
        lml (= lk0 of :379), niter, stop_reason and the per-iteration traces."""
        cfg = _lib.VbnmfCfg()
        cfg.itmax = int(Itmax)
        cfg.tol = float(Tol)
        for i in range(4):
            cfg.hyper_update[i] = int(bool(hyper_update[i]))
        cfg.n0, cfg.dn, cfg.fudge = int(n0), int(dn), float(fudge)
        hy = hyper_vec(hyper)
        trace = np.full(cfg.itmax, np.nan)
        htrace = np.full((cfg.itmax, 4), np.nan)
        niter, reason, lml = C.c_int(0), C.c_int(0), C.c_double(0.0)
        self._ck(self.lib.vbnmf_run(self.handle, C.byref(cfg), _dp(hy), _dp(trace), _dp(htrace),
                                    C.byref(niter), C.byref(lml), C.byref(reason)))
        it = niter.value
        return dict(hyper=hyper_dict(hy), lml=lml.value, niter=it, stop_reason=reason.value,
                    lkh_trace=trace[:it].copy(), hyper_trace=htrace[:it].copy())

    def cluster_id(self):
        cid = np.zeros(self.m, dtype=np.int32)
        self._ck(self.lib.vbnmf_cluster_id(self.handle, cid.ctypes.data_as(_lib.c_i32p)))
        return cid

    def uniform_columns(self, tol):
        fl = np.zeros(self.r, dtype=np.int32)
        self._ck(self.lib.vbnmf_uniform_columns(self.handle, float(tol),
                                                fl.ctypes.data_as(_lib.c_i32p)))
        return fl.astype(bool)

    # -- ML path -------------------------------------------------------------------------------
    def ml_run(self, w0, h0, Itmax=10000, Tol=1e-5, criterion="likelihood", ncnn_step=40):
        """it-loop of factorize() (R/factorize.R:189-212) with either stopping criterion:
        'likelihood' (:207) or 'connectivity' (:194-204, unchanged cell co-clustering for
        ncnn_step iterations)."""
        if criterion not in ("likelihood", "connectivity"):
            raise ValueError("Unknown stopping criterion.")
        w0 = np.asfortranarray(w0, dtype=np.float64)
        h0 = np.asfortranarray(h0, dtype=np.float64)
        r = w0.shape[1]
        w = np.zeros((self.n, r), order="F")
        h = np.zeros((r, self.m), order="F")
        trace = np.full(int(Itmax), np.nan)
        nch = np.full(int(Itmax), np.nan)
        niter = C.c_int(0)
        self._ck(self.lib.mlnmf_run2(self.handle, r, _dp(w0), _dp(h0), int(Itmax), float(Tol),
                                     int(criterion == "connectivity"), int(ncnn_step), _dp(w),
                                     _dp(h), _dp(trace), _dp(nch), C.byref(niter)))
        self.r = r
        it = niter.value
        return dict(w=w, h=h, niter=it, lik_trace=trace[:it].copy(), lik=float(trace[it - 1]),
                    nchange_trace=nch[:it].copy())

    # -- measurement ---------------------------------------------------------------------------
    def bench_iterations(self, hyper, iters, fudge=EPS, hyper_on=False):
        """`iters` iterations of the device-controlled product loop, CUDA-event timed.  hyper_on:
        hyper_update after every iteration (the loop's steady state past hyper.update.n0); the
        updated hyper-parameters come back in the result."""
        hy = hyper_vec(hyper)
        ms = np.zeros(4)
        launches = C.c_int64(0)
        lkh = C.c_double(0.0)
        self._ck(self.lib.vbnmf_bench_iterations(self.handle, _dp(hy), float(fudge), int(iters),
                                                 int(bool(hyper_on)), _dp(ms), C.byref(launches),
                                                 C.byref(lkh)))
        return dict(ms_total=ms[0], ms_cols=ms[1], ms_rows=ms[2], ms_other=ms[3],
                    launches=launches.value, lkh=lkh.value, hyper=hyper_dict(hy))


def set_host_threads(n):
    """Threads that stage host -> device uploads (process-wide); pass cores / processes when one
    process drives each GPU."""
    _lib.check(_lib.load().vbnmf_set_host_threads(int(n)))


def trim_pool(device=0):
    _lib.check(_lib.load().vbnmf_trim_pool(int(device)))


def consensus(labels, device=0, tree=True, max_groups=0):
    """Consensus measures of restarts on the device (vbnmf_consensus, R/factorize.R:51-78).
    labels: nrun x m integers 0 ... K-1 (one row per run).  Returns dict(s1, s2) -- the sums of a
    and a^2 over cell pairs, a = runs in which both cells share a label -- and with tree=True also
    ngroups (G), merges ((G-1) x 5 int64: a, b, IP_ab, N_a, N_b of every average-linkage merge)
    and rescans.  More groups than max_groups (0: what device memory allows) raise VbnmfError with
    code ERR_MEMORY and the number of groups in its `ngroups`."""
    L = np.ascontiguousarray(np.atleast_2d(labels), dtype=np.int32)
    nrun, m = L.shape
    K = int(L.max()) + 1 if L.size else 1
    mom = np.zeros(2, dtype=np.int64)
    ng, resc = C.c_int64(0), C.c_int64(0)
    merges = None
    cap = 0
    if tree:
        cap = min(m, K ** nrun) - 1                              # G <= min(m, K^nrun)
        merges = np.zeros((max(cap, 1), 5), dtype=np.int64)
    lib = _lib.load()
    rc = lib.vbnmf_consensus(int(device), m, nrun, K, L.ctypes.data_as(_lib.c_i32p), int(max_groups),
                             mom.ctypes.data_as(_lib.c_i64p), C.byref(ng),
                             None if merges is None else merges.ctypes.data_as(_lib.c_i64p), cap,
                             C.byref(resc))
    try:
        _lib.check(rc)
    except _lib.VbnmfError as err:
        err.ngroups = ng.value
        raise
    out = dict(s1=int(mom[0]), s2=int(mom[1]))
    if tree:
        G = ng.value
        out.update(ngroups=G, merges=merges[:max(G - 1, 0)].copy(), rescans=resc.value)
    return out


class Comm:
    """Process-level NCCL communicator for cell-sharded factorizations (vbnmf_comm)."""

    def __init__(self, nranks, rank, uid, device=0):
        self.lib = _lib.load()
        self.ptr = C.c_void_p()
        buf = (C.c_char * 128).from_buffer_copy(uid)
        _lib.check(self.lib.vbnmf_comm_create(C.byref(self.ptr), int(nranks), int(rank), buf,
                                              int(device)))
        self.nranks, self.rank = int(nranks), int(rank)

    def close(self):
        if self.ptr and self.ptr.value:
            self.lib.vbnmf_comm_destroy(self.ptr)
            self.ptr = C.c_void_p()
