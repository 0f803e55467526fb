"""vb_init(initializer='svd') (R/bayesian.R:116-149) computed on the GPU (Engine.init_svd,
vbnmf_init_svd): the randomized truncated SVD of the resident matrix, each pair of singular vectors
k >= 1 oriented, then the reference formula.  Checked against the CPU restatement
(synth.device_svd_init_reference) on an exact SVD of the golden matrices, through a state round
trip, the front end, the argument errors, the R shim, at C2 size and, with 2 GPUs, sharded."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_counts

pytestmark = pytest.mark.gpu

HYPER = dict(aw=1.0, bw=1.0, ah=1.0, bh=1.0)


def exact_svd(X, rank):
    u, d, vt = np.linalg.svd(np.asarray(X.todense()), full_matrices=False)
    return u[:, :rank], d[:rank], vt[:rank].T


def oriented_reference(u, d, v, w_got, h_got):
    """synth.device_svd_init_reference, except that a component whose P and N differ by less
    than 1e-6 relative takes whichever orientation is closer to what the device returned."""
    from ccfindr_b200 import api, synth
    w, h = synth.device_svd_init_reference(u, d, v)
    uo, vo = synth.orient_svd_pairs(u, v)
    for k in range(1, len(d)):
        P = np.linalg.norm(np.maximum(uo[:, k], 0)) * np.linalg.norm(np.maximum(vo[:, k], 0))
        N = np.linalg.norm(np.minimum(uo[:, k], 0)) * np.linalg.norm(np.minimum(vo[:, k], 0))
        if abs(P - N) >= 1e-6 * max(P, N):
            continue
        uf, vf = uo.copy(), vo.copy()
        uf[:, k], vf[:, k] = -uf[:, k], -vf[:, k]
        wf, hf = api.svd_init_from(uf, d, vf)
        if np.abs(wf[:, k] - w_got[:, k]).max() < np.abs(w[:, k] - w_got[:, k]).max():
            w[:, k], h[k] = wf[:, k], hf[k]
    return w, h


@pytest.mark.parametrize("counts", ["pbmc", "c1s1", "c1s2", "c1s3"])
def test_device_svd_initializer_matches_the_oriented_restatement(counts):
    from ccfindr_b200.engine import Engine
    X = load_counts(counts)
    u, d, v = exact_svd(X, 10)
    with Engine(X) as eng:
        for rank in (2, 3, 5, 10):
            eng.init_svd(rank, seed=5)
            st = eng.get_state()
            w, h = oriented_reference(u[:, :rank], d[:rank], v[:, :rank], st["lw"], st["lh"])
            for got, ref in ((st["lw"], w), (st["lh"], h), (st["ew"], w), (st["eh"], h)):
                assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 1e-6, (counts, rank)
            assert not st["dw"].any() and not st["dh"].any()   # dw = dh = 0 (:161-162)


def test_state_after_init_svd_round_trips_through_set_state():
    """The state downloaded after init_svd, loaded by set_state into a fresh handle, reads back
    unchanged and gives the same run bit for bit: the device holds exactly what it reports."""
    from ccfindr_b200.engine import Engine
    X = load_counts("pbmc")
    with Engine(X) as a:
        a.init_svd(5, seed=3)
        st = a.get_state()
        ra = a.run(HYPER, Itmax=40, Tol=1e-7)
    with Engine(X) as b:
        b.set_state(st["lw"], st["lh"], st["ew"], st["eh"])
        back = b.get_state()
        for k in ("lw", "lh", "ew", "eh", "dw", "dh"):
            assert np.array_equal(back[k], st[k]), k
        rb = b.run(HYPER, Itmax=40, Tol=1e-7)
    assert ra["niter"] == rb["niter"] and ra["stop_reason"] == rb["stop_reason"]
    assert np.array_equal(ra["lkh_trace"], rb["lkh_trace"])
    assert np.array_equal(ra["hyper_trace"], rb["hyper_trace"])


def test_vb_factorize_with_device_svd_equals_the_restated_initializer():
    from ccfindr_b200 import api, synth
    X = load_counts("pbmc")
    ranks = [3, 4]
    u, d, v = exact_svd(X, max(ranks))
    inits = {(1, r): synth.device_svd_init_reference(u[:, :r], d[:r], v[:, :r]) for r in ranks}
    kw = dict(ranks=ranks, nrun=1, verbose=0, Itmax=30, initializer="svd")
    a = api.vb_factorize(api.scNMFSet(X), device_init=True, **kw)
    b = api.vb_factorize(api.scNMFSet(X), inits=inits, **kw)
    assert list(a.ranks) == list(b.ranks) == ranks
    assert np.max(np.abs(a.measure["lml"] - b.measure["lml"]) / np.abs(b.measure["lml"])) < 1e-6


def test_init_svd_argument_errors():
    from ccfindr_b200 import _lib
    from ccfindr_b200.engine import Engine
    X = load_counts("tiny")                                     # 39 genes x 25 cells
    assert _lib.load().vbnmf_init_svd(None, 2, 1, 0) == _lib.ERR_ARG
    with Engine(X) as eng:
        for rank, offset, text in ((0, 0, "rank must be in 1..64"), (65, 0, "rank must be in 1..64"),
                                   (2, -1, "cell_offset must be >= 0"),
                                   (26, 0, "rank exceeds min(n, m)")):
            with pytest.raises(_lib.VbnmfError) as e:
                eng.init_svd(rank, cell_offset=offset)
            assert e.value.code == _lib.ERR_ARG and text in str(e.value), (rank, offset)
        eng.init_svd(3)                                         # the handle is still usable
        st = eng.get_state(("lw", "lh"))
        assert np.isfinite(st["lw"]).all() and np.isfinite(st["lh"]).all()
        assert (st["lw"][:, 1:] >= 0).all() and (st["lh"][1:] >= 0).all()


@pytest.fixture(scope="module")
def shim():
    """r-shim/src/vbnmf_shim.c built against the stand-in R runtime as tests/test_rshim.py builds
    it, into a library of its own."""
    from ccfindr_b200 import _lib, build as vb_build
    from test_rshim import SHIM_C, STUB
    vb_build.build()
    out = os.path.join(STUB, "_build", "libshimtest_svd.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-shared", "-fPIC", "-O1", "-Wall", "-Wextra", "-Werror",
           "-Wno-cast-function-type", "-I", STUB, "-I", os.path.join(ROOT, "include"), SHIM_C,
           os.path.join(STUB, "rstub.c"), "-L", libdir, "-lvbnmf", "-Wl,-rpath," + libdir,
           "-o", out]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    lib = C.CDLL(out)
    lib.rstub_init()
    for name in ("rstub_real", "rstub_int", "rstub_data", "VECTOR_ELT"):
        getattr(lib, name).restype = C.c_void_p
    lib.rstub_real.argtypes = [C.c_void_p, C.c_ssize_t, C.c_int, C.c_int]
    lib.rstub_int.argtypes = [C.c_void_p, C.c_ssize_t, C.c_int]
    lib.rstub_data.argtypes = [C.c_void_p]
    lib.VECTOR_ELT.argtypes = [C.c_void_p, C.c_ssize_t]
    lib.R_init_ccfindRgpu(None)
    yield lib
    lib.rstub_free_all()


def test_r_shim_svd_entry_points_match_the_ctypes_path(shim):
    from ccfindr_b200.engine import Engine
    X = load_counts("c1s1")
    n, m = X.shape
    r, seed = 4, 9
    hyper = np.array([1.0, 1.0, 1.0, 0.6])

    def real(a, nrow=0, ncol=0):
        a = np.asfortranarray(a, dtype=np.float64)
        return C.c_void_p(shim.rstub_real(a.ctypes.data_as(C.c_void_p), a.size, nrow, ncol))

    def ints(a, logical=0):
        a = np.ascontiguousarray(a, dtype=np.int32)
        return C.c_void_p(shim.rstub_int(a.ctypes.data_as(C.c_void_p), a.size, logical))

    def state(h):
        st = C.c_void_p(shim.C_vbnmf_get_state(h))
        out = {}
        for i, k in enumerate(("lw", "lh", "ew", "eh", "dw", "dh")):
            shape = (n, r) if k[1] == "w" else (r, m)
            p = shim.rstub_data(C.c_void_p(shim.VECTOR_ELT(st, i)))
            buf = (C.c_double * (shape[0] * shape[1])).from_address(p)
            out[k] = np.frombuffer(buf, dtype=np.float64).reshape(shape, order="F").copy()
        return out

    for f in ("C_vbnmf_create", "C_vbnmf_init_svd", "C_vbnmf_init_svd2", "C_vbnmf_get_state",
              "C_vbnmf_destroy"):
        getattr(shim, f).restype = C.c_void_p
    h = C.c_void_p(shim.C_vbnmf_create(ints(X.indptr), ints(X.indices), real(X.data),
                                       ints([n, m]), ints([0])))
    shim.C_vbnmf_init_svd(h, ints([r]), real([float(seed)]))
    got_svd = state(h)
    shim.C_vbnmf_init_svd2(h, ints([r]), real(hyper), real([float(seed)]))
    got_svd2 = state(h)
    shim.C_vbnmf_destroy(h)
    with Engine(X) as eng:
        eng.init_svd(r, seed=seed)
        ref_svd = eng.get_state()
        eng.init_svd2(r, hyper, seed=seed)
        ref_svd2 = eng.get_state()
    # the sketch is accumulated with fp64 atomics: equal to rounding, not bit for bit
    for got, ref in ((got_svd, ref_svd), (got_svd2, ref_svd2)):
        for k in ("lw", "lh", "ew", "eh"):
            assert np.max(np.abs(got[k] - ref[k])) / np.max(np.abs(ref[k])) < 1e-9, k
        assert not got["dw"].any() and not got["dh"].any()


def test_init_svd_at_c2_size():
    """20k genes x 100k cells (synth.tenx_like_device, the C2 matrix), rank 10: finite, w and h
    nonnegative for k >= 1.  The unit norm of the singular vectors is read off the factors:
    |w_0| / |h_0| = |u_0|, and with 'svd2' from the same seed (w2 = |U| / scale, mean(h2) = bh)
    |u_k| = |w2_k| |h2_0| / |h_0|^2 for every k."""
    import torch
    import bench
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    wl = bench.WORKLOADS["c2"]
    n, m, r = wl["n"], wl["m_per_gpu"], 10
    dev = torch.device("cuda", 0)
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    with Engine.from_device_csc(n, m, int(rowidx.numel()), colptr, rowidx, values) as eng:
        eng.init_svd(r, seed=2)
        st = eng.get_state(("lw", "lh"))
        eng.init_svd2(r, HYPER, seed=2)
        st2 = eng.get_state(("lw", "lh"))
    w, h = st["lw"], st["lh"]
    assert np.isfinite(w).all() and np.isfinite(h).all()
    assert (w[:, 1:] >= 0).all() and (h[1:] >= 0).all()
    assert (np.linalg.norm(w, axis=0) > 0).all()
    h0 = np.linalg.norm(h[0])
    assert abs(np.linalg.norm(w[:, 0]) / h0 - 1.0) < 1e-7
    unorm = np.linalg.norm(st2["lw"], axis=0) * np.linalg.norm(st2["lh"][0]) / h0 ** 2
    assert np.max(np.abs(unorm - 1.0)) < 1e-7, unorm


def test_two_gpu_sharded_init_svd_equals_one_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29737",
           os.path.join(ROOT, "tests", "mgpu_svd_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MGPU_SVD_OK" in res.stdout
