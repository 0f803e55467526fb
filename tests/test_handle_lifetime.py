"""Device memory of the handle paths: every create path and the temporary handle of
vbnmf_consensus give back all they took, on success and on the argument errors found after the
device was touched, and the export functions of a live handle keep no scratch.  The library
allocates only from the device's default memory pool, whose used bytes the driver reports
(cuMemPoolGetAttribute, CU_MEMPOOL_ATTR_USED_MEM_CURRENT).

The argument errors found before the device is touched must stay ERR_ARG on a machine without a
GPU too (a check moved behind the device set-up would turn them into ERR_CUDA): that test needs
no device."""
import ctypes as C
import gc

import numpy as np
import pytest
import scipy.sparse as sp

CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


def _lib():
    from ccfindr_b200 import _lib
    return _lib


@pytest.fixture
def pool_used():
    """used_bytes() of the default memory pool of device 0, read once the device is idle."""
    import torch
    cuda = C.CDLL("libcuda.so.1")
    assert cuda.cuInit(0) == 0
    dev = C.c_int()
    assert cuda.cuDeviceGet(C.byref(dev), 0) == 0
    pool = C.c_void_p()
    assert cuda.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0

    def used_bytes():
        gc.collect()  # an Engine dropped earlier must not be destroyed in the middle of a reading
        torch.cuda.synchronize(0)
        v = C.c_uint64()
        assert cuda.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(v)) == 0
        return v.value
    return used_bytes


def _counts():
    from ccfindr_b200 import synth
    return sp.csc_matrix(synth.simulate_whx(nrow=300, ncol=120, rank=3, seed=5)["x"])


def _write_mtx(path, x, duplicate=False):
    x = sp.coo_matrix(x)
    rows, cols, vals = list(x.row), list(x.col), list(x.data)
    if duplicate:
        rows.append(rows[0]); cols.append(cols[0]); vals.append(vals[0])
    with open(path, "w") as f:
        f.write("%%%%MatrixMarket matrix coordinate integer general\n%d %d %d\n"
                % (x.shape[0], x.shape[1], len(vals)))
        for i, j, v in zip(rows, cols, vals):
            f.write("%d %d %d\n" % (i + 1, j + 1, int(v)))


def _create_host(lib, n, m, colptr, rowidx, values):
    h = C.c_void_p()
    colptr = np.ascontiguousarray(colptr, dtype=np.int64)
    rowidx = np.ascontiguousarray(rowidx, dtype=np.int32)
    values = np.ascontiguousarray(values, dtype=np.float64)
    rc = lib.vbnmf_create(C.byref(h), n, m, len(values), None, colptr.ctypes.data_as(_lib().c_i64p),
                          rowidx.ctypes.data_as(_lib().c_i32p), values.ctypes.data_as(_lib().c_dp), 0)
    return rc, h


def _consensus(lib, labels, K, cap):
    L = np.ascontiguousarray(labels, dtype=np.int32)
    nrun, m = L.shape
    mom = np.zeros(2, dtype=np.int64)
    ng, resc = C.c_int64(0), C.c_int64(0)
    mg = np.zeros((max(m, 1), 5), dtype=np.int64)
    return lib.vbnmf_consensus(0, m, nrun, K, L.ctypes.data_as(_lib().c_i32p), 0,
                               mom.ctypes.data_as(_lib().c_i64p), C.byref(ng),
                               mg.ctypes.data_as(_lib().c_i64p), cap, C.byref(resc)), ng.value


def test_argument_errors_before_the_device():
    from ccfindr_b200 import build
    build.build()
    lib = _lib().load()
    ERR_ARG = _lib().ERR_ARG
    h = C.c_void_p()
    one64 = np.zeros(2, dtype=np.int64)
    one32 = np.zeros(1, dtype=np.int32)
    ones = np.ones(1)
    # vbnmf_create: NULL row indices, and n above the int32 range
    assert lib.vbnmf_create(C.byref(h), 1, 1, 1, None, one64.ctypes.data_as(_lib().c_i64p), None,
                            ones.ctypes.data_as(_lib().c_dp), 0) == ERR_ARG
    assert lib.vbnmf_create(C.byref(h), 2 ** 31, 1, 1, None, one64.ctypes.data_as(_lib().c_i64p),
                            one32.ctypes.data_as(_lib().c_i32p), ones.ctypes.data_as(_lib().c_dp),
                            0) == ERR_ARG
    assert b"2^31" in lib.vbnmf_last_error(None)
    assert lib.vbnmf_create_from_device(C.byref(h), 1, 1, 1, None, None, None, 0) == ERR_ARG
    assert lib.vbnmf_create_from_mtx(C.byref(h), b"/nonexistent/matrix.mtx", 0, None) == ERR_ARG
    assert b"cannot open" in lib.vbnmf_last_error(None)
    assert lib.vbnmf_create_subset(C.byref(h), None, None, None, None) == ERR_ARG
    assert lib.vbnmf_create_shuffled(C.byref(h), None, 1) == ERR_ARG
    assert not h.value
    assert _consensus(lib, np.zeros((2, 4)), 0, 3)[0] == ERR_ARG  # nlabels = 0
    assert b"nlabels" in lib.vbnmf_last_error(None)


@pytest.mark.gpu
def test_create_paths_give_back_their_memory(pool_used, tmp_path):
    import torch
    from ccfindr_b200.engine import Engine
    x = _counts()
    mtx = tmp_path / "matrix.mtx"
    _write_mtx(mtx, x)
    dev = torch.device("cuda", 0)
    colptr = torch.tensor(x.indptr, dtype=torch.int64, device=dev)
    rowidx = torch.tensor(x.indices, dtype=torch.int32, device=dev)
    values = torch.tensor(x.data, dtype=torch.float32, device=dev)
    with Engine(x) as src:
        keep = np.ones(x.shape[0], bool), np.arange(x.shape[1]) % 2 == 0
        for make in (lambda: Engine(x), lambda: Engine(x * 0.3),  # fp32 and fp64 values
                     lambda: Engine.from_device_csc(*x.shape, x.nnz, colptr, rowidx, values),
                     lambda: Engine.from_mtx(mtx), lambda: src.subset(*keep),
                     lambda: src.subset(*keep, col_scale=np.linspace(0.3, 2.0, x.shape[1])),
                     lambda: src.shuffle(7)):
            before = pool_used()
            eng = make()
            assert eng.nnz > 0
            eng.close()
            assert pool_used() == before


@pytest.mark.gpu
def test_refused_creates_give_back_their_memory(pool_used, tmp_path):
    from ccfindr_b200._lib import VbnmfError
    from ccfindr_b200.engine import Engine
    lib = _lib().load()
    ERR_ARG = _lib().ERR_ARG
    x = _counts()
    dup = tmp_path / "dup.mtx"
    _write_mtx(dup, x, duplicate=True)
    diag = sp.csc_matrix(np.diag([1.0, 2.0, 3.0]))
    rep = sp.csc_matrix((np.ones(4), np.array([0, 0, 1, 1]), np.array([0, 3, 4])), shape=(2, 2))
    with Engine(diag) as d, Engine(rep) as r:
        before = pool_used()
        rc, h = _create_host(lib, 3, 2, [0, 1, 2], [0, 1, 2], [1.0, 1.0, 1.0])  # colptr ends at 2
        assert rc == ERR_ARG and not h.value and b"span nnz" in lib.vbnmf_last_error(None)
        assert pool_used() == before
        with pytest.raises(VbnmfError, match="duplicate entries"):
            Engine.from_mtx(dup)
        assert pool_used() == before
        with pytest.raises(VbnmfError, match="holds no entries"):
            d.subset(np.array([True, False, False]), np.array([False, True, True]))
        assert pool_used() == before
        with pytest.raises(VbnmfError, match="more entries"):
            r.shuffle(1)
        assert pool_used() == before
        labels = np.array([[0, 1, 2, 3, 0, 1], [0, 0, 1, 1, 2, 2]])   # 6 groups
        assert _consensus(lib, labels, 4, 3) == (ERR_ARG, 6)        # merge_cap 3 < G - 1
        assert pool_used() == before
        assert _consensus(lib, labels, 4, 5) == (0, 6)
        assert pool_used() == before


@pytest.mark.gpu
def test_exports_keep_no_scratch(pool_used):
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    x = _counts()
    hyper = dict(aw=1.0, bw=1.0, ah=1.0, bh=1.0)
    w0, h0 = synth.random_init(*x.shape, 3, hyper, seed=2)
    with Engine(x) as eng:
        eng.set_state(w0, h0)
        eng.step(hyper)
        calls = {"get_state": eng.get_state, "cluster_id": eng.cluster_id,
                 "uniform_columns": lambda: eng.uniform_columns(1e-3), "qc_stats": eng.qc_stats,
                 "init_svd": lambda: eng.init_svd(3, seed=1)}
        for name, call in calls.items():
            call()
            first = pool_used()
            call()
            assert pool_used() == first, name
