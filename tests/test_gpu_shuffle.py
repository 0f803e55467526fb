"""GPU tests of the column shuffle: Engine.shuffle (csrc/shuffle.cuh, vbnmf_create_shuffled)
against the NumPy restatement synth.shuffle_columns_reference, and factorize(randomize=True,
device_shuffle=True) against the same front end fed with host-shuffled matrices."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_counts
from test_gpu_qc import c2_device_matrix, check_csc_equal, fp64_counts, real_counts, with_zeros

pytestmark = pytest.mark.gpu

HYPER = dict(aw=1.0, bw=1.0, ah=1.0, bh=1.0)
KINDS = {"int": lambda X: X, "int-fp64": fp64_counts, "zeros": with_zeros, "real": real_counts}


def runs(eng, r=3):
    """One ML run and one VB run from fixed starts: results and factors."""
    from ccfindr_b200 import synth
    w0, h0 = synth.uniform_init(eng.n, eng.m, r, 5)
    ml = eng.ml_run(w0, h0, Itmax=30)
    eng.init_random(r, HYPER, seed=17)
    vb = eng.run(HYPER, Itmax=30, hyper_update=(False,) * 4)
    st = eng.get_state(("ew", "eh"))
    return [ml["w"], ml["h"], ml["lik_trace"], vb["lkh_trace"], np.array([vb["lml"]]), st["ew"],
            st["eh"]]


def assert_same_runs(a, b):
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


# ---- 1. bitwise equal to the restatement --------------------------------------------------------
@pytest.mark.parametrize("name", ["pbmc", "c1s1", "c1s2", "c1s3", "tiny"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_shuffle_matches_reference(name, kind):
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    X = KINDS[kind](load_counts(name))
    with Engine(X) as src:
        for seed in (1, 2**40 + 7):
            with src.shuffle(seed) as sh:
                assert (sh.n, sh.m, sh.nnz) == (src.n, src.m, src.nnz)
                check_csc_equal(sh.csc(), synth.shuffle_columns_reference(X, seed))
        check_csc_equal(src.csc(), sp.csc_matrix(X))


@pytest.mark.parametrize("shape", ["dense_column", "one_row", "one_by_one"])
def test_shuffle_degenerate_shapes(shape):
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    rng = np.random.default_rng(8)
    if shape == "dense_column":   # k = n: the draw must collect every row
        D = (rng.random((3000, 6)) < 0.1) * rng.integers(1, 9, (3000, 6)).astype(float)
        D[:, 2] = rng.integers(1, 9, 3000)
    elif shape == "one_row":
        D = np.array([[3.0, 0.0, 1.0, 7.0, 0.0, 2.0]])
    else:
        D = np.array([[4.0]])
    X = sp.csc_matrix(D)
    with Engine(X) as src, src.shuffle(3) as sh:
        Y = sh.csc()
        check_csc_equal(Y, synth.shuffle_columns_reference(X, 3))
    if shape == "dense_column":
        assert np.array_equal(Y.indices[Y.indptr[2]:Y.indptr[3]], np.arange(3000))
        assert not np.array_equal(Y.data[Y.indptr[2]:Y.indptr[3]], D[:, 2])


# ---- 2. the same handle as a host upload; source and repeatability ------------------------------
@pytest.mark.parametrize("name,kind", [("pbmc", "int"), ("c1s3", "int-fp64"), ("c1s2", "real"),
                                       ("c1s1", "int")])
def test_shuffled_handle_equals_host_upload(name, kind):
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    X = KINDS[kind](load_counts(name))
    ref = synth.shuffle_columns_reference(X, 31)
    assert ref.getnnz(axis=1).min() > 0
    with Engine(X) as src:
        before = runs(src)
        with src.shuffle(31) as a, src.shuffle(31) as b, Engine(ref) as host:
            check_csc_equal(a.csc(), b.csc())
            got, again, want = runs(a), runs(b), runs(host)
            assert a.layout_info() == host.layout_info()
            assert_same_runs(got, want)
            assert_same_runs(again, want)
        assert_same_runs(runs(src), before)
        check_csc_equal(src.csc(), sp.csc_matrix(X))


# ---- 3. C2 size ---------------------------------------------------------------------------------
def test_shuffle_at_c2_size():
    """20k genes x 100k cells (~1.6e8 nonzeros) generated on the device: colptr kept, rows
    strictly increasing, every column's values kept, and 5000 sampled columns bitwise equal to the
    restatement."""
    import torch
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    (colptr, rowidx, values), X = c2_device_matrix()
    n, m = X.shape
    seed = 123
    with Engine.from_device_csc(n, m, X.nnz, colptr, rowidx, values) as src:
        with src.shuffle(seed) as sh:
            Y = sh.csc()
    assert np.array_equal(Y.indptr, X.indptr)
    col = np.repeat(np.arange(m, dtype=np.int64), np.diff(X.indptr))
    step = np.diff(Y.indices.astype(np.int64))
    assert np.all(step[col[1:] == col[:-1]] > 0)
    # per-column multisets of the (integer) counts: sort (column, value) keys on the device
    assert np.all(X.data == np.round(X.data))
    vmax = int(max(X.data.max(), Y.data.max())) + 1
    dev = torch.device("cuda", 0)
    c = torch.from_numpy(col).to(dev) * vmax
    kx = torch.sort(c + torch.from_numpy(X.data.astype(np.int64)).to(dev)).values
    ky = torch.sort(c + torch.from_numpy(Y.data.astype(np.int64)).to(dev)).values
    assert torch.equal(kx, ky)
    del c, kx, ky
    for j in np.sort(np.random.default_rng(5).choice(m, 5000, replace=False)):
        b, e = X.indptr[j], X.indptr[j + 1]
        s = synth.shuffle_rows(seed, j, n, e - b)
        o = np.argsort(s)
        assert np.array_equal(Y.indices[b:e], s[o]), j
        assert np.array_equal(Y.data[b:e], X.data[b:e][o]), j


# ---- 4. empty genes and errors ------------------------------------------------------------------
def test_shuffle_that_empties_a_gene():
    from ccfindr_b200 import synth
    from ccfindr_b200._lib import VbnmfError
    from ccfindr_b200.engine import Engine
    n, m = 8, 4   # every gene holds one entry
    X = sp.csc_matrix((np.arange(1.0, 9.0), np.arange(8), np.arange(0, 9, 2)), shape=(n, m))
    seed = next(s for s in range(100)
                if (synth.shuffle_columns_reference(X, s).getnnz(axis=1) == 0).any())
    ref = synth.shuffle_columns_reference(X, seed)
    empty = ref.getnnz(axis=1) == 0
    w0, h0 = synth.uniform_init(n, m, 2, 1)
    with Engine(X) as src, src.shuffle(seed) as sh, Engine(ref) as host:
        check_csc_equal(sh.csc(), ref)
        cells = sh.qc_stats()["gene_cells"]
        assert np.all(cells[empty] == 0) and np.all(cells[~empty] > 0)
        for eng in (sh, host):
            with pytest.raises(VbnmfError) as e:
                eng.ml_run(w0, h0, Itmax=5)
            assert e.value.code == 6
        src.ml_run(w0, h0, Itmax=5)   # the source has no empty gene


def test_shuffle_errors():
    from ccfindr_b200._lib import VbnmfError
    from ccfindr_b200.engine import Engine
    tall = sp.csc_matrix((np.ones(3), np.array([0, 5, 3999999]), np.array([0, 2, 3])),
                         shape=(4000000, 2))
    with Engine(tall) as eng:
        with pytest.raises(VbnmfError, match="929792") as e:
            eng.shuffle(1)
        assert e.value.code == 1
    # a column with more stored entries than rows (repeated entries): k distinct rows cannot exist
    rep = sp.csc_matrix((np.ones(4), np.array([0, 0, 1, 1]), np.array([0, 3, 4])), shape=(2, 2))
    with Engine(rep) as eng:
        with pytest.raises(VbnmfError, match="more entries") as e:
            eng.shuffle(1)
        assert e.value.code == 1
        with eng.subset(np.ones(2, bool), np.array([False, True])) as ok:  # still usable
            assert ok.nnz == 1


# ---- 5. front end -------------------------------------------------------------------------------
def test_factorize_device_shuffle_equals_host_shuffled_input(monkeypatch):
    from ccfindr_b200 import api, synth
    from ccfindr_b200.engine import Engine
    X = load_counts("pbmc")
    kw = dict(ranks=[2, 3], nrun=2, randomize=True, nsmpl=2, Itmax=40, verbose=0, seed=4)
    with pytest.raises(ValueError):
        api.factorize(api.scNMFSet(X), ranks=[2], device_shuffle=True)

    uploads = []
    init = Engine.__init__

    def counting_init(self, counts=None, *a, **k):
        if counts is not None:
            uploads.append(counts.shape)
        init(self, counts, *a, **k)

    def no_dense(*a, **k):
        raise AssertionError("the counts were densified")

    with monkeypatch.context() as mp:
        mp.setattr(Engine, "__init__", counting_init)
        mp.setattr(sp.csc_matrix, "todense", no_dense)
        dev = api.factorize(api.scNMFSet(X), device_shuffle=True, **kw)
    assert uploads == [X.shape]

    seeds = []

    def host_shuffle(self, seed):
        seeds.append(seed)
        return Engine(synth.shuffle_columns_reference(self.csc(), seed))

    with monkeypatch.context() as mp:
        mp.setattr(Engine, "shuffle", host_shuffle)
        host = api.factorize(api.scNMFSet(X), device_shuffle=True, **kw)
    assert seeds == [4 * 100003 + 1000 * r + 37 * i for r in (2, 3) for i in (1, 2)]
    for k in range(2):
        assert np.array_equal(dev.basis[k], host.basis[k])
        assert np.array_equal(dev.coeff[k], host.coeff[k])
    assert sorted(dev.measure) == sorted(host.measure)
    for key in dev.measure:
        assert np.array_equal(dev.measure[key], host.measure[key], equal_nan=True), key
    assert np.all(np.isfinite(dev.measure["r_se"]))
