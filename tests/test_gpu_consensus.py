"""GPU tests of the consensus measures: engine.consensus (csrc/consensus.cuh, vbnmf_consensus)
against the NumPy restatement oracle/oracle_consensus.py, bit for bit, and factorize /
vb_factorize with device_consensus=True against the host measures."""
import ctypes as C
import re

import numpy as np
import pytest

from conftest import load_counts
from oracle import oracle_consensus as oc
from test_api_cpu import _label_runs

pytestmark = pytest.mark.gpu


def planted(m, nrun, K, p, seed):
    return np.stack(_label_runs(np.random.default_rng(seed), m, nrun, K, p)) - 1


def tie_heavy(m, nrun, K, seed):
    return np.random.default_rng(seed).integers(0, K, size=(nrun, m))


CASES = {
    "tie_G27": lambda: tie_heavy(1000, 3, 3, 1),
    "tie_G600": lambda: tie_heavy(5000, 4, 5, 2),
    "tie_G4k": lambda: tie_heavy(30000, 6, 4, 3),
    "planted_G5k": lambda: planted(100000, 20, 15, 0.01, 4),
    "planted_G11k": lambda: planted(100000, 20, 15, 0.02, 5),
}


@pytest.mark.parametrize("case", list(CASES))
def test_device_tree_equals_the_restatement(case):
    from ccfindr_b200 import api, engine
    L = CASES[case]()
    nrun, m = L.shape
    got = engine.consensus(L)
    s1, s2, G, merges = oc.tree(L)
    assert (got["s1"], got["s2"], got["ngroups"]) == (s1, s2, G)
    assert np.array_equal(got["merges"], merges)
    assert got["rescans"] >= G - 1
    assert engine.consensus(L, tree=False) == dict(s1=s1, s2=s2)
    d, c = api.consensus_from_labels(list(L + 1))
    assert d == api.dispersion_from_moments(s1, s2, m, nrun)
    assert c == api.cophenet_from_merges(s1, s2, m, nrun, merges)
    assert abs(d - api.dispersion_from_labels(list(L + 1))) < 1e-12


def test_repeated_calls_are_identical():
    from ccfindr_b200 import engine
    L = CASES["planted_G5k"]()
    a, b = engine.consensus(L), engine.consensus(L)
    assert a.keys() == b.keys()
    assert all(np.array_equal(a[k], b[k]) for k in a)


def test_structure_at_1_3m_cells():
    """1.3M cells x 20 runs, G ~ 7e4 groups (the host cophenetic value is NaN past 6,000)."""
    from ccfindr_b200 import api, engine
    L = planted(1300000, 20, 15, 0.02, 7).astype(np.int32)
    nrun, m = L.shape
    res = engine.consensus(L)
    G, mg = res["ngroups"], res["merges"]
    assert G >= 50000 and mg.shape == (G - 1, 5)
    a, b = mg[:, 0], mg[:, 1]
    assert (a < b).all() and len(np.unique(b)) == G - 1       # every group but one retired once
    retired = np.zeros(G, dtype=np.int64)
    retired[b] = np.arange(1, G)
    assert ((retired[a] == 0) | (retired[a] > np.arange(1, G))).all()   # a still active
    _, sz = np.unique(L.T, axis=0, return_counts=True)
    assert len(sz) == G
    P = m * (m - 1) // 2
    assert int((mg[:, 3] * mg[:, 4]).sum()) + int((sz.astype(np.int64) * (sz - 1) // 2).sum()) == P
    h = 1.0 - mg[:, 2] / (nrun * mg[:, 3] * mg[:, 4]).astype(np.float64)
    assert (h >= 0).all() and (h <= 1).all()
    mom = oc.moments(L)
    assert (res["s1"], res["s2"]) == mom
    d, c = api.consensus_from_labels(list(L + 1))
    assert np.isfinite(c) and 0 < c <= 1
    assert np.isnan(api.cophenet_from_labels(list(L + 1)))
    assert d == api.dispersion_from_moments(*mom, m, nrun)


def test_max_groups_refusal():
    from ccfindr_b200 import api, engine
    from ccfindr_b200._lib import ERR_MEMORY, VbnmfError
    L = CASES["tie_G600"]()
    G = oc.tree(L)[2]
    with pytest.raises(VbnmfError) as e:
        engine.consensus(L, max_groups=G - 1)
    assert e.value.code == ERR_MEMORY and e.value.ngroups == G
    assert engine.consensus(L, max_groups=G)["ngroups"] == G
    with pytest.warns(UserWarning, match="label groups"):
        d, c = api.consensus_from_labels(list(L + 1), max_groups=10)
    assert np.isnan(c) and d == api.consensus_from_labels(list(L + 1), tree=False)[0]


def test_argument_errors():
    from ccfindr_b200 import _lib
    from ccfindr_b200._lib import ERR_ARG
    lib = _lib.load()

    def call(L, nrun, m, K, merges=True, cap=None):
        L = np.ascontiguousarray(L, dtype=np.int32)
        mom = np.zeros(2, dtype=np.int64)
        ng, resc = C.c_int64(0), C.c_int64(0)
        mg = np.zeros((64, 5), dtype=np.int64)
        rc = lib.vbnmf_consensus(0, m, nrun, K, L.ctypes.data_as(_lib.c_i32p), 0,
                                 mom.ctypes.data_as(_lib.c_i64p), C.byref(ng),
                                 mg.ctypes.data_as(_lib.c_i64p) if merges else None,
                                 m - 1 if cap is None else cap, C.byref(resc))
        return rc, ng.value
    L = tie_heavy(50, 3, 4, 9)
    assert call(L, 3, 50, 4) == (0, oc.tree(L)[2])
    assert call(L, 3, 50, 3)[0] == ERR_ARG                    # label 3 outside 0 ... K-1
    bad = L.copy(); bad[1, 7] = -1
    assert call(bad, 3, 50, 4)[0] == ERR_ARG
    assert call(L, 3, 50, 241)[0] == ERR_ARG                  # K x K table above shared memory
    assert call(L, 0, 50, 4)[0] == ERR_ARG
    assert call(L, 3, 0, 4)[0] == ERR_ARG
    assert call(L[:1, :1], 1, 200000000, 4)[0] == ERR_ARG     # nrun ceil(m/2)^2 >= 2^53
    G = oc.tree(L)[2]
    assert call(L, 3, 50, 4, cap=G - 2) == (ERR_ARG, G)       # merge_cap < G - 1
    assert b"merge_cap" in lib.vbnmf_last_error(None)


def test_factorize_device_consensus_on_pbmc():
    from ccfindr_b200 import api
    X = load_counts("pbmc")
    kw = dict(ranks=[2, 3], nrun=5, Itmax=200, verbose=0, store_connectivity=True)
    host = api.factorize(api.scNMFSet(X), **kw)
    dev = api.factorize(api.scNMFSet(X), device_consensus=True, **kw)
    assert np.array_equal(host.measure["likelihood"], dev.measure["likelihood"])
    for a, b in zip(host.basis + host.coeff, dev.basis + dev.coeff):
        assert np.array_equal(a, b)
    assert np.max(np.abs(host.measure["dispersion"] - dev.measure["dispersion"])) < 1e-12
    assert np.max(np.abs(host.measure["cophenetic"] - dev.measure["cophenetic"])) < 5e-3
    L = np.stack(dev.metadata["labels"]) - 1
    s1, s2, G, merges = oc.tree(L)
    m = L.shape[1]
    assert dev.measure["cophenetic"][-1] == api.cophenet_from_merges(s1, s2, m, 5, merges)
    assert dev.measure["dispersion"][-1] == api.dispersion_from_moments(s1, s2, m, 5)
    with pytest.raises(ValueError, match="average"):
        api.factorize(api.scNMFSet(X), linkage="single", device_consensus=True, **kw)


def test_vb_factorize_device_dispersion(capsys):
    from ccfindr_b200 import api
    X = load_counts("pbmc")
    kw = dict(ranks=[2, 3], nrun=3, Itmax=50, verbose=2, progress_bar=False)
    disp = {}
    for flag in (False, True):
        api.vb_factorize(api.scNMFSet(X), device_consensus=flag, **kw)
        disp[flag] = [float(v) for v in re.findall(r"dispersion = (\S+)", capsys.readouterr().out)]
    assert len(disp[True]) == len(disp[False]) >= 2
    assert np.max(np.abs(np.array(disp[True]) - np.array(disp[False]))) < 1e-12
