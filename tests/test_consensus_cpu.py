"""CPU tests of the consensus measures assembled from integer moments and the merge list
(api.dispersion_from_moments, api.cophenet_from_merges) and of their NumPy restatement
(oracle/oracle_consensus.py), the reference for the device path (vbnmf_consensus)."""
import numpy as np
import pytest

from ccfindr_b200 import api
from oracle import oracle_consensus as oc
from oracle import oracle_dense as od
from test_api_cpu import _label_runs


def _tie_heavy(rng, nrun, K, m):
    return rng.integers(0, K, size=(nrun, m))


def _conav(L):
    """the literal m(m-1)/2 average connectivity vector (R/factorize.R:51-60)"""
    nrun, m = L.shape
    conav = np.zeros(m * (m - 1) // 2)
    for lab in L:
        h = np.zeros((int(lab.max()) + 1, m))
        h[lab, np.arange(m)] = 1.0
        conav += od.connectivity(h)
    return conav / nrun


def _cophenet_direct(L, merges):
    """cor(d, c) over all cell pairs with the G x G cophenetic matrix of the merge list built
    explicitly (same-group pairs contribute d = c = 0), weighted by n_a n_b."""
    tup, sz = oc.groups(L)
    nrun = L.shape[0]
    G = len(sz)
    agree = np.zeros((G, G))
    for t in range(nrun):
        agree += tup[:, t][:, None] == tup[:, t][None, :]
    D = 1.0 - agree / nrun
    C = np.zeros((G, G))
    members = [[g] for g in range(G)]
    for a, b, ip, na, nb in merges:
        h = 1.0 - ip / (nrun * na * nb)
        C[np.ix_(members[a], members[b])] = h
        C[np.ix_(members[b], members[a])] = h
        members[a] += members[b]
    iu = np.triu_indices(G, 1)
    w = (sz[:, None] * sz[None, :]).astype(float)[iu]
    d, c = D[iu], C[iu]
    same = float(np.sum(sz * (sz - 1) / 2))
    N = same + w.sum()
    md, mc = (w * d).sum() / N, (w * c).sum() / N
    vd = (w * (d - md) ** 2).sum() + same * md ** 2
    vc = (w * (c - mc) ** 2).sum() + same * mc ** 2
    cov = (w * (d - md) * (c - mc)).sum() + same * md * mc
    return float(cov / np.sqrt(vd * vc))


@pytest.mark.parametrize("nrun,K,m", [(1, 3, 40), (2, 2, 60), (5, 4, 150), (10, 6, 200)])
def test_moments_equal_the_pairwise_definition(nrun, K, m):
    L = _tie_heavy(np.random.default_rng(nrun * K), nrun, K, m)
    s1, s2 = oc.moments(L)
    assert (s1, s2) == oc.moments_pairwise(L)
    disp = api.dispersion_from_moments(s1, s2, m, nrun)
    assert abs(disp - api.dispersion_from_labels(list(L + 1))) < 1e-12
    assert abs(disp - od.dispersion(_conav(L), m)) < 1e-12


@pytest.mark.parametrize("nrun", [1, 2, 3, 4, 6, 10])
@pytest.mark.parametrize("K", [2, 3, 6])
def test_row_cached_greedy_reproduces_the_literal_greedy(nrun, K):
    """Tie-heavy labels: few runs and labels make equal q values common."""
    rng = np.random.default_rng(100 * nrun + K)
    L = _tie_heavy(rng, nrun, K, 400)
    tup, sz = oc.groups(L)
    assert len(sz) <= 400
    ip = oc.ip_matrix(tup, sz)
    lit = oc.greedy_literal(ip, sz, nrun)
    cached, rescans = oc.greedy_cached(ip, sz, nrun)
    assert lit.shape == (len(sz) - 1, 5)
    assert np.array_equal(lit, cached)
    assert rescans >= len(sz) - 1


@pytest.mark.parametrize("nrun,K,m", [(3, 3, 80), (5, 4, 150), (8, 5, 250)])
def test_assembled_cophenetic_equals_the_direct_weighted_computation(nrun, K, m):
    L = _tie_heavy(np.random.default_rng(m), nrun, K, m)
    s1, s2, G, merges = oc.tree(L)
    got = api.cophenet_from_merges(s1, s2, m, nrun, merges)
    assert abs(got - _cophenet_direct(L, merges)) < 1e-12


@pytest.mark.parametrize("m,nrun,rank,noise", [(40, 4, 3, 0.2), (150, 6, 4, 0.1), (300, 10, 5, 0.3)])
def test_assembled_measures_match_the_literal_ones(m, nrun, rank, noise):
    """the cases of test_api_cpu.py::test_consensus_measures_from_label_groups_match_the_literal_ones"""
    rng = np.random.default_rng(m + nrun)
    L = np.stack(_label_runs(rng, m, nrun, rank, noise)) - 1
    conav = _conav(L)
    s1, s2, G, merges = oc.tree(L)
    assert abs(api.dispersion_from_moments(s1, s2, m, nrun) - od.dispersion(conav, m)) < 1e-12
    got = api.cophenet_from_merges(s1, s2, m, nrun, merges)
    assert abs(got - od.cophenet(conav, m, "average")) < 5e-3


def test_edge_cases():
    # one run: every distance is 0 or 1; the tree joins the clusters at height 1
    L = np.array([[0, 0, 1, 1, 2, 2, 2]])
    s1, s2, G, merges = oc.tree(L)
    assert G == 3 and (s1, s2) == (5, 5)
    assert api.cophenet_from_merges(s1, s2, 7, 1, merges) == pytest.approx(1.0, abs=1e-15)
    assert abs(api.dispersion_from_moments(s1, s2, 7, 1) - od.dispersion(_conav(L), 7)) < 1e-15
    # one group: no variance
    L = np.zeros((4, 9), dtype=int)
    s1, s2, G, merges = oc.tree(L)
    assert G == 1 and merges.shape == (0, 5)
    assert np.isnan(api.cophenet_from_merges(s1, s2, 9, 4, merges))
    assert api.dispersion_from_moments(s1, s2, 9, 4) == pytest.approx(1.0, abs=1e-15)
    # m = 2: one pair, NaN as cophenet_from_labels
    L = np.array([[0, 1], [0, 0]])
    s1, s2, G, merges = oc.tree(L)
    assert np.isnan(api.cophenet_from_merges(s1, s2, 2, 2, merges))
    assert abs(api.dispersion_from_moments(s1, s2, 2, 2) - api.dispersion_from_labels(list(L + 1))) < 1e-15
    # unused label values change nothing
    rng = np.random.default_rng(4)
    L = rng.integers(0, 3, size=(5, 60))
    assert oc.tree(L * 2 + 1)[:3] == oc.tree(L)[:3]
    assert np.array_equal(oc.tree(L * 2 + 1)[3], oc.tree(L)[3])
