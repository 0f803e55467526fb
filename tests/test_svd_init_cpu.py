"""CPU tests of the 'svd' initializer as Engine.init_svd computes it (no GPU): every pair of
singular vectors k >= 1 oriented (synth.orient_svd_pairs), then the reference formula of
R/bayesian.R:116-149 (api.svd_init_from, which api.vb_init calls).  Checked on exact SVDs of the
golden matrices: equal to the literal formula where the pair is already dominant, independent of
the signs the SVD returned, and finite where the literal formula divides 0 by 0."""
import numpy as np
import pytest

from conftest import load_counts
from ccfindr_b200 import api, synth


def exact_svd(X, rank):
    u, d, vt = np.linalg.svd(np.asarray(X.todense()), full_matrices=False)
    return u[:, :rank], d[:rank], vt[:rank].T


def dominant(u, v, k):
    P = np.linalg.norm(np.maximum(u[:, k], 0)) * np.linalg.norm(np.maximum(v[:, k], 0))
    N = np.linalg.norm(np.minimum(u[:, k], 0)) * np.linalg.norm(np.minimum(v[:, k], 0))
    return P >= N


@pytest.mark.parametrize("counts", ["pbmc", "c1s1", "c1s2", "c1s3"])
def test_oriented_formula_equals_the_literal_one_on_dominant_pairs(counts):
    X = load_counts(counts)
    u, d, v = exact_svd(X, 10)
    w, h = synth.device_svd_init_reference(u, d, v)
    wl, hl = api.svd_init_from(u, d, v)
    for k in range(10):
        if k == 0 or dominant(u, v, k):
            assert np.array_equal(w[:, k], wl[:, k]) and np.array_equal(h[k], hl[k]), k
        else:
            assert not np.allclose(w[:, k], wl[:, k])
    # the oriented SVD is dominant everywhere: the literal formula then gives the same factors
    uo, vo = synth.orient_svd_pairs(u, v)
    assert all(dominant(uo, vo, k) for k in range(1, 10))
    wo, ho = api.svd_init_from(uo, d, vo)
    assert np.array_equal(w, wo) and np.array_equal(h, ho)


def test_vb_init_svd_is_the_helper_on_its_svd():
    """api.vb_init(..., 'svd') is svd_init_from on the SVD it takes (the dense branch here, so
    the SVD can be repeated exactly): the host behaviour is the reference formula, unchanged."""
    X = load_counts("tiny")
    n, m = X.shape
    hyper = dict(aw=1.0, bw=1.0, ah=1.0, bh=1.0)
    for rank in (13, 20):               # rank >= min(n, m) / 2: np.linalg.svd in vb_init
        w, h = api.vb_init(n, m, X, rank, hyper, "svd", seed=3)
        u, d, v = exact_svd(X, rank)
        wl, hl = api.svd_init_from(u, d, v)
        assert np.array_equal(w, wl) and np.array_equal(h, hl)
        if all(dominant(u, v, k) for k in range(1, rank)):
            wd, hd = synth.device_svd_init_reference(u, d, v)
            assert np.array_equal(w, wd) and np.array_equal(h, hd)


@pytest.mark.parametrize("counts", ["pbmc", "c1s3"])
def test_oriented_formula_does_not_depend_on_the_signs_of_the_svd(counts):
    X = load_counts(counts)
    u, d, v = exact_svd(X, 8)
    w, h = synth.device_svd_init_reference(u, d, v)
    rng = np.random.default_rng(1)
    for _ in range(6):
        s = rng.choice([-1.0, 1.0], size=8)
        ws, hs = synth.device_svd_init_reference(u * s, d, v * s)
        assert np.array_equal(ws, w) and np.array_equal(hs, h)
    assert (w[:, 1:] >= 0).all() and (h[1:] >= 0).all()
    # w_k and h_k carry the same norm sqrt(d_k P) for k >= 1, sqrt(d_0) for k = 0
    assert np.allclose(np.linalg.norm(w, axis=0), np.linalg.norm(h, axis=1), rtol=1e-12, atol=0)
    assert abs(np.linalg.norm(w[:, 0]) ** 2 - d[0]) < 1e-12 * d[0]


def test_oriented_formula_is_finite_where_the_literal_one_is_nan():
    """Two blocks: the second singular pair lives on genes 2-3 and cells 2-3 only.  Returned
    as (-u_1, -v_1) it has no positive part, and the literal formula divides 0 by 0."""
    X = np.array([[3.0, 3.0, 0.0, 0.0], [3.0, 3.0, 0.0, 0.0],
                  [0.0, 0.0, 1.0, 1.0], [0.0, 0.0, 1.0, 1.0]])
    s = np.sqrt(0.5)
    u = np.array([[s, 0.0], [s, 0.0], [0.0, -s], [0.0, -s]])
    v = u.copy()
    d = np.array([6.0, 2.0])
    assert np.allclose(u @ np.diag(d) @ v.T, X)
    with np.errstate(invalid="ignore", divide="ignore"):
        wl, hl = api.svd_init_from(u, d, v)
    assert np.isnan(wl[:, 1]).all() and np.isnan(hl[1]).all()
    w, h = synth.device_svd_init_reference(u, d, v)
    assert np.isfinite(w).all() and np.isfinite(h).all()
    assert (w >= 0).all() and (h >= 0).all()
    assert np.allclose(w @ h, X)               # two disjoint rank-one blocks: NNDSVD is exact
