"""CPU checks of synth.shuffle_columns_reference, the NumPy restatement of the on-device column
shuffle (csrc/shuffle.cuh) that the GPU tests compare Engine.shuffle against bit for bit."""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy import stats

from conftest import load_counts
from ccfindr_b200 import synth


def test_umulhi_is_the_high_word_of_the_product():
    u = np.random.default_rng(0).integers(0, 2**64, size=2000, dtype=np.uint64, endpoint=False)
    u[:4] = [0, 1, 2**64 - 1, 2**63]
    for n in (1, 3, 20000, 2**31 - 1):
        got = synth._umulhi(u, n)
        assert [int(v) for v in got] == [(int(x) * n) >> 64 for x in u]


def test_draws_are_the_counter_stream_of_tag_3():
    for seed, j in ((1, 0), (7, 12345), (2**63 + 5, 2**31 - 1)):
        st = synth._Stream(seed, (3 << 62) | j)
        want = [st.next() for _ in range(100)]
        assert [int(v) for v in synth._shuffle_draws(seed, j, 100)] == want


def test_rows_are_the_first_distinct_draws():
    for seed, j, n, k in ((3, 0, 20000, 1600), (3, 1, 200, 50), (5, 9, 7, 7), (5, 2, 1, 1)):
        rows = synth.shuffle_rows(seed, j, n, k)
        st = synth._Stream(seed, (3 << 62) | j)
        seen, want = set(), []
        while len(want) < k:
            r = (st.next() * n) >> 64
            if r not in seen:
                seen.add(r)
                want.append(r)
        assert rows.tolist() == want


def check_shuffled(X, Y):
    X, Y = sp.csc_matrix(X), sp.csc_matrix(Y)
    n, m = X.shape
    assert Y.shape == X.shape
    assert np.array_equal(Y.indptr, X.indptr)
    assert Y.indices.min(initial=0) >= 0 and Y.indices.max(initial=0) < n
    for j in range(m):
        b, e = X.indptr[j], X.indptr[j + 1]
        assert np.all(np.diff(Y.indices[b:e]) > 0), j          # distinct and sorted
        assert np.array_equal(np.sort(Y.data[b:e]), np.sort(X.data[b:e])), j


def with_zeros(X):
    """X with an appended gene that stores explicit zeros in the first two cells."""
    n, m = X.shape
    C = X.tocoo()
    Y = sp.csc_matrix((np.concatenate([C.data, [0.0, 0.0]]),
                       (np.concatenate([C.row, [n, n]]), np.concatenate([C.col, [0, 1]]))),
                      shape=(n + 1, m))
    Y.sort_indices()
    return Y


@pytest.mark.parametrize("name", ["tiny", "pbmc"])
def test_columns_keep_pointers_and_values(name):
    X = load_counts(name)
    for M in (X, with_zeros(X)):
        Y = synth.shuffle_columns_reference(M, 11)
        check_shuffled(M, Y)
        assert Y.nnz == M.nnz and (Y.data == 0).sum() == (M.data == 0).sum()
        assert not np.array_equal(Y.indices, M.indices)


def test_full_column_is_a_permutation_and_one_row_works():
    n = 64
    X = sp.csc_matrix(np.arange(1.0, n * 3 + 1).reshape(n, 3))
    Y = synth.shuffle_columns_reference(X, 5)
    check_shuffled(X, Y)
    for j in range(3):
        assert Y.indices[Y.indptr[j]:Y.indptr[j + 1]].tolist() == list(range(n))
        assert not np.array_equal(Y.data[Y.indptr[j]:Y.indptr[j + 1]], X[:, j].toarray().ravel())
    one = sp.csc_matrix(np.array([[2.0, 0.0, 5.0]]))
    check_shuffled(one, synth.shuffle_columns_reference(one, 1))
    assert (synth.shuffle_columns_reference(one, 1) != one).nnz == 0


def test_same_seed_same_result_other_seed_differs():
    X = load_counts("pbmc")
    a = synth.shuffle_columns_reference(X, 21)
    b = synth.shuffle_columns_reference(X, 21)
    c = synth.shuffle_columns_reference(X, 22)
    assert np.array_equal(a.indices, b.indices) and np.array_equal(a.data, b.data)
    assert not np.array_equal(a.indices, c.indices)


def test_unsorted_input_and_too_many_entries():
    X = load_counts("tiny")
    rev = np.concatenate([np.arange(X.indptr[j], X.indptr[j + 1])[::-1] for j in range(X.shape[1])])
    U = sp.csc_matrix((X.data[rev], X.indices[rev], X.indptr), shape=X.shape)
    assert not U.has_sorted_indices
    a = synth.shuffle_columns_reference(U, 3)
    b = synth.shuffle_columns_reference(X, 3)
    assert np.array_equal(a.indices, b.indices) and np.array_equal(a.data, b.data)
    with pytest.raises(ValueError):
        synth.shuffle_rows(1, 0, 3, 4)


def uniform_sample_matrix(m=20000, n=200, k=50):
    """m columns of k entries in n rows; entry t of every column holds the value t + 1."""
    indptr = np.arange(m + 1, dtype=np.int64) * k
    indices = np.tile(np.arange(k, dtype=np.int32) * (n // k), m)
    data = np.tile(np.arange(1.0, k + 1), m)
    return sp.csc_matrix((data, indices, indptr), shape=(n, m))


def test_rows_are_uniform_and_values_are_permuted():
    n, k = 200, 50
    X = uniform_sample_matrix(n=n, k=k)
    Y = synth.shuffle_columns_reference(X, 2024)
    hits = np.bincount(Y.indices, minlength=n)
    p = stats.chisquare(hits).pvalue
    assert p > 1e-3, p
    # value t + 1 lands at the rank of s_t among the column's rows: rank must not follow t
    rank = np.tile(np.arange(k), X.shape[1])
    t = Y.data.astype(np.int64) - 1
    rho = stats.spearmanr(rank, t).statistic
    assert abs(rho) < 0.02, rho
