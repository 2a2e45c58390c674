"""The dense EASE oracle (oracle/ease_dense_oracle.py) against scipy and the reference's matrix formulas; no GPU."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.ease_dense_oracle import canon_dense_scores, canon_dense_topn, canon_ease_from_inverse, canon_gram
from oracle.signed_oracle import canon_predict_signed


def _tied_model(I, seed):
    """Small integers times 0.125: exact ties, zeros, negatives, and rows that cancel."""
    rng = np.random.default_rng(seed)
    B = rng.integers(-4, 5, size=(I, I)).astype(np.float64) * 0.125
    B[:, 3] = 0.0
    B[0, 5], B[1, 5] = 0.75, -0.75  # column 5 of a user holding items 0 and 1 sums to exactly 0.0
    B[:, 7] = -np.abs(B[:, 7]) - 0.125  # negative only
    B[9] = -np.abs(B[9]) - 0.125  # a user holding only item 9 has negative scores only
    return B


def _interactions(U, I, seed):
    rng = np.random.default_rng(seed)
    X = (rng.random((U, I)) < 0.2).astype(np.float64)
    X[0] = 0.0  # empty history
    X[1] = 0.0
    X[1, [0, 1]] = 1.0
    X[2] = 1.0  # every item held
    X[3] = 0.0
    X[3, 9] = 1.0
    return csr_matrix(X)


def test_gram_counts():
    X = _interactions(50, 30, 1)
    Xd = X.toarray().astype(np.int64)
    G = canon_gram(X)
    assert G.dtype == np.int64 and np.array_equal(G, Xd.T @ Xd)


@pytest.mark.parametrize("mask", [False, True])
def test_scores_are_scipy_csr_at_dense(mask):
    I = 40
    B = _tied_model(I, 2)
    X = _interactions(60, I, 3)
    S = canon_dense_scores(X.indptr, X.indices, B, mask_history=mask)
    want = (X.astype(bool).astype(np.float64) @ B)
    if mask:
        want[X.toarray() > 0] = 0.0
    assert np.array_equal(S.view(np.int64), np.asarray(want).view(np.int64))  # bit for bit, signed zeros included
    assert S[1, 5] == 0.0 and np.all(S[0] == 0.0)
    # gathered rows give the same bits as the whole B
    items = np.unique(X.indices)
    assert np.array_equal(canon_dense_scores(X.indptr, X.indices, (items, B[items]), mask).view(np.int64), S.view(np.int64))


@pytest.mark.parametrize("N", [1, 5, 40, 100])
@pytest.mark.parametrize("mask", [False, True])
def test_topn_agrees_with_the_signed_oracle(N, mask):
    I = 40
    B = _tied_model(I, 4)
    X = _interactions(60, I, 5)
    got = canon_dense_topn(canon_dense_scores(X.indptr, X.indices, B, mask_history=mask), N)
    want = canon_predict_signed(X, csr_matrix(B), N, remove_history=mask)
    for k in ("idx", "val", "len"):
        assert np.array_equal(got[k], want[k]), k
    assert got["len"][0] == 0 and np.all(got["idx"][0] == -1)
    assert got["len"][3] > 0 and np.all(got["val"][3, : got["len"][3]] < 0)  # negative scores are ranked too


def test_topn_rejects_nan():
    with pytest.raises(AssertionError):
        canon_dense_topn(np.array([[1.0, np.nan]]), 2)


@pytest.mark.parametrize("with_w", ["none", "finite", "inf"])
def test_closed_form_agrees_with_the_reference_formula(with_w):
    rng = np.random.default_rng(6)
    I = 30
    A = rng.standard_normal((I, I))
    P = A @ A.T + I * np.identity(I)
    P[4, :] = 0.0  # an item nobody saw: P_4j = P_j4 = 0 off the diagonal
    P[:, 4] = 0.0
    P[4, 4] = 0.5
    w = None if with_w == "none" else 1.0 / rng.integers(1, 9, I).astype(np.float64) ** 0.5
    if with_w == "inf":
        w[4] = np.inf
    B = canon_ease_from_inverse(P, w)
    with np.errstate(invalid="ignore", over="ignore"):
        ref = np.identity(I) - P @ np.diag(1.0 / np.diag(P))
        np.fill_diagonal(ref, 0.0)
        if w is not None:
            ref = ref @ np.diag(w)
    fin = np.isfinite(ref)
    assert np.array_equal(B[fin], ref[fin])
    nan_col = np.zeros((I, I), dtype=bool)
    if with_w == "inf":
        nan_col[:, 4] = True  # -(0 * (1 / P_44)) * inf; the reference's diagonal entry 0 * inf is NaN as well
        nan_col[4, 4] = False
    assert np.array_equal(np.isnan(B), nan_col)
    assert np.array_equal(np.isnan(ref), nan_col | (np.eye(I, dtype=bool) & nan_col.any(axis=0)[None, :]))
    assert np.all(np.diag(B) == 0.0) and not np.signbit(np.diag(B)).any()
