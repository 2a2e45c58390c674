"""CPU checks of the factor-model oracle (oracle/factor_oracle.py, DESIGN.md 2 "Factor models" and 4.10): the
canonical definition against the reference's recipe (lil_matrix + numpy @), zeros not stored, float32 factors, and the
emulated two-scale screen within its bound."""
import os
import sys

import numpy as np
import pytest
from scipy.sparse import csr_matrix, lil_matrix

from oracle.factor_oracle import (canon_factor_full, canon_factor_scores, canon_factor_topn, emulate_factor_screen,
                                  factor_screen_delta, ref_factor_predict)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(U=300, I=500, D=24, density=0.03, seed=0, dtype=np.float64):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((U, D)).astype(dtype)
    Q = rng.standard_normal((I, D)).astype(dtype)
    X = csr_matrix((rng.random((U, I)) < density).astype(np.float64))
    return P, Q, X


def _bound(P, Q):
    """A few ulp * D of ||p_u|| ||q_j||: the distance between two summation orders of the same products."""
    D = P.shape[1]
    rp = np.linalg.norm(np.asarray(P, np.float64), axis=1)
    rq = np.linalg.norm(np.asarray(Q, np.float64), axis=1)
    return 4 * (D + 2) * 2.0**-53 * np.outer(rp, rq)


def _same_lists_outside_near_ties(got, S, N, bound):
    """Canonical lists against the reference's scores S [U x I] (dense): every listed value within the bound of the
    reference's, and the item sets equal except inside groups of values closer than 2 * bound."""
    for u in range(S.shape[0]):
        n = got["len"][u]
        if n == 0:
            continue
        idx = got["idx"][u, :n]
        assert np.all(np.abs(got["val"][u, :n] - S[u, idx]) <= bound[u, idx])
        order = np.lexsort((np.arange(S.shape[1]), -S[u]))[:n]
        for a, b in zip(idx, order):
            if a != b:
                assert abs(S[u, a] - S[u, b]) <= 2 * max(bound[u, a], bound[u, b])


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_canonical_against_the_reference_recipe(dtype):
    P, Q, X = _model(dtype=dtype)
    X[::7] = 0  # users without history
    X.eliminate_zeros()
    ref = ref_factor_predict(P, Q, X)
    full = canon_factor_full(P.astype(np.float64), Q.astype(np.float64), X)
    canon = csr_matrix(full)
    ref.sort_indices()
    assert np.array_equal(canon.indptr, ref.indptr) and np.array_equal(canon.indices, ref.indices)
    # float32 factors: the reference computes in float32, the definition in float64 on the widened values
    tol = _bound(P, Q) if dtype == np.float64 else 2.0**-22 * P.shape[1] * np.outer(
        np.linalg.norm(P.astype(np.float64), axis=1), np.linalg.norm(Q.astype(np.float64), axis=1))
    r, c = canon.nonzero()
    assert np.all(np.abs(canon.data - np.asarray(ref[r, c]).ravel()) <= tol[r, c])
    top = canon_factor_topn(P.astype(np.float64), Q.astype(np.float64), X, 20)
    _same_lists_outside_near_ties(top, ref.toarray(), 20, tol)
    assert np.all(top["len"][np.diff(X.indptr) == 0] == 0)


def test_zero_scores_are_not_stored_by_lil_matrix():
    P = np.array([[1.0, 0.0], [0.0, 0.0], [1.0, 1.0]])
    Q = np.array([[0.0, 1.0], [1.0, 0.0], [1.0, -1.0], [2.0, 3.0]])
    X = csr_matrix(np.ones((3, 4)))
    ref = ref_factor_predict(P, Q, X)
    want = P @ Q.T
    assert ref.nnz == np.count_nonzero(want)  # user 0: q_0 gives 0.0, user 1: all 0.0, user 2: q_2 gives 0.0
    assert np.diff(ref.indptr).tolist() == [3, 0, 3]
    assert np.array_equal(csr_matrix(canon_factor_full(P, Q, X)).toarray(), ref.toarray())
    top = canon_factor_topn(P, Q, X, 4)
    assert top["len"].tolist() == [3, 0, 3]


def test_definition_is_the_left_fold():
    rng = np.random.default_rng(3)
    P = rng.standard_normal((5, 9)) * np.exp2(rng.integers(-30, 30, size=(5, 9)))
    Q = rng.standard_normal((6, 9)) * np.exp2(rng.integers(-30, 30, size=(6, 9)))
    S = canon_factor_scores(P, Q, np.arange(5))
    for u in range(5):
        for j in range(6):
            s = P[u, 0] * Q[j, 0]
            for d in range(1, 9):
                s = s + P[u, d] * Q[j, d]
            assert S[u, j] == s


def test_history_filter_and_order():
    P, Q, X = _model(U=40, I=60, D=5, density=0.2, seed=4)
    allowed = np.ones(60, dtype=bool)
    allowed[::5] = False
    full = canon_factor_full(P, Q, X, remove_history=True, allowed=allowed)
    top = canon_factor_topn(P, Q, X, 7, remove_history=True, allowed=allowed)
    for u in range(40):
        n = top["len"][u]
        idx = top["idx"][u, :n]
        assert not np.any(np.isin(idx, X.indices[X.indptr[u] : X.indptr[u + 1]]))
        assert np.all(allowed[idx])
        cols = np.flatnonzero(full[u] != 0.0)
        order = cols[np.lexsort((cols, -full[u, cols]))][:7]
        assert np.array_equal(idx, order) and np.array_equal(top["val"][u, :n], full[u, order])


@pytest.mark.parametrize("D", [1, 7, 128, 1024])
def test_emulated_screen_within_the_bound(D):
    rng = np.random.default_rng(D)
    U, I = (60, 50) if D == 1024 else (200, 150)
    for scale_p, scale_q in ((0, 0), (40, -40), (-40, 40), (-300, -300)):
        P = rng.standard_normal((U, D)) * np.exp2(scale_p + rng.integers(-3, 3, size=(U, 1)))
        Q = rng.standard_normal((I, D)) * np.exp2(scale_q + rng.integers(-3, 3, size=(I, 1)))
        S_hat = emulate_factor_screen(P, Q)
        S = canon_factor_scores(P, Q, np.arange(U))
        ratio = np.abs(S_hat - S) / factor_screen_delta(P, Q)
        assert np.all(ratio <= 1.0), (D, scale_p, scale_q, ratio.max())


def test_reference_predict_is_the_restated_recipe():
    """With the reference installed (baseline/_ref): its own FactorizationAlgorithm._predict on a small model equals the
    restatement, and its shape check raises AssertionError."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "recpack")):
        pytest.skip("baseline/_ref not installed")
    sys.path.insert(0, ref_dir)
    try:
        import recpack.algorithms.base as rb
    finally:
        sys.path.remove(ref_dir)
    P, Q, X = _model(U=50, I=70, D=6, seed=5)
    X[::4] = 0
    X.eliminate_zeros()
    algo = rb.FactorizationAlgorithm(num_components=6)
    algo.user_embedding_, algo.item_embedding_ = P, Q
    got = csr_matrix(algo._predict(X))
    want = ref_factor_predict(P, Q, X)
    got.sort_indices()
    want.sort_indices()
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data)
    with pytest.raises(AssertionError):
        algo._predict(X[:, :60])
