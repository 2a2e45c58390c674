"""Scoring of signed similarity models: float64, bit-identical to scipy's ``X @ S`` (DESIGN.md 2, "Signed models").

A model with a negative value is loaded with rpk_model_load_signed_csr and scored by k_predict_signed (top-N) or by
the float64 row kernel (full CSR, and the users k_predict_signed hands over).  Every case compares lists, lengths and
scores with np.array_equal against oracle.signed_oracle.canon_predict_signed, in both modes and with and without
history removal.  The path cases build one branch of the kernel each, assert on the oracle side that the construction
reaches it, and, with the instrumented build (-DRPK_PHASE_PROF, one "[predict signed paths]" line per call), that the
kernel's counter of that branch moved."""
import re
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.signed_oracle import canon_predict_signed

DBG_MULTI_PASS, DBG_MANY_PASS = 4, 32
SG_EXACT_D = 2048  # histories at least this long go to the float64 row kernel (predict.cu)
CAP = 256          # survivors a list of N <= 128 holds (predict.cu: max(256, next_pow2(2N)))


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.debug_flags(0)
    eng.predict_item_filter(None)


def _signed_class():
    from recpack_b200 import ItemSimilarityMatrixAlgorithm

    class FixedModel(ItemSimilarityMatrixAlgorithm):
        """An algorithm whose model is given: the reference's base class contract with a signed similarity_matrix_."""

        def __init__(self, S, predict_topK=None, remove_history=False):
            super().__init__()
            self.similarity_matrix_ = csr_matrix(S)
            self.predict_topK = predict_topK
            self.remove_history = remove_history

        def _fit(self, X):
            return self

    return FixedModel


def _csr(rows, I):
    """rows: {row: {col: value}} -> CSR [max row + 1 or I x I]."""
    indptr, indices, data = [0], [], []
    for r in range(I):
        cols = sorted(rows.get(r, {}))
        indices += cols
        data += [rows[r][c] for c in cols]
        indptr.append(len(indices))
    return csr_matrix((np.array(data, dtype=np.float64), np.array(indices, dtype=np.int32), np.array(indptr)), shape=(I, I))


def _hist(lists, I):
    indptr = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(h) for h in lists], out=indptr[1:])
    indices = np.concatenate([np.sort(np.asarray(h, dtype=np.int32)) for h in lists] + [np.zeros(0, np.int32)])
    return csr_matrix((np.ones(len(indices)), indices, indptr), shape=(len(lists), I))


def _paths(err):
    """Counters of the instrumented build's lines, summed over the calls (empty without instrumentation)."""
    tot = {}
    for line in err.splitlines():
        if "[predict signed paths]" in line:
            for k, v in re.findall(r"([a-zA-Z][a-zA-Z ]*?)=(\d+)", line.split("]", 1)[1]):
                tot[k.strip()] = tot.get(k.strip(), 0) + int(v)
    return tot


def _check(engine, capfd, S, X, N, allowed=None, flags=0):
    """Top-N and full CSR, with and without history removal, against the oracle bit for bit.  Returns the counters."""
    U, I = X.shape
    engine.debug_flags(flags)
    engine.model_load_signed_csr(I, S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data.astype(np.float64))
    engine._model_key = None  # not an estimator's model: the next estimator's predict uploads its own
    engine.predict_item_filter(None if allowed is None else np.asarray(allowed, dtype=np.uint8))
    indptr, indices = X.indptr.astype(np.int64), X.indices.astype(np.int32)
    capfd.readouterr()
    try:
        for mask in (False, True):
            want = canon_predict_signed(X, S, N, remove_history=mask, allowed=allowed)
            for want_val in (True, False):
                got = engine.predict_topn(U, indptr, indices, N, mask_history=mask, want_val=want_val)
                assert np.array_equal(got["len"], want["len"])
                assert np.array_equal(got["idx"], want["idx"])
                if want_val:
                    assert np.array_equal(got["val"], want["val"])
            full = canon_predict_signed(X, S, None, remove_history=mask, allowed=allowed)
            o_ptr, o_idx, o_val = engine.predict_csr(U, indptr, indices, mask_history=mask)
            assert np.array_equal(o_ptr, full.indptr)
            assert np.array_equal(o_idx, full.indices)
            assert np.array_equal(o_val, full.data)
    finally:
        engine.debug_flags(0)
        engine.predict_item_filter(None)
    return _paths(capfd.readouterr().err)


def _moved(paths, name, at_least=1):
    if paths:  # instrumented build
        print(f"path counter {name!r}: {paths.get(name, 0)}, required >= {at_least}")
        assert paths.get(name, 0) >= at_least


def _random_signed(rng, I, density, neg=0.4):
    S = (rng.random((I, I)) < density) * rng.standard_normal((I, I))
    S[rng.random((I, I)) < neg] *= -1
    return csr_matrix(S)


# ---------------------------------------------------------------------------------------------------------------
# hand-built models


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 5, 20])
def test_mixed_signs(engine, capfd, N):
    rng = np.random.default_rng(N)
    I = 60
    S = _random_signed(rng, I, 0.3)
    X = csr_matrix((rng.random((80, I)) < 0.1).astype(np.float64))
    _check(engine, capfd, S, X, N)


@pytest.mark.gpu
def test_cancellation_to_zero_removes_the_entry_and_the_list_refills(engine, capfd):
    I = 12
    S = _csr({0: {5: 1.0, 6: 0.25, 7: -0.5}, 1: {5: -1.0, 8: 0.125}, 2: {5: 0.5, 9: -0.75}}, I)
    X = _hist([[0, 1], [0, 1, 2], [1]], I)
    full = canon_predict_signed(X, S)
    assert 5 not in full.indices[full.indptr[0] : full.indptr[1]]  # touched, summed to exactly 0.0, not stored
    _check(engine, capfd, S, X, 3)


@pytest.mark.gpu
def test_order_sensitive_sums_follow_the_history_order(engine, capfd):
    I = 8
    S = _csr({0: {3: 1.0, 4: 1e16}, 1: {3: 1e16, 4: -1e16}, 2: {3: -1e16, 4: 1.0, 5: -2.0}}, I)
    X = _hist([[0, 1, 2]], I)
    full = canon_predict_signed(X, S)
    assert list(full.indices) == [4, 5] and full.data[0] == 1.0  # (1 + 1e16) - 1e16 = 0 is dropped, (1e16 - 1e16) + 1 = 1
    _check(engine, capfd, S, X, 3)


@pytest.mark.gpu
def test_equal_scores_are_ordered_by_column(engine, capfd):
    I = 40
    S = _csr({0: {j: (0.5 if j % 3 else -0.5) for j in range(1, 40)}, 1: {j: 0.25 for j in range(20, 30)}}, I)
    X = _hist([[0], [0, 1], [1]], I)
    _check(engine, capfd, S, X, 7)


@pytest.mark.gpu
def test_users_with_fewer_stored_scores_than_n_list_negative_scores(engine, capfd):
    I = 10
    S = _csr({0: {1: 0.5, 2: -0.25, 3: -0.75}, 4: {5: -1.0}}, I)
    X = _hist([[0], [4], [0, 4]], I)
    want = canon_predict_signed(X, S, 5)
    assert want["len"].tolist() == [3, 1, 4] and (want["val"][1, 0] < 0)
    _check(engine, capfd, S, X, 5)


@pytest.mark.gpu
def test_empty_histories_and_an_all_negative_model(engine, capfd):
    rng = np.random.default_rng(3)
    I = 30
    S = -abs(_random_signed(rng, I, 0.4))
    S.eliminate_zeros()
    X = _hist([[], [1, 2], [], list(range(0, 30, 2))], I)
    _check(engine, capfd, S, X, 6)


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_nan_and_inf_are_rejected(engine, bad):
    from recpack_b200._lib import RpkError

    S = _csr({0: {1: -0.5, 2: bad}}, 4)
    with pytest.raises(RpkError):
        engine.model_load_signed_csr(4, S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data)


@pytest.mark.gpu
def test_public_class_predicts_signed_models_in_both_modes():
    rng = np.random.default_rng(7)
    I = 50
    S = _random_signed(rng, I, 0.25)
    X = csr_matrix((rng.random((70, I)) < 0.12).astype(np.float64))
    cls = _signed_class()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for mask in (False, True):
            full = cls(S, None, mask).predict(X)
            want = canon_predict_signed(X, S, None, remove_history=mask)
            full.sort_indices()
            assert np.array_equal(full.indptr, want.indptr) and np.array_equal(full.indices, want.indices)
            assert np.array_equal(full.data, want.data)
            top = cls(S, 8, mask).predict(X)
            w = canon_predict_signed(X, S, 8, remove_history=mask)
            assert getattr(top, "_rpk_topn_dev", None) is not None
            for u in range(X.shape[0]):
                lo, hi = top.indptr[u], top.indptr[u + 1]
                assert np.array_equal(top.indices[lo:hi], w["idx"][u, : w["len"][u]])
                assert np.array_equal(top.data[lo:hi], w["val"][u, : w["len"][u]])


# ---------------------------------------------------------------------------------------------------------------
# post-filters


@pytest.mark.gpu
def test_item_filter_refills_the_lists_and_spgemm_stays_unfiltered(engine, capfd):
    rng = np.random.default_rng(11)
    I = 70
    S = _random_signed(rng, I, 0.3)
    X = csr_matrix((rng.random((60, I)) < 0.1).astype(np.float64))
    allowed = rng.random(I) < 0.6
    _check(engine, capfd, S, X, 10, allowed=allowed)
    # the TARS classes call the same float64 row kernel: after a filtered predict it is unfiltered
    engine.model_load_signed_csr(I, S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data)
    engine.predict_item_filter(allowed.astype(np.uint8))
    try:
        engine.predict_topn(X.shape[0], X.indptr.astype(np.int64), X.indices.astype(np.int32), 10)
        A = csr_matrix(X)
        A.sort_indices()
        indptr, indices, values = engine.spgemm_csr(A, S)
        want = csr_matrix(A @ S)
        want.sort_indices()
        assert np.array_equal(indptr, want.indptr) and np.array_equal(indices, want.indices)
        assert np.array_equal(values, want.data)
    finally:
        engine.predict_item_filter(None)


@pytest.mark.gpu
def test_public_class_postfilters_refill_the_lists():
    from recpack_b200 import ExcludeItems

    rng = np.random.default_rng(13)
    I = 40
    S = _random_signed(rng, I, 0.3)
    X = csr_matrix((rng.random((30, I)) < 0.15).astype(np.float64))
    banned = np.arange(0, I, 3)
    allowed = np.ones(I, dtype=bool)
    allowed[banned] = False
    algo = _signed_class()(S, 6, True).set_postfilters([ExcludeItems(banned)])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        top = algo.predict(X)
    w = canon_predict_signed(X, S, 6, remove_history=True, allowed=allowed)
    assert np.array_equal(np.diff(top.indptr), w["len"])
    for u in range(X.shape[0]):
        lo, hi = top.indptr[u], top.indptr[u + 1]
        assert np.array_equal(top.indices[lo:hi], w["idx"][u, : w["len"][u]])
        assert np.array_equal(top.data[lo:hi], w["val"][u, : w["len"][u]])


# ---------------------------------------------------------------------------------------------------------------
# the branches of k_predict_signed


@pytest.mark.gpu
def test_intervals_overlapping_at_the_nth_place(engine, capfd):
    """50 equal scores around the 5th place: all of them survive the screen and are folded exactly."""
    I = 200
    S = _csr({0: {j: 0.5 for j in range(1, 51)} | {j: -0.25 for j in range(60, 120)}, 1: {j: 0.125 for j in range(150, 160)}}, I)
    X = _hist([[0], [0, 1], [1]], I)
    want = canon_predict_signed(X, S, 5)
    assert np.count_nonzero(want["val"][0] == 0.5) == 5  # a tie group larger than the list at the N-th place
    _moved(_check(engine, capfd, S, X, 5), "overlap ranges", 2)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, DBG_MULTI_PASS])
def test_more_survivors_than_the_list_holds(engine, capfd, flags):
    I = 1200
    S = _csr({0: {j: 0.5 for j in range(1, 700)}, 1: {j: -0.5 for j in range(700, 1100)}}, I)
    X = _hist([[0], [0, 1], [1, 2]], I)
    assert 699 > CAP  # one tie group at the N-th place, larger than the list
    _moved(_check(engine, capfd, S, X, 5, flags=flags), "overflow users", 4)


@pytest.mark.gpu
def test_exact_zeros_that_empty_the_list(engine, capfd):
    """100 items cancel to exactly 0.0 next to the screen's N-th value; only 2 positive scores remain, and the
    strongly negative items screened out belong to the list: the user goes to the float64 row kernel."""
    I = 400
    rows = {0: {}, 1: {}}
    for j in range(10, 110):
        rows[0][j] = 1.0 + j / 1024
        rows[1][j] = -(1.0 + j / 1024)
    rows[0].update({200: 1.0, 201: 0.5})
    rows[0].update({j: -4.0 - j / 512 for j in range(300, 340)})
    S = _csr(rows, I)
    X = _hist([[0, 1]], I)
    want = canon_predict_signed(X, S, 5)
    full = canon_predict_signed(X, S)
    assert full.nnz == 2 + 40 and want["len"][0] == 5 and (want["val"][0, 2:] < -4).all()
    _moved(_check(engine, capfd, S, X, 5), "zero users", 2)


@pytest.mark.gpu
def test_heavy_histories(engine, capfd):
    rng = np.random.default_rng(17)
    I = 2600
    S = csr_matrix((rng.random((I, I)) < 0.004) * rng.standard_normal((I, I)))
    X = _hist([rng.choice(I, 2100, replace=False), rng.choice(I, SG_EXACT_D - 1, replace=False), [1, 2, 3]], I)
    assert np.diff(X.indptr).max() >= SG_EXACT_D
    _moved(_check(engine, capfd, S, X, 20), "heavy users", 4)


@pytest.mark.gpu
def test_long_model_rows(engine, capfd):
    """Dense model rows: segments of thousands of entries, swept by the same strided loop."""
    rng = np.random.default_rng(19)
    I = 3000
    dense = rng.standard_normal((4, I))
    rows = {i: {j: float(dense[i, j]) for j in range(I)} for i in range(4)}
    rows[5] = {j: 0.5 for j in range(0, I, 7)}
    S = _csr(rows, I)
    X = _hist([[0], [0, 1, 2, 3], [1, 5], [5]], I)
    assert np.diff(S.indptr).max() == I
    _moved(_check(engine, capfd, S, X, 20), "long segments", 1)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [DBG_MULTI_PASS, DBG_MANY_PASS])
def test_several_item_ranges_by_flag(engine, capfd, flags):
    rng = np.random.default_rng(flags)
    I = 300
    S = _random_signed(rng, I, 0.05)
    X = csr_matrix((rng.random((50, I)) < 0.05).astype(np.float64))
    paths = _check(engine, capfd, S, X, 10, flags=flags)
    if paths:
        assert paths["P"] >= (4 if flags == DBG_MANY_PASS else 2) * 4  # 4 top-N calls per _check


@pytest.mark.gpu
def test_several_item_ranges_at_a_large_item_count(engine, capfd):
    rng = np.random.default_rng(23)
    I, K = 120_000, 16
    rows = np.repeat(np.arange(I), K)
    cols = rng.integers(0, I, I * K)
    S = csr_matrix((rng.standard_normal(I * K), (rows, cols)), shape=(I, I))
    S.sum_duplicates()
    S.eliminate_zeros()
    hist = [rng.choice(I, int(d), replace=False) for d in rng.integers(1, 60, 200)]
    X = _hist(hist, I)
    paths = _check(engine, capfd, S, X, 20)
    if paths:
        assert paths["P"] >= 3 * 4


# ---------------------------------------------------------------------------------------------------------------
# end to end and full size


@pytest.mark.gpu
def test_pearson_model_end_to_end_with_metrics():
    from recpack_b200 import NDCGK, RecallK, pearson_top_k

    rng = np.random.default_rng(29)
    U, I = 600, 120
    R = (rng.random((U, I)) < 0.15) * rng.integers(1, 6, (U, I))
    X = csr_matrix(R.astype(np.float64))
    S = pearson_top_k(X, 100)  # most of each row: the negative correlations stay in the model
    assert S.data.min() < 0
    train = csr_matrix((rng.random((U, I)) < 0.06).astype(np.float64))
    test_out = csr_matrix((rng.random((U, I)) < 0.03).astype(np.float64))
    algo = _signed_class()(S, 10, True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = algo.predict(train)
    want = canon_predict_signed(train, S, 10, remove_history=True)
    assert np.array_equal(np.diff(pred.indptr), want["len"])
    plain = csr_matrix((pred.data.copy(), pred.indices.copy(), pred.indptr.copy()), shape=pred.shape)
    for cls in (NDCGK, RecallK):
        a, b = cls(10), cls(10)
        a.calculate(test_out, pred)   # the device lists attached to the prediction
        b.calculate(test_out, plain)  # the host CSR
        assert a.value == b.value


@pytest.mark.gpu
def test_nonnegative_models_keep_the_fixed_point_route(engine, capfd):
    from oracle import recpack_oracle as orc

    rng = np.random.default_rng(31)
    I = 80
    S = abs(_random_signed(rng, I, 0.2))
    X = csr_matrix((rng.random((40, I)) < 0.1).astype(np.float64))
    engine.model_load_csr(I, S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data)
    capfd.readouterr()
    got = engine.predict_topn(X.shape[0], X.indptr.astype(np.int64), X.indices.astype(np.int32), 10)
    err = capfd.readouterr().err
    want = orc.canon_predict_topn(X, S, 10)
    assert np.array_equal(got["idx"], want["idx"]) and np.array_equal(got["val"], want["val"])
    assert "[predict signed paths]" not in err


@pytest.mark.gpu
def test_full_size_signed_itemknn_against_the_spgemm_route(engine):
    from recpack_b200 import ItemKNN
    from recpack_b200.synth import make_dataset

    train, _, _ = make_dataset("ml25m")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        S = csr_matrix(ItemKNN(K=200).fit(train).similarity_matrix_)
    S.sort_indices()
    rows = np.repeat(np.arange(S.shape[0], dtype=np.uint64), np.diff(S.indptr))
    h = (rows * np.uint64(0x9E3779B1) + S.indices.astype(np.uint64) * np.uint64(0x85EBCA77) + np.uint64(12345)) % np.uint64(3)
    S.data[h == 0] *= -1
    U, I = train.shape
    X = csr_matrix(train, dtype=np.float64)
    X.sort_indices()
    X.data[:] = 1.0
    engine.model_load_signed_csr(I, S.indptr.astype(np.int64), S.indices.astype(np.int32), S.data)
    got = engine.predict_topn(U, X.indptr.astype(np.int64), X.indices.astype(np.int32), 20, mask_history=True)
    ref = engine.spgemm_topn(X, S, 20, mask_history=True)
    assert U == 162_541
    assert np.array_equal(got["len"], ref["len"])
    assert np.array_equal(got["idx"], ref["idx"])
    assert np.array_equal(got["val"], ref["val"])
    sample = np.random.default_rng(0).choice(U, 1000, replace=False)
    want = canon_predict_signed(X[sample], S, 20, remove_history=True)
    assert np.array_equal(got["idx"][sample], want["idx"]) and np.array_equal(got["val"][sample], want["val"])


# ---------------------------------------------------------------------------------------------------------------
# the oracle itself (no GPU)


def test_oracle_follows_scipy_order_and_drops_zero_sums():
    X = csr_matrix(np.ones((1, 3)))
    S = csr_matrix(np.array([[1.0, 1e16], [1e16, -1e16], [-1e16, 1.0]]))
    full = canon_predict_signed(X, S)
    assert full.indices.tolist() == [1] and full.data.tolist() == [1.0]
    top = canon_predict_signed(X, S, 2)
    assert top["len"].tolist() == [1] and top["idx"].tolist() == [[1, -1]]


def test_oracle_removals_and_order():
    X = csr_matrix(np.array([[1.0, 0, 0, 0], [0, 1.0, 0, 0]]))
    S = csr_matrix(np.array([[0.5, -0.5, -0.5, 0.25], [0, 0, 2.0, -1.0], [0, 0, 0, 0], [0, 0, 0, 0]]))
    top = canon_predict_signed(X, S, 3, remove_history=True)
    assert top["idx"].tolist() == [[3, 1, 2], [2, 3, -1]] and top["val"][0].tolist() == [0.25, -0.5, -0.5]
    top = canon_predict_signed(X, S, 3, allowed=[True, True, False, True])
    assert top["idx"].tolist() == [[0, 3, 1], [3, -1, -1]]
