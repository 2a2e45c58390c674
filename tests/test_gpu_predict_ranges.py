"""Top-N scoring over several item ranges per user: the 32-bit kernel runs the ranges of a user one after the other,
carries the survivor bound of the earlier ranges into the later ones and merges every range's survivors into one
running list; the two-limb kernel (DBG_WIDE_ACC) offers its running list to the next range's selection as extra
candidates.  Each case below puts the deciding entries in a different place across the ranges; the lists (and the
scores, when asked for) must be the oracle's, bit for bit."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle import recpack_oracle as orc

pytestmark = pytest.mark.gpu

DBG_WIDE_ACC, DBG_TINY_LIST, DBG_MULTI_PASS, DBG_MANY_PASS = 1, 2, 4, 32  # two ranges / four ranges (at 64 items: 16 each)
I = 64


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.debug_flags(0)
    eng.predict_item_filter(None)


def _model(cols_of_row, val_of_row):
    K = max(len(c) for c in cols_of_row)
    idx = np.zeros((I, K), dtype=np.int32)
    val = np.zeros((I, K))
    ln = np.zeros(I, dtype=np.int32)
    for i in range(I):
        c = np.asarray(cols_of_row[i], dtype=np.int32)
        o = np.argsort(c)
        ln[i] = len(c)
        idx[i, : len(c)] = c[o]
        val[i, : len(c)] = np.asarray(val_of_row[i])[o]
    return K, idx, val, ln


def _users(rows):
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    indices = np.concatenate([np.sort(np.asarray(r, dtype=np.int32)) for r in rows] + [np.zeros(0, np.int32)]).astype(np.int32)
    X = csr_matrix((np.ones(len(indices), dtype=np.int32), indices, indptr), shape=(len(rows), I))
    return X, indptr, indices


def _want(X, S, N, allowed):
    if allowed is None:
        return orc.canon_predict_topn(X, S, N, remove_history=True)
    full = orc.canon_predict_topn(X, S, I, remove_history=True)
    U = X.shape[0]
    want = {"idx": np.full((U, N), -1, np.int32), "val": np.zeros((U, N)), "len": np.zeros(U, np.int32)}
    for u in range(U):
        keep = [t for t in range(full["len"][u]) if allowed[full["idx"][u, t]]][:N]
        want["idx"][u, : len(keep)] = full["idx"][u, keep]
        want["val"][u, : len(keep)] = full["val"][u, keep]
        want["len"][u] = len(keep)
    return want


def _check(engine, model, rows, N, flags, allowed=None):
    K, idx, val, ln = model
    S = orc.topk_to_csr(idx, val, ln, I)
    engine.model_load_topk(I, K, idx, val, ln)
    X, indptr, indices = _users(rows)
    want = _want(X, S, N, allowed)
    engine.debug_flags(flags)
    engine.predict_item_filter(None if allowed is None else allowed.astype(np.uint8))
    try:
        lists = engine.predict_topn(len(rows), indptr, indices, N, mask_history=True, want_val=False)
        full = engine.predict_topn(len(rows), indptr, indices, N, mask_history=True)
    finally:
        engine.debug_flags(0)
        engine.predict_item_filter(None)
    for got in (lists, full):
        assert np.array_equal(got["len"], want["len"])
        assert np.array_equal(got["idx"], want["idx"])
    assert np.array_equal(full["val"], want["val"])


def _random_rows(rng, U, lo=1, hi=12):
    rows = [rng.choice(I, size=rng.integers(lo, hi), replace=False) for _ in range(U)]
    rows[3] = []  # a user without history
    return rows


FLAGS = [DBG_MULTI_PASS, DBG_MANY_PASS, DBG_MANY_PASS | DBG_TINY_LIST,
         DBG_WIDE_ACC | DBG_MULTI_PASS, DBG_WIDE_ACC | DBG_MANY_PASS, DBG_WIDE_ACC | DBG_MANY_PASS | DBG_TINY_LIST]


@pytest.mark.parametrize("flags", FLAGS)
def test_top_n_in_the_last_range(engine, flags):
    rng = np.random.default_rng(11)
    cols = [np.unique(np.r_[rng.choice(48, 4, replace=False), 48 + rng.choice(16, 4, replace=False)]) for _ in range(I)]
    vals = [np.where(c >= 48, 0.6 + 0.3 * rng.random(len(c)), 0.05 + 0.2 * rng.random(len(c))) for c in cols]
    _check(engine, _model(cols, vals), _random_rows(rng, 60), 5, flags)


@pytest.mark.parametrize("flags", FLAGS)
def test_tie_at_the_nth_place_across_ranges(engine, flags):
    rng = np.random.default_rng(12)
    targets = np.array([3, 9, 20, 35, 47, 60])  # ranges 0, 0, 1, 2, 2, 3 of four; 0, 0, 0, 1, 1, 1 of two
    cols, vals = [], []
    for i in range(I):
        others = rng.choice(np.setdiff1d(np.arange(I), targets), 3, replace=False)
        base = 0.25 + 0.5 * rng.random()
        # even rows: the six targets exactly equal (ties broken by item index, the N-th place among them);
        # odd rows: equal up to the last bits of the fixed-point scores (only exact sums order them)
        t = np.full(6, base) if i % 2 == 0 else base * (1.0 + rng.integers(-3, 4, size=6) * 2.0**-36)
        cols.append(np.r_[targets, others])
        vals.append(np.r_[t, 0.01 + 0.1 * rng.random(3)])
    rows = [rng.choice(np.setdiff1d(np.arange(I), targets), size=rng.integers(1, 20), replace=False) for _ in range(50)]
    rows[3] = []
    rows[4] = [0, 2]  # even rows only: exact ties
    _check(engine, _model(cols, vals), rows, 5, flags)


@pytest.mark.parametrize("flags", FLAGS)
def test_earlier_ranges_with_fewer_than_n_candidates(engine, flags):
    rng = np.random.default_rng(13)
    # every row reaches one item below 32 (the first range of two, of four: the first range; the second and third
    # of four are empty) and many in the last quarter
    cols = [np.r_[rng.integers(0, 16), 48 + rng.choice(16, 6, replace=False)] for _ in range(I)]
    vals = [0.05 + rng.random(len(c)) for c in cols]
    _check(engine, _model(cols, vals), _random_rows(rng, 60), 8, flags)


@pytest.mark.parametrize("flags", FLAGS)
def test_range_emptied_by_the_history_mask_or_the_item_filter(engine, flags):
    rng = np.random.default_rng(14)
    # rows reach items 0..7 (first range) and 40..47 (third of four, second of two) only
    cols = [np.r_[rng.choice(8, 3, replace=False), 40 + rng.choice(8, 3, replace=False)] for _ in range(I)]
    vals = [0.05 + rng.random(6) for _ in range(I)]
    model = _model(cols, vals)
    rows = _random_rows(rng, 40)
    rows[5] = list(range(8))  # the history masks every candidate of the first range
    rows[6] = list(range(8)) + [20, 33]
    rows[7] = list(range(40, 48))  # ... of the third
    _check(engine, model, rows, 5, flags)
    allowed = np.ones(I, dtype=bool)
    allowed[40:48] = False  # the filter empties the third range
    _check(engine, model, rows, 5, flags, allowed)
    allowed[:] = True
    allowed[:8] = False  # ... the first
    _check(engine, model, rows, 5, flags, allowed)
