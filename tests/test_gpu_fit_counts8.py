"""Dense-leg counts in 8 bits: with at most 255 dense users the tensor-core Gram writes its count strip as uint8
through TMA tensor stores, and k_fit_rows expands each strip row into its packed 16-bit counters.  The fit must
stay bit for bit the oracle's, at the largest count 8 bits hold, across row strips, and for item-range passes
whose first column is not 16-aligned."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle import recpack_oracle as orc

pytestmark = pytest.mark.gpu

DBG_WIDE_ACC, DBG_MULTI_PASS = 1, 4


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.fit_config(-1)
    eng.fit_strip_rows(0)
    eng.debug_flags(0)


def _fit(engine, X, K, sim="cosine", dense_users=-1, flags=0, strip_rows=0, item_begin=0, item_end=None):
    from recpack_b200.matrix import binary_structure

    Xc, indptr, indices = binary_structure(X)
    U, I = Xc.shape
    engine.debug_flags(flags)
    engine.fit_config(dense_users)
    engine.fit_strip_rows(strip_rows)
    try:
        got = engine.fit_topk(U, I, indptr, indices, K, similarity=sim, item_begin=item_begin, item_end=item_end)
        dense = engine.last_timings()["dense_users"]
    finally:
        engine.fit_strip_rows(0)
        engine.fit_config(-1)
        engine.debug_flags(0)
    return got, dense


def _assert_fit_equal(got, want):
    assert np.array_equal(got["len"], want["len"])
    assert np.array_equal(got["idx"], want["idx"])
    assert np.array_equal(got["cnt"], want["cnt"])
    assert np.array_equal(got["val"], want["val"])  # bit-identical float64


def _heavy_pair_matrix(n_dense, seed):
    """n_dense users with 60+ items each that all hold items 0 and 1 (their Gram count is n_dense), and 1,745
    users with short histories (< 32 items: never dense)."""
    rng = np.random.default_rng(seed)
    I = 1003  # not a multiple of 16 or of 256: the strip rows end in a partial vector
    rows = []
    for _ in range(n_dense):
        rows.append(np.r_[0, 1, 2 + rng.choice(I - 2, 60, replace=False)])
    for _ in range(1745):
        rows.append(rng.choice(I, int(rng.integers(1, 20)), replace=False))
    indptr = np.r_[0, np.cumsum([len(r) for r in rows])]
    indices = np.concatenate(rows)
    X = csr_matrix((np.ones(len(indices), np.int32), indices, indptr), shape=(len(rows), I))
    X.sum_duplicates()
    X.sort_indices()
    return X


@pytest.mark.parametrize("flags", [0, DBG_WIDE_ACC, DBG_MULTI_PASS])
@pytest.mark.parametrize("sim", ["cosine", "conditional_probability"])
def test_dense_count_of_255_fits_8_bits(engine, sim, flags):
    """255 dense users share items 0 and 1: the 8-bit strip holds a count of 255, and the fit equals the fit
    without a dense leg and the oracle."""
    X = _heavy_pair_matrix(255, seed=3)
    K = 40
    want = orc.canon_fit(X, K=K, similarity=sim)
    got8, dense = _fit(engine, X, K, sim, dense_users=255, flags=flags)
    assert dense == 255
    sparse, dense0 = _fit(engine, X, K, sim, dense_users=0, flags=flags)
    assert dense0 == 0
    _assert_fit_equal(got8, sparse)
    _assert_fit_equal(got8, want)
    row0 = got8["idx"][0][: got8["len"][0]]
    assert 1 in row0 and got8["cnt"][0][list(row0).index(1)] >= 255


def test_256_dense_users_take_16_bit_counts(engine):
    """One dense user more than 8 bits can count: the 16-bit strip, same results."""
    X = _heavy_pair_matrix(256, seed=4)
    K = 40
    got, dense = _fit(engine, X, K, dense_users=256)
    assert dense == 256
    _assert_fit_equal(got, orc.canon_fit(X, K=K))


@pytest.mark.parametrize("flags", [0, DBG_WIDE_ACC, DBG_MULTI_PASS])
@pytest.mark.parametrize("strip_rows", [128, 384])
def test_8bit_strips_over_several_row_strips(engine, strip_rows, flags):
    """The 8-bit count strip in several row strips, over the whole range and an unaligned item shard."""
    from recpack_b200.synth import synth_interactions

    U, I, nnz, K = 943, 1003, 100_000, 200
    X = synth_interactions(U, I, nnz, seed=7)
    want = orc.canon_fit(X, K=K)
    got, dense = _fit(engine, X, K, dense_users=200, flags=flags, strip_rows=strip_rows)
    assert 0 < dense <= 200
    _assert_fit_equal(got, want)
    b, e = I // 7 + 3, I - I // 5
    part, _ = _fit(engine, X, K, dense_users=200, flags=flags, strip_rows=strip_rows, item_begin=b, item_end=e)
    for key in ("idx", "cnt", "val", "len"):
        assert np.array_equal(part[key], want[key][b:e]), key


def test_8bit_gram_with_more_tiles_than_ctas(engine):
    """I = 5,000: 40 x 20 Gram tiles, more than one per CTA, so every epilogue warp refills its staging boxes after
    the previous tile's TMA stores have read them."""
    from recpack_b200.synth import synth_interactions

    U, I, nnz, K = 3000, 5000, 300_000, 100
    X = synth_interactions(U, I, nnz, seed=9)
    want = orc.canon_fit(X, K=K)
    got, dense = _fit(engine, X, K, dense_users=255)
    assert 0 < dense <= 255
    _assert_fit_equal(got, want)
