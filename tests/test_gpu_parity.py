"""GPU parity tests: the CUDA path (through the public classes and the C ABI) against the oracle
and against golden vectors produced by the real reference.  Integer / index results are compared
bit for bit; similarity values too (they are reproduced with the reference's operation order);
metric values to 1e-12 against the canonical oracle and tie-aware against the reference."""
import math
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from conftest import load_golden, unpack
from oracle import recpack_oracle as orc

pytestmark = pytest.mark.gpu

UNIT = ["unit_cosine", "unit_empty_col", "unit_condprob", "unit_condprob_pd1", "unit_condprob_pd0.2", "unit_condprob_pd0.5"]
SMALL = ["small_cosine", "small_condprob", "small_condprob_pd"]
FLAG_SETS = [0, 1, 2, 4, 5, 6, 8, 10]  # bit0: 32-bit counters (fit) / wide accumulators (predict); bit1: tiny lists; bit2: multi-pass; bit3: heavy rows counted in pieces


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.debug_flags(0)


def _params(g):
    pd_ = float(g["pop_discount"]) if "pop_discount" in g else float("nan")
    sim = str(g["similarity"]) if "similarity" in g else "cosine"
    return int(g["K"]), sim, (None if math.isnan(pd_) else pd_)


def _fit_lists(engine, X, K, sim="cosine", pd_=None, item_begin=0, item_end=None):
    from recpack_b200.matrix import binary_structure

    Xc, indptr, indices = binary_structure(X)
    U, I = Xc.shape
    item_pow = None
    if sim == "conditional_probability" and pd_:
        n = np.bincount(indices, minlength=I)
        item_pow = np.zeros(I)
        item_pow[n > 0] = np.power(1 / n[n > 0], pd_)
    return engine.fit_topk(U, I, indptr, indices, K, similarity=sim, item_pow=item_pow, item_begin=item_begin, item_end=item_end)


def _assert_fit_equal(got, want):
    assert np.array_equal(got["len"], want["len"])
    assert np.array_equal(got["idx"], want["idx"])
    assert np.array_equal(got["cnt"], want["cnt"])
    assert np.array_equal(got["val"], want["val"])  # bit-identical float64


# ------------------------------------------------------------------------------- fit
@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("name", UNIT + SMALL)
def test_fit_matches_canonical_oracle_on_golden_inputs(engine, name, flags):
    g = load_golden(name)
    K, sim, pd_ = _params(g)
    X = unpack(g, "X")
    engine.debug_flags(flags)
    got = _fit_lists(engine, X, K, sim, pd_)
    engine.debug_flags(0)
    _assert_fit_equal(got, orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_))


@pytest.mark.parametrize("name", UNIT + SMALL + ["mid_cosine"])
def test_fit_vs_reference_golden_tie_aware(engine, name):
    """Against the unmodified reference's similarity_matrix_: same row sizes, same values, item
    differences only inside the boundary tie group; identical float64 values on common entries."""
    g = load_golden(name)
    K, sim, pd_ = _params(g)
    X = unpack(g, "X")
    S_ref = unpack(g, "S")
    got = _fit_lists(engine, X, K, sim, pd_)
    S = orc.topk_to_csr(got["idx"], got["val"], got["len"], X.shape[1])
    if pd_:
        np.testing.assert_allclose(np.sort(S.data), np.sort(S_ref.data), rtol=1e-12)
        return
    # mid_cosine keeps a seeded sample of the reference's rows (S_rows) to stay small
    rows = g["S_rows"] if "S_rows" in g else np.arange(X.shape[1])
    stats = orc.compare_topk_tie_aware(S_ref, got, orc.binarize(X), similarity=sim, rows=rows)
    assert stats["rows_checked"] == len(rows)
    S = S[rows]
    common = S.multiply(S_ref.astype(bool)).tocsr()
    ref_common = S_ref.multiply(S.astype(bool)).tocsr()
    common.sort_indices()
    ref_common.sort_indices()
    assert np.array_equal(common.data, ref_common.data)


def test_reference_unit_vectors_through_public_api():
    """recpack/tests/test_algorithms/test_nearest_neighbour.py:44-70,119-181 with the drop-in class."""
    from recpack_b200 import ItemKNN

    data = csr_matrix(([1] * 7, ([0, 0, 1, 1, 2, 2, 2], [1, 2, 0, 2, 0, 1, 2])), shape=(4, 3))
    e = 2 / math.sqrt(6)
    algo = ItemKNN(K=2)
    algo.fit(data)
    expected = np.array([[0, 0.5, e], [0.5, 0, e], [e, e, 0]])
    np.testing.assert_almost_equal(algo.similarity_matrix_.toarray(), expected)
    _in = csr_matrix(([1, 1, 1], ([0, 1, 2], [0, 1, 2])), shape=(3, 3))
    np.testing.assert_almost_equal(algo.predict(_in).toarray(), expected)
    _in = csr_matrix(([1, 1], ([0, 0], [0, 1])), shape=(1, 3))
    np.testing.assert_almost_equal(algo.predict(_in).toarray(), [[0.5, 0.5, 4 / math.sqrt(6)]])

    algo = ItemKNN(K=2, normalize_sim=True)
    algo.fit(data)
    np.testing.assert_array_almost_equal(algo.similarity_matrix_.sum(axis=1), 1)

    data_empty_col = csr_matrix(([1] * 5, ([0, 0, 1, 1, 2], [1, 2, 2, 1, 2])))
    algo = ItemKNN(K=2)
    with pytest.warns(UserWarning, match="ItemKNN missing similar items for 1 items."):
        algo.fit(data_empty_col)
    np.testing.assert_almost_equal(algo.similarity_matrix_.toarray(), [[0, 0, 0], [0, 0, e], [0, e, 0]])

    algo = ItemKNN(K=2, similarity="conditional_probability")
    algo.fit(data)
    np.testing.assert_almost_equal(algo.similarity_matrix_.toarray(), [[0, 1 / 2, 1], [1 / 2, 0, 1], [2 / 3, 2 / 3, 0]])
    for pdc in (1, 0.2, 0.5):
        algo = ItemKNN(K=2, similarity="conditional_probability", pop_discount=pdc)
        algo.fit(data)
        exp = np.array(
            [
                [0, 1 / (2 * 2**pdc), 2 / (2 * 3**pdc)],
                [1 / (2 * 2**pdc), 0, 2 / (2 * 3**pdc)],
                [2 / (3 * 2**pdc), 2 / (3 * 2**pdc), 0],
            ]
        )
        np.testing.assert_almost_equal(algo.similarity_matrix_.toarray(), exp)


CASES = [
    # U, I, nnz, K, similarity, pop_discount
    (200, 64, 1500, 5, "cosine", None),
    (500, 300, 9000, 50, "cosine", None),
    (943, 1682, 100_000, 200, "cosine", None),
    (500, 300, 9000, 50, "conditional_probability", None),
    (500, 300, 9000, 50, "conditional_probability", 0.3),
    (60, 2000, 6000, 100, "conditional_probability", None),  # few users, many items: huge tie groups
    (60, 2000, 6000, 100, "cosine", None),
    (1500, 40, 20_000, 64, "cosine", None),  # K >= I: every positive neighbour is kept
]


@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("case", CASES)
def test_fit_matches_oracle_on_synthetic(engine, case, flags):
    from recpack_b200.synth import synth_interactions

    U, I, nnz, K, sim, pd_ = case
    X = synth_interactions(U, I, nnz, seed=U + I)
    engine.debug_flags(flags)
    got = _fit_lists(engine, X, K, sim, pd_)
    engine.debug_flags(0)
    _assert_fit_equal(got, orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_))


@pytest.mark.parametrize("flags", [0, 1, 4])
@pytest.mark.parametrize("dense_users", [16, 200, 4096])
@pytest.mark.parametrize("case", [CASES[1], CASES[2], CASES[3], CASES[7]])
def test_fit_hybrid_dense_users_gives_identical_results(engine, case, dense_users, flags):
    """The users with the longest histories go through the tcgen05 Gram, the rest through the sparse
    kernel: counts, lists and values must not change."""
    from recpack_b200.synth import synth_interactions

    U, I, nnz, K, sim, pd_ = case
    X = synth_interactions(U, I, nnz, seed=U + I)
    engine.debug_flags(flags)
    engine.fit_config(dense_users)
    try:
        got = _fit_lists(engine, X, K, sim, pd_)
    finally:
        engine.fit_config(-1)
        engine.debug_flags(0)
    _assert_fit_equal(got, orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_))


@pytest.mark.parametrize("flags", [0, 1, 4])
@pytest.mark.parametrize("strip_rows,dense_users", [(128, 64), (256, 4096), (128, 0)])
@pytest.mark.parametrize("case", [CASES[2], CASES[3], CASES[5]])
def test_fit_in_row_strips_gives_identical_results(engine, case, strip_rows, dense_users, flags):
    """The fit cuts its row range into strips so that only one strip of the dense leg's count matrix exists at a time
    (rpk_fit_strip_rows): later strips reuse the item counts, the dense / sparse split and the dense operand of the first.
    Whole range and an unaligned item shard."""
    from recpack_b200.synth import synth_interactions

    U, I, nnz, K, sim, pd_ = case
    X = synth_interactions(U, I, nnz, seed=U + I)
    want = orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_)
    engine.debug_flags(flags)
    engine.fit_config(dense_users)
    engine.fit_strip_rows(strip_rows)
    try:
        got = _fit_lists(engine, X, K, sim, pd_)
        b, e = I // 7 + 3, I - I // 5
        part = _fit_lists(engine, X, K, sim, pd_, item_begin=b, item_end=e)
    finally:
        engine.fit_strip_rows(0)
        engine.fit_config(-1)
        engine.debug_flags(0)
    _assert_fit_equal(got, want)
    _assert_fit_equal(part, {k: v[b:e] for k, v in want.items()})


@pytest.mark.parametrize("flags", [0, 2, 6])
def test_fit_total_ties(engine, flags):
    """Every pair ties: 3 users who all saw all items.  The canonical pick is the lowest indices."""
    I, K = 700, 40
    X = csr_matrix(np.ones((3, I), dtype=np.int32))
    engine.debug_flags(flags)
    for sim in ("cosine", "conditional_probability"):
        got = _fit_lists(engine, X, K, sim)
        for i in (0, 1, 350, I - 1):
            want = [j for j in range(I) if j != i][:K]
            assert got["idx"][i].tolist() == want
            assert np.all(got["cnt"][i] == 3)
    engine.debug_flags(0)


def test_fit_item_shards_concatenate(engine):
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(400, 250, 6000, seed=3)
    full = _fit_lists(engine, X, 30)
    parts = [_fit_lists(engine, X, 30, item_begin=b, item_end=e) for b, e in ((0, 100), (100, 101), (101, 250))]
    for key in ("idx", "cnt", "val", "len"):
        assert np.array_equal(np.concatenate([p[key] for p in parts]), full[key])
    counts = engine.fit_item_counts(250)
    assert np.array_equal(counts, np.bincount(X.indices, minlength=250))


def test_fit_input_coercion_and_edges(engine):
    from recpack_b200 import ItemKNN, UnsupportedTypeError

    # counts > 1, duplicates, explicit zeros and unsorted indices are binarised away (base.py:129-139)
    rows = np.array([0, 0, 0, 1, 1, 2, 2, 2, 2])
    cols = np.array([2, 1, 1, 0, 2, 0, 1, 2, 3])
    vals = np.array([5, 1, 1, 2, 1, 1, 7, 1, 0])
    X = csr_matrix((vals, (rows, cols)), shape=(4, 5))
    Xb = csr_matrix((np.ones(7), ([0, 0, 1, 1, 2, 2, 2], [1, 2, 0, 2, 0, 1, 2])), shape=(4, 5))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a = ItemKNN(K=2).fit(X)
        b = ItemKNN(K=2).fit(Xb)
    assert (a.similarity_matrix_ != b.similarity_matrix_).nnz == 0
    assert a.similarity_matrix_.dtype == np.float64
    with pytest.raises(UnsupportedTypeError):
        ItemKNN(K=2).fit(np.ones((3, 3)))
    with pytest.raises(ValueError):
        ItemKNN(similarity="jaccard")
    with pytest.warns(UserWarning):
        ItemKNN(pop_discount=0.5)
    with pytest.raises(ValueError):
        ItemKNN(similarity="conditional_probability", pop_discount=1.5)
    # empty matrix
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        algo = ItemKNN(K=3).fit(csr_matrix((5, 4), dtype=np.int32))
    assert algo.similarity_matrix_.nnz == 0 and algo.similarity_matrix_.shape == (4, 4)
    # dimension mismatch in predict is a ValueError like scipy's matmul
    with pytest.raises(ValueError):
        b.predict(csr_matrix((2, 7), dtype=np.int32))


# ------------------------------------------------------------------------------- predict
def _load_model_from_oracle(engine, X, K, sim="cosine", pd_=None):
    want = orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_)
    I = X.shape[1]
    engine.model_load_topk(I, K, want["idx"], want["val"], want["len"])
    return orc.topk_to_csr(want["idx"], want["val"], want["len"], I)


@pytest.mark.parametrize("flags", [0, 1, 2, 4, 7, 16, 20])
@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[2], CASES[3], CASES[5]])
def test_predict_topn_matches_oracle(engine, case, flags):
    from recpack_b200.matrix import binary_structure
    from recpack_b200.synth import synth_interactions, weak_generalization_split

    U, I, nnz, K, sim, pd_ = case
    X = synth_interactions(U, I, nnz, seed=U + I)
    train, _ = weak_generalization_split(X, 0.8, seed=5)
    S = _load_model_from_oracle(engine, train, K, sim, pd_)
    Xc, indptr, indices = binary_structure(train)
    engine.debug_flags(flags)
    for N, mask in ((20, True), (7, False)):
        got = engine.predict_topn(U, indptr, indices, N, mask_history=mask)
        want = orc.canon_predict_topn(train, S, N, remove_history=mask)
        assert np.array_equal(got["len"], want["len"])
        assert np.array_equal(got["idx"], want["idx"])
        assert np.array_equal(got["val"], want["val"])
        # lists only (no scores asked for): most lists are settled by the approximate sums, the rest are scored
        # again exactly -- the lists must be the same
        lists = engine.predict_topn(U, indptr, indices, N, mask_history=mask, want_val=False)
        assert np.array_equal(lists["len"], want["len"])
        assert np.array_equal(lists["idx"], want["idx"])
    engine.debug_flags(0)


@pytest.mark.parametrize("flags", [0, 2, 4, 6])
def test_predict_lists_only_near_ties_take_the_exact_pass(engine, flags):
    """Scores that differ only in the lowest bits of the fixed-point sums -- inside one item range and across two
    ranges (flag 4: two passes) -- cannot be ordered by the 32-bit approximate sums: those users must come out of
    the second, exact pass (or the in-kernel exact sweep) with the oracle's order."""
    from recpack_b200.matrix import binary_structure

    I, K, U, N = 64, 6, 40, 5
    rng = np.random.default_rng(3)
    # every row: the same few target items spread over both halves of the item range, values equal up to ~1e-11
    base = rng.random(I) * 0.5 + 0.25
    idx = np.zeros((I, K), dtype=np.int32)
    val = np.zeros((I, K))
    targets = np.array([3, 9, 20, 35, 47, 60], dtype=np.int32)
    for i in range(I):
        idx[i] = targets
        val[i] = base[i] * (1.0 + rng.integers(-3, 4, size=K) * 2.0**-36)
    ln = np.full(I, K, dtype=np.int32)
    S = orc.topk_to_csr(idx, val, ln, I)
    engine.model_load_topk(I, K, idx, val, ln)
    rows = [np.sort(rng.choice(np.setdiff1d(np.arange(I), targets), size=rng.integers(1, 30), replace=False)) for _ in range(U)]
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    indices = np.concatenate(rows).astype(np.int32)
    X = csr_matrix((np.ones(len(indices), dtype=np.int32), indices, indptr), shape=(U, I))
    engine.debug_flags(flags)
    want = orc.canon_predict_topn(X, S, N, remove_history=True)
    got = engine.predict_topn(U, indptr, indices, N, mask_history=True, want_val=False)
    full = engine.predict_topn(U, indptr, indices, N, mask_history=True)
    engine.debug_flags(0)
    assert np.array_equal(got["idx"], want["idx"]) and np.array_equal(got["len"], want["len"])
    assert np.array_equal(full["idx"], want["idx"]) and np.array_equal(full["val"], want["val"])


@pytest.mark.parametrize("flags", [0, 1, 4, 32, 33])  # 32: four item ranges (the last holds 24 of the 120 items)
def test_predict_full_csr_matches_oracle_and_reference(engine, flags):
    from recpack_b200.matrix import binary_structure

    g = load_golden("small_cosine")
    S_ref = unpack(g, "S")
    Xin = unpack(g, "Xin")
    S_ref.sort_indices()
    engine.model_load_csr(S_ref.shape[0], S_ref.indptr.astype(np.int64), S_ref.indices.astype(np.int32), S_ref.data)
    Xc, indptr, indices = binary_structure(Xin)
    engine.debug_flags(flags)
    for mask in (False, True):
        o_ptr, o_idx, o_val = engine.predict_csr(Xin.shape[0], indptr, indices, mask_history=mask)
        want = orc.canon_predict_csr(Xin, S_ref, remove_history=mask)
        assert np.array_equal(o_ptr, want.indptr) and np.array_equal(o_idx, want.indices)
        assert np.array_equal(o_val, want.data)
        ref = unpack(g, "pred_nohist" if mask else "pred")
        ref.sort_indices()
        assert np.array_equal(o_idx, ref.indices) and np.array_equal(o_ptr, ref.indptr)
        np.testing.assert_allclose(o_val, ref.data, rtol=1e-9, atol=1e-10)  # the reference's float64 sums
    engine.debug_flags(0)


def test_predict_small_similarities_keep_relative_resolution():
    """Conditional probability with pop_discount = 1 gives similarities ~ c / (n_i n_j) << 1 (round-1 advice: a fixed
    2^-39 absolute resolution lost 1e-4 .. 1e-2 relative there).  The fixed-point scale is chosen per model from its
    largest value, so scores stay within d_u * vmax * 2^-40 of the float64 sums X @ S -- here ~1e-12 relative."""
    from recpack_b200 import ItemKNN
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(3000, 400, 90_000, seed=5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        algo = ItemKNN(K=60, similarity="conditional_probability", pop_discount=1.0).fit(X)
        pred = algo.predict(X)
    S = algo.similarity_matrix_
    vmax = float(S.data.max())
    assert vmax < 1e-2  # similarities far below 1: the regime the advice describes
    ref = csr_matrix(csr_matrix(X).astype(np.float64) @ S)
    ref.sort_indices()
    pred = csr_matrix(pred)
    pred.sort_indices()
    assert np.array_equal(pred.indptr, ref.indptr) and np.array_equal(pred.indices, ref.indices)
    d = np.repeat(np.diff(csr_matrix(X).indptr), np.diff(ref.indptr)).astype(np.float64)
    err = np.abs(pred.data - ref.data)
    assert np.all(err <= d * vmax * 2.0**-40 + 1e-300)
    assert float((err / ref.data).max()) < 1e-9


def test_predict_heavy_user_limb_chunks(engine):
    """A user with more than 4095 history items crosses the limb-normalisation path; identical
    similarity rows with value ~1 force the high-limb bound check."""
    from recpack_b200.matrix import binary_structure

    I, K = 6000, 8
    rng = np.random.default_rng(0)
    idx = np.stack([rng.choice(I, size=K, replace=False) for _ in range(I)]).astype(np.int32)
    val = rng.random((I, K)) * 0.999 + 0.0005
    val[:, 0] = 1.0
    idx[:, 0] = 17  # every row points at item 17 with weight 1 -> score(17) ~ history length
    for r in range(I):  # keep columns unique inside a row
        seen = set()
        for t in range(K):
            while int(idx[r, t]) in seen or (t > 0 and idx[r, t] == 17):
                idx[r, t] = rng.integers(0, I)
            seen.add(int(idx[r, t]))
    ln = np.full(I, K, dtype=np.int32)
    engine.model_load_topk(I, K, idx, val, ln)
    S = orc.topk_to_csr(idx, val, ln, I)
    hist = np.sort(rng.choice(I, size=5000, replace=False)).astype(np.int32)
    X = csr_matrix((np.ones(5003, dtype=np.int32), np.concatenate([hist, [1, 2, 3]]).astype(np.int32), np.array([0, 5000, 5000, 5003])), shape=(3, I))
    Xc, indptr, indices = binary_structure(X)
    for flags in (0, 1):
        engine.debug_flags(flags)
        got = engine.predict_topn(3, indptr, indices, 25, mask_history=False)
        want = orc.canon_predict_topn(X, S, 25, remove_history=False)
        assert np.array_equal(got["idx"], want["idx"]) and np.array_equal(got["val"], want["val"])
        assert got["len"].tolist() == want["len"].tolist()
    engine.debug_flags(0)


def test_model_rejects_bad_values(engine):
    from recpack_b200.engine import RpkError

    idx = np.array([[1], [0]], dtype=np.int32)
    ln = np.array([1, 1], dtype=np.int32)
    for bad in (-0.5, float("nan"), float("inf")):
        with pytest.raises(RpkError):
            engine.model_load_topk(2, 1, idx, np.array([[bad], [0.1]]), ln)
    engine.model_load_topk(2, 1, idx, np.array([[2.5], [0.1]]), ln)  # any non-negative magnitude is representable


@pytest.mark.parametrize("scale", [1.0, 3.7e-9, 5.0e6])
def test_fixed_point_scale_is_relative_to_the_largest_similarity(engine, scale):
    """ADVICE r1: the resolution of the scores must not depend on the magnitude of the similarities
    (conditional probability with pop_discount ~ 1 on a large catalogue gives values ~1e-8..1e-10): scaling every
    value of the model by a constant scales the scores by it and leaves the lists alone; scores agree with the
    float64 product to 1e-11 relative."""
    from recpack_b200.matrix import binary_structure
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(300, 200, 4000, seed=5)
    K, N = 15, 10
    want = orc.canon_fit(X, K=K)
    _, indptr, indices = binary_structure(X)
    engine.model_load_topk(200, K, want["idx"], want["val"], want["len"])
    base = engine.predict_topn(300, indptr, indices, N)
    engine.model_load_topk(200, K, want["idx"], want["val"] * scale, want["len"])
    got = engine.predict_topn(300, indptr, indices, N)
    S = orc.topk_to_csr(want["idx"], want["val"] * scale, want["len"], 200)
    oracle = orc.canon_predict_topn(X, S, N, remove_history=True)
    assert np.array_equal(got["idx"], oracle["idx"]) and np.array_equal(got["val"], oracle["val"])
    ref = (orc.binarize(X).astype(np.float64) @ S).toarray()  # float64 scores of the reference's X @ S
    m = got["idx"] >= 0
    rows = np.repeat(np.arange(300), N).reshape(300, N)
    np.testing.assert_allclose(got["val"][m], ref[rows[m], got["idx"][m]], rtol=1e-10)
    if scale != 1.0 and np.log2(scale) != np.floor(np.log2(scale)):
        # the lists of the scaled model agree with the unscaled model's except where rounding moves a near tie
        assert np.mean(got["idx"] == base["idx"]) > 0.99
    # full CSR output carries the same scale
    o_ptr, o_idx, o_val = engine.predict_csr(300, indptr, indices)
    full = csr_matrix((o_val, o_idx, o_ptr), shape=(300, 200)).toarray()
    np.testing.assert_allclose(full[ref > 0], ref[ref > 0], rtol=1e-10)


# ------------------------------------------------------------------------------- metrics / ranking
def test_metric_unit_vectors_through_public_api():
    """recpack/tests/test_metrics/test_dcg.py:30-156, test_recall.py:13-42; numbers from the reference."""
    from recpack_b200 import CalibratedRecallK, DCGK, NDCGK, RecallK

    g = load_golden("metrics_unit")
    pred = unpack(g, "pred")
    classes = {"ndcg": NDCGK, "recall": RecallK, "dcg": DCGK, "calibrated_recall": CalibratedRecallK}
    for tname in ("true", "simplified", "unrecommended"):
        yt = unpack(g, "true_" + tname)
        for kind, cls in classes.items():
            for k in (1, 2, 3):
                m = cls(k)
                m.calculate(yt, pred)
                np.testing.assert_allclose(m.value, float(g[f"{tname}_{kind}{k}_value"]), rtol=1e-12)
                res = m.results
                order = np.argsort(g[f"{tname}_{kind}{k}_users"])
                assert np.array_equal(res["user_id"].to_numpy(), g[f"{tname}_{kind}{k}_users"][order])
                np.testing.assert_allclose(res["score"].to_numpy(), g[f"{tname}_{kind}{k}_scores"][order], rtol=1e-12, atol=1e-15)
                assert m.name == f"{cls.__name__}_{k}"
    m = NDCGK(2)
    m.calculate(unpack(g, "true_unrecommended"), pred)
    assert m.num_users == 3 and m.num_items == 5
    with pytest.raises(AssertionError):
        NDCGK(2).calculate(csr_matrix((10, 6)), pred)


def test_top_k_ranks_fixture_and_random(engine):
    from recpack_b200 import get_top_K_ranks, get_top_K_values

    g = load_golden("topk_ranks")
    mat = unpack(g, "mat")
    assert (get_top_K_ranks(mat, 20) != unpack(g, "ranks20")).nnz == 0
    rng = np.random.default_rng(1)
    for flags in (0, 2):
        engine.debug_flags(flags)
        dense = np.round(rng.random((40, 900)) * 50) / 50 * (rng.random((40, 900)) < 0.4) - 0.2 * (rng.random((40, 900)) < 0.05)
        Y = csr_matrix(dense)
        for K in (1, 10, 64):
            got = get_top_K_ranks(Y, K)
            want = orc.canon_top_k_ranks(Y, K)
            assert (got != want).nnz == 0
        assert (get_top_K_ranks(Y, None) != orc.canon_top_k_ranks(Y, None)).nnz == 0
    engine.debug_flags(0)
    data_knn = csr_matrix(([0.3, 0.2, 0.1, 0.23, 0.3, 0.5], ([0, 0, 0, 2, 2, 2], [0, 2, 3, 1, 3, 4])), shape=(10, 5))
    topK = csr_matrix(([0.3, 0.2, 0.3, 0.5], ([0, 0, 2, 2], [0, 2, 3, 4])), shape=(10, 5))
    np.testing.assert_almost_equal(topK.todense(), get_top_K_values(data_knn, 2).todense())  # tests/test_util.py:49-62


@pytest.mark.parametrize("name", SMALL)
def test_pipeline_fit_predict_metrics_vs_oracle_and_reference(name):
    """End to end through the drop-in classes: fit -> predict(top-N, history removed) -> NDCG@10 /
    Recall@20.  Bit-exact lists and 1e-12 metrics against the canonical oracle; against the reference's
    own numbers the difference is bounded by the users whose lists differ by tie picks."""
    from recpack_b200 import ItemKNN, NDCGK, RecallK

    g = load_golden(name)
    K, sim, pd_ = _params(g)
    X = unpack(g, "X")
    ytrue = unpack(g, "ytrue")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        algo = ItemKNN(K=K, similarity=sim, pop_discount=pd_, predict_topK=20, remove_history=True).fit(X)
        pred = algo.predict(X)
    want_fit = orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_)
    S = orc.topk_to_csr(want_fit["idx"], want_fit["val"], want_fit["len"], X.shape[1])
    got_S = algo.similarity_matrix_.copy()
    got_S.sort_indices()
    assert np.array_equal(got_S.indices, S.indices) and np.array_equal(got_S.data, S.data)
    want = orc.canon_predict_topn(X, S, 20, remove_history=True)
    idx, ln = pred._rpk_topn
    assert np.array_equal(idx, want["idx"]) and np.array_equal(ln, want["len"])
    res = orc.canon_metrics_from_lists(want["idx"], want["len"], ytrue, [("ndcg", 10), ("recall", 20)])
    for cls, kind, k in ((NDCGK, "ndcg", 10), (RecallK, "recall", 20)):
        m = cls(k)
        m.calculate(ytrue, pred)
        value, per_user, users = res[(kind, k)]
        np.testing.assert_allclose(m.value, value, rtol=1e-12)
        np.testing.assert_allclose(m.results["score"].to_numpy(), per_user, rtol=1e-12, atol=1e-15)
        assert np.array_equal(m.results["user_id"].to_numpy(), users)
        # same metric from a plain CSR (no attached lists): goes through rpk_topk_csr
        plain = csr_matrix(pred)
        m2 = cls(k)
        m2.calculate(ytrue, plain)
        np.testing.assert_allclose(m2.value, value, rtol=1e-12)
        # reference's number: reported difference must stay small (tie picks only)
        ref_value = float(g[f"{kind}{k}_value"])
        # (cond. prob. on 120 items is tie-dominated: the reference's arbitrary picks move it by percents)
        assert abs(m.value - ref_value) <= (0.02 if sim == "cosine" else 0.10) * max(ref_value, 1e-9)


def test_mid_shape_metrics_vs_reference_numbers():
    """ML-100K shape, K=200: metric values next to the unmodified reference's (tie picks move NDCG by
    a few 1e-5 relative, SURVEY.md 0.2) -- asserted at 1e-3, the exact comparison is against the oracle."""
    from recpack_b200 import ItemKNN, NDCGK, RecallK

    g = load_golden("mid_cosine")
    X, ytrue = unpack(g, "X"), unpack(g, "ytrue")
    algo = ItemKNN(K=200, predict_topK=20, remove_history=True).fit(X)
    pred = algo.predict(X)
    for cls, tag, k in ((NDCGK, "ndcg", 10), (RecallK, "recall", 20)):
        m = cls(k)
        m.calculate(ytrue, pred)
        ref = float(g[f"{tag}{k}_value"])
        assert abs(m.value - ref) <= 1e-3 * ref, (tag, m.value, ref)


def test_predict_after_pickle_and_model_reuse():
    """The fitted estimator pickles (similarity_matrix_ is a plain scipy CSR); predict gives the same lists
    whether the model comes from the device-resident fit result, from the host lists or from the CSR."""
    import pickle

    from recpack_b200 import ItemKNN
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(400, 250, 6000, seed=9)
    algo = ItemKNN(K=30, predict_topK=15, remove_history=True).fit(X)
    a = algo.predict(X)                                   # model from the device-resident fit result
    other = ItemKNN(K=7).fit(synth_interactions(50, 40, 300, seed=1))  # invalidates the resident result
    b = algo.predict(X)                                   # model rebuilt from the host lists
    clone = pickle.loads(pickle.dumps(algo))
    clone._fit_lists = None
    c = clone.predict(X)                                  # model from similarity_matrix_ (CSR path)
    for other_pred in (b, c):
        assert np.array_equal(a._rpk_topn[0], other_pred._rpk_topn[0])
        assert np.array_equal(a.data, other_pred.data)
    assert other.similarity_matrix_.shape == (40, 40)


def test_model_load_from_padded_shards(engine):
    """rpk_model_load_topk_rows: model rows read through a row map from padded, gathered per-rank shards."""
    from recpack_b200.matrix import binary_structure
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(300, 200, 4000, seed=21)
    K, N = 12, 10
    want = orc.canon_fit(X, K=K)
    cuts, maxrows = [0, 90, 97, 200], 103
    g_idx = np.full((3 * maxrows, K), -1, dtype=np.int32)
    g_val = np.zeros((3 * maxrows, K))
    g_len = np.zeros(3 * maxrows, dtype=np.int32)
    src = np.empty(200, dtype=np.int64)
    for r in range(3):
        b, e = cuts[r], cuts[r + 1]
        g_idx[r * maxrows : r * maxrows + e - b] = want["idx"][b:e]
        g_val[r * maxrows : r * maxrows + e - b] = want["val"][b:e]
        g_len[r * maxrows : r * maxrows + e - b] = want["len"][b:e]
        src[b:e] = r * maxrows + np.arange(e - b)
    _, indptr, indices = binary_structure(X)
    engine.model_load_topk(200, K, want["idx"], want["val"], want["len"])
    a = engine.predict_topn(300, indptr, indices, N)
    engine.model_load_topk_rows(200, K, 3 * maxrows, g_idx, g_val, g_len, src)
    b_ = engine.predict_topn(300, indptr, indices, N)
    # the same exchange in the packed format: rows packed per shard, loaded through the same row map
    g_ent = np.full((3 * maxrows, K), ~np.uint64(0), dtype=np.uint64)
    for r in range(3):
        b, e = cuts[r], cuts[r + 1]
    exps = [engine.model_scale_exp(K, np.ascontiguousarray(want["val"][cuts[r] : cuts[r + 1]]), np.ascontiguousarray(want["len"][cuts[r] : cuts[r + 1]])) for r in range(3)]
    e_all = min(exps)  # what the all-reduce(MIN) of the ranks gives
    assert e_all == orc.scale_exp(want["val"][np.arange(K)[None, :] < want["len"][:, None]])
    for r in range(3):
        b, e = cuts[r], cuts[r + 1]
        g_ent[r * maxrows : r * maxrows + e - b] = engine.model_pack_rows(200, K, want["idx"][b:e], want["val"][b:e], want["len"][b:e], e_all)
    engine.model_load_packed_rows(200, K, 3 * maxrows, g_ent, g_len, e_all, src)
    c_ = engine.predict_topn(300, indptr, indices, N)
    for key in ("idx", "val", "len"):
        assert np.array_equal(a[key], b_[key]) and np.array_equal(a[key], c_[key])
    from recpack_b200.engine import RpkError

    with pytest.raises(RpkError):  # rows must be in column order
        bad = g_ent.copy()
        r = int(src[np.flatnonzero(want["len"] >= 2)[0]])
        bad[r, :2] = bad[r, 1::-1]
        engine.model_load_packed_rows(200, K, 3 * maxrows, bad, g_len, e_all, src)
    engine.model_load_topk(200, K, want["idx"], want["val"], want["len"])  # leave a valid model behind


@pytest.mark.parametrize("flags,dense_users", [(0, 0), (0, 64), (4, 0), (1, 0), (8, 0), (8, 64)])
def test_fit_items_seen_by_more_than_65535_users(engine, flags, dense_users):
    """Counts between two items that both exceed 65,535 users do not fit the packed 16-bit counters: they come
    from the exact pair kernel (or, with flag 1, from the 32-bit counter path)."""
    rng = np.random.default_rng(4)
    U, I, K = 70_000, 40, 12
    p = np.concatenate([[0.99, 0.97, 0.95, 0.945], rng.random(I - 4) * 0.5 + 0.02])
    X = csr_matrix((rng.random((U, I)) < p[None, :]).astype(np.int32))
    assert (np.bincount(X.indices, minlength=I) >= 65536).sum() >= 3
    engine.debug_flags(flags)
    engine.fit_config(dense_users)
    try:
        got = _fit_lists(engine, X, K)
    finally:
        engine.fit_config(-1)
        engine.debug_flags(0)
    _assert_fit_equal(got, orc.canon_fit(X, K=K))


@pytest.mark.parametrize("flags,dense_users", [(0, 0), (0, 64), (4, 0), (8, 0), (8, 64)])
def test_fit_wrapped_counter_does_not_leak_into_neighbour(engine, flags, dense_users):
    """A packed 16-bit counter in an even slot that passes 65,535 carries into the odd slot next to it; the
    carried amount (known from the exact pair count) is taken back, so the ordinary neighbour column keeps
    its exact count."""
    rng = np.random.default_rng(11)
    U, I, K = 70_000, 40, 39  # K = I - 1: every count of a row is compared
    p = rng.random(I) * 0.5 + 0.02
    p[[0, 2, 6, 9]] = [0.99, 0.97, 0.96, 0.95]   # heavy columns in even slots 0, 2, 6 with ordinary neighbours
    X = csr_matrix((rng.random((U, I)) < p[None, :]).astype(np.int32))
    n = np.bincount(X.indices, minlength=I)
    assert (n >= 65536).sum() == 4 and n[1] < 65536 and n[3] < 65536 and n[7] < 65536
    engine.debug_flags(flags)
    engine.fit_config(dense_users)
    try:
        got = _fit_lists(engine, X, K)
    finally:
        engine.fit_config(-1)
        engine.debug_flags(0)
    _assert_fit_equal(got, orc.canon_fit(X, K=K))


def test_fit_result_stays_on_device_until_used():
    """fit keeps the top-K lists on the device: similarity_matrix_ is built on first access, an assigned matrix
    replaces the device copy, pickles carry the host matrix only, and metrics read the device-resident lists."""
    import pickle

    from recpack_b200 import ItemKNN, NDCGK
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(300, 180, 5000, seed=4)
    Y = synth_interactions(300, 180, 1500, seed=5)
    algo = ItemKNN(K=25, predict_topK=10, remove_history=True).fit(X)
    assert algo.__dict__["_similarity_host"] is None and algo.__dict__["_fit_dev"] is not None
    pred = algo.predict(X)                       # model straight from the device lists
    assert algo.__dict__["_similarity_host"] is None
    assert hasattr(pred, "_rpk_topn_dev")
    m = NDCGK(10)
    m.calculate(Y, pred)
    m_host = NDCGK(10)
    m_host.calculate(Y, csr_matrix(pred))        # plain CSR: ranked again from the host copy
    assert m.value == m_host.value
    S = algo.similarity_matrix_                  # first access builds the CSR
    assert S.shape == (180, 180) and S is algo.similarity_matrix_
    want = orc.canon_fit(X, K=25)
    ref = orc.topk_to_csr(want["idx"], want["val"], want["len"], 180)
    got = S.copy()
    got.sort_indices()
    assert np.array_equal(got.indices, ref.indices) and np.array_equal(got.data, ref.data)
    clone = pickle.loads(pickle.dumps(algo))
    assert clone.__dict__["_fit_dev"] is None
    assert np.array_equal(clone.predict(X)._rpk_topn[0], pred._rpk_topn[0])
    # assigning a matrix replaces the fit result (the reference lets users do this)
    S2 = S.copy()
    S2.data[:] = 1.0
    algo.similarity_matrix_ = S2
    assert algo.__dict__["_fit_dev"] is None
    assert not np.array_equal(algo.predict(X).data, pred.data)


def test_precision_and_reciprocal_rank_through_public_api():
    """PrecisionK / ReciprocalRankK (recpack/metrics/precision.py:41-50, reciprocal_rank.py:37-40) from the same
    top-N lists: reference values on its own fixtures, reference per-user scores on a tie-free matrix, and the
    oracle on lists produced by predict."""
    from recpack_b200 import ItemKNN, PrecisionK, ReciprocalRankK
    from recpack_b200.metrics import precision_k, reciprocal_rank_k
    from recpack_b200.synth import synth_interactions

    g = load_golden("metrics_more")
    cases = [(t, unpack(g, "true_" + t), unpack(g, "pred"), (1, 2, 3)) for t in ("true", "simplified", "unrecommended")]
    cases.append(("big", unpack(g, "big_true"), unpack(g, "big_pred"), (1, 5, 10)))
    for tname, yt, pred, ks in cases:
        for k in ks:
            for cls, kind in ((PrecisionK, "precision"), (ReciprocalRankK, "reciprocal_rank")):
                m = cls(k)
                m.calculate(yt, pred)
                assert m.name == f"{cls.__name__}_{k}"
                np.testing.assert_allclose(m.value, float(g[f"{tname}_{kind}{k}_value"]), rtol=1e-12)
                res = m.results
                order = np.argsort(g[f"{tname}_{kind}{k}_users"])
                assert np.array_equal(res["user_id"].to_numpy(), g[f"{tname}_{kind}{k}_users"][order])
                if tname == "big":
                    np.testing.assert_allclose(res["score"].to_numpy(), g[f"{tname}_{kind}{k}_scores"][order], rtol=1e-12, atol=0)
    np.testing.assert_almost_equal(precision_k(unpack(g, "true_true"), unpack(g, "pred"), 2), 0.75)
    np.testing.assert_almost_equal(reciprocal_rank_k(unpack(g, "true_true"), unpack(g, "pred"), 2), 0.75)
    # device-resident lists from predict
    X = synth_interactions(250, 90, 2500, seed=6)
    Y = synth_interactions(250, 90, 900, seed=8)
    pred = ItemKNN(K=15, predict_topK=12, remove_history=True).fit(X).predict(X)
    idx, ln = pred._rpk_topn
    want = orc.canon_metrics_from_lists(idx, ln, Y, [("precision", 10), ("reciprocal_rank", 10)])
    for cls, kind in ((PrecisionK, "precision"), (ReciprocalRankK, "reciprocal_rank")):
        m = cls(10)
        m.calculate(Y, pred)
        value, per_user, users = want[(kind, 10)]
        np.testing.assert_allclose(m.value, value, rtol=1e-12)
        np.testing.assert_allclose(m.results["score"].to_numpy(), per_user, rtol=1e-12, atol=0)
