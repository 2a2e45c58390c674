"""Pin the oracle (oracle/recpack_oracle.py) to outputs of the real reference.

The fixtures in tests/golden/ were produced by tests/golden/make_golden.py, which imports
the unmodified reference from /root/reference.  CPU only."""
import math

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from conftest import load_golden, unpack
from oracle import recpack_oracle as orc

UNIT = ["unit_cosine", "unit_empty_col", "unit_condprob", "unit_condprob_pd1", "unit_condprob_pd0.2", "unit_condprob_pd0.5"]
SMALL = ["small_cosine", "small_condprob", "small_condprob_pd"]


def _params(g):
    pd_ = float(g["pop_discount"])
    return int(g["K"]), str(g["similarity"]), (None if math.isnan(pd_) else pd_)


def _same_csr(A, B):
    A, B = csr_matrix(A), csr_matrix(B)
    A.sort_indices()
    B.sort_indices()
    return A.shape == B.shape and np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices) and np.array_equal(A.data, B.data)


@pytest.mark.parametrize("name", UNIT + SMALL)
def test_ref_tier_reproduces_reference_bit_for_bit(name):
    g = load_golden(name)
    K, sim, pd_ = _params(g)
    S = orc.ref_fit(unpack(g, "X"), K=K, similarity=sim, pop_discount=pd_)
    assert _same_csr(S, unpack(g, "S"))
    pred = orc.ref_predict(unpack(g, "Xin"), S)
    assert _same_csr(pred, unpack(g, "pred"))
    assert _same_csr(orc.ref_remove_history(pred, unpack(g, "Xin")), unpack(g, "pred_nohist"))


def test_ref_tier_normalize_sim():
    g = load_golden("unit_normalize_sim")
    S = orc.ref_fit(unpack(g, "X"), K=2, normalize_sim=True)
    assert _same_csr(S, unpack(g, "S"))


def test_ref_row_blocked_equals_unblocked():
    g = load_golden("small_cosine")
    X = unpack(g, "X")
    S = orc.ref_fit_row_blocked(X, K=int(g["K"]), block=32)
    assert _same_csr(S, unpack(g, "S"))


def test_unit_closed_forms():
    """recpack/tests/test_algorithms/test_nearest_neighbour.py:44-70,119-152."""
    g = load_golden("unit_cosine")
    got = orc.canon_fit(unpack(g, "X"), K=2)
    S = orc.topk_to_csr(got["idx"], got["val"], got["len"], 3).toarray()
    e = 2 / math.sqrt(6)
    np.testing.assert_almost_equal(S, [[0, 0.5, e], [0.5, 0, e], [e, e, 0]])
    g = load_golden("unit_condprob")
    got = orc.canon_fit(unpack(g, "X"), K=2, similarity="conditional_probability")
    S = orc.topk_to_csr(got["idx"], got["val"], got["len"], 3).toarray()
    np.testing.assert_almost_equal(S, [[0, 0.5, 1], [0.5, 0, 1], [2 / 3, 2 / 3, 0]])
    g = load_golden("unit_empty_col")
    got = orc.canon_fit(unpack(g, "X"), K=2)
    S = orc.topk_to_csr(got["idx"], got["val"], got["len"], 3).toarray()
    np.testing.assert_almost_equal(S, [[0, 0, 0], [0, 0, e], [0, e, 0]])
    assert got["len"].tolist() == [0, 1, 1]


@pytest.mark.parametrize("name", UNIT + SMALL + ["mid_cosine"])
def test_canonical_fit_vs_reference_tie_aware(name):
    g = load_golden(name)
    K = int(g["K"])
    sim = str(g["similarity"]) if "similarity" in g else "cosine"
    pd_ = None
    if "pop_discount" in g and not math.isnan(float(g["pop_discount"])):
        pd_ = float(g["pop_discount"])
    X = unpack(g, "X")
    S_ref = unpack(g, "S")
    got = orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_)
    Xb = orc.binarize(X)
    if pd_:
        # irrational keys: the canonical order is the float64 key; compare values only
        S = orc.topk_to_csr(got["idx"], got["val"], got["len"], X.shape[1])
        a, b = np.sort(S.data), np.sort(S_ref.data)
        np.testing.assert_allclose(a, b, rtol=1e-12)
        return
    # mid_cosine keeps a seeded sample of the reference's rows (S_rows) to stay small
    rows = g["S_rows"] if "S_rows" in g else np.arange(X.shape[1])
    stats = orc.compare_topk_tie_aware(S_ref, got, Xb, similarity=sim, rows=rows)
    assert stats["rows_checked"] == len(rows)
    # kept values are reproduced with the reference's own operation order: wherever the two
    # sides keep the same item the float64 value must be IDENTICAL
    S = orc.topk_to_csr(got["idx"], got["val"], got["len"], X.shape[1])[rows]
    common = S.multiply(S_ref.astype(bool)).tocsr()
    ref_common = S_ref.multiply(S.astype(bool)).tocsr()
    common.sort_indices()
    ref_common.sort_indices()
    assert np.array_equal(common.data, ref_common.data)
    if name == "mid_cosine":
        assert stats["rows_with_diff"] > 0  # the reference's tie picks are arbitrary (SURVEY 0.2)


@pytest.mark.parametrize("name", SMALL)
def test_canonical_predict_and_metrics_vs_reference(name):
    g = load_golden(name)
    S_ref = unpack(g, "S")
    Xin = unpack(g, "Xin")
    # scoring with the REFERENCE's S isolates the scoring / metric definitions from fit ties
    full = orc.canon_predict_csr(Xin, S_ref)
    ref_pred = unpack(g, "pred")
    ref_pred.sort_indices()
    assert np.array_equal(full.indices, ref_pred.indices) and np.array_equal(full.indptr, ref_pred.indptr)
    np.testing.assert_allclose(full.data, ref_pred.data, rtol=1e-9, atol=1e-10)
    top = orc.canon_predict_topn(Xin, S_ref, 20, remove_history=True)
    ytrue = unpack(g, "ytrue")
    nohist = unpack(g, "pred_nohist")
    # (1) the restated reference metrics reproduce the reference's numbers (same arbitrary ties)
    np.testing.assert_allclose(orc.ref_ndcg(ytrue, nohist, 10)[0], float(g["ndcg10_value"]), rtol=1e-12)
    np.testing.assert_allclose(orc.ref_recall(ytrue, nohist, 20)[0], float(g["recall20_value"]), rtol=1e-12)
    # (2) canonical lists vs the reference's own rank matrix: identical score multisets per user;
    #     item differences are tie picks (metrics/base.py:189 -> util.py:68 argpartition)
    ref_ranks = orc.ref_top_k_ranks(nohist, 20)
    nohist.sort_indices()
    same_list = np.zeros(Xin.shape[0], dtype=bool)
    for u in range(Xin.shape[0]):
        row = ref_ranks[u]
        ref_items = row.indices[np.argsort(row.data)]
        m = int(top["len"][u])
        assert len(ref_items) == m
        dense = nohist[u].toarray().ravel()
        np.testing.assert_allclose(np.sort(dense[ref_items]), np.sort(top["val"][u, :m]), rtol=1e-9, atol=1e-11)
        same_list[u] = np.array_equal(ref_items, top["idx"][u, :m])
    res = orc.canon_metrics_from_lists(top["idx"], top["len"], ytrue, [("ndcg", 10), ("recall", 20), ("dcg", 10), ("calibrated_recall", 20)])
    for (kind, k), (value, per_user, users) in res.items():
        order = np.argsort(g[f"{kind}{k}_users"])
        assert np.array_equal(np.sort(g[f"{kind}{k}_users"]), users)
        ref_scores = g[f"{kind}{k}_scores"][order]
        ok = same_list[users]
        np.testing.assert_allclose(per_user[ok], ref_scores[ok], rtol=1e-12, atol=1e-15)
        if ok.all():
            np.testing.assert_allclose(value, float(g[f"{kind}{k}_value"]), rtol=1e-12)
    if name == "small_cosine":
        assert same_list.mean() > 0.5


def test_metric_unit_vectors():
    """recpack/tests/test_metrics/test_dcg.py:30-156, test_recall.py:13-42 (values from the reference)."""
    g = load_golden("metrics_unit")
    pred = unpack(g, "pred")
    for tname in ("true", "simplified", "unrecommended"):
        yt = unpack(g, "true_" + tname)
        for k in (1, 2, 3):
            ranks = orc.canon_top_k_ranks(pred, k)
            U = pred.shape[0]
            idx = np.full((U, k), -1, dtype=np.int32)
            ln = np.zeros(U, dtype=np.int32)
            for u in range(U):
                row = ranks[u]
                for c, r in zip(row.indices, row.data):
                    idx[u, int(r) - 1] = c
                ln[u] = row.nnz
            res = orc.canon_metrics_from_lists(idx, ln, yt, [("ndcg", k), ("recall", k), ("dcg", k), ("calibrated_recall", k)])
            for (kind, kk), (value, per_user, users) in res.items():
                np.testing.assert_allclose(value, float(g[f"{tname}_{kind}{kk}_value"]), rtol=1e-12)
                assert np.array_equal(np.sort(g[f"{tname}_{kind}{kk}_users"]), users)
            # restated reference metrics agree as well
            np.testing.assert_allclose(orc.ref_ndcg(yt, pred, k)[0], float(g[f"{tname}_ndcg{k}_value"]), rtol=1e-12)
            np.testing.assert_allclose(orc.ref_recall(yt, pred, k)[0], float(g[f"{tname}_recall{k}_value"]), rtol=1e-12)
    # closed forms quoted in the reference tests
    np.testing.assert_almost_equal(float(g["true_recall2_value"]), 2 / 3)
    np.testing.assert_almost_equal(float(g["unrecommended_recall2_value"]), 4 / 9)
    idcg2 = 1 + 1 / np.log2(3)
    np.testing.assert_almost_equal(float(g["true_ndcg2_value"]), ((1 / np.log2(3)) / idcg2 + (1 + 1 / np.log2(3)) / idcg2) / 2)


def test_top_k_ranks_fixture():
    """recpack/tests/test_util.py:14-25."""
    g = load_golden("topk_ranks")
    mat = unpack(g, "mat")
    ref = unpack(g, "ranks20")
    got = orc.canon_top_k_ranks(mat, 20)
    assert (got != ref).nnz == 0  # no ties in this fixture -> identical
    assert _same_csr(orc.ref_top_k_ranks(mat, 20), ref)


def _lists_from_ranks(pred, k):
    ranks = orc.canon_top_k_ranks(pred, k)
    U = pred.shape[0]
    idx = np.full((U, k), -1, dtype=np.int32)
    ln = np.zeros(U, dtype=np.int32)
    for u in range(U):
        row = ranks[u]
        for c, r in zip(row.indices, row.data):
            idx[u, int(r) - 1] = c
        ln[u] = row.nnz
    return idx, ln


def test_precision_and_reciprocal_rank_vs_reference():
    """recpack/metrics/precision.py:41-50, reciprocal_rank.py:37-40: values and per-user scores produced by the
    reference (tests/golden/make_golden.py more) on its own metric fixtures and on a tie-free random matrix."""
    g = load_golden("metrics_more")
    cases = [(t, unpack(g, "true_" + t), unpack(g, "pred"), (1, 2, 3)) for t in ("true", "simplified", "unrecommended")]
    cases.append(("big", unpack(g, "big_true"), unpack(g, "big_pred"), (1, 5, 10)))
    for tname, yt, pred, ks in cases:
        for k in ks:
            idx, ln = _lists_from_ranks(pred, k)
            res = orc.canon_metrics_from_lists(idx, ln, yt, [("precision", k), ("reciprocal_rank", k)])
            for (kind, kk), (value, per_user, users) in res.items():
                np.testing.assert_allclose(value, float(g[f"{tname}_{kind}{kk}_value"]), rtol=1e-12)
                order = np.argsort(g[f"{tname}_{kind}{kk}_users"])
                assert np.array_equal(g[f"{tname}_{kind}{kk}_users"][order], users)
                if tname == "big":  # no score ties: the per-user numbers are the reference's
                    np.testing.assert_allclose(per_user, g[f"{tname}_{kind}{kk}_scores"][order], rtol=1e-12, atol=0)
    # closed forms quoted in the reference tests (recpack/tests/test_metrics/test_precision.py:16-21,
    # test_reciprocal_rank.py:14-19)
    np.testing.assert_almost_equal(float(g["true_precision2_value"]), 0.75)
    np.testing.assert_almost_equal(float(g["true_reciprocal_rank2_value"]), 0.75)


# ---- real-valued interaction matrices (ItemKNN(normalize_X=True), Pearson): fixtures of tests/golden/make_golden_real.py
REAL_NORMX = ["real_unit_normx_cosine", "real_unit_normx_condprob", "real_small_normx_cosine", "real_small_normx_condprob",
              "real_small_normx_condprob_pd", "real_mid_normx_cosine"]
REAL_PEARSON = ["real_unit_pearson", "real_small_pearson"]


def _kept_sets_tie_aware(canon, ref_S, full, K):
    """Row by row: same number of kept entries, same multiset of values, and every item picked by only one side carries
    the boundary value (the reference's introselect breaks ties arbitrarily, SURVEY.md 0.2)."""
    ref_S, full = csr_matrix(ref_S), csr_matrix(full)
    for r in range(full.shape[0]):
        n = int(canon["len"][r])
        mine = dict(zip(canon["idx"][r, :n].tolist(), canon["val"][r, :n].tolist()))
        lo, hi = ref_S.indptr[r], ref_S.indptr[r + 1]
        theirs = dict(zip(ref_S.indices[lo:hi].tolist(), ref_S.data[lo:hi].tolist()))
        assert len(mine) == len(theirs), r
        assert sorted(mine.values()) == sorted(theirs.values()), r
        only = set(mine) ^ set(theirs)
        if only:
            boundary = min(mine.values())
            for j in only:
                assert (mine.get(j, theirs.get(j))) == boundary, (r, j)
        for j in set(mine) & set(theirs):
            assert mine[j] == theirs[j]


@pytest.mark.parametrize("name", REAL_NORMX)
def test_real_valued_oracle_reproduces_reference_normalize_X(name):
    g = load_golden(name)
    K, sim, pd_ = _params(g)
    full = orc.ref_real_full(orc.ref_normalize_X(unpack(g, "X")), sim, pd_)
    assert _same_csr(full, unpack(g, "full"))
    S = orc.ref_fit(unpack(g, "X"), K=K, similarity=sim, pop_discount=pd_, normalize_X=True)
    assert _same_csr(S, unpack(g, "S"))
    _kept_sets_tie_aware(orc.canon_topk_of_full(unpack(g, "full"), K), unpack(g, "S"), unpack(g, "full"), K)


@pytest.mark.parametrize("name", REAL_PEARSON)
def test_real_valued_oracle_reproduces_reference_pearson(name):
    g = load_golden(name)
    K = int(g["K"])
    full = orc.ref_real_full(unpack(g, "X"), "pearson")
    assert _same_csr(full, unpack(g, "full"))
    _kept_sets_tie_aware(orc.canon_topk_of_full(unpack(g, "full"), K), unpack(g, "S"), unpack(g, "full"), K)


def test_normalize_X_closed_form():
    """recpack/tests/test_algorithms/test_nearest_neighbour.py:73-107."""
    g = load_golden("real_unit_normx_cosine")
    got = orc.canon_topk_of_full(unpack(g, "full"), 2)
    S = orc.topk_to_csr(got["idx"], got["val"], got["len"], 3).toarray()
    a, b = 1 / 9, 1 / 9 + 1 / 4
    d = math.sqrt(1 / 4 + 1 / 9)
    f = math.sqrt(2 / 4 + 1 / 9)
    np.testing.assert_almost_equal(S, [[0, a / (d * d), b / (d * f)], [a / (d * d), 0, b / (d * f)], [b / (d * f), b / (d * f), 0]])


@pytest.mark.parametrize("name", ["split_small", "split_heavy"])
def test_fraction_split_oracle_reproduces_reference(name):
    """Fixtures of tests/golden/make_golden_split.py (the reference's FractionInteractionSplitter.split)."""
    g = load_golden(name)
    mask = orc.ref_fraction_split_mask(g["uid"], float(g["in_frac"]), int(g["seed"]))
    assert np.array_equal(np.sort(g["interactionid"][mask]), g["in_ids"])
    assert np.array_equal(np.sort(g["interactionid"][~mask]), g["out_ids"])


@pytest.mark.parametrize("name", ["tars_cosine_exp", "tars_condprob_linear", "tars_pearson_vaz", "tars_pearson_bigK", "tars_liu2012",
                                  "tars_lee", "tars_ding_nofitdecay"])
def test_tars_goldens_canonical_topk_is_the_references_up_to_ties(name):
    """Fixtures of tests/golden/make_golden_tars.py: the canonical selection from the reference's full similarity matrix
    keeps what the reference's get_top_K_values keeps (tie-aware), negatives and the competing diagonal zero included."""
    g = load_golden(name)
    K = int(g["K"])
    _kept_sets_tie_aware(orc.canon_topk_of_full(unpack(g, "full"), K), unpack(g, "S"), unpack(g, "full"), K)
