"""Generate golden vectors by running the REAL reference (imported from /root/reference).

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Writes tests/golden/*.npz.  Every array is an input or an output of unmodified
reference code: recpack.algorithms.ItemKNN, recpack.metrics.NDCGK / RecallK,
recpack.util.get_top_K_ranks.  The fixtures are small on purpose (committed).
"""
import os
import sys
import warnings

import numpy as np
from scipy.sparse import csr_matrix

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)

from recpack.algorithms import ItemKNN  # noqa: E402  (the reference)
from recpack.metrics import NDCGK, RecallK  # noqa: E402
from recpack.metrics.dcg import DCGK  # noqa: E402
from recpack.metrics.recall import CalibratedRecallK  # noqa: E402
from recpack.util import get_top_K_ranks  # noqa: E402

from recpack_b200.synth import synth_interactions, weak_generalization_split  # noqa: E402


def pack(prefix, M, out):
    M = csr_matrix(M)
    out[prefix + "_indptr"] = M.indptr.astype(np.int64)
    out[prefix + "_indices"] = M.indices.astype(np.int32)
    out[prefix + "_data"] = M.data.astype(np.float64)
    out[prefix + "_shape"] = np.array(M.shape, dtype=np.int64)


def knn_case(name, X, K, similarity="cosine", pop_discount=None, X_pred_in=None, y_true=None, normalize_sim=False):
    out = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        algo = ItemKNN(K=K, similarity=similarity, pop_discount=pop_discount, normalize_sim=normalize_sim)
        algo.fit(X)
        pack("X", X, out)
        pack("S", algo.similarity_matrix_, out)
        out["K"] = np.array(K)
        out["similarity"] = np.array(similarity)
        out["pop_discount"] = np.array(np.nan if pop_discount is None else pop_discount)
        out["normalize_sim"] = np.array(normalize_sim)
        if X_pred_in is not None:
            pred = algo.predict(X_pred_in)
            pack("Xin", X_pred_in, out)
            pack("pred", pred, out)
            Xin_b = csr_matrix(X_pred_in).astype(bool).astype(np.int64)
            pred_nohist = csr_matrix(pred - pred.multiply(Xin_b))  # pipelines/pipeline.py:174-175
            pack("pred_nohist", pred_nohist, out)
            if y_true is not None:
                pack("ytrue", y_true, out)
                for cls, tag, k in ((NDCGK, "ndcg", 10), (RecallK, "recall", 20), (DCGK, "dcg", 10), (CalibratedRecallK, "calibrated_recall", 20)):
                    m = cls(k)
                    m.calculate(csr_matrix(y_true), pred_nohist)
                    out[f"{tag}{k}_value"] = np.array(m.value)
                    res = m.results
                    out[f"{tag}{k}_users"] = res["user_id"].to_numpy().astype(np.int64)
                    out[f"{tag}{k}_scores"] = res["score"].to_numpy().astype(np.float64)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "S nnz", algo.similarity_matrix_.nnz)


def main():
    # 1. the reference's own unit-test matrices (tests/test_algorithms/test_nearest_neighbour.py:24-41)
    data = csr_matrix(([1] * 7, ([0, 0, 1, 1, 2, 2, 2], [1, 2, 0, 2, 0, 1, 2])), shape=(4, 3))
    data_empty_col = csr_matrix(([1] * 5, ([0, 0, 1, 1, 2], [1, 2, 2, 1, 2])))
    eye_in = csr_matrix(([1, 1, 1], ([0, 1, 2], [0, 1, 2])), shape=(3, 3))
    knn_case("unit_cosine", data, 2, X_pred_in=eye_in)
    knn_case("unit_empty_col", data_empty_col, 2, X_pred_in=csr_matrix(data_empty_col))
    knn_case("unit_condprob", data, 2, similarity="conditional_probability", X_pred_in=eye_in)
    for pd_ in (1, 0.2, 0.5):
        knn_case(f"unit_condprob_pd{pd_}", data, 2, similarity="conditional_probability", pop_discount=pd_, X_pred_in=eye_in)
    knn_case("unit_normalize_sim", data, 2, normalize_sim=True, X_pred_in=eye_in)

    # 2. seeded power-law matrices through fit -> predict -> history removal -> metrics
    for name, (U, I, nnz), K, sim, pdisc in (
        ("small_cosine", (300, 120, 3000), 10, "cosine", None),
        ("small_condprob", (300, 120, 3000), 10, "conditional_probability", None),
        ("small_condprob_pd", (300, 120, 3000), 10, "conditional_probability", 0.5),
        ("mid_cosine", (943, 1682, 100_000), 200, "cosine", None),
    ):
        X = synth_interactions(U, I, nnz, seed=7)
        train, test_out = weak_generalization_split(X, 0.8, seed=11)
        if name == "mid_cosine":
            # keep the committed fixture small: inputs, scalar metric values and a seeded sample of 512 rows of S
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                algo = ItemKNN(K=K).fit(train)
                pred = algo.predict(train)
                pred = csr_matrix(pred - pred.multiply(train))
                out = {}
                pack("X", train, out)
                pack("ytrue", test_out, out)
                S = csr_matrix(algo.similarity_matrix_)
                rows = np.sort(np.random.default_rng(0).choice(S.shape[0], size=512, replace=False))
                pack("S", S[rows], out)
                out["S_rows"] = rows.astype(np.int64)
                out["K"] = np.array(K)
                for cls, tag, k in ((NDCGK, "ndcg", 10), (RecallK, "recall", 20)):
                    m = cls(k)
                    m.calculate(test_out, pred)
                    out[f"{tag}{k}_value"] = np.array(m.value)
                np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
                print(name, "S nnz", algo.similarity_matrix_.nnz)
        else:
            knn_case(name, train, K, similarity=sim, pop_discount=pdisc, X_pred_in=train, y_true=test_out)

    # 3. get_top_K_ranks on the reference's seeded fixture (tests/test_util.py:14-25)
    import scipy.sparse

    mat = scipy.sparse.random(2, 100, density=0.10, random_state=np.random.RandomState(13940)).tocsr()
    out = {}
    pack("mat", mat, out)
    pack("ranks20", get_top_K_ranks(mat, 20), out)
    np.savez_compressed(os.path.join(HERE, "topk_ranks.npz"), **out)

    # 4. metric fixtures (tests/test_metrics/conftest.py:29-74)
    X_pred = csr_matrix(([0.3, 0.2, 0.1, 0.23, 0.3, 0.5], ([0, 0, 0, 2, 2, 2], [0, 2, 3, 1, 3, 4])), shape=(10, 5))
    truths = {
        "true": csr_matrix(([1] * 5, ([0, 0, 2, 2, 2], [0, 2, 0, 1, 3])), shape=(10, 5)),
        "simplified": csr_matrix(([1] * 2, ([0, 2], [2, 4])), shape=(10, 5)),
        "unrecommended": csr_matrix(([1] * 6, ([0, 0, 2, 2, 2, 3], [0, 2, 0, 1, 3, 1])), shape=(10, 5)),
    }
    out = {}
    pack("pred", X_pred, out)
    for tname, yt in truths.items():
        pack("true_" + tname, yt, out)
        for cls, tag in ((NDCGK, "ndcg"), (RecallK, "recall"), (DCGK, "dcg"), (CalibratedRecallK, "calibrated_recall")):
            for k in (1, 2, 3):
                m = cls(k)
                m.calculate(yt, X_pred)
                out[f"{tname}_{tag}{k}_value"] = np.array(m.value)
                out[f"{tname}_{tag}{k}_scores"] = m.results["score"].to_numpy().astype(np.float64)
                out[f"{tname}_{tag}{k}_users"] = m.results["user_id"].to_numpy().astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "metrics_unit.npz"), **out)
    more_metrics(X_pred, truths)
    print("done")


def more_metrics(X_pred=None, truths=None):
    """5. PrecisionK / ReciprocalRankK on the same fixtures (tests/test_metrics/test_precision.py,
    test_reciprocal_rank.py use them) and on a seeded prediction matrix without score ties."""
    from recpack.metrics.precision import PrecisionK
    from recpack.metrics.reciprocal_rank import ReciprocalRankK

    if X_pred is None:
        X_pred = csr_matrix(([0.3, 0.2, 0.1, 0.23, 0.3, 0.5], ([0, 0, 0, 2, 2, 2], [0, 2, 3, 1, 3, 4])), shape=(10, 5))
        truths = {
            "true": csr_matrix(([1] * 5, ([0, 0, 2, 2, 2], [0, 2, 0, 1, 3])), shape=(10, 5)),
            "simplified": csr_matrix(([1] * 2, ([0, 2], [2, 4])), shape=(10, 5)),
            "unrecommended": csr_matrix(([1] * 6, ([0, 0, 2, 2, 2, 3], [0, 2, 0, 1, 3, 1])), shape=(10, 5)),
        }
    rng = np.random.default_rng(3)
    dense = rng.permutation(60 * 40).reshape(60, 40).astype(np.float64) + 1.0  # distinct scores: no tie picks
    dense[rng.random((60, 40)) < 0.7] = 0.0
    big_pred = csr_matrix(dense)
    big_true = csr_matrix((rng.random((60, 40)) < 0.15).astype(np.int64))
    out = {}
    pack("pred", X_pred, out)
    pack("big_pred", big_pred, out)
    pack("big_true", big_true, out)
    cases = [(t, yt, X_pred, (1, 2, 3)) for t, yt in truths.items()] + [("big", big_true, big_pred, (1, 5, 10))]
    for tname, yt, pr, ks in cases:
        if tname != "big":
            pack("true_" + tname, yt, out)
        for cls, tag in ((PrecisionK, "precision"), (ReciprocalRankK, "reciprocal_rank")):
            for k in ks:
                m = cls(k)
                m.calculate(yt, pr)
                out[f"{tname}_{tag}{k}_value"] = np.array(m.value)
                out[f"{tname}_{tag}{k}_scores"] = m.results["score"].to_numpy().astype(np.float64)
                out[f"{tname}_{tag}{k}_users"] = m.results["user_id"].to_numpy().astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "metrics_more.npz"), **out)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "more":
    more_metrics()  # only the fixture added later; the others are left as committed
elif __name__ == "__main__":
    main()
