"""CPU oracle for RecPack's item-similarity hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module.  The product
(``recpack_b200``) never does: it fails loudly when the CUDA library is missing.

Two tiers live here (SURVEY.md section 8c):

* ``ref_*``   -- a restatement of the reference's own calls (scikit-learn
  ``cosine_similarity``, scipy ``csr @ csr``, numpy ``argpartition``).  The
  arithmetic of the reference lives in those third-party packages (pinned in
  the reference's setup.py:15-17 as numpy/scipy/scikit-learn ``==1.*``; this
  image has numpy 2.3, scipy 1.18, scikit-learn 1.9), so the restatement calls
  the same entry points in the same order.  Its top-K ties are arbitrary, like
  the reference's.  This tier is what the CPU baseline times.
* ``canon_*`` -- the canonical, deterministic definition the CUDA path is
  bit-compared with: exact integer co-occurrence counts, top-K by exact key
  with ties broken by ascending item index, similarity values reproduced with
  the reference's own floating-point operation order, fixed-point scoring.

Parity pinning: ``tests/test_oracle_golden.py`` checks both tiers against
fixtures in ``tests/golden/`` produced by importing the real reference
(``tests/golden/make_golden.py``), and against the closed-form vectors of the
reference's own tests (recpack/tests/test_algorithms/test_nearest_neighbour.py:44-181,
recpack/tests/test_metrics/test_dcg.py:30-156, test_recall.py:13-42).

Reference citations are relative to /root/reference.
"""
from __future__ import annotations

import itertools
from fractions import Fraction

import numpy as np
import scipy.sparse as sp
from scipy.sparse import csr_matrix

# Fixed-point scoring definition (see canon_quantize): the scale 2^e is chosen per model so that the largest
# similarity lands in [2^39, 2^40).
Q_BITS = 39


def scale_exp(values) -> int:
    """e = 39 - floor(log2(vmax)); 39 for an empty / all-zero model."""
    v = np.asarray(values, dtype=np.float64)
    vmax = float(v.max()) if v.size else 0.0
    if not vmax > 0.0:
        return Q_BITS
    return Q_BITS - int(np.floor(np.log2(vmax))) if np.isfinite(vmax) else Q_BITS


# --------------------------------------------------------------------------
# Input coercion  (recpack/algorithms/base.py:129-151, recpack/util.py:99-109)
# --------------------------------------------------------------------------
def binarize(X) -> csr_matrix:
    """Binary CSR with sorted, unique indices and no stored zeros.

    The reference does ``X.astype(bool).astype(X.dtype)`` (util.py:107); a stored
    zero stays in the structure as 0 and contributes nothing to any product,
    so dropping it is equivalent for everything downstream.
    """
    X = csr_matrix(X, copy=True)
    X.sum_duplicates()
    X.eliminate_zeros()
    X.sort_indices()
    X.data = np.ones_like(X.data, dtype=np.int64)
    return X.astype(np.int64)


# --------------------------------------------------------------------------
# Tier A: restatement of the reference's own calls
# --------------------------------------------------------------------------
def ref_cosine(X: csr_matrix) -> csr_matrix:
    """nearest_neighbour.py:69-84 -- cosine between item columns, diagonal set to 0."""
    from sklearn.metrics.pairwise import cosine_similarity

    S = cosine_similarity(X.T, dense_output=False)
    S.setdiag(0)
    return S


def ref_conditional_probability(X: csr_matrix, pop_discount=0) -> csr_matrix:
    """nearest_neighbour.py:22-66 (+ algorithms/util.py:118-133 for the inverse)."""
    Xb = X.astype(bool).astype(X.dtype)
    co = Xb.T @ X
    freq = np.asarray(Xb.sum(axis=0)).ravel()
    D = sp.diags(freq).tocsr()
    A = csr_matrix(D.shape)
    nz = D.nonzero()
    A[nz] = 1 / D[nz]
    S = A @ co @ A.power(pop_discount) if pop_discount else A @ co
    S.setdiag(0)
    return S


def ref_top_k_ranks(X: csr_matrix, K=None) -> csr_matrix:
    """util.py:50-77 -- per row, rank (1 = largest) of the K largest stored values."""
    rows, cols, ranks = [], [], []
    for r in range(X.shape[0]):
        lo, hi = X.indptr[r], X.indptr[r + 1]
        k = hi - lo if K is None else min(K, hi - lo)
        if k == 0:
            continue
        part = np.argpartition(X.data[lo:hi], list(range(-k, 0)))[-k:]
        picked = X.indices[lo + part]
        for rank, c in enumerate(picked[::-1], start=1):
            rows.append(r)
            cols.append(c)
            ranks.append(rank)
    return csr_matrix((ranks, (rows, cols)), shape=X.shape)


def ref_top_k_values(X: csr_matrix, K=None) -> csr_matrix:
    """util.py:80-96."""
    mask = ref_top_k_ranks(X, K)
    mask[mask > 0] = 1
    return mask.multiply(X)


def ref_fit(X, K=200, similarity="cosine", pop_discount=None, normalize_X=False, normalize_sim=False) -> csr_matrix:
    """ItemKNN._fit, nearest_neighbour.py:204-224, after the binarising wrapper base.py:129-139."""
    from sklearn.preprocessing import Normalizer

    X = csr_matrix(X)
    X = X.astype(bool).astype(X.dtype)
    tr = Normalizer(norm="l1", copy=False)
    if normalize_X:
        X = tr.transform(X)
    if similarity == "cosine":
        S = ref_cosine(X)
    elif similarity == "conditional_probability":
        S = ref_conditional_probability(X, pop_discount)
    else:
        raise ValueError(f"similarity {similarity} not supported")
    S = ref_top_k_values(csr_matrix(S), K)
    if normalize_sim:
        S = tr.transform(S)
    return csr_matrix(S)


def ref_fit_row_blocked(X, K=200, block=2048, rows=None) -> csr_matrix:
    """Row-blocked cosine fit (SURVEY.md 8d): the same calls on item-row blocks.

    ``cosine_similarity(Xt[blk], Xt)`` is bit-identical per row to the unblocked
    call; the explicit diagonal zero the reference stores (nearest_neighbour.py:81)
    is reproduced so that it competes in the selection exactly as it does there.
    ``rows`` restricts the work to a sample of item rows (CPU-baseline sampling).
    """
    from sklearn.metrics.pairwise import cosine_similarity

    X = csr_matrix(X).astype(bool).astype(np.float64)
    Xt = X.T.tocsr()
    n_items = Xt.shape[0]
    row_ids = np.arange(n_items) if rows is None else np.asarray(rows)
    out = []
    for s in range(0, len(row_ids), block):
        blk = row_ids[s : s + block]
        Sb = csr_matrix(cosine_similarity(Xt[blk], Xt, dense_output=False))
        # setdiag(0) on the full matrix overwrites the stored diagonal in place; do the same
        # here without disturbing the SpGEMM's entry order (argpartition's tie picks depend on it)
        for r, i in enumerate(blk):
            lo, hi = Sb.indptr[r], Sb.indptr[r + 1]
            hit = np.flatnonzero(Sb.indices[lo:hi] == i)
            if len(hit):
                Sb.data[lo + hit[0]] = 0
        out.append(ref_top_k_values(Sb, K))
    return sp.vstack(out).tocsr() if out else csr_matrix((0, n_items))


def ref_ease(X, l2=1e3, alpha=0) -> csr_matrix:
    """EASE._fit, recpack/algorithms/ease.py:63-95 (without the optional pruning)."""
    X = csr_matrix(X)
    X = X.astype(bool).astype(X.dtype)
    XTX = (X.T @ X).toarray()
    P = np.linalg.inv(XTX + l2 * np.identity((X.shape[1]), dtype=np.float32))
    B = np.identity(X.shape[1]) - P @ np.diag(1.0 / np.diag(P))
    B[np.diag_indices(B.shape[0])] = 0.0
    if alpha != 0:
        w = 1 / np.diag(XTX) ** alpha
        B = B @ np.diag(w)
    return csr_matrix(B)


def ref_predict(X, S) -> csr_matrix:
    """ItemSimilarityMatrixAlgorithm._predict, algorithms/base.py:237-255."""
    X = csr_matrix(X)
    return csr_matrix(X.astype(bool).astype(X.dtype) @ S)


def ref_remove_history(X_pred: csr_matrix, X_in: csr_matrix) -> csr_matrix:
    """pipelines/pipeline.py:174-175."""
    hist = csr_matrix(X_in).astype(bool).astype(np.int64)
    return csr_matrix(X_pred - X_pred.multiply(hist))


def _ref_eliminate_empty(y_true, y_pred):
    """metrics/base.py:106-123."""
    users = sorted(set(y_true.nonzero()[0]))
    return np.array(users, dtype=np.int64), y_true[users, :], y_pred[users, :]


def ref_ndcg(y_true, y_pred, K):
    """MetricTopK.calculate + NDCGK._calculate, metrics/base.py:172-193, metrics/dcg.py:98-128.

    Returns (value, per-user scores, user ids)."""
    y_true, y_pred = csr_matrix(y_true), csr_matrix(y_pred)
    users, yt, yp = _ref_eliminate_empty(y_true, y_pred)
    ranks = ref_top_k_ranks(yp, K)
    disc = 1.0 / np.log2(np.arange(2, K + 2))
    idcg = np.array([1] + list(itertools.accumulate(disc)))
    den = ranks.multiply(yt).tocsr()
    den.data = np.log2(den.data + 1)
    inv = den.copy()
    inv.data = 1 / inv.data
    dcg = np.asarray(yt.multiply(inv).sum(axis=1)).ravel()
    hist = np.asarray(yt.sum(axis=1)).ravel().astype(np.int32)
    hist[hist > K] = K
    per_user = dcg / idcg[hist]
    return (per_user.mean() if len(per_user) else np.nan), per_user, users


def ref_recall(y_true, y_pred, K):
    """RecallK._calculate, metrics/recall.py:38-46."""
    y_true, y_pred = csr_matrix(y_true), csr_matrix(y_pred)
    users, yt, yp = _ref_eliminate_empty(y_true, y_pred)
    ranks = ref_top_k_ranks(yp, K)
    hits = np.asarray(ranks.multiply(yt).astype(bool).sum(axis=1)).ravel()
    per_user = hits / np.asarray(yt.sum(axis=1)).ravel()
    return (per_user.mean() if len(per_user) else np.nan), per_user, users


# --------------------------------------------------------------------------
# Tier B: canonical exact definition
# --------------------------------------------------------------------------
def item_counts(Xb: csr_matrix) -> np.ndarray:
    return np.bincount(Xb.indices, minlength=Xb.shape[1]).astype(np.int64)


class Prepared:
    """Binarised matrix, its transpose and the item popularities, computed once (the sampled-row checks
    at the 100 M / 500 M interaction shapes would otherwise redo the transpose per row block)."""

    def __init__(self, X):
        self.Xb = binarize(X)
        self.Xt = self.Xb.T.tocsr()
        self.n = item_counts(self.Xb)
        self.shape = self.Xb.shape


def prepare(X) -> "Prepared":
    return X if isinstance(X, Prepared) else Prepared(X)


def cooccurrence_rows(Xb, rows) -> np.ndarray:
    """Exact integer co-occurrence counts c[i, :] for the given item rows
    (nearest_neighbour.py:48: ``to_binary(X).T @ X`` restricted to rows)."""
    if isinstance(Xb, Prepared):
        return np.asarray((Xb.Xt[rows] @ Xb.Xb).todense())
    Xt = Xb.T.tocsr().astype(np.int64)
    return np.asarray((Xt[rows] @ Xb.astype(np.int64)).todense())


def seq_sum(p: np.ndarray, c: np.ndarray) -> np.ndarray:
    """s = (((p + p) + p) + ...) with c terms, float64.

    scipy's csr_matmat adds the c identical products fl(a_i * a_j) one at a time
    (scipy/sparse/_compressed.py:444-465 -> sparsetools csr_matmat), so this is the
    reference's value bit for bit (verified in tests/golden/make_golden.py)."""
    p = np.asarray(p, dtype=np.float64)
    c = np.asarray(c, dtype=np.int64)
    s = np.zeros_like(p)
    for t in range(int(c.max()) if c.size else 0):
        live = c > t
        s[live] = s[live] + p[live]
    return s


def _pow_table(n: np.ndarray, pop_discount: float) -> np.ndarray:
    """(1/n_j) ** alpha exactly as ``A.power(pop_discount)`` computes it
    (nearest_neighbour.py:58); items never seen get 0 (they cannot be candidates)."""
    out = np.zeros(len(n), dtype=np.float64)
    nz = n > 0
    out[nz] = np.power(1 / n[nz], pop_discount)
    return out


def canon_order(similarity, pop_discount, c, n_j, pw_j, idx):
    """Permutation sorting candidates best-first under the canonical total order.

    cosine:        exact c^2/n_j descending (n_i is constant inside a row), index ascending
    cond. prob.:   exact integer c descending, index ascending
    with discount: float64 key fl(c * pw_j) descending, index ascending (documented: the
                   key c / n_j^alpha is irrational, float64 is its definition here)
    """
    c = np.asarray(c, dtype=np.int64)
    idx = np.asarray(idx, dtype=np.int64)
    if similarity == "cosine":
        key = (c * c).astype(np.float64) / n_j.astype(np.float64)
    elif pop_discount:
        key = c.astype(np.float64) * pw_j
    else:
        key = c.astype(np.float64)
    order = np.lexsort((idx, -key))
    if similarity == "cosine" and len(order) > 1:
        # float64 division is monotone, so only runs of equal float keys can be
        # mis-ordered; re-sort those runs with exact rationals.
        ks = key[order]
        run_start = np.flatnonzero(np.r_[True, ks[1:] != ks[:-1]])
        run_end = np.r_[run_start[1:], len(ks)]
        for a, b in zip(run_start, run_end):
            if b - a < 2:
                continue
            sub = order[a:b]
            pairs = {(int(c[t]), int(n_j[t])) for t in sub}
            if len({Fraction(cc * cc, nn) for cc, nn in pairs}) > 1:
                sub = sorted(sub, key=lambda t: (-Fraction(int(c[t]) ** 2, int(n_j[t])), int(idx[t])))
                order[a:b] = sub
    return order


def canon_values(similarity, pop_discount, c, n_i, n_j, pw_j):
    """Similarity values with the reference's floating-point operation order."""
    c = np.asarray(c, dtype=np.int64)
    if similarity == "cosine":
        a_i = 1.0 / np.sqrt(np.float64(n_i))  # sklearn sparsefuncs_fast.pyx:578-604
        a_j = 1.0 / np.sqrt(n_j.astype(np.float64))
        return seq_sum(a_i * a_j, c)
    inv_i = 1 / np.float64(n_i)  # algorithms/util.py:132
    v = inv_i * c.astype(np.float64)  # A @ co  (one product per entry)
    if pop_discount:
        v = v * pw_j  # (A @ co) @ A^alpha
    return v


def canon_fit(X, K=200, similarity="cosine", pop_discount=None, rows=None, block=256):
    """Canonical ItemKNN fit.  Returns dict(idx, cnt, val, len) with rows in rank order
    (best first), ``idx`` padded with -1.  ``rows`` restricts to a subset of item rows."""
    Xb = prepare(X)  # a Prepared object may be passed instead of a matrix
    n = Xb.n
    I = Xb.shape[1]
    row_ids = np.arange(I) if rows is None else np.asarray(rows, dtype=np.int64)
    pw = _pow_table(n, pop_discount) if pop_discount else None
    Kc = int(min(K, max(I - 1, 0)))
    idx = np.full((len(row_ids), K), -1, dtype=np.int32)
    cnt = np.zeros((len(row_ids), K), dtype=np.int32)
    val = np.zeros((len(row_ids), K), dtype=np.float64)
    ln = np.zeros(len(row_ids), dtype=np.int32)
    for s in range(0, len(row_ids), block):
        blk = row_ids[s : s + block]
        C = cooccurrence_rows(Xb, blk)
        for r, i in enumerate(blk):
            crow = C[r].copy()
            crow[i] = 0  # diagonal never survives (nearest_neighbour.py:64,81 + util.py:96)
            cand = np.flatnonzero(crow)
            if len(cand) == 0:
                continue
            cc = crow[cand]
            order = canon_order(similarity, pop_discount, cc, n[cand], pw[cand] if pw is not None else None, cand)
            keep = order[:Kc]
            m = len(keep)
            j = cand[keep]
            idx[s + r, :m] = j
            cnt[s + r, :m] = cc[keep]
            val[s + r, :m] = canon_values(similarity, pop_discount, cc[keep], n[i], n[j], pw[j] if pw is not None else None)
            ln[s + r] = m
    return {"idx": idx, "cnt": cnt, "val": val, "len": ln}


def topk_to_csr(idx, val, ln, n_cols) -> csr_matrix:
    """[rows x K] rank-ordered lists -> CSR with sorted column indices."""
    rows = np.repeat(np.arange(len(ln)), ln)
    mask = np.arange(idx.shape[1])[None, :] < np.asarray(ln)[:, None]
    S = csr_matrix((val[mask], (rows, idx[mask])), shape=(len(ln), n_cols))
    S.sort_indices()
    return S


def canon_quantize(values: np.ndarray, e: int = None) -> np.ndarray:
    """Fixed-point image of the similarity values of ONE model: q = clip(rint(v * 2^e), 1, 2^40 - 1) with the
    model's scale exponent e (scale_exp of all its values unless given).

    Scores are exact integer sums of q, hence independent of summation order; a stored entry never
    vanishes (|q * 2^-e - v| <= 2^-(e+1) unless v < 2^-(e+1))."""
    v = np.asarray(values, dtype=np.float64)
    if np.any(~(v >= 0)) or np.any(~np.isfinite(v)):
        raise ValueError("similarity values must be finite and non-negative")
    e = scale_exp(v) if e is None else e
    sv = np.ldexp(v, e)
    if np.any(sv >= float(1 << 40)):
        raise ValueError("similarity values do not fit 40 bits at this scale")
    # a stored entry never vanishes; a value within half a step of 2^40 would round up to it: clamped
    return np.clip(np.rint(sv).astype(np.int64), 1, (1 << 40) - 1)


def canon_scores_q(X, S: csr_matrix) -> csr_matrix:
    """Exact fixed-point scores  sum_{i in hist(u)} q_ij  as an int64 CSR (users x items)."""
    Xb = binarize(X)
    Sq = csr_matrix(S, copy=True)
    Sq.sum_duplicates()
    Sq.eliminate_zeros()
    Sq = csr_matrix((canon_quantize(Sq.data), Sq.indices, Sq.indptr), shape=Sq.shape)
    out = (Xb.astype(np.int64) @ Sq).tocsr()
    out.sort_indices()
    return out


def canon_score_scale(S: csr_matrix) -> float:
    """2^-e of the model: exact scores are score_q * this."""
    Sq = csr_matrix(S, copy=True)
    Sq.sum_duplicates()
    Sq.eliminate_zeros()
    return float(np.ldexp(1.0, -scale_exp(Sq.data)))


def canon_predict_topn(X, S, N, remove_history=True):
    """Canonical top-N lists: (score desc, item index asc); history masked before truncation
    (pipeline.py:174-175 happens before metrics/base.py:189 in the reference).

    Returns dict(idx [U,N] -1 padded, score_q [U,N] int64, val [U,N] float64, len [U])."""
    Xb = binarize(X)
    scores = canon_scores_q(Xb, S)
    U = Xb.shape[0]
    idx = np.full((U, N), -1, dtype=np.int32)
    sq = np.zeros((U, N), dtype=np.int64)
    ln = np.zeros(U, dtype=np.int32)
    for u in range(U):
        lo, hi = scores.indptr[u], scores.indptr[u + 1]
        cols = scores.indices[lo:hi]
        vals = scores.data[lo:hi]
        if remove_history and hi > lo:
            keep = ~np.isin(cols, Xb.indices[Xb.indptr[u] : Xb.indptr[u + 1]])
            cols, vals = cols[keep], vals[keep]
        if len(cols) == 0:
            continue
        order = np.lexsort((cols, -vals))[:N]
        m = len(order)
        idx[u, :m] = cols[order]
        sq[u, :m] = vals[order]
        ln[u] = m
    return {"idx": idx, "score_q": sq, "val": sq.astype(np.float64) * canon_score_scale(S), "len": ln}


def canon_predict_csr(X, S, remove_history=False) -> csr_matrix:
    """Full canonical score matrix (float64 = score_q * 2^-39), reference layout of predict()."""
    Xb = binarize(X)
    sc = canon_scores_q(Xb, S)
    out = csr_matrix((sc.data.astype(np.float64) * canon_score_scale(S), sc.indices, sc.indptr), shape=sc.shape)
    if remove_history:
        out = csr_matrix(out - out.multiply(Xb))
        out.eliminate_zeros()
    return out


def discount_tables(K):
    """metrics/dcg.py:98-104: discount template and IDCG cache (IDCG[0] = 1 guard)."""
    disc = 1.0 / np.log2(np.arange(2, K + 2))
    idcg = np.array([1] + list(itertools.accumulate(disc)), dtype=np.float64)
    return disc, idcg


def canon_metrics_from_lists(top_idx, top_len, y_true, metrics):
    """NDCG@K / Recall@K / DCG@K / CalibratedRecall@K / Precision@K / ReciprocalRank@K from rank-ordered lists.

    ``metrics`` is a list of (kind, K).  Users with an empty y_true row are dropped
    (metrics/base.py:106-123); a user with true items but no recommendations scores 0.
    Returns {(kind, K): (value, per_user, user_ids)}."""
    yt = binarize(y_true)
    true_len = np.diff(yt.indptr)
    users = np.flatnonzero(true_len > 0)
    out = {}
    for kind, K in metrics:
        disc, idcg = discount_tables(K)
        per_user = np.zeros(len(users), dtype=np.float64)
        for t, u in enumerate(users):
            truth = yt.indices[yt.indptr[u] : yt.indptr[u + 1]]
            m = min(int(top_len[u]), K, top_idx.shape[1])
            hit = np.isin(top_idx[u, :m], truth)
            if kind in ("ndcg", "dcg"):
                dcg = float(np.sum(disc[:m][hit]))
                per_user[t] = dcg / idcg[min(len(truth), K)] if kind == "ndcg" else dcg
            elif kind == "recall":
                per_user[t] = hit.sum() / len(truth)
            elif kind == "calibrated_recall":
                per_user[t] = hit.sum() / min(len(truth), K)
            elif kind == "precision":  # metrics/precision.py:41-50: divided by K even when fewer were recommended
                per_user[t] = hit.sum() / K
            elif kind == "reciprocal_rank":  # metrics/reciprocal_rank.py:37-40
                where = np.flatnonzero(hit)
                per_user[t] = 1.0 / (where[0] + 1) if len(where) else 0.0
            else:
                raise ValueError(kind)
        out[(kind, K)] = (per_user.mean() if len(users) else float("nan"), per_user, users)
    return out


def canon_top_k_ranks(Y: csr_matrix, K) -> csr_matrix:
    """get_top_K_ranks (util.py:50-77) with the canonical tie rule (value desc, column asc)."""
    Y = csr_matrix(Y)
    rows, cols, ranks = [], [], []
    for r in range(Y.shape[0]):
        lo, hi = Y.indptr[r], Y.indptr[r + 1]
        order = np.lexsort((Y.indices[lo:hi], -Y.data[lo:hi]))
        k = hi - lo if K is None else min(K, hi - lo)
        for rank, t in enumerate(order[:k], start=1):
            rows.append(r)
            cols.append(Y.indices[lo + t])
            ranks.append(rank)
    return csr_matrix((ranks, (rows, cols)), shape=Y.shape)


# --------------------------------------------------------------------------
# Real-valued interaction matrices: ItemKNN(normalize_X=True), Pearson (SURVEY.md 8f-2)
# --------------------------------------------------------------------------
def ref_normalize_X(X) -> csr_matrix:
    """nearest_neighbour.py:205-210 after the binarising wrapper (base.py:129-139): l1-normalised binary rows."""
    from sklearn.preprocessing import Normalizer

    X = csr_matrix(X)
    X = X.astype(bool).astype(X.dtype)
    return Normalizer(norm="l1", copy=False).transform(X)


def ref_pearson(X: csr_matrix) -> csr_matrix:
    """nearest_neighbour.py:87-111 -- cosine of the matrix centred per item over its positive entries."""
    if (X == 1).sum() == X.nnz:
        raise ValueError("Pearson similarity can not be computed on a binary matrix.")
    count = (X > 0).sum(axis=0).A
    avg = X.sum(axis=0).A.astype(float)
    avg[count > 0] = avg[count > 0] / count[count > 0]
    X = X - (X > 0).multiply(avg)
    return ref_cosine(csr_matrix(X))


def ref_real_full(X, similarity="cosine", pop_discount=None) -> csr_matrix:
    """The full item x item matrix of a real-valued X, as compute_cosine_similarity / compute_conditional_probability
    return it (explicit zeros on the diagonal)."""
    X = csr_matrix(X)
    if similarity == "cosine":
        return csr_matrix(ref_cosine(X))
    if similarity == "conditional_probability":
        return csr_matrix(ref_conditional_probability(X, pop_discount))
    if similarity == "pearson":
        return csr_matrix(ref_pearson(X))
    raise ValueError(f"similarity {similarity} not supported")


def canon_topk_of_full(full: csr_matrix, K: int):
    """Canonical get_top_K_values (util.py:50-96) of a full similarity matrix: per row the min(K, stored) best STORED
    entries by (value descending, item ascending) -- explicit zeros such as the diagonal compete (util.py:63-68) --
    and entries equal to zero then drop out of the product (util.py:96).  Returns dict(idx, val, len), rank order."""
    full = csr_matrix(full)
    rows = full.shape[0]
    idx = np.full((rows, K), -1, dtype=np.int32)
    val = np.zeros((rows, K), dtype=np.float64)
    ln = np.zeros(rows, dtype=np.int32)
    for r in range(rows):
        lo, hi = full.indptr[r], full.indptr[r + 1]
        cols = full.indices[lo:hi]
        vals = full.data[lo:hi].astype(np.float64)
        order = np.lexsort((cols, -vals))[: min(K, hi - lo)]
        keep = order[vals[order] != 0.0]
        ln[r] = keep.size
        idx[r, : keep.size] = cols[keep]
        val[r, : keep.size] = vals[keep]
    return {"idx": idx, "val": val, "len": ln}


def canon_fit_real(X, K, similarity="cosine", pop_discount=None):
    """Canonical top-K of the reference's own float64 similarity values for a real-valued X."""
    return canon_topk_of_full(ref_real_full(X, similarity, pop_discount), K)


# --------------------------------------------------------------------------
# Data side: FractionInteractionSplitter (SURVEY.md 8f-4)
# --------------------------------------------------------------------------
def ref_fraction_split_mask(user_ix: np.ndarray, in_frac: float, seed: int) -> np.ndarray:
    """scenarios/splitters.py:233-263 -- per user (ascending id, rows in table order, as pandas groupby yields them)
    shuffle the row positions with np.random.RandomState(seed + u) and send the first ceil(n * in_frac) to data_in.
    Returns the boolean mask of the table rows that end up in data_in.  The generator is numpy's (MT19937 + legacy
    shuffle; not vendored in the reference)."""
    user_ix = np.asarray(user_ix, dtype=np.int64)
    order = np.argsort(user_ix, kind="stable")
    su = user_ix[order]
    bounds = np.flatnonzero(np.r_[True, su[1:] != su[:-1], True])
    mask = np.zeros(user_ix.shape[0], dtype=bool)
    for b, e in zip(bounds[:-1], bounds[1:]):
        hist = order[b:e].copy()
        np.random.RandomState(int(seed) + int(su[b])).shuffle(hist)
        cut = int(np.ceil((e - b) * in_frac))
        mask[hist[:cut]] = True
    return mask


# --------------------------------------------------------------------------
# Tie-aware comparison against the unmodified reference (SURVEY.md 8c (3))
# --------------------------------------------------------------------------
def compare_topk_tie_aware(ref_S: csr_matrix, got, Xb: csr_matrix, similarity="cosine", rel=1e-5, rows=None):
    """Compare reference top-K rows (arbitrary ties) with canonical lists ``got``.

    Per row: the sorted kept values must agree to ``rel``; items kept by only one side
    must all sit in the boundary tie group (exact key equal to the K-th exact key, widened
    by 4*c*2^-53 relative because the reference's own sums carry that much rounding noise).
    Row r of ``ref_S`` is item ``rows[r]`` (default: item r), so a sample of the reference's
    rows can be checked against the full lists.
    Returns dict(rows_checked, rows_with_diff, max_rel_err)."""
    ref_S = csr_matrix(ref_S)
    n = item_counts(Xb)
    stats = {"rows_checked": 0, "rows_with_diff": 0, "max_rel_err": 0.0}
    for r in range(ref_S.shape[0]):
        i = r if rows is None else int(rows[r])
        lo, hi = ref_S.indptr[r], ref_S.indptr[r + 1]
        rj, rv = ref_S.indices[lo:hi], ref_S.data[lo:hi]
        m = int(got["len"][i])
        gj, gv, gc = got["idx"][i, :m], got["val"][i, :m], got["cnt"][i, :m]
        assert len(rj) == m, f"row {i}: reference keeps {len(rj)} entries, canonical {m}"
        stats["rows_checked"] += 1
        if m == 0:
            continue
        a, b = np.sort(rv), np.sort(gv)
        err = float(np.max(np.abs(a - b) / np.maximum(np.abs(a), 1e-300)))
        stats["max_rel_err"] = max(stats["max_rel_err"], err)
        assert err <= rel, f"row {i}: kept values differ by {err}"
        only = np.setxor1d(rj, gj)
        if len(only) == 0:
            continue
        stats["rows_with_diff"] += 1
        c_last, j_last = int(gc[m - 1]), int(gj[m - 1])
        if similarity == "cosine":
            k_last = Fraction(c_last * c_last, int(n[j_last]))
        else:
            k_last = Fraction(c_last)
        crow = cooccurrence_rows(Xb, [i])[0]
        for j in only:
            cj = int(crow[j])
            kj = Fraction(cj * cj, int(n[j])) if similarity == "cosine" else Fraction(cj)
            tol = Fraction(4 * max(cj, c_last) * 4, 1 << 53)  # squared key: twice the relative noise, doubled for safety
            assert abs(kj - k_last) <= tol * k_last, f"row {i}: item {j} differs outside the boundary tie group"
    return stats
