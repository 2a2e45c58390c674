"""Oracle of the dense EASE chain (DESIGN.md 2, 4.7): the exact Gram, the closed form from the inverse and scipy's
``binary(X) @ B`` with a dense float64 model, in plain numpy.

* ``canon_gram``: ``X.T @ X`` as int64 counts (``ease.py:79``).
* ``canon_ease_from_inverse``: ``B_ij = -fl(P_ij * fl(1 / P_jj)) * w_j``, ``B_ii = +0.0`` -- the elementwise form of
  ``I - P @ diag(1 / diag(P))`` and ``@ diag(w)`` (``ease.py:83-88``) in the order of the reference's products.
* ``canon_dense_scores``: scipy's ``csr_matvecs`` order -- every score starts at ``0.0`` and adds ``B[i, j]`` over
  the history items ``i`` in ascending order, one rounding per add -- then optionally zeroes the history columns.
* ``canon_dense_topn``: the N largest scores ``!= 0.0`` by (value desc, column asc), the stored entries of
  ``csr_matrix(scores)``."""
import numpy as np


def canon_gram(X):
    """Exact co-occurrence counts ``X.T @ X`` of the binary interaction matrix X (scipy sparse or dense), int64."""
    from scipy.sparse import csr_matrix

    Xb = csr_matrix(X, copy=True)
    Xb.data[:] = 1
    Xb = Xb.astype(np.int64)
    return np.asarray((Xb.T @ Xb).toarray(), dtype=np.int64)


def canon_ease_from_inverse(P, w=None):
    """B from the inverse P [I, I]: off the diagonal ``-(P_ij * (1 / P_jj))``, then ``* w_j`` when w is given (inf in w
    gives NaN where P_ij = 0 and ±inf elsewhere, as the reference's matrix products do); the diagonal is ``+0.0``."""
    P = np.asarray(P, dtype=np.float64)
    inv = 1.0 / np.diag(P)
    with np.errstate(invalid="ignore", over="ignore"):
        B = -(P * inv[None, :])
        if w is not None:
            B = B * np.asarray(w, dtype=np.float64)[None, :]
    np.fill_diagonal(B, 0.0)
    return B


def _rows_lookup(rows_of_B):
    """(item ids, rows): the full B [I, I], or a pair (sorted item ids, their rows of B)."""
    if isinstance(rows_of_B, tuple):
        items, rows = rows_of_B
        return np.asarray(items, dtype=np.int64), np.asarray(rows, dtype=np.float64)
    rows = np.asarray(rows_of_B, dtype=np.float64)
    return np.arange(rows.shape[0], dtype=np.int64), rows


def canon_dense_scores(indptr, indices, rows_of_B, mask_history=False):
    """Scores [U, I] of the users of the CSR structure (indptr, indices; indices ascending within a row) against B.

    rows_of_B: B itself, or ``(items, rows)`` with ``rows[k] = B[items[k]]`` for sorted ``items`` that cover every
    history item (so that a large B need not be on the host).  The additions run by history position over all users
    at once; each element still sees the adds of its own user in ascending item order, starting from 0.0."""
    indptr = np.asarray(indptr, dtype=np.int64)
    indices = np.asarray(indices, dtype=np.int64)
    items, rows = _rows_lookup(rows_of_B)
    U = indptr.shape[0] - 1
    I = rows.shape[1]
    d = np.diff(indptr)
    owner = np.repeat(np.arange(U), d)
    assert np.all((np.diff(indices) > 0) | (np.diff(owner) != 0)), "history items must ascend within a user"
    pos = np.searchsorted(items, indices)
    assert np.all(pos < items.shape[0]) and np.array_equal(items[np.minimum(pos, items.shape[0] - 1)], indices), \
        "rows_of_B does not cover the history"
    S = np.zeros((U, I), dtype=np.float64)
    for k in range(int(d.max()) if U else 0):
        us = np.flatnonzero(d > k)
        S[us] += rows[pos[indptr[us] + k]]
    if mask_history:
        S[owner, indices] = 0.0
    return S


def canon_dense_topn(scores, N):
    """dict(idx [U, N] -1 padded, val [U, N] 0.0 padded, len [U]): per row the N largest values ``!= 0.0`` by
    (value desc, column asc).  NaN scores have no place in that order: the rows must hold none."""
    scores = np.asarray(scores, dtype=np.float64)
    U = scores.shape[0]
    assert not np.isnan(scores).any(), "NaN scores are not ranked"
    idx = np.full((U, N), -1, dtype=np.int32)
    val = np.zeros((U, N), dtype=np.float64)
    ln = np.zeros(U, dtype=np.int32)
    for u in range(U):
        cols = np.flatnonzero(scores[u] != 0.0)
        if cols.size == 0:
            continue
        v = scores[u, cols]
        order = np.lexsort((cols, -v))[:N]
        m = order.shape[0]
        idx[u, :m] = cols[order]
        val[u, :m] = v[order]
        ln[u] = m
    return {"idx": idx, "val": val, "len": ln}
