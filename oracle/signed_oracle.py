"""Oracle of the float64 scoring of signed similarity models (DESIGN.md 2, "Signed models").

The reference's ``ItemSimilarityMatrixAlgorithm._predict`` is ``X @ similarity_matrix_`` (algorithms/base.py:237-255),
which scipy computes with csr_matmat: every score is the left fold, in float64, of ``s_ij`` over the user's history
items in their stored (ascending) order, and a sum of exactly 0.0 is not stored.  The lists are then built from the
stored entries only."""
import numpy as np
from scipy.sparse import csr_matrix


def canon_predict_signed(X, S, N=None, remove_history=False, allowed=None):
    """scipy's ``binary(X) @ S``, then the history removal (pipelines/pipeline.py:174-175) and the item filter
    (``allowed``: bool / 0-1 per item, postprocessing/filters.py:58-101).

    N None: the CSR of the remaining stored scores (ascending columns).  Else dict(idx [U, N] -1 padded,
    val [U, N] 0 padded, len [U]): the N largest stored scores per user by (value desc, column asc)."""
    X = csr_matrix(X, dtype=np.float64, copy=True)
    X.sort_indices()
    X.data[:] = 1.0
    S = csr_matrix(S, dtype=np.float64)
    P = csr_matrix(X @ S)  # csr_matmat: stored entries are the non-zero sums
    P.sort_indices()
    U, I = P.shape
    drop = np.zeros(P.nnz, dtype=bool)
    rows = np.repeat(np.arange(U), np.diff(P.indptr))
    if remove_history:
        for u in np.flatnonzero(np.diff(P.indptr)):
            lo, hi = P.indptr[u], P.indptr[u + 1]
            drop[lo:hi] |= np.isin(P.indices[lo:hi], X.indices[X.indptr[u] : X.indptr[u + 1]])
    if allowed is not None:
        drop |= ~np.asarray(allowed, dtype=bool)[P.indices]
    keep = ~drop
    counts = np.bincount(rows[keep], minlength=U)
    indptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(counts, out=indptr[1:])
    out = csr_matrix((P.data[keep], P.indices[keep], indptr), shape=(U, I))
    if N is None:
        return out
    idx = np.full((U, N), -1, dtype=np.int32)
    val = np.zeros((U, N))
    ln = np.zeros(U, dtype=np.int32)
    for u in range(U):
        lo, hi = out.indptr[u], out.indptr[u + 1]
        if hi == lo:
            continue
        cols, vals = out.indices[lo:hi], out.data[lo:hi]
        order = np.lexsort((cols, -vals))[:N]
        m = len(order)
        idx[u, :m] = cols[order]
        val[u, :m] = vals[order]
        ln[u] = m
    return {"idx": idx, "val": val, "len": ln}
