"""Oracle of factor-model scoring (DESIGN.md 2, "Factor models"; rpk_factor_topn / rpk_factor_full).

The definition, restated in numpy operation by operation:
  score   s_uj = left fold over d of fl(p_ud * q_jd), starting from the first product; separate multiply and add
  users   only users with a stored entry in X are scored (the reference's users = set(X.nonzero()[0]))
  stored  the scores != 0.0 (lil_matrix.__setitem__ drops zeros)
  lists   remove_history removes the user's history columns, `allowed` (the item filter) the filtered columns, then
          the N largest stored scores by (value desc, column asc)
The fold is vectorised over a block of users and sequential over d (numpy's elementwise multiply and add round once
each, so no FMA enters).

`ref_factor_predict` restates the reference's own recipe (FactorizationAlgorithm._predict: lil_matrix rows assigned
from numpy's `@`, BLAS order).  `emulate_factor_screen` is the two-operand, two-scale form of
embed_oracle.emulate_screen."""
from concurrent.futures import ThreadPoolExecutor
import os

import numpy as np
from scipy.sparse import csr_matrix, lil_matrix

from oracle.embed_oracle import screen_eps, screen_scale, tf32_rna


def canon_factor_scores(P, Q, rows):
    """s[rows, :] as float64 [len(rows) x I], the left fold over d."""
    P = np.asarray(P, dtype=np.float64)
    QT = np.ascontiguousarray(np.asarray(Q, dtype=np.float64).T)
    A = P[np.asarray(rows, dtype=np.int64)]
    acc = A[:, 0, None] * QT[0][None, :]
    tmp = np.empty_like(acc)
    for d in range(1, P.shape[1]):
        np.multiply(A[:, d, None], QT[d][None, :], out=tmp)
        np.add(acc, tmp, out=acc)
    return acc


def _hist(X, u):
    return X.indices[X.indptr[u] : X.indptr[u + 1]]


def canon_factor_full(P, Q, X, remove_history=False, allowed=None, block=256):
    """Every score as float64 [U x I]: 0.0 for users without history, history columns (remove_history) and filtered
    columns."""
    X = csr_matrix(X)
    U, I = X.shape
    out = np.zeros((U, I))
    users = np.flatnonzero(np.diff(X.indptr) > 0)
    for b0 in range(0, len(users), block):
        ub = users[b0 : b0 + block]
        out[ub] = canon_factor_scores(P, Q, ub)
    if remove_history:
        for u in users:
            out[u, _hist(X, u)] = 0.0
    if allowed is not None:
        out[:, ~np.asarray(allowed, dtype=bool)] = 0.0
    return out


def canon_factor_topn(P, Q, X, N, remove_history=False, allowed=None, users=None, block=64, threads=None):
    """dict(idx int32 [R x N] -1 padded, val float64 [R x N] 0 padded, len int32 [R]) for the users `users` (default:
    all rows of X, in order)."""
    X = csr_matrix(X)
    U, I = X.shape
    users = np.arange(U) if users is None else np.asarray(users, dtype=np.int64)
    R = len(users)
    idx = np.full((R, N), -1, dtype=np.int32)
    val = np.zeros((R, N))
    ln = np.zeros(R, dtype=np.int32)
    ok = None if allowed is None else np.asarray(allowed, dtype=bool)

    def work(b0):
        ub = users[b0 : b0 + block]
        S = canon_factor_scores(P, Q, ub)
        for t, u in enumerate(ub):
            if X.indptr[u + 1] == X.indptr[u]:
                continue
            v = S[t]
            if remove_history:
                v[_hist(X, u)] = 0.0
            if ok is not None:
                v[~ok] = 0.0
            cols = np.flatnonzero(v != 0.0)
            order = np.lexsort((cols, -v[cols]))[:N]
            idx[b0 + t, : len(order)] = cols[order]
            val[b0 + t, : len(order)] = v[cols[order]]
            ln[b0 + t] = len(order)

    n_threads = threads or min(32, os.cpu_count() or 1)
    with ThreadPoolExecutor(n_threads) as ex:
        list(ex.map(work, range(0, R, block)))
    return {"idx": idx, "val": val, "len": ln}


def ref_factor_predict(P, Q, X):
    """The reference's recipe: users = set(X.nonzero()[0]); result[users] = P[users] @ Q.T into a lil_matrix."""
    users = list(set(X.nonzero()[0]))
    result = lil_matrix(X.shape)
    result[users] = P[users] @ Q.T
    return result.tocsr()


# ---- the screen's error bound with two operands (DESIGN.md 4.10) ------------------------------------------------
def factor_screen_delta(P, Q):
    """delta_uj in the units of s: eps_D r_u r_j + beta, r = row norms, beta = 2^-100 2^-(sp+sq) + (2D+2) 2^-1074."""
    D = P.shape[1]
    sp, sq = screen_scale(P), screen_scale(Q)
    rp = np.sqrt(np.einsum("ij,ij->i", P, P)) * (1 + 2.0**-40)
    rq = np.sqrt(np.einsum("ij,ij->i", Q, Q)) * (1 + 2.0**-40)
    beta = 2.0**-100 * 2.0 ** (-(sp + sq)) + (2 * D + 2) * 2.0**-1074
    return screen_eps(D) * np.outer(rp, rq) + beta


def emulate_factor_screen(P, Q):
    """Pessimistic emulation of the tensor-core screen with two operands, each scaled by its own power of two: tf32
    operands, exact fp32 products, an fp32 accumulation that truncates at every one of the D additions.  Returns s^ in
    the units of s (float64)."""
    sp, sq = screen_scale(P), screen_scale(Q)
    A = tf32_rna(np.ldexp(P, sp).astype(np.float32)).astype(np.float64)
    B = tf32_rna(np.ldexp(Q, sq).astype(np.float32)).astype(np.float64)
    acc = np.zeros((A.shape[0], B.shape[0]), dtype=np.float32)
    for d in range(A.shape[1]):
        p = (A[:, d, None] * B[None, :, d]).astype(np.float32)  # exact: 11 x 11 significant bits
        exact = acc.astype(np.float64) + p.astype(np.float64)
        acc = exact.astype(np.float32)
        over = np.abs(acc.astype(np.float64)) > np.abs(exact)  # round-to-nearest went away from zero: step back
        acc[over] = np.nextafter(acc[over], np.float32(0))
    return np.ldexp(acc.astype(np.float64), -(sp + sq))
