"""Oracle of the item neighbours of a dense embedding matrix (DESIGN.md 2, "Embedding neighbours"; rpk_embed_topk).

The definition, restated in numpy operation by operation:
  dot     s_ij = left fold over d of fl(e_id * e_jd), starting from the first product; separate multiply and add
  cosine  the same fold over xhat_i = fl(e_i / n_i), n_i = fl(sqrt(left fold of fl(e_id * e_id))); n_i == 0 leaves the row
  lists   per row i, over j != i, the K largest values that are not exactly 0.0, by (value desc, column asc)
The fold is vectorised over the pairs of a row block and sequential over d (numpy's elementwise multiply and add round
once each, so no FMA enters); row blocks run in threads (numpy releases the GIL)."""
from concurrent.futures import ThreadPoolExecutor
import os

import numpy as np


def canon_rows(E, similarity):
    """The rows the fold runs over: E itself (dot) or the canonical normalised rows (cosine)."""
    E = np.ascontiguousarray(E, dtype=np.float64)
    if similarity == "dot":
        return E
    if similarity != "cosine":
        raise ValueError(similarity)
    ss = E[:, 0] * E[:, 0]
    for d in range(1, E.shape[1]):
        ss = ss + E[:, d] * E[:, d]
    n = np.sqrt(ss)
    with np.errstate(invalid="ignore", divide="ignore"):
        X = E / np.where(n == 0.0, 1.0, n)[:, None]
    return np.where((n == 0.0)[:, None], E, X)


def canon_block(X, rows):
    """s[rows, :] as float64 [len(rows) x I], the left fold over d."""
    XT = np.ascontiguousarray(X.T)
    A = X[rows]
    acc = A[:, 0, None] * XT[0][None, :]
    tmp = np.empty_like(acc)
    for d in range(1, X.shape[1]):
        np.multiply(A[:, d, None], XT[d][None, :], out=tmp)
        np.add(acc, tmp, out=acc)
    return acc


def _select(vals, row, K):
    vals = vals.copy()
    vals[row] = 0.0
    cols = np.flatnonzero(vals != 0.0)
    order = np.lexsort((cols, -vals[cols]))[:K]
    return cols[order].astype(np.int32), vals[cols[order]]


def canon_embed_topk(E, K, similarity="cosine", rows=None, block=64, threads=None):
    """dict(idx int32 [R x K] -1 padded, val float64 [R x K] 0 padded, len int32 [R]) for the item rows `rows`
    (default: all, in order) against all I columns."""
    X = canon_rows(E, similarity)
    I = X.shape[0]
    rows = np.arange(I) if rows is None else np.asarray(rows, dtype=np.int64)
    R = len(rows)
    idx = np.full((R, K), -1, dtype=np.int32)
    val = np.zeros((R, K))
    ln = np.zeros(R, dtype=np.int32)

    def work(b0):
        rb = rows[b0 : b0 + block]
        S = canon_block(X, rb)
        for t, r in enumerate(rb):
            c, v = _select(S[t], r, K)
            idx[b0 + t, : len(c)] = c
            val[b0 + t, : len(c)] = v
            ln[b0 + t] = len(c)

    n_threads = threads or min(32, os.cpu_count() or 1)
    with ThreadPoolExecutor(n_threads) as ex:
        list(ex.map(work, range(0, R, block)))
    return {"idx": idx, "val": val, "len": ln}


# ---- the screen's error bound (DESIGN.md 4.9) ------------------------------------------------------------------
def screen_scale(X):
    """sigma: the largest row norm of 2^sigma X lies in [1, 2) (0 for an all-zero matrix)."""
    q = float(np.max(np.einsum("ij,ij->i", X, X))) if X.size else 0.0
    if q == 0.0:
        return 0
    return 1 - int(np.frexp(np.sqrt(q))[1])


def screen_eps(D):
    return 2.0**-10 + (D + 2) * 2.0**-22


def screen_delta(X, sigma):
    """delta_ij in the units of s: eps_D r_i r_j + beta, r = row norms of 2^sigma X (scaled back)."""
    D = X.shape[1]
    r = np.sqrt(np.einsum("ij,ij->i", X, X)) * (1 + 2.0**-40)
    beta = 2.0**-100 * 2.0 ** (-2 * sigma) + (2 * D + 2) * 2.0**-1074
    return screen_eps(D) * np.outer(r, r) + beta


def tf32_rna(f32):
    """cvt.rna.tf32.f32: round to 10 fraction bits, ties away from zero; values below 2^-126 flushed first."""
    f = np.where(np.abs(f32) < np.float32(2.0**-126), np.float32(0), f32).astype(np.float32)
    b = f.view(np.uint32).astype(np.uint64)
    b = (b + 0x1000) & 0xFFFFE000
    return b.astype(np.uint32).view(np.float32)


def emulate_screen(X, sigma):
    """Pessimistic emulation of the tensor-core screen: tf32 operands, exact fp32 products, and an fp32 accumulation
    that truncates (rounds toward zero) at every one of the D additions.  Returns s^ in the units of s (float64)."""
    A = tf32_rna(np.ldexp(X, sigma).astype(np.float32)).astype(np.float64)
    I, D = A.shape
    acc = np.zeros((I, I), dtype=np.float32)
    for d in range(D):
        p = (A[:, d, None] * A[None, :, d]).astype(np.float32)  # exact: 11 x 11 significant bits
        exact = acc.astype(np.float64) + p.astype(np.float64)
        acc = exact.astype(np.float32)
        over = np.abs(acc.astype(np.float64)) > np.abs(exact)  # round-to-nearest went away from zero: step back
        acc[over] = np.nextafter(acc[over], np.float32(0))
    return np.ldexp(acc.astype(np.float64), -2 * sigma)
