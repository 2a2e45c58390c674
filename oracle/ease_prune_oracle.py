"""Oracle of EASE's pruning (``EASE(density=...)``, recpack/algorithms/ease.py:97-109; DESIGN.md 2, "Pruning").

``ref_ease_prune`` restates the reference's ``_prune``; ``canon_ease_prune`` is the canonical definition the GPU path
implements: the reference leaves the pick inside the group of equal magnitudes at the cut to ``argpartition``, the
canonical rule takes those entries in row-major order."""
import numpy as np
from scipy.sparse import csr_matrix

_NAN_KEY = np.uint64(0x7FF0000000000001)  # one key above +inf (0x7ff0000000000000) for every NaN


def ref_ease_prune(S, density) -> csr_matrix:
    """``EASE._prune`` on ``similarity_matrix_ = csr_matrix(B)``, run only ``if self.density`` (``np.product`` is
    ``np.prod``, removed under numpy 2)."""
    S = csr_matrix(S, dtype=np.float64, copy=True)
    if not density:
        return S
    K = min(int(density * np.prod(S.shape)), S.nnz)
    S.data[np.argpartition(abs(S.data), -K)[0:-K]] = 0
    S.eliminate_zeros()
    return S


def prune_keys(values) -> np.ndarray:
    """The ordering key of a value: the bit pattern of |v| as uint64, every NaN one key above +inf."""
    k = np.ascontiguousarray(values, dtype=np.float64).view(np.uint64) & np.uint64(0x7FFFFFFFFFFFFFFF)
    return np.minimum(k, _NAN_KEY)


def canon_prune_topk(S, keep) -> csr_matrix:
    """The min(keep, nnz) stored entries (values != 0.0) with the largest |v|, ties by row-major position, as a canonical
    CSR with the values unchanged (rpk_ease_prune)."""
    S = csr_matrix(S, dtype=np.float64, copy=True)
    S.sum_duplicates()
    S.eliminate_zeros()  # also drops -0.0
    rows = np.repeat(np.arange(S.shape[0], dtype=np.int64), np.diff(S.indptr))
    K = min(int(keep), S.nnz)
    order = np.lexsort((S.indices, rows, ~prune_keys(S.data)))[:K]  # key descending, then row, then column
    kept = np.zeros(S.nnz, dtype=bool)
    kept[order] = True
    counts = np.bincount(rows[kept], minlength=S.shape[0])
    indptr = np.zeros(S.shape[0] + 1, dtype=np.int64)
    np.cumsum(counts, out=indptr[1:])
    return csr_matrix((S.data[kept], S.indices[kept], indptr), shape=S.shape)


def canon_ease_prune(S, density) -> csr_matrix:
    """The canonical ``_prune``: nothing when ``density`` is falsy; else K = min(int(density * (rows*cols)), nnz), one
    float64 product of the exact integer size, and K = 0 keeps every entry, as the reference's ``[0:-0]`` does."""
    S = csr_matrix(S, dtype=np.float64, copy=True)
    if not density:
        return S
    n = int(S.shape[0]) * int(S.shape[1])
    K = int(float(density) * n)
    return canon_prune_topk(S, K if K > 0 else n)
