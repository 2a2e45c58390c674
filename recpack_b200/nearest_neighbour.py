"""ItemKNN on the GPU -- drop-in for recpack.algorithms.ItemKNN.

With ``recpack`` importable this class subclasses the reference's own ``ItemKNN``
(recpack/algorithms/nearest_neighbour.py:114-224): constructor validation, warnings and attributes are inherited,
``_fit`` calls rpk_fit_topk instead of sklearn / scipy / numpy, ``_predict`` is the GPU scorer of
``GpuSimilarityMixin``."""
from __future__ import annotations

from typing import Optional

import numpy as np
from scipy.sparse import csr_matrix

from . import _ref
from .base import GpuSimilarityMixin, lists_to_csr
from .engine import get_engine
from .matrix import device_structure, to_host

if _ref.HAVE_RECPACK:
    _ItemKNNBase = _ref.ref_nn.ItemKNN
else:
    from ._mirror import ItemKNNArgs as _ItemKNNBase


class ItemKNN(GpuSimilarityMixin, _ItemKNNBase):
    """Item K Nearest Neighbours (Deshpande & Karypis 2004), cosine or conditional-probability
    similarity, K most similar items per item.  See the reference docstring
    (nearest_neighbour.py:114-167) for the model; arguments are identical.

    :param predict_topK: optional, keep only this many scores per user in ``predict``.
    :param remove_history: optional, drop history items inside ``predict``.
    """

    def __init__(
        self,
        K=200,
        similarity: str = "cosine",
        pop_discount: Optional[float] = None,
        normalize_X: bool = False,
        normalize_sim: bool = False,
        predict_topK: Optional[int] = None,
        remove_history: bool = False,
    ):
        super().__init__(K=K, similarity=similarity, pop_discount=pop_discount, normalize_X=normalize_X,
                         normalize_sim=normalize_sim)
        self.predict_topK = predict_topK
        self.remove_history = remove_history

    def _fit(self, X: csr_matrix) -> None:
        engine = get_engine()
        X, indptr, indices, ptr_d, idx_d = device_structure(X, engine.device)
        U, I = X.shape
        item_pow = None
        if self.similarity == "conditional_probability" and self.pop_discount:
            # A.power(pop_discount) of the reference (nearest_neighbour.py:58), same numpy call
            n = np.bincount(indices, minlength=I)
            item_pow = np.zeros(I, dtype=np.float64)
            nz = n > 0
            item_pow[nz] = np.power(1 / n[nz], self.pop_discount)
        K = int(self.K)
        # the rank-ordered lists stay on the device (torch tensors owned by this estimator); similarity_matrix_
        # is built from them on first use
        if self.normalize_X:
            # Normalizer(norm="l1") on the binary rows (nearest_neighbour.py:207-210): every entry of user u becomes
            # fl(1 / d_u); the real-valued Gram kernel sums in the reference's order (rpk_fit_topk_real)
            import torch

            d = ptr_d[1:] - ptr_d[:-1]
            values = torch.repeat_interleave(1.0 / d.to(torch.float64), d)
            torch.cuda.current_stream(values.device).synchronize()  # the library runs on its own stream
            out = engine.fit_topk_real(U, I, ptr_d, idx_d, values, K, similarity=self.similarity, item_pow=item_pow)
            out["cnt"] = None
        else:
            out = engine.fit_topk(U, I, ptr_d, idx_d, K, similarity=self.similarity, item_pow=item_pow, want_cnt=False)
        if self.normalize_sim:
            # Normalizer(norm="l1") over the kept entries of each row (nearest_neighbour.py:220-222), on the host
            idx, val, ln = to_host(out["idx"], out["val"], out["len"])
            mask = np.arange(idx.shape[1])[None, :] < ln[:, None]
            row_sum = np.where(mask, np.abs(val), 0.0).sum(axis=1)
            row_sum[row_sum == 0] = 1.0
            self.similarity_matrix_ = lists_to_csr(idx, np.ascontiguousarray(val / row_sum[:, None]), ln, I)
        else:
            self._set_device_fit(out, I, engine.device)


def pearson_centred(X: csr_matrix) -> csr_matrix:
    """The matrix compute_pearson_similarity hands to the cosine (nearest_neighbour.py:100-108): every positive entry
    minus the mean of its item's positive entries; entries that become zero are not stored."""
    if not isinstance(X, csr_matrix):
        raise TypeError("expected a scipy csr_matrix")
    X = X.astype(np.float64).tocsr()
    X.sum_duplicates()
    X.eliminate_zeros()
    if (X.data == 1).sum() == X.nnz:
        raise ValueError("Pearson similarity can not be computed on a binary matrix.")
    I = X.shape[1]
    pos = X.data > 0
    count = np.bincount(X.indices[pos], minlength=I)
    avg = np.bincount(X.indices, weights=X.data, minlength=I).astype(np.float64)
    nz = count > 0
    avg[nz] = avg[nz] / count[nz]
    data = X.data.copy()
    data[pos] = data[pos] - avg[X.indices[pos]]
    C = csr_matrix((data, X.indices.copy(), X.indptr.copy()), shape=X.shape)
    C.eliminate_zeros()  # the sparse subtraction of the reference stores no zero results
    return C


def real_top_k(X: csr_matrix, K: int, similarity: str = "cosine") -> csr_matrix:
    """``get_top_K_values(compute_<similarity>(X), K)`` for a real-valued CSR X on the GPU (rpk_fit_topk_real);
    similarity in {"cosine", "conditional_probability", "pearson"}."""
    if similarity == "pearson":
        X, similarity = pearson_centred(X), "cosine"
    else:
        X = csr_matrix(X).astype(np.float64)
        X.sum_duplicates()
        X.eliminate_zeros()
    U, I = X.shape
    out = get_engine().fit_topk_real(U, I, np.ascontiguousarray(X.indptr, dtype=np.int64),
                                     np.ascontiguousarray(X.indices, dtype=np.int32),
                                     np.ascontiguousarray(X.data, dtype=np.float64), int(K), similarity=similarity)
    return lists_to_csr(out["idx"], out["val"], out["len"], I)


def pearson_top_k(X: csr_matrix, K: int) -> csr_matrix:
    """``get_top_K_values(compute_pearson_similarity(X), K)`` (nearest_neighbour.py:87-111, util.py:80-96) without the
    item x item matrix: ratings are centred per item over the positive entries, the cosine Gram of the centred matrix and
    the per-row selection run on the GPU (rpk_fit_topk_real).  Similarities can be negative: set as the
    ``similarity_matrix_`` of an ``ItemSimilarityMatrixAlgorithm`` the result is scored in float64 (scipy's ``X @ S``
    bit for bit), and the TARSItemKNN family scores it through rpk_spgemm_*."""
    return real_top_k(X, K, "pearson")
