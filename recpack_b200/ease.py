"""EASE on the GPU -- drop-in for recpack.algorithms.EASE (recpack/algorithms/ease.py:19-109).

``_fit``: the dense Gram ``X^T X`` comes from the tensor-core kernel (exact integer counts, rpk_gram_dense_f64), the
inverse of ``X^T X + l2 I`` from cuSOLVER (Cholesky factorisation + inverse through ``torch.linalg``: the matrix is
symmetric positive definite), the closed form ``B = -P / diag(P)`` with zero diagonal and the optional popularity
scaling from rpk_ease_from_inverse.  The model stays on the device as a dense float64 matrix; ``similarity_matrix_``
(a scipy CSR like the reference's) is built on first access.

``_predict``: ``X @ B`` with the dense scorer (rpk_predict_dense_*): every score is the float64 sum over the user's
history in ascending item order -- the order of scipy's ``csr @ dense`` -- so equal models give bit-identical scores;
``predict_topK`` / ``remove_history`` as for ItemKNN.  A NaN in the model (``alpha != 0`` with an item nobody
interacted with) stays NaN in the full scores, as in the reference; top-N raises ``RpkError`` when a score it would
rank is NaN.

``density`` (``_prune``, ease.py:97-109): after the closed form the model is pruned on the device to its
``K = min(int(density * I*I), nnz)`` largest-magnitude entries (rpk_ease_prune; ``K = 0`` keeps every entry, as the
reference's ``argpartition(..., -0)[0:-0]`` does) and the dense model is dropped.  Ties at the cut go to the entries
first in row-major order.  The pruned model is scored like every signed similarity model, in float64 and bit for bit
scipy's ``X @ S`` (rpk_model_load_signed_csr); its values must be finite there.  The loaded model is keyed by
(estimator, version) like ``GpuSimilarityMixin``'s: after editing ``similarity_matrix_`` in place, call
``invalidate_device_model()``.  A negative ``density`` raises ``ValueError`` (the reference computes a negative K and
zeroes the |K| smallest entries instead, or fails in ``argpartition`` when |K| >= nnz).

The reference inverts with LAPACK's LU (``np.linalg.inv``); Cholesky on the GPU agrees with it to rounding
(~1e-12 relative on B), not bit for bit -- the tolerance of the tests."""
from __future__ import annotations

from typing import Optional

import numpy as np
from scipy.sparse import csr_matrix
from sklearn.utils.validation import check_is_fitted

from . import _ref
from .base import canonical_csr, lists_to_csr, matrix_signature, predict_with_model
from .engine import get_engine
from .matrix import binary_structure, device_structure, to_csr_matrix, to_host

if _ref.HAVE_RECPACK:
    import importlib

    _EaseBase = importlib.import_module(_ref.ref_base.__name__.rsplit(".", 1)[0] + ".ease").EASE
else:
    from ._mirror import ItemSimilarityMatrixAlgorithm as _MirrorBase

    class _EaseBase(_MirrorBase):
        def __init__(self, l2=1e3, alpha=0, density=None):
            super().__init__()
            self.l2 = l2
            self.alpha = alpha
            self.density = density


class EASE(_EaseBase):
    """Embarrassingly Shallow Autoencoder (Steck 2019); arguments as in the reference (ease.py:19-62).

    :param predict_topK: optional, keep only this many scores per user in ``predict``.
    :param remove_history: optional, drop history items inside ``predict``.
    """

    def __init__(self, l2=1e3, alpha=0, density=None, predict_topK: Optional[int] = None, remove_history: bool = False):
        super().__init__(l2=l2, alpha=alpha, density=density)
        self.predict_topK = predict_topK
        self.remove_history = remove_history

    # -- fit ------------------------------------------------------------------------------
    def _transform_fit_input(self, X):
        return to_csr_matrix(X, binary=True)

    def _transform_predict_input(self, X):
        return to_csr_matrix(X, binary=True)

    def _fit(self, X: csr_matrix) -> None:
        import torch

        if self.density and self.density < 0:
            raise ValueError("density must be non-negative")
        engine = get_engine()
        X, indptr, indices, ptr_d, idx_d = device_structure(X, engine.device)
        U, I = X.shape
        G = engine.gram_dense_f64(U, I, ptr_d, idx_d)  # exact counts as float64
        engine.sync()
        n = torch.diagonal(G).clone()  # item popularities = diag(X^T X)
        # l2 * np.identity(I, dtype=float32) promotes to float64 in the sum (ease.py:80)
        torch.diagonal(G).add_(float(np.float32(self.l2)))
        L = torch.linalg.cholesky(G)       # cuSOLVER potrf
        del G
        P = torch.cholesky_inverse(L).contiguous()  # cuSOLVER potri (the result comes back column-major)
        del L
        w = None
        if self.alpha != 0:
            w = 1.0 / n.cpu().numpy() ** self.alpha  # 1 / np.diag(XTX) ** alpha (ease.py:87), inf for unseen items as there
        torch.cuda.current_stream(P.device).synchronize()
        B = engine.ease_from_inverse(P, w)  # in place
        engine.sync()
        d = self.__dict__
        d["_similarity_host"] = None
        d["_model_version"] = d.get("_model_version", 0) + 1
        if self.density:
            S = engine.ease_prune(B, prune_keep(self.density, I))
            del B, P
            d["_B_dev"] = None
            d["_S_dev"] = S
        else:
            d["_B_dev"] = B
            d["_S_dev"] = None

    # -- similarity_matrix_: the dense model as the reference stores it, built on demand -------------------
    @property
    def similarity_matrix_(self):
        d = self.__dict__
        S = d.get("_similarity_host")
        if S is None:
            B, S_dev = d.get("_B_dev"), d.get("_S_dev")
            if B is not None:
                S = csr_matrix(B.cpu().numpy())
            elif S_dev is not None:
                I = int(S_dev[0].shape[0]) - 1
                S = csr_matrix(tuple(t.cpu().numpy() for t in S_dev[::-1]), shape=(I, I))
            else:
                raise AttributeError(f"{type(self).__name__} object has no attribute 'similarity_matrix_'")
            d["_similarity_host"] = S
        return S

    @similarity_matrix_.setter
    def similarity_matrix_(self, S):
        d = self.__dict__
        d["_similarity_host"] = S
        d["_B_dev"] = None
        d["_S_dev"] = None
        d["_model_version"] = d.get("_model_version", 0) + 1

    def __sklearn_is_fitted__(self):
        d = self.__dict__
        return any(d.get(k) is not None for k in ("_similarity_host", "_B_dev", "_S_dev"))

    def __getstate__(self):
        d = self.__dict__
        if d.get("_B_dev") is not None or d.get("_S_dev") is not None:
            self.similarity_matrix_  # pickles carry the host matrix, never device memory
        state = dict(super().__getstate__())
        state["_B_dev"] = None
        state["_S_dev"] = None
        return state

    def _check_fit_complete(self):
        import warnings

        import torch

        check_is_fitted(self)
        B, S_dev = self.__dict__.get("_B_dev"), self.__dict__.get("_S_dev")
        if B is not None:
            missing = int((B != 0).sum(dim=1).eq(0).sum().item())
        elif S_dev is not None:
            missing = int(torch.diff(S_dev[0]).eq(0).sum().item())
        else:
            S = csr_matrix(self.similarity_matrix_)
            missing = int(S.shape[0] - np.count_nonzero(np.asarray((S != 0).sum(axis=1)).ravel()))
        if missing > 0:
            warnings.warn(f"{self.name} missing similar items for {missing} items.")

    def _check_prediction(self, X_pred: csr_matrix, X: csr_matrix) -> None:
        import warnings

        has_hist = np.diff(X.indptr) > 0
        has_pred = np.asarray((X_pred != 0).sum(axis=1)).ravel() > 0 if X_pred.nnz and not np.all(X_pred.data) else np.diff(X_pred.indptr) > 0
        missing = int(np.count_nonzero(has_hist & ~has_pred))
        if missing > 0:
            warnings.warn(f"{self.name} failed to recommend any items for {missing} users")

    # -- predict --------------------------------------------------------------------------
    def _device_model(self, engine):
        import torch

        d = self.__dict__
        B = d.get("_B_dev")
        if B is None or B.device.index != engine.device:
            S = self.similarity_matrix_
            dense = np.ascontiguousarray(S.toarray() if hasattr(S, "toarray") else np.asarray(S), dtype=np.float64)
            B = torch.from_numpy(dense).to(torch.device("cuda", engine.device))
            torch.cuda.current_stream(B.device).synchronize()
            d["_B_dev"] = B
        return B

    def _ensure_sparse_model(self, engine):
        """Loads the pruned model as a signed model (float64 scoring) unless it is the engine's resident one; the key
        (estimator, version) is that of ``GpuSimilarityMixin._ensure_device_model``."""
        d = self.__dict__
        key = (id(self), d.get("_model_version", 0))
        with engine.model_lock:
            if engine._model_key == key:
                return
            engine._model_key = None  # a failed load leaves no model behind
            S_dev = d.get("_S_dev")
            if S_dev is not None and S_dev[0].device.index == engine.device:
                ptr, idx, val = S_dev
            else:
                S = canonical_csr(self.similarity_matrix_)
                ptr, idx, val = (np.ascontiguousarray(S.indptr, dtype=np.int64), np.ascontiguousarray(S.indices, dtype=np.int32),
                                 np.ascontiguousarray(S.data, dtype=np.float64))
            engine.model_load_signed_csr(int(ptr.shape[0]) - 1, ptr, idx, val)
            engine._model_key = key
            engine._model_owner = self

    def invalidate_device_model(self):
        """Call after editing ``similarity_matrix_`` in place: the next predict takes the model from the host matrix
        again instead of the device copy that the fit (or an earlier predict) left behind."""
        d = self.__dict__
        if d.get("_similarity_host") is not None:
            d["_S_dev"] = None
            d["_B_dev"] = None
        d["_model_version"] = d.get("_model_version", 0) + 1

    def _n_items(self):
        d = self.__dict__
        if d.get("_S_dev") is not None:
            return int(d["_S_dev"][0].shape[0]) - 1
        if d.get("_B_dev") is not None:
            return int(d["_B_dev"].shape[0])
        return self.similarity_matrix_.shape[0]

    def _predict(self, X: csr_matrix) -> csr_matrix:
        engine = get_engine()
        if self.density:  # a pruned model: float64 sparse scoring, the route of every signed similarity model
            I = self._n_items()
            if X.shape[1] != I:
                raise ValueError("matmul: dimension mismatch with signature (n?,k),(k,m?)->(n?,m?)")
            return predict_with_model(engine, self._ensure_sparse_model, X, I, self.predict_topK, self.remove_history)
        B = self._device_model(engine)
        I = int(B.shape[0])
        if X.shape[1] != I:
            raise ValueError("matmul: dimension mismatch with signature (n?,k),(k,m?)->(n?,m?)")
        U = X.shape[0]
        X, _, _, ptr_d, idx_d = device_structure(X, engine.device)
        if self.predict_topK is None:
            scores = engine.predict_dense_full(U, ptr_d, idx_d, B, mask_history=bool(self.remove_history))
            engine.sync()
            return csr_matrix(scores.cpu().numpy())
        N = int(self.predict_topK)
        top = engine.predict_dense_topn(U, ptr_d, idx_d, B, N, mask_history=bool(self.remove_history))
        engine.sync()
        idx, val, ln = to_host(top["idx"], top["val"], top["len"])
        M = lists_to_csr(idx, val, ln, I, attach=True)
        M._rpk_topn_dev = (top["idx"], top["len"], engine.device)
        M._rpk_topn_sig = matrix_signature(M)
        return M


def prune_keep(density, I: int) -> int:
    """How many entries ``_prune`` keeps of an I x I model, before the cap at its nnz: ``int(density * (I*I))`` as one
    float64 product of the exact integer I*I (ease.py:105); 0 there means every entry stays (``argpartition(a, -0)[0:-0]``
    is empty), so I*I is returned instead."""
    K = int(float(density) * (int(I) * int(I)))
    return K if K > 0 else int(I) * int(I)
