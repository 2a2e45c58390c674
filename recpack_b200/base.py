"""Item-similarity algorithm bases whose scoring runs on the GPU.

With ``recpack`` importable the classes here subclass the reference's own
``recpack.algorithms.base.ItemSimilarityMatrixAlgorithm`` / ``TopKItemSimilarityMatrixAlgorithm``
(base.py:220-304): ``fit`` / ``predict`` wrappers, ``name``, ``identifier`` and the constructor are inherited,
and only what computes is replaced -- ``_predict`` (rpk_predict_*), the input coercion (structure only,
memoised per matrix) and the two O(nnz) Python-set checks (same warnings, computed from row pointers).
Without ``recpack`` a small mirror of those wrappers stands in (``_mirror.py``).  There is no CPU path."""
from __future__ import annotations

import warnings

import numpy as np
from scipy.sparse import csr_matrix
from sklearn.utils.validation import check_is_fitted

from . import _ref
from .engine import get_engine
from .matrix import binary_structure, device_structure, to_csr_matrix, to_host

if _ref.HAVE_RECPACK:
    Algorithm = _ref.ref_base.Algorithm
    _SimilarityBase = _ref.ref_base.ItemSimilarityMatrixAlgorithm
    _TopKBase = _ref.ref_base.TopKItemSimilarityMatrixAlgorithm
else:
    from . import _mirror

    Algorithm = _mirror.Algorithm
    _SimilarityBase = _mirror.ItemSimilarityMatrixAlgorithm
    _TopKBase = _mirror.TopKItemSimilarityMatrixAlgorithm


class GpuPredictMixin:
    """What every GPU ``_predict`` of this package adds to the reference's contract: ``predict_topK``,
    ``remove_history`` and ``set_postfilters`` (below), the predict input coercion (structure only, memoised per
    matrix) and the reference's "failed to recommend" check computed from row pointers."""

    predict_topK = None
    remove_history = False
    _postfilters = ()

    def set_postfilters(self, filters):
        """Post-filters (``recpack_b200.postprocessing.ExcludeItems`` / ``SelectItems``) applied inside predict,
        before the truncation to ``predict_topK``: the filtered items are never recommended and the lists are
        refilled from the items that remain (postprocessing/filters.py:58-101 on an untruncated matrix)."""
        self._postfilters = tuple(filters or ())
        return self

    def _transform_predict_input(self, X):
        return to_csr_matrix(X, binary=True)

    def _check_prediction(self, X_pred: csr_matrix, X: csr_matrix) -> None:
        """Warn when a user with history got no recommendation (base.py:108-127)."""
        has_hist = np.diff(X.indptr) > 0
        has_pred = np.diff(X_pred.indptr) > 0
        if X_pred.nnz and not np.all(X_pred.data):  # explicit zeros do not count as recommendations
            has_pred = np.asarray((X_pred != 0).sum(axis=1)).ravel() > 0
        missing = int(np.count_nonzero(has_hist & ~has_pred))
        if missing > 0:
            warnings.warn(f"{self.name} failed to recommend any items for {missing} users")


class GpuSimilarityMixin(GpuPredictMixin):
    """GPU implementation of the ``ItemSimilarityMatrixAlgorithm`` contract (base.py:220-279): predict =
    X @ similarity_matrix_.

    Two additions follow the reference's own precedent ``predict_topK`` ("Use when the user x item
    output matrix would become too large for RAM", base.py:427-430):

    * ``predict_topK``: keep only the N best scores per user (score desc, item index asc);
    * ``remove_history``: drop the user's own history items inside predict -- before the truncation,
      which is where the pipeline removes them (pipelines/pipeline.py:174-175).

    With both unset ``predict`` returns every non-zero score like the reference.  Scores are exact sums
    of the similarities in fixed point relative to the largest similarity of the model
    (``q = rint(v * 2^e)`` with ``2^e * vmax`` in ``[2^39, 2^40)``, see DESIGN.md 2): they agree with the
    reference's float64 sums to ``d_u * vmax * 2^-40`` and do not depend on summation order.

    A model with at least one negative value (Pearson neighbours, embedding cosines, any signed weights) is scored
    in float64 instead: ``predict`` is then scipy's ``X @ similarity_matrix_`` bit for bit (each score the left fold
    over the user's history items in ascending order; sums of exactly 0.0 are not stored), and ``predict_topK``
    keeps the N largest stored scores, negative ones included when fewer than N positive ones exist (DESIGN.md 2).
    Similarity values must be finite."""

    def truncated(self, K: int):
        """The same model cut to the K (<= self.K) best neighbours per item, without fitting again: the fitted lists
        are in rank order, so the first K places ARE the fit at K -- a sweep over K fits once at the largest value
        (recpack/algorithms/nearest_neighbour.py:360-397 refits for every K)."""
        from sklearn.base import clone

        dev = self.__dict__.get("_fit_dev")
        if dev is None:
            raise ValueError("truncated() needs the rank-ordered lists of a GPU fit (fit on this object first)")
        K = int(K)
        if not 1 <= K <= dev["idx"].shape[1]:
            raise ValueError(f"K must be in [1, {dev['idx'].shape[1]}]")
        other = clone(self)
        other.set_params(K=K)
        out = {"idx": dev["idx"][:, :K].contiguous(), "val": dev["val"][:, :K].contiguous(), "len": dev["len"].clamp(max=K)}
        other._set_device_fit(out, dev["I"], dev["device"])
        other._postfilters = self._postfilters
        return other

    # -- similarity_matrix_: host CSR, materialised on first use when the fit result lives on the device ----
    @property
    def similarity_matrix_(self):
        d = self.__dict__
        S = d.get("_similarity_host")
        if S is None:
            if d.get("_fit_dev") is None:
                raise AttributeError(f"{type(self).__name__} object has no attribute 'similarity_matrix_'")
            S = self._materialize_similarity()
        return S

    @similarity_matrix_.setter
    def similarity_matrix_(self, S):
        d = self.__dict__
        d["_similarity_host"] = S
        d["_fit_dev"] = None  # an assigned matrix replaces the device-resident fit result
        d["_model_version"] = d.get("_model_version", 0) + 1

    def _materialize_similarity(self):
        dev = self.__dict__["_fit_dev"]
        idx, val, ln = to_host(dev["idx"], dev["val"], dev["len"])
        S = lists_to_csr(idx, val, ln, dev["I"])
        self.__dict__["_similarity_host"] = S
        return S

    def _set_device_fit(self, out, I, device):
        """Keep the rank-ordered top-K lists of a fit on the device (torch tensors owned by this object)."""
        d = self.__dict__
        get_engine(device).sync()  # the lists are complete before torch touches them (streams may differ)
        d["_similarity_host"] = None
        d["_model_version"] = d.get("_model_version", 0) + 1
        d["_fit_dev"] = {"idx": out["idx"], "val": out["val"], "len": out["len"], "I": int(I), "device": int(device),
                         "empty_rows": int((out["len"] == 0).sum().item())}

    def __sklearn_is_fitted__(self):
        d = self.__dict__
        return d.get("_similarity_host") is not None or d.get("_fit_dev") is not None

    def __getstate__(self):
        if self.__dict__.get("_fit_dev") is not None:
            self.similarity_matrix_  # pickles carry the host matrix, never device memory
        state = dict(super().__getstate__())
        state["_fit_dev"] = None
        return state

    # -- device model management ---------------------------------------------------------------
    def _ensure_device_model(self, engine):
        """Loads this estimator's similarity model into the engine unless it is the resident one.  The key is
        (estimator, version): the version is bumped whenever ``similarity_matrix_`` is assigned or a fit finishes;
        arrays edited in place afterwards need ``invalidate_device_model()``."""
        d = self.__dict__
        key = (id(self), d.get("_model_version", 0))
        with engine.model_lock:
            if engine._model_key == key:
                return
            engine._model_key = None  # a failed load leaves no model behind (the C side drops it too)
            dev = d.get("_fit_dev")
            if dev is not None and dev["device"] == engine.device:
                engine.model_load_topk(dev["I"], dev["idx"].shape[1], dev["idx"], dev["val"], dev["len"])
            else:
                S = canonical_csr(self.similarity_matrix_)
                # a model with a negative value is scored in float64 (X @ S bit for bit), any other in fixed point
                load = engine.model_load_signed_csr if S.nnz and np.any(S.data < 0) else engine.model_load_csr
                load(S.shape[0], np.ascontiguousarray(S.indptr, dtype=np.int64), np.ascontiguousarray(S.indices, dtype=np.int32),
                     np.ascontiguousarray(S.data, dtype=np.float64))
            engine._model_key = key
            engine._model_owner = self  # keeps id(self) unique while it is the resident model

    def invalidate_device_model(self):
        """Call after editing ``similarity_matrix_`` in place: the next predict uploads it again."""
        self.__dict__["_model_version"] = self.__dict__.get("_model_version", 0) + 1

    def _n_items(self):
        dev = self.__dict__.get("_fit_dev")
        return dev["I"] if dev is not None else self.similarity_matrix_.shape[0]

    def _predict(self, X: csr_matrix) -> csr_matrix:
        engine = get_engine()
        I = self._n_items()
        if X.shape[1] != I:
            raise ValueError("matmul: dimension mismatch with signature (n?,k),(k,m?)->(n?,m?)")
        return predict_with_model(engine, self._ensure_device_model, X, I, self.predict_topK, self.remove_history,
                                  self._postfilters)

    # -- the reference's checks, without Python sets over nonzero() -------------------------------------
    def _transform_fit_input(self, X):
        return to_csr_matrix(X, binary=True)

    def _check_fit_complete(self):
        """check_is_fitted + "missing similar items" (base.py:257-279); the device-resident fit result answers
        from its row lengths without building the host matrix."""
        check_is_fitted(self)
        assert self.__sklearn_is_fitted__()
        dev = self.__dict__.get("_fit_dev")
        if dev is not None:
            missing = dev["empty_rows"]
        else:
            S = csr_matrix(self.similarity_matrix_)
            rows_with_score = np.diff(S.indptr) > 0
            if S.nnz and not np.all(S.data):
                rows_with_score = np.asarray((S != 0).sum(axis=1)).ravel() > 0
            missing = int(S.shape[0] - np.count_nonzero(rows_with_score))
        if missing > 0:
            warnings.warn(f"{self.name} missing similar items for {missing} items.")


class ItemSimilarityMatrixAlgorithm(GpuSimilarityMixin, _SimilarityBase):
    """recpack/algorithms/base.py:220-279 with ``_predict`` on the GPU: any algorithm that sets a sparse
    ``similarity_matrix_`` in ``_fit`` scores through rpk_predict_* -- in fixed point when it is non-negative, in
    float64 (scipy's ``X @ S`` bit for bit) when it has a negative value."""


class TopKItemSimilarityMatrixAlgorithm(GpuSimilarityMixin, _TopKBase):
    """recpack/algorithms/base.py:282-304."""


def canonical_csr(S) -> csr_matrix:
    """S as a CSR with sorted, unique column indices and no stored zeros (copied only when it is not one already)."""
    if not isinstance(S, csr_matrix):
        S = csr_matrix(S)
    if not S.has_canonical_format:
        S = S.copy()
        S.sum_duplicates()
    if S.nnz and not np.all(S.data):
        S = S.copy()
        S.eliminate_zeros()
    return S


def predict_with_model(engine, ensure_model, X: csr_matrix, I: int, predict_topK, remove_history, postfilters=()) -> csr_matrix:
    """Scores X with the model that ``ensure_model(engine)`` makes resident: the full CSR of the scores when
    ``predict_topK`` is None, else the top-N lists as a CSR that carries them (host and device) for the metrics."""
    from .postprocessing import combined_mask

    U = X.shape[0]
    with engine.model_lock:  # load + score as one step: the engine holds one model at a time
        ensure_model(engine)
        engine.predict_item_filter(combined_mask(postfilters, I))
        if predict_topK is None:
            X, indptr, indices = binary_structure(X)
            o_ptr, o_idx, o_val = engine.predict_csr(U, indptr, indices, mask_history=bool(remove_history))
            return csr_matrix((o_val, o_idx, o_ptr), shape=(U, I))
        N = int(predict_topK)
        X, _, _, ptr_d, idx_d = device_structure(X, engine.device)
        top = engine.predict_topn(U, ptr_d, idx_d, N, mask_history=bool(remove_history))
        engine.sync()
    return topn_result(top, I, engine.device)


def topn_result(top, I: int, device: int) -> csr_matrix:
    """The CSR of device-resident top-N lists (dict(idx, val, len), rank order) that carries them for the metrics."""
    idx, val, ln = to_host(top["idx"], top["val"], top["len"])
    M = lists_to_csr(idx, val, ln, I, attach=True)
    # the metrics read the lists where they are, as long as the matrix still is what predict returned
    M._rpk_topn_dev = (top["idx"], top["len"], device)
    M._rpk_topn_sig = matrix_signature(M)
    return M


def matrix_signature(M: csr_matrix):
    """Cheap identity of a CSR's content as predict returned it (array addresses, nnz and a checksum of the
    values): an in-place edit of ``data`` / ``indices`` or a re-assignment changes it."""
    return (M.data.ctypes.data, M.indices.ctypes.data, M.indptr.ctypes.data, M.nnz, M.shape,
            float(M.data.sum()) if M.nnz else 0.0)


def lists_to_csr(idx, val, ln, n_cols, attach=False) -> csr_matrix:
    """[rows x K] rank-ordered lists (-1 padded) -> CSR whose rows keep the rank order.

    When every row is full the arrays are used as they are (no copy)."""
    rows, K = idx.shape
    ln = np.asarray(ln)
    if rows and int(ln.min()) == K:
        indptr = np.arange(rows + 1, dtype=np.int64) * K
        M = csr_matrix((val.reshape(-1), idx.reshape(-1), indptr), shape=(rows, n_cols))
    else:
        mask = np.arange(K, dtype=np.int32)[None, :] < ln[:, None]
        indptr = np.zeros(rows + 1, dtype=np.int64)
        np.cumsum(ln, out=indptr[1:])
        M = csr_matrix((val[mask], idx[mask], indptr), shape=(rows, n_cols))
    if attach:
        M._rpk_topn = (idx, ln)
    return M
