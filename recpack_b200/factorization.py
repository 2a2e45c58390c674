"""Factorization models on the GPU -- RecPack's ``FactorizationAlgorithm`` (recpack/algorithms/base.py:307-369) and
drop-ins for every class of ``recpack.algorithms`` that subclasses it (``SVD`` and ``NMF``, algorithms/factorization.py).

The reference predicts ``user_embedding_[users] @ item_embedding_.T`` for the users with history into a
``lil_matrix`` -- a dense users x items product (77 GB at ML-25M shape) built on the host.  Here ``_predict`` runs on
the GPU (rpk_factor_*, DESIGN.md 2 "Factor models" and 4.10): every score is the float64 left fold over d of
``fl(p_ud * q_jd)``; scores of exactly 0.0 are not stored, as ``lil_matrix`` drops them; users without history get an
empty row.  With ``predict_topK`` the N best stored scores per user (score desc, item asc) come back as lists that the
metrics read in place -- the product is screened on the tensor cores and never materialised; ``remove_history`` and
``set_postfilters`` apply inside predict as for the similarity models.  ``predict_topK`` is limited to 1,024.

Relation to the reference: BLAS sums in an unspecified order (and in float32 for float32 factors), so values agree
to a few ulp * D of ``||p_u|| ||q_j||`` and lists agree except inside groups of scores within that distance.

The factors are uploaded once per model version: assigning ``user_embedding_`` / ``item_embedding_`` bumps it; after
editing them in place call ``invalidate_device_model()``.  ``_fit`` is the reference's own (sklearn); the drop-ins exist
only when ``recpack`` is importable."""
from __future__ import annotations

import inspect

import numpy as np
from scipy.sparse import csr_matrix, vstack

from . import _ref
from .base import GpuPredictMixin, topn_result
from .engine import get_engine
from .matrix import device_structure

if _ref.HAVE_RECPACK:
    _FactorBase = _ref.ref_base.FactorizationAlgorithm
else:
    from ._mirror import FactorizationAlgorithm as _FactorBase

__all__ = ["FactorizationAlgorithm"]

MAX_TOPK = 1024
_FULL_BLOCK_BYTES = 1 << 30  # full predict: users per block so that one block of float64 scores stays below this


def _factor(name):
    """A fitted factor matrix, stored in the instance dict under its own name (sklearn's ``check_is_fitted`` and
    pickling see it as a plain attribute); assigning it drops the device copy."""

    def get(self):
        try:
            return self.__dict__[name]
        except KeyError:
            raise AttributeError(f"{type(self).__name__} object has no attribute {name!r}") from None

    def set_(self, value):
        d = self.__dict__
        d[name] = value
        d["_factors_dev"] = None
        d["_model_version"] = d.get("_model_version", 0) + 1

    return property(get, set_)


class GpuFactorizationMixin(GpuPredictMixin):
    """``_predict`` of ``FactorizationAlgorithm`` on the GPU (see the module docstring)."""

    user_embedding_ = _factor("user_embedding_")
    item_embedding_ = _factor("item_embedding_")

    def invalidate_device_model(self):
        """Call after editing the factors in place: the next predict uploads them again."""
        d = self.__dict__
        d["_factors_dev"] = None
        d["_model_version"] = d.get("_model_version", 0) + 1

    def __getstate__(self):
        state = dict(super().__getstate__())
        state["_factors_dev"] = None  # pickles carry the host factors, never device memory
        return state

    def _device_factors(self, engine):
        import torch

        d = self.__dict__
        key = (d.get("_model_version", 0), engine.device)
        dev = d.get("_factors_dev")
        if dev is None or dev[0] != key:
            where = torch.device("cuda", engine.device)
            P, Q = (torch.as_tensor(np.asarray(F) if not torch.is_tensor(F) else F).to(device=where, dtype=torch.float64)
                    .contiguous() for F in (self.user_embedding_, self.item_embedding_))
            if P.dim() != 2 or Q.dim() != 2 or P.shape[1] != Q.shape[1]:
                raise ValueError(f"factors of shapes {tuple(P.shape)} and {tuple(Q.shape)} do not form a product")
            torch.cuda.current_stream(where).synchronize()
            dev = d["_factors_dev"] = (key, P, Q)
        return dev[1], dev[2]

    def _predict(self, X: csr_matrix) -> csr_matrix:
        from .postprocessing import combined_mask

        engine = get_engine()
        P, Q = self._device_factors(engine)
        U, I = int(P.shape[0]), int(Q.shape[0])
        if X.shape != (U, I):  # the reference's assert (base.py:307-369)
            raise AssertionError(f"X has shape {X.shape}, the factors give ({U}, {I})")
        if self.predict_topK is not None and not 1 <= int(self.predict_topK) <= MAX_TOPK:
            raise ValueError(f"predict_topK must be in [1, {MAX_TOPK}] for factorization models, got {self.predict_topK}")
        X, _, _, ptr_d, idx_d = device_structure(X, engine.device)
        mask_history = bool(self.remove_history)
        with engine.model_lock:  # the item filter is state of the engine
            engine.predict_item_filter(combined_mask(self._postfilters, I))
            if self.predict_topK is None:
                return self._predict_full(engine, P, Q, X, ptr_d, idx_d, mask_history)
            top = engine.factor_topn(P, Q, ptr_d, idx_d, int(self.predict_topK), mask_history=mask_history)
            engine.sync()
        return topn_result(top, I, engine.device)

    @staticmethod
    def _predict_full(engine, P, Q, X, ptr_d, idx_d, mask_history):
        """Every stored score as a CSR, in blocks of users (rpk_factor_full)."""
        U, I = X.shape
        rows = max(1, _FULL_BLOCK_BYTES // (8 * I))
        blocks = []
        for a in range(0, U, rows):
            b = min(U, a + rows)
            lo, hi = int(X.indptr[a]), int(X.indptr[b])
            S = engine.factor_full(P[a:b], Q, (ptr_d[a : b + 1] - lo).contiguous(), idx_d[lo:hi], mask_history=mask_history)
            engine.sync()
            blocks.append(csr_matrix(S.cpu().numpy()))  # drops the 0.0 scores, as lil_matrix does
        return vstack(blocks, format="csr") if len(blocks) > 1 else (blocks[0] if blocks else csr_matrix((U, I)))


class FactorizationAlgorithm(GpuFactorizationMixin, _FactorBase):
    """recpack/algorithms/base.py:307-369 with ``_predict`` on the GPU.  Assign ``user_embedding_`` ([U, D], one row
    per row of the X passed to predict) and ``item_embedding_`` ([I, D]) in ``_fit``, or on a fitted object.

    :param num_components: the dimension of the factors (the reference's argument).
    :param predict_topK: optional, keep only this many scores per user in ``predict`` (at most 1,024).
    :param remove_history: optional, drop history items inside ``predict``.
    """

    def __init__(self, num_components=100, predict_topK=None, remove_history=False):
        super().__init__(num_components=num_components)
        self.predict_topK = predict_topK
        self.remove_history = remove_history


if _ref.HAVE_RECPACK:
    import importlib

    _algorithms = importlib.import_module(_ref.ref_base.__name__.rsplit(".", 1)[0])
    for _name, _cls in sorted(vars(_algorithms).items()):
        if inspect.isclass(_cls) and issubclass(_cls, _FactorBase) and _cls is not _FactorBase:
            globals()[_name] = type(_name, (GpuFactorizationMixin, _cls),
                                    {"__doc__": f"GPU drop-in for recpack's {_name}: the reference's fit, the predict of "
                                                "recpack_b200.factorization (see its docstring).",
                                     "__module__": __name__})
            __all__.append(_name)
