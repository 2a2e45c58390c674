"""Item neighbours of a dense embedding matrix: the ``similarity_matrix_`` of Prod2Vec-style models.

The reference's ``Prod2Vec`` / ``Prod2VecClustered`` build their model from the cosine similarities of the item
embeddings, cut per row with ``get_top_K_values`` (recpack/algorithms/p2v.py:213-242); users do the same with any
item-factor matrix (SVD, NMF, BPR, WMF, an external encoder).  ``embedding_top_k`` computes that model on the GPU
(rpk_embed_topk) without ever forming the I x I matrix: the tensor cores screen candidates, every kept value and every
order decision is made in float64 on the definition of DESIGN.md 2 ("Embedding neighbours").

Typical use::

    algo = ItemSimilarityMatrixAlgorithm()        # or any subclass whose fit is the embedding model
    algo.similarity_matrix_ = embedding_top_k(item_factors, K=200)
    algo.predict(X)                               # scored by the existing kernels, post-filters and metrics apply

A model with a negative value is scored in float64 (scipy's ``X @ S`` bit for bit), any other in fixed point.
"""
from __future__ import annotations

import numpy as np
from scipy.sparse import csr_matrix

from .base import lists_to_csr
from .engine import _is_torch, get_engine
from .matrix import to_host


def embedding_top_k(E, K: int, similarity: str = "cosine") -> csr_matrix:
    """Per item row of ``E`` [I x D], the ``K`` largest stored similarities to the other items as an [I x I] CSR.

    :param E: numpy array or torch tensor (host or CUDA), float32 or float64; float32 is widened to float64 (exact).
    :param K: neighbours per item, 1 <= K <= 1024.  Rows with fewer stored values (exact zeros are not stored) are shorter.
    :param similarity: ``"cosine"`` (rows L2-normalised first; a zero row stays zero) or ``"dot"``.
    :raises RpkError: NaN / inf in ``E``, or sizes outside 1 <= D <= 1024, I < 2^24.
    """
    if similarity not in ("cosine", "dot"):
        raise ValueError(f"similarity must be 'cosine' or 'dot', got {similarity!r}")
    if _is_torch(E):
        import torch

        if E.dtype not in (torch.float32, torch.float64):
            raise TypeError(f"E must be float32 or float64, got {E.dtype}")
        if E.dim() != 2:
            raise ValueError("E must be a 2-d matrix [items x dimensions]")
        E = E.to(torch.float64).contiguous()
        device = E.device.index if E.is_cuda else None
        if not E.is_cuda:
            E = E.numpy()
    else:
        E = np.asarray(E)
        if E.dtype not in (np.float32, np.float64):
            raise TypeError(f"E must be float32 or float64, got {E.dtype}")
        if E.ndim != 2:
            raise ValueError("E must be a 2-d matrix [items x dimensions]")
        E = np.ascontiguousarray(E, dtype=np.float64)
        device = None
    I = int(E.shape[0])
    out = get_engine(device).embed_topk(E, int(K), similarity)
    idx, val, ln = (out["idx"], out["val"], out["len"]) if device is None else to_host(out["idx"], out["val"], out["len"])
    return lists_to_csr(idx, val, ln, I)
