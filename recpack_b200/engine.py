"""Thin Python driver over the C ABI: one Engine = one rpk context on one GPU.

Arrays may be numpy arrays (host: the library copies them in / out inside the call) or torch
CUDA tensors (device: passed by address, nothing is copied, the call is stream-ordered)."""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _lib
from ._lib import RpkError

SIM_CODES = {"cosine": 0, "conditional_probability": 1}
EMBED_SIM_CODES = {"cosine": 0, "dot": 2}
METRIC_CODES = {"ndcg": 0, "recall": 1, "dcg": 2, "calibrated_recall": 3, "precision": 4, "reciprocal_rank": 5, "hits": 6}

DBG_WIDE_ACC, DBG_TINY_LIST, DBG_MULTI_PASS, DBG_SPLIT_ROWS, DBG_EXACT_SCORES, DBG_MANY_PASS = 1, 2, 4, 8, 16, 32


def _is_torch(x):
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda")


def _addr(x, dtype=None, allow_none=False):
    """Address of a C-contiguous numpy array or torch tensor (None -> NULL)."""
    if x is None:
        if allow_none:
            return None
        raise ValueError("array argument must not be None")
    if _is_torch(x):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        if dtype is not None and str(x.dtype).replace("torch.", "") != np.dtype(dtype).name:
            raise TypeError(f"tensor dtype {x.dtype}, expected {np.dtype(dtype).name}")
        return x.data_ptr()
    if not isinstance(x, np.ndarray):
        raise TypeError(f"expected numpy array or torch tensor, got {type(x).__name__}")
    if dtype is not None and x.dtype != np.dtype(dtype):
        raise TypeError(f"array dtype {x.dtype}, expected {np.dtype(dtype).name}")
    if not x.flags.c_contiguous:
        raise ValueError("array must be C-contiguous")
    return x.ctypes.data


def _empty_like_kind(ref, shape, dtype):
    """Allocate an output next to the inputs: torch CUDA tensor if ref is one, else numpy."""
    if _is_torch(ref):
        import torch

        return torch.empty(shape, dtype=getattr(torch, np.dtype(dtype).name), device=ref.device)
    return np.empty(shape, dtype=dtype)


class Engine:
    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        if self._lib.rpk_create(int(device), C.byref(h)) != 0:
            raise RpkError("rpk_create failed: " + self._lib.rpk_last_error(None).decode())
        self._h = h
        self.device = int(device)
        import secrets

        self.nonce = secrets.randbits(62)  # identifies this context in (picklable) fit tokens
        self.model_lock = threading.RLock()  # the context holds ONE similarity model: load + score under this lock
        self._model_key = None
        self._model_owner = None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rpk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RpkError(self._lib.rpk_last_error(self._h).decode())

    # -- plumbing -------------------------------------------------------------------------
    def set_stream(self, stream_ptr):
        self._check(self._lib.rpk_set_stream(self._h, C.c_void_p(stream_ptr or 0)))

    def use_torch_stream(self):
        import torch

        self.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def sync(self):
        self._check(self._lib.rpk_sync(self._h))

    def trace(self, on: bool = True):
        """rpk_trace: record named marks at the phase boundaries of every later call."""
        self._check(self._lib.rpk_trace(self._h, int(bool(on))))

    def trace_report(self) -> str:
        """rpk_trace_report: 'name  ms since the previous mark' lines of the marks since the last report."""
        return self._lib.rpk_trace_report(self._h).decode()

    def launch_count(self) -> int:
        return int(self._lib.rpk_launch_count(self._h))

    def debug_flags(self, flags: int):
        self._check(self._lib.rpk_debug_flags(self._h, int(flags)))

    # -- fit ------------------------------------------------------------------------------
    def fit_topk(self, U, I, indptr, indices, K, similarity="cosine", item_pow=None, item_begin=0, item_end=None,
                 want_cnt=True, want_val=True, out=None):
        """rpk_fit_topk (binary X).  Returns dict(idx, cnt, val, len); rows in rank order."""
        item_end = I if item_end is None else item_end
        rows = item_end - item_begin
        nnz = int(indices.shape[0])
        if out is None:
            out = {
                "idx": _empty_like_kind(indices, (rows, K), np.int32),
                "cnt": _empty_like_kind(indices, (rows, K), np.int32) if want_cnt else None,
                "val": _empty_like_kind(indices, (rows, K), np.float64) if want_val else None,
                "len": _empty_like_kind(indices, (rows,), np.int32),
            }
        self._check(self._lib.rpk_fit_topk(
            self._h, U, I, nnz, _addr(indptr, np.int64), _addr(indices, np.int32), SIM_CODES[similarity],
            _addr(item_pow, np.float64, allow_none=True), int(K), int(item_begin), int(item_end),
            _addr(out["idx"], np.int32), _addr(out.get("cnt"), np.int32, allow_none=True),
            _addr(out.get("val"), np.float64, allow_none=True), _addr(out["len"], np.int32)))
        return out

    def fit_topk_real(self, U, I, indptr, indices, values, K, similarity="cosine", item_pow=None, item_begin=0,
                      item_end=None, out=None):
        """rpk_fit_topk_real (real-valued X: one float64 per stored entry).  Returns dict(idx, val, len)."""
        item_end = I if item_end is None else item_end
        rows = item_end - item_begin
        nnz = int(indices.shape[0])
        if out is None:
            out = {
                "idx": _empty_like_kind(indices, (rows, K), np.int32),
                "val": _empty_like_kind(indices, (rows, K), np.float64),
                "len": _empty_like_kind(indices, (rows,), np.int32),
            }
        self._check(self._lib.rpk_fit_topk_real(
            self._h, U, I, nnz, _addr(indptr, np.int64), _addr(indices, np.int32), _addr(values, np.float64),
            SIM_CODES[similarity], _addr(item_pow, np.float64, allow_none=True), int(K), int(item_begin), int(item_end),
            _addr(out["idx"], np.int32), _addr(out["val"], np.float64), _addr(out["len"], np.int32)))
        return out

    def fit_item_counts(self, I, like=None):
        out = _empty_like_kind(like, (I,), np.int32)
        self._check(self._lib.rpk_fit_item_counts(self._h, _addr(out, np.int32), int(I)))
        return out

    def last_timings(self):
        """dict(gram_tc_ms, fit_rows_ms, predict_ms): device time of the dominant kernels of the last calls."""
        out = np.zeros(5, dtype=np.float64)
        self._check(self._lib.rpk_last_timings(self._h, _addr(out)))
        return {"gram_tc_ms": float(out[0]), "fit_rows_ms": float(out[1]), "predict_ms": float(out[2]),
                "dense_users": int(out[3]), "dense_kd": int(out[4])}

    def fit_config(self, dense_users: int = -1):
        self._check(self._lib.rpk_fit_config(self._h, int(dense_users)))

    # -- real-valued scoring: C = A @ S in float64, scipy's summation order ------------------------------
    @staticmethod
    def _csr_args(M):
        return (np.ascontiguousarray(M.indptr, dtype=np.int64), np.ascontiguousarray(M.indices, dtype=np.int32),
                np.ascontiguousarray(M.data, dtype=np.float64))

    def spgemm_topn(self, A, S, N, mask_history=False):
        """rpk_spgemm_topn for scipy CSR A [rows x I] and S [I x I] (sorted indices).  Returns dict(idx, val, len)."""
        rows, I = A.shape
        ap, ai, av = self._csr_args(A)
        sp_, si, sv = self._csr_args(S)
        out = {"idx": np.empty((rows, N), dtype=np.int32), "val": np.empty((rows, N), dtype=np.float64),
               "len": np.empty((rows,), dtype=np.int32)}
        self._check(self._lib.rpk_spgemm_topn(self._h, int(rows), int(ai.shape[0]), _addr(ap), _addr(ai), _addr(av), int(I),
                                              int(si.shape[0]), _addr(sp_), _addr(si), _addr(sv), int(N), int(bool(mask_history)),
                                              _addr(out["idx"]), _addr(out["val"]), _addr(out["len"])))
        return out

    def spgemm_csr(self, A, S, mask_history=False):
        """A @ S as (indptr int64, indices int32, values float64), ascending columns (rpk_spgemm_count + _fill)."""
        rows, I = A.shape
        ap, ai, av = self._csr_args(A)
        sp_, si, sv = self._csr_args(S)
        cnt = np.zeros(rows, dtype=np.int64)
        self._check(self._lib.rpk_spgemm_count(self._h, int(rows), int(ai.shape[0]), _addr(ap), _addr(ai), _addr(av), int(I),
                                               int(si.shape[0]), _addr(sp_), _addr(si), _addr(sv), int(bool(mask_history)),
                                               _addr(cnt)))
        indptr = np.zeros(rows + 1, dtype=np.int64)
        np.cumsum(cnt, out=indptr[1:])
        nnz = int(indptr[-1])
        indices = np.empty(nnz, dtype=np.int32)
        values = np.empty(nnz, dtype=np.float64)
        self._check(self._lib.rpk_spgemm_fill(self._h, int(rows), int(ai.shape[0]), _addr(ap), _addr(ai), _addr(av), int(I),
                                              int(si.shape[0]), _addr(sp_), _addr(si), _addr(sv), int(bool(mask_history)),
                                              _addr(indptr), nnz, _addr(indices), _addr(values)))
        return indptr, indices, values

    def split_fraction(self, uids, seg, rows, in_frac, seed):
        """rpk_split_fraction: uint8 mask over the table rows, 1 = data_in (see include/rpk.h)."""
        n_rows = int(rows.shape[0])
        out = _empty_like_kind(rows, (n_rows,), np.uint8)
        self._check(self._lib.rpk_split_fraction(self._h, int(uids.shape[0]), _addr(uids, np.int64), _addr(seg, np.int64),
                                                 _addr(rows, np.int64), n_rows, float(in_frac), int(seed), _addr(out, np.uint8)))
        return out

    def fit_strip_rows(self, rows: int = 0):
        """rpk_fit_strip_rows: item rows per strip of the fit (0 = automatic)."""
        self._check(self._lib.rpk_fit_strip_rows(self._h, int(rows)))

    def gram_dense_u16(self, A):
        """G = A A^T on the tensor cores for a 0/1 uint8 matrix A [I, Kd] (verification entry)."""
        I, Kd = A.shape
        out = _empty_like_kind(A, (I, I), np.uint16)
        self._check(self._lib.rpk_gram_dense_u16(self._h, int(I), int(Kd), _addr(A, np.uint8), _addr(out, np.uint16)))
        return out

    # -- item neighbours of a dense embedding matrix ---------------------------------------
    def embed_topk(self, E, K, similarity="cosine", item_begin=0, item_end=None, want_val=True):
        """rpk_embed_topk for a float64 [I, D] matrix (numpy or torch CUDA).  Returns dict(idx, val, len), rank order."""
        I, D = (int(n) for n in E.shape)
        item_end = I if item_end is None else int(item_end)
        rows = max(item_end - int(item_begin), 0)
        out = {
            "idx": _empty_like_kind(E, (rows, K), np.int32),
            "val": _empty_like_kind(E, (rows, K), np.float64) if want_val else None,
            "len": _empty_like_kind(E, (rows,), np.int32),
        }
        self._check(self._lib.rpk_embed_topk(self._h, I, D, _addr(E, np.float64), EMBED_SIM_CODES[similarity], int(K),
                                             int(item_begin), int(item_end), _addr(out["idx"], np.int32),
                                             _addr(out["val"], np.float64, allow_none=True), _addr(out["len"], np.int32)))
        return out

    def embed_screen_f32(self, E, similarity="cosine"):
        """rpk_embed_screen_f32: the screen's approximate [I, I] float32 matrix (verification entry)."""
        I, D = (int(n) for n in E.shape)
        out = _empty_like_kind(E, (I, I), np.float32)
        self._check(self._lib.rpk_embed_screen_f32(self._h, I, D, _addr(E, np.float64), EMBED_SIM_CODES[similarity],
                                                   _addr(out, np.float32)))
        return out

    # -- EASE: dense Gram, closed-form model, dense scoring ----------------------------------
    def gram_dense_f64(self, U, I, indptr, indices):
        """rpk_gram_dense_f64: exact X^T X of all users as float64 [I, I] (torch CUDA tensor when the inputs are)."""
        out = _empty_like_kind(indices, (I, I), np.float64)
        self._check(self._lib.rpk_gram_dense_f64(self._h, int(U), int(I), int(indices.shape[0]), _addr(indptr, np.int64),
                                                 _addr(indices, np.int32), _addr(out, np.float64)))
        return out

    def ease_from_inverse(self, P, w=None, out=None):
        """rpk_ease_from_inverse on device matrices: B = -P / diag(P) (columns), zero diagonal, optional column scale w."""
        I = int(P.shape[0])
        out = P if out is None else out
        self._check(self._lib.rpk_ease_from_inverse(self._h, I, _addr(P, np.float64), _addr(w, np.float64, allow_none=True),
                                                    _addr(out, np.float64)))
        return out

    def ease_prune(self, B, keep):
        """rpk_ease_prune: the min(keep, nnz(B)) largest-magnitude entries of the device matrix B [I, I] as a canonical
        CSR of device tensors (indptr int64, indices int32, values float64), trimmed to the kept count."""
        import torch

        I = int(B.shape[0])
        keep = int(keep)
        cap = max(1, min(keep, I * I))
        indptr = torch.empty(I + 1, dtype=torch.int64, device=B.device)
        indices = torch.empty(cap, dtype=torch.int32, device=B.device)
        values = torch.empty(cap, dtype=torch.float64, device=B.device)
        nnz = np.zeros(1, dtype=np.int64)
        self._check(self._lib.rpk_ease_prune(self._h, I, _addr(B, np.float64), keep, _addr(indptr, np.int64),
                                             _addr(indices, np.int32), _addr(values, np.float64), _addr(nnz)))
        n = int(nnz[0])
        if n < cap:  # let the unused part of the output go
            indices, values = indices[:n].clone(), values[:n].clone()
        return indptr, indices, values

    def predict_dense_topn(self, U, indptr, indices, B, N, mask_history=True, want_val=True):
        out = {
            "idx": _empty_like_kind(indices, (U, N), np.int32),
            "val": _empty_like_kind(indices, (U, N), np.float64) if want_val else None,
            "len": _empty_like_kind(indices, (U,), np.int32),
        }
        self._check(self._lib.rpk_predict_dense_topn(
            self._h, int(U), int(indices.shape[0]), _addr(indptr, np.int64), _addr(indices, np.int32), int(B.shape[0]),
            _addr(B, np.float64), int(N), int(bool(mask_history)), _addr(out["idx"], np.int32),
            _addr(out["val"], np.float64, allow_none=True), _addr(out["len"], np.int32)))
        return out

    def predict_dense_full(self, U, indptr, indices, B, mask_history=False):
        """All scores X @ B as a float64 [U, I] array next to the inputs (torch CUDA tensor or numpy)."""
        out = _empty_like_kind(indices, (U, int(B.shape[0])), np.float64)
        self._check(self._lib.rpk_predict_dense_full(
            self._h, int(U), int(indices.shape[0]), _addr(indptr, np.int64), _addr(indices, np.int32), int(B.shape[0]),
            _addr(B, np.float64), int(bool(mask_history)), _addr(out, np.float64)))
        return out

    # -- model ----------------------------------------------------------------------------
    def model_load_topk(self, I, K, idx, val, ln):
        self._check(self._lib.rpk_model_load_topk(self._h, int(I), int(K), _addr(idx, np.int32), _addr(val, np.float64),
                                                  _addr(ln, np.int32)))

    def model_load_topk_rows(self, I, K, rows_in, idx, val, ln, row_src):
        self._check(self._lib.rpk_model_load_topk_rows(self._h, int(I), int(K), int(rows_in), _addr(idx, np.int32),
                                                       _addr(val, np.float64), _addr(ln, np.int32), _addr(row_src, np.int64)))

    def model_scale_exp(self, K, val, ln) -> int:
        """rpk_model_scale_exp: exponent e of the fixed-point scale 2^e these lists would get as a model of their own."""
        e = C.c_int32(0)
        self._check(self._lib.rpk_model_scale_exp(self._h, int(K), int(val.shape[0]), _addr(val, np.float64), _addr(ln, np.int32),
                                                  C.byref(e)))
        return int(e.value)

    def model_pack_rows(self, I, K, idx, val, ln, scale_exp, out=None):
        """rpk_model_pack_rows: rank-ordered lists -> packed model rows (uint64 bit patterns; torch tensors carry
        them as int64) at the scale 2^scale_exp.  `out`: [rows, K] buffer to fill."""
        rows = int(idx.shape[0])
        if out is None:
            out = _empty_like_kind(idx, (rows, K), np.int64 if _is_torch(idx) else np.uint64)
        self._check(self._lib.rpk_model_pack_rows(self._h, int(I), int(K), rows, _addr(idx, np.int32), _addr(val, np.float64),
                                                  _addr(ln, np.int32), int(scale_exp), _addr(out)))
        return out

    def model_load_packed_rows(self, I, K, rows_in, ent, ln, scale_exp, row_src=None):
        self._check(self._lib.rpk_model_load_packed_rows(self._h, int(I), int(K), int(rows_in), _addr(ent), _addr(ln, np.int32),
                                                         _addr(row_src, np.int64, allow_none=True), int(scale_exp)))

    def model_vmax(self, K, val, ln, out):
        """rpk_model_vmax: the largest value of the lists into `out` (one float64, device tensor: stream-ordered)."""
        self._check(self._lib.rpk_model_vmax(self._h, int(K), int(val.shape[0]), _addr(val, np.float64), _addr(ln, np.int32),
                                             _addr(out, np.float64)))
        return out

    def model_pack_rows_v(self, I, K, idx, val, ln, vmax, out):
        self._check(self._lib.rpk_model_pack_rows_v(self._h, int(I), int(K), int(idx.shape[0]), _addr(idx, np.int32),
                                                    _addr(val, np.float64), _addr(ln, np.int32), _addr(vmax, np.float64), _addr(out)))
        return out

    def model_load_packed_rows_v(self, I, K, rows_in, ent, ln, vmax, row_src=None):
        self._check(self._lib.rpk_model_load_packed_rows_v(self._h, int(I), int(K), int(rows_in), _addr(ent), _addr(ln, np.int32),
                                                           _addr(row_src, np.int64, allow_none=True), _addr(vmax, np.float64)))

    def fit_token(self) -> int:
        return int(self._lib.rpk_fit_token(self._h))

    def model_load_last_fit(self, token: int):
        self._check(self._lib.rpk_model_load_last_fit(self._h, int(token)))

    def model_load_csr(self, I, indptr, indices, values):
        self._check(self._lib.rpk_model_load_csr(self._h, int(I), int(indices.shape[0]), _addr(indptr, np.int64),
                                                 _addr(indices, np.int32), _addr(values, np.float64)))

    def model_load_signed_csr(self, I, indptr, indices, values):
        """A model of any sign, scored in float64: predictions are scipy's ``X @ S`` bit for bit."""
        self._check(self._lib.rpk_model_load_signed_csr(self._h, int(I), int(indices.shape[0]), _addr(indptr, np.int64),
                                                        _addr(indices, np.int32), _addr(values, np.float64)))

    # -- predict --------------------------------------------------------------------------
    def predict_topn(self, U, indptr, indices, N, mask_history=True, want_val=True, out=None):
        if out is None:
            out = {
                "idx": _empty_like_kind(indices, (U, N), np.int32),
                "val": _empty_like_kind(indices, (U, N), np.float64) if want_val else None,
                "len": _empty_like_kind(indices, (U,), np.int32),
            }
        self._check(self._lib.rpk_predict_topn(
            self._h, int(U), int(indices.shape[0]), _addr(indptr, np.int64), _addr(indices, np.int32), int(N),
            int(bool(mask_history)), _addr(out["idx"], np.int32), _addr(out.get("val"), np.float64, allow_none=True),
            _addr(out["len"], np.int32)))
        return out

    def predict_item_filter(self, allowed):
        """rpk_predict_item_filter: uint8[I] mask of the items that may be recommended (None removes the filter)."""
        if allowed is None:
            self._check(self._lib.rpk_predict_item_filter(self._h, None, 0))
        else:
            self._check(self._lib.rpk_predict_item_filter(self._h, _addr(allowed, np.uint8), int(allowed.shape[0])))

    def predict_csr(self, U, indptr, indices, mask_history=False):
        """Full score matrix as (indptr int64, indices int32, data float64) numpy arrays."""
        nnz = int(indices.shape[0])
        row_nnz = np.empty(U, dtype=np.int64)
        self._check(self._lib.rpk_predict_csr_count(self._h, int(U), nnz, _addr(indptr, np.int64), _addr(indices, np.int32),
                                                    int(bool(mask_history)), _addr(row_nnz, np.int64)))
        out_indptr = np.zeros(U + 1, dtype=np.int64)
        np.cumsum(row_nnz, out=out_indptr[1:])
        total = int(out_indptr[-1])
        out_indices = np.empty(total, dtype=np.int32)
        out_values = np.empty(total, dtype=np.float64)
        if U > 0:
            self._check(self._lib.rpk_predict_csr_fill(
                self._h, int(U), nnz, _addr(indptr, np.int64), _addr(indices, np.int32), int(bool(mask_history)),
                _addr(out_indptr, np.int64), _addr(out_indices, np.int32), _addr(out_values, np.float64)))
        return out_indptr, out_indices, out_values

    # -- ranking / metrics ----------------------------------------------------------------
    def topk_csr(self, rows, indptr, indices, values, K):
        out_idx = _empty_like_kind(indices, (rows, K), np.int32)
        out_len = _empty_like_kind(indices, (rows,), np.int32)
        self._check(self._lib.rpk_topk_csr(self._h, int(rows), int(indices.shape[0]), _addr(indptr, np.int64),
                                           _addr(indices, np.int32), _addr(values, np.float64), int(K),
                                           _addr(out_idx, np.int32), _addr(out_len, np.int32)))
        return out_idx, out_len

    def metrics_topn(self, U, N, top_idx, top_len, true_indptr, true_indices, metrics, want_per_user=True, out_sums=None,
                     out_n_users=None):
        """metrics: list of (kind, K).  Returns (sums float64[m], n_users int, per_user float64[m, U] or None).
        The discount / IDCG tables are built here with numpy exactly as recpack/metrics/dcg.py:98-104 does.
        out_sums (float64[m]) / out_n_users (int64[1]) as torch CUDA tensors keep the reduction on the device: the call
        is then stream-ordered without a host round trip and returns the two tensors instead of host values."""
        import itertools

        kinds = np.array([METRIC_CODES[k] for k, _ in metrics], dtype=np.int32)
        Ks = np.array([k for _, k in metrics], dtype=np.int32)
        maxK = int(Ks.max())
        disc = 1.0 / np.log2(np.arange(2, maxK + 2))
        idcg = np.array([1] + list(itertools.accumulate(disc, lambda x, y: x + y)), dtype=np.float64)
        m = len(metrics)
        per_user = _empty_like_kind(top_idx, (m, U), np.float64) if want_per_user else None
        on_device = out_sums is not None and out_n_users is not None
        sums = out_sums if on_device else np.empty(m, dtype=np.float64)
        n_users = out_n_users if on_device else np.zeros(1, dtype=np.int64)
        self._check(self._lib.rpk_metrics_topn(
            self._h, int(U), int(N), _addr(top_idx, np.int32), _addr(top_len, np.int32), _addr(true_indptr, np.int64),
            _addr(true_indices, np.int32), int(true_indices.shape[0]), m, _addr(kinds), _addr(Ks),
            _addr(np.ascontiguousarray(disc)), _addr(idcg), maxK, _addr(per_user, np.float64, allow_none=True),
            _addr(sums, np.float64), _addr(n_users, np.int64)))
        if on_device:
            return sums, n_users, per_user
        return sums, int(n_users[0]), per_user


    def coverage_topn(self, U, N, K, I, top_idx, top_len, true_indptr, want_flags=False):
        """rpk_coverage_topn: (number of covered items, uint8[I] flags or None)."""
        count = np.zeros(1, dtype=np.int64)
        flags = np.zeros(I, dtype=np.uint8) if want_flags else None
        self._check(self._lib.rpk_coverage_topn(self._h, int(U), int(N), int(K), int(I), _addr(top_idx, np.int32),
                                                _addr(top_len, np.int32), _addr(true_indptr, np.int64), _addr(count),
                                                _addr(flags, np.uint8, allow_none=True)))
        return int(count[0]), flags


_engines = {}
_lock = threading.Lock()


def get_engine(device: int | None = None) -> Engine:
    """Process-wide engine of a device (default: LOCAL_RANK, else 0)."""
    import os

    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    with _lock:
        eng = _engines.get(device)
        if eng is None:
            eng = _engines[device] = Engine(device)
        return eng
