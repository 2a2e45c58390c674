#!/usr/bin/env python
"""Top-20 scoring of a signed model at the ML-25M shape, remove_history on: three routes timed in one process,
alternating, warm, with CUDA events over the same launches.

  signed   rpk_predict_topn on the signed model (k_predict_signed + the float64 row kernel for handed-over users)
  spgemm   rpk_spgemm_topn with unit left values: the same lists through k_real_rows
  a32      rpk_predict_topn on |S| (the fixed-point k_predict_a32), for scale

The model is ItemKNN cosine K=200 with a seeded, hash-chosen third of its entries negated.  Histories and model are
device-resident for all three, so each time is the call on the stream.  Prints the card name and power limit.
usage: probe_signed.py [reps]"""
import os
import subprocess
import sys
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from scipy.sparse import csr_matrix

from recpack_b200 import ItemKNN
from recpack_b200.engine import Engine
from recpack_b200.synth import make_dataset

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                   text=True)
print(f"card: {q.stdout.strip()}", flush=True)
train, _, _ = make_dataset("ml25m")
with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    S = csr_matrix(ItemKNN(K=200).fit(train).similarity_matrix_)
S.sort_indices()
rows = np.repeat(np.arange(S.shape[0], dtype=np.uint64), np.diff(S.indptr))
h = (rows * np.uint64(0x9E3779B1) + S.indices.astype(np.uint64) * np.uint64(0x85EBCA77) + np.uint64(12345)) % np.uint64(3)
S.data[h == 0] *= -1
U, I = train.shape
print(f"U={U} I={I} history nnz={train.nnz} model nnz={S.nnz} negative={np.count_nonzero(S.data < 0)}", flush=True)

dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
X = csr_matrix(train, dtype=np.float64)
X.sort_indices()
ptr, idx, ones = dev(X.indptr, np.int64), dev(X.indices, np.int32), torch.ones(X.nnz, dtype=torch.float64, device="cuda")
s_ptr, s_idx, s_val = dev(S.indptr, np.int64), dev(S.indices, np.int32), dev(S.data, np.float64)
N = 20
eng_s, eng_g, eng_a = Engine(0), Engine(0), Engine(0)
for e in (eng_s, eng_g, eng_a):
    e.use_torch_stream()
eng_s.model_load_signed_csr(I, s_ptr, s_idx, s_val)
eng_a.model_load_csr(I, s_ptr, s_idx, s_val.abs())
outs = {k: {"idx": torch.empty((U, N), dtype=torch.int32, device="cuda"), "val": torch.empty((U, N), dtype=torch.float64, device="cuda"),
            "len": torch.empty(U, dtype=torch.int32, device="cuda")} for k in ("signed", "spgemm", "a32")}
lib = eng_g._lib


def signed():
    eng_s.predict_topn(U, ptr, idx, N, mask_history=True, out=outs["signed"])


def spgemm():
    o = outs["spgemm"]
    eng_g._check(lib.rpk_spgemm_topn(eng_g._h, U, X.nnz, ptr.data_ptr(), idx.data_ptr(), ones.data_ptr(), I, S.nnz, s_ptr.data_ptr(),
                                     s_idx.data_ptr(), s_val.data_ptr(), N, 1, o["idx"].data_ptr(), o["val"].data_ptr(),
                                     o["len"].data_ptr()))


def a32():
    eng_a.predict_topn(U, ptr, idx, N, mask_history=True, out=outs["a32"])


routes = {"signed": signed, "spgemm": spgemm, "a32": a32}
for f in routes.values():  # warm-up: module loads, geometry tables, scratch buffers
    f()
torch.cuda.synchronize()
same = all(torch.equal(outs["signed"][k], outs["spgemm"][k]) for k in ("idx", "val", "len"))
print(f"signed lists == spgemm lists for all {U} users: {same}", flush=True)
times = {k: [] for k in routes}
for r in range(reps):
    for k, f in routes.items():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        f()
        b.record()
        b.synchronize()
        times[k].append(a.elapsed_time(b))
for k, t in times.items():
    t = np.array(t)
    print(f"{k:7s} median {np.median(t):8.2f} ms  min {t.min():8.2f}  max {t.max():8.2f}  over {len(t)} calls", flush=True)
print(f"signed last_timings (scoring slot, ms): {eng_s.last_timings()}", flush=True)
