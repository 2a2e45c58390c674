#!/usr/bin/env python
"""EASE l2=200 at a named shape (default msd: 571,355 x 41,140, 33.6 M interactions) for density None, 0.01 and 0.001:
device-event time of each fit phase (Gram, inverse, finish, prune), predict(top-20, remove_history) for all users, NDCG@10,
Recall@20 and the entries kept, with the card's name and power limit read in the same run.  For the pruned models it
also reports the device time of each stage of rpk_ease_prune (its trace marks), both for the call timed as a phase and
for the call inside the class's fit, and the number of candidates (entries of the top-digit bin that holds the cut).

The phases are the calls of ``EASE._fit`` in its order, each between two CUDA events on the stream both torch and the
engine use; "fit (class)" is the whole ``_fit`` of the drop-in class, timed the same way.  Usage:
    python profiles/probe_ease_density.py [shape]"""
import os
import subprocess
import sys
import time
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from recpack_b200 import EASE, NDCGK, RecallK  # noqa: E402
from recpack_b200.ease import prune_keep  # noqa: E402
from recpack_b200.engine import get_engine  # noqa: E402
from recpack_b200.matrix import device_structure  # noqa: E402
from recpack_b200.synth import make_dataset  # noqa: E402

L2 = 200.0
NAN_KEY = 0x7FF0000000000001


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def phases(train, density):
    """Device time (ms) of each step of EASE._fit, in its order."""
    eng = get_engine(0)
    X, _, _, ptr_d, idx_d = device_structure(train, eng.device)
    U, I = X.shape
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ev[0].record()
    G = eng.gram_dense_f64(U, I, ptr_d, idx_d)
    eng.sync()
    ev[1].record()
    torch.diagonal(G).add_(float(np.float32(L2)))
    L = torch.linalg.cholesky(G)
    del G
    P = torch.cholesky_inverse(L).contiguous()
    del L
    ev[2].record()
    torch.cuda.current_stream().synchronize()
    B = eng.ease_from_inverse(P, None)
    eng.sync()
    ev[3].record()
    eng.trace_report()  # drop the marks of the calls above
    stages, n_cand = None, 0
    if density:
        _, _, val = eng.ease_prune(B, prune_keep(density, I))
        ev[4].record()
        torch.cuda.synchronize()
        stages = prune_stages(eng.trace_report())
        nnz = int(val.shape[0])
        # entries of the top-digit bin that holds the cut: the candidates of the selection
        cut = int(((val.view(torch.int64) & 0x7FFFFFFFFFFFFFFF).clamp(max=NAN_KEY)).min().item())
        keys = (B.view(torch.int64) & 0x7FFFFFFFFFFFFFFF).clamp_(max=NAN_KEY)
        n_cand = int(((keys >> 48) == (cut >> 48)).logical_and_(keys != 0).sum().item())
        del val, keys
    else:
        nnz = int((B != 0).sum().item())
        ev[4].record()
        torch.cuda.synchronize()
    del B, P
    torch.cuda.empty_cache()
    names = ["gram", "inverse", "finish", "prune"]
    out = {n: ev[k].elapsed_time(ev[k + 1]) for k, n in enumerate(names)}
    if not density:
        out["prune"] = 0.0
    return out, nnz, stages, n_cand


def prune_stages(report):
    """Device time (ms) of the stages of one rpk_ease_prune call from its trace marks (a mark's time is the time since
    the mark before it, so a stage's time is that of the mark which ends it)."""
    marks = [(name.strip(), float(ms)) for name, ms, _ in (ln.rsplit(None, 2) for ln in report.splitlines() if ln.strip())]
    names = [n for n, _ in marks]
    if "prune_hist" not in names or "prune_end" not in names:
        return None
    i = names.index("prune_hist")
    ends = {"prune_collect": "hist", "prune_select": "collect", "prune_counts": "select", "prune_fill": "counts+scans",
            "prune_end": "fill"}
    out = {ends[n]: ms for n, ms in marks[i + 1:] if n in ends}
    out["total"] = sum(out.values())
    return out


def fmt_stages(st):
    return "n/a" if st is None else " ".join(f"{k} {v:.1f}" for k, v in st.items()) + " ms"


def main():
    shape = sys.argv[1] if len(sys.argv) > 1 else "msd"
    print(f"card: {card()}", flush=True)
    t0 = time.time()
    train, test_out, gen = make_dataset(shape, generator="auto")
    U, I = train.shape
    print(f"[{shape}] data {time.time() - t0:.1f} s gen={gen} U={U} I={I} nnz={train.nnz}", flush=True)
    eng = get_engine(0)
    eng.trace(True)
    for density in (None, 0.01, 0.001):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for rep in range(2):  # the first repetition warms up every shape
                ph, kept, st_phase, n_cand = phases(train, density)
                algo = EASE(l2=L2, density=density, predict_topK=20, remove_history=True)
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                Xf = algo._transform_fit_input(train)
                eng.trace_report()
                e[0].record()
                algo._fit(Xf)
                e[1].record()
                torch.cuda.synchronize()
                st_class = prune_stages(eng.trace_report())
                Xp = algo._transform_predict_input(train)
                pred = algo._predict(Xp)
                e[2].record()
                torch.cuda.synchronize()
                m = NDCGK(10)
                m.calculate(test_out, pred)
                r = RecallK(20)
                r.calculate(test_out, pred)
                print(f"[{shape}] density={density} rep{rep}  gram {ph['gram']:.1f} ms  inverse {ph['inverse']:.1f} ms  "
                      f"finish {ph['finish']:.1f} ms  prune {ph['prune']:.1f} ms  | fit (class) {e[0].elapsed_time(e[1]):.1f} ms  "
                      f"predict(top-20, remove_history, {U} users) {e[1].elapsed_time(e[2]):.1f} ms  "
                      f"NDCG@10 {m.value:.6f}  Recall@20 {r.value:.6f}  kept {kept} of {I * I}  "
                      f"torch peak {torch.cuda.max_memory_allocated() / 1e9:.1f} GB", flush=True)
                if density:
                    print(f"[{shape}] density={density} rep{rep}  boundary-bin entries (candidates) {n_cand}  "
                          f"prune stages, phases(): {fmt_stages(st_phase)}  |  inside EASE._fit: {fmt_stages(st_class)}",
                          flush=True)
                del algo, pred
                torch.cuda.empty_cache()
    print(f"card: {card()}", flush=True)


if __name__ == "__main__":
    main()
