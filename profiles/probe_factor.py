"""Factor-model scoring (rpk_factor_topn) at full size: the ML-25M shape (D = 128, N = 20) and 1M x 200k (D = 128,
N = 100), remove_history, seeded Gaussian factors, the interactions of synth.make_dataset.

Per shape: the card's name and power limit; CUDA-event time per call (after a warm-up call, mean over >= 3 calls); the
phase marks of one traced call (prep, screen chunks, compactions, exact pass, exact rows); the screen's achieved
TFLOP/s (2 U_scored I D over the summed chunk time) against the data-sheet 1,125 TFLOP/s of dense TF32.  For comparison,
in the same run: cuBLAS fp32 torch.mm in user blocks + history mask + torch.topk (not exact: a speed reference only), and
a CPU estimate of the reference's recipe (P[users] @ Q.T into a lil_matrix, then the top N) on a user sample,
extrapolated.  With RPK_LIB pointing at a -DRPK_PHASE_PROF build the library also prints its "[factor paths]" counters.

    python profiles/probe_factor.py [--shapes ml25m,large] [--calls 3]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.sparse import csr_matrix, lil_matrix

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from recpack_b200.engine import get_engine  # noqa: E402
from recpack_b200.synth import make_dataset  # noqa: E402

N_OF = {"ml25m": 20, "large": 100}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fn, calls):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="ml25m,large")
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--D", type=int, default=128)
    args = ap.parse_args()
    print(f"# card: {card()}")
    eng = get_engine(0)
    eng.use_torch_stream()
    D = args.D
    dev = torch.device("cuda", 0)
    for shape in args.shapes.split(","):
        N = N_OF[shape]
        train, _, _ = make_dataset(shape, seed=0)
        if not isinstance(train, csr_matrix):
            train = csr_matrix(train)
        U, I = train.shape
        ptr = torch.from_numpy(np.ascontiguousarray(train.indptr, dtype=np.int64)).to(dev)
        idx = torch.from_numpy(np.ascontiguousarray(train.indices, dtype=np.int32)).to(dev)
        g = torch.Generator(device="cuda").manual_seed(U)
        P = torch.randn((U, D), dtype=torch.float64, device=dev, generator=g)
        Q = torch.randn((I, D), dtype=torch.float64, device=dev, generator=g)
        scored = int(((ptr[1:] - ptr[:-1]) > 0).sum())
        ms = timed(lambda: eng.factor_topn(P, Q, ptr, idx, N, mask_history=True), args.calls)
        print(f"{shape}: U={U} (scored {scored}) I={I} nnz={train.nnz} D={D} N={N} remove_history: {ms:.2f} ms per call "
              f"(CUDA events, mean of {args.calls} after a warm-up)")
        eng.trace(True)
        eng.factor_topn(P, Q, ptr, idx, N, mask_history=True)
        eng.trace(False)
        rep = eng.trace_report()
        phases, gemm = {}, 0.0
        for line in rep.splitlines():
            name, t = line.rsplit(None, 2)[0].strip(), float(line.rsplit(None, 2)[1])
            phases[name] = phases.get(name, 0.0) + t
            if name == "factor: screen chunk":
                gemm += t
        print("  phases (ms, summed over chunks / row groups): " + ", ".join(f"{k} {v:.2f}" for k, v in phases.items()))
        flop = 2.0 * scored * I * D
        tf = flop / (gemm * 1e-3) / 1e12
        print(f"  screen: {flop / 1e12:.2f} TFLOP in {gemm:.2f} ms = {tf:.1f} TFLOP/s "
              f"({100 * tf / 1125:.1f} % of the 1,125 TFLOP/s dense TF32 data-sheet rate)")
        # cuBLAS fp32 + history mask + torch.topk in user blocks (not exact; speed reference)
        Pf, Qf = P.float(), Q.float()
        B = max(1, min(U, (8 << 30) // (4 * I)))
        users = torch.repeat_interleave(torch.arange(U, device=dev), ptr[1:] - ptr[:-1])

        def blas():
            for r0 in range(0, U, B):
                r1 = min(U, r0 + B)
                S = Pf[r0:r1] @ Qf.T
                lo, hi = int(ptr[r0]), int(ptr[r1])
                S[users[lo:hi] - r0, idx[lo:hi].long()] = -float("inf")
                torch.topk(S, N, dim=1)

        ms_b = timed(blas, 1)
        print(f"  cuBLAS fp32 torch.mm + history mask + torch.topk in blocks of {B} users: {ms_b:.2f} ms per call (not exact)")
        del Pf, Qf, users
        # CPU estimate of the reference's recipe on a user sample
        Pn, Qn = P.cpu().numpy(), Q.cpu().numpy()
        sample = np.sort(np.random.default_rng(0).choice(U, size=min(U, 1000 if I < 100_000 else 200), replace=False))
        Xs = train[sample]
        t0 = time.perf_counter()
        for r0 in range(0, len(sample), 50):
            Xb = Xs[r0 : r0 + 50]
            us = list(set(Xb.nonzero()[0]))
            res = lil_matrix(Xb.shape)
            res[us] = Pn[sample[r0 : r0 + 50]][us] @ Qn.T
            R = res.tocsr()
            R = R - R.multiply(Xb)  # remove_history, as the pipeline does
            Rd = R.toarray()
            np.argpartition(Rd, -N, axis=1)[:, -N:]
        t_cpu = (time.perf_counter() - t0) * U / len(sample)
        print(f"  CPU estimate (the reference's lil_matrix recipe + history removal + argpartition on {len(sample)} users = "
              f"{100 * len(sample) / U:.2f} %, extrapolated, {os.cpu_count()} CPUs): {t_cpu:.1f} s")
        del P, Q, ptr, idx
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
