"""Embedding neighbours (rpk_embed_topk) at full size: I in {200,000, 1,000,000}, D = 128, K = 100, cosine.

Per shape: the card's name and power limit; CUDA-event time per call (after a warm-up call, mean over >= 5 calls);
the phase marks of one traced call (prep, each screen chunk, each compaction, exact pass, exact rows); the screen's
achieved TFLOP/s (2 I^2 D over the summed chunk GEMM time) against the data-sheet 1,125 TFLOP/s of dense TF32.
For comparison, in the same run: cuBLAS fp32 torch.mm in row blocks + torch.topk (not exact: a speed reference only),
and a CPU estimate (sklearn cosine_similarity + the reference's top-K on a sample of rows, extrapolated).
With RPK_LIB pointing at a -DRPK_PHASE_PROF build the library also prints its "[embed paths]" counters (stderr).

    python profiles/probe_embed.py [--sizes 200000,1000000] [--calls 5]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from recpack_b200.engine import get_engine  # noqa: E402


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
    ap.add_argument("--sizes", default="200000,1000000")
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--D", type=int, default=128)
    ap.add_argument("--K", type=int, default=100)
    args = ap.parse_args()
    print(f"# card: {card()}")
    eng = get_engine(0)
    eng.use_torch_stream()
    D, K = args.D, args.K
    for I in (int(s) for s in args.sizes.split(",")):
        g = torch.Generator(device="cuda").manual_seed(I)
        E = torch.randn((I, D), dtype=torch.float64, device="cuda", generator=g)
        ms = timed(lambda: eng.embed_topk(E, K, "cosine"), args.calls)
        print(f"I={I} D={D} K={K} cosine: {ms:.2f} ms per call (CUDA events, mean of {args.calls} after a warm-up)")
        eng.trace(True)
        eng.embed_topk(E, K, "cosine")
        eng.trace(False)
        rep = eng.trace_report()
        phases = {}
        gemm = 0.0
        for line in rep.splitlines():
            name, t = line.rsplit(None, 2)[0].strip(), float(line.rsplit(None, 2)[1])
            phases[name] = phases.get(name, 0.0) + t
            if name == "embed: screen chunk":
                gemm += t
        print("  phases (ms, summed over chunks / row groups): " + ", ".join(f"{k} {v:.2f}" for k, v in phases.items()))
        tf = 2.0 * I * I * D / (gemm * 1e-3) / 1e12
        print(f"  screen: {2.0 * I * I * D / 1e12:.2f} TFLOP in {gemm:.2f} ms = {tf:.1f} TFLOP/s "
              f"({100 * tf / 1125:.1f} % of the 1,125 TFLOP/s dense TF32 data-sheet rate)")
        # cuBLAS fp32 + torch.topk in row blocks (not exact; speed reference)
        Xn = torch.nn.functional.normalize(E, dim=1).float()
        B = max(1, min(I, (8 << 30) // (4 * I)))

        def blas():
            for r0 in range(0, I, B):
                S = Xn[r0 : r0 + B] @ Xn.T
                S[torch.arange(S.shape[0], device="cuda"), torch.arange(r0, r0 + S.shape[0], device="cuda")] = -2
                torch.topk(S, K, dim=1)

        ms_b = timed(blas, 2)
        print(f"  cuBLAS fp32 torch.mm + torch.topk in blocks of {B} rows: {ms_b:.2f} ms per call (not exact)")
        del Xn
        # CPU estimate on a row sample
        from sklearn.metrics.pairwise import cosine_similarity

        En = E.cpu().numpy()
        rows = np.random.default_rng(0).choice(I, size=min(I, 2000), replace=False)
        t0 = time.perf_counter()
        for r0 in range(0, len(rows), 250):
            S = cosine_similarity(En[rows[r0 : r0 + 250]], En)
            S[np.arange(S.shape[0]), rows[r0 : r0 + 250]] = 0.0
            part = np.argpartition(S, -K, axis=1)[:, -K:]
            np.take_along_axis(S, part, axis=1)
        t_cpu = (time.perf_counter() - t0) * I / len(rows)
        print(f"  CPU estimate (sklearn cosine_similarity + argpartition top-K on {len(rows)} rows = "
              f"{100 * len(rows) / I:.2f} %, extrapolated, {os.cpu_count()} CPUs): {t_cpu:.1f} s")
        del E
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
