#!/usr/bin/env python
"""Benchmark of the item-similarity hot path: ItemKNN fit -> predict (top-N, history masked) ->
NDCG@10 / Recall@20 on a synthetic ML-25M-shape matrix (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            # this repo, N GPUs (torchrun for N > 1)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle restatement)
  python bench.py --steps K --warmup W --dump-outputs DIR  # also writes the last timed step's results to DIR/*.npy

One "step" = one full pass: fit of this rank's item rows, all-gather of the pruned similarity lists
(N > 1), scoring + top-20 + NDCG@10 / Recall@20 of this rank's users, all-reduce of the metric sums.
`value` = evaluated users / step time with all inputs resident in HBM; `e2e` = the same through the
public classes with host (pinned) scipy inputs, host<->device copies inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ItemKNN fit + predict + NDCG@10/Recall@20 throughput (evaluated users / second per full pass)"
UNIT = "users/s"
N_LIST = 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (full passes); the e2e leg times as many")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--shape", default="ml25m", help="ml100k | ml1m | ml25m | netflix | msd | large (recpack_b200/synth.py SHAPES)")
    ap.add_argument("--similarity", default="cosine", choices=["cosine", "conditional_probability"])
    ap.add_argument("--K", type=int, default=200, help="neighbours kept per item")
    ap.add_argument("--generator", default="auto", choices=["auto", "numpy", "cuda"], help="synthetic data generator (synth.make_dataset)")
    ap.add_argument("--trace", action="store_true", help="print rank 0's device-time trace of one extra step (rpk_trace) to stderr")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--ref-fraction", type=float, default=0.02, help="fraction of a full pass one step of the reference arm / CPU baseline does")
    ap.add_argument("--cpu-procs", type=int, default=0, help="worker processes of --impl reference's setup (0 = one per host core, at most 64)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs); "
                                                          "one GPU only")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl b200 and --gpus 1")
    return args


def make_data(args):
    """(train, test_out) of the named shape; the generator used is recorded in args.generator_used."""
    from recpack_b200.synth import make_dataset

    train, test_out, gen = make_dataset(args.shape, seed=0, split_seed=42, generator=args.generator)
    args.generator_used = gen
    return train, test_out


def workload_name(args, train, n_eval=None):
    U, I = train.shape
    sim = "cosine" if args.similarity == "cosine" else "conditional-probability"
    tail = f" over {n_eval} users" if n_eval is not None else ""
    return (f"ItemKNN {sim} K={args.K}, {args.shape} shape {U}x{I}, {train.nnz} train interactions (80% WeakGeneralization split), "
            f"top-{N_LIST} with history masked, NDCG@10 + Recall@20{tail}")


def workload_stats(train, K, N, test_out):
    d = np.diff(train.indptr).astype(np.float64)
    dout = np.diff(test_out.indptr).astype(np.float64)
    U, I = train.shape
    return {
        "sum_d2": float((d * d).sum()),
        # SURVEY.md 8(d): bytes per user = d_u*(4 + K*8) + 8 + N*8 + d_out*4
        "score_bytes": float((d * (4 + K * 8) + 8 + N * 8 + dout * 4).sum()),
        # sparse Gram: every (user, item) incidence re-reads that user's row (4 B / index) + CSC + output lists
        "fit_bytes": float((d * d).sum() * 4 + train.nnz * 8 + I * K * 8),
        "dense_equiv_ops": 2.0 * U * I * I,
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, device=0):
        self.rows = []
        self.proc = None
        self.device = device

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (baseline/_ref, unmodified), row-blocked -- baseline/ref_runner.py
# ----------------------------------------------------------------------------------------------
def bench_config(args, train, test_out):
    """The `config` object: identical for the GPU arm and the reference arm of the same command line."""
    n_eval = int(np.count_nonzero(np.diff(test_out.indptr)))
    return {"workload": workload_name(args, train, n_eval),
            "l2": "256 MB buffer written between timed iterations (L2 flush)", "seeds": {"data": 0, "split": 42},
            "generator": args.generator_used,
            "parallelism": f"item rows x{args.gpus} (fit), users x{args.gpus} (scoring)"}


def cpu_baseline(args, train, test_out, S_host, fraction, steps=1, seed0=0):
    """One (or a few) bounded steps of the reference on ONE host thread -- the reference's sparse path is
    single-threaded (scipy SpGEMM, sklearn normalise, the Python top-K loops).  A step fits a random `fraction` of
    the item rows and scores + evaluates the same fraction of the users against the real fitted S, so its time is
    that fraction of a full pass and users-in-the-sample / seconds estimates the full-pass throughput."""
    from baseline.ref_runner import RefRunner

    r = RefRunner(train, test_out, args.K, args.similarity)
    r.set_model(S_host)
    outs = [r.step(fraction, seed0 + k) for k in range(steps)]
    U, I = train.shape
    v = float(np.mean([o["users"] / o["seconds"] for o in outs]))
    o = outs[-1]
    return {
        "value": v, "unit": UNIT, "cores": 1, "kind": r.kind,
        "sample": f"{steps} step(s) of {o['rows']} of {I} item rows fitted + {o['users']} of {U} users scored and evaluated "
                  f"({100 * fraction:.1f} % of a full pass: fit {o['fit_seconds']:.1f} s + scoring {o['score_seconds']:.1f} s); "
                  + ("recpack's own get_top_K_values / ItemKNN._predict / NDCGK / RecallK from baseline/_ref on sklearn cosine_similarity row blocks"
                     if r.kind == "reference" else "oracle/recpack_oracle.py ref_* (recpack not importable)")
                  + f", 1 thread of {os.cpu_count()} host cores",
        "step_seconds": [round(x["seconds"], 3) for x in outs],
        "fit_seconds_full_pass_estimate": float(np.mean([x["fit_seconds"] for x in outs])) / fraction,
        "scoring_users_per_s": float(np.mean([x["users"] / x["score_seconds"] for x in outs])),
        "ndcg10_sample": float(o["ndcg10"]), "recall20_sample": float(o["recall20"]),
    }


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  Setup (untimed): the data and the
    complete similarity matrix, fitted by the reference's calls on all host cores (row blocks are independent).
    Timed: `steps` bounded steps on one thread, each a random `--ref-fraction` of a full pass (see cpu_baseline)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from baseline.ref_runner import RefRunner, parallel_steps

    t_start = time.perf_counter()
    train, test_out = make_data(args)
    U, I = train.shape
    r = RefRunner(train, test_out, args.K, args.similarity)
    procs = max(1, min(args.cpu_procs or (os.cpu_count() or 1), os.cpu_count() or 1, 64))
    t0 = time.perf_counter()
    d = np.diff(train.indptr).astype(np.float64)
    full_fit = float((d * d).sum()) <= 6e10  # ML-25M / Netflix shapes: minutes of CPU in all; beyond that a stand-in
    if full_fit:
        S = r.fit_all(procs)
        s_note = f"the reference's own row-blocked fit of all {I} rows on {procs} worker processes ({time.perf_counter() - t0:.0f} s, untimed setup)"
    else:
        rng = np.random.default_rng(1)
        from scipy.sparse import csr_matrix

        pop = np.sqrt(np.bincount(train.indices, minlength=I).astype(np.float64) + 1.0)
        idx = rng.choice(I, size=(I, args.K), p=pop / pop.sum()).astype(np.int32)
        S = csr_matrix((rng.random(I * args.K) * 0.5 + 1e-3, idx.ravel(), np.arange(I + 1, dtype=np.int64) * args.K), shape=(I, I))
        S.sum_duplicates()
        s_note = "a stand-in K-sparse S (neighbours ~ sqrt(popularity)): the complete reference fit of this shape takes hours of CPU"
    r.set_model(S)
    f = args.ref_fraction
    outs = []
    for s in range(args.warmup + args.steps):
        o = r.step(f, 1000 + s)
        if s >= args.warmup:
            outs.append(o)
    v = float(np.mean([o["users"] / o["seconds"] for o in outs]))
    ms = 1000.0 * float(np.mean([o["seconds"] for o in outs]))
    o = outs[-1]
    # what all host cores deliver together on independent blocks (one more round, every worker one step)
    par, wall = parallel_steps(r, f, [5000 + k for k in range(procs)])
    v_all = float(sum(x["users"] for x in par) / wall)
    sample = (f"each step: {o['rows']} of {I} item rows fitted + {o['users']} of {U} users scored and evaluated = {100 * f:.1f} % of a full pass, "
              f"measured (fit {o['fit_seconds']:.1f} s + scoring {o['score_seconds']:.1f} s); scoring against {s_note}; "
              + ("recpack's own get_top_K_values / ItemKNN._predict / NDCGK / RecallK from baseline/_ref on sklearn cosine_similarity row blocks"
                 if r.kind == "reference" else "oracle/recpack_oracle.py ref_* (recpack not importable)")
              + f"; 1 thread (the reference's sparse path is single-threaded) of {os.cpu_count()} host cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args, train, test_out),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": r.kind, "sample": sample,
                         "all_cores": {"value": v_all, "cores": procs,
                                       "sample": f"{procs} worker processes, one such step each, at once ({wall:.1f} s wall)"}},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "step_fraction_of_full_pass": f,
        "full_pass_seconds_estimate": U / v,
        "fit_seconds_full_pass_estimate": float(np.mean([x["fit_seconds"] for x in outs])) / f,
        "scoring_users_per_s": float(np.mean([x["users"] / x["score_seconds"] for x in outs])),
        "ndcg10_sample": float(o["ndcg10"]), "recall20_sample": float(o["recall20"]),
        "setup_seconds": t0 - t_start, "model_seconds": time.perf_counter() - t0,
    }
    _emit(line)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch

    # a user of the drop-in has recpack installed: with the reference on the path (baseline/_ref, installed by
    # baseline/install_ref.sh) the classes timed by the e2e leg SUBCLASS the reference's own (recpack_b200/_ref.py)
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "recpack")):
        for p_ in (os.path.join(ROOT, "baseline", "stubs"), ref_dir):
            if p_ not in sys.path:
                sys.path.insert(0, p_)

    from recpack_b200.distributed import ShardExchange, fit_work_per_item, score_work_per_user, shard_bounds
    from recpack_b200.engine import get_engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (recpack_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    train, test_out = make_data(args)
    U, I = train.shape
    K_NEIGH, SIM = args.K, args.similarity
    stats = workload_stats(train, K_NEIGH, N_LIST, test_out)
    eng = get_engine(local_rank)
    eng.use_torch_stream()

    # ---- shards: item rows for fit (balanced by popularity-weighted work), users for scoring (by history)
    d_u = np.diff(train.indptr).astype(np.float64)
    item_work = fit_work_per_item(train)
    icut = shard_bounds(item_work, world)
    ucut = shard_bounds(score_work_per_user(train, K_NEIGH), world)
    ib, ie = icut[rank], icut[rank + 1]
    ub, ue = ucut[rank], ucut[rank + 1]

    # ---- resident inputs
    t_ptr_full = torch.from_numpy(train.indptr.astype(np.int64)).to(dev)
    t_idx_full = torch.from_numpy(train.indices.astype(np.int32)).to(dev)
    my_ptr_h = train.indptr[ub:ue + 1].astype(np.int64)
    my_lo, my_hi = int(my_ptr_h[0]), int(my_ptr_h[-1])
    u_ptr = torch.from_numpy(my_ptr_h - my_lo).to(dev)
    u_idx = t_idx_full[my_lo:my_hi].contiguous()
    y_ptr_h = test_out.indptr[ub:ue + 1].astype(np.int64)
    y_ptr = torch.from_numpy(y_ptr_h - y_ptr_h[0]).to(dev)
    y_idx = torch.from_numpy(test_out.indices[int(y_ptr_h[0]):int(y_ptr_h[-1])].astype(np.int32)).to(dev)
    nU = ue - ub

    rows = ie - ib
    exchange = ShardExchange(icut, K_NEIGH, dev, dist) if world > 1 else None
    if world > 1:
        fit_out = exchange.local_out()  # the fit writes straight into the all-gather send buffers
    else:
        fit_out = {"idx": torch.empty((rows, K_NEIGH), dtype=torch.int32, device=dev), "cnt": None,
                   "val": torch.empty((rows, K_NEIGH), dtype=torch.float64, device=dev),
                   "len": torch.empty((rows,), dtype=torch.int32, device=dev)}
    top_out = {"idx": torch.empty((nU, N_LIST), dtype=torch.int32, device=dev), "val": None,
               "len": torch.empty((nU,), dtype=torch.int32, device=dev)}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.int32, device=dev)  # > L2 (126 MB)
    red_d = torch.zeros(3, dtype=torch.float64, device=dev)
    n_d = torch.zeros(1, dtype=torch.int64, device=dev)
    metrics = [("ndcg", 10), ("recall", 20)]
    phase_ms = {"fit": [], "exchange": [], "score": [], "gram_tc": [], "fit_rows": [], "predict": []}

    def one_step(record):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        eng.fit_topk(U, I, t_ptr_full, t_idx_full, K_NEIGH, similarity=SIM, item_begin=ib, item_end=ie, out=fit_out)
        ev[1].record()
        if world > 1:
            g_ent, g_len = exchange.gather_packed(eng)  # rows travel in the model's packed format
            eng.model_load_packed_rows_v(I, K_NEIGH, g_ent.shape[0], g_ent, g_len, exchange.vmax, exchange.row_source())
        else:
            eng.model_load_topk(I, K_NEIGH, fit_out["idx"], fit_out["val"], fit_out["len"])
        ev[2].record()
        eng.predict_topn(nU, u_ptr, u_idx, N_LIST, mask_history=True, out=top_out)
        # the metric sums stay on the device (no host round trip before the all-reduce): red = [sum NDCG, sum Recall, users]
        eng.metrics_topn(nU, N_LIST, top_out["idx"], top_out["len"], y_ptr, y_idx, metrics, want_per_user=False,
                         out_sums=red_d[:2], out_n_users=n_d)
        red_d[2:3].copy_(n_d)
        red = red_d
        if world > 1:
            dist.all_reduce(red)
        ev[3].record()
        torch.cuda.synchronize()
        if record:
            kt = eng.last_timings()
            phase_ms["gram_tc"].append(kt["gram_tc_ms"])
            phase_ms["fit_rows"].append(kt["fit_rows_ms"])
            phase_ms["predict"].append(kt["predict_ms"])
            phase_ms["dense_kd"] = kt["dense_kd"]
            phase_ms["dense_users"] = kt["dense_users"]
            phase_ms["fit"].append(ev[0].elapsed_time(ev[1]))
            phase_ms["exchange"].append(ev[1].elapsed_time(ev[2]))
            phase_ms["score"].append(ev[2].elapsed_time(ev[3]))
        return ev[0].elapsed_time(ev[3]), red.cpu().numpy()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        flush.fill_(1)
        one_step(False)
    sampler = ClockSampler(local_rank)
    launches0 = eng.launch_count()
    barrier()
    if rank == 0:
        sampler.start()
    step_ms = []
    red = None
    for _ in range(args.steps):
        flush.fill_(1)  # L2 flush between timed iterations (outside the event-timed region)
        barrier()
        ms, red = one_step(True)
        step_ms.append(ms)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        if world > 1:
            raise SystemExit("--dump-outputs needs a single process (--gpus 1)")
        dump_outputs(args.dump_outputs, fit_out, top_out, red)
    if args.trace:  # one more step with the library's marks on (after the timed region)
        eng.trace(True)
        one_step(False)
        rep = eng.trace_report()
        eng.trace(False)
        if rank == 0:
            sys.stderr.write("[trace of one step, rank 0: device ms since the previous mark]\n" + rep)
    launches = eng.launch_count() - launches0
    t = torch.tensor([float(np.sum(step_ms)), float(np.mean(phase_ms["fit"])), float(np.mean(phase_ms["score"])),
                      float(np.mean(phase_ms["exchange"]))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, fit_ms, score_ms, exch_ms = [float(x) for x in t.cpu().numpy()]
    ms_per_step = total_ms / args.steps
    n_eval = int(red[2])
    ndcg10, recall20 = float(red[0] / red[2]), float(red[1] / red[2])

    # ---- end to end through the public classes, host inputs (N = 1 rank-local: each rank does its shard)
    e2e = None
    if not args.no_e2e and world == 1:
        e2e = run_e2e(args, train, test_out, eng, steps=args.steps)
    elif not args.no_e2e:
        # N > 1: the same sharded step through the C ABI with HOST input buffers (pinned), every copy inside the
        # timed region, wall clock bracketed by barriers, max over ranks
        def pin(a):
            return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

        hx_ptr, hx_idx = pin(train.indptr.astype(np.int64)), pin(train.indices.astype(np.int32))
        hu_ptr, hu_idx = pin(my_ptr_h - my_lo), pin(train.indices[my_lo:my_hi].astype(np.int32))
        hy_ptr, hy_idx = pin(y_ptr_h - y_ptr_h[0]), pin(test_out.indices[int(y_ptr_h[0]):int(y_ptr_h[-1])].astype(np.int32))
        h2d_rank = sum(int(t.numel() * t.element_size()) for t in (hx_ptr, hx_idx, hu_ptr, hu_idx, hy_ptr, hy_idx))
        h_top_idx = torch.empty((nU, N_LIST), dtype=torch.int32).pin_memory()
        h_top_len = torch.empty((nU,), dtype=torch.int32).pin_memory()
        e_times = []
        e_red = None
        for s_ in range(args.steps + 1):
            barrier()
            t0 = time.perf_counter()
            eng.fit_topk(U, I, hx_ptr.numpy(), hx_idx.numpy(), K_NEIGH, similarity=SIM, item_begin=ib, item_end=ie, out=fit_out)
            g_ent, g_len = exchange.gather_packed(eng)
            eng.model_load_packed_rows_v(I, K_NEIGH, g_ent.shape[0], g_ent, g_len, exchange.vmax, exchange.row_source())
            eng.predict_topn(nU, hu_ptr.numpy(), hu_idx.numpy(), N_LIST, mask_history=True, out=top_out)
            sums, n_users, _ = eng.metrics_topn(nU, N_LIST, top_out["idx"], top_out["len"], hy_ptr.numpy(), hy_idx.numpy(), metrics,
                                                want_per_user=False)
            r_ = torch.tensor([sums[0], sums[1], float(n_users)], dtype=torch.float64, device=dev)
            dist.all_reduce(r_)
            e_red = r_.cpu().numpy()  # the step's result on the host
            h_top_idx.copy_(top_out["idx"], non_blocking=True)  # ... and this rank's top-N lists
            h_top_len.copy_(top_out["len"], non_blocking=True)
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            if s_ > 0:
                e_times.append(float(dt.item()))
        tot = torch.tensor([float(h2d_rank)], dtype=torch.float64, device=dev)
        dist.all_reduce(tot)
        te = float(np.median(e_times))
        e2e = {"value": U / te, "unit": UNIT, "seconds": te, "step_seconds": [round(x, 5) for x in e_times],
               "h2d_bytes_per_step": int(tot.item()), "d2h_bytes_per_step": int(U * (N_LIST * 4 + 4) + world * (2 * 8 + 8 + 24)),
               "ndcg10": float(e_red[0] / e_red[2]), "recall20": float(e_red[1] / e_red[2]),
               "path": "C ABI per rank with pinned host inputs (X, the rank's user rows, y_true); the rank's top-N lists and the "
                       "metric sums come back to the host; the top-K similarity lists stay on the device"}

    if rank == 0:
        peak, peak_src = measured_peaks()
        fit_frac_share = (ie - ib) / I
        k_gram, k_rows, k_pred = (float(np.mean(phase_ms[k])) for k in ("gram_tc", "fit_rows", "predict"))
        # measured DRAM bytes per launch come from an `ncu --set full` capture of THIS shape / configuration when one is
        # committed (profiles/r2_traffic.json, keyed "<shape>/<similarity>/K<k>/gpus<n>"); otherwise null
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(f"{args.shape}/{args.similarity}/K{args.K}/gpus{world}", {})
        # both big kernels against the HBM roofline: algorithmic bytes per launch (DESIGN.md 4.1 / 4.3) / CUDA-event time
        alg_pred = stats["score_bytes"] * (d_u[ub:ue].sum() / d_u.sum())
        alg_rows = stats["fit_bytes"] * (item_work[ib:ie].sum() / item_work.sum())
        notes = {
            "k_predict_a32": "algorithmic bytes per launch (SURVEY 8d: d_u*(4+8K)+8+8N+4*d_out per user) / CUDA-event duration of the "
                             "scoring kernels; S and X are L2-resident, so measured DRAM traffic is far below the algorithmic bytes: "
                             "the kernel is bound by instruction issue and the shared-memory pipe (one 32-bit atomic per similarity "
                             "entry), not by HBM",
            "k_fit_rows": "algorithmic bytes per launch (4 B per co-occurrence update + CSC + output lists) / CUDA-event duration of the "
                          "row kernels; X is L2-resident, the kernel is bound by instruction issue and shared-memory atomics, not by HBM",
        }
        per_kernel = []
        for nm_, ms_, alg_ in (("k_predict_a32", k_pred, alg_pred), ("k_fit_rows", k_rows, alg_rows)):
            if ms_ > 0:
                a_ = alg_ / (ms_ * 1e-3) / 1e9
                per_kernel.append({"bound": "hbm", "kernel": nm_, "achieved": a_, "peak": peak, "unit": "GB/s", "frac": a_ / peak,
                                   "traffic": traffic.get(nm_), "kernel_ms": ms_, "algorithmic_bytes": alg_, "note": notes[nm_]})
        dom = max(per_kernel, key=lambda r_: r_["kernel_ms"])
        kname, kms, ach = dom["kernel"], dom["kernel_ms"], dom["achieved"]
        tensor = None
        if k_gram > 0:
            bf16 = None
            mp = os.path.join(ROOT, "MEASURED_PEAKS.json")
            if os.path.exists(mp):
                with open(mp) as f:
                    bf16 = float(json.load(f)["bf16_tflops"])
            ops = 2.0 * phase_ms.get("dense_kd", 0) * (ie - ib) * I  # 2 * Kd * rows * I (Kd = dense users, padded to 128)
            tops = ops / (k_gram * 1e-3) / 1e12
            tensor = {"bound": "tensor", "kernel": "k_gram_i8_tc", "achieved": tops, "unit": "TOP/s (int8)", "ms": k_gram, "dense_users": phase_ms.get("dense_users", 0),
                      "peak": 2 * bf16 if bf16 else 4500.0,
                      "peak_source": "2 x measured bf16 cuBLAS burst (MEASURED_PEAKS.json): int8 issues at twice the bf16 rate" if bf16 else "nominal dense int8",
                      "frac": tops / (2 * bf16 if bf16 else 4500.0), "traffic": traffic.get("k_gram_i8_tc")}
        line = {
            "metric": METRIC, "value": U / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int32 counts / u64 fixed-point scores / f64 values", "data": "synthetic",
            "config": bench_config(args, train, test_out),
            "fit_seconds": fit_ms * 1e-3, "scoring_users_per_s": U / (score_ms * 1e-3), "exchange_ms": exch_ms,
            "ndcg10": ndcg10, "recall20": recall20, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": traffic.get(kname), "peak_source": peak_src, "kernel_ms": kms,
                         "note": notes[kname]},
            "roofline_kernels": per_kernel,
            "roofline_tensor": tensor,
            "phases_ms": {"fit": fit_ms, "exchange": exch_ms, "score": score_ms},
            "kernels_ms": {"k_gram_i8_tc": k_gram, "k_fit_rows": k_rows, "k_predict_a32": k_pred},
            "dense_equiv_int8_ops_per_s": stats["dense_equiv_ops"] * fit_frac_share / (fit_ms * 1e-3),
            "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if not args.no_cpu_baseline and world == 1:
            from recpack_b200.base import lists_to_csr

            S_host = lists_to_csr(fit_out["idx"].cpu().numpy(), fit_out["val"].cpu().numpy(), fit_out["len"].cpu().numpy(), I)
            S_host.sort_indices()
            line["cpu_baseline"] = cpu_baseline(args, train, test_out, S_host, args.ref_fraction, steps=1)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 60_000_000  # all files of --dump-outputs together stay below 64 MB (.npy headers included)


def dump_outputs(out_dir, fit_out, top_out, red):
    """What the last timed step computed, as DIR/<name>.npy in float64 (ids and counts are exact):

      metric_sums                          [sum of NDCG@10, sum of Recall@20, evaluated users]
      topn_users, topn_idx, topn_len       top-N lists (-1 padded) of every user, or of a seeded sample of users
      fit_items, fit_idx, fit_val, fit_len top-K similarity lists (-1 padded) of every item row, or of a seeded sample

    The samples depend only on the shape and the arguments, so two builds run with the same arguments write
    the same rows and their files can be compared one to one."""
    import torch

    os.makedirs(out_dir, exist_ok=True)

    def sample(n, row_bytes):
        keep = min(n, max(1, DUMP_BYTES // 2 // row_bytes))  # half for the top-N lists, half for the similarity lists
        if keep == n:
            return np.arange(n, dtype=np.int64)
        return np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))

    def rows_of(t, sel):
        return t[torch.from_numpy(sel).to(t.device)].cpu().numpy().astype(np.float64)

    nU, N = top_out["idx"].shape
    I, K = fit_out["idx"].shape
    users = sample(nU, 8 * (N + 2))
    items = sample(I, 8 * (2 * K + 2))
    arrays = {
        "metric_sums": np.asarray(red, dtype=np.float64),
        "topn_users": users.astype(np.float64), "topn_idx": rows_of(top_out["idx"], users), "topn_len": rows_of(top_out["len"], users),
        "fit_items": items.astype(np.float64), "fit_idx": rows_of(fit_out["idx"], items), "fit_val": rows_of(fit_out["val"], items),
        "fit_len": rows_of(fit_out["len"], items),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_e2e(args, train, test_out, eng, steps):
    """fit(X) -> predict(X) -> NDCGK/RecallK.calculate through the drop-in classes, scipy CSR inputs whose
    arrays live in pinned host memory; every copy is inside the timed region."""
    import warnings

    import torch
    from scipy.sparse import csr_matrix

    from recpack_b200 import ItemKNN, NDCGK, RecallK

    def pinned_arrays(M):
        ptr = torch.from_numpy(M.indptr.astype(np.int64)).pin_memory()
        idx = torch.from_numpy(M.indices.astype(np.int32)).pin_memory()
        dat = torch.ones(M.nnz, dtype=torch.int32).pin_memory()
        return ptr, idx, dat

    def fresh_csr(pins, shape):
        # a new matrix object over the same pinned arrays: the package memoises device copies per matrix
        # object, so every step uploads its inputs again
        ptr, idx, dat = pins
        out = csr_matrix((dat.numpy(), idx.numpy(), ptr.numpy()), shape=shape)
        out.has_canonical_format = True
        return out

    px, py = pinned_arrays(train), pinned_arrays(test_out)
    U, I = train.shape
    times = []
    for s in range(steps + 1):
        Xh, Yh = fresh_csr(px, train.shape), fresh_csr(py, test_out.shape)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            algo = ItemKNN(K=args.K, similarity=args.similarity, predict_topK=N_LIST, remove_history=True).fit(Xh)
            pred = algo.predict(Xh)
        m1, m2 = NDCGK(10), RecallK(20)
        m1.calculate(Yh, pred)
        m2.calculate(Yh, pred)
        v = (m1.value, m2.value)
        torch.cuda.synchronize()
        if s > 0:
            times.append(time.perf_counter() - t0)
        del algo, pred, m1, m2
    t = float(np.median(times))  # host-side timing: the median is robust against a stray slow step
    # inputs: X (fit and predict share one upload) and y_true (both metrics share one upload)
    h2d = (train.nnz * 4 + (U + 1) * 8) + (test_out.nnz * 4 + (U + 1) * 8)
    # results: the top-N prediction matrix (idx + val + len) and each metric's per-user values + sums.  The
    # top-K similarity lists stay on the device (similarity_matrix_ is built on first access, not here).
    d2h = U * N_LIST * 12 + U * 4 + 2 * (U * 8 + 16) + 8
    return {"value": U / t, "unit": UNIT, "seconds": t, "step_seconds": [round(x, 5) for x in times], "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "ndcg10": float(v[0]), "recall20": float(v[1]),
            "classes": "subclasses of recpack's ItemKNN / NDCGK / RecallK (reference importable from baseline/_ref)"
                       if _have_recpack() else "stand-alone mirror classes (recpack not importable)",
            "path": "drop-in classes: ItemKNN(...).fit(X) -> predict(X) -> NDCGK(10) / RecallK(20).calculate with scipy CSR inputs in pinned "
                    "host memory; the top-N prediction matrix (indices, scores) and the per-user metric values come back to the host",
            "note": "similarity_matrix_ is not materialised inside the timed region: the top-K lists stay on the device until the "
                    "attribute is first read (the reference's fit leaves S on the host; here that is 142 MB D2H + one CSR build on demand)"}


def _have_recpack():
    from recpack_b200 import _ref

    return bool(_ref.HAVE_RECPACK)


def _emit(line):
    """The JSON line is the only thing written to the real stdout (libraries such as NCCL print banners there)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # anything else that writes to fd 1 goes to stderr
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_gpu(a)
