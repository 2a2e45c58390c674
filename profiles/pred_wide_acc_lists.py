# Device time of the two-limb top-N kernel (k_predict) when it scores every user: lists only, N = 20, history
# masked, DBG_WIDE_ACC, at a bench shape.  No benchmark workload runs this; it stands for the large-model fallback
# (a block table beyond 32 bits) and sets the duration of test_lists_only_full_size.  To compare two builds, run
# the script once per library:
#   RPK_LIB=<librpk.so> python profiles/pred_wide_acc_lists.py [shape] [calls]
# It prints predict_ms (CUDA events around the scoring kernels) of every call after a warm-up call.
import os
import sys

sys.path.insert(0, ".")
from recpack_b200.engine import get_engine
from recpack_b200.matrix import binary_structure
from recpack_b200.synth import make_dataset

DBG_WIDE_ACC = 1
shape = sys.argv[1] if len(sys.argv) > 1 else "ml25m"
calls = int(sys.argv[2]) if len(sys.argv) > 2 else 5
train, _, _ = make_dataset(shape, seed=0, split_seed=42, generator="auto")
X, indptr, indices = binary_structure(train)
U, I = X.shape
eng = get_engine()
fit = eng.fit_topk(U, I, indptr, indices, 200)
eng.model_load_topk(I, 200, fit["idx"], fit["val"], fit["len"])
times = {}
for flags in (0, DBG_WIDE_ACC):
    eng.debug_flags(flags)
    eng.predict_topn(U, indptr, indices, 20, mask_history=True, want_val=False)
    times[flags] = []
    for _ in range(calls):
        eng.predict_topn(U, indptr, indices, 20, mask_history=True, want_val=False)
        eng.sync()
        times[flags].append(eng.last_timings()["predict_ms"])
eng.debug_flags(0)
lib = os.environ.get("RPK_LIB", "in-tree librpk.so")
for flags, t in times.items():
    print(f"{shape} U={U} I={I} N=20 lists only flags={flags} lib={lib}: predict_ms "
          + " ".join(f"{v:.2f}" for v in t) + f"  (median {sorted(t)[len(t) // 2]:.2f})")
