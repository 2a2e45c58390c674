# Phase profile of the top-N scoring kernel in lists-only mode (the metrics path of bench.py) at a bench shape.
# Run with an instrumented library: make -C recpack_b200/csrc EXTRA=-DRPK_PHASE_PROF into a separate build, then
#   RPK_LIB=<that librpk.so> python profiles/pred_phase_lists.py [shape]
# The kernel prints its phases (cycles of thread 0 per user or work item) to stderr after every call.
import sys

sys.path.insert(0, ".")
from recpack_b200.engine import get_engine
from recpack_b200.matrix import binary_structure
from recpack_b200.synth import make_dataset

shape = sys.argv[1] if len(sys.argv) > 1 else "ml25m"
train, _, _ = make_dataset(shape, seed=0, split_seed=42, generator="auto")
X, indptr, indices = binary_structure(train)
U, I = X.shape
eng = get_engine()
fit = eng.fit_topk(U, I, indptr, indices, 200)
eng.model_load_topk(I, 200, fit["idx"], fit["val"], fit["len"])
for _ in range(2):
    eng.predict_topn(U, indptr, indices, 20, mask_history=True, want_val=False)
