"""Factor models on the GPU (rpk_factor_topn / _full / _screen_f32, FactorizationAlgorithm; DESIGN.md 2 "Factor
models" and 4.10).

Every comparison is bit for bit on idx, val and len against oracle.factor_oracle.canon_factor_topn.  The crafted cases
build one path each (exact ties, exact zeros -> the zero hand-off, items ordered by similarity -> buffer overflow and
the exact row kernel, a heavy history of the user's best items -> masked in the screen); with the instrumented build
(-DRPK_PHASE_PROF, one "[factor paths]" line per call) they also assert that the path's counter moved."""
import os
import pickle
import re
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.factor_oracle import canon_factor_full, canon_factor_scores, canon_factor_topn, factor_screen_delta

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    eng.predict_item_filter(None)
    yield eng
    eng.predict_item_filter(None)


def _paths(err):
    tot = {}
    for line in err.splitlines():
        if "[factor paths]" in line:
            for k, v in re.findall(r"([a-zA-Z][a-zA-Z ]*?)=(\d+)", line.split("]", 1)[1]):
                tot[k.strip()] = tot.get(k.strip(), 0) + int(v)
    return tot


def _moved(paths, name):
    if paths:  # instrumented build
        print(f"path counter {name!r}: {paths.get(name, 0)}")
        assert paths.get(name, 0) >= 1, (name, paths)


def _same(got, want, N):
    """got: lists of N; want: oracle lists of N' >= N (a prefix of the same total order)."""
    got = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in got.items()}
    assert np.array_equal(got["len"], np.minimum(want["len"], N))
    assert np.array_equal(got["idx"], want["idx"][:, :N])
    assert np.array_equal(got["val"], want["val"][:, :N])


def _csr(X):
    X = csr_matrix(X)
    return np.ascontiguousarray(X.indptr, dtype=np.int64), np.ascontiguousarray(X.indices, dtype=np.int32)


def _run(engine, capfd, P, Q, X, N, remove_history=True, allowed=None, want=None):
    ptr, idx = _csr(X)
    engine.predict_item_filter(None if allowed is None else np.asarray(allowed, dtype=np.uint8))
    capfd.readouterr()
    try:
        got = engine.factor_topn(P, Q, ptr, idx, N, mask_history=remove_history)
    finally:
        paths = _paths(capfd.readouterr().err)
        engine.predict_item_filter(None)
    if want is None:
        want = canon_factor_topn(P, Q, X, N, remove_history, allowed)
    _same(got, want, N)
    return paths


def _interactions(rng, U, I, density, empty_every=0):
    X = csr_matrix((rng.random((U, I)) < density).astype(np.float64))
    if empty_every:
        X[::empty_every] = 0
        X.eliminate_zeros()
    return X


@pytest.mark.parametrize("D", [1, 7, 64, 128, 300, 1024])
def test_gaussian(engine, capfd, D):
    rng = np.random.default_rng(D)
    U, I = (600, 3000) if D == 1024 else (1500, 5000)
    P, Q = rng.standard_normal((U, D)), rng.standard_normal((I, D))
    X = _interactions(rng, U, I, 0.01, empty_every=9)
    for rh in (False, True):
        want = canon_factor_topn(P, Q, X, 1024, rh)
        assert np.all(want["len"][::9] == 0)
        for N in (1, 10, 20, 200, 1024):
            _run(engine, capfd, P, Q, X, N, rh, want=want)


def test_item_filters(engine, capfd):
    from recpack_b200 import ExcludeItems, SelectItems
    from recpack_b200.postprocessing import combined_mask

    rng = np.random.default_rng(41)
    U, I, D = 800, 4000, 32
    P, Q = rng.standard_normal((U, D)), rng.standard_normal((I, D))
    X = _interactions(rng, U, I, 0.02)
    ex, sel = ExcludeItems(rng.choice(I, 1500, replace=False)), SelectItems(rng.choice(I, 2500, replace=False))
    for filters in ([ex], [sel], [ex, sel]):
        allowed = combined_mask(filters, I).astype(bool)
        for N in (10, 300):
            _run(engine, capfd, P, Q, X, N, True, allowed)


def test_ties_negative_scores_short_rows(engine, capfd):
    rng = np.random.default_rng(43)
    U, D = 700, 12
    B = rng.standard_normal((900, D))
    Q = np.concatenate([B, B, B[:300]])[rng.permutation(2100)]  # exact ties: duplicated item rows
    P = rng.standard_normal((U, D))
    X = _interactions(rng, U, 2100, 0.01, empty_every=5)
    for N in (5, 64, 1024):
        _run(engine, capfd, P, Q, X, N)
    # only negative scores: p >= 0, q <= 0
    _run(engine, capfd, np.abs(P) + 0.1, -np.abs(Q) - 0.1, X, 50)
    # fewer eligible stored scores than N: 300 items, most of them in the users' histories
    Xs = _interactions(rng, U, 300, 0.7)
    _run(engine, capfd, P, Q[:300], Xs, 200)


def test_exact_zeros_zero_handoff(engine, capfd):
    """Integer factors on disjoint blocks of dimensions: most scores are exactly 0.0 and users have fewer than N stored
    scores; I fits the first chunk, so the rows reach the exact pass, which hands them over."""
    rng = np.random.default_rng(47)
    U, I, D = 600, 1500, 40
    P, Q = np.zeros((U, D)), np.zeros((I, D))
    for M in (P, Q):
        for i in range(M.shape[0]):
            b = rng.integers(0, 10)
            M[i, 4 * b : 4 * b + 4] = rng.integers(-2, 3, size=4)
    X = _interactions(rng, U, I, 0.01)
    paths = _run(engine, capfd, P, Q, X, 400)
    _moved(paths, "zero handoffs")


def test_items_ordered_by_similarity_overflow(engine, capfd):
    """Items along a smooth curve in item order, users at points of the same curve: each user's best items sit next
    to each other, so the chunk that holds them appends almost every column and the row goes to the exact row kernel."""
    rng = np.random.default_rng(53)
    I, D = 6000, 8
    t = np.linspace(0, 3 * np.pi, I)[:, None]
    Q = np.concatenate([np.cos(t * (k + 1) / 4) for k in range(D)], axis=1) + 1e-3 * rng.standard_normal((I, D))
    P = Q[rng.choice(I, 400, replace=False)] + 1e-3 * rng.standard_normal((400, D))
    X = _interactions(rng, 400, I, 0.002)
    paths = _run(engine, capfd, P, Q, X, 50)
    _moved(paths, "overflow rows")
    _moved(paths, "exact rows")


def test_heavy_history_is_masked_in_the_screen(engine, capfd):
    """A user whose 20,000-item history is made of their highest-scoring items: those columns are never appended
    (masked-skip counter moves, no buffer overflows), and the list is the best of the remaining items."""
    rng = np.random.default_rng(59)
    U, I, D = 300, 30000, 64
    P, Q = rng.standard_normal((U, D)), rng.standard_normal((I, D))
    X = _interactions(rng, U, I, 0.001).tolil()
    s = canon_factor_scores(P, Q, [7])[0]
    X[7, :] = 0
    X[7, np.sort(np.argsort(-s)[:20000])] = 1
    X = csr_matrix(X)
    X.eliminate_zeros()
    assert X.indptr[8] - X.indptr[7] == 20000
    paths = _run(engine, capfd, P, Q, X, 100)
    _moved(paths, "masked skips")
    if paths:
        assert paths.get("overflow rows", 0) == 0, paths


def test_float32_torch_and_bad_input(engine):
    import torch

    from recpack_b200._lib import RpkError

    rng = np.random.default_rng(61)
    P = rng.standard_normal((500, 30)).astype(np.float32)
    Q = rng.standard_normal((900, 30)).astype(np.float32)
    X = _interactions(rng, 500, 900, 0.02, empty_every=4)
    ptr, idx = _csr(X)
    want = canon_factor_topn(P.astype(np.float64), Q.astype(np.float64), X, 12, True)
    for tp in (lambda a: a.astype(np.float64), lambda a: torch.from_numpy(a).double().cuda()):
        ptr_in, idx_in = (ptr, idx) if isinstance(tp(P[:1]), np.ndarray) else (torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda())
        _same(engine.factor_topn(tp(P), tp(Q), ptr_in, idx_in, 12), want, 12)
    Pf = P.astype(np.float64)
    Qf = Q.astype(np.float64)
    for bad in (np.nan, np.inf, -np.inf):
        F = Pf.copy()
        F[17, 2] = bad
        with pytest.raises(RpkError):
            engine.factor_topn(F, Qf, ptr, idx, 5)
        G = Qf.copy()
        G[3, 1] = bad
        with pytest.raises(RpkError):
            engine.factor_full(Pf, G, ptr, idx)
    with pytest.raises(RpkError):
        engine.factor_topn(np.full((500, 3), 1e300), np.ascontiguousarray(Qf[:, :3]), ptr, idx, 3)  # squared norms overflow
    for N in (0, 1025):
        with pytest.raises(RpkError):
            engine.factor_topn(Pf, Qf, ptr, idx, N)
    with pytest.raises(RpkError):  # columns out of range
        engine.factor_topn(np.ascontiguousarray(Pf[:, :5]), np.ascontiguousarray(Qf[:800, :5]), ptr, idx, 5)
    unsorted = idx.copy()
    r = int(np.argmax(np.diff(ptr)))
    unsorted[ptr[r] : ptr[r + 1]] = unsorted[ptr[r] : ptr[r + 1]][::-1]
    with pytest.raises(RpkError):
        engine.factor_topn(Pf, Qf, ptr, unsorted, 5)
    with pytest.raises(RpkError):
        engine.factor_topn(np.zeros((500, 1025)), np.zeros((900, 1025)), ptr, idx, 5)


@pytest.mark.parametrize("D", [7, 128, 1024])
def test_screen_bound_on_the_hardware(engine, D):
    rng = np.random.default_rng(67 + D)
    U = I = 4000
    P = rng.standard_normal((U, D)) * np.exp2(rng.integers(-10, 10, size=(U, 1)) + 40)
    Q = rng.standard_normal((I, D)) * np.exp2(rng.integers(-10, 10, size=(I, 1)) - 40)
    S_hat = engine.factor_screen_f32(P, Q).astype(np.float64)
    S = canon_factor_scores(P, Q, np.arange(U))
    ratio = np.abs(S_hat - S) / factor_screen_delta(P, Q)
    print(f"factor screen D={D}: largest |s^ - s| / delta = {ratio.max():.4f}")
    assert np.all(ratio <= 1.0)


def test_full_scores_with_masks(engine):
    rng = np.random.default_rng(71)
    U, I, D = 400, 700, 19
    P, Q = rng.standard_normal((U, D)), rng.standard_normal((I, D))
    P[5] = 0.0
    X = _interactions(rng, U, I, 0.03, empty_every=6)
    ptr, idx = _csr(X)
    allowed = np.ones(I, dtype=bool)
    allowed[::3] = False
    for rh in (False, True):
        for ok in (None, allowed):
            engine.predict_item_filter(None if ok is None else ok.astype(np.uint8))
            try:
                got = engine.factor_full(P, Q, ptr, idx, mask_history=rh)
            finally:
                engine.predict_item_filter(None)
            assert np.array_equal(got, canon_factor_full(P, Q, X, rh, ok))


def _algo(P, Q, **kw):
    from recpack_b200 import FactorizationAlgorithm

    a = FactorizationAlgorithm(num_components=P.shape[1], **kw)
    a.user_embedding_, a.item_embedding_ = P, Q
    return a


def test_class_predict_metrics_pickle(engine):
    from recpack_b200 import NDCGK, RecallK, ExcludeItems
    from oracle.recpack_oracle import canon_metrics_from_lists

    rng = np.random.default_rng(73)
    U, I, D = 900, 1200, 16
    P, Q = rng.standard_normal((U, D)), rng.standard_normal((I, D)).astype(np.float32)
    P[3] = 0.0  # every score 0.0: an empty row and the warning
    X = _interactions(rng, U, I, 0.02, empty_every=10)
    X[3, 0] = 1.0
    y_true = _interactions(rng, U, I, 0.01)
    Qd = Q.astype(np.float64)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        full = _algo(P, Q).predict(X)
    assert any("failed to recommend any items for 1 users" in str(m.message) for m in w)
    want = csr_matrix(canon_factor_full(P, Qd, X))
    full.sort_indices()
    assert np.array_equal(full.indptr, want.indptr) and np.array_equal(full.indices, want.indices)
    assert np.array_equal(full.data, want.data)

    banned = np.arange(0, I, 11)
    allowed = np.ones(I, dtype=bool)
    allowed[banned] = False
    algo = _algo(P, Q, predict_topK=20, remove_history=True).set_postfilters([ExcludeItems(banned)])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        top = algo.predict(X)
    ref = canon_factor_topn(P, Qd, X, 20, True, allowed)
    assert top._rpk_topn_dev is not None
    assert np.array_equal(np.diff(top.indptr), ref["len"])
    assert np.array_equal(top._rpk_topn[0], ref["idx"])
    want_m = canon_metrics_from_lists(ref["idx"], ref["len"], y_true, [("ndcg", 10), ("recall", 20)])
    for M, key in ((NDCGK(10), ("ndcg", 10)), (RecallK(20), ("recall", 20))):
        M.calculate(y_true, top)
        assert M.value == pytest.approx(want_m[key][0], rel=1e-12, abs=1e-15)

    clone = pickle.loads(pickle.dumps(algo))
    assert clone.__dict__.get("_factors_dev") is None
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        again = clone.predict(X)
    assert np.array_equal(again.indices, top.indices) and np.array_equal(again.data, top.data)
    with pytest.raises(AssertionError):
        algo.predict(X[:, :1000])
    with pytest.raises(ValueError):
        _algo(P, Q, predict_topK=1025).predict(X)


def test_reference_dropins():
    """With the reference installed (baseline/_ref): SVD / NMF drop-ins fit by the reference's own _fit score like the
    canonical lists, the reference's own _predict agrees tie-aware, and its registry accepts them."""
    from recpack_b200 import _ref

    if not _ref.HAVE_RECPACK:
        pytest.skip("recpack (baseline/_ref) not importable")
    import recpack_b200
    from recpack_b200 import factorization

    rng = np.random.default_rng(79)
    X = _interactions(rng, 300, 200, 0.05)
    for name in ("SVD", "NMF"):
        assert name in factorization.__all__, factorization.__all__
        cls = getattr(recpack_b200, name)
        base = next(b for b in cls.__mro__[1:] if b.__name__ == name)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            algo = cls(num_components=8).fit(X)
            algo.predict_topK, algo.remove_history = 10, True
            top = algo.predict(X)
            ref_full = csr_matrix(base._predict(algo, X))
        P = np.asarray(algo.user_embedding_, dtype=np.float64)
        Q = np.asarray(algo.item_embedding_, dtype=np.float64)
        want = canon_factor_topn(P, Q, X, 10, True)
        assert np.array_equal(top._rpk_topn[0], want["idx"])
        canon = csr_matrix(canon_factor_full(P, Q, X))
        assert np.array_equal(canon.indptr, ref_full.indptr)
        r, c = canon.nonzero()
        tol = 4 * (P.shape[1] + 2) * 2.0**-53 * np.linalg.norm(P, axis=1)[r] * np.linalg.norm(Q, axis=1)[c]
        assert np.all(np.abs(canon.data - np.asarray(ref_full[r, c]).ravel()) <= tol)
        from recpack.pipelines import ALGORITHM_REGISTRY

        sub = type(name + "B200", (cls,), {})
        if sub.__name__ not in ALGORITHM_REGISTRY:
            ALGORITHM_REGISTRY.register(sub.__name__, sub)
        assert sub.__name__ in ALGORITHM_REGISTRY


def test_full_size_ml25m(engine):
    import torch

    from recpack_b200.synth import make_dataset

    engine.predict_item_filter(None)  # a class predict above leaves its post-filter set on the process-wide engine
    train, _, _ = make_dataset("ml25m", seed=0)
    X = csr_matrix(train)
    X.sort_indices()
    U, I = X.shape
    D, N = 128, 20
    rng = np.random.default_rng(83)
    P, Q = rng.standard_normal((U, D)), rng.standard_normal((I, D))
    dev = torch.device("cuda", 0)
    ptr, idx = (torch.from_numpy(a).to(dev) for a in _csr(X))
    got = engine.factor_topn(torch.from_numpy(P).to(dev), torch.from_numpy(Q).to(dev), ptr, idx, N, mask_history=True)
    gi, gv, gl = got["idx"].long(), got["val"], got["len"].long()
    has = (ptr[1:] - ptr[:-1]) > 0
    assert torch.equal(gl, torch.where(has, N, 0))
    pos = torch.arange(N, device=dev)[None, :] < gl[:, None]
    v0, v1, i0, i1 = gv[:, :-1], gv[:, 1:], gi[:, :-1], gi[:, 1:]
    ordered = (v0 > v1) | ((v0 == v1) & (i0 < i1)) | ~pos[:, 1:]
    assert bool(ordered.all())
    # no history item: every listed (user, item) pair is absent from X
    users = torch.arange(U, device=dev)[:, None].expand(U, N)[pos]
    items = gi[pos]
    key = users * I + items
    hist_users = torch.repeat_interleave(torch.arange(U, device=dev), ptr[1:] - ptr[:-1])
    hist_key = torch.sort(hist_users * I + idx.long()).values
    at = torch.searchsorted(hist_key, key).clamp(max=hist_key.numel() - 1)
    assert not bool((hist_key[at] == key).any())
    sample = np.sort(rng.choice(U, size=1000, replace=False))
    want = canon_factor_topn(P, Q, X, N, True, users=sample)
    for k in ("idx", "val", "len"):
        assert np.array_equal(got[k].cpu().numpy()[sample], want[k])
