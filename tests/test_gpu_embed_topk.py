"""Item neighbours of dense embeddings on the GPU (rpk_embed_topk, DESIGN.md 2 "Embedding neighbours" and 4.9).

Every comparison is bit for bit on idx, val and len against oracle.embed_oracle.canon_embed_topk.  The crafted cases
build one path each (exact ties, exact zeros -> the zero hand-off, rows ordered by similarity -> buffer overflow and
the exact row kernel); with the instrumented build (-DRPK_PHASE_PROF, one "[embed paths]" line per call) they also
assert that the path's counter moved."""
import re
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.embed_oracle import canon_block, canon_embed_topk, canon_rows, screen_delta, screen_scale
from oracle.signed_oracle import canon_predict_signed

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.predict_item_filter(None)  # the post-filter of the end-to-end case stays set on the process-wide engine


def _paths(err):
    tot = {}
    for line in err.splitlines():
        if "[embed paths]" in line:
            for k, v in re.findall(r"([a-zA-Z][a-zA-Z ]*?)=(\d+)", line.split("]", 1)[1]):
                tot[k.strip()] = tot.get(k.strip(), 0) + int(v)
    return tot


def _moved(paths, name):
    if paths:  # instrumented build
        print(f"path counter {name!r}: {paths.get(name, 0)}")
        assert paths.get(name, 0) >= 1, (name, paths)


def _same(got, want, K):
    """got: lists of K; want: oracle lists of K' >= K (a prefix of the same total order)."""
    assert np.array_equal(got["len"], np.minimum(want["len"], K))
    assert np.array_equal(got["idx"], want["idx"][:, :K])
    assert np.array_equal(got["val"], want["val"][:, :K])


def _run(engine, capfd, E, K, similarity, want=None):
    capfd.readouterr()
    got = engine.embed_topk(E, K, similarity)
    paths = _paths(capfd.readouterr().err)
    _same(got, canon_embed_topk(E, K, similarity) if want is None else want, K)
    return paths


@pytest.mark.parametrize("D", [1, 7, 64, 128, 300, 1024])
@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_gaussian(engine, capfd, D, similarity):
    E = np.random.default_rng(D).standard_normal((5000, D))
    want = canon_embed_topk(E, 1024, similarity)
    for K in (1, 10, 200, 1024):
        _run(engine, capfd, E, K, similarity, want)


@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_k_covers_the_row(engine, capfd, similarity):
    """K >= I - 1: every stored value of the row, in order."""
    E = np.random.default_rng(3).standard_normal((700, 20))
    want = canon_embed_topk(E, 1024, similarity)
    for K in (699, 1024):
        _run(engine, capfd, E, K, similarity, want)


@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_ties_negations_zero_rows(engine, capfd, similarity):
    rng = np.random.default_rng(5)
    B = rng.standard_normal((1000, 33))
    E = np.concatenate([B, B, -B, np.zeros((200, 33))])[rng.permutation(3200)]
    for K in (5, 64):
        _run(engine, capfd, E, K, similarity)


@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_exact_zeros_zero_handoff(engine, capfd, similarity):
    """Integer embeddings in orthogonal blocks: most pairs are exactly 0.0 and rows have fewer than K stored values.
    I fits the first chunk, so no buffer overflows and the rows reach the exact pass, which hands them over."""
    rng = np.random.default_rng(7)
    I, D = 1500, 40  # 10 groups of ~150 items, each group on its own 4 of the 40 dimensions
    E = np.zeros((I, D))
    for i in range(I):
        b = rng.integers(0, 10)
        E[i, 4 * b : 4 * b + 4] = rng.integers(-2, 3, size=4)
    paths = _run(engine, capfd, E, 400, similarity)
    _moved(paths, "zero handoffs")


@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_rows_ordered_by_similarity_overflow(engine, capfd, similarity):
    """Items along a smooth curve in item order: each row's neighbours sit next to it, so the chunk that holds them
    appends almost every column and the row goes to the exact row kernel."""
    rng = np.random.default_rng(9)
    I, D = 6000, 8
    t = np.linspace(0, 3 * np.pi, I)[:, None]
    E = np.concatenate([np.cos(t * (k + 1) / 4) for k in range(D)], axis=1) + 1e-3 * rng.standard_normal((I, D))
    paths = _run(engine, capfd, E, 50, similarity)
    _moved(paths, "overflow rows")
    _moved(paths, "exact rows")


def test_dot_norms_spread_and_odd_d(engine, capfd):
    rng = np.random.default_rng(13)
    I, D = 3000, 13
    E = rng.standard_normal((I, D)) * np.exp2(rng.uniform(-60, 60, size=(I, 1)))
    for K in (1, 37, 300):
        _run(engine, capfd, E, K, "dot")


@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_shards_concatenate(engine, similarity):
    E = np.random.default_rng(17).standard_normal((4100, 48))
    full = engine.embed_topk(E, 25, similarity)
    a = 1337
    lo = engine.embed_topk(E, 25, similarity, item_begin=0, item_end=a)
    hi = engine.embed_topk(E, 25, similarity, item_begin=a, item_end=4100)
    for k in ("idx", "val", "len"):
        assert np.array_equal(np.concatenate([lo[k], hi[k]]), full[k])
    empty = engine.embed_topk(E, 25, similarity, item_begin=a, item_end=a)
    assert empty["idx"].shape == (0, 25)


def test_torch_inputs(engine):
    import torch

    from recpack_b200 import embedding_top_k

    E = np.random.default_rng(19).standard_normal((900, 30)).astype(np.float32)
    want = canon_embed_topk(E.astype(np.float64), 12, "cosine")
    for src in (E, torch.from_numpy(E), torch.from_numpy(E).cuda()):
        S = embedding_top_k(src, 12)
        assert S.shape == (900, 900)
        assert np.array_equal(np.diff(S.indptr), want["len"])
        assert np.array_equal(S.indices, want["idx"][want["idx"] >= 0])
        assert np.array_equal(S.data, want["val"][want["idx"] >= 0])


@pytest.mark.parametrize("similarity,D", [("cosine", 128), ("dot", 128), ("cosine", 1024), ("dot", 7)])
def test_screen_bound_on_the_hardware(engine, similarity, D):
    rng = np.random.default_rng(23 + D)
    I = 4000
    E = rng.standard_normal((I, D))
    if similarity == "dot":
        E *= np.exp2(rng.integers(-10, 10, size=(I, 1)))
    S_hat = engine.embed_screen_f32(E, similarity).astype(np.float64)
    X = canon_rows(E, similarity)
    S = canon_block(X, np.arange(I))
    ratio = np.abs(S_hat - S) / screen_delta(X, screen_scale(X))
    print(f"screen D={D} {similarity}: largest |s^ - s| / delta = {ratio.max():.4f}")
    assert np.all(ratio <= 1.0)


def test_rejects_bad_input(engine):
    from recpack_b200._lib import RpkError

    E = np.random.default_rng(29).standard_normal((50, 4))
    for bad in (np.nan, np.inf, -np.inf):
        F = E.copy()
        F[17, 2] = bad
        with pytest.raises(RpkError):
            engine.embed_topk(F, 5)
    with pytest.raises(RpkError):
        engine.embed_topk(np.full((10, 3), 1e300), 3, "dot")  # squared norms overflow
    for K in (0, 1025):
        with pytest.raises(RpkError):
            engine.embed_topk(E, K)
    with pytest.raises(RpkError):
        engine.embed_topk(np.zeros((10, 1025)), 3)
    with pytest.raises(RpkError):
        engine.embed_topk(E, 5, item_begin=10, item_end=5)
    with pytest.raises(RpkError):
        engine.embed_topk(E, 5, item_begin=0, item_end=51)
    with pytest.raises(RpkError):  # D = 0
        engine._check(engine._lib.rpk_embed_topk(engine._h, 50, 0, E.ctypes.data, 0, 5, 0, 50, np.zeros(250, np.int32).ctypes.data,
                                                 None, np.zeros(50, np.int32).ctypes.data))
    with pytest.raises(RpkError):  # unknown similarity
        engine._check(engine._lib.rpk_embed_topk(engine._h, 50, 4, E.ctypes.data, 1, 5, 0, 50, np.zeros(250, np.int32).ctypes.data,
                                                 None, np.zeros(50, np.int32).ctypes.data))


def test_end_to_end_scoring(engine):
    from recpack_b200 import ExcludeItems, ItemSimilarityMatrixAlgorithm, embedding_top_k

    class EmbeddingModel(ItemSimilarityMatrixAlgorithm):
        def __init__(self, S, predict_topK=None, remove_history=False):
            super().__init__()
            self.similarity_matrix_ = S
            self.predict_topK = predict_topK
            self.remove_history = remove_history

        def _fit(self, X):
            return self

    rng = np.random.default_rng(31)
    I = 180  # K = 100 of 179 neighbours: the model holds negative values and is scored in float64
    E = rng.standard_normal((I, 16))
    S = embedding_top_k(E, 100)
    assert np.any(S.data < 0)
    X = csr_matrix((rng.random((400, I)) < 0.05).astype(np.float64))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        full = EmbeddingModel(S).predict(X)
    want = csr_matrix(X @ S)
    want.sort_indices()
    full = csr_matrix(full)
    full.sort_indices()
    assert np.array_equal(full.indptr, want.indptr) and np.array_equal(full.indices, want.indices)
    assert np.array_equal(full.data, want.data)

    banned = np.arange(0, I, 7)
    allowed = np.ones(I, dtype=bool)
    allowed[banned] = False
    algo = EmbeddingModel(S, 20, True).set_postfilters([ExcludeItems(banned)])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        top = algo.predict(X)
    w = canon_predict_signed(X, S, 20, remove_history=True, allowed=allowed)
    assert np.array_equal(np.diff(top.indptr), w["len"])
    for u in range(X.shape[0]):
        lo, hi = top.indptr[u], top.indptr[u + 1]
        assert np.array_equal(top.indices[lo:hi], w["idx"][u, : w["len"][u]])
        assert np.array_equal(top.data[lo:hi], w["val"][u, : w["len"][u]])


def test_full_size_cosine(engine):
    import torch

    I, D, K = 200_000, 128, 100
    rng = np.random.default_rng(37)
    E = rng.standard_normal((I, D))
    got = engine.embed_topk(torch.from_numpy(E).cuda(), K, "cosine")
    idx, val, ln = (got[k].cpu().numpy() for k in ("idx", "val", "len"))
    assert np.all(ln == K)
    assert np.all(idx != np.arange(I)[:, None])
    assert np.all(val != 0.0)
    assert np.all((val[:, :-1] > val[:, 1:]) | ((val[:, :-1] == val[:, 1:]) & (idx[:, :-1] < idx[:, 1:])))
    rows = np.sort(rng.choice(I, size=2000, replace=False))
    want = canon_embed_topk(E, K, "cosine", rows=rows)
    assert np.array_equal(idx[rows], want["idx"])
    assert np.array_equal(val[rows], want["val"])
    assert np.array_equal(ln[rows], want["len"])
