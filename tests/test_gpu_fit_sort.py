"""The fit's finishing kernel (k_fit_sort_rows, fit.cu): the exact top K of the survivors k_fit_rows defers, and the
similarity values of every row.

  sort order           the float64 sort key decides only where it provably agrees with the exact order; every other
                       comparison goes to the exact one (128-bit c^2 n_j products, or the untruncated float64 key), then
                       to the index.  DBG_COARSE_SORT_KEY keeps 24 bits of each key and widens the margin to 2^40 bit
                       patterns, so almost every comparison is settled exactly: the results must not move.
  values               a cosine value is the c-fold left sum of fl(a_i a_j) (scipy's csr_matmat order), taken in
                       O(log c) real additions: every step inside one binade of the running sum adds the same
                       increment once a step inside that binade has been taken.  A numpy mirror of that loop against
                       the one-at-a-time sum (no device needed), and a fit whose counts cross many binades.

With the instrumented build (-DRPK_PHASE_PROF, which prints one "[fit sort]" line per fit call), the coarse-key cases
also check that the exact-comparison counter moved."""
import re
import struct

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from conftest import load_golden, unpack
from oracle import recpack_oracle as orc

DBG_TINY_LIST, DBG_MULTI_PASS, DBG_COARSE_SORT_KEY = 2, 4, 64


# ---------------------------------------------------------------------------------------------------------------
# the O(log c) repeated sum, mirrored on the host


def _bits(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


def _double(b):
    return struct.unpack("<d", struct.pack("<q", b))[0]


def _repeat_sum(x, c):
    """repeat_sum of fit.cu in Python floats (IEEE float64, round to nearest even)."""
    s, r = 0.0, 0
    while r < c:
        s0 = s
        s = s + x
        r += 1
        b = _bits(s)
        if r == c or s0 == 0.0 or (_bits(s0) >> 52) != (b >> 52):
            continue
        s1 = s + x
        r += 1
        b1 = _bits(s1)
        s = s1
        if r == c or (b1 >> 52) != (b >> 52):
            continue
        d = b1 - b
        room = (((b >> 52) + 1) << 52) - 1 - b1
        t = c - r
        if d > 0 and room // d < t:
            t = room // d
        s = _double(b1 + t * d)
        r += t
    return s


def _check_mirror(x, c):
    got = np.array([_repeat_sum(float(a), int(k)) for a, k in zip(x, c)])
    want = orc.seq_sum(x, c)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{len(bad)} mismatches, first x={x[bad[0]]!r} c={c[bad[0]]}"


def test_repeat_sum_mirror_matches_the_sequential_sum():
    rng = np.random.default_rng(1)
    # cosine-shaped products fl(fl(1/sqrt(n_i)) fl(1/sqrt(n_j)))
    ni = rng.integers(1, 200_000, size=1500)
    nj = rng.integers(1, 200_000, size=1500)
    x = (1.0 / np.sqrt(ni.astype(np.float64))) * (1.0 / np.sqrt(nj.astype(np.float64)))
    c = np.minimum(rng.integers(1, 30_000, size=1500), np.minimum(ni, nj))
    _check_mirror(x, c)
    # exact half-ulp ties: odd mantissas scaled so that the last bit falls at half an ulp of many partial sums
    m = rng.integers(1, 1 << 20, size=1500) * 2 + 1
    x = np.ldexp(m.astype(np.float64), -rng.integers(20, 60, size=1500))
    c = rng.integers(1, 20_000, size=1500)
    _check_mirror(x, c)
    # arbitrary x, small c; and every c below 3,000 for one x
    x = rng.random(2000) * 10.0 ** rng.integers(-12, 3, size=2000)
    c = rng.integers(1, 64, size=2000)
    _check_mirror(x, c)
    x1 = (1.0 / np.sqrt(7919.0)) * (1.0 / np.sqrt(104729.0))
    _check_mirror(np.full(2999, x1), np.arange(1, 3000))
    # increments that vanish (x below half an ulp of the sum) and exactly half an ulp
    _check_mirror(np.array([1.0, 2.0 ** -53, 1.0 + 2.0 ** -52]), np.array([5, 7, 9]))
    assert _repeat_sum(2.0 ** -53, 1 << 60) == 2.0 ** -53 * (1 << 53)  # the sum stops growing at 1.0


# ---------------------------------------------------------------------------------------------------------------
# GPU: coarse sort keys leave every output unchanged


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.debug_flags(0)
    eng.fit_config(-1)


class ExactCount:
    """Sums the exact-comparison counter of the "[fit sort]" lines; nothing to check under the normal build."""

    def __init__(self):
        self.total, self.lines = 0, 0

    def add(self, text):
        for line in text.splitlines():
            if line.startswith("[fit sort]"):
                self.lines += 1
                self.total += int(re.search(r"\bexact_cmp=(\d+)", line).group(1))

    def require_moved(self):
        if not self.lines:
            print("exact-comparison counter: no [fit sort] line (normal build), not checked")
            return
        print(f"exact comparisons: {self.total} in {self.lines} fit calls")
        assert self.total > 0


def _fit(engine, capfd, X, K, sim="cosine", pd_=None, flags=0, count=None):
    from recpack_b200.matrix import binary_structure

    Xc, indptr, indices = binary_structure(X)
    U, I = Xc.shape
    item_pow = None
    if sim == "conditional_probability" and pd_:
        n = np.bincount(indices, minlength=I)
        item_pow = np.zeros(I)
        item_pow[n > 0] = np.power(1 / n[n > 0], pd_)
    out = {"idx": np.full((I, K), -2, np.int32), "cnt": np.full((I, K), -3, np.int32),
           "val": np.full((I, K), np.nan), "len": np.full(I, -4, np.int32)}
    capfd.readouterr()
    engine.debug_flags(flags)
    try:
        engine.fit_topk(U, I, indptr, indices, K, similarity=sim, item_pow=item_pow, out=out)
        engine.sync()
    finally:
        engine.debug_flags(0)
    if count is not None:
        count.add(capfd.readouterr().err)
    return out


def _same(got, want, what):
    for key in ("len", "idx", "cnt", "val"):
        bad = np.flatnonzero(np.any((got[key] != want[key]).reshape(len(got[key]), -1), axis=1))
        assert len(bad) == 0, f"{what}: {key} differs in {len(bad)} rows, first {bad[:8].tolist()}"


COARSE = [DBG_COARSE_SORT_KEY, DBG_COARSE_SORT_KEY | DBG_TINY_LIST, DBG_COARSE_SORT_KEY | DBG_MULTI_PASS]
SYNTH = [
    # U, I, nnz, K, similarity, pop_discount (cases of test_gpu_parity.py)
    (500, 300, 9000, 50, "cosine", None),
    (943, 1682, 100_000, 200, "cosine", None),
    (500, 300, 9000, 50, "conditional_probability", 0.3),
    (60, 2000, 6000, 100, "conditional_probability", None),
    (60, 2000, 6000, 100, "cosine", None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("flags", COARSE)
def test_coarse_keys_golden_and_synthetic(engine, capfd, flags):
    count = ExactCount()
    for name in ("unit_cosine", "unit_condprob_pd0.5", "small_cosine", "small_condprob", "small_condprob_pd"):
        g = load_golden(name)
        pd_ = float(g["pop_discount"]) if "pop_discount" in g else float("nan")
        pd_ = None if np.isnan(pd_) else pd_
        sim = str(g["similarity"]) if "similarity" in g else "cosine"
        X = unpack(g, "X")
        K = int(g["K"])
        _same(_fit(engine, capfd, X, K, sim, pd_, flags, count), orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_),
              f"{name} flags={flags}")
    from recpack_b200.synth import synth_interactions

    for U, I, nnz, K, sim, pd_ in SYNTH:
        X = synth_interactions(U, I, nnz, seed=U + I)
        _same(_fit(engine, capfd, X, K, sim, pd_, flags, count), orc.canon_fit(X, K=K, similarity=sim, pop_discount=pd_),
              f"synthetic {U}x{I} {sim} flags={flags}")
    if flags == DBG_COARSE_SORT_KEY:  # the other two sort inside the row kernel or merge: no row is deferred
        count.require_moved()


@pytest.mark.gpu
def test_coarse_keys_total_ties(engine, capfd):
    """Every pair ties (3 users saw all 700 items): the lowest indices, whatever settles the comparisons."""
    I, K = 700, 40
    X = csr_matrix(np.ones((3, I), dtype=np.int32))
    count = ExactCount()
    for sim in ("cosine", "conditional_probability"):
        for flags in (0, DBG_COARSE_SORT_KEY):
            got = _fit(engine, capfd, X, K, sim, flags=flags, count=count)
            _same(got, orc.canon_fit(X, K=K, similarity=sim), f"total ties {sim} flags={flags}")
    count.require_moved()


@pytest.mark.gpu
@pytest.mark.parametrize("similarity,K", [("cosine", 200), ("conditional_probability", 100)])
def test_coarse_keys_mid_shape_every_row(engine, capfd, similarity, K):
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(40000, 8000, 1_200_000, seed=21)  # the matrix of test_mid_shape_every_row
    prep = orc.prepare(X)
    want = orc.canon_fit(prep, K=K, similarity=similarity, block=512)
    count = ExactCount()
    _same(_fit(engine, capfd, X, K, similarity, flags=DBG_COARSE_SORT_KEY, count=count), want, f"mid {similarity}")
    count.require_moved()


@pytest.fixture(scope="module")
def sweep_case():
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(12000, 5000, 240_000, seed=11, item_exp=1.0)  # the matrix of test_k_sweep
    prep = orc.prepare(X)
    return X, prep, orc.canon_fit(prep, K=4096)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 33, 200, 512, 513, 2048, 4096])
def test_coarse_keys_k_sweep(engine, capfd, sweep_case, K):
    X, prep, full = sweep_case
    want = {"idx": full["idx"][:, :K], "cnt": full["cnt"][:, :K], "val": full["val"][:, :K],
            "len": np.minimum(full["len"], K)}
    count = ExactCount()
    _same(_fit(engine, capfd, X, K, flags=DBG_COARSE_SORT_KEY, count=count), want, f"K={K}")
    if K in (33, 513):
        _same(_fit(engine, capfd, X, K, "conditional_probability", flags=DBG_COARSE_SORT_KEY, count=count),
              orc.canon_fit(prep, K=K, similarity="conditional_probability"), f"K={K} conditional probability")
    count.require_moved()


# ---------------------------------------------------------------------------------------------------------------
# GPU: values whose counts cross many binades


def _fold(p, c):
    """orc.seq_sum with the entries sorted by count, so that the live entries of each step are a prefix."""
    order = np.argsort(-c, kind="stable")
    ps, cs = p[order], c[order]
    s = np.zeros_like(ps)
    live = len(cs)
    for t in range(int(cs.max()) if len(cs) else 0):
        while live and cs[live - 1] <= t:
            live -= 1
        s[:live] += ps[:live]
    out = np.empty_like(s)
    out[order] = s
    return out


@pytest.mark.gpu
def test_values_with_counts_across_binades(engine, capfd):
    """300,000 users over 240 items with popularities up to ~0.6 U: co-occurrence counts up to ~10^5."""
    rng = np.random.default_rng(7)
    U, I = 300_000, 240
    prob = 0.6 * np.exp(-np.arange(I) / 40.0) + 1e-4
    cols = [np.flatnonzero(rng.random(U) < q) for q in prob]
    rows = np.concatenate(cols).astype(np.int64)
    items = np.concatenate([np.full(len(u), j, np.int32) for j, u in enumerate(cols)])
    X = csr_matrix((np.ones(len(rows), np.int32), (rows, items)), shape=(U, I))
    K = 200
    got = _fit(engine, capfd, X, K)
    n = np.asarray(X.sum(axis=0)).ravel().astype(np.int64)
    ln = got["len"]
    mask = np.arange(K)[None, :] < ln[:, None]
    ii = np.repeat(np.arange(I), ln)
    jj = got["idx"][mask].astype(np.int64)
    cc = got["cnt"][mask].astype(np.int64)
    assert cc.max() > 50_000
    # the lists against the oracle's order (values checked below)
    C = np.asarray((X.T @ X).todense())
    for i in range(I):
        crow = C[i].copy()
        crow[i] = 0
        cand = np.flatnonzero(crow)
        order = orc.canon_order("cosine", None, crow[cand], n[cand], None, cand)[:K]
        assert ln[i] == len(order) and np.array_equal(got["idx"][i, : ln[i]], cand[order]), i
        assert np.array_equal(got["cnt"][i, : ln[i]], crow[cand[order]]), i
    p = (1.0 / np.sqrt(n[ii].astype(np.float64))) * (1.0 / np.sqrt(n[jj].astype(np.float64)))
    want = _fold(p, cc)
    small = np.flatnonzero(cc < 3000)[:500]
    assert np.array_equal(want[small], orc.seq_sum(p[small], cc[small]))
    bad = np.flatnonzero(got["val"][mask] != want)
    assert len(bad) == 0, f"{len(bad)} values differ, first (i, j, c) = {(ii[bad[0]], jj[bad[0]], cc[bad[0]])}"
    assert np.all(got["val"][~mask] == 0.0)
