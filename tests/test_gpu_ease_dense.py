"""The dense EASE chain on the GPU (csrc/ease.cu) against oracle/ease_dense_oracle.py, bit for bit, at the geometry it
runs at: the exact Gram over user chunks (``run_gram_dense_f64`` -> ``k_gram_i8_tc`` -> ``k_acc_g16``), the closed
form (``k_ease_finish``) and the dense scorer (``k_predict_dense`` -> ``k_dense_finalize``).

The scorer's item ranges (P ranges of R columns, 256 / 512 / 1,024 threads) are chosen from shared memory; the
natural-geometry cases sit on each side of each boundary.  With the instrumented build (-DRPK_PHASE_PROF, one
"[dense paths] P=.. R=.. nt=.." line per call) they also assert that the geometry was reached."""
import re
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.ease_dense_oracle import canon_dense_scores, canon_dense_topn, canon_ease_from_inverse, canon_gram

pytestmark = pytest.mark.gpu

DBG_MULTI_PASS, DBG_MANY_PASS = 4, 32


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    eng.debug_flags(0)
    yield eng
    eng.debug_flags(0)


def _paths(err):
    return [{k: int(v) for k, v in re.findall(r"(\w+)=(\d+)", line.split("]", 1)[1])}
            for line in err.splitlines() if "[dense paths]" in line]


def _bits_equal(a, b):
    """Same float64 values bit for bit, NaN positions included (any NaN payload)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    ok = ~np.isnan(a)
    return np.array_equal(a[ok].view(np.int64), b[ok].view(np.int64))


def _same_lists(got, want, want_val=True):
    assert np.array_equal(got["len"], want["len"]), "len"
    assert np.array_equal(got["idx"], want["idx"]), "idx"
    if want_val:
        assert _bits_equal(got["val"], want["val"]), "val"
    else:
        assert got["val"] is None


# ------------------------------------------------------------------------------------------
# Geometry of run_predict_dense (csrc/ease.cu), mirrored here:
#   cap = max(256, next_pow2(2 N)); fixed = sel_smem_bytes(cap); avail = smem_max - fixed - 1024
#   P = 1, 2, ...: R = (ceil(I / P) + 1) & ~1 until R * 8 <= avail
#   nt = R >= 8192 ? 1024 : (R >= 2048 ? 512 : 256)
# sel_smem_bytes (csrc/select.cuh): (cap + SEL_RANK_MAX = 64) 16-byte Entry slots + SEL_BINS = 4096 ints + SelShared
# (4 u64, one Entry, 39 ints: 204 bytes, 208 with the 16-byte alignment of Entry).  A wrong mirror shows up as a
# geometry mismatch against the instrumented build's path line.
# ------------------------------------------------------------------------------------------
def _sel_smem_bytes(cap):
    return (cap + 64) * 16 + 4096 * 4 + 208


def _avail(N, smem_max):
    cap = 256
    while cap < 2 * N:
        cap *= 2
    return smem_max - _sel_smem_bytes(cap) - 1024


def _geometry(I, N, smem_max):
    avail = _avail(N, smem_max)
    P = 1
    while True:
        R = (-(-I // P) + 1) & ~1
        if R * 8 <= avail:
            break
        P += 1
    nt = 1024 if R >= 8192 else (512 if R >= 2048 else 256)
    return P, R, nt


def _largest_one_range(N, smem_max):
    """Largest I scored in one range: R = I for even I, and R * 8 <= avail."""
    return (_avail(N, smem_max) // 8) & ~1


def _smem_max():
    import torch

    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


# ------------------------------------------------------------------------------------------
# Scorer, crafted models with exact ties
# ------------------------------------------------------------------------------------------
def _tied_model(I, seed):
    """B = small integers * 0.125 on the device: sums are exact, so scores tie often, also across item ranges."""
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    B = torch.randint(-3, 5, (I, I), generator=g, device="cuda", dtype=torch.int64).to(torch.float64) * 0.125
    B[:, 3] = 0.0                                    # a column nobody scores
    B[0, :] = 0.0
    B[1, :] = 0.0
    B[0, 10::7], B[1, 10::7] = 0.75, -0.75           # user {0, 1}: these columns cancel to exactly 0.0
    B[0, 11::7], B[1, 11::7] = 0.5, 0.25
    B[9] = -(B[9].abs()) - 0.125                     # user {9}: negative scores only
    B.fill_diagonal_(0.0)
    return B


def _tied_users(I, seed):
    rng = np.random.default_rng(seed)
    X = (rng.random((300, I)) < 0.04).astype(np.int8)
    X[0] = 0                 # empty history
    X[1] = 0
    X[1, [0, 1]] = 1         # cancelling columns
    X[2] = 1                 # every item held: with the history mask, every candidate is masked
    X[3] = 0
    X[3, 9] = 1              # negative only
    X[4] = 0
    X[4, [0, 1, I - 1]] = 1  # cancellation plus the last item
    X[5, ::2] = 1            # a long history
    return csr_matrix(X)


@pytest.mark.parametrize("flags", [0, DBG_MULTI_PASS, DBG_MANY_PASS])
@pytest.mark.parametrize("I", [120, 1001])
def test_crafted_ties(engine, capfd, I, flags):
    B = _tied_model(I, I + flags)
    X = _tied_users(I, I)
    B_host = B.cpu().numpy()
    U = X.shape[0]
    indptr, indices = X.indptr.astype(np.int64), X.indices.astype(np.int32)
    seen = []
    engine.debug_flags(flags)
    try:
        for mask in (False, True):
            want_scores = canon_dense_scores(indptr, indices, B_host, mask_history=mask)
            capfd.readouterr()
            full = engine.predict_dense_full(U, indptr, indices, B, mask_history=mask)
            assert _bits_equal(full, want_scores)
            for N in (1, 20, 2048):
                want = canon_dense_topn(want_scores, N)
                for want_val in (True, False):
                    got = engine.predict_dense_topn(U, indptr, indices, B, N, mask_history=mask, want_val=want_val)
                    _same_lists(got, want, want_val)
            if mask:
                assert want["len"][2] == 0  # every candidate masked
            assert want["len"][0] == 0 and want["len"][3] > 0 and np.all(want["val"][3, : want["len"][3]] < 0)
            paths = _paths(capfd.readouterr().err)
            if paths:
                Ps = sorted({p["P"] for p in paths})
                seen.append(f"mask={mask}: P={Ps}")
                assert Ps[0] >= {0: 1, DBG_MULTI_PASS: 2, DBG_MANY_PASS: 4}[flags]
    finally:
        engine.debug_flags(0)
    if seen:
        print(f"I={I} flags={flags}: " + ", ".join(seen))
    assert canon_dense_scores(indptr, indices, B_host)[1, 10] == 0.0  # the cancelling columns are there


# ------------------------------------------------------------------------------------------
# Scorer, natural geometry (no flags)
# ------------------------------------------------------------------------------------------
def _users(I, seed):
    """512 users: mostly short histories, two of several thousand items, one empty, one holding item I - 1."""
    rng = np.random.default_rng(seed)
    d = np.minimum(rng.geometric(1 / 40, size=512), I)
    d[5], d[6], d[7] = min(I, 2000), min(I, 3000), 0
    rows = [np.sort(rng.choice(I, size=int(k), replace=False)) for k in d]
    rows[8] = np.array(sorted(set(rows[8].tolist()) | {I - 1}), dtype=np.int64)
    indptr = np.zeros(513, dtype=np.int64)
    np.cumsum([len(r) for r in rows], out=indptr[1:])
    return indptr, np.concatenate(rows).astype(np.int32)


def _natural_cases():
    # (name, N, I as a function of the largest one-range item count at that N)
    return [
        ("nt256", 20, lambda m: 2046),        # R = 2046
        ("nt512", 20, lambda m: 2047),        # R = 2048 (rounded up to even)
        ("nt512_top", 20, lambda m: 8190),    # R = 8190
        ("nt1024", 20, lambda m: 8191),       # R = 8192
        ("p1_max", 20, lambda m: m),          # the largest I with one range
        ("p2_min", 20, lambda m: m + 2),      # two ranges
        ("p1_max_n2048", 2048, lambda m: m),
        ("p2_min_n2048", 2048, lambda m: m + 2),
        ("msd", 20, lambda m: 41_140),
        ("ml25m", 20, lambda m: 59_047),
    ]


@pytest.mark.parametrize("name,N,I_of", _natural_cases(), ids=[c[0] for c in _natural_cases()])
def test_natural_geometry(engine, capfd, name, N, I_of):
    import torch

    smem_max = _smem_max()
    I = I_of(_largest_one_range(N, smem_max))
    P, R, nt = _geometry(I, N, smem_max)
    full_geom = _geometry(I, 1, smem_max)  # the full scores need no list: the workspace of N = 1
    expect = {"nt256": (1, 256), "nt512": (1, 512), "nt512_top": (1, 512), "nt1024": (1, 1024), "p1_max": (1, 1024),
              "p2_min": (2, 1024), "p1_max_n2048": (1, 1024), "p2_min_n2048": (2, 1024), "msd": (2, 1024),
              "ml25m": (3, 1024)}[name]
    assert (P, nt) == expect, (name, I, P, R, nt)

    g = torch.Generator(device="cuda").manual_seed(I)
    B = torch.randn((I, I), generator=g, device="cuda", dtype=torch.float64)
    indptr, indices = _users(I, I)
    U = 512
    ptr_d = torch.from_numpy(indptr).cuda()
    idx_d = torch.from_numpy(indices).cuda()
    capfd.readouterr()
    full = engine.predict_dense_full(U, ptr_d, idx_d, B, mask_history=True)
    top = engine.predict_dense_topn(U, ptr_d, idx_d, B, N, mask_history=True)
    engine.sync()
    paths = _paths(capfd.readouterr().err)
    print(f"{name}: I={I} N={N} -> lists P={P} R={R} nt={nt}, full P={full_geom[0]} R={full_geom[1]} nt={full_geom[2]} "
          f"(shared memory opt-in {smem_max} B); path lines: {[(p['P'], p['R'], p['nt']) for p in paths]}")
    if paths:
        assert [(p["P"], p["R"], p["nt"]) for p in paths] == [full_geom, (P, R, nt)], paths
    full_h = full.cpu().numpy()
    got = {k: v.cpu().numpy() for k, v in top.items()}
    del full, top

    # full rows of a sample (the heavy users, the empty one, the one holding item I - 1) against the oracle
    sample = np.array([5, 6, 7, 8] + list(range(9, 41)) + [511])
    s_ptr = np.zeros(len(sample) + 1, dtype=np.int64)
    np.cumsum(np.diff(indptr)[sample], out=s_ptr[1:])
    s_idx = np.concatenate([indices[indptr[u]:indptr[u + 1]] for u in sample])
    items = np.unique(s_idx)
    rows = B[torch.from_numpy(items).cuda()].cpu().numpy()
    del B
    torch.cuda.empty_cache()
    want_s = canon_dense_scores(s_ptr, s_idx, (items, rows), mask_history=True)
    assert _bits_equal(full_h[sample], want_s)
    want_top_s = canon_dense_topn(want_s, N)
    _same_lists({k: v[sample] for k, v in got.items()}, want_top_s)
    # the lists of every user against the full rows of the same kernel
    _same_lists(got, canon_dense_topn(full_h, N))


# ------------------------------------------------------------------------------------------
# Closed form
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("I", [1, 2, 255, 257, 3000])
@pytest.mark.parametrize("w_kind", ["none", "finite", "inf"])
@pytest.mark.parametrize("in_place", [True, False])
def test_closed_form(engine, I, w_kind, in_place):
    import torch

    rng = np.random.default_rng(I)
    P = rng.standard_normal((I, I)) * 1e-3
    P[np.arange(I), np.arange(I)] = rng.random(I) + 0.5
    j0 = I // 2  # an item nobody saw: a zero row and column of P off the diagonal
    P[j0, np.arange(I) != j0] = 0.0
    P[np.arange(I) != j0, j0] = 0.0
    w = None
    if w_kind != "none":
        w = 1.0 / rng.integers(1, 50, I).astype(np.float64) ** 0.5
        if w_kind == "inf":
            w[j0] = np.inf
    want = canon_ease_from_inverse(P, w)
    Pd = torch.from_numpy(P).cuda()
    out = None if in_place else torch.full_like(Pd, 7.0)
    got = engine.ease_from_inverse(Pd, w, out=out)
    engine.sync()
    if in_place:
        assert got.data_ptr() == Pd.data_ptr()
    else:
        assert np.array_equal(Pd.cpu().numpy(), P)  # the input is untouched
    got = got.cpu().numpy()
    assert _bits_equal(got, want)
    assert np.array_equal(np.diag(got).view(np.int64), np.zeros(I, dtype=np.int64))  # +0.0 exactly
    assert np.isnan(got).sum() == (I - 1 if w_kind == "inf" else 0)


# ------------------------------------------------------------------------------------------
# Gram
# ------------------------------------------------------------------------------------------
def _gram_users(U, I, seed, empty=()):
    """Every user holds items 1 and 2 (count U); three random items each in [4, I); item 3 nobody holds; user 0 holds
    I - 1; the users in `empty` hold nothing."""
    rng = np.random.default_rng(seed)
    cols = np.concatenate([np.ones((U, 1), np.int64), np.full((U, 1), 2), rng.integers(4, I, (U, 3))], axis=1)
    cols[0, 2] = I - 1
    keep = np.ones(U, dtype=bool)
    keep[list(empty)] = False
    rows = np.repeat(np.arange(U), 5)[np.repeat(keep, 5)]
    X = csr_matrix((np.ones(rows.shape[0], np.int32), (rows, cols[keep].ravel())), shape=(U, I))
    X.sum_duplicates()
    X.data[:] = 1
    X.sort_indices()
    return X


@pytest.mark.parametrize("U,empty", [(32_768, ()), (32_769, (7, 32_768)), (65_537, ()), (65_540, (0, 40_000, 65_539))])
@pytest.mark.parametrize("I", [1000, 4097])
def test_gram_exact(engine, U, empty, I):
    X = _gram_users(U, I, U + I, empty)
    G = engine.gram_dense_f64(U, I, X.indptr.astype(np.int64), X.indices.astype(np.int32))
    want = canon_gram(X)
    assert want[1, 2] == U - len(empty) and want[3].max() == 0 and want[I - 1, I - 1] >= 1
    assert np.array_equal(G, want.astype(np.float64))


def test_gram_no_users(engine):
    G = engine.gram_dense_f64(0, 257, np.zeros(1, np.int64), np.zeros(0, np.int32))
    assert G.shape == (257, 257) and np.array_equal(G, np.zeros((257, 257)))


def test_gram_u16_full_chunk(engine):
    rng = np.random.default_rng(11)
    A = (rng.random((300, 32_768)) < 0.01).astype(np.uint8)
    A[[0, 5, 299]] = 1  # count 32,768
    G = engine.gram_dense_u16(A)
    Af = A.astype(np.float64)
    want = (Af @ Af.T).astype(np.int64)  # exact: counts < 2^53
    assert G[0, 5] == 32_768 and np.array_equal(G.astype(np.int64), want)
    A1 = np.ones((1, 32_768), dtype=np.uint8)
    assert engine.gram_dense_u16(A1).tolist() == [[32_768]]
    A1[0, ::3] = 0
    assert engine.gram_dense_u16(A1).tolist() == [[int(A1.sum())]]


# ------------------------------------------------------------------------------------------
# End to end at the ML-1M shape, exact against the oracle on the fitted model
# ------------------------------------------------------------------------------------------
def test_ml1m_shape_exact(engine):
    from recpack_b200 import EASE
    from recpack_b200.synth import make_dataset

    train, _, _ = make_dataset("ml1m")
    algo = EASE(l2=200.0).fit(train)
    B = algo._B_dev.cpu().numpy()
    X = csr_matrix(train, copy=True)
    X.sort_indices()
    full = algo.predict(train)
    want = canon_dense_scores(X.indptr, X.indices, B)
    assert _bits_equal(full.toarray(), want)
    algo.set_params(predict_topK=20, remove_history=True)
    pred = algo.predict(train)
    idx, ln = pred._rpk_topn
    want[np.repeat(np.arange(X.shape[0]), np.diff(X.indptr)), X.indices] = 0.0  # canon_dense_scores(mask_history=True)
    top = canon_dense_topn(want, 20)
    assert np.array_equal(ln, top["len"]) and np.array_equal(idx, top["idx"])
    dense = pred.toarray()
    r = np.repeat(np.arange(X.shape[0]), 20).reshape(-1, 20)
    ok = top["idx"] >= 0
    assert _bits_equal(dense[r[ok], top["idx"][ok]], top["val"][ok])


# ------------------------------------------------------------------------------------------
# A NaN column: full scores as scipy computes them, top-N refused
# ------------------------------------------------------------------------------------------
def test_nan_column(engine):
    from recpack_b200 import EASE
    from recpack_b200._lib import RpkError
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(400, 150, 6000, seed=9).tolil()
    X[:, 77] = 0  # nobody interacted with item 77: w_77 = inf, column 77 of B is NaN off the diagonal
    X = csr_matrix(X)
    X.eliminate_zeros()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        algo = EASE(l2=20.0, alpha=0.5).fit(X)
    B = algo._B_dev.cpu().numpy()
    assert np.isnan(B[:, 77]).sum() == 149 and not np.isnan(np.delete(B, 77, axis=1)).any()
    full = algo.predict(X).toarray()
    want = np.asarray(X.astype(bool).astype(np.float64) @ B)
    assert np.isnan(want[:, 77]).any() and _bits_equal(full, want)
    for remove_history in (False, True):
        algo.set_params(predict_topK=10, remove_history=remove_history)
        with pytest.raises(RpkError, match="NaN"):
            algo.predict(X)
    # a user holding items 5 and 77: NaN at column 77 unless the history mask removes it
    ptr = np.array([0, 2], dtype=np.int64)
    idx = np.array([5, 77], dtype=np.int32)
    with pytest.raises(RpkError, match="NaN"):
        engine.predict_dense_topn(1, ptr, idx, algo._B_dev, 10, mask_history=False)
    got = engine.predict_dense_topn(1, ptr, idx, algo._B_dev, 10, mask_history=True)
    _same_lists(got, canon_dense_topn(canon_dense_scores(ptr, idx, B, mask_history=True), 10))
