"""Every selection path of the fit's row kernel (k_fit_rows) and its shared-memory geometry, compared with the oracle.

The row kernel counts one item row in shared memory and selects its top K there (block_select_topk, select.cuh).  Each
case below builds an interaction matrix that forces one path of that selection:

  direct path          rows with at most direct_cap candidates; the rank sort (<= 64 survivors) and the bitonic sort,
                       deferred to k_fit_sort_rows (P == 1), in the kernel (DBG_TINY_LIST) or merged by k_fit_merge
                       (DBG_MULTI_PASS)
  guess accepted       B0: the 1-in-16 sampled threshold guess leaves between K and cap survivors, with the coded
                       reciprocal and with the exact one
  guess rejected       the count bound overestimates the candidates (a clique), or the sample holds only weak keys
  queue overflow       more than 4,096 slots pass the pre-filter of the queued copy: the direct visit runs instead
  band select          phase C: more than cap candidates whose approximate keys are equal (one count, one popularity
                       code) and whose exact keys differ; with one exact class larger than the room, the index radix
  code rounding        popularities at a half step of the 12-per-octave code, on both sides of the K-th place
  fp32 keys            counts above 4,096 (c^2 is not exact in fp32) and pairs with c1^2 n2 - c2^2 n1 = +-1
  K sweep              K from 1 to 4,096 on one matrix, and K >= I - 1
  geometry edges       the item counts where P changes, where the coded keys stop fitting, and the bands where the
                       shared memory of a block was over-committed before the static tables were counted
  mid shape            40,000 x 8,000, every row

Outputs are poisoned beforehand (idx = -2, cnt = -3, val = NaN, len = -4), so that a row no kernel writes fails.  Each
case asserts on the oracle side that its construction reaches the path (a numpy mirror of the host geometry and of
the B0 guess), and, with the instrumented build (-DRPK_PHASE_PROF, which prints one "[fit paths]" line per fit call),
that the kernel's counter of that path moved."""
import math
import re

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle import recpack_oracle as orc

pytestmark = pytest.mark.gpu

DBG_TINY_LIST, DBG_MULTI_PASS, DBG_SPLIT_ROWS = 2, 4, 8
SEL_BINS, SEL_RANK_MAX, SEL_SAMPLE, SEL_GUESS_MIN, QUEUE_CAP = 4096, 64, 16, 4096, 4096
SEL_SHARED_BYTES = 208  # sizeof(SelShared) rounded up to 16
SMEM_OPTIN_B200 = 232448  # sharedMemPerBlockOptin of sm_100
STATIC16 = 2320  # static shared memory of k_fit_rows<true> (ptxas -v, sm_100a)
COUNTERS = ("guess_ok", "guess_rejected", "queue_overflow", "band", "index_radix", "deferred", "merged", "P", "R",
            "code", "smem", "static")
F32 = np.float32


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    yield eng
    eng.debug_flags(0)
    eng.fit_config(-1)


@pytest.fixture(scope="module")
def smem_max():
    import torch

    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


# ---------------------------------------------------------------------------------------------------------------
# the host geometry of fit_range, mirrored


def _np2(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def _geom(I, K, U=100_000, cosine=True, flags=0, smem_max=SMEM_OPTIN_B200, static=STATIC16, reserved=None):
    """cap, direct_cap, use_code, P, R and the dynamic shared memory of the 16-bit row kernel.  `reserved`: what the
    host takes off for static shared memory (the kernel's static size; the parent commit took a fixed 2,048)."""
    tiny = bool(flags & DBG_TINY_LIST)
    cap = max(64 if tiny else 1024, _np2(2 * K))
    direct_cap = K if tiny else min(cap, max(2 * K, 64))
    fixed = (cap + SEL_RANK_MAX) * 16 + SEL_BINS * 4 + SEL_SHARED_BYTES
    avail = smem_max - fixed - (static if reserved is None else reserved)
    use_code = cosine and I + 65536 < avail and U < (1 << 21)
    code = ((I + 512 + 15) & ~15) if use_code else 0
    rmax = ((avail - code) // 2) & ~7
    P = max(1, -(-I // rmax))
    if flags & DBG_MULTI_PASS and P < 2 and I >= 16:
        P = 2
    R = (-(-I // P) + 7) & ~7
    smem = fixed + 2 * R + code
    return {"cap": cap, "direct_cap": direct_cap, "use_code": use_code, "P": P, "R": R, "smem": smem,
            "over": smem + static - smem_max, "defer": P == 1 and not tiny}


def _bands(K, cosine, hi=300_000):
    """Item counts at which the parent's fixed 2 KB reservation over-committed a block's shared memory."""
    bands, start, prev = [], None, None
    for I in range(2, hi):
        if _geom(I, K, cosine=cosine, reserved=2048)["over"] > 0:
            if start is None or I != prev + 1:
                if start is not None:
                    bands.append((start, prev))
                start = I
            prev = I
    if start is not None:
        bands.append((start, prev))
    return bands


def _last_p1(K, cosine, flags=0):
    """Largest I with P == 1 (the boundary moves by the code bytes; search downward from an upper bound)."""
    lo, hi = 2, 300_000
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if _geom(mid, K, cosine=cosine, flags=flags)["P"] == 1:
            lo = mid
        else:
            hi = mid - 1
    return lo


def _code_limit(K):
    """Largest I that keeps the coded keys (cosine)."""
    I = 2
    while _geom(I + 4096, K)["use_code"]:
        I += 4096
    while _geom(I + 1, K)["use_code"]:
        I += 1
    return I


def test_geometry_mirror_pins_the_shared_memory_bands():
    """The mirror reproduces the over-committed bands of the parent's 2 KB reservation, and the reservation of the
    kernel's static size leaves none."""
    assert _bands(200, True)[:5] == [(65201, 65296), (97809, 97936), (117361, 117528), (130401, 130592),
                                     (196129, 196400)]
    assert _bands(512, True)[:1] == [(65201, 65296)]
    assert _bands(200, False)[:2] == [(98065, 98200), (196129, 196400)]
    assert _bands(1024, True)[:1] == [(59745, 59832)]
    for cosine in (True, False):
        assert _bands(4096, cosine)[:2] == [(40721, 40856), (81441, 81712)]
    g = _geom(65201, 200, reserved=2048)
    assert g["use_code"] and g["P"] == 1 and 0 < g["over"] <= 272
    for K in (200, 1024, 4096):
        for cosine in (True, False):
            assert all(_geom(I, K, cosine=cosine)["over"] <= 0 for I in range(2, 300_000, 7))
    # the coded keys stop at I + 65536 < avail: 130,863 with the 2 KB reservation, 272 items earlier now; the ML-25M
    # shape keeps P = 1 and the same R with them
    assert _geom(130_863, 200, reserved=2048)["use_code"] and not _geom(130_864, 200, reserved=2048)["use_code"]
    assert _code_limit(200) == 130_591 and not _geom(130_592, 200)["use_code"]
    ml = _geom(59_047, 200, U=162_541)
    assert ml["P"] == 1 and ml["use_code"]
    assert _geom(59_047, 200, U=162_541, reserved=2048)["R"] == ml["R"]
    # caps and their changes at K = 32, 512, 513
    assert [_geom(1000, K)["direct_cap"] for K in (31, 32, 33, 512, 513)] == [64, 64, 66, 1024, 1026]
    assert [_geom(1000, K)["cap"] for K in (512, 513, 4096)] == [1024, 2048, 8192]


# ---------------------------------------------------------------------------------------------------------------
# matrices


def _csr(hists, I):
    hists = [np.unique(np.asarray(h, dtype=np.int32)) for h in hists]
    indptr = np.concatenate([[0], np.cumsum([len(h) for h in hists])]).astype(np.int64)
    indices = np.concatenate(hists + [np.zeros(0, np.int32)]).astype(np.int32)
    return csr_matrix((np.ones(len(indices), dtype=np.int32), indices, indptr), shape=(len(hists), I))


def _star(I, targets, c, n, extra_users=()):
    """Users such that every target item co-occurs c[j] times with item j and item j is seen by n[j] users (c[j] <= n[j];
    c = 0: no co-occurrence).  Co-user k holds the targets and {j : c[j] > k}; filler user k holds {j : n[j] - c[j] > k}."""
    c = np.asarray(c, dtype=np.int64)
    n = np.asarray(n, dtype=np.int64)
    assert np.all(c <= n)
    targets = np.asarray(targets, dtype=np.int32)
    free = np.ones(I, bool)
    free[targets] = False
    c = np.where(free, c, 0)
    n = np.where(free, n, 0)
    hists = []
    for k in range(int(c.max())):
        hists.append(np.concatenate([targets, np.flatnonzero(c > k)]))
    rest = n - c
    for k in range(int(rest.max()) if rest.size else 0):
        hists.append(np.flatnonzero(rest > k))
    hists += list(extra_users)
    return _csr(hists, I)


def _append_empty_users(X, count):
    indptr = np.concatenate([X.indptr.astype(np.int64), np.full(count, X.indptr[-1], dtype=np.int64)])
    return csr_matrix((X.data, X.indices, indptr), shape=(X.shape[0] + count, X.shape[1]))


# ---------------------------------------------------------------------------------------------------------------
# the B0 guess of block_select_topk, mirrored (16-bit counters, one item range, no dense leg)


def _code_tab():
    return np.exp2(-np.arange(256, dtype=F32) / F32(12)).astype(F32)


def _codes(n):
    with np.errstate(divide="ignore"):
        v = np.rint(F32(12) * np.log2(np.maximum(n, 1).astype(F32)))
    return np.clip(v, 0, 255).astype(np.int64)


def _bits(x):
    return np.asarray(x, dtype=F32).view(np.uint32).astype(np.int64)


def _b0(X, prep, i, K, coded, flags=0):
    """For row i: (candidate count bound, guess accepted, slots queued by the pre-filter)."""
    n = prep.n
    I = X.shape[1]
    g = _geom(I, K, U=X.shape[0], flags=flags)
    row = orc.cooccurrence_rows(prep, [i])[0].astype(np.int64)
    row[i] = 0
    slots = np.flatnonzero(row)
    cs = row[slots]
    cf = cs.astype(F32)
    if coded:
        r = _code_tab()[_codes(n[slots])]
    else:
        r = (F32(1) / n[slots].astype(F32)).astype(F32)
    key = _bits((cf * cf).astype(F32) * r)
    kmin = int(_bits(F32(F32(1) / F32(n.max())) * F32(0.94)))
    if coded:
        X_ = prep.Xb
        work = int(np.diff(X_.indptr)[X_[:, i].nonzero()[0]].sum())
        n_c = min(I, work)
        kmax = int(_bits(F32(n[i]) * F32(n[i])))
        M = 1 << 20
    else:
        n_c = len(slots)
        kmax = int(_bits(F32(cs.max()) * F32(cs.max()))) if len(cs) else 0
        M = 32
    if n_c <= g["direct_cap"] or n_c < SEL_GUESS_MIN or kmax <= kmin:
        return n_c, None, 0
    rng_ = kmax - kmin
    shift = max(0, rng_.bit_length() - 12)
    nb = (rng_ >> shift) + 1
    sk = key[(slots % SEL_SAMPLE) == 0]
    sk = sk[(sk >= kmin) & (sk <= kmax)]
    h = np.bincount((sk - kmin) >> shift, minlength=nb)
    ks = -(-K // SEL_SAMPLE)
    sd = math.isqrt(ks - 1) + 1 if ks > 1 else 1
    need = ks + 3 * sd + 3
    suffix = np.cumsum(h[::-1])[::-1]
    bstar = int(np.flatnonzero(suffix >= need).max()) if suffix[0] >= need else 0
    edge = kmin + (bstar << shift)
    thr = edge - M if edge > M else 0
    count2 = int(np.count_nonzero(key >= edge))
    got = int(np.count_nonzero(key >= thr))
    queued = 0
    if coded and thr > 0:
        tf = np.array([thr], dtype=np.uint32).view(F32)[0]
        tab = _code_tab()
        cq = np.ceil((np.sqrt(tf / tab) * F32(0.9999)).astype(F32))
        cq = np.clip(cq, 1, 65535).astype(np.int64)
        queued = int(np.count_nonzero(cs >= cq[_codes(n[slots])]))
    return n_c, (count2 >= K and got <= g["cap"]), queued


# ---------------------------------------------------------------------------------------------------------------
# fit calls into poisoned outputs, the path counters of the instrumented build


def _lines(text):
    out = []
    for line in text.splitlines():
        if line.startswith("[fit paths]"):
            out.append({k: int(re.search(r"\b" + k + r"=(\d+)", line).group(1)) for k in COUNTERS})
    return out


class Paths:
    """Path counters of the fit calls of one case; empty under the normal build."""

    def __init__(self):
        self.lines = []

    def require(self, key, at_least=1):
        if not self.lines:
            print(f"path counter '{key}': no [fit paths] line (normal build), not checked")
            return
        n = sum(line[key] for line in self.lines)
        print(f"path counter '{key}': {n}, required >= {at_least}")
        assert n >= at_least, f"the case did not reach its path: '{key}' = {n}"

    def geometry(self, g):
        for line in self.lines:
            assert line["P"] == g["P"] and line["R"] == g["R"] and line["code"] == int(g["use_code"]), (line, g)
            assert line["static"] == STATIC16 and line["smem"] == g["smem"], (line, g)


def _fit(engine, capfd, X, K, similarity="cosine", flags=0, dense=-1, device=False, rows=None, paths=None):
    U, I = X.shape
    b, e = (0, I) if rows is None else rows
    nr = e - b
    indptr = np.ascontiguousarray(X.indptr, dtype=np.int64)
    indices = np.ascontiguousarray(X.indices, dtype=np.int32)
    if device:
        import torch

        indptr, indices = torch.from_numpy(indptr).cuda(), torch.from_numpy(indices).cuda()
        out = {"idx": torch.full((nr, K), -2, dtype=torch.int32, device="cuda"),
               "cnt": torch.full((nr, K), -3, dtype=torch.int32, device="cuda"),
               "val": torch.full((nr, K), float("nan"), dtype=torch.float64, device="cuda"),
               "len": torch.full((nr,), -4, dtype=torch.int32, device="cuda")}
        torch.cuda.synchronize()
    else:
        out = {"idx": np.full((nr, K), -2, np.int32), "cnt": np.full((nr, K), -3, np.int32),
               "val": np.full((nr, K), np.nan), "len": np.full(nr, -4, np.int32)}
    print(capfd.readouterr().out, end="")  # keep what the case printed so far
    engine.debug_flags(flags)
    engine.fit_config(dense)
    try:
        engine.fit_topk(U, I, indptr, indices, K, similarity=similarity, item_begin=b, item_end=e, out=out)
        engine.sync()
    finally:
        engine.debug_flags(0)
        engine.fit_config(-1)
    if device:
        out = {k: v.cpu().numpy() for k, v in out.items()}
    if paths is not None:
        paths.lines += _lines(capfd.readouterr().err)
    return out


def _same(got, want, what, rows=None):
    for key in ("len", "idx", "cnt", "val"):
        g = got[key] if rows is None else got[key][rows]
        w = want[key]
        bad = np.flatnonzero(np.any((g != w).reshape(len(g), -1), axis=1))
        assert len(bad) == 0, (f"{what}: {key} differs in {len(bad)} rows, first {bad[:8].tolist()}; row {bad[0]}: "
                               f"got {g[bad[0]].ravel()[:10].tolist()} want {w[bad[0]].ravel()[:10].tolist()}")


def _run(engine, capfd, X, K, want, similarity="cosine", variants=((0, -1),), device=False, paths=None):
    """The fit in each (flags, dense_users) variant against the oracle's full output."""
    paths = Paths() if paths is None else paths
    for flags, dense in variants:
        for dev in ((False, True) if device else (False,)):
            got = _fit(engine, capfd, X, K, similarity, flags, dense, dev, paths=paths)
            _same(got, want, f"K={K} {similarity} flags={flags} dense={dense} {'device' if dev else 'host'}")
    return paths


# ---------------------------------------------------------------------------------------------------------------
# direct path and both sorts


@pytest.mark.parametrize("flags", [0, DBG_TINY_LIST, DBG_MULTI_PASS])
def test_direct_path_rank_and_bitonic_sorts(engine, capfd, flags):
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(1500, 1200, 9000, seed=3)
    prep = orc.prepare(X)
    K = 200
    g = _geom(1200, K, U=1500, flags=flags)
    want = orc.canon_fit(prep, K=K)
    # candidates per row: some rank-sorted (<= 64), some bitonic (65 .. direct_cap), all on the direct path
    cand = np.array([np.count_nonzero(r) - (r[i] > 0) for i, r in
                     enumerate(orc.cooccurrence_rows(prep, np.arange(1200)))])
    work = np.asarray(prep.Xt @ np.diff(prep.Xb.indptr)).ravel()
    direct = np.minimum(work, 1200) <= g["direct_cap"]
    assert np.count_nonzero(direct & (cand <= SEL_RANK_MAX) & (cand > 1)) > 50
    assert np.count_nonzero(direct & (cand > SEL_RANK_MAX)) > 20
    paths = _run(engine, capfd, X, K, want, variants=((flags, -1),), device=flags == 0)
    for sim, Ks in (("conditional_probability", 30), ("cosine", 10)):
        _run(engine, capfd, X, Ks, orc.canon_fit(prep, K=Ks, similarity=sim), sim, variants=((flags, -1),), paths=paths)
    if flags == 0:
        paths.require("deferred", at_least=100)
    if flags == DBG_MULTI_PASS:
        paths.require("merged", at_least=1000)


# ---------------------------------------------------------------------------------------------------------------
# B0: the sampled threshold guess


def _guess_matrix(seed=5):
    """Four target rows that co-occur with every other item; counts 1-4 and popularities spread over 300 values, so the
    sample represents the keys and the guess stands."""
    I = 6000
    rng = np.random.default_rng(seed)
    c = rng.integers(1, 5, size=I)
    n = c + rng.integers(0, 300, size=I)
    return _star(I, [11, 2222, 3333, 5999], c, n)


def test_guess_accepted_coded_and_exact_reciprocal(engine, capfd):
    X = _guess_matrix()
    prep = orc.prepare(X)
    K = 200
    want = orc.canon_fit(prep, K=K)
    for i in (11, 2222, 3333, 5999):
        for coded in (True, False):
            n_c, ok, queued = _b0(X, prep, i, K, coded)
            assert n_c >= SEL_GUESS_MIN and ok, (i, coded, n_c, ok)
            assert not coded or 0 < queued <= QUEUE_CAP
    paths = _run(engine, capfd, X, K, want, device=True)
    paths.require("guess_ok", at_least=4)
    # U >= 2^21 turns the coded keys off and changes no count: the same oracle output
    Xe = _append_empty_users(X, (1 << 21) - X.shape[0] + 5)
    assert not _geom(6000, K, U=Xe.shape[0])["use_code"]
    pe = _run(engine, capfd, Xe, K, want)
    pe.require("guess_ok", at_least=4)


def test_guess_rejected_count_bound_of_a_clique(engine, capfd):
    """50 users share 100 items: the bound min(I, work) = 5,000 starts B0, but there are only 99 real candidates."""
    I = 5000
    rng = np.random.default_rng(6)
    hists = [np.arange(100) for _ in range(50)]
    hists += [rng.choice(np.arange(100, I), size=rng.integers(2, 30), replace=False) for _ in range(3000)]
    X = _csr(hists, I)
    prep = orc.prepare(X)
    K = 200
    for i in (0, 57, 99):
        n_c, ok, _ = _b0(X, prep, i, K, True)
        assert n_c >= SEL_GUESS_MIN and ok is False
    want = orc.canon_fit(prep, K=K)
    assert np.all(want["len"][:100] == 99)
    paths = _run(engine, capfd, X, K, want, variants=((0, -1), (DBG_TINY_LIST, -1)))
    paths.require("guess_rejected", at_least=200)


def _low_guess_matrix(strong):
    """Target rows whose sampled slots (items = 0 mod 16) hold weak keys (c = 1, n = 4) while `strong` other items hold
    strong ones (c = 8, n = 8 .. 207): the guessed threshold lets all strong items and the sample through."""
    I = 8192
    j = np.arange(I)
    c = np.ones(I, np.int64)
    n = np.full(I, 8, np.int64)  # the remaining items: c = 1, n = 8, below the sample's keys
    samp = j % 16 == 0
    n[samp] = 4
    others = np.flatnonzero(~samp)
    pick = others[np.linspace(0, len(others) - 1, strong).astype(np.int64)]
    c[pick] = 8
    n[pick] = 8 + (pick % 200)
    return _star(I, [8181, 8182, 8183], c, n)


@pytest.mark.parametrize("strong,overflow", [(2000, False), (5000, True)])
def test_guess_rejected_low_sample_and_queue_overflow(engine, capfd, strong, overflow):
    X = _low_guess_matrix(strong)
    prep = orc.prepare(X)
    K = 200
    for i in (8181, 8182, 8183):
        n_c, ok, queued = _b0(X, prep, i, K, True)
        assert n_c >= SEL_GUESS_MIN and ok is False
        assert (queued > QUEUE_CAP) == overflow, queued
    want = orc.canon_fit(prep, K=K)
    paths = _run(engine, capfd, X, K, want, variants=((0, -1), (DBG_MULTI_PASS, -1), (0, 64)), device=True)
    paths.require("guess_rejected", at_least=3)
    if overflow:
        paths.require("queue_overflow", at_least=3)


# ---------------------------------------------------------------------------------------------------------------
# phase C: band quick-select under coded keys, index radix


def _band_matrix(big_class):
    """Target rows 0..2 co-occur twice with 2,400 items whose popularities lie in [1024, 1053] (all code 120): identical
    approximate keys, exact keys ordered by popularity.  big_class: the K-th place lies in a class of about 1,150 items
    that share n = 1030 (one exact class larger than the list)."""
    I = 4096
    j = np.arange(I)
    c = np.zeros(I, np.int64)
    n = np.zeros(I, np.int64)
    grp = np.arange(8, 8 + 2400)
    c[grp] = 2
    n[grp] = 1024 + (grp * 7) % 30
    if big_class:  # 50 better, 1,300 tied at n = 1030 around the K-th place, 1,050 worse
        n[grp] = np.where(grp % 48 == 0, 1024, np.where(grp % 2 == 0, 1030, 1040 + grp % 14))
    rng = np.random.default_rng(9)
    extra = [rng.choice(np.arange(2410, I), size=20, replace=False) for _ in range(200)]
    return _star(I, [0, 1, 2], c, n, extra_users=extra)


@pytest.mark.parametrize("big_class", [False, True])
def test_band_select_under_coded_keys(engine, capfd, big_class):
    X = _band_matrix(big_class)
    prep = orc.prepare(X)
    n = prep.n
    grp = np.arange(8, 8 + 2400)
    assert np.all(_codes(n[grp]) == 120) and np.all((n[grp] >= 1024) & (n[grp] <= 1053))
    K = 200
    want = orc.canon_fit(prep, K=K)
    # the K-th place lies inside the group, and inside one exact class
    nk = n[want["idx"][0, K - 1]]
    assert np.count_nonzero(n[grp] < nk) < K < np.count_nonzero(n[grp] <= nk)
    if big_class:
        assert nk == 1030 and np.count_nonzero(n[grp] == 1030) > _geom(X.shape[1], K)["cap"]
    variants = ((0, -1), (DBG_TINY_LIST, -1), (DBG_MULTI_PASS, -1), (DBG_SPLIT_ROWS, -1), (0, 64))
    paths = _run(engine, capfd, X, K, want, variants=variants)
    paths.require("band", at_least=3 * len(variants))
    if big_class:
        paths.require("index_radix", at_least=3)


def _half_step_pops(lo=200, hi=4000, count=3):
    """Popularities whose 12 log2(n) lies closest to a half code step (either rounding is possible on the GPU)."""
    nn = np.arange(lo, hi)
    frac = np.abs((12 * np.log2(nn)) % 1 - 0.5)
    return nn[np.argsort(frac)[:count]]


def test_code_rounding_edges(engine, capfd):
    I = 3000
    c = np.zeros(I, np.int64)
    n = np.zeros(I, np.int64)
    cols = np.arange(10, 10 + 6 * 120)
    pops = []
    for h in _half_step_pops(300, 700):
        pops += [h - 1, h, h + 1]
    pops = np.array(pops[:6])
    for t, p in enumerate(pops):
        sl = cols[t * 120 : (t + 1) * 120]
        c[sl] = 3
        n[sl] = p
    X = _star(I, [0, 1], c, n)
    prep = orc.prepare(X)
    K = 200
    want = orc.canon_fit(prep, K=K)
    kth = prep.n[want["idx"][0, K - 1]]
    # neighbours of the half step on both sides of the K-th place
    assert np.any(prep.n[want["idx"][0, :K]] > kth - 2) and np.count_nonzero(n[cols] > kth) > 0
    for K2 in (200, 300, 121, 359):
        w2 = orc.canon_fit(prep, K=K2)
        _run(engine, capfd, X, K2, w2, variants=((0, -1), (DBG_TINY_LIST, -1), (DBG_MULTI_PASS, -1)))


# ---------------------------------------------------------------------------------------------------------------
# fp32 keys with counts above 4,096


def _unit_pairs(cmin=4097, cmax=4400, nmax=20000, want=4):
    """(c1, n1, c2, n2) with c1^2 n2 - c2^2 n1 = +-1, c <= n <= nmax."""
    out = []
    for c1 in range(cmin, cmax):
        m = c1 * c1
        for c2 in range(c1 + 1, cmax):
            if math.gcd(c1, c2) != 1:
                continue
            inv = pow(c2 * c2, -1, m)
            for s in (1, -1):
                n1 = (-s * inv) % m  # c2^2 n1 = -s (mod c1^2)
                if c2 <= n1 <= nmax:
                    n2 = (c2 * c2 * n1 + s) // (c1 * c1)
                    if c1 <= n2 <= nmax and c1 * c1 * n2 - c2 * c2 * n1 == s:
                        out.append((c1, n1, c2, n2))
                        if len(out) >= want:
                            return out
    return out


def test_fp32_key_precision_with_unit_gaps(engine, capfd):
    pairs = _unit_pairs()
    assert len(pairs) >= 2
    K = 10
    blocks = []
    base = 0
    for (c1, n1, c2, n2) in pairs[:3]:
        # target row t; 9 items clearly better (c = n = 4500), then the pair at places 10 / 11, then 20 weaker
        I_b = 64
        c = np.zeros(I_b, np.int64)
        n = np.zeros(I_b, np.int64)
        c[1:10], n[1:10] = 4500, 4500
        c[10], n[10] = c1, n1
        c[11], n[11] = c2, n2
        c[12:32], n[12:32] = 100, 20000
        blocks.append(_star(I_b, [0], c, n))
        base += I_b
    I = base
    hists = []
    for b, Xb in enumerate(blocks):
        for u in range(Xb.shape[0]):
            hists.append(Xb.indices[Xb.indptr[u] : Xb.indptr[u + 1]] + 64 * b)
    X = _csr(hists, I)
    prep = orc.prepare(X)
    assert prep.n[0] > 4096
    want = orc.canon_fit(prep, K=K)
    for b, (c1, n1, c2, n2) in enumerate(pairs[:3]):
        a = int(np.flatnonzero(want["idx"][64 * b] == 64 * b + 10)[0]) if 64 * b + 10 in want["idx"][64 * b] else K
        bb = int(np.flatnonzero(want["idx"][64 * b] == 64 * b + 11)[0]) if 64 * b + 11 in want["idx"][64 * b] else K
        assert {a, bb} == {9, K}  # exactly one of the pair keeps the K-th place
        assert int(F32(c1) * F32(c1)) != c1 * c1 or int(F32(c2) * F32(c2)) != c2 * c2  # c^2 is rounded in fp32
    _run(engine, capfd, X, K, want, variants=((0, -1), (DBG_TINY_LIST, -1), (DBG_MULTI_PASS, -1)))
    _run(engine, capfd, X, 11, orc.canon_fit(prep, K=11))


# ---------------------------------------------------------------------------------------------------------------
# K sweep


KS = [1, 2, 31, 32, 33, 63, 64, 65, 255, 256, 511, 512, 513, 1024, 2048, 4096]


@pytest.fixture(scope="module")
def sweep_case():
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(12000, 5000, 240_000, seed=11, item_exp=1.0)
    prep = orc.prepare(X)
    return X, prep, orc.canon_fit(prep, K=4096)


@pytest.mark.parametrize("K", KS)
def test_k_sweep(engine, capfd, sweep_case, K):
    X, prep, full = sweep_case
    want = {"idx": full["idx"][:, :K], "cnt": full["cnt"][:, :K], "val": full["val"][:, :K],
            "len": np.minimum(full["len"], K)}
    assert np.any(full["len"] > K) or K >= 2048
    assert np.any((full["len"] < K) & (full["len"] > 0)) or K <= 2
    g = _geom(5000, K, U=12000)
    assert g["cap"] == max(1024, _np2(2 * K)) and g["P"] == 1 and g["use_code"]
    paths = _run(engine, capfd, X, K, want, device=K in (1, 513, 4096))
    paths.geometry(g)
    _run(engine, capfd, X, K, want, variants=((DBG_MULTI_PASS, -1),))
    if K in (1, 64, 513, 4096):
        _run(engine, capfd, X, K, orc.canon_fit(prep, K=K, similarity="conditional_probability"),
             "conditional_probability")


@pytest.mark.parametrize("K", [49, 50, 64, 4096])
def test_k_at_least_the_item_count(engine, capfd, K):
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(400, 50, 3000, seed=12)
    prep = orc.prepare(X)
    for sim in ("cosine", "conditional_probability"):
        _run(engine, capfd, X, K, orc.canon_fit(prep, K=K, similarity=sim), sim,
             variants=((0, -1), (DBG_TINY_LIST, -1), (DBG_MULTI_PASS, -1)))


# ---------------------------------------------------------------------------------------------------------------
# geometry edges


def _sparse(I, U=30000, seed=0):
    rng = np.random.default_rng(seed)
    d = rng.integers(2, 12, size=U)
    hists = [rng.choice(I, size=k, replace=False) for k in d]
    # a few heavier users so that some rows have more than K candidates
    hists += [rng.choice(I, size=3000, replace=False) for _ in range(4)]
    return _csr(hists, I)


def _edge_cases():
    cases = []
    for K in (200, 1024, 4096):
        for sim in ("cosine", "conditional_probability"):
            cos = sim == "cosine"
            last = _last_p1(K, cos)
            Is = {last, last + 1}
            for lo, hi in _bands(K, cos)[:2]:
                Is.add((lo + hi) // 2)
            if K == 200 and cos:
                Is |= {_code_limit(K), _code_limit(K) + 1}
            for I in sorted(Is):
                cases.append((K, sim, I))
    return cases


def _properties(got, X, prep, K, cosine, rows):
    n = prep.n
    idx, cnt, ln = got["idx"], got["cnt"].astype(np.int64), got["len"]
    mask = np.arange(K)[None, :] < ln[:, None]
    assert np.all(ln >= 0) and np.all(idx[mask] >= 0) and np.all(idx[~mask] == -1) and np.all(cnt[~mask] == 0)
    assert not np.any(idx == np.arange(rows[0], rows[1])[:, None])
    nj = n[np.maximum(idx, 0)]
    assert np.all(cnt[mask] >= 1) and np.all(cnt[mask] <= np.minimum(n[rows[0]:rows[1], None], nj)[mask])
    both = mask[:, 1:]
    a, b = (cnt[:, :-1] ** 2 * nj[:, 1:], cnt[:, 1:] ** 2 * nj[:, :-1]) if cosine else (cnt[:, :-1], cnt[:, 1:])
    assert np.all((a >= b)[both])
    assert np.all((idx[:, :-1] < idx[:, 1:])[(a == b) & both])
    assert not np.any(np.isnan(got["val"]))


@pytest.mark.parametrize("K,similarity,I", _edge_cases())
def test_geometry_edges(engine, capfd, K, similarity, I):
    cosine = similarity == "cosine"
    X = _sparse(I, seed=I % 1000)
    prep = orc.prepare(X)
    g = _geom(I, K, U=X.shape[0], cosine=cosine)
    assert g["over"] <= 0
    rows = (I - 1536, I)  # the geometry depends on I alone; the tail rows keep the outputs small at K = 4096
    paths = Paths()
    for dev in (False, True):
        got = _fit(engine, capfd, X, K, similarity, device=dev, rows=rows, paths=paths)
        _properties(got, X, prep, K, cosine, rows)
        sample = np.random.default_rng(I).choice(rows[1] - rows[0], size=64, replace=False)
        sample = np.unique(np.concatenate([sample, [0, rows[1] - rows[0] - 1]]))
        want = orc.canon_fit(prep, K=K, similarity=similarity, rows=rows[0] + sample, block=16)
        _same(got, want, f"I={I} K={K} {similarity} {'device' if dev else 'host'}", rows=sample)
    paths.geometry(g)


def test_geometry_mirror_matches_the_device(smem_max):
    assert smem_max == SMEM_OPTIN_B200


# ---------------------------------------------------------------------------------------------------------------
# mid shape, every row


@pytest.fixture(scope="module")
def mid_case():
    from recpack_b200.synth import synth_interactions

    X = synth_interactions(40000, 8000, 1_200_000, seed=21)
    prep = orc.prepare(X)
    return X, prep, {"cosine": orc.canon_fit(prep, K=200, block=512),
                     "conditional_probability": orc.canon_fit(prep, K=100, similarity="conditional_probability", block=512)}


@pytest.mark.parametrize("similarity,K", [("cosine", 200), ("conditional_probability", 100)])
def test_mid_shape_every_row(engine, capfd, mid_case, similarity, K):
    X, prep, wants = mid_case
    want = wants[similarity]
    if similarity == "cosine":
        guessed = sum(_b0(X, prep, i, K, True)[1] is True for i in np.argsort(-prep.n)[:40])
        assert guessed >= 20
    paths = _run(engine, capfd, X, K, want, similarity, variants=((0, -1), (0, 64)), device=True)
    if similarity == "cosine":
        paths.require("guess_ok", at_least=100)
        paths.require("deferred", at_least=1000)
