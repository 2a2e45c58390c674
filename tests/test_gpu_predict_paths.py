"""Every fallback branch of the 32-bit top-N kernel (k_predict_a32), compared with the oracle bit for bit.

The kernel runs the item ranges of a user one after the other on approximate 32-bit sums and leaves them only where it
cannot prove the order.  Each case below builds a model and users that force one such branch:

  handoff              more survivors than the list holds: the user goes to the two-limb kernel (k_predict, which
                       writes the final lists of the handed-over users only)
  carried retry        the bound carried from the earlier ranges lets more than cap - N items of a later range through:
                       that range is swept again with its own bound
  exact restart        an approximate entry of an earlier range is too close to a later range's exact one: the user is
                       run again with exact sums throughout
  history lengths      more than one staged chunk of rows, exact sums from the start (d >= 2048), two 20-bit limbs up
                       to d = 4095 and 64-bit adds above, sums that reach the bound of the per-user shift
  long segments        model row segments of more than 96 entries (the tail loop of the row sweep)
  N sweep              warp ranking, counting and bitonic ordering of the list, lists larger than a user's candidates
  production geometry  I = 59,047 with more users than CTAs, the default and the one-CTA geometry
  geometry cache       one model, calls whose N and flags change the number of item ranges

Every call runs in both modes (lists only, and lists with scores) into outputs poisoned beforehand, so that a row
that no kernel writes fails.  Each case asserts on the oracle side that its construction reaches the branch, and,
with the instrumented build (-DRPK_PHASE_PROF, which prints one "[predict32 phases]" line per call), that the
kernel's counter of that branch moved.  The last tests compare lists-only mode at the full ML-25M and Netflix shapes
with the two-limb kernel for every user, and with the oracle on a sample."""
import re

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle import recpack_oracle as orc

pytestmark = pytest.mark.gpu

DBG_WIDE_ACC, DBG_TINY_LIST, DBG_MULTI_PASS, DBG_MANY_PASS = 1, 2, 4, 32
A32_EXACT_D = 2048  # histories at least this long get exact sums from the start (predict.cu)
Q_MAX = (1 << 40) - (1 << 10)  # q of v = 1 - 2^-30, the largest value of a model whose scale exponent is 40
COUNTERS = ("carried retries", "exact range passes", "exact restarts", "overflow users", "P", "R")


@pytest.fixture(scope="module")
def engine():
    from recpack_b200.engine import get_engine

    eng = get_engine(0)
    with pytest.MonkeyPatch.context() as mp:
        mp.delenv("RPK_PRED_CTAS", raising=False)
        yield eng
        eng.debug_flags(0)
        eng.predict_item_filter(None)


# ---------------------------------------------------------------------------------------------------------------
# models, users, the oracle side


def _q(v):
    """Values that are multiples of 2^-40 below 1: with the model's largest value in [0.5, 1) the scale is 2^40 and
    q = v * 2^40 exactly."""
    return np.asarray(v, dtype=np.float64) * 2.0**-40


def _finish(I, idx, val, ln):
    S = orc.topk_to_csr(idx, val, ln, I)
    q = orc.canon_quantize(S.data)
    rowmax = np.zeros(I, dtype=np.int64)
    nz = np.flatnonzero(np.diff(S.indptr) > 0)
    if len(nz):
        rowmax[nz] = np.maximum.reduceat(q, S.indptr[nz])
    Sq = csr_matrix((q, S.indices, S.indptr), shape=S.shape)
    return {"I": I, "K": idx.shape[1], "idx": idx, "val": val, "ln": ln, "S": S, "Sq": Sq, "rowmax": rowmax}


def _model(I, rows):
    """rows: {item: (columns, q values)}; items not named have empty rows."""
    K = max([len(c) for c, _ in rows.values()] + [1])
    idx = np.zeros((I, K), dtype=np.int32)
    val = np.zeros((I, K))
    ln = np.zeros(I, dtype=np.int32)
    for i, (c, q) in rows.items():
        c = np.asarray(c, dtype=np.int32)
        assert len(np.unique(c)) == len(c)
        o = np.argsort(c)
        ln[i] = len(c)
        idx[i, : len(c)] = c[o]
        val[i, : len(c)] = _q(np.asarray(q, dtype=np.int64)[o])
    return _finish(I, idx, val, ln)


def _users(I, hists):
    hists = [np.unique(np.asarray(h, dtype=np.int32)) for h in hists]
    indptr = np.concatenate([[0], np.cumsum([len(h) for h in hists])]).astype(np.int64)
    indices = np.concatenate(hists + [np.zeros(0, np.int32)]).astype(np.int32)
    X = csr_matrix((np.ones(len(indices), dtype=np.int32), indices, indptr), shape=(len(hists), I))
    return {"U": len(hists), "hists": hists, "X": X, "indptr": indptr, "indices": indices}


def _load(engine, model):
    engine.model_load_topk(model["I"], model["K"], model["idx"], model["val"], model["ln"])


def _shift(model, hist):
    """The kernel's shift of one user's 32-bit sums: B = sum over the history rows of ceil(rowmax_q / 2^20) * 2^20,
    s = the smallest shift with (B >> s) + d <= 2^32 - 1."""
    d = len(hist)
    b20 = int(np.sum((model["rowmax"][np.asarray(hist, dtype=np.int64)] + (1 << 20) - 1) >> 20))
    B = b20 << 20
    s = 0
    while (B >> s) + d > (1 << 32) - 1:
        s += 1
    return s


def _margin(model, hist):
    """Width 2 d * 2^s (in q units) of the interval an approximate sum stands for."""
    return (2 * len(hist)) << _shift(model, hist)


def _scores(model, hist, mask=True, allowed=None):
    """(candidate items, exact q sums) of one user, best first by (score desc, index asc)."""
    row = np.asarray(model["Sq"][np.asarray(hist, dtype=np.int64)].sum(axis=0)).ravel().astype(np.int64)
    ok = row > 0
    if mask:
        ok[np.asarray(hist, dtype=np.int64)] = False
    if allowed is not None:
        ok &= allowed
    items = np.flatnonzero(ok)
    sc = row[items]
    o = np.lexsort((items, -sc))
    return items[o], sc[o]


def _cap(N, flags):
    return max(64 if flags & DBG_TINY_LIST else 256, 1 << max(0, (2 * N - 1).bit_length()))


def _range_len(I, flags):
    P = 4 if flags & DBG_MANY_PASS else 2 if flags & DBG_MULTI_PASS else 1
    return ((I + P - 1) // P + 3) & ~3


def _want(model, users, N, mask, allowed):
    X, S = users["X"], model["S"]
    if allowed is None:
        return orc.canon_predict_topn(X, S, N, remove_history=mask)
    full = orc.canon_predict_topn(X, S, model["I"], remove_history=mask)
    U = users["U"]
    want = {"idx": np.full((U, N), -1, np.int32), "val": np.zeros((U, N)), "len": np.zeros(U, np.int32)}
    for u in range(U):
        keep = [t for t in range(full["len"][u]) if allowed[full["idx"][u, t]]][:N]
        want["idx"][u, : len(keep)] = full["idx"][u, keep]
        want["val"][u, : len(keep)] = full["val"][u, keep]
        want["len"][u] = len(keep)
    return want


def _truncate(want, N):
    return {"idx": want["idx"][:, :N], "val": want["val"][:, :N], "len": np.minimum(want["len"], N)}


# ---------------------------------------------------------------------------------------------------------------
# calls into poisoned outputs, the phase counters of the instrumented build


def _phase_lines(text):
    out = []
    for line in text.splitlines():
        if line.startswith("[predict32 phases]"):
            out.append({k: int(re.search(r"\b" + k + r"=(\d+)", line).group(1)) for k in COUNTERS})
    return out


def _predict(engine, capfd, users, N, mask, want_val, device):
    U = users["U"]
    if device:
        import torch

        indptr = torch.from_numpy(users["indptr"]).cuda()
        indices = torch.from_numpy(users["indices"]).cuda()
        out = {"idx": torch.full((U, N), -2, dtype=torch.int32, device="cuda"),
               "val": torch.full((U, N), float("nan"), dtype=torch.float64, device="cuda") if want_val else None,
               "len": torch.full((U,), -3, dtype=torch.int32, device="cuda")}
        torch.cuda.synchronize()
    else:
        indptr, indices = users["indptr"], users["indices"]
        out = {"idx": np.full((U, N), -2, np.int32), "val": np.full((U, N), np.nan) if want_val else None,
               "len": np.full(U, -3, np.int32)}
    capfd.readouterr()
    engine.predict_topn(U, indptr, indices, N, mask_history=mask, want_val=want_val, out=out)
    if device:
        engine.sync()
        out = {k: (v.cpu().numpy() if v is not None else None) for k, v in out.items()}
    return out, _phase_lines(capfd.readouterr().err)


def _assert_same(got, want, what):
    for key in ("len", "idx", "val"):
        if got.get(key) is None:
            continue
        g, w = got[key], want[key]
        bad = np.flatnonzero(np.any((g != w).reshape(len(g), -1), axis=1))
        assert len(bad) == 0, (f"{what}: {key} differs for {len(bad)} users, first {bad[:8].tolist()}; "
                               f"user {bad[0]}: got {g[bad[0]].ravel()[:12].tolist()} want {w[bad[0]].ravel()[:12].tolist()}")


class Paths:
    """Phase counters of the calls of one case, per mode; empty under the normal build."""

    def __init__(self):
        self.lines = {"lists": [], "scores": []}

    def total(self, key, mode=None):
        modes = [mode] if mode else list(self.lines)
        return sum(line[key] for m in modes for line in self.lines[m])

    def seen(self, mode=None):
        modes = [mode] if mode else list(self.lines)
        return any(self.lines[m] for m in modes)

    def require(self, key, mode=None, at_least=1):
        """The named counter moved in this case's calls (instrumented build only; the comparisons do not depend on it)."""
        if not self.seen(mode):
            print(f"path counter '{key}': no phase line (normal build), not checked")
            return
        n = self.total(key, mode)
        print(f"path counter '{key}' ({mode or 'both modes'}): {n}, required >= {at_least}")
        assert n >= at_least, f"the case did not reach its branch: '{key}' = {n}"

    def forbid(self, key, mode=None):
        if self.seen(mode):
            n = self.total(key, mode)
            print(f"path counter '{key}' ({mode or 'both modes'}): {n}, required 0")
            assert n == 0, f"'{key}' = {n}"

    def geometry(self, P=None, R=None):
        for lines in self.lines.values():
            for line in lines:
                if P is not None:
                    assert line["P"] == P, line
                if R is not None:
                    assert line["R"] == R, line


def _check(engine, capfd, model, users, N, flags=0, mask=True, allowed=None, device=False, want=None, paths=None):
    """Both modes against the oracle (model already loaded); returns the phase counters."""
    want = _want(model, users, N, mask, allowed) if want is None else want
    paths = Paths() if paths is None else paths
    engine.debug_flags(flags)
    engine.predict_item_filter(None if allowed is None else allowed.astype(np.uint8))
    try:
        for mode, want_val in (("lists", False), ("scores", True)):
            for dev in ((False, True) if device else (False,)):
                got, lines = _predict(engine, capfd, users, N, mask, want_val, dev)
                paths.lines[mode] += lines
                _assert_same(got, want, f"N={N} flags={flags} mask={mask} filter={allowed is not None} {mode} "
                                        f"{'device' if dev else 'host'} outputs")
    finally:
        engine.debug_flags(0)
        engine.predict_item_filter(None)
    return paths


# ---------------------------------------------------------------------------------------------------------------
# 1, 3: handoff to the two-limb kernel

I_HUB = 1024
HUB_ITEMS = np.arange(100, 500)  # 400 items: 156 in the first range of four, 244 in the second
HUB_Q = 3 << 37


def _hub_case(seed):
    """Hub rows 600..609 hold the 400 hub items at one value (exact ties), rows 610..619 the same items a few q units
    apart (near ties); every other row is an ordinary weaker row."""
    rng = np.random.default_rng(seed)
    rows = {}
    for h in range(600, 610):
        rows[h] = (HUB_ITEMS, np.full(400, HUB_Q))
    for h in range(610, 620):
        rows[h] = (HUB_ITEMS, HUB_Q + rng.integers(0, 8, size=400))
    for i in range(I_HUB):
        if i not in rows:
            c = rng.choice(I_HUB, size=rng.integers(1, 24), replace=False)
            rows[i] = (c, rng.integers(1 << 30, 1 << 38, size=len(c)))
    model = _model(I_HUB, rows)
    ordinary = [rng.choice(np.setdiff1d(np.arange(I_HUB), np.arange(600, 620)), size=rng.integers(1, 12), replace=False)
                for _ in range(40)]
    ordinary[5] = []
    hubs = [[600], [603, 607], [610], [612, 615]]
    hists = ordinary[:10] + hubs[:2] + ordinary[10:25] + hubs[2:] + ordinary[25:]  # hub users 10, 11, 27, 28
    hub_users = [10, 11, 27, 28]
    return model, _users(I_HUB, hists), hub_users


def _close_group(model, hist, N, allowed=None, lo=0, hi=None):
    """Candidates in [lo, hi) whose exact scores lie within the margin of the N-th best one's: they survive any bound."""
    items, sc = _scores(model, hist, allowed=allowed)
    sel = (items >= lo) & (items < (model["I"] if hi is None else hi))
    items, sc = items[sel], sc[sel]
    if len(sc) == 0:
        return 0
    nth = sc[min(N, len(sc)) - 1]
    return int(np.count_nonzero(sc >= nth - _margin(model, hist)))


@pytest.mark.parametrize("flags", [0, DBG_MULTI_PASS, DBG_TINY_LIST, DBG_MULTI_PASS | DBG_TINY_LIST])
def test_handoff_of_tie_groups_larger_than_the_list(engine, capfd, flags):
    model, users, hub_users = _hub_case(21)
    N = 10
    for u in hub_users:  # every hub item survives any bound, all of them in the first range
        assert _close_group(model, users["hists"][u], N, hi=_range_len(I_HUB, flags)) > _cap(N, flags)
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, flags, device=flags == 0)
    _check(engine, capfd, model, users, N, flags, mask=False, paths=paths)
    paths.require("overflow users", "lists", at_least=len(hub_users))
    paths.require("overflow users", "scores", at_least=len(hub_users))


def test_handoff_honours_the_item_filter(engine, capfd):
    model, users, hub_users = _hub_case(22)
    N = 10
    allowed = np.random.default_rng(23).random(I_HUB) < 0.8
    allowed[[101, 102, 103]] = False  # the best-indexed ties
    for u in hub_users:
        assert _close_group(model, users["hists"][u], N, allowed) > _cap(N, 0)
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, 0, allowed=allowed, device=True)
    paths.require("overflow users", at_least=2 * len(hub_users))


@pytest.mark.parametrize("flags", [DBG_MANY_PASS])
def test_carried_retry_then_handoff(engine, capfd, flags):
    model, users, hub_users = _hub_case(24)
    N = 20
    R = _range_len(I_HUB, flags)
    cap = _cap(N, flags)
    for u in hub_users:
        h = users["hists"][u]
        # range 0 fills the list with ties; range 1 has more close ones than the places left
        assert N <= _close_group(model, h, N, hi=R) <= cap
        assert _close_group(model, h, N, lo=R, hi=2 * R) > cap - N
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, flags)
    for mode in ("lists", "scores"):
        paths.require("carried retries", mode, at_least=len(hub_users))
        paths.require("overflow users", mode, at_least=len(hub_users))


# ---------------------------------------------------------------------------------------------------------------
# 2: carried retry that succeeds


def test_carried_retry_that_fits(engine, capfd):
    I, N, flags = 1024, 10, DBG_MULTI_PASS
    R = _range_len(I, flags)
    assert R == 512
    rng = np.random.default_rng(31)
    weak = np.arange(20)
    strong = 520 + np.arange(300)
    rows = {1000: (np.r_[weak, strong], np.r_[(1 << 20) + (weak << 14), (np.float64(1 << 39) * 0.96 ** np.arange(300)).astype(np.int64)]),
            1001: (np.r_[weak[:15], strong[::2]], np.r_[(1 << 21) + (weak[:15] << 15), (np.float64(1 << 38) * 0.93 ** np.arange(150)).astype(np.int64)])}
    for i in range(I):
        if i not in rows:
            c = rng.choice(I, size=rng.integers(1, 16), replace=False)
            rows[i] = (c, rng.integers(1 << 20, 1 << 36, size=len(c)))
    model = _model(I, rows)
    hists = [rng.choice(1000, size=rng.integers(1, 10), replace=False) for _ in range(30)]
    hists[7] = [1000]
    hists[19] = [1001, 1000]
    users = _users(I, hists)
    for u in (7, 19):
        items, sc = _scores(model, users["hists"][u])
        r0 = sc[items < R]
        assert len(r0) >= N
        # every range-1 candidate beats the list the first range leaves: the carried bound passes them all
        assert np.count_nonzero((items >= R) & (sc > r0[0])) > _cap(N, flags) - N
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, flags)
    paths.require("carried retries", "lists", at_least=2)
    paths.require("carried retries", "scores", at_least=2)
    paths.forbid("overflow users")


# ---------------------------------------------------------------------------------------------------------------
# 4: exact restart


def _restart_rows(rng, first, last, place, loose, N):
    """Three model rows (d = 3) with item x in `first` and item y in `last` at list places `place` and `place + 1`.
    One of the two is "loose": each of its q is an even multiple of 2^s, so its approximate sum stands 2 d units of 2^s
    above its exact one; the other is "tight": odd multiples plus 2^s - 1, 3 q units above.  The tight one is exactly
    2^(s+1) - 3 ahead, the loose one ahead by 4 units in the approximate order, so neither half the margin nor a carried
    bound without the - d proves the right order.  The other places are well separated; the ones ahead of x are in
    `first`, so that at place N - 1 x is the N-th entry of the list the first range leaves."""
    ahead = rng.choice(first, size=place, replace=False)  # x is at place `place` of its own range
    others = np.r_[ahead, rng.choice(np.setdiff1d(np.r_[first, last], ahead), size=N + 4 - place, replace=False)]
    x = int(rng.choice(np.setdiff1d(first, others)))
    y = int(rng.choice(np.setdiff1d(last, others)))
    levels = (1 << 39) - np.arange(N + 6, dtype=np.int64) * (1 << 33)
    B = 3 * (((int(levels[0]) + (1 << 20) - 1) >> 20) << 20)
    s = 0
    while (B >> s) + 3 > (1 << 32) - 1:
        s += 1
    M = int(levels[place] >> s) | 1
    q_loose = np.array([M + 1, M + 1, M - 1], dtype=np.int64) << s  # sum 3M + 1 units of 2^s, approximate 3M + 4
    q_tight = (np.full(3, M, dtype=np.int64) << s) + (1 << s) - 1  # sum (3M + 3) 2^s - 3, approximate 3M
    qx, qy = (q_loose, q_tight) if loose == "x" else (q_tight, q_loose)
    q_other = np.r_[levels[:place], levels[place + 2 :]][: len(others)]
    rows = [(np.r_[others, x, y], np.r_[q_other, qx[k], qy[k]]) for k in range(3)]
    return rows, x, y


@pytest.mark.parametrize("flags", [DBG_MULTI_PASS, DBG_MANY_PASS])
def test_exact_restart_on_a_near_tie_across_ranges(engine, capfd, flags):
    I, N = 1024, 6
    R = _range_len(I, flags)
    P = -(-I // R)
    rng = np.random.default_rng(41 + flags)
    first, last = np.arange(0, R), np.arange((P - 1) * R, 990)
    rows, pairs, hists = {}, [], []
    h = 990
    for place in (0, N // 2, N - 1):
        for loose in ("x", "y"):
            three, x, y = _restart_rows(rng, first, last, place, loose, N)
            for k in range(3):
                rows[h + k] = three[k]
            pairs.append((len(hists), x, y, place))
            hists.append([h, h + 1, h + 2])
            h += 3
    for i in range(I):
        if i not in rows:
            c = rng.choice(I, size=rng.integers(1, 8), replace=False)
            rows[i] = (c, rng.integers(1 << 10, 1 << 25, size=len(c)))
    hists += [rng.choice(990, size=rng.integers(1, 6), replace=False) for _ in range(10)]
    model = _model(I, rows)
    users = _users(I, hists)
    for u, x, y, place in pairs:
        hist = users["hists"][u]
        items, sc = _scores(model, hist)
        W = _margin(model, hist)
        px, py = int(np.flatnonzero(items == x)[0]), int(np.flatnonzero(items == y)[0])
        assert {px, py} == {place, place + 1}
        assert abs(int(sc[px]) - int(sc[py])) < W  # closer than the margin
        rest = np.delete(sc, [px, py])
        assert np.min(np.abs(rest - sc[px])) > 4 * W  # well separated from everything else
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, flags)
    paths.require("exact restarts", "lists", at_least=len(pairs))
    paths.forbid("exact restarts", "scores")


# ---------------------------------------------------------------------------------------------------------------
# 5: history lengths

I_LONG = 6000
A_ITEM, B_ITEM = 7, 5990  # in every row, at the model's largest value (B one q unit lower)
LONG_D = [511, 512, 513, 1024, 2047, 2048, 4095, 4096, 5000]


def _long_case(seed):
    rng = np.random.default_rng(seed)
    I = I_LONG
    K = 16
    cols = np.empty((I, K), dtype=np.int64)
    pool = np.setdiff1d(np.arange(I), [A_ITEM, B_ITEM])
    for i in range(I):
        cols[i, :2] = (A_ITEM, B_ITEM)
        cols[i, 2:] = rng.choice(pool, size=K - 2, replace=False)
    qv = rng.integers(1 << 20, 1 << 38, size=(I, K))
    qv[:, 0], qv[:, 1] = Q_MAX, Q_MAX - 1
    o = np.argsort(cols, axis=1)
    idx = np.take_along_axis(cols, o, axis=1).astype(np.int32)
    val = _q(np.take_along_axis(qv, o, axis=1))
    model = _finish(I, idx, val, np.full(I, K, dtype=np.int32))
    hists = [rng.choice(pool, size=d, replace=False) for d in LONG_D]
    hists += [rng.choice(pool, size=d, replace=False) for d in (1, 2, 3, 100, 700)]
    hists.append([])
    return model, _users(I, hists)


@pytest.mark.parametrize("flags", [0, DBG_MULTI_PASS, DBG_MANY_PASS])
def test_history_lengths_and_sums_at_the_shift_bound(engine, capfd, flags):
    model, users = _long_case(51)
    N = 20
    for hist in users["hists"][: len(LONG_D)]:
        d = len(hist)
        s = _shift(model, hist)
        top = d * ((Q_MAX >> s) | 1)  # approximate sum of A
        assert top + d <= (1 << 32) - 1 and 2 * (top + d) > (1 << 32) - 1  # in the top octave of the 32-bit sums
        items, sc = _scores(model, hist)
        assert items[0] == A_ITEM and items[1] == B_ITEM and sc[0] - sc[1] == d < _margin(model, hist)
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, flags)
    if flags == 0:
        _check(engine, capfd, model, users, N, flags, mask=False, paths=paths)
    paths.geometry(P={0: 1, DBG_MULTI_PASS: 2, DBG_MANY_PASS: 4}[flags])
    paths.require("exact range passes", "lists")


# ---------------------------------------------------------------------------------------------------------------
# 6: long row segments


@pytest.mark.parametrize("flags", [0, DBG_MULTI_PASS])
def test_long_row_segments(engine, capfd, flags):
    I = 1024
    rng = np.random.default_rng(61)
    lengths = [96, 97, 128, 400]
    rows = {}
    for k in range(40):  # rows 900..939, every entry in the first range of two
        n = lengths[k % 4]
        rows[900 + k] = (rng.choice(512, size=n, replace=False), rng.integers(1 << 24, 1 << 39, size=n))
    for i in range(I):
        if i not in rows:
            c = rng.choice(I, size=rng.integers(1, 10), replace=False)
            rows[i] = (c, rng.integers(1 << 20, 1 << 30, size=len(c)))
    model = _model(I, rows)
    hists = [[900], [901], [902], [903], [900, 901, 903], [901, 902, 903], list(range(900, 940)), list(range(910, 950))]
    hists += [rng.choice(I, size=rng.integers(1, 8), replace=False) for _ in range(8)]
    users = _users(I, hists)
    _load(engine, model)
    for N in (10, 50):
        _check(engine, capfd, model, users, N, flags)
    _check(engine, capfd, model, users, 10, flags, mask=False)


# ---------------------------------------------------------------------------------------------------------------
# 7, 9: N sweep and the geometry cache


def _sweep_case():
    I, K = 4096, 64
    rng = np.random.default_rng(71)
    pop = rng.random(I) ** 3  # skewed item popularity
    pop /= pop.sum()
    idx = np.zeros((I, K), dtype=np.int32)
    val = np.zeros((I, K))
    ln = rng.integers(1, K + 1, size=I).astype(np.int32)
    for i in range(I):
        c = np.sort(rng.choice(I, size=ln[i], replace=False, p=pop))
        idx[i, : ln[i]] = c
        val[i, : ln[i]] = _q(rng.integers(1 << 20, 1 << 39, size=ln[i]))
    model = _finish(I, idx, val, ln)
    hists = [rng.choice(I, size=1 + u % 80, replace=False) for u in range(400)]
    return model, _users(I, hists)


@pytest.fixture(scope="module")
def sweep():
    model, users = _sweep_case()
    want = orc.canon_predict_topn(users["X"], model["S"], 2048, remove_history=True)
    return model, users, want


@pytest.mark.parametrize("N", [1, 31, 32, 33, 64, 65, 129, 513, 2048])
def test_n_sweep(engine, capfd, sweep, N):
    model, users, want = sweep
    assert np.any(want["len"] < N) or N < 64  # lists longer than some users' candidates
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, want=_truncate(want, N))
    cand = [len(_scores(model, h)[0]) for h in users["hists"]]
    over = sum(c > _cap(N, 0) for c in cand)
    if N > 512 and over:  # the own bound cannot cut: users with more candidates than the list are handed over
        paths.require("overflow users", "lists", at_least=over)


def test_geometry_cache_between_calls(engine, capfd, sweep):
    model, users, want = sweep
    _load(engine, model)
    for N, flags in [(5, 0), (2048, 0), (5, 0), (5, DBG_MANY_PASS), (5, 0), (2048, DBG_MANY_PASS), (5, 0)]:
        _check(engine, capfd, model, users, N, flags, want=_truncate(want, N))


# ---------------------------------------------------------------------------------------------------------------
# 8: production geometry, mixed batch

I_PROD, K_PROD = 59_047, 200


def _prod_case():
    """Random skewed rows at the ML-25M item count, plus the constructions of the cases above remapped into the
    catalogue, and users without history, with empty history rows only and with every candidate in their history."""
    rng = np.random.default_rng(81)
    I, K = I_PROD, K_PROD
    pop = rng.random(I) ** 4
    cols = np.minimum((rng.random((I, 2 * K)) ** 2.5 * I).astype(np.int64), I - 1)
    cols = rng.permutation(I)[cols]  # the popular items spread over the catalogue
    cols.sort(axis=1)
    dup = np.zeros_like(cols, dtype=bool)
    dup[:, 1:] = cols[:, 1:] == cols[:, :-1]
    key = np.where(dup, 2.0, rng.random(cols.shape))
    o = np.argsort(key, axis=1)[:, :K]
    cols = np.take_along_axis(cols, o, axis=1)
    n_uniq = (~dup).sum(axis=1)
    ln = np.minimum(n_uniq, np.maximum(1, (rng.pareto(1.0, I) * 12).astype(np.int64))).clip(max=K)
    ln[rng.choice(I, 40, replace=False)] = 0  # empty rows
    qv = (np.float64(1 << 39) * 0.5 ** rng.exponential(4.0, size=(I, K)) * (0.9 + 0.1 * pop[cols])).astype(np.int64) + 1
    special = {}
    # case 1: two users whose two hub rows hold 200 items each at one value (400 ties over all three ranges),
    # one with near ties
    hub_items = rng.choice(19_000, size=800, replace=False)  # all in the first range
    hub_rows = rng.choice(np.flatnonzero(ln > 0), size=6, replace=False)
    for k, r in enumerate(hub_rows):
        its = hub_items[(k % 4) * 200 : (k % 4) * 200 + 200]
        special[r] = (its, np.full(200, HUB_Q) + (rng.integers(0, 8, 200) if k >= 4 else 0))
    # case 4: x in the first range, y in the last (three ranges of 19,684, two of the one-CTA geometry)
    restart_users = []
    free = np.setdiff1d(np.flatnonzero(ln > 0), list(special))
    for k, (place, loose) in enumerate(((0, "x"), (3, "y"), (5, "x"))):
        three, _, _ = _restart_rows(rng, np.arange(0, 19_000), np.arange(40_000, I), place, loose, 6)
        hr = free[[3 * k, 3 * k + 1, 3 * k + 2]]
        for r, row in zip(hr, three):
            special[r] = row
        restart_users.append(list(hr))
    # case 5: 5,000 rows that point to A and B at the model's largest value
    a, b = 12_345, 51_234
    long_rows = rng.choice(np.setdiff1d(np.arange(I), np.r_[list(special), a, b]), size=5000, replace=False)
    # the users whose every candidate is in their history: eight rows pointing only to each other
    clique = rng.choice(np.setdiff1d(np.arange(I), np.r_[list(special), long_rows, a, b]), size=8, replace=False)
    idx = np.zeros((I, K), dtype=np.int32)
    val = np.zeros((I, K))
    for r, (c, q) in special.items():
        o = np.argsort(c)
        ln[r] = len(c)
        idx[r, : len(c)], val[r, : len(c)] = np.asarray(c)[o], _q(np.asarray(q)[o])
    plain = np.setdiff1d(np.arange(I), list(special))
    in_clique, in_long = set(clique.tolist()), set(long_rows.tolist())
    for r in plain:
        n = int(ln[r])
        c, q = cols[r, :n], qv[r, :n]
        if r in in_clique:
            c, q, n = np.setdiff1d(clique, [r]), qv[r, :7], 7
        elif r in in_long:
            keep = (c != a) & (c != b)
            c, q = np.r_[a, b, c[keep]][: max(n, 2)], np.r_[Q_MAX, Q_MAX - 1, q[keep]][: max(n, 2)]
            n = len(c)
        o = np.argsort(c)
        ln[r] = n
        idx[r, :n], val[r, :n] = c[o], _q(q[o])
    model = _finish(I, idx, val, ln.astype(np.int32))
    # users: heavy-tailed history lengths over skewed items, then the special ones
    d = np.minimum((rng.pareto(1.1, 3200) * 6).astype(np.int64) + 1, 3000)
    hists = [rng.choice(I, size=k, replace=False, p=pop / pop.sum()) if k < 200 else rng.choice(I, size=k, replace=False)
             for k in d]
    empty_rows = np.flatnonzero(ln == 0)
    specials = [list(hub_rows[0:2]), list(hub_rows[2:4]), list(hub_rows[4:6])] + restart_users
    specials += [long_rows[:k] for k in (511, 2047, 4095, 5000)]
    specials += [[], [], list(empty_rows[:1]), list(empty_rows[:12]), list(clique), list(clique)]
    for k, h in enumerate(specials):
        hists.insert(37 * k + 11, h)
    return model, _users(I, hists)


@pytest.fixture(scope="module")
def prod():
    model, users = _prod_case()
    want = orc.canon_predict_topn(users["X"], model["S"], 2048, remove_history=True)
    return model, users, want


@pytest.mark.parametrize("N", [20, 2048])
@pytest.mark.parametrize("ctas", ["default", "1"])
def test_production_geometry_mixed_batch(engine, capfd, monkeypatch, prod, ctas, N):
    model, users, want = prod
    assert users["U"] > 2 * 148
    assert np.count_nonzero(want["len"] == 0) >= 6  # no history, empty rows only, every candidate in the history
    if ctas != "default":
        monkeypatch.setenv("RPK_PRED_CTAS", ctas)
    _load(engine, model)
    paths = _check(engine, capfd, model, users, N, device=True, want=_truncate(want, N))
    if N == 20:
        paths.geometry(P=3 if ctas == "default" else 2)
        paths.require("overflow users", "lists", at_least=3)
        paths.require("exact restarts", "lists")


# ---------------------------------------------------------------------------------------------------------------
# lists-only mode at full size: every user against the two-limb kernel, a sample against the oracle

FULL = {
    "ml25m_cosine": dict(shape="ml25m", similarity="cosine", K=200, generator="numpy"),
    "netflix_condprob": dict(shape="netflix", similarity="conditional_probability", K=100, generator="cuda"),
}


@pytest.mark.parametrize("name", list(FULL))
def test_lists_only_full_size(engine, capfd, name):
    import torch

    from recpack_b200.base import lists_to_csr
    from recpack_b200.matrix import binary_structure
    from recpack_b200.synth import make_dataset

    cfg, N = FULL[name], 20
    train, _, _ = make_dataset(cfg["shape"], seed=0, split_seed=42, generator=cfg["generator"])
    U, I = train.shape
    _, indptr, indices = binary_structure(train)
    ptr_d = torch.from_numpy(indptr).cuda()
    idx_d = torch.from_numpy(indices).cuda()
    engine.debug_flags(0)
    fit = engine.fit_topk(U, I, ptr_d, idx_d, cfg["K"], similarity=cfg["similarity"], want_cnt=False)
    engine.model_load_topk(I, cfg["K"], fit["idx"], fit["val"], fit["len"])
    paths = Paths()
    got = {}
    try:
        for flags in (0, DBG_WIDE_ACC):
            engine.debug_flags(flags)
            out = {"idx": torch.full((U, N), -2, dtype=torch.int32, device="cuda"),
                   "len": torch.full((U,), -3, dtype=torch.int32, device="cuda")}
            torch.cuda.synchronize()
            capfd.readouterr()
            engine.predict_topn(U, ptr_d, idx_d, N, mask_history=True, want_val=False, out=out)
            engine.sync()
            paths.lines["lists"] += _phase_lines(capfd.readouterr().err)
            got[flags] = {k: v.cpu().numpy() for k, v in out.items()}
        engine.sync()
        fit = {k: v.cpu().numpy() for k, v in fit.items() if v is not None}
    finally:
        engine.debug_flags(0)
    del ptr_d, idx_d
    torch.cuda.empty_cache()
    _assert_same(got[0], got[DBG_WIDE_ACC], f"{name}: lists-only vs the two-limb kernel")
    S = lists_to_csr(fit["idx"], fit["val"], fit["len"], I)
    S.sort_indices()
    d = np.diff(train.indptr)
    rng = np.random.default_rng(91)
    users = np.unique(np.r_[np.argsort(-d, kind="stable")[:20], rng.choice(U, size=1000, replace=False)])
    want = orc.canon_predict_topn(train[users], S, N, remove_history=True)
    _assert_same({k: v[users] for k, v in got[0].items()}, want, f"{name}: lists-only vs the oracle")
    if name == "ml25m_cosine":
        paths.require("exact restarts", "lists")
