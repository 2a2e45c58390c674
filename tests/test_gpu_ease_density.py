"""EASE(density=...) on the GPU: rpk_ease_prune against the canonical pruning (oracle/ease_prune_oracle.py) bit for
bit, the drop-in class against the oracle, the reference class and the signed scoring oracle, and the MSD shape
(BASELINE.json configs[3]) at density 0.01 checked on the device."""
import pickle
import warnings

import numpy as np
import pytest
from scipy.sparse import csr_matrix

from conftest import HAVE_REF
from oracle import signed_oracle
from oracle.ease_prune_oracle import canon_ease_prune, canon_prune_topk

pytestmark = pytest.mark.gpu

NAN_KEY = 0x7FF0000000000001


def _bits_equal(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.uint64), np.asarray(b, dtype=np.float64).view(np.uint64))


def _assert_csr_equal(got, want):
    got, want = csr_matrix(got), csr_matrix(want)
    assert got.shape == want.shape
    assert np.array_equal(got.indptr, want.indptr)
    assert np.array_equal(got.indices, want.indices)
    assert _bits_equal(got.data, want.data)


def _crafted():
    rng = np.random.default_rng(5)
    out = {}
    out["one_zero"] = np.zeros((1, 1))
    out["one"] = np.array([[-3.5]])
    out["two"] = np.array([[0.0, -2.0], [2.0, 1.0]])
    B = rng.choice([-3.0, -2.0, -1.0, 0.0, 1.0, 2.0, 3.0], size=(37, 37))  # tie groups across rows, +-x pairs
    out["ties_across_rows"] = B
    v = np.exp(rng.uniform(-5, 5, size=(37, 37)))
    out["pm_pairs"] = np.where(rng.random((37, 37)) < 0.5, v, -v) * (rng.random((37, 37)) < 0.7)
    out["pm_pairs"][:, 20] = -out["pm_pairs"][:, 3]  # every magnitude of column 3 again, negated
    out["all_equal"] = np.where(rng.random((37, 37)) < 0.5, 1.5, -1.5)
    B = np.where(rng.random((37, 37)) < 0.5, 0.0, -0.0)
    B[rng.random((37, 37)) < 0.1] = 4.0
    out["signed_zeros"] = B
    B = rng.standard_normal((37, 37))
    B[rng.random((37, 37)) < 0.1] = np.inf
    B[rng.random((37, 37)) < 0.1] = -np.inf
    B[rng.random((37, 37)) < 0.1] = np.nan
    B[3, 4] = -np.nan
    B[5, 6] = np.array([0x7FF0000000000123], dtype=np.uint64).view(np.float64)[0]  # a NaN with a payload
    out["nonfinite"] = B
    B = rng.standard_normal((37, 37)) + 10.0
    B[::3] *= 1e-6  # rows that pruning empties
    out["emptied_rows"] = B
    out["small_set_1000"] = rng.choice([-1.0, -0.5, -0.25, 0.0, 0.25, 0.5, 1.0], size=(1000, 1000), p=[.05, .1, .2, .3, .2, .1, .05])
    out["continuous_1000"] = rng.standard_normal((1000, 1000)) * (rng.random((1000, 1000)) < 0.4)
    return out


CRAFTED = _crafted()


@pytest.mark.parametrize("name", sorted(CRAFTED))
def test_entry_point_against_the_canonical_pruning(name):
    import torch

    from recpack_b200.engine import get_engine

    B = CRAFTED[name]
    nnz = int(np.count_nonzero(B != 0.0))  # NaN != 0.0: stored
    Bt = torch.from_numpy(np.ascontiguousarray(B)).cuda()
    eng = get_engine(0)
    keeps = sorted({0, 1, max(nnz - 1, 0), nnz, nnz + 7, nnz // 3, B.size})
    for keep in keeps:
        ptr, idx, val = eng.ease_prune(Bt, keep)
        got = csr_matrix((val.cpu().numpy(), idx.cpu().numpy(), ptr.cpu().numpy()), shape=B.shape)
        want = canon_prune_topk(csr_matrix(B), keep)
        assert got.nnz == min(keep, nnz)
        _assert_csr_equal(got, want)


def test_entry_point_with_host_outputs():
    import torch

    from recpack_b200.engine import get_engine

    B = CRAFTED["small_set_1000"]
    keep = 123_457
    eng = get_engine(0)
    Bt = torch.from_numpy(B).cuda()
    ptr = np.full(B.shape[0] + 1, -2, dtype=np.int64)
    idx = np.full(keep, -2, dtype=np.int32)
    val = np.full(keep, np.nan)
    nnz = np.zeros(1, dtype=np.int64)
    eng._check(eng._lib.rpk_ease_prune(eng._h, B.shape[0], Bt.data_ptr(), keep, ptr.ctypes.data, idx.ctypes.data,
                                       val.ctypes.data, nnz.ctypes.data))
    assert int(nnz[0]) == keep
    _assert_csr_equal(csr_matrix((val, idx, ptr), shape=B.shape), canon_prune_topk(csr_matrix(B), keep))


def _device_check(Bt, keep, ptr, idx, val):
    """The canonical pruning of a device matrix verified on the device: exactly K kept, the threshold found by bisection
    over the key, every key above it kept, and the ties taken the first ones in row-major order."""
    import torch

    I = Bt.shape[0]
    keys = Bt.view(torch.int64) & 0x7FFFFFFFFFFFFFFF
    keys.clamp_(max=NAN_KEY)
    nnz = int((keys != 0).sum().item())
    K = min(int(keep), nnz)
    assert int(ptr[-1].item()) == K and idx.shape[0] == K and val.shape[0] == K
    lo, hi = 1, NAN_KEY  # largest t with #(key >= t) >= K
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if int((keys >= mid).sum().item()) >= K:
            lo = mid
        else:
            hi = mid - 1
    T = lo
    row_gt = (keys > T).sum(dim=1)
    row_eq = (keys == T).sum(dim=1)
    q = K - int(row_gt.sum().item())
    assert 1 <= q <= int(row_eq.sum().item())
    eq_before = torch.cumsum(row_eq, 0) - row_eq
    take = (q - eq_before).clamp(min=0).minimum(row_eq)
    want_ptr = torch.zeros(I + 1, dtype=torch.int64, device=Bt.device)
    want_ptr[1:] = torch.cumsum(row_gt + take, 0)
    assert torch.equal(ptr, want_ptr)
    chunk = max(1, (1 << 30) // I)
    for r0 in range(0, I, chunk):
        r1 = min(I, r0 + chunk)
        k = keys[r0:r1]
        eq = k == T
        rank = torch.cumsum(eq.to(torch.int32), dim=1)
        mask = (k > T) | (eq & (rank <= take[r0:r1, None]))
        a, b = int(ptr[r0].item()), int(ptr[r1].item())
        assert torch.equal(idx[a:b].long(), mask.nonzero()[:, 1])
        assert torch.equal(val[a:b].view(torch.int64), Bt[r0:r1][mask].view(torch.int64))
    return K, T


def test_beyond_l2_20000():
    """I = 20,000 (3.2 GB, far beyond the 126 MB L2): magnitudes from a small set, so that the cut falls inside a tie
    group of tens of millions of entries, and a cut in the continuous part."""
    import torch

    from recpack_b200.engine import get_engine

    I = 20_000
    g = torch.Generator(device="cuda").manual_seed(3)
    Bt = torch.randn((I, I), generator=g, device="cuda", dtype=torch.float64)
    coarse = torch.randint(-4, 5, (I, I), generator=g, device="cuda").to(torch.float64) * 0.25
    Bt = torch.where(torch.rand((I, I), generator=g, device="cuda") < 0.7, coarse, Bt)
    del coarse
    n_above = int((Bt.abs() > 0.75).sum().item())
    eng = get_engine(0)
    for keep in (n_above + 12_345_678, I * I // 50):
        ptr, idx, val = eng.ease_prune(Bt, keep)
        _device_check(Bt, keep, ptr, idx, val)
        del ptr, idx, val


# -- the class ----------------------------------------------------------------------------------------------------------
def _data(seed=13, U=500, I=200, nnz=9000, unseen=0):
    from recpack_b200.synth import synth_interactions, weak_generalization_split

    X = synth_interactions(U, I, nnz, seed=seed)
    train, test_out = weak_generalization_split(X, 0.8, seed=2)
    if unseen:  # items nobody saw: with alpha != 0 their columns are 0 * inf = NaN
        keep = np.ones(I, dtype=bool)
        keep[-unseen:] = False
        train = csr_matrix(train.multiply(keep[None, :]))
        train.eliminate_zeros()
    return train, test_out


@pytest.mark.parametrize("alpha", [0, 0.5])
def test_class_against_the_canonical_pruning_of_the_dense_fit(alpha):
    from recpack_b200 import EASE

    train, _ = _data()
    I = train.shape[1]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        S_dense = EASE(l2=50.0, alpha=alpha).fit(train).similarity_matrix_
        again = EASE(l2=50.0, alpha=alpha).fit(train).similarity_matrix_
        _assert_csr_equal(again, S_dense)  # two fits of the same data on the device give the same bits
        for d in (0.5 / (I * I), 0.01, 0.3, 1.0, 0.0, None):
            algo = EASE(l2=50.0, alpha=alpha, density=d).fit(train)
            _assert_csr_equal(algo.similarity_matrix_, canon_ease_prune(S_dense, d))
            if d:
                assert algo.__dict__["_B_dev"] is None  # the dense model does not outlive the fit


def test_missing_items_warning_pickle_and_predict():
    from recpack_b200 import EASE
    from recpack_b200._lib import RpkError

    train, _ = _data()
    algo = EASE(l2=50.0, density=0.002)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        algo.fit(train)
    S = algo.similarity_matrix_
    empty = int(np.count_nonzero(np.diff(S.indptr) == 0))
    assert empty > 0
    msgs = [str(x.message) for x in w if "missing similar items" in str(x.message)]
    assert msgs == [f"EASE missing similar items for {empty} items."]

    users = train
    for N, rh in ((20, True), (None, True), (None, False), (7, False)):
        algo.set_params(predict_topK=N, remove_history=rh)
        fresh = EASE(l2=50.0, density=0.002).fit(train)  # a device model of another estimator is resident in between
        fresh.set_params(predict_topK=N, remove_history=rh)
        fresh.predict(users)
        for model in (algo, pickle.loads(pickle.dumps(algo))):
            pred = model.predict(users)
            want = signed_oracle.canon_predict_signed(users, S, N=N, remove_history=rh)
            if N is None:
                _assert_csr_equal(pred, want)
            else:
                idx, ln = pred._rpk_topn
                assert np.array_equal(ln, want["len"]) and np.array_equal(idx, want["idx"])
                vals = np.where(want["idx"] >= 0, np.asarray(pred[np.arange(users.shape[0])[:, None], np.maximum(want["idx"], 0)].todense()), 0.0)
                assert _bits_equal(vals, want["val"])
    clone = pickle.loads(pickle.dumps(algo))
    assert clone.__dict__.get("_S_dev") is None and clone.__dict__.get("_B_dev") is None
    _assert_csr_equal(clone.similarity_matrix_, S)

    # an assigned pruned matrix is scored the same way
    other = EASE(l2=50.0, density=0.002, predict_topK=20, remove_history=True)
    other.similarity_matrix_ = S.copy()
    want = signed_oracle.canon_predict_signed(users, S, N=20, remove_history=True)
    assert np.array_equal(other.predict(users)._rpk_topn[0], want["idx"])

    # NaN in the model (alpha with unseen items): the signed scorer refuses it
    train_u, _ = _data(unseen=3)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        bad = EASE(l2=50.0, alpha=0.5, density=0.3, predict_topK=10).fit(train_u)
        assert np.isnan(bad.similarity_matrix_.data).any()
        with pytest.raises(RpkError):
            bad.predict(train_u)


def test_invalidate_device_model_after_an_in_place_edit():
    from recpack_b200 import EASE

    train, _ = _data()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        algo = EASE(l2=50.0, density=0.05, predict_topK=10, remove_history=True).fit(train)
        S = algo.similarity_matrix_
        before = signed_oracle.canon_predict_signed(train, S, N=10, remove_history=True)
        assert np.array_equal(algo.predict(train)._rpk_topn[0], before["idx"])
        S.data *= -1.0  # reverses every ranking
        algo.invalidate_device_model()
        after = signed_oracle.canon_predict_signed(train, S, N=10, remove_history=True)
        assert not np.array_equal(after["idx"], before["idx"])
        assert np.array_equal(algo.predict(train)._rpk_topn[0], after["idx"])


@pytest.mark.skipif(not HAVE_REF, reason="baseline/_ref not installed")
def test_against_the_reference_class(monkeypatch):
    import recpack.algorithms
    import recpack.metrics

    from recpack_b200 import EASE, NDCGK

    monkeypatch.setattr(np, "product", np.prod, raising=False)  # removed under numpy 2; the reference's _prune calls it
    train, test_out = _data()
    for d in (0.01, 0.1):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = recpack.algorithms.EASE(l2=50.0, density=d).fit(train)
            ours = EASE(l2=50.0, density=d).fit(train)
            R, S = csr_matrix(ref.similarity_matrix_), csr_matrix(ours.similarity_matrix_)
            assert R.nnz == S.nnz
            kth = np.sort(np.abs(S.data))[::-1][S.nnz - 1]
            Rm, Sm = R.astype(bool).toarray(), S.astype(bool).toarray()
            diff = Rm ^ Sm
            dense_ref = EASE(l2=50.0).fit(train).similarity_matrix_.toarray()
            assert np.all(np.abs(np.abs(dense_ref[diff]) - kth) <= 1e-8 * kth)
            both = Rm & Sm
            np.testing.assert_allclose(S.toarray()[both], R.toarray()[both], rtol=1e-8)
            p_ref = ref.predict(train)
            p_ref = p_ref - p_ref.multiply(train.astype(bool))
            ours.set_params(predict_topK=20, remove_history=True)
            p_ours = ours.predict(train)
        m_ref, m_ours = recpack.metrics.NDCGK(10), NDCGK(10)
        m_ref.calculate(test_out, p_ref)
        m_ours.calculate(test_out, p_ours)
        # equal kept sets: the models agree to rounding and so do the metrics; an entry at the cut that LU and Cholesky
        # round to opposite sides changes a few scores by about the K-th magnitude, and a ranking with them
        assert m_ours.value == pytest.approx(m_ref.value, rel=1e-9 if not diff.any() else 1e-3)


def test_msd_shape_density_001():
    """MSD shape (571,355 x 41,140, 33.6 M interactions), density 0.01: the pruned model of the class equals
    rpk_ease_prune of the dense fit, which the device check confirms; top-20 lists of all users equal rpk_spgemm_topn
    on the same model, and 1,000 sampled users equal the signed scoring oracle."""
    import torch

    from recpack_b200 import EASE
    from recpack_b200.engine import get_engine
    from recpack_b200.matrix import binary_structure
    from recpack_b200.synth import make_dataset

    train, _, _ = make_dataset("msd", generator="auto")
    U, I = train.shape
    eng = get_engine(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dense = EASE(l2=200.0)
        dense._fit(dense._transform_fit_input(train))
        Bt = dense.__dict__["_B_dev"]
        keep = int(0.01 * (I * I))
        ptr, idx, val = eng.ease_prune(Bt, keep)
        _device_check(Bt, keep, ptr, idx, val)
        del dense, Bt
        torch.cuda.empty_cache()
        algo = EASE(l2=200.0, density=0.01, predict_topK=20, remove_history=True)
        algo._fit(algo._transform_fit_input(train))
    S_dev = algo.__dict__["_S_dev"]
    assert torch.equal(S_dev[0], ptr) and torch.equal(S_dev[1], idx) and torch.equal(S_dev[2].view(torch.int64), val.view(torch.int64))
    del ptr, idx, val
    S = algo.similarity_matrix_
    X, _, _ = binary_structure(train)
    pred = algo._predict(X)
    idx_g, ln_g = pred._rpk_topn
    A = csr_matrix((np.ones(X.nnz), X.indices, X.indptr), shape=X.shape)
    want = eng.spgemm_topn(A, S, 20, mask_history=True)
    assert np.array_equal(ln_g, want["len"]) and np.array_equal(idx_g, want["idx"])
    users = np.random.default_rng(0).choice(U, size=1000, replace=False)
    ref = signed_oracle.canon_predict_signed(X[users], S, N=20, remove_history=True)
    assert np.array_equal(idx_g[users], ref["idx"]) and np.array_equal(ln_g[users], ref["len"])
    got_val = pred[users]
    vals = np.where(ref["idx"] >= 0, np.asarray(got_val[np.arange(1000)[:, None], np.maximum(ref["idx"], 0)].todense()), 0.0)
    assert _bits_equal(vals, ref["val"])
