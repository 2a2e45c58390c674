"""EASE(density=...): the pruning oracle against the reference's ``_prune`` (recpack/algorithms/ease.py:97-109) and
the keep count of the drop-in class, on the CPU."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.ease_prune_oracle import canon_ease_prune, canon_prune_topk, prune_keys, ref_ease_prune


def _same(a, b):
    a, b = csr_matrix(a), csr_matrix(b)
    a.sort_indices()
    b.sort_indices()
    return (a.shape == b.shape and np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
            and np.array_equal(a.data.view(np.uint64), b.data.view(np.uint64)))


def _model(I, seed, zeros=0.3):
    rng = np.random.default_rng(seed)
    B = rng.standard_normal((I, I)) * np.exp(rng.uniform(-8, 8, (I, I)))  # distinct magnitudes
    B[rng.random((I, I)) < zeros] = 0.0
    np.fill_diagonal(B, 0.0)
    return csr_matrix(B)


@pytest.mark.parametrize("density", [0.004, 0.01, 0.1, 0.3, 0.5, 0.69])
def test_canon_equals_reference_without_ties(density):
    S = _model(60, seed=int(density * 1000))
    assert len(np.unique(np.abs(S.data))) == S.nnz
    assert _same(canon_ease_prune(S, density), ref_ease_prune(S, density))


@pytest.mark.parametrize("seed", range(4))
def test_ties_differ_only_inside_the_group_at_the_cut(seed):
    rng = np.random.default_rng(seed)
    B = rng.choice([-3.0, -1.0, 1.0, 2.0, 3.0, 0.0], size=(40, 40))
    S = csr_matrix(B)
    for density in (0.05, 0.2, 0.4):
        c, r = canon_ease_prune(S, density), ref_ease_prune(S, density)
        assert c.nnz == r.nnz
        kth = np.sort(np.abs(S.data))[::-1][c.nnz - 1]
        diff = (c != r).tocoo()
        assert np.all(np.abs(B[diff.row, diff.col]) == kth)
        # the canonical pick inside the group: the first ties in row-major order
        Cd = c.toarray()
        tie_pos = np.flatnonzero(np.abs(B.ravel()) == kth)
        taken = Cd.ravel()[tie_pos] != 0
        assert np.all(taken[: taken.sum()])


def test_everything_stays_for_k0_knnz_density_ge_1_and_falsy_density():
    S = _model(30, seed=1)
    I = S.shape[0]
    for density in (None, 0.0, 0.5 / (I * I), 0.99 / (I * I), (S.nnz + 0.5) / (I * I), 0.9, 1.0, 3.0):
        for f in (canon_ease_prune, ref_ease_prune):
            assert _same(f(S, density), S), (f.__name__, density)


def test_nan_and_inf_rank_first():
    B = np.array([[0.0, np.nan, -np.inf], [1e300, -0.0, np.nan], [np.inf, -5.0, 2.0]])
    S = csr_matrix(B)
    assert S.nnz == 7  # -0.0 is not stored, NaN is
    for K, want in [(1, [(0, 1)]), (2, [(0, 1), (1, 2)]), (4, [(0, 1), (0, 2), (1, 2), (2, 0)]),
                    (5, [(0, 1), (0, 2), (1, 0), (1, 2), (2, 0)])]:
        c = canon_prune_topk(S, K).tocoo()
        assert sorted(zip(c.row.tolist(), c.col.tolist())) == want
        r = ref_ease_prune(S, K / 9 + 1e-9).tocoo()
        assert sorted(zip(r.row.tolist(), r.col.tolist())) == want


def test_keys_order_magnitudes_and_tie_signs():
    v = np.array([0.0, -0.0, 5e-324, -1.0, 1.0, np.inf, -np.inf, np.nan, -np.nan])
    k = prune_keys(v)
    assert k[0] == k[1] == 0 and k[3] == k[4] and k[5] == k[6] and k[7] == k[8] > k[5] > k[4] > k[2] > 0


def test_keep_count_is_one_float64_product_and_k0_keeps_all():
    from recpack_b200.ease import prune_keep

    assert prune_keep(0.01, 41_140) == int(np.float64(0.01) * np.prod((41_140, 41_140)))
    # a density where density * I * I (two roundings) and density * (I * I) truncate differently
    hits = [(d, I) for I in range(2, 400) for d in (0.07, 0.29, 0.57, 0.58)
            if int(d * I * I) != int(d * (I * I))]
    assert hits
    for d, I in hits:
        assert prune_keep(d, I) == int(np.float64(d) * np.prod((I, I)))
    assert prune_keep(0.9 / 100, 10) == 100  # int(0.9) == 0: the reference keeps everything
    assert prune_keep(1.0, 10) == 100
