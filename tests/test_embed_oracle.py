"""CPU checks of the embedding-neighbour definition (DESIGN.md 2, "Embedding neighbours") and of the screen's error
bound (DESIGN.md 4.9).

* oracle.embed_oracle.canon_embed_topk agrees with the reference's recipe -- get_top_K_values of sklearn's
  cosine_similarity (BLAS) with the diagonal zeroed -- up to BLAS's summation order: values within a few ulp * D, and
  lists equal except inside groups of values that lie within that distance of each other.
* A pessimistic numpy emulation of the tensor-core screen (tf32 operands, exact products, fp32 accumulation truncated
  at every addition) stays within delta_ij on every pair."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from oracle.embed_oracle import canon_block, canon_embed_topk, canon_rows, emulate_screen, screen_delta, screen_scale


def _reference_topk(E, K, similarity):
    """The reference's recipe: sklearn's cosine_similarity (or E @ E.T), setdiag(0), get_top_K_values."""
    from sklearn.metrics.pairwise import cosine_similarity

    S = cosine_similarity(E) if similarity == "cosine" else E @ E.T
    np.fill_diagonal(S, 0.0)
    S = csr_matrix(S)
    S.eliminate_zeros()
    I = S.shape[0]
    idx = np.full((I, K), -1, dtype=np.int64)
    val = np.zeros((I, K))
    ln = np.zeros(I, dtype=np.int64)
    for i in range(I):
        lo, hi = S.indptr[i], S.indptr[i + 1]
        c, v = S.indices[lo:hi], S.data[lo:hi]
        o = np.lexsort((c, -v))[:K]
        idx[i, : len(o)], val[i, : len(o)], ln[i] = c[o], v[o], len(o)
    return idx, val, ln


def _tie_aware_equal(want, idx, val, ln, tol):
    """Lists equal up to a reordering of values within tol of each other; per rank the values agree within tol."""
    for i in range(len(ln)):
        n = int(want["len"][i])
        m = int(ln[i])
        a_v, b_v = want["val"][i, :n], val[i, :m]
        k = min(n, m)
        assert np.all(np.abs(a_v[:k] - b_v[:k]) <= tol[i]), i
        if n != m:  # only values within tol of zero may be stored on one side and not on the other
            extra = a_v[k:] if n > m else b_v[k:]
            assert np.all(np.abs(extra) <= tol[i]), i
        a_c, b_c = set(want["idx"][i, :k].tolist()), set(idx[i, :k].tolist())
        if a_c != b_c:  # the differing columns lie within 2 tol of the cut
            cut = min(a_v[k - 1], b_v[k - 1])
            for c in a_c ^ b_c:
                v = a_v[list(want["idx"][i, :k]).index(c)] if c in a_c else b_v[list(idx[i, :k]).index(c)]
                assert abs(v - cut) <= 2 * tol[i], (i, c)


def _crafted(rng, I, D):
    """Duplicate and negated rows (exact ties and +- pairs), zero rows, integer values (exact zeros)."""
    B = rng.integers(-2, 3, size=(I // 4, D)).astype(np.float64)
    E = np.concatenate([B, B, -B, np.zeros((I - 3 * (I // 4), D))])
    return E[rng.permutation(I)]


@pytest.mark.parametrize("similarity", ["cosine", "dot"])
@pytest.mark.parametrize("case", ["gauss", "crafted", "wide"])
def test_oracle_matches_reference_recipe(similarity, case):
    rng = np.random.default_rng(11)
    if case == "gauss":
        E, K = rng.standard_normal((400, 24)), 15
    elif case == "crafted":
        E, K = _crafted(rng, 400, 9), 30
    else:
        E, K = rng.standard_normal((300, 200)) * np.exp2(rng.integers(-8, 8, size=(300, 1))), 40
    want = canon_embed_topk(E, K, similarity)
    idx, val, ln = _reference_topk(E, K, similarity)
    X = canon_rows(E, similarity)
    r = np.sqrt(np.einsum("ij,ij->i", X, X))
    D = E.shape[1]
    tol = 4 * (D + 2) * 2.0**-52 * r * r.max() + 1e-300  # |fold - any other order| <= ~D ulp of ||x_i|| ||x_j||
    _tie_aware_equal(want, idx, val, ln, tol)


def test_oracle_definition_details():
    """No self neighbour, exact zeros dropped, negatives kept when fewer than K positives, (value desc, column asc)."""
    E = np.array([[1.0, 0.0], [1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, 0.0]])
    out = canon_embed_topk(E, 4, "dot")
    assert out["len"].tolist() == [2, 2, 0, 2, 0]
    assert out["idx"][0].tolist() == [1, 3, -1, -1] and out["val"][0].tolist() == [1.0, -1.0, 0.0, 0.0]
    assert out["idx"][3].tolist() == [0, 1, -1, -1]
    # the fold is left to right in float64 without FMA
    E = np.array([[1.0, 1e-16, -1.0], [1.0, 1.0, 1.0]])
    assert canon_block(E, np.array([0]))[0, 1] == (1.0 + 1e-16) - 1.0


@pytest.mark.parametrize("D", [1, 7, 128, 1024])
@pytest.mark.parametrize("similarity", ["cosine", "dot"])
def test_screen_emulation_within_bound(D, similarity):
    rng = np.random.default_rng(D)
    I = 96 if D == 1024 else 160
    E = rng.standard_normal((I, D)) * (np.exp2(rng.integers(-20, 20, size=(I, 1))) if similarity == "dot" else 1.0)
    X = canon_rows(E, similarity)
    sigma = screen_scale(X)
    S = canon_block(X, np.arange(I))
    err = np.abs(emulate_screen(X, sigma) - S)
    ratio = err / screen_delta(X, sigma)
    print(f"D={D} {similarity}: largest |s^ - s| / delta = {ratio.max():.3f}")
    assert np.all(ratio <= 1.0)
