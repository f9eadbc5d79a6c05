"""CPU: pins the numpy oracle (oracle/similarity_oracle.py) against
  (1) golden vectors produced by the unmodified reference (tests/golden/make_golden.py),
  (2) the compiled reference itself when oracle/_ref holds it,
  (3) the dense-control recipes of the reference's own (stale) unit tests,
      Base/Similarity/Compute_similarity_test.py:31-439."""
import numpy as np
import pytest
import scipy.sparse as sps

from golden_util import load_golden, same_sparse, tie_free
from oracle import ref_loader
from oracle.similarity_oracle import SimilarityOracle, check_topk_against_dense
from recsys2019_deeplearning_evaluation_b200.synth import synth_urm

URMS, CASES, KNN = load_golden()


@pytest.mark.parametrize("n", range(len(CASES)))
def test_oracle_matches_golden(n):
    values, kw, W = CASES[n]
    X = URMS[values]
    orc = SimilarityOracle(X, **kw)
    Wo = orc.compute_similarity()
    signed = kw["similarity"] in ("adjusted", "pearson")
    if tie_free(kw, values):
        # exact: same index sets, values to fp32 rounding -- against the reference's numpy implementation always,
        # and against the Cython class wherever it is not in its stale-slot regime (signed similarities)
        assert same_sparse(Wo, W["py"], rtol=1e-5)
        if not signed:
            assert same_sparse(Wo, W["cy"], rtol=1e-5)
    # tie-aware validity of the reference outputs w.r.t. the oracle's dense values (all cases)
    check_topk_against_dense(W["py"], orc, np.arange(150), rtol=1e-5)
    if not signed:
        check_topk_against_dense(W["cy"], orc, np.arange(150), rtol=1e-5)


def test_golden_urms_regenerate_from_seed():
    for v, X in URMS.items():
        Y = synth_urm(400, 150, 0.06, seed=17, values=v)
        assert (X.indptr == Y.indptr).all() and (X.indices == Y.indices).all() and np.array_equal(X.data, Y.data)


@pytest.mark.skipif(ref_loader.load("Compute_Similarity_Cython") is None, reason="oracle/_ref not built")
@pytest.mark.parametrize("kind", ["cosine", "asymmetric", "jaccard", "dice", "tversky"])
def test_oracle_vs_compiled_reference_live(kind):
    cy = ref_loader.load("Compute_Similarity_Cython").Compute_Similarity_Cython
    X = synth_urm(900, 260, 0.03, seed=5, values="continuous" if kind in ("cosine", "asymmetric") else "binary")
    kw = dict(topK=20, shrink=4, similarity=kind, asymmetric_alpha=0.6, tversky_alpha=0.5, tversky_beta=1.5)
    Wr = cy(X, **kw).compute_similarity()
    orc = SimilarityOracle(X, **kw)
    if kind in ("cosine", "asymmetric"):
        assert same_sparse(orc.compute_similarity(), Wr, rtol=1e-5)
    check_topk_against_dense(Wr, orc, np.arange(260), rtol=1e-5)


def test_shrink_truncated_like_c_int():
    """Appendix A quirk 3 (`cdef int shrink`, pyx:65)."""
    X = URMS["continuous"]
    a = SimilarityOracle(X, topK=10, shrink=10.9).compute_similarity()
    b = SimilarityOracle(X, topK=10, shrink=10).compute_similarity()
    assert same_sparse(a, b, rtol=0, atol=0)


def test_recipe_xtx_diag_zero():
    """Compute_similarity_test.py:31-56: topK=n, shrink=0, normalize=False => W == X^T X with zero diagonal."""
    rng = np.random.default_rng(1)
    D = (rng.random((50, 20)) * (rng.random((50, 20)) < 0.5)).astype(np.float32)
    W = SimilarityOracle(sps.csr_matrix(D), topK=20, shrink=0, normalize=False).compute_similarity().toarray()
    G = D.astype(np.float64).T @ D.astype(np.float64)
    np.fill_diagonal(G, 0)
    assert np.allclose(W, G, atol=1e-4)  # the recipe's atol


def test_recipe_cosine_vs_definition_and_jaccard_vs_sets():
    """Compute_similarity_test.py:91-156: cosine against the textbook formula, jaccard against set arithmetic."""
    rng = np.random.default_rng(2)
    D = (rng.random((80, 15)) * (rng.random((80, 15)) < 0.4)).astype(np.float32)
    X = sps.csr_matrix(D)
    W = SimilarityOracle(X, topK=15, shrink=0, normalize=True).compute_similarity().toarray()
    n = np.linalg.norm(D.astype(np.float64), axis=0)
    C = (D.astype(np.float64).T @ D.astype(np.float64)) / (np.outer(n, n) + 1e-6)
    np.fill_diagonal(C, 0)
    assert np.allclose(W, C, atol=1e-4)
    Wj = SimilarityOracle(X, topK=15, shrink=0, similarity="jaccard").compute_similarity().toarray()
    Bm = D > 0
    for i in range(15):
        for j in range(15):
            if i != j:
                inter = np.sum(Bm[:, i] & Bm[:, j]); union = np.sum(Bm[:, i] | Bm[:, j])
                assert abs(Wj[j, i] - inter / (union + 1e-6)) < 1e-4


def test_topk_matches_similarityMatrixTopK_recipe():
    """Compute_similarity_test.py:377-439: top-K output == column-wise top-K of the full matrix."""
    X = URMS["continuous"]
    full = SimilarityOracle(X, topK=150, shrink=2).compute_similarity().toarray()
    top = SimilarityOracle(X, topK=9, shrink=2).compute_similarity().toarray()
    for c in range(150):
        keep = np.argsort(-full[:, c], kind="stable")[:9]
        ref = np.zeros(150); ref[keep] = full[keep, c]
        assert np.allclose(top[:, c], ref, atol=1e-7)


# ------------------------------------------------------------------ euclidean (Compute_Similarity_Euclidean.py)
from golden_util import load_euclid_golden  # noqa: E402
from oracle.similarity_oracle import EuclideanOracle  # noqa: E402

EU_CASES = load_euclid_golden()


@pytest.mark.parametrize("n", range(len(EU_CASES)))
def test_euclidean_oracle_matches_golden(n):
    """The reference class computes in fp32; the restatement in fp64: values within 1e-4 (the reference's own
    Compute_similarity_euclidean_test.py:59-84 checks 1e-4 absolute against a dense control), index sets identical on
    the tie-free (continuous) inputs, tie-aware otherwise."""
    values, kw, W = EU_CASES[n]
    orc = EuclideanOracle(URMS[values], **kw)
    check_topk_against_dense(W, orc, np.arange(150), rtol=1e-4)
    if values == "continuous":
        assert same_sparse(orc.compute_similarity(), W, rtol=1e-4)


def test_euclidean_oracle_dense_control():
    """Recipe of Base/Similarity/Compute_similarity_euclidean_test.py:59-84: 1/(1 + scipy euclidean distance), topK = n."""
    rng = np.random.default_rng(1)
    D = (rng.random((40, 12)) * (rng.random((40, 12)) < 0.5)).astype(np.float32)
    S = EuclideanOracle(sps.csr_matrix(D), topK=12, shrink=1, similarity_from_distance_mode="lin").compute_similarity().toarray()
    diff = D.astype(np.float64)[:, :, None] - D.astype(np.float64)[:, None, :]
    ctrl = 1.0 / (np.sqrt((diff ** 2).sum(axis=0)) + 1.0 + 1e-9)
    np.fill_diagonal(ctrl, 0.0)
    assert np.allclose(S, ctrl, atol=1e-6)


def test_reference_comparer_on_tied_binary_data():
    """compare_topk_with_reference (bench.py's parity gate) accepts the oracle's result against the compiled reference's
    own output (stored in similarity_golden.npz) on binary data, where the K boundary is full of ties the two resolve
    differently, and rejects corrupted results."""
    from oracle.similarity_oracle import compare_topk_with_reference, cosine_pair_values
    values, kw, W = CASES[16]
    assert values == "binary" and kw["similarity"] == "cosine"
    X, K, n = URMS[values], kw["topK"], 150
    Wr = W["cy"]
    Wo = SimilarityOracle(X, **kw).compute_similarity()
    Xc = sps.csc_matrix(X)
    pv = lambda jj, cc: cosine_pair_values(Xc, jj, cc, kw["shrink"])
    res = compare_topk_with_reference(Wo, Wr, np.arange(n), K, pair_values=pv)
    assert res["ok"], res
    assert res["tie_cols"] > 0 and res["tie_pairs_checked"] > 0  # the case really exercises the tie path
    # a wrong value on one entry
    bad = sps.csc_matrix(Wo, copy=True)
    bad.data[7] *= 1.01
    assert not compare_topk_with_reference(bad, Wr, np.arange(n), K, pair_values=pv)["ok"]
    # a wrong neighbour carrying the K-th value (only the exact pair evaluation can see it)
    bad = sps.lil_matrix(Wo)
    c = 11
    col = sps.csc_matrix(Wo)[:, c]
    jmin = col.indices[np.argmin(col.data)]
    free = np.setdiff1d(np.arange(n), np.r_[col.indices, sps.csc_matrix(Wr)[:, c].indices, [c]])
    bad[free[0], c] = col.data.min()
    bad[jmin, c] = 0
    assert not compare_topk_with_reference(sps.csc_matrix(bad), Wr, np.arange(n), K, pair_values=pv)["ok"]
    # a missing neighbour
    bad = sps.lil_matrix(Wo)
    bad[jmin, c] = 0
    assert not compare_topk_with_reference(sps.csc_matrix(bad), Wr, np.arange(n), K, pair_values=pv)["ok"]
