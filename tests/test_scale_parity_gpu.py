"""-m gpu: one parity case per BASELINE.json config at (a slice of) its REAL shape -- the toy-sized cases of the other files
never reach the kernel variants the benchmark times (multi-window / bitmap kernel at 200 K columns, f = 128 row gathers,
f = 256 normal equations, multi-block Cholesky).

  configs[0]  C1 10 K x 5 K, 1 %      ItemKNN cosine, every column, against the compiled reference (oracle/_ref)
  configs[1]  C2 6 040 x 3 706        SLIM-BPR, one epoch of the reference's default recipe, against the C oracle
  configs[2]  C3 138 K x 27 K         BPR-MF f = 128, batch 1000, one epoch on the replayed glibc stream, against the C oracle
  configs[3]  C4-shaped rows          IALS f = 256 (user profiles ~208 like C4) + EASE_R on a 2 048-item slice at C4 density
  configs[4]  C5 1 M x 200 K, 0.05 %  ItemKNN cosine, binary: 500 columns of the benchmarked run against the compiled
                                      reference -- bitmap kernel (default) and the packed-counter window kernel

The C1 and C5 ItemKNN cases also run against the reference's fp64 restatement (oracle/similarity_oracle.py), so that they
are checked where the compiled reference is not built.
"""
import numpy as np
import pytest
import scipy.sparse as sps

from oracle import ref_loader
from oracle.similarity_oracle import SimilarityOracle, check_topk_against_dense, compare_topk_with_reference, cosine_pair_values
from recsys2019_deeplearning_evaluation_b200.synth import synth_config, synth_urm

pytestmark = pytest.mark.gpu
KW = dict(topK=200, shrink=100, normalize=True, similarity="cosine")  # SURVEY.md 8(d)


def _ref_cls():
    mod = ref_loader.load("Compute_Similarity_Cython")
    if mod is None:
        pytest.skip("oracle/_ref not built")
    return mod.Compute_Similarity_Cython


def _sim_cls():
    from recsys2019_deeplearning_evaluation_b200.similarity import Compute_Similarity_Cython
    return Compute_Similarity_Cython


def _against_reference(X, W, W_ref, cols):
    Xc = sps.csc_matrix(X)
    res = compare_topk_with_reference(W, W_ref, cols, KW["topK"],
                                      pair_values=lambda jj, cc: cosine_pair_values(Xc, jj, cc, KW["shrink"]))
    assert res["ok"], res
    return res


def _c1_every_column(values, reference):
    X = synth_config("C1", values=values)
    W = _sim_cls()(X, **KW).compute_similarity()
    W_ref = reference(X, **KW).compute_similarity()
    assert W.nnz == W_ref.nnz
    _against_reference(X, W, W_ref, np.arange(X.shape[1]))


@pytest.mark.parametrize("values", ["binary", "ratings"])
def test_c1_itemknn_every_column_against_the_compiled_reference(values):
    _c1_every_column(values, _ref_cls())


@pytest.mark.parametrize("values", ["binary", "ratings"])
def test_c1_itemknn_every_column_against_the_oracle(values):
    """The same check against the fp64 restatement of the reference (oracle/similarity_oracle.py, pinned to the reference's
    stored outputs by tests/test_oracle_similarity.py), which runs where the compiled reference is not built."""
    _c1_every_column(values, SimilarityOracle)


def _c5_benchmarked_kernels(monkeypatch, reference):
    """The run bench.py times (C5, binary): columns [66666, 67166) of the full-range output, produced (a) by the default
    routing (bitmap kernel K1-C, window kernel for what it hands back) and (b) by the packed 16-bit-counter window kernel
    alone (B200REC_K1C=0), both against `reference` on the same URM."""
    X = synth_config("C5", values="binary")
    n = X.shape[1]
    lo, hi = 66666, 67166
    W_ref = reference(X, **KW).compute_similarity(start_col=lo, end_col=hi)
    Xc = sps.csc_matrix(X)
    pv = lambda jj, cc: cosine_pair_values(Xc, jj, cc, KW["shrink"])
    for k1c in ("1", "0"):
        monkeypatch.setenv("B200REC_K1C", k1c)
        sim = _sim_cls()(X, **KW)
        assert sim.binary_path
        tab = sim.compute_topk_device(0, n)  # the whole range, as timed
        idx, val, cnt = (t[lo:hi].cpu().numpy() for t in (tab.idx, tab.val, tab.cnt))
        keep = np.arange(idx.shape[1])[None, :] < cnt[:, None]
        cols = np.broadcast_to(np.arange(lo, hi)[:, None], idx.shape)[keep]
        G = sps.csc_matrix((val[keep], (idx[keep], cols)), shape=(n, n))
        res = compare_topk_with_reference(G, W_ref, np.arange(lo, hi), KW["topK"], pair_values=pv)
        assert res["ok"], (k1c, res)
        assert (tab.cnt == KW["topK"]).all()  # every C5 column has far more than K co-rated neighbours
        # a column sub-range (the multi-GPU shard path) gives the same rows
        part = sim.compute_topk_device(lo, hi)
        assert np.array_equal(part.cnt.cpu().numpy(), cnt)
        assert np.array_equal(np.sort(part.idx.cpu().numpy(), 1), np.sort(idx, 1))
        sim._dealloc()


def test_c5_itemknn_benchmarked_kernels_against_the_compiled_reference(monkeypatch):
    _c5_benchmarked_kernels(monkeypatch, _ref_cls())


def test_c5_itemknn_benchmarked_kernels_against_the_oracle(monkeypatch):
    """The same check against the fp64 restatement of the reference, as for C1."""
    _c5_benchmarked_kernels(monkeypatch, SimilarityOracle)


def test_c2_slim_bpr_one_epoch_of_the_reference_recipe():
    """SLIM_BPR_Cython defaults (SLIM_BPR_Cython.py:67-74): symmetric, adagrad, lr 1e-4, lambda 0, topK 200."""
    from oracle.sgd_oracle import SLIMOracle
    from recsys2019_deeplearning_evaluation_b200.slim_bpr_epoch import SLIM_BPR_Cython_Epoch
    X = synth_config("C2", values="binary")
    kw = dict(learning_rate=1e-4, li_reg=0.0, lj_reg=0.0, topK=200, symmetric=True, random_seed=42, sgd_mode="adagrad")
    g, o = SLIM_BPR_Cython_Epoch(X, **kw), SLIMOracle(X, **kw)
    g.epochIteration_Cython()
    o.epochIteration_Cython()
    S, R = g.get_S_dense().astype(np.float64), o.S_full()
    np.fill_diagonal(R, 0)
    assert np.abs(R).max() > 0
    assert np.allclose(S, R, rtol=1e-4, atol=1e-9), float(np.abs(S - R).max())


def test_c3_bprmf_f128_one_epoch_on_the_reference_stream():
    from oracle.sgd_oracle import MFOracle
    from recsys2019_deeplearning_evaluation_b200.mf_epoch import MatrixFactorization_Cython_Epoch
    X = synth_config("C3", values="binary")
    kw = dict(n_factors=128, algorithm_name="MF_BPR", batch_size=1000, learning_rate=1e-3, random_seed=42, sgd_mode="sgd",
              user_reg=1e-4, positive_reg=1e-4, negative_reg=1e-4)
    g, o = MatrixFactorization_Cython_Epoch(X, **kw), MFOracle(X, **kw)
    U0 = g.get_USER_factors()
    g.epochIteration_Cython()
    o.epochIteration_Cython()
    assert g.samples_last_epoch() == (X.shape[0] // 1000 + 1) * 1000
    U, V = g.get_USER_factors(), g.get_ITEM_factors()
    assert np.abs(U - U0).max() > 0
    assert np.allclose(U, o.get_USER_factors(), rtol=1e-4, atol=2e-6)
    assert np.allclose(V, o.get_ITEM_factors(), rtol=1e-4, atol=2e-6)
    # the device sampler + device-side dependency tracking on the same shape: replayed through the oracle
    g2 = MatrixFactorization_Cython_Epoch(X, sampler="philox", **kw)
    init = (g2.get_USER_factors(), g2.get_ITEM_factors())
    g2.epochIteration_Cython()
    o2 = MFOracle(X, init_factors=init, samples=g2.get_samples(), **kw)
    o2.epochIteration_Cython()
    assert np.allclose(g2.get_USER_factors(), o2.get_USER_factors(), rtol=1e-4, atol=2e-6)
    assert np.allclose(g2.get_ITEM_factors(), o2.get_ITEM_factors(), rtol=1e-4, atol=2e-6)


def test_c4_ials_f256_on_c4_shaped_rows():
    """f = 256 with user profiles of ~208 entries (C4's) and item profiles of ~280; 3 500 normal-equation solves per epoch
    in the numpy restatement (MatrixFactorization/IALSRecommender.py:137-201)."""
    from threadpoolctl import threadpool_limits
    from oracle.ials_oracle import confidence, run_epoch
    from recsys2019_deeplearning_evaluation_b200.recommenders import IALSRecommender
    f = 256
    X = synth_urm(2000, 1500, 0.139, seed=44, values="binary")
    np.random.seed(5)
    V0 = f ** -0.5 * np.random.random_sample((1500, f))
    np.random.seed(5)
    r = IALSRecommender(X, verbose=False)
    r.fit(epochs=1, num_factors=f, alpha=1.0, reg=1e-3)
    C = confidence(X, "linear", 1.0)
    with threadpool_limits(limits=4):
        U, V = run_epoch(C, np.zeros((2000, f)), V0.copy(), 1e-3)
    assert np.allclose(r.USER_factors, U, rtol=1e-4, atol=1e-8), float(np.abs(r.USER_factors - U).max())
    assert np.allclose(r.ITEM_factors, V, rtol=1e-4, atol=1e-8), float(np.abs(r.ITEM_factors - V).max())


def test_c4_ease_on_a_2048_item_slice():
    """EASE_R (EASE_R_Recommender.py:55-69) at C4's density on 2 048 items = 16 Cholesky blocks, l2_norm 1e3."""
    from oracle.ease_oracle import ease_B
    from recsys2019_deeplearning_evaluation_b200.recommenders import EASE_R_Recommender
    X = synth_urm(60_000, 2048, 0.0118, seed=45, values="binary")
    r = EASE_R_Recommender(X, verbose=False)
    r.fit(topK=None, l2_norm=1e3, verbose=False)
    B = ease_B(X, 1e3)
    G = np.asarray(r.W_sparse)
    assert float(np.abs(G - B).max() / np.abs(B).max()) < 1e-4
