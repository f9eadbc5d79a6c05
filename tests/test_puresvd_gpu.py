"""-m gpu: the randomized-SVD kernels (csrc/rsvd.cu) piece by piece against scipy / numpy, the device randomized_svd against
the fp64 oracle (oracle/svd_oracle.py) on the same Omega, PureSVDRecommender end to end, and a full-shape C3 fit against
scikit-learn's own float32 call."""
import ctypes
import os
import tempfile

import numpy as np
import pytest
import scipy.sparse as sps

from oracle import svd_oracle
from oracle.evaluator_oracle import evaluate_scores
from recsys2019_deeplearning_evaluation_b200 import _lib, rsvd
from recsys2019_deeplearning_evaluation_b200.synth import synth_urm, synth_config

pytestmark = pytest.mark.gpu


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _st():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev_csr(M):
    return _t(M.indptr.astype(np.int32)), _t(M.indices.astype(np.int32)), _t(M.data.astype(np.float32))


def _spmm(M, X):
    import torch
    p, i, v = _dev_csr(M)
    Y = torch.empty((M.shape[0], X.shape[1]), dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().b200_csr_spmm_dense_device(M.shape[0], p.data_ptr(), i.data_ptr(), v.data_ptr(), _t(X).data_ptr(),
                                                       X.shape[1], Y.data_ptr(), _st()))
    return Y.cpu().numpy()


def _transpose(M):
    import torch
    p, i, v = _dev_csr(M)
    tp = torch.empty(M.shape[1] + 1, dtype=torch.int32, device="cuda")
    ti = torch.empty(max(M.nnz, 1), dtype=torch.int32, device="cuda")
    tv = torch.empty(max(M.nnz, 1), dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().b200_csr_transpose_device(M.shape[0], M.shape[1], M.nnz, p.data_ptr(), i.data_ptr(), v.data_ptr(),
                                                      tp.data_ptr(), ti.data_ptr(), tv.data_ptr(), _st()))
    return sps.csr_matrix((tv.cpu().numpy()[:M.nnz], ti.cpu().numpy()[:M.nnz], tp.cpu().numpy()), shape=(M.shape[1], M.shape[0]))


def _orth(Y, l, seed=0):
    Yd = _t(Y)
    bd = ctypes.c_int32(-1)
    _lib.check(_lib.load().b200_orthonormalize_device(Y.shape[0], l, Y.shape[1], Yd.data_ptr(), seed, ctypes.byref(bd), _st()))
    return Yd.cpu().numpy(), bd.value


def _skewed_urm():
    """Empty rows, and one Zipf-drawn row with more than 10 000 stored entries."""
    X = synth_urm(600, 15000, 0.002, seed=21, values="ratings", popularity=1.0).tolil()
    X[0:3, :] = 0
    rng = np.random.default_rng(4)
    X[7, rng.choice(15000, 11000, replace=False)] = rng.integers(1, 6, 11000).astype(np.float32)
    X = sps.csr_matrix(X, dtype=np.float32)
    X.eliminate_zeros()
    X.sort_indices()
    assert X.getnnz(axis=1).max() > 10000 and (X.getnnz(axis=1) == 0).sum() >= 3
    return X


@pytest.mark.parametrize("l", [1, 3, 11, 32, 110, 360, 512])
def test_spmm_and_transpose_against_scipy(l):
    X = _skewed_urm()
    ld = (l + 3) // 4 * 4
    rng = np.random.default_rng(l)
    T = _transpose(X)
    ref_t = X.T.tocsr()
    ref_t.sort_indices()
    assert np.array_equal(T.indptr, ref_t.indptr) and np.array_equal(T.indices, ref_t.indices) and np.array_equal(T.data, ref_t.data)
    for A in (X, T):
        D = np.zeros((A.shape[1], ld), np.float32)
        D[:, :l] = rng.standard_normal((A.shape[1], l))
        Y = _spmm(A, D)
        ref = A.astype(np.float64) @ D.astype(np.float64)
        # relative to the row norm of |A| |X|, the scale of the summed terms (a cancelling sum has a small result)
        rn = np.linalg.norm(abs(A).astype(np.float64) @ np.abs(D.astype(np.float64)), axis=1, keepdims=True)
        assert np.all(np.abs(Y - ref) <= 1e-5 * rn), np.max(np.abs(Y - ref) / np.maximum(rn, 1e-30))
        assert not Y[:, l:].any()


def _conditioned(n, l, cond, seed):
    rng = np.random.default_rng(seed)
    U, _ = np.linalg.qr(rng.standard_normal((n, l)))
    V, _ = np.linalg.qr(rng.standard_normal((l, l)))
    return ((U * np.logspace(0, -np.log10(cond), l)) @ V.T).astype(np.float32)


@pytest.mark.parametrize("l,cond", [(40, 1.0), (40, 1e3), (40, 1e6), (110, 1e6), (300, 1e3), (300, 1e6)])
def test_orthonormalize(l, cond):
    n = 6000
    ld = (l + 3) // 4 * 4
    Y = np.zeros((n, ld), np.float32)
    Y[:, :l] = _conditioned(n, l, cond, seed=l)
    Q, bd = _orth(Y, l)
    Q64, Y64 = Q[:, :l].astype(np.float64), Y[:, :l].astype(np.float64)
    assert bd == 0 and not Q[:, l:].any()
    assert np.max(np.abs(Q64.T @ Q64 - np.eye(l))) <= 1e-5
    assert np.linalg.norm(Y64 - Q64 @ (Q64.T @ Y64)) <= 1e-5 * np.linalg.norm(Y64)
    assert np.array_equal(_orth(Y, l)[0], Q)  # deterministic


def test_orthonormalize_rank_deficient():
    n, l = 3000, 24
    rng = np.random.default_rng(2)
    Y = np.zeros((n, l), np.float32)
    Y[:, :] = rng.standard_normal((n, 5)) @ rng.standard_normal((5, l))
    Y[:, 9] = Y[:, 2]  # an exact copy
    Y[:, 15] = 0       # and an empty column
    Q, bd = _orth(Y, l, seed=7)
    Q64, Y64 = Q.astype(np.float64), Y.astype(np.float64)
    assert bd >= 1 and np.isfinite(Q).all()
    assert np.max(np.abs(Q64.T @ Q64 - np.eye(l))) <= 1e-5
    assert np.linalg.norm(Y64 - Q64 @ (Q64.T @ Y64)) <= 1e-5 * np.linalg.norm(Y64)
    Q0, _ = _orth(np.zeros((200, 8), np.float32), 8)  # nothing to span: still an orthonormal basis
    assert np.max(np.abs(Q0.T.astype(np.float64) @ Q0 - np.eye(8))) <= 1e-5


def _rank5():
    rng = np.random.default_rng(5)
    M = (rng.random((300, 5)) @ rng.random((5, 400))).astype(np.float32)
    return sps.csr_matrix(M)


def _cold():
    X = synth_urm(2500, 900, 0.02, seed=31, values="ratings").tolil()
    X[::7, :] = 0
    X[:, ::11] = 0
    X = sps.csr_matrix(X, dtype=np.float32)
    X.eliminate_zeros()
    return X


RSVD_CASES = {
    "c1_like_k100": (lambda: synth_urm(10000, 5000, 0.01, seed=1), 100),
    "c2_like_ratings_k50": (lambda: synth_urm(6040, 3706, 0.0447, seed=2, values="ratings"), 50),
    "transposed_k100": (lambda: synth_urm(3000, 8000, 0.01, seed=3), 100),
    "zipf_k300": (lambda: synth_urm(20000, 6000, 0.005, seed=4, popularity=1.0), 300),
    "n_iter4_k60": (lambda: synth_urm(2000, 600, 0.03, seed=5), 60),
    "oversample_past_min": (lambda: synth_urm(150, 40, 0.2, seed=6, values="ratings"), 35),
    "rank5_k8": (_rank5, 8),
    "cold_users_items": (_cold, 40),
}


def _oracle(X, k, seed):
    _, transpose, l, _, _ = rsvd.plan(X.shape, k)
    return svd_oracle.randomized_svd(X, k, rsvd.draw_omega(seed, X.shape[0] if transpose else X.shape[1], l))


def _separated(s, rel=1e-3):
    gap = np.full(len(s), np.inf)
    d = np.abs(np.diff(s)) / s[0]
    gap[:-1] = np.minimum(gap[:-1], d)
    gap[1:] = np.minimum(gap[1:], d)
    return gap > rel


@pytest.mark.parametrize("name", list(RSVD_CASES))
def test_randomized_svd_against_oracle(name):
    make, k = RSVD_CASES[name]
    X = make()
    U, s, Vt = rsvd.randomized_svd(X, k, random_state=17)
    Uo, so, Vto = _oracle(X, k, 17)
    kk = min(k, min(X.shape))
    assert U.shape == (X.shape[0], kk) and s.shape == (kk,) and Vt.shape == (kk, X.shape[1])
    assert U.dtype == s.dtype == Vt.dtype == np.float32
    assert np.isfinite(U).all() and np.isfinite(s).all() and np.isfinite(Vt).all()
    top = 5 if name == "rank5_k8" else kk
    assert np.all(np.abs(s[:top] - so[:top]) <= 1e-5 * so[:top]), np.max(np.abs(s[:top] - so[:top]) / so[:top])
    if name == "rank5_k8":
        assert np.all(s[5:] <= 1e-5 * s[0])
    users = np.linspace(0, X.shape[0] - 1, min(200, X.shape[0])).astype(np.int64)
    sc, ref = (U[users] * s) @ Vt, (Uo[users] * so) @ Vto
    assert np.max(np.abs(sc - ref)) <= 1e-4 * np.max(np.abs(ref))
    sep = _separated(so[:top])
    for a, b in ((U[:, :top], Uo[:, :top]), (Vt[:top].T, Vto[:top].T)):
        cos = np.sum(a[:, sep] * b[:, sep], axis=0) / (np.linalg.norm(a[:, sep], axis=0) * np.linalg.norm(b[:, sep], axis=0))
        assert np.all(cos >= 1 - 1e-5), (name, cos.min())


def test_fit_is_deterministic():
    X = synth_urm(8000, 3000, 0.01, seed=9)
    a = rsvd.randomized_svd(X, 64, random_state=3)
    b = rsvd.randomized_svd(X, 64, random_state=3)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def _ref_recommend(URM, scores, users, cutoff):
    out = []
    for r, u in enumerate(users):
        s = scores[r].astype(np.float64).copy()
        s[URM.indices[URM.indptr[u]:URM.indptr[u + 1]]] = -np.inf
        order = np.lexsort((np.arange(len(s)), -s))[:cutoff]
        out.append(order[np.isfinite(s[order])].tolist())
    return out


def test_puresvd_recommender():
    from recsys2019_deeplearning_evaluation_b200.evaluation import EvaluatorHoldout
    from recsys2019_deeplearning_evaluation_b200.recommenders import PureSVDRecommender
    X = synth_urm(3000, 1200, 0.02, seed=12, values="ratings", popularity=0.8)
    rec = PureSVDRecommender(X, verbose=False)
    rec.fit(num_factors=50, random_seed=4)
    assert rec.USER_factors.shape == (3000, 50) and rec.ITEM_factors.shape == (1200, 50)
    assert rec.USER_factors.dtype == rec.ITEM_factors.dtype == np.float32
    _, transpose, l, _, _ = rsvd.plan(X.shape, 50)
    Uo, Vo = svd_oracle.pure_svd_factors(X, 50, rsvd.draw_omega(4, X.shape[1], l))
    users = np.arange(0, 3000, 13)
    sc = rec._compute_item_score(users)
    ref = Uo[users] @ Vo.T
    assert np.max(np.abs(sc - ref)) <= 1e-4 * np.max(np.abs(ref))
    assert np.allclose(sc, rec.USER_factors[users] @ rec.ITEM_factors.T, rtol=1e-4, atol=1e-5 * np.abs(sc).max())
    lists = rec.recommend(users, cutoff=10)
    want = _ref_recommend(rec.URM_train, sc, users, 10)
    assert sum(a == b for a, b in zip(lists, want)) >= len(users) - 2  # near-equal scores may swap at the 1e-7 level
    assert sum(len(a) for a in lists) == 10 * len(users)
    test = synth_urm(3000, 1200, 0.004, seed=13, values="ratings")
    kw = dict(cutoff_list=[5, 10], min_ratings_per_user=1)
    res, _ = EvaluatorHoldout(test, verbose=False, **kw).evaluateRecommender(rec)
    ev_ref = evaluate_scores(rec.URM_train, test, rec._compute_item_score(np.arange(3000)), **kw)
    for c in ev_ref:
        for m in ("PRECISION", "RECALL", "MAP", "NDCG"):
            assert abs(res[c][m] - ev_ref[c][m]) <= 1e-4 * max(1.0, abs(ev_ref[c][m])), (c, m)
    with tempfile.TemporaryDirectory() as d:
        rec.save_model(d + os.sep)
        rec2 = PureSVDRecommender(X, verbose=False)
        rec2.load_model(d + os.sep)
        assert np.array_equal(rec2.USER_factors, rec.USER_factors) and np.array_equal(rec2.ITEM_factors, rec.ITEM_factors)
        assert rec2.recommend(users, cutoff=10) == lists


def test_puresvd_unseeded_uses_the_global_stream():
    from recsys2019_deeplearning_evaluation_b200.recommenders import PureSVDRecommender
    X = synth_urm(900, 400, 0.03, seed=14)
    np.random.seed(8)
    a = PureSVDRecommender(X, verbose=False)
    a.fit(num_factors=12)
    after = np.random.random_sample(3)
    b = PureSVDRecommender(X, verbose=False)
    b.fit(num_factors=12, random_seed=8)  # RandomState(8) gives the same normals as the global stream seeded with 8
    assert np.array_equal(a.USER_factors, b.USER_factors) and np.array_equal(a.ITEM_factors, b.ITEM_factors)
    np.random.seed(8)
    np.random.normal(size=(400, 22))  # the reference's one draw: (n_items, num_factors + 10)
    assert np.array_equal(np.random.random_sample(3), after)


def test_c3_full_shape_against_sklearn():
    """Singular values within 1e-5 of scikit-learn's float32 call.  The scores are checked against the fp64 oracle on the same
    Omega: at C3 the spectrum around component 100 is nearly flat, so the float32 LU-normalised reference itself lands about
    1e-3 (relative to the largest score) away from the exact answer; the device result must be within 1e-4 of it and no
    farther from it than scikit-learn is."""
    ext = pytest.importorskip("sklearn.utils.extmath")
    X = synth_config("C3")
    U, s, Vt = rsvd.randomized_svd(X, 100, random_state=0)
    Us, ss, Vts = ext.randomized_svd(X, n_components=100, random_state=0)
    assert np.all(np.abs(s - ss) <= 1e-5 * ss), np.max(np.abs(s - ss) / ss)
    Uo, so, Vto = _oracle(X, 100, 0)
    users = np.linspace(0, X.shape[0] - 1, 1000).astype(np.int64)
    sc, sk, ref = ((A[users].astype(np.float64) * b) @ C for A, b, C in ((U, s, Vt), (Us, ss, Vts), (Uo, so, Vto)))
    err, err_sk = np.max(np.abs(sc - ref)), np.max(np.abs(sk - ref))
    assert err <= 1e-4 * np.max(np.abs(ref)) and err <= max(err_sk, 2e-4 * np.max(np.abs(ref))), (err, err_sk)
