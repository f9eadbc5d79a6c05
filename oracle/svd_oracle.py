"""fp64 numpy restatement of sklearn.utils.extmath.randomized_svd as MatrixFactorization/PureSVDRecommender.py:36-55 calls it
(TEST INFRASTRUCTURE; third-party arithmetic, not under the reference tree).  The Gaussian start Omega is an argument (drawn by
the caller from numpy's stream, as sklearn draws it); every normaliser is an economic QR, which spans the same subspace as
sklearn's LU.  Pinned to scikit-learn's own float32 output by tests/golden/puresvd_golden.npz."""
import numpy as np
import scipy.sparse as sps


def auto_rules(shape, n_components):
    """(n_iter, transpose) of randomized_svd with n_iter='auto', transpose='auto'."""
    return (7 if n_components < 0.1 * min(shape) else 4), shape[0] < shape[1]


def randomized_svd(M, n_components, Omega, n_iter=None, transpose=None):
    """(U, s, Vt) in fp64 like randomized_svd(M, n_components, n_oversamples=Omega.shape[1] - n_components): the user side
    (rows of M) decides the signs, every column's largest-magnitude entry positive, first index on ties."""
    auto_iter, auto_t = auto_rules(M.shape, n_components)
    n_iter = auto_iter if n_iter is None else n_iter
    transpose = auto_t if transpose is None else transpose
    A = sps.csr_matrix(M, dtype=np.float64)
    if transpose:
        A = A.T.tocsr()
    Q = np.asarray(Omega, np.float64)
    for _ in range(n_iter):
        Q, _ = np.linalg.qr(A @ Q)
        Q, _ = np.linalg.qr(A.T @ Q)
    Q, _ = np.linalg.qr(A @ Q)
    B = np.asarray((A.T @ Q).T)
    Uhat, s, Vt = np.linalg.svd(B, full_matrices=False)
    U = Q @ Uhat
    user, item = (Vt.T, U) if transpose else (U, Vt.T)
    arg = np.argmax(np.abs(user), axis=0)
    sign = np.where(user[arg, np.arange(user.shape[1])] < 0, -1.0, 1.0)
    user, item = user * sign, item * sign
    k = min(n_components, len(s))
    return user[:, :k], s[:k], item[:, :k].T


def pure_svd_factors(M, num_factors, Omega):
    """PureSVDRecommender.fit: USER_factors = U, ITEM_factors = (diag(s) Vt)^T."""
    U, s, Vt = randomized_svd(M, num_factors, Omega)
    return U, (s[:, None] * Vt).T
