"""Randomized truncated SVD on the device: `sklearn.utils.extmath.randomized_svd` as
MatrixFactorization/PureSVDRecommender.py:36-55 calls it (power_iteration_normalizer='auto', flip_sign=True), without
scikit-learn.

The host part is what sklearn decides before any arithmetic -- the argument checks, the `n_iter` and `transpose` rules and
the Gaussian start Omega, drawn from numpy's stream exactly like `check_random_state(random_state).normal(...)`.  Everything
else runs in csrc/rsvd.cu: the power iterations (CSR x dense products, shifted-CholeskyQR3 normalisation), B^T = A^T Q and
its QR, and the final products, sign flip and Sigma scaling.  The one host step in between is the SVD of the l x l
triangular factor in fp64 numpy (l = n_components + n_oversamples).

Declared deviations: the normaliser (CholeskyQR instead of LU / QR; the subspaces agree in exact arithmetic); computation
in float32 / float64-accumulated whatever the input dtype; when l exceeds min(shape), the first min(shape) columns of
Omega start the iteration (the full Omega is still drawn, so numpy's stream advances as in sklearn)."""
import ctypes
import numbers
import time

import numpy as np
import scipy.sparse as sps

from . import _lib

MAX_L = 512  # n_components + n_oversamples, capped at min(shape), must not exceed this


def check_random_state(seed):
    """sklearn.utils.check_random_state restated with numpy only."""
    if seed is None or seed is np.random:
        return np.random.mtrand._rand
    if isinstance(seed, numbers.Integral):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError("%r cannot be used to seed a numpy.random.RandomState instance" % (seed,))


def plan(shape, n_components, n_oversamples=10, n_iter="auto", transpose="auto"):
    """The host rules of sklearn's _randomized_svd for a matrix of `shape`: (n_iter, transpose, l, l_eff, k_eff) with l the
    width of Omega, l_eff = min(l, min(shape)) the width of the range, k_eff = min(n_components, l_eff) the components
    returned.  Raises ValueError on bad arguments."""
    if isinstance(n_components, (bool, np.bool_)) or not isinstance(n_components, numbers.Integral) or n_components < 1:
        raise ValueError("n_components must be an integer >= 1, got %r" % (n_components,))
    if isinstance(n_oversamples, (bool, np.bool_)) or not isinstance(n_oversamples, numbers.Integral) or n_oversamples < 0:
        raise ValueError("n_oversamples must be an integer >= 0, got %r" % (n_oversamples,))
    n_rows, n_cols = int(shape[0]), int(shape[1])
    if n_rows < 1 or n_cols < 1:
        raise ValueError("randomized_svd needs a non-empty matrix, got shape %r" % (tuple(shape),))
    if isinstance(n_iter, str):
        if n_iter != "auto":
            raise ValueError("n_iter must be 'auto' or an integer >= 0, got %r" % (n_iter,))
        n_iter = 7 if n_components < 0.1 * min(n_rows, n_cols) else 4
    elif isinstance(n_iter, (bool, np.bool_)) or not isinstance(n_iter, numbers.Integral) or n_iter < 0:
        raise ValueError("n_iter must be 'auto' or an integer >= 0, got %r" % (n_iter,))
    if isinstance(transpose, str):
        if transpose != "auto":
            raise ValueError("transpose must be 'auto' or a bool, got %r" % (transpose,))
        transpose = n_rows < n_cols
    l = int(n_components) + int(n_oversamples)
    l_eff = min(l, n_rows, n_cols)
    if l_eff > MAX_L:
        raise ValueError("n_components + n_oversamples = %d is above the supported %d" % (l_eff, MAX_L))
    return int(n_iter), bool(transpose), l, l_eff, min(int(n_components), l_eff)


def draw_omega(random_state, n_rows, l):
    """Omega = check_random_state(random_state).normal(size=(n_rows, l)) cast to float32 (sklearn's draw for float32 data)."""
    return check_random_state(random_state).normal(size=(n_rows, l)).astype(np.float32)


class DeviceSVD(object):
    """Result of `rsvd_device`: `user` [n_rows(M), k] and `item` [n_cols(M), k] float32 CUDA tensors (the item side multiplied
    by `s` when asked), `s` (k,) float32 ndarray, `timings` (dict, seconds / device milliseconds) and `breakdowns`."""

    def __init__(self, user, item, s, timings, breakdowns):
        self.user, self.item, self.s, self.timings, self.breakdowns = user, item, s, timings, breakdowns


def rsvd_device(M, n_components, n_oversamples=10, n_iter="auto", transpose="auto", random_state=None, scale_item_side=False,
                timed=False):
    """The whole of randomized_svd on the current CUDA device.  M: scipy sparse (or dense) matrix, cast to CSR float32.
    With `timed`, per-phase device times (CUDA events) are recorded at the cost of extra synchronisation."""
    import torch
    n_iter, transpose, l, l_eff, k_eff = plan(M.shape, n_components, n_oversamples, n_iter, transpose)
    M = sps.csr_matrix(M, dtype=np.float32)
    if not M.has_sorted_indices:
        M = M.sorted_indices()
    n_users, n_items = M.shape
    if M.nnz >= 2 ** 31 - 1:
        raise ValueError("randomized_svd: nnz must fit int32")
    t0 = time.perf_counter()
    omega = draw_omega(random_state, n_users if transpose else n_items, l)
    t_omega = time.perf_counter() - t0
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timed else None
    m_ptr = torch.from_numpy(np.ascontiguousarray(M.indptr, np.int32)).to(dev)
    m_idx = torch.from_numpy(np.ascontiguousarray(M.indices, np.int32)).to(dev)
    m_val = torch.from_numpy(np.ascontiguousarray(M.data, np.float32)).to(dev)
    t_ptr = torch.empty(n_items + 1, dtype=torch.int32, device=dev)
    t_idx = torch.empty(max(M.nnz, 1), dtype=torch.int32, device=dev)
    t_val = torch.empty(max(M.nnz, 1), dtype=torch.float32, device=dev)
    if timed:
        ev[0].record()
    _lib.check(lib.b200_csr_transpose_device(n_users, n_items, M.nnz, m_ptr.data_ptr(), m_idx.data_ptr(), m_val.data_ptr(),
                                             t_ptr.data_ptr(), t_idx.data_ptr(), t_val.data_ptr(), st))
    if timed:
        ev[1].record()
    Mcsr, Mtcsr = (m_ptr, m_idx, m_val), (t_ptr, t_idx, t_val)
    (a, at), (n_rows, n_cols) = ((Mtcsr, Mcsr), (n_items, n_users)) if transpose else ((Mcsr, Mtcsr), (n_users, n_items))
    ld = (l_eff + 3) // 4 * 4
    om = np.zeros((n_cols, ld), np.float32)
    om[:, :l_eff] = omega[:, :l_eff]
    d_om = torch.from_numpy(om).to(dev)
    Q = torch.empty((n_rows, ld), dtype=torch.float32, device=dev)
    Qb = torch.empty((n_cols, ld), dtype=torch.float32, device=dev)
    Rb = torch.empty((l_eff, l_eff), dtype=torch.float64, device=dev)
    ms = (ctypes.c_float * 2)()
    breakdowns = ctypes.c_int32(0)
    _lib.check(lib.b200_rsvd_range_device(n_rows, n_cols, a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), at[0].data_ptr(),
                                          at[1].data_ptr(), at[2].data_ptr(), d_om.data_ptr(), l_eff, ld, n_iter, 0, Q.data_ptr(),
                                          Qb.data_ptr(), Rb.data_ptr(), ms if timed else None, ctypes.byref(breakdowns), st))
    # the host step: svd(Rb^T) = W diag(s) Z^T, l_eff x l_eff in fp64 (B = Rb^T Qb^T = W diag(s) (Qb Z)^T)
    t0 = time.perf_counter()
    W, s, Zt = np.linalg.svd(Rb.cpu().numpy().T)
    t_svd = time.perf_counter() - t0
    W, Z = np.ascontiguousarray(W), np.ascontiguousarray(Zt.T)
    s32 = np.ascontiguousarray(s[:k_eff], np.float32)
    user = torch.empty((n_users, k_eff), dtype=torch.float32, device=dev)
    item = torch.empty((n_items, k_eff), dtype=torch.float32, device=dev)
    if timed:
        ev[2].record()
    _lib.check(lib.b200_rsvd_finish_device(n_rows, n_cols, Q.data_ptr(), Qb.data_ptr(), l_eff, ld, _lib.ptr(W), _lib.ptr(Z),
                                           _lib.ptr(s32), k_eff, int(transpose), int(bool(scale_item_side)), user.data_ptr(),
                                           item.data_ptr(), st))
    timings = {"n_iter": n_iter, "transpose": transpose, "l": l_eff, "host_omega_s": t_omega, "host_svd_s": t_svd}
    if timed:
        ev[3].record()
        torch.cuda.synchronize()
        timings.update(transpose_ms=ev[0].elapsed_time(ev[1]), spmm_ms=float(ms[0]), orth_ms=float(ms[1]),
                       finish_ms=ev[2].elapsed_time(ev[3]))
    return DeviceSVD(user, item, s32, timings, int(breakdowns.value))


def randomized_svd(M, n_components, n_oversamples=10, n_iter="auto", transpose="auto", random_state=None):
    """sklearn.utils.extmath.randomized_svd(M, n_components, n_oversamples=10, n_iter='auto', transpose='auto',
    random_state=None) with power_iteration_normalizer='auto' and flip_sign=True: float32 (U, s, Vt) of shapes
    (n_rows, k), (k,), (k, n_cols) with k = min(n_components, min(shape))."""
    r = rsvd_device(M, n_components, n_oversamples, n_iter, transpose, random_state)
    return r.user.cpu().numpy(), r.s, np.ascontiguousarray(r.item.cpu().numpy().T)
