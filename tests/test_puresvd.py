"""CPU: the host rules of the device randomized_svd (rsvd.py) and the fp64 oracle (oracle/svd_oracle.py), pinned to
scikit-learn's own randomized_svd output (tests/golden/puresvd_golden.npz, tests/golden/make_golden_puresvd.py)."""
import json
import os

import numpy as np
import pytest

from recsys2019_deeplearning_evaluation_b200 import rsvd
from recsys2019_deeplearning_evaluation_b200.synth import synth_urm
from oracle import svd_oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "puresvd_golden.npz")


def golden_cases():
    z = np.load(GOLDEN, allow_pickle=False)
    n = 0
    while "case%d_meta" % n in z.files:
        meta = json.loads(str(z["case%d_meta" % n]))
        nu, ni, d, seed, values, pop = meta["urm"]
        X = synth_urm(nu, ni, d, seed=seed, values=values, popularity=pop)
        g = {k: z["case%d_%s" % (n, k)] for k in ("s", "V", "users", "scores") if "case%d_%s" % (n, k) in z.files}
        yield n, X, meta["k"], meta["random_state"], g
        n += 1


def oracle_run(X, k, random_state):
    _, transpose, l, _, _ = rsvd.plan(X.shape, k)
    Omega = rsvd.draw_omega(random_state, X.shape[0] if transpose else X.shape[1], l)
    return svd_oracle.randomized_svd(X, k, Omega)


def separated(s, rel=1e-3):
    """Components whose singular value is more than `rel` (relative) away from both neighbours."""
    gap = np.full(len(s), np.inf)
    d = np.abs(np.diff(s)) / s[0]
    gap[:-1] = np.minimum(gap[:-1], d)
    gap[1:] = np.minimum(gap[1:], d)
    return gap > rel


@pytest.mark.parametrize("case", list(range(6)))
def test_oracle_matches_sklearn_golden(case):
    n, X, k, rs, g = list(golden_cases())[case]
    U, s, Vt = oracle_run(X, k, rs)
    kk = min(k, min(X.shape))
    assert U.shape == (X.shape[0], kk) and s.shape == (kk,) == g["s"].shape and Vt.shape == (kk, X.shape[1])
    assert np.all(np.abs(s - g["s"]) <= 1e-5 * g["s"]), np.max(np.abs(s - g["s"]) / g["s"])
    sc = (U[g["users"]] * s) @ Vt
    assert np.max(np.abs(sc - g["scores"])) <= 2e-4 * np.max(np.abs(g["scores"]))
    if "V" in g:
        sep = separated(g["s"])
        cos = np.sum(Vt.T[:, sep] * g["V"][:, sep], axis=0) / np.linalg.norm(g["V"][:, sep], axis=0)
        assert np.all(cos >= 1 - 1e-5), cos.min()


def test_golden_records_its_library():
    z = np.load(GOLDEN, allow_pickle=False)
    assert str(z["sklearn_version"])


def test_n_iter_and_transpose_rules():
    # k < 0.1 * min(shape) -> 7 power iterations, otherwise 4 (k == 0.1 * min(shape) gives 4)
    assert rsvd.plan((1000, 500), 49)[0] == 7
    assert rsvd.plan((1000, 500), 50)[0] == 4
    assert rsvd.plan((500, 1000), 50)[0] == 4
    assert rsvd.plan((1000, 500), 10, n_iter=2)[0] == 2
    assert rsvd.plan((1000, 500), 10)[1] is False and rsvd.plan((500, 1000), 10)[1] is True
    assert rsvd.plan((500, 500), 10)[1] is False and rsvd.plan((1000, 500), 10, transpose=True)[1] is True
    # (n_iter, transpose, l, l_eff, k_eff): the range is capped at min(shape), and so are the components
    assert rsvd.plan((150, 40), 35)[2:] == (45, 40, 35)
    assert rsvd.plan((120, 30), 40)[2:] == (50, 30, 30)
    assert rsvd.plan((30, 120), 40)[2:] == (50, 30, 30)


def test_omega_draw_matches_sklearn():
    ext = pytest.importorskip("sklearn.utils.extmath")
    from sklearn.utils import check_random_state
    for seed in (0, 12345):
        a = rsvd.draw_omega(seed, 37, 13)
        b = check_random_state(seed).normal(size=(37, 13)).astype(np.float32)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    ra, rb = np.random.RandomState(7), np.random.RandomState(7)
    assert np.array_equal(rsvd.draw_omega(ra, 20, 5), check_random_state(rb).normal(size=(20, 5)).astype(np.float32))
    assert np.array_equal(ra.random_sample(3), rb.random_sample(3))  # both instances advanced alike
    # None: numpy's global stream, left where sklearn's own call leaves it
    np.random.seed(99)
    a = rsvd.draw_omega(None, 25, 9)
    after_ours = np.random.random_sample(4)
    np.random.seed(99)
    b = check_random_state(None).normal(size=(25, 9)).astype(np.float32)
    after_sklearn = np.random.random_sample(4)
    assert np.array_equal(a, b) and np.array_equal(after_ours, after_sklearn)
    # and the whole of randomized_svd consumes exactly one (A.shape[1], k + 10) draw
    X = synth_urm(60, 90, 0.1, seed=3)
    np.random.seed(5)
    ext.randomized_svd(X, n_components=4, random_state=None)
    ref_next = np.random.random_sample(3)
    np.random.seed(5)
    _, transpose, l, _, _ = rsvd.plan(X.shape, 4)
    rsvd.draw_omega(None, X.shape[0] if transpose else X.shape[1], l)
    assert np.array_equal(np.random.random_sample(3), ref_next)


def test_argument_errors_come_before_any_device_work(monkeypatch):
    from recsys2019_deeplearning_evaluation_b200 import _lib

    def no_device(*a, **k):
        raise AssertionError("device work started before the arguments were checked")

    monkeypatch.setattr(_lib, "load", no_device)
    X = synth_urm(50, 20, 0.2)
    for bad in (0, -3, 2.5, "10", True, None):
        with pytest.raises(ValueError):
            rsvd.randomized_svd(X, bad)
    with pytest.raises(ValueError):
        rsvd.randomized_svd(X, 5, n_iter=-1)
    with pytest.raises(ValueError):
        rsvd.randomized_svd(X, 5, n_iter="many")
    with pytest.raises(ValueError):
        rsvd.randomized_svd(X, 5, transpose="sometimes")
    with pytest.raises(ValueError):
        rsvd.randomized_svd(X, 5, n_oversamples=-1)
    with pytest.raises(ValueError):
        rsvd.randomized_svd(X, 5, random_state="seed")
    with pytest.raises(ValueError):
        rsvd.randomized_svd(synth_urm(900, 800, 0.01), 600)  # l = 610 above the supported 512
