"""Generates tests/golden/puresvd_golden.npz: scikit-learn's own randomized_svd (what MatrixFactorization/
PureSVDRecommender.py:36-55 runs) on small synthetic URMs, float32 as the recommender passes them.

    python tests/golden/make_golden_puresvd.py

Per case: `caseN_meta` (JSON: the synth_urm arguments, k and the random_state), `caseN_s` (the singular values),
`caseN_V` (Vt^T, only for n_items <= 400), `caseN_users` and `caseN_scores` (U[users] diag(s) Vt for 20 sampled users);
`sklearn_version` records the library that produced them."""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from recsys2019_deeplearning_evaluation_b200.synth import synth_urm  # noqa: E402

# (n_users, n_items, density, synth seed, values, popularity), k, random_state -- what each case exercises:
CASES = [
    ((1000, 500, 0.02, 1, "binary", None), 20, 0),      # n_iter 7
    ((604, 370, 0.045, 2, "ratings", None), 30, 3),     # ratings, n_iter 7
    ((300, 800, 0.03, 3, "binary", None), 25, 5),       # wide: transposed orientation
    ((2000, 600, 0.02, 4, "binary", 1.0), 60, 7),       # Zipf items; k == 0.1 min(shape) -> n_iter 4
    ((150, 40, 0.2, 5, "ratings", None), 35, 9),        # k + 10 > min(shape)
    ((120, 30, 0.3, 6, "binary", None), 40, 11),        # k > min(shape)
]


def case_urm(meta):
    nu, ni, d, seed, values, pop = meta["urm"]
    return synth_urm(nu, ni, d, seed=seed, values=values, popularity=pop)


def main():
    import sklearn
    from sklearn.utils.extmath import randomized_svd
    out = {"sklearn_version": np.array(sklearn.__version__)}
    for n, (urm, k, rs) in enumerate(CASES):
        meta = {"urm": list(urm), "k": k, "random_state": rs}
        X = case_urm(meta)
        U, s, Vt = randomized_svd(X, n_components=k, random_state=rs)
        users = np.linspace(0, X.shape[0] - 1, 20).astype(np.int32)
        out["case%d_meta" % n] = np.array(json.dumps(meta))
        out["case%d_s" % n] = s
        if X.shape[1] <= 400:
            out["case%d_V" % n] = Vt.T
        out["case%d_users" % n] = users
        out["case%d_scores" % n] = ((U[users] * s) @ Vt).astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "puresvd_golden.npz"), **out)


if __name__ == "__main__":
    main()
