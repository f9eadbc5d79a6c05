"""PureSVD timing on one GPU: the device randomized_svd (rsvd.py / csrc/rsvd.cu) at the BASELINE.json shapes, one JSON line
per measurement.

    python tools/puresvd_bench.py --out profiles/r03_puresvd.jsonl [--configs C3 C4 C5] [--ks 100 350] [--sklearn C3]

Per (config, k): device time per fit split into SpMM / orthonormalisation / finish (CUDA events; the URM transpose
separately), the end-to-end fit() time with the host Omega draw reported on its own, and the two SpMM products timed alone
with their achieved bytes/s from nnz (8 + 4 ld) + 4 ld (n_rows + n_cols) and whether the gathered dense matrix fits the
126 MB L2.  `--sklearn` configs also time scikit-learn's randomized_svd once (k = 100) and report the parity of the device
output against it (singular values, scores of 1 000 users).  The first line names the card and its power limit."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from recsys2019_deeplearning_evaluation_b200 import _lib, rsvd  # noqa: E402
from recsys2019_deeplearning_evaluation_b200.recommenders import PureSVDRecommender  # noqa: E402
from recsys2019_deeplearning_evaluation_b200.synth import synth_config  # noqa: E402

L2_BYTES = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in q.split(","))
    return {"card": name, "power_limit": power, "max_sm_clock": clock}


def spmm_time(csr, n_rows, n_cols, ld, reps=10):
    """ms per product Y[n_rows, ld] = A X[n_cols, ld] (CUDA events over `reps` launches after one warm-up)."""
    import torch
    X = torch.randn((n_cols, ld), dtype=torch.float32, device="cuda")
    Y = torch.empty((n_rows, ld), dtype=torch.float32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib = _lib.load()

    def run():
        _lib.check(lib.b200_csr_spmm_dense_device(n_rows, csr[0].data_ptr(), csr[1].data_ptr(), csr[2].data_ptr(), X.data_ptr(), ld,
                                                  Y.data_ptr(), st))
    run()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        run()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", nargs="+", default=["C3", "C4", "C5"])
    ap.add_argument("--ks", nargs="+", type=int, default=[100, 350])
    ap.add_argument("--sklearn", nargs="*", default=["C3"])
    args = ap.parse_args()
    torch.cuda.set_device(0)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    info = card()
    out = open(args.out, "a")

    def emit(d):
        d = dict(info, **d)
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    emit({"what": "session", "device": _lib.device_info()[0]})
    rsvd.rsvd_device(synth_config("C1"), 20, random_state=0)  # module load, first launches
    torch.cuda.synchronize()
    for name in args.configs:
        t0 = time.perf_counter()
        X = synth_config(name)
        t_gen = time.perf_counter() - t0
        n_users, n_items = X.shape
        for k in args.ks:
            n_iter, transpose, _, l, _ = rsvd.plan(X.shape, k)
            ld = (l + 3) // 4 * 4
            r = rsvd.rsvd_device(X, k, random_state=0, timed=True)
            tm = r.timings
            torch.cuda.synchronize()
            rec = PureSVDRecommender(X, verbose=False)
            t0 = time.perf_counter()
            rec.fit(num_factors=k, random_seed=0)
            torch.cuda.synchronize()
            t_fit = time.perf_counter() - t0
            n_rows, n_cols = (n_items, n_users) if transpose else (n_users, n_items)
            from recsys2019_deeplearning_evaluation_b200.recommenders import _dev_csr
            A = _dev_csr(X.T.tocsr() if transpose else X)
            At = _dev_csr(X if transpose else X.T.tocsr())
            legs = {}
            for leg, csr, rows, cols in (("A_Q", A, n_rows, n_cols), ("At_Y", At, n_cols, n_rows)):
                ms = spmm_time(csr, rows, cols, ld)
                byts = X.nnz * (8 + 4 * ld) + 4 * ld * (rows + cols)
                legs[leg] = {"ms": ms, "bytes": byts, "GBps": byts / ms / 1e6, "gathered_MB": cols * ld * 4 / 1e6,
                             "gathered_fits_L2": cols * ld * 4 <= L2_BYTES}
            del A, At
            emit({"what": "fit", "config": name, "k": k, "l": l, "ld": ld, "n_iter": n_iter, "transpose": transpose,
                  "shape": [n_users, n_items], "nnz": int(X.nnz), "breakdowns": r.breakdowns,
                  "device_ms": {"transpose": tm["transpose_ms"], "spmm": tm["spmm_ms"], "orth": tm["orth_ms"],
                                "finish": tm["finish_ms"]},
                  "host_omega_s": tm["host_omega_s"], "host_svd_s": tm["host_svd_s"], "fit_e2e_s": t_fit,
                  "n_spmm_per_fit": 2 * n_iter + 2, "spmm": legs, "synth_s": t_gen})
            del rec, r
            torch.cuda.empty_cache()
        if name in args.sklearn:
            from sklearn.utils.extmath import randomized_svd as sk_rsvd
            import sklearn
            t0 = time.perf_counter()
            Us, ss, Vts = sk_rsvd(X, n_components=100, random_state=0)
            t_sk = time.perf_counter() - t0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            U, s, Vt = rsvd.randomized_svd(X, 100, random_state=0)
            t_gpu = time.perf_counter() - t0
            users = np.linspace(0, n_users - 1, 1000).astype(np.int64)
            sc, ref = (U[users] * s) @ Vt, (Us[users] * ss) @ Vts
            emit({"what": "sklearn", "config": name, "k": 100, "sklearn_version": sklearn.__version__, "sklearn_s": t_sk,
                  "device_randomized_svd_s": t_gpu, "sigma_max_rel_err": float(np.max(np.abs(s - ss) / ss)),
                  "scores_max_abs_err_over_max": float(np.max(np.abs(sc - ref)) / np.max(np.abs(ref)))})
        del X
    out.close()


if __name__ == "__main__":
    main()
