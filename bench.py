#!/usr/bin/env python3
"""Benchmark of the hot path BASELINE.json names: ItemKNN cosine top-K rows/sec (and BPR samples/sec as a
secondary figure) on a synthetic CSR URM.

    python bench.py --gpus N --steps K --warmup W [--impl b200|reference] [--workload C5] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one full pass of the similarity hot path over the workload
(all n_items columns: accumulate + normalise + top-K, plus the all-gather when N > 1) with the URM already
resident in HBM.  `--dump-outputs DIR` writes the top-K table of the last timed step to DIR (dump_topk_table) so that
two builds can be compared output for output; the URM is generated from a fixed seed, so the inputs are the same in
every run with the same arguments.  `e2e` is the same metric through the reference-facing Python call
(Compute_Similarity_Cython(URM, ...).compute_similarity() -> scipy CSR) with HOST buffers: H2D of the CSR,
device-side constructor work, kernel, CSR assembly and D2H all inside the timed region.

`--impl reference` times the reference's own Cython (oracle/_ref, compiled unmodified) on the host cores,
column-sharded over worker processes with the reference's own start_col/end_col hook.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ItemKNN cosine top-K rows/sec"
SIM_KW = dict(topK=200, shrink=100, normalize=True, similarity="cosine")  # SURVEY.md 8(d) hyper-parameters


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Everything any library writes to stdout (NCCL prints its version banner there) is diverted to stderr; the ONE JSON
# line goes to the original stdout through emit_json().
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit_json(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled every 200 ms while the timed region runs (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch(workload):
    """dram bytes per launch of the top-K kernel from the committed ncu summary of this workload, or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(workload)
        except Exception:
            return None
    return None


# ----------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """Reference arm: the unmodified reference Cython class on host cores (oracle/_ref), or the numpy port when
    the compiled reference is absent.  Rank 0 only."""
    if rank != 0:
        return
    from recsys2019_deeplearning_evaluation_b200.synth import synth_config, CONFIGS
    from oracle import ref_loader
    t0 = time.time()
    X = synth_config(args.workload, values=args.values)
    n_items = X.shape[1]
    log("[reference] URM %s nnz=%d generated in %.1fs" % (X.shape, X.nnz, time.time() - t0))
    mod = ref_loader.load("Compute_Similarity_Cython")
    kind = "reference" if mod is not None else "port"
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, args.ref_workers))
    slice_cols = args.ref_slice
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    conns, procs = [], []
    for w in range(workers):
        a, b = ctx.Pipe()
        pr = ctx.Process(target=_ref_worker, args=(b, X, kind, w), daemon=True)
        pr.start()
        conns.append(a)
        procs.append(pr)
    ctor_s = max(c.recv() for c in conns)  # constructors run concurrently; the slowest one
    log("[reference] %d workers constructed (%s) in %.1fs" % (workers, kind, ctor_s))
    rng = np.random.default_rng(0)

    def one_step():
        starts = rng.integers(1, max(2, n_items - slice_cols - 1), size=workers)
        t = time.perf_counter()
        for c, s in zip(conns, starts):
            c.send((int(s), int(s) + slice_cols))
        for c in conns:
            c.recv()
        return time.perf_counter() - t

    for _ in range(args.warmup):
        one_step()
    times = [one_step() for _ in range(args.steps)]
    for c in conns:
        c.send(None)
    total = sum(times)
    cols = workers * slice_cols * args.steps
    rate = cols / total
    e2e_rate = n_items / (ctor_s + n_items / rate)
    nu, ni, dens = CONFIGS[args.workload]
    sample = "%d workers x %d-column slices via start_col/end_col, %d steps; constructor %.1fs excluded from value, included in e2e (projected full fit)" % (
        workers, slice_cols, args.steps, ctor_s)
    out = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s ItemKNN cosine topK=200 shrink=100 on %dx%d density %.4g %s URM" % (
            args.workload, nu, ni, dens, args.values), "timing": "bounded sample of the column axis per step"},
        "cpu_baseline": {"value": rate, "unit": "rows/s", "cores": workers, "kind": kind, "sample": sample},
        "e2e": {"value": e2e_rate, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cores": cores,
    }
    emit_json(out)


def _ref_worker(conn, X, kind, w):
    from oracle import ref_loader
    t = time.perf_counter()
    if kind == "reference":
        cls = ref_loader.load("Compute_Similarity_Cython").Compute_Similarity_Cython
        obj = cls(X, **SIM_KW)
    else:
        from oracle.similarity_oracle import SimilarityOracle
        obj = SimilarityOracle(X, **SIM_KW)
    conn.send(time.perf_counter() - t)
    devnull = open(os.devnull, "w")
    while True:
        msg = conn.recv()
        if msg is None:
            return
        so = os.dup(1)
        os.dup2(devnull.fileno(), 1)  # the reference prints a progress line per call
        try:
            obj.compute_similarity(start_col=msg[0], end_col=msg[1])
        finally:
            sys.stdout.flush()
            os.dup2(so, 1)
            os.close(so)
        conn.send(1)


def cpu_baseline_leg(X, budget_cols):
    """Reference Cython (1 thread, as shipped) on a bounded slice of the same URM, for the b200 arm's JSON.
    Returns (the cpu_baseline dict, the reference's W for those columns, lo, hi): parity_gate() compares the GPU
    table of the same run against it."""
    from oracle import ref_loader
    mod = ref_loader.load("Compute_Similarity_Cython")
    kind = "reference" if mod is not None else "port"
    t = time.perf_counter()
    if mod is not None:
        obj = mod.Compute_Similarity_Cython(X, **SIM_KW)
    else:
        from oracle.similarity_oracle import SimilarityOracle
        obj = SimilarityOracle(X, **SIM_KW)
    ctor = time.perf_counter() - t
    n = X.shape[1]
    lo = max(1, n // 3)
    hi = min(n - 1, lo + budget_cols)
    so = os.dup(1)
    devnull = open(os.devnull, "w")
    os.dup2(devnull.fileno(), 1)
    try:
        t = time.perf_counter()
        W_ref = obj.compute_similarity(start_col=lo, end_col=hi)
        dt = time.perf_counter() - t
    finally:
        sys.stdout.flush()
        os.dup2(so, 1)
        os.close(so)
    return ({"value": (hi - lo) / dt, "unit": "rows/s", "cores": 1, "kind": kind,
             "sample": "columns [%d,%d) of the same URM in %.1fs, 1 thread (the reference is single-threaded); constructor %.1fs not counted" % (lo, hi, dt, ctor)},
            W_ref, lo, hi)


def parity_gate(X, table, W_ref, lo, hi, K, kind):
    """The timed run's own output against the reference's columns [lo, hi) of the same URM (the checker, not the thing
    measured): tie-aware index sets + 1e-4 relative values (oracle.similarity_oracle.compare_topk_with_reference);
    entries that only the GPU holds (ties at the K-th value) are re-evaluated exactly in fp64 from the URM columns."""
    import scipy.sparse as sps
    from oracle.similarity_oracle import compare_topk_with_reference, cosine_pair_values
    idx, val, cnt = (t[lo:hi].cpu().numpy() for t in table)
    keep = np.arange(idx.shape[1])[None, :] < cnt[:, None]
    cols = np.broadcast_to(np.arange(lo, hi)[:, None], idx.shape)[keep]
    n = X.shape[1]
    G = sps.csc_matrix((val[keep], (idx[keep], cols)), shape=(n, n))
    t = time.perf_counter()
    Xc = sps.csc_matrix(X)
    res = compare_topk_with_reference(G, W_ref, np.arange(lo, hi), K,
                                      pair_values=lambda jj, cc: cosine_pair_values(Xc, jj, cc, SIM_KW["shrink"]))
    res.update({"against": "%s Compute_Similarity_Cython, columns [%d,%d) of the timed run's output table" % (kind, lo, hi),
                "rule": "tie-aware index sets, rtol 1e-4", "seconds": time.perf_counter() - t})
    return res


DUMP_COLS = 16384  # at K = 200: 16384 x 200 x (8 + 4) B = 39 MB of neighbour ids and values


def dump_topk_table(path, table):
    """Writes the [n_items, K] top-K table (idx, val, cnt) as path/<name>.npy for a fixed, seeded sample of DUMP_COLS target
    columns (all of them when there are fewer): columns.npy (the sampled target columns), neighbours.npy and similarities.npy
    ([columns, K]) and counts.npy.  The kernel's slot order within a column is unspecified, so each column's entries are put
    in ascending neighbour order -- the order of a column of the CSR matrix compute_similarity() returns -- with the unused
    slots (at and beyond counts) last, as neighbour -1 and similarity 0.  Ids are stored as float64, which holds them exactly."""
    import torch
    idx, val, cnt = table
    n, K = idx.shape
    cols = np.arange(n) if n <= DUMP_COLS else np.sort(np.random.default_rng(0).choice(n, DUMP_COLS, replace=False))
    sel = torch.from_numpy(cols).to(idx.device)
    i, v, c = (t.index_select(0, sel).cpu().numpy() for t in (idx, val, cnt))
    unused = np.arange(K)[None, :] >= c[:, None]
    i, v = np.where(unused, -1, i), np.where(unused, 0.0, v)
    order = np.argsort(np.where(unused, np.iinfo(np.int64).max, i.astype(np.int64)), axis=1, kind="stable")
    os.makedirs(path, exist_ok=True)
    for name, a in (("columns", cols.astype(np.float64)), ("neighbours", np.take_along_axis(i, order, 1).astype(np.float64)),
                    ("similarities", np.take_along_axis(v, order, 1).astype(np.float32)), ("counts", c.astype(np.float64))):
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------
def pinned_csr(X):
    """scipy CSR whose three arrays live in pinned host memory (so the e2e H2D runs at PCIe speed)."""
    import torch
    import scipy.sparse as sps
    bufs = []
    for a in (X.data.astype(np.float32, copy=False), X.indices.astype(np.int32, copy=False),
              X.indptr.astype(np.int32, copy=False)):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        bufs.append(t)
    M = sps.csr_matrix((bufs[0].numpy(), bufs[1].numpy(), bufs[2].numpy()), shape=X.shape, copy=False)
    M.has_sorted_indices = True
    M._pinned = bufs
    return M


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from recsys2019_deeplearning_evaluation_b200.synth import synth_config, CONFIGS
    from recsys2019_deeplearning_evaluation_b200.similarity import Compute_Similarity_Cython, topk_table_to_csr
    from recsys2019_deeplearning_evaluation_b200 import _lib
    from recsys2019_deeplearning_evaluation_b200.dist import balanced_ranges, allgather_topk_tables, SymmetricTopKTable
    assert torch.cuda.is_available(), "bench.py --impl b200 needs CUDA (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    t0 = time.time()
    X = synth_config(args.workload, values=args.values)
    n_users, n_items = X.shape
    log("[rank %d] URM %s nnz=%d generated in %.1fs" % (rank, X.shape, X.nnz, time.time() - t0))
    Xp = pinned_csr(X)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- resident-input arm: handle built once, a step = kernel (+ all-gather)
    sim = Compute_Similarity_Cython(Xp, **SIM_KW)
    bounds = balanced_ranges(sim.column_work(), world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])

    # N > 1: the full table lives in symmetric memory and the kernel of every rank stores its rows into every rank's copy
    # (dist.SymmetricTopKTable); NCCL all-gathers of the ranks' slabs are the fallback when symmetric memory cannot be set up
    table, gather = None, "1 GPU"
    if world > 1:
        try:
            if args.gather == "nccl":
                raise RuntimeError("--gather nccl")
            table = SymmetricTopKTable(n_items, sim.K)
            gather = "kernel stores every finished row into all %d ranks' tables over NVLink (symmetric memory) + barrier" % world
        except Exception as ex:
            log("[rank %d] symmetric-memory table unavailable (%r): NCCL all-gather" % (rank, ex))
            gather = "NCCL all-gather of [n_items/N, K] idx/val/cnt slabs"
        flag = torch.tensor([1 if table is not None else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            table = None

    out_tab = sim.compute_topk_device(lo, hi) if table is None else None  # the output table is allocated once, every step refills it

    def step():
        if table is not None:
            return table.fill(sim, lo, hi)
        tab = sim.compute_topk_device(lo, hi, out=out_tab)
        if world > 1:
            return allgather_topk_tables(tab.idx, tab.val, tab.cnt, bounds)
        return tab.idx, tab.val, tab.cnt

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out = step()
    ev1.record()
    barrier()
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([elapsed_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    value = n_items * args.steps / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_topk_table(args.dump_outputs, out)

    # ---- kernel-only roofline leg (CUDA events around the kernel on its launching stream, inside the library)
    kms = []
    scratch = sim.compute_topk_device(lo, hi)
    for _ in range(args.steps):
        sim.compute_topk_device(lo, hi, out=scratch)
        kms.append(sim.last_kernel_ms())
    del scratch
    kernel_avg_ms = float(np.mean(kms))
    ent = sim.gathered_entries(lo, hi)
    bpe = 4 if sim.binary_path else 8
    share = (hi - lo) / float(n_items)
    # SURVEY.md 8(d): bytes = bpe * sum_u len_u^2 (row gathers) + CSR + CSC read once + 8*K*n_items written
    alg_bytes = bpe * ent + 2 * bpe * X.nnz * share + 8 * sim.K * (hi - lo)
    peak, peak_src = measured_peaks()
    achieved = alg_bytes / 1e9 / (kernel_avg_ms * 1e-3)
    traffic = ncu_traffic_per_launch(args.workload) if world == 1 else None
    import ctypes
    en, ctas, nb, nw = (ctypes.c_int32() for _ in range(4))
    _lib.check(_lib.load().b200_sim_debug_k1c(sim._h, -1, ctypes.byref(en), ctypes.byref(ctas), ctypes.byref(nb), ctypes.byref(nw)))
    kname = ("sim_k1d_kernel (4-bit counters, %d CTAs/SM): %d columns; sim_topk_kernel (window kernel): %d columns" % (
        ctas.value, nb.value - (nw.value - (hi - lo - nb.value)), nw.value)) if en.value else "sim_topk_kernel"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": kname, "kernel_ms": kernel_avg_ms,
                "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                "bytes_model": "%d B x %d gathered row entries + CSR/CSC once + 8 B x K x columns" % (bpe, ent)}

    # ---- e2e arm: host scipy CSR in -> scipy CSR out through the reference-facing class; inputs in page-locked memory (the
    # contract's case) and in ordinary pageable numpy arrays (what a caller's scipy matrix is)
    e2e_steps = max(3, args.e2e_steps)
    h2d = X.data.nbytes + X.indices.nbytes + X.indptr.nbytes
    d2h = 0

    def e2e_arm(Xin):
        nonlocal d2h
        times, parts = [], []
        W = None
        for it in range(e2e_steps + 1):  # first pass is a warm-up
            W = None  # a caller that refits drops its previous model first: the page-locked result arrays are reused, not reallocated
            barrier()
            t = time.perf_counter()
            s2 = Compute_Similarity_Cython(Xin, **SIM_KW)
            torch.cuda.synchronize()
            t_create = time.perf_counter() - t
            if table is not None:
                gi, gv, gc = table.fill(s2, lo, hi)
            else:
                tab = s2.compute_topk_device(lo, hi)
                if world > 1:
                    gi, gv, gc = allgather_topk_tables(tab.idx, tab.val, tab.cnt, bounds)
                else:
                    gi, gv, gc = tab.idx, tab.val, tab.cnt
            torch.cuda.synchronize()
            t_kernel = time.perf_counter() - t - t_create
            if rank == 0:
                W = topk_table_to_csr(n_items, s2.K, gi.contiguous(), gv.contiguous(), gc.contiguous())
                d2h = W.data.nbytes + W.indices.nbytes + W.indptr.nbytes
            barrier()
            dt = time.perf_counter() - t
            s2._dealloc()
            if it > 0:
                times.append(dt)
                parts.append({"create_h2d_s": t_create, "kernel_gather_s": t_kernel, "csr_assembly_d2h_s": dt - t_create - t_kernel})
        if world > 1:  # every sample: max over ranks
            tt = torch.tensor(times, device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            times = [float(x) for x in tt.tolist()]
        k = int(np.argsort(times)[len(times) // 2])
        return {"seconds_median": times[k], "seconds_min": min(times), "seconds_all": times, "breakdown_median_fit": parts[k]}

    e2e_pinned = e2e_arm(Xp)
    e2e_pageable = e2e_arm(X)
    e2e_s = e2e_pinned["seconds_median"]

    sim_K = sim.K
    sim._dealloc()
    secondary = None
    if world > 1 and not args.no_bpr:
        try:
            secondary = bpr_leg_sharded(args, X, rank, world)
        except Exception as ex:
            secondary = {"metric": "BPR-MF samples/sec", "error": repr(ex)}
    if rank != 0:
        return
    if world == 1 and not args.no_bpr:
        try:
            secondary = bpr_leg(args, X)
        except Exception as ex:
            secondary = {"metric": "BPR-MF samples/sec", "error": repr(ex)}
    cpu, parity = None, None
    if not args.no_cpu_baseline:
        try:
            # N = 1: the cpu_baseline slice; N > 1: a shorter slice, only for the parity of the gathered table
            cpu, W_ref, c_lo, c_hi = cpu_baseline_leg(X, args.cpu_cols if world == 1 else max(200, args.cpu_cols // 4))
        except Exception as ex:  # the GPU numbers stand without it
            cpu = {"value": None, "unit": "rows/s", "cores": 1, "kind": "unavailable", "sample": repr(ex)}
        else:
            try:
                parity = parity_gate(X, out, W_ref, c_lo, c_hi, sim_K, cpu["kind"])
            except Exception as ex:
                parity = {"ok": False, "error": repr(ex)}
            if world > 1:
                cpu = None  # reported at N = 1 only
    tensor = None
    if world == 1 and not args.no_tensor:
        try:
            tensor = tensor_leg(args)
        except Exception as ex:
            tensor = {"error": repr(ex)}
    nu, ni, dens = CONFIGS[args.workload]
    name, sms, mem = _lib.device_info()
    out = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None,
        "dtype": "i32 counts + f32" if sim.binary_path else "f32", "data": "synthetic",
        "config": {"workload": "%s ItemKNN cosine topK=200 shrink=100 on %dx%d density %.4g %s URM" % (
            args.workload, nu, ni, dens, args.values),
            "windows": sim.n_windows, "binary_path": sim.binary_path,
            "parallelism": ("item-sharded x%d; " % world + gather) if world > 1 else "1 GPU",
            "timing": "inputs (CSR+CSC %.2f GB) larger than the 126 MB L2; no explicit flush" % (2 * bpe * X.nnz / 1e9)},
        "clocks": clocks,
        "e2e": {"value": n_items / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "seconds_per_fit": e2e_s, "steps": e2e_steps, "pinned_inputs": e2e_pinned,
                "pageable_inputs": dict(e2e_pageable, value=n_items / e2e_pageable["seconds_median"]),
                "what": "Compute_Similarity_Cython(host scipy CSR).compute_similarity() -> scipy CSR; value = median fit with the three "
                        "input arrays in page-locked memory, pageable_inputs = the same with ordinary numpy arrays"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "secondary": secondary,
        "hot_path_iii": tensor,
        "device": name,
    }
    emit_json(out)


def bpr_leg_sharded(args, X, rank, world):
    """N > 1: user-sharded Hogwild BPR-MF (dist.ShardedBPR): every rank samples its own user range, the item factors are
    replicated and every rank's movement of the table is exchanged once per epoch with an all-reduce that runs on a side
    stream behind the next epoch's training kernel (one epoch of staleness).  Two runs: "weak" -- every rank draws a full
    reference epoch ((n_users / 1000 + 1) * 1000 samples) per step, the data-parallel reading of samples/sec -- and
    "strong" -- the reference epoch split over the ranks.  Time = device events, max over ranks, pipeline flushed inside."""
    import torch
    import torch.distributed as dist
    from recsys2019_deeplearning_evaluation_b200.dist import ShardedBPR
    f = 128
    from recsys2019_deeplearning_evaluation_b200.synth import synth_config
    out = {}
    for scaling, Xw in (("weak", X), ("strong", X), ("c3_weak", None), ("c3_strong", None)):
        if Xw is None:
            Xw = synth_config("C3", values="binary")  # BASELINE.json configs[2]: 138 K x 27 K
        tr = ShardedBPR(Xw, scaling=scaling.replace("c3_", ""), n_factors=f, batch_size=1000, learning_rate=1e-3, random_seed=42, sgd_mode="sgd")
        for _ in range(3):
            tr.epoch()
        tr.flush()
        torch.cuda.synchronize(); dist.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = args.steps
        ev0.record()
        n = 0
        for _ in range(steps):
            n += tr.epoch()
        tr.flush()
        ev1.record()
        torch.cuda.synchronize(); dist.barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        out[scaling] = {"value": n / (ms * 1e-3), "ms_per_step": ms / steps, "samples_per_step": n // steps}
        del tr
        torch.cuda.empty_cache()
    return {"metric": "BPR-MF samples/sec", "unit": "samples/s", "value": out["weak"]["value"], "scaling": "weak",
            "ms_per_epoch": out["weak"]["ms_per_step"], "samples_per_epoch": out["weak"]["samples_per_step"],
            "strong_scaling": out["strong"],
            "c3": {"workload": "C3 (configs[2]) MF_BPR n_factors=%d, same sharding" % f, "weak": out["c3_weak"], "strong": out["c3_strong"]},
            "config": {"workload": "%s MF_BPR n_factors=%d sgd lr=1e-3" % (args.workload, f),
                       "parallelism": "user-sharded hogwild x%d, item factors replicated, one NCCL all-reduce of the ranks' item-factor movement (%.0f MB) per epoch, overlapped with the next epoch" % (
                           world, X.shape[1] * f * 4 / 1e6)}}


def bpr_leg(args, X):
    """Second half of BASELINE.json's metric: BPR-MF samples/sec (MatrixFactorization_Cython_Epoch,
    algorithm_name='MF_BPR', 128 factors, the wrapper's default batch_size=1000, sgd) on the same URM, 1 GPU.
    A step is one epochIteration_Cython(); device time by CUDA events on the launching stream, wall time around the
    call (the glibc sampler runs on the host inside it)."""
    import torch
    from recsys2019_deeplearning_evaluation_b200.mf_epoch import MatrixFactorization_Cython_Epoch
    f = 128
    peak, peak_src = measured_peaks()
    res = {"metric": "BPR-MF samples/sec", "unit": "samples/s",
           "config": {"workload": "%s MF_BPR n_factors=%d sgd lr=1e-3" % (args.workload, f),
                      "bytes_per_sample": 6 * f * 4, "timing": "factor tables (%.2f GB) larger than L2" % ((X.shape[0] + X.shape[1]) * f * 4 / 1e9)},
           "modes": {}}
    for label, kw in (("minibatch_bs1000_glibc_stream", dict(batch_size=1000, sampler="glibc")),
                      ("minibatch_bs1000_philox", dict(batch_size=1000, sampler="philox")),
                      ("hogwild_philox", dict(batch_size=1000, sampler="philox", hogwild=True))):
        m = MatrixFactorization_Cython_Epoch(X, n_factors=f, algorithm_name="MF_BPR", learning_rate=1e-3, random_seed=42,
                                             sgd_mode="sgd", **kw)
        for _ in range(3):
            m.epochIteration_Cython()
        torch.cuda.synchronize()
        walls, devs = [], []
        for _ in range(args.steps):
            t = time.perf_counter()
            m.epochIteration_Cython()
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t)
            devs.append(m.last_epoch_ms() * 1e-3)
        n = m.samples_last_epoch()
        dev = float(np.mean(devs))
        res["modes"][label] = {"value": n / dev, "e2e_value": n / float(np.mean(walls)), "samples_per_epoch": n,
                               "device_ms_per_epoch": 1e3 * dev,
                               "roofline": {"bound": "hbm", "achieved": n * 6 * f * 4 / 1e9 / dev, "peak": peak, "unit": "GB/s",
                                            "frac": n * 6 * f * 4 / 1e9 / dev / peak, "peak_source": peak_src}}
        m._dealloc()
    if not args.no_cpu_baseline:
        # parity of the reference-semantics mode at the benchmarked shape: one epoch of the dataflow kernel on a device-drawn
        # stream, the same stream and initial factors replayed through the C oracle (itself pinned to the compiled reference)
        try:
            from oracle.sgd_oracle import MFOracle
            kw = dict(n_factors=f, algorithm_name="MF_BPR", batch_size=1000, learning_rate=1e-3, random_seed=7, sgd_mode="sgd",
                      user_reg=1e-4, positive_reg=1e-4, negative_reg=1e-4)
            t = time.perf_counter()
            g = MatrixFactorization_Cython_Epoch(X, sampler="philox", **kw)
            init = (g.get_USER_factors(), g.get_ITEM_factors())
            g.epochIteration_Cython()
            o = MFOracle(X, init_factors=init, samples=g.get_samples(), **kw)
            o.epochIteration_Cython()
            U, V = g.get_USER_factors(), g.get_ITEM_factors()
            ok = bool(np.allclose(U, o.get_USER_factors(), rtol=1e-4, atol=2e-6) and np.allclose(V, o.get_ITEM_factors(), rtol=1e-4, atol=2e-6))
            moved = float(np.abs(V - init[1]).max())
            res["parity"] = {"ok": ok, "max_abs_diff": float(max(np.abs(U - o.get_USER_factors()).max(), np.abs(V - o.get_ITEM_factors()).max())),
                             "max_abs_movement": moved, "samples": int(g.samples_last_epoch()),
                             "against": "oracle/sgd_oracle.c mf_epoch on the epoch's own (u, i, j) stream, rtol 1e-4 atol 2e-6",
                             "seconds": time.perf_counter() - t}
            g._dealloc()
            del o, init, U, V
        except Exception as ex:
            res["parity"] = {"ok": False, "error": repr(ex)}
    res["value"] = res["modes"]["hogwild_philox"]["value"]
    res["reference_semantics_value"] = res["modes"]["minibatch_bs1000_philox"]["value"]
    # BASELINE.json configs[2] as written: BPRMF, 128 factors, MovieLens-20M-shape URM (C3: 138 K x 27 K)
    try:
        from recsys2019_deeplearning_evaluation_b200.synth import synth_config
        X3 = synth_config("C3", values="binary")
        c3 = {"workload": "C3 (configs[2]) MF_BPR n_factors=%d sgd lr=1e-3, epoch = %d samples" % (f, (X3.shape[0] // 1000 + 1) * 1000)}
        for label, kw in (("minibatch_bs1000_philox", dict(batch_size=1000, sampler="philox")),
                          ("hogwild_philox", dict(batch_size=1000, sampler="philox", hogwild=True))):
            m = MatrixFactorization_Cython_Epoch(X3, n_factors=f, algorithm_name="MF_BPR", learning_rate=1e-3, random_seed=42,
                                                 sgd_mode="sgd", **kw)
            for _ in range(3):
                m.epochIteration_Cython()
            torch.cuda.synchronize()
            devs = []
            for _ in range(args.steps):
                m.epochIteration_Cython()
                torch.cuda.synchronize()
                devs.append(m.last_epoch_ms() * 1e-3)
            c3[label] = {"value": m.samples_last_epoch() / float(np.mean(devs)), "device_ms_per_epoch": 1e3 * float(np.mean(devs))}
            m._dealloc()
        res["c3"] = c3
    except Exception as ex:
        res["c3"] = {"error": repr(ex)}
    if not args.no_cpu_baseline:
        from oracle import ref_loader
        mod = ref_loader.load("MatrixFactorization_Cython_Epoch")
        if mod is not None:
            ref_loader.numpy_alias_shim()
            r = mod.MatrixFactorization_Cython_Epoch(X, n_factors=f, algorithm_name="MF_BPR", batch_size=1000, learning_rate=1e-3,
                                                     random_seed=42, sgd_mode="sgd")
            t = time.perf_counter()
            r.epochIteration_Cython()
            dt = time.perf_counter() - t
            n = (X.shape[0] // 1000 + 1) * 1000
            res["cpu_baseline"] = {"value": n / dt, "unit": "samples/s", "cores": 1, "kind": "reference",
                                   "sample": "one epochIteration_Cython (%d samples) in %.1fs, 1 thread" % (n, dt)}
    return res


def tensor_leg(args):
    """Hot path (iii) as BASELINE.json configs[3] writes it: IALS with 256 factors and EASE_R on the Netflix-shape synthetic
    URM (C4, 480 K x 17.7 K, binary), one GPU.  Flops per SURVEY.md 8(d): IALS epoch = sum over rows of 2 len f^2 (Gram of the
    gathered factor rows) + (2/3) f^3 + 2 f^2 (Cholesky + two triangular solves); EASE = 2 sum_u len_u^2 (sparse Gram) + n^3
    (Cholesky + inverse from the factor).  Roofline bound: tensor (dense contraction); peak = the measured sustained bf16
    throughput (MEASURED_PEAKS.json), the denominator the contract names -- the kernels compute in 3xTF32 / fp64."""
    import torch
    from recsys2019_deeplearning_evaluation_b200.synth import synth_config, CONFIGS
    from recsys2019_deeplearning_evaluation_b200 import recommenders as R
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak_tf, peak_src = (float(json.load(open(pk))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)") \
        if os.path.exists(pk) else (1500.0, "fallback (B200_PROFILING.md)")
    t0 = time.time()
    X = synth_config("C4", values="binary")
    nu, ni = X.shape
    log("[tensor leg] C4 URM %s nnz=%d generated in %.1fs" % (X.shape, X.nnz, time.time() - t0))
    res = {"config": {"workload": "C4 (configs[3]): IALS num_factors=256 alpha=1 reg=1e-3 linear, EASE_R l2_norm=1e3 on %dx%d density %.4g binary URM" % CONFIGS["C4"]},
           "peak_tflops": peak_tf, "peak_source": peak_src}
    f = 256
    try:
        np.random.seed(42)
        rec = R.IALSRecommender(X, verbose=False)
        rec.fit(epochs=1, num_factors=f, alpha=1.0, reg=1e-3)  # builds the device state and runs the first epoch (warm-up)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        rec._run_epoch(1)
        ev1.record()
        torch.cuda.synchronize()
        sec = ev0.elapsed_time(ev1) * 1e-3
        flops = float(2 * 2 * f * f * X.nnz + (nu + ni) * (2.0 * f ** 3 / 3.0 + 2.0 * f * f))
        res["ials"] = {"metric": "IALS row-solves/sec", "value": (nu + ni) / sec, "unit": "rows/s", "seconds_per_epoch": sec, "n_factors": f,
                       "roofline": {"bound": "tensor", "achieved": flops / sec / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                                    "frac": flops / sec / 1e12 / peak_tf, "flops_per_epoch": flops},
                       "path": getattr(rec, "last_path", None)}
        del rec
    except Exception as ex:
        res["ials"] = {"error": repr(ex)}
    torch.cuda.empty_cache()
    try:
        ease = R.EASE_R_Recommender(X, verbose=False)
        secs = []
        for _ in range(2):
            torch.cuda.synchronize()
            t = time.perf_counter()
            ease.fit(topK=None, l2_norm=1e3, verbose=False)
            torch.cuda.synchronize()
            secs.append(time.perf_counter() - t)
        lens = np.diff(X.indptr).astype(np.float64)
        flops = float(2.0 * (lens ** 2).sum() + float(ni) ** 3)
        sec = min(secs)
        res["ease"] = {"metric": "EASE_R fit seconds", "value": sec, "unit": "s", "higher_is_better": False, "seconds_all": secs,
                       "what": "EASE_R_Recommender(host URM).fit(): H2D, Gram (similarity kernel, dense mode), blocked Cholesky inverse on tcgen05 (3xTF32), B on the device",
                       "roofline": {"bound": "tensor", "achieved": flops / sec / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                                    "frac": flops / sec / 1e12 / peak_tf, "flops_per_fit": flops}}
        del ease
    except Exception as ex:
        res["ease"] = {"error": repr(ex)}
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C5", help="C1..C5 (synth.CONFIGS); the metric is quoted on C5")
    ap.add_argument("--values", default="binary", choices=["binary", "ratings", "continuous"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-cols", type=int, default=2000, help="columns in the CPU-baseline slice")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bpr", action="store_true", help="skip the BPR-MF samples/sec leg")
    ap.add_argument("--no-tensor", action="store_true", help="skip the C4 IALS / EASE_R leg (hot path iii)")
    ap.add_argument("--ref-workers", type=int, default=64, help="worker processes of the reference arm (capped by the host core count)")
    ap.add_argument("--ref-slice", type=int, default=250)
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"], help="N > 1: how the ranks' rows reach every rank")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the top-K table of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the output of --impl b200; the reference arm times column slices and keeps no output")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
