"""Batched CV searches over arbitrary splits against sklearn's per-fit loop, and the rate of slm_gram_rows_update.

    python tools/splitter_probe.py [--out FILE] [--loop-cells 24] [--quick]

Workloads (seeded): Lasso with 50 alphas on RepeatedKFold(5, 3) and on ShuffleSplit(10, test_size=0.2,
train_size=0.6), n = 5000, p = 1000; SparseGroupLasso with 30 alphas on LeaveOneOut, n = 300, p = 120 (the
fused small-design kernel).  The batched search is timed end to end (GridSearchCV.fit, search + refit) with
CUDA events after one warm-up fit.  The per-fit loop is what sklearn's GridSearchCV does per (candidate, split)
cell: clone, fit on X[train] (H2D copy, packing, Gram, one-column solve), score X[test]; a subset of
`--loop-cells` cells is timed and the total is extrapolated (reported as such).

slm_gram_rows_update is timed at |idx| in {64, 1024, 16000} rows drawn from n = 256 000 (16 problems per call,
p = 1000: pa = 1008), flops |idx| pa (pa + 1) per problem, next to slm_gram_blocks on the same number of
contiguous rows (16 disjoint ranges, hence n = 16 x 16000) and to the FP64 matrix product of torch (cuBLAS DGEMM,
8192^3) as the DGEMM reference rate.  One JSON line per number.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def _events_ms(torch, fn, reps=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def _workloads(quick):
    from sklearn.model_selection import LeaveOneOut, RepeatedKFold, ShuffleSplit

    from sparselm_b200.model import Lasso, SparseGroupLasso

    out = []
    n, p = (1500, 300) if quick else (5000, 1000)
    rng = np.random.default_rng(0)
    X = rng.standard_normal((n, p))
    y = X[:, :20] @ rng.standard_normal(20) + 0.5 * rng.standard_normal(n)
    amax = np.abs(X.T @ y).max() / n
    alphas = list(amax * np.logspace(-3, -0.3, 50))
    out.append(("lasso_repeated_kfold_5x3", Lasso(), {"alpha": alphas}, RepeatedKFold(n_splits=5, n_repeats=3,
                                                                                       random_state=0), X, y))
    out.append(("lasso_shuffle_split_10", Lasso(), {"alpha": alphas},
                ShuffleSplit(10, test_size=0.2, train_size=0.6, random_state=0), X, y))
    n2, p2 = 300, 120
    X2 = rng.standard_normal((n2, p2))
    y2 = X2[:, :8] @ rng.standard_normal(8) + 0.3 * rng.standard_normal(n2)
    groups = np.repeat(np.arange(30), 4)
    amax2 = np.abs(X2.T @ y2).max() / n2
    out.append(("sgl_leave_one_out", SparseGroupLasso(groups=groups, l1_ratio=0.5),
                {"alpha": list(amax2 * np.logspace(-3, -0.3, 30))}, LeaveOneOut(), X2, y2))
    return out


def probe_searches(torch, loop_cells, quick, emit):
    from sklearn.base import clone
    from sklearn.metrics import get_scorer

    from sparselm_b200.model_selection import GridSearchCV

    scorer = get_scorer("neg_root_mean_squared_error")
    for name, est, grid, cv, X, y in _workloads(quick):
        splits = list(cv.split(X, y))
        cands = [{"alpha": a} for a in grid["alpha"]]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            gs = GridSearchCV(est, grid, cv=cv).fit(X, y)  # warm-up: modules, kernels, allocator
            assert gs.batched_
            ms = _events_ms(torch, lambda: GridSearchCV(est, grid, cv=cv).fit(X, y))
            # the per-fit loop: evenly spaced cells of the (candidate, split) grid
            cells = [(c, s) for s in range(len(splits)) for c in range(len(cands))]
            pick = np.linspace(0, len(cells) - 1, min(loop_cells, len(cells))).astype(int)
            clone(est).set_params(**cands[0]).fit(X[splits[0][0]], y[splits[0][0]])  # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in pick:
                c, s = cells[i]
                tr, te = splits[s]
                e = clone(est).set_params(**cands[c]).fit(X[tr], y[tr])
                scorer(e, X[te], y[te])
            torch.cuda.synchronize()
            loop_s = (time.perf_counter() - t0) / len(pick) * len(cells)
        emit(dict(probe="search", workload=name, n=X.shape[0], p=X.shape[1], n_candidates=len(cands),
                  n_splits=len(splits), batched_ms=round(ms, 2), per_fit_loop_ms=round(1e3 * loop_s, 1),
                  per_fit_loop_extrapolated_from_cells=f"{len(pick)} of {len(cells)}",
                  speedup=round(1e3 * loop_s / ms, 1)))


def probe_rows_update(torch, quick, emit):
    from sparselm_b200.engine import get_engine

    eng = get_engine()
    S = 16
    sizes = (64, 1024, 16000) if not quick else (64, 256, 1000)
    # the contiguous comparison takes S disjoint row ranges of the largest size: the design has that many rows
    n, p = S * sizes[-1], (1000 if not quick else 200)
    rng = np.random.default_rng(1)
    gen = torch.Generator(device=eng.device).manual_seed(1)
    X = torch.randn((n, p), dtype=torch.float64, device=eng.device, generator=gen)
    Xa = eng.pack(X, torch.randn(n, dtype=torch.float64, device=eng.device, generator=gen))
    del X
    pa = Xa.shape[1]
    G = torch.zeros((S, pa, pa), dtype=torch.float64, device=eng.device)
    for m in sizes:
        lists = [np.sort(rng.choice(n, m, replace=False)) for _ in range(S)]
        ptr = np.arange(S + 1, dtype=np.int64) * m
        rows = eng.to_device(np.concatenate(lists).astype(np.int32))
        flops = S * m * pa * (pa + 1)
        reps = max(3, int(2e12 // max(flops, 1)) // 4)
        res = {}
        for tma in (15, 0):
            eng.set_option("tma", tma)
            eng.gram_rows_update(Xa, ptr, rows, G)
            res["tma" if tma else "cp_async"] = _events_ms(torch, lambda: eng.gram_rows_update(Xa, ptr, rows, G), reps)
            res[("tma" if tma else "cp_async") + "_downdate"] = _events_ms(
                torch, lambda: eng.gram_rows_update(Xa, ptr, rows, G, accumulate=True, negate=True), reps)
        eng.set_option("tma", 15)
        rp = np.arange(S + 1, dtype=np.int64) * m  # contiguous rows, same count: the dense Gram build
        assert rp[-1] <= n
        eng.gram_blocks(Xa, rp)
        dense_ms = _events_ms(torch, lambda: eng.gram_blocks(Xa, rp), reps)
        emit(dict(probe="gram_rows_update", rows=m, problems=S, pa=pa, gflop=round(flops / 1e9, 3),
                  **{f"{k}_ms": round(v, 4) for k, v in res.items()},
                  **{f"{k}_tflops": round(flops / v / 1e9, 2) for k, v in res.items()},
                  gram_blocks_contiguous_ms=round(dense_ms, 4), gram_blocks_contiguous_tflops=round(flops / dense_ms / 1e9, 2)))
    k = 8192 if not quick else 2048
    A = torch.randn((k, k), dtype=torch.float64, device=eng.device)
    torch.mm(A, A)
    ms = _events_ms(torch, lambda: torch.mm(A, A), 5)
    emit(dict(probe="dgemm_reference", shape=f"{k}^3", ms=round(ms, 3), tflops=round(2 * k ** 3 / ms / 1e9, 2)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--loop-cells", type=int, default=24, help="cells of the per-fit loop to time per workload")
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("splitter_probe needs a CUDA device: there is nothing to measure without one")
    gpu = _gpu_info()

    def emit(d):
        d = dict(gpu=gpu, **d)
        line = json.dumps(d)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    probe_rows_update(torch, args.quick, emit)
    probe_searches(torch, args.loop_cells, args.quick, emit)


if __name__ == "__main__":
    main()
