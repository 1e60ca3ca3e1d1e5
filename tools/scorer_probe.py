"""Cost of the residual-statistics scorers in batched CV searches, against r2 and against sklearn's per-fit loop.

    python tools/scorer_probe.py [--out FILE] [--loop-cells 24] [--quick]

Workloads (seeded): bench.py's C2 design searched with GridSearchCV (Lasso, 100 alphas x KFold(5), n = 10 000,
p = 2 000) and the RepeatedKFold(5, 3) Lasso search of tools/splitter_probe.py (50 alphas, n = 5 000, p = 1 000).
For each workload GridSearchCV.fit (search + refit) runs with scoring="r2" and with each statistics scorer, the
scorers alternating, and the median of three CUDA-event timings after one warm-up is reported.  The statistics
kernels are timed on their own on the workload's test folds with the search's column count: slm_cv_score_stats
with every statistic, and with the median only, against slm_cv_score_many on the same problems (the difference is
the statistics kernels' time).  The per-fit loop is what sklearn's GridSearchCV does per (candidate, split) cell
with the median scorer: clone, fit on X[train], score X[test]; `--loop-cells` cells are timed and the total is
extrapolated (reported as such).  One JSON line per number.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from splitter_probe import _events_ms, _gpu_info  # noqa: E402

SCORERS = ["r2", "neg_median_absolute_error", "neg_max_error", "neg_mean_absolute_percentage_error",
           "d2_absolute_error_score"]


def _workloads(quick):
    from sklearn.model_selection import KFold

    import bench
    import splitter_probe

    if quick:
        rng = np.random.default_rng(0)
        X = rng.standard_normal((2000, 400))
        y = X[:, :20] @ rng.standard_normal(20) + 0.5 * rng.standard_normal(2000)
        from sparselm_b200.model import Lasso

        alphas = np.abs(X.T @ y).max() / 2000 * np.logspace(0, -3, 20)
        c2 = ("c2_lasso_kfold5", Lasso(solver_options={"tol": bench.TOL}), {"alpha": list(alphas)}, KFold(5), X, y)
    else:
        w = bench.workload("c2")
        c2 = ("c2_lasso_kfold5", w["est"], {"alpha": list(w["alphas"])}, KFold(w["F"]), w["X"], w["y"])
    return [c2, splitter_probe._workloads(quick)[0]]


def probe(torch, loop_cells, quick, emit):
    from sklearn.base import clone
    from sklearn.metrics import get_scorer

    from sparselm_b200 import _lib
    from sparselm_b200.engine import get_engine
    from sparselm_b200.model_selection import GridSearchCV

    eng = get_engine()
    for name, est, grid, cv, X, y in _workloads(quick):
        splits = list(cv.split(X, y))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for sc in SCORERS:  # warm-up of every path
                assert GridSearchCV(est, grid, cv=cv, scoring=sc).fit(X, y).batched_
            times = {sc: [] for sc in SCORERS}
            for _ in range(3):
                for sc in SCORERS:
                    times[sc].append(_events_ms(torch, lambda: GridSearchCV(est, grid, cv=cv, scoring=sc).fit(X, y)))
        med = {sc: float(np.median(v)) for sc, v in times.items()}
        for sc in SCORERS:
            emit(dict(probe="search", workload=name, n=X.shape[0], p=X.shape[1], n_candidates=len(grid["alpha"]),
                      n_splits=len(splits), scoring=sc, search_ms=round(med[sc], 2),
                      runs_ms=[round(t, 2) for t in times[sc]], vs_r2=round(med[sc] / med["r2"], 3)))
        # the statistics kernels on the test rows of the first min(16, splits) splits, the search's column count
        K = len(grid["alpha"])
        p = X.shape[1]
        Xa = eng.pack(X, y)
        B = eng.to_device(np.random.default_rng(1).standard_normal((p, K)) * 1e-2)
        items = [(eng.to_device(np.sort(te).astype(np.int32)), B, K, None) for _, te in splits[:16]]
        res = {}
        for label, fn in (("sums_only", lambda: eng.cv_score_rows(Xa, p, items)),
                          ("all_statistics", lambda: eng.cv_score_stats(
                              Xa, p, items, stats=_lib.SLM_STAT_MAX | _lib.SLM_STAT_MAPE | _lib.SLM_STAT_MEDIAN)),
                          ("median_only", lambda: eng.cv_score_stats(Xa, p, items, stats=_lib.SLM_STAT_MEDIAN))):
            fn()
            res[label] = _events_ms(torch, fn, 20)
        emit(dict(probe="statistics_kernels", workload=name, problems=len(items), rows_per_problem=len(splits[0][1]),
                  columns=K, **{f"{k}_ms": round(v, 4) for k, v in res.items()},
                  statistics_ms=round(res["all_statistics"] - res["sums_only"], 4),
                  median_ms=round(res["median_only"] - res["sums_only"], 4)))
        del Xa
        # sklearn's per-fit loop with the median scorer, evenly spaced cells, extrapolated
        scorer = get_scorer("neg_median_absolute_error")
        cands = [{"alpha": a} for a in grid["alpha"]]
        cells = [(c, s) for s in range(len(splits)) for c in range(len(cands))]
        pick = np.linspace(0, len(cells) - 1, min(loop_cells, len(cells))).astype(int)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
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
        emit(dict(probe="per_fit_loop", workload=name, scoring="neg_median_absolute_error", cells=len(cells),
                  per_fit_loop_ms=round(1e3 * loop_s, 1), extrapolated_from_cells=f"{len(pick)} of {len(cells)}",
                  speedup_vs_batched=round(1e3 * loop_s / med["neg_median_absolute_error"], 1)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--loop-cells", type=int, default=24, help="cells of the per-fit loop to time per workload")
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("scorer_probe needs a CUDA device: there is nothing to measure without one")
    gpu = _gpu_info()

    def emit(d):
        line = json.dumps(dict(gpu=gpu, **d))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    probe(torch, args.loop_cells, args.quick, emit)


if __name__ == "__main__":
    main()
