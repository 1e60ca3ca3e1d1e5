"""Cost of StabilitySelection on the batched engine, of its count kernel, and of sklearn's equivalent loop.

    python tools/stability_probe.py [--out FILE] [--loop-cells 24] [--quick]

Workloads (seeded, 100 complementary-pair subsamples of half the rows each):
  * Lasso, 50 alphas, n = 5 000, p = 1 000;
  * SparseGroupLasso (100 groups of 10, l1_ratio 0.5), 30 alphas, same shape;
  * GroupLasso (20 groups of 6), 30 alphas, n = 2 000, p = 120: the small-design (fused) kernel.
StabilitySelection.fit is timed end to end with CUDA events, median of three runs after one warm-up.
slm_support_counts is timed alone (20 calls) on a chunk's table shape, [16][p][ldz] with the workload's column
count.  sklearn's loop is clone(est).set_params(**c).fit(X[rows], y[rows]) per (candidate, subsample) cell:
`--loop-cells` evenly spaced cells are timed and the total is extrapolated (reported as such).  One JSON line per
number, each with the card's name, power limit and max SM clock read at start.
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
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
    from sparselm_b200.model import GroupLasso, Lasso, SparseGroupLasso

    out = []
    n, p = (1500, 300) if quick else (5000, 1000)
    rng = np.random.default_rng(0)
    X = rng.standard_normal((n, p))
    y = X[:, :20] @ rng.standard_normal(20) + 0.5 * rng.standard_normal(n)
    amax = np.abs(X.T @ y).max() / n
    out.append(("lasso", Lasso(), {"alpha": list(amax * np.logspace(-3, -0.3, 50))}, X, y))
    groups = np.arange(p) // (p // 100)
    out.append(("sgl_100_groups", SparseGroupLasso(groups=groups, l1_ratio=0.5),
                {"alpha": list(amax * np.logspace(-2.5, -0.3, 30))}, X, y))
    n2, p2 = (600, 120) if quick else (2000, 120)
    X2 = rng.standard_normal((n2, p2))
    y2 = X2[:, :12] @ rng.standard_normal(12) + 0.5 * rng.standard_normal(n2)
    amax2 = np.abs(X2.T @ y2).max() / n2
    out.append(("group_small_p120", GroupLasso(groups=np.arange(p2) // 6),
                {"alpha": list(amax2 * np.logspace(-2.5, -0.3, 30))}, X2, y2))
    return out


def probe(torch, loop_cells, quick, emit):
    from sklearn.base import clone

    from sparselm_b200 import _lib
    from sparselm_b200.engine import get_engine
    from sparselm_b200.stability import StabilitySelection

    eng = get_engine()
    n_sub = 100
    for name, est, grid, X, y in _workloads(quick):
        n, p = X.shape
        make = lambda: StabilitySelection(est, grid, n_subsamples=n_sub, random_state=0)  # noqa: E731
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sel = make().fit(X, y)  # warm-up
            runs = [_events_ms(torch, lambda: make().fit(X, y)) for _ in range(3)]
        K = len(grid["alpha"])
        emit(dict(probe="fit", workload=name, n=n, p=p, n_candidates=K, n_subsamples=n_sub, cells=K * n_sub,
                  fit_ms=round(float(np.median(runs)), 2), runs_ms=[round(t, 2) for t in runs],
                  selected_size=sel.selected_size_, n_scores_ge_threshold=int(sel.get_support().sum()),
                  max_iterations=int(sel.solver_info_["n_iter"].max())))
        # the count kernel alone on one chunk's table: [SLM_MAX_FOLDS][p][ldz]
        F = _lib.SLM_MAX_FOLDS
        ldz = max(8, (K + 7) // 8 * 8)
        tab = np.random.default_rng(1).standard_normal((F, p, ldz))
        tab[np.random.default_rng(2).random(tab.shape) < 0.7] = 0.0
        coef = eng.to_device(tab)
        counts = torch.zeros((p, K), dtype=torch.int32, device=eng.device)
        union = torch.zeros((F, p), dtype=torch.uint8, device=eng.device)
        eng.support_counts(coef, K, 1e-6, counts, union)
        ms = _events_ms(torch, lambda: eng.support_counts(coef, K, 1e-6, counts, union), 20)
        nbytes = 2 * F * p * K * 8  # two passes over the candidate columns of the table
        emit(dict(probe="support_counts", workload=name, F=F, p=p, ldz=ldz, K=K, ms=round(ms, 4),
                  bytes_read=nbytes, gbytes_per_s=round(nbytes / ms / 1e6, 1),
                  chunks_per_fit=-(-n_sub // F), share_of_fit=round(ms * -(-n_sub // F) / float(np.median(runs)), 4)))
        del coef
        # sklearn's loop of engine fits, evenly spaced cells, extrapolated
        cands = [{"alpha": a} for a in grid["alpha"]]
        cells = [(c, s) for s in range(n_sub) for c in range(K)]
        pick = np.linspace(0, len(cells) - 1, min(loop_cells, len(cells))).astype(int)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            rows0 = sel.subsamples_[0]
            clone(est).set_params(**cands[0]).fit(X[rows0], y[rows0])  # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in pick:
                c, s = cells[i]
                rows = sel.subsamples_[s]
                clone(est).set_params(**cands[c]).fit(X[rows], y[rows])
            torch.cuda.synchronize()
        loop_s = (time.perf_counter() - t0) / len(pick) * len(cells)
        emit(dict(probe="per_fit_loop", workload=name, cells=len(cells), per_fit_loop_ms=round(1e3 * loop_s, 1),
                  extrapolated_from_cells=f"{len(pick)} of {len(cells)}",
                  speedup_vs_batched=round(1e3 * loop_s / float(np.median(runs)), 1)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--loop-cells", type=int, default=24, help="cells of sklearn's loop to time per workload")
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("stability_probe needs a CUDA device: there is nothing to measure without one")
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
