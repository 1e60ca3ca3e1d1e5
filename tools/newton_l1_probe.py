"""The l1 Newton phase (solver_options={"newton": "l1"}) against the first-order iterations alone, on an AR(1)
rho = 0.99 design (n = 5000, p = 1000, 30 true coefficients): a single AdaptiveLasso fit, and GridSearchCV over
20 alphas x 5 folds for Lasso and for SparseGroupLasso (l1_ratio 0.5, 100 groups of 10).

One JSON line per configuration and mode: ms per fit or search (CUDA events around the call, after one warm-up
call of the same mode; median of --reps timed calls, the modes alternating), total iterations, unconverged
columns, the Newton phase's stats (phases, factorisations, columns, ms inside the phase), and the largest
coefficient / score difference against the plain mode.  For a search the stats of the search itself (every
candidate x fold column) and of the refit of the best candidate are reported separately; the time covers both.
Modes: first-order only (newton False), "l1", and "l1" with Engine.NEWTON_L1_SHRINK_IS_PROGRESS off ("l1_strict":
every unfinished phase counts towards the three after which a column stays first-order).
Last, one l1 Newton step of Lasso columns (slm_newton_step_l1) at p = 1000 with Lasso's single zero-weight group
against the same step with p singleton zero-weight groups (identical arithmetic on the group terms).
The GPU's name and power limit lead.
Usage: python tools/newton_l1_probe.py [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import sparselm_b200.model._base as _base  # noqa: E402
import sparselm_b200.model_selection as _ms  # noqa: E402
from sparselm_b200.model import AdaptiveLasso, Lasso, SparseGroupLasso  # noqa: E402
from sparselm_b200.model_selection import GridSearchCV  # noqa: E402


def ar1(seed, n=5000, p=1000, rho=0.99, n_true=30):
    rng = np.random.default_rng(seed)
    X = np.empty((n, p))
    X[:, 0] = rng.standard_normal(n)
    for j in range(1, p):
        X[:, j] = rho * X[:, j - 1] + np.sqrt(1 - rho * rho) * rng.standard_normal(n)
    b = np.zeros(p)
    b[rng.choice(p, n_true, replace=False)] = rng.standard_normal(n_true) * 3.0
    return X, X @ b + rng.standard_normal(n) + 2.0


# the Newton stats of the last call: the estimators and the search keep only the solver's per-column info.
# A plain fit (and the refit of a search) goes through model._base.solve_specs; the search's own batches through
# model_selection.batched_cv (which calls its own import of solve_specs, not the wrapper below)
_last = {}
_solve_specs, _batched_cv = _base.solve_specs, _ms.batched_cv


def _capture_fit(*a, **k):
    out = _solve_specs(*a, **k)
    _last["fit"] = dict(iterations=int(out["n_iter"][0, 0]), unconverged=int(out["n_unconverged"]),
                        newton_stats=out.get("newton") or None)
    return out


def _capture_cv(*a, **k):
    out = _batched_cv(*a, **k)
    _last["search"] = dict(iterations=int(out["info"]["n_iter"].sum()), unconverged=int(out["n_unconverged"]),
                           newton_stats=out.get("newton") or None)
    return out


_base.solve_specs, _ms.batched_cv = _capture_fit, _capture_cv


def configs():
    X, y = ar1(0)
    amax = np.abs((X - X.mean(0)).T @ (y - y.mean())).max() / len(y)
    alphas = list(amax * np.geomspace(0.5, 1e-3, 20))
    groups = np.repeat(np.arange(100), 10)
    yield "adaptive_lasso_fit", X, y, lambda nw: AdaptiveLasso(alpha=1e-2 * amax, fit_intercept=True, solver_options=nw)
    yield "lasso_cv_20x5", X, y, lambda nw: GridSearchCV(Lasso(fit_intercept=True, solver_options=nw), {"alpha": alphas}, cv=5)
    yield "sgl_cv_20x5", X, y, lambda nw: GridSearchCV(SparseGroupLasso(groups=groups, l1_ratio=0.5, fit_intercept=True,
                                                                        solver_options=nw), {"alpha": alphas}, cv=5)


def run(make, X, y, mode):
    from sparselm_b200.engine import Engine

    Engine.NEWTON_L1_SHRINK_IS_PROGRESS = mode != "l1_strict"
    est = make({"tol": 1e-10, "max_iter": 200000, "newton": "l1" if mode == "l1_strict" else mode})
    _last.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        e0.record()
        est.fit(X, y)
        e1.record()
    e1.synchronize()
    Engine.NEWTON_L1_SHRINK_IS_PROGRESS = True
    return est, e0.elapsed_time(e1), dict(_last)


def answer(est):
    if isinstance(est, GridSearchCV):
        scores = np.concatenate([est.cv_results_[f"split{f}_test_score"] for f in range(5)])
        return est.best_estimator_.coef_, scores
    return est.coef_, np.array([est.intercept_])


def step_timing(m, k=16, p=1000, calls=30):
    """ms per slm_newton_step_l1 call on k Lasso columns with m non-zero coordinates each: one zero-weight group of
    all p coordinates (what the engine passes for Lasso) against p singleton zero-weight groups."""
    import ctypes

    from sparselm_b200.engine import get_engine

    eng = get_engine(None)
    dev = eng.device
    X, y = ar1(0)
    n = X.shape[0]
    pa = eng.padded_cols(p)
    Xa = torch.zeros((n, pa), dtype=torch.float64, device=dev)
    Xa[:, :p] = torch.from_numpy(X).to(dev)
    Xa[:, p] = torch.from_numpy(y).to(dev)
    G = (Xa.T @ Xa).contiguous()[None]
    rng = np.random.default_rng(1)
    ldv = (p + 7) // 8 * 8
    X0 = np.zeros((k, ldv))
    for c in range(k):
        X0[c, rng.choice(p, m, replace=False)] = rng.standard_normal(m)
    X0 = torch.from_numpy(X0).to(dev)
    W1 = torch.full((k, ldv), 0.01, dtype=torch.float64, device=dev)
    nobs = torch.full((k,), float(n), dtype=torch.float64, device=dev)
    fh = np.zeros(k, dtype=np.int32)
    out = torch.zeros((k, 4), dtype=torch.float64, device=dev)
    res = {}
    for name, gptr in (("one_group", np.array([0, p])), ("singletons", np.arange(p + 1))):
        Gn = len(gptr) - 1
        gptr_d = torch.from_numpy(gptr.astype(np.int32)).to(dev)
        gid_d = torch.from_numpy(np.repeat(np.arange(Gn), np.diff(gptr)).astype(np.int32)).to(dev)
        W2 = torch.zeros((k, Gn), dtype=torch.float64, device=dev)
        nbytes = eng.lib.slm_newton_workspace(p, Gn, k, 1)
        work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        Xw = X0.clone()

        def call():
            Xw.copy_(X0)
            eng._ck(eng.lib.slm_newton_step_l1(
                eng.h, eng._ptr(G), pa * pa, pa, p, 1, k, fh.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                eng._ptr(nobs), eng._ptr(Xw), eng._ptr(W2), None, eng._ptr(W1), eng._ptr(gptr_d), eng._ptr(gid_d), Gn,
                eng._ptr(work), nbytes, eng._ptr(out), eng.stream), "slm_newton_step_l1")

        for _ in range(3):
            call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            call()
        e1.record()
        e1.synchronize()
        res[name] = (e0.elapsed_time(e1) / calls, Xw.cpu().numpy(), out.cpu().numpy())
    same = float(np.abs(res["one_group"][1] - res["singletons"][1]).max())
    return dict(config="lasso_l1_step", p=p, k=k, m=m, calls=calls, ms_one_group=res["one_group"][0],
                ms_singletons=res["singletons"][0], max_x_diff=same,
                accepted=int(res["one_group"][2][:, 0].sum()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("newton_l1_probe: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [json.dumps({"gpu": smi[0] if smi else torch.cuda.get_device_name()})]
    print(lines[-1], flush=True)
    for name, X, y, make in configs():
        modes = (False, "l1", "l1_strict")
        for nw in modes:
            run(make, X, y, nw)  # warm-up: compile-free, but loads modules and fills the allocator's pool
        ms = {nw: [] for nw in modes}
        res = {}
        for _ in range(args.reps):
            for nw in modes:
                est, t, st = run(make, X, y, nw)
                ms[nw].append(t)
                res[nw] = (est, st)
        c0, s0 = answer(res[False][0])
        for nw in modes:
            est, st = res[nw]
            c, s = answer(est)
            row = dict(config=name, newton=nw, ms=float(np.median(ms[nw])), ms_all=[round(v, 2) for v in ms[nw]])
            if "search" in st:
                row.update(search=st["search"], refit=st["fit"])
            else:
                row.update(st["fit"])
            row.update(max_coef_diff=float(np.abs(c - c0).max()), coef_scale=float(np.abs(c0).max()),
                       max_score_diff=float(np.abs(s - s0).max()), score_scale=float(np.abs(s0).max()))
            lines.append(json.dumps(row))
            print(lines[-1], flush=True)
    for m in (50, 300):
        lines.append(json.dumps(step_timing(m)))
        print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
