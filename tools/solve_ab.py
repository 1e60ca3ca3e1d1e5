"""Record every batched solve of a fixed set of workloads that covers each iteration mode of slm_solve_batch:
the fused and the two-kernel per-iteration kernels, the small-design kernel, the cooperative and cluster kernels,
adaptive passes and both Newton phases.  Two builds of the package are compared run by run: the results must be
bitwise equal and the kernel sequences identical.

usage: python tools/solve_ab.py record --root DIR --out FILE.npz   (DIR holds the sparselm_b200 package to load)
       python tools/solve_ab.py compare A.npz B.npz [--json OUT]

record keeps, per Engine.solve call, B, gap, n_iter, status, iters_run and the slm_launch_count delta, and per case
the ordered names of the device activities (torch.profiler; the run is not a timing run)."""

from __future__ import annotations

import argparse
import json
import sys

import numpy as np


def _problem(n, p, n_groups, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    w = np.zeros(p)
    k = max(4, p // 12)
    w[rng.choice(p, k, replace=False)] = 2 * rng.standard_normal(k)
    y = X @ w + 0.3 * rng.standard_normal(n)
    groups = rng.integers(0, n_groups, size=p)
    groups[:n_groups] = np.arange(n_groups)
    return X, y, groups


def _ar1_problem(n, p, rho, seed):
    """strongly correlated columns: slow for the first-order iterations, so the Newton phases run"""
    rng = np.random.default_rng(seed)
    X = np.empty((n, p))
    X[:, 0] = rng.standard_normal(n)
    for j in range(1, p):
        X[:, j] = rho * X[:, j - 1] + np.sqrt(1 - rho * rho) * rng.standard_normal(n)
    b = np.zeros(p)
    b[rng.choice(p, 30, replace=False)] = 3.0 * rng.standard_normal(30)
    return X, X @ b + rng.standard_normal(n)


def _alphas(X, y, hi, lo, k):
    return list(np.abs(X.T @ y).max() / X.shape[0] * np.logspace(hi, lo, k))


def cases():
    from sparselm_b200.engine import get_engine
    from sparselm_b200.model import AdaptiveLasso, AdaptiveSparseGroupLasso, GroupLasso, Lasso, SparseGroupLasso
    from sparselm_b200.model_selection import GridSearchCV

    eng = get_engine()
    X1, y1, g1 = _problem(2500, 1000, 100, 1)
    a1 = _alphas(X1, y1, -0.3, -2.3, 10)
    opts = {"tol": 1e-10}

    def grid(est, X, y, alphas, cv=5):
        return lambda: GridSearchCV(est, {"alpha": alphas}, cv=cv).fit(X, y)

    def two_kernel(fn):
        def run():
            eng.set_option("fused_prox", 0)
            try:
                fn()
            finally:
                eng.set_option("fused_prox", 1)
        return run

    X2, y2, g2 = _problem(600, 120, 12, 2)
    X3, y3, g3 = _problem(300, 420, 30, 21)  # the cluster case of tests/test_gpu_coop.py
    X4, y4, g4 = _problem(800, 500, 50, 4)
    X5, y5 = _ar1_problem(1200, 300, 0.99, 1)
    a5 = list(np.abs(X5.T @ y5).max() / len(y5) * np.array([0.5, 0.1, 0.01, 3e-3, 1e-3]))
    newton_opts = {"tol": 1e-10, "max_iter": 200000}
    return [
        ("fused_lasso", grid(Lasso(solver_options=opts), X1, y1, a1)),
        ("fused_sgl", grid(SparseGroupLasso(groups=g1, l1_ratio=0.5, solver_options=opts), X1, y1, a1)),
        ("two_kernel_lasso", two_kernel(grid(Lasso(solver_options=opts), X1, y1, a1))),
        ("two_kernel_sgl", two_kernel(grid(SparseGroupLasso(groups=g1, l1_ratio=0.5, solver_options=opts), X1, y1, a1))),
        ("small", grid(SparseGroupLasso(groups=g2, l1_ratio=0.5, solver_options=opts), X2, y2, _alphas(X2, y2, -0.3, -2, 8))),
        ("coop_lasso", lambda: Lasso(alpha=a1[5], solver_options=opts).fit(X1, y1)),
        ("coop_sgl", lambda: SparseGroupLasso(groups=g1, alpha=a1[5], solver_options=opts).fit(X1, y1)),
        ("cluster_sgl", grid(SparseGroupLasso(groups=g3, solver_options={"tol": 1e-11}), X3, y3,
                             _alphas(X3, y3, -0.3, -2.2, 7), cv=3)),
        ("cluster_lasso", grid(Lasso(solver_options={"tol": 1e-11}), X3, y3, _alphas(X3, y3, -0.3, -2.2, 7), cv=3)),
        ("adaptive_lasso", grid(AdaptiveLasso(solver_options=opts), X4, y4, _alphas(X4, y4, -0.5, -2, 6))),
        ("adaptive_sgl", grid(AdaptiveSparseGroupLasso(groups=g4, solver_options=opts), X4, y4, _alphas(X4, y4, -0.5, -2, 6))),
        ("newton_group", grid(GroupLasso(groups=np.repeat(np.arange(100), 3), solver_options=newton_opts), X5, y5, a5)),
        ("newton_l1", grid(Lasso(solver_options={**newton_opts, "newton": "l1"}), X5, y5, a5)),
    ]


def record(root, out):
    sys.path.insert(0, root)
    import torch
    from torch.profiler import ProfilerActivity, profile

    import sparselm_b200
    from sparselm_b200.engine import Engine

    print("package:", sparselm_b200.__file__, flush=True)
    solves = []
    orig = Engine.solve

    def solve(self, *a, **k):
        l0 = self.launch_count()
        res = orig(self, *a, **k)
        torch.cuda.synchronize()
        solves.append({"B": res["B"].cpu().numpy(), "gap": res["gap"].copy(), "n_iter": res["n_iter"].copy(),
                       "status": res["status"].copy(), "iters_run": res["iters_run"],
                       "launches": self.launch_count() - l0,
                       "newton_phases": int((res.get("newton") or {}).get("phases", 0))})
        return res

    Engine.solve = solve
    arrays, meta = {}, {}
    for name, fn in cases():
        n0 = len(solves)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        acts = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
        seq = [e.name for e in acts]
        meta[name] = {"n_solves": len(solves) - n0, "device_activities": seq,
                      "iters_run": [s["iters_run"] for s in solves[n0:]],
                      "launches": [s["launches"] for s in solves[n0:]],
                      "newton_phases": [s["newton_phases"] for s in solves[n0:]]}
        for i, s in enumerate(solves[n0:]):
            for key in ("B", "gap", "n_iter", "status"):
                arrays[f"{name}/{i}/{key}"] = s[key]
        print(f"{name}: {len(solves) - n0} solves, {len(seq)} device activities, iters_run {meta[name]['iters_run']}, "
              f"Newton phases {meta[name]['newton_phases']}", flush=True)
    np.savez(out, meta=np.array(json.dumps(meta)), **arrays)


def compare(a_path, b_path, out_json):
    A, B = np.load(a_path), np.load(b_path)
    ma, mb = json.loads(str(A["meta"])), json.loads(str(B["meta"]))
    ok = sorted(A.files) == sorted(B.files) and list(ma) == list(mb)
    rows = {}
    for name in ma:
        keys = [k for k in A.files if k.startswith(name + "/")]
        arrays_equal = all(k in B.files and A[k].dtype == B[k].dtype and A[k].shape == B[k].shape
                           and A[k].tobytes() == B[k].tobytes() for k in keys)
        seq_equal = ma[name]["device_activities"] == mb.get(name, {}).get("device_activities")
        same = {f: ma[name][f] == mb.get(name, {}).get(f) for f in ("n_solves", "iters_run", "launches", "newton_phases")}
        rows[name] = {"solves": ma[name]["n_solves"], "arrays_compared": len(keys), "arrays_bitwise_equal": arrays_equal,
                      "device_activities": len(ma[name]["device_activities"]),
                      "device_activity_sequence_equal": seq_equal, **{f + "_equal": v for f, v in same.items()},
                      "iters_run": ma[name]["iters_run"], "launches": ma[name]["launches"],
                      "newton_phases": ma[name]["newton_phases"]}
        ok = ok and arrays_equal and seq_equal and all(same.values())
    res = {"identical": ok, "cases": rows}
    text = json.dumps(res, indent=1)
    print(text)
    if out_json:
        with open(out_json, "w") as f:
            f.write(text + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    r = sub.add_parser("record")
    r.add_argument("--root", required=True)
    r.add_argument("--out", required=True)
    c = sub.add_parser("compare")
    c.add_argument("a")
    c.add_argument("b")
    c.add_argument("--json")
    args = ap.parse_args()
    if args.cmd == "record":
        record(args.root, args.out)
    else:
        sys.exit(compare(args.a, args.b, args.json))
