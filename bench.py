"""Benchmark of the hot path: CV grid fits/sec (alpha x fold), device-timed.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference]
                    [--workload c3|c2|c1|c4|c5] [--dump-outputs DIR]

One "step" = one full cross-validated grid search of the workload (every
(alpha, fold) problem solved to the duality-gap tolerance and scored).

--dump-outputs DIR writes what the last timed step of the device-resident arm returned as DIR/<name>.npy
(float64): the test-score table, the solver info per (alpha, fold) and every alpha's warm-start solution.
The inputs are generated from fixed seeds, so two builds run with the same arguments can be compared
output for output.  bench_outputs/ is the directory git ignores for this.

* value     : fits/sec with X, y already resident in HBM when the timed region starts
              (Gram build + Lipschitz + batched solve + CV scoring, CUDA events, max over ranks)
* e2e       : the same through the public API, sparselm_b200.model_selection.GridSearchCV.fit on
              HOST (pinned) arrays: H2D copy of X, y and D2H of scores/coefficients inside the
              timed region, refit on the full data included
* roofline  : the dominant kernel (FP64 DMMA Gram apply) against the FP64 tensor peak, which
              MEASURED_PEAKS.json does not hold: it is measured here with cuBLAS DGEMM 8192^3
* cpu_baseline / --impl reference : the CPU oracle (oracle/) on the host cores.  Two arms: "gram_path"
              = what a careful CPU implementation of the same search does (per-fold Grams built once with
              BLAS, block coordinate descent in Gram form, every alpha warm-started from the previous
              one, OpenMP over fold x path-segment tasks) on the WHOLE workload -- this is the value of
              `--impl reference`; and "per_fit" = one independent residual-form solve per (alpha, fold)
              cell, one cell per thread, the structural analogue of the reference's joblib fan-out of
              cvxpy solves, on a bounded sample.  The reference's own cvxpy path cannot run in this
              image (cvxpy is not installed); both arms are far faster than it would be.
* tall      : (default workload only) the tall-design config C5 (n=400k, p=8k, X row-sharded, Gram
              all-reduce) as a companion object, 3 steps; `--workload c5` gives it a full line.
"""

from __future__ import annotations

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

TOL = 1e-9  # relative duality gap (SURVEY section 8d: one decade inside the 1e-8 parity spec)


# --------------------------------------------------------------------------- #
# workloads (SURVEY.md section 8d)
# --------------------------------------------------------------------------- #
def make_data(n, p, seed=0, noise=10.0):
    """make_regression-style synthetic data (X ~ N(0,1), p/10 informative coefficients
    100*U(0,1), y = Xw + noise*N(0,1)); generated with numpy for speed."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    w = np.zeros(p)
    idx = rng.choice(p, p // 10, replace=False)
    w[idx] = 100.0 * rng.random(p // 10)
    y = X @ w + noise * rng.standard_normal(n)
    return X, y


def workload(name):
    from sparselm_b200.model import AdaptiveLasso, AdaptiveOverlapGroupLasso, Lasso, SparseGroupLasso

    opts = {"tol": TOL}
    opts.update(json.loads(os.environ.get("BENCH_SOLVER_OPTIONS", "{}")))  # experiments: check_every, ...
    if name == "c3":
        n, p, G, K, F = 20000, 4000, 200, 100, 5
        X, y = make_data(n, p)
        rng = np.random.default_rng(1)
        groups = rng.permutation(np.repeat(np.arange(G), p // G))  # shuffled labels (dataset.py:129-134)
        est = SparseGroupLasso(groups=groups, l1_ratio=0.5, solver_options=opts)
        desc = "SparseGroupLasso, 200 groups, 100 alphas x 5 folds, n=20000 p=4000 (BASELINE configs[2])"
        oracle = dict(name="SparseGroupLasso", groups=groups, l1_ratio=0.5)
    elif name == "c2":
        n, p, K, F = 10000, 2000, 100, 5
        X, y = make_data(n, p)
        est = Lasso(solver_options=opts)
        desc = ("Lasso LineSearchCV, 100 alphas x 5 folds, n=10000 p=2000 (BASELINE configs[1]): n_iter = 2 lines of "
                "the alpha grid + a refit per line")
        oracle = dict(name="Lasso")
        lines = 2
    elif name == "c1":
        from sklearn.datasets import make_regression

        n, p, K, F = 100, 80, 10, 5
        X, y = make_regression(n_samples=100, n_features=80, n_informative=10, random_state=0)
        est = AdaptiveLasso(solver_options={"tol": TOL})
        alphas = np.logspace(-8, 2, 10)
        desc = "AdaptiveLasso GridSearchCV, 10 alphas x 5 folds, make_regression n=100 p=80 (README, configs[0])"
        return dict(X=X, y=y, est=est, alphas=alphas, F=F, desc=desc, name=name,
                    oracle=dict(name="AdaptiveLasso"))
    elif name == "c4":
        n, p, G, K, F = 5000, 1500, 150, 20, 5
        X, y = make_data(n, p)
        rng = np.random.default_rng(2)
        base = rng.permutation(np.repeat(np.arange(G), p // G))
        extra = rng.random(p) < 0.3
        group_list = [[int(base[j])] + ([int((base[j] + 1 + rng.integers(G - 1)) % G)] if extra[j] else [])
                      for j in range(p)]
        est = AdaptiveOverlapGroupLasso(group_list=group_list, solver_options={**opts, "max_iter": 50000})
        desc = "AdaptiveOverlapGroupLasso, 30% overlap, 3 reweight passes, 20 alphas x 5 folds, n=5000 p=1500 (configs[3])"
        oracle = dict(name="AdaptiveOverlapGroupLasso", group_list=group_list)
    elif name == "c5":
        # tall design: X (25.6 GB) is generated on the device of every rank from the same seed
        from sparselm_b200.model import RidgedGroupLasso

        n, p, G, K, F = 400000, 8000, 400, 100, 5
        rng = np.random.default_rng(3)
        groups = rng.permutation(np.repeat(np.arange(G), p // G))
        est = RidgedGroupLasso(groups=groups, delta=(1.0,), solver_options=opts)
        desc = ("RidgedGroupLasso tall design, 400 groups, delta=1, 100 alphas x 5 folds, n=400000 p=8000, "
                "X row-sharded with an NCCL Gram all-reduce (BASELINE configs[4])")
        return dict(X=None, y=None, est=est, alphas=None, F=F, desc=desc, name=name, n=n, p=p, K=K,
                    device_gen=True, oracle=dict(name="RidgedGroupLasso", groups=groups, delta=(1.0,)))
    else:
        raise SystemExit(f"unknown workload {name}")
    alpha_max = np.abs(X.T @ y).max() / n
    alphas = alpha_max * np.logspace(0, -3, K)
    return dict(X=X, y=y, est=est, alphas=alphas, F=F, desc=desc, name=name, oracle=oracle,
                lines=lines if name == "c2" else 1)


# --------------------------------------------------------------------------- #
# clocks
# --------------------------------------------------------------------------- #
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.samples, self.stop_flag = None, [], False

    def start(self):
        # NVML polled every ~10 ms from a thread (a timed region of five 33 ms steps sees ~15 samples; the solver
        # loop runs inside ctypes calls, which release the GIL); nvidia-smi -lms 100 when NVML is not importable
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.handle
        while not self.stop_flag:
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)))
            except Exception:
                break
            time.sleep(0.01)

    def _stop_nvml(self):
        self.stop_flag = True
        self.thread.join(timeout=2)
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        sm = [a for a, _, _ in self.samples]
        reasons = sorted(nm for nm, b in bits.items() if any(r & b for _, _, r in self.samples))
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(m for _, m, _ in self.samples)) if sm else None,
                "samples": len(sm), "source": "nvml", "reasons": reasons}

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            return self._stop_nvml()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- #
# CPU baseline: the oracle on a bounded sample, all host threads
# --------------------------------------------------------------------------- #
def device_data(wl, torch, dev):
    """make_regression-style data generated on the device (same seed on every rank => the
    same matrix): X ~ N(0,1), p/10 informative coefficients 100 U(0,1), noise 10."""
    n, p, K = wl["n"], wl["p"], wl["K"]
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    X = torch.empty((n, p), dtype=torch.float64, device=dev)
    step = 1 << 15
    for r in range(0, n, step):  # row chunks keep the generator's scratch small
        X[r:r + step].normal_(generator=g)
    w = torch.zeros(p, dtype=torch.float64, device=dev)
    idx = torch.randperm(p, generator=g, device=dev)[: p // 10]
    w[idx] = 100.0 * torch.rand(p // 10, generator=g, device=dev, dtype=torch.float64)
    y = X @ w + 10.0 * torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    alpha_max = float((X.T @ y).abs().max().item()) / n
    wl["X"], wl["y"] = X, y.cpu().numpy()
    wl["alphas"] = alpha_max * np.logspace(0, -3, K)
    return wl


def cpu_sample_problem(wl, n_fits):
    """One training fold + n_fits alphas spread over the grid, as inputs of slmo_bcd_many."""
    import oracle.reference as R

    if wl.get("device_gen"):
        return None
    X, y, o = wl["X"], wl["y"], wl["oracle"]
    n, p = X.shape
    te = np.arange(0, n // wl["F"])  # fold 0 of KFold(F)
    tr = np.setdiff1d(np.arange(n), te)
    Xt, yt = X[tr], y[tr]
    name = o["name"]
    if name not in ("Lasso", "SparseGroupLasso"):
        return None
    if name == "Lasso":
        labels, G = np.arange(p), p
        l1r = 1.0
    else:
        labels, G = R.group_labels(o["groups"], p)
        l1r = o["l1_ratio"]
    sel = np.unique(np.linspace(0, len(wl["alphas"]) - 1, n_fits).round().astype(int))
    alphas = wl["alphas"][sel]
    order = np.argsort(labels, kind="stable")
    gptr = np.concatenate([[0], np.cumsum(np.bincount(labels, minlength=G))]).astype(np.int64)
    Xc = np.asfortranarray(Xt[:, order])
    return dict(Xc=Xc, y=np.ascontiguousarray(yt), gptr=gptr, G=G, p=p, n=len(tr), alphas=alphas, l1r=l1r,
                name=name)


def cpu_run(sp):
    import ctypes

    import oracle.reference as R

    lib = R._load()
    K, p, G = len(sp["alphas"]), sp["p"], sp["G"]
    w1 = np.repeat((sp["l1r"] * sp["alphas"])[:, None], p, axis=1).copy()
    w2 = np.repeat(((1 - sp["l1r"]) * sp["alphas"])[:, None], G, axis=1).copy()
    dl = np.zeros((K, G))
    betas = np.zeros((K, p))
    infos = np.zeros((K, 4))
    ns = np.full(K, sp["n"], dtype=np.int64)
    dp = ctypes.POINTER(ctypes.c_double)
    Xs = (dp * K)(*[R._dp(sp["Xc"])] * K)
    ys = (dp * K)(*[R._dp(sp["y"])] * K)
    t0 = time.perf_counter()
    lib.slmo_bcd_many(K, R._ip(ns), p, Xs, ys, G, R._ip(sp["gptr"]), R._dp(w1), R._dp(w2), R._dp(dl),
                      TOL, 1e-14, 100000, 2, R._dp(betas), R._dp(infos))
    dt = time.perf_counter() - t0
    return K / dt, dt, infos


def cpu_gram_path_problem(wl):
    """Inputs of the Gram-form path arm: features in group order, fold edges, penalty tables."""
    import oracle.reference as R

    if wl.get("device_gen") or wl["oracle"]["name"] not in ("Lasso", "SparseGroupLasso"):
        return None
    X, y, o, F = wl["X"], wl["y"], wl["oracle"], wl["F"]
    n, p = X.shape
    if o["name"] == "Lasso":
        labels, G, l1r = np.arange(p), p, 1.0
    else:
        labels, G = R.group_labels(o["groups"], p)
        l1r = o["l1_ratio"]
    order = np.argsort(labels, kind="stable")
    gptr = np.concatenate([[0], np.cumsum(np.bincount(labels, minlength=G))]).astype(np.int64)
    return dict(Xo=np.ascontiguousarray(X[:, order]), y=y, F=F, n=n, p=p, G=G, gptr=gptr, l1r=l1r,
                alphas=np.asarray(wl["alphas"], dtype=float), edges=np.linspace(0, n, F + 1).astype(int))


def cpu_gram_path_run(gp, threads):
    """One whole CV search on the host: fold Grams (BLAS), then fold x path-segment tasks of
    warm-started Gram-form BCD (slmo_gram_path_many).  Returns (fits/s, seconds, infos)."""
    import ctypes

    import oracle.reference as R

    lib = R._load()
    F, n, p, G, alphas, edges = gp["F"], gp["n"], gp["p"], gp["G"], gp["alphas"], gp["edges"]
    t0 = time.perf_counter()
    blocks = []
    for f in range(F):
        Xf, yf = gp["Xo"][edges[f]:edges[f + 1]], gp["y"][edges[f]:edges[f + 1]]
        blocks.append((Xf.T @ Xf, Xf.T @ yf, float(yf @ yf)))
    Gtot, ctot, ytot = sum(b[0] for b in blocks), sum(b[1] for b in blocks), sum(b[2] for b in blocks)
    Gs = [Gtot - b[0] for b in blocks]
    cs = [ctot - b[1] for b in blocks]
    K = len(alphas)
    nseg = max(1, min(K // 8, -(-threads // F)))  # enough tasks for every thread, paths of >= 8 alphas
    segs = np.linspace(0, K, nseg + 1).astype(int)
    tasks = [(f, segs[i], segs[i + 1]) for i in range(nseg) for f in range(F)]
    T = len(tasks)
    koff = np.concatenate([[0], np.cumsum([b - a for _, a, b in tasks])]).astype(np.int64)
    Kt = int(koff[-1])
    w1, w2, dl = np.zeros((Kt, p)), np.zeros((Kt, G)), np.zeros((Kt, G))
    for t, (f, a, b) in enumerate(tasks):
        w1[koff[t]:koff[t + 1]] = (gp["l1r"] * alphas[a:b])[:, None]
        w2[koff[t]:koff[t + 1]] = ((1 - gp["l1r"]) * alphas[a:b])[:, None]
    dp = ctypes.POINTER(ctypes.c_double)
    Gp = (dp * T)(*[R._dp(Gs[f]) for f, _, _ in tasks])
    cp = (dp * T)(*[R._dp(cs[f]) for f, _, _ in tasks])
    yty = np.array([ytot - blocks[f][2] for f, _, _ in tasks])
    ns = np.array([float(n - (edges[f + 1] - edges[f])) for f, _, _ in tasks])
    betas, infos = np.zeros((Kt, p)), np.zeros((Kt, 4))
    lib.slmo_gram_path_many(T, p, Gp, cp, R._dp(yty), R._dp(ns), G, R._ip(gp["gptr"]), R._ip(koff), R._dp(w1),
                            R._dp(w2), R._dp(dl), TOL, 1e-14, 100000, 2, R._dp(betas), R._dp(infos))
    dt = time.perf_counter() - t0
    return Kt / dt, dt, infos


def cpu_baseline(wl, n_fits=None):
    import oracle.reference as R

    R.build()
    threads = R.num_threads()
    n_fits = n_fits or max(4, min(threads, 16))
    sp = cpu_sample_problem(wl, n_fits)
    if sp is None:
        return {"value": None, "unit": "fits/s", "cores": threads, "kind": "port",
                "sample": "not timed for this workload"}
    v, dt, infos = cpu_run(sp)
    per_fit = {"value": v, "unit": "fits/s", "cores": threads,
               "sample": f"{len(sp['alphas'])} of the {len(wl['alphas'])} alphas on training fold 0 "
                         f"(n={sp['n']}, p={sp['p']}), one independent residual-form BCD solve per thread to gap "
                         f"{TOL:g}, {dt:.1f} s, mean sweeps {infos[:, 0].mean():.0f}"}
    gp = cpu_gram_path_problem(wl)
    if gp is None:
        return {**per_fit, "kind": "port", "sample": per_fit["sample"] + "; cvxpy not installed: reference path not timed"}
    v2, dt2, infos2 = cpu_gram_path_run(gp, threads)
    return {"value": v2, "unit": "fits/s", "cores": threads, "kind": "port",
            "sample": f"the whole workload ({len(infos2)} fits): per-fold Grams by BLAS + Gram-form BCD along "
                      f"warm-started alpha paths (OpenMP over fold x segment tasks) to gap {TOL:g}, {dt2:.1f} s, "
                      f"mean sweeps {infos2[:, 0].mean():.1f}, {int((infos2[:, 3] == 1).sum())} unconverged; "
                      f"cvxpy not installed: reference path not timed",
            "per_fit": per_fit}


# --------------------------------------------------------------------------- #
def dist_init(n_gpus):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def _all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0 alone and is
    meant to use every host core it may run on (set before the OpenMP runtime of the oracle loads)."""
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 or "OMP_NUM_THREADS" not in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(ncpu)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _all_host_threads()
    wl = workload(args.workload)
    import oracle.reference as R

    R.build()
    threads = R.num_threads()
    gp = cpu_gram_path_problem(wl)
    sp = None if gp is not None else cpu_sample_problem(wl, max(4, min(threads, 16)))
    if gp is None and sp is None:
        print(json.dumps({"impl": "reference", "unavailable": "CPU oracle arm not wired for this workload"}))
        return
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, _ = cpu_gram_path_run(gp, threads) if gp is not None else cpu_run(sp)
        if i >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    if gp is not None:
        sample = (f"the whole workload per step ({len(wl['alphas'])} alphas x {wl['F']} folds): per-fold Grams by BLAS + "
                  f"Gram-form block coordinate descent along warm-started alpha paths (C, OpenMP over fold x segment "
                  f"tasks) to gap {TOL:g}; cvxpy is not installed so the reference's own solve cannot be timed")
    else:
        sample = (f"{len(sp['alphas'])} of {len(wl['alphas'])} alphas x 1 of {wl['F']} folds per step, oracle BCD "
                  f"(C, OpenMP over fits) to gap {TOL:g}; cvxpy is not installed so the reference's own solve "
                  f"cannot be timed")
    line = {
        "impl": "reference", "metric": "cv_grid_fits_per_sec", "value": value, "unit": "fits/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "tol": TOL},
        "cpu_baseline": {"value": value, "unit": "fits/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def measure_fp64_peak(torch, dev):
    N = 8192
    a = torch.randn(N, N, dtype=torch.float64, device=dev)
    b = torch.randn(N, N, dtype=torch.float64, device=dev)
    best = 1e9
    for i in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2.0 * N ** 3 / best / 1e9  # TFLOP/s


def run_engine(args):
    import torch

    rank, world, local = dist_init(args.gpus)
    from sklearn.base import clone
    from sklearn.model_selection import KFold

    from sparselm_b200.engine import get_engine
    from sparselm_b200.model_selection import GridSearchCV, batched_cv

    wl = workload(args.workload)
    engine = get_engine(local)
    dev = engine.device
    if wl.get("device_gen"):
        wl = device_data(wl, torch, dev)
    X, y, est, alphas, F = wl["X"], wl["y"], wl["est"], wl["alphas"], wl["F"]
    n, p = X.shape
    lines = int(wl.get("lines", 1))  # line searches per step (LineSearchCV: the Grams are built once)
    n_fits = len(alphas) * F * lines
    shard = None
    if world > 1:
        from sparselm_b200.parallel import GridShard

        shard = GridShard(rank, world)

    peak = measure_fp64_peak(torch, dev)

    # ---- device-resident arm ------------------------------------------------------
    Xd = X if isinstance(X, torch.Tensor) else torch.from_numpy(X).to(dev)
    folds = [te for _, te in KFold(F).split(np.empty((n, 1)))]
    # candidates described the way GridSearchCV._batch_plan does it: one working estimator
    # re-parametrised per alpha
    from types import SimpleNamespace

    work = clone(est)
    ests, specs = [], []
    for a in alphas:
        work.set_params(alpha=a)
        specs.append(work._problem_spec(p))
        ests.append(SimpleNamespace(fit_intercept=bool(work.fit_intercept)))
    opts = est._engine_options()

    def step_device(sh=shard):
        if lines == 1:
            return batched_cv(engine, Xd, y, folds, ests, specs, dict(opts), "neg_root_mean_squared_error", shard=sh)
        cache = {}  # what LineSearchCV keeps between its lines: the device-resident design and Grams
        for _ in range(lines):
            out = batched_cv(engine, Xd, y, folds, ests, specs, dict(opts), "neg_root_mean_squared_error", shard=sh,
                             cache=cache, cache_key="bench")
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        res = step_device()
    barrier()
    engine.timing_enable(True)
    engine.timing_reset()
    launches0 = engine.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    times = []
    for _ in range(args.steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = step_device()
        e1.record()
        barrier()
        times.append(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    launches = engine.launch_count() - launches0
    tim = engine.timing_read()
    exec_flops, dense_flops = engine.apply_stats()
    engine.timing_enable(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, len(alphas))
    ms = float(np.mean(times))
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n_fits / (ms / 1e3)

    # ---- weak-scaling companion (N > 1): the grid grows with the GPUs -------------------
    # the named config is a FIXED 100 x 5 grid (strong scaling, the headline `value`); the
    # usual way such a search grows is a second hyper-parameter (sparse-lm's own SGL example
    # sweeps alpha x l1_ratio), so next to it: N l1_ratio values x 100 alphas x 5 folds on N GPUs
    weak = None
    if world > 1 and args.workload == "c3" and not args.no_weak:
        weak = run_weak(args, torch, engine, Xd, y, folds, work, alphas, F, p, opts, shard, barrier, world, dev)

    # ---- sharded search against the un-sharded one (outside every timed region) ----------------
    parity = None
    if world > 1:
        try:
            if rank == 0:
                single = step_device(None)
                a, b = np.asarray(res["test_scores"]), np.asarray(single["test_scores"])
                parity = {"sharded_vs_single_rel_err": float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))),
                          "what": "max relative difference of the (alpha, fold) test-score table between the sharded "
                                  f"search on {world} GPUs and the same search on rank 0 alone"}
        except Exception as exc:  # noqa: BLE001
            parity = {"sharded_vs_single_rel_err": None, "error": f"{type(exc).__name__}: {exc}"[:300]}
        barrier()

    # ---- tall-design companion (BASELINE configs[4]) ---------------------------------------------
    tall = None
    if args.workload == "c3" and not args.no_tall:
        tall = run_tall(args, torch, engine, shard, barrier, world, rank, dev, peak)

    # ---- end-to-end arm: public API on host (pinned) arrays --------------------------
    if wl.get("device_gen"):
        e2e = None  # 25.6 GB design generated on the device: no host copy to start from
    else:
        e2e = run_e2e(args, torch, wl, shard, barrier, world, dev)
    finish(args, wl, res, engine, tim, exec_flops, dense_flops, ms, value, e2e, launches, clocks, peak, world, rank,
           weak, parity, tall)


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, res, n_cand):
    """Write what batched_cv returned to its caller as out_dir/<name>.npy (float64): the test-score table
    [alpha, fold], the solver info tables [alpha, fold] (info_*), the iteration and unconverged counts, and
    each alpha's warm-start solution [alpha, feature] (its solution on the first training fold that solved it,
    in the solver's feature order: the start point of the refit; NaN rows were solved by another rank)."""
    arrays = {"test_scores": res["test_scores"], "iters_run": res["iters_run"], "n_unconverged": res["n_unconverged"]}
    arrays.update({f"info_{k}": v for k, v in res["info"].items()})
    warm = [res["warm"].get(ci) for ci in range(n_cand)]
    pe = next(w.numel() for w in warm if w is not None)
    arrays["warm_start_coef"] = np.stack([np.full(pe, np.nan) if w is None else w.cpu().numpy() for w in warm])
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_tall(args, torch, engine, shard, barrier, world, rank, dev, peak):
    """C5 next to the headline: RidgedGroupLasso, n=400000, p=8000, 100 alphas x 5 folds, rows of the
    Gram build sharded over the ranks (one all-reduce), 3 timed steps.  A failure here must not cost
    the headline line: it is reported inside the object instead."""
    import gc
    from types import SimpleNamespace

    from sklearn.base import clone
    from sklearn.model_selection import KFold

    from sparselm_b200.model_selection import batched_cv

    try:
        wl = device_data(workload("c5"), torch, dev)
        X, y, est, alphas, F = wl["X"], wl["y"], wl["est"], wl["alphas"], wl["F"]
        n, p = X.shape
        work = clone(est)
        ests, specs = [], []
        for a in alphas:
            work.set_params(alpha=a)
            specs.append(work._problem_spec(p))
            ests.append(SimpleNamespace(fit_intercept=bool(work.fit_intercept)))
        opts = est._engine_options()
        folds = [te for _, te in KFold(F).split(np.empty((n, 1)))]

        def step():
            return batched_cv(engine, X, y, folds, ests, specs, dict(opts), "neg_root_mean_squared_error", shard=shard)

        for _ in range(3):
            res = step()
        barrier()
        engine.timing_enable(True)
        engine.timing_reset()
        ts = []
        for _ in range(3):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = step()
            e1.record()
            barrier()
            ts.append(e0.elapsed_time(e1))
        tim = engine.timing_read()
        engine.timing_enable(False)
        ms = float(np.mean(ts))
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        gb = tim["gram_build"]
        build_tf = gb["flops"] / (gb["ms"] * 1e-3) / 1e12 if gb["ms"] > 0 else None
        out = {"workload": wl["desc"], "value": len(alphas) * F / (ms / 1e3), "unit": "fits/s", "ms_per_step": ms,
               "steps": 3, "warmup": 3, "n_gpus": world, "unconverged": int(res["n_unconverged"]),
               "iterations_per_step": int(res["iters_run"]),
               "roofline": {"bound": "tensor", "kernel": "gemm_f64_tma_kernel<SYM> (this rank's share of the Gram build, "
                                                         "FP64 DMMA, SYRK flop count)",
                            "achieved": build_tf, "peak": peak, "unit": "TFLOP/s",
                            "frac": build_tf / peak if build_tf else None,
                            "step_ms_by_kernel_family": {k: v["ms"] / 3 for k, v in tim.items()}}}
        del X, wl, res
        gc.collect()
        torch.cuda.empty_cache()
        return out
    except Exception as exc:  # noqa: BLE001
        return {"value": None, "unit": "fits/s", "error": f"{type(exc).__name__}: {exc}"[:300]}


def run_weak(args, torch, engine, Xd, y, folds, work, alphas, F, p, opts, shard, barrier, world, dev):
    """Weak-scaling companion: `world` l1_ratio lines of the named config on `world` GPUs.  A failure
    here must not cost the headline line: it is reported inside the object instead."""
    from types import SimpleNamespace

    from sparselm_b200.model_selection import batched_cv

    try:
        ratios = np.linspace(0.2, 0.8, world)
        w_ests, w_specs = [], []
        for r in ratios:
            work.set_params(l1_ratio=float(r))
            for a in alphas:
                work.set_params(alpha=a)
                w_specs.append(work._problem_spec(p))
                w_ests.append(SimpleNamespace(fit_intercept=bool(work.fit_intercept)))

        def step_weak():
            return batched_cv(engine, Xd, y, folds, w_ests, w_specs, dict(opts), "neg_root_mean_squared_error",
                              shard=shard)

        for _ in range(2):
            wres = step_weak()
        wt = []
        for _ in range(args.steps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            wres = step_weak()
            e1.record()
            barrier()
            wt.append(e0.elapsed_time(e1))
        wms = float(np.mean(wt))
        import torch.distributed as dist

        t = torch.tensor([wms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wms = float(t.item())
        weak = {"value": len(w_specs) * F / (wms / 1e3), "unit": "fits/s", "ms_per_step": wms,
                "n_fits_per_step": len(w_specs) * F, "unconverged": int(wres["n_unconverged"]),
                "grid": f"{world} l1_ratio values x {len(alphas)} alphas x {F} folds "
                        f"(one l1_ratio line of the named config per GPU)"}
        return weak
    except Exception as exc:  # noqa: BLE001
        return {"value": None, "unit": "fits/s", "error": f"{type(exc).__name__}: {exc}"[:300]}


def run_e2e(args, torch, wl, shard, barrier, world, dev):
    from sklearn.base import clone

    from sparselm_b200.model_selection import GridSearchCV, LineSearchCV

    X, y, est, alphas, F = wl["X"], wl["y"], wl["est"], wl["alphas"], wl["F"]
    n, p = X.shape
    lines = int(wl.get("lines", 1))
    n_fits = len(alphas) * F * lines
    Xp = torch.from_numpy(X).pin_memory()
    Xh = Xp.numpy()
    grid = {"alpha": list(alphas)}

    def step_e2e():
        if lines > 1:  # BASELINE configs[1]: LineSearchCV, n_iter = 2 * n_params lines, a refit per line
            gs = LineSearchCV(clone(est), [("alpha", list(alphas))], cv=F)
        else:
            gs = GridSearchCV(clone(est), grid, cv=F)
        if shard is not None:
            gs._shard = shard
        gs.fit(Xh, y)
        return gs

    for _ in range(max(1, args.warmup // 2)):
        gs = step_e2e()
    e2e_times = []
    for _ in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        gs = step_e2e()
        torch.cuda.synchronize()
        e2e_times.append((time.perf_counter() - t0) * 1e3)
    e2e_ms = float(np.mean(e2e_times))
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    h2d = X.nbytes + y.nbytes
    d2h = 8 * (n_fits * 2 + n_fits + lines * (p + 1))  # residual sums, per-fit info, refit coefficients
    api = "LineSearchCV.fit (2 lines, pinned host X uploaded once, a refit per line)" if lines > 1 else \
        "GridSearchCV.fit (pinned host X, refit included)"
    return {"value": n_fits / (e2e_ms / 1e3), "unit": "fits/s", "ms_per_step": e2e_ms,
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "api": "sparselm_b200.model_selection." + api}


def finish(args, wl, res, engine, tim, exec_flops, dense_flops, ms, value, e2e, launches, clocks, peak, world, rank,
           weak=None, parity=None, tall=None):
    if rank != 0:
        return
    X, alphas, F = wl["X"], wl["alphas"], wl["F"]
    n, p = X.shape
    n_fits = len(alphas) * F * int(wl.get("lines", 1))
    xbytes = n * p * 8
    ap = tim["gram_apply"]
    apply_ms = ap["ms"] / max(ap["launches"], 1)
    # the row-sparse apply contracts only over the support rows of each column chunk:
    # `achieved` counts the flops it really executes for real columns (2 p |S| K_chunk); the
    # dense-equivalent figure 2 p^2 K_active (SURVEY 8d) is reported next to it
    achieved = exec_flops / (ap["ms"] * 1e-3) / 1e12 if ap["ms"] > 0 else None
    dense_equiv = ap["flops"] / (ap["ms"] * 1e-3) / 1e12 if ap["ms"] > 0 else None
    # DRAM bytes per launch of the dominant kernel from an ncu --set full capture of THIS workload on one GPU
    # (profiles/): a constant of that capture, so it is only quoted for the configuration it was taken on
    traffic, traffic_src, traffic_build = None, None, None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if world == 1 and os.path.exists(tpath):
        ent = json.load(open(tpath)).get(args.workload, {})
        traffic, traffic_src = ent.get("gram_apply_dram_bytes_per_launch"), ent.get("source")
        traffic_build = ent.get("gram_build_dram_bytes_per_launch")
    step_ms = {k: v["ms"] / args.steps for k, v in tim.items()}
    info = res["info"]
    gb = tim["gram_build"]
    build_tf = gb["flops"] / (gb["ms"] * 1e-3) / 1e12 if gb["ms"] > 0 else None
    src = "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 figure)"
    roof_build = {"bound": "tensor", "kernel": "gemm_f64_tma_kernel<SYM> (Gram build, TMA-fed FP64 DMMA, SYRK flop count)",
                  "achieved": build_tf, "peak": peak, "unit": "TFLOP/s", "frac": build_tf / peak if build_tf else None,
                  "peak_source": src, "avg_launch_ms": gb["ms"] / max(gb["launches"], 1),
                  "launches_per_step": gb["launches"] / args.steps, "traffic": traffic_build,
                  "traffic_source": None if traffic_build is None else "ncu --set full capture of this workload's build "
                                    "launch on one GPU (profiles/r02z_ncu.md): dram__bytes_read.sum + dram__bytes_write.sum"}
    roof_apply = {"bound": "tensor", "kernel": "gemm_f64_tma_kernel (row-sparse Gram apply, TMA gather4-fed FP64 DMMA)",
                  "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                  "peak_source": src, "dense_equivalent_tflops": dense_equiv,
                  "support_fraction": (exec_flops / dense_flops) if dense_flops > 0 else None,
                  "avg_launch_ms": apply_ms, "launches_per_step": ap["launches"] / args.steps,
                  "traffic": traffic, "traffic_source": traffic_src}
    # the roofline object describes the kernel family with the largest share of the step (tall designs: the Gram
    # build; C3 on one GPU: build and apply are within a few per cent of each other); the other tensor-core
    # family is reported next to it with the same fields
    if gb["ms"] > ap["ms"]:
        roof = dict(roof_build, gram_apply_tflops=achieved, second_kernel=roof_apply)
    else:
        roof = dict(roof_apply, gram_build_tflops=build_tf, second_kernel=roof_build)
    roof["step_ms_by_kernel_family"] = step_ms
    nw = res.get("newton") or {}
    if nw.get("factorizations"):  # second-order phase of the last timed step (csrc/newton_kernels.cuh)
        torch_model = os.environ.get("SLM_NEWTON_TORCH", "0") == "1"
        roof["newton_phase"] = {"ms_per_step": float(nw["ms"]), "factorizations_per_step": int(nw["factorizations"]),
                                "phases_per_step": int(nw["phases"]),
                                "note": ("SLM_NEWTON_TORCH=1: the torch / cuSOLVER model of the phase (A/B run)" if torch_model else
                                         "lock-step Newton steps on the active groups of the slow columns, this repo's kernels: "
                                         "Hessian assembly from the Gram, batched blocked Cholesky with tensor-core trailing "
                                         "updates, blocked triangular solves, device-side line search (slm_newton_step)")}
    line = {
        "metric": "cv_grid_fits_per_sec", "value": value, "unit": "fits/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "tol": TOL, "n_fits_per_step": n_fits,
                   "iterations_per_step": int(res["iters_run"]), "mean_iterations_per_fit": float(info["n_iter"].mean()),
                   "unconverged": int(res["n_unconverged"]),
                   "l2": "inputs larger than L2 between iterations (X %.0f MB, fold Grams %.0f MB vs 126 MB L2)"
                         % (xbytes / 1e6, (F + 1) * (p + 8) ** 2 * 8 / 1e6),
                   "parallelism": f"rows (Gram build) + grid (solve) sharded x{world}" if world > 1 else "single GPU"},
        "roofline": roof,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if weak is not None:
        line["weak_scaling"] = weak
    if parity is not None:
        line["sharded_parity"] = parity
    if tall is not None:
        line["tall"] = tall
    line["tma_launches"] = int(engine.tma_launch_count())
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(wl)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling companion run (N > 1)")
    ap.add_argument("--no-tall", action="store_true", help="skip the tall-design (C5) companion object")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (engine only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs needs --impl engine")
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        try:
            import torch.distributed as dist

            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    main()
