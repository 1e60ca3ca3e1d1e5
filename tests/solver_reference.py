"""Float64 references of the solver kernels (csrc/solver_kernels.cuh, coop_kernels.cuh), shared by
tests/test_gpu_solver_kernels.py and its CPU counterpart tests/test_solver_reference.py.

- `certificate`: what gap_partial_kernel + gap_final_kernel report in final mode (primal, gap, dual norm,
  status) for an arbitrary iterate, from the Gram form of engine_model (bisection dual norm, independent of
  the kernel's Newton iteration).
- `fused_iterates`: m steps of the accelerated proximal-gradient iteration (engine_model.solve_fused without
  convergence checks), recording how close the run came to the switch points of the iteration (restart test,
  soft threshold, group shrink): an iterate comparison is only fair when no decision is within rounding of its
  threshold.
- the problems of both test modules, so that the CPU test checks the margins at exactly the seeds the GPU
  test runs.
"""

from __future__ import annotations

import numpy as np

import engine_model as M

MARGIN = 1e-8  # smallest relative distance from a switch point an iterate comparison accepts


def design(seed, n, p, n_support=None, shift=0.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p)) + shift
    s = n_support or max(4, p // 10)
    w = np.zeros(p)
    w[rng.choice(p, s, replace=False)] = 2.0 * rng.standard_normal(s)
    y = X @ w + 0.5 * rng.standard_normal(n)
    return X, y, rng


def gptr_of(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)


def problem_from_gram(Gf, p, n, gptr, W1, W2, D2, L=None):
    """engine_model.BatchProblem on an engine Gram [pa, pa] (G in [:p, :p], c in row p, y'y at [p, p])."""
    Gf = np.asarray(Gf, dtype=float)
    return M.BatchProblem(Gf[:p, :p], Gf[p, :p].copy(), Gf[p, p], n, gptr, W1, W2, D2, L)


def problem_from_design(X, y, gptr, W1, W2, D2, L=None):
    return M.BatchProblem(X.T @ X, X.T @ y, y @ y, X.shape[0], gptr, W1, W2, D2, L)


def dual_norms(pb, B):
    """Dual norm omega of every column (smooth rows excluded, as in the gap kernels)."""
    g = (pb.c[:, None] - pb.G @ B) / pb.n - pb.D2[pb.gid] * B
    g = np.where(M.smooth_rows(pb), 0.0, g)
    om = np.zeros(pb.K)
    for gi in range(len(pb.gptr) - 1):
        a, b = pb.gptr[gi], pb.gptr[gi + 1]
        om = np.maximum(om, M.group_dual_norm(g[a:b], pb.W1[a:b], pb.W2[gi]))
    return om


def certificate(pb, B, tol, floor_rel=1e-14):
    """Final-mode certificate of every column: primal, gap, omega, status and the scale of the relative test,
    plus `ratio` = gap / (tol * scale) and `dD` = |change of the dual value| per relative error of omega."""
    with np.errstate(invalid="ignore", over="ignore"):
        GB = pb.G @ B
        P, D, gap = M.gap_terms(pb, B, GB)
        om = dual_norms(pb, B)
        scale = np.maximum(np.abs(P), max(floor_rel, 4e-15 / tol) * pb.yty / (2 * pb.n))
        finite = np.isfinite(P) & np.isfinite(gap)
        ok = M.smooth_ok(pb, B, GB)
        status = np.where(~finite, 2, np.where((gap <= tol * scale) & ok, 0, 1))
        # D(s) = (2 s yr - s^2 rr_aug) / 2n with s = 1/omega for omega > 1: dD/d(log omega) = -s (yr - s rr_aug) / n
        ss = np.add.reduceat(B * B, pb.gptr[:-1], axis=0)
        rr_aug = pb.yty - 2 * (pb.c @ B) + (B * GB).sum(0) + pb.n * (pb.D2 * ss).sum(0)
        yr = pb.yty - pb.c @ B
        s = np.where(om > 1, 1 / np.where(om > 1, om, 1), 1.0)
        dD = np.where((om > 1) & np.isfinite(om), np.abs(s * (yr - s * rr_aug)) / pb.n, 0.0)
    return {"primal": P, "gap": gap, "omega": om, "status": status, "scale": scale, "ratio": gap / (tol * scale),
            "dD": dD, "smooth_ok": ok}


def fused_iterates(pb, B0, m):
    """m steps of engine_model.solve_fused from B0 (no convergence checks) and the smallest relative distances
    of the run from its switch points: restart dot / sum |terms| (exact zeros excepted), ||v| - step w1| /
    (step w1) and |‖u_g‖ - step w2| / (step w2)."""
    step = 1.0 / pb.L
    W = B0.copy()
    Wold = W.copy()
    GWold = np.zeros_like(W)
    tm = np.ones(pb.K)
    dot = np.zeros(pb.K)
    mg = {"restart": np.inf, "soft": np.inf, "shrink": np.inf}
    t1 = step * pb.W1
    t2 = step * pb.W2
    for it in range(m):
        GW = pb.G @ W
        if it == 0:
            th, tn = np.zeros(pb.K), tm.copy()
        else:
            tn = (1 + np.sqrt(1 + 4 * tm * tm)) / 2
            th = np.where(dot > 0, 0.0, (tm - 1) / tn)
            tn = np.where(dot > 0, 1.0, tn)
        Z = W + th * (W - Wold)
        GZ = GW + th * (GW - GWold)
        V = Z - step * (GZ - pb.c[:, None]) / pb.n
        if (t1 > 0).any():
            mg["soft"] = min(mg["soft"], float((np.abs(np.abs(V) - t1) / np.where(t1 > 0, t1, 1))[t1 > 0].min()))
        U = M.soft(V, t1)
        nrm = np.sqrt(np.add.reduceat(U * U, pb.gptr[:-1], axis=0))
        if (t2 > 0).any():
            mg["shrink"] = min(mg["shrink"], float((np.abs(nrm - t2) / np.where(t2 > 0, t2, 1))[t2 > 0].min()))
        with np.errstate(divide="ignore", invalid="ignore"):
            sc = np.where(nrm > 0, np.maximum(0.0, 1.0 - t2 / np.where(nrm > 0, nrm, 1)), 0.0)
        Wn = U * (sc / (1.0 + step * pb.D2))[pb.gid]
        terms = (Z - Wn) * (Wn - W)
        dot_new = terms.sum(0)
        size = np.abs(terms).sum(0)
        live = (dot_new != 0) & (size > 0)
        if live.any() and it < m - 1:  # the last step's restart test decides nothing
            mg["restart"] = min(mg["restart"], float((np.abs(dot_new) / np.where(size > 0, size, 1))[live].min()))
        Wold, GWold, W, tm, dot = W, GW, Wn, tn, dot_new
    return W, mg


def assert_margins(mg, what=""):
    for k, v in mg.items():
        assert v >= MARGIN, f"{what}: the reference run came within {v:.2e} of a {k} switch point"


# ---- problems of the m-step iterate tests ----------------------------------------------------------------------
# name -> (p, n, group sizes (None: Lasso), kind, K per fold, m, cold start)
def _sizes(p, top, seed):
    """group sizes 1..top covering p rows, the largest equal to top"""
    rng = np.random.default_rng(seed)
    out = [top]
    while sum(out) < p:
        out.append(int(rng.integers(1, top + 1)))
    out[-1] -= sum(out) - p
    if out[-1] == 0:
        out.pop()
    return out


ITER_CASES = {
    "small_sgl_p100": (100, 160, 6, "sgl", [6], 40, True),
    "small_group_p150": (150, 200, 8, "group", [5], 40, False),
    "small_lasso_p150": (150, 200, None, "lasso", [7], 40, True),
    "lasso_p240": (240, 300, None, "lasso", [9], 30, True),
    "rc2_p240": (240, 300, 8, "sgl", [8], 30, True),
    "rc3_p240": (240, 300, 12, "group", [6], 30, False),
    "rc5_p240": (240, 300, 20, "ridged", [7], 30, True),
    "rc8_p240": (240, 300, 32, "sgl", [5], 30, True),
    "twopass_p240": (240, 300, 45, "group", [6], 30, True),
    "few_lasso_p300": (300, 360, None, "lasso", [3], 40, True),
    "few_sgl_p300": (300, 360, 10, "sgl", [4], 40, False),
    "many_sgl_p400": (400, 300, 10, "sgl", [20], 40, True),
    "folds_sgl_p260": (260, 330, 9, "sgl", [13, 8, 5], 40, True),
}


def iter_case(name):
    """Design, group table and per-fold penalty columns (W1 (p, K), W2 (Gn, K), D2 (Gn, K)) and start points."""
    p, n, top, kind, Ks, m, cold = ITER_CASES[name]
    seed = sum(map(ord, name))
    X, y, rng = design(seed, n, p)
    gptr = np.arange(p + 1, dtype=np.int32) if top is None else gptr_of(_sizes(p, top, seed))
    Gn = len(gptr) - 1
    gw = np.sqrt(np.diff(gptr)).astype(float)
    amax = np.abs(X.T @ y).max() / n
    cols = []
    for f, K in enumerate(Ks):
        alphas = amax * np.geomspace(0.5, 0.03, K) * (1.0 + 0.05 * f)
        W1 = np.zeros((p, K))
        W2 = np.zeros((Gn, K))
        D2 = np.zeros((Gn, K))
        if kind == "lasso":
            W1[:] = alphas
        elif kind == "sgl":
            W1[:] = 0.5 * alphas
            W2[:] = gw[:, None] * (0.3 * alphas)[None, :]
        else:
            W2[:] = gw[:, None] * (0.5 * alphas)[None, :]
            if kind == "ridged":
                D2[:] = 0.2 + rng.random((Gn, 1))
        B0 = np.zeros((p, K))
        if not cold:
            B0 = np.where(rng.random((p, K)) < 0.15, rng.standard_normal((p, K)), 0.0)
        cols.append((W1, W2, D2, B0))
    return X, y, gptr, Ks, m, cols, kind
